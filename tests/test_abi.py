"""CPU checks of the drop-in boundary: the C-ABI library builds, loads, and exports every symbol the header declares."""
import ctypes
import os
import re

import danbo_b200
from danbo_b200 import _lib, build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    text = open(os.path.join(ROOT, "include", "danbo_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\bint\s+(danbo_\w+)\s*\(", text)))


def test_header_and_library_agree():
    build.build()
    lib = ctypes.CDLL(_lib.path())
    syms = header_symbols()
    assert len(syms) >= 10
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/danbo_b200.h but not exported"
    assert sorted(_lib.EXPORTS) == syms, "ctypes signatures must cover exactly the header's entry points"
    assert lib.danbo_version() == _lib.ABI_VERSION


def test_kernels_refuse_cpu_tensors():
    import pytest
    import torch
    with pytest.raises(RuntimeError):
        danbo_b200.kernels.nearfar(torch.zeros(4, 8), torch.zeros(1, 5), torch.zeros(1, 24, 4, 4), 4,
                                   torch.zeros(24, 4, 4), torch.ones(24, 3))


def test_unsupported_flags_raise():
    import pytest
    for kw in ({"agg_type": "relu"}, {"agg_type": "sum"}, {"gnn_backbone": "PNBGNN"}, {"netwidth": 128},
               {"nerf_type": "nerf"}, {"single_net": False}):
        with pytest.raises(NotImplementedError):
            danbo_b200.raycaster.check_args(danbo_b200.make_args("danbo_base", **kw))
    # both aggregation types of danbo.py:431-435 that a config can reach pass the check; softmax needs mask_vol_prob
    for agg in ("sigmoid", "softmax"):
        danbo_b200.raycaster.check_args(danbo_b200.make_args("danbo_base", agg_type=agg, lindisp=True))
    from danbo_b200.networks import DanboField
    with pytest.raises(NotImplementedError):
        DanboField(agg_type="softmax", mask_vol_prob=False)


def test_anerf_flag_subset():
    """nerf_type='nerf' (A-NeRF, BASELINE config #4): the preset passes the flag check, anything outside the shipped
    anerf_base.txt subset raises (no silent fallback)."""
    import pytest
    import danbo_b200 as db
    from danbo_b200 import anerf
    args = db.make_args("anerf_base", no_reload=True)
    anerf.check_anerf_args(args)
    for k, v in (("netwidth", 256), ("multires", 10), ("cutoff_viewdir", False), ("view_type", "world"),
                 ("bone_type", "axisang"), ("cutoff_mm", 400.0)):
        bad = db.make_args("anerf_base", no_reload=True, **{k: v})
        with pytest.raises(NotImplementedError):
            anerf.check_anerf_args(bad)
    # parameter inventory = the reference's state_dict (probe in oracle/gen_golden.py), minus the embedder constants
    from danbo_b200 import params
    shapes = params.anerf_param_shapes()
    assert shapes["pts_linears.0.weight"] == (448, 432) and shapes["pts_linears.5.weight"] == (448, 880)
    assert shapes["views_linears.0.weight"] == (224, 1224) and shapes["rgb_linear.weight"] == (3, 224)
    net = anerf.AnerfField()
    sd = net.state_dict()
    assert set(shapes) <= set(sd) and {"pe_fn.cutoff_dist", "pe_fn.tau", "dirs_pe_fn.cutoff_dist", "dirs_pe_fn.tau"} <= set(sd)
    for k, shp in shapes.items():
        assert tuple(sd[k].shape) == tuple(shp), k


def header_declarations():
    """name -> list of parameter strings, parsed from include/danbo_b200.h."""
    text = open(os.path.join(ROOT, "include", "danbo_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    out = {}
    for m in re.finditer(r"\bint\s+(danbo_\w+)\s*\(([^;]*?)\)\s*;", text, flags=re.S):
        params = [p.strip() for p in m.group(2).replace("\n", " ").split(",")]
        out[m.group(1)] = [] if params in ([""], ["void"]) else params
    return out


def test_ctypes_signatures_match_header_parameters():
    """Every ctypes signature has the header's parameter count, and pointer / int / float kinds line up (an argument
    added on one side only would shift every later argument of a call)."""
    decls = header_declarations()
    assert set(decls) == set(_lib.EXPORTS)
    kinds = {ctypes.c_void_p: "ptr", ctypes.c_int: "int", ctypes.c_float: "float", ctypes.c_longlong: "longlong"}
    for name, params in decls.items():
        sig = _lib._SIGNATURES[name]
        assert len(sig) == len(params), (name, len(sig), len(params))
        for i, (p, t) in enumerate(zip(params, sig)):
            if "*" in p:
                want = "ptr"
            elif re.match(r"(const\s+)?long long\b", p):
                want = "longlong"
            elif re.match(r"(const\s+)?float\b", p):
                want = "float"
            else:
                want = "int"
            assert kinds[t] == want, (name, i, p, kinds[t])


def test_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the unmodified reference from baseline/_ref or $DANBO_REFERENCE on the host cores; the
    oracle port only where neither exists) prints one JSON line with the keys the driver reads."""
    import json
    import subprocess
    import sys
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ref_harness
    env = dict(os.environ, DANBO_REF_SAMPLE_RAYS="4096")          # one reference chunk: keeps the CPU suite short
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in line, k
    assert line["impl"] == "reference" and line["unit"] == "rays/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == ("reference" if ref_harness.available() else "port")
    assert line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and "workload" in line["config"]


def test_header_compiles_as_c_and_links():
    """include/danbo_b200.h is plain C: a gcc-compiled program that includes it, takes the address of every declared
    entry point and calls danbo_version() links against the library and runs (no GPU needed)."""
    import subprocess
    import tempfile
    build.build()
    syms = header_symbols()
    src = ['#include <stdio.h>', '#include "danbo_b200.h"', "int main(void) {", "    const void* fns[] = {"]
    src += [f"        (const void*)&{s}," for s in syms]
    src += ["    };", "    unsigned n = 0;", "    for (unsigned i = 0; i < sizeof(fns) / sizeof(fns[0]); ++i) n += fns[i] != 0;",
            '    printf("%u %d\\n", n, danbo_version());', "    return 0;", "}"]
    with tempfile.TemporaryDirectory() as d:
        c, exe = os.path.join(d, "abi.c"), os.path.join(d, "abi")
        open(c, "w").write("\n".join(src) + "\n")
        libdir = os.path.dirname(_lib.path())
        cmd = ["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), c, "-o", exe,
               "-L", libdir, "-l:libdanbo_b200.so", f"-Wl,-rpath,{libdir}", "-Wl,-rpath,/usr/local/cuda/lib64",
               "-L", "/usr/local/cuda/lib64"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr[-3000:]
        out = subprocess.run([exe], capture_output=True, text=True, timeout=60)
        assert out.returncode == 0, out.stderr[-2000:]
        n, ver = out.stdout.split()
        assert int(n) == len(syms) and int(ver) == _lib.ABI_VERSION


def test_entry_points_validate_arguments_without_touching_the_gpu():
    """Error behaviour of the C ABI (include/danbo_b200.h: 0 = ok, < 0 = invalid argument): empty inputs are a no-op and
    invalid arguments are refused before anything is launched, so these calls need no GPU."""
    build.build()
    lib = _lib.load()
    N = None                                         # NULL pointer
    # empty inputs -> 0
    assert lib.danbo_nearfar(N, 8, 0, N, 3, N, 1, 1, N, N, 0, 0, 1.3, 1.3001, N, N, N, 1, N, N, N) == 0
    assert lib.danbo_sample_mask(N, 8, 0, 32, N, N, N, N, N, N, N, 1, 1, N, N, N, N, 0, 0, 0, N) == 0
    assert lib.danbo_field_agg(N, 8, 0, 32, N, N, N, N, 0, N, N, 1, 1, N, N, N, N, N, N, N, 0, 148, 0, N) == 0
    assert lib.danbo_composite_resample(N, 8, 0, 32, 16, N, N, N, N, 1.0, N, N, N, N, N, N, N, N, N, N, N, 1, N) == 0
    assert lib.danbo_graph_net_fwd(N, 0, N, N, N, N) == 0
    assert lib.danbo_train_loss(N, N, N, N, N, N, 1.0, 1, 0, 0, 1.0, 1.0, N, N, N, N, 0, 0.0, N, N, 0.0, N, N, N, N, N, N, N, N) == 0
    # invalid arguments -> negative, nothing launched
    assert lib.danbo_nearfar(N, 4, 16, N, 3, N, 1, 1, N, N, 0, 0, 1.3, 1.3001, N, N, N, 1, N, N, N) < 0        # ray_stride < 8
    assert lib.danbo_sample_mask(N, 8, 16, 32, N, N, N, N, N, N, N, 1, 1, N, N, N, N, 16, 0, 0, N) < 0       # no near/far/z_in
    assert lib.danbo_sample_mask(N, 8, 1 << 20, 1 << 12, N, N, N, N, N, N, N, 1, 1, N, N, N, N, 16, 0, 0, N) < 0   # ids overflow int32
    assert lib.danbo_field_agg(N, 8, 16, 32, N, N, N, N, 64, N, N, 1, 1, N, N, N, N, N, N, N, 0, 148, 0, N) < 0   # no logits / workspace
    assert lib.danbo_composite_resample(N, 8, 16, 2, 16, N, N, N, N, 1.0, N, N, N, N, N, N, N, N, N, N, N, 1, N) < 0     # S < 3
    assert lib.danbo_composite_resample(N, 8, 16, 128, 64, N, N, N, N, 1.0, N, N, N, N, N, N, N, N, N, N, N, 1, N) < 0  # S + S_f > 160
    assert lib.danbo_composite_resample(N, 8, 16, 32, 16, N, N, N, N, 1.0, N, N, N, N, N, N, N, N, N, N, N, 1, N) < 0   # no u_vals / u_rand
    assert lib.danbo_merge_composite(N, 8, 16, 128, 64, N, N, N, N, N, N, N, 1.0, N, N, N, N, N, N, N, N, N, N, N) < 0
    assert lib.danbo_graph_net_fwd(N, 4, N, N, N, N) < 0
    assert lib.danbo_pack_agg_frags(N, N, N) < 0                                                             # no table
    assert lib.danbo_agg_frag_bytes() == 4 * 24 * (2 * 4 * 32 * 2 + 2 * 2 * 4 * 32 * 2)                     # W0 + W1 fragments
    assert lib.danbo_train_loss(N, N, N, N, N, N, 1.0, 1, 16, 0, 1.0, 1.0, N, N, N, N, 0, 0.0, N, N, 0.0, N, N, N, N, N, N, N, N) < 0
