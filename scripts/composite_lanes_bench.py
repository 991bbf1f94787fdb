"""Lanes per ray of the forward compositing kernels: times `danbo_composite_resample` and `danbo_merge_composite` built
with several lane tables, and optionally a reference build of another composite.cu (the parent commit's, say), on
seeded synthetic inputs at the sample counts in use; counts the output elements that differ from the reference bit for bit.

    python scripts/composite_lanes_bench.py --out FILE.json [--ref OLD_composite.cu]
        [--variant CR/MC ...]          CR, MC: lanes per ray for kEo = 1..5 (kEo = ceil(S / 32)), e.g. 8,16,16,32,32/8,16,32,32,32

Each variant replaces the `kCrLanes` / `kMcLanes` tables of csrc/composite.cu in a copy compiled into a temporary
directory (same nvcc flags as the package build); nothing in the tree is written.  In the output, a timing key is the
variant string ("ref" for --ref), each value a list of rounds (builds alternate within a round) of median CUDA-event
times in µs of one launch over 30 launches; `differ_from_ref` lists, per variant, every output with its count of
differing elements and largest absolute difference (empty: bit-identical).  The card's name, power limit and SM clock
limit are recorded in the same file."""
import argparse, concurrent.futures, ctypes, json, os, re, shutil, subprocess, sys, tempfile
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "danbo-pytorch_b200", "csrc")
sys.path.insert(0, os.path.join(ROOT, "danbo-pytorch_b200"))
from build import NVCC_FLAGS                                    # noqa: E402

P, I, F = ctypes.c_void_p, ctypes.c_int, ctypes.c_float
SIG_CR = [P, I, I, I, I, P, P, P, P, F, P, P, P, P, P, P, P, P, P, P, P, I, P]
SIG_MC = [P, I, I, I, I, P, P, P, P, P, P, P, F, P, P, P, P, P, P, P, P, P, P, P]
DEFAULT_VARIANTS = ["8,16,16,32,32/8,16,32,32,32", "16,16,16,32,32/16,16,16,32,32", "8,8,32,32,32/8,8,16,32,32",
                    "32,32,32,32,32/32,32,32,32,32"]
# (rays, S, S_f, train): the bench image, config #3's training shape, A-NeRF's coarse pass and its fine composite
SHAPES = [(261121, 32, 16, False), (261121, 32, 16, True), (131072, 64, 16, False), (131072, 64, 16, True),
          (65536, 96, 48, False), (65536, 144, 0, False)]
dev = torch.device("cuda")
ptr = lambda t: None if t is None else t.data_ptr()


def compile_lib(src_text, tmp, name):
    d = os.path.join(tmp, name)
    os.makedirs(d)
    shutil.copy(os.path.join(CSRC, "common.cuh"), d)
    with open(os.path.join(d, "composite.cu"), "w") as f:
        f.write(src_text)
    lib = os.path.join(d, "lib.so")
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    subprocess.run([nvcc] + NVCC_FLAGS + ["-shared", os.path.join(d, "composite.cu"), "-o", lib], check=True)
    h = ctypes.CDLL(lib)
    h.danbo_composite_resample.argtypes = SIG_CR
    h.danbo_merge_composite.argtypes = SIG_MC
    return h


def with_tables(src, variant):
    cr, mc = variant.split("/")
    for name, vals in (("kCrLanes", cr), ("kMcLanes", mc)):
        assert len(vals.split(",")) == 5 and all(v in ("8", "16", "32") for v in vals.split(",")), variant
        src, n = re.subn(r"constexpr int %s\[5\] = \{[^}]*\};" % name, "constexpr int %s[5] = {%s};" % (name, vals), src)
        assert n == 1, name
    return src


def inputs(N, S, S_f, train, seed=0):
    g = torch.Generator(device=dev).manual_seed(seed)
    scale = torch.tensor([2., 2., 2., 20.], device=dev)
    x = dict(rays=torch.randn(N, 8, device=dev, generator=g))
    t = (torch.arange(S, device=dev) + torch.rand(N, S, device=dev, generator=g)) / S
    x["z"] = (2.0 + torch.rand(N, 1, device=dev, generator=g) + 4.0 * t).contiguous()
    x["raw"] = torch.randn(N * S + N, 4, device=dev, generator=g) * scale
    x["mask"] = (torch.rand(N, S, device=dev, generator=g) < 0.35).int() * 7        # sparse, like DANBO's coarse masks
    x["raw1"] = torch.randn(N * S_f, 4, device=dev, generator=g) * scale
    x["mask1"] = (torch.rand(N, S_f, device=dev, generator=g) < 0.5).int() * 7
    x["u_vals"] = torch.linspace(0., 1., S_f).to(dev)
    x["u_rand"] = torch.rand(N, S_f, device=dev, generator=g) if train else None
    x["noise"] = torch.randn(N, S, device=dev, generator=g) if train else None
    x["noise1"] = torch.randn(N, S + S_f, device=dev, generator=g) if train else None
    x["confd0"] = torch.randn(N * S, 24, device=dev, generator=g) if train else None
    x["confd1"] = torch.randn(N * S_f, 24, device=dev, generator=g) if train else None
    return x


def run(lib, x, N, S, S_f, train, reps=30):
    f = lambda *s: torch.empty(*s, device=dev)
    St = S + S_f
    o = dict(w=f(N, S), a=f(N, S), rgb=f(N, 3), disp=f(N), acc=f(N), zs=f(N, S_f), z_all=f(N, St),
             order=torch.empty(N, St, dtype=torch.int32, device=dev))
    m = dict(w=f(N, St), a=f(N, St), rgb=f(N, 3), disp=f(N), acc=f(N))
    if train:
        m["confd"], m["invalid"] = f(N, St, 24), f(N, St, 24)
    s = torch.cuda.current_stream().cuda_stream

    def cr():
        assert lib.danbo_composite_resample(ptr(x["rays"]), 8, N, S, S_f, ptr(x["raw"]), ptr(x["mask"]), ptr(x["z"]),
                                            ptr(x["noise"]), 1.0, ptr(x["u_vals"]), ptr(x["u_rand"]), ptr(o["w"]),
                                            ptr(o["a"]), ptr(o["rgb"]), ptr(o["disp"]), ptr(o["acc"]), ptr(o["zs"]),
                                            ptr(o["z_all"]), ptr(o["order"]), None, 0 if train else 1, s) == 0

    def mc():
        assert lib.danbo_merge_composite(ptr(x["rays"]), 8, N, S, S_f, ptr(x["raw"]), ptr(x["mask"]), ptr(x["raw1"]),
                                         ptr(x["mask1"]), ptr(o["z_all"]), ptr(o["order"]), ptr(x["noise1"]), 1.0,
                                         ptr(m["w"]), ptr(m["a"]), ptr(m["rgb"]), ptr(m["disp"]), ptr(m["acc"]), None,
                                         ptr(x["confd0"]), ptr(x["confd1"]), ptr(m.get("confd")), ptr(m.get("invalid")),
                                         s) == 0
    times = {}
    for name, fn in (("composite_resample", cr), ("merge_composite", mc))[: 2 if S_f > 0 else 1]:
        for _ in range(3):
            cr(); fn()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * reps)]
        for r in range(reps):
            if fn is mc:
                cr()                                             # the merge reads this coarse call's order
            ev[2 * r].record(); fn(); ev[2 * r + 1].record()
        torch.cuda.synchronize()
        ts = sorted(ev[2 * r].elapsed_time(ev[2 * r + 1]) * 1e3 for r in range(reps))
        times[name] = round(ts[reps // 2], 1)
    cr()
    outs = {"composite_resample." + k: v for k, v in o.items() if S_f > 0 or k in ("w", "a", "rgb", "disp", "acc")}
    if S_f > 0:
        mc()
        outs.update({"merge_composite." + k: v for k, v in m.items()})
    torch.cuda.synchronize()
    return times, {k: v.clone() for k, v in outs.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--ref", default=None, help="another composite.cu to time and compare against")
    ap.add_argument("--variant", action="append", default=None)
    opt = ap.parse_args()
    variants = opt.variant or DEFAULT_VARIANTS
    src = open(os.path.join(CSRC, "composite.cu")).read()
    tmp = tempfile.mkdtemp(prefix="composite_lanes_")
    try:
        jobs = [(v, with_tables(src, v)) for v in variants] + ([("ref", open(opt.ref).read())] if opt.ref else [])
        with concurrent.futures.ThreadPoolExecutor(len(jobs)) as ex:
            built = list(ex.map(lambda ij: compile_lib(ij[1][1], tmp, "v%d" % ij[0]), enumerate(jobs)))
        libs = {name: lib for (name, _), lib in zip(jobs, built)}
        gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True).stdout.strip()
        res = {"gpu": gpu, "shapes": []}
        for N, S, S_f, train in SHAPES:
            x = inputs(N, S, S_f, train)
            row = {"rays": N, "S": S, "S_f": S_f, "mode": "train" if train else "eval", "times_us": {}}
            outs = {}
            for _ in range(2):
                for name, lib in libs.items():
                    t, outs[name] = run(lib, x, N, S, S_f, train)
                    row["times_us"].setdefault(name, []).append(t)
            if "ref" in outs:
                row["differ_from_ref"] = {
                    name: {k: [int((v != outs["ref"][k]).sum()), float((v.double() - outs["ref"][k].double()).abs().max())]
                           for k, v in o.items() if not torch.equal(v, outs["ref"][k])}
                    for name, o in outs.items() if name != "ref"}
            print(json.dumps(row), flush=True)
            res["shapes"].append(row)
        with open(opt.out, "w") as f:
            json.dump(res, f, indent=1)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
