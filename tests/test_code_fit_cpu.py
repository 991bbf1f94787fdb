"""CPU checks of frame-code fitting with a frozen field (training.PoseFitStep(code_kwargs=..., code_optimizer=...)):
the fp64 statement of the code gradient (tests/code_fit_ref.py) against torch autograd through the folded view
layer, every refusal raised before any device work with nothing on the caster or the pose layer moved, and the
ctypes signature of danbo_ray_bias_codes_bwd against the header."""
import ctypes
import os
import re
import sys
import types

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)
import danbo_b200                                    # noqa: E402,F401
from danbo_b200 import _lib, autograd, pose_opt as po, raycaster, render, training   # noqa: E402
from code_fit_ref import code_rows, codes_grad_fp64, folded_view_bias   # noqa: E402
from util import make_caster                         # noqa: E402

FX = np.load(os.path.join(ROOT, "tests", "golden", "popt.npz"))


def _cams(n, n_codes, run, seed):
    """Image-major runs of `run` rays with cams in [-2, n_codes + 2] (negatives and values above the last row), and
    a few single rays of another cam inside 16-ray groups (mixed runs)."""
    g = torch.Generator().manual_seed(seed)
    cams = torch.randint(-2, n_codes + 3, (n // run,), generator=g).repeat_interleave(run)
    for i in torch.randint(0, n, (max(n // 64, 4),), generator=g).tolist():
        cams[i] = int(torch.randint(-2, n_codes + 3, (1,), generator=g))
    return cams.to(torch.int32)


def test_code_gradient_statement_matches_autograd():
    g = torch.Generator().manual_seed(3)
    n, n_codes = 3072, 6
    cam = _cams(n, n_codes, 192, 0)
    dirs = torch.nn.functional.normalize(torch.randn(n, 3, generator=g, dtype=torch.float64), dim=-1)
    w_view = torch.randn(128, 411, generator=g, dtype=torch.float64) * 0.05
    b_view = torch.randn(128, generator=g, dtype=torch.float64) * 0.05
    codes = torch.randn(n_codes, 128, generator=g, dtype=torch.float64).requires_grad_(True)
    mean = torch.randn(128, generator=g, dtype=torch.float64).requires_grad_(True)
    d_rb = torch.randn(n, 128, generator=g, dtype=torch.float64)
    rb = folded_view_bias(dirs, cam, w_view, b_view, codes, mean)
    (rb * d_rb).sum().backward()
    want = codes_grad_fp64(cam, w_view, d_rb, n_codes)
    assert torch.allclose(codes.grad, want, rtol=1e-12, atol=1e-12)
    # every row is reached (clamped cams land on the last one); the mean code takes what the negative cams read
    rows = code_rows(cam, n_codes)
    assert set(rows.tolist()) == set(range(-1, n_codes))
    assert float(mean.grad.abs().max()) > 0 and float(want[-1].abs().max()) > 0


# ---------------------------------------------------------------------------------------------------- refusals
def _popt():
    args = types.SimpleNamespace(opt_rot6d=False, opt_pose_lrate=1e-2, init_poseopt=None, no_poseopt_reload=False,
                                 use_ckpt_anchor=False, opt_pose_cache=False, opt_pose_tol=0.0, opt_pose_coef=2.0,
                                 use_temp_loss=False, ext_scale=0.001, lrate=1e-2, loss_fn="L1", agg_type="sigmoid")
    attrs = {"rest_pose": FX["rest_pose"], "betas": np.zeros((1, 10), np.float32), "kp3d": FX["init_kps"],
             "bones": FX["init_bones"]}
    opt, popt = po.create_popt(args, attrs)
    return args, opt, popt


def _snapshot(caster, popt):
    return ({k: v.clone() for k, v in caster.state_dict()["network_fn_state_dict"].items()},
            {k: v.clone() for k, v in popt["popt_layer"].state_dict().items()})


def _unchanged(caster, popt, snap):
    sd, layer = snap
    assert all(p.grad is None for p in caster.parameters())
    assert all(torch.equal(v, sd[k]) for k, v in caster.state_dict()["network_fn_state_dict"].items())
    assert all(torch.equal(v, layer[k]) for k, v in popt["popt_layer"].state_dict().items())
    assert not hasattr(caster, "grads_in_place") and caster._packed is None and caster._packed_t is None


def _table(rows=4, requires_grad=True, **kw):
    return torch.nn.Parameter(torch.zeros(rows, 128, **kw), requires_grad=requires_grad)


@pytest.mark.parametrize("case,exc,word", [
    ("no_codes", NotImplementedError, "no frame codes"),
    ("width", ValueError, r"\(rows >= 1, 128\)"),
    ("dtype", ValueError, "fp32"),
    ("device", ValueError, "is on meta"),
    ("adam", NotImplementedError, "FlatAdam"),
    ("half", ValueError, "both code_kwargs"),
])
def test_code_fit_refusals(case, exc, word):
    """Refused in PoseFitStep's constructor, before the pose checks and any device work (the pose optimizer here is
    not even a FlatAdam: the code refusals come first)."""
    args, opt, popt = _popt()
    flags = {"opt_framecode": False, "loss_fn": "MSE"} if case == "no_codes" else {}
    caster, _, _ = make_caster("danbo_fast", device="cpu", train=True, **flags)
    snap = _snapshot(caster, popt)
    table = {"width": lambda: torch.nn.Parameter(torch.zeros(4, 64)),
             "dtype": lambda: torch.nn.Parameter(torch.zeros(4, 128, dtype=torch.float64)),
             "device": lambda: torch.nn.Parameter(torch.zeros(4, 128, device="meta"))}.get(case, _table)()
    code_opt = torch.optim.Adam([table], lr=1e-2)
    kwargs = {"code_kwargs": {"frame_codes": table}, "code_optimizer": code_opt}
    if case == "half":
        kwargs = {"code_kwargs": {"frame_codes": table}}
    for graph in (False, True):
        with pytest.raises(exc, match=word):
            training.PoseFitStep(caster, args, popt, opt, graph=graph, **kwargs)
    _unchanged(caster, popt, snap)
    if table.device.type != "meta":
        assert torch.equal(table.detach(), torch.zeros_like(table)) and table.grad is None


def test_create_code_fit_refuses_a_field_without_codes():
    caster, _, _ = make_caster("danbo_fast", device="cpu", opt_framecode=False, loss_fn="MSE")
    with pytest.raises(NotImplementedError, match="no frame codes"):
        training.create_code_fit(caster, 4)


def test_render_refusals():
    """render_rays / render_images / render_graphed / scenes refuse a fitted table they do not implement, before any
    device work."""
    caster, args, _ = make_caster("danbo_fast", device="cpu")
    sd = {k: v.clone() for k, v in caster.state_dict()["network_fn_state_dict"].items()}
    n = 8
    kw = dict(N_samples=8, kp_batch=torch.zeros(n, 24, 3), skts=torch.zeros(n, 24, 4, 4), cyls=torch.zeros(n, 5),
              bones=torch.zeros(n, 24, 3), cams=torch.zeros(n, 1, dtype=torch.long), N_importance=4)
    rays = torch.zeros(n, 8)
    with pytest.raises(ValueError, match=r"\(rows >= 1, 128\)"):
        caster(rays, frame_codes=torch.zeros(3, 127), **kw)
    with pytest.raises(ValueError, match="is on meta"):
        caster(rays, frame_codes=torch.zeros(3, 128, device="meta"), **kw)
    with pytest.raises(NotImplementedError, match="render_graphed"):
        caster.render_graphed(rays, frame_codes=torch.zeros(3, 128), **kw)
    pose = {"kps": np.zeros((24, 3)), "skts": np.zeros((24, 4, 4)), "bones": np.zeros((24, 3)), "cyl": np.zeros(5)}
    for extra, word in (({"graphed": True}, "graphed"), ({"distributed": True}, "distributed")):
        with pytest.raises(NotImplementedError, match=word):
            render.render_images(caster, args, [np.eye(4)], [pose], 8, 8, frame_codes=torch.zeros(3, 128), **extra)
    inst = {"caster": caster, "kps": torch.zeros(1, 24, 3), "skts": torch.zeros(1, 24, 4, 4),
            "bones": torch.zeros(1, 24, 3), "cyls": torch.zeros(1, 5), "cams": 0, "frame_codes": torch.zeros(3, 128)}
    with torch.no_grad(), pytest.raises(NotImplementedError, match="frame_codes"):
        raycaster.check_scene([inst], 8, 4)
    plain, pargs, _ = make_caster("danbo_fast", device="cpu", opt_framecode=False, loss_fn="MSE")
    with pytest.raises(NotImplementedError, match="no frame codes"):
        plain(rays, frame_codes=torch.zeros(3, 128), **kw)
    anerf = types.SimpleNamespace(_supports_frame_codes=False, network=None)
    with pytest.raises(NotImplementedError, match="DANBO field only"):
        raycaster.RayCaster.check_frame_codes(anerf, torch.zeros(3, 128))
    assert all(torch.equal(v, sd[k]) for k, v in caster.state_dict()["network_fn_state_dict"].items())
    assert caster._packed is None


def test_render_block_refuses_codes_fitted_beside_a_trained_network():
    caster, _, _ = make_caster("danbo_fast", device="cpu", train=True)
    with pytest.raises(NotImplementedError, match="while the network trains"):
        autograd.render_block_with_grad(caster, None, 1, None, None, None, None, None, None, None, 8, 8, 1.0, 0., 0.,
                                        None, {}, None, frame_codes=_table())
    assert all(p.grad is None for p in caster.parameters())


def test_codes_entry_point_matches_the_header():
    text = open(os.path.join(ROOT, "include", "danbo_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    args = [a.strip() for a in re.search(r"\bint\s+danbo_ray_bias_codes_bwd\s*\(([^)]*)\)", text).group(1).split(",")]
    sig = _lib._SIGNATURES["danbo_ray_bias_codes_bwd"]
    assert len(sig) == len(args) == 7
    for a, t in zip(args, sig):
        assert (t is ctypes.c_void_p) == ("*" in a), (a, t)
    assert _lib.ABI_VERSION == 5          # a new entry point: no existing signature changed


def test_codes_entry_point_validates_without_the_gpu():
    from danbo_b200 import build
    build.build()
    lib = _lib.load()
    N = None
    assert lib.danbo_ray_bias_codes_bwd(N, 0, 4, N, N, N, N) == 0          # no rays: nothing to do
    assert lib.danbo_ray_bias_codes_bwd(N, 16, 4, N, N, N, N) < 0          # missing pointers: refused, nothing launched
