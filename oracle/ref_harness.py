"""Runs the UNMODIFIED reference, an original DANBO-pytorch checkout: the directory named by $DANBO_REFERENCE, else
the git-ignored copy under baseline/_ref/ that scripts/vendor_ref.sh makes.  Without either, the tests that need it
skip.  TEST / BASELINE INFRASTRUCTURE - nothing in the product imports this.

Used by oracle/gen_golden.py to pin the oracle, by tests/test_oracle_vs_reference.py, by the drop-in tests
(tests/test_gpu_dropin.py: the reference's own Trainer / render_path driving this repo's ray caster) and by bench.py's
reference arm / cpu_baseline (the reference's own `render`, core/trainer.py:96-162, on the host cores).  Needs only import stubs for packages that are not installed
(SURVEY §8c): pytorch3d's three rotation conversions (published formula), empty plotly/matplotlib, an argparse
shim for configargparse, and empty h5py/imageio/deepdish/smplx/pytorch_msssim.  Two compatibility shims:
F6 (np.float32 widths into a tensor under numpy 2) and F5 (A-NeRF ctor kwargs).
"""
import os
import sys
import tempfile

import numpy as np
import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
_CANDIDATES = [os.environ.get("DANBO_REFERENCE"), os.path.join(os.path.dirname(_HERE), "baseline", "_ref")]
REF = next((c for c in _CANDIDATES if c and os.path.isdir(os.path.join(c, "core"))), _CANDIDATES[-1])
STUBS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ref_stubs")


def available():
    return os.path.isdir(os.path.join(REF, "core"))


def _imports():
    for p in (STUBS, REF):
        if p not in sys.path:
            sys.path.insert(0, p)
    import core.raycasters as rc                      # noqa
    import run_nerf                                   # noqa
    return rc, run_nerf


def parse_args(config="h36m_zju/danbo_fast.txt", extra=()):
    rc, run_nerf = _imports()
    tmp = tempfile.mkdtemp(prefix="danbo_ref_")
    argv = ["--config", os.path.join(REF, "configs", config), "--no_reload", "--basedir", tmp,
            "--expname", "probe"] + list(extra)
    args = run_nerf.config_parser().parse_args(argv)
    os.makedirs(os.path.join(tmp, "probe"), exist_ok=True)
    return args


def build(args, rest_pose, n_views=8, near=1.0, far=5.0, seed=0, device="cpu"):
    """create_raycaster under the shims -> the bare (non-DataParallel) reference ray caster, on `device` (the reference
    wraps its caster in nn.DataParallel, which MOVES the module to the GPU when exactly one is visible)."""
    rc, _ = _imports()
    from core.utils.skeleton_utils import SMPLSkeleton

    orig_profile = rc.get_skel_profile_from_rest_pose

    def profile_f64(*a, **k):                          # F6
        prof = orig_profile(*a, **k)
        return {k_: (v.astype(np.float64) if k_.endswith("_width") else v) for k_, v in prof.items()}

    orig_create = rc.create_nerf

    def create_nerf(args_, kwargs, data_attrs):        # F5
        if args_.nerf_type == "nerf":
            kwargs = {k_: v for k_, v in kwargs.items() if k_ not in ("mask_vol_prob", "agg_type")}
        return orig_create(args_, kwargs, data_attrs)

    rc.get_skel_profile_from_rest_pose = profile_f64
    rc.create_nerf = create_nerf
    try:
        torch.manual_seed(seed)
        data_attrs = {"skel_type": SMPLSkeleton, "near": near, "far": far, "n_views": n_views,
                      "rest_pose": rest_pose}
        import contextlib, io
        with contextlib.redirect_stdout(io.StringIO()):
            _, kw_test, _, _, _, _ = rc.create_raycaster(args, data_attrs)
    finally:
        rc.get_skel_profile_from_rest_pose = orig_profile
        rc.create_nerf = orig_create
    kw_test["ray_caster"].to(device)
    return kw_test["ray_caster"], kw_test


def load_weights(caster, sd):
    """Overwrite the reference network's parameters with `sd` (reference names); returns the full dict."""
    net = caster.network
    own = net.state_dict()
    for k, v in sd.items():
        assert k in own and tuple(own[k].shape) == tuple(v.shape), (k, v.shape)
        own[k] = v.clone()
    net.load_state_dict(own)
    return {k: v.clone() for k, v in net.state_dict().items()}


def reference_render_setup(preset_config="h36m_zju/danbo_fast.txt", device="cpu", weight_seed=0, extra=()):
    """-> (render_fn, kw_test): the reference ray caster with this repo's synthetic weights on `device`, and the reference's
    own `render` (core/trainer.py:96-162: ray batch assembly + `batchify_rays` in `chunk`s)."""
    rc, _ = _imports()
    from core.trainer import render
    root = os.path.dirname(_HERE)
    if root not in sys.path:
        sys.path.insert(0, root)
    from danbo_b200 import synthetic as syn
    args = parse_args(preset_config, extra)
    caster, kw_test = build(args, syn.rest_pose())
    load_weights(caster, syn.synthetic_params(weight_seed))
    caster.to(device)
    caster.eval()
    return render, kw_test, args


def reference_render_rays(render, kw_test, args, rays_o, rays_d, pose, cams, H, W, focal, device="cpu"):
    """One call of the reference's `render` on a ray set of one pose (what `render_path` does per image,
    run_nerf.py:92-96).  pose: dict with kps / skts / bones / cyl arrays.  -> dict of outputs."""
    n = rays_o.shape[0]
    t = lambda a: torch.as_tensor(a, dtype=torch.float32, device=device)[None].expand(n, *np.shape(a))
    with torch.no_grad():
        return render(H, W, focal, rays=(rays_o.to(device), rays_d.to(device)), chunk=args.chunk,
                      kp_batch=t(pose["kps"]), skts=t(pose["skts"]), cyls=t(pose["cyl"]), bones=t(pose["bones"]),
                      cams=cams.to(device), **kw_test)
