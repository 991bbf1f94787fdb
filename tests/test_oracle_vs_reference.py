"""Live comparison of the CPU oracle with the UNMODIFIED reference on inputs that are NOT among the committed fixtures
(other poses, ray subsets and weight seeds).  Needs an original DANBO-pytorch checkout ($DANBO_REFERENCE or the copy
under baseline/_ref/, see oracle/ref_harness.py) and skips without one."""
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import ref_harness as rh  # noqa: E402

pytestmark = pytest.mark.skipif(not rh.available(), reason="needs the original DANBO-pytorch (DANBO_REFERENCE or baseline/_ref)")


def _render_both(config, extra, pose_seed, weight_seed, n_rays, agg_type="sigmoid", lindisp=False):
    import danbo_oracle as orc
    from danbo_b200 import params, synthetic as syn
    from util import align_A
    args = rh.parse_args(config, list(extra))
    caster, kw = rh.build(args, syn.rest_pose())
    caster.eval()
    rh.load_weights(caster, syn.synth_state_dict(params.danbo_param_shapes(), weight_seed))
    pose = syn.make_pose(pose_seed)
    full = syn.render_batch(pose, 48, 48)
    g = torch.Generator().manual_seed(pose_seed)
    pick = torch.sort(torch.randperm(full["ray_batch"].shape[0], generator=g)[:n_rays]).values
    b = {k: (v[pick].contiguous() if torch.is_tensor(v) and v.shape[0] == full["ray_batch"].shape[0] else v)
         for k, v in full.items()}
    kwargs = {k: v for k, v in kw.items() if k not in ("ray_caster", "N_samples", "use_viewdirs")}
    with torch.no_grad():
        want = caster(b["ray_batch"], N_samples=args.N_samples, kp_batch=b["kp_batch"], skts=b["skts"], cyls=b["cyls"],
                      bones=b["bones"], cams=b["cams"], N_uniques=1, **kwargs)
        t = lambda a: torch.as_tensor(a)[None]
        got = orc.render_rays(b["ray_batch"], t(pose["skts"]), t(pose["bones"]), t(pose["cyl"]), b["cams"], align_A(),
                              syn.synthetic_params(weight_seed), args.N_samples, args.N_importance, rays_per_pose=n_rays,
                              use_volume_near_far=bool(args.use_volume_near_far), agg_type=agg_type, lindisp=lindisp)
    return got, want, n_rays


@pytest.mark.parametrize("config,extra,kw", [
    ("h36m_zju/danbo_fast.txt", (), {}),
    ("h36m_zju/danbo_base.txt", ("--N_samples", "40", "--N_importance", "24"), {}),
    ("h36m_zju/danbo_fast.txt", ("--agg_type", "softmax"), {"agg_type": "softmax"}),
    ("h36m_zju/danbo_fast.txt", ("--lindisp",), {"lindisp": True}),
])
def test_oracle_matches_live_reference(config, extra, kw):
    got, want, N = _render_both(config, extra, pose_seed=11, weight_seed=2, n_rays=96, **kw)
    for k in ("rgb_map", "acc_map", "disp_map", "rgb0", "acc0"):
        err = (got[k] - want[k]).abs().reshape(N, -1).max(-1).values
        scale = max(float(want[k].abs().max()), 1.0)
        # a sample within rounding of a bone-box face flips its mask and moves that ray discontinuously (see
        # test_oracle_golden.test_render_rays_end_to_end): 98 % of rays within 2e-5 of scale
        assert float((err <= 2e-5 * scale).float().mean()) >= 0.98, (k, float(err.max()))


def test_anerf_oracle_matches_live_reference():
    """AN1 live: another pose, other weights and sample counts than the committed `render_anerf` fixture."""
    import danbo_oracle as orc
    from danbo_b200 import params, synthetic as syn
    from util import align_A
    args = rh.parse_args("h36m_zju/anerf_base.txt", ["--N_samples", "20", "--N_importance", "10"])
    caster, kw = rh.build(args, syn.rest_pose())
    caster.eval()
    sd = syn.synth_state_dict(params.anerf_param_shapes(), 5)
    rh.load_weights(caster, sd)
    pose = syn.make_pose(13)
    full = syn.render_batch(pose, 40, 40)
    g = torch.Generator().manual_seed(13)
    N = 48
    pick = torch.sort(torch.randperm(full["ray_batch"].shape[0], generator=g)[:N]).values
    b = {k: (v[pick].contiguous() if torch.is_tensor(v) and v.shape[0] == full["ray_batch"].shape[0] else v)
         for k, v in full.items()}
    kwargs = {k: v for k, v in kw.items() if k not in ("ray_caster", "N_samples", "use_viewdirs")}
    with torch.no_grad():
        want = caster(b["ray_batch"], N_samples=args.N_samples, kp_batch=b["kp_batch"], skts=b["skts"], cyls=b["cyls"],
                      bones=b["bones"], cams=b["cams"], N_uniques=1, **kwargs)
        P = {k: torch.as_tensor(v) for k, v in sd.items()}
        t = lambda a: torch.as_tensor(a)[None]
        got = orc.anerf_render_rays(b["ray_batch"], t(pose["skts"]), t(pose["cyl"]), b["cams"], align_A(), P,
                                    args.N_samples, args.N_importance, rays_per_pose=N,
                                    tau=float(caster.network.pe_fn.get_tau()))
    for k in ("rgb_map", "acc_map", "rgb0", "acc0"):
        err = (got[k] - want[k]).abs().reshape(N, -1).max(-1).values
        # the 64x-amplified top octave of the cutoff PE moves raw by ~1e-4; a ray whose importance samples flip a bin moves more
        assert float((err <= 2e-4).float().mean()) >= 0.95, (k, float(err.max()))


@pytest.mark.parametrize("config", ["h36m_zju/danbo_base.txt", "h36m_zju/danbo_fast.txt", "h36m_zju/anerf_base.txt",
                                    "h36m_zju/anerf_h.txt", "perfcap/danbo_base.txt", "perfcap/danbo_fast.txt",
                                    "perfcap/anerf_base.txt", "surreal/danbo_base.txt", "surreal/danbo_fast.txt"])
def test_flag_defaults_and_config_reader_match_the_reference_parser(config):
    """`config.DEFAULTS` + `read_config_file` against the reference's own argparse (run_nerf.py:186-572) on the shipped
    configs: every flag this path looks at must come out with the reference's value; the presets are those configs."""
    import danbo_b200 as db
    from danbo_b200 import config as cfg, raycaster, anerf
    want = vars(rh.parse_args(config, []))
    got = vars(db.make_args(config_file=os.path.join(rh.REF, "configs", config)))
    skip = {"expname", "basedir", "no_reload"}                      # set by the harness itself
    bad = {k: (got[k], want[k]) for k in cfg.DEFAULTS if k in want and k not in skip and got[k] != want[k]}
    assert not bad, bad
    args = db.make_args(config_file=os.path.join(rh.REF, "configs", config), no_reload=True)
    (anerf.check_anerf_args if args.nerf_type == "nerf" else raycaster.check_args)(args)       # the path accepts them
    preset = {"h36m_zju/danbo_base.txt": "danbo_base", "h36m_zju/danbo_fast.txt": "danbo_fast",
              "h36m_zju/anerf_base.txt": "anerf_base"}.get(config)
    if preset:
        p = vars(db.make_args(preset))
        bad = {k: (p[k], want[k]) for k in cfg.DEFAULTS if k in want and k not in skip and p[k] != want[k]}
        assert not bad, bad


def test_setup_constants_match_live_reference():
    """S0 / S1: the bone-align transforms (raycasters.py:548-591) and the initial per-bone half extents
    (misc.py:675-724, gnn_backbone.py:777-785) of the reference's freshly constructed caster, for two rest poses."""
    import numpy as np
    from danbo_b200 import skeleton as sk, synthetic as syn
    for scale in (0.5, 0.43):
        rest = (sk.SMPL_REST_POSE * scale).astype(np.float32)
        args = rh.parse_args("h36m_zju/danbo_fast.txt", [])
        caster, _ = rh.build(args, rest)
        A, child = sk.bone_align_transforms(rest)
        want_A = caster.transforms.detach().numpy().reshape(24, 4, 4)
        assert np.abs(A - want_A).max() <= 1e-6, np.abs(A - want_A).max()
        assert list(np.asarray(child)) == list(np.asarray(caster.child_idxs))
        got = sk.initial_axis_scale(sk.skeleton_profile(rest), 0.4)
        want = caster.network.graph_net.axis_scale.detach()
        assert float((got - want).abs().max()) <= 1e-6 * float(want.abs().max()), float((got - want).abs().max())
