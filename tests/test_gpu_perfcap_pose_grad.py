"""Pose refinement on the perfcap configs on the GPU (run with -m gpu): `danbo_view_root_bwd`'s d skts against oracle
autograd, the whole training step's d loss / d skts with root-local view directions, and a --opt_pose TrainStep on a
perfcap caster."""
import numpy as np
import pytest
import torch

import danbo_oracle as orc
from util import load_fixture, params_for, align_A, make_caster, preset_of, config_flags_of, field_mlp_bf16_ste
from test_perfcap_pose_grad_cpu import CASES, perfcap_case, oracle_skts_grad, random_ray_bias_grad

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(300, method="thread")]   # a hung kernel must not hang the box
DEV = "cuda"


def _rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm())


def _cos(a, b):
    a, b = a.reshape(-1).double(), b.reshape(-1).double()
    return float(torch.dot(a, b) / (a.norm() * b.norm() + 1e-30))


@pytest.mark.parametrize("name", CASES)
def test_view_root_bwd_matches_oracle_autograd(name):
    """Stage level: the kernel's d skts for a random d ray_bias against fp64 autograd of the oracle on the same fp32
    inputs.  The kernel reduces 32 rays per block: render_perfcap (160 rays, one pose) and train_perfcap (4 poses x 48
    rays) have blocks of one pose and blocks holding two; train_perfcap_straddle (43 rays) a first block with both of
    its poses and a partial second block."""
    from danbo_b200 import kernels as K
    rays, pose_skts, rpp, Wv, cams = perfcap_case(name)
    N = rays.shape[0]
    d_rb = random_ray_bias_grad(N, 7)
    d = lambda t: t.to(DEV).float().contiguous()
    got = torch.zeros(pose_skts.shape, device=DEV)
    K.view_root_bwd(d(rays), d(pose_skts), rpp, d(Wv), d(d_rb), got)
    torch.cuda.synchronize()
    got = got.cpu()
    want = oracle_skts_grad(rays.double(), pose_skts.double(), rpp, Wv.double(), cams, d_rb.double())
    rel = _rel(got, want)
    per_pose = [_rel(got[g], want[g]) for g in range(pose_skts.shape[0])]
    print(f"[perfcap popt] view_root_bwd {name}: {N} rays, {pose_skts.shape[0]} poses, |g| {float(want.norm()):.3e} "
          f"rel {rel:.2e}, per pose max {max(per_pose):.2e}")
    assert float(got[:, 0, :, 3].abs().max()) == 0.0 and float(got[:, 0, 3].abs().max()) == 0.0
    assert float(got[:, 1:].abs().max()) == 0.0
    assert rel <= 1e-5, rel
    assert max(per_pose) <= 1e-5, per_pose                      # a misrouted ray or block shows here


def _perfcap_step(caster, args, fx, b, rand, skts, bones, stages=None):
    out = caster.render_rays(b["ray_batch"], N_samples=args.N_samples, kp_batch=b["kp_batch"], skts=skts,
                             cyls=b["cyls"], bones=bones, cams=b["cams"], N_uniques=int(fx["n_poses"]), perturb=1.0,
                             N_importance=args.N_importance, raw_noise_std=0.,
                             _rand={k: v.to(DEV) for k, v in rand.items()}, _stages=stages)
    P = {"graph_net.axis_scale": caster.network.graph_net.axis_scale}
    from danbo_b200 import skeleton as sk, synthetic as syn
    init_scale = sk.initial_axis_scale(sk.skeleton_profile(syn.rest_pose()), 0.4)
    loss = orc.training_loss(out, b["target_s"].to(DEV), b["bgs"].to(DEV), P, init_scale.to(DEV))
    caster.network.zero_grad(set_to_none=True)
    loss.backward()
    torch.cuda.synchronize()
    grads = {n: p.grad.detach().cpu().clone() for n, p in caster.network.named_parameters() if p.grad is not None}
    return loss, grads


def _oracle_step(fx, b, rand, z_samples, detach_view):
    """Oracle d loss / d (pose skts, pose bones) at the given importance samples, with the kernel's bf16 operand rounding
    (`util.field_mlp_bf16_ste`).  detach_view: the view branch sees skts.detach(), i.e. no root-local view term."""
    from danbo_b200 import skeleton as sk, synthetic as syn
    rpp = int(fx["rays_per_pose"])
    P = params_for(fx)
    pose_skts = b["skts"][::rpp].clone().requires_grad_(True)
    pose_bones = b["bones"][::rpp].clone().requires_grad_(True)
    view_directions = orc.view_directions
    if detach_view:
        orc.view_directions = lambda rays_d, skts, mode="world": view_directions(rays_d, skts.detach(), mode)
    try:
        ref = orc.render_rays(b["ray_batch"], pose_skts, pose_bones, b["cyls"][::rpp], b["cams"], align_A(), P,
                              int(fx["N_samples"]), int(fx["N_importance"]), rays_per_pose=rpp,
                              use_volume_near_far=bool(fx["use_volume_near_far"]), training=True, rand=rand,
                              raw_noise_std=0., z_samples=z_samples, view_mode="root_local", mlp_fn=field_mlp_bf16_ste)
    finally:
        orc.view_directions = view_directions
    init_scale = sk.initial_axis_scale(sk.skeleton_profile(syn.rest_pose()), 0.4)
    loss = orc.training_loss(ref, b["target_s"], b["bgs"], P, init_scale)
    loss.backward()
    return float(loss.detach()), pose_skts.grad, pose_bones.grad


def test_training_step_pose_gradients():
    """Whole step on train_perfcap: the per-ray world-to-bone matrices and bone parameters enter the perfcap caster as
    leaves; their per-pose gradients against the oracle at the kernel path's own importance samples.  Both sides run
    with raw_noise_std = 0 (see test_gpu_configs.py::test_training_step_other_shipped_configs).  Joint 0's rotation
    block must be closer to the full oracle than to one without the view term, and that term must be a visible part of
    the block: otherwise a kernel that adds nothing would pass the bounds."""
    from danbo_b200 import synthetic as syn
    fx = load_fixture("train_perfcap")
    caster, args, _ = make_caster(preset_of(fx), train=True, **config_flags_of(fx))
    assert caster.view_mode == "root_local"
    n_poses, rpp = int(fx["n_poses"]), int(fx["rays_per_pose"])
    b = syn.training_batch(n_poses, rpp, seed=int(fx["batch_seed"]))
    rand = {k: fx["rand." + k] for k in ("t_rand", "noise0", "u", "noise1")}
    skts_leaf = b["skts"].clone().to(DEV).requires_grad_(True)
    bones_leaf = b["bones"].clone().to(DEV).requires_grad_(True)
    stages = {}
    loss, _ = _perfcap_step(caster, args, fx, b, rand, skts_leaf, bones_leaf, stages)
    per_pose = lambda g: g.reshape(n_poses, rpp, *g.shape[1:]).sum(1).cpu()
    got_skts, got_bones = per_pose(skts_leaf.grad), per_pose(bones_leaf.grad)
    z = stages["z_samples"].cpu()
    ref_loss, want_skts, want_bones = _oracle_step(fx, b, rand, z, detach_view=False)
    _, det_skts, _ = _oracle_step(fx, b, rand, z, detach_view=True)
    assert abs(float(loss.detach()) - ref_loss) <= 5e-4
    assert float(got_skts[:, :, 3].abs().max()) == 0.0                   # the homogeneous row of every joint
    for nm, got, want in (("skts", got_skts, want_skts), ("bones", got_bones, want_bones)):
        cos, rel = _cos(got, want), _rel(got, want)
        print(f"[perfcap popt] step d {nm}: |g| {float(want.norm()):.3e} cos {cos:.5f} rel {rel:.3e}")
        assert cos >= 0.985 and rel <= 0.2, (nm, cos, rel)         # the DANBO pose path's bounds
    blk = lambda t: t[:, 0, :3, :3]
    view_term = float((blk(want_skts) - blk(det_skts)).norm())
    to_full = float((blk(got_skts) - blk(want_skts)).norm())
    to_detached = float((blk(got_skts) - blk(det_skts)).norm())
    share = view_term / float(blk(want_skts).norm())
    print(f"[perfcap popt] joint 0 rotation block: |oracle| {float(blk(want_skts).norm()):.3e}, view term {view_term:.3e} "
          f"({100 * share:.1f} %); kernels to full oracle {to_full:.3e}, to oracle without the view term {to_detached:.3e}")
    assert share >= 0.02, share
    assert to_full < to_detached, (to_full, to_detached)


def test_parameter_gradients_unchanged_by_the_pose_leaf():
    """The network's parameter gradients with and without a skts leaf agree to within the run-to-run floor of the atomic
    reductions: the pose gradient adds launches, it does not change what the others compute."""
    from danbo_b200 import synthetic as syn
    fx = load_fixture("train_perfcap")
    caster, args, _ = make_caster(preset_of(fx), train=True, **config_flags_of(fx))
    n_poses, rpp = int(fx["n_poses"]), int(fx["rays_per_pose"])
    b = syn.training_batch(n_poses, rpp, seed=int(fx["batch_seed"]))
    rand = {k: fx["rand." + k] for k in ("t_rand", "noise0", "u", "noise1")}
    _, g_a = _perfcap_step(caster, args, fx, b, rand, b["skts"], b["bones"])
    _, g_b = _perfcap_step(caster, args, fx, b, rand, b["skts"], b["bones"])
    leaf = b["skts"].clone().to(DEV).requires_grad_(True)
    _, g_c = _perfcap_step(caster, args, fx, b, rand, leaf, b["bones"])
    assert leaf.grad is not None and float(leaf.grad.norm()) > 0
    assert set(g_c) == set(g_a)
    floor = max(_rel(g_b[k], g_a[k]) for k in g_a if float(g_a[k].norm()) > 0)
    worst = max(_rel(g_c[k], g_a[k]) for k in g_a if float(g_a[k].norm()) > 0)
    print(f"[perfcap popt] {len(g_a)} parameter gradients with a pose leaf: rel {worst:.2e} (run-to-run floor {floor:.2e})")
    assert worst <= max(2 * floor, 1e-5), (worst, floor)


def test_train_step_with_pose_layer_and_feed():
    """--opt_pose on a perfcap caster end to end: device feed -> pose layer -> render -> fused loss + pose regulariser ->
    both optimisers.  With opt_pose_coef = 0 the regulariser's gradient is zero, so the poses of the frames drawn move
    only through the render loss and the others must not move.  Then 20 steps on one batch: the loss falls."""
    import danbo_b200 as db
    from danbo_b200 import feed as fd, pose_opt as po, training, synthetic as syn
    flags = dict(view_type="relray", ray_tr_type="root_local", nerf_type="graph")     # configs/perfcap/danbo_fast.txt
    caster, _, _ = make_caster("danbo_fast", train=True, **flags)
    args = db.make_args("danbo_fast", no_reload=True, opt_pose=True, **flags)
    assert caster.view_mode == "root_local"
    n_images = 12
    arrays = fd.synthetic_arrays(n_images=n_images, H=64, W=64, seed=2)
    feed = fd.RayFeed.from_arrays(arrays, syn.NEAR, syn.FAR, N_rand=4 * 48, N_sample_images=4, device=DEV, seed=1,
                                  cam_idxs=np.arange(n_images) % 8)
    args.opt_pose_coef, args.opt_pose_tol, args.opt_pose_lrate = 0.0, 0.0, 1e-3
    attrs = {"rest_pose": syn.rest_pose()[None], "betas": torch.zeros(1, 10).numpy(), "kp3d": arrays["kp3d"],
             "bones": arrays["bones"]}
    pose_optimizer, kw = po.create_popt(args, attrs, device=DEV)
    layer = kw["popt_layer"]
    before = layer.bones.detach().clone()
    step = training.TrainStep(caster, args, popt_kwargs=kw, pose_optimizer=pose_optimizer)
    with pytest.raises(NotImplementedError):
        training.TrainStep(caster, args, graph=True, popt_kwargs=kw, pose_optimizer=pose_optimizer)
    g = torch.Generator(device=DEV).manual_seed(0)
    touched = set()
    for _ in range(2):
        batch = feed.next_batch(g)
        touched.update(feed.last_idxs[0].tolist())
        loss, preds = step(batch)
        assert preds["rgb_map"].shape == (4 * 48, 3) and float(loss) == float(loss)
    torch.cuda.synchronize()
    moved = (layer.bones.detach() - before).abs().amax(dim=(1, 2)).cpu()
    print("[perfcap popt] touched", sorted(touched), "moved", [f"{float(v):.1e}" for v in moved])
    assert len(touched) < n_images
    for i in range(n_images):
        assert (float(moved[i]) > 0) == (i in touched), (i, float(moved[i]), sorted(touched))
    losses = [float(step(batch)[0]) for _ in range(20)]
    torch.cuda.synchronize()
    print("[perfcap popt] losses", ["%.4f" % v for v in losses])
    assert all(v == v for v in losses) and losses[-1] < losses[0] - 0.01
    assert bool(torch.isfinite(layer.bones).all()) and bool(torch.isfinite(layer.pelvis).all())
