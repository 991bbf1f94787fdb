"""Pose fitting with a frozen DANBO field on the GPU (run with -m gpu): training.PoseFitStep against training's own pose
gradient, the network left untouched, the captured step against the eager one, no weight-gradient launch, the
pose-only kernel variants against their full versions, a fit that recovers perturbed poses, and checkpoints between
fitting and training."""
import os

import numpy as np
import pytest
import torch

from util import make_caster

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900, method="thread")]   # a hung kernel must not hang the box
DEV = "cuda"
PERFCAP = dict(view_type="relray", ray_tr_type="root_local", nerf_type="graph")     # configs/perfcap/danbo_fast.txt
CONFIGS = pytest.mark.parametrize("flags", [{}, PERFCAP], ids=["h36m_zju", "perfcap"])
# Kernels of one uncaptured TrainStep(graph=True)._step with a pose layer (kernels._count), as measured on the parent
# commit of PoseFitStep on a B200: training's launch sequence must not change.
TRAIN_LAUNCHES = {"world": 58, "root_local": 59}


def _rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp(min=1e-30))


def _setup(flags, coef=1.0, lr=1e-3, n_images=12, rays_per_image=48):
    import danbo_b200 as db
    from danbo_b200 import feed as fd, synthetic as syn
    args = db.make_args("danbo_fast", no_reload=True, opt_pose=True, **flags)
    args.perturb, args.raw_noise_std = 0., 0.
    args.opt_pose_coef, args.opt_pose_tol, args.opt_pose_lrate = coef, 0.0, lr
    arrays = fd.synthetic_arrays(n_images=n_images, H=64, W=64, seed=2)
    feed = fd.RayFeed.from_arrays(arrays, syn.NEAR, syn.FAR, N_rand=4 * rays_per_image, N_sample_images=4, device=DEV,
                                  seed=1, cam_idxs=np.arange(n_images) % 8)
    attrs = {"rest_pose": syn.rest_pose()[None], "betas": torch.zeros(1, 10).numpy(), "kp3d": arrays["kp3d"],
             "bones": arrays["bones"]}
    return args, feed, attrs, arrays


def _fresh(flags, args, attrs):
    """The seeded caster and a pose layer off its anchors (the regulariser is active)."""
    from danbo_b200 import pose_opt as po
    caster, _, _ = make_caster("danbo_fast", train=True, **flags)
    opt, kw = po.create_popt(args, attrs, device=DEV, flat=True)
    with torch.no_grad():
        kw["popt_layer"].bones[:, 1:] += 0.02
    return caster, opt, kw


def _vol_scale_loss(args, caster):
    gn = caster.network.graph_net
    if not getattr(args, "opt_vol_scale", False) or not gn.axis_scale.requires_grad:
        return 0.0
    s = gn.axis_scale.detach().double().abs().clamp(min=gn.init_scale.to(gn.axis_scale.device).double() * 0.05)
    return float((s[:, 0] * s[:, 1] * s[:, 2]).sum() * args.vol_scale_penalty)


def _train_once(flags, args, attrs, batch):
    from danbo_b200 import training
    caster, opt, kw = _fresh(flags, args, attrs)
    vol = _vol_scale_loss(args, caster)
    step = training.TrainStep(caster, args, graph=True, popt_kwargs=kw, pose_optimizer=opt)
    loss, _ = step._step(batch)
    torch.cuda.synchronize()
    return float(loss) - vol, opt.bucket.flat.clone()


def _fit_once(flags, args, attrs, batch, graph=False):
    from danbo_b200 import training
    caster, opt, kw = _fresh(flags, args, attrs)
    step = training.PoseFitStep(caster, args, kw, opt, graph=graph)
    loss, _ = step(batch)
    torch.cuda.synchronize()
    return float(loss), opt.bucket.flat.clone(), float(opt.step_dev)


@CONFIGS
def test_pose_gradient_equals_training_pose_gradient(flags):
    """One PoseFitStep against one uncaptured kernel-path TrainStep step from the same seeded state and batch: the pose
    gradient bucket agrees to the atomics' reordering, the loss is training's loss without vol_scale_loss."""
    args, feed, attrs, _ = _setup(flags)
    batch = feed.next_batch(torch.Generator(device=DEV).manual_seed(0))
    f1, f2 = _fit_once(flags, args, attrs, batch), _fit_once(flags, args, attrs, batch)
    t = _train_once(flags, args, attrs, batch)
    spread, err = _rel(f2[1], f1[1]), _rel(f1[1], t[1])
    loss_rel = abs(f1[0] - t[0]) / abs(t[0])
    print(f"[fit vs train {flags.get('ray_tr_type', 'world')}] loss {f1[0]:.7f} vs {t[0]:.7f} (rel {loss_rel:.1e}); "
          f"pose grads rel {err:.2e} (fit spread {spread:.2e})")
    assert float(f1[1].abs().max()) > 0
    assert err <= max(1e-4, 2 * spread)
    assert loss_rel <= 1e-6


@CONFIGS
def test_fitting_leaves_the_network_untouched(flags):
    from danbo_b200 import training
    args, feed, attrs, _ = _setup(flags)
    batch = feed.next_batch(torch.Generator(device=DEV).manual_seed(0))
    caster, opt, kw = _fresh(flags, args, attrs)
    net = caster.network
    marked = dict(net.named_parameters())["pts_linears.2.weight"]
    marked.grad = torch.randn_like(marked)                       # a gradient a user left behind must survive
    params = {n: p.detach().clone() for n, p in net.named_parameters()}
    grads = {n: (None if p.grad is None else p.grad.clone()) for n, p in net.named_parameters()}
    flags_rg = {n: p.requires_grad for n, p in net.named_parameters()}
    sd = {k: v.clone() for k, v in caster.state_dict()["network_fn_state_dict"].items()}
    poses = kw["popt_layer"].bones.detach().clone()
    step = training.PoseFitStep(caster, args, kw, opt, graph=True)
    for _ in range(10):
        step(batch)
    torch.cuda.synchronize()
    for n, p in net.named_parameters():
        assert torch.equal(p.detach(), params[n]), n
        assert (p.grad is None) if grads[n] is None else torch.equal(p.grad, grads[n]), n
        assert p.requires_grad == flags_rg[n], n
    assert all(torch.equal(v, sd[k]) for k, v in caster.state_dict()["network_fn_state_dict"].items())
    assert float(opt.step_dev) == 10.0
    assert float((kw["popt_layer"].bones.detach() - poses).abs().max()) > 0


@CONFIGS
def test_captured_step_equals_eager_step(flags):
    args, feed, attrs, _ = _setup(flags)
    batch = feed.next_batch(torch.Generator(device=DEV).manual_seed(0))
    e1, e2 = _fit_once(flags, args, attrs, batch), _fit_once(flags, args, attrs, batch)
    g = _fit_once(flags, args, attrs, batch, graph=True)
    spread, err = _rel(e2[1], e1[1]), _rel(g[1], e1[1])
    loss_rel = abs(g[0] - e1[0]) / abs(e1[0])
    print(f"[captured vs eager fit {flags.get('ray_tr_type', 'world')}] loss rel {loss_rel:.1e}; pose grads rel "
          f"{err:.2e} (eager spread {spread:.2e})")
    assert g[2] == 1.0                                           # capture applied no pose step
    assert err <= max(1e-4, 2 * spread)
    assert loss_rel <= 1e-6


@CONFIGS
def test_no_weight_gradient_work(flags):
    """The kernels of one eager fitting step: no wgrad / transpose / colsum / ray-bias backward launch, one Adam (the
    pose layer's), no weight pack once the pack is current.  TrainStep's own launch count is that of the parent
    commit."""
    from torch.profiler import profile, ProfilerActivity
    from danbo_b200 import kernels as K, training
    args, feed, attrs, _ = _setup(flags)
    batch = feed.next_batch(torch.Generator(device=DEV).manual_seed(0))
    caster, opt, kw = _fresh(flags, args, attrs)
    step = training.PoseFitStep(caster, args, kw, opt)
    step(batch)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step(batch)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    kern = [n for n in names if not (n.startswith("Memcpy") or n.startswith("Memset"))]
    tag = flags.get("ray_tr_type", "world")
    print(f"[fit launches {tag}] {len(kern)} kernels")
    for bad in ("wgrad", "transpose_kernel", "colsum", "ray_bias_bwd", "pack_dgrad", "pack_mlp"):
        assert not any(bad in n for n in kern), (bad, [n for n in kern if bad in n])
    assert sum("adam" in n for n in kern) == 1
    assert any("dgrad_kernel<false>" in n for n in kern) and not any("dgrad_kernel<true>" in n for n in kern)
    assert any("pair_logits_bwd_kernel<false, false>" in n for n in kern)
    gn = [n for n in kern if "gn::bwd_kernel<" in n]
    assert len(gn) == 3 and all(", false>" in n for n in gn), gn
    assert any("view_root_bwd" in n for n in kern) == (tag == "root_local")
    # training's launch sequence is unchanged
    caster, opt, kw = _fresh(flags, args, attrs)
    tstep = training.TrainStep(caster, args, graph=True, popt_kwargs=kw, pose_optimizer=opt)
    tstep._step(batch)
    K.PROFILE = {"mlp": [], "launches": 0}
    try:
        tstep._step(batch)
        torch.cuda.synchronize()
        n_train = K.PROFILE["launches"]
    finally:
        K.PROFILE = None
    print(f"[train launches {tag}] kernels._count {n_train} (parent commit: {TRAIN_LAUNCHES[tag]})")
    assert n_train == TRAIN_LAUNCHES[tag]


@CONFIGS
def test_kernel_variants_match_full_versions(flags, monkeypatch):
    """Inside one training backward (training-size blocks): the dX-only danbo_mlp_dgrad gives dX bit for bit, the
    pose-only danbo_field_agg_bwd gives d vol and d skts equal to the full call within the atomics' spread, and
    danbo_graph_net_bwd without grads gives `work`, then d pose bones, bit for bit."""
    from danbo_b200 import kernels as K, training
    args, feed, attrs, _ = _setup(flags)
    batch = feed.next_batch(torch.Generator(device=DEV).manual_seed(0))
    rec = {"mlp": [], "field": [], "gn": []}
    mlp_tc, field_bwd, gn_bwd, gn_pose = K.mlp_backward_tc, K.field_agg_bwd, K.graph_net_bwd, K.graph_net_bwd_pose

    def mlp_tc_rec(P, G, d_raw, active, fo, save, d_ray_bias, ws, **kw):
        dX = mlp_tc(P, G, d_raw, active, fo, save, d_ray_bias, ws, **kw)
        torch.cuda.synchronize()
        dX2 = K.mlp_backward_pose(P, d_raw, active, fo, save, K.PackedDgrad(d_raw.device).pack(P))
        torch.cuda.synchronize()
        rows = int(active.count)
        rec["mlp"].append((rows, dX[:rows].clone(), dX2[:rows].clone()))
        return dX

    def field_rec(rays, S, z, mask, active, pose_skts, pose_vol, rpp, consts, fo, dX, gl, grads, d_skts=None):
        torch.cuda.synchronize()
        outs = []
        for full in (True, True, False):
            g = [torch.zeros_like(t) for t in grads]
            if not full:
                g = [None] * 7 + [g[7], None]
            ds = torch.zeros_like(d_skts)
            field_bwd(rays, S, z, mask, active, pose_skts, pose_vol, rpp, consts, fo, dX, gl, g, d_skts=ds)
            torch.cuda.synchronize()
            outs.append((g[7], ds))
        rec["field"].append(outs)
        return field_bwd(rays, S, z, mask, active, pose_skts, pose_vol, rpp, consts, fo, dX, gl, grads, d_skts=d_skts)

    def gn_rec(saved, d_vol, grads):
        work = gn_bwd(saved, d_vol, grads)
        w_full = gn_bwd(saved, d_vol, [torch.zeros_like(g) for g in grads])
        w_pose = gn_bwd(saved, d_vol, None)
        rec["gn"].append((saved, w_full, w_pose))
        return work

    monkeypatch.setattr(K, "mlp_backward_tc", mlp_tc_rec)
    monkeypatch.setattr(K, "field_agg_bwd", field_rec)
    monkeypatch.setattr(K, "graph_net_bwd", gn_rec)
    caster, opt, kw = _fresh(flags, args, attrs)
    step = training.TrainStep(caster, args, graph=True, popt_kwargs=kw, pose_optimizer=opt)
    bones_seen = {}

    def gn_pose_rec(saved, work, pose_bones):
        bones_seen["b"] = pose_bones
        return gn_pose(saved, work, pose_bones)
    monkeypatch.setattr(K, "graph_net_bwd_pose", gn_pose_rec)
    step._step(batch)
    torch.cuda.synchronize()
    tag = flags.get("ray_tr_type", "world")
    assert len(rec["mlp"]) == 2 and len(rec["field"]) == 2 and len(rec["gn"]) == 1
    for rows, full, pose in rec["mlp"]:
        print(f"[dgrad variant {tag}] {rows} rows: dX bit-identical {torch.equal(full, pose)}")
        assert rows > 128 and torch.equal(full, pose)
    for (v1, s1), (v2, s2), (vp, sp) in rec["field"]:
        for nm, a, b, c in (("d vol", v1, v2, vp), ("d skts", s1, s2, sp)):
            spread, err = _rel(b, a), _rel(c, a)
            print(f"[field variant {tag}] {nm}: rel {err:.2e} (full-call spread {spread:.2e})")
            assert float(a.abs().max()) > 0 and err <= max(1e-6, 2 * spread), (nm, err, spread)
    saved, w_full, w_pose = rec["gn"][0]
    assert torch.equal(w_full, w_pose)
    b = bones_seen["b"]
    assert torch.equal(gn_pose(saved, w_full, b), gn_pose(saved, w_pose, b))


def _angle_err(bones, truth):
    """Mean geodesic angle (rad) between the non-root joint rotations of two (F,24,3) axis-angle tables."""
    from danbo_b200 import networks
    R, T = networks.axis_angle_to_matrix(bones[:, 1:].double()), networks.axis_angle_to_matrix(truth[:, 1:].double())
    tr = (R.transpose(-1, -2) @ T).diagonal(dim1=-2, dim2=-1).sum(-1)
    return float(torch.arccos(((tr - 1) / 2).clamp(-1, 1)).mean())


@CONFIGS
def test_fitting_recovers_perturbed_poses(flags):
    """A field trained for 400 iterations on synthetic images renders target images at the known poses (4 images x
    1 024 rays); the non-root axis-angles are perturbed by seeded N(0, 0.05 rad) noise and 50 captured fitting
    iterations (opt_pose_coef = 0, lr 1e-3) run on those targets.  The photometric loss and the mean joint-angle error
    of the fitted frames must both fall.  Measured on one B200 (1 000 W power limit): h36m_zju loss 0.2033 -> 0.1733,
    mean angle error 0.0831 -> 0.0780 rad; perfcap loss 0.2169 -> 0.2012, 0.0831 -> 0.0796 rad (both curves in
    profiles/r9_pose_fit_gpu_tests.txt).  (With 192 rays per batch most joints get almost no photometric gradient, and
    Adam moves every parameter by about lr per step whatever its gradient's size: those joints random-walk and the
    mean angle error grows while the loss falls.)"""
    from danbo_b200 import pose_opt as po, training
    args, feed, attrs, arrays = _setup(flags, coef=0.0, lr=1e-3, rays_per_image=1024)
    caster, _, _ = make_caster("danbo_fast", train=True, **flags)
    gen = torch.Generator(device=DEV).manual_seed(0)
    train = training.TrainStep(caster, args, graph=True)
    for _ in range(400):
        train(feed.next_batch(gen))
    torch.cuda.synchronize()
    batch = feed.next_batch(gen)
    frames = sorted(set(feed.last_idxs[0].tolist()))
    truth = torch.as_tensor(arrays["bones"], device=DEV).float()
    # targets: the frozen field at the known poses, on the batch's rays (cams < 0: the mean frame code)
    batch = dict(batch, cams=torch.full_like(batch["cams"], -1))
    with torch.no_grad():
        a = args
        preds = caster(batch["ray_batch"], N_samples=a.N_samples, kp_batch=batch["kp_batch"], skts=batch["skts"],
                       cyls=batch["cyls"], bones=batch["bones"], cams=batch["cams"], N_uniques=batch["N_uniques"],
                       perturb=0., N_importance=a.N_importance, raw_noise_std=0.)
        bgs = batch.get("bgs", 1.0)
        target = preds["rgb_map"] + (1. - preds["acc_map"])[..., None] * bgs
    batch["target_s"] = target.detach().clone()
    opt, kw = po.create_popt(args, attrs, device=DEV, flat=True)
    layer = kw["popt_layer"]
    with torch.no_grad():
        g = torch.Generator(device=DEV).manual_seed(7)
        layer.bones[:, 1:] += 0.05 * torch.randn(layer.bones[:, 1:].shape, device=DEV, generator=g)
    fit = training.PoseFitStep(caster, args, kw, opt, graph=True)
    losses, errs = [], [_angle_err(layer.bones.detach()[frames], truth[frames])]
    for _ in range(50):
        loss, _ = fit(batch)
        losses.append(float(loss))
        errs.append(_angle_err(layer.bones.detach()[frames], truth[frames]))
    torch.cuda.synchronize()
    tag = flags.get("ray_tr_type", "world")
    print(f"[fit {tag}] frames {frames}")
    print(f"[fit {tag}] loss  " + " ".join("%.5f" % v for v in losses[::5] + losses[-1:]))
    print(f"[fit {tag}] angle " + " ".join("%.4f" % v for v in errs[::5] + errs[-1:]))
    assert all(v == v for v in losses)
    assert losses[-1] < losses[0]
    assert errs[-1] < errs[0]


def test_checkpoints_between_fitting_and_training(tmp_path):
    from danbo_b200 import training
    args, feed, attrs, _ = _setup({})
    batch = feed.next_batch(torch.Generator(device=DEV).manual_seed(0))
    caster, opt, kw = _fresh({}, args, attrs)
    fit = training.PoseFitStep(caster, args, kw, opt, graph=True)
    for _ in range(3):
        fit(batch)
    path = os.path.join(tmp_path, "fit.tar")
    fit.save(path, 3)
    ck = torch.load(path, map_location="cpu", weights_only=False)
    assert ck["optimizer_state_dict"] is None and ck["network_fn_state_dict"] is not None
    caster2, opt2, kw2 = _fresh({}, args, attrs)
    train = training.TrainStep(caster2, args, graph=True, popt_kwargs=kw2, pose_optimizer=opt2)
    assert train.resume(ck) == 3
    assert float(opt2.step_dev) == 3.0
    for p, q in zip(kw["popt_layer"].parameters(), kw2["popt_layer"].parameters()):
        assert torch.equal(p.detach(), q.detach())
    assert torch.equal(opt.exp_avg, opt2.exp_avg) and torch.equal(opt.exp_avg_sq, opt2.exp_avg_sq)
    train(batch)
    path = os.path.join(tmp_path, "train.tar")
    train.save(path, 4)
    ck = torch.load(path, map_location="cpu", weights_only=False)
    caster3, opt3, kw3 = _fresh({}, args, attrs)
    fit3 = training.PoseFitStep(caster3, args, kw3, opt3)
    assert fit3.resume(ck) == 4
    assert float(opt3.step_dev) == 4.0
    for p, q in zip(kw2["popt_layer"].parameters(), kw3["popt_layer"].parameters()):
        assert torch.equal(p.detach(), q.detach())
    assert torch.equal(opt2.exp_avg, opt3.exp_avg)
    loss, _ = fit3(batch)
    assert float(loss) == float(loss) and float(opt3.step_dev) == 5.0
