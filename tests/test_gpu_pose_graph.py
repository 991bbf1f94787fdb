"""A captured --opt_pose training iteration on the GPU (run with -m gpu): the pose kernels (danbo_pose_fwd / _bwd,
danbo_graph_net_bwd_pose) against the reference's fixture and autograd, one graphed step against one eager step from
the same state and batch, graphed training with a feed, and checkpoints between the two paths."""
import os

import numpy as np
import pytest
import torch

from util import make_caster

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600, method="thread")]   # a hung kernel must not hang the box
DEV = "cuda"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FX = np.load(os.path.join(ROOT, "tests", "golden", "popt.npz"))
PERFCAP = dict(view_type="relray", ray_tr_type="root_local", nerf_type="graph")     # configs/perfcap/danbo_fast.txt


def _rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp(min=1e-30))


def _fixture_layer(tag):
    from danbo_b200 import pose_opt as po
    sd = {k[len(tag) + 4:]: torch.tensor(FX[k]) for k in FX.files if k.startswith(tag + ".sd.")}
    return po.load_poseopt_from_state_dict({"poseopt_layer_state_dict": sd}).to(DEV)


def _kernel_layer(layer):
    d = {n: p.detach() for n, p in layer.named_parameters()}
    d["rest_pose"] = layer.rest_pose
    if layer.kp_map is not None:
        d["kp_map"] = layer.kp_map
    return d


@pytest.mark.parametrize("tag", ["axisang", "multiview"])
def test_pose_kernels_match_the_reference_fixture(tag):
    """Kernel 1's kps / skts / bones against the reference's outputs, kernel 2's parameter gradients against the
    reference's own (taken with probe weights on kps and skts); frames that were not drawn get exactly zero."""
    from danbo_b200 import kernels as K
    layer = _fixture_layer(tag)
    L = _kernel_layer(layer)
    idx = torch.tensor(FX["idxs"], device=DEV)
    kps, bones, skts, stats = K.pose_fwd(L, idx, 1, len(idx))
    assert stats is None
    for nm, t in (("kps", kps), ("skts", skts), ("bones", bones)):
        ref = torch.tensor(FX[f"{tag}.out.{nm}"])
        err = float((t.cpu() - ref).abs().max())
        print(f"[pose fwd {tag}] {nm}: max abs err {err:.2e}")
        assert err <= 2e-6 * max(1.0, float(ref.abs().max())), (nm, err)
    g = torch.Generator().manual_seed(0)                                  # test_pose_opt._probe_weights
    wk, ws = torch.randn(len(idx), 24, 3, generator=g), torch.randn(len(idx), 24, 4, 4, generator=g)
    grads = {n: torch.zeros_like(p) for n, p in layer.named_parameters()}
    K.pose_bwd(L, idx, 1, len(idx), ws.to(DEV), grads, d_kps=wk.to(DEV))
    for nm, gr in grads.items():
        ref = torch.tensor(FX[f"{tag}.grad.{nm}"])
        err = float((gr.cpu() - ref).abs().max())
        print(f"[pose bwd {tag}] {nm}: max abs err {err:.2e} (scale {float(ref.abs().max()):.2e})")
        assert err <= 2e-5 * max(1.0, float(ref.abs().max())), (nm, err)
    # a draw of two frames, one of them twice: every other row of every gradient is exactly zero
    idx2 = torch.tensor([1, 4, 4], device=DEV)
    grads = {n: torch.zeros_like(p) for n, p in layer.named_parameters()}
    K.pose_bwd(L, idx2, 1, 3, ws[:3].to(DEV), grads, d_kps=wk[:3].to(DEV))
    rows = {"pelvis": [1, 4], "root_bones": [1, 4]}
    if layer.kp_map is not None:
        rows["bones"] = sorted(set(layer.kp_map[[1, 4]].tolist()))
    else:
        rows["bones"] = [1, 4]
    for nm, gr in grads.items():
        other = [i for i in range(gr.shape[0]) if i not in rows[nm]]
        assert torch.equal(gr[other], torch.zeros_like(gr[other])), nm
        assert float(gr[rows[nm]].abs().sum()) > 0, nm


def test_pose_kernels_with_regulariser_and_rest_table_match_autograd():
    """Kernels 1 and 2 with everything the training step hands them: a two-row rest-pose table indexed per frame, the
    regulariser and MPJPC against anchors, d bones, d kps and d kp_loss, duplicate and near-zero-angle poses; against
    fp64 autograd of `calculate_kinematic` + `kp_loss` on the same fp32 parameters."""
    import types
    from danbo_b200 import kernels as K, pose_opt as po
    g = torch.Generator().manual_seed(3)
    kps0, bones0 = torch.tensor(FX["init_kps"]), torch.tensor(FX["init_bones"])
    bones = bones0 + 0.03 * torch.randn(bones0.shape, generator=g)
    bones[2] *= 1e-8                                                      # the small-angle branch
    rest = torch.cat([torch.tensor(FX["rest_pose"]), torch.tensor(FX["rest_pose"]) * 1.1], 0)
    table = np.array([0, 1, 0, 1, 1, 0, 1])
    layer = po.PoseOptLayer(kps0, bones, rest, rest_pose_idxs=table).to(DEV)
    idxs = np.array([2, 3, 3, 5, 1, 6])
    G = len(idxs)
    args = types.SimpleNamespace(opt_rot6d=False, opt_pose_tol=5e-4, opt_pose_coef=2.0, use_temp_loss=False,
                                 ext_scale=0.001)
    L = _kernel_layer(layer)
    L["rest_idx"] = torch.tensor(table, device=DEV).long()
    idx = torch.tensor(idxs, device=DEV)
    anchors = {"kps": kps0.to(DEV).contiguous(), "bones": bones0.to(DEV).contiguous()}
    kps, kb, skts, stats = K.pose_fwd(L, idx, 1, G, anchors=anchors, tol=args.opt_pose_tol, coef=args.opt_pose_coef,
                                      ext_scale=args.ext_scale)
    ref = po.PoseOptLayer(kps0, bones, rest, rest_pose_idxs=table).double()
    rk, rb, rs, _, _ = ref.calculate_kinematic(idxs)
    a64 = {"kps": kps0.double(), "bones": bones0.double(), "rots": None}
    losses, st = po.kp_loss(args, a64, idxs, {"kp_batch": rk, "bones": rb, "rots": None})
    for nm, t, r in (("kps", kps, rk), ("skts", skts, rs), ("bones", kb, rb)):
        err = float((t.cpu().double() - r.detach()).abs().max())
        assert err <= 2e-6 * max(1.0, float(r.detach().abs().max())), (nm, err)
    reg, mpjpc = float(stats[0]), float(stats[1])
    print(f"[pose fwd, regulariser] kp_loss {reg:.7e} vs {float(losses['kp_loss']):.7e}; MPJPC {mpjpc:.5f} vs "
          f"{float(st['MPJPC']):.5f}")
    assert float(losses["kp_loss"]) > 0 and abs(reg - float(losses["kp_loss"])) <= 1e-5 * float(losses["kp_loss"])
    assert abs(mpjpc - float(st["MPJPC"])) <= 1e-5 * float(st["MPJPC"])
    wk, ws, wb = (torch.randn(G, 24, *s_, generator=g) for s_ in ((3,), (4, 4), (3,)))
    d_reg = 0.7
    ((rk * wk).sum() + (rs * ws).sum() + (rb * wb).sum() + d_reg * losses["kp_loss"]).backward()
    grads = {n: torch.zeros_like(p) for n, p in layer.named_parameters()}
    K.pose_bwd(L, idx, 1, G, ws.to(DEV), grads, d_bones=wb.to(DEV), d_kps=wk.to(DEV), anchor_bones=anchors["bones"],
               d_reg=torch.tensor(d_reg, device=DEV), tol=args.opt_pose_tol, coef=args.opt_pose_coef)
    for nm, p in ref.named_parameters():
        err = float((grads[nm].cpu().double() - p.grad).abs().max())
        print(f"[pose bwd, regulariser and rest table] {nm}: max abs err {err:.2e} (scale {float(p.grad.abs().max()):.2e})")
        assert err <= 2e-5 * max(1.0, float(p.grad.abs().max())), (nm, err)
    untouched = [i for i in range(7) if i not in idxs]
    assert torch.equal(grads["bones"][untouched], torch.zeros_like(grads["bones"][untouched]))


def test_graph_net_pose_gradient_matches_autograd():
    from danbo_b200 import autograd as ag, networks
    torch.manual_seed(0)
    net = networks.DanboField().to(DEV)
    G = 16
    aa = (torch.randn(G, 24, 3, device=DEV) * 0.6)
    aa[3, 7] *= 1e-8
    aa.requires_grad_(True)
    vol = ag.graph_net_volumes(net, aa)
    d_vol = torch.randn_like(vol)
    (vol * d_vol).sum().backward()
    got = aa.grad.detach().cpu().double()
    gn = networks.GraphNet().double()
    gn.load_state_dict({k: v.double().cpu() for k, v in net.graph_net.state_dict().items()})
    ref_aa = aa.detach().cpu().double().requires_grad_(True)
    w = networks.pe_embed(networks.axis_angle_to_matrix(ref_aa)[..., :3, :2].flatten(start_dim=-2), 5)
    (gn(w) * d_vol.cpu().double()).sum().backward()
    assert torch.equal(got[:, 0], torch.zeros_like(got[:, 0]))
    worst = max(_rel(got[g], ref_aa.grad[g]) for g in range(G))
    print(f"[graph net d pose] worst per-pose rel {worst:.2e}")
    assert worst <= 1e-5, worst


def _setup(flags, coef=1.0, lr=1e-3, n_images=12):
    import danbo_b200 as db
    from danbo_b200 import feed as fd, synthetic as syn
    args = db.make_args("danbo_fast", no_reload=True, opt_pose=True, **flags)
    args.perturb, args.raw_noise_std = 0., 0.
    args.opt_pose_coef, args.opt_pose_tol, args.opt_pose_lrate = coef, 0.0, lr
    arrays = fd.synthetic_arrays(n_images=n_images, H=64, W=64, seed=2)
    feed = fd.RayFeed.from_arrays(arrays, syn.NEAR, syn.FAR, N_rand=4 * 48, N_sample_images=4, device=DEV, seed=1,
                                  cam_idxs=np.arange(n_images) % 8)
    attrs = {"rest_pose": syn.rest_pose()[None], "betas": torch.zeros(1, 10).numpy(), "kp3d": arrays["kp3d"],
             "bones": arrays["bones"]}
    return args, feed, attrs


def _one_step(flags, args, attrs, batch, mode, nudge=0.0):
    """One training step from a fresh, seeded state.  mode: "torch" (eager TrainStep: the PyTorch pose ops), "kernel"
    (what TrainStep(graph=True) captures, run without capture) or "graph" (the captured step, replayed once).
    nudge: relative size of a seeded random change of the pose parameters, a few fp32 ulps."""
    from danbo_b200 import pose_opt as po, training
    caster, _, _ = make_caster("danbo_fast", train=True, **flags)
    opt, kw = po.create_popt(args, attrs, device=DEV, flat=True)
    layer = kw["popt_layer"]
    with torch.no_grad():
        layer.bones[:, 1:] += 0.02                          # off the anchors: the regulariser is active
        g = torch.Generator(device=DEV).manual_seed(5)
        for p in layer.parameters():
            p.mul_(1 + nudge * torch.randn(p.shape, device=DEV, generator=g))
    before = {n: p.detach().clone() for n, p in layer.named_parameters()}
    step = training.TrainStep(caster, args, graph=mode != "torch", popt_kwargs=kw, pose_optimizer=opt)
    loss, _ = step._step(batch) if mode == "kernel" else step(batch)
    torch.cuda.synchronize()
    after = {n: p.detach().clone() for n, p in layer.named_parameters()}
    return (float(loss), step.bucket.flat.clone(), opt.bucket.flat.clone(), before, after,
            float(opt.step_dev), float(step.optimizer.step_dev), float(step.last_stats["MPJPC"]))


def _cos(a, b):
    a, b = a.reshape(-1).double(), b.reshape(-1).double()
    return float(torch.dot(a, b) / (a.norm() * b.norm() + 1e-30))


@pytest.mark.parametrize("flags", [{}, PERFCAP], ids=["h36m_zju", "perfcap"])
def test_graphed_step_matches_eager_step(flags):
    """The captured step against the same step run without capture (the pose kernels and the fused graph net in
    both): loss, gradients and the poses after the step agree to the atomics' reordering, and capture applied no extra
    step.  Then the kernel path against the eager PyTorch pose path.  The two compute skts and the graph net's features
    in different fp32 orders, and the render amplifies such last-bit differences (a sample near a bone box's face or a
    bf16 rounding boundary changes side), so that comparison is bounded by the same path's own sensitivity: the eager
    step with the pose parameters nudged by 3e-7 relative."""
    args, feed, attrs = _setup(flags)
    batch = feed.next_batch(torch.Generator(device=DEV).manual_seed(0))
    k1 = _one_step(flags, args, attrs, batch, "kernel")
    k2 = _one_step(flags, args, attrs, batch, "kernel")
    g = _one_step(flags, args, attrs, batch, "graph")
    t = _one_step(flags, args, attrs, batch, "torch")
    tn = _one_step(flags, args, attrs, batch, "torch", nudge=3e-7)
    tag = flags.get("ray_tr_type", "world")
    assert g[5] == 1.0 and g[6] == 1.0                       # one step of each optimiser: capture applied none
    loss_rel = abs(g[0] - k1[0]) / abs(k1[0])
    net_spread, pose_spread = _rel(k2[1], k1[1]), _rel(k2[2], k1[2])
    net_rel, pose_rel = _rel(g[1], k1[1]), _rel(g[2], k1[2])
    print(f"[graphed vs uncaptured {tag}] loss {g[0]:.7f} vs {k1[0]:.7f} (rel {loss_rel:.1e}); network grads rel "
          f"{net_rel:.2e} (uncaptured spread {net_spread:.2e}); pose grads rel {pose_rel:.2e} (spread {pose_spread:.2e})")
    t_loss = abs(t[0] - k1[0]) / abs(t[0])
    t_net, t_pose = _rel(k1[1], t[1]), _rel(k1[2], t[2])
    c_net, c_pose = _cos(k1[1], t[1]), _cos(k1[2], t[2])
    f_loss, f_net, f_pose = abs(tn[0] - t[0]) / abs(t[0]), _rel(tn[1], t[1]), _rel(tn[2], t[2])
    print(f"[kernels vs PyTorch pose ops {tag}] loss {k1[0]:.7f} vs {t[0]:.7f} (rel {t_loss:.1e}); network grads rel "
          f"{t_net:.2e} cos {c_net:.6f}; pose grads rel {t_pose:.2e} cos {c_pose:.6f}; MPJPC {k1[7]:.5f} vs {t[7]:.5f}")
    print(f"[PyTorch pose ops, poses nudged by 3e-7 {tag}] loss rel {f_loss:.1e}; network grads rel {f_net:.2e} cos "
          f"{_cos(tn[1], t[1]):.6f}; pose grads rel {f_pose:.2e} cos {_cos(tn[2], t[2]):.6f}")
    assert loss_rel <= 1e-6
    assert net_rel <= max(1e-4, 2 * net_spread)
    assert pose_rel <= max(1e-4, 2 * pose_spread)
    lr = args.opt_pose_lrate
    for n in g[4]:
        moved = float((g[4][n] - g[3][n]).abs().max())
        diff = float((g[4][n] - k1[4][n]).abs().max())
        assert 0.5 * lr < moved < 1.5 * lr, (n, moved)        # one Adam step moves a parameter by at most ~lr
        assert diff <= 0.5 * lr, (n, diff)
    # the poses after the step: one Adam step moves an entry by about lr in the direction of its gradient's sign
    p_diff = max(float((k1[4][n] - t[4][n]).abs().mean()) for n in t[4]) / lr
    p_floor = max(float((tn[4][n] - t[4][n]).abs().mean()) for n in t[4]) / lr
    print(f"[kernels vs PyTorch pose ops {tag}] poses after the step: mean |diff| {p_diff:.3f} lr (nudged eager: "
          f"{p_floor:.3f} lr)")
    assert abs(k1[7] - t[7]) <= 1e-5 * abs(t[7])
    assert t_loss <= 3 * f_loss + 1e-6, (t_loss, f_loss)
    assert t_net <= 3 * f_net + 1e-4 and t_pose <= 3 * f_pose + 1e-4, (t_net, f_net, t_pose, f_pose)
    assert c_net >= 1 - 3 * (1 - _cos(tn[1], t[1])) - 1e-6 and c_pose >= 1 - 3 * (1 - _cos(tn[2], t[2])) - 1e-6
    assert p_diff <= 3 * p_floor + 0.01, (p_diff, p_floor)


@pytest.mark.parametrize("flags", [{}, PERFCAP], ids=["h36m_zju", "perfcap"])
def test_step_pose_gradient_wiring(flags, monkeypatch):
    """Inside one training step on the kernel path: the d bones that reach danbo_pose_bwd are the graph net's d pose
    (danbo_graph_net_bwd_pose), d kp_loss is 1, and the pose layer's gradient bucket equals fp64 autograd of
    `calculate_kinematic` + `kp_loss` seeded with the very d skts / d bones the render's backward produced (on perfcap
    these include danbo_view_root_bwd's share of joint 0)."""
    from danbo_b200 import kernels as K, pose_opt as po, training
    args, feed, attrs = _setup(flags, coef=2.0)
    batch = feed.next_batch(torch.Generator(device=DEV).manual_seed(0))
    rec = {}
    pose_bwd, gn_pose = K.pose_bwd, K.graph_net_bwd_pose

    def rec_pose_bwd(layer, idx, stride, G, d_skts, grads, **kw):
        rec.update(idx=idx[::stride][:G].cpu(), d_skts=d_skts.clone(), **{k: (v.clone() if torch.is_tensor(v) else v)
                                                                            for k, v in kw.items()})
        return pose_bwd(layer, idx, stride, G, d_skts, grads, **kw)

    def rec_gn_pose(*a):
        rec["gn"] = gn_pose(*a)
        return rec["gn"]
    monkeypatch.setattr(K, "pose_bwd", rec_pose_bwd)
    monkeypatch.setattr(K, "graph_net_bwd_pose", rec_gn_pose)
    caster, _, _ = make_caster("danbo_fast", train=True, **flags)
    opt, kw = po.create_popt(args, attrs, device=DEV, flat=True)
    layer = kw["popt_layer"]
    with torch.no_grad():
        layer.bones[:, 1:] += 0.02 * torch.randn(layer.bones[:, 1:].shape, device=DEV,
                                                 generator=torch.Generator(device=DEV).manual_seed(1))
    ref = po.load_poseopt_from_state_dict({"poseopt_layer_state_dict": {k: v.cpu() for k, v in layer.state_dict().items()}})
    ref = ref.double()
    step = training.TrainStep(caster, args, graph=True, popt_kwargs=kw, pose_optimizer=opt)
    step._step(batch)
    torch.cuda.synchronize()
    assert float(rec["d_reg"]) == 1.0
    assert torch.equal(rec["d_bones"], rec["gn"])
    d_skts = rec["d_skts"].cpu().double()
    assert float(d_skts[:, 0, :3, :3].abs().max()) > 0
    idxs = rec["idx"].numpy()
    rk, rb, rs, _, _ = ref.calculate_kinematic(idxs)
    a = kw["popt_anchors"]
    losses, _ = po.kp_loss(args, {"kps": a["kps"].cpu().double(), "bones": a["bones"].cpu().double(), "rots": None},
                           idxs, {"kp_batch": rk, "bones": rb, "rots": None})
    total = (rs * d_skts).sum() + (rb * rec["d_bones"].cpu().double()).sum() + losses["kp_loss"]
    if rec["d_kps"] is not None:
        total = total + (rk * rec["d_kps"].cpu().double()).sum()
    total.backward()
    off = 0
    for (nm, p), q in zip(ref.named_parameters(), layer.parameters()):
        got = opt.bucket.flat[off:off + q.numel()].view_as(q).cpu().double()
        off += q.numel()
        err = _rel(got, p.grad)
        print(f"[step wiring {flags.get('ray_tr_type', 'world')}] d {nm}: rel {err:.2e} against fp64 autograd "
              f"(|g| {float(p.grad.norm()):.3e})")
        assert err <= 2e-5, (nm, err)


def test_graphed_training_with_a_feed():
    """20 graphed iterations: with opt_pose_coef = 0 exactly the frames drawn move; the loss falls on a repeated batch;
    both optimisers count 20 steps."""
    from danbo_b200 import pose_opt as po, training
    n_images = 12
    args, feed, attrs = _setup(PERFCAP, coef=0.0, n_images=n_images)
    caster, _, _ = make_caster("danbo_fast", train=True, **PERFCAP)
    opt, kw = po.create_popt(args, attrs, device=DEV, flat=True)
    layer = kw["popt_layer"]
    before = layer.bones.detach().clone()
    step = training.TrainStep(caster, args, graph=True, popt_kwargs=kw, pose_optimizer=opt)
    gen = torch.Generator(device=DEV).manual_seed(0)
    touched = set()
    for _ in range(2):
        batch = feed.next_batch(gen)
        touched.update(feed.last_idxs[0].tolist())
        step(batch)
    torch.cuda.synchronize()
    moved = (layer.bones.detach() - before).abs().amax(dim=(1, 2)).cpu()
    print("[graphed popt] touched", sorted(touched), "moved", [f"{float(v):.1e}" for v in moved])
    assert len(touched) < n_images
    for i in range(n_images):
        assert (float(moved[i]) > 0) == (i in touched), (i, float(moved[i]), sorted(touched))
    losses = [float(step(batch)[0]) for _ in range(18)]
    torch.cuda.synchronize()
    print("[graphed popt] losses", ["%.4f" % v for v in losses])
    assert all(v == v for v in losses) and losses[-1] < losses[0]
    assert float(opt.step_dev) == 20.0 and float(step.optimizer.step_dev) == 20.0
    assert bool(torch.isfinite(layer.bones).all()) and bool(torch.isfinite(layer.pelvis).all())


def test_checkpoints_between_graphed_and_eager(tmp_path):
    from danbo_b200 import pose_opt as po, training
    args, feed, attrs = _setup({})
    gen = torch.Generator(device=DEV).manual_seed(0)
    batch = feed.next_batch(gen)
    # graphed -> the reference's torch.optim.Adam over the layer's parameters
    caster, _, _ = make_caster("danbo_fast", train=True)
    opt, kw = po.create_popt(args, attrs, device=DEV, flat=True)
    step = training.TrainStep(caster, args, graph=True, popt_kwargs=kw, pose_optimizer=opt)
    for _ in range(3):
        step(batch)
    path = os.path.join(tmp_path, "graphed.tar")
    step.save(path, 3)
    ck = torch.load(path, map_location="cpu", weights_only=False)
    _, kw2 = po.create_popt(args, attrs, ckpt=ck)
    adam = torch.optim.Adam(list(kw2["popt_layer"].parameters()), lr=args.opt_pose_lrate)
    adam.load_state_dict(ck["pose_optimizer_state_dict"])
    for i, p in enumerate(kw["popt_layer"].parameters()):
        st = adam.state[list(kw2["popt_layer"].parameters())[i]]
        assert float(st["step"]) == 3.0
        assert torch.equal(st["exp_avg"], opt.exp_avg[sum(q.numel() for q in list(kw["popt_layer"].parameters())[:i]):][:p.numel()].view_as(p).cpu())
        assert torch.equal(kw2["popt_layer"].state_dict()[[n for n, _ in kw["popt_layer"].named_parameters()][i]],
                           p.detach().cpu())
    # eager with torch.optim.Adam -> resumed under graph capture
    caster, _, _ = make_caster("danbo_fast", train=True)
    opt_e, kw_e = po.create_popt(args, attrs, device=DEV)
    step_e = training.TrainStep(caster, args, popt_kwargs=kw_e, pose_optimizer=opt_e)
    for _ in range(2):
        step_e(batch)
    path = os.path.join(tmp_path, "eager.tar")
    step_e.save(path, 2)
    ck = torch.load(path, map_location="cpu", weights_only=False)
    caster, _, _ = make_caster("danbo_fast", train=True)
    opt_g, kw_g = po.create_popt(args, attrs, device=DEV, ckpt=ck, flat=True)
    step_g = training.TrainStep(caster, args, graph=True, popt_kwargs=kw_g, pose_optimizer=opt_g)
    assert step_g.resume(ck) == 2
    assert float(opt_g.step_dev) == 2.0
    for i, p in enumerate(kw_e["popt_layer"].parameters()):
        q = list(kw_g["popt_layer"].parameters())[i]
        assert torch.equal(p.detach(), q.detach())
        assert torch.equal(opt_e.state[p]["exp_avg"], opt_g.exp_avg[sum(r.numel() for r in list(kw_g["popt_layer"].parameters())[:i]):][:q.numel()].view_as(q))
    loss, _ = step_g(batch)
    torch.cuda.synchronize()
    assert float(loss) == float(loss) and float(opt_g.step_dev) == 3.0
