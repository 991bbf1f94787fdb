"""The 2D keypoint reprojection term on the GPU (run with -m gpu): danbo_pose_kp2d against its fp64 twin
(pose_opt.kp2d_loss), the pose-parameter gradient of the term through the pose layer against fp64 autograd, the captured
PoseFitStep / TrainStep against their uncaptured runs with the term on, a fit of perturbed limbs to projected
keypoints, and steps without the term running the launches they ran before the term existed."""
import numpy as np
import pytest
import torch

from test_kp2d_cpu import _scene
from util import make_caster

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900, method="thread")]   # a hung kernel must not hang the box
DEV = "cuda"
PERFCAP = dict(view_type="relray", ray_tr_type="root_local", nerf_type="graph")     # configs/perfcap/danbo_fast.txt
CONFIGS = pytest.mark.parametrize("flags", [{}, PERFCAP], ids=["h36m_zju", "perfcap"])
# kernels._count of one uncaptured step with a pose layer and a batch without 2D keypoints, as measured on the parent
# commit of the 2D keypoint term on a B200: the launch sequence of such a step must not change.
TRAIN_LAUNCHES = {"world": 58, "root_local": 59}
FIT_LAUNCHES = {"world": 39, "root_local": 42}
# The loss of one captured step of that batch from the seeded state of _fresh, as the parent commit computes it on a
# B200 (bit for bit the same in every run there)
PARENT_LOSS = {("fit", "world"): 0.6799911856651306, ("train", "world"): 0.6801741123199463,
               ("fit", "root_local"): 0.6797281503677368, ("train", "root_local"): 0.6799110770225525}
LIMBS = [1, 2, 4, 5, 7, 8, 16, 17, 18, 19, 20, 21]          # SMPL hips, knees, ankles, shoulders, elbows, wrists


def _rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp(min=1e-30))


@pytest.mark.parametrize("G,sigma,coef", [(1, 100., 1.0), (5, 30., 0.5), (37, 100., 2.0)])
def test_kernel_matches_fp64_twin(G, sigma, coef):
    from danbo_b200 import kernels as K, pose_opt as po
    kps, kp2d, proj = _scene(G=G, seed=G, at_centre=False)
    k32, d32, p32 = (t.float().to(DEV).contiguous() for t in (kps, kp2d, proj))
    loss, px, d_kps = K.pose_kp2d(k32, d32, p32, sigma, coef)
    torch.cuda.synchronize()
    x = k32.double().cpu().requires_grad_(True)
    r_loss, r_px = po.kp2d_loss(x, d32.double().cpu(), p32.double().cpu(), sigma, coef)
    r_loss.backward()
    ref = x.grad
    l_rel = abs(float(loss) - float(r_loss.detach())) / abs(float(r_loss.detach()))
    p_rel = abs(float(px) - float(r_px)) / abs(float(r_px))
    d_err = float((d_kps.cpu().double() - ref).abs().max()) / float(ref.abs().max())
    print(f"[kp2d kernel G={G}] loss rel {l_rel:.1e}; kp2d_px rel {p_rel:.1e}; d kps max err / scale {d_err:.1e}")
    assert l_rel <= 1e-5 and p_rel <= 1e-5 and d_err <= 1e-5
    # joints behind the camera (w <= 1e-6) and joints with c = 0: exactly 0
    X = torch.cat([k32, torch.ones_like(k32[..., :1])], -1)
    w = torch.einsum("gc,gjc->gj", p32[:, 2], X)
    dead = (w <= 1e-6) | (d32[..., 2] == 0)
    assert bool(dead.any()) and torch.equal(d_kps[dead], torch.zeros_like(d_kps[dead]))


def _layer(kind):
    """A pose layer of 7 synthetic frames: a two-row rest-pose table indexed per frame, or the multi-view split
    (kp_map)."""
    from danbo_b200 import pose_opt as po, synthetic as syn
    poses = [syn.make_pose(40 + f) for f in range(7)]
    kps0 = torch.tensor(np.stack([p["kps"] for p in poses]))
    bones0 = torch.tensor(np.stack([p["bones"] for p in poses]))
    rest = torch.tensor(syn.rest_pose())[None]
    kw = {}
    if kind == "rest_table":
        rest = torch.cat([rest, rest * 1.1], 0)
        kw["rest_pose_idxs"] = np.array([0, 1, 0, 1, 1, 0, 1])
    else:
        kw["kp_map"], kw["kp_uidxs"] = np.array([0, 1, 1, 2, 0, 2, 1]), np.array([0, 1, 3])
    return po.PoseOptLayer(kps0, bones0, rest, **kw), kps0, bones0, kw


@pytest.mark.parametrize("kind", ["rest_table", "kp_map"])
def test_pose_layer_gradient_of_the_term(kind):
    """autograd.pose_layer -> autograd.pose_kp2d -> backward (danbo_pose_fwd, danbo_pose_kp2d, danbo_pose_bwd with the
    term's d kps) against fp64 autograd through calculate_kinematic + kp2d_loss, the 2D term alone."""
    from danbo_b200 import autograd as ag, pose_opt as po, render, synthetic as syn
    layer, kps0, bones0, kw = _layer(kind)
    ref = po.PoseOptLayer(kps0, bones0, layer.rest_pose.clone(), **kw).double()
    ref.load_state_dict({k: v.double() for k, v in layer.state_dict().items()})
    layer = layer.to(DEV)
    idxs = np.array([2, 3, 3, 5, 1, 6])
    G = len(idxs)
    g = torch.Generator().manual_seed(4)
    with torch.no_grad():
        truth = ref.calculate_kinematic(idxs)[0]
    proj = torch.tensor(render.projection_matrix(syn.bullet_time_cameras(syn.camera(), G), 256, 256, 307.2))
    X = torch.cat([truth, torch.ones_like(truth[..., :1])], -1)
    h = torch.einsum("grc,gjc->gjr", proj, X)
    det = h[..., :2] / h[..., 2:] + 20 * torch.randn(G, 24, 2, generator=g, dtype=torch.float64)
    kp2d = torch.cat([det, torch.rand(G, 24, 1, generator=g, dtype=torch.float64)], -1).float()
    proj = proj.float()
    sigma, coef = 50., 1.5
    rest_idx = torch.as_tensor(kw["rest_pose_idxs"], device=DEV).long() if kind == "rest_table" else None
    anchors = {"kps": kps0.to(DEV).contiguous(), "bones": bones0.to(DEV).contiguous()}
    kps, _, _, _, _ = ag.pose_layer(layer, torch.tensor(idxs, device=DEV), 1, G, anchors, rest_idx=rest_idx)
    loss, px = ag.pose_kp2d(kps, kp2d.to(DEV), proj.to(DEV), sigma, coef)
    loss.backward()
    rk = ref.calculate_kinematic(idxs)[0]
    r_loss, r_px = po.kp2d_loss(rk, kp2d.double(), proj.double(), sigma, coef)
    r_loss.backward()
    print(f"[kp2d through the pose layer, {kind}] loss {float(loss.detach()):.6e} vs {float(r_loss):.6e}; kp2d_px {float(px):.4f}")
    assert abs(float(loss) - float(r_loss)) <= 1e-5 * abs(float(r_loss))
    for nm, p in ref.named_parameters():
        got = dict(layer.named_parameters())[nm].grad
        err = float((got.cpu().double() - p.grad).abs().max())
        print(f"[kp2d through the pose layer, {kind}] {nm}: max abs err {err:.2e} (scale {float(p.grad.abs().max()):.2e})")
        assert float(p.grad.abs().max()) > 0
        assert err <= 2e-5 * max(1.0, float(p.grad.abs().max())), (nm, err)


def _setup(flags, n_images=12, rays_per_image=48, H=64, kp2d_coef=1.0, lr=1e-3, opt_pose_coef=1.0):
    import danbo_b200 as db
    from danbo_b200 import feed as fd, synthetic as syn
    args = db.make_args("danbo_fast", no_reload=True, opt_pose=True, kp2d_coef=kp2d_coef, kp2d_sigma=100., **flags)
    args.perturb, args.raw_noise_std = 0., 0.
    args.opt_pose_coef, args.opt_pose_tol, args.opt_pose_lrate = opt_pose_coef, 0.0, lr
    arrays = fd.synthetic_arrays(n_images=n_images, H=H, W=H, seed=2)
    feed = fd.RayFeed.from_arrays(arrays, syn.NEAR, syn.FAR, N_rand=4 * rays_per_image, N_sample_images=4, device=DEV,
                                  seed=1, cam_idxs=np.arange(n_images) % 8)
    attrs = {"rest_pose": syn.rest_pose()[None], "betas": torch.zeros(1, 10).numpy(), "kp3d": arrays["kp3d"],
             "bones": arrays["bones"]}
    return args, feed, attrs, arrays


def _detections(layer, arrays, frames, H, noise=0.0, seed=0):
    """Keypoints of the layer's current poses of `frames`, projected through the frames' cameras (+ seeded pixel noise,
    confidence 1) and the projection matrices: the batch keys kp2d, kp2d_proj."""
    from danbo_b200 import render
    with torch.no_grad():
        kps = layer.calculate_kinematic(np.asarray(frames))[0].double().cpu()
    proj = torch.tensor(render.projection_matrix(arrays["c2ws"][frames], H, H, float(arrays["focals"][0])))
    X = torch.cat([kps, torch.ones_like(kps[..., :1])], -1)
    h = torch.einsum("grc,gjc->gjr", proj, X)
    uv = h[..., :2] / h[..., 2:]
    uv = uv + noise * torch.randn(uv.shape, generator=torch.Generator().manual_seed(seed), dtype=torch.float64)
    kp2d = torch.cat([uv, torch.ones_like(uv[..., :1])], -1)
    return {"kp2d": kp2d.float().to(DEV), "kp2d_proj": proj.float().to(DEV)}


def _fresh(flags, args, attrs):
    from danbo_b200 import pose_opt as po
    caster, _, _ = make_caster("danbo_fast", train=True, **flags)
    opt, kw = po.create_popt(args, attrs, device=DEV, flat=True)
    with torch.no_grad():
        kw["popt_layer"].bones[:, 1:] += 0.02
    return caster, opt, kw


def _batch_with_detections(flags, args, attrs, arrays, feed):
    batch = feed.next_batch(torch.Generator(device=DEV).manual_seed(0))
    frames = feed.last_idxs[0].cpu().numpy()
    _, _, kw = _fresh(flags, args, attrs)
    # detections 8 px off the true projections of the anchors; the layer starts 0.02 rad off them
    with torch.no_grad():
        kw["popt_layer"].bones[:, 1:] -= 0.02
    return dict(batch, **_detections(kw["popt_layer"], arrays, frames, 64, noise=8.0))


def _run(flags, args, attrs, batch, kind, mode, steps=3):
    """`steps` iterations of a fresh, seeded step.  kind: "fit" (PoseFitStep) or "train" (TrainStep with a pose layer);
    mode: "graph" (captured, replayed) or "kernel" (the same function run without capture)."""
    from danbo_b200 import training
    caster, opt, kw = _fresh(flags, args, attrs)
    if kind == "fit":
        step = training.PoseFitStep(caster, args, kw, opt, graph=mode == "graph")
        call = step
    else:
        step = training.TrainStep(caster, args, graph=True, popt_kwargs=kw, pose_optimizer=opt)

        def call(b):
            if mode == "graph":
                return step(b)
            out = step._step({k: v for k, v in b.items() if k not in ("kp_batch", "skts", "bones")})
            step._after_step()
            return out
    losses, px = [], []
    for _ in range(steps):
        loss, _ = call(batch)
        losses.append(float(loss))
        px.append(float(step.last_stats["kp2d_px"]))
    torch.cuda.synchronize()
    poses = {n: p.detach().clone() for n, p in kw["popt_layer"].named_parameters()}
    return losses, px, poses, float(opt.step_dev)


@pytest.mark.parametrize("kind", ["fit", "train"])
@CONFIGS
def test_captured_step_equals_uncaptured_with_the_term(flags, kind):
    args, feed, attrs, arrays = _setup(flags)
    batch = _batch_with_detections(flags, args, attrs, arrays, feed)
    e1, e2 = _run(flags, args, attrs, batch, kind, "kernel"), _run(flags, args, attrs, batch, kind, "kernel")
    g = _run(flags, args, attrs, batch, kind, "graph")
    tag = flags.get("ray_tr_type", "world")
    lr = args.opt_pose_lrate
    spread = max(float((e2[2][n] - e1[2][n]).abs().max()) for n in e1[2])
    diff = max(float((g[2][n] - e1[2][n]).abs().max()) for n in e1[2])
    print(f"[captured vs uncaptured {kind} {tag}] losses {g[0]} vs {e1[0]}; kp2d_px {g[1]} vs {e1[1]}; poses after 3 "
          f"steps max |diff| {diff / lr:.3f} lr (uncaptured spread {spread / lr:.3f} lr)")
    assert g[3] == 3.0 and e1[3] == 3.0                             # capture applied no pose step
    assert abs(g[0][0] - e1[0][0]) <= 1e-6 * abs(e1[0][0])
    assert abs(g[1][0] - e1[1][0]) <= 1e-6 * abs(e1[1][0])
    assert e1[1][0] > 1.0                                           # the term is active: pixels off the detections
    assert diff <= max(0.5 * lr, 2 * spread)


def _count_launches(fn):
    from danbo_b200 import kernels as K
    K.PROFILE = {"mlp": [], "launches": 0}
    try:
        fn()
        torch.cuda.synchronize()
        return K.PROFILE["launches"]
    finally:
        K.PROFILE = None


@CONFIGS
def test_no_change_without_the_term(flags):
    """A batch without 2D keypoints runs the launches it ran before the term existed (kernels._count, measured on the
    parent commit) and gives the parent commit's loss bit for bit; a batch that carries them with kp2d_coef = 0 runs the
    same launches with the same loss.  The pose update is formed from atomically added gradients, so it is compared
    within the run-to-run spread (on a B200 up to 3e-8 after one step, the same on the parent commit).  With the term on,
    a fitting step runs one launch more (danbo_pose_kp2d: its gradient rides on danbo_pose_bwd's d_kps)."""
    from danbo_b200 import training
    tag = flags.get("ray_tr_type", "world")
    args, feed, attrs, arrays = _setup(flags, kp2d_coef=0.0)
    batch = _batch_with_detections(flags, args, attrs, arrays, feed)
    plain = {k: v for k, v in batch.items() if k not in training.KP2D_KEYS}
    strip = lambda b: {k: v for k, v in b.items() if k not in ("kp_batch", "skts", "bones")}
    for kind in ("fit", "train"):
        counts, results = {}, {}
        for name, b in (("plain", plain), ("plain again", plain), ("keys, coef 0", batch)):
            caster, opt, kw = _fresh(flags, args, attrs)
            if kind == "fit":
                step = training.PoseFitStep(caster, args, kw, opt)
                step(b)                                             # first call: weight packs
                counts[name] = _count_launches(lambda: step(b))
                caster, opt, kw = _fresh(flags, args, attrs)
                step = training.PoseFitStep(caster, args, kw, opt, graph=True)
            else:
                step = training.TrainStep(caster, args, graph=True, popt_kwargs=kw, pose_optimizer=opt)
                step._step(strip(b))
                counts[name] = _count_launches(lambda: step._step(strip(b)))
                caster, opt, kw = _fresh(flags, args, attrs)
                step = training.TrainStep(caster, args, graph=True, popt_kwargs=kw, pose_optimizer=opt)
            loss, _ = step(b)
            torch.cuda.synchronize()
            results[name] = (float(loss), torch.cat([p.detach().reshape(-1) for p in kw["popt_layer"].parameters()]),
                             sorted(step.last_stats))
        want = (FIT_LAUNCHES if kind == "fit" else TRAIN_LAUNCHES)[tag]
        (l0, p0, s0), (l1, p1, _), (l2, p2, s2) = results["plain"], results["plain again"], results["keys, coef 0"]
        spread, diff = float((p1 - p0).abs().max()), float((p2 - p0).abs().max())
        print(f"[no term {kind} {tag}] launches {counts} (parent commit: {want}); losses {l0!r} {l1!r} {l2!r}; poses "
              f"after the step max |diff| {diff:.3e} (plain vs plain {spread:.3e})")
        assert counts["plain"] == counts["plain again"] == counts["keys, coef 0"] == want
        assert s0 == s2 == ["MPJPC"]
        assert l0 == l1 == l2 == PARENT_LOSS[kind, tag]
        assert diff <= max(2 * spread, 2e-7)
    args.kp2d_coef = 1.0
    caster, opt, kw = _fresh(flags, args, attrs)
    step = training.PoseFitStep(caster, args, kw, opt)
    step(batch)
    n_on = _count_launches(lambda: step(batch))
    print(f"[term on, fit {tag}] kernels._count {n_on}")
    assert n_on == FIT_LAUNCHES[tag] + 1


# Step budget of the recovery fit, calibrated on one B200 (profiles/r11_kp2d_gpu_tests.txt has the measured curves).
RECOVERY_STEPS = 250


@CONFIGS
def test_fit_recovers_perturbed_limbs_from_detections(flags):
    """Detections are the true joints of the batch's frames projected through their cameras (256 x 256 images).  The
    axis-angles of the limb joints are perturbed by seeded N(0, 0.25 rad) noise; PoseFitStep(graph=True) with the 2D
    term (kp2d_coef = 100, sigma = 100 px; no pose regulariser) must cut the mean pixel error kp2d_px by 10x within
    RECOVERY_STEPS iterations, whatever the untrained field's photometric term pulls toward.  Measured on one B200
    (1 000 W): 9.55 px at the first step, 10x lower at step 159, 0.63 px at step 250 (both configs)."""
    from danbo_b200 import pose_opt as po, training
    H = 256
    args, feed, attrs, arrays = _setup(flags, H=H, kp2d_coef=100.0, lr=5e-3, opt_pose_coef=0.0, rays_per_image=192)
    batch = feed.next_batch(torch.Generator(device=DEV).manual_seed(0))
    frames = feed.last_idxs[0].cpu().numpy()
    caster, _, _ = make_caster("danbo_fast", train=True, **flags)
    opt, kw = po.create_popt(args, attrs, device=DEV, flat=True)
    layer = kw["popt_layer"]
    batch = dict(batch, **_detections(layer, arrays, frames, H))
    with torch.no_grad():
        g = torch.Generator(device=DEV).manual_seed(7)
        layer.bones[:, LIMBS] += 0.25 * torch.randn(layer.bones[:, LIMBS].shape, device=DEV, generator=g)
    fit = training.PoseFitStep(caster, args, kw, opt, graph=True)
    px = []
    for _ in range(RECOVERY_STEPS):
        fit(batch)
        px.append(float(fit.last_stats["kp2d_px"]))
    tag = flags.get("ray_tr_type", "world")
    first10 = next((i for i, v in enumerate(px) if v <= px[0] / 10), None)
    print(f"[kp2d recovery {tag}] kp2d_px every 10 steps: " + " ".join("%.3f" % v for v in px[::10] + px[-1:]))
    print(f"[kp2d recovery {tag}] 10x below the first step's {px[0]:.3f} px at step {first10}; last {px[-1]:.4f} px")
    assert all(v == v for v in px)
    assert px[0] > 2.0
    assert px[-1] <= px[0] / 10
