"""Frame-code fitting with a frozen DANBO field on the GPU (run with -m gpu): danbo_ray_bias_codes_bwd against the fp64
statement (tests/code_fit_ref.py) and against danbo_ray_bias_bwd's code gradient; PoseFitStep(code_kwargs=...) against
training's frame-code gradient, against pose fitting with the mean code, with the network left untouched, captured
against eager; a fit of codes toward images rendered with known codes; rendering with a fitted table; and the launch
sequences of training, pose fitting and the plain render, which code fitting must leave as they were."""
import os

import numpy as np
import pytest
import torch

from code_fit_ref import codes_grad_fp64
from util import make_caster

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900, method="thread")]   # a hung kernel must not hang the box
DEV = "cuda"
PERFCAP = dict(view_type="relray", ray_tr_type="root_local", nerf_type="graph")     # configs/perfcap/danbo_fast.txt
CONFIGS = pytest.mark.parametrize("flags", [{}, PERFCAP], ids=["h36m_zju", "perfcap"])
# kernels._count of one uncaptured TrainStep(graph=True)._step with a pose layer, one eager PoseFitStep without codes
# and one eval render of the same 192-ray batch, measured on a B200 at the parent commit of code fitting.
PARENT_LAUNCHES = {"world": {"train": 58, "fit": 39, "render": 24},
                   "root_local": {"train": 59, "fit": 42, "render": 24}}


def _rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp(min=1e-30))


# ---------------------------------------------------------------------------------------------------- kernel
def _cams(n, n_codes, run, seed):
    """Image-major runs of `run` rays with cams in [-2, n_codes + 2] (the mean code, and values above the last row),
    and single rays of another cam inside 16-ray groups (mixed runs)."""
    g = torch.Generator().manual_seed(seed)
    cams = torch.randint(-2, n_codes + 3, (n // run,), generator=g).repeat_interleave(run)
    for i in torch.randint(0, n, (max(n // 64, 4),), generator=g).tolist():
        cams[i] = int(torch.randint(-2, n_codes + 3, (1,), generator=g))
    cams[5], cams[6] = 1, 2 * n_codes                                # a mixed 16-ray group, one ray clamped
    return cams.to(torch.int32)


def _kernel_inputs(n, run, seed=0, n_codes=8):
    g = torch.Generator().manual_seed(seed)
    cam = _cams(n, n_codes, run, seed)
    w_view = torch.randn(128, 411, generator=g) * 0.05
    d_rb = torch.randn(n, 128, generator=g) * 1e-3
    return cam, w_view, d_rb, n_codes


@pytest.mark.parametrize("n,run", [(3072, 192), (262144, 4096)])
def test_codes_kernel_matches_fp64(n, run):
    """Bound per element: 1e-5 of the same sum over |W_v| and |d ray_bias| (fp32 run sums of up to 4 096 rays, a
    128-term dot product and one atomic per run)."""
    from danbo_b200 import kernels as K
    cam, w_view, d_rb, n_codes = _kernel_inputs(n, run)
    d_codes = torch.zeros(n_codes, 128, device=DEV)
    K.ray_bias_codes_bwd(cam.to(DEV), w_view.to(DEV), d_rb.to(DEV), d_codes)
    torch.cuda.synchronize()
    want = codes_grad_fp64(cam, w_view, d_rb, n_codes)
    scale = codes_grad_fp64(cam, w_view.abs(), d_rb.abs(), n_codes)
    err = (d_codes.cpu().double() - want).abs()
    ratio = float((err / scale.clamp(min=1e-30)).max())
    print(f"[codes kernel n={n}] max |err| {float(err.max()):.2e}, max err / scale {ratio:.2e}, "
          f"rel {_rel(d_codes.cpu(), want):.2e}")
    assert float(want.abs().min()) > 0                          # every row is reached
    assert bool((err <= 1e-5 * scale + 1e-12).all())


def test_codes_kernel_matches_ray_bias_bwd():
    """danbo_ray_bias_codes_bwd's d codes against danbo_ray_bias_bwd's on identical inputs (the same statement,
    summed in 16-ray groups there and in runs here)."""
    from danbo_b200 import kernels as K
    n = 3072
    cam, w_view, d_rb, n_codes = _kernel_inputs(n, 192, seed=1)
    g = torch.Generator().manual_seed(2)
    rays = torch.cat([torch.randn(n, 3, generator=g), torch.nn.functional.normalize(torch.randn(n, 3, generator=g)),
                      torch.full((n, 2), 2.0)], -1).to(DEV)
    codes = torch.randn(n_codes + 1, 128, generator=g).to(DEV)
    cam_d, w_d, rb_d = cam.to(DEV), w_view.to(DEV), d_rb.to(DEV)
    full = torch.zeros(n_codes, 128, device=DEV)
    K.ray_bias_bwd(rays, cam_d, codes, w_d, rb_d, torch.zeros(128, 411, device=DEV), torch.zeros(128, device=DEV), full)
    only = K.ray_bias_codes_bwd(cam_d, w_d, rb_d, torch.zeros(n_codes, 128, device=DEV))
    torch.cuda.synchronize()
    scale = codes_grad_fp64(cam, w_view.abs(), d_rb.abs(), n_codes)
    err = (only.cpu().double() - full.cpu().double()).abs()
    print(f"[codes kernel vs ray_bias_bwd] rel {_rel(only, full):.2e}")
    assert float(full.abs().max()) > 0 and bool((err <= 2e-5 * scale + 1e-12).all())


# ---------------------------------------------------------------------------------------------------- step
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
    batch = feed.next_batch(torch.Generator(device=DEV).manual_seed(0))
    return args, feed, attrs, batch


def _fresh(flags, args, attrs, codes=None, code_lr=1e-3, perturb=0.02):
    """The seeded caster, a pose layer off its anchors and, with `codes` (rows or an (rows,128) tensor), a fitted
    code table from training.create_code_fit set to those values."""
    from danbo_b200 import pose_opt as po, training
    caster, _, _ = make_caster("danbo_fast", train=True, **flags)
    opt, kw = po.create_popt(args, attrs, device=DEV, flat=True)
    with torch.no_grad():
        kw["popt_layer"].bones[:, 1:] += perturb
    if codes is None:
        return caster, opt, kw, {}
    rows = codes if isinstance(codes, int) else codes.shape[0]
    copt, ckw = training.create_code_fit(caster, rows, lr=code_lr)
    if torch.is_tensor(codes):
        with torch.no_grad():
            ckw["frame_codes"].copy_(codes)
    return caster, opt, kw, {"code_kwargs": ckw, "code_optimizer": copt}


def _test_codes(caster, seed=5):
    w = caster.network.framecodes.codes.weight.detach()
    g = torch.Generator(device=DEV).manual_seed(seed)
    return w + 0.5 * w.std() * torch.randn(w.shape, device=DEV, generator=g)


def _fit_code_grad(flags, args, attrs, batch, codes):
    from danbo_b200 import training
    caster, opt, kw, ck = _fresh(flags, args, attrs, codes=codes)
    step = training.PoseFitStep(caster, args, kw, opt, **ck)
    loss, _ = step(batch)
    torch.cuda.synchronize()
    return float(loss), ck["code_optimizer"].bucket.flat.view(-1, 128).clone(), opt.bucket.flat.clone()


@CONFIGS
def test_code_gradient_equals_training_code_gradient(flags):
    """The d codes of one fitting step against the framecodes.codes.weight gradient of one uncaptured training step
    (TrainStep with a pose layer) on the same batch, with the network's table set to the fitted rows.  Tolerance:
    2x the run-to-run spread of the fitting gradient, at least 1e-4 relative.  The two backward passes differ in
    their MLP dgrad variant and sum d ray_bias with fp32 atomics in another order, and training forms the code
    gradient in 16-ray groups (danbo_ray_bias_bwd) where fitting sums runs (danbo_ray_bias_codes_bwd)."""
    from danbo_b200 import pose_opt as po, training
    args, _, attrs, batch = _setup(flags)
    probe, _, _ = make_caster("danbo_fast", train=True, **flags)
    codes = _test_codes(probe)
    f1, f2 = _fit_code_grad(flags, args, attrs, batch, codes), _fit_code_grad(flags, args, attrs, batch, codes)
    caster, _, _ = make_caster("danbo_fast", train=True, **flags)
    with torch.no_grad():
        caster.network.framecodes.codes.weight.copy_(codes)
    opt, kw = po.create_popt(args, attrs, device=DEV, flat=True)
    with torch.no_grad():
        kw["popt_layer"].bones[:, 1:] += 0.02
    tstep = training.TrainStep(caster, args, graph=True, popt_kwargs=kw, pose_optimizer=opt)
    tstep._step(batch)
    torch.cuda.synchronize()
    t = caster.network.framecodes.codes.weight.grad.clone()
    spread, err = _rel(f2[1], f1[1]), _rel(f1[1], t)
    used = sorted(set(batch["cams"].reshape(-1).tolist()))
    tag = flags.get("ray_tr_type", "world")
    print(f"[code grad vs train {tag}] rows {used}: rel {err:.2e} (fit spread {spread:.2e}); pose grads rel "
          f"{_rel(f1[2], opt.bucket.flat):.2e}")
    assert float(f1[1].abs().max()) > 0
    assert err <= max(1e-4, 2 * spread)
    unused = [r for r in range(t.shape[0]) if r not in used]
    assert float(f1[1][unused].abs().max()) == 0 and float(t[unused].abs().max()) == 0


@CONFIGS
def test_mean_codes_step_equals_mean_code_step(flags):
    """Codes at the network's mean and the batch's cams pointing at fitted rows against pose fitting without codes and
    cams = -1: the same rgb_map and loss, and the pose gradient within the run-to-run spread."""
    from danbo_b200 import training
    args, _, attrs, batch = _setup(flags)
    caster, opt, kw, ck = _fresh(flags, args, attrs, codes=8)
    loss_c, preds_c = training.PoseFitStep(caster, args, kw, opt, **ck)(batch)
    torch.cuda.synchronize()
    rgb_c, grad_c = preds_c["rgb_map"].detach().clone(), opt.bucket.flat.clone()
    mean_batch = dict(batch, cams=torch.full_like(batch["cams"], -1))
    runs = []
    for _ in range(2):
        caster, opt, kw, _ = _fresh(flags, args, attrs)
        loss_m, preds_m = training.PoseFitStep(caster, args, kw, opt)(mean_batch)
        torch.cuda.synchronize()
        runs.append((float(loss_m), preds_m["rgb_map"].detach().clone(), opt.bucket.flat.clone()))
    spread, err = _rel(runs[1][2], runs[0][2]), _rel(grad_c, runs[0][2])
    d_rgb = float((rgb_c - runs[0][1]).abs().max())
    tag = flags.get("ray_tr_type", "world")
    print(f"[mean codes {tag}] rgb bit-equal {torch.equal(rgb_c, runs[0][1])} (max |diff| {d_rgb:.1e}); loss "
          f"{float(loss_c):.7f} vs {runs[0][0]:.7f}; pose grads rel {err:.2e} (spread {spread:.2e})")
    assert d_rgb <= 1e-6
    assert abs(float(loss_c) - runs[0][0]) <= 1e-6 * abs(runs[0][0])
    assert err <= max(1e-5, 2 * spread)


@CONFIGS
def test_code_fitting_leaves_the_network_untouched(flags):
    from danbo_b200 import training
    args, _, attrs, batch = _setup(flags)
    caster, opt, kw, ck = _fresh(flags, args, attrs, codes=8, code_lr=1e-2)
    net = caster.network
    marked = dict(net.named_parameters())["framecodes.codes.weight"]
    marked.grad = torch.randn_like(marked)                       # a gradient a user left behind must survive
    params = {n: p.detach().clone() for n, p in net.named_parameters()}
    grads = {n: (None if p.grad is None else p.grad.clone()) for n, p in net.named_parameters()}
    sd = {k: v.clone() for k, v in caster.state_dict()["network_fn_state_dict"].items()}
    codes0 = ck["code_kwargs"]["frame_codes"].detach().clone()
    step = training.PoseFitStep(caster, args, kw, opt, graph=True, **ck)
    for _ in range(6):
        step(batch)
    torch.cuda.synchronize()
    for n, p in net.named_parameters():
        assert torch.equal(p.detach(), params[n]), n
        assert (p.grad is None) if grads[n] is None else torch.equal(p.grad, grads[n]), n
    assert all(torch.equal(v, sd[k]) for k, v in caster.state_dict()["network_fn_state_dict"].items())
    moved = (ck["code_kwargs"]["frame_codes"].detach() - codes0).abs().amax(1)
    used = sorted(set(batch["cams"].reshape(-1).tolist()))
    assert float(ck["code_optimizer"].step_dev) == 6.0 and float(opt.step_dev) == 6.0
    assert all(float(moved[r]) > 0 for r in used) and all(float(moved[r]) == 0 for r in range(8) if r not in used)


def _run(flags, args, attrs, batch, graph, n=5):
    from danbo_b200 import training
    caster, opt, kw, ck = _fresh(flags, args, attrs, codes=8, code_lr=1e-3)
    step = training.PoseFitStep(caster, args, kw, opt, graph=graph, **ck)
    losses = [float(step(batch)[0]) for _ in range(n)]
    torch.cuda.synchronize()
    return losses, ck["code_kwargs"]["frame_codes"].detach().clone(), opt.flat.clone()


@CONFIGS
def test_captured_code_fit_equals_eager(flags):
    """5 steps captured against 5 eager steps.  The first loss (nothing updated yet) agrees to 1e-6 relative.  After
    that, Adam divides each entry's gradient by its own magnitude, so an entry whose gradient is close to zero changes
    sign with the fp32 atomics' summation order and moves by about lr either way.  Eager runs therefore differ from
    one another too, by 6e-5 .. 1.1e-3 relative in losses, codes and poses on a B200.  The bound is 4x the measured
    eager spread, and at least 3e-3 relative."""
    args, _, attrs, batch = _setup(flags)
    e1, e2 = _run(flags, args, attrs, batch, False), _run(flags, args, attrs, batch, False)
    g = _run(flags, args, attrs, batch, True)
    tag = flags.get("ray_tr_type", "world")
    for i, name in ((1, "codes"), (2, "poses")):
        spread, err = _rel(e2[i], e1[i]), _rel(g[i], e1[i])
        print(f"[captured vs eager code fit {tag}] {name} rel {err:.2e} (eager spread {spread:.2e})")
        assert err <= max(3e-3, 4 * spread), name
    lspread = max(abs(a - b) / abs(b) for a, b in zip(e2[0], e1[0]))
    lerr = max(abs(a - b) / abs(b) for a, b in zip(g[0], e1[0]))
    print(f"[captured vs eager code fit {tag}] losses {['%.6f' % v for v in g[0]]}: rel {lerr:.1e} "
          f"(spread {lspread:.1e})")
    assert abs(g[0][0] - e1[0][0]) <= 1e-6 * abs(e1[0][0])
    assert lerr <= max(3e-3, 4 * lspread)


@CONFIGS
def test_fitting_recovers_frame_codes(flags):
    """Targets rendered by the field at the known poses with its own frame codes (cams 0..7, one per image); fitting
    starts at the mean code with the poses at the truth and a pose learning rate of 0 (only codes move), 40 captured
    iterations at lr 1e-2.  The photometric loss must fall below 0.9x its first value and the mean distance of the
    fitted rows to the true codes below 0.98x its first value.  Measured on one B200 (1 000 W power limit), which set
    these thresholds: h36m_zju loss 0.00818 -> 0.00672 (0.82x), distance 3.341 -> 3.144 (0.94x); perfcap loss
    0.00812 -> 0.00668, distance 3.341 -> 3.150 (profiles/r14_code_fit_gpu_tests.txt).  (Adam moves each entry by
    about lr per step, so 40 steps close only part of the distance.)"""
    from danbo_b200 import training
    args, feed, attrs, _ = _setup(flags, coef=0.0, lr=0.0, rays_per_image=512)
    batch = feed.next_batch(torch.Generator(device=DEV).manual_seed(3))
    caster, opt, kw, ck = _fresh(flags, args, attrs, codes=8, code_lr=1e-2, perturb=0.0)
    truth = caster.network.framecodes.codes.weight.detach().clone()
    caster.eval()
    with torch.no_grad():
        a = args
        preds = caster(batch["ray_batch"], N_samples=a.N_samples, kp_batch=batch["kp_batch"], skts=batch["skts"],
                       cyls=batch["cyls"], bones=batch["bones"], cams=batch["cams"], N_uniques=batch["N_uniques"],
                       perturb=0., N_importance=a.N_importance, raw_noise_std=0.)
        target = preds["rgb_map"] + (1. - preds["acc_map"])[..., None] * batch.get("bgs", 1.0)
    batch["target_s"] = target.detach().clone()
    codes = ck["code_kwargs"]["frame_codes"]
    used = sorted(set(batch["cams"].reshape(-1).tolist()))
    dist = lambda: float((codes.detach()[used] - truth[used]).norm(dim=1).mean())
    fit = training.PoseFitStep(caster, args, kw, opt, graph=True, **ck)
    losses, dists = [], [dist()]
    for _ in range(40):
        losses.append(float(fit(batch)[0]))
        dists.append(dist())
    torch.cuda.synchronize()
    tag = flags.get("ray_tr_type", "world")
    print(f"[code fit {tag}] rows {used}")
    print(f"[code fit {tag}] loss " + " ".join("%.5f" % v for v in losses[::5] + losses[-1:]))
    print(f"[code fit {tag}] |code - truth| " + " ".join("%.4f" % v for v in dists[::5] + dists[-1:]))
    assert all(v == v for v in losses)
    assert losses[-1] < 0.9 * losses[0] and dists[-1] < 0.98 * dists[0]


@CONFIGS
def test_render_with_the_network_table_is_bit_identical(flags):
    """frame_codes = the network's own table renders like the plain call, bit for bit (render_rays and
    render.render_images); another table changes the pixels of the rays that read it."""
    from danbo_b200 import render, synthetic as syn
    caster, args, _ = make_caster("danbo_fast", **flags)
    args, _, attrs, batch = _setup(flags)
    a = args
    table = caster.network.framecodes.codes.weight.detach().clone()
    kw = dict(N_samples=a.N_samples, kp_batch=batch["kp_batch"], skts=batch["skts"], cyls=batch["cyls"],
              bones=batch["bones"], cams=batch["cams"], N_uniques=batch["N_uniques"], perturb=0.,
              N_importance=a.N_importance, raw_noise_std=0.)
    plain = caster(batch["ray_batch"], **kw)
    same = caster(batch["ray_batch"], frame_codes=table, **kw)
    other = caster(batch["ray_batch"], frame_codes=_test_codes(caster), **kw)
    for k in ("rgb_map", "acc_map", "disp_map", "rgb0"):
        assert torch.equal(plain[k], same[k]), k
    assert float((other["rgb_map"] - plain["rgb_map"]).abs().max()) > 0
    pose = syn.make_pose(0)
    c2ws = [syn.camera()]
    img = render.render_images(caster, a, c2ws, [pose], 32, 32, cam_idx=3)
    img_t = render.render_images(caster, a, c2ws, [pose], 32, 32, cam_idx=3, frame_codes=table)
    assert torch.equal(img, img_t)


@CONFIGS
def test_launch_sequences_are_the_parents(flags):
    """TrainStep, PoseFitStep without codes and the plain eval render launch what they launched at the parent commit
    (kernels._count); code fitting adds the head backward where pose fitting skips it, the code kernel and one Adam."""
    from torch.profiler import profile, ProfilerActivity
    from danbo_b200 import kernels as K, training
    args, _, attrs, batch = _setup(flags)
    tag = flags.get("ray_tr_type", "world")

    def counted(fn):
        fn()
        torch.cuda.synchronize()
        K.PROFILE = {"mlp": [], "launches": 0}
        try:
            fn()
            torch.cuda.synchronize()
            return K.PROFILE["launches"]
        finally:
            K.PROFILE = None

    caster, opt, kw, _ = _fresh(flags, args, attrs)
    tstep = training.TrainStep(caster, args, graph=True, popt_kwargs=kw, pose_optimizer=opt)
    caster, opt, kw, _ = _fresh(flags, args, attrs)
    fstep = training.PoseFitStep(caster, args, kw, opt)
    caster, opt, kw, ck = _fresh(flags, args, attrs, codes=8)
    cstep = training.PoseFitStep(caster, args, kw, opt, **ck)
    rcaster, _, _ = make_caster("danbo_fast", **flags)
    a = args

    def render():
        with torch.no_grad():
            rcaster(batch["ray_batch"], N_samples=a.N_samples, kp_batch=batch["kp_batch"], skts=batch["skts"],
                    cyls=batch["cyls"], bones=batch["bones"], cams=batch["cams"], N_uniques=batch["N_uniques"],
                    perturb=0., N_importance=a.N_importance, raw_noise_std=0.)
    got = {"train": counted(lambda: tstep._step(batch)), "fit": counted(lambda: fstep(batch)), "render": counted(render)}
    n_codes = counted(lambda: cstep(batch))
    print(f"[launches {tag}] {got}, code fitting {n_codes} (parent: {PARENT_LAUNCHES[tag]})")
    assert got == PARENT_LAUNCHES[tag]
    assert n_codes == got["fit"] + (2 if tag == "root_local" else 4)
    # the code step's extra kernels, by name: two head backwards on h36m (perfcap runs them already), one code kernel,
    # one more Adam
    names = {}
    for key, fn in (("fit", lambda: fstep(batch)), ("codes", lambda: cstep(batch))):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        names[key] = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    count = lambda key, s: sum(s in n for n in names[key])
    assert count("codes", "ray_bias_codes_bwd_kernel") == 1 and count("fit", "ray_bias_codes_bwd_kernel") == 0
    assert count("codes", "adam_kernel") == 2 and count("fit", "adam_kernel") == 1
    assert count("codes", "head_bwd_kernel<false, true>") == 2
    assert count("fit", "head_bwd_kernel<false, true>") == (2 if tag == "root_local" else 0)
    assert not any(s in n for n in names["codes"] for s in ("wgrad", "ray_bias_bwd_kernel", "head_bwd_kernel<true"))


def test_checkpoint_round_trip_with_codes(tmp_path):
    from danbo_b200 import training
    args, _, attrs, batch = _setup({})
    caster, opt, kw, ck = _fresh({}, args, attrs, codes=8, code_lr=1e-2)
    fit = training.PoseFitStep(caster, args, kw, opt, graph=True, **ck)
    for _ in range(3):
        fit(batch)
    path = os.path.join(tmp_path, "fit.tar")
    fit.save(path, 3)
    ck_file = torch.load(path, map_location="cpu", weights_only=False)
    assert set(ck_file["framecode_fit"]) == {"codes", "optimizer_state_dict"}
    caster2, opt2, kw2, ck2 = _fresh({}, args, attrs, codes=8, code_lr=1e-2)
    fit2 = training.PoseFitStep(caster2, args, kw2, opt2, **ck2)
    assert fit2.resume(ck_file) == 3
    assert torch.equal(ck2["code_kwargs"]["frame_codes"].detach(), ck["code_kwargs"]["frame_codes"].detach())
    assert torch.equal(ck2["code_optimizer"].exp_avg, ck["code_optimizer"].exp_avg)
    assert float(ck2["code_optimizer"].step_dev) == 3.0
    # without code fitting the checkpoint keeps exactly its keys
    caster3, opt3, kw3, _ = _fresh({}, args, attrs)
    plain = training.PoseFitStep(caster3, args, kw3, opt3)
    plain(batch)
    path3 = os.path.join(tmp_path, "plain.tar")
    plain.save(path3, 1)
    keys = set(torch.load(path3, map_location="cpu", weights_only=False))
    assert keys == set(ck_file) - {"framecode_fit"}
