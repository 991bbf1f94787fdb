"""A-NeRF pose refinement on the GPU (run with -m gpu): the MLP's input gradient, `danbo_anerf_embed_bwd`'s d skts, the
whole training step's d loss / d skts, and a --opt_pose TrainStep on an A-NeRF caster."""
import numpy as np
import pytest
import torch

import danbo_oracle as orc
from util import load_fixture, align_A, decode_tile_image, anerf_mlp_bf16_reference
from test_anerf_pose_grad_cpu import CASES, anerf_case, fixture_of, oracle_skts_grad, random_input_grads
from test_gpu_anerf import make_anerf_caster, anerf_params

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(300, method="thread")]   # a hung kernel must not hang the box
DEV = "cuda"


def _K():
    from danbo_b200 import kernels
    return kernels


def _rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm())


@pytest.mark.parametrize("name", CASES)
def test_embed_bwd_matches_oracle_autograd(name):
    """Stage level, fp32 on both sides: d skts of the encodings for a random d xd / d xv.  The kernel reduces 4 rays per
    block.  render_anerf (64 rays, one pose) and train_anerf (2 poses x 24 rays) fill whole blocks of one pose, so only the
    block reduction runs; train_anerf_straddle (2 poses x 22 rays, last ray dropped: 43 rays) has a block holding both
    poses (the per-ray atomics) and a last block with a ray-less warp."""
    K = _K()
    fx = load_fixture(fixture_of(name))
    caster, args, _ = make_anerf_caster(fx)
    rays, z, pose_skts, rpp, tau = anerf_case(name)
    N, S = z.shape
    d_xd, d_xv = random_input_grads(N * S, 7)
    d = lambda t: t.to(DEV).float().contiguous()
    cams = torch.zeros(N, device=DEV, dtype=torch.int32)
    enc, _ = K.anerf_ray_encode(d(rays), d(pose_skts), rpp, cams, caster._codes_with_mean(), caster._packed_mlp())
    d_skts = torch.zeros(pose_skts.shape, device=DEV)
    K.anerf_embed_bwd(d(rays), S, d(z), d(pose_skts), rpp, caster._align(), enc, tau, d(d_xd), d(d_xv), d_skts)
    again = torch.zeros_like(d_skts)
    K.anerf_embed_bwd(d(rays), S, d(z), d(pose_skts), rpp, caster._align(), enc, tau, d(d_xd), d(d_xv), again)
    torch.cuda.synchronize()
    want = oracle_skts_grad(rays, z, pose_skts, rpp, align_A(), tau, d_xd, d_xv)
    got = d_skts.cpu()
    rel = _rel(got, want)
    print(f"[anerf popt] embed bwd {name}: {pose_skts.shape[0]} poses |g| {float(want.norm()):.3e} rel {rel:.3e} "
          f"run-to-run {_rel(again.cpu(), got):.1e}")
    assert float(got[:, :, 3].abs().max()) == 0.0
    assert rel <= 2e-4, rel
    for g in range(pose_skts.shape[0]):                          # each pose on its own: a misrouted block shows here
        assert _rel(got[g], want[g]) <= 2e-4, (g, _rel(got[g], want[g]))


def test_mlp_input_gradient():
    """d xd / d xv of anerf_mlp_backward(want_dx=True) against autograd of the bf16-emulating restatement on the kernel's
    own untiled inputs.  The weights are rounded to bf16 first: the backward chain multiplies by the fp32 weights, the
    restatement by their bf16 roundings.  What remains is the forward: the restatement recomputes it, so a bf16
    activation can round to the neighbouring value and a pre-activation within rounding of zero can fall on the other
    side of a ReLU than in the kernel's saved activations, over ten layers (measured on a B200: rel 1.8e-2 for d xd).
    The parameter gradients must not change with want_dx."""
    K = _K()
    fx = load_fixture("render_anerf")
    caster, args, P = make_anerf_caster(fx)
    Pb = {k: (v.to(torch.bfloat16).float() if k != "framecodes.codes.weight" else v) for k, v in P.items()}
    caster.network.load_state_dict(Pb, strict=False)
    rays, z, pose_skts, rpp, tau = anerf_case("render_anerf")
    N, S = z.shape
    rows = N * S
    d = lambda t: t.to(DEV).float().contiguous()
    cams = fx["cams"].reshape(-1).to(DEV).to(torch.int32)
    packed = caster._packed_mlp()
    codes = caster._codes_with_mean()
    enc, cb = K.anerf_ray_encode(d(rays), d(pose_skts), rpp, cams, codes, packed)
    xd, xv = K.anerf_embed(d(rays), S, d(z), d(pose_skts), rpp, caster._align(), enc, tau)
    raw = torch.empty(rows + N, 4, device=DEV)
    sv = K.anerf_save_buffer(rows, DEV)
    K.anerf_mlp(xd, xv, packed, cb, rows, S, raw, save=sv)
    torch.manual_seed(2)
    d_raw = torch.zeros(rows + N, 4, device=DEV)
    d_raw[:rows] = torch.randn(rows, 4, device=DEV)
    Pd = {k: v.to(DEV) for k, v in Pb.items()}
    G = {k: torch.zeros_like(v) for k, v in Pd.items()}
    G_plain = {k: torch.zeros_like(v) for k, v in Pd.items()}
    dXd, dXv = K.anerf_mlp_backward(Pd, G, d_raw, rows, S, xd, xv, sv, cb, cams, codes, want_dx=True)
    assert K.anerf_mlp_backward(Pd, G_plain, d_raw, rows, S, xd, xv, sv, cb, cams, codes) is None
    torch.cuda.synchronize()
    for k in G:                                                   # the parameter gradients do not depend on want_dx
        assert _rel(G[k].cpu(), G_plain[k].cpu()) <= 1e-5 or float(G_plain[k].norm()) == 0.0, k
    xd_f = decode_tile_image(xd, rows, 7, 432).cpu().requires_grad_(True)
    xv_f = decode_tile_image(xv, rows, 11, 648).cpu().requires_grad_(True)
    out = anerf_mlp_bf16_reference(xd_f, xv_f, cb.cpu().repeat_interleave(S, 0), {k: v.cpu() for k, v in Pb.items()})
    (out * d_raw[:rows].cpu()).sum().backward()
    for nm, got, want in (("d xd", dXd.cpu(), xd_f.grad), ("d xv", dXv.cpu(), xv_f.grad)):
        rel = _rel(got, want)
        print(f"[anerf popt] mlp {nm}: |g| {float(want.norm()):.3e} rel {rel:.3e}")
        cos = float(torch.dot(got.reshape(-1).double(), want.reshape(-1).double()) / (got.double().norm() * want.double().norm()))
        print(f"[anerf popt] mlp {nm}: cos {cos:.6f}")
        assert got.shape == want.shape and rel <= 4e-2 and cos >= 0.999, (nm, rel, cos)


def _anerf_step(caster, args, fx, b, rand, skts):
    stages = {}
    out = caster.render_rays(b["ray_batch"], N_samples=args.N_samples, kp_batch=b["kp_batch"], skts=skts, cyls=b["cyls"],
                             bones=b["bones"], cams=b["cams"], N_uniques=int(fx["n_poses"]), perturb=1.0,
                             N_importance=args.N_importance, raw_noise_std=float(fx["raw_noise_std"]), nerf_type="nerf",
                             _rand={k: v.to(DEV) for k, v in rand.items()}, _stages=stages)
    tgt, bgs = b["target_s"].to(DEV), b["bgs"].to(DEV)
    l1 = lambda rgb, acc: torch.mean(torch.abs(rgb + (1. - acc)[..., None] * bgs - tgt))
    loss = l1(out["rgb_map"], out["acc_map"]) + l1(out["rgb0"], out["acc0"])
    caster.network.zero_grad(set_to_none=True)
    loss.backward()
    torch.cuda.synchronize()
    grads = {n: p.grad.detach().cpu().clone() for n, p in caster.network.named_parameters() if p.grad is not None}
    return loss, grads, stages


def test_training_step_pose_gradients():
    """Whole step: the per-ray world-to-bone matrices enter the A-NeRF caster as a leaf; their per-pose gradient against
    oracle autograd at the kernel's own importance samples, and the 25 parameter gradients unchanged by the pose leaf."""
    from danbo_b200 import synthetic as syn
    fx = load_fixture("train_anerf")
    caster, args, _ = make_anerf_caster(fx)
    caster.train()
    n_poses, rpp = int(fx["n_poses"]), int(fx["rays_per_pose"])
    b = syn.training_batch(n_poses, rpp, seed=int(fx["batch_seed"]))
    rand = {k: fx["rand." + k] for k in ("t_rand", "noise0", "u", "noise1")}
    _, g_a, _ = _anerf_step(caster, args, fx, b, rand, b["skts"])
    _, g_b, _ = _anerf_step(caster, args, fx, b, rand, b["skts"])
    leaf = b["skts"].clone().to(DEV).requires_grad_(True)
    loss, g_c, stages = _anerf_step(caster, args, fx, b, rand, leaf)
    assert len(g_a) == 25 and set(g_c) == set(g_a)
    floor = max(_rel(g_b[k], g_a[k]) for k in g_a if float(g_a[k].norm()) > 0)
    worst = max(_rel(g_c[k], g_a[k]) for k in g_a if float(g_a[k].norm()) > 0)
    print(f"[anerf popt] parameter gradients with a pose leaf: rel {worst:.2e} (run-to-run floor {floor:.2e})")
    assert worst <= max(2 * floor, 1e-5), (worst, floor)
    got = leaf.grad.reshape(n_poses, rpp, 24, 4, 4).sum(1).cpu()
    P = anerf_params(fx)
    pose_skts = b["skts"][::rpp].clone().requires_grad_(True)
    ref = orc.anerf_render_rays(b["ray_batch"], pose_skts, b["cyls"][::rpp], b["cams"], align_A(), P, int(fx["N_samples"]),
                                int(fx["N_importance"]), rays_per_pose=rpp, training=True, rand=rand,
                                raw_noise_std=float(fx["raw_noise_std"]), z_samples=stages["z_samples"].cpu())
    l1 = lambda rgb, acc: torch.mean(torch.abs(rgb + (1. - acc)[..., None] * b["bgs"] - b["target_s"]))
    ref_loss = l1(ref["rgb_map"], ref["acc_map"]) + l1(ref["rgb0"], ref["acc0"])
    ref_loss.backward()
    assert abs(float(loss.detach()) - float(ref_loss.detach())) <= 5e-3
    a, r = got.reshape(-1).double(), pose_skts.grad.reshape(-1).double()
    cos = float(torch.dot(a, r) / (a.norm() * r.norm() + 1e-30))
    rel = float((a - r).norm() / r.norm())
    print(f"[anerf popt] step d skts: |g| {float(r.norm()):.3e} cos {cos:.5f} rel {rel:.3e}")
    assert float(got[:, :, 3].abs().max()) == 0.0
    # same bounds as the DANBO path's pose gradients (bf16 forward MLP, the raw-noise gate)
    assert cos >= 0.985 and rel <= 0.2, (cos, rel)


def test_train_step_with_pose_layer_and_feed():
    """--opt_pose on an A-NeRF caster end to end: device feed -> pose layer -> render -> fused loss + pose regulariser ->
    both optimisers.  With opt_pose_coef = 0 the regulariser's gradient is zero, so the poses of the frames drawn move
    only through the render loss; the others must not move, and everything stays finite."""
    import danbo_b200 as db
    from danbo_b200 import feed as fd, pose_opt as po, training, synthetic as syn
    fx = load_fixture("train_anerf")
    caster, _, _ = make_anerf_caster(fx)
    args = db.make_args("anerf_base", no_reload=True, N_samples=int(fx["N_samples"]), N_importance=int(fx["N_importance"]))
    n_images = 12
    arrays = fd.synthetic_arrays(n_images=n_images, H=64, W=64, seed=2)
    # frame codes: the caster has 8 (n_views), so the images cycle through them as in feed.synthetic_feed
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
    losses, touched = [], set()
    for _ in range(2):
        batch = feed.next_batch(g)
        touched.update(feed.last_idxs[0].tolist())
        loss, preds = step(batch)
        losses.append(float(loss))
        assert preds["rgb_map"].shape == (4 * 48, 3)
    torch.cuda.synchronize()
    print("[anerf popt] losses", [f"{v:.4f}" for v in losses], "touched", sorted(touched))
    assert all(l == l and l < 10 for l in losses)
    moved = (layer.bones.detach() - before).abs().amax(dim=(1, 2)).cpu()
    assert bool(torch.isfinite(layer.bones).all()) and bool(torch.isfinite(layer.pelvis).all())
    assert len(touched) < n_images
    for i in range(n_images):
        assert (float(moved[i]) > 0) == (i in touched), (i, float(moved[i]), sorted(touched))
