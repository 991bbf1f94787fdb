"""anerf_h training on the GPU (run with -m gpu): A-NeRF with a separate fine network (single_net = False,
configs/h36m_zju/anerf_h.txt).  The fine network runs on all S_c + S_f merged samples, so its backward is the compositing
backward at the merged length and a second MLP backward over n * (S_c + S_f) rows.  Pinned to the oracle's autograd,
whose separate-fine-network forward is pinned by render_anerf_h.npz and whose training composition by train_anerf.npz
(the draws used here: t_rand, noise0, u and noise1 of shape (N, S_c + S_f))."""
import os
import tempfile

import pytest
import torch

import danbo_oracle as orc
import ref_harness as rh
from util import load_fixture, align_A
from test_gpu_anerf import anerf_params

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600, method="thread")]
DEV = "cuda"


def _K():
    from danbo_b200 import kernels
    return kernels


def _attrs():
    from danbo_b200 import synthetic as syn, skeleton as sk
    return {"skel_type": sk.SMPLSkeleton, "near": syn.NEAR, "far": syn.FAR, "n_views": 8, "rest_pose": syn.rest_pose()}


def fine_params(fx):
    from danbo_b200 import params, synthetic as syn
    return syn.synth_state_dict(params.anerf_param_shapes(), int(fx["weight_seed"]) + 1)


def make_anerf_h_caster(fx, **overrides):
    """create_raycaster for anerf_h at the fixture's sample counts; coarse weights of the fixture's seed, fine weights of
    seed + 1 (as render_anerf_h.npz).  -> caster, args, grad_vars, optimizer."""
    import danbo_b200 as db
    args = db.make_args("anerf_base", no_reload=True, single_net=False, N_samples=int(fx["N_samples"]),
                        N_importance=int(fx["N_importance"]), **overrides)
    _, kw_test, _, grad_vars, optimizer, _ = db.create_raycaster(args, _attrs(), device=DEV)
    caster = kw_test["ray_caster"]
    assert caster.network_fine is not caster.network and not caster.single_net
    for net, P in ((caster.network, anerf_params(fx)), (caster.network_fine, fine_params(fx))):
        missing = net.load_state_dict(P, strict=False)
        assert not missing.unexpected_keys and all("pe_fn" in k for k in missing.missing_keys), missing
    return caster, args, grad_vars, optimizer


def _rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm())


def _l1(out, tgt, bgs):
    return torch.mean(torch.abs(out[0] + (1. - out[1])[..., None] * bgs - tgt))


def _fixture_batch(fx):
    from danbo_b200 import synthetic as syn
    b = syn.training_batch(int(fx["n_poses"]), int(fx["rays_per_pose"]), seed=int(fx["batch_seed"]))
    rand = {k: fx["rand." + k] for k in ("t_rand", "noise0", "u", "noise1")}
    return b, rand


def _render(caster, args, fx, b, rand, skts=None, raw_noise_std=None, stages=None):
    std = float(fx["raw_noise_std"]) if raw_noise_std is None else raw_noise_std
    return caster.render_rays(b["ray_batch"], N_samples=args.N_samples, kp_batch=b["kp_batch"],
                              skts=b["skts"] if skts is None else skts, cyls=b["cyls"], bones=b["bones"], cams=b["cams"],
                              N_uniques=int(fx["n_poses"]), perturb=1.0, N_importance=args.N_importance,
                              raw_noise_std=std, nerf_type="nerf", _rand={k: v.to(DEV) for k, v in rand.items()},
                              _stages=stages)


def _grads(caster):
    """-> {"coarse <name>" / "fine <name>": gradient} of the 50 trainable tensors."""
    return {f"{which} {n}": p.grad.detach().cpu().clone() for which, net in (("coarse", caster.network),
                                                                            ("fine", caster.network_fine))
            for n, p in net.named_parameters() if p.requires_grad}


def _step(caster, args, fx, b, rand, skts=None, terms="both"):
    """Train-mode forward at the fixture's draws, the trainer's L1 terms (fine, coarse or both), backward.
    -> loss, the 50 parameter gradients (coarse then fine), stages."""
    stages = {}
    out = _render(caster, args, fx, b, rand, skts=skts, stages=stages)
    tgt, bgs = b["target_s"].to(DEV), b["bgs"].to(DEV)
    fine_t = _l1((out["rgb_map"], out["acc_map"]), tgt, bgs)
    coarse_t = _l1((out["rgb0"], out["acc0"]), tgt, bgs)
    loss = {"both": fine_t + coarse_t, "fine": fine_t, "coarse": coarse_t}[terms]
    caster.network.zero_grad(set_to_none=True)
    caster.network_fine.zero_grad(set_to_none=True)
    loss.backward()
    torch.cuda.synchronize()
    return loss.detach(), _grads(caster), stages


def _oracle(fx, b, rand, stages, pose_skts=None):
    rpp = int(fx["rays_per_pose"])
    P = {k: v.clone().requires_grad_(v.dtype.is_floating_point) for k, v in anerf_params(fx).items()}
    Pf = {k: v.clone().requires_grad_(v.dtype.is_floating_point) for k, v in fine_params(fx).items()}
    skts = b["skts"][::rpp] if pose_skts is None else pose_skts
    ref = orc.anerf_render_rays(b["ray_batch"], skts, b["cyls"][::rpp], b["cams"], align_A(), P, int(fx["N_samples"]),
                                int(fx["N_importance"]), rays_per_pose=rpp, training=True, rand=rand,
                                raw_noise_std=float(fx["raw_noise_std"]), z_samples=stages["z_samples"].cpu(), P_fine=Pf)
    loss = _l1((ref["rgb_map"], ref["acc_map"]), b["target_s"], b["bgs"]) + \
        _l1((ref["rgb0"], ref["acc0"]), b["target_s"], b["bgs"])
    loss.backward()
    return loss.detach(), P, Pf


# ---------------------------------------------------------------------------------------------------------------- 1
@pytest.mark.parametrize("S", [36, 144])
def test_fine_composite_backward_at_merged_length(S):
    """danbo_composite_bwd over S_t dense samples (the fine network's composite; 24+12 and 96+48), with density noise and
    inv_B != 1, on 37 rays (not a multiple of the rays of a block): d raw against fp64 autograd of the oracle's
    compositing; the n empty tail rows stay exactly 0 (every sample carries its own field value)."""
    torch.manual_seed(S)
    N, B = 37, 1.7
    rays = torch.randn(N, 8)
    rays[:, 3:6] = torch.nn.functional.normalize(torch.randn(N, 3), dim=-1) * (0.8 + 0.4 * torch.rand(N, 1))
    z = torch.sort(torch.rand(N, S) * 3 + 1, -1).values
    raw = torch.randn(N, S, 4) * torch.tensor([1., 1., 1., 5.])
    noise = torch.randn(N, S) * 0.7
    g_rgb, g_acc = torch.randn(N, 3), torch.randn(N)
    torch.set_default_dtype(torch.float64)                  # the oracle's constants follow the default dtype
    try:
        r = raw.double().requires_grad_(True)
        out = orc.composite(r, z.double(), rays[:, 3:6].double(), noise.double(), B=B)
        ((out["rgb_map"] * g_rgb.double()).sum() + (out["acc_map"] * g_acc.double()).sum()).backward()
    finally:
        torch.set_default_dtype(torch.float32)
    d = lambda t: t.to(DEV).contiguous()
    raw_buf = d(torch.cat([raw.reshape(N * S, 4), torch.randn(N, 4)], 0))
    d_raw = torch.zeros(N * S + N, 4, device=DEV)
    _K().composite_bwd(d(rays), S, raw_buf, torch.ones(N, S, dtype=torch.int32, device=DEV), d(z), d(noise), 1.0 / B,
                       d(g_rgb), d(g_acc), d_raw)
    torch.cuda.synchronize()
    got, want = d_raw[:N * S].reshape(N, S, 4).cpu().double(), r.grad
    err, scale = float((got - want).abs().max()), float(want.abs().max())
    print(f"[anerf_h] composite bwd S_t={S}: err {err:.3e} scale {scale:.3e} rel {err / scale:.2e}")
    assert err <= 1e-6 * scale, (err, scale)
    assert float(d_raw[N * S:].abs().max()) == 0.0


# ---------------------------------------------------------------------------------------------------------------- 2
def test_anerf_h_training_step_gradients():
    """Train-mode anerf_h step at the fixture's draws: loss and all 50 parameter gradients against the oracle's autograd
    at the kernel's own importance samples; the fine terms reach only the fine network and the coarse terms only the
    coarse one (the importance samples are detached)."""
    fx = load_fixture("train_anerf")
    caster, args, _, _ = make_anerf_h_caster(fx)
    caster.train()
    b, rand = _fixture_batch(fx)
    loss, got, stages = _step(caster, args, fx, b, rand)
    ref_loss, P, Pf = _oracle(fx, b, rand, stages)
    print(f"[anerf_h train] loss cuda {float(loss):.6f} oracle {float(ref_loss):.6f}")
    assert abs(float(loss) - float(ref_loss)) <= 5e-3
    want = {f"coarse {k}": v.grad for k, v in P.items() if v.grad is not None}
    want.update({f"fine {k}": v.grad for k, v in Pf.items() if v.grad is not None})
    assert len(got) == 50 and set(want) == set(got)
    big = max(float(w.norm()) for w in want.values())
    bad = []
    for k, r in want.items():
        a, r = got[k].reshape(-1).double(), r.reshape(-1).double()
        cos = float(torch.dot(a, r) / (a.norm() * r.norm() + 1e-30))
        rel = float((a - r).norm() / max(float(r.norm()), 1e-3 * big))
        print(f"[anerf_h train] {k:38s} |g| {float(r.norm()):.3e} cos {cos:.5f} rel {rel:.3e}")
        if (float(r.norm()) > 1e-3 * big and cos < 0.97) or rel > 0.3:
            bad.append((k, cos, rel))
    assert not bad, bad
    _, g_fine, _ = _step(caster, args, fx, b, rand, terms="fine")
    _, g_coarse, _ = _step(caster, args, fx, b, rand, terms="coarse")
    for k in got:
        only, other = (g_coarse, g_fine) if k.startswith("coarse") else (g_fine, g_coarse)
        assert float(other[k].abs().max()) == 0.0, (k, "gradient from the other network's outputs")
        assert float(only[k].abs().max()) > 0.0, (k, "no gradient from its own outputs")


# ---------------------------------------------------------------------------------------------------------------- 3
def test_anerf_h_train_mode_noise():
    """The fine composite takes the draw `noise1` in train mode with and without gradients: the fine outputs of a no-grad
    train-mode call equal those of the same call with gradients, and both differ from raw_noise_std = 0."""
    fx = load_fixture("train_anerf")
    caster, args, _, _ = make_anerf_h_caster(fx)
    caster.train()
    b, rand = _fixture_batch(fx)
    with torch.no_grad():
        ng = _render(caster, args, fx, b, rand)
        quiet = _render(caster, args, fx, b, rand, raw_noise_std=0.)
    wg = _render(caster, args, fx, b, rand)
    assert wg["rgb_map"].requires_grad and not ng["rgb_map"].requires_grad
    for k in ("rgb_map", "acc_map", "alpha", "T_i"):
        err = float((ng[k] - wg[k].detach()).abs().max())
        diff = float((quiet[k] - wg[k].detach()).abs().max())
        print(f"[anerf_h noise] {k}: no-grad vs grad {err:.2e}, vs raw_noise_std 0 {diff:.2e}")
        assert err <= 1e-6, (k, err)
        assert diff > 1e-3, (k, diff)


# ---------------------------------------------------------------------------------------------------------------- 4
def _anerf_mlp_bf16(x, view, P):
    """The oracle's A-NeRF MLP with the kernel's roundings (as util.anerf_mlp_bf16_reference: bf16 operands and stored
    activations, fp32 accumulation, sigma from the unrounded last activation), differentiable: each rounding passes the
    gradient straight through."""
    import torch.nn.functional as F

    def bf(t):
        return t + (t.to(torch.bfloat16).float() - t).detach()
    xb = bf(x)
    h, a = xb, None
    for i in range(8):
        a = F.relu(h @ bf(P[f"pts_linears.{i}.weight"]).t() + P[f"pts_linears.{i}.bias"])
        h = bf(a)
        if i == 4:
            h = torch.cat([xb, h], -1)
    sigma = a @ P["alpha_linear.weight"].t() + P["alpha_linear.bias"]
    feat = bf(h @ bf(P["feature_linear.weight"]).t() + P["feature_linear.bias"])
    Wv = P["views_linears.0.weight"]
    g = F.relu(feat @ bf(Wv[:, :448]).t() + bf(view[:, :648]) @ bf(Wv[:, 448:1096]).t() + view[:, 648:] @ Wv[:, 1096:].t()
               + P["views_linears.0.bias"])
    return torch.cat([g @ P["rgb_linear.weight"].t() + P["rgb_linear.bias"], sigma], -1)


def _cos_rel(a, r):
    a, r = a.reshape(-1).double(), r.reshape(-1).double()
    return float(torch.dot(a, r) / (a.norm() * r.norm() + 1e-30)), float((a - r).norm() / r.norm())


def test_anerf_h_pose_gradients(monkeypatch):
    """skts as a leaf: per-pose d skts of the whole anerf_h step (coarse pass at z0, fine pass at z_all with S_t samples)
    against the oracle's autograd through both networks; the 50 parameter gradients are unchanged by the leaf.

    The fine network's d skts is ill-conditioned to the bf16 rounding of the forward at this fixture: the fp32 oracle with
    only the MLP's roundings added (`_anerf_mlp_bf16`) is at cos 0.926 / rel 0.38 from the plain fp32 oracle (anerf_base:
    0.994 / 0.11).  So the bound of the anerf_base test (cos >= 0.985, rel <= 0.2) applies against that bf16 oracle, and
    against the fp32 oracle the kernel may be no further off than the bf16 oracle is, with 25 % margin."""
    fx = load_fixture("train_anerf")
    caster, args, _, _ = make_anerf_h_caster(fx)
    caster.train()
    n_poses, rpp = int(fx["n_poses"]), int(fx["rays_per_pose"])
    b, rand = _fixture_batch(fx)
    _, g_a, _ = _step(caster, args, fx, b, rand)
    _, g_b, _ = _step(caster, args, fx, b, rand)
    leaf = b["skts"].clone().to(DEV).requires_grad_(True)
    loss, g_c, stages = _step(caster, args, fx, b, rand, skts=leaf)
    assert len(g_a) == len(g_c) == 50
    assert set(g_c) == set(g_a)
    floor = max(_rel(g_b[k], g_a[k]) for k in g_a if float(g_a[k].norm()) > 0)
    worst = max(_rel(g_c[k], g_a[k]) for k in g_a if float(g_a[k].norm()) > 0)
    print(f"[anerf_h popt] parameter gradients with a pose leaf: rel {worst:.2e} (run-to-run floor {floor:.2e})")
    assert worst <= max(2 * floor, 1e-5), (worst, floor)
    got = leaf.grad.reshape(n_poses, rpp, 24, 4, 4).sum(1).cpu()
    assert float(got[:, :, 3].abs().max()) == 0.0
    ref = {}
    for name in ("fp32", "bf16"):
        if name == "bf16":
            monkeypatch.setattr(orc, "anerf_mlp", _anerf_mlp_bf16)
        pose_skts = b["skts"][::rpp].clone().requires_grad_(True)
        ref_loss, _, _ = _oracle(fx, b, rand, stages, pose_skts=pose_skts)
        assert abs(float(loss) - float(ref_loss)) <= 5e-3
        ref[name] = pose_skts.grad
        cos, rel = _cos_rel(got, pose_skts.grad)
        print(f"[anerf_h popt] step d skts vs the {name} oracle: |g| {float(pose_skts.grad.norm()):.3e} cos {cos:.5f} "
              f"rel {rel:.3e}")
    cos, rel = _cos_rel(got, ref["bf16"])
    assert cos >= 0.985 and rel <= 0.2, (cos, rel)
    cos32, rel32 = _cos_rel(got, ref["fp32"])
    cos_b, rel_b = _cos_rel(ref["bf16"], ref["fp32"])
    print(f"[anerf_h popt] bf16 oracle vs fp32 oracle: cos {cos_b:.5f} rel {rel_b:.3e}")
    assert rel32 <= 1.25 * rel_b and 1. - cos32 <= 1.25 * (1. - cos_b), (cos32, rel32, cos_b, rel_b)


# ---------------------------------------------------------------------------------------------------------------- 5
def _train_args(fx):
    import danbo_b200 as db
    return db.make_args("anerf_base", no_reload=True, single_net=False, N_samples=int(fx["N_samples"]),
                        N_importance=int(fx["N_importance"]))


def _flat(params):
    return torch.cat([p.detach().reshape(-1) for p in params]).cpu()


def test_anerf_h_train_step_trains_both_networks():
    """training.TrainStep on anerf_h: the bucket holds create_raycaster's grad_vars in their order; the loss goes down and
    both networks train (and stay two networks)."""
    from danbo_b200 import synthetic as syn, training
    fx = load_fixture("train_anerf")
    caster, _, grad_vars, _ = make_anerf_h_caster(fx)
    targs = _train_args(fx)
    with pytest.raises(NotImplementedError):
        training.TrainStep(caster, targs, graph=True)
    b = syn.training_batch(2, 48, seed=4)
    b = {k: (v.to(DEV) if torch.is_tensor(v) else v) for k, v in b.items()}
    step = training.TrainStep(caster, targs)
    assert len(step.bucket.params) == 50 and all(p is q for p, q in zip(step.bucket.params, grad_vars))
    coarse0 = _flat(caster.network.parameters())
    fine0 = _flat(caster.network_fine.parameters())
    torch.manual_seed(3)
    losses = [float(step(b)[0]) for _ in range(15)]
    torch.cuda.synchronize()
    print("[anerf_h train] losses", ["%.4f" % l for l in losses])
    assert all(l == l for l in losses) and losses[-1] < losses[0] - 0.01
    coarse1, fine1 = _flat(caster.network.parameters()), _flat(caster.network_fine.parameters())
    assert float((coarse1 - coarse0).abs().max()) > 0 and float((fine1 - fine0).abs().max()) > 0
    assert not torch.equal(coarse1, fine1)


# ---------------------------------------------------------------------------------------------------------------- 6
def test_anerf_h_checkpoint_round_trip():
    """TrainStep.save writes both networks and a 50-entry optimizer state in torch.optim.Adam's format (it loads into the
    Adam create_raycaster returns); a fresh caster resumed from the file takes the same next step."""
    from danbo_b200 import synthetic as syn, training
    fx = load_fixture("train_anerf")
    caster, _, _, _ = make_anerf_h_caster(fx)
    targs = _train_args(fx)
    b = syn.training_batch(2, 48, seed=6)
    b = {k: (v.to(DEV) if torch.is_tensor(v) else v) for k, v in b.items()}
    step = training.TrainStep(caster, targs)
    torch.manual_seed(5)
    for _ in range(3):
        step(b)
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "003.tar")
        step.save(path, 3)
        ckpt = torch.load(path, map_location=DEV, weights_only=False)
    assert {"network_fn_state_dict", "network_fine_state_dict", "optimizer_state_dict"} <= set(ckpt)
    sd = ckpt["optimizer_state_dict"]
    assert len(sd["state"]) == 50 and sd["param_groups"][0]["params"] == list(range(50))
    caster2, _, grad_vars2, optimizer2 = make_anerf_h_caster(fx)
    for i, p in enumerate(grad_vars2):
        assert tuple(sd["state"][i]["exp_avg"].shape) == tuple(p.shape), i
    optimizer2.load_state_dict(sd)                                    # the reference's Adam over grad_vars takes it
    caster2.load_state_dict(ckpt)
    step2 = training.TrainStep(caster2, targs)
    assert step2.resume(ckpt) == 3
    torch.manual_seed(9)
    loss_a, _ = step(b)
    torch.manual_seed(9)
    loss_b, _ = step2(b)
    torch.cuda.synchronize()
    pa, pb = _flat(step.bucket.params), _flat(step2.bucket.params)
    print(f"[anerf_h ckpt] next loss {float(loss_a):.6f} resumed {float(loss_b):.6f}  params max diff "
          f"{float((pa - pb).abs().max()):.3e}")
    assert abs(float(loss_a) - float(loss_b)) <= 1e-5 * abs(float(loss_a))
    assert float((pa - pb).abs().max()) <= 2e-4                       # one Adam step moves a weight by about lr


# ---------------------------------------------------------------------------------------------------------------- 7
@pytest.mark.skipif(not rh.available(), reason="no reference copy (run scripts/vendor_ref.sh)")
def test_reference_trainer_on_anerf_h_caster():
    """The reference's own Trainer.train_batch (core/trainer.py:257-300) with configs/h36m_zju/anerf_h.txt on this caster:
    same loss as TrainStep on the same batch and seed, same parameters after the step."""
    import danbo_b200 as db
    from danbo_b200 import training
    from test_gpu_dropin import N_POSES, RPP, _attrs as dropin_attrs, _ref_batch, _reference_cuda_defaults
    rc, run_nerf = rh._imports()
    from core.trainer import Trainer
    args = rh.parse_args("h36m_zju/anerf_h.txt", ["--N_rand", str(N_POSES * RPP), "--N_sample_images", str(N_POSES)])
    assert not args.single_net
    fx = {"weight_seed": 0}

    def load(caster):
        caster.network.load_state_dict(anerf_params(fx), strict=False)
        caster.network_fine.load_state_dict(fine_params(fx), strict=False)

    db.install()
    try:
        kw_train, kw_test, _, grad_vars, optimizer, _ = run_nerf.create_raycaster(args, dropin_attrs(),
                                                                                  device=torch.device(DEV))
    finally:
        db.uninstall()
    caster = kw_test["ray_caster"]
    assert isinstance(caster, db.RayCaster) and caster.network_fine is not caster.network and len(grad_vars) == 50
    load(caster)
    trainer = Trainer(args, dropin_attrs(), optimizer, None, kw_train, kw_test, popt_kwargs=None, device=torch.device(DEV))
    batch, b = _ref_batch(DEV)
    torch.manual_seed(11)
    caster.train()
    with _reference_cuda_defaults():
        loss_dict, _ = trainer.train_batch(batch, i=1, global_step=1)
    torch.cuda.synchronize()
    got = float(loss_dict["total_loss"])
    p_after = _flat(grad_vars)

    args2 = db.make_args("anerf_base", no_reload=True, single_net=False, N_samples=args.N_samples,
                         N_importance=args.N_importance, perturb=args.perturb, raw_noise_std=args.raw_noise_std,
                         lrate=args.lrate, loss_fn=args.loss_fn)
    _, kw2, _, grad_vars2, _, _ = db.create_raycaster(args2, dropin_attrs(), device=DEV)
    caster2 = kw2["ray_caster"]
    load(caster2)
    step = training.TrainStep(caster2, args2)
    b2 = {k: (v.to(DEV) if torch.is_tensor(v) else v) for k, v in b.items()}
    torch.manual_seed(11)
    loss2, _ = step(b2)
    torch.cuda.synchronize()
    p2 = _flat(grad_vars2)
    print(f"[anerf_h dropin] reference Trainer on this caster {got:.6f}  TrainStep {float(loss2):.6f}  params max diff "
          f"{float((p_after - p2).abs().max()):.3e}")
    assert abs(got - float(loss2)) <= 2e-5 * max(abs(float(loss2)), 1.0)
    assert float((p_after - p2).abs().max()) <= 2e-4
