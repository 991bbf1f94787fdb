"""A-NeRF pose refinement without a GPU: the closed form `danbo_anerf_embed_bwd` implements (d loss / d skts of the
A-NeRF encodings, given d loss / d the density and view inputs), restated in plain torch, against torch autograd of the
oracle's `anerf_inputs` with the world-to-bone matrices as a leaf.  fp64 on both sides, so the comparison pins the
derivation itself.  A second test compares the oracle's d skts with the original A-NeRF encoders' own autograd when a
copy of the original is given (it is the only check that would see a `.detach()` inside them)."""
import os
import sys

import pytest
import torch

import danbo_oracle as orc
from util import load_fixture, align_A, pose_tensors

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import ref_harness as rh  # noqa: E402

CUTOFF = orc.ANERF_CUTOFF


# "train_anerf_straddle": the train_anerf draw with 22 rays per pose and the last ray dropped (43 rays): danbo_anerf_embed_bwd
# reduces 4 rays per block, so one block holds rays of both poses and the last block has a ray-less warp.
CASES = ["render_anerf", "train_anerf", "train_anerf_straddle"]


def fixture_of(name):
    return "train_anerf" if name.startswith("train_anerf") else name


def anerf_case(name):
    """-> rays (N,8), z (N,S), pose_skts (G,24,4,4), rays_per_pose, tau: the coarse samples of a committed A-NeRF case."""
    fx = load_fixture(fixture_of(name))
    if name == "render_anerf":
        rays = fx["ray_batch"]
        return rays, fx["st.z.0"], pose_tensors(fx)[0], rays.shape[0], float(fx["tau"])
    from danbo_b200 import synthetic as syn
    n_poses, rpp = int(fx["n_poses"]), int(fx["rays_per_pose"])
    if name == "train_anerf_straddle":
        rpp = 22
    b = syn.training_batch(n_poses, rpp, seed=int(fx["batch_seed"]))
    if name == "train_anerf_straddle":
        b = {k: (v[:-1] if torch.is_tensor(v) and v.shape[0] == n_poses * rpp else v) for k, v in b.items()}
    rays = b["ray_batch"]
    near, far = orc.cylinder_near_far(rays[:, 0:3], rays[:, 3:6], b["cyls"], rays[:, 6:7], rays[:, 7:8])
    z = orc.coarse_z(near, far, int(fx["N_samples"]))
    return rays, z.contiguous(), b["skts"][::rpp].contiguous(), rpp, 20.


def oracle_skts_grad(rays, z, pose_skts, rpp, A, tau, d_xd, d_xv):
    """Autograd of sum(d_xd * density_inputs) + sum(d_xv * view_inputs[:, :648]) with respect to pose_skts."""
    N = rays.shape[0]
    leaf = pose_skts.clone().requires_grad_(True)
    pose = torch.clamp(torch.arange(N) // rpp, max=pose_skts.shape[0] - 1)
    pts = orc.ray_points(rays[:, 0:3], rays[:, 3:6], z)
    P = {"framecodes.codes.weight": torch.zeros(1, 128, dtype=rays.dtype)}
    dens, view, _ = orc.anerf_inputs(pts, rays[:, 3:6], torch.zeros(N, dtype=torch.long), leaf[pose], A, P, True, tau)
    ((dens * d_xd).sum() + (view[:, :648] * d_xv).sum()).backward()
    return leaf.grad


def closed_form_skts_grad(rays, z, pose_skts, rpp, A, tau, d_xd, d_xv, c=CUTOFF):
    """What danbo_anerf_embed_bwd computes, in plain torch (see csrc/anerf_bwd.cu for the derivation)."""
    N, S = z.shape
    G = pose_skts.shape[0]
    pose = torch.clamp(torch.arange(N) // rpp, max=G - 1)
    sk = pose_skts[pose]                                                   # (N,24,4,4)
    R, t = sk[:, :, :3, :3], sk[:, :, :3, 3]
    A3, a3 = A[:, :3, :3], A[:, :3, 3]
    o, d_ray = rays[:, 0:3], rays[:, 3:6]
    p = o[:, None, :] + d_ray[:, None, :] * z[..., None]                   # (N,S,3)
    q = torch.einsum("njab,nsb->nsja", R, p) + t[:, None]
    q = torch.einsum("jab,nsjb->nsja", A3, q) + a3                         # (N,S,24,3)
    v = q.norm(dim=-1)
    r = q / v[..., None]
    w = 1. - torch.sigmoid(tau * (v - c))
    wp = -tau * w * (1. - w)
    s = (c - v) * (2. / c) - 1.
    gd = d_xd.reshape(N, S, 432)
    gpe, gr = gd[..., :360].reshape(N, S, 15, 24), gd[..., 360:].reshape(N, S, 24, 3)
    fr = (2. ** torch.arange(7, dtype=z.dtype))[:, None]
    sn, cs = torch.sin(fr * s[..., None, :]), torch.cos(fr * s[..., None, :])            # (N,S,7,24)
    T = gpe[..., 0, :] * (c - v) + (gpe[..., 1::2, :] * sn + gpe[..., 2::2, :] * cs).sum(-2)
    B = -gpe[..., 0, :] - (2. / c) * (fr * (gpe[..., 1::2, :] * cs - gpe[..., 2::2, :] * sn)).sum(-2)
    # per ray: d_j = normalize(R_j d_ray) and its 4-octave encoding, rows [d, sin(2^f d), cos(2^f d)]
    lr = torch.einsum("njab,nb->nja", R, d_ray)
    ln = lr.norm(dim=-1)
    dj = lr / ln[..., None]                                                # (N,24,3)
    f4 = (2. ** torch.arange(4, dtype=z.dtype))[:, None, None]
    sd, cd = torch.sin(f4 * dj[:, None]), torch.cos(f4 * dj[:, None])      # (N,4,24,3)
    enc = torch.cat([dj[:, None], torch.stack([sd, cd], 2).flatten(1, 2)], 1)                         # (N,9,24,3)
    denc = torch.cat([torch.ones_like(dj)[:, None], torch.stack([f4 * cd, -f4 * sd], 2).flatten(1, 2)], 1)
    gv = d_xv.reshape(N, S, 9, 24, 3)
    T = T + (gv * enc[:, None]).sum((-3, -1))
    dd = (w[..., None] * (gv * denc[:, None]).sum(-3)).sum(1)             # (N,24,3)
    dv = wp * T + w * B
    dq = dv[..., None] * r + (gr - (r * gr).sum(-1, keepdim=True) * r) / v[..., None]
    dl = torch.einsum("jab,nsja->nsjb", A3, dq)                           # A^T dq
    ph = torch.cat([p, torch.ones_like(p[..., :1])], -1)
    g = torch.einsum("nsja,nsc->njac", dl, ph)                            # (N,24,3,4)
    dm = (dd - (dj * dd).sum(-1, keepdim=True) * dj) / ln[..., None]
    g[..., :3] = g[..., :3] + torch.einsum("nja,nb->njab", dm, d_ray)
    out = torch.zeros(G, 24, 4, 4, dtype=z.dtype)
    out[:, :, :3, :] = torch.zeros(G, 24, 3, 4, dtype=z.dtype).index_add_(0, pose, g)
    return out


def random_input_grads(n_rows, seed, dtype=torch.float32):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(n_rows, 432, generator=g).to(dtype), torch.randn(n_rows, 648, generator=g).to(dtype)


@pytest.mark.parametrize("name", CASES)
def test_closed_form_matches_oracle_autograd(name):
    rays, z, pose_skts, rpp, tau = anerf_case(name)
    N, S = z.shape
    d_xd, d_xv = random_input_grads(N * S, 7, torch.float64)
    dt = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        args = (rays.double(), z.double(), pose_skts.double(), rpp, align_A().double(), tau, d_xd, d_xv)
        want = oracle_skts_grad(*args)
        got = closed_form_skts_grad(*args)
    finally:
        torch.set_default_dtype(dt)
    rel = float((got - want).norm() / want.norm())
    print(f"[anerf pose grad] {name}: {pose_skts.shape[0]} poses, |g| {float(want.norm()):.3e} rel {rel:.3e}")
    assert float(want[:, :, 3].abs().max()) == 0.0 and float(got[:, :, 3].abs().max()) == 0.0
    assert rel <= 1e-6, rel


@pytest.mark.skipif(not rh.available(), reason="needs the original DANBO-pytorch (DANBO_REFERENCE or baseline/_ref)")
def test_oracle_pose_grad_matches_reference_encoders():
    """The original's A-NeRF encoders (encode_pts / encode_views of its NeRF network, reached through its own ray caster)
    under autograd, with the world-to-bone matrices as a leaf, against the oracle's d skts on the same coarse samples."""
    from danbo_b200 import params, synthetic as syn
    args = rh.parse_args("h36m_zju/anerf_base.txt", ["--N_samples", "16", "--N_importance", "8"])
    caster, kw = rh.build(args, syn.rest_pose())
    caster.eval()
    rh.load_weights(caster, syn.synth_state_dict(params.anerf_param_shapes(), 3))
    pose = syn.make_pose(9)
    full = syn.render_batch(pose, 32, 32)
    g = torch.Generator().manual_seed(9)
    N = 24
    pick = torch.sort(torch.randperm(full["ray_batch"].shape[0], generator=g)[:N]).values
    b = {k: (v[pick].contiguous() if torch.is_tensor(v) and v.shape[0] == full["ray_batch"].shape[0] else v)
         for k, v in full.items()}
    leaf = torch.as_tensor(pose["skts"])[None].float().clone().requires_grad_(True)
    net, seen = caster.network, {}
    orig_pts, orig_views, orig_sample = net.encode_pts, net.encode_views, caster.sample_pts

    def enc_pts(*a, **k):
        out = orig_pts(*a, **k)
        seen.setdefault("dens", out[0])
        return out

    def enc_views(*a, **k):
        out = orig_views(*a, **k)
        seen.setdefault("view", out[0])
        return out

    def sample_pts(*a, **k):
        out = orig_sample(*a, **k)
        seen.setdefault("z", out[1])
        return out
    net.encode_pts, net.encode_views, caster.sample_pts = enc_pts, enc_views, sample_pts
    try:
        kwargs = {k: v for k, v in kw.items() if k not in ("ray_caster", "N_samples", "use_viewdirs")}
        with torch.enable_grad():
            caster(b["ray_batch"], N_samples=args.N_samples, kp_batch=b["kp_batch"], skts=leaf.expand(N, -1, -1, -1),
                   cyls=b["cyls"], bones=b["bones"], cams=b["cams"], N_uniques=1, **kwargs)
    finally:
        del net.encode_pts, net.encode_views, caster.sample_pts
    z = seen["z"].detach().reshape(N, -1)
    S = z.shape[1]
    d_xd, d_xv = random_input_grads(N * S, 11)
    loss = (seen["dens"].reshape(N * S, -1) * d_xd).sum() + (seen["view"].reshape(N * S, -1)[:, :648] * d_xv).sum()
    assert loss.requires_grad, "the original's encoders do not depend on skts under autograd"
    (want,) = torch.autograd.grad(loss, leaf)
    got = oracle_skts_grad(b["ray_batch"], z, leaf.detach(), N, align_A(), float(net.pe_fn.get_tau()), d_xd, d_xv)
    rel = float((got - want).norm() / want.norm())
    print(f"[anerf pose grad] original's encoders: |g| {float(want.norm()):.3e} rel {rel:.3e}")
    assert rel <= 1e-4, rel
