"""Pose refinement on the perfcap configs without a GPU.  There the view branch encodes the ray direction in the root
joint's frame (ray_tr_type=root_local, view_type=relray), so d loss / d ray_bias also reaches the root rotation.  The
closed form `danbo_view_root_bwd` implements is restated in plain torch and compared with fp64 autograd of the oracle's
`view_inputs(view_directions(rays_d, skts, "root_local"))` contracted with W_v[:, 256:] and a random d ray_bias, with
the world-to-bone matrices as a leaf."""
import pytest
import torch

import danbo_oracle as orc
from util import load_fixture, params_for, pose_tensors

# "train_perfcap_straddle": the train_perfcap draw at 2 poses x 22 rays with the last ray dropped (43 rays).  The kernel
# reduces 32 rays per block, so its first block holds rays of both poses and its second has lanes without a ray.
# "train_perfcap_unnormalised": the train_perfcap rays with each direction scaled by a factor in [0.3, 3).
CASES = ["render_perfcap", "train_perfcap", "train_perfcap_straddle", "train_perfcap_unnormalised"]


def fixture_of(name):
    return "train_perfcap" if name.startswith("train_perfcap") else name


def perfcap_case(name):
    """-> rays (N,>=8), pose_skts (G,24,4,4), rays_per_pose, W_v (128,411), cams (N,): a committed perfcap case."""
    fx = load_fixture(fixture_of(name))
    Wv = params_for(fx)["views_linears.0.weight"]
    if name == "render_perfcap":
        rays = fx["ray_batch"]
        return rays, pose_tensors(fx)[0], rays.shape[0], Wv, fx["cams"].reshape(-1)
    from danbo_b200 import synthetic as syn
    n_poses, rpp = int(fx["n_poses"]), int(fx["rays_per_pose"])
    if name == "train_perfcap_straddle":
        n_poses, rpp = 2, 22
    b = syn.training_batch(n_poses, rpp, seed=int(fx["batch_seed"]))
    rays = b["ray_batch"].clone()
    if name == "train_perfcap_straddle":
        b = {k: (v[:-1] if torch.is_tensor(v) and v.shape[0] == n_poses * rpp else v) for k, v in b.items()}
        rays = b["ray_batch"].clone()
    if name == "train_perfcap_unnormalised":
        g = torch.Generator().manual_seed(4)
        rays[:, 3:6] *= 0.3 + 2.7 * torch.rand(rays.shape[0], 1, generator=g)
    return rays.contiguous(), b["skts"][::rpp].contiguous(), rpp, Wv, b["cams"].reshape(-1)


def random_ray_bias_grad(n, seed, dtype=torch.float32):
    return torch.randn(n, 128, generator=torch.Generator().manual_seed(seed)).to(dtype)


def oracle_skts_grad(rays, pose_skts, rpp, Wv, cams, d_ray_bias):
    """Autograd of sum(d_ray_bias * (view_inputs . W_v[:, 256:]^T)) with respect to pose_skts."""
    N = rays.shape[0]
    leaf = pose_skts.clone().requires_grad_(True)
    pose = torch.clamp(torch.arange(N) // rpp, max=pose_skts.shape[0] - 1)
    P = {"framecodes.codes.weight": torch.randn(8, 128, generator=torch.Generator().manual_seed(1)).to(rays.dtype)}
    v = orc.view_inputs(orc.view_directions(rays[:, 3:6], leaf[pose], "root_local"), cams, P, True)
    ((v @ Wv[:, 256:].t()) * d_ray_bias).sum().backward()
    return leaf.grad


def closed_form_skts_grad(rays, pose_skts, rpp, Wv, d_ray_bias):
    """What danbo_view_root_bwd computes, in plain torch (see csrc/backward_mlp.cu for the derivation)."""
    N, G = rays.shape[0], pose_skts.shape[0]
    pose = torch.clamp(torch.arange(N) // rpp, max=G - 1)
    d = rays[:, 3:6]
    m = (pose_skts[pose, 0, :3, :3] @ d[..., None])[..., 0]
    nrm = m.norm(dim=-1, keepdim=True).clamp_min(1e-12)
    dn = m / nrm
    g = d_ray_bias @ Wv[:, 256:283]                                     # (N,27) = [dn, (sin, cos)(2^f dn) for f < 4]
    fr = (2. ** torch.arange(4, dtype=rays.dtype))[:, None]             # (4,1)
    x = dn[:, None, :] * fr                                             # (N,4,3)
    gsc = g[:, 3:].reshape(N, 4, 2, 3)
    ddn = g[:, :3] + (fr * (gsc[:, :, 0] * torch.cos(x) - gsc[:, :, 1] * torch.sin(x))).sum(1)
    dm = (ddn - (dn * ddn).sum(-1, keepdim=True) * dn) / nrm
    out = torch.zeros(G, 24, 4, 4, dtype=rays.dtype)
    out[:, 0, :3, :3] = torch.zeros(G, 3, 3, dtype=rays.dtype).index_add_(0, pose, dm[:, :, None] * d[:, None, :])
    return out


@pytest.mark.parametrize("name", CASES)
def test_closed_form_matches_oracle_autograd(name):
    rays, pose_skts, rpp, Wv, cams = perfcap_case(name)
    N = rays.shape[0]
    d_rb = random_ray_bias_grad(N, 7, torch.float64)
    args = (rays.double(), pose_skts.double(), rpp, Wv.double())
    want = oracle_skts_grad(*args, cams, d_rb)
    got = closed_form_skts_grad(*args, d_rb)
    rel = float((got - want).norm() / want.norm())
    print(f"[perfcap pose grad] {name}: {N} rays, {pose_skts.shape[0]} poses, |g| {float(want.norm()):.3e} rel {rel:.3e}")
    assert rel <= 1e-12, rel
    for g in range(pose_skts.shape[0]):                                 # every pose receives its own rays' share
        assert float((got[g] - want[g]).norm()) <= 1e-12 * float(want.norm())
        assert float(want[g, 0, :3, :3].norm()) > 0
    # only the root rotation depends on the view branch: joint 0's translation column, its homogeneous row and
    # joints 1-23 get exactly zero, from autograd and from the closed form
    for t in (want, got):
        assert float(t[:, 0, :, 3].abs().max()) == 0.0 and float(t[:, 0, 3, :].abs().max()) == 0.0
        assert float(t[:, 1:].abs().max()) == 0.0


def test_entry_point_validates_arguments_without_touching_the_gpu():
    from danbo_b200 import _lib, build, kernels
    build.build()
    lib = _lib.load()
    N = None
    assert lib.danbo_view_root_bwd(N, 11, 0, N, 1, 1, N, N, N, N) == 0                 # no rays: nothing to do
    assert lib.danbo_view_root_bwd(N, 11, 16, N, 16, 1, N, N, N, N) < 0                # NULL pointers
    with pytest.raises(RuntimeError):                                                  # no CPU path
        kernels.view_root_bwd(torch.zeros(4, 11), torch.zeros(1, 24, 4, 4), 4, torch.zeros(128, 411),
                              torch.zeros(4, 128), torch.zeros(1, 24, 4, 4))
