"""The closed forms the pose kernels compute (csrc/pose.cu, danbo_graph_net_bwd_pose in csrc/graphnet.cu,
csrc/rotation.cuh), restated in torch and held against fp64 autograd of the PyTorch pose path; and what a captured
--opt_pose step refuses.  CPU only."""
import os
import sys
import types

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import danbo_b200                                    # noqa: E402,F401
from danbo_b200 import networks, pose_opt as po, skeleton as sk, training   # noqa: E402

FX = np.load(os.path.join(ROOT, "tests", "golden", "popt.npz"))
T = lambda k: torch.tensor(FX[k]).double()
PARENTS = [int(p) for p in sk.JOINT_PARENTS]


def rel(a, b):
    return float((a - b).abs().max() / b.abs().max().clamp(min=1e-30))


# ---- closed forms (the kernels' arithmetic, in fp64) ---------------------------------------------------------------
def aa_bwd(aa, g):
    """d aa of axisang_to_rot for d R = g (...,3,3): rotation.cuh axisang_to_rot_bwd."""
    ax, ay, az = aa.unbind(-1)
    ang = aa.norm(dim=-1)
    half = 0.5 * ang
    small = ang.abs() < 1e-6
    sh, ch = torch.sin(half), torch.cos(half)
    safe = torch.where(small, torch.ones_like(ang), ang)
    k = torch.where(small, 0.5 - ang * ang / 48, sh / safe)
    r, i, j, kk = ch, ax * k, ay * k, az * k
    s = 2.0 / (r * r + i * i + j * j + kk * kk)
    g = g.reshape(*g.shape[:-2], 9).unbind(-1)
    ds = (-(j * j + kk * kk) * g[0] + (i * j - kk * r) * g[1] + (i * kk + j * r) * g[2] + (i * j + kk * r) * g[3]
          - (i * i + kk * kk) * g[4] + (j * kk - i * r) * g[5] + (i * kk - j * r) * g[6] + (j * kk + i * r) * g[7]
          - (i * i + j * j) * g[8])
    dn = -0.5 * s * s * ds
    dr = s * (-kk * g[1] + j * g[2] + kk * g[3] - i * g[5] - j * g[6] + i * g[7]) + 2 * r * dn
    di = s * (j * g[1] + kk * g[2] + j * g[3] - 2 * i * g[4] - r * g[5] + kk * g[6] + r * g[7] - 2 * i * g[8]) + 2 * i * dn
    dj = s * (-2 * j * g[0] + i * g[1] + r * g[2] + i * g[3] + kk * g[5] - r * g[6] + kk * g[7] - 2 * j * g[8]) + 2 * j * dn
    dk = s * (-2 * kk * g[0] - r * g[1] + i * g[2] + r * g[3] - 2 * kk * g[4] + j * g[5] + i * g[6] + j * g[7]) + 2 * kk * dn
    dkk = di * ax + dj * ay + dk * az
    dkdang = torch.where(small, -ang / 24, (0.5 * ch * ang - sh) / (safe * safe))
    dang = -0.5 * sh * dr + dkdang * dkk
    u = torch.where(ang > 0, dang / torch.where(ang > 0, ang, torch.ones_like(ang)), torch.zeros_like(ang))
    return torch.stack([di * k + u * ax, dj * k + u * ay, dk * k + u * az], -1)


def chain_bwd(aa, rest, pelvis, d_skts, d_kps):
    """danbo_pose_bwd's chain: d (skts, kps) of G poses -> d aa (G,24,3), d pelvis (G,3)."""
    Rl = po.axisang_to_rot(aa)
    G = aa.shape[0]
    R, t = [None] * 24, [None] * 24
    R[0], t[0] = Rl[:, 0], rest[:, 0]
    for jj in range(1, 24):
        p = PARENTS[jj]
        R[jj] = R[p] @ Rl[:, jj]
        t[jj] = (R[p] @ (rest[:, jj] - rest[:, p])[..., None])[..., 0] + t[p]
    R, t = torch.stack(R, 1), torch.stack(t, 1) + pelvis[:, None]
    db = d_skts[..., :3, 3]
    dR = d_skts[..., :3, :3].transpose(-1, -2) - t[..., :, None] * db[..., None, :]
    dt = -(R @ db[..., None])[..., 0] + d_kps
    dR, dt = list(dR.unbind(1)), list(dt.unbind(1))
    for jj in range(23, 0, -1):                           # parents precede children in the SMPL table
        p = PARENTS[jj]
        off = rest[:, jj] - rest[:, p]
        dR[p] = dR[p] + dR[jj] @ Rl[:, jj].transpose(-1, -2) + dt[jj][..., :, None] * off[..., None, :]
        dt[p] = dt[p] + dt[jj]
    dRl = torch.stack([dR[0]] + [R[:, PARENTS[jj]].transpose(-1, -2) @ dR[jj] for jj in range(1, 24)], 1)
    return aa_bwd(aa, dRl), dt[0]


def pe_rot6d_bwd(aa, keep, dw):
    """danbo_graph_net_bwd_pose after d w_in: through the 5-octave PE (sin / cos from the saved inputs) and rot6d."""
    dx = dw[..., :6].clone()
    for f in range(5):
        dx = dx + 2.0 ** f * (keep[..., 12 + 12 * f:18 + 12 * f] * dw[..., 6 + 12 * f:12 + 12 * f]
                              - keep[..., 6 + 12 * f:12 + 12 * f] * dw[..., 12 + 12 * f:18 + 12 * f])
    g = torch.zeros(*aa.shape[:-1], 3, 3, dtype=aa.dtype)
    g[..., :, :2] = dx.reshape(*aa.shape[:-1], 3, 2)
    return aa_bwd(aa, g)


def _gather_case(tag, idxs):
    """(layer in fp64, per-pose aa, rest, pelvis, scatter of per-pose d aa / d pelvis into the parameter gradients)."""
    sd = {k[len(tag) + 4:]: torch.tensor(FX[k]) for k in FX.files if k.startswith(tag + ".sd.")}
    layer = po.load_poseopt_from_state_dict({"poseopt_layer_state_dict": sd}).double()
    idx = torch.as_tensor(idxs)
    pelvis, aa = layer.idx_to_params(idx)
    rest = layer.get_rest_pose(idx).expand(len(idx), 24, 3)

    def scatter(d_aa, d_pel):
        g = {"pelvis": torch.zeros_like(layer.pelvis).index_add_(0, idx, d_pel)}
        if layer.kp_map is None:
            g["bones"] = torch.zeros_like(layer.bones).index_add_(0, idx, d_aa)
        else:
            g["root_bones"] = torch.zeros_like(layer.root_bones).index_add_(0, idx, d_aa[:, 0])
            g["bones"] = torch.zeros_like(layer.bones).index_add_(0, layer.kp_map[idx], d_aa[:, 1:])
        return g
    return layer, aa.detach(), rest.detach(), pelvis.detach(), scatter


def _check_layer(layer, idxs, aa, rest, pelvis, scatter, seed=0):
    gen = torch.Generator().manual_seed(seed)
    wk = torch.randn(len(idxs), 24, 3, generator=gen, dtype=torch.float64)
    ws = torch.randn(len(idxs), 24, 4, 4, generator=gen, dtype=torch.float64)
    wb = torch.randn(len(idxs), 24, 3, generator=gen, dtype=torch.float64)
    kps, bones, skts, _, _ = layer.calculate_kinematic(idxs)
    ((kps * wk).sum() + (skts * ws).sum() + (bones * wb).sum()).backward()
    d_aa, d_pel = chain_bwd(aa, rest, pelvis, ws, wk)
    got = scatter(d_aa + wb, d_pel)
    for n, p in layer.named_parameters():
        assert rel(got[n], p.grad) < 1e-12, (n, rel(got[n], p.grad))


# ---- tests ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tag", ["axisang", "multiview"])
def test_chain_backward_matches_autograd_on_the_fixture(tag):
    idxs = FX["idxs"]                                     # 12 draws of 7 frames: duplicates included
    assert len(set(idxs.tolist())) < len(idxs)
    layer, aa, rest, pelvis, scatter = _gather_case(tag, idxs)
    _check_layer(layer, idxs, aa, rest, pelvis, scatter)


def test_chain_backward_with_per_frame_rest_poses_and_small_angles():
    bones = T("init_bones").clone()
    bones[2] *= 1e-8                                      # the small-angle branch
    bones[3, :5] = 0.0                                    # exactly zero: the norm gets no gradient
    rest = torch.cat([T("rest_pose"), T("rest_pose") * 1.1], 0)
    table = np.array([0, 1, 0, 1, 1, 0, 1])
    layer = po.PoseOptLayer(T("init_kps"), bones, rest, rest_pose_idxs=table).double()
    idxs = np.array([2, 3, 3, 5, 1, 2])
    idx = torch.as_tensor(idxs)
    pelvis, aa = layer.idx_to_params(idx)

    def scatter(d_aa, d_pel):
        return {"pelvis": torch.zeros_like(layer.pelvis).index_add_(0, idx, d_pel),
                "bones": torch.zeros_like(layer.bones).index_add_(0, idx, d_aa)}
    _check_layer(layer, idxs, aa.detach(), layer.rest_pose[torch.as_tensor(table)[idx]], pelvis.detach(), scatter, seed=3)


def test_axisang_backward_small_and_zero_angles():
    rng = np.random.RandomState(0)
    aa = torch.tensor(rng.randn(64, 3))
    aa[:8] *= 1e-8
    aa[8:10] = 0.0
    aa[10] = torch.tensor([3.1, 0.2, -0.1])
    aa.requires_grad_(True)
    g = torch.randn(64, 3, 3, dtype=torch.float64, generator=torch.Generator().manual_seed(1))
    (po.axisang_to_rot(aa) * g).sum().backward()
    got = aa_bwd(aa.detach(), g)
    assert float((got - aa.grad).abs().max()) <= 1e-12 * float(aa.grad.abs().max())
    assert torch.equal(got[8:10], aa.grad[8:10])


def test_graph_net_pose_backward_matches_autograd():
    """d pre0 -> d axis-angle: the transposed adjacency mix, W0[j], mask_root, the PE and rot6d (graphnet.cu)."""
    torch.manual_seed(0)
    gn = networks.GraphNet().double()
    G = 5
    aa = torch.randn(G, 24, 3, dtype=torch.float64) * 0.7
    aa[1, 4] *= 1e-9
    aa.requires_grad_(True)
    w = networks.pe_embed(networks.axis_angle_to_matrix(aa)[..., :3, :2].flatten(start_dim=-2), 5)
    pre0 = gn.layers[0](gn.mask * w)
    d_pre0 = torch.randn_like(pre0)
    (pre0 * d_pre0).sum().backward()
    A = gn.layers[0].get_adjw().detach()[0]                                   # (24,24)
    d_lin = torch.einsum("jk,gjc->gkc", A, d_pre0)
    dw = torch.einsum("kic,gkc->gki", gn.layers[0].lin.weight.detach(), d_lin) * gn.mask
    keep = (w * gn.mask).detach()                                             # what the forward saves (root zeroed)
    got = pe_rot6d_bwd(aa.detach(), keep, dw)
    assert torch.equal(got[:, 0], torch.zeros_like(got[:, 0]))
    for g in range(G):
        assert rel(got[g], aa.grad[g]) < 1e-12, (g, rel(got[g], aa.grad[g]))


@pytest.mark.parametrize("tol", [0.0, 0.002])
def test_regulariser_closed_form_matches_kp_loss(tol):
    G, skip = 4, 3
    frames = torch.tensor([1, 4, 6, 4])
    anchors = {"kps": T("init_kps"), "bones": T("init_bones"), "rots": None}
    per_pose = (T("init_bones")[frames] + 0.05 * torch.randn(G, 24, 3, dtype=torch.float64,
                                                             generator=torch.Generator().manual_seed(2))).requires_grad_(True)
    kps = T("init_kps")[frames] + 0.01
    ex = lambda t: t[:, None].expand(G, skip, *t.shape[1:]).reshape(G * skip, *t.shape[1:])
    args = types.SimpleNamespace(opt_rot6d=False, opt_pose_tol=tol, opt_pose_coef=2.0, use_temp_loss=False, ext_scale=0.001)
    losses, stats = po.kp_loss(args, anchors, frames.repeat_interleave(skip), {"kp_batch": ex(kps), "bones": ex(per_pose),
                                                                                "rots": None})
    losses["kp_loss"].backward()
    # danbo_pose_fwd / danbo_pose_bwd on the G poses: coef * mean over (pose, joint >= 1) of the hinge, gradient
    # coef * 2 (aa - anchor) / (G * 23) where the square exceeds tol
    e = (per_pose.detach() - anchors["bones"][frames])[:, 1:]
    hinge = torch.where(e * e > tol, e * e - tol, torch.zeros_like(e))
    assert abs(float(hinge.sum() / (G * 23) * 2.0) - float(losses["kp_loss"].detach())) <= 1e-12
    grad = torch.zeros_like(per_pose)
    grad[:, 1:] = torch.where(e * e > tol, 2.0 * 2.0 * e / (G * 23), torch.zeros_like(e))
    assert rel(grad, per_pose.grad) < 1e-12
    mpjpc = (anchors["kps"][frames] - kps).norm(dim=-1).mean() / 0.001
    assert abs(float(mpjpc) - float(stats["MPJPC"])) <= 1e-9 * float(mpjpc)


def _stand_in(graph_net=True, fine=False):
    class Net(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.w = torch.nn.Parameter(torch.full((3,), 0.5))
            if graph_net:
                self.graph_net = torch.nn.Linear(1, 1)

    class Caster(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.network = Net()
            if fine:
                self.network_fine = Net()
    return Caster()


def _popt(**kw):
    args = types.SimpleNamespace(opt_rot6d=False, opt_pose_lrate=1e-2, init_poseopt=None, no_poseopt_reload=False,
                                 use_ckpt_anchor=False, opt_pose_cache=False, opt_pose_tol=0.0, opt_pose_coef=2.0,
                                 use_temp_loss=False, ext_scale=0.001, lrate=1e-2, loss_fn="L1", agg_type="sigmoid")
    for k, v in kw.items():
        setattr(args, k, v)
    attrs = {"rest_pose": FX["rest_pose"], "betas": np.zeros((1, 10), np.float32), "kp3d": FX["init_kps"],
             "bones": FX["init_bones"]}
    opt, popt = po.create_popt(args, attrs)
    return args, opt, popt


@pytest.mark.parametrize("case,word", [("anerf", "A-NeRF"), ("fine", "fine network"), ("world", "world_size"),
                                       ("rot6d", "opt_rot6d"), ("temp", "use_temp_loss"), ("cache", "opt_pose_cache"),
                                       ("adam", "FlatAdam")])
def test_graph_capture_refusals(case, word):
    args, opt, popt = _popt(opt_rot6d=case == "rot6d", use_temp_loss=case == "temp", opt_pose_cache=case == "cache")
    caster = _stand_in(graph_net=case != "anerf", fine=case == "fine")
    grads = [p.grad for p in caster.network.parameters()]
    with pytest.raises(NotImplementedError, match=word):
        training.TrainStep(caster, args, popt_kwargs=popt, pose_optimizer=opt, graph=True,
                           world_size=2 if case == "world" else 1)
    assert [p.grad for p in caster.network.parameters()] == grads        # refused before anything was set up


def test_graph_capture_refuses_batches_without_equal_runs():
    assert training.pose_batch_poses({"kp_idx": torch.zeros(12, dtype=torch.long), "N_uniques": 4}) == (4, 3)
    with pytest.raises(NotImplementedError, match="unique"):
        training.pose_batch_poses({"kp_idx": torch.zeros(10, dtype=torch.long), "N_uniques": 4})


def test_flat_pose_optimizer_needs_cuda():
    args = types.SimpleNamespace(opt_pose_lrate=1e-3)
    attrs = {"rest_pose": FX["rest_pose"], "betas": np.zeros((1, 10), np.float32), "kp3d": FX["init_kps"],
             "bones": FX["init_bones"]}
    with pytest.raises(RuntimeError, match="CUDA"):
        po.create_popt(args, attrs, flat=True)
