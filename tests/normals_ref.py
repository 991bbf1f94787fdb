"""fp64 reference of d sigma / d p for the surface-normal tests: the body of `danbo_oracle.density_grid` at arbitrary
points, differentiable, with the feature window optionally kept in the graph (the oracle's `bone_features` detaches it,
as training does; a surface normal needs the true derivative)."""
import torch
import torch.nn.functional as F

import danbo_oracle as orc


def bone_features(pts_t, vol, axis_scale, rays_per_pose, detach_window=True, res=16, feat=5):
    """`danbo_oracle.bone_features` (same closed form of the grid_sample call) with `detach_window` as a choice:
    pts_t (N,S,24,3), vol (G,24,240), axis_scale (24,3) -> h (N,S,24,15), invalid (N,S,24)."""
    N, S = pts_t.shape[:2]
    J = orc.J
    x = pts_t / axis_scale.reshape(1, 1, -1, 3).abs()
    win = torch.exp(-2 * ((x ** 6).sum(-1)))
    if detach_window:
        win = win.detach()                                          # gnn_backbone.py:804
    invalid = ((x.abs() > 1).sum(-1) > 0).to(x.dtype)
    G = vol.shape[0]
    pose = torch.clamp(torch.arange(N) // rays_per_pose, max=G - 1)
    table = vol.reshape(G, J, feat, res, 3)[pose]                        # (N,24,5,16,3)
    iy = ((x + 1.) * res - 1.) / 2.
    i0 = torch.floor(iy)
    w1 = iy - i0
    w0 = 1. - w1
    i0 = i0.long()
    i1 = i0 + 1

    def tap(idx):
        ok = ((idx >= 0) & (idx < res)).to(x.dtype)
        idc = idx.clamp(0, res - 1)
        t = table[:, None].expand(N, S, J, feat, res, 3)
        g = torch.gather(t, 4, idc[:, :, :, None, None, :].expand(N, S, J, feat, 1, 3)).squeeze(4)
        return g * ok[:, :, :, None, :]

    val = tap(i0) * w0[:, :, :, None, :] + tap(i1) * w1[:, :, :, None, :]
    return val.flatten(start_dim=-2) * win[..., None], invalid


def _hbar(pts, skts, bones, A, P, agg_type, detach_window):
    pts = pts.reshape(-1, 1, 3)
    vol = orc.graph_net(orc.graph_inputs(bones), P)
    pts_t = orc.world_to_bone(pts, skts.expand(pts.shape[0], -1, -1, -1), A)
    h, invalid = bone_features(pts_t, vol, P["graph_net.axis_scale"], pts.shape[0], detach_window=detach_window)
    hf = h.reshape(-1, orc.J, 15)
    p = orc.agg_prob(orc.agg_net(hf, P), invalid.reshape(-1, orc.J), agg_type)
    return (hf * p[..., None]).sum(-2)


def density_at_points(pts, skts, bones, A, P, agg_type="sigmoid", detach_window=True):
    """Raw sigma (M,) at world points pts (M,3) for one pose (skts (1,24,4,4), bones (1,24,3)): what
    `danbo_oracle.density_grid` evaluates at its lattice points, differentiable in pts, skts and P (run it in fp64 for
    gradient references).  detach_window=False differentiates the feature window as well."""
    x = orc.pe_embed(_hbar(pts, skts, bones, A, P, agg_type, detach_window), 6)
    return F.linear(orc.density_trunk(x, P), P["alpha_linear.weight"], P["alpha_linear.bias"])[:, 0]


def density_bf16_trunk(pts, skts, bones, A, P, agg_type="sigmoid"):
    """density_at_points (window differentiated) with the MLP trunk's operands rounded as the tensor-core kernel rounds
    them (bf16 weights, inputs and stored activations, fp32 sigma head), through a straight-through estimator: forward
    values are the kernel's arithmetic, the backward is calculus on them (as `util.field_mlp_bf16_ste`)."""
    bf = lambda t: t + (t.to(torch.bfloat16).to(t.dtype) - t).detach()
    xb = bf(orc.pe_embed(_hbar(pts, skts, bones, A, P, agg_type, False), 6))
    x, a = xb, None
    for i in range(8):
        a = F.relu(x @ bf(P[f"pts_linears.{i}.weight"]).t() + P[f"pts_linears.{i}.bias"])
        x = bf(a)
        if i == 4:
            x = torch.cat([xb, x], -1)
    return (a @ P["alpha_linear.weight"].t() + P["alpha_linear.bias"])[:, 0]
