"""CPU oracle for the DANBO per-sample body-field hot path.  TEST INFRASTRUCTURE ONLY.

This file restates, in plain torch-on-CPU tensor arithmetic (fp32, fp64 where the reference uses it),
the algorithm of the reference for every row of SURVEY.md §8(a).  Only tests/, __graft_entry__.smoke()
and bench.py's cpu_baseline / --impl reference legs may import it; the product path (the package under
danbo-pytorch_b200/) never does and fails loudly when its CUDA library is missing.

Pinning: the reference ships no tests or golden vectors (SURVEY §4), so the pins are outputs of the reference
itself, produced by oracle/gen_golden.py (which imports the reference) and committed under tests/golden/.
tests/test_oracle_golden.py checks every function below against them.

Every function names the reference file:line it follows.  `P` is a flat dict of parameters keyed by the
reference's own state_dict names (SURVEY appendix A), e.g. P["pts_linears.0.weight"].
"""
import math
import numpy as np
import torch
import torch.nn.functional as F

J = 24
PARENTS = [0, 0, 0, 0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 9, 9, 12, 13, 14, 16, 17, 18, 19, 20, 21]


# ----------------------------------------------------------------------------------------------------------
# NF1  core/utils/ray_utils.py:294-346  get_near_far_in_cylinder
# ----------------------------------------------------------------------------------------------------------
def cylinder_near_far(rays_o, rays_d, cyl, near, far):
    """2-D ray/circle intersection in the x-z ground plane; NaN rows take the chunk-wide nanmean (F8)."""
    g = [0, -1]
    r_near = (rays_o + rays_d * near)[..., g]
    r_far = (rays_o + rays_d * far)[..., g]
    radius, center = cyl[..., 2:3], cyl[..., :2]
    nc = center - r_near
    nf = r_far - r_near
    nf_norm = torch.norm(nf, dim=-1, p=2)
    scale = torch.norm(rays_d[..., g], dim=-1, p=2)[..., None]
    cross = nc[..., 0] * nf[..., 1] - nc[..., 1] * nf[..., 0]
    dist = (torch.abs(cross) / nf_norm)[..., None]
    Q = (radius.pow(2) - dist.pow(2)).pow(0.5)
    K = ((nc * nf).sum(-1) / nf_norm)[..., None]
    mask = (Q < K).float()
    new_near = near + mask * (K - Q) / scale
    new_far = near + (K + Q) / scale
    if torch.isnan(new_near).any():
        idx = torch.where(torch.isnan(Q))[0]
        avg_near = np.nanmean(new_near.numpy())
        new_near[idx, :] = float(avg_near) if not np.isnan(avg_near) else near[idx, :]
        avg_far = np.nanmean(new_far.numpy())
        new_far[idx, :] = float(avg_far) if not np.isnan(avg_far) else far[idx, :]
    return new_near, new_far


# ----------------------------------------------------------------------------------------------------------
# NF2  core/raycasters.py:648-707 GraphCaster.get_near_far + core/utils/ray_utils.py:383-417
# ----------------------------------------------------------------------------------------------------------
def box_near_far(rays_o, rays_d, skts, A, axis_scale, near, far, bound=1.3, eps=1e-4):
    """Per-bone OBB test in fp64; a box counts only with exactly two of six plane hits inside (F7).
    Returns near, far (N,1) and the masks p_valid (N,24,6), v_valid (N,24)."""
    B = rays_o.shape[0]
    o_t = (skts[..., :3, :3] @ rays_o.reshape(B, 1, 3, 1) + skts[..., :3, -1:]).reshape(B, J, 3)
    d_t = (skts[..., :3, :3] @ rays_d.reshape(B, 1, 3, 1)).reshape(B, J, 3)
    A1 = A[None]                                            # (1,24,4,4)
    o_t = ((A1[..., :3, :3] @ o_t[..., None]) + A1[..., :3, -1:]).reshape(B, J, 3)
    d_t = (A1[..., :3, :3] @ d_t[..., None]).reshape(B, J, 3)
    s = axis_scale.reshape(1, J, 3).abs()
    o_s, d_s = o_t / s, d_t / s
    bounds = bound * torch.ones(1, J, 2, 3)
    bounds[..., 0, :] *= -1
    t = (bounds.double() - o_s[..., None, :]) / d_s[..., None, :]
    t = t.reshape(B, J, 6, 1)
    hit = (t * d_s[..., None, :] + o_s[..., None, :]).float()
    inside = torch.ones(hit.shape[:-1], dtype=torch.bool)
    for a in range(3):
        inside = inside & (hit[..., a] <= (bound + eps)) & (hit[..., a] >= (-bound - eps))
    v_valid = inside.sum(-1) == 2
    seg = hit[v_valid][inside[v_valid]].reshape(-1, 2, 3)
    seg = seg * s.expand(B, J, 3)[v_valid][..., None, :]
    nrm = d_t[v_valid].norm(dim=-1)
    steps = (seg - o_t[v_valid][..., None, :]).norm(dim=-1) / nrm[..., None]
    v_near = 100000 * torch.ones(B, J)
    v_far = -100000 * torch.ones(B, J)
    v_near[v_valid] = steps.min(dim=-1).values
    v_far[v_valid] = steps.max(dim=-1).values
    v_near = v_near.min(dim=-1).values
    v_far = v_far.max(dim=-1).values
    ray_valid = v_valid.sum(-1) > 0
    new_near, new_far = near.clone(), far.clone()
    new_near[ray_valid, 0] = v_near[ray_valid]
    new_far[ray_valid, 0] = v_far[ray_valid]
    return new_near, new_far, inside, v_valid


# ----------------------------------------------------------------------------------------------------------
# SM1  core/utils/ray_utils.py:206-253 sample_from_lineseg ; core/raycasters.py:455-468
# ----------------------------------------------------------------------------------------------------------
def coarse_z(near, far, S, t_rand=None, lindisp=False):
    """z = near(1-t)+far*t on t=linspace(0,1,S) (lindisp: linear in inverse depth, ray_utils.py:226-227);
    stratified jitter when t_rand (N,S) is given."""
    t = torch.linspace(0., 1., steps=S).expand([near.size(0), S])
    if not lindisp:
        z = near * (1. - t) + far * t
    else:
        z = 1. / (1. / near * (1. - t) + 1. / far * t)
    if t_rand is not None:
        mids = .5 * (z[..., 1:] + z[..., :-1])
        upper = torch.cat([mids, z[..., -1:]], -1)
        lower = torch.cat([z[..., :1], mids], -1)
        z = lower + (upper - lower) * t_rand
    return z


def ray_points(rays_o, rays_d, z):
    return rays_o[..., None, :] + rays_d[..., None, :] * z[..., :, None]


# ----------------------------------------------------------------------------------------------------------
# T1/T2/T3  core/encoders.py:288-303 transform_batch_pts ; :442-444 bone align ; :639-651 RelDist
# ----------------------------------------------------------------------------------------------------------
def world_to_bone(pts, skts, A):
    """pts (N,S,3), skts (N,24,4,4), A (24,4,4) -> pts_t (N,S,24,3): A_j (R_j p + t_j) + a_j, two steps."""
    N, S = pts.shape[:2]
    hom = torch.cat([pts, torch.ones(N, S, 1)], -1)                     # (N,S,4)
    loc = torch.einsum("njab,nsb->nsja", skts, hom)[..., :3]            # (N,S,24,3)
    A1 = A[None, None]
    return (A1[..., :3, :3] @ loc[..., None]).squeeze(-1) + A1[..., :3, -1]


# ----------------------------------------------------------------------------------------------------------
# PE  core/cutoff_embedder.py:22-73 Embedder
# ----------------------------------------------------------------------------------------------------------
def pe_embed(x, n_freq):
    """[x, sin(2^0 x), cos(2^0 x), ..., sin(2^(L-1) x), cos(2^(L-1) x)] along the last dim."""
    out = [x]
    for k in range(n_freq):
        f = float(2.0 ** k)
        out += [torch.sin(x * f), torch.cos(x * f)]
    return torch.cat(out, -1)


# ----------------------------------------------------------------------------------------------------------
# GN1  core/encoders.py:460-473,859-877 ; core/utils/skeleton_utils.py:411-418 (pytorch3d axis_angle_to_matrix)
# ----------------------------------------------------------------------------------------------------------
def axis_angle_to_matrix(aa):
    """pytorch3d's published route: axis-angle -> quaternion (Taylor branch below 1e-6) -> matrix.
    pytorch3d is an un-vendored, unpinned dependency of the reference (README.md:31-33)."""
    ang = torch.norm(aa, p=2, dim=-1, keepdim=True)
    half = ang * 0.5
    small = ang.abs() < 1e-6
    k = torch.where(small, 0.5 - (ang * ang) / 48, torch.sin(half) / torch.where(small, torch.ones_like(ang), ang))
    q = torch.cat([torch.cos(half), aa * k], dim=-1)
    r, i, j, kk = torch.unbind(q, -1)
    two_s = 2.0 / (q * q).sum(-1)
    m = torch.stack((1 - two_s * (j * j + kk * kk), two_s * (i * j - kk * r), two_s * (i * kk + j * r),
                     two_s * (i * j + kk * r), 1 - two_s * (i * i + kk * kk), two_s * (j * kk - i * r),
                     two_s * (i * kk - j * r), two_s * (j * kk + i * r), 1 - two_s * (i * i + j * j)), -1)
    return m.reshape(q.shape[:-1] + (3, 3))


def graph_inputs(pose_bones, n_freq=5):
    """pose_bones (G,24,3) -> w (G,24,66): rot6d = first two columns of R, row-major, then PE."""
    R = axis_angle_to_matrix(pose_bones)
    rot6d = R[..., :3, :2].flatten(start_dim=-2)
    return pe_embed(rot6d, n_freq)


# ----------------------------------------------------------------------------------------------------------
# GN2  core/networks/gnn_backbone.py:683-704 BodyGNN.forward on FactorizeGNN, layers :249-266 / misc.py:174-183
# ----------------------------------------------------------------------------------------------------------
def _adjw(P, prefix):
    return P[f"{prefix}.adj_w"] * P[f"{prefix}.adj"]                     # get_adjw gnn_backbone.py:225-247


def graph_net(w, P, prefix="graph_net"):
    """w (G,24,66) -> per-bone feature lines (G,24,240).  The first layer's output is doubled (F3)."""
    mask = torch.ones(1, J, 1)
    mask[:, 0] = 0.                                                      # mask_root
    n = mask * w
    # layer 0: DensePNGCN, shared bias, then `n = n + first_n` because skip_gcn=False == 0
    n = torch.einsum("bkl,klj->bkj", n, P[f"{prefix}.layers.0.lin.weight"])
    n = torch.matmul(_adjw(P, f"{prefix}.layers.0"), n) + P[f"{prefix}.layers.0.bias"]
    n = F.relu(n + n)
    # layer 1: DensePNGCN
    n = torch.einsum("bkl,klj->bkj", n, P[f"{prefix}.layers.1.lin.weight"])
    n = torch.matmul(_adjw(P, f"{prefix}.layers.1"), n) + P[f"{prefix}.layers.1.bias"]
    n = F.relu(n)
    # layer 2: ParallelLinear (gcn_fc_D = 1)
    n = F.relu(torch.einsum("bkl,klj->bkj", n, P[f"{prefix}.layers.2.weight"]) + P[f"{prefix}.layers.2.bias"])
    # layer 3: ParallelLinear -> 240 = feat(5) x bin(16) x axis(3)
    return torch.einsum("bkl,klj->bkj", n, P[f"{prefix}.layers.3.weight"]) + P[f"{prefix}.layers.3.bias"]


# ----------------------------------------------------------------------------------------------------------
# G1/G2  core/networks/gnn_backbone.py:787-828 sample_from_volume ; core/networks/misc.py:331-351
# ----------------------------------------------------------------------------------------------------------
def bone_features(pts_t, vol, axis_scale, rays_per_pose, res=16, feat=5):
    """pts_t (N,S,24,3), vol (G,24,240), axis_scale (24,3) -> h (N,S,24,15), invalid (N,S,24), x (N,S,24,3).

    Closed form of the 4-D F.grid_sample(bilinear, zeros, align_corners=False) call: the grid x coordinate
    {-2/3,0,2/3} picks the axis column exactly, the y coordinate interpolates linearly over 16 bins with
    zero padding.  240 = f*48 + bin*3 + axis; output channel = f*3 + axis; times exp(-2*sum x^6)."""
    N, S = pts_t.shape[:2]
    x = pts_t / axis_scale.reshape(1, 1, -1, 3).abs()
    win = torch.exp(-2 * ((x ** 6).sum(-1))).detach()               # gnn_backbone.py:804 detaches the window
    invalid = ((x.abs() > 1).sum(-1) > 0).float()
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
        ok = ((idx >= 0) & (idx < res)).float()                          # (N,S,24,3)
        idc = idx.clamp(0, res - 1)
        # gather table[n, j, f, idc[n,s,j,a], a] -> (N,S,24,5,3)
        t = table[:, None].expand(N, S, J, feat, res, 3)
        g = torch.gather(t, 4, idc[:, :, :, None, None, :].expand(N, S, J, feat, 1, 3)).squeeze(4)
        return g * ok[:, :, :, None, :]

    val = tap(i0) * w0[:, :, :, None, :] + tap(i1) * w1[:, :, :, None, :]   # (N,S,24,5,3)
    h = val.flatten(start_dim=-2) * win[..., None]
    return h, invalid, x


# ----------------------------------------------------------------------------------------------------------
# A1  core/networks/danbo.py:201-216 -> MixGNN gnn_backbone.py:567-591,608-629
# ----------------------------------------------------------------------------------------------------------
def agg_net(h, P, prefix="prob_linears"):
    """h (P,24,15) -> blend logits a (P,24)."""
    o = torch.einsum("bkl,klj->bkj", h, P[f"{prefix}.layers.0.lin.weight"])
    o = F.relu(torch.matmul(_adjw(P, f"{prefix}.layers.0"), o) + P[f"{prefix}.layers.0.bias"])
    o = F.relu(torch.einsum("bkl,klj->bkj", o, P[f"{prefix}.layers.1.weight"]) + P[f"{prefix}.layers.1.bias"])
    a = torch.einsum("bkl,klj->bkj", o, P[f"{prefix}.layers.2.weight"]) + P[f"{prefix}.layers.2.bias"]
    return a[..., 0]


# A2  core/networks/danbo.py:388-415,431-440
def agg_prob(a, invalid, agg_type="sigmoid", mask_vol_prob=True, eps=1e-7):
    if agg_type == "sigmoid":
        return (torch.sigmoid(a) * 1.002 - 0.001) * (1 - invalid)
    if agg_type == "softmax":
        if not mask_vol_prob:
            return F.softmax(a, dim=-1)
        valid = 1 - invalid
        e = torch.exp(a - a.max(dim=-1, keepdim=True)[0]) * valid
        return e / torch.sum(e + eps, dim=-1, keepdim=True).clamp(min=eps)
    raise NotImplementedError(agg_type)


# ----------------------------------------------------------------------------------------------------------
# V1  core/networks/nerf.py:252-279 ; core/networks/embedding.py:86-108
# ----------------------------------------------------------------------------------------------------------
def view_inputs(rays_d, cams, P, training, n_freq=4):
    """Per-ray (N,155): PE(un-normalised rays_d) (27) ++ frame code (128); mean code when eval and idx<0."""
    if "framecodes.codes.weight" not in P:                   # opt_framecode=False (configs/surreal): no code (nerf.py:262-279)
        return pe_embed(rays_d, n_freq)
    codes = P["framecodes.codes.weight"]
    if (not training) and cams.max() < 0:
        c = codes.mean(0, keepdim=True).expand(len(cams), -1)
    else:
        c = codes[cams.reshape(-1).long()]
    return torch.cat([pe_embed(rays_d, n_freq), c], -1)


# ----------------------------------------------------------------------------------------------------------
# M1  core/networks/nerf.py:176-209
# ----------------------------------------------------------------------------------------------------------
def density_trunk(x, P):
    h = x
    for i in range(8):
        h = F.relu(F.linear(h, P[f"pts_linears.{i}.weight"], P[f"pts_linears.{i}.bias"]))
        if i == 4:
            h = torch.cat([x, h], -1)
    return h


def field_mlp(x, view, P):
    """x (P,195), view (P,155) -> raw (P,4) = [rgb, sigma]."""
    h = density_trunk(x, P)
    alpha = F.linear(h, P["alpha_linear.weight"], P["alpha_linear.bias"])
    f = F.linear(h, P["feature_linear.weight"], P["feature_linear.bias"])
    g = F.relu(F.linear(torch.cat([f, view], -1), P["views_linears.0.weight"], P["views_linears.0.bias"]))
    rgb = F.linear(g, P["rgb_linear.weight"], P["rgb_linear.bias"])
    return torch.cat([rgb, alpha], -1)


# ----------------------------------------------------------------------------------------------------------
# C1  core/networks/nerf.py:281-347 raw2outputs
# ----------------------------------------------------------------------------------------------------------
def composite(raw, z, rays_d, noise=None, B=1.0):
    """noise (N,S) is the already-scaled density noise (randn * raw_noise_std * B) or None."""
    d = z[..., 1:] - z[..., :-1]
    d = torch.cat([d, torch.Tensor([1e10]).expand(d[..., :1].shape)], -1)
    d = d * torch.norm(rays_d[..., None, :], dim=-1)
    rgb = torch.sigmoid(raw[..., :3]) * 1.002 - 0.001
    n = 0. if noise is None else noise
    alpha = 1. - torch.exp(-(F.relu(raw[..., 3] / B + n)) * d)
    T = torch.cumprod(torch.cat([torch.ones((alpha.shape[0], 1)), 1. - alpha + 1e-10], -1), -1)[:, :-1]
    w = alpha * T
    rgb_map = torch.sum(w[..., None] * rgb, -2)
    depth = torch.sum(w * z, -1)
    wsum = torch.sum(w, -1)
    disp = 1. / torch.max(1e-10 * torch.ones_like(depth), depth / (wsum + 1e-10))
    disp = disp * (~torch.isclose(wsum, torch.tensor(0.))).float()
    acc = torch.minimum(wsum, torch.tensor(1.))
    return {"rgb_map": rgb_map, "disp_map": disp, "acc_map": acc, "weights": w, "alpha": alpha}


# ----------------------------------------------------------------------------------------------------------
# R1  core/utils/ray_utils.py:159-203 sample_pdf, :257-291 isample_from_lineseg (is_only=True)
# ----------------------------------------------------------------------------------------------------------
def importance_sample(z, weights, S_f, u=None, alpha_base=0.01, is_only=True):
    """Returns z_all (N,S_t) sorted, z_samples (N,S_f), sorted_idxs (N,S_t) int64, inds (N,S_f) int64.
    u=None -> deterministic linspace(0,1,S_f) (eval); else the caller's uniform draws (train).
    is_only = single_net (raycasters.py:348): smoothed weights + alpha_base; False: the interior weights themselves
    (ray_utils.py:272-281)."""
    mid = .5 * (z[..., 1:] + z[..., :-1])
    wl, wk, wu = weights[..., 0:-2], weights[..., 1:-1], weights[..., 2:]
    dw = 0.5 * (torch.maximum(wl, wk) + torch.maximum(wk, wu)) + alpha_base if is_only else wk
    dw = dw + 1e-5
    pdf = dw / torch.sum(dw, -1, keepdim=True)
    cdf = torch.cumsum(pdf, -1)
    cdf = torch.cat([torch.zeros_like(cdf[..., :1]), cdf], -1)
    if u is None:
        u = torch.linspace(0., 1., steps=S_f).expand(list(cdf.shape[:-1]) + [S_f])
    u = u.contiguous()
    inds = torch.searchsorted(cdf, u, right=True)
    below = torch.clamp(inds - 1, min=0)
    above = torch.clamp(inds, max=cdf.shape[-1] - 1)
    cdf_b, cdf_a = torch.gather(cdf, 1, below), torch.gather(cdf, 1, above)
    bin_b, bin_a = torch.gather(mid, 1, below), torch.gather(mid, 1, above)
    den = cdf_a - cdf_b
    den = torch.where(den < 1e-5, torch.ones_like(den), den)
    zs = (bin_b + (u - cdf_b) / den * (bin_a - bin_b)).detach()       # ray_utils.py:287
    z_all, order = torch.sort(torch.cat([z, zs], -1), -1)
    return z_all, zs, order, inds


# R2  core/raycasters.py:484-514,745-761
def merge_sorted(coarse, fine, order):
    cat = torch.cat([coarse, fine], dim=1)
    idx = order
    while idx.dim() < cat.dim():
        idx = idx[..., None]
    return torch.gather(cat, 1, idx.expand(*order.shape, *cat.shape[2:]))


# ----------------------------------------------------------------------------------------------------------
# whole path: core/raycasters.py:245-377 render_rays (single_net=True, N_importance>0)
# ----------------------------------------------------------------------------------------------------------
def view_directions(rays_d, skts, view_mode="world"):
    """What V1 encodes.  "world" (ray_tr_type=world, view_type=identity; h36m_zju and surreal configs): the un-normalised
    rays_d.  "root_local" (ray_tr_type=root_local, view_type=relray; perfcap configs): the direction rotated into the
    root joint's frame and normalised (RootLocalEncoder encoders.py:570-578, VecNormEncoder :774-795)."""
    if view_mode == "world":
        return rays_d
    if view_mode == "root_local":
        return F.normalize((skts[:, 0, :3, :3] @ rays_d[..., None])[..., 0], dim=-1, p=2)
    raise NotImplementedError(view_mode)


def field_eval(pts, rays_d, cams, skts, A, vol, P, rays_per_pose, training, agg_type="sigmoid", view_mode="world",
               mlp_fn=None):
    """T1..A3 + V1 + M1 for points (N,S,3) -> raw (N,S,4), confd (N,S,24), invalid (N,S,24), stage dict.
    mlp_fn (test hook): replaces `field_mlp` (same signature), e.g. by a restatement with the CUDA kernel's bf16 operand
    rounding, so that a comparison can separate "declared bf16 arithmetic" from everything else."""
    N, S = pts.shape[:2]
    pts_t = world_to_bone(pts, skts, A)
    h, invalid, x = bone_features(pts_t, vol, P["graph_net.axis_scale"], rays_per_pose)
    hf = h.reshape(N * S, J, -1)
    a = agg_net(hf, P)
    p = agg_prob(a, invalid.reshape(N * S, J), agg_type)
    hbar = (hf * p[..., None]).sum(-2)
    dens_in = pe_embed(hbar, 6)
    v_ray = view_inputs(view_directions(rays_d, skts, view_mode), cams, P, training)
    v = v_ray[:, None].expand(N, S, -1).reshape(N * S, -1)
    raw = (mlp_fn or field_mlp)(dens_in, v, P).reshape(N, S, 4)
    stages = {"pts_t": pts_t, "x": x, "h": h, "p": p.reshape(N, S, J), "hbar": hbar.reshape(N, S, -1), "view_inputs": v_ray}
    return raw, a.reshape(N, S, J), invalid, stages


def render_rays(ray_batch, pose_skts, pose_bones, pose_cyls, cams, A, P, S_c, S_f, rays_per_pose,
                use_volume_near_far=False, training=False, rand=None, raw_noise_std=0., agg_type="sigmoid",
                return_stages=False, z_samples=None, lindisp=False, view_mode="world", mlp_fn=None):
    """ray_batch (N,>=8); pose_* are per unique pose (G,...); ray n belongs to pose n // rays_per_pose.
    rand (training) = dict(t_rand (N,S_c), noise0 (N,S_c), u (N,S_f), noise1 (N,S_t)) drawn by the caller in
    the reference's order (SURVEY §7 hard part 4)."""
    N = ray_batch.shape[0]
    G = pose_skts.shape[0]
    pose = torch.clamp(torch.arange(N) // rays_per_pose, max=G - 1)
    skts, cyls = pose_skts[pose], pose_cyls[pose]
    rays_o, rays_d = ray_batch[:, 0:3], ray_batch[:, 3:6]
    near, far = ray_batch[:, 6:7], ray_batch[:, 7:8]
    near, far = cylinder_near_far(rays_o, rays_d, cyls, near, far)
    nf_cyl = (near.clone(), far.clone())
    if use_volume_near_far:
        with torch.no_grad():                                            # raycasters.py:648 @torch.no_grad()
            near, far, _, _ = box_near_far(rays_o, rays_d, skts, A, P["graph_net.axis_scale"], near, far)
    vol = graph_net(graph_inputs(pose_bones), P)
    rand = rand or {}
    z = coarse_z(near, far, S_c, rand.get("t_rand"), lindisp)
    pts = ray_points(rays_o, rays_d, z)
    raw0, confd0, inv0, st0 = field_eval(pts, rays_d, cams, skts, A, vol, P, rays_per_pose, training, agg_type, view_mode,
                                         mlp_fn)
    n0 = rand["noise0"] * raw_noise_std if "noise0" in rand else None
    out0 = composite(raw0, z, rays_d, n0)
    z_all, zs, order, inds = importance_sample(z, out0["weights"], S_f, rand.get("u"))
    if z_samples is not None:
        # test hook: evaluate the fine pass at externally supplied (detached) importance samples, so a comparison
        # against an implementation whose coarse weights differ in the last bits is not dominated by resampling
        zs = z_samples
        z_all, order = torch.sort(torch.cat([z, zs], -1), -1)
    pts_f = ray_points(rays_o, rays_d, zs)
    raw1, confd1, inv1, st1 = field_eval(pts_f, rays_d, cams, skts, A, vol, P, rays_per_pose, training, agg_type, view_mode,
                                         mlp_fn)
    raw = merge_sorted(raw0, raw1, order)
    confd = merge_sorted(confd0, confd1, order)
    inv = merge_sorted(inv0, inv1, order)
    n1 = rand["noise1"] * raw_noise_std if "noise1" in rand else None
    out = composite(raw, z_all, rays_d, n1)
    ret = {"rgb_map": out["rgb_map"], "disp_map": out["disp_map"], "acc_map": out["acc_map"],
           "alpha": out["alpha"], "T_i": out["weights"],
           "rgb0": out0["rgb_map"], "disp0": out0["disp_map"], "acc0": out0["acc_map"], "alpha0": out0["alpha"]}
    if training:
        ret["confd"] = confd
        ret["part_invalid"] = inv
    if return_stages:
        ret["_stages"] = {"near_cyl": nf_cyl[0], "far_cyl": nf_cyl[1], "near": near, "far": far, "vol": vol,
                          "z_coarse": z, "raw0": raw0, "weights0": out0["weights"], "z_samples": zs,
                          "z_all": z_all, "sorted_idxs": order, "inds": inds, "raw1": raw1, "raw": raw,
                          "confd0": confd0, "invalid0": inv0, "coarse": st0, "fine": st1}
    return ret


# ----------------------------------------------------------------------------------------------------------
# AN1  A-NeRF field (nerf_type=nerf, configs/h36m_zju/anerf_base.txt): core/networks/nerf.py:222-279 encode_pts /
# encode_views ; core/cutoff_embedder.py:151-214 CutoffEmbedder._embed ; core/encoders.py:639-651 RelDistEncoder,
# :774-795 VecNormEncoder, :305-317 transform_batch_rays ; MLP nerf.py:164-209 with W=448, view_W=224.
# ----------------------------------------------------------------------------------------------------------
ANERF_CUTOFF = 500 * 0.001          # cutoff_mm * ext_scale (encoders.py:62, run_nerf.py:498)


def anerf_cutoff_weight(dist, tau, cutoff=ANERF_CUTOFF):
    """cutoff_embedder.py:177-184: w = 1 - sigmoid(tau * (dist - cutoff))."""
    return 1. - torch.sigmoid(tau * (dist - cutoff))


def anerf_dist_pe(v, tau, n_freq=7, cutoff=ANERF_CUTOFF):
    """pe_fn of A-NeRF (cut_to_cutoff, shift_inputs, cutoff_inputs, include_input; dist_inputs False):
    v (...,24) -> (...,15*24): rows [c - v, sin(2^0 s), cos(2^0 s), ..., cos(2^6 s)] each times w, s = (c-v)*2/c - 1;
    flattened row-major (row, joint)."""
    inp = cutoff - v
    shifted = inp * (2. / cutoff) - 1.
    freqs = 2. ** torch.linspace(0., n_freq - 1, steps=n_freq)
    x = freqs.view(1, -1, 1) * shifted[..., None, :]                       # (..., F, 24)
    w = anerf_cutoff_weight(v, tau, cutoff)[..., None, :]
    emb = torch.stack([torch.sin(x), torch.cos(x)], dim=-2).flatten(start_dim=-3, end_dim=-2)   # (..., 2F, 24)
    emb = torch.cat([inp[..., None, :], emb], dim=-2) * w
    return emb.flatten(start_dim=-2)


def anerf_dir_pe(d, v, tau, n_freq=4, cutoff=ANERF_CUTOFF):
    """dirs_pe_fn (dist_inputs=True): d (...,72) per-joint unit vectors, v (...,24) -> (...,9*72); joint j's weight is
    repeated over its three components."""
    dist = v[..., None].expand(*v.shape, 3).flatten(start_dim=-2)           # (..., 72)
    freqs = 2. ** torch.linspace(0., n_freq - 1, steps=n_freq)
    x = freqs.view(1, -1, 1) * d[..., None, :]
    w = anerf_cutoff_weight(dist, tau, cutoff)[..., None, :]
    emb = torch.stack([torch.sin(x), torch.cos(x)], dim=-2).flatten(start_dim=-3, end_dim=-2)
    emb = torch.cat([d[..., None, :], emb], dim=-2) * w
    return emb.flatten(start_dim=-2)


def anerf_inputs(pts, rays_d, cams, skts, A, P, training, tau=20.):
    """pts (N,S,3) -> density_inputs (N*S,432), view_inputs (N*S,776), stage dict."""
    N, S = pts.shape[:2]
    pts_t = world_to_bone(pts, skts, A)                                     # (N,S,24,3) incl. bone alignment (T2)
    v = torch.norm(pts_t, dim=-1, p=2)                                      # RelDistEncoder
    r = F.normalize(pts_t, dim=-1, p=2).flatten(start_dim=2)                # VecNormEncoder on pts_t (bone_type reldir)
    dens = torch.cat([anerf_dist_pe(v, tau), r], -1).reshape(N * S, -1)
    rays_t = (skts[..., :3, :3] @ rays_d.reshape(N, 1, 3, 1)).reshape(N, 1, J, 3)     # transform_batch_rays (rotation only)
    d = F.normalize(rays_t, dim=-1, p=2).flatten(start_dim=2).expand(N, S, -1)
    d_pe = anerf_dir_pe(d, v, tau)
    codes = P["framecodes.codes.weight"]
    if (not training) and cams.max() < 0:
        c = codes.mean(0, keepdim=True).expand(len(cams), -1)
    else:
        c = codes[cams.reshape(-1).long()]
    view = torch.cat([d_pe, c[:, None].expand(N, S, -1)], -1).reshape(N * S, -1)
    return dens, view, {"pts_t": pts_t, "v": v, "r": r, "d": d}


def anerf_mlp(x, view, P):
    """nerf.py:176-209 with the skip after layer 4 ([x ; h]); W read from the parameter shapes."""
    h = x
    for i in range(8):
        h = F.relu(F.linear(h, P[f"pts_linears.{i}.weight"], P[f"pts_linears.{i}.bias"]))
        if i == 4:
            h = torch.cat([x, h], -1)
    alpha = F.linear(h, P["alpha_linear.weight"], P["alpha_linear.bias"])
    f = F.linear(h, P["feature_linear.weight"], P["feature_linear.bias"])
    g = F.relu(F.linear(torch.cat([f, view], -1), P["views_linears.0.weight"], P["views_linears.0.bias"]))
    rgb = F.linear(g, P["rgb_linear.weight"], P["rgb_linear.bias"])
    return torch.cat([rgb, alpha], -1)


def anerf_render_rays(ray_batch, pose_skts, pose_cyls, cams, A, P, S_c, S_f, rays_per_pose, training=False, rand=None,
                      raw_noise_std=0., tau=20., return_stages=False, z_samples=None, lindisp=False, P_fine=None):
    """RayCaster.render_rays (raycasters.py:245-377) for nerf_type=nerf: cylinder near/far only (:419-420), the field
    evaluated on every sample, single_net fine pass on the S_f new samples (F9).  P_fine: parameters of a separate
    fine network (single_net = False, configs/h36m_zju/anerf_h.txt): importance weights are the raw interior coarse
    weights and the fine network is evaluated on all S_c + S_f merged samples (raycasters.py:350-371)."""
    N = ray_batch.shape[0]
    G = pose_skts.shape[0]
    pose = torch.clamp(torch.arange(N) // rays_per_pose, max=G - 1)
    skts, cyls = pose_skts[pose], pose_cyls[pose]
    rays_o, rays_d = ray_batch[:, 0:3], ray_batch[:, 3:6]
    near, far = cylinder_near_far(rays_o, rays_d, cyls, ray_batch[:, 6:7], ray_batch[:, 7:8])
    rand = rand or {}
    z = coarse_z(near, far, S_c, rand.get("t_rand"), lindisp)
    x0, v0, st0 = anerf_inputs(ray_points(rays_o, rays_d, z), rays_d, cams, skts, A, P, training, tau)
    raw0 = anerf_mlp(x0, v0, P).reshape(N, S_c, 4)
    n0 = rand["noise0"] * raw_noise_std if "noise0" in rand else None
    out0 = composite(raw0, z, rays_d, n0)
    z_all, zs, order, inds = importance_sample(z, out0["weights"], S_f, rand.get("u"), is_only=P_fine is None)
    if z_samples is not None:                                               # test hook, see render_rays
        zs = z_samples
        z_all, order = torch.sort(torch.cat([z, zs], -1), -1)
    if P_fine is None:
        x1, v1, st1 = anerf_inputs(ray_points(rays_o, rays_d, zs), rays_d, cams, skts, A, P, training, tau)
        raw1 = anerf_mlp(x1, v1, P).reshape(N, S_f, 4)
        raw = merge_sorted(raw0, raw1, order)
    else:
        pts_all = merge_sorted(ray_points(rays_o, rays_d, z), ray_points(rays_o, rays_d, zs), order)
        x1, v1, st1 = anerf_inputs(pts_all, rays_d, cams, skts, A, P_fine, training, tau)
        raw1 = raw = anerf_mlp(x1, v1, P_fine).reshape(N, S_c + S_f, 4)
    n1 = rand["noise1"] * raw_noise_std if "noise1" in rand else None
    out = composite(raw, z_all, rays_d, n1)
    ret = {"rgb_map": out["rgb_map"], "disp_map": out["disp_map"], "acc_map": out["acc_map"],
           "alpha": out["alpha"], "T_i": out["weights"],
           "rgb0": out0["rgb_map"], "disp0": out0["disp_map"], "acc0": out0["acc_map"], "alpha0": out0["alpha"]}
    if return_stages:
        ret["_stages"] = {"near": near, "far": far, "z_coarse": z, "dens_in0": x0, "view_in0": v0, "raw0": raw0,
                          "weights0": out0["weights"], "z_samples": zs, "z_all": z_all, "sorted_idxs": order,
                          "raw1": raw1, "raw": raw, "v0": st0["v"]}
    return ret


# ----------------------------------------------------------------------------------------------------------
# D1  core/raycasters.py:421-453 render_mesh_density ; core/networks/nerf.py:136-154
# ----------------------------------------------------------------------------------------------------------
def density_grid(kps, skts, bones, A, P, radius, res, agg_type="sigmoid"):
    """Raw sigma on a (res+1)^3 lattice centred on the root joint, x/y swapped like the reference."""
    t = np.linspace(-radius, radius, res + 1)
    grid = np.stack(np.meshgrid(t, t, t), axis=-1).astype(np.float32)
    sh = grid.shape
    pts = (torch.tensor(grid.reshape(-1, 3)) + kps[0, 0]).reshape(-1, 1, 3)
    vol = graph_net(graph_inputs(bones), P)
    pts_t = world_to_bone(pts, skts.expand(pts.shape[0], -1, -1, -1), A)
    h, invalid, _ = bone_features(pts_t, vol, P["graph_net.axis_scale"], pts.shape[0])
    hf = h.reshape(-1, J, 15)
    p = agg_prob(agg_net(hf, P), invalid.reshape(-1, J), agg_type)
    x = pe_embed((hf * p[..., None]).sum(-2), 6)
    sigma = F.linear(density_trunk(x, P), P["alpha_linear.weight"], P["alpha_linear.bias"])
    return sigma.reshape(*sh[:-1]).transpose(1, 0)


def anerf_density_grid(kps, skts, A, P, radius, res, tau=20.):
    """The same lattice query for the A-NeRF field (nerf.py:136-154 forward_pts -> encode_pts :222-250): raw sigma =
    alpha_linear of the W=448 trunk on [cutoff PE(v) ; r]; the view branch is not evaluated."""
    t = np.linspace(-radius, radius, res + 1)
    grid = np.stack(np.meshgrid(t, t, t), axis=-1).astype(np.float32)
    sh = grid.shape
    pts = (torch.tensor(grid.reshape(-1, 3)) + kps[0, 0]).reshape(-1, 1, 3)
    n = pts.shape[0]
    pts_t = world_to_bone(pts, skts.expand(n, -1, -1, -1), A)
    v = torch.norm(pts_t, dim=-1, p=2)
    r = F.normalize(pts_t, dim=-1, p=2).flatten(start_dim=2)
    x = torch.cat([anerf_dist_pe(v, tau), r], -1).reshape(n, -1)
    h = x
    for i in range(8):
        h = F.relu(F.linear(h, P[f"pts_linears.{i}.weight"], P[f"pts_linears.{i}.bias"]))
        if i == 4:
            h = torch.cat([x, h], -1)
    sigma = F.linear(h, P["alpha_linear.weight"], P["alpha_linear.bias"])
    return sigma.reshape(*sh[:-1]).transpose(1, 0)


# ----------------------------------------------------------------------------------------------------------
# L*  core/trainer.py:396-422,507-553 (losses stay in PyTorch in the product too; here for the training parity test)
# ----------------------------------------------------------------------------------------------------------
def training_loss(ret, target, bgs, P, init_scale, soft_coef=0.001, vol_coef=0.001, coarse_weight=1.0, agg_type="sigmoid",
                  loss_fn="L1"):
    def l1(rgb, acc):                                               # img2l1 / img2mse, core/trainer.py:164-187
        d = rgb + (1. - acc)[..., None] * bgs - target
        return torch.mean(torch.abs(d)) if loss_fn == "L1" else torch.mean(d ** 2)
    loss = l1(ret["rgb_map"], ret["acc_map"]) + coarse_weight * l1(ret["rgb0"], ret["acc0"])
    if agg_type == "sigmoid":                                       # trainer.py:372: only with sigmoid blend weights
        labels = ((ret["T_i"] * ret["alpha"]) > 0).float()
        valid = 1 - ret["part_invalid"]
        p = torch.sigmoid(ret["confd"]) * 1.002 - 0.001
        loss = loss + soft_coef * (labels - (p * valid).sum(-1)).pow(2.).mean()
    scale = P["graph_net.axis_scale"].abs().clamp(min=init_scale * 0.05)
    loss = loss + vol_coef * torch.prod(scale, dim=-1).sum()
    return loss
