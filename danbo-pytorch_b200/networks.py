"""Host-side mirror of the reference's DANBO field module: same parameter names and shapes (SURVEY appendix A,
params.py), so reference checkpoints load unchanged; the forward work is done by the CUDA kernels.

Only the per-pose graph net (GN1 + GN2: at most 16 poses x 24 nodes per call) runs as PyTorch ops, as SURVEY §8(a)
prescribes; everything per sample goes through libdanbo_b200.so.

Reference: core/networks/danbo.py:9-185, nerf.py:13-105, gnn_backbone.py:184-274,517-629,631-704,737-831,
misc.py:129-183, embedding.py:4-50.
"""
import math

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import skeleton as sk

J = sk.N_JOINTS


class ParallelLinear(nn.Module):
    """One (in,out) matrix per joint; weight (joint,in,out), bias (1,joint,out) (misc.py:129-183)."""

    def __init__(self, n_parallel, in_feat, out_feat, bias=True):
        super().__init__()
        self.n_parallel, self.in_feat, self.out_feat = n_parallel, in_feat, out_feat
        self.weight = nn.Parameter(torch.empty(n_parallel, in_feat, out_feat))
        if bias:
            self.bias = nn.Parameter(torch.zeros(1, n_parallel, out_feat))
        else:
            self.register_parameter("bias", None)
        for n in range(n_parallel):
            nn.init.kaiming_uniform_(self.weight[n].T.data, a=math.sqrt(5))

    def forward(self, x):
        out = torch.einsum("bkl,klj->bkj", x, self.weight)
        return out if self.bias is None else out + self.bias


class DenseGCN(nn.Module):
    """Per-joint linear followed by a learned mix over the skeleton tree (gnn_backbone.py:184-274)."""

    def __init__(self, adj, in_ch, out_ch, init_adj_w=0.05):
        super().__init__()
        adj = adj.clone()
        idx = torch.arange(adj.shape[-1])
        adj[:, idx, idx] = 1
        adj_w = adj.clone() * (init_adj_w + (torch.rand_like(adj) - 0.5) * 0.1).clamp(min=0.01, max=1.0)
        adj_w[:, idx, idx] = 1.0
        self.lin = ParallelLinear(adj.shape[-1], in_ch, out_ch, bias=False)
        self.bias = nn.Parameter(torch.zeros(out_ch))
        self.register_buffer("adj", adj)
        self.adj_w = nn.Parameter(adj_w)

    def get_adjw(self):
        return self.adj_w * self.adj

    def forward(self, x):
        return torch.matmul(self.get_adjw(), self.lin(x)) + self.bias


def _tree_adj():
    return torch.from_numpy(sk.skeleton_adjacency()).view(1, J, J)


class GraphNet(nn.Module):
    """FactorizeGNN ('FGNNcat'): pose -> three 16-bin feature lines x 5 channels per bone (gnn_backbone.py:737-831)."""

    def __init__(self, in_ch=66, W=128, voxel_res=16, voxel_feat=5, skel_profile=None, base_scale=0.4, opt_scale=True):
        super().__init__()
        adj = _tree_adj()
        self.voxel_res, self.voxel_feat = voxel_res, voxel_feat
        self.layers = nn.ModuleList([DenseGCN(adj, in_ch, W), DenseGCN(adj, W, W), ParallelLinear(J, W, W),
                                     ParallelLinear(J, W, voxel_res * voxel_feat * 3)])
        scale = torch.ones(J, 3) * base_scale
        if skel_profile is not None:
            scale = sk.initial_axis_scale(skel_profile, base_scale)
        # plain attribute in the reference (gnn_backbone.py:784); a non-persistent buffer here so it follows .to(device)
        self.register_buffer("init_scale", scale.clone(), persistent=False)
        self.axis_scale = nn.Parameter(scale, requires_grad=opt_scale)
        mask = torch.ones(1, J, 1)
        mask[:, 0] = 0.                                         # mask_root
        # non-persistent buffer: follows .to(device) (a per-call host->device copy would synchronise the stream) but
        # stays out of the state_dict, like the reference's plain attribute (gnn_backbone.py:669-670)
        self.register_buffer("mask", mask, persistent=False)

    def get_axis_scale(self):
        return self.axis_scale

    def get_adjw(self):
        return [m.get_adjw() for m in self.layers if isinstance(m, DenseGCN)]

    def forward(self, w):
        """w (G,24,66) -> (G,24,240).  Layer 0's output is doubled, as in the reference (SURVEY F3:
        `if i == skip_gcn` with skip_gcn=False, gnn_backbone.py:695-699)."""
        n = self.mask * w
        n = self.layers[0](n)
        n = F.relu(n + n)
        n = F.relu(self.layers[1](n))
        n = F.relu(self.layers[2](n))
        return self.layers[3](n)


class AggNet(nn.Module):
    """'vox_MIXGNN' blend-weight net 15 -> 32 -> 32 -> 1 per bone (gnn_backbone.py:602-629); evaluated by the
    field_agg kernel, kept here as the parameter owner (and for `get_adjw`)."""

    def __init__(self, in_ch=15, W=32):
        super().__init__()
        self.layers = nn.ModuleList([DenseGCN(_tree_adj(), in_ch, W), ParallelLinear(J, W, W), ParallelLinear(J, W, 1)])

    def get_adjw(self):
        return [self.layers[0].get_adjw()]


class Optcodes(nn.Module):
    """Per-frame appearance codes (embedding.py:4-50)."""

    def __init__(self, n_codes, code_ch):
        super().__init__()
        self.n_codes, self.code_ch = n_codes, code_ch
        self.codes = nn.Embedding(n_codes, code_ch)
        nn.init.xavier_normal_(self.codes.weight)


class _NoCutoffPE:
    """Stands in for the reference's Embedder where the trainer only asks for its tau (trainer.py:297-300)."""

    def get_tau(self):
        return 0.0

    def update_threshold(self, *a, **k):
        pass


def pe_embed(x, n_freq):
    out = [x]
    for k in range(n_freq):
        out += [torch.sin(x * float(2.0 ** k)), torch.cos(x * float(2.0 ** k))]
    return torch.cat(out, -1)


def axis_angle_to_matrix(aa):
    """Axis-angle -> quaternion -> rotation matrix, the route pytorch3d documents (skeleton_utils.py:411-418)."""
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


class DanboField(nn.Module):
    """Parameter owner of the DANBO field (`network` / `network_fine` of the ray caster)."""

    def __init__(self, n_framecodes=8, W=256, D=8, view_W=128, node_W=128, agg_W=32, voxel_feat=5, voxel_res=16,
                 multires_voxel=6, multires_graph=5, multires_views=4, framecode_ch=128, skel_profile=None,
                 opt_scale=True, agg_type="sigmoid", mask_vol_prob=True, opt_framecode=True):
        super().__init__()
        if D != 8 or W != 256 or view_W != 128 or agg_W != 32 or voxel_feat != 5 or voxel_res != 16 \
                or multires_voxel != 6 or framecode_ch != 128 or multires_views != 4:
            raise NotImplementedError("the sm_100a kernels are specialised for netdepth=8, netwidth=256, agg_W=32, "
                                      "voxel_feat=5, voxel_res=16, multires_voxel=6, multires_views=4, framecode_size=128")
        if agg_type not in ("sigmoid", "softmax"):
            raise NotImplementedError(f"agg_type={agg_type!r} is not implemented (supported: 'sigmoid', 'softmax')")
        if agg_type == "softmax" and not mask_vol_prob:
            # plain F.softmax (danbo.py:389-390) gives bones that do not see the sample a non-zero weight, so a sample no
            # bone sees no longer has h = 0 and the sparse evaluation (DESIGN.md §3) is not result-identical
            raise NotImplementedError("agg_type='softmax' needs mask_vol_prob=True (as in every shipped config)")
        self.W, self.D, self.view_W = W, D, view_W
        self.multires_voxel, self.multires_graph, self.multires_views = multires_voxel, multires_graph, multires_views
        self.agg_type, self.mask_vol_prob = agg_type, mask_vol_prob
        x_ch = voxel_feat * 3 * (1 + 2 * multires_voxel)
        v_ch = 3 * (1 + 2 * multires_views)
        layers = [nn.Linear(x_ch, W)]
        for i in range(D - 1):
            layers.append(nn.Linear(W + x_ch, W) if i == 4 else nn.Linear(W, W))
        self.pts_linears = nn.ModuleList(layers)
        self.alpha_linear = nn.Linear(W, 1)
        self.opt_framecode = bool(opt_framecode)        # False (configs/surreal): no per-frame code in the view layer
        self.views_linears = nn.ModuleList([nn.Linear(v_ch + (framecode_ch if opt_framecode else 0) + 2 * view_W, view_W)])
        self.feature_linear = nn.Linear(W, 2 * view_W)
        self.rgb_linear = nn.Linear(view_W, 3)
        self.framecodes = Optcodes(n_framecodes, framecode_ch) if opt_framecode else None
        self.graph_net = GraphNet(6 * (1 + 2 * multires_graph), node_W, voxel_res, voxel_feat, skel_profile,
                                  opt_scale=opt_scale)
        self.prob_linears = AggNet(voxel_feat * 3, agg_W)
        self.pe_fn = _NoCutoffPE()

    # ---- surface the trainer touches (trainer.py:294-300,509-546) -------------------------------------------
    def sigmoid(self, logit, invalid, mask_invalid=True, clamp=True, eps=1e-7, sigmoid_eps=0.001):
        p = torch.sigmoid(logit) * (1 + 2 * sigmoid_eps) - sigmoid_eps
        if mask_invalid:
            p = p * (1 - invalid.flatten(end_dim=-2))
        return p

    def softmax(self, logit, invalid, eps=1e-7, temp=1.0):
        """danbo.py:388-404 (torch ops; the kernels compute the same inside field_rows)."""
        if not self.mask_vol_prob:
            return torch.softmax(logit / temp, dim=-1)
        logit = logit / temp
        valid = 1 - invalid.flatten(end_dim=-2)
        nominator = torch.exp(logit - logit.max(dim=-1, keepdim=True)[0]) * valid
        return nominator / torch.sum(nominator + eps, dim=-1, keepdim=True).clamp(min=eps)

    def get_agg(self, logit, invalid, eps=1e-7):
        return self.softmax(logit, invalid, eps=eps) if self.agg_type == "softmax" else self.sigmoid(logit, invalid, eps=eps)

    @property
    def agg_mode(self):
        """`agg_mode` argument of danbo_field_agg / danbo_field_agg_bwd."""
        return 1 if self.agg_type == "softmax" else 0

    def get_adjw(self):
        return self.graph_net.get_adjw() + self.prob_linears.get_adjw()

    def update_embed_fns(self, global_step, args):
        pass                                                     # no cutoff / frequency schedule in DANBO configs

    # ---- GN1 + GN2 (PyTorch, per unique pose) ---------------------------------------------------------------
    fused_graph_net = True        # GN1 + GN2 as danbo_graph_net_fwd/_bwd (CUDA tensors); False: the PyTorch ops below
    # set by training.TrainStep around the forward pass of its pose-kernel path (a captured --opt_pose iteration): the
    # pose's gradient then comes from the graph-net kernels (danbo_graph_net_bwd_pose) too
    pose_kernels = False

    def bone_volumes(self, pose_bones):
        """pose_bones (G,24,3) axis-angle -> (G,24,240) feature lines (encoders.py:460-473,859-877; danbo.py:190-194)."""
        # a pose that itself needs a gradient (pose layer under --opt_pose) takes the PyTorch ops below unless the pose
        # kernels serve the step: eager training with a pose layer keeps them as its reference path
        pose_grad = torch.is_grad_enabled() and pose_bones.requires_grad and not self.pose_kernels
        six = pose_bones.shape[-1] == 6          # a rot6d pose layer hands its parameters over as they are (encoders.py:873-877)
        if self.fused_graph_net and pose_bones.is_cuda and not pose_grad and not six:
            from .autograd import graph_net_volumes
            return graph_net_volumes(self, pose_bones)
        rot6d = pose_bones if six else axis_angle_to_matrix(pose_bones)[..., :3, :2].flatten(start_dim=-2)
        return self.graph_net(pe_embed(rot6d, self.multires_graph))

    def agg_tensors(self):
        l = self.prob_linears.layers
        return {"w0": l[0].lin.weight, "adj_w": l[0].adj_w, "adj": l[0].adj, "b0": l[0].bias,
                "w1": l[1].weight, "b1": l[1].bias, "w2": l[2].weight, "b2": l[2].bias}
