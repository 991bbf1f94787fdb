"""Pose layer (SURVEY §8f rank 2, forward half): learnable per-frame poses -> kinematic chain -> the `kps / bones / skts`
tables the body-field path consumes, with the reference's state-dict keys so pose-refined checkpoints load.

Mirrors core/pose_opt.py: `PoseOptLayer` (:132-339: parameters `pelvis` (N,3), `bones` (N,24,3) axis-angle or (N,24,6)
with `use_rot6d`; buffer `rest_pose`; the multi-view split `root_bones` / `bones` / `kp_map` / `kp_uidxs`),
`create_popt` (:14-83), `load_poseopt_from_state_dict` (:104-130), `load_bones_from_state_dict` (:95-102),
`pose_ckpt_to_pose_data` (:415-451) and the trainer's pose regulariser (`Trainer._compute_kp_loss`,
core/trainer.py:446-505).

Built differently from the reference: the chain is evaluated per tree LEVEL for any parent table (the reference hard-codes
the SMPL unrolling, :374-413) on rotation / translation pairs instead of 4x4 products, and world-to-bone matrices are
the closed-form rigid inverse [R^T | -R^T t] instead of `torch.inverse` (24 LU factorisations per pose and its backward)
- all plain torch ops on the parameters' device, differentiable by autograd.  Poses are evaluated once per UNIQUE index
(`N_uniques` image-major batches skip even the unique()) and returned as stride-0 expands, which is what the ray caster
reduces back to per-pose tables (raycaster._prepare).

The gradient of the rendered colours with respect to the layer's outputs comes from the CUDA path: d loss / d skts from
`danbo_field_agg_bwd` (`grads[9]`, csrc/backward_field.cu; the render block's autograd node takes the per-pose matrices
as an input) and d loss / d bones through the graph net's PyTorch ops (`networks.DanboField.bone_volumes`); `kp_batch`
receives none in the DANBO field, as in the reference.  `training.TrainStep(popt_kwargs=..., pose_optimizer=...)` runs
the whole --opt_pose iteration.  That gradient path was written after round 1's GPU minutes were spent: it is pinned on
the CPU (oracle vs the reference's own pose gradients, tests/golden/train_fast_popt.npz) and its GPU tests
(tests/test_gpu_zzy_pose_grad.py) have not run on hardware yet.
"""
import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import skeleton as sk


# ---- rotations (core/utils/skeleton_utils.py:397-439; pytorch3d.transforms published formulas) -------------------
def axisang_to_rot(axisang):
    """(…,3) -> (…,3,3) via the unit quaternion, as pytorch3d.axis_angle_to_matrix does (skeleton_utils.py:411)."""
    ang = torch.norm(axisang, p=2, dim=-1, keepdim=True)
    half = ang * 0.5
    small = ang.abs() < 1e-6
    safe = torch.where(small, torch.ones_like(ang), ang)
    k = torch.where(small, 0.5 - ang * ang / 48, torch.sin(half) / safe)
    q = torch.cat([torch.cos(half), axisang * k], -1)
    r, i, j, k_ = torch.unbind(q, -1)
    two_s = 2.0 / (q * q).sum(-1)
    o = torch.stack((1 - two_s * (j * j + k_ * k_), two_s * (i * j - k_ * r), two_s * (i * k_ + j * r),
                     two_s * (i * j + k_ * r), 1 - two_s * (i * i + k_ * k_), two_s * (j * k_ - i * r),
                     two_s * (i * k_ - j * r), two_s * (j * k_ + i * r), 1 - two_s * (i * i + j * j)), -1)
    return o.reshape(q.shape[:-1] + (3, 3))


def rot6d_to_rotmat(x):
    """(…,6) -> (…,3,3): Gram-Schmidt of the two stored columns (Zhou et al. 2019; skeleton_utils.py:423-439)."""
    shape = x.shape[:-1]
    x = x.reshape(-1, 3, 2)
    a1, a2 = x[:, :, 0], x[:, :, 1]
    b1 = F.normalize(a1)
    b2 = F.normalize(a2 - (b1 * a2).sum(-1, keepdim=True) * b1)
    b3 = torch.cross(b1, b2, dim=-1)
    return torch.stack((b1, b2, b3), dim=-1).reshape(*shape, 3, 3)


def rot_to_rot6d(rot):
    return rot[..., :3, :2].flatten(start_dim=-2)


def rot_to_axisang(rot):
    """(…,3,3) -> (…,3) via the quaternion with the largest component (pytorch3d.matrix_to_axis_angle's route,
    skeleton_utils.py:405); the rotation angle is reduced to [0, pi]."""
    m = rot[..., :3, :3]
    m00, m01, m02 = m[..., 0, 0], m[..., 0, 1], m[..., 0, 2]
    m10, m11, m12 = m[..., 1, 0], m[..., 1, 1], m[..., 1, 2]
    m20, m21, m22 = m[..., 2, 0], m[..., 2, 1], m[..., 2, 2]
    q_abs = torch.sqrt(torch.clamp(torch.stack([1 + m00 + m11 + m22, 1 + m00 - m11 - m22,
                                                1 - m00 + m11 - m22, 1 - m00 - m11 + m22], -1), min=0))
    cand = torch.stack([torch.stack([q_abs[..., 0] ** 2, m21 - m12, m02 - m20, m10 - m01], -1),
                        torch.stack([m21 - m12, q_abs[..., 1] ** 2, m10 + m01, m02 + m20], -1),
                        torch.stack([m02 - m20, m10 + m01, q_abs[..., 2] ** 2, m12 + m21], -1),
                        torch.stack([m10 - m01, m20 + m02, m21 + m12, q_abs[..., 3] ** 2], -1)], -2)
    cand = cand / (2.0 * q_abs[..., None].clamp(min=0.1))
    best = q_abs.argmax(-1)
    q = torch.gather(cand, -2, best[..., None, None].expand(*best.shape, 1, 4))[..., 0, :]
    q = torch.where(q[..., :1] < 0, -q, q)
    norms = torch.norm(q[..., 1:], p=2, dim=-1, keepdim=True)
    half = torch.atan2(norms, q[..., :1])
    ang = 2 * half
    small = ang.abs() < 1e-6
    k = torch.where(small, 0.5 - ang * ang / 48, torch.sin(half) / torch.where(small, torch.ones_like(ang), ang))
    return q[..., 1:] / k


def rot6d_to_axisang(rot6d):
    return rot_to_axisang(rot6d_to_rotmat(rot6d))


def bones_to_rot(bones):
    if bones.shape[-1] == 3:
        return axisang_to_rot(bones)
    if bones.shape[-1] == 6:
        return rot6d_to_rotmat(bones)
    raise NotImplementedError(f"bone parameters of width {bones.shape[-1]}")


# ---- kinematic chain -------------------------------------------------------------------------------------------
def _levels(parents):
    """Joints grouped by depth below the root: [(joint ids, parent ids), ...] (SMPL: 8 levels of 3,3,3,5,3,2,2,2)."""
    parents = np.asarray(parents)
    depth = np.zeros(len(parents), dtype=np.int64)
    for j in range(len(parents)):                     # parents precede children in SMPL's table; general tables: walk up
        d, p = 0, j
        while parents[p] != p:
            p = parents[p]
            d += 1
        depth[j] = d
    return [(np.nonzero(depth == d)[0], parents[depth == d]) for d in range(1, int(depth.max()) + 1)]


def kinematic_chain(rots, rest_pose, parents=sk.JOINT_PARENTS, pelvis=None):
    """rots (N,J,3,3), rest_pose (1|N,J,3) -> l2ws (N,J,4,4), skts (N,J,4,4), kps (N,J,3).

    Joint j's local-to-world is the product of [R_a | rest_a - rest_parent(a)] along the path root..j, the root's
    translation being its rest position (pose_opt.py:264-339, :341-372); `pelvis` (N,3) shifts every joint."""
    N, J = rots.shape[:2]
    rest = rest_pose.expand(N, J, 3)
    root = int(np.nonzero(np.asarray(parents) == np.arange(J))[0][0])
    R = [None] * J
    t = [None] * J
    R[root], t[root] = rots[:, root], rest[:, root]
    for ids, par in _levels(parents):
        Rp = torch.stack([R[p] for p in par], 1)                                     # (N,L,3,3)
        tp = torch.stack([t[p] for p in par], 1)
        off = (rest[:, ids] - rest[:, par])[..., None]
        Rl = Rp @ rots[:, ids]
        tl = (Rp @ off)[..., 0] + tp
        for n, j in enumerate(ids):
            R[j], t[j] = Rl[:, n], tl[:, n]
    R, t = torch.stack(R, 1), torch.stack(t, 1)
    if pelvis is not None:
        t = t + pelvis[:, None]
    bottom = torch.tensor([0., 0., 0., 1.], dtype=R.dtype, device=R.device).expand(N, J, 1, 4)
    l2ws = torch.cat([torch.cat([R, t[..., None]], -1), bottom], -2)
    Rt = R.transpose(-1, -2)
    skts = torch.cat([torch.cat([Rt, -(Rt @ t[..., None])], -1), bottom], -2)        # rigid inverse
    return l2ws, skts, t


def get_kinematic_chain_T(rest_pose, bones, parents=sk.JOINT_PARENTS):
    """pose_opt.py:341-372: (kps, bones, skts, l2ws, rots) for bones (N,J,3|6) without a pelvis shift."""
    N, J, D = bones.shape
    rots = bones_to_rot(bones.reshape(-1, D)).reshape(N, J, 3, 3)
    l2ws, skts, kps = kinematic_chain(rots, rest_pose.reshape(-1, J, 3), parents)
    return kps, bones, skts, l2ws, rots


class PoseOptLayer(nn.Module):
    """pose_opt.py:132-339.  `forward(idxs)` -> (kps, bones, skts, l2ws, rots), one row per requested index."""

    def __init__(self, kps, bones, rest_pose, skel_type=None, kp_map=None, kp_uidxs=None, use_cache=False,
                 use_rot6d=False, beta=None, rest_pose_idxs=None):
        super().__init__()
        self.skel_type = skel_type if skel_type is not None else sk.SMPLSkeleton
        if list(np.asarray(self.skel_type.joint_trees)) != list(sk.JOINT_PARENTS):
            raise NotImplementedError("only support SMPLSkeleton now")                  # pose_opt.py:160
        self.parents = np.asarray(self.skel_type.joint_trees)
        self.root_id = int(self.skel_type.root_id)
        self.use_cache, self.use_rot6d = bool(use_cache), bool(use_rot6d)
        self.rest_pose_idxs = rest_pose_idxs
        if kp_map is not None:
            self.register_buffer("kp_map", torch.as_tensor(np.asarray(kp_map)).long())
            self.register_buffer("kp_uidxs", torch.as_tensor(np.asarray(kp_uidxs)).long())
        else:
            self.kp_map = self.kp_uidxs = None
        kps, bones = torch.as_tensor(kps).float(), torch.as_tensor(bones).float()
        self.beta = None if beta is None else torch.as_tensor(beta)
        self.register_buffer("rest_pose", torch.as_tensor(rest_pose).float().clone())
        self.pelvis = nn.Parameter(kps[:, self.root_id].clone())
        if self.use_rot6d:
            NJ = bones.shape[1]
            bones = rot_to_rot6d(axisang_to_rot(bones.reshape(-1, 3)).reshape(-1, NJ, 3, 3))
        if self.kp_map is None:
            self.bones = nn.Parameter(bones.clone())
        else:                                               # multi-view: one root rotation per frame, the rest shared
            self.root_bones = nn.Parameter(bones[:, self.root_id].clone())
            self.bones = nn.Parameter(bones[self.kp_uidxs, self.root_id + 1:].clone())
        self.N_kps = self.pelvis.shape[0]
        self._cache = None
        if self.use_cache:
            self.update_cache()

    # -- parameters of the requested frames (pose_opt.py:210-224)
    def idx_to_params(self, idx):
        idx = torch.as_tensor(idx, device=self.pelvis.device).long().reshape(-1)
        pelvis = self.pelvis[idx]
        if self.kp_map is None:
            return pelvis, self.bones[idx]
        return pelvis, torch.cat([self.root_bones[idx, None, :], self.bones[self.kp_map[idx]]], 1)

    def get_pelvis(self, idx=None):
        return self.idx_to_params(np.arange(self.N_kps) if idx is None else idx)[0]

    def get_beta(self):
        return self.beta

    def get_bones(self, idx=None):
        bones = self.idx_to_params(np.arange(self.N_kps) if idx is None else idx)[1]
        return rot6d_to_axisang(bones) if self.use_rot6d else bones

    def get_rest_pose(self, kp_idxs=None, rest_pose_idxs=None):
        if len(self.rest_pose) == 1:
            return self.rest_pose
        if rest_pose_idxs is not None:
            return self.rest_pose[rest_pose_idxs]
        table = torch.as_tensor(self.rest_pose_idxs, device=self.rest_pose.device).long()
        return self.rest_pose[table[torch.as_tensor(kp_idxs, device=table.device).long()]]

    @torch.no_grad()
    def update_cache(self):
        self._cache = None
        self._cache = tuple(t.detach() for t in self.calculate_kinematic(np.arange(self.N_kps)))
        self.cache_kps, self.cache_bones, self.cache_skts, self.cache_l2ws, self.cache_rots = self._cache

    def _apply(self, fn, *args, **kwargs):
        out = super()._apply(fn, *args, **kwargs)             # .to(device) / .float(): the cache follows the parameters
        if getattr(self, "_cache", None) is not None:
            self.update_cache()
        return out

    def forward(self, idxs, rest_pose_idxs=None, N_uniques=None):
        if self.use_cache and self._cache is not None:
            idx = torch.as_tensor(idxs, device=self.pelvis.device).long().reshape(-1)
            return tuple(c[idx] for c in self._cache)
        return self.calculate_kinematic(idxs, rest_pose_idxs, N_uniques)

    def calculate_kinematic(self, idxs, rest_pose_idxs=None, N_uniques=None):
        """`N_uniques`: the batch is image-major with equal runs (what `ray_collate_fn` builds, dataset.py:980-987), so
        the unique poses are `idxs[::len // N_uniques]` and the per-ray rows are stride-0 expands - no unique(), no
        host round trip.  Otherwise the indices are reduced with unique() as the reference does (:273)."""
        dev = self.pelvis.device
        if idxs is None:
            idxs = np.arange(self.N_kps)
        idx = torch.as_tensor(idxs, device=dev).long().reshape(-1)
        n = idx.shape[0]
        if N_uniques is not None and n % int(N_uniques) == 0:
            skip = n // int(N_uniques)
            uniq, inverse = idx[::skip], None
        else:
            skip = None
            uniq, inverse = torch.unique(idx, return_inverse=True)
        rest = self.get_rest_pose(uniq, rest_pose_idxs)
        pelvis, bone = self.idx_to_params(uniq)
        N, J, D = bone.shape
        rots = bones_to_rot(bone.reshape(-1, D)).reshape(N, J, 3, 3)
        l2ws, skts, kps = kinematic_chain(rots, rest, self.parents, pelvis)
        outs = (kps, bone, skts, l2ws, rots)
        if inverse is not None:
            return tuple(t[inverse] for t in outs)
        return tuple(t[:, None].expand(N, skip, *t.shape[1:]).reshape(n, *t.shape[1:]) for t in outs)


# ---- construction / checkpoints ---------------------------------------------------------------------------------
def create_popt(args, data_attrs, ckpt=None, device=None, flat=False):
    """pose_opt.py:14-83 -> (pose_optimizer, {'popt_anchors', 'popt_layer', 'skel_type'}).

    flat=True: the optimizer is a `training.FlatAdam` over a `parallel.GradBucket` of the layer's parameters (CUDA
    only) instead of `torch.optim.Adam`: one launch per step, and what `training.TrainStep(graph=True)` needs to capture
    an --opt_pose iteration.  Its state_dict is in torch.optim.Adam's format, so checkpoints load either way."""
    skel_type = data_attrs.get("skel_type", sk.SMPLSkeleton)
    J = len(skel_type.joint_names)
    rest_pose = torch.as_tensor(np.asarray(data_attrs["rest_pose"])).reshape(-1, J, 3).float()
    beta = torch.as_tensor(np.asarray(data_attrs["betas"]))
    init_kps = torch.as_tensor(np.asarray(data_attrs["kp3d"])).float()
    init_bones = torch.as_tensor(np.asarray(data_attrs["bones"])).float()
    layer = PoseOptLayer(init_kps.clone(), init_bones.clone(), rest_pose, beta=beta, skel_type=skel_type,
                         kp_map=data_attrs.get("kp_map"), kp_uidxs=data_attrs.get("kp_uidxs"),
                         rest_pose_idxs=data_attrs.get("rest_pose_idxs"), use_cache=False,
                         use_rot6d=bool(getattr(args, "opt_rot6d", False))).to(device)
    params, lr = list(layer.parameters()), getattr(args, "opt_pose_lrate", 5e-4)
    if flat:
        from . import parallel, training
        optimizer = training.FlatAdam(params, parallel.GradBucket(params), lr=lr, betas=(0.9, 0.999))
    else:
        optimizer = torch.optim.Adam(params=params, lr=lr, betas=(0.9, 0.999))
    anchor_kps, anchor_bones, anchor_beta = init_kps, init_bones, beta
    init = getattr(args, "init_poseopt", None)
    if (ckpt is not None or init is not None) and not getattr(args, "no_poseopt_reload", False):
        pose_ckpt = torch.load(init, map_location="cpu", weights_only=False) if init is not None else ckpt
        layer.load_state_dict(pose_ckpt["poseopt_layer_state_dict"])
        if "poseopt_anchors" in pose_ckpt:
            a = pose_ckpt["poseopt_anchors"]
            anchor_kps, anchor_bones, anchor_beta = a["kps"], a["bones"], a["beta"]
        if getattr(args, "use_ckpt_anchor", False):
            with torch.no_grad():
                anchor_kps, anchor_bones = (t.cpu().clone() for t in layer(torch.arange(anchor_bones.shape[0]))[:2])
            anchor_beta = layer.get_beta()
    anchor_rots = bones_to_rot(anchor_bones.reshape(-1, anchor_bones.shape[-1])).reshape(*anchor_kps.shape[:2], 3, 3)
    if getattr(args, "opt_pose_cache", False):
        layer.use_cache = True
        layer.update_cache()
    optimizer.zero_grad()
    return optimizer, {"popt_anchors": {"kps": anchor_kps, "bones": anchor_bones, "rots": anchor_rots,
                                        "beta": anchor_beta}, "popt_layer": layer, "skel_type": skel_type}


def load_bones_from_state_dict(state_dict, device="cpu"):
    """pose_opt.py:95-102: axis-angle bones whatever the stored representation."""
    bones = state_dict["poseopt_layer_state_dict"]["bones"]
    if bones.shape[-1] == 6:
        bones = rot6d_to_axisang(bones)
    return bones.to(device)


def load_poseopt_from_state_dict(state_dict):
    """pose_opt.py:104-130: a layer shaped after the checkpoint's tensors, then `load_state_dict`."""
    sd = state_dict["poseopt_layer_state_dict"]
    pelvis, bones = sd["pelvis"], sd["bones"]
    kp_map = kp_uidxs = None
    if "kp_map" in sd:
        kp_map, kp_uidxs = sd["kp_map"].cpu().numpy(), sd["kp_uidxs"].cpu().numpy()
    N, NJ, ND = pelvis.shape[0], bones.shape[1], bones.shape[2]
    if kp_map is not None:
        NJ += 1                                             # the root bone is stored apart
    layer = PoseOptLayer(torch.zeros(N, NJ, 3), torch.zeros(N, NJ, 3), torch.zeros(1, NJ, 3), use_rot6d=ND == 6,
                         kp_map=kp_map, kp_uidxs=kp_uidxs)
    layer.load_state_dict(sd)
    return layer


def pose_ckpt_to_pose_data(path=None, popt_sd=None, ext_scale=0.001, legacy=False):
    """pose_opt.py:415-451: refined poses of a checkpoint as the arrays the renderer's data loading uses:
    (kp3d, bones, skts, cyls, rest_pose, pelvis), float32 numpy; the chain is evaluated in float64 as the reference's
    numpy path (`get_smpl_l2ws`, skeleton_utils.py:334-376) does."""
    if legacy:
        raise NotImplementedError("legacy (A-NeRF v1, y/z-swapped) pose checkpoints are not implemented")
    if popt_sd is None:
        popt_sd = torch.load(path, map_location="cpu", weights_only=False)["poseopt_layer_state_dict"]
    layer = load_poseopt_from_state_dict({"poseopt_layer_state_dict": popt_sd})
    with torch.no_grad():
        pelvis = layer.get_pelvis().cpu().numpy()
        bones = layer.get_bones().cpu().numpy()
        rest_pose = layer.get_rest_pose()[0].cpu().numpy()
    l2ws = np.stack([sk.forward_kinematics(b, rest_pose, 1.0, layer.parents) for b in bones])
    l2ws[..., :3, -1] += pelvis[:, None]
    kp3d = l2ws[..., :3, -1].copy().astype(np.float32)
    skts = np.linalg.inv(l2ws).astype(np.float32)
    cyls = sk.bounding_cylinder(kp3d, ext_scale=ext_scale, extend_mm=250, head="-y").astype(np.float32)
    return kp3d, bones, skts, cyls, rest_pose, pelvis


# ---- the trainer's pose regulariser (core/trainer.py:446-505) ----------------------------------------------------
def kp_loss(args, anchors, kp_idx, kp_opts, popt_layer=None, temp_val=None):
    """-> ({'kp_loss'[, 'temp_loss']}, {'MPJPC'}).  `kp_opts`: {'kp_batch', 'bones', 'rots'} from the layer's forward."""
    kp_idx = torch.as_tensor(kp_idx).long()
    dev = kp_opts["bones"].device
    pick = lambda t: t[kp_idx.to(t.device)].to(dev)       # anchors kept on the layer's device are indexed there (no sync)
    if getattr(args, "opt_rot6d", False):
        reg = rot_to_rot6d(pick(anchors["rots"]))
        bones = rot_to_rot6d(kp_opts["rots"])
    else:
        reg = pick(anchors["bones"])
        bones = kp_opts["bones"]
    assert len(reg) == len(bones)
    tol = float(getattr(args, "opt_pose_tol", 0.))
    d = (reg - bones).pow(2.)[:, 1:]                                        # root excluded
    d = torch.where(d > tol, d - tol, torch.zeros_like(d)).sum(-1)          # hinge at the tolerance
    losses = {"kp_loss": d.mean() * float(getattr(args, "opt_pose_coef", 0.))}
    if getattr(args, "use_temp_loss", False):
        n_frames = len(popt_layer.bones)
        prev_k, prev_b, _, _, prev_r = popt_layer(kp_idx - 1)
        next_k, next_b, _, _, next_r = popt_layer((kp_idx + 1) % n_frames)
        if getattr(args, "opt_rot6d", False):
            prev_b, next_b = rot_to_rot6d(prev_r), rot_to_rot6d(next_r)
        prev_k, prev_b, next_k, next_b = (t.detach() for t in (prev_k, prev_b, next_k, next_b))
        kps = kp_opts["kp_batch"]
        ang = ((bones - prev_b) - (next_b - bones)).pow(2.).sum(-1)
        vel = ((kps - prev_k) - (next_k - kps)).pow(2.).sum(-1)
        losses["temp_loss"] = ((ang + vel) * temp_val[..., None].to(dev)).mean() * float(args.temp_coef)
    pjpc = (pick(anchors["kps"]) - kp_opts["kp_batch"].detach()).pow(2.).sum(-1).pow(0.5)
    return losses, {"MPJPC": pjpc.mean() / float(getattr(args, "ext_scale", 0.001))}


# ---- 2D keypoint reprojection term (the torch statement of danbo_pose_kp2d, csrc/pose.cu) ---------------------------
def kp2d_loss(kps, kp2d, proj, sigma, coef):
    """kps (G,24,3) world-frame joints, kp2d (G,24,3) detections (pixel u, pixel v, confidence c >= 0) in SMPL joint
    order, proj (G,3,4) projection matrices.  -> (loss, kp2d_px): coef / (G*24) * sum c (rho(r_u) + rho(r_v)) with the
    Geman-McClure rho(r) = sigma^2 r^2 / (sigma^2 + r^2) on the pixel residuals, and the mean |r| over the joints with
    c > 0 (detached).  Joints at or behind the camera (w = P2 [kps, 1] <= 1e-6) contribute nothing, gradient included."""
    G, J = kps.shape[:2]
    X = torch.cat([kps, torch.ones_like(kps[..., :1])], -1)
    h = (proj[:, None] @ X[..., None])[..., 0]                                 # (G,J,3)
    front = h[..., 2] > 1e-6
    w = torch.where(front, h[..., 2], torch.ones_like(h[..., 2]))
    r = h[..., :2] / w[..., None] - kp2d[..., :2]
    r = torch.where(front[..., None], r, torch.zeros_like(r))
    s2 = float(sigma) ** 2
    rho = (s2 * r * r / (s2 + r * r)).sum(-1)
    c = kp2d[..., 2]
    loss = (c * rho).sum() * (float(coef) / (G * J))
    seen = (front & (c > 0)).to(r.dtype)
    px = (r.detach().norm(dim=-1) * seen).sum() / seen.sum().clamp(min=1)
    return loss, px
