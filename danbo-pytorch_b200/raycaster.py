"""Drop-in mirror of the reference's ray caster for the DANBO hot path (SURVEY §8b).

Same class surface as core/raycasters.py:205-716 (RayCaster / GraphCaster): construction through
`create_raycaster(args, data_attrs)`, `forward(*args, fwd_type=..., **kwargs)`, `render_rays(...)` with the
reference's argument names, `render_mesh_density`, `render_pts_density`, the custom `state_dict` key scheme
(`network_fn_state_dict`, `network_fine_state_dict`), `.network`, `.network_fine`, `.transforms`, `.rest_poses`,
`update_embed_fns`, `get_networks`.  The work itself is a fixed sequence of CUDA kernels from libdanbo_b200.so.

Unsupported flag combinations raise NotImplementedError (never a silent fallback).
"""
import os

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import kernels as K
from . import skeleton as sk
from .networks import DanboField

MAX_RAYS_PER_LAUNCH = 262144          # multiple of every sane `chunk`; bounds the size of the X tile buffer (1.5 GB at danbo_fast density)
# Opt-in (not yet measured on hardware): an eval call of one pose is cut into this many ray blocks whose launch
# sequences are issued on separate streams, so that the issue-/LSU-bound kernels of one block can fill the SM time the
# tensor-bound MLP kernel of the other leaves (and the gaps between dependent launches).  1 = one stream, as measured.
BLOCK_STREAMS = int(os.environ.get("DANBO_BLOCK_STREAMS", "1"))
# Rows (samples) per launch sequence of the surface-normal paths (render_pts_gradient, render_rays(want_normals=True)):
# they keep the bf16 MLP activations and the encoded rows for a backward pass, about 7 KB per row, so 2^18 rows hold
# about 1.8 GB.
NORMAL_BLOCK_ROWS = 1 << 18


class RayCaster(nn.Module):
    """GraphCaster of the reference (raycasters.py:642-716) on B200 kernels."""

    _supports_fine_network = False        # a separate fine network (single_net=False): the A-NeRF caster only
    _supports_normals = True              # density gradients / normals (render_pts_gradient, want_normals): DANBO only
    _supports_parts = True                # body-part maps (render_pts_parts, want_parts): a field with an aggregation net

    def __init__(self, network, network_fine=None, single_net=True, rest_poses=None, align_bones="align",
                 skel_type=None, use_volume_near_far=False, view_mode="world", **kwargs):
        super().__init__()
        separate = (not single_net) and network_fine is not None and network_fine is not network
        if (not single_net or (network_fine is not None and network_fine is not network)) and not (
                separate and self._supports_fine_network):
            raise NotImplementedError("single_net=False (separate fine network) is implemented for nerf_type='nerf' only "
                                      "(configs/*/anerf_h.txt); every DANBO config ships single_net=True")
        if align_bones != "align":
            raise NotImplementedError(f"align_bones={align_bones!r}: only 'align' is implemented")
        self.network = network
        self.network_fine = network_fine if separate else network
        self.single_net = not separate
        self.rest_poses = rest_poses
        self.skel_type = skel_type if skel_type is not None else sk.SMPLSkeleton
        self.align_bones = align_bones
        self.use_volume_near_far = bool(use_volume_near_far)
        if view_mode not in ("world", "root_local"):
            raise NotImplementedError(f"view_mode={view_mode!r}")
        self.view_mode = view_mode                # what V1 encodes: rays_d as they are, or in the root joint's frame
        A, child = sk.bone_align_transforms(rest_poses)          # S0
        self.transforms = torch.from_numpy(A)[None]               # (1,24,4,4) like the reference attribute
        self.child_idxs = child
        self._packed = None
        self._packed_key = None
        self._pack_gen = 0                        # bumped by every weight pack: the transposed pack follows it
        self._packed_t = None
        self._packed_t_gen = -1
        self._align_dev = None
        self._graphed = None
        self.block_streams = BLOCK_STREAMS
        self._side_streams = []

    # ------------------------------------------------------------------------------------------------ dispatch
    def forward(self, *args, fwd_type="", **kwargs):
        if fwd_type == "density":
            return self.render_pts_density(*args, **kwargs)
        if fwd_type == "mesh":
            return self.render_mesh_density(*args, **kwargs)
        if fwd_type == "density_color":
            raise NotImplementedError("fwd_type='density_color' is broken in the reference (render_pts_density has no "
                                      "`color` argument, raycasters.py:236-237)")
        if not self.training:
            with torch.no_grad():
                return self.render_rays(*args, **kwargs)
        return self.render_rays(*args, **kwargs)

    def get_networks(self):
        return self.network, self.network_fine

    def render_graphed(self, ray_batch, N_samples, kp_batch=None, skts=None, cyls=None, bones=None, cams=None,
                       N_uniques=1, N_importance=0, nanmean_chunk=None, preproc_kwargs=None, lindisp=False, **ignored):
        """Eval-mode render replayed from a CUDA graph (one graph per ray count).  Same inputs and returned dict as the
        plain call; the returned tensors are static buffers that the next graphed call overwrites."""
        from .graphs import GraphedFn
        if self.training:
            raise RuntimeError("render_graphed is for eval mode")
        if ignored.get("want_normals"):
            raise NotImplementedError("want_normals is not implemented for render_graphed (normals are not captured): "
                                      "use the plain call")
        if ignored.get("want_parts"):
            raise NotImplementedError("want_parts is not implemented for render_graphed (part maps are not captured): "
                                      "use the plain call")
        if ignored.get("ray_noise_std", 0.) > 0 or ignored.get("pytest"):
            raise NotImplementedError("ray_noise_std > 0 and pytest are not implemented")
        B = float((preproc_kwargs or {}).get("density_scale", 1.0))
        rays, pose_skts, pose_bones, pose_cyls, cam_idx, skip = self._prepare(ray_batch, skts, cyls, bones, cams, N_uniques)
        if self._graphed is None:
            def run(rays, pose_skts, pose_bones, pose_cyls, cam_idx, _param_ptrs=None, **kw):
                with torch.no_grad():
                    return self._render_prepared(rays, pose_skts, pose_bones, pose_cyls, cam_idx, **kw)
            self._graphed = GraphedFn(run, self._device())
        # A captured graph reads the parameters through the raw pointers they had at capture time (the weight pack, the
        # graph net and the aggregation net all read them live, so value changes are always seen); the pointers are part
        # of the graph key, so re-pointed storage (`.to()`, an optimizer's flat arena) gets a fresh capture.
        ptrs = hash(tuple(p.data_ptr() for p in self.parameters()))
        self._packed_mlp()                    # eager: repacks (into the buffers the graph reads) iff the weights changed
        return self._graphed(rays=rays, pose_skts=pose_skts, pose_bones=pose_bones, pose_cyls=pose_cyls, cam_idx=cam_idx,
                             skip=skip, N_samples=N_samples, N_importance=N_importance, B=B, nanmean_chunk=nanmean_chunk,
                             lindisp=bool(lindisp), _param_ptrs=ptrs)

    def update_embed_fns(self, global_step, args):
        self.network.update_embed_fns(global_step, args)
        if self.network_fine is not self.network:                      # raycasters.py:596-597
            self.network_fine.update_embed_fns(global_step, args)

    # custom key scheme of raycasters.py:601-637
    def state_dict(self, *args, **kwargs):
        sd = self.network.state_dict()
        fine = sd if self.network_fine is self.network else self.network_fine.state_dict()
        return {"network_fn_state_dict": sd, "network_fine_state_dict": fine}

    @staticmethod
    def _load_into(net, sd, strict):
        own = net.state_dict()
        try:
            net.load_state_dict(sd, strict=strict)
        except (KeyError, RuntimeError):
            filt = {k: v for k, v in sd.items() if k in own and tuple(own[k].shape) == tuple(v.shape)}
            net.load_state_dict(filt, strict=False)

    def load_state_dict(self, ckpt, strict=True):
        sd = ckpt["network_fn_state_dict"] if "network_fn_state_dict" in ckpt else ckpt
        self._load_into(self.network, sd, strict)
        if self.network_fine is not self.network and "network_fine_state_dict" in ckpt:
            self._load_into(self.network_fine, ckpt["network_fine_state_dict"], strict)
        self._packed_key = None

    # ------------------------------------------------------------------------------------------------ helpers
    def _device(self):
        return self.network.alpha_linear.weight.device

    def _consts(self):
        net = self.network
        dev = self._device()
        if self._align_dev is None or self._align_dev.device != dev:
            self._align_dev = self.transforms[0].to(dev).float().contiguous()      # once; a per-call H2D copy would sync
        return K.FieldConsts(self._align_dev, net.graph_net.axis_scale, net.agg_tensors())

    def _packed_mlp(self):
        net = self.network
        names = [f"pts_linears.{i}.{w}" for i in range(8) for w in ("weight", "bias")] + [
            "alpha_linear.weight", "alpha_linear.bias", "feature_linear.weight", "feature_linear.bias",
            "views_linears.0.weight", "views_linears.0.bias", "rgb_linear.weight", "rgb_linear.bias"]
        P = dict(net.named_parameters())
        key = tuple((P[n].data_ptr(), P[n]._version) for n in names)
        if self._packed is None or self._packed.wstream.device != self._device():
            self._packed = K.PackedMLP(self._device())
            self._packed_key = None
        # The host-side key cannot see an update made by a kernel through raw pointers, and a replayed CUDA graph never
        # runs this Python at all.  So the pack is unconditional in every train-mode forward with gradients - eager or
        # being captured: the pack launches then belong to the training graph and every replay packs the weights the
        # previous replay's Adam wrote.  Eval calls rely on the key: it changes with every torch in-place op
        # (`_version`), `load_state_dict`, `TrainStep` (which invalidates it after every iteration) and `FlatAdam.step`
        # (which bumps the parameters' versions); `render_graphed` checks it EAGERLY before each replay and repacks into
        # the same static buffers, so an eval graph holds no pack launch and still never sees stale weights.  A train-mode
        # forward in which no MLP weight needs a gradient (training.PoseFitStep: the field is frozen) is keyed the same
        # way; PoseFitStep checks the key eagerly before each replay of its graph.
        force = self.training and torch.is_grad_enabled() and any(P[n].requires_grad for n in names)
        # a forced (training) pack skips the empty-sample constants, which only calls without a backward pass read
        if force or key != self._packed_key or not self._packed.has_empty:
            tensors = {n: P[n] for n in names}
            if not getattr(net, "opt_framecode", True):
                # no frame code: the kernels' view layer keeps its 411-input layout with zero weights (and zero codes,
                # `_codes_with_mean`) in the code columns, which adds exact zeros
                tensors["views_linears.0.weight"] = F.pad(P["views_linears.0.weight"].detach(), (0, 128))
            self._packed.pack(tensors, want_empty=not force)
            self._packed_key = key
            self._pack_gen += 1
        return self._packed

    def _packed_dgrad(self):
        """The transposed weight tiles of the MLP's data-gradient chain for a backward that trains no weight (the
        pose-only path): repacked only when `_packed_mlp` last repacked, so it follows the same key.  (A training
        backward packs them into its own workspace every iteration, autograd._RenderBlock.)"""
        packed = self._packed_mlp()
        if self._packed_t is None or self._packed_t.wstream.device != self._device():
            self._packed_t = K.PackedDgrad(self._device())
            self._packed_t_gen = -1
        if self._packed_t_gen != self._pack_gen:
            P = dict(self.network.named_parameters())
            tensors = {n: P[n] for n in ["feature_linear.weight", "views_linears.0.weight"] +
                       [f"pts_linears.{i}.weight" for i in range(8)]}
            if not getattr(self.network, "opt_framecode", True):     # the kernels' 411-column view layout, as above
                tensors["views_linears.0.weight"] = F.pad(P["views_linears.0.weight"].detach(), (0, 128))
            self._packed_t.pack(tensors)
            self._packed_t_gen = self._pack_gen
        return self._packed_t

    def _codes_with_mean(self):
        if not getattr(self.network, "opt_framecode", True):
            return torch.zeros(2, 128, device=self._device())
        w = self.network.framecodes.codes.weight.detach()
        return torch.cat([w, w.mean(0, keepdim=True)], 0).contiguous()

    @staticmethod
    def _unique(t, skip):
        return t[::skip].contiguous().float()

    def _view_rays(self, rays, p_skts, skip):
        """The rays whose direction columns V1 encodes.  "world" (ray_tr_type=world + view_type=identity, the h36m_zju
        and surreal configs): the rays themselves.  "root_local" (ray_tr_type=root_local + view_type=relray, the perfcap
        configs; RootLocalEncoder encoders.py:570-578, VecNormEncoder :774-795): a copy whose direction is rotated into
        the root joint's frame of the ray's pose and normalised - a per-ray quantity, so the folded view layer
        (`ray_bias`) takes it unchanged."""
        if self.view_mode == "world":
            return rays
        n, G = rays.shape[0], p_skts.shape[0]
        if G == 1:
            d = rays[:, 3:6] @ p_skts[0, 0, :3, :3].t()
        else:
            pose = torch.clamp(torch.arange(n, device=rays.device) // skip, max=G - 1)
            d = (p_skts[pose, 0, :3, :3] @ rays[:, 3:6, None])[..., 0]
        out = rays[:, :8].clone()
        out[:, 3:6] = F.normalize(d, dim=-1, p=2)
        return out

    # ------------------------------------------------------------------------------------------------ render
    def render_rays(self, ray_batch, N_samples, kp_batch, skts=None, cyls=None, bones=None, cams=None,
                    subject_idxs=None, retraw=False, lindisp=False, perturb=0., N_importance=0, network_fine=None,
                    raw_noise_std=0., ray_noise_std=0., verbose=False, ext_scale=0.001, pytest=False, N_uniques=1,
                    render_confd=False, render_entropy=False, preproc_kwargs=None, netchunk=1024 * 64,
                    nerf_type="danbo", use_viewdirs=True, nanmean_chunk=None, want_normals=False, want_parts=False,
                    _rand=None, _stages=None):
        """Same arguments and returned dict as raycasters.py:245-377,516-546,710-716.

        Extra (optional) keywords: `nanmean_chunk` keeps the reference's per-chunk near/far fill (F8) when more than
        one reference chunk is passed in a single call; `want_normals` adds `normal_map` (n,3), the composite of the
        samples' unit normals (`_render_normals`; eval mode without gradients only); `want_parts` adds `part_map` (n,24),
        the composite of the samples' aggregation weights p_j (eval mode without gradients only; not together with
        `want_normals`); `_rand`/`_stages` are test hooks (inject the four random tensors / collect stage tensors)."""
        if want_normals:
            self._refuse_normals("render_rays(want_normals=True)")
            if self.training or torch.is_grad_enabled():
                raise NotImplementedError("want_normals is for eval mode without gradients (caster.eval(), torch.no_grad()): "
                                          "normals in training are not implemented")
        if want_parts:
            self._refuse_parts("render_rays(want_parts=True)")
            if self.training or torch.is_grad_enabled():
                raise NotImplementedError("want_parts is for eval mode without gradients (caster.eval(), torch.no_grad()): "
                                          "part maps in training are not implemented")
            if want_normals:
                raise NotImplementedError("want_parts together with want_normals in one call is not implemented: make two "
                                          "calls")
        # render_confd / render_entropy / verbose / retraw are accepted and ignored, as in the reference's render_rays
        # (raycasters.py:245-377 never reads them)
        if ray_noise_std > 0 or pytest:
            raise NotImplementedError("ray_noise_std > 0 (samples moved off their ray) and pytest (numpy's fixed random "
                                      "numbers) are not implemented")
        if N_importance <= 0:
            raise NotImplementedError("N_importance must be > 0 (the reference itself requires it, SURVEY F10)")
        if skts is None or bones is None or cyls is None:
            raise ValueError("skts, bones and cyls are required")
        if cams is None and getattr(self.network, "opt_framecode", True):
            raise ValueError("cams are required (the field has per-frame codes)")
        pk = preproc_kwargs or {}
        if pk.get("density_fn", F.relu) is not F.relu:
            raise NotImplementedError("density_type other than 'relu' is not implemented")
        B = float(pk.get("density_scale", 1.0))
        rays, pose_skts, pose_bones, pose_cyls, cam_idx, skip = self._prepare(ray_batch, skts, cyls, bones, cams, N_uniques)
        if want_normals:
            return self._render_normals(rays, pose_skts, pose_bones, pose_cyls, cam_idx, skip, N_samples, N_importance, B,
                                        nanmean_chunk, bool(lindisp), _stages)
        return self._render_prepared(rays, pose_skts, pose_bones, pose_cyls, cam_idx, skip=skip, N_samples=N_samples,
                                     N_importance=N_importance, B=B, raw_noise_std=raw_noise_std, perturb=perturb,
                                     nanmean_chunk=nanmean_chunk, lindisp=bool(lindisp), _rand=_rand, _stages=_stages,
                                     **({"want_parts": True} if want_parts else {}))

    def _prepare(self, ray_batch, skts, cyls, bones, cams, N_uniques):
        """Host-side reduction of the reference's per-ray stride-0 expands to per-pose tables (encoders.py:465-471)."""
        dev = self._device()
        N = ray_batch.shape[0]
        skip = max(N // max(int(N_uniques), 1), 1)
        rays = ray_batch.to(dev, non_blocking=True).float().contiguous()
        pose_skts = self._unique(skts, skip).to(dev, non_blocking=True)
        pose_bones = self._unique(bones, skip).to(dev, non_blocking=True)
        pose_cyls = self._unique(cyls, skip).to(dev, non_blocking=True)
        if cams is None or not getattr(self.network, "opt_framecode", True):
            cam_idx = torch.zeros(N, device=dev, dtype=torch.int32)       # no frame codes: row 0 of the zero table
        else:
            cam_idx = cams.reshape(N, -1)[:, 0].to(dev, non_blocking=True).to(torch.int32).contiguous()
        return rays, pose_skts, pose_bones, pose_cyls, cam_idx, skip

    def _render_prepared(self, rays, pose_skts, pose_bones, pose_cyls, cam_idx, skip=1, N_samples=64, N_importance=16,
                         B=1.0, raw_noise_std=0., perturb=0., nanmean_chunk=None, lindisp=False, _rand=None, _stages=None,
                         want_parts=False):
        dev = self._device()
        N = rays.shape[0]
        net = self.network
        consts = self._consts()
        packed = self._packed_mlp()
        vol = net.bone_volumes(pose_bones).float().contiguous()            # GN1 + GN2 (PyTorch, <= 16 poses; autograd)
        codes = self._codes_with_mean()
        training = self.training
        rand = _rand or {}
        if training and perturb > 0 and "t_rand" not in rand:
            # the reference's draw order (SURVEY §7 hard part 4): rand, randn, rand, randn
            S_t = N_samples + N_importance
            rand = {"t_rand": torch.rand(N, N_samples, device=dev),
                    "noise0": torch.randn(N, N_samples, device=dev), "u": torch.rand(N, N_importance, device=dev),
                    "noise1": torch.randn(N, S_t, device=dev)}
        if training and torch.is_grad_enabled():
            from .autograd import render_block_with_grad
            if N > MAX_RAYS_PER_LAUNCH:
                raise NotImplementedError(f"training batches above {MAX_RAYS_PER_LAUNCH} rays are not implemented")
            return render_block_with_grad(self, rays, skip, pose_skts, pose_cyls, vol, cam_idx, codes, consts, packed,
                                          N_samples, N_importance, B, raw_noise_std, perturb, nanmean_chunk,
                                          {k: v.to(dev).contiguous() for k, v in rand.items()}, _stages, lindisp=lindisp)
        outs = []
        # internal launches: any split works for a single pose; with several poses a block holds whole poses
        G = pose_skts.shape[0]
        block, n_streams = self._plan_blocks(N, G, skip, nanmean_chunk,
                                             self.block_streams if (not training and _stages is None) else 1)
        cur = torch.cuda.current_stream(dev) if n_streams > 1 else None
        while len(self._side_streams) < (n_streams if n_streams > 1 else 0):
            self._side_streams.append(torch.cuda.Stream(device=dev))
        used = []
        for i, s0 in enumerate(range(0, N, block)):
            s1 = min(N, s0 + block)
            sub_rand = {k: v[s0:s1].to(dev).contiguous() for k, v in rand.items()}
            args = (rays[s0:s1], s0, skip, pose_skts, pose_cyls, vol, cam_idx[s0:s1], codes, consts, packed, N_samples,
                    N_importance, B, raw_noise_std, perturb, training, nanmean_chunk, sub_rand, _stages)
            if n_streams > 1:
                side = self._side_streams[i % n_streams]
                if side not in used:
                    side.wait_stream(cur)                                   # inputs, packed weights, bone volumes
                    used.append(side)
                with torch.cuda.stream(side):
                    out = self._render_block(*args, lindisp=lindisp, want_parts=want_parts)
                if not torch.cuda.is_current_stream_capturing():           # a captured graph's memory is static anyway
                    for t in out.values():
                        t.record_stream(cur)                                # consumed (cat) on the caller's stream
                outs.append(out)
            else:
                outs.append(self._render_block(*args, lindisp=lindisp, want_parts=want_parts))
        for side in used:
            cur.wait_stream(side)
        if len(outs) == 1:
            return outs[0]
        return {k: torch.cat([o[k] for o in outs], 0) for k in outs[0]}

    @staticmethod
    def _plan_blocks(N, G, skip, nanmean_chunk, want_streams):
        """-> (rays per internal launch block, streams to issue the blocks on).  One pose: any split gives the same
        pixels as long as blocks are whole near/far fill chunks (F8); several poses: a block holds whole poses.  More than
        one stream only for a single pose, with `nanmean_chunk` given (so the split cannot change a pixel) and a call
        large enough to be worth it."""
        block = MAX_RAYS_PER_LAUNCH if G == 1 else max((MAX_RAYS_PER_LAUNCH // skip) * skip, skip)
        n_streams = int(want_streams) if (G == 1 and nanmean_chunk and N >= 32768 and want_streams > 1) else 1
        if n_streams > 1:
            unit = int(nanmean_chunk)
            block = min(block, -(-(-(-N // n_streams)) // unit) * unit)     # ceil(N / n_streams) rounded up to the unit
        if nanmean_chunk and G == 1:
            block = max((block // int(nanmean_chunk)) * int(nanmean_chunk), int(nanmean_chunk))
        return block, n_streams

    def _render_block(self, rays, ray0, skip, pose_skts, pose_cyls, vol, cam_idx, codes, consts, packed, S_c, S_f, B,
                      raw_noise_std, perturb, training, nanmean_chunk, rand, stages, keep=None, lindisp=False,
                      nearfar=None, want_parts=False):
        """One launch sequence over <= MAX_RAYS_PER_LAUNCH rays.  `keep` (dict) receives every intermediate the
        backward pass needs (train mode with gradients, and the normal map).  `nearfar`: the block's (near, far), when
        the caller computed them over a larger range of rays (the normal map's blocks).  `want_parts` (eval): the fine
        composite also writes `part_map` (danbo_merge_composite_parts)."""
        n = rays.shape[0]
        # poses of this block: ray (ray0 + i) -> pose (ray0 + i) // skip
        if pose_skts.shape[0] == 1:
            p0 = 0
        else:
            assert ray0 % skip == 0
            p0 = ray0 // skip
        p_skts, p_cyls, p_vol = pose_skts[p0:], pose_cyls[p0:], vol[p0:]
        seg = 0 if not nanmean_chunk else int(nanmean_chunk)
        if nearfar is None:
            near, far = K.nearfar(rays, p_cyls, p_skts, skip, consts.align, consts.axis_scale, seg_len=seg,
                                  use_box=self.use_volume_near_far, bound=1.3)
        else:
            near, far = nearfar
        rays_v = self._view_rays(rays, p_skts, skip)
        rbias = K.ray_bias(rays_v, cam_idx, codes, packed)
        inv_B = 1.0 / B
        save = keep is not None
        # A sample no bone sees has MLP input PE(0): its output depends on the ray only through the view bias.  Without a
        # backward pass the n per-ray rows come from the weight pack's constants (K.mlp_empty_rows) instead of the MLP
        # (9 % of the rows of a 512x512 image); with one they stay MLP rows, so that their gradient takes the same path.
        const_empty = not save
        raw0 = torch.empty(n * S_c + n, 4, device=rays.device, dtype=torch.float32)
        if const_empty:
            K.mlp_empty_rows(rbias, packed, raw0[n * S_c:])
        # ---- coarse pass
        t_rand = rand.get("t_rand") if (training and perturb > 0) or "t_rand" in rand else None
        z0, mask0, act0 = K.sample_mask(rays, S_c, p_skts, skip, consts, near=near, far=far, t_rand=t_rand,
                                        append_empty=not const_empty, lindisp=lindisp)
        agg_mode = self.network.agg_mode
        f0 = K.field_agg(rays, S_c, z0, mask0, act0, p_skts, p_vol, skip, consts, want_hbar=save, want_xrows=save,
                         agg_mode=agg_mode)
        sv0 = sv1 = None
        if save:
            sv0 = K.ActSave(act0.capacity, rays.device)
            K.mlp_forward_save(f0.xtiles, packed, rbias, act0, f0.row_ray, raw0, sv0)
        else:
            K.mlp_forward(f0.xtiles, packed, rbias, act0, f0.row_ray, raw0)
        noise0 = (rand["noise0"] * (raw_noise_std * B)).contiguous() if ("noise0" in rand and raw_noise_std > 0) else None
        c0 = K.composite_resample(rays, S_c, S_f, raw0, mask0, z0, noise=noise0, inv_B=inv_B, u_rand=rand.get("u"),
                                  want_inds=stages is not None, want_weights=stages is not None)
        if "z_fine" in rand:
            # test hook: evaluate the fine pass at given importance samples (z_fine, z_all, order as the reference
            # produced them) instead of this pass's own - cuts the coarse -> fine coupling for stage-wise parity checks
            c0 = dict(c0, z_samples=rand["z_fine"].float().contiguous(), z_all=rand["z_all"].float().contiguous(),
                      order=rand["order"].to(torch.int32).contiguous())
        # ---- fine pass: only the S_f new samples go through the field (single_net, SURVEY F9)
        z1, mask1, act1 = K.sample_mask(rays, S_f, p_skts, skip, consts, z_in=c0["z_samples"], append_empty=False)
        f1 = K.field_agg(rays, S_f, z1, mask1, act1, p_skts, p_vol, skip, consts, want_hbar=save, want_xrows=save,
                         agg_mode=agg_mode)
        raw1 = torch.empty(n * S_f, 4, device=rays.device, dtype=torch.float32)
        if save:
            sv1 = K.ActSave(act1.capacity, rays.device)
            K.mlp_forward_save(f1.xtiles, packed, rbias, act1, f1.row_ray, raw1, sv1)
        else:
            K.mlp_forward(f1.xtiles, packed, rbias, act1, f1.row_ray, raw1)
        noise1 = (rand["noise1"] * (raw_noise_std * B)).contiguous() if ("noise1" in rand and raw_noise_std > 0) else None
        if want_parts:
            c1 = K.merge_composite_parts(rays, S_c, S_f, raw0, mask0, raw1, mask1, c0["z_all"], c0["order"], f0.logits,
                                         f1.logits, agg_mode, noise=noise1, inv_B=inv_B, want_raw=stages is not None)
        else:
            c1 = K.merge_composite(rays, S_c, S_f, raw0, mask0, raw1, mask1, c0["z_all"], c0["order"], noise=noise1,
                                   inv_B=inv_B, want_raw=stages is not None, confd0=f0.logits if training else None,
                                   confd1=f1.logits if training else None, want_invalid=training)
        ret = {"rgb_map": c1["rgb_map"], "disp_map": c1["disp_map"], "acc_map": c1["acc_map"], "alpha": c1["alpha"],
               "T_i": c1["weights"], "rgb0": c0["rgb_map"], "disp0": c0["disp_map"], "acc0": c0["acc_map"],
               "alpha0": c0["alpha"]}
        if training:
            ret["confd"] = c1["confd"]
            ret["part_invalid"] = c1["part_invalid"]
        if want_parts:
            ret["part_map"] = c1["part_map"]
        if save:
            keep.update(dict(rays=rays, rays_v=rays_v, cam_idx=cam_idx, codes=codes, p_skts=p_skts, p_vol=p_vol, p0=p0, skip=skip,
                             consts=consts, S_c=S_c, S_f=S_f, inv_B=inv_B, z0=z0, mask0=mask0, act0=act0, f0=f0, raw0=raw0,
                             sv0=sv0, noise0=noise0, z1=z1, mask1=mask1, act1=act1, f1=f1, raw1=raw1, sv1=sv1,
                             noise1=noise1, z_all=c0["z_all"], order=c0["order"]))
        if stages is not None:
            stages.update({"near": near, "far": far, "vol": vol, "z_coarse": z0, "mask0": mask0, "raw0": raw0,
                           "weights0": c0["weights"], "z_samples": c0["z_samples"], "z_all": c0["z_all"],
                           "sorted_idxs": c0["order"], "inds": c0.get("inds"), "mask1": mask1, "raw1": raw1,
                           "raw": c1.get("raw"), "n_active0": act0.count, "n_active1": act1.count,
                           "ray_bias": rbias})
        return ret

    # ------------------------------------------------------------------------------------------------ normals
    def _refuse_normals(self, what):
        if not self._supports_normals:
            raise NotImplementedError(f"{what}: density gradients are implemented for the DANBO field only (the A-NeRF "
                                      "field's density depends on the point through its cut-off encodings as well)")

    def _pass_gradient(self, rays, S, z, mask, act, fo, sv, p_skts, p_vol, skip, consts, packed_t):
        """d raw sigma / d p of every sample of one saved pass, from one backward pass seeded with d raw = (0,0,0,1) on
        every row (rows are independent, so each sample gets its own gradient) -> (n*S, 3).  A sample no bone sees has
        no active row and gets exactly 0."""
        dev = rays.device
        n = rays.shape[0]
        d_raw = torch.zeros(n * S + n, 4, device=dev)           # covers the appended empty entries (ids >= n*S) too
        d_raw[:, 3] = 1.
        P = dict(self.network.named_parameters())
        dX = K.mlp_backward_pose({k: P[k].detach() for k in ("rgb_linear.weight", "alpha_linear.weight")}, d_raw, act,
                                 fo, sv, packed_t)
        d_pts = torch.zeros(n * S, 3, device=dev)
        K.field_agg_bwd_pts(rays, S, z, mask, act, p_skts, p_vol, skip, consts, fo, dX, d_pts)
        return d_pts

    @staticmethod
    def _unit_normals(grad):
        """-grad / |grad| (the outward normal of a density level set); exactly 0 where the gradient is 0."""
        nrm = grad.norm(dim=-1, keepdim=True)
        return torch.where(nrm > 0, -grad / torch.where(nrm > 0, nrm, torch.ones_like(nrm)), torch.zeros_like(grad))

    @torch.no_grad()
    def render_pts_gradient(self, pts, kps, skts, bones, netchunk=NORMAL_BLOCK_ROWS):
        """Raw sigma and its gradient with respect to the point, in world coordinates, at points (P,1,3) or (P,3) for
        ONE pose -> (sigma (P,1), grad (P,3)).  sigma is what render_pts_density returns.  The gradient is the field's
        true derivative (the feature window is differentiated, where training detaches it); a point no bone sees gets
        exactly 0.  Points go in chunks of `netchunk` (the saved activations take about 7 KB per point).  No autograd:
        the network's parameters and their .grad are untouched."""
        self._refuse_normals("render_pts_gradient")
        if kps.shape[0] != 1 or skts.shape[0] != 1 or bones.shape[0] != 1:
            raise NotImplementedError("render_pts_gradient takes one pose (kps, skts, bones with a leading 1)")
        dev = self._device()
        P = pts.shape[0]
        p_all = pts.reshape(P, 3).to(dev).float()
        consts, packed, packed_t = self._consts(), self._packed_mlp(), self._packed_dgrad()
        p_skts = skts.to(dev).float().contiguous()
        vol = self.network.bone_volumes(bones.to(dev).float()).float().contiguous()
        agg_mode = self.network.agg_mode
        sigma = torch.empty(P, device=dev)
        grad = torch.empty(P, 3, device=dev)
        chunk = max(int(netchunk), 1)
        for c0 in range(0, P, chunk):
            c1 = min(P, c0 + chunk)
            m = c1 - c0
            rays = torch.zeros(m, 8, device=dev)                    # "rays" with o = point, d = 0, z = 0
            rays[:, :3] = p_all[c0:c1]
            z = torch.zeros(m, 1, device=dev)
            # append_empty=2: one extra entry (id 2m-1) carries sigma of a point that no bone sees, as in render_pts_density
            _, mask, act = K.sample_mask(rays, 1, p_skts, m, consts, z_in=z, append_empty=2, capacity=m + 1)
            fo = K.field_agg(rays, 1, z, mask, act, p_skts, vol, m, consts, want_hbar=True, want_xrows=True,
                             agg_mode=agg_mode)
            if not torch.cuda.is_current_stream_capturing() and fo.overflowed():
                fo = K.field_agg(rays, 1, z, mask, act, p_skts, vol, m, consts, want_hbar=True, want_xrows=True,
                                 agg_mode=agg_mode, pairs_per_row=K.J)
            raw = torch.empty(2 * m, 4, device=dev)
            sv = K.ActSave(act.capacity, dev)
            # the colour head reads a view bias; sigma does not, and its backward seed has no colour component
            K.mlp_forward_save(fo.xtiles, packed, torch.zeros(m, 128, device=dev), act, fo.row_ray, raw, sv)
            grad[c0:c1] = self._pass_gradient(rays, 1, z, mask, act, fo, sv, p_skts, vol, m, consts, packed_t)
            sigma[c0:c1] = torch.where(mask.reshape(-1) != 0, raw[:m, 3], raw[2 * m - 1, 3])
        return (sigma.reshape(P, 1, 1) if pts.dim() == 3 else sigma.reshape(P, 1)), grad

    def _render_normals(self, rays, pose_skts, pose_bones, pose_cyls, cam_idx, skip, S_c, S_f, B, nanmean_chunk,
                        lindisp, stages):
        """render_rays(want_normals=True): the eval render (no perturbation, no noise) with its intermediates kept, the
        seeded backward of render_pts_gradient on both passes, and normal_map = sum_m w_m n_m over the merged samples
        with the fine composite's weights (world frame, not renormalised).  The plain call's blocks (and their near /
        far fill segments) are kept; each is cut into ray blocks of at most NORMAL_BLOCK_ROWS samples of a single
        pose."""
        dev = self._device()
        N = rays.shape[0]
        net = self.network
        consts, packed, packed_t = self._consts(), self._packed_mlp(), self._packed_dgrad()
        vol = net.bone_volumes(pose_bones).float().contiguous()
        codes = self._codes_with_mean()
        G = pose_skts.shape[0]
        block, _ = self._plan_blocks(N, G, skip, nanmean_chunk, 1)
        seg = 0 if not nanmean_chunk else int(nanmean_chunk)
        sub_rays = max(1, NORMAL_BLOCK_ROWS // (S_c + S_f + 1))
        outs = []
        for s0 in range(0, N, block):
            s1 = min(N, s0 + block)
            p0 = 0 if G == 1 else s0 // skip
            near, far = K.nearfar(rays[s0:s1], pose_cyls[p0:], pose_skts[p0:], skip, consts.align, consts.axis_scale,
                                  seg_len=seg, use_box=self.use_volume_near_far, bound=1.3)
            # sub-blocks of one pose each: ray i of the call belongs to pose min(i // skip, G - 1)
            a = s0
            while a < s1:
                g = min(a // skip, G - 1)
                pose_end = s1 if g == G - 1 else min(s1, (g + 1) * skip)
                b = min(pose_end, a + sub_rays)
                keep = {}
                ret = self._render_block(rays[a:b], 0, b - a, pose_skts[g:g + 1], pose_cyls[g:g + 1], vol[g:g + 1],
                                         cam_idx[a:b], codes, consts, packed, S_c, S_f, B, 0., 0., False, nanmean_chunk,
                                         {}, stages, keep=keep, lindisp=lindisp,
                                         nearfar=(near[a - s0:b - s0], far[a - s0:b - s0]))
                k = keep
                n = b - a
                g0 = self._pass_gradient(k["rays"], S_c, k["z0"], k["mask0"], k["act0"], k["f0"], k["sv0"], k["p_skts"],
                                         k["p_vol"], k["skip"], consts, packed_t)
                g1 = self._pass_gradient(k["rays"], S_f, k["z1"], k["mask1"], k["act1"], k["f1"], k["sv1"], k["p_skts"],
                                         k["p_vol"], k["skip"], consts, packed_t)
                nrm = self._unit_normals(torch.cat([g0.reshape(n, S_c, 3), g1.reshape(n, S_f, 3)], 1))
                nrm = torch.gather(nrm, 1, k["order"].long()[..., None].expand(-1, -1, 3))      # merge order (z_all)
                ret["normal_map"] = (ret["T_i"][..., None] * nrm).sum(1)
                outs.append(ret)
                a = b
        if len(outs) == 1:
            return outs[0]
        return {k: torch.cat([o[k] for o in outs], 0) for k in outs[0]}

    # ------------------------------------------------------------------------------------------------ density grid
    @torch.no_grad()
    def render_pts_density(self, pts, kps, skts, bones, netchunk=1024 * 64, network=None):
        """Raw sigma at points (P,1,3) or (P,3) for ONE pose (raycasters.py:439-453, nerf.py:136-154)."""
        assert kps.shape[0] == 1, f"Assuming only one poses are provided, got {kps.shape[0]} instead"
        out, _, _ = self._pts_field(pts, skts, bones)
        return out.reshape(pts.shape[0], 1, 1) if pts.dim() == 3 else out.reshape(pts.shape[0], 1)

    def _pts_field(self, pts, skts, bones):
        """render_pts_density's launches -> (raw sigma (P,), visibility masks (P,) int32, FieldOut of the points)."""
        dev = self._device()
        P = pts.shape[0]
        p = pts.reshape(P, 3).to(dev).float()
        rays = torch.zeros(P, 8, device=dev)                         # "rays" with o = point, d = 0, z = 0
        rays[:, :3] = p
        consts, packed = self._consts(), self._packed_mlp()
        p_skts = skts.to(dev).float().contiguous()
        vol = self.network.bone_volumes(bones.to(dev).float()).float().contiguous()
        z = torch.zeros(P, 1, device=dev)
        # append_empty=2: one extra entry (id 2P-1) carries sigma of a point that no bone sees (h = 0)
        _, mask, act = K.sample_mask(rays, 1, p_skts, P, consts, z_in=z, append_empty=2, capacity=P + 1)
        fo = K.field_agg(rays, 1, z, mask, act, p_skts, vol, P, consts, agg_mode=self.network.agg_mode)
        if not torch.cuda.is_current_stream_capturing() and fo.overflowed():
            # a dense lattice inside the body: more than 6 visible bones per point on average -> worst-case workspace
            fo = K.field_agg(rays, 1, z, mask, act, p_skts, vol, P, consts, agg_mode=self.network.agg_mode,
                             pairs_per_row=K.J)
        sigma = torch.empty(2 * P, device=dev)
        K.mlp_forward(fo.xtiles, packed, None, act, fo.row_ray, sigma, density_only=True)
        return torch.where(mask.reshape(-1) != 0, sigma[:P], sigma[2 * P - 1]), mask.reshape(-1), fo

    # ------------------------------------------------------------------------------------------------ part maps
    def _refuse_parts(self, what):
        if not self._supports_parts:
            raise NotImplementedError(f"{what}: body-part weights are implemented for the DANBO field only (the A-NeRF "
                                      "field has no per-bone aggregation)")

    @torch.no_grad()
    def render_pts_parts(self, pts, kps, skts, bones):
        """Raw sigma and the aggregation weights p_j of every bone at points (P,1,3) or (P,3) for ONE pose
        -> (sigma (P,1) or (P,1,1), p (P,24)).  sigma is render_pts_density's; p = network.get_agg(logits, invalid) with
        the field's logits and visibility masks of the same launches, 0 for a point no bone sees."""
        self._refuse_parts("render_pts_parts")
        if kps.shape[0] != 1 or skts.shape[0] != 1 or bones.shape[0] != 1:
            raise NotImplementedError("render_pts_parts takes one pose (kps, skts, bones with a leading 1)")
        P = pts.shape[0]
        sigma, mask, fo = self._pts_field(pts, skts, bones)
        vis = ((mask.long()[:, None] >> torch.arange(K.J, device=mask.device)) & 1).bool()
        # entries danbo_field_agg did not write are uninitialised (and x 0 may still be NaN): a sigmoid pass writes the
        # visible bones only, a softmax pass all 24 of a row some bone sees (its max runs over all of them)
        written = vis if self.network.agg_type == "sigmoid" else vis.any(-1, keepdim=True)
        logits = torch.where(written, fo.logits[:P], torch.zeros((), device=mask.device))
        p = self.network.get_agg(logits, (~vis).float())
        return (sigma.reshape(P, 1, 1) if pts.dim() == 3 else sigma.reshape(P, 1)), p

    @torch.no_grad()
    def render_mesh_density(self, kps, skts, bones, subject_idxs=None, radius=1.0, res=64, render_kwargs=None,
                            netchunk=1024 * 64, v=None):
        """(res+1)^3 lattice of raw sigma around the root joint, x/y swapped (raycasters.py:421-437)."""
        t = np.linspace(-radius, radius, res + 1)
        grid = np.stack(np.meshgrid(t, t, t), axis=-1).astype(np.float32)
        sh = grid.shape
        pts = torch.tensor(grid.reshape(-1, 3)).to(self._device()) + kps[0, 0].to(self._device())
        sigma = self.render_pts_density(pts.reshape(-1, 1, 3), kps, skts, bones, netchunk)[..., :1]
        return sigma.reshape(*sh[:-1]).transpose(1, 0)


GraphCaster = RayCaster


# ------------------------------------------------------------------------------------------------------ factory
_SUPPORTED = {"nerf_type": ("danbo", "graph"), "gnn_backbone": ("FGNNcat",), "agg_backbone": ("vox_MIXGNN",),
              "agg_type": ("sigmoid", "softmax"), "align_bones": ("align",), "density_type": ("relu",),
              "kp_dist_type": ("reldist",), "view_type": ("identity", "relray"), "ray_tr_type": ("world", "root_local"),
              "pts_tr_type": ("local",), "bone_type": ("Nope",), "graph_input_type": ("rot6d",)}
_REQUIRED = {"netdepth": 8, "netwidth": 256, "agg_W": 32, "agg_D": 3, "node_W": 128, "gcn_D": 4, "gcn_fc_D": 1,
             "voxel_res": 16, "voxel_feat": 5, "multires_voxel": 6, "multires_graph": 5, "multires_views": 4,
             "framecode_size": 128, "single_net": True, "use_viewdirs": True,
             "mask_root": True, "attenuate_feat": True, "attenuate_invalid": False, "use_cutoff": False,
             "opt_posecode": False, "gnn_concat": False, "no_adj": False, "adj_self_one": False,
             "align_corners": False, "vol_cal_scale": True}


def _flag(args, k):
    """A flag's value; a flag the namespace does not carry has the reference CLI's own default (run_nerf.py:186-572,
    config.DEFAULTS), exactly what the reference's parser would have filled in - never "whatever is supported"."""
    from .config import DEFAULTS
    if hasattr(args, k):
        return getattr(args, k)
    if k in DEFAULTS:
        return DEFAULTS[k]
    raise NotImplementedError(f"flag {k!r} is missing from args and has no reference default on record")


def check_args(args):
    """The flag subset that selects this path (SURVEY §8a 'config' row); anything else raises."""
    for k, allowed in _SUPPORTED.items():
        v = _flag(args, k)
        if v not in allowed:
            raise NotImplementedError(f"{k}={v!r} is not implemented by danbo_b200 (supported: {allowed})")
    for k, want in _REQUIRED.items():
        v = _flag(args, k)
        if v != want:
            raise NotImplementedError(f"{k}={v!r} is not implemented by danbo_b200 (kernels are built for {k}={want!r})")
    if _flag(args, "netwidth_view") not in (None, 128):
        raise NotImplementedError("netwidth_view must be None/128")
    view = (_flag(args, "view_type"), _flag(args, "ray_tr_type"))
    if view not in (("identity", "world"), ("relray", "root_local")):
        raise NotImplementedError(f"view_type / ray_tr_type = {view}: the shipped pairs are identity + world "
                                  "(h36m_zju, surreal) and relray + root_local (perfcap)")


def create_raycaster(args, data_attrs, device=None):
    """Mirror of core/raycasters.py:17-143: returns (render_kwargs_train, render_kwargs_test, start, grad_vars,
    optimizer, loaded_ckpt).  `render_kwargs_train['ray_caster']` exposes `.module` like nn.DataParallel does."""
    is_anerf = getattr(args, "nerf_type", "danbo") == "nerf"
    if is_anerf:
        from . import anerf as _anerf                 # A-NeRF field behind the reference's plain RayCaster (config #4)
        _anerf.check_anerf_args(args)
    else:
        check_args(args)
    device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    skel_type = data_attrs.get("skel_type", sk.SMPLSkeleton)
    rest_pose = np.asarray(data_attrs["rest_pose"], dtype=np.float32)
    n_framecodes = data_attrs["n_views"] if getattr(args, "n_framecodes", None) is None else args.n_framecodes
    profile = sk.skeleton_profile(rest_pose)
    data_attrs["skel_profile"] = profile
    if is_anerf:
        net = _anerf.AnerfField(n_framecodes=n_framecodes)
        single = bool(getattr(args, "single_net", True))
        net_fine = net if single else _anerf.AnerfField(n_framecodes=n_framecodes)        # networks/__init__.py:64-67
        caster = _anerf.AnerfCaster(net, network_fine=net_fine, single_net=single, rest_poses=rest_pose,
                                    align_bones=args.align_bones, skel_type=skel_type)
    else:
        net = DanboField(n_framecodes=n_framecodes, skel_profile=profile, opt_scale=bool(getattr(args, "opt_vol_scale", True)),
                         agg_type=args.agg_type, mask_vol_prob=bool(getattr(args, "mask_vol_prob", True)),
                         opt_framecode=bool(getattr(args, "opt_framecode", True)))
        caster = RayCaster(net, network_fine=net, single_net=True, rest_poses=rest_pose, align_bones=args.align_bones,
                           skel_type=skel_type, use_volume_near_far=bool(getattr(args, "use_volume_near_far", False)),
                           view_mode="root_local" if getattr(args, "ray_tr_type", "world") == "root_local" else "world")
    caster.to(device)
    grad_vars = [p for p in net.parameters() if p.requires_grad]
    if caster.network_fine is not net:                                 # raycasters.py:188
        grad_vars += [p for p in caster.network_fine.parameters() if p.requires_grad]
    wd = getattr(args, "weight_decay", None)
    if wd is None:
        optimizer = torch.optim.Adam(params=grad_vars, lr=args.lrate, betas=(0.9, 0.999))
    else:
        optimizer = torch.optim.AdamW(params=grad_vars, lr=args.lrate, betas=(0.9, 0.999), weight_decay=wd)
    start, loaded = 0, None
    ft = getattr(args, "ft_path", None)
    ckpts = []
    if ft is not None and ft != "None":
        ckpts = [ft]
    else:
        d = os.path.join(getattr(args, "basedir", "./logs"), getattr(args, "expname", ""))
        if os.path.isdir(d):
            ckpts = [os.path.join(d, f) for f in sorted(os.listdir(d)) if "tar" in f and "pose" not in f]
    if ckpts and not getattr(args, "no_reload", False):
        loaded = torch.load(ckpts[-1], map_location=device, weights_only=False)
        caster.load_state_dict(loaded)
        finetune = getattr(args, "finetune", False) or getattr(args, "finetune_light", False)
        if not finetune:
            start = loaded.get("global_step", 0)
            if "optimizer_state_dict" in loaded:
                optimizer.load_state_dict(loaded["optimizer_state_dict"])
    kw_train = {"ray_caster": _ModuleHandle(caster), "perturb": args.perturb, "N_importance": args.N_importance,
                "N_samples": args.N_samples, "use_viewdirs": args.use_viewdirs, "raw_noise_std": args.raw_noise_std,
                "ray_noise_std": getattr(args, "ray_noise_std", 0.), "ext_scale": getattr(args, "ext_scale", 0.001),
                "preproc_kwargs": {"density_scale": getattr(args, "density_scale", 1.0), "density_fn": F.relu},
                "lindisp": bool(getattr(args, "lindisp", False)), "nerf_type": args.nerf_type}
    kw_test = dict(kw_train)
    kw_test.update({"ray_caster": caster, "perturb": False, "raw_noise_std": 0., "ray_noise_std": 0.})
    optimizer.zero_grad()
    return kw_train, kw_test, start, grad_vars, optimizer, loaded


class _ModuleHandle(nn.Module):
    """What the trainer expects where the reference wraps the caster in nn.DataParallel (raycasters.py:116):
    callable, with `.module`.  One process drives one GPU here; multi-GPU is torch.distributed (parallel.py)."""

    def __init__(self, module):
        super().__init__()
        self.module = module

    def forward(self, *a, **k):
        return self.module(*a, **k)
