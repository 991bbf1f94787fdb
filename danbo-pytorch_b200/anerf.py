"""A-NeRF (nerf_type = nerf, BASELINE config #4) behind the reference's plain `RayCaster` (SURVEY §8a row AN1).

`AnerfField` owns the parameters under the reference's names (core/networks/nerf.py:73-105 with W = 448, view_W = 224,
plus the cutoff embedders' `cutoff_dist` / `tau` entries, cutoff_embedder.py:128-133) so reference checkpoints load.
`AnerfCaster` mirrors raycasters.py:205-546 for this network type: cylinder near/far only (:419-420), every sample
goes through the field, single_net fine pass on the S_f new samples (F9), or a separate fine network on all S_c + S_f
merged samples (anerf_h).  Train mode: the forward keeps every layer's activation tile image (`danbo_anerf_mlp_save`)
and `_AnerfBlock.backward` turns d (rgb, acc) into the MLP / frame-code gradients of each network with the compositing
backward kernels and `kernels.anerf_mlp_backward`; when the poses require a gradient (--opt_pose) it also returns
d loss / d skts through `kernels.anerf_embed_bwd`.
"""
import torch
import torch.nn as nn

from . import kernels as K
from .networks import Optcodes
from .raycaster import RayCaster, MAX_RAYS_PER_LAUNCH

J = 24
CUTOFF = 500 * 0.001                     # cutoff_mm * ext_scale (encoders.py:62, run_nerf.py:498)


class _CutoffPE(nn.Module):
    """State of a CutoffEmbedder (cutoff_embedder.py:100-150): a frozen per-joint cutoff and the temperature buffer."""

    def __init__(self, init_tau=20.):
        super().__init__()
        self.init_tau = init_tau
        self.cutoff_dist = nn.Parameter(torch.ones(J) * CUTOFF, requires_grad=False)
        self.register_buffer("tau", torch.tensor(init_tau))

    def get_tau(self):
        return self.tau.item()

    def update_tau(self, global_step, step, rate):
        self.tau = (self.init_tau * torch.ones_like(self.tau) * rate ** (global_step / float(step * 1000))).clamp(max=2000.)


class AnerfField(nn.Module):
    def __init__(self, n_framecodes=8, W=448, D=8, view_W=224, multires=7, multires_views=4, framecode_ch=128):
        super().__init__()
        if (W, D, view_W, multires, multires_views, framecode_ch) != (448, 8, 224, 7, 4, 128):
            raise NotImplementedError("the sm_100a A-NeRF kernels are specialised for netwidth=448, netdepth=8, "
                                      "multires=7, multires_views=4, framecode_size=128 (configs/*/anerf_base.txt)")
        self.W, self.D, self.view_W = W, D, view_W
        x_ch = J * (1 + 2 * multires) + J * 3
        v_ch = J * 3 * (1 + 2 * multires_views)
        layers = [nn.Linear(x_ch, W)]
        for i in range(D - 1):
            layers.append(nn.Linear(W + x_ch, W) if i == 4 else nn.Linear(W, W))
        self.pe_fn = _CutoffPE()
        self.dirs_pe_fn = _CutoffPE()
        self.pts_linears = nn.ModuleList(layers)
        self.alpha_linear = nn.Linear(W, 1)
        self.views_linears = nn.ModuleList([nn.Linear(v_ch + framecode_ch + 2 * view_W, view_W)])
        self.feature_linear = nn.Linear(W, 2 * view_W)
        self.rgb_linear = nn.Linear(view_W, 3)
        self.framecodes = Optcodes(n_framecodes, framecode_ch)

    def update_embed_fns(self, global_step, args):
        """trainer.py:294-300: the cutoff temperature schedule."""
        step, rate = getattr(args, "tau_step", None), getattr(args, "tau_rate", None)
        if step and rate:
            self.pe_fn.update_tau(global_step, step, rate)
            self.dirs_pe_fn.update_tau(global_step, step, rate)


class AnerfCaster(RayCaster):
    """The reference's base RayCaster (raycasters.py:205-546) over the A-NeRF field, on B200 kernels.  With a separate
    fine network (single_net=False, configs/*/anerf_h.txt) the importance weights are the unsmoothed coarse weights and the
    fine network is evaluated on all S_c + S_f merged samples (raycasters.py:345-371)."""
    _supports_fine_network = True
    _supports_normals = False             # its density also depends on the point through the cut-off encodings
    _supports_parts = False               # no per-bone aggregation: every bone's encoding goes into one MLP
    _supports_scene = False               # render_scene_rays composites the DANBO render block's merge inputs
    _supports_frame_codes = False         # its code table feeds its own view branch (danbo_anerf_ray_encode)

    def __init__(self, network, network_fine=None, single_net=True, rest_poses=None, align_bones="align", skel_type=None,
                 **kwargs):
        super().__init__(network, network_fine=network_fine, single_net=single_net, rest_poses=rest_poses,
                         align_bones=align_bones, skel_type=skel_type, use_volume_near_far=False)
        self._unit_scale = None

    # ---- helpers --------------------------------------------------------------------------------------------
    def _align(self):
        dev = self._device()
        if self._align_dev is None or self._align_dev.device != dev:
            self._align_dev = self.transforms[0].to(dev).float().contiguous()
            self._unit_scale = torch.ones(J, 3, device=dev)
        return self._align_dev

    def _tau(self, net=None):
        """Cutoff temperature as a host float; read back from the buffer only when the buffer changed."""
        net = self.network if net is None else net
        t = net.pe_fn.tau
        key = (t.data_ptr(), t._version)
        cache = self.__dict__.setdefault("_tau_cache", {})
        if cache.get(id(net), (None, None))[0] != key:
            cache[id(net)] = (key, float(t.item()))
        return cache[id(net)][1]

    def _packed_mlp(self, net=None):
        net = self.network if net is None else net
        names = [f"pts_linears.{i}.{w}" for i in range(8) for w in ("weight", "bias")] + [
            "alpha_linear.weight", "alpha_linear.bias", "feature_linear.weight", "feature_linear.bias",
            "views_linears.0.weight", "views_linears.0.bias", "rgb_linear.weight", "rgb_linear.bias"]
        P = dict(net.named_parameters())
        key = tuple((P[n].data_ptr(), P[n]._version) for n in names)
        cache = self.__dict__.setdefault("_packed_cache", {})
        if self._packed_key is None:                         # set by load_state_dict / an optimizer step: repack everything
            cache.clear()
            self._packed_key = "valid"
        ent = cache.get(id(net))
        if ent is None or ent[1].wstream.device != self._device():
            ent = cache[id(net)] = [None, K.AnerfPacked(self._device())]
        # same rule as RayCaster._packed_mlp: in a train-mode forward with gradients the pack is unconditional
        force = self.training and torch.is_grad_enabled()
        if force or ent[0] != key:
            ent[1].pack({n: P[n] for n in names})
            ent[0] = key
        return ent[1]

    def _codes_of(self, net):
        w = net.framecodes.codes.weight.detach()
        return torch.cat([w, w.mean(0, keepdim=True)], 0).contiguous()

    # ---- render ---------------------------------------------------------------------------------------------
    def _render_prepared(self, rays, pose_skts, pose_bones, pose_cyls, cam_idx, skip=1, N_samples=96, N_importance=48,
                         B=1.0, raw_noise_std=0., perturb=0., nanmean_chunk=None, lindisp=False, _rand=None,
                         _stages=None):
        N = rays.shape[0]
        align = self._align()
        packed = self._packed_mlp()
        codes = self._codes_with_mean()
        tau = self._tau()
        G = pose_skts.shape[0]
        dev = rays.device
        rand = dict(_rand or {})
        if self.training and perturb > 0 and "t_rand" not in rand:
            # the reference's draw order (SURVEY §7 hard part 4): rand, randn, rand, randn
            S_t = N_samples + N_importance
            rand = {"t_rand": torch.rand(N, N_samples, device=dev), "noise0": torch.randn(N, N_samples, device=dev),
                    "u": torch.rand(N, N_importance, device=dev), "noise1": torch.randn(N, S_t, device=dev)}
        rand = {k: v.to(dev).contiguous() for k, v in rand.items()}
        if self.training and torch.is_grad_enabled():
            # rows the networks evaluate per ray: a separate fine network runs on all S_c + S_f merged samples
            rows = N_samples + (N_samples + N_importance if not self.single_net else N_importance)
            max_train = max(MAX_RAYS_PER_LAUNCH * 24 // rows // 4096, 1) * 4096
            if not self.single_net:
                self._packed_mlp(self.network_fine)         # the unconditional train-mode pack, as for the coarse network
            if N > max_train:
                raise NotImplementedError(f"A-NeRF training batches above {max_train} rays are not implemented")
            return _anerf_block_with_grad(self, rays, skip, pose_skts, pose_cyls, cam_idx, codes, align, packed, tau,
                                          N_samples, N_importance, B, nanmean_chunk, lindisp, rand, raw_noise_std, _stages)
        # every sample is evaluated: bound the rows of one launch sequence (operand images are 2.3 KB per row)
        max_rays = max(MAX_RAYS_PER_LAUNCH * 24 // (N_samples + N_importance) // 4096, 1) * 4096
        block = max_rays if G == 1 else max((max_rays // skip) * skip, skip)
        if nanmean_chunk and G == 1:
            block = max((block // int(nanmean_chunk)) * int(nanmean_chunk), int(nanmean_chunk))
        outs = []
        for s0 in range(0, N, block):
            s1 = min(N, s0 + block)
            outs.append(self._render_block_anerf(rays[s0:s1], s0, skip, pose_skts, pose_cyls, cam_idx[s0:s1], codes, align,
                                                 packed, tau, N_samples, N_importance, B, nanmean_chunk, _stages,
                                                 lindisp=lindisp, rand={k: v[s0:s1] for k, v in rand.items()},
                                                 raw_noise_std=raw_noise_std if self.training else 0.))
        if len(outs) == 1:
            return outs[0]
        return {k: torch.cat([o[k] for o in outs], 0) for k in outs[0]}

    def _render_block_anerf(self, rays, ray0, skip, pose_skts, pose_cyls, cam_idx, codes, align, packed, tau, S_c, S_f, B,
                            nanmean_chunk, stages, lindisp=False, rand=None, raw_noise_std=0., keep=None):
        """rand: the four random tensors of a train-mode call (stratified jitter, density noise, importance u); keep
        (dict): receives what the backward pass needs, and makes the MLP keep its activations."""
        rand = rand or {}
        save = keep is not None
        n = rays.shape[0]
        dev = rays.device
        if pose_skts.shape[0] == 1:
            p0 = 0
        else:
            assert ray0 % skip == 0
            p0 = ray0 // skip
        p_skts, p_cyls = pose_skts[p0:], pose_cyls[p0:]
        seg = 0 if not nanmean_chunk else int(nanmean_chunk)
        near, far = K.nearfar(rays, p_cyls, p_skts, skip, align, self._unit_scale, seg_len=seg, use_box=False)   # NF1
        enc, code_bias = K.anerf_ray_encode(rays, p_skts, skip, cam_idx, codes, packed)
        # SM1 (ray_utils.py:206-253, eval): z = near (1 - t) + far t, the reference's own two-product form
        t = torch.linspace(0., 1., steps=S_c, device=dev)
        if not lindisp:
            z0 = (near[:, None] * (1. - t) + far[:, None] * t).contiguous()
        else:                                                # ray_utils.py:226-227, the reference's own expression
            z0 = (1. / (1. / near[:, None] * (1. - t) + 1. / far[:, None] * t)).contiguous()
        if "t_rand" in rand:                                 # stratified jitter, ray_utils.py:233-248 (the reference's ops)
            mids = .5 * (z0[..., 1:] + z0[..., :-1])
            upper, lower = torch.cat([mids, z0[..., -1:]], -1), torch.cat([z0[..., :1], mids], -1)
            z0 = (lower + (upper - lower) * rand["t_rand"]).contiguous()
        xd, xv = K.anerf_embed(rays, S_c, z0, p_skts, skip, align, enc, tau)
        raw0 = torch.empty(n * S_c + n, 4, device=dev, dtype=torch.float32)
        sv0 = K.anerf_save_buffer(n * S_c, dev) if save else None
        K.anerf_mlp(xd, xv, packed, code_bias, n * S_c, S_c, raw0, save=sv0)
        ones0 = torch.ones(n, S_c, device=dev, dtype=torch.int32)          # every sample carries its own field value
        inv_B = 1.0 / B
        noise0 = (rand["noise0"] * (raw_noise_std * B)).contiguous() if ("noise0" in rand and raw_noise_std > 0) else None
        c0 = K.composite_resample(rays, S_c, S_f, raw0, ones0, z0, noise=noise0, inv_B=inv_B, u_rand=rand.get("u"),
                                  want_inds=stages is not None, smooth=self.single_net, want_weights=stages is not None)
        z1 = c0["z_samples"]
        if save:
            keep.update(dict(rays=rays, cam_idx=cam_idx, codes=codes, code_bias=code_bias, S_c=S_c, S_f=S_f, inv_B=inv_B,
                             z0=z0, raw0=raw0, ones0=ones0, noise0=noise0, xd0=xd, xv0=xv, sv0=sv0, ray_enc=enc,
                             p_skts=p_skts, skip=skip, align=align, tau=tau))
        if not self.single_net:
            return self._fine_network_pass(rays, p_skts, skip, cam_idx, align, S_c, S_f, B, c0, near, far, z0, raw0, stages,
                                           rand=rand, raw_noise_std=raw_noise_std, keep=keep)
        if save:                                             # the coarse pass's operand images are read again by the backward
            xd1, xv1 = K.anerf_embed(rays, S_f, z1, p_skts, skip, align, enc, tau)
        else:
            xd1, xv1 = K.anerf_embed(rays, S_f, z1, p_skts, skip, align, enc, tau, xd=xd, xv=xv)
        raw1 = torch.empty(n * S_f, 4, device=dev, dtype=torch.float32)
        sv1 = K.anerf_save_buffer(n * S_f, dev) if save else None
        K.anerf_mlp(xd1, xv1, packed, code_bias, n * S_f, S_f, raw1, save=sv1)
        ones1 = torch.ones(n, S_f, device=dev, dtype=torch.int32)
        noise1 = (rand["noise1"] * (raw_noise_std * B)).contiguous() if ("noise1" in rand and raw_noise_std > 0) else None
        c1 = K.merge_composite(rays, S_c, S_f, raw0, ones0, raw1, ones1, c0["z_all"], c0["order"], noise=noise1,
                               inv_B=inv_B, want_raw=stages is not None)
        if save:
            keep.update(dict(raw1=raw1, ones1=ones1, noise1=noise1, xd1=xd1, xv1=xv1, sv1=sv1, z_all=c0["z_all"],
                             order=c0["order"], z1=z1))
        ret = {"rgb_map": c1["rgb_map"], "disp_map": c1["disp_map"], "acc_map": c1["acc_map"], "alpha": c1["alpha"],
               "T_i": c1["weights"], "rgb0": c0["rgb_map"], "disp0": c0["disp_map"], "acc0": c0["acc_map"],
               "alpha0": c0["alpha"]}
        if stages is not None:
            stages.update({"near": near, "far": far, "z_coarse": z0, "raw0": raw0, "weights0": c0["weights"],
                           "z_samples": z1, "z_all": c0["z_all"], "sorted_idxs": c0["order"], "raw1": raw1,
                           "raw": c1.get("raw"), "ray_enc": enc, "code_bias": code_bias})
        return ret

    def _fine_network_pass(self, rays, p_skts, skip, cam_idx, align, S_c, S_f, B, c0, near, far, z0, raw0, stages,
                           rand=None, raw_noise_std=0., keep=None):
        """single_net=False (raycasters.py:350-376): the fine network on all S_c + S_f merged samples, then raw2outputs
        (with the train-mode density noise `noise1`, as raw2outputs adds it whenever raw_noise_std > 0).  keep: as in
        _render_block_anerf."""
        rand = rand or {}
        n, dev = rays.shape[0], rays.device
        fine = self.network_fine
        S_t = S_c + S_f
        packed_f = self._packed_mlp(fine)
        codes_f, tau_f = self._codes_of(fine), self._tau(fine)
        enc_f, code_bias_f = K.anerf_ray_encode(rays, p_skts, skip, cam_idx, codes_f, packed_f)
        z_all = c0["z_all"]
        xd, xv = K.anerf_embed(rays, S_t, z_all, p_skts, skip, align, enc_f, tau_f)
        raw = torch.empty(n * S_t + n, 4, device=dev, dtype=torch.float32)       # tail rows: unused empty entries
        sv = K.anerf_save_buffer(n * S_t, dev) if keep is not None else None
        K.anerf_mlp(xd, xv, packed_f, code_bias_f, n * S_t, S_t, raw, save=sv)
        ones = torch.ones(n, S_t, device=dev, dtype=torch.int32)
        inv_B = 1.0 / B
        noise1 = (rand["noise1"] * (raw_noise_std * B)).contiguous() if ("noise1" in rand and raw_noise_std > 0) else None
        c1 = K.composite_resample(rays, S_t, 0, raw, ones, z_all, noise=noise1, inv_B=inv_B)
        if keep is not None:
            keep.update(dict(raw_f=raw, ones_f=ones, z_all=z_all, noise1=noise1, xd_f=xd, xv_f=xv, sv_f=sv,
                             code_bias_f=code_bias_f, codes_f=codes_f, ray_enc_f=enc_f, tau_f=tau_f))
        ret = {"rgb_map": c1["rgb_map"], "disp_map": c1["disp_map"], "acc_map": c1["acc_map"], "alpha": c1["alpha"],
               "T_i": c1["weights"], "rgb0": c0["rgb_map"], "disp0": c0["disp_map"], "acc0": c0["acc_map"],
               "alpha0": c0["alpha"]}
        if stages is not None:
            stages.update({"near": near, "far": far, "z_coarse": z0, "raw0": raw0, "weights0": c0["weights"],
                           "z_samples": c0["z_samples"], "z_all": z_all, "sorted_idxs": c0["order"],
                           "raw": raw[: n * S_t].reshape(n, S_t, 4)})
        return ret

    # ---- density queries (D1 for this field; not part of config #4) ------------------------------------------
    @torch.no_grad()
    def render_pts_density(self, pts, kps, skts, bones=None, netchunk=1024 * 64, network=None):
        """Raw sigma at points (P,1,3) or (P,3) for ONE pose (raycasters.py:439-453, nerf.py:136-154 forward_pts).
        Each point is a one-sample ray (o = point, z = 0) through the render path's own kernels; sigma is the head of the
        density trunk and does not depend on the view branch, which runs on an arbitrary unit direction."""
        assert kps.shape[0] == 1, f"Assuming only one poses are provided, got {kps.shape[0]} instead"
        dev = self._device()
        P = pts.shape[0]
        p = pts.reshape(P, 3).to(dev).float()
        align, packed, codes, tau = self._align(), self._packed_mlp(), self._codes_with_mean(), self._tau()
        p_skts = skts.to(dev).float().contiguous()
        out = torch.empty(P, device=dev)
        block = MAX_RAYS_PER_LAUNCH * 8                     # rows per launch sequence (operand images: 2.3 KB per row)
        for s0 in range(0, P, block):
            s1 = min(P, s0 + block)
            n = s1 - s0
            rays = torch.zeros(n, 8, device=dev)
            rays[:, :3] = p[s0:s1]
            rays[:, 5] = 1.0
            cam = torch.zeros(n, device=dev, dtype=torch.int32)
            enc, code_bias = K.anerf_ray_encode(rays, p_skts, n, cam, codes, packed)
            z = torch.zeros(n, 1, device=dev)
            xd, xv = K.anerf_embed(rays, 1, z, p_skts, n, align, enc, tau)
            raw = torch.empty(n, 4, device=dev, dtype=torch.float32)
            K.anerf_mlp(xd, xv, packed, code_bias, n, 1, raw)
            out[s0:s1] = raw[:, 3]
        return out.reshape(P, 1, 1) if pts.dim() == 3 else out.reshape(P, 1)

    # render_mesh_density: inherited (lattice around the root joint -> render_pts_density)


ANERF_PARAM_NAMES = [f"pts_linears.{i}.{w}" for i in range(8) for w in ("weight", "bias")] + [
    "alpha_linear.weight", "alpha_linear.bias", "feature_linear.weight", "feature_linear.bias",
    "views_linears.0.weight", "views_linears.0.bias", "rgb_linear.weight", "rgb_linear.bias", "framecodes.codes.weight"]
ANERF_OUT_KEYS = ["rgb_map", "disp_map", "acc_map", "alpha", "T_i", "rgb0", "disp0", "acc0", "alpha0"]
ANERF_DIFF_KEYS = ("rgb_map", "acc_map", "rgb0", "acc0")


class _AnerfBlock(torch.autograd.Function):
    """Autograd root of A-NeRF training: forward = the render kernels with saved activations; backward = compositing
    backward kernels (composite.cu) + kernels.anerf_mlp_backward.  Differentiable outputs are what the trainer's losses
    read (core/trainer.py:396-422): rgb_map, acc_map, rgb0, acc0.  The per-pose world-to-bone matrices are an input:
    when they require a gradient (the pose layer under --opt_pose, core/trainer.py:314-341) each pass also forms the MLP's
    input gradient and `danbo_anerf_embed_bwd` turns it into d loss / d skts.  `params`: the 25 tensors of the network in
    ANERF_PARAM_NAMES order, then those of a separate fine network (single_net=False)."""

    @staticmethod
    def forward(ctx, caster, cfg, pose_skts, *params):
        keep = {}
        with torch.no_grad():
            ret = caster._render_block_anerf(cfg["rays"], 0, cfg["skip"], pose_skts, cfg["pose_cyls"], cfg["cam_idx"],
                                             cfg["codes"], cfg["align"], cfg["packed"], cfg["tau"], cfg["S_c"], cfg["S_f"],
                                             cfg["B"], cfg["nanmean_chunk"], cfg["stages"], lindisp=cfg["lindisp"],
                                             rand=cfg["rand"], raw_noise_std=cfg["raw_noise_std"], keep=keep)
        ctx.keep, ctx.params = keep, params
        ctx.mark_non_differentiable(*[ret[k] for k in ANERF_OUT_KEYS if k not in ANERF_DIFF_KEYS])
        return tuple(ret[k] for k in ANERF_OUT_KEYS)

    @staticmethod
    def backward(ctx, *gouts):
        k = ctx.keep
        g = dict(zip(ANERF_OUT_KEYS, gouts))
        rays, dev = k["rays"], k["rays"].device
        n, S_c, S_f = rays.shape[0], k["S_c"], k["S_f"]
        zeros = lambda *s: torch.zeros(*s, device=dev, dtype=torch.float32)
        cg = lambda t, *s: zeros(*s) if t is None else t.contiguous().float()
        P = dict(zip(ANERF_PARAM_NAMES, ctx.params))
        G = {name: torch.zeros_like(p, dtype=torch.float32) for name, p in P.items()}
        separate = "raw_f" in k
        if separate:
            # the fine network's composite over all S_t merged samples; the importance samples are detached
            # (ray_utils.py:287), so the fine outputs reach only the fine network and the coarse outputs only the coarse
            S_t = S_c + S_f
            P_f = dict(zip(ANERF_PARAM_NAMES, ctx.params[len(ANERF_PARAM_NAMES):]))
            G_f = {name: torch.zeros_like(p, dtype=torch.float32) for name, p in P_f.items()}
            d_raw_f, d_raw0 = zeros(n * S_t + n, 4), zeros(n * S_c + n, 4)
            K.composite_bwd(rays, S_t, k["raw_f"], k["ones_f"], k["z_all"], k["noise1"], k["inv_B"], cg(g["rgb_map"], n, 3),
                            cg(g["acc_map"], n), d_raw_f)
        else:
            d_raw0, d_raw1 = zeros(n * S_c + n, 4), zeros(n * S_f, 4)
            K.merge_composite_bwd(rays, S_c, S_f, k["raw0"], k["ones0"], k["raw1"], k["ones1"], k["z_all"], k["order"],
                                  k["noise1"], k["inv_B"], cg(g["rgb_map"], n, 3), cg(g["acc_map"], n), None, d_raw0,
                                  d_raw1, None, None)
        K.composite_bwd(rays, S_c, k["raw0"], k["ones0"], k["z0"], k["noise0"], k["inv_B"], cg(g["rgb0"], n, 3),
                        cg(g["acc0"], n), d_raw0)
        want_pose = ctx.needs_input_grad[2]
        d_skts = zeros(*k["p_skts"].shape) if want_pose else None         # p0 == 0: a training block holds every pose
        coarse = (P, G, d_raw0, S_c, k["z0"], k["xd0"], k["xv0"], k["sv0"], k["code_bias"], k["codes"], k["ray_enc"],
                  k["tau"])
        if separate:
            fine = (P_f, G_f, d_raw_f, S_t, k["z_all"], k["xd_f"], k["xv_f"], k["sv_f"], k["code_bias_f"], k["codes_f"],
                    k["ray_enc_f"], k["tau_f"])
        else:
            fine = (P, G, d_raw1, S_f, k["z1"], k["xd1"], k["xv1"], k["sv1"], k["code_bias"], k["codes"], k["ray_enc"],
                    k["tau"])
        for Pn, Gn, d_raw, S, z, xd, xv, sv, code_bias, codes, enc, tau in (coarse, fine):
            dx = K.anerf_mlp_backward(Pn, Gn, d_raw, n * S, S, xd, xv, sv, code_bias, k["cam_idx"], codes, want_dx=want_pose)
            if want_pose:
                K.anerf_embed_bwd(rays, S, z, k["p_skts"], k["skip"], k["align"], enc, tau, dx[0], dx[1], d_skts)
                del dx
        ctx.keep = None
        grads = tuple(G[name] for name in ANERF_PARAM_NAMES)
        if separate:
            grads += tuple(G_f[name] for name in ANERF_PARAM_NAMES)
        return (None, None, d_skts) + grads


def _anerf_block_with_grad(caster, rays, skip, pose_skts, pose_cyls, cam_idx, codes, align, packed, tau, S_c, S_f, B,
                           nanmean_chunk, lindisp, rand, raw_noise_std, stages):
    params = [dict(caster.network.named_parameters())[n] for n in ANERF_PARAM_NAMES]
    if not caster.single_net:
        params += [dict(caster.network_fine.named_parameters())[n] for n in ANERF_PARAM_NAMES]
    cfg = dict(rays=rays, skip=skip, pose_cyls=pose_cyls, cam_idx=cam_idx, codes=codes, align=align,
               packed=packed, tau=tau, S_c=S_c, S_f=S_f, B=B, nanmean_chunk=nanmean_chunk, lindisp=lindisp, rand=rand,
               raw_noise_std=raw_noise_std, stages=stages)
    outs = _AnerfBlock.apply(caster, cfg, pose_skts, *params)
    return dict(zip(ANERF_OUT_KEYS, outs))


_ANERF_REQUIRED = {"netdepth": 8, "netwidth": 448, "multires": 7, "multires_views": 4, "multires_bones": 0,
                   "framecode_size": 128, "opt_framecode": True, "use_viewdirs": True,
                   "use_cutoff": True, "cutoff_viewdir": True, "cutoff_inputs": True, "cutoff_shift": True,
                   "cut_to_dist": True, "cutoff_bones": False, "normalize_cutoff": False, "opt_cutoff": False,
                   "freq_schedule": False, "cutoff_mm": 500.0, "ext_scale": 0.001, "i_embed": 0}
_ANERF_SUPPORTED = {"align_bones": ("align",), "density_type": ("relu",), "kp_dist_type": ("reldist",),
                    "view_type": ("relray",), "ray_tr_type": ("local",), "pts_tr_type": ("local",), "bone_type": ("reldir",)}


def check_anerf_args(args):
    """The flag subset of configs/*/anerf_base.txt that selects this path; anything else raises."""
    from .raycaster import _flag
    for k, allowed in _ANERF_SUPPORTED.items():
        v = _flag(args, k)
        if v not in allowed:
            raise NotImplementedError(f"{k}={v!r} is not implemented for nerf_type='nerf' (supported: {allowed})")
    for k, want in _ANERF_REQUIRED.items():
        v = _flag(args, k)
        if v != want:
            raise NotImplementedError(f"{k}={v!r} is not implemented for nerf_type='nerf' (kernels are built for {k}={want!r})")
    if getattr(args, "netwidth_view", None) not in (None, 224):
        raise NotImplementedError("netwidth_view must be None/224")
