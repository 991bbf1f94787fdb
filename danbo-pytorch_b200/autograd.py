"""Autograd root of the training path: one torch.autograd.Function around a render block.

Forward = the same kernel sequence as inference (train mode keeps the bf16 MLP activations, the encoded rows and the
pair lists); backward = hand-written kernels for compositing, MLP, aggregation net, feature gather and ray bias
(csrc/backward_*.cu, composite.cu).  Gradient sources are rgb_map, acc_map, rgb0, acc0 and confd, exactly the tensors the
trainer's losses read (core/trainer.py:396-422,507-536); disp / alpha / T_i / part_invalid are non-differentiable, as in
the reference where they are used only under comparisons.  The per-pose graph net is its own node (`_GraphNet`, or the
PyTorch ops when the pose itself needs a gradient): its output `vol` is an input of this Function and receives d vol.
The per-pose world-to-bone matrices are an input too: when they require a gradient (the pose layer under --opt_pose,
core/trainer.py:314-341) `danbo_field_agg_bwd` also accumulates d loss / d skts, and with root-local view directions
(perfcap configs) `danbo_view_root_bwd` adds the view branch's part.

When no network parameter needs a gradient and the poses do (training.PoseFitStep fits poses to a frozen field), both
nodes take the pose-only path: the same data-gradient chain through compositing, MLP, field and graph net, with the
kernel variants that form no weight gradient (no K = rows GEMMs, transposes, bias sums, aggregation-net or graph-net
weight atomics, no ray-bias backward) and a transposed weight pack that is keyed on the weights instead of redone per
call (RayCaster._packed_dgrad).  A fitted frame-code table (PoseFitStep's code fitting) is one more input of the render
block; the pose-only backward then also forms its gradient (danbo_ray_bias_codes_bwd), never the network's.
"""
import torch

from . import kernels as K

MLP_NAMES = [f"pts_linears.{i}.{w}" for i in range(8) for w in ("weight", "bias")] + [
    "alpha_linear.weight", "alpha_linear.bias", "feature_linear.weight", "feature_linear.bias",
    "views_linears.0.weight", "views_linears.0.bias", "rgb_linear.weight", "rgb_linear.bias"]
AGG_NAMES = ["prob_linears.layers.0.lin.weight", "prob_linears.layers.0.adj_w", "prob_linears.layers.0.bias",
             "prob_linears.layers.1.weight", "prob_linears.layers.1.bias", "prob_linears.layers.2.weight",
             "prob_linears.layers.2.bias"]
OTHER_NAMES = ["framecodes.codes.weight", "graph_net.axis_scale"]
PARAM_NAMES = MLP_NAMES + AGG_NAMES + OTHER_NAMES
OUT_KEYS = ["rgb_map", "disp_map", "acc_map", "alpha", "T_i", "rgb0", "disp0", "acc0", "alpha0", "confd", "part_invalid"]
DIFF_KEYS = ("rgb_map", "acc_map", "rgb0", "acc0", "confd")
N_TRAINED = len(MLP_NAMES) + len(AGG_NAMES)      # parameters every training configuration trains (OTHER_NAMES may not)


def weight_grads(flags, core=None):
    """Whether a backward node trains the network's weights, from the requires-grad flags of its parameter inputs.
    True when each of the first `core` flags (default: all) is set - the others may be constants, as axis_scale without
    opt_scale or the zero code table of a field without frame codes; False when no flag is set (the pose-only path).
    Anything in between is refused: a backward that trains some of the field's weights is not implemented."""
    flags = [bool(f) for f in flags]
    core = len(flags) if core is None else int(core)
    if all(flags[:core]):
        return True
    if not any(flags):
        return False
    raise NotImplementedError("a backward in which only some of the field's parameters need a gradient is not implemented: "
                              "train all of them (training.TrainStep) or none (training.PoseFitStep)")


class _RenderBlock(torch.autograd.Function):

    @staticmethod
    def forward(ctx, caster, cfg, vol, pose_skts, frame_codes, *params):
        keep = {}
        with torch.no_grad():
            ret = caster._render_block(cfg["rays"], 0, cfg["skip"], pose_skts, cfg["pose_cyls"], vol, cfg["cam_idx"],
                                       cfg["codes"], cfg["consts"], cfg["packed"], cfg["S_c"], cfg["S_f"], cfg["B"],
                                       cfg["raw_noise_std"], cfg["perturb"], True, cfg["nanmean_chunk"], cfg["rand"],
                                       cfg["stages"], keep=keep, lindisp=cfg["lindisp"])
        ctx.keep = keep
        ctx.caster = caster
        ctx.params = params
        ctx.vol_shape = vol.shape
        ctx.codes_shape = None if frame_codes is None else frame_codes.shape
        outs = tuple(ret[k] for k in OUT_KEYS)
        ctx.mark_non_differentiable(*[ret[k] for k in OUT_KEYS if k not in DIFF_KEYS])
        return outs

    @staticmethod
    def backward(ctx, *gouts):
        k = ctx.keep
        g = dict(zip(OUT_KEYS, gouts))
        rays, dev = k["rays"], k["rays"].device
        n, S_c, S_f = rays.shape[0], k["S_c"], k["S_f"]
        zeros = lambda *s: torch.zeros(*s, device=dev, dtype=torch.float32)
        cg = lambda t, *s: zeros(*s) if t is None else t.contiguous().float()
        g_rgb, g_acc = cg(g["rgb_map"], n, 3), cg(g["acc_map"], n)
        g_rgb0, g_acc0 = cg(g["rgb0"], n, 3), cg(g["acc0"], n)
        g_confd = None if g["confd"] is None else g["confd"].contiguous().float()
        P = dict(zip(PARAM_NAMES, ctx.params))
        if not weight_grads(ctx.needs_input_grad[5:], N_TRAINED):
            return _RenderBlock._pose_only(ctx, P, g_rgb, g_acc, g_rgb0, g_acc0, g_confd)
        # Every backward kernel ACCUMULATES into its gradient buffers.  When the trainer keeps all gradients in one flat,
        # pre-zeroed bucket (parallel.GradBucket, opted in through caster.grads_in_place) the kernels add straight into
        # the parameters' .grad views and this node returns no parameter gradients: that removes one zero-fill and one
        # AccumulateGrad add per parameter tensor (86 launches per iteration).
        in_place = bool(getattr(ctx.caster, "grads_in_place", False)) and all(
            p.grad is not None and p.grad.dtype == torch.float32 and p.grad.is_contiguous() and p.grad.shape == p.shape
            for p in ctx.params)
        if in_place:
            G = {name: p.grad for name, p in P.items()}
        else:
            G = {name: torch.zeros_like(p, dtype=torch.float32) for name, p in P.items()}
        d_raw0, d_raw1 = zeros(n * S_c + n, 4), zeros(n * S_f, 4)
        gl0 = gl1 = None
        if g_confd is not None:
            gl0 = torch.empty(n * S_c, K.J, device=dev, dtype=torch.float32)
            gl1 = torch.empty(n * S_f, K.J, device=dev, dtype=torch.float32)
        # compositing (fine/merged then coarse)
        K.merge_composite_bwd(rays, S_c, S_f, k["raw0"], k["mask0"], k["raw1"], k["mask1"], k["z_all"], k["order"],
                              k["noise1"], k["inv_B"], g_rgb, g_acc, g_confd, d_raw0, d_raw1, gl0, gl1)
        K.composite_bwd(rays, S_c, k["raw0"], k["mask0"], k["z0"], k["noise0"], k["inv_B"], g_rgb0, g_acc0, d_raw0)
        if getattr(ctx.caster, "_debug_bwd", None) is not None:     # diagnostics (scripts/mlp_bwd_e2e_check.py): what the MLP
            ctx.caster._debug_bwd.update(d_raw0=d_raw0.clone(), d_raw1=d_raw1.clone(), keep=dict(k))   # backward was fed
        # MLP + field, per pass
        d_ray_bias = zeros(n, 128)
        d_vol = zeros(*ctx.vol_shape)
        d_vol_blk = d_vol[k["p0"]:]
        agg_grads = [G[nm] for nm in AGG_NAMES] + [d_vol_blk, G["graph_net.axis_scale"]]
        d_skts = zeros(*k["p_skts"].shape) if ctx.needs_input_grad[3] else None      # p0 == 0: a block holds every pose
        # Two launch streams (K.BACKWARD_STREAMS): after a pass's dgrad the weight-gradient launches (transposes, wgrad,
        # reduce, bias sums; then the ray-bias backward) and the field backward (feature gather + aggregation net) are
        # independent - they read what dgrad wrote and add into disjoint gradient tensors - so the first group goes to a
        # side stream.  At training sizes (3 072 rays) every one of these kernels is a partial wave, latency bound.
        tc = K.BACKWARD_IMPL == "tc"
        cur = torch.cuda.current_stream(dev)
        side = None
        if tc and K.BACKWARD_STREAMS > 1:
            side = getattr(ctx.caster, "_bwd_side_stream", None)
            if side is None or side.device != dev:
                side = ctx.caster._bwd_side_stream = torch.cuda.Stream(device=dev)
        wss = []
        alive = []          # tensors read by side-stream launches: must not return to the allocator before the streams join
        first = True
        side2 = None
        if side is not None:
            # a third stream for the coarse pass's field backward: it only needs that pass's dX, so the fine pass's head /
            # dgrad launches (main stream) need not wait for it.  Both passes' field backward add into the aggregation
            # net / bone volume gradients with atomics, so they may overlap.
            side2 = getattr(ctx.caster, "_bwd_side_stream2", None)
            if side2 is None or side2.device != dev:
                side2 = ctx.caster._bwd_side_stream2 = torch.cuda.Stream(device=dev)
        for ip, (d_raw, S, z, mask, act, fo, sv, gl) in enumerate((
                (d_raw0, S_c, k["z0"], k["mask0"], k["act0"], k["f0"], k["sv0"], gl0),
                (d_raw1, S_f, k["z1"], k["mask1"], k["act1"], k["f1"], k["sv1"], gl1))):
            if tc:
                if side is not None or not wss:            # a workspace per pass when the passes' launches overlap
                    wss.append(K.BwdWorkspace(act.capacity if side is not None else max(k["act0"].capacity, k["act1"].capacity), dev))
                ws = wss[-1]
                if not first:
                    ws.wstream = wss[0].wstream            # the packed transposed weights are the same for both passes
                dX = K.mlp_backward_tc(P, G, d_raw, act, fo, sv, d_ray_bias, ws, repack=first, wgrad_stream=side)
                first = False
            else:
                dX = K.mlp_backward(P, G, d_raw, act, fo, sv, d_ray_bias)
            alive.append(dX)
            if side2 is not None and ip == 0:
                side2.wait_stream(cur)
                with torch.cuda.stream(side2):
                    K.field_agg_bwd(rays, S, z, mask, act, k["p_skts"], k["p_vol"], k["skip"], k["consts"], fo, dX, gl,
                                    agg_grads, d_skts=d_skts)
            else:
                K.field_agg_bwd(rays, S, z, mask, act, k["p_skts"], k["p_vol"], k["skip"], k["consts"], fo, dX, gl,
                                agg_grads, d_skts=d_skts)
        if side2 is not None:
            cur.wait_stream(side2)
        # root-local view directions (perfcap configs) depend on the root rotation: with a pose leaf, d ray_bias also
        # flows to d skts (adds into the same tensor as field_agg_bwd's atomics)
        view_root = d_skts is not None and getattr(ctx.caster, "view_mode", "world") == "root_local"
        if side is not None:
            # d_ray_bias is complete once the second pass's head backward has run: the side stream already waits for it
            with torch.cuda.stream(side):
                K.ray_bias_bwd(k["rays_v"], k["cam_idx"], k["codes"], P["views_linears.0.weight"], d_ray_bias,
                               G["views_linears.0.weight"], G["views_linears.0.bias"], G["framecodes.codes.weight"])
                if view_root:
                    K.view_root_bwd(rays, k["p_skts"], k["skip"], P["views_linears.0.weight"], d_ray_bias, d_skts)
            cur.wait_stream(side)
        else:
            K.ray_bias_bwd(k["rays_v"], k["cam_idx"], k["codes"], P["views_linears.0.weight"], d_ray_bias,
                           G["views_linears.0.weight"], G["views_linears.0.bias"], G["framecodes.codes.weight"])
            if view_root:
                K.view_root_bwd(rays, k["p_skts"], k["skip"], P["views_linears.0.weight"], d_ray_bias, d_skts)
        ctx.keep = None
        del alive, wss
        if in_place:
            return (None, None, d_vol, d_skts, None) + (None,) * len(PARAM_NAMES)
        return (None, None, d_vol, d_skts, None) + tuple(G[name] for name in PARAM_NAMES)

    @staticmethod
    def _pose_only(ctx, P, g_rgb, g_acc, g_rgb0, g_acc0, g_confd):
        """Backward to d vol, d skts and the fitted frame codes only.  Compositing as in training; per pass the dX-only
        MLP chain (head backward only where d ray_bias is read: root-local view directions, fitted frame codes) and the
        field backward without the aggregation-net and axis-scale accumulators; no ray-bias weight backward;
        danbo_ray_bias_codes_bwd for fitted frame codes, danbo_view_root_bwd on root-local view directions."""
        if K.BACKWARD_IMPL != "tc":
            raise NotImplementedError("the pose-only backward runs on the tensor-core MLP kernels (BACKWARD_IMPL='tc')")
        k = ctx.keep
        rays, dev = k["rays"], k["rays"].device
        n, S_c, S_f = rays.shape[0], k["S_c"], k["S_f"]
        zeros = lambda *s: torch.zeros(*s, device=dev, dtype=torch.float32)
        d_raw0, d_raw1 = zeros(n * S_c + n, 4), zeros(n * S_f, 4)
        gl0 = gl1 = None
        if g_confd is not None:
            gl0 = torch.empty(n * S_c, K.J, device=dev, dtype=torch.float32)
            gl1 = torch.empty(n * S_f, K.J, device=dev, dtype=torch.float32)
        K.merge_composite_bwd(rays, S_c, S_f, k["raw0"], k["mask0"], k["raw1"], k["mask1"], k["z_all"], k["order"],
                              k["noise1"], k["inv_B"], g_rgb, g_acc, g_confd, d_raw0, d_raw1, gl0, gl1)
        K.composite_bwd(rays, S_c, k["raw0"], k["mask0"], k["z0"], k["noise0"], k["inv_B"], g_rgb0, g_acc0, d_raw0)
        d_vol = zeros(*ctx.vol_shape)
        grads = [None] * 7 + [d_vol[k["p0"]:], None]
        d_skts = zeros(*k["p_skts"].shape) if ctx.needs_input_grad[3] else None
        view_root = d_skts is not None and getattr(ctx.caster, "view_mode", "world") == "root_local"
        want_codes = ctx.needs_input_grad[4]
        d_ray_bias = zeros(n, 128) if (view_root or want_codes) else None
        packed_t = ctx.caster._packed_dgrad()
        cur = torch.cuda.current_stream(dev)
        side2 = None
        if K.BACKWARD_STREAMS > 1:
            # as in training: the coarse pass's field backward overlaps the fine pass's MLP backward
            side2 = getattr(ctx.caster, "_bwd_side_stream2", None)
            if side2 is None or side2.device != dev:
                side2 = ctx.caster._bwd_side_stream2 = torch.cuda.Stream(device=dev)
        alive = []
        for ip, (d_raw, S, z, mask, act, fo, sv, gl) in enumerate((
                (d_raw0, S_c, k["z0"], k["mask0"], k["act0"], k["f0"], k["sv0"], gl0),
                (d_raw1, S_f, k["z1"], k["mask1"], k["act1"], k["f1"], k["sv1"], gl1))):
            dX = K.mlp_backward_pose(P, d_raw, act, fo, sv, packed_t, d_ray_bias)
            alive.append(dX)
            if side2 is not None and ip == 0:
                side2.wait_stream(cur)
                with torch.cuda.stream(side2):
                    K.field_agg_bwd(rays, S, z, mask, act, k["p_skts"], k["p_vol"], k["skip"], k["consts"], fo, dX, gl,
                                    grads, d_skts=d_skts)
            else:
                K.field_agg_bwd(rays, S, z, mask, act, k["p_skts"], k["p_vol"], k["skip"], k["consts"], fo, dX, gl,
                                grads, d_skts=d_skts)
        d_codes = None
        if want_codes:
            # d_ray_bias is complete after the second pass's head backward (this stream): the code gradient overlaps
            # the coarse pass's field backward on side2
            d_codes = K.ray_bias_codes_bwd(k["cam_idx"], P["views_linears.0.weight"], d_ray_bias,
                                           zeros(*ctx.codes_shape))
        if side2 is not None:
            cur.wait_stream(side2)
        if view_root:
            K.view_root_bwd(rays, k["p_skts"], k["skip"], P["views_linears.0.weight"], d_ray_bias, d_skts)
        ctx.keep = None
        del alive
        return (None, None, d_vol if ctx.needs_input_grad[2] else None, d_skts, d_codes) + (None,) * len(PARAM_NAMES)


def render_block_with_grad(caster, rays, skip, pose_skts, pose_cyls, vol, cam_idx, codes, consts, packed, S_c, S_f, B,
                           raw_noise_std, perturb, nanmean_chunk, rand, stages, lindisp=False, frame_codes=None):
    """`codes` is the code table the kernels read ((rows + 1,128), last row the mean code).  `frame_codes`: the fitted
    table whose rows are codes[:-1] (training.PoseFitStep), an input of the node; when it requires a gradient the
    pose-only backward forms d frame_codes (danbo_ray_bias_codes_bwd).  A backward that trains the network as well
    is not implemented."""
    named = dict(caster.network.named_parameters())
    if not getattr(caster.network, "opt_framecode", True):
        # no frame codes (configs/surreal): the kernels keep the view layer's 411-input layout, so the node gets a
        # zero-padded view weight (F.pad is differentiable: the gradient of the 283 real columns flows back to the
        # parameter, the rest is dropped) and a zero code table that takes no gradient.  These temporaries have no
        # .grad, so the backward pass returns its gradients through autograd instead of adding them in place.
        named["views_linears.0.weight"] = torch.nn.functional.pad(named["views_linears.0.weight"], (0, 128))
        named["framecodes.codes.weight"] = torch.zeros(1, 128, device=rays.device)
    params = [named[n] for n in PARAM_NAMES]
    trains = weight_grads([p.requires_grad for p in params], N_TRAINED)  # a mixed set is refused before any launch
    if trains and frame_codes is not None and frame_codes.requires_grad:
        raise NotImplementedError("fitting frame codes while the network trains is not implemented: fit them with the "
                                  "field frozen (training.PoseFitStep(code_kwargs=...))")
    cfg = dict(rays=rays, skip=skip, pose_cyls=pose_cyls, cam_idx=cam_idx, codes=codes, consts=consts,
               packed=packed, S_c=S_c, S_f=S_f, B=B, raw_noise_std=raw_noise_std, perturb=perturb,
               nanmean_chunk=nanmean_chunk, rand=rand, stages=stages, lindisp=lindisp)
    outs = _RenderBlock.apply(caster, cfg, vol, pose_skts, frame_codes, *params)
    return dict(zip(OUT_KEYS, outs))


class _GraphNet(torch.autograd.Function):
    """GN1 + GN2 (pose -> bone feature lines) as four launches each way; gradients go to the ten graph-net parameters
    and, when the pose requires one (the pose layer's kernel path, `pose_layer`), one more launch gives d pose_bones."""

    @staticmethod
    def forward(ctx, net, pose_bones, *params):
        named = {n: p for n, p in zip(K.GN_GRADS, params)}
        gn = net.graph_net
        named["layers.0.adj"], named["layers.1.adj"] = gn.layers[0].adj, gn.layers[1].adj
        pose_bones = pose_bones.detach().float().contiguous()
        vol, saved = K.graph_net_fwd(pose_bones, [named[n].detach() for n in K.GN_PARAMS])
        ctx.saved_bufs, ctx.net, ctx.params, ctx.pose_bones = saved, net, params, pose_bones
        return vol

    @staticmethod
    def backward(ctx, d_vol):
        params = ctx.params
        if not weight_grads(ctx.needs_input_grad[2:]):
            # pose-only (training.PoseFitStep): the transposed products only, then d pose as below
            work = K.graph_net_bwd(ctx.saved_bufs, d_vol, None)
            d_pose = K.graph_net_bwd_pose(ctx.saved_bufs, work, ctx.pose_bones)
            ctx.saved_bufs = ctx.pose_bones = None
            return (None, d_pose) + (None,) * len(params)
        # same contract as _RenderBlock: with a pre-zeroed flat gradient bucket the kernels add straight into .grad
        in_place = bool(getattr(ctx.net, "grads_in_place", False)) and all(
            p.grad is not None and p.grad.dtype == torch.float32 and p.grad.is_contiguous() and p.grad.shape == p.shape
            for p in params)
        grads = [p.grad if in_place else torch.zeros_like(p, dtype=torch.float32) for p in params]
        work = K.graph_net_bwd(ctx.saved_bufs, d_vol, grads)
        # a pose that needs a gradient (the pose layer's kernel path): d pose_bones through layer 0's inputs
        d_pose = K.graph_net_bwd_pose(ctx.saved_bufs, work, ctx.pose_bones) if ctx.needs_input_grad[1] else None
        ctx.saved_bufs = ctx.pose_bones = None
        if in_place:
            return (None, d_pose) + (None,) * len(params)
        return (None, d_pose) + tuple(grads)


def graph_net_volumes(net, pose_bones):
    named = dict(net.graph_net.named_parameters())
    params = [named[n] for n in K.GN_GRADS]
    if torch.is_grad_enabled() and (pose_bones.requires_grad or any(p.requires_grad for p in params)):
        weight_grads([p.requires_grad for p in params])                  # a mixed set is refused before any launch
        return _GraphNet.apply(net, pose_bones, *params)
    named["layers.0.adj"], named["layers.1.adj"] = net.graph_net.layers[0].adj, net.graph_net.layers[1].adj
    return K.graph_net_fwd(pose_bones, [named[n].detach() for n in K.GN_PARAMS])[0]


class _PoseLayer(torch.autograd.Function):
    """The pose layer's forward (`pose_opt.PoseOptLayer.calculate_kinematic` for the batch's unique poses) and the
    trainer's pose regulariser (`pose_opt.kp_loss` without the temporal term) as one launch (danbo_pose_fwd); the
    backward of both as one launch (danbo_pose_bwd) that adds into the layer's parameter gradients."""

    @staticmethod
    def forward(ctx, spec, idx, *params):
        layer = dict(spec["buffers"], **{n: p.detach() for n, p in zip(spec["names"], params)})
        kps, bones, skts, stats = K.pose_fwd(layer, idx, spec["skip"], spec["G"], anchors=spec["anchors"],
                                             tol=spec["tol"], coef=spec["coef"], ext_scale=spec["ext_scale"])
        ctx.spec, ctx.layer, ctx.idx, ctx.params = spec, layer, idx, params
        mpjpc = stats[1]
        ctx.mark_non_differentiable(mpjpc)
        return kps, bones, skts, stats[0], mpjpc

    @staticmethod
    def backward(ctx, d_kps, d_bones, d_skts, d_reg, _d_mpjpc):
        spec, params = ctx.spec, ctx.params
        # with a pose optimizer over one flat, pre-zeroed gradient bucket (training.FlatAdam) the kernel adds straight
        # into the parameters' .grad views, as the render block does for the network
        in_place = spec["grads_in_place"] and all(
            p.grad is not None and p.grad.dtype == torch.float32 and p.grad.is_contiguous() and p.grad.shape == p.shape
            for p in params)
        grads = {n: (p.grad if in_place else torch.zeros_like(p, dtype=torch.float32)) for n, p in zip(spec["names"], params)}
        c = lambda t: None if t is None else t.float().contiguous()
        if d_skts is None:
            d_skts = torch.zeros(spec["G"], K.J, 4, 4, device=ctx.idx.device)
        K.pose_bwd(ctx.layer, ctx.idx, spec["skip"], spec["G"], c(d_skts), grads, d_bones=c(d_bones), d_kps=c(d_kps),
                   anchor_bones=spec["anchors"]["bones"] if d_reg is not None else None,
                   d_reg=None if d_reg is None else c(d_reg).reshape(()), tol=spec["tol"], coef=spec["coef"])
        ctx.layer = ctx.params = None
        if in_place:
            return (None, None) + (None,) * len(params)
        return (None, None) + tuple(grads[n] for n in spec["names"])


def pose_layer(layer, idx, skip, G, anchors, rest_idx=None, tol=0., coef=0., ext_scale=0.001, grads_in_place=False):
    """Poses idx[0], idx[skip], ... (G of them, idx int64 on the layer's device) of a `pose_opt.PoseOptLayer`
    (axis-angle; the multi-view split too) through the kernels.  anchors: {'kps', 'bones'} fp32 (F,24,3) on the layer's
    device; rest_idx: the layer's `rest_pose_idxs` as an int64 device tensor when it holds several rest poses.
    -> kps (G,24,3), bones (G,24,3), skts (G,24,4,4), kp_loss (differentiable scalar), MPJPC (scalar)."""
    names = [n for n, _ in layer.named_parameters()]
    buffers = {"rest_pose": layer.rest_pose.float().contiguous()}
    if layer.kp_map is not None:
        buffers["kp_map"] = layer.kp_map
    if layer.rest_pose.shape[0] > 1:
        if rest_idx is None:
            raise ValueError("pose_layer: a layer with several rest poses needs rest_idx")
        buffers["rest_idx"] = rest_idx
    spec = dict(names=names, buffers=buffers, skip=int(skip), G=int(G), anchors=anchors, tol=float(tol),
                coef=float(coef), ext_scale=float(ext_scale), grads_in_place=bool(grads_in_place))
    return _PoseLayer.apply(spec, idx, *[p for _, p in layer.named_parameters()])


class _PoseKp2d(torch.autograd.Function):
    """The 2D keypoint reprojection term (`pose_opt.kp2d_loss`) as one launch (danbo_pose_kp2d), which writes d loss /
    d kps with the loss; the backward scales it.  Under the pose layer, that gradient reaches danbo_pose_bwd as its
    d_kps (`_PoseLayer.backward`)."""

    @staticmethod
    def forward(ctx, kps, kp2d, proj, sigma, coef):
        loss, px, d_kps = K.pose_kp2d(kps.detach().contiguous(), kp2d, proj, sigma, coef)
        ctx.save_for_backward(d_kps)
        ctx.mark_non_differentiable(px)
        return loss, px

    @staticmethod
    def backward(ctx, d_loss, _d_px):
        (d_kps,) = ctx.saved_tensors
        return d_loss * d_kps, None, None, None, None


def pose_kp2d(kps, kp2d, proj, sigma, coef):
    """kps (G,24,3) fp32 (the pose layer's output), kp2d (G,24,3) detections (u, v, confidence), proj (G,3,4), both
    contiguous fp32 on kps' device.  -> (loss, kp2d_px): the differentiable scalar term and the mean pixel error."""
    return _PoseKp2d.apply(kps, kp2d, proj, float(sigma), float(coef))
