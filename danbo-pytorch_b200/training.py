"""Training step around the hot path: the trainer's losses (they stay PyTorch elementwise ops, SURVEY §8a row L*),
Adam, and the data-parallel gradient exchange.  Mirrors core/trainer.py:257-300 (train_batch), :348-422,507-553
(losses), :563-576 (optimize) for the flags the shipped DANBO configs use."""
import os

import torch
import torch.nn.functional as F

from . import parallel


def _img_loss(kind, x, y, beta=0.1):
    if kind == "L1":
        return torch.mean(torch.abs(x - y))
    if kind == "MSE":
        return torch.mean((x - y) ** 2)
    if kind == "Huber":
        return F.smooth_l1_loss(x, y, reduction="mean", beta=beta)
    raise NotImplementedError(f"loss_fn {kind}")


def compute_loss(args, preds, batch, network):
    """total loss + dict of terms: rgb (fine + coarse), soft-softmax on confd, volume-scale penalty."""
    bgs = batch.get("bgs", 1.0)
    terms = {}

    def rgb_term(rgb, acc):
        if getattr(args, "use_background", True):
            rgb = rgb + (1. - acc)[..., None] * bgs
        return _img_loss(args.loss_fn, rgb, batch["target_s"], getattr(args, "loss_beta", 0.1)) * getattr(args, "rgb_loss_coef", 1.0)

    terms["rgb_loss"] = rgb_term(preds["rgb_map"], preds["acc_map"])
    if "rgb0" in preds:
        terms["rgb_loss0"] = rgb_term(preds["rgb0"], preds["acc0"]) * getattr(args, "coarse_weight", 1.0)
    if "confd" in preds and getattr(args, "agg_type", None) == "sigmoid":
        labels = ((preds["T_i"] * preds["alpha"]) > 0).float()
        valid = 1 - preds["part_invalid"]
        p = network.sigmoid(preds["confd"], preds["part_invalid"], mask_invalid=False, clamp=False)
        terms["soft_softmax_loss"] = args.soft_softmax_loss_coef * (labels - (p * valid).sum(-1)).pow(2.).mean()
    if getattr(args, "opt_vol_scale", False) and hasattr(network, "graph_net"):
        gn = network.graph_net
        scale = gn.axis_scale.abs().clamp(min=gn.init_scale.to(gn.axis_scale.device) * 0.05)
        # product written out: torch.prod's backward inspects the input for zeros on the host (a sync, illegal in capture)
        terms["vol_scale_loss"] = (scale[:, 0] * scale[:, 1] * scale[:, 2]).sum() * args.vol_scale_penalty
    return sum(terms.values()), terms


def fused_loss_supported(args, preds):
    return args.loss_fn in ("L1", "MSE") and preds["rgb_map"].is_cuda


def fused_loss_backward(args, preds, batch, network, extra_loss=None):
    """compute_loss + backward as ONE kernel launch (danbo_train_loss) followed by the path's own backward: the loss terms
    and d loss / d (rgb_map, acc_map, rgb0, acc0, confd) come out of the same pass, the volume-scale gradient is added to
    axis_scale.grad directly, and autograd is entered at the render block's outputs.  `extra_loss` (a scalar with its own
    autograd graph, e.g. the pose regulariser) is back-propagated in the same sweep.  -> (total loss, dict of terms)."""
    from . import kernels as K
    soft = args.soft_softmax_loss_coef if ("confd" in preds and getattr(args, "agg_type", None) == "sigmoid") else None
    gn = getattr(network, "graph_net", None)                # the A-NeRF field has no graph net / bone volumes
    vol = gn is not None and bool(getattr(args, "opt_vol_scale", False)) and gn.axis_scale.requires_grad
    if vol and gn.axis_scale.grad is None:
        gn.axis_scale.grad = torch.zeros_like(gn.axis_scale)
    terms, g = K.train_loss(preds, batch["target_s"], batch.get("bgs", 1.0), args.loss_fn, getattr(args, "rgb_loss_coef", 1.0),
                            getattr(args, "coarse_weight", 1.0), soft_coef=soft,
                            axis_scale=gn.axis_scale if vol else None, init_scale=gn.init_scale if vol else None,
                            vol_coef=getattr(args, "vol_scale_penalty", 0.) if vol else 0.,
                            g_axis_scale=gn.axis_scale.grad if vol else None,
                            use_background=getattr(args, "use_background", True))
    keys = [k for k in ("rgb_map", "acc_map", "rgb0", "acc0", "confd") if k in g and preds[k].requires_grad]
    roots, seeds = [preds[k] for k in keys], [g[k] for k in keys]
    if extra_loss is not None:
        roots, seeds = roots + [extra_loss], seeds + [torch.ones_like(extra_loss)]
    torch.autograd.backward(roots, seeds)
    names = ("rgb_loss", "rgb_loss0", "soft_softmax_loss", "vol_scale_loss")
    total = terms.sum().float()
    if extra_loss is not None:
        total = total + extra_loss.detach().float()
    return total, {n: terms[i] for i, n in enumerate(names)}


def adam_state_to_dict(params, exp_avg, exp_avg_sq, step, group):
    """Flat moment arenas -> a state dict in torch.optim.Adam's own format (so checkpoints written here resume under the
    reference's `torch.optim.Adam`, core/raycasters.py:71-78,99-101, and the other way round)."""
    state, off = {}, 0
    for i, p in enumerate(params):
        n = p.numel()
        state[i] = {"step": torch.tensor(float(step)), "exp_avg": exp_avg[off:off + n].view_as(p).clone(),
                    "exp_avg_sq": exp_avg_sq[off:off + n].view_as(p).clone()}
        off += n
    pg = {"lr": group["lr"], "betas": tuple(group["betas"]), "eps": group["eps"], "weight_decay": 0, "amsgrad": False,
          "maximize": False, "foreach": None, "capturable": False, "differentiable": False, "fused": None,
          "params": list(range(len(params)))}
    return {"state": state, "param_groups": [pg]}


def adam_state_from_dict(sd, params, exp_avg, exp_avg_sq):
    """Inverse of adam_state_to_dict for a torch.optim.Adam state dict over the same parameters (one group, any
    steps).  Fills the flat arenas in place -> (step, lr).  Parameters without state (never stepped) get zeros."""
    ids = [i for g in sd["param_groups"] for i in g["params"]]
    if len(ids) != len(params):
        raise ValueError(f"optimizer state holds {len(ids)} parameters, the model has {len(params)}")
    off, step = 0, 0.0
    for i, p in zip(ids, params):
        n = p.numel()
        st = sd["state"].get(i)
        if st is None:
            exp_avg[off:off + n].zero_()
            exp_avg_sq[off:off + n].zero_()
        else:
            if tuple(st["exp_avg"].shape) != tuple(p.shape):
                raise ValueError(f"optimizer state {i}: shape {tuple(st['exp_avg'].shape)} vs parameter {tuple(p.shape)}")
            exp_avg[off:off + n].copy_(st["exp_avg"].reshape(-1))
            exp_avg_sq[off:off + n].copy_(st["exp_avg_sq"].reshape(-1))
            step = max(step, float(st["step"]))
        off += n
    return step, float(sd["param_groups"][0]["lr"])


def save_checkpoint(path, global_step, caster, optimizer, popt_kwargs=None, pose_optimizer=None):
    """Trainer.save_nerf (core/trainer.py:597-618): the same keys, so `create_raycaster` here or in the reference resumes
    from the file."""
    popt_sd = poptim_sd = anchors = None
    if popt_kwargs is not None and popt_kwargs.get("popt_layer") is not None:
        popt_sd = popt_kwargs["popt_layer"].state_dict()
        poptim_sd = pose_optimizer.state_dict() if pose_optimizer is not None else None
        anchors = popt_kwargs.get("popt_anchors")
    torch.save({"global_step": global_step,
                "optimizer_state_dict": optimizer.state_dict() if optimizer is not None else None,
                "poseopt_layer_state_dict": popt_sd, "pose_optimizer_state_dict": poptim_sd, "poseopt_anchors": anchors,
                **caster.state_dict()}, path)


class FlatAdam(torch.optim.Optimizer):
    """torch.optim.Adam (lr, betas, eps; no weight decay / amsgrad) as ONE kernel launch: parameters, gradients and both
    moments live in flat fp32 arenas and every nn.Parameter is a view of the parameter arena.  `step` and `lr` are device
    scalars, so the update can sit inside a captured CUDA graph (set the rate with `set_lr`)."""

    def __init__(self, params, bucket, lr=5e-4, betas=(0.9, 0.999), eps=1e-8):
        params = [p for p in params if p.requires_grad]
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps))
        assert [id(p) for p in params] == [id(p) for p in bucket.params], "FlatAdam needs the GradBucket's parameter order"
        dev = params[0].device
        if dev.type != "cuda":
            raise RuntimeError("FlatAdam runs on CUDA tensors only (there is no CPU path)")
        self.bucket = bucket
        n = bucket.flat.numel()
        self.flat = torch.empty(n, device=dev, dtype=torch.float32)
        off = 0
        with torch.no_grad():
            for p in params:
                self.flat[off:off + p.numel()].copy_(p.data.reshape(-1))
                p.data = self.flat[off:off + p.numel()].view_as(p)
                off += p.numel()
        self.exp_avg = torch.zeros_like(self.flat)
        self.exp_avg_sq = torch.zeros_like(self.flat)
        self.step_dev = torch.zeros(1, device=dev, dtype=torch.float32)
        self.lr_dev = torch.full((1,), float(lr), device=dev, dtype=torch.float32)

    def set_lr(self, lr):
        self.param_groups[0]["lr"] = float(lr)
        self.lr_dev.fill_(float(lr))

    def zero_grad(self, set_to_none=True):
        """Zeroes the gradient bucket in place: the parameters' .grad must stay views of it (set_to_none is ignored)."""
        self.bucket.zero()

    def state_dict(self):
        """torch.optim.Adam's format (one host read of the step counter)."""
        return adam_state_to_dict(self.bucket.params, self.exp_avg, self.exp_avg_sq, float(self.step_dev.item()),
                                  self.param_groups[0])

    def load_state_dict(self, sd):
        step, lr = adam_state_from_dict(sd, self.bucket.params, self.exp_avg, self.exp_avg_sq)
        self.step_dev.fill_(step)
        self.set_lr(lr)

    @torch.no_grad()
    def step(self, closure=None):
        from . import kernels as K, _lib
        g = self.param_groups[0]
        self.step_dev += 1
        idx = self.flat.device.index if self.flat.device.index is not None else torch.cuda.current_device()
        _lib.check(_lib.load().danbo_adam_step(K._p(self.flat), K._p(self.bucket.flat), K._p(self.exp_avg),
                                               K._p(self.exp_avg_sq), self.flat.numel(), K._p(self.lr_dev),
                                               float(g["betas"][0]), float(g["betas"][1]), float(g["eps"]),
                                               K._p(self.step_dev), K.num_sms(idx), K._stream()), "danbo_adam_step")
        K._count(1)
        if not torch.cuda.is_current_stream_capturing():
            # the kernel wrote through raw pointers: bump the tensors' versions so that version-keyed caches (the packed
            # bf16 weights of an eval caster) see the update; a captured replay is covered by TrainStep._after_step
            for p in self.bucket.params:
                torch.autograd.graph.increment_version(p)


def pose_batch_poses(batch):
    """(G, skip) of an --opt_pose batch: the poses are kp_idx[::skip], one per image of an image-major batch of
    N_uniques equal runs (what the data feed builds).  A batch that does not divide so is refused: finding its poses
    would need torch.unique, a host synchronisation, which a captured step cannot hold."""
    n, G = int(batch["kp_idx"].shape[0]), int(batch["N_uniques"])
    if G <= 0 or n % G:
        raise NotImplementedError(f"a captured --opt_pose step needs N_uniques ({G}) to divide the batch ({n} rays): "
                                  "other batches need torch.unique, a host synchronisation")
    return G, n // G


KP2D_KEYS = ("kp2d", "kp2d_proj")


def kp2d_batch(args, batch, pose_layer=True):
    """The 2D keypoint term's inputs of a batch: (kp2d (G,24,3) detections (u, v, confidence), kp2d_proj (G,3,4)),
    G = N_uniques, when the batch carries both and args.kp2d_coef > 0; None when the term is off.  A batch with one of
    the two keys, with other shapes, or with the term on and no pose layer raises ValueError (host-side checks only:
    nothing has run on the device yet)."""
    has = [k in batch for k in KP2D_KEYS]
    if not any(has):
        return None
    if not all(has):
        raise ValueError(f"the 2D keypoint term needs both batch['kp2d'] and batch['kp2d_proj'] (got only "
                         f"{KP2D_KEYS[has.index(True)]!r})")
    G = int(batch["N_uniques"])
    kp2d, proj = batch["kp2d"], batch["kp2d_proj"]
    if tuple(kp2d.shape) != (G, 24, 3) or tuple(proj.shape) != (G, 3, 4):
        raise ValueError(f"batch['kp2d'] must be (N_uniques, 24, 3) = ({G}, 24, 3) and batch['kp2d_proj'] ({G}, 3, 4); "
                         f"got {tuple(kp2d.shape)} and {tuple(proj.shape)}")
    if G <= 0 or int(batch["kp_idx"].shape[0]) % G:
        raise ValueError(f"the 2D keypoint term needs an image-major batch of N_uniques ({G}) equal runs")
    if not float(getattr(args, "kp2d_coef", 0.)) > 0:
        return None
    if not pose_layer:
        raise ValueError("the 2D keypoint term (kp2d_coef > 0) needs a pose layer (popt_kwargs of pose_opt.create_popt)")
    if not float(getattr(args, "kp2d_sigma", 100.)) > 0:
        raise ValueError("kp2d_sigma must be positive")
    return kp2d, proj


def _kp2d_term(args, kps, kp2d, kernels):
    """(loss, kp2d_px) of the 2D keypoint term on the pose layer's (G,24,3) kps: the kernel (autograd.pose_kp2d) or the
    PyTorch ops (pose_opt.kp2d_loss)."""
    from . import autograd, pose_opt
    det, proj = (t.to(device=kps.device, dtype=torch.float32).contiguous() for t in kp2d)
    sigma, coef = float(getattr(args, "kp2d_sigma", 100.)), float(args.kp2d_coef)
    if kernels:
        return autograd.pose_kp2d(kps, det, proj, sigma, coef)
    return pose_opt.kp2d_loss(kps, det, proj, sigma, coef)


def _refuse_pose_graph(args, caster, world_size, pose_optimizer, layer,
                       what="graph capture of a training step with a pose layer"):
    """What a captured iteration with a pose layer (and PoseFitStep, which runs the same kernels) does not cover: raise,
    naming the reason, before any device work."""
    why = None
    if getattr(caster.network, "graph_net", None) is None:
        why = "the A-NeRF field (the pose kernels serve the DANBO field's graph net and bone transforms)"
    elif getattr(caster, "network_fine", caster.network) is not caster.network:
        why = "a separate fine network"
    elif world_size > 1:
        why = "world_size > 1 (the pose gradients' all-reduce is not part of the captured step)"
    elif layer.use_rot6d or getattr(args, "opt_rot6d", False):
        why = "opt_rot6d (the pose kernels take axis-angle parameters)"
    elif getattr(args, "use_temp_loss", False):
        why = "use_temp_loss (the temporal pose term is not part of the pose kernels)"
    elif layer.use_cache or getattr(args, "opt_pose_cache", False):
        why = "opt_pose_cache (the cache is refreshed on the host after every pose step)"
    elif not isinstance(pose_optimizer, FlatAdam):
        why = ("a pose optimizer that is not a training.FlatAdam (pass pose_opt.create_popt(..., flat=True)): a captured "
               "backward writes into fixed gradient storage, which zero_grad(set_to_none=True) would detach")
    if why is not None:
        raise NotImplementedError(f"{what} is not implemented for {why}")


class TrainStep:
    """forward -> losses -> backward -> (all-reduce of one flat fp32 gradient bucket) -> Adam."""

    def __init__(self, caster, args, optimizer=None, world_size=1, graph=False, fused_loss=True, popt_kwargs=None,
                 pose_optimizer=None):
        """`popt_kwargs` / `pose_optimizer`: what `pose_opt.create_popt` returns (--opt_pose, core/trainer.py:314-341):
        the batch's poses then come from the pose layer (indexed by `batch['kp_idx']`), the pose regulariser
        (`pose_opt.kp_loss`) joins the loss and the pose optimiser steps with the network's.  A batch with `kp2d` and
        `kp2d_proj` adds the 2D keypoint term when args.kp2d_coef > 0 (`kp2d_batch`): danbo_pose_kp2d in a captured
        step, `pose_opt.kp2d_loss` in an eager one; `last_stats["kp2d_px"]` is its mean pixel error."""
        self.caster, self.args, self.world = caster, args, world_size
        # flags the reference trainer honours and this step does not implement: raise, never ignore (no shipped config
        # sets any of them)
        for flag, ok in (("opt_pose_step", (None, 1)), ("opt_pose_stop", (None, False, 0)), ("weight_decay", (None, 0, 0.0)),
                         ("reg_fn", (None, "", "None")), ("use_lpips_loss", (None, False))):
            if getattr(args, flag, None) not in ok:
                raise NotImplementedError(f"{flag}={getattr(args, flag)!r} is not implemented by danbo_b200.TrainStep")
        self.popt = popt_kwargs if (popt_kwargs and popt_kwargs.get("popt_layer") is not None) else None
        self.pose_optimizer = pose_optimizer
        self.last_stats = {}
        self.n_steps = 0                        # optimizer steps taken (the `step` of Adam's state; restored by resume())
        self.lrate = float(args.lrate)
        # a captured iteration runs the pose layer, its regulariser and their backward as kernels (autograd.pose_layer);
        # eager steps keep the PyTorch ops of pose_opt
        self._pose_kernels = self.popt is not None and graph
        if self.popt is not None:
            layer = self.popt["popt_layer"]
            if graph:
                _refuse_pose_graph(args, caster, world_size, pose_optimizer, layer)
            dev = next(caster.network.parameters()).device
            layer.to(dev)
            # anchors on the layer's device once: indexing them by the batch's kp_idx then needs no host round trip
            self.popt["popt_anchors"] = {k: (v.to(dev) if torch.is_tensor(v) else v)
                                         for k, v in self.popt["popt_anchors"].items()}
            if self._pose_kernels:
                a = self.popt["popt_anchors"]
                self._pose_anchors = {k: a[k].float().contiguous() for k in ("kps", "bones")}
                self._rest_idx = None
                if layer.rest_pose.shape[0] > 1:
                    self._rest_idx = torch.as_tensor(layer.rest_pose_idxs, device=dev).long()
        self.fused_loss = fused_loss           # False: the trainer's losses as PyTorch ops + autograd (compute_loss)
        # create_raycaster's grad_vars order (raycasters.py:188): the network, then a separate fine network.  The bucket,
        # the optimizer state and so the checkpoints index the reference's Adam over grad_vars.
        nets = [caster.network]
        fine = getattr(caster, "network_fine", caster.network)
        if fine is not caster.network:
            if graph:
                raise NotImplementedError("graph capture of a training step with a separate fine network is not implemented")
            nets.append(fine)
        params = [p for net in nets for p in net.parameters() if p.requires_grad]
        self.bucket = parallel.GradBucket(params)
        caster.grads_in_place = True            # backward kernels add into the bucket's views (see autograd._RenderBlock)
        caster.network.grads_in_place = True    # ... and so does the graph net's backward (autograd._GraphNet)
        cuda = params[0].is_cuda
        if optimizer is None:
            # default: the single-launch Adam over flat arenas; pass a torch optimizer to keep the reference's
            optimizer = FlatAdam(params, self.bucket, lr=args.lrate, betas=(0.9, 0.999)) if cuda else \
                torch.optim.Adam(params, lr=args.lrate, betas=(0.9, 0.999))
        self.optimizer = optimizer
        self._graphed = None
        self._graph_whole = False
        if graph:
            from .graphs import GraphedFn
            flat = isinstance(optimizer, FlatAdam)
            # The whole iteration - forward, losses, backward, the NCCL all-reduce of the gradient bucket and the
            # single-launch Adam - is ONE captured graph (NCCL collectives are capturable; DANBO_GRAPH_ALLREDUCE=0 keeps
            # the all-reduce and Adam as ordinary stream work after the replay).  A torch optimizer cannot be captured,
            # so it always steps outside.  The weight pack is part of the captured forward (RayCaster._packed_mlp), so a
            # replay always evaluates the weights the previous replay's Adam wrote.
            self._graph_whole = flat and (world_size == 1 or os.environ.get("DANBO_GRAPH_ALLREDUCE", "1") == "1")

            def run(**b):
                loss, preds = self._step(b) if self._graph_whole else self._fwd_bwd(b)
                out = {"loss": loss, "rgb_map": preds["rgb_map"], "acc_map": preds["acc_map"]}
                if self.popt is not None:
                    out.update(self.last_stats)
                return out
            # building the graph must not train: parameters, moments and the step counters (the network's and the
            # pose layer's) are restored after capture
            state = [optimizer.flat, optimizer.exp_avg, optimizer.exp_avg_sq, optimizer.step_dev] if flat else []
            if self.popt is not None:
                po = pose_optimizer
                state += [po.flat, po.exp_avg, po.exp_avg_sq, po.step_dev]
            self._graphed = GraphedFn(run, params[0].device, warmup=3, state=state if self._graph_whole else [],
                                      capture_error_mode="thread_local" if world_size > 1 else "global")

    def __call__(self, batch):
        kp2d = kp2d_batch(self.args, batch, self.popt is not None)     # refused before any device work
        if kp2d is None and any(k in batch for k in KP2D_KEYS):
            batch = {k: v for k, v in batch.items() if k not in KP2D_KEYS}     # the term is off: nothing of it runs
        if self._graphed is not None:
            if self.popt is not None:
                pose_batch_poses(batch)          # refused before any device work
                # the poses come from the layer: the feed's tables would only be copied into static buffers
                batch = {k: v for k, v in batch.items() if k not in ("kp_batch", "skts", "bones")}
            out = self._graphed(**batch)
            if self.popt is not None:
                self.last_stats = {k: out[k] for k in ("MPJPC", "kp2d_px") if k in out}
            if not self._graph_whole:
                if self.world > 1:
                    self.bucket.allreduce(average=True)
                self._optimizer_step()
            self._after_step()
            return out["loss"], out
        out = self._step(batch)
        self._after_step()
        return out

    def _step(self, batch):
        loss, preds = self._fwd_bwd(batch)
        if self.world > 1:
            self.bucket.allreduce(average=True)
        self._optimizer_step()
        return loss, preds

    def save(self, path, global_step):
        """Checkpoint in the reference's format (Trainer.save_nerf, core/trainer.py:597-618)."""
        save_checkpoint(path, global_step, self.caster, self.optimizer, self.popt, self.pose_optimizer)

    def resume(self, ckpt):
        """Optimizer (and pose layer) state of a loaded checkpoint dict; the network weights are loaded by
        `create_raycaster` / `caster.load_state_dict`.  -> global_step."""
        if ckpt.get("optimizer_state_dict") is not None:
            self.optimizer.load_state_dict(ckpt["optimizer_state_dict"])
        if self.popt is not None and ckpt.get("poseopt_layer_state_dict") is not None:
            self.popt["popt_layer"].load_state_dict(ckpt["poseopt_layer_state_dict"])
            if self.pose_optimizer is not None and ckpt.get("pose_optimizer_state_dict") is not None:
                self.pose_optimizer.load_state_dict(ckpt["pose_optimizer_state_dict"])
        self.caster._packed_key = None
        sd = ckpt.get("optimizer_state_dict")
        if sd is not None and sd.get("state"):
            self.n_steps = int(max(float(st["step"]) for st in sd["state"].values()))
            self.lrate = None                   # force the rate of the resumed step count at the next iteration
        return int(ckpt.get("global_step", 0))

    def decayed_lrate(self):
        """decay_optimizer_lrate (core/trainer.py:189-200): lrate * rate ** ((steps // decay_unit) / lrate_decay)."""
        a = self.args
        decay, unit = getattr(a, "lrate_decay", None), int(getattr(a, "decay_unit", 1000))
        if not decay:
            return float(a.lrate)
        return float(a.lrate) * float(getattr(a, "lrate_decay_rate", 0.1)) ** ((self.n_steps // unit) / decay)

    def _after_step(self):
        """Steps 4-5 of train_batch (core/trainer.py:286-294): learning-rate decay and the encoders' schedules."""
        self.n_steps += 1
        # a replayed graph runs no Python: invalidate the eager-eval weight pack here, once per iteration, as well
        self.caster._packed_key = None
        new = self.decayed_lrate()
        if new != self.lrate:                   # a staircase in units of decay_unit steps: rarely changes
            self.lrate = new
            if hasattr(self.optimizer, "set_lr"):
                self.optimizer.set_lr(new)      # device scalar: also seen by a captured graph
            else:
                for g in self.optimizer.param_groups:
                    g["lr"] = new
        # the pose optimiser's rate stays constant: the reference defines update_pose_opt_params (core/pose_opt.py:454-463)
        # but its trainer never calls it
        update = getattr(self.caster, "update_embed_fns", None)
        if update is not None and not getattr(self.args, "finetune", False):
            update(self.n_steps, self.args)

    def _optimizer_step(self):
        self.optimizer.step()
        if self.popt is not None and self.pose_optimizer is not None:
            if self.world > 1:                  # every rank saw other frames: average like the network's gradients
                import torch.distributed as dist
                for p in self.popt["popt_layer"].parameters():
                    if p.grad is not None:
                        dist.all_reduce(p.grad)
                        p.grad /= self.world
            self.pose_optimizer.step()
            if self.popt["popt_layer"].use_cache:                # pose_opt.py:577-578
                self.popt["popt_layer"].update_cache()
        self.caster._packed_key = None          # weights changed (a raw-pointer update does not bump tensor versions)

    def _fwd_bwd(self, batch):
        a = self.args
        self.caster.train()
        self.bucket.zero()
        extra = None
        kp2d = kp2d_batch(a, batch, self.popt is not None)
        if self._pose_kernels:
            from .autograd import pose_layer
            G, skip = pose_batch_poses(batch)
            n = G * skip
            self.pose_optimizer.zero_grad()
            kps, bones, skts, extra, mpjpc = pose_layer(
                self.popt["popt_layer"], batch["kp_idx"].long(), skip, G, self._pose_anchors, rest_idx=self._rest_idx,
                tol=getattr(a, "opt_pose_tol", 0.), coef=getattr(a, "opt_pose_coef", 0.),
                ext_scale=getattr(a, "ext_scale", 0.001), grads_in_place=True)
            # per-ray rows as stride-0 expands, as PoseOptLayer.calculate_kinematic returns them
            ex = lambda t: t[:, None].expand(G, skip, *t.shape[1:]).reshape(n, *t.shape[1:])
            batch = dict(batch, kp_batch=ex(kps), skts=ex(skts), bones=ex(bones))
            self.last_stats = {"MPJPC": mpjpc}
            if kp2d is not None:
                l2d, self.last_stats["kp2d_px"] = _kp2d_term(a, kps, kp2d, kernels=True)
                extra = extra + l2d
        elif self.popt is not None:
            from . import pose_opt
            layer = self.popt["popt_layer"]
            if self.pose_optimizer is not None:
                self.pose_optimizer.zero_grad(set_to_none=True)
            # not the layer's cache: the poses must carry their graph (the cache is refreshed after the pose step)
            kps, bones, skts, _, rots = layer.calculate_kinematic(batch["kp_idx"], N_uniques=batch["N_uniques"])
            batch = dict(batch, kp_batch=kps, skts=skts, bones=bones)
            losses, self.last_stats = pose_opt.kp_loss(a, self.popt["popt_anchors"], batch["kp_idx"],
                                                       {"kp_batch": kps, "bones": bones, "rots": rots}, popt_layer=layer,
                                                       temp_val=batch.get("temp_val"))
            extra = sum(losses.values())
            if kp2d is not None:
                skip = int(batch["kp_idx"].shape[0]) // int(batch["N_uniques"])      # one row per pose of the batch
                l2d, self.last_stats["kp2d_px"] = _kp2d_term(a, kps[::skip], kp2d, kernels=False)
                extra = extra + l2d
        net = self.caster.network
        net.pose_kernels = self._pose_kernels        # the graph net's kernels then also return d pose
        try:
            preds = self.caster(batch["ray_batch"], N_samples=a.N_samples, kp_batch=batch["kp_batch"], skts=batch["skts"],
                                cyls=batch["cyls"], bones=batch["bones"], cams=batch["cams"], N_uniques=batch["N_uniques"],
                                perturb=a.perturb, N_importance=a.N_importance, raw_noise_std=a.raw_noise_std)
        finally:
            net.pose_kernels = False
        # every rank holds 1/world of the batch: mean-reduced data terms are averaged by the all-reduce; the parameter-only
        # volume penalty is identical on every rank, so averaging leaves it unchanged
        if self.fused_loss and fused_loss_supported(a, preds):
            loss, terms = fused_loss_backward(a, preds, batch, self.caster.network, extra_loss=extra)
            return loss, preds
        loss, terms = compute_loss(a, preds, batch, self.caster.network)
        if extra is not None:
            loss = loss + extra
        loss.backward()
        return loss.detach(), preds


class PoseFitStep:
    """Fits the SMPL poses of frames to their images with the field frozen: forward -> losses -> pose-only backward ->
    pose backward -> the pose optimizer's Adam.  Call shape of TrainStep: `loss, preds = step(batch)`,
    `step.last_stats["MPJPC"]`, `step.save(path, global_step)`, `step.resume(ckpt)`.

    Only the pose layer's parameters change, through `pose_optimizer` (a FlatAdam, `pose_opt.create_popt(..., flat=True)`).
    The network's parameters, their .grad, `caster.state_dict()` and any network optimizer are left as they are: the
    network's parameters are passed to the render with requires_grad off for the duration of a call, so its backward
    nodes take the pose-only path (autograd.weight_grads) and form no weight gradient.  No learning-rate decay and no
    `update_embed_fns` schedule is applied to the network.

    Loss: the trainer's image terms as TrainStep computes them (rgb_loss, rgb_loss0, soft_softmax_loss) plus the pose
    regulariser (kp_loss, danbo_pose_fwd), and the 2D keypoint reprojection term when the batch carries `kp2d` and
    `kp2d_proj` and args.kp2d_coef > 0 (`kp2d_batch`; danbo_pose_kp2d; `last_stats["kp2d_px"]`).  vol_scale_loss
    depends on the network's axis_scale only, has no pose gradient and is left out.  Frames the field was not trained
    on have no frame code: give them cams < 0 in the batch and they are rendered with the mean code (danbo_ray_bias's
    last code row).

    graph=True captures the whole iteration as one CUDA graph (graphs.GraphedFn); capture applies no pose step (the pose
    arena, its moments and its step counter are restored).  The MLP weight packs are keyed on the weights and checked
    before each replay, outside the graph, so a `caster.load_state_dict` between steps is seen.  graph=False runs the
    same kernels eagerly.  Refused (NotImplementedError, before any device work): the A-NeRF field, a separate fine
    network, world_size > 1, opt_rot6d, use_temp_loss, opt_pose_cache, a pose optimizer that is not a FlatAdam, and a
    batch whose N_uniques does not divide it."""

    def __init__(self, caster, args, popt_kwargs, pose_optimizer, graph=False, world_size=1):
        if not popt_kwargs or popt_kwargs.get("popt_layer") is None:
            raise ValueError("PoseFitStep needs the pose layer of pose_opt.create_popt (popt_kwargs['popt_layer'])")
        layer = popt_kwargs["popt_layer"]
        _refuse_pose_graph(args, caster, world_size, pose_optimizer, layer, what="pose fitting (PoseFitStep)")
        self.caster, self.args, self.popt, self.pose_optimizer = caster, args, popt_kwargs, pose_optimizer
        self.last_stats = {}
        dev = next(caster.network.parameters()).device
        layer.to(dev)
        self.popt["popt_anchors"] = {k: (v.to(dev) if torch.is_tensor(v) else v)
                                     for k, v in self.popt["popt_anchors"].items()}
        a = self.popt["popt_anchors"]
        self._pose_anchors = {k: a[k].float().contiguous() for k in ("kps", "bones")}
        self._rest_idx = None
        if layer.rest_pose.shape[0] > 1:
            self._rest_idx = torch.as_tensor(layer.rest_pose_idxs, device=dev).long()
        self._graphed = None
        if graph:
            from .graphs import GraphedFn

            def run(_param_ptrs=None, **b):
                loss, preds = self._step(b)
                return dict(self.last_stats, loss=loss, rgb_map=preds["rgb_map"], acc_map=preds["acc_map"])
            po = pose_optimizer
            self._graphed = GraphedFn(run, dev, warmup=3, state=[po.flat, po.exp_avg, po.exp_avg_sq, po.step_dev])

    def _frozen(self):
        """Context: the network's parameters with requires_grad off (restored on exit)."""
        import contextlib
        nets = [self.caster.network]

        @contextlib.contextmanager
        def ctx():
            saved = [(p, p.requires_grad) for net in nets for p in net.parameters()]
            try:
                for p, _ in saved:
                    p.requires_grad_(False)
                yield
            finally:
                for p, r in saved:
                    p.requires_grad_(r)
        return ctx()

    def __call__(self, batch):
        pose_batch_poses(batch)                  # refused before any device work
        kp2d = kp2d_batch(self.args, batch)
        if kp2d is None and any(k in batch for k in KP2D_KEYS):
            batch = {k: v for k, v in batch.items() if k not in KP2D_KEYS}     # the term is off: nothing of it runs
        if self._graphed is None:
            return self._step(batch)
        # the poses come from the layer: the feed's tables would only be copied into static buffers
        batch = {k: v for k, v in batch.items() if k not in ("kp_batch", "skts", "bones")}
        self.caster.train()
        with self._frozen():
            # eager, outside the graph: repack the MLP weights (both packs, into the buffers the graph reads) iff they
            # changed since the last pack
            self.caster._packed_dgrad()
        # the graph reads the parameters through the raw pointers they had at capture: re-pointed storage recaptures
        ptrs = hash(tuple(p.data_ptr() for p in self.caster.network.parameters()))
        out = self._graphed(_param_ptrs=ptrs, **batch)
        self.last_stats = {k: out[k] for k in ("MPJPC", "kp2d_px") if k in out}
        return out["loss"], out

    def _step(self, batch):
        from .autograd import pose_layer
        a = self.args
        caster, net = self.caster, self.caster.network
        caster.train()
        G, skip = pose_batch_poses(batch)
        n = G * skip
        self.pose_optimizer.zero_grad()
        kps, bones, skts, reg, mpjpc = pose_layer(
            self.popt["popt_layer"], batch["kp_idx"].long(), skip, G, self._pose_anchors, rest_idx=self._rest_idx,
            tol=getattr(a, "opt_pose_tol", 0.), coef=getattr(a, "opt_pose_coef", 0.),
            ext_scale=getattr(a, "ext_scale", 0.001), grads_in_place=True)
        ex = lambda t: t[:, None].expand(G, skip, *t.shape[1:]).reshape(n, *t.shape[1:])
        self.last_stats = {"MPJPC": mpjpc}
        kp2d = kp2d_batch(a, batch)
        if kp2d is not None:
            l2d, self.last_stats["kp2d_px"] = _kp2d_term(a, kps, kp2d, kernels=True)
            reg = reg + l2d
        batch = dict(batch, kp_batch=ex(kps), skts=ex(skts), bones=ex(bones))
        net.pose_kernels = True                  # the graph net's kernels return d pose
        try:
            with self._frozen():
                preds = caster(batch["ray_batch"], N_samples=a.N_samples, kp_batch=batch["kp_batch"],
                               skts=batch["skts"], cyls=batch["cyls"], bones=batch["bones"], cams=batch["cams"],
                               N_uniques=batch["N_uniques"], perturb=a.perturb, N_importance=a.N_importance,
                               raw_noise_std=a.raw_noise_std)
                if fused_loss_supported(a, preds):
                    # axis_scale needs no gradient here, so the fused loss forms no volume-scale term
                    loss, _ = fused_loss_backward(a, preds, batch, net, extra_loss=reg)
                else:
                    _, terms = compute_loss(a, preds, batch, net)
                    terms.pop("vol_scale_loss", None)
                    total = sum(terms.values()) + reg
                    total.backward()
                    loss = total.detach()
        finally:
            net.pose_kernels = False
        self.pose_optimizer.step()
        return loss, preds

    def save(self, path, global_step):
        """Checkpoint in the reference's format with the (unchanged) network, the pose layer and the pose optimizer;
        there is no network optimizer state (optimizer_state_dict is None)."""
        save_checkpoint(path, global_step, self.caster, None, self.popt, self.pose_optimizer)

    def resume(self, ckpt):
        """The pose layer and pose optimizer state of a loaded checkpoint dict (nothing of the network).
        -> global_step."""
        if ckpt.get("poseopt_layer_state_dict") is not None:
            self.popt["popt_layer"].load_state_dict(ckpt["poseopt_layer_state_dict"])
            if ckpt.get("pose_optimizer_state_dict") is not None:
                self.pose_optimizer.load_state_dict(ckpt["pose_optimizer_state_dict"])
        return int(ckpt.get("global_step", 0))
