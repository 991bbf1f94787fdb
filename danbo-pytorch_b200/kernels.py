"""Thin torch-side wrappers of the C ABI (include/danbo_b200.h): allocate outputs, pass raw pointers + sizes.

Every function requires CUDA tensors and enqueues on torch's current stream.  There is no CPU path."""
import ctypes
import functools
import os

import torch

from . import _lib

J = 24
TILE_M = 128
X_TILE_BYTES = 128 * 256 * 2

# bench.py sets this to {"mlp": [], "launches": 0} to count this library's kernel launches and to time the
# dominant kernel with CUDA events on the launching stream; None in normal operation.
PROFILE = None


def _count(n):
    if PROFILE is not None:
        PROFILE["launches"] += n


# True (or DANBO_NVTX=1): every stage wrapper opens an NVTX range (`ncu --nvtx --nvtx-include "field_agg/"`)
NVTX = os.environ.get("DANBO_NVTX", "") == "1"


class _Timed:
    """with _Timed("name"): ... -> CUDA-event pair appended to PROFILE["stages"] when stage timing is on; an NVTX range
    of the same name when NVTX is on."""

    def __init__(self, name):
        self.name = name

    def __enter__(self):
        self.on = PROFILE is not None and "stages" in PROFILE
        self.nvtx = NVTX
        if self.nvtx:
            torch.cuda.nvtx.range_push(self.name)
        if self.on:
            self.e0, self.e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            self.e0.record()

    def __exit__(self, *exc):
        if self.on:
            self.e1.record()
            PROFILE["stages"].append((self.name, self.e0, self.e1))
        if self.nvtx:
            torch.cuda.nvtx.range_pop()


def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("danbo_b200 kernels need CUDA tensors; there is no CPU fallback for this path")


@functools.lru_cache(maxsize=8)
def num_sms(device_index):
    return torch.cuda.get_device_properties(device_index).multi_processor_count


@functools.lru_cache(maxsize=64)
def _linspace01(S, device_index):
    # torch's CPU linspace is the oracle's definition of t; S floats, cached per device
    return torch.linspace(0., 1., steps=S).to(torch.device("cuda", device_index))


def f32c(t):
    return t.detach().to(torch.float32).contiguous()


# "mma" (default since round 2): the aggregation net on tensor cores, split-bf16 mma.sync (csrc/field_mma.cu; logits
# within 2e-5 of the fp32 kernel's, 0.85 -> 0.57 ms for the coarse field_agg call of a 512x512 image).  "ffma": the fp32
# FFMA kernel of round 1 (`DANBO_PAIR_LOGITS=ffma`, or set this before building a caster).
PAIR_LOGITS_IMPL = os.environ.get("DANBO_PAIR_LOGITS", "mma")


class FieldConsts:
    """Device pointers to the ten constant tensors the field kernels read, plus the optional MMA fragment table of the
    aggregation net (see danbo_b200.h)."""

    def __init__(self, align, axis_scale, agg, pair_logits_impl=None):
        self.tensors = [f32c(align), f32c(axis_scale), f32c(agg["w0"]), f32c(agg["adj_w"]), f32c(agg["adj"]),
                        f32c(agg["b0"]), f32c(agg["w1"]), f32c(agg["b1"]), f32c(agg["w2"]), f32c(agg["b2"])]
        _need_cuda(*self.tensors)
        impl = PAIR_LOGITS_IMPL if pair_logits_impl is None else pair_logits_impl
        if impl not in ("ffma", "mma"):
            raise ValueError(f"pair-logits implementation {impl!r}: 'ffma' or 'mma'")
        self.frags = None
        ptrs = [t.data_ptr() for t in self.tensors] + [None]
        if impl == "mma":
            lib = _lib.load()
            self.frags = torch.empty(int(lib.danbo_agg_frag_bytes()), device=self.tensors[0].device, dtype=torch.uint8)
            ptrs[10] = self.frags.data_ptr()
        self.array = (ctypes.c_void_p * 11)(*ptrs)
        if impl == "mma":
            _lib.check(lib.danbo_pack_agg_frags(self.array, _p(self.frags), _stream()), "danbo_pack_agg_frags")
            _count(1)

    @property
    def align(self):
        return self.tensors[0]

    @property
    def axis_scale(self):
        return self.tensors[1]


def nearfar(rays, pose_cyl, pose_skts, rays_per_pose, align, axis_scale, seg_len=0, use_box=False, bound=1.3,
            return_masks=False):
    """NF1 (+NF2).  rays (n,>=8) contiguous; pose_cyl (G,>=3); pose_skts (G,24,4,4).  -> near (n), far (n)."""
    _need_cuda(rays, pose_cyl, pose_skts, align, axis_scale)
    lib = _lib.load()
    n = rays.shape[0]
    near = torch.empty(n, device=rays.device, dtype=torch.float32)
    far = torch.empty_like(near)
    n_seg = 1 if seg_len <= 0 else (n + seg_len - 1) // seg_len
    acc = torch.empty(4 * max(n_seg, 1), device=rays.device, dtype=torch.float64)
    pv = vv = None
    if return_masks:
        pv = torch.zeros(n, J, device=rays.device, dtype=torch.uint8)
        vv = torch.zeros(n, J, device=rays.device, dtype=torch.uint8)
    import numpy as np
    bound_hi = float(np.float32(bound + 1e-4))        # torch compares the fp32 hits with fp32(bound_range + eps)
    with _Timed("nearfar"):
        _lib.check(lib.danbo_nearfar(_p(rays), rays.stride(0), n, _p(pose_cyl), pose_cyl.stride(0), _p(pose_skts),
                                     int(rays_per_pose), pose_skts.shape[0], _p(align), _p(axis_scale), int(seg_len),
                                     int(bool(use_box)), float(bound), bound_hi, _p(near), _p(far), _p(acc), n_seg,
                                     _p(pv), _p(vv), _stream()), "danbo_nearfar")
    _count(2)
    if return_masks:
        return near, far, pv, vv
    return near, far


class ActiveList:
    """Compacted ids of the samples at least one bone sees (+ one empty entry per ray in the coarse pass)."""

    def __init__(self, capacity, device):
        self.capacity = int(capacity)
        self.ids = torch.empty(self.capacity, device=device, dtype=torch.int32)
        self.count = torch.zeros(1, device=device, dtype=torch.int32)


def sample_mask(rays, S, pose_skts, rays_per_pose, consts, near=None, far=None, t_rand=None, z_in=None,
                append_empty=False, capacity=None, lindisp=False):
    """-> z (n,S), mask (n,S) uint32-as-int32, ActiveList."""
    _need_cuda(rays, pose_skts, near, far, t_rand, z_in)
    lib = _lib.load()
    n = rays.shape[0]
    dev = rays.device
    cap = n * S + (n if append_empty else 0) if capacity is None else int(capacity)
    active = ActiveList(max(cap, 1), dev)
    mask = torch.empty(n, S, device=dev, dtype=torch.int32)
    if z_in is None:
        z = torch.empty(n, S, device=dev, dtype=torch.float32)
        t_vals = _linspace01(S, dev.index if dev.index is not None else torch.cuda.current_device())
        z_out = z
    else:
        z = z_in.contiguous()
        t_vals, z_out = None, None
    with _Timed("sample_mask"):
        _lib.check(lib.danbo_sample_mask(_p(rays), rays.stride(0), n, S, _p(near), _p(far), _p(t_vals), _p(t_rand),
                                         _p(z if z_in is not None else None), _p(z_out), _p(pose_skts),
                                         int(rays_per_pose), pose_skts.shape[0], consts.array, _p(mask), _p(active.ids),
                                         _p(active.count), active.capacity, int(append_empty), int(bool(lindisp)),
                                         _stream()), "danbo_sample_mask")
    _count(1)
    return z, mask, active


class FieldOut:
    """What danbo_field_agg produced for one pass (kept whole in train mode: the backward reuses the pair lists)."""
    __slots__ = ("xtiles", "row_ray", "logits", "hbar", "x_rows", "work", "pair_cap", "agg_mode")

    def overflowed(self):
        """True if the call saw more visible (row, bone) pairs than its workspace held (host read: synchronises).  The
        call's rows are NaN in that case."""
        return bool(self.work[48].item())


AGG_MODES = {"sigmoid": 0, "softmax": 1}


WORST_CASE_PAIR_ROWS = 65536      # up to this many rows the pair workspace is sized for 24 visible bones per row


def field_agg(rays, S, z, mask, active, pose_skts, pose_vol, rays_per_pose, consts, want_hbar=False,
              want_xrows=False, pairs_per_row=None, agg_mode=0):
    """-> FieldOut: xtiles (uint8 tiles), row_ray (cap) int32, logits (n*S,24) [visible entries only; all 24 entries
    of every active row with agg_mode 1], hbar (cap,16) / x_rows (cap,208 bf16) when asked.
    agg_mode: AGG_MODES[agg_type] (0 sigmoid, 1 masked softmax, which evaluates every bone of an active row)."""
    _need_cuda(rays, z, mask, pose_skts, pose_vol)
    lib = _lib.load()
    n = rays.shape[0]
    dev = rays.device
    n_tiles = (active.capacity + TILE_M - 1) // TILE_M
    o = FieldOut()
    o.xtiles = torch.empty(n_tiles * X_TILE_BYTES, device=dev, dtype=torch.uint8)
    o.row_ray = torch.empty(active.capacity, device=dev, dtype=torch.int32)
    o.logits = torch.empty(n * S, J, device=dev, dtype=torch.float32)
    o.hbar = torch.empty(active.capacity, 16, device=dev, dtype=torch.float32) if want_hbar else None
    o.x_rows = torch.empty(active.capacity, 208, device=dev, dtype=torch.bfloat16) if want_xrows else None
    if pairs_per_row is None:
        # a sample can lie in all 24 bone boxes, but `capacity` of the render / training calls counts every sample of
        # the batch while only the samples inside at least one box (15 % on the 512x512 image, with 1.3 visible bones
        # each) own pairs: 6 per row of capacity is > 24 per active row as long as <= 25 % of the samples are active.
        # Small calls (density queries at points that may all sit inside the torso) get the exact worst case.  Beyond
        # that an overflow is detected on the device: work[48] is set and every row of the call becomes NaN
        # (`FieldOut.overflowed()` reads the flag; render_pts_density re-runs with the worst-case size).
        pairs_per_row = J if active.capacity <= WORST_CASE_PAIR_ROWS else 6
    if agg_mode == 1:
        pairs_per_row = J
    o.pair_cap = int(pairs_per_row * active.capacity) + 24 * 32
    o.agg_mode = int(agg_mode)
    o.work = torch.empty(64 + o.pair_cap, device=dev, dtype=torch.int32)
    idx = dev.index if dev.index is not None else torch.cuda.current_device()
    with _Timed("field_agg"):
        _lib.check(lib.danbo_field_agg(_p(rays), rays.stride(0), n, S, _p(z), _p(mask), _p(active.ids), _p(active.count),
                                       active.capacity, _p(pose_skts), _p(pose_vol), int(rays_per_pose),
                                       pose_skts.shape[0], consts.array, _p(o.xtiles), _p(o.row_ray), _p(o.logits),
                                       _p(o.hbar), _p(o.x_rows), _p(o.work), o.pair_cap, num_sms(idx), o.agg_mode,
                                       _stream()), "danbo_field_agg")
    _count(4)
    return o


class PackedMLP:
    """bf16 stage stream + fp32 heads + per-ray view slice, packed from the module's fp32 nn.Linear weights."""

    def __init__(self, device):
        lib = _lib.load()
        a, b, c = ctypes.c_longlong(), ctypes.c_longlong(), ctypes.c_longlong()
        lib.danbo_mlp_workspace_bytes(ctypes.byref(a), ctypes.byref(b), ctypes.byref(c))
        self.wstream = torch.empty(a.value, device=device, dtype=torch.uint8)
        self.heads = torch.empty(b.value // 4, device=device, dtype=torch.float32)
        self.wv_ray = torch.empty(c.value // 4, device=device, dtype=torch.float32)
        self.key = None
        self.has_empty = False

    def pack(self, P, want_empty=True):
        """P: mapping with the reference's names (pts_linears.i.weight ...) -> fp32 CUDA tensors.  want_empty: also compute
        the empty-sample constants (`mlp_empty_rows` reads them; a training pack does not need them)."""
        lib = _lib.load()
        lib.danbo_mlp_set_pack_empty(int(bool(want_empty)))
        self.has_empty = bool(want_empty)
        ws = [f32c(P[f"pts_linears.{i}.weight"]) for i in range(8)]
        bs = [f32c(P[f"pts_linears.{i}.bias"]) for i in range(8)]
        others = [f32c(P[k]) for k in ("alpha_linear.weight", "alpha_linear.bias", "feature_linear.weight",
                                       "feature_linear.bias", "views_linears.0.weight", "views_linears.0.bias",
                                       "rgb_linear.weight", "rgb_linear.bias")]
        _need_cuda(*ws, *bs, *others)
        wa = (ctypes.c_void_p * 8)(*[t.data_ptr() for t in ws])
        ba = (ctypes.c_void_p * 8)(*[t.data_ptr() for t in bs])
        _lib.check(lib.danbo_pack_mlp_weights(wa, ba, *[_p(t) for t in others], _p(self.wstream), _p(self.heads),
                                              _p(self.wv_ray), _stream()), "danbo_pack_mlp_weights")
        self._keep = (ws, bs, others)          # keep sources alive until the stream has consumed them
        _count(2 if want_empty else 1)
        return self


def ray_bias(rays, cam_idx, codes_with_mean, packed):
    """-> (n,128).  codes_with_mean (n_codes+1,128): last row = mean code (used when cam_idx < 0)."""
    _need_cuda(rays, cam_idx, codes_with_mean)
    lib = _lib.load()
    n = rays.shape[0]
    out = torch.empty(n, 128, device=rays.device, dtype=torch.float32)
    table = torch.empty(codes_with_mean.shape[0], 128, device=rays.device, dtype=torch.float32)
    with _Timed("ray_bias"):
        _lib.check(lib.danbo_ray_bias(_p(rays), rays.stride(0), n, _p(cam_idx), _p(codes_with_mean),
                                      codes_with_mean.shape[0] - 1, _p(packed.wv_ray), _p(table), _p(out), _stream()),
                   "danbo_ray_bias")
    _count(2)
    return out


def mlp_empty_rows(rbias, packed, raw_tail):
    """raw_tail (n,4) <- the field's output for "a sample no bone sees" of every ray, from the constants the weight pack
    left behind the heads and the ray's view bias (danbo_mlp_empty_rows): these rows then need not go through the MLP."""
    _need_cuda(rbias, raw_tail)
    n = rbias.shape[0]
    assert raw_tail.shape[0] == n and raw_tail.is_contiguous() and raw_tail.dtype == torch.float32
    if not packed.has_empty:
        raise RuntimeError("the packed weights carry no empty-sample constants (packed by a training forward): repack")
    dev = rbias.device
    idx = dev.index if dev.index is not None else torch.cuda.current_device()
    with _Timed("ray_bias"):
        _lib.check(_lib.load().danbo_mlp_empty_rows(_p(rbias), n, _p(packed.heads), _p(raw_tail), num_sms(idx), _stream()),
                   "danbo_mlp_empty_rows")
    _count(1)


def set_mlp_cta_pair(enable):
    """Kernel variant of the fused MLP forward: CTA pairs (cta_group::2, default) or one CTA per tile.  -> previous."""
    return bool(_lib.load().danbo_mlp_set_cta_pair(int(bool(enable))))


def mlp_forward(xtiles, packed, rbias, active, row_ray, out, density_only=False, trace=None):
    """Runs the fused MLP over the active rows; row r is written to out[active.ids[r]].
    trace: optional int64 CUDA tensor of 480 entries -> clock64 timeline of CTA 0 (profiling aid)."""
    lib = _lib.load()
    if trace is not None:
        dev = xtiles.device
        idx = dev.index if dev.index is not None else torch.cuda.current_device()
        _lib.check(lib.danbo_mlp_forward_trace(_p(xtiles), _p(packed.wstream), _p(packed.heads), _p(rbias),
                                               _p(active.ids), _p(row_ray), _p(active.count), active.capacity, _p(out),
                                               out.shape[0] if not density_only else out.numel(),
                                               int(bool(density_only)), num_sms(idx), _p(trace), _stream()),
                   "danbo_mlp_forward_trace")
        _count(1)
        return out
    dev = xtiles.device
    idx = dev.index if dev.index is not None else torch.cuda.current_device()
    if PROFILE is not None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    _lib.check(lib.danbo_mlp_forward(_p(xtiles), _p(packed.wstream), _p(packed.heads), _p(rbias), _p(active.ids),
                                     _p(row_ray), _p(active.count), active.capacity, _p(out),
                                     out.shape[0] if not density_only else out.numel(), int(bool(density_only)),
                                     num_sms(idx), _stream()), "danbo_mlp_forward")
    if PROFILE is not None:
        e1.record()
        PROFILE["mlp"].append((e0, e1, active.count))
    _count(1)
    return out


def composite_resample(rays, S, S_f, raw, mask, z, noise=None, inv_B=1.0, u_rand=None, want_inds=False, smooth=True,
                       want_weights=True):
    """C1 + R1 on the coarse samples.  raw (n*S+n,4).  -> dict.  smooth: single_net importance weights (is_only);
    S_f = 0: compositing only.  want_weights=False: no "weights" entry, and the (n, S) weight row is not written."""
    _need_cuda(rays, raw, mask, z, noise, u_rand)
    lib = _lib.load()
    n = rays.shape[0]
    dev = rays.device
    f = lambda *s: torch.empty(*s, device=dev, dtype=torch.float32)
    out = {"alpha": f(n, S), "rgb_map": f(n, 3), "disp_map": f(n), "acc_map": f(n)}
    if want_weights:
        out["weights"] = f(n, S)
    u_vals = None
    if S_f > 0:
        out["z_samples"], out["z_all"] = f(n, S_f), f(n, S + S_f)
        out["order"] = torch.empty(n, S + S_f, device=dev, dtype=torch.int32)
        if want_inds:
            out["inds"] = torch.empty(n, S_f, device=dev, dtype=torch.int32)
        if u_rand is None:
            u_vals = _linspace01(S_f, dev.index if dev.index is not None else torch.cuda.current_device())
    with _Timed("composite_resample"):
        _lib.check(lib.danbo_composite_resample(_p(rays), rays.stride(0), n, S, S_f, _p(raw), _p(mask), _p(z), _p(noise),
                                                float(inv_B), _p(u_vals), _p(u_rand), _p(out.get("weights")), _p(out["alpha"]),
                                                _p(out["rgb_map"]), _p(out["disp_map"]), _p(out["acc_map"]),
                                                _p(out.get("z_samples")), _p(out.get("z_all")), _p(out.get("order")),
                                                _p(out.get("inds")), int(bool(smooth)), _stream()), "danbo_composite_resample")
    _count(1)
    return out


def merge_composite(rays, S_c, S_f, raw0, mask0, raw1, mask1, z_all, order, noise=None, inv_B=1.0, want_raw=False,
                    confd0=None, confd1=None, want_invalid=False):
    """R2 + C1 on the merged samples -> dict (rgb_map, disp_map, acc_map, alpha, weights [, raw, confd, part_invalid])."""
    lib = _lib.load()
    n = rays.shape[0]
    dev = rays.device
    St = S_c + S_f
    f = lambda *s: torch.empty(*s, device=dev, dtype=torch.float32)
    out = {"weights": f(n, St), "alpha": f(n, St), "rgb_map": f(n, 3), "disp_map": f(n), "acc_map": f(n)}
    if want_raw:
        out["raw"] = f(n, St, 4)
    if confd0 is not None:
        out["confd"] = f(n, St, J)
    if want_invalid:
        out["part_invalid"] = f(n, St, J)
    with _Timed("merge_composite"):
        _lib.check(lib.danbo_merge_composite(_p(rays), rays.stride(0), n, S_c, S_f, _p(raw0), _p(mask0), _p(raw1), _p(mask1),
                                             _p(z_all), _p(order), _p(noise), float(inv_B), _p(out["weights"]),
                                             _p(out["alpha"]), _p(out["rgb_map"]), _p(out["disp_map"]), _p(out["acc_map"]),
                                             _p(out.get("raw")), _p(confd0), _p(confd1), _p(out.get("confd")),
                                             _p(out.get("part_invalid")), _stream()), "danbo_merge_composite")
    _count(1)
    return out


def merge_composite_parts(rays, S_c, S_f, raw0, mask0, raw1, mask1, z_all, order, logits0, logits1, agg_mode,
                          noise=None, inv_B=1.0, want_raw=False):
    """merge_composite (eval mode) plus part_map (n,24) = sum_m w_m p_m, p_m the aggregation weights of merged sample m
    from its pass's field_agg logits (`logits0` (n*S_c,24), `logits1` (n*S_f,24)) and visibility mask; the other
    outputs are bit-identical to merge_composite's -> dict (rgb_map, disp_map, acc_map, alpha, weights, part_map [, raw])."""
    _need_cuda(rays, raw0, mask0, raw1, mask1, z_all, order, logits0, logits1, noise)
    n = rays.shape[0]
    if tuple(logits0.shape) != (n * S_c, J) or tuple(logits1.shape) != (n * S_f, J):
        raise ValueError(f"logits (n*S_c,24) and (n*S_f,24) expected, got {tuple(logits0.shape)}, {tuple(logits1.shape)}")
    if agg_mode not in (0, 1):
        raise ValueError(f"agg_mode {agg_mode!r}: 0 (sigmoid) or 1 (softmax)")
    lib = _lib.load()
    dev = rays.device
    St = S_c + S_f
    f = lambda *s: torch.empty(*s, device=dev, dtype=torch.float32)
    out = {"weights": f(n, St), "alpha": f(n, St), "rgb_map": f(n, 3), "disp_map": f(n), "acc_map": f(n),
           "part_map": f(n, J)}
    if want_raw:
        out["raw"] = f(n, St, 4)
    with _Timed("merge_composite"):
        _lib.check(lib.danbo_merge_composite_parts(_p(rays), rays.stride(0), n, S_c, S_f, _p(raw0), _p(mask0), _p(raw1),
                                                   _p(mask1), _p(z_all), _p(order), _p(noise), float(inv_B),
                                                   _p(out["weights"]), _p(out["alpha"]), _p(out["rgb_map"]),
                                                   _p(out["disp_map"]), _p(out["acc_map"]), _p(out.get("raw")),
                                                   _p(logits0), _p(logits1), int(agg_mode),
                                                   _p(out["part_map"]), _stream()), "danbo_merge_composite_parts")
    _count(1)
    return out


# ------------------------------------------------------------------------------------------------------ backward
class ActSave:
    """bf16 activations of the fused MLP kept for the backward pass."""

    def __init__(self, cap, device):
        self.cap = int(cap)
        self.act = torch.empty(9, self.cap, 256, device=device, dtype=torch.bfloat16)
        self.g = torch.empty(self.cap, 128, device=device, dtype=torch.bfloat16)


def mlp_forward_save(xtiles, packed, rbias, active, row_ray, out, save):
    lib = _lib.load()
    dev = xtiles.device
    idx = dev.index if dev.index is not None else torch.cuda.current_device()
    _lib.check(lib.danbo_mlp_forward_save(_p(xtiles), _p(packed.wstream), _p(packed.heads), _p(rbias), _p(active.ids),
                                          _p(row_ray), _p(active.count), active.capacity, _p(out), out.shape[0],
                                          num_sms(idx), _p(save.act), _p(save.g), save.cap, _stream()),
               "danbo_mlp_forward_save")
    _count(1)
    return out


def composite_bwd(rays, S, raw, mask, z, noise, inv_B, g_rgb, g_acc, d_raw):
    lib = _lib.load()
    _lib.check(lib.danbo_composite_bwd(_p(rays), rays.stride(0), rays.shape[0], S, _p(raw), _p(mask), _p(z), _p(noise),
                                       float(inv_B), _p(g_rgb), _p(g_acc), _p(d_raw), _stream()), "danbo_composite_bwd")
    _count(1)


def merge_composite_bwd(rays, S_c, S_f, raw0, mask0, raw1, mask1, z_all, order, noise, inv_B, g_rgb, g_acc, g_confd,
                        d_raw0, d_raw1, d_logit0, d_logit1):
    lib = _lib.load()
    _lib.check(lib.danbo_merge_composite_bwd(_p(rays), rays.stride(0), rays.shape[0], S_c, S_f, _p(raw0), _p(mask0),
                                             _p(raw1), _p(mask1), _p(z_all), _p(order), _p(noise), float(inv_B),
                                             _p(g_rgb), _p(g_acc), _p(g_confd), _p(d_raw0), _p(d_raw1), _p(d_logit0),
                                             _p(d_logit1), _stream()), "danbo_merge_composite_bwd")
    _count(1)


def _dgrad(A, B, ldb, D, ldd, active, N, K, accumulate=False, mask=None):
    lib = _lib.load()
    _lib.check(lib.danbo_gemm_dgrad(_p(A), int(A.dtype == torch.bfloat16), A.stride(0), _p(B), int(ldb), _p(D), int(ldd),
                                    _p(active.count), active.capacity, int(N), int(K), int(bool(accumulate)),
                                    _p(mask), 0 if mask is None else mask.stride(0), _stream()), "danbo_gemm_dgrad")
    _count(1)


def _wgrad(A, B, dW, ldw, active, M, N):
    lib = _lib.load()
    _lib.check(lib.danbo_gemm_wgrad(_p(A), A.stride(0), _p(B), int(B.dtype == torch.bfloat16), B.stride(0), _p(dW),
                                    int(ldw), _p(active.count), active.capacity, int(M), int(N), _stream()),
               "danbo_gemm_wgrad")
    _count(1)


def _colsum(A, db, active, N):
    lib = _lib.load()
    _lib.check(lib.danbo_colsum(_p(A), A.stride(0), _p(db), _p(active.count), active.capacity, int(N), _stream()),
               "danbo_colsum")
    _count(1)


def _off(t, elems):
    """Device pointer `elems` elements into tensor t (for column slices of row-major weights)."""
    return ctypes.c_void_p(t.data_ptr() + elems * t.element_size())


class _Ptr:
    """Minimal tensor-like view (pointer + row stride + dtype) so GEMM wrappers can address column slices."""

    def __init__(self, t, col0=0, ld=None):
        self.t, self.col0, self.dtype, self.ld = t, col0, t.dtype, ld

    def data_ptr(self):
        return self.t.data_ptr() + self.col0 * self.t.element_size()

    def stride(self, d):
        return self.ld if (self.ld is not None and d == 0) else self.t.stride(d)


def mlp_backward(P, G, d_raw, active, fo, save, d_ray_bias):
    """Backward of the fused MLP over the rows of one pass.
    P: fp32 parameter tensors by reference name; G: same-named fp32 gradient accumulators (added to).
    fo: FieldOut of the pass (row_ray, x_rows); save: ActSave.  -> dX (cap,208) fp32."""
    lib = _lib.load()
    dev = d_raw.device
    cap = active.capacity
    idx = dev.index if dev.index is not None else torch.cuda.current_device()
    f32 = lambda *s: torch.empty(*s, device=dev, dtype=torch.float32)
    delta9, cur, nxt, d_feat, dX = f32(cap, 128), f32(cap, 256), f32(cap, 256), f32(cap, 256), f32(cap, 208)
    a = save.act
    _lib.check(lib.danbo_mlp_head_bwd(_p(d_raw), _p(active.ids), _p(fo.row_ray), _p(active.count), cap, _p(save.g),
                                      _p(a[7]), _p(P["rgb_linear.weight"]), _p(P["alpha_linear.weight"]), _p(delta9),
                                      _p(cur), _p(G["rgb_linear.weight"]), _p(G["rgb_linear.bias"]),
                                      _p(G["alpha_linear.weight"]), _p(G["alpha_linear.bias"]), _p(d_ray_bias),
                                      num_sms(idx), _stream()), "danbo_mlp_head_bwd")
    _count(1)
    Wv, Wf = P["views_linears.0.weight"], P["feature_linear.weight"]
    # views_linears.0 (feature part): dW[:, :256] += delta9^T . feat ; d feat = delta9 . Wv[:, :256]
    _wgrad(delta9, a[8], G["views_linears.0.weight"], 411, active, 128, 256)
    _dgrad(delta9, Wv, 411, d_feat, 256, active, 256, 128)
    # feature_linear (no activation): bias, weight, and d a7 += d feat . Wf, then the relu mask of layer 7
    _colsum(d_feat, G["feature_linear.bias"], active, 256)
    _wgrad(d_feat, a[7], G["feature_linear.weight"], 256, active, 256, 256)
    _dgrad(d_feat, Wf, 256, cur, 256, active, 256, 256, accumulate=True, mask=a[7])
    for L in range(7, 0, -1):
        W = P[f"pts_linears.{L}.weight"]
        _colsum(cur, G[f"pts_linears.{L}.bias"], active, 256)
        if L == 5:
            dW = G["pts_linears.5.weight"]
            _wgrad(cur, fo.x_rows, dW, 451, active, 256, 195)
            _wgrad(cur, a[4], _Ptr(dW.view(-1), 195), 451, active, 256, 256)
            _dgrad(cur, W, 451, dX, 208, active, 195, 256)
            _dgrad(cur, _Ptr(W.view(-1), 195), 451, nxt, 256, active, 256, 256, mask=a[4])
        else:
            _wgrad(cur, a[L - 1], G[f"pts_linears.{L}.weight"], 256, active, 256, 256)
            _dgrad(cur, W, 256, nxt, 256, active, 256, 256, mask=a[L - 1])
        cur, nxt = nxt, cur
    _colsum(cur, G["pts_linears.0.bias"], active, 256)
    _wgrad(cur, fo.x_rows, G["pts_linears.0.weight"], 195, active, 256, 195)
    _dgrad(cur, P["pts_linears.0.weight"], 195, dX, 208, active, 195, 256, accumulate=True)
    return dX


BACKWARD_IMPL = "tc"          # "tc": tcgen05 dgrad/wgrad kernels; "simt": the fp32 SIMT GEMM chain (kept as a cross-check)
# 2: the weight-gradient launches of the training backward run on a side stream beside the field backward (autograd.py);
# 1: one stream.  DANBO_BWD_STREAMS overrides.
BACKWARD_STREAMS = int(os.environ.get("DANBO_BWD_STREAMS", "2"))


class BwdWorkspace:
    """Buffers of the tensor-core MLP backward for one row capacity (reused by the coarse and fine passes)."""

    def __init__(self, cap, device):
        lib = _lib.load()
        sizes = [ctypes.c_longlong() for _ in range(5)]
        ns = ctypes.c_int()
        lib.danbo_mlp_bwd_workspace(int(cap), *[ctypes.byref(x) for x in sizes], ctypes.byref(ns))
        u8 = lambda n: torch.empty(int(n), device=device, dtype=torch.uint8)
        self.cap = int(cap)
        self.wstream, self.delta, self.deltaT, self.actT, self.partial = [u8(x.value) for x in sizes]
        self.packed_key = None


def mlp_backward_tc(P, G, d_raw, active, fo, save, d_ray_bias, ws, repack=True, wgrad_stream=None):
    """Tensor-core backward of the fused MLP over the rows of one pass -> dX (cap,208) fp32; parameter grads added to G.
    wgrad_stream: a side stream for the weight-gradient launches (transposes, wgrad, reduce, bias column sums).  They
    depend only on what dgrad wrote and touch only the MLP's gradient tensors, so they can run beside the field backward
    (which consumes dX on the calling stream); the caller joins the side stream before it returns."""
    lib = _lib.load()
    dev = d_raw.device
    cap = active.capacity
    assert ws.cap >= cap and save.cap == cap
    idx = dev.index if dev.index is not None else torch.cuda.current_device()
    # rgb / alpha heads, ray-bias gradient (small fp32 reductions)
    _lib.check(lib.danbo_mlp_head_bwd(_p(d_raw), _p(active.ids), _p(fo.row_ray), _p(active.count), cap, _p(save.g),
                                      _p(save.act[7]), _p(P["rgb_linear.weight"]), _p(P["alpha_linear.weight"]), None,
                                      None, _p(G["rgb_linear.weight"]), _p(G["rgb_linear.bias"]),
                                      _p(G["alpha_linear.weight"]), _p(G["alpha_linear.bias"]), _p(d_ray_bias),
                                      num_sms(idx), _stream()), "danbo_mlp_head_bwd")
    if repack:
        wa = (ctypes.c_void_p * 8)(*[P[f"pts_linears.{i}.weight"].data_ptr() for i in range(8)])
        _lib.check(lib.danbo_pack_mlp_dgrad(wa, _p(P["feature_linear.weight"]), _p(P["views_linears.0.weight"]),
                                            _p(ws.wstream), _stream()), "danbo_pack_mlp_dgrad")
        _count(1)
    dX = torch.empty(cap, 208, device=dev, dtype=torch.float32)
    _lib.check(lib.danbo_mlp_dgrad(_p(ws.wstream), _p(P["rgb_linear.weight"]), _p(P["alpha_linear.weight"]), _p(d_raw),
                                   _p(active.ids), _p(active.count), cap, _p(save.act), _p(save.g), cap, _p(ws.delta),
                                   _p(ws.deltaT), _p(dX), num_sms(idx), _stream()), "danbo_mlp_dgrad")
    dw_names = ["views_linears.0.weight", "feature_linear.weight"] + [f"pts_linears.{i}.weight" for i in range(7, -1, -1)]
    db_names = ["feature_linear.bias"] + [f"pts_linears.{i}.bias" for i in range(7, -1, -1)]
    dw = (ctypes.c_void_p * 10)(*[G[n].data_ptr() for n in dw_names])
    db = (ctypes.c_void_p * 9)(*[G[n].data_ptr() for n in db_names])

    def wgrad():
        _lib.check(lib.danbo_mlp_wgrad(_p(save.act), _p(fo.x_rows), _p(ws.delta), cap, _p(active.count), cap, _p(ws.deltaT), 1,
                                       _p(ws.actT), _p(ws.partial), dw, db, _stream()), "danbo_mlp_wgrad")
    if wgrad_stream is None:
        wgrad()
    else:
        wgrad_stream.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(wgrad_stream):
            wgrad()
    _count(8)
    return dX


class PackedDgrad:
    """The transposed bf16 weight tiles danbo_mlp_dgrad reads, kept across calls: a backward that trains no weight
    (the pose-only path) repacks them only when the weights changed (`RayCaster._packed_dgrad`), not per iteration."""

    def __init__(self, device):
        sizes = [ctypes.c_longlong() for _ in range(5)]
        ns = ctypes.c_int()
        _lib.load().danbo_mlp_bwd_workspace(1, *[ctypes.byref(x) for x in sizes], ctypes.byref(ns))
        self.wstream = torch.empty(sizes[0].value, device=device, dtype=torch.uint8)

    def pack(self, P):
        """P: the reference's parameter names -> fp32 CUDA tensors (pts_linears.i.weight, feature_linear.weight,
        views_linears.0.weight)."""
        ws = [f32c(P[f"pts_linears.{i}.weight"]) for i in range(8)]
        wf, wv = f32c(P["feature_linear.weight"]), f32c(P["views_linears.0.weight"])
        _need_cuda(*ws, wf, wv)
        wa = (ctypes.c_void_p * 8)(*[t.data_ptr() for t in ws])
        _lib.check(_lib.load().danbo_pack_mlp_dgrad(wa, _p(wf), _p(wv), _p(self.wstream), _stream()),
                   "danbo_pack_mlp_dgrad")
        self._keep = (ws, wf, wv)              # sources alive until the stream has consumed them
        _count(1)
        return self


def mlp_backward_pose(P, d_raw, active, fo, save, packed_t, d_ray_bias=None):
    """Backward of the fused MLP when no weight needs a gradient (pose-only path) -> dX (cap,208) fp32.  The head
    backward runs only for d_ray_bias ((n,128) fp32, added to; None: not formed, and then no head launch at all); the
    data-gradient chain is the dX-only variant of danbo_mlp_dgrad (no delta planes).  packed_t: a PackedDgrad of the
    current weights.  No transposes, no K = rows GEMMs, no bias sums."""
    lib = _lib.load()
    dev = d_raw.device
    cap = active.capacity
    assert save.cap == cap
    idx = dev.index if dev.index is not None else torch.cuda.current_device()
    if d_ray_bias is not None:
        _lib.check(lib.danbo_mlp_head_bwd(_p(d_raw), _p(active.ids), _p(fo.row_ray), _p(active.count), cap, _p(save.g),
                                          _p(save.act[7]), _p(P["rgb_linear.weight"]), _p(P["alpha_linear.weight"]),
                                          None, None, None, None, None, None, _p(d_ray_bias), num_sms(idx), _stream()),
                   "danbo_mlp_head_bwd")
        _count(1)
    dX = torch.empty(cap, 208, device=dev, dtype=torch.float32)
    _lib.check(lib.danbo_mlp_dgrad(_p(packed_t.wstream), _p(P["rgb_linear.weight"]), _p(P["alpha_linear.weight"]),
                                   _p(d_raw), _p(active.ids), _p(active.count), cap, _p(save.act), _p(save.g), cap, None,
                                   None, _p(dX), num_sms(idx), _stream()), "danbo_mlp_dgrad")
    _count(1)
    return dX


def ray_bias_bwd(rays, cam_idx, codes_with_mean, w_view, d_ray_bias, d_w_view, d_b_view, d_codes):
    lib = _lib.load()
    _lib.check(lib.danbo_ray_bias_bwd(_p(rays), rays.stride(0), rays.shape[0], _p(cam_idx), _p(codes_with_mean),
                                      codes_with_mean.shape[0] - 1, _p(w_view), _p(d_ray_bias), _p(d_w_view),
                                      _p(d_b_view), _p(d_codes), _stream()), "danbo_ray_bias_bwd")
    _count(1)


def view_root_bwd(rays, pose_skts, rays_per_pose, w_view, d_ray_bias, d_skts):
    """d skts (n_poses,24,4,4) += d loss / d skts through root-local view directions (perfcap configs under --opt_pose,
    danbo_view_root_bwd): rows 0-2, columns 0-2 of joint 0 only.  rays (n,>=6) with unit column stride, w_view the
    (128,411) view weight, d_ray_bias (n,128) the gradient of danbo_ray_bias's output."""
    tensors = dict(rays=rays, pose_skts=pose_skts, w_view=w_view, d_ray_bias=d_ray_bias, d_skts=d_skts)
    _need_cuda(*tensors.values())
    for name, t in tensors.items():
        if t.dtype != torch.float32:
            raise ValueError(f"view_root_bwd: {name} must be fp32, got {t.dtype}")
        if t.device != rays.device:
            raise ValueError(f"view_root_bwd: {name} is on {t.device}, rays on {rays.device}")
    n = rays.shape[0]
    if rays.dim() != 2 or rays.shape[1] < 6 or rays.stride(1) != 1:
        raise ValueError("view_root_bwd: rays must be (n, >=6) with contiguous rows")
    if pose_skts.dim() != 4 or tuple(pose_skts.shape[1:]) != (J, 4, 4) or not pose_skts.is_contiguous():
        raise ValueError("view_root_bwd: pose_skts must be a contiguous (n_poses,24,4,4) tensor")
    if tuple(w_view.shape) != (128, 411) or not w_view.is_contiguous():
        raise ValueError("view_root_bwd: w_view must be a contiguous (128,411) tensor")
    if tuple(d_ray_bias.shape) != (n, 128) or not d_ray_bias.is_contiguous() or d_ray_bias.data_ptr() % 16:
        raise ValueError("view_root_bwd: d_ray_bias must be a contiguous, 16-byte aligned (n,128) tensor")
    if d_skts.shape != pose_skts.shape or not d_skts.is_contiguous():
        raise ValueError("view_root_bwd: d_skts must be a contiguous tensor of pose_skts' shape")
    if int(rays_per_pose) <= 0:
        raise ValueError("view_root_bwd: rays_per_pose must be positive")
    with _Timed("view_root_bwd"):
        _lib.check(_lib.load().danbo_view_root_bwd(_p(rays), rays.stride(0), n, _p(pose_skts), int(rays_per_pose),
                                                   pose_skts.shape[0], _p(w_view), _p(d_ray_bias), _p(d_skts),
                                                   _stream()), "danbo_view_root_bwd")
    _count(1)
    return d_skts


def field_agg_bwd(rays, S, z, mask, active, pose_skts, pose_vol, rays_per_pose, consts, fo, dX, g_logit_ext, grads,
                  d_skts=None):
    """grads: list of the 9 fp32 parameter / volume accumulators in the order of danbo_field_agg_bwd (see danbo_b200.h);
    entries 0-6 and 8 (aggregation net, axis_scale) all None select the pose-only kernel variant, entry 7 (d vol) is
    always required.  d_skts: (n_poses,24,4,4) fp32 accumulator of the gradient w.r.t. the world-to-bone matrices, or
    None."""
    lib = _lib.load()
    dev = rays.device
    n = rays.shape[0]
    d_hbar = torch.empty(active.capacity, 16, device=dev, dtype=torch.float32)
    d_logit = torch.empty(n * S, J, device=dev, dtype=torch.float32)
    if len(grads) != 9:
        raise ValueError("field_agg_bwd takes 9 accumulators (+ d_skts)")
    n_weight = sum(g is not None for i, g in enumerate(grads) if i != 7)
    if grads[7] is None or n_weight not in (0, 8):
        raise ValueError("field_agg_bwd: d vol (grads[7]) is required; the other 8 accumulators are all given or all None")
    if d_skts is not None:
        _need_cuda(d_skts)
        if d_skts.dtype != torch.float32 or not d_skts.is_contiguous() or tuple(d_skts.shape) != (pose_skts.shape[0], J, 4, 4):
            raise ValueError("d_skts must be a contiguous fp32 (n_poses,24,4,4) tensor")
    ga = (ctypes.c_void_p * 10)(*([None if g is None else g.data_ptr() for g in grads] +
                                  [None if d_skts is None else d_skts.data_ptr()]))
    idx = dev.index if dev.index is not None else torch.cuda.current_device()
    _lib.check(lib.danbo_field_agg_bwd(_p(rays), rays.stride(0), n, S, _p(z), _p(mask), _p(active.ids), _p(active.count),
                                       active.capacity, _p(pose_skts), _p(pose_vol), int(rays_per_pose),
                                       pose_skts.shape[0], consts.array, _p(fo.logits), _p(fo.hbar), _p(dX),
                                       _p(g_logit_ext), _p(d_hbar), _p(d_logit), _p(fo.work), fo.pair_cap, ga,
                                       num_sms(idx), fo.agg_mode, _stream()), "danbo_field_agg_bwd")
    _count(2)


def field_agg_bwd_pts(rays, S, z, mask, active, pose_skts, pose_vol, rays_per_pose, consts, fo, dX, d_pts, d_vol=None,
                      d_skts=None):
    """d / d (sample position) of the field's output through the same chain as field_agg_bwd (danbo_field_agg_bwd_pts):
    d_pts (n*S,3) fp32, added to, is required; d_vol (pose_vol's shape) and d_skts (n_poses,24,4,4) are optional
    accumulators (None: not formed).  The feature window's derivative is included (training detaches it), so these are
    the field's true derivatives.  fo: the forward field_agg of the same call, with want_hbar."""
    lib = _lib.load()
    dev = rays.device
    n = rays.shape[0]
    if fo.hbar is None:
        raise ValueError("field_agg_bwd_pts: the forward field_agg must keep hbar (want_hbar=True)")
    for name, t, shape in (("d_pts", d_pts, (n * S, 3)), ("d_vol", d_vol, tuple(pose_vol.shape)),
                           ("d_skts", d_skts, (pose_skts.shape[0], J, 4, 4))):
        if t is None:
            if name == "d_pts":
                raise ValueError("field_agg_bwd_pts: d_pts is required")
            continue
        _need_cuda(t)
        if t.dtype != torch.float32 or not t.is_contiguous() or tuple(t.shape) != shape or t.device != dev:
            raise ValueError(f"field_agg_bwd_pts: {name} must be a contiguous fp32 {shape} tensor on {dev}")
    if tuple(dX.shape) != (active.capacity, 208) or dX.dtype != torch.float32 or not dX.is_contiguous():
        raise ValueError("field_agg_bwd_pts: dX must be the contiguous fp32 (capacity,208) output of the MLP backward")
    d_hbar = torch.empty(active.capacity, 16, device=dev, dtype=torch.float32)
    d_logit = torch.empty(n * S, J, device=dev, dtype=torch.float32)
    idx = dev.index if dev.index is not None else torch.cuda.current_device()
    _lib.check(lib.danbo_field_agg_bwd_pts(_p(rays), rays.stride(0), n, S, _p(z), _p(mask), _p(active.ids),
                                           _p(active.count), active.capacity, _p(pose_skts), _p(pose_vol),
                                           int(rays_per_pose), pose_skts.shape[0], consts.array, _p(fo.logits),
                                           _p(fo.hbar), _p(dX), None, _p(d_hbar), _p(d_logit), _p(fo.work), fo.pair_cap,
                                           _p(d_pts), _p(d_vol), _p(d_skts), num_sms(idx), fo.agg_mode, _stream()),
               "danbo_field_agg_bwd_pts")
    _count(2)
    return d_pts


GN_PARAMS =["layers.0.lin.weight", "layers.0.adj_w", "layers.0.adj", "layers.0.bias", "layers.1.lin.weight",
             "layers.1.adj_w", "layers.1.adj", "layers.1.bias", "layers.2.weight", "layers.2.bias", "layers.3.weight",
             "layers.3.bias"]                                    # order of danbo_graph_net_fwd's params[12]
GN_GRADS = [n for n in GN_PARAMS if not n.endswith(".adj")]     # order of danbo_graph_net_bwd's grads[10]


def graph_net_fwd(pose_bones, tensors):
    """GN1 + GN2 in four launches.  pose_bones (G,24,3); tensors: the 12 GN_PARAMS tensors (fp32, CUDA).
    -> vol (G,24,240), saved (what graph_net_bwd needs)."""
    lib = _lib.load()
    pb = f32c(pose_bones)
    tensors = [f32c(t) for t in tensors]
    _need_cuda(pb, *tensors)
    G, dev = pb.shape[0], pb.device
    bufs = [torch.empty(G, J, 66, device=dev)] + [torch.empty(G, J, 128, device=dev) for _ in range(5)]
    vol = torch.empty(G, J, 240, device=dev)
    pa = (ctypes.c_void_p * 12)(*[t.data_ptr() for t in tensors])
    sa = (ctypes.c_void_p * 6)(*[t.data_ptr() for t in bufs])
    _lib.check(lib.danbo_graph_net_fwd(_p(pb), G, pa, sa, _p(vol), _stream()), "danbo_graph_net_fwd")
    _count(4)
    return vol, (tensors, bufs)


def graph_net_bwd(saved, d_vol, grads):
    """grads: the 10 fp32 accumulators in GN_GRADS order (added to), or None: the pose-only variant (three launches,
    no weight gradient), whose `work` graph_net_bwd_pose reads all the same."""
    lib = _lib.load()
    tensors, bufs = saved
    d_vol = f32c(d_vol)
    G, dev = d_vol.shape[0], d_vol.device
    work = torch.empty(2 * G * J * 128, device=dev)
    pa = (ctypes.c_void_p * 12)(*[t.data_ptr() for t in tensors])
    sa = (ctypes.c_void_p * 6)(*[t.data_ptr() for t in bufs])
    ga = None if grads is None else (ctypes.c_void_p * 10)(*[g.data_ptr() for g in grads])
    _lib.check(lib.danbo_graph_net_bwd(G, pa, sa, _p(d_vol), ga, _p(work), _stream()), "danbo_graph_net_bwd")
    _count(3 if grads is None else 4)
    return work


def graph_net_bwd_pose(saved, work, pose_bones):
    """d loss / d pose_bones (G,24,3) of the graph net (danbo_graph_net_bwd_pose), after graph_net_bwd returned `work`
    for the same `saved`; pose_bones is what graph_net_fwd read.  The root's row is zero (mask_root)."""
    tensors, bufs = saved
    _need_cuda(pose_bones, work)
    G = bufs[0].shape[0]
    if pose_bones.dtype != torch.float32 or tuple(pose_bones.shape) != (G, J, 3) or not pose_bones.is_contiguous():
        raise ValueError(f"graph_net_bwd_pose: pose_bones must be a contiguous fp32 ({G},24,3) tensor")
    if work.dtype != torch.float32 or work.numel() != 2 * G * J * 128 or not work.is_contiguous():
        raise ValueError("graph_net_bwd_pose: work must be graph_net_bwd's workspace of the same poses")
    if pose_bones.device != work.device or bufs[0].device != work.device:
        raise ValueError("graph_net_bwd_pose: pose_bones, work and saved must be on one device")
    d_bones = torch.empty(G, J, 3, device=work.device)
    pa = (ctypes.c_void_p * 12)(*[t.data_ptr() for t in tensors])
    sa = (ctypes.c_void_p * 6)(*[t.data_ptr() for t in bufs])
    with _Timed("graph_net_bwd_pose"):
        _lib.check(_lib.load().danbo_graph_net_bwd_pose(_p(pose_bones), G, pa, sa, _p(work), _p(d_bones), _stream()),
                   "danbo_graph_net_bwd_pose")
    _count(1)
    return d_bones


def _pose_layer_args(fn, layer, idx, idx_stride, n_poses):
    """Checks the pose layer's tensors for pose_fwd / pose_bwd -> the leading arguments of danbo_pose_fwd/_bwd."""
    pelvis, bones, rest = layer["pelvis"], layer["bones"], layer["rest_pose"]
    root_bones, kp_map, rest_idx = layer.get("root_bones"), layer.get("kp_map"), layer.get("rest_idx")
    _need_cuda(pelvis, bones, rest, idx, root_bones, kp_map, rest_idx)
    dev = pelvis.device
    for name, t, dt in (("pelvis", pelvis, torch.float32), ("bones", bones, torch.float32), ("rest_pose", rest, torch.float32),
                        ("root_bones", root_bones, torch.float32), ("kp_map", kp_map, torch.int64),
                        ("rest_idx", rest_idx, torch.int64), ("idx", idx, torch.int64)):
        if t is None:
            continue
        if t.dtype != dt or not t.is_contiguous() or t.device != dev:
            raise ValueError(f"{fn}: {name} must be a contiguous {dt} tensor on {dev}")
    F_ = pelvis.shape[0]
    if tuple(pelvis.shape) != (F_, 3):
        raise ValueError(f"{fn}: pelvis must be (F,3)")
    if (root_bones is None) != (kp_map is None):
        raise ValueError(f"{fn}: root_bones and kp_map go together (the multi-view split)")
    if root_bones is None:
        if tuple(bones.shape) != (F_, J, 3):
            raise ValueError(f"{fn}: bones must be (F,24,3) axis-angle")
    elif tuple(root_bones.shape) != (F_, 3) or bones.dim() != 3 or tuple(bones.shape[1:]) != (J - 1, 3) \
            or tuple(kp_map.shape) != (F_,):
        raise ValueError(f"{fn}: the multi-view split needs root_bones (F,3), bones (U,23,3) and kp_map (F)")
    if rest.dim() != 3 or tuple(rest.shape[1:]) != (J, 3):
        raise ValueError(f"{fn}: rest_pose must be (R,24,3)")
    if rest.shape[0] > 1 and (rest_idx is None or tuple(rest_idx.shape) != (F_,)):
        raise ValueError(f"{fn}: several rest poses need a per-frame row table rest_idx (F)")
    if idx.dim() != 1 or int(idx_stride) <= 0 or (int(n_poses) - 1) * int(idx_stride) >= max(idx.shape[0], 1):
        raise ValueError(f"{fn}: idx must be 1-D and hold n_poses entries at stride idx_stride")
    return [_p(pelvis), _p(bones), _p(root_bones), _p(kp_map), _p(rest), rest.shape[0],
            _p(rest_idx if rest.shape[0] > 1 else None), _p(idx), int(idx_stride), int(n_poses)]


def pose_fwd(layer, idx, idx_stride, n_poses, anchors=None, tol=0., coef=0., ext_scale=0.001):
    """The pose layer's forward for poses idx[0], idx[stride], ... (danbo_pose_fwd).  layer: dict of the parameter and
    buffer tensors (pelvis, bones[, root_bones, kp_map], rest_pose[, rest_idx]); anchors: {'kps', 'bones'} (F,24,3)
    for the regulariser and MPJPC, or None.  -> kps (G,24,3), bones (G,24,3), skts (G,24,4,4), stats (2,) or None."""
    args = _pose_layer_args("pose_fwd", layer, idx, idx_stride, n_poses)
    dev, F_ = layer["pelvis"].device, layer["pelvis"].shape[0]
    ak = ab = stats = None
    if anchors is not None:
        ak, ab = anchors["kps"], anchors["bones"]
        for name, t in (("kps", ak), ("bones", ab)):
            _need_cuda(t)
            if t.dtype != torch.float32 or not t.is_contiguous() or t.device != dev or tuple(t.shape) != (F_, J, 3):
                raise ValueError(f"pose_fwd: anchor {name} must be a contiguous fp32 ({F_},24,3) tensor on {dev}")
        if not float(ext_scale) > 0:
            raise ValueError("pose_fwd: ext_scale must be positive")
        stats = torch.empty(2, device=dev)
    G = int(n_poses)
    kps, bones, skts = torch.empty(G, J, 3, device=dev), torch.empty(G, J, 3, device=dev), torch.empty(G, J, 4, 4, device=dev)
    with _Timed("pose_fwd"):
        _lib.check(_lib.load().danbo_pose_fwd(*args, _p(ak), _p(ab), float(tol), float(coef), float(ext_scale), _p(kps),
                                              _p(bones), _p(skts), _p(stats), _stream()), "danbo_pose_fwd")
    _count(1)
    return kps, bones, skts, stats


def pose_bwd(layer, idx, idx_stride, n_poses, d_skts, grads, d_bones=None, d_kps=None, anchor_bones=None, d_reg=None,
             tol=0., coef=0.):
    """Backward of pose_fwd (danbo_pose_bwd): ADDS d loss / d parameters into grads {'pelvis', 'bones'[,
    'root_bones']} (fp32, the parameters' shapes).  d_reg: device scalar d loss / d kp_loss, or None (no regulariser)."""
    args = _pose_layer_args("pose_bwd", layer, idx, idx_stride, n_poses)
    dev, G = layer["pelvis"].device, int(n_poses)
    for name, t, shape in (("d_skts", d_skts, (G, J, 4, 4)), ("d_bones", d_bones, (G, J, 3)), ("d_kps", d_kps, (G, J, 3)),
                           ("d_reg", d_reg, ()), ("anchor_bones", anchor_bones, (layer["pelvis"].shape[0], J, 3))):
        if t is None:
            continue
        _need_cuda(t)
        if t.dtype != torch.float32 or not t.is_contiguous() or t.device != dev or tuple(t.shape) != shape:
            raise ValueError(f"pose_bwd: {name} must be a contiguous fp32 {shape} tensor on {dev}")
    if d_skts is None:
        raise ValueError("pose_bwd: d_skts is required")
    if d_reg is not None and anchor_bones is None:
        raise ValueError("pose_bwd: the regulariser's gradient needs anchor_bones")
    names = ("pelvis", "bones") + (("root_bones",) if layer.get("root_bones") is not None else ())
    if set(grads) != set(names):
        raise ValueError(f"pose_bwd: grads must hold exactly {names}")
    for nm in names:
        g = grads[nm]
        _need_cuda(g)
        if g.dtype != torch.float32 or not g.is_contiguous() or g.device != dev or g.shape != layer[nm].shape:
            raise ValueError(f"pose_bwd: grads[{nm!r}] must be a contiguous fp32 tensor of the parameter's shape")
    with _Timed("pose_bwd"):
        _lib.check(_lib.load().danbo_pose_bwd(*args, _p(d_skts), _p(d_bones), _p(d_kps), _p(anchor_bones), _p(d_reg),
                                              float(tol), float(coef), _p(grads["pelvis"]), _p(grads["bones"]),
                                              _p(grads.get("root_bones")), _stream()), "danbo_pose_bwd")
    _count(1)


def pose_kp2d(kps, kp2d, proj, sigma, coef):
    """The 2D keypoint reprojection term (danbo_pose_kp2d) of kps (G,24,3) against detections kp2d (G,24,3) = (u, v,
    confidence) through projection matrices proj (G,3,4), all contiguous fp32 on one device.
    -> loss (scalar), kp2d_px (scalar, mean pixel error over the joints with confidence > 0), d loss / d kps (G,24,3)."""
    _need_cuda(kps, kp2d, proj)
    dev, G = kps.device, kps.shape[0]
    for name, t, shape in (("kps", kps, (G, J, 3)), ("kp2d", kp2d, (G, J, 3)), ("proj", proj, (G, 3, 4))):
        if t.dtype != torch.float32 or not t.is_contiguous() or t.device != dev or tuple(t.shape) != shape:
            raise ValueError(f"pose_kp2d: {name} must be a contiguous fp32 {shape} tensor on {dev}")
    if not float(sigma) > 0:
        raise ValueError("pose_kp2d: sigma must be positive")
    d_kps = torch.empty(G, J, 3, device=dev)
    stats = torch.empty(2, device=dev)
    with _Timed("pose_kp2d"):
        _lib.check(_lib.load().danbo_pose_kp2d(_p(kps), _p(kp2d), _p(proj), int(G), float(sigma), float(coef),
                                               _p(d_kps), _p(stats), _stream()), "danbo_pose_kp2d")
    _count(1)
    return stats[0], stats[1], d_kps


LOSS_KINDS = {"L1": 0, "MSE": 1}


def train_loss(preds, target, bgs, loss_kind, rgb_coef, coarse_weight, soft_coef=None, axis_scale=None, init_scale=None,
               vol_coef=0., g_axis_scale=None, use_background=True):
    """L*: the trainer's losses and their gradients in one launch (danbo_train_loss).
    preds: the caster's train-mode dict.  bgs: (n,3) tensor or a float.  soft_coef None -> no soft-softmax term;
    axis_scale None -> no volume-scale term (otherwise its gradient is ADDED to g_axis_scale (24,3)).
    -> terms (4,) float64 [rgb, rgb coarse, soft-softmax, volume-scale], grads dict keyed like preds."""
    lib = _lib.load()
    rgb, acc = preds["rgb_map"], preds["acc_map"]
    _need_cuda(rgb, acc, target, axis_scale)
    n, dev = rgb.shape[0], rgb.device
    c = lambda t: None if t is None else t.detach().float().contiguous()
    rgb0, acc0 = c(preds.get("rgb0")), c(preds.get("acc0"))
    confd = pinv = Ti = al = None
    S_t = 0
    if soft_coef is not None:
        confd, pinv, Ti, al = c(preds["confd"]), c(preds["part_invalid"]), c(preds["T_i"]), c(preds["alpha"])
        S_t = confd.shape[1]
    bg_t = c(bgs).expand(n, 3).contiguous() if torch.is_tensor(bgs) else None
    terms = torch.empty(4, device=dev, dtype=torch.float64)
    g = {"rgb_map": torch.empty(n, 3, device=dev), "acc_map": torch.empty(n, device=dev)}
    if rgb0 is not None:
        g["rgb0"], g["acc0"] = torch.empty(n, 3, device=dev), torch.empty(n, device=dev)
    if confd is not None:
        g["confd"] = torch.empty_like(confd)
    _lib.check(lib.danbo_train_loss(_p(c(rgb)), _p(c(acc)), _p(rgb0), _p(acc0), _p(c(target)), _p(bg_t),
                                    0.0 if bg_t is not None else float(bgs), int(bool(use_background)), n,
                                    LOSS_KINDS[loss_kind], float(rgb_coef), float(coarse_weight), _p(confd), _p(pinv), _p(Ti),
                                    _p(al), int(S_t), float(soft_coef or 0.), _p(c(axis_scale)), _p(c(init_scale)),
                                    float(vol_coef), _p(terms), _p(g["rgb_map"]), _p(g["acc_map"]), _p(g.get("rgb0")),
                                    _p(g.get("acc0")), _p(g.get("confd")), _p(g_axis_scale), _stream()), "danbo_train_loss")
    _count(1)
    return terms, g


# ------------------------------------------------------------------------------------------------------------
# AN1: A-NeRF field (nerf_type = nerf, BASELINE config #4)
ANERF_XD_TILE_BYTES = 7 * 16384
ANERF_XV_TILE_BYTES = 11 * 16384


class AnerfPacked:
    """Packed weights + per-CTA activation scratch of the A-NeRF MLP (W = 448)."""

    def __init__(self, device):
        lib = _lib.load()
        idx = device.index if device.index is not None else torch.cuda.current_device()
        sizes = [ctypes.c_longlong() for _ in range(4)]
        lib.danbo_anerf_workspace_bytes(num_sms(idx), *[ctypes.byref(x) for x in sizes])
        self.wstream = torch.empty(sizes[0].value, device=device, dtype=torch.uint8)
        self.heads = torch.empty(sizes[1].value // 4, device=device, dtype=torch.float32)
        self.w_code = torch.empty(sizes[2].value // 4, device=device, dtype=torch.float32)
        self.scratch = torch.empty(sizes[3].value, device=device, dtype=torch.uint8)

    def pack(self, P):
        lib = _lib.load()
        ws = [f32c(P[f"pts_linears.{i}.weight"]) for i in range(8)]
        bs = [f32c(P[f"pts_linears.{i}.bias"]) for i in range(8)]
        others = [f32c(P[k]) for k in ("alpha_linear.weight", "alpha_linear.bias", "feature_linear.weight",
                                       "feature_linear.bias", "views_linears.0.weight", "views_linears.0.bias",
                                       "rgb_linear.weight", "rgb_linear.bias")]
        _need_cuda(*ws, *bs, *others)
        wa = (ctypes.c_void_p * 8)(*[t.data_ptr() for t in ws])
        ba = (ctypes.c_void_p * 8)(*[t.data_ptr() for t in bs])
        _lib.check(lib.danbo_anerf_pack_weights(wa, ba, *[_p(t) for t in others], _p(self.wstream), _p(self.heads),
                                                _p(self.w_code), _stream()), "danbo_anerf_pack_weights")
        self._keep = (ws, bs, others)
        _count(1)
        return self


def anerf_ray_encode(rays, pose_skts, rays_per_pose, cam_idx, codes_with_mean, packed):
    """-> ray_enc (n,648), code_bias (n,224)."""
    _need_cuda(rays, pose_skts, cam_idx, codes_with_mean)
    lib = _lib.load()
    n = rays.shape[0]
    enc = torch.empty(n, 648, device=rays.device, dtype=torch.float32)
    cb = torch.empty(n, 224, device=rays.device, dtype=torch.float32)
    with _Timed("anerf_ray_encode"):
        _lib.check(lib.danbo_anerf_ray_encode(_p(rays), rays.stride(0), n, _p(pose_skts), int(rays_per_pose),
                                              pose_skts.shape[0], _p(cam_idx), _p(codes_with_mean),
                                              codes_with_mean.shape[0] - 1, _p(packed.w_code), _p(enc), _p(cb), _stream()),
                   "danbo_anerf_ray_encode")
    _count(1)
    return enc, cb


def anerf_embed(rays, S, z, pose_skts, rays_per_pose, align, ray_enc, tau, xd=None, xv=None):
    """z (n,S) -> operand tile images xd, xv (uint8) of the n*S dense rows."""
    _need_cuda(rays, z, pose_skts, align, ray_enc)
    lib = _lib.load()
    rows = rays.shape[0] * S
    tiles = (rows + 127) // 128
    if xd is None:
        xd = torch.empty(tiles * ANERF_XD_TILE_BYTES, device=rays.device, dtype=torch.uint8)
    if xv is None:
        xv = torch.empty(tiles * ANERF_XV_TILE_BYTES, device=rays.device, dtype=torch.uint8)
    assert xd.numel() >= tiles * ANERF_XD_TILE_BYTES and xv.numel() >= tiles * ANERF_XV_TILE_BYTES
    with _Timed("anerf_embed"):
        _lib.check(lib.danbo_anerf_embed(_p(rays), rays.stride(0), int(S), _p(z), rows, _p(pose_skts), int(rays_per_pose),
                                         pose_skts.shape[0], _p(align), _p(ray_enc), float(tau), _p(xd), _p(xv), _stream()),
                   "danbo_anerf_embed")
    _count(1)
    return xd, xv


ANERF_ACT_TILE_BYTES = 7 * 16384          # one layer's activation tile image (128 rows x 448 bf16, operand layout)


def anerf_save_buffer(rows, device):
    """Train mode: room for the nine activation tile images ([tile][9]) danbo_anerf_mlp_save keeps per 128-row tile."""
    n = ctypes.c_longlong()
    _lib.check(_lib.load().danbo_anerf_save_bytes(int(rows), ctypes.byref(n)), "danbo_anerf_save_bytes")
    return torch.empty(n.value, device=device, dtype=torch.uint8)


def anerf_untile(img, tile_stride, rows, n_chunks, byte_offset=0):
    """Operand tile images -> row-major bf16 (rows, 64 * n_chunks).  byte_offset / tile_stride select one layer's plane of
    the [tile][9] activation save."""
    _need_cuda(img)
    out = torch.empty(rows, 64 * n_chunks, device=img.device, dtype=torch.bfloat16)
    src = ctypes.c_void_p(img.data_ptr() + int(byte_offset))
    _lib.check(_lib.load().danbo_anerf_untile(src, int(tile_stride), int(rows), int(n_chunks), _p(out), _stream()),
               "danbo_anerf_untile")
    _count(1)
    return out


def anerf_mlp(xd, xv, packed, code_bias, rows, S, out, trace=None, save=None):
    """out (>= rows, 4) <- [rgb, sigma] of the dense rows.  trace: optional int64 CUDA tensor (320) for a clock64 timeline.
    save: train mode, a buffer from anerf_save_buffer(rows) that receives every layer's activation tile image."""
    _need_cuda(xd, xv, code_bias, out)
    lib = _lib.load()
    idx = out.device.index if out.device.index is not None else torch.cuda.current_device()
    if save is not None:
        with _Timed("anerf_mlp"):
            _lib.check(lib.danbo_anerf_mlp_save(_p(xd), _p(xv), _p(packed.wstream), _p(packed.heads), _p(code_bias),
                                                _p(packed.scratch), int(rows), int(S), _p(out), out.shape[0], num_sms(idx),
                                                _p(save), _stream()), "danbo_anerf_mlp_save")
        _count(1)
        return out
    with _Timed("anerf_mlp"):
        _lib.check(lib.danbo_anerf_mlp(_p(xd), _p(xv), _p(packed.wstream), _p(packed.heads), _p(code_bias),
                                       _p(packed.scratch), int(rows), int(S), _p(out), out.shape[0], num_sms(idx),
                                       _p(trace), _stream()),
                   "danbo_anerf_mlp")
    _count(1)
    return out


class _RowCount:
    """Device row counter for the generic GEMM kernels (they read the row count from device memory)."""

    def __init__(self, rows, device):
        self.count = torch.full((1,), int(rows), device=device, dtype=torch.int32)
        self.capacity = int(rows)


def anerf_mlp_backward(P, G, d_raw, rows, S, xd, xv, save, code_bias, cam_idx, codes_with_mean, want_dx=False):
    """Backward of the A-NeRF MLP (core/networks/nerf.py:164-209 under autograd, trainer.py:573) over the `rows` dense
    rows of one pass: parameter gradients are ADDED to G (reference names).  The encodings have no trainable parameter
    (opt_cutoff = False), so the input gradient is only formed when the poses are optimised (want_dx): then
    -> (d xd (rows,432), d xv (rows,648)) fp32, d xd = delta0 . W0 + delta5 . W5[:, :432] (layer 0 and the skip input of
    layer 5), d xv = delta9 . Wv[:, 448:1096], three more danbo_gemm_dgrad launches.  Otherwise None, and the launch
    sequence is the one without them.

    d_raw (>= rows,4) [d rgb, d sigma]; xd / xv: the pass's operand tile images; save: what danbo_anerf_mlp_save kept;
    code_bias (n_rays,224) from danbo_anerf_ray_encode.  Built from the generic fp32 GEMM kernels of backward_mlp.cu
    (danbo_gemm_dgrad / _wgrad / danbo_colsum) on row-major copies of the tile images: correct first, not yet on tensor
    cores (the DANBO field's backward is: mlp_bwd_tcgen05.cu)."""
    dev = d_raw.device
    W, VW, XD, XV = 448, 224, 432, 648
    n_rays = rows // S
    rc = _RowCount(rows, dev)
    rcr = _RowCount(n_rays, dev)
    f32 = lambda *s: torch.empty(*s, device=dev, dtype=torch.float32)
    act = lambda L: anerf_untile(save, 9 * ANERF_ACT_TILE_BYTES, rows, 7, byte_offset=L * ANERF_ACT_TILE_BYTES)
    xd_r = anerf_untile(xd, 7 * 16384, rows, 7)
    xv_r = anerf_untile(xv, 11 * 16384, rows, 11)
    Wv, Wf = f32c(P["views_linears.0.weight"]), f32c(P["feature_linear.weight"])
    WvT = Wv.t().contiguous()                                        # (1224, 224): the forward product needs B = W^T
    feat, a7 = act(8), act(7)
    # view layer pre-activation, recomputed: z9 = feat . Wv[:, :448]^T + xv . Wv[:, 448:1096]^T + code_bias[ray]
    z9 = code_bias[:n_rays].repeat_interleave(S, dim=0).contiguous()
    _dgrad(feat, WvT, VW, z9, VW, rc, VW, W, accumulate=True)
    _dgrad(xv_r, _Ptr(WvT.view(-1), W * VW), VW, z9, VW, rc, VW, XV, accumulate=True)
    g = torch.relu(z9)
    # rgb head
    d9 = f32(rows, VW)
    _dgrad(_Ptr(d_raw.view(-1), 0, ld=4), f32c(P["rgb_linear.weight"]), VW, d9, VW, rc, VW, 3, mask=z9.to(torch.bfloat16))
    dXd = dXv = None
    if want_dx:
        dXv = f32(rows, XV)
        with _Timed("anerf_mlp_dx"):
            _dgrad(d9, _Ptr(Wv.view(-1), W), W + XV + 128, dXv, XV, rc, XV, VW)
    _wgrad(_Ptr(d_raw.view(-1), 0, ld=4), g, G["rgb_linear.weight"], VW, rc, 3, VW)
    _colsum(_Ptr(d_raw.view(-1), 0, ld=4), G["rgb_linear.bias"], rc, 3)
    # view layer: weights of the feature / direction / frame-code column blocks, bias, frame codes
    GWv = G["views_linears.0.weight"]
    _wgrad(d9, feat, GWv, W + XV + 128, rc, VW, W)
    _wgrad(d9, xv_r, _Ptr(GWv.view(-1), W), W + XV + 128, rc, VW, XV)
    d_cb = d9.view(n_rays, S, VW).sum(1).contiguous()                # the code / bias part is per ray
    code_rows = codes_with_mean[cam_idx[:n_rays].long()].contiguous()
    _wgrad(d_cb, code_rows, _Ptr(GWv.view(-1), W + XV), W + XV + 128, rcr, VW, 128)
    _colsum(d_cb, G["views_linears.0.bias"], rcr, VW)
    d_code = f32(n_rays, 128)
    _dgrad(d_cb, _Ptr(Wv.view(-1), W + XV), W + XV + 128, d_code, 128, rcr, 128, VW)
    G["framecodes.codes.weight"].index_add_(0, cam_idx[:n_rays].long(), d_code)
    # feature layer (no activation) and the sigma head into d a7
    d_feat = f32(rows, W)
    _dgrad(d9, Wv, W + XV + 128, d_feat, W, rc, W, VW)
    _colsum(d_feat, G["feature_linear.bias"], rc, W)
    _wgrad(d_feat, a7, G["feature_linear.weight"], W, rc, W, W)
    cur, nxt = f32(rows, W), f32(rows, W)
    _dgrad(_Ptr(d_raw.view(-1), 3, ld=4), f32c(P["alpha_linear.weight"]), W, cur, W, rc, W, 1)
    _wgrad(_Ptr(d_raw.view(-1), 3, ld=4), a7, G["alpha_linear.weight"], W, rc, 1, W)
    _colsum(_Ptr(d_raw.view(-1), 3, ld=4), G["alpha_linear.bias"], rc, 1)
    _dgrad(d_feat, Wf, W, cur, W, rc, W, W, accumulate=True, mask=a7)
    a_prev = a7
    for L in range(7, 0, -1):
        Wl = f32c(P[f"pts_linears.{L}.weight"])
        a_in = act(L - 1)
        _colsum(cur, G[f"pts_linears.{L}.bias"], rc, W)
        if L == 5:                                                   # skip layer: input = [xd (432) ; a4 (448)]
            dW = G["pts_linears.5.weight"]
            _wgrad(cur, xd_r, dW, XD + W, rc, W, XD)
            _wgrad(cur, a_in, _Ptr(dW.view(-1), XD), XD + W, rc, W, W)
            _dgrad(cur, _Ptr(Wl.view(-1), XD), XD + W, nxt, W, rc, W, W, mask=a_in)
            if want_dx:
                dXd = f32(rows, XD)
                with _Timed("anerf_mlp_dx"):
                    _dgrad(cur, Wl, XD + W, dXd, XD, rc, XD, W)
        else:
            _wgrad(cur, a_in, G[f"pts_linears.{L}.weight"], W, rc, W, W)
            _dgrad(cur, Wl, W, nxt, W, rc, W, W, mask=a_in)
        cur, nxt = nxt, cur
    _colsum(cur, G["pts_linears.0.bias"], rc, W)
    _wgrad(cur, xd_r, G["pts_linears.0.weight"], XD, rc, W, XD)
    if want_dx:
        with _Timed("anerf_mlp_dx"):
            _dgrad(cur, f32c(P["pts_linears.0.weight"]), XD, dXd, XD, rc, XD, W, accumulate=True)
        return dXd, dXv
    return None


def anerf_embed_bwd(rays, S, z, pose_skts, rays_per_pose, align, ray_enc, tau, d_xd, d_xv, d_skts):
    """d skts (n_poses,24,4,4) += d loss / d skts of one pass's encodings (danbo_anerf_embed_bwd), given the MLP's input
    gradient d_xd (n*S,432), d_xv (n*S,648) and the pass's forward inputs (z (n,S), ray_enc from anerf_ray_encode)."""
    _need_cuda(rays, z, pose_skts, align, ray_enc, d_xd, d_xv, d_skts)
    n = rays.shape[0]
    f32 = torch.float32
    assert rays.dtype == f32 and rays.dim() == 2 and rays.shape[1] >= 6 and rays.stride(1) == 1
    assert z.dtype == f32 and z.shape == (n, S) and z.is_contiguous()
    assert ray_enc.dtype == f32 and ray_enc.shape[0] >= n and ray_enc.shape[1] == 648 and ray_enc.is_contiguous()
    assert pose_skts.dtype == f32 and pose_skts.shape[1:] == (24, 4, 4) and pose_skts.is_contiguous()
    assert align.dtype == f32 and align.shape == (24, 4, 4) and align.is_contiguous()
    assert d_xd.dtype == f32 and d_xv.dtype == f32
    assert d_xd.shape == (n * S, 432) and d_xv.shape == (n * S, 648) and d_xd.is_contiguous() and d_xv.is_contiguous()
    assert d_skts.shape == pose_skts.shape and d_skts.dtype == torch.float32 and d_skts.is_contiguous()
    with _Timed("anerf_embed_bwd"):
        _lib.check(_lib.load().danbo_anerf_embed_bwd(_p(rays), rays.stride(0), n, int(S), _p(z), _p(pose_skts),
                                                     int(rays_per_pose), pose_skts.shape[0], _p(align), _p(ray_enc),
                                                     float(tau), _p(d_xd), _p(d_xv), _p(d_skts), _stream()),
                   "danbo_anerf_embed_bwd")
    _count(1)
    return d_skts
