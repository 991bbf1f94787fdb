"""Shared helpers for the parity tests: fixture loading and parameter rebuilding."""
import contextlib
import os

import numpy as np
import torch

import danbo_b200  # noqa: F401
from danbo_b200 import skeleton as sk, synthetic as syn

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_fixture(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False)
    out = {}
    for k in z.files:
        v = z[k]
        out[k] = torch.from_numpy(v) if v.dtype.kind in "fiub" and v.ndim > 0 else v.item() if v.ndim == 0 else v
    return out


def params_for(fx):
    return syn.synthetic_params(int(fx["weight_seed"]), opt_framecode=bool(int(fx.get("opt_framecode", 1))))


def config_flags_of(fx):
    """Flags (beyond the preset) of the shipped config a fixture was rendered with: perfcap's root-local view
    directions, surreal's missing frame codes."""
    cfg = str(fx.get("config", ""))
    flags = {}
    if "perfcap" in cfg:
        flags.update(view_type="relray", ray_tr_type="root_local", nerf_type="graph")
    if not int(fx.get("opt_framecode", 1)):
        flags.update(opt_framecode=False, loss_fn="MSE")
    return flags


def align_A():
    A, _ = sk.bone_align_transforms(syn.rest_pose())
    return torch.from_numpy(A)


def pose_tensors(fx):
    return (fx["pose_skts"][None] if fx["pose_skts"].dim() == 3 else fx["pose_skts"],
            fx["pose_bones"][None] if fx["pose_bones"].dim() == 2 else fx["pose_bones"],
            fx["pose_cyl"][None] if fx["pose_cyl"].dim() == 1 else fx["pose_cyl"])


def mask_mismatch_report(x, got_invalid, want_invalid, ulps=16):
    """Bone-visibility masks are a bit-exact target except where |x| sits within a few ulp of the box face.
    Returns (#mismatches, #mismatches explained by the margin)."""
    bad = got_invalid != want_invalid
    n_bad = int(bad.sum())
    if n_bad == 0:
        return 0, 0
    margin = (x.abs() - 1.0).abs().min(-1).values            # distance of the closest coordinate to a face
    near = margin <= ulps * 1.1920929e-07
    return n_bad, int((bad & near).sum())


# ---------------------------------------------------------------------------------------------------- GPU helpers
def sw128_offsets(n_cols=208):
    """Byte offsets of (row r, col k) inside one 64 KB X tile, mirroring csrc/common.cuh::sw128_offset."""
    r = np.arange(128)[:, None]
    k = np.arange(n_cols)[None, :]
    chunk, kk = k >> 6, k & 63
    return chunk * (128 * 128) + (r >> 3) * 1024 + (r & 7) * 128 + (((kk >> 3) ^ (r & 7)) << 4) + ((kk & 7) << 1)


def decode_xtiles(xtiles, n_rows, n_cols=195):
    """uint8 tile buffer -> float32 (n_rows, n_cols) matrix of the bf16 rows the field kernel wrote."""
    off = torch.from_numpy(sw128_offsets(208).astype(np.int64)).to(xtiles.device)        # (128,208)
    n_tiles = (n_rows + 127) // 128
    words = xtiles[: n_tiles * 65536].view(torch.int16).view(n_tiles, 32768)
    idx = (off // 2).reshape(1, -1).expand(n_tiles, -1)
    vals = torch.gather(words, 1, idx).reshape(n_tiles * 128, 208)
    return vals.view(torch.bfloat16).float()[:n_rows, :n_cols]


def make_caster(preset, weight_seed=0, device="cuda", train=False, **flags):
    import danbo_b200 as db
    args = db.make_args(preset, no_reload=True, **flags)
    data_attrs = {"skel_type": sk.SMPLSkeleton, "near": syn.NEAR, "far": syn.FAR, "n_views": 8,
                  "rest_pose": syn.rest_pose()}
    kw_train, kw_test, *_ = db.create_raycaster(args, data_attrs, device=device)
    caster = kw_test["ray_caster"]
    P = syn.synthetic_params(weight_seed, opt_framecode=bool(getattr(args, "opt_framecode", True)))
    caster.network.load_state_dict(P)
    caster.train(train)
    return caster, args, {k: v.to(device) for k, v in P.items()}


def agg_type_of(fx):
    """Aggregation type of a fixture (`--agg_type softmax` in its extra flags; the configs ship sigmoid)."""
    return "softmax" if "agg_type softmax" in str(fx.get("extra", "")) else "sigmoid"


def view_mode_of(fx):
    """"root_local" for fixtures of the perfcap configs (ray_tr_type=root_local, view_type=relray), else "world"."""
    return "root_local" if "perfcap" in str(fx.get("config", "")) else "world"


def lindisp_of(fx):
    return "--lindisp" in str(fx.get("extra", ""))


def preset_of(fx):
    cfg = str(fx["config"])
    if "fast" in cfg:
        return "danbo_fast"
    return "danbo_cfg3" if "N_samples 64" in str(fx.get("extra", "")) else "danbo_base"


def mlp_bf16_reference(x, view_bias, P, bf=None):
    """The fused kernel's arithmetic restated in torch: bf16 operands, fp32 accumulation, activations rounded to
    bf16 where the kernel writes them back to tensor memory; sigma and rgb heads in fp32.  bf: the rounding applied to
    operands and stored activations (default bf16 round-to-nearest-even returned as fp32)."""
    if bf is None:
        bf = lambda t: t.to(torch.bfloat16).float()
    xb = bf(x)
    h = xb
    a = None
    for i in range(8):
        W = bf(P[f"pts_linears.{i}.weight"])
        a = torch.relu(h @ W.t() + P[f"pts_linears.{i}.bias"])
        h = bf(a)
        if i == 4:
            h = torch.cat([xb, h], -1)
    sigma = a @ P["alpha_linear.weight"].t() + P["alpha_linear.bias"]
    feat = bf(h @ bf(P["feature_linear.weight"]).t() + P["feature_linear.bias"])
    g = torch.relu(feat @ bf(P["views_linears.0.weight"][:, :256]).t() + view_bias)
    rgb = g @ P["rgb_linear.weight"].t() + P["rgb_linear.bias"]
    return torch.cat([rgb, sigma], -1)


def decode_tile_image(buf, n_rows, n_chunks, n_cols):
    """uint8 operand tile images ([tile][chunk][128 rows x 64 k] bf16, 128B-swizzled) -> float32 (n_rows, n_cols)."""
    off = torch.from_numpy(sw128_offsets(n_chunks * 64).astype(np.int64)).to(buf.device)
    n_tiles = (n_rows + 127) // 128
    tile_bytes = n_chunks * 16384
    words = buf[: n_tiles * tile_bytes].view(torch.int16).view(n_tiles, tile_bytes // 2)
    idx = (off // 2).reshape(1, -1).expand(n_tiles, -1)
    vals = torch.gather(words, 1, idx).reshape(n_tiles * 128, n_chunks * 64)
    return vals.view(torch.bfloat16).float()[:n_rows, :n_cols]


def anerf_mlp_bf16_reference(xd, xv, code_bias, P):
    """The A-NeRF kernel's arithmetic restated in torch: bf16 operands and stored activations, fp32 accumulation,
    sigma / rgb heads in fp32 from the unrounded last activations."""
    bf = lambda t: t.to(torch.bfloat16).float()
    xb = bf(xd)
    h, a = xb, None
    for i in range(8):
        a = torch.relu(h @ bf(P[f"pts_linears.{i}.weight"]).t() + P[f"pts_linears.{i}.bias"])
        h = bf(a)
        if i == 4:
            h = torch.cat([xb, h], -1)
    sigma = a @ P["alpha_linear.weight"].t() + P["alpha_linear.bias"]
    feat = bf(h @ bf(P["feature_linear.weight"]).t() + P["feature_linear.bias"])
    Wv = P["views_linears.0.weight"]
    g = torch.relu(feat @ bf(Wv[:, :448]).t() + bf(xv) @ bf(Wv[:, 448:448 + 648]).t() + code_bias)
    rgb = g @ P["rgb_linear.weight"].t() + P["rgb_linear.bias"]
    return torch.cat([rgb, sigma], -1)


def pixel_parity(caster, fx, kw, name, dev="cuda"):
    """Rendered pixels against the reference fixture, with the coarse -> fine coupling accounted for.

    The fine pass places its samples by inverse-CDF sampling of the coarse weights (ray_utils.py:140-204), which is
    ill-conditioned where the coarse pdf is flat: a bf16-sized change of the coarse weights moves importance samples by
    up to a few per cent of the ray span, and the random-init field differs there.  So the comparison is made twice:
      (a) with the fine pass evaluated at the REFERENCE's importance samples (test hook `_rand[z_fine]`): visibility masks
          must be bit-identical, the merged raw values within the bf16 MLP tolerance, every pixel within 1.5e-2 and at most
          5 % of the rays above 5e-3 (this is the stated pixel tolerance of the bf16 path; measured 0 - 4 %);
      (b) free-running: every ray above 5e-3 must be EXPLAINED - its importance samples moved by >= 5e-4 of the ray span,
          or it already exceeds 2.5e-3 in (a).  Unexplained outliers fail.  -> dict of the measured numbers."""
    import torch
    N = fx["ray_batch"].shape[0]
    st_free, st_inj = {}, {}
    free = caster(fx["ray_batch"], _stages=st_free, **kw)
    inj = caster(fx["ray_batch"], _stages=st_inj, **kw,
                 _rand={"z_fine": fx["st.z_samples.0"].to(dev), "z_all": fx["st.z_all.0"].to(dev),
                        "order": fx["st.sorted_idxs.0"].to(dev)})
    torch.cuda.synchronize()
    err = lambda o, k: (o[k].cpu() - fx["out." + k]).abs().reshape(N, -1).max(-1).values
    span = (fx["st.far.0"] - fx["st.near.0"]).reshape(N).clamp_min(1e-6)
    # (a)
    invalid_inj = ((st_inj["mask1"].cpu().long()[..., None] >> torch.arange(24)) & 1) == 0
    assert torch.equal(invalid_inj, fx["st.invalid.1"] != 0), "fine-pass visibility masks at the reference's samples"
    scale = float(fx["st.raw.1"].abs().max())
    raw_err = float((st_inj["raw"].cpu() - fx["st.raw.1"]).abs().max())
    assert raw_err <= 3e-2 * scale, (raw_err, scale)
    rep = {"raw_err_of_scale": raw_err / scale}
    for k in ("rgb0", "acc0", "rgb_map", "acc_map"):
        e = err(inj, k)
        rep[k + "@ref_samples"] = (float(e.mean()), float(e.max()), int((e > 5e-3).sum()))
        assert float(e.max()) <= 1.5e-2 and float(e.mean()) <= 1e-3 and int((e > 5e-3).sum()) <= max(2, N // 20), (name, k, rep)
    # (b)
    shift = (st_free["z_samples"].cpu() - fx["st.z_samples.0"]).abs().max(-1).values / span
    for k in ("rgb_map", "acc_map"):
        e = err(free, k)
        big = e > 5e-3
        explained = (shift >= 5e-4) | (err(inj, k) > 2.5e-3)
        rep[k] = (float(e.mean()), float(e.max()), int(big.sum()), int((big & ~explained).sum()))
        assert float(e.mean()) <= 4e-3 and float(e.max()) <= 0.2, (name, k, rep)
        assert not bool((big & ~explained).any()), (name, k, "unexplained outliers", rep)
    print(f"[pixels] {name}: " + "  ".join(f"{k} {v}" for k, v in rep.items()))
    return rep


def field_mlp_bf16_ste(x, view, P):
    """`danbo_oracle.field_mlp` with the CUDA kernel's operand rounding (see mlp_bf16_reference) made differentiable by a
    straight-through estimator: forward values are those of the bf16 tensor-core kernel, the backward is fp32 calculus on
    them.  Passed as `mlp_fn` to the oracle, it splits an end-to-end gradient difference into "the declared bf16
    arithmetic of the forward pass" and "anything else" (which must then be at rounding level)."""
    import torch
    bf = lambda t: t + (t.to(torch.bfloat16).float() - t).detach()
    xb = bf(x)
    h, a = xb, None
    for i in range(8):
        a = torch.relu(h @ bf(P[f"pts_linears.{i}.weight"]).t() + P[f"pts_linears.{i}.bias"])
        h = bf(a)
        if i == 4:
            h = torch.cat([xb, h], -1)
    sigma = a @ P["alpha_linear.weight"].t() + P["alpha_linear.bias"]
    feat = bf(h @ bf(P["feature_linear.weight"]).t() + P["feature_linear.bias"])
    Wv = P["views_linears.0.weight"]
    g = torch.relu(feat @ bf(Wv[:, :256]).t() + view @ Wv[:, 256:].t() + P["views_linears.0.bias"])
    rgb = g @ P["rgb_linear.weight"].t() + P["rgb_linear.bias"]
    return torch.cat([rgb, sigma], -1)


def reference_core(tmp_path):
    """-> a directory holding the reference's `core/` and `run_nerf.py`: the reference itself when a copy is given
    ($DANBO_REFERENCE or the vendored baseline/_ref), else a stand-in with just the seam the drop-in hook works on - a
    `core.raycasters` that defines `create_raycaster` and a `run_nerf` that copies the name (run_nerf.py:20)."""
    import ref_harness as rh
    if rh.available():
        return rh.REF
    root = tmp_path / "stand_in"
    (root / "core").mkdir(parents=True)
    (root / "core" / "__init__.py").write_text("")
    (root / "core" / "raycasters.py").write_text(
        "import os\n\nRAY_CHUNK = 4096\n\n\ndef create_raycaster(args, data_attrs, device=None):\n"
        "    raise AssertionError('the stand-in factory must not be called')\n")
    (root / "run_nerf.py").write_text("from core.raycasters import create_raycaster\n")
    return str(root)


@contextlib.contextmanager
def reference_modules(tmp_path):
    """-> (core.raycasters, run_nerf) of the reference copy when one is given, else of the `reference_core` stand-in.
    The stand-in's modules and path entry are gone again on exit, and modules of those names that were loaded
    before are put back."""
    import importlib
    import sys
    import ref_harness as rh
    if rh.available():
        yield rh._imports()
        return
    root = reference_core(tmp_path)
    names = ("core", "core.raycasters", "run_nerf")
    saved = {n: sys.modules.pop(n) for n in names if n in sys.modules}
    sys.path.insert(0, root)
    try:
        yield importlib.import_module("core.raycasters"), importlib.import_module("run_nerf")
    finally:
        sys.path.remove(root)
        for n in names:
            sys.modules.pop(n, None)
        sys.modules.update(saved)


# ------------------------------------------------------------ layer-local fp64 oracle of the tcgen05 MLP kernels
# Every stage of the fused MLP (forward, dgrad chain, K = rows weight gradients) consumes bf16 operands that the kernels
# also save (act_save, g_save, the delta planes, x_rows) and bf16-RN weights.  A stage is therefore checked on its own:
# fp64 of exactly those operands, never of an earlier stage's reference, so that nothing propagates between layers.
# Each reference is (r, s, K): the fp64 value, the sum of the magnitudes of its terms and the accumulation length.
#
# Bounds (per entry), with u = 2^-8 the unit roundoff of bf16 (8-bit significand: |x - bf16_rn(x)| <= 2^-8 |x|) and
# gamma = K * 2^-22, 4x the IEEE fp32 worst case K * 2^-24 (tensor-core accumulation order and alignment are not
# IEEE-specified):
#   bf16 outputs      |got - r| <= u |r| + 2 gamma s    (the fp32 sum is within gamma s of r, its bf16 rounding within
#                                                         u |sum| <= u |r| + u gamma s of the sum; 2 gamma covers both)
#   fp32, small K     |got - r| <= 2 gamma s
#   K = rows sums     the fp32 per-entry bound, and ||got - r|| <= 1e-5 ||r - prefill||: the per-entry bound grows with
#                     the row count, the norm bound does not; one dropped 64-row block of 40 000 rows moves dW by ~1e-3.
# A gated entry (relu of the saved activation <= 0) has r = s = 0, so the kernel must write exactly 0 there.
# bf16 outputs must also be correctly rounded (a nearest bf16 of r; either neighbour at a tie) on at least
# MIN_NEAREST_BF16 of their non-zero entries: a consistent 1-ulp bias on 5 % of them fails that.
BF16_U = 2.0 ** -8
GAMMA_PER_K = 2.0 ** -22
REDUCTION_REL = 1e-5
MIN_NEAREST_BF16 = 0.98         # measured on a B200: 0.9961 for one row (1 of 256 entries), >= 0.9995 for more rows
MLP_LAYERS = [f"pts_linears.{i}" for i in range(8)] + ["feature_linear", "views_linears.0"]


def random_mlp_params(seed, width=256, n_x=195, n_view=411):
    """fp32 (CPU) parameters of the field MLP in the reference's names, scaled so that activations stay O(1).  The
    A-NeRF MLP is width 448, n_x 432, n_view 1224 (its view layer is 224 wide)."""
    g = torch.Generator().manual_seed(seed)
    r = lambda *s: torch.randn(*s, generator=g)
    P = {}
    for i in range(8):
        n_in = n_x if i == 0 else n_x + width if i == 5 else width
        P[f"pts_linears.{i}.weight"] = r(width, n_in) * (2.0 / n_in) ** 0.5
        P[f"pts_linears.{i}.bias"] = r(width) * 0.1
    vw = width // 2
    P["alpha_linear.weight"], P["alpha_linear.bias"] = r(1, width) / 16, r(1)
    P["feature_linear.weight"], P["feature_linear.bias"] = r(width, width) / 16, r(width) * 0.1
    P["views_linears.0.weight"], P["views_linears.0.bias"] = r(vw, n_view) * (2.0 / n_view) ** 0.5, r(vw) * 0.1
    P["rgb_linear.weight"], P["rgb_linear.bias"] = r(3, vw) / vw ** 0.5, r(3)
    return P


def bf16_rn(t):
    """bf16 round-to-nearest-even of t, returned in t's dtype."""
    return t.to(torch.bfloat16).to(t.dtype)


def mlp_bf16_weights(P, dtype=torch.float64):
    """The operands the packs hand the tensor cores: bf16-RN matrices of the ten MMA layers (danbo_pack_mlp_weights,
    danbo_pack_mlp_dgrad), fp32 biases and head weights, all widened to `dtype`."""
    W = {}
    for n in MLP_LAYERS:
        W[n + ".weight"] = bf16_rn(P[n + ".weight"].float()).to(dtype)
        if n != "views_linears.0":
            W[n + ".bias"] = P[n + ".bias"].float().to(dtype)
    for n in ("alpha_linear.weight", "alpha_linear.bias", "rgb_linear.weight", "rgb_linear.bias"):
        W[n] = P[n].float().to(dtype)
    return W


def lin_ref(parts, bias=None):
    """parts: [(input (n,k), weight (m,k))] -> (r, s, K) of sum_i input_i . weight_i^T (+ bias)."""
    r = sum(a @ w.t() for a, w in parts)
    s = sum(a.abs() @ w.abs().t() for a, w in parts)
    K = sum(a.shape[1] for a, _ in parts)
    if bias is not None:
        r, s, K = r + bias, s + bias.abs(), K + 1
    return r, s, K


def _gate(ref, act):
    r, s, K = ref
    keep = (act > 0).to(r.dtype)
    return r * keep, s * keep, K


def fwd_plane_ref(L, x, acts, W, rbias_rows=None):
    """Layer-local reference of forward plane L: 0..7 = pts_linears.L after relu, 8 = feature_linear, 9 = relu of the
    view layer (g_save; rbias_rows = the fp32 per-ray part of each row).  x (n,195) and acts[0..L-1] are the bf16
    values the kernel consumed.  -> (r, s, K)."""
    if L == 0:
        parts = [(x, W["pts_linears.0.weight"])]
    elif L == 5:
        W5 = W["pts_linears.5.weight"]
        parts = [(x, W5[:, :195]), (acts[4], W5[:, 195:])]
    elif L < 9:
        parts = [(acts[L - 1], W[f"{MLP_LAYERS[L]}.weight"])]
    else:
        r, s, K = lin_ref([(acts[8], W["views_linears.0.weight"][:, :256])], rbias_rows)
        return r.clamp_min(0), s, K
    r, s, K = lin_ref(parts, W[f"{MLP_LAYERS[L]}.bias"])
    return (r.clamp_min(0) if L < 8 else r), s, K


def head_refs(a7, g, W):
    """sigma = w_alpha . a7 + b_alpha and rgb = W_rgb . g + b_rgb from the saved bf16 planes -> {name: (r, bound)}.
    The kernel forms both heads from its fp32 activations, which it never saves: the bound adds their bf16 rounding,
    1.01 u sum |w a|, to the fp32 accumulation bound."""
    out = {}
    for name, a, w, b in (("sigma", a7, W["alpha_linear.weight"], W["alpha_linear.bias"]),
                          ("rgb", g, W["rgb_linear.weight"], W["rgb_linear.bias"])):
        r, s, K = lin_ref([(a, w)], b)
        prod = a.abs() @ w.abs().t()
        out[name] = (r, 1.01 * BF16_U * prod + 2 * (K + 4) * GAMMA_PER_K * s)
    return out


def delta9_ref(g_out, g_save, W):
    """Delta plane 0 (views_linears.0, 128 wide) = (d rgb . W_rgb) [g > 0], from the fp32 d raw rows -> (r, s, K)."""
    return _gate(lin_ref([(g_out[:, :3], W["rgb_linear.weight"].t())]), g_save)


# dgrad planes 1..9: (weight and its column slice, relu-gate activation plane or None); plane p reads plane p-1
_DGRAD = {1: ("views_linears.0", slice(0, 256), None), 2: ("feature_linear", slice(None), 7),
          3: ("pts_linears.7", slice(None), 6), 4: ("pts_linears.6", slice(None), 5),
          5: ("pts_linears.5", slice(195, 451), 4), 6: ("pts_linears.4", slice(None), 3),
          7: ("pts_linears.3", slice(None), 2), 8: ("pts_linears.2", slice(None), 1), 9: ("pts_linears.1", slice(None), 0)}


def dgrad_plane_ref(p, D, acts, g_out, W, sigma_term=True, gate_plane=None):
    """Layer-local reference of delta plane p (1..9) from the saved plane p-1: D[p-1] . bf16(W)[:, cols], plus the
    sigma head's d sigma w_alpha in plane 2, gated by the saved activation named in _DGRAD.  sigma_term / gate_plane
    exist to plant errors in the predicate tests.  -> (r, s, K)."""
    name, cols, gate = _DGRAD[p]
    parts = [(D[p - 1], W[name + ".weight"][:, cols].t())]
    if p == 2 and sigma_term:
        parts.append((g_out[:, 3:4], W["alpha_linear.weight"].t()))
    ref = lin_ref(parts)
    gate = gate if gate_plane is None else gate_plane
    return ref if gate is None else _gate(ref, acts[gate])


def dx_ref(D, W):
    """dX (n,195) = D[4] . bf16(W5)[:, :195] + D[9] . bf16(W0) (dgrad stages 4 and 10) -> (r, s, K)."""
    return lin_ref([(D[4], W["pts_linears.5.weight"][:, :195].t()), (D[9], W["pts_linears.0.weight"].t())])


# weight gradients (K = rows): (destination, column slice, delta plane, input: activation plane index or "x")
WGRAD_ITEMS = [("views_linears.0.weight", slice(0, 256), 0, 8), ("feature_linear.weight", slice(None), 1, 7),
               ("pts_linears.7.weight", slice(None), 2, 6), ("pts_linears.6.weight", slice(None), 3, 5),
               ("pts_linears.5.weight", slice(0, 195), 4, "x"), ("pts_linears.5.weight", slice(195, 451), 4, 4),
               ("pts_linears.4.weight", slice(None), 5, 3), ("pts_linears.3.weight", slice(None), 6, 2),
               ("pts_linears.2.weight", slice(None), 7, 1), ("pts_linears.1.weight", slice(None), 8, 0),
               ("pts_linears.0.weight", slice(None), 9, "x")]
BIAS_ITEMS = [("feature_linear.bias", 1)] + [(f"pts_linears.{7 - i}.bias", 2 + i) for i in range(8)]


def wgrad_refs(D, acts, x):
    """D: the ten delta planes (plane 0 is 128 wide) -> [(name, cols, (r, s, K))] of dW[:, cols] = D^T . input and
    [(name, (r, s, K))] of db = column sums."""
    w = []
    for name, cols, p, src in WGRAD_ITEMS:
        a = x if src == "x" else acts[src]
        w.append((name, cols, (D[p].t() @ a, D[p].t().abs() @ a.abs(), D[p].shape[0])))
    b = [(name, (D[p].sum(0), D[p].abs().sum(0), D[p].shape[0])) for name, p in BIAS_ITEMS]
    return w, b


def head_bwd_refs(g_out, g_save, a7, row_ray, n_rays, W):
    """Heads of the backward (danbo_mlp_head_bwd): rgb / alpha weight and bias gradients and d ray_bias (n_rays,128),
    scattered by row_ray -> {name: (r, s, K)} (K = rows, or 3 + rows for d ray_bias)."""
    n = g_out.shape[0]
    out = {"rgb_linear.weight": (g_out[:, :3].t() @ g_save, g_out[:, :3].t().abs() @ g_save.abs(), n),
           "rgb_linear.bias": (g_out[:, :3].sum(0), g_out[:, :3].abs().sum(0), n),
           "alpha_linear.weight": (g_out[:, 3:4].t() @ a7, g_out[:, 3:4].t().abs() @ a7.abs(), n),
           "alpha_linear.bias": (g_out[:, 3].sum(0, keepdim=True), g_out[:, 3].abs().sum(0, keepdim=True), n)}
    r, s, _ = delta9_ref(g_out, g_save, W)
    idx = row_ray.long()
    zr = torch.zeros(n_rays, 128, dtype=r.dtype, device=r.device)
    out["d_ray_bias"] = (zr.index_add(0, idx, r), zr.index_add(0, idx, s), 3 + n)
    return out


def _where(bad):
    i = int(bad.reshape(-1).nonzero()[0])
    return tuple(int(v) for v in np.unravel_index(i, tuple(bad.shape))) if bad.dim() else ()


def nearest_bf16_fraction(got, r):
    """Fraction of the non-zero entries of r whose got is a nearest bf16 of r (either neighbour at an exact tie)."""
    nz = r != 0
    if not bool(nz.any()):
        return 1.0
    _, e = torch.frexp(r[nz])                                # |r| in [2^(e-1), 2^e): bf16 spacing 2^(e-8)
    half_ulp = torch.ldexp(torch.ones_like(r[nz]), (e - 9).to(torch.int32))
    return float(((got[nz] - r[nz]).abs() <= half_ulp).double().mean())


def check_bf16(name, got, ref, min_nearest=MIN_NEAREST_BF16):
    """bf16 output against its layer-local reference: the per-entry bound and the correct-rounding fraction.
    -> (max error / bound, nearest fraction)."""
    r, s, K = ref
    got = got.to(r.dtype)
    bound = BF16_U * r.abs() + 2 * K * GAMMA_PER_K * s
    err = (got - r).abs()
    bad = ~(err <= bound)
    assert not bool(bad.any()), (f"{name}: {int(bad.sum())} of {bad.numel()} entries outside the bound, first at "
                                 f"{_where(bad)}: got {float(got[bad][0]):.6e} want {float(r[bad][0]):.6e}")
    near = nearest_bf16_fraction(got, r)
    assert near >= min_nearest, f"{name}: only {near:.4f} of the entries are correctly rounded (>= {min_nearest})"
    return float((err / bound.clamp_min(1e-300)).max()) if err.numel() else 0.0, near


def check_fp32(name, got, ref, bound=None):
    """fp32 output against its reference: |got - r| <= 2 gamma s per entry (or the given bound).  -> max error / bound."""
    r, s, K = ref
    got = got.to(r.dtype)
    if bound is None:
        bound = 2 * K * GAMMA_PER_K * s
    err = (got - r).abs()
    bad = ~(err <= bound)
    assert not bool(bad.any()), (f"{name}: {int(bad.sum())} of {bad.numel()} entries outside the bound, first at "
                                 f"{_where(bad)}: got {float(got[bad][0]):.6e} want {float(r[bad][0]):.6e}")
    return float((err / bound.clamp_min(1e-300)).max()) if err.numel() else 0.0


def check_reduction(name, got, ref, prefill):
    """K = rows reduction added to `prefill`: the per-entry fp32 bound on prefill + r, and ||got - (prefill + r)|| <=
    REDUCTION_REL ||r||.  -> (max error / bound, relative norm error)."""
    r, s, K = ref
    pre = prefill.to(r.dtype)
    ratio = check_fp32(name, got, (pre + r, pre.abs() + s, K + 1))
    rn = float(r.norm())
    rel = float((got.to(r.dtype) - pre - r).norm()) / rn if rn > 0 else float((got.to(r.dtype) - pre).norm())
    assert rel <= REDUCTION_REL, f"{name}: relative error {rel:.3e} > {REDUCTION_REL:.0e}"
    return ratio, rel


def encode_tile_image(vals, n_chunks):
    """Row-major (n_rows, <= 64 n_chunks) values -> uint8 operand tile images ([tile][chunk][128 rows x 64 k] bf16,
    128B-swizzled; the inverse of decode_tile_image).  Missing columns and rows of the last tile are zero."""
    n_rows = vals.shape[0]
    n_tiles = max((n_rows + 127) // 128, 1)
    full = torch.zeros(n_tiles * 128, n_chunks * 64, dtype=torch.bfloat16, device=vals.device)
    full[:n_rows, :vals.shape[1]] = vals.to(torch.bfloat16)
    off = torch.from_numpy(sw128_offsets(n_chunks * 64).astype(np.int64)).to(vals.device)
    buf = torch.zeros(n_tiles * n_chunks * 16384, dtype=torch.uint8, device=vals.device)
    words = buf.view(torch.int16).view(n_tiles, -1)
    words.scatter_(1, (off // 2).reshape(1, -1).expand(n_tiles, -1), full.view(torch.int16).reshape(n_tiles, -1))
    return buf
