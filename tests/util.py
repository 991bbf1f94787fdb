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


def mlp_bf16_reference(x, view_bias, P):
    """The fused kernel's arithmetic restated in torch: bf16 operands, fp32 accumulation, activations rounded to
    bf16 where the kernel writes them back to tensor memory; sigma and rgb heads in fp32."""
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
