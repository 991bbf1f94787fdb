"""Body-part maps of the DANBO field on the GPU (danbo_merge_composite_parts, RayCaster.render_rays(want_parts=True),
render_pts_parts, render_images(parts=True), part-coloured meshes of render_mesh(parts=True)) with both aggregation
types, against the oracle and against what the plain calls produce.  Measured numbers are printed."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)
import danbo_oracle as orc                           # noqa: E402
from danbo_b200 import kernels as K, mesh, raycaster, render, synthetic as syn   # noqa: E402
from util import (agg_type_of, align_A, lindisp_of, load_fixture, make_caster, mask_mismatch_report,  # noqa: E402
                  params_for, pose_tensors, preset_of)

pytestmark = pytest.mark.gpu
DEV = "cuda"
AGG = ["sigmoid", "softmax"]
FIXTURE = {"sigmoid": "render_fast", "softmax": "render_fast_softmax"}
# launches of one eval render_rays block of one pose once the weights are packed (the parent commit's sequence):
# field constants 1, graph net 4, nearfar 2, ray_bias 2, empty rows 1, per pass sample_mask 1 + field_agg 4 + mlp 1,
# composite_resample 1, merge 1
PLAIN_EVAL_LAUNCHES = 24


@pytest.fixture(autouse=True)
def _keep_global_rng():
    """Building a caster draws from torch's global generators (module initialisation): restore them, so that tests
    which run later in the same process see the random streams they would see without this module."""
    cpu, cuda = torch.get_rng_state(), torch.cuda.get_rng_state_all()
    yield
    torch.set_rng_state(cpu)
    torch.cuda.set_rng_state_all(cuda)


def _bits(mask):
    return ((mask.long()[..., None] >> torch.arange(24, device=mask.device)) & 1).bool()


def _image(agg_type, seed=3, H=64):
    caster, args, P = make_caster("danbo_fast", agg_type=agg_type)
    caster.eval()
    pose = syn.make_pose(seed)
    b = syn.render_batch(pose, H, H)
    kw = dict(N_samples=args.N_samples, kp_batch=b["kp_batch"], skts=b["skts"], cyls=b["cyls"], bones=b["bones"],
              cams=b["cams"], N_uniques=1, perturb=False, N_importance=args.N_importance, raw_noise_std=0.,
              nanmean_chunk=args.chunk)
    return caster, args, pose, b, kw


@pytest.mark.parametrize("agg_type", AGG)
def test_part_map_against_oracle(agg_type):
    """part_map at the oracle's own importance samples (the `_rand` z_fine hook of util.pixel_parity) against
    sum_m w_m get_agg(confd_m, part_invalid_m) built from the oracle's train-mode outputs (no perturbation, no noise).
    The merged visibility must be bit-identical; per ray, max_j |diff| is held to the bounds pixel_parity applies to
    acc_map: max 1.5e-2, mean 1e-3, at most 5 % of the rays above 5e-3 (both are weighted sums of the same weights)."""
    fx = load_fixture(FIXTURE[agg_type])
    assert agg_type_of(fx) == agg_type
    caster, args, P = make_caster(preset_of(fx), agg_type=agg_type, lindisp=lindisp_of(fx))
    caster.eval()
    skts, bones, cyl = pose_tensors(fx)
    N = fx["ray_batch"].shape[0]
    ex = lambda t: t.expand(N, *t.shape[1:])
    kw = dict(N_samples=args.N_samples, kp_batch=ex(fx["pose_kps"][None]), skts=ex(skts), cyls=ex(cyl), bones=ex(bones),
              cams=fx["cams"], N_uniques=1, perturb=False, N_importance=args.N_importance, raw_noise_std=0.,
              lindisp=args.lindisp)
    st = {}
    with torch.no_grad():
        ret = caster.render_rays(fx["ray_batch"], want_parts=True, _stages=st, **kw,
                                 _rand={"z_fine": fx["st.z_samples.0"].to(DEV), "z_all": fx["st.z_all.0"].to(DEV),
                                        "order": fx["st.sorted_idxs.0"].to(DEV)})
    torch.cuda.synchronize()
    ref = orc.render_rays(fx["ray_batch"], skts, bones, cyl, fx["cams"], align_A(), params_for(fx), args.N_samples,
                          args.N_importance, N, use_volume_near_far=bool(int(fx["use_volume_near_far"])), training=True,
                          agg_type=agg_type, z_samples=fx["st.z_samples.0"], lindisp=lindisp_of(fx))
    # visibility of the merged samples, bit for bit
    merged = torch.gather(torch.cat([st["mask0"], st["mask1"]], 1), 1, st["sorted_idxs"].long()).cpu()
    assert torch.equal(~_bits(merged), ref["part_invalid"] != 0)
    p = orc.agg_prob(ref["confd"].double(), ref["part_invalid"].double(), agg_type)
    want = (ref["T_i"].double()[..., None] * p).sum(1)
    got = ret["part_map"].double().cpu()
    e = (got - want).abs().max(-1).values
    e_acc = (ret["acc_map"].double().cpu() - ref["acc_map"].double()).abs()
    print(f"[parts] {agg_type}: part_map vs oracle per ray max |diff| max {float(e.max()):.3e} mean {float(e.mean()):.3e}, "
          f"{int((e > 5e-3).sum())} of {N} rays above 5e-3 (acc_map: max {float(e_acc.max()):.3e} mean "
          f"{float(e_acc.mean()):.3e}); max part weight {float(want.max()):.3f}")
    # the comparison is not between zeros: the reference's largest weight is 10x the bound held to
    assert float(want.max()) > 10 * 1.5e-2
    assert float(e.max()) <= 1.5e-2 and float(e.mean()) <= 1e-3 and int((e > 5e-3).sum()) <= max(2, N // 20)


@pytest.mark.parametrize("agg_type", AGG)
def test_parts_leave_the_render_unchanged(agg_type):
    """A want_parts call returns the plain call's maps bit for bit, and runs the plain call's launch sequence with the
    merge kernel swapped: the same count, which is the count of the parent commit's eval block."""
    caster, args, pose, b, kw = _image(agg_type)
    with torch.no_grad():
        caster.render_rays(b["ray_batch"], **kw)                        # packs the weights
        K.PROFILE = {"mlp": [], "launches": 0}
        try:
            plain = caster.render_rays(b["ray_batch"], **kw)
            n_plain = K.PROFILE["launches"]
            K.PROFILE["launches"] = 0
            parts = caster.render_rays(b["ray_batch"], want_parts=True, **kw)
            n_parts = K.PROFILE["launches"]
        finally:
            K.PROFILE = None
    print(f"[parts] {agg_type}: launches plain {n_plain}, want_parts {n_parts}")
    assert n_plain == PLAIN_EVAL_LAUNCHES and n_parts == n_plain
    assert set(parts) == set(plain) | {"part_map"}
    for k in plain:
        assert torch.equal(parts[k], plain[k]), k


@pytest.mark.parametrize("agg_type", AGG)
def test_part_map_bounds_and_background(agg_type):
    """Softmax: sum_j part_map <= acc_map + 1e-6; sigmoid: part_map >= -0.001 acc_map - 1e-7.  Rays whose samples no
    bone sees get exactly 0, and so does the background of render_images(parts=True), whose images are the plain
    call's."""
    caster, args, pose, b, kw = _image(agg_type)
    st = {}
    with torch.no_grad():
        ret = caster.render_rays(b["ray_batch"], want_parts=True, _stages=st, **kw)
    pm, acc = ret["part_map"], ret["acc_map"]
    assert pm.shape == (b["ray_batch"].shape[0], 24) and bool(torch.isfinite(pm).all())
    if agg_type == "softmax":
        assert bool((pm.sum(-1) <= acc + 1e-6).all())
    else:
        assert bool((pm >= -0.001 * acc[:, None] - 1e-7).all())
    miss = ((st["mask0"] == 0).all(1) & (st["mask1"] == 0).all(1))
    hit_sum = pm.sum(-1)[~miss]
    print(f"[parts] {agg_type}: {int(miss.sum())} of {miss.numel()} rays miss every box; sum_j part_map on the others: "
          f"mean {float(hit_sum.mean()):.3f}, max {float(hit_sum.max()):.3f}; mean acc {float(acc[~miss].mean()):.3f}")
    assert int(miss.sum()) > 0 and torch.equal(pm[miss], torch.zeros(int(miss.sum()), 24, device=DEV))
    assert float(pm.max()) > 0.3
    H = W = 64
    imgs, pmaps = render.render_images(caster, args, [syn.camera()], [pose], H, W, parts=True)
    imgs0 = render.render_images(caster, args, [syn.camera()], [pose], H, W)
    assert pmaps.shape == (1, H, W, 24) and torch.equal(imgs, imgs0)
    bg = torch.ones(H * W, dtype=torch.bool, device=DEV)
    bg[b["pixel_idx"].to(DEV)] = False
    assert torch.equal(pmaps.reshape(-1, 24)[bg], torch.zeros(int(bg.sum()), 24, device=DEV))
    # the random-init test weights leave the body translucent (mean acc_map 0.07 on the rays that hit a box), so the
    # labels are taken at half the image's largest weight rather than at the default 0.5
    lab = render.part_labels(pmaps, min_weight=0.5 * float(pmaps.max()))
    assert bool((lab.reshape(-1)[bg] == -1).all()) and int((lab >= 0).sum()) > 0


@pytest.mark.parametrize("agg_type", AGG)
def test_part_map_across_blocks_and_poses(agg_type, monkeypatch):
    """A call of one pose cut into several launch blocks (MAX_RAYS_PER_LAUNCH lowered to 1024, nanmean_chunk 256), and
    a call of two poses (N_uniques=2, one block each), give the part maps of the one-block single-pose calls."""
    caster, args, _, _, _ = _image(agg_type)
    m = 2048
    batches = [syn.render_batch(syn.make_pose(s), 96, 96) for s in (3, 5)]
    assert all(bb["ray_batch"].shape[0] >= m for bb in batches)
    kw_of = lambda bb, sl: dict(N_samples=args.N_samples, kp_batch=bb["kp_batch"][sl], skts=bb["skts"][sl],
                                cyls=bb["cyls"][sl], bones=bb["bones"][sl], cams=bb["cams"][sl], perturb=False,
                                N_importance=args.N_importance, raw_noise_std=0., nanmean_chunk=256)
    sl = slice(0, m)
    with torch.no_grad():
        single = [caster.render_rays(bb["ray_batch"][sl], want_parts=True, N_uniques=1, **kw_of(bb, sl))
                  for bb in batches]
        monkeypatch.setattr(raycaster, "MAX_RAYS_PER_LAUNCH", 1024)
        cut = caster.render_rays(batches[0]["ray_batch"][sl], want_parts=True, N_uniques=1, **kw_of(batches[0], sl))
        cat = lambda k: torch.cat([bb[k][sl] for bb in batches], 0)
        two = caster.render_rays(cat("ray_batch"), want_parts=True, N_uniques=2, N_samples=args.N_samples,
                                 kp_batch=cat("kp_batch"), skts=cat("skts"), cyls=cat("cyls"), bones=cat("bones"),
                                 cams=cat("cams"), perturb=False, N_importance=args.N_importance, raw_noise_std=0.,
                                 nanmean_chunk=256)
    assert raycaster.RayCaster._plan_blocks(m, 1, m, 256, 1)[0] == 1024          # the cut call ran two blocks
    want = torch.cat([s["part_map"] for s in single], 0)
    d_cut = float((cut["part_map"] - single[0]["part_map"]).abs().max())
    d_two = float((two["part_map"] - want).abs().max())
    print(f"[parts] {agg_type}: blocks vs one block max |diff| {d_cut:.3e}; two poses vs single calls {d_two:.3e}")
    assert d_cut <= 1e-6 and d_two <= 1e-6
    assert torch.equal(cut["acc_map"] > 0, single[0]["acc_map"] > 0)
    for s in single:
        assert float(s["part_map"].max()) > 0.3


def _points(kps, n_lattice=12, n_random=1500, seed=0):
    """A lattice around the body (root +- 0.9), random points scattered around the joints, and three far away."""
    root = kps[0]
    g = torch.linspace(-0.9, 0.9, n_lattice)
    L = torch.stack(torch.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3) + root
    gen = torch.Generator().manual_seed(seed)
    R = kps[torch.randint(0, 24, (n_random,), generator=gen)] + 0.1 * torch.randn(n_random, 3, generator=gen)
    far = root + torch.tensor([[25., 0., 0.], [0., -30., 0.], [0., 0., 40.]])
    return torch.cat([L, R, far], 0).float().contiguous()


@pytest.mark.parametrize("agg_type", AGG)
def test_render_pts_parts_against_oracle(agg_type):
    """render_pts_parts against the oracle's field_eval at the same points: visibility bit for bit (except within a
    few ulp of a box face), p within 1e-4 of the logits' scale (the bound the aggregation-net kernels are held to);
    sigma equals render_pts_density's bit for bit; points no bone sees get p = 0 exactly."""
    fx = load_fixture(FIXTURE[agg_type])
    caster, _, _ = make_caster(preset_of(fx), agg_type=agg_type)
    caster.eval()
    skts, bones, _ = pose_tensors(fx)
    kps = fx["pose_kps"]
    pts = _points(kps)
    M = pts.shape[0]
    d = lambda t: t.to(DEV)
    sig, p = caster.render_pts_parts(d(pts), d(kps[None]), d(skts), d(bones))
    assert sig.shape == (M, 1) and p.shape == (M, 24)
    assert torch.equal(sig, caster.render_pts_density(d(pts), d(kps[None]), d(skts), d(bones)))
    s3, p3 = caster.render_pts_parts(d(pts).reshape(M, 1, 3), d(kps[None]), d(skts), d(bones))
    assert s3.shape == (M, 1, 1) and torch.equal(s3.reshape(M, 1), sig) and torch.equal(p3, p)
    Pc = params_for(fx)
    vol = orc.graph_net(orc.graph_inputs(bones), Pc)
    with torch.no_grad():
        _, a, invalid, stg = orc.field_eval(pts[:, None], torch.zeros(M, 3), torch.zeros(M, 1, dtype=torch.long),
                                            skts.expand(M, -1, -1, -1), align_A(), vol, Pc, M, False, agg_type)
    p_ref, invalid = stg["p"][:, 0].double(), invalid[:, 0] != 0
    _, mask, _ = caster._pts_field(d(pts), d(skts), d(bones))              # the masks render_pts_parts used
    vis = _bits(mask).cpu()
    n_bad, n_near = mask_mismatch_report(stg["x"][:, 0], (~vis).float(), invalid.float())
    same = (vis == ~invalid).all(-1)
    got = p.double().cpu()
    scale = max(float(a[:, 0][~invalid].abs().max()), 1.)
    err = float((got[same] - p_ref[same]).abs().max())
    print(f"[parts] {agg_type}: render_pts_parts vs oracle: {int(vis.any(-1).sum())} of {M} points seen, visibility "
          f"differs at {n_bad} (point, bone) pairs ({n_near} within 16 ulp of a box face), p max |diff| {err:.3e} "
          f"(logit scale {scale:.3e})")
    assert n_bad == n_near and int(same.sum()) >= M - 4
    assert err <= 1e-4 * scale
    assert bool((got[~vis] == 0).all()) and torch.equal(p[-3:], torch.zeros(3, 24, device=DEV))
    assert int(vis.any(-1).sum()) > M // 4
    if agg_type == "softmax":
        assert bool((got.sum(-1) <= 1. + 1e-6).all())


@pytest.mark.parametrize("agg_type", AGG)
def test_mesh_parts_and_normals(agg_type, tmp_path):
    """render_mesh(parts=True, normals=True) at res 64: the plain call's vertices and triangles, one normal per vertex,
    (V,24) weights equal to render_pts_parts at root + 2 radius v, and a PLY that read_ply returns with
    vertices, normals and the PART_COLORS entry of each vertex's arg-max bone."""
    caster, _, pose, _, _ = _image(agg_type)
    t = lambda a: torch.as_tensor(a)[None].to(DEV)
    kps, skts, bones = t(pose["kps"]), t(pose["skts"]), t(pose["bones"])
    res, radius = 64, 1.0
    raw = caster(kps=kps, skts=skts, bones=bones, radius=radius, res=res, fwd_type="mesh")
    thr = float(torch.relu(raw).max()) * 0.25
    (v0, t0), = mesh.render_mesh(caster, kps, skts, bones, radius=radius, res=res, threshold=thr)
    (v, tr, n, p), = mesh.render_mesh(caster, kps, skts, bones, radius=radius, res=res, threshold=thr, normals=True,
                                      parts=True, out_dir=str(tmp_path))
    (v1, t1, p1), = mesh.render_mesh(caster, kps, skts, bones, radius=radius, res=res, threshold=thr, parts=True)
    assert torch.equal(v, v0) and torch.equal(tr, t0) and torch.equal(v1, v) and tr.shape[0] > 100
    assert n.shape == v.shape and torch.equal(p1, p)
    _, want = caster.render_pts_parts(kps[0, 0] + 2. * radius * v, kps, skts, bones)
    assert p.shape == (v.shape[0], 24) and torch.equal(p, want)
    rv, rt, rn, rc = mesh.read_ply(os.path.join(str(tmp_path), "meshes", "000.ply"), with_normals=True, with_colors=True)
    assert np.array_equal(rv, v.cpu().numpy()) and np.array_equal(rt, tr.cpu().numpy())
    assert np.array_equal(rn, n.cpu().numpy())
    assert np.array_equal(rc, mesh.PART_COLORS[p.argmax(-1).cpu().numpy()])
    used = np.unique(p.argmax(-1).cpu().numpy())
    print(f"[parts] {agg_type}: mesh {v.shape[0]} vertices, {len(used)} parts coloured, vertices no bone sees "
          f"{int((p == 0).all(-1).sum())}")
    assert len(used) >= 5
