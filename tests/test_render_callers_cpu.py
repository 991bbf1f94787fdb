"""Ray generation and box culling (SURVEY §8f rank 1: `render.rays_in_box`, `synthetic.cylinder_image_box` /
`pinhole_rays`, `skeleton.bounding_cylinder`) against the reference's `kp_to_valid_rays` (core/utils/ray_utils.py:84-138).

CPU: these are torch / numpy ops that run on whatever device is asked for.  tests/golden/rays_box.npz comes from the
UNMODIFIED reference (oracle/gen_golden_rays.py)."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import danbo_b200                                    # noqa: E402,F401
import ref_harness                                   # noqa: E402
from danbo_b200 import render, skeleton as sk, synthetic as syn  # noqa: E402

FX = np.load(os.path.join(ROOT, "tests", "golden", "rays_box.npz"))
H, W, N_VIEWS, FOCAL = int(FX["H"]), int(FX["W"]), int(FX["n_views"]), float(FX["focal"])


def _inputs():
    poses = [syn.make_pose(int(s), render_cylinder=False) for s in FX["pose_seeds"]]
    c2ws = syn.bullet_time_cameras(syn.camera(), N_VIEWS).astype(np.float32)
    return poses, c2ws


def test_render_cylinder_from_keypoints():
    """kp_to_valid_rays derives the cylinder from the key points with the render-time expansion ratios (top 1.6,
    bottom 1.1, 250 mm; ray_utils.py:86-107)."""
    poses, _ = _inputs()
    for p, want in zip(poses, FX["derived.cyls"]):
        got = sk.bounding_cylinder(p["kps"], ext_scale=0.001, extend_mm=250, top_expand_ratio=1.6, bot_expand_ratio=1.1,
                                   head="-y")
        np.testing.assert_allclose(got, want, rtol=0, atol=1e-6)


@pytest.mark.parametrize("tag", ["derived", "given"])
def test_rays_in_box_match_reference(tag):
    """Pixel box of the projected cylinder caps (bit-exact pixel indices) and the pinhole rays of those pixels."""
    poses, c2ws = _inputs()
    cyls = FX[f"{tag}.cyls"]
    n_rays = set()
    for i in range(N_VIEWS):
        cyl = cyls[i % len(poses)]                                      # poses are reused cyclically (ray_utils.py:116)
        tl, br = syn.cylinder_image_box(cyl, H, W, FOCAL, c2ws[i])
        np.testing.assert_array_equal(tl, FX[f"{tag}.{i}.tl"])
        np.testing.assert_array_equal(br, FX[f"{tag}.{i}.br"])
        ro, rd, idx = render.rays_in_box(H, W, FOCAL, c2ws[i], cyl, "cpu")
        np.testing.assert_array_equal(idx.numpy(), FX[f"{tag}.{i}.valid_idx"])
        np.testing.assert_allclose(ro.numpy(), FX[f"{tag}.{i}.rays_o"], rtol=0, atol=1e-7)
        np.testing.assert_allclose(rd.numpy(), FX[f"{tag}.{i}.rays_d"], rtol=0, atol=3e-7)
        # the same rays through the host-side helper used by the fixtures / bench
        ro2, rd2, idx2 = syn.render_rays_for_pose(dict(poses[i % len(poses)], cyl=cyl), H, W, FOCAL, c2ws[i])
        assert torch.equal(idx2, idx) and float((rd2 - rd).abs().max()) < 3e-7 and float((ro2 - ro).abs().max()) < 1e-7
        n_rays.add(int(idx.shape[0]))
        assert 0 < idx.shape[0] < H * W                                 # the box really culls
    assert len(n_rays) > 1                                              # ... differently from view to view


@pytest.mark.skipif(not ref_harness.available(), reason="needs the original DANBO-pytorch (DANBO_REFERENCE or baseline/_ref)")
def test_live_reference_other_cameras():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import gen_golden_rays as gg
    poses = [syn.make_pose(21, render_cylinder=False)]
    c2ws = syn.bullet_time_cameras(syn.camera(tz=4.0), 7).astype(np.float32)[[1, 4, 6]]
    old = (gg.H, gg.W)
    gg.H, gg.W = 64, 72
    try:
        rays, valid, cyls, boxes = gg.run_reference(poses, c2ws, 50.0, given_cyls=False)
    finally:
        gg.H, gg.W = old
    for i in range(3):
        ro, rd, idx = render.rays_in_box(64, 72, 50.0, c2ws[i], cyls[0], "cpu")
        np.testing.assert_array_equal(idx.numpy(), valid[i].numpy())
        np.testing.assert_allclose(rd.numpy(), rays[i][1].numpy(), rtol=0, atol=3e-7)


class _Recorder:
    """Stand-in ray caster: records what it is called with and returns per-ray tensors derived from the rays."""

    def __init__(self):
        self.calls = []

    def __call__(self, ray_batch, **kw):
        self.calls.append((ray_batch.clone(), {k: (v.clone() if torch.is_tensor(v) else v) for k, v in kw.items()}))
        return {"rgb_map": ray_batch[:, 3:6] * 2, "acc_map": ray_batch[:, 6], "T_i": ray_batch[:, None, :4].expand(-1, 5, -1)}


def _render_inputs(n=10):
    g = torch.Generator().manual_seed(0)
    rays = (torch.randn(n, 3, generator=g), torch.randn(n, 3, generator=g))
    kw = dict(kp_batch=torch.randn(n, 24, 3, generator=g), skts=torch.randn(n, 24, 4, 4, generator=g),
              cams=torch.arange(n)[:, None], N_uniques=1, perturb=0.)
    return rays, kw


def test_render_chunks_like_batchify_rays():
    """`render(single_call=False)` = the reference's loop: every tensor kwarg sliced per chunk, results concatenated;
    `single_call=True` hands the whole batch over once with nanmean_chunk = chunk."""
    rays, kw = _render_inputs()
    a, b = _Recorder(), _Recorder()
    ra = render.render(8, 8, 10., chunk=4, rays=rays, near=1., far=5., use_viewdirs=True, single_call=False, ray_caster=a, **kw)
    rb = render.render(8, 8, 10., chunk=4, rays=rays, near=1., far=5., use_viewdirs=True, single_call=True, ray_caster=b, **kw)
    assert [c[0].shape[0] for c in a.calls] == [4, 4, 2] and len(b.calls) == 1 and b.calls[0][1]["nanmean_chunk"] == 4
    full = torch.cat([c[0] for c in a.calls], 0)
    assert torch.equal(full, b.calls[0][0]) and full.shape == (10, 11)
    assert torch.equal(full[:, 6], torch.ones(10)) and torch.equal(full[:, 7], torch.full((10,), 5.))
    assert float((full[:, 8:].norm(dim=-1) - 1).abs().max()) < 1e-6
    assert torch.equal(a.calls[1][1]["skts"], kw["skts"][4:8]) and a.calls[1][1]["N_uniques"] == 1
    for k in ra:
        assert torch.equal(ra[k], rb[k])
    assert ra["rgb_map"].shape == (10, 3) and ra["T_i"].shape == (10, 5, 4)


@pytest.mark.skipif(not ref_harness.available(), reason="needs the original DANBO-pytorch (DANBO_REFERENCE or baseline/_ref)")
def test_render_hands_the_caster_what_the_reference_does():
    ref_harness._imports()
    import core.trainer as tr
    rays, kw = _render_inputs()
    a, b = _Recorder(), _Recorder()
    want = tr.render(8, 8, 10., chunk=4, rays=rays, near=1., far=5., use_viewdirs=True, ray_caster=a, **kw)
    got = render.render(8, 8, 10., chunk=4, rays=rays, near=1., far=5., use_viewdirs=True, single_call=False, ray_caster=b, **kw)
    assert len(a.calls) == len(b.calls) == 3
    for (ra, ka), (rb, kb) in zip(a.calls, b.calls):
        assert torch.equal(ra, rb) and set(ka) == set(kb)
        assert all(torch.equal(ka[k], kb[k]) if torch.is_tensor(ka[k]) else ka[k] == kb[k] for k in ka)
    assert set(want) == set(got) and all(torch.equal(want[k], got[k]) for k in want)
