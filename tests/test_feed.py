"""Training data feed (SURVEY §8f rank 3, `feed.RayFeed`) against the reference's data pipeline (core/dataset.py).

CPU only: the feed is torch ops on whatever device holds the arrays.  `tests/golden/feed_*.npz` are batches of the
UNMODIFIED reference `BaseH5Dataset` + `ray_collate_fn` on the synthetic training set (oracle/gen_golden_feed.py); the
feed replays the image / pixel indices the reference drew.  The random draws themselves are checked by their
properties."""
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
from danbo_b200 import feed as fd                    # noqa: E402
from danbo_b200 import synthetic as syn              # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")


def _feed_for(fx, **kw):
    n, H, W, seed, centers = (int(v) for v in fx["spec"])
    arrays = fd.synthetic_arrays(n, H, W, seed, centers=bool(centers))
    assert int(arrays["imgs"].astype(np.int64).sum()) == int(fx["imgs_checksum"][0]), "synthetic data set drifted"
    return fd.RayFeed.from_arrays(arrays, syn.NEAR, syn.FAR, N_rand=48, N_sample_images=4, perturb_bg=False, **kw), arrays


@pytest.mark.parametrize("name", ["feed_plain", "feed_centers"])
def test_feed_reproduces_reference_batch(name):
    fx = np.load(os.path.join(GOLD, name + ".npz"))
    feed, _ = _feed_for(fx)
    b = feed.next_batch(image_idxs=fx["image_idxs"][::-1].copy(), pixel_idxs=fx["pixel_idxs"])   # unsorted: the feed sorts
    n = fx["rays_o"].shape[0]
    rays = b["ray_batch"].numpy()
    assert rays.shape == (n, 11)
    np.testing.assert_array_equal(rays[:, 0:3], fx["rays_o"])
    np.testing.assert_allclose(rays[:, 3:6], fx["rays_d"], rtol=0, atol=2e-7)       # fp32 dot product, summation order
    np.testing.assert_array_equal(rays[:, 6], np.full(n, syn.NEAR, np.float32))
    np.testing.assert_array_equal(rays[:, 7], np.full(n, syn.FAR, np.float32))
    d = fx["rays_d"]
    np.testing.assert_allclose(rays[:, 8:11], d / np.linalg.norm(d, axis=-1, keepdims=True), atol=3e-7)
    # image data: uint8 -> float, background compositing (dataset.py:281-305) -- bit-exact
    np.testing.assert_array_equal(b["target_s"].numpy(), fx["target_s"])
    np.testing.assert_array_equal(b["fgs"].numpy(), fx["fgs"])
    np.testing.assert_array_equal(b["bgs"].numpy(), fx["bgs"])
    # per-ray pose expansion (dataset.py:399-421), image-major (ray_collate_fn)
    np.testing.assert_array_equal(b["kp_batch"].numpy(), fx["kp3d"])
    np.testing.assert_array_equal(b["bones"].numpy(), fx["bones"])
    np.testing.assert_array_equal(b["skts"].numpy(), fx["skts"])
    np.testing.assert_array_equal(b["cyls"].numpy(), fx["cyls"])
    assert b["N_uniques"] == 4
    np.testing.assert_array_equal(b["kp_idx"].numpy(), fx["kp_idx"])                # the queried index (dataset.py:424-430)
    img, pix = feed.last_idxs
    np.testing.assert_array_equal(img.numpy(), fx["image_idxs"])
    np.testing.assert_array_equal(pix.numpy(), fx["pixel_idxs"])


def test_cam_idxs_default_is_the_queried_index():
    """dataset.py:432-438: the camera code index is the queried image index unless a subclass maps it."""
    fx = np.load(os.path.join(GOLD, "feed_plain.npz"))
    feed, _ = _feed_for(fx)
    b = feed.next_batch(image_idxs=fx["image_idxs"], pixel_idxs=fx["pixel_idxs"])
    assert b["cams"].shape == (48, 1) and b["cams"].dtype == torch.int64
    np.testing.assert_array_equal(b["cams"][:, 0].numpy(), fx["cam_idxs"])


@pytest.mark.parametrize("sparse", [False, True])
def test_sample_pixels_properties(sparse):
    """dataset.py:307-356: N_rand pixels per image, without replacement, inside the sampling mask, increasing; the whole
    image when the mask holds fewer pixels than requested; every mask pixel equally likely.  Both samplers: random keys
    over the image (small masks) and first-R-distinct-of-2R candidates (masks of >= 64 R pixels)."""
    if sparse:
        feed = fd.synthetic_feed(n_images=4, H=48, W=48, N_rand=4 * 8, N_sample_images=4)      # disc: ~886 px >= 64 * 8
        B, R, reps = 4, 8, 3000
    else:
        feed = fd.synthetic_feed(n_images=8, H=16, W=16, N_rand=8 * 20, N_sample_images=8)
        B, R, reps = 8, 20, 400
    assert feed._sparse_draw == sparse
    HW = feed.H * feed.W
    g = torch.Generator().manual_seed(0)
    idx = torch.arange(B)
    mask = feed.sampling_masks > 0
    counts = torch.zeros(HW)
    for _ in range(reps):
        pix = feed.sample_pixels(idx, g)
        assert pix.shape == (B, R) and pix.dtype == torch.int64
        assert (pix[:, 1:] > pix[:, :-1]).all()                       # increasing => distinct
        assert torch.gather(mask, 1, pix).all()
        counts += torch.bincount(pix.reshape(-1), minlength=HW)
    m = mask[0]
    assert counts[~m].sum() == 0
    expect = reps * B * R / int(m.sum())
    assert (counts[m] - expect).abs().max() < 6 * expect ** 0.5       # ~binomial spread
    assert abs(float(counts[m].mean()) - expect) < 1e-3
    # mask smaller than the request -> whole image (dataset.py:318-319)
    feed.sampling_masks[3] = 0
    feed.sampling_masks[3, :5] = 1
    feed.rebuild_sampling_index()
    assert int(feed._n_valid[3]) == HW and not (sparse and HW < 64 * R and feed._sparse_draw)
    seen_outside = False
    for _ in range(20):
        pix = feed.sample_pixels(torch.tensor([3]), g)
        assert (pix[:, 1:] > pix[:, :-1]).all()
        seen_outside |= bool((pix >= 5).any())
    assert seen_outside


def test_sparse_draw_repeats_are_skipped_in_draw_order():
    """The 2R-candidate sampler on a mask barely above its threshold, where repeated candidates are common: the result
    must still be R distinct candidate pixels, and pairs of pixels equally likely (no bias from the dedupe)."""
    feed = fd.synthetic_feed(n_images=1, H=24, W=24, N_rand=3, N_sample_images=1)
    feed.sampling_masks[:] = 0
    feed.sampling_masks[0, 100:292] = 1                               # 192 = 64 * 3 candidates
    feed.rebuild_sampling_index()
    assert feed._sparse_draw and int(feed._n_valid[0]) == 192
    g = torch.Generator().manual_seed(3)
    counts = torch.zeros(576)
    reps = 20000
    for _ in range(reps // 50):
        pix = feed.sample_pixels(torch.zeros(50, dtype=torch.long), g)        # 50 independent draws of the same image
        assert (pix[:, 1:] > pix[:, :-1]).all() and int(pix.min()) >= 100 and int(pix.max()) < 292
        counts += torch.bincount(pix.reshape(-1), minlength=576)
    expect = reps * 3 / 192
    assert (counts[100:292] - expect).abs().max() < 6 * expect ** 0.5


def test_image_sampler_passes_and_rank_shares():
    """RayImageSampler (dataset.py:941-976): consecutive entries of a permutation, so every image appears once per pass;
    batches sorted.  With world_size 2 the ranks' shares concatenated are the single-process batch."""
    mk = lambda **kw: fd.synthetic_feed(n_images=12, H=8, W=8, N_rand=4 * 2, N_sample_images=4, seed=5, **kw)
    one, r0, r1 = mk(), mk(rank=0, world_size=2), mk(rank=1, world_size=2)
    seen = []
    for step in range(9):                                              # 3 passes over 12 images
        full = one.draw_images()
        assert full.shape == (4,) and (full[1:] >= full[:-1]).all()
        assert torch.equal(torch.cat([r0.draw_images(), r1.draw_images()]), full)
        seen += full.tolist()
        if step % 3 == 2:
            assert sorted(seen) == list(range(12))                     # one pass = every image exactly once
            seen = []
    b0 = r0.next_batch(torch.Generator().manual_seed(0))
    assert b0["N_uniques"] == 2 and b0["ray_batch"].shape == (4, 11)
    with pytest.raises(ValueError):
        mk(world_size=3)
    # a batch that straddles two passes continues into a fresh permutation (dataset.py:964-970)
    odd = fd.synthetic_feed(n_images=5, H=8, W=8, N_rand=4 * 2, N_sample_images=4, seed=1)
    flat = [i for _ in range(5) for i in odd.draw_images().tolist()]
    assert len(flat) == 20 and sorted(flat) == sorted(list(range(5)) * 4)          # 4 whole passes in 5 batches


def test_next_batch_draws_distinct_sorted_images_and_perturbs_background_only():
    feed = fd.synthetic_feed(n_images=12, H=16, W=16, N_rand=6 * 10, N_sample_images=6, perturb_bg=True, mask_img=True)
    g = torch.Generator().manual_seed(1)
    seen = set()
    for _ in range(30):
        b = feed.next_batch(g)
        img, pix = feed.last_idxs
        assert img.shape == (6,) and (img[1:] > img[:-1]).all()       # 12 images, 6 per batch: distinct; np.sort (dataset.py:959-975)
        seen.update(img.tolist())
        fg = b["fgs"]
        plain = torch.gather(feed.bkgds[feed.bkgd_idxs[img]], 1, pix[..., None].expand(-1, -1, 3)).float().reshape(-1, 3) / 255.
        inside = fg[:, 0] > 0
        assert torch.equal(b["bgs"][inside], plain[inside])            # foreground keeps the stored background
        if (~inside).any():
            assert not torch.equal(b["bgs"][~inside], plain[~inside])  # the rest is noise in [0, 1)
            assert (b["bgs"][~inside] >= 0).all() and (b["bgs"][~inside] < 1).all()
            raw = torch.gather(feed.imgs[img], 1, pix[..., None].expand(-1, -1, 3)).float().reshape(-1, 3) / 255.
            assert torch.equal(b["target_s"][~inside], b["bgs"][~inside])      # mask_img: background pixels show bg
            assert torch.equal(b["target_s"][inside], raw[inside])
        assert b["ray_batch"].shape == (60, 11) and b["ray_batch"].is_contiguous()
        assert b["skts"].shape == (60, 24, 4, 4) and b["kp_batch"].shape == (60, 24, 3)
        assert b["N_uniques"] == 6
        # the pose tensors are per-image expands: ray r belongs to pose r // rays_per_image (encoders.py:465-471)
        assert torch.equal(b["skts"][::10], feed.skts[img])
    assert len(seen) == 12


def test_unsupported_flags_raise():
    with pytest.raises(NotImplementedError):
        fd.synthetic_feed(n_images=2, H=8, W=8, patch_size=2)
    with pytest.raises(NotImplementedError):
        fd.synthetic_feed(n_images=2, H=8, W=8, N_nms=1)


@pytest.mark.skipif(not ref_harness.available(), reason="needs the original DANBO-pytorch (DANBO_REFERENCE or baseline/_ref)")
def test_live_reference_other_draws():
    """The unmodified reference data pipeline, live, on draws that are not among the fixtures (focal per axis,
    identity camera rotation short-cut of dataset.py:393-394, no background arrays)."""
    import gen_golden_feed as gg
    arrays = fd.synthetic_arrays(n_images=5, H=18, W=14, seed=9, centers=True)
    arrays["focals"] = np.stack([arrays["focals"], arrays["focals"] * 1.1], -1)     # (N, 2): fx, fy
    arrays["c2ws"][1, :3, :3] = np.eye(3, dtype=np.float32)
    for drop_bg in (False, True):
        a = {k: v for k, v in arrays.items() if not (drop_bg and k.startswith("bkgd"))}
        ref = gg.run_reference(a, np.array([1, 3, 4]), rays_per_image=9, seed=5)
        feed = fd.RayFeed.from_arrays(a, 1.0, 5.0, N_rand=27, N_sample_images=3, perturb_bg=False)
        b = feed.next_batch(image_idxs=ref["image_idxs"], pixel_idxs=ref["pixel_idxs"])
        np.testing.assert_array_equal(b["ray_batch"][:, :3].numpy(), ref["rays_o"])
        np.testing.assert_allclose(b["ray_batch"][:, 3:6].numpy(), ref["rays_d"], rtol=0, atol=2e-7)
        np.testing.assert_array_equal(b["target_s"].numpy(), ref["target_s"])
        np.testing.assert_array_equal(b["fgs"].numpy(), ref["fgs"])
        assert ("bgs" in b) == (not drop_bg)
        if not drop_bg:
            np.testing.assert_array_equal(b["bgs"].numpy(), ref["bgs"])


def test_prefetch_on_the_cpu_is_next_batch():
    a = fd.synthetic_feed(n_images=6, H=12, W=12, N_rand=3 * 5, N_sample_images=3, seed=2, perturb_bg=False)
    b = fd.synthetic_feed(n_images=6, H=12, W=12, N_rand=3 * 5, N_sample_images=3, seed=2, perturb_bg=False)
    ga, gb = torch.Generator().manual_seed(4), torch.Generator().manual_seed(4)
    for _ in range(3):
        x, y = a.prefetch(ga), b.next_batch(gb)
        assert all(torch.equal(x[k], y[k]) for k in x if torch.is_tensor(x[k]))
