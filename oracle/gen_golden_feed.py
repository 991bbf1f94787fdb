"""Generates tests/golden/feed_*.npz by running the UNMODIFIED reference data pipeline (see oracle/ref_harness.py).
TEST INFRASTRUCTURE.

    python oracle/gen_golden_feed.py       # needs the reference ($DANBO_REFERENCE or baseline/_ref); writes tests/golden/feed_plain.npz, feed_centers.npz

Pins `danbo-pytorch_b200/feed.py` (SURVEY §8f rank 3): the reference's `BaseH5Dataset.__getitem__`
(core/dataset.py:61-129) is run on a synthetic training set stored under the reference's HDF5 keys (read through the
npz-backed h5py stub, oracle/ref_stubs/h5py.py), for the sorted image indices a `RayImageSampler` would yield
(:941-976), and collated with the reference's `ray_collate_fn` (:980-987).  The pixel indices its `sample_pixels` drew
are recorded so the test can replay them.  The data set itself is not stored: `feed.synthetic_arrays` regenerates it
from (n_images, H, W, seed), and a checksum of the images guards against drift."""
import os
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import ref_harness                                   # noqa: E402
import danbo_b200                                    # noqa: E402
from danbo_b200 import feed                          # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
SPEC = dict(n_images=6, H=20, W=24, seed=3)


def run_reference(arrays, image_idxs, rays_per_image, seed, mask_img=True, perturb_bg=False):
    """-> dict of the collated batch + the pixel indices drawn, all numpy."""
    ref_harness._imports()
    import core.dataset as ds
    tmp = os.path.join(tempfile.mkdtemp(prefix="danbo_feed_"), "train.npz")
    np.savez(tmp, **arrays)
    data = ds.BaseH5Dataset(tmp, N_samples=rays_per_image, mask_img=mask_img, perturb_bg=perturb_bg)
    drawn = []
    orig = data.sample_pixels

    def sample_pixels(idx, q_idx):
        p = orig(idx, q_idx)
        drawn.append(p.copy())
        return p
    data.sample_pixels = sample_pixels
    np.random.seed(seed)
    items = [data[int(i)] for i in np.sort(image_idxs)]
    if not data.has_bg:
        for it in items:
            it.pop("bgs")
    batch = ds.ray_collate_fn(items)
    out = {k: v.numpy() for k, v in batch.items()}
    out["pixel_idxs"] = np.stack(drawn)
    out["image_idxs"] = np.sort(image_idxs)
    return out


def main():
    if not ref_harness.available():
        raise SystemExit("needs the reference ($DANBO_REFERENCE or baseline/_ref)")
    for name, centers in (("feed_plain", False), ("feed_centers", True)):
        arrays = feed.synthetic_arrays(centers=centers, **SPEC)
        out = run_reference(arrays, np.array([4, 0, 5, 2]), rays_per_image=12, seed=11)
        out["spec"] = np.array([SPEC["n_images"], SPEC["H"], SPEC["W"], SPEC["seed"], int(centers)])
        out["imgs_checksum"] = np.array([int(arrays["imgs"].astype(np.int64).sum())])
        np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)
        print(name, {k: v.shape for k, v in out.items()})


if __name__ == "__main__":
    main()
