"""Generates tests/golden/rays_box.npz by running the UNMODIFIED reference ray generation (see oracle/ref_harness.py).
TEST INFRASTRUCTURE.

    python oracle/gen_golden_rays.py       # needs the reference ($DANBO_REFERENCE or baseline/_ref)

Pins SURVEY §8f rank 1 (`render.rays_in_box`, `synthetic.cylinder_image_box`, `skeleton.bounding_cylinder`): the
reference's `kp_to_valid_rays` (core/utils/ray_utils.py:84-138: `get_rays` :7-29, `get_kp_bounding_cylinder`
skeleton_utils.py:568-631, `cylinder_to_box_2d` :633-720) for bullet-time cameras around synthetic poses, once with the
cylinders derived from the key points (render-time expansion ratios) and once with given cylinders."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import ref_harness                                   # noqa: E402
import danbo_b200                                    # noqa: E402,F401
from danbo_b200 import synthetic as syn              # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "rays_box.npz")
H, W, N_VIEWS, POSE_SEEDS = 96, 80, 5, (3, 8)


def inputs():
    poses = [syn.make_pose(s, render_cylinder=False) for s in POSE_SEEDS]
    c2ws = syn.bullet_time_cameras(syn.camera(), N_VIEWS).astype(np.float32)
    return poses, c2ws, float(0.45 * H)          # short focal length: the boxes lie inside the image


def run_reference(poses, c2ws, focal, given_cyls):
    ref_harness._imports()
    from core.utils.ray_utils import kp_to_valid_rays
    kps = torch.tensor(np.stack([p["kps"] for p in poses]))
    cyl = torch.tensor(np.stack([p["cyl"] for p in poses])) if given_cyls else None
    rays, valid, cyls, boxes = kp_to_valid_rays(torch.tensor(c2ws), H, W, focal, kps=kps, cylinder_params=cyl,
                                                ext_scale=0.001)
    return rays, valid, cyls.numpy(), boxes


def main():
    if not ref_harness.available():
        raise SystemExit("needs the reference ($DANBO_REFERENCE or baseline/_ref)")
    poses, c2ws, focal = inputs()
    out = {"H": H, "W": W, "n_views": N_VIEWS, "pose_seeds": np.array(POSE_SEEDS), "focal": focal}
    for tag, given in (("derived", False), ("given", True)):
        rays, valid, cyls, boxes = run_reference(poses, c2ws, focal, given)
        out[f"{tag}.cyls"] = cyls
        for i in range(N_VIEWS):
            out[f"{tag}.{i}.rays_o"], out[f"{tag}.{i}.rays_d"] = rays[i][0].numpy(), rays[i][1].numpy()
            out[f"{tag}.{i}.valid_idx"] = valid[i].numpy()
            out[f"{tag}.{i}.tl"], out[f"{tag}.{i}.br"] = np.asarray(boxes[i][0]), np.asarray(boxes[i][1])
    np.savez_compressed(OUT, **out)
    print(OUT, os.path.getsize(OUT) / 1e6, "MB", [out[f"derived.{i}.valid_idx"].shape[0] for i in range(N_VIEWS)])


if __name__ == "__main__":
    main()
