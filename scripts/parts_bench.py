"""Cost of the body-part paths against the plain calls they extend, on the bench pose with danbo_fast weights.

Prints, with the card's name, power limit and max SM clock read in the same run:
  - a 512x512 eval render with and without want_parts (the h36m_zju danbo_fast bench pose and camera), and the merge
    kernel alone in both renders (CUDA events around the launch, kernels.PROFILE stage timing);
  - the res-255 mesh of the pose with and without parts=True, and render_pts_parts against render_pts_density on its
    vertices.
Each pair is timed in alternating windows with CUDA events after a warm-up of both; the median window is reported.

    python scripts/parts_bench.py [--out FILE] [--reps N]      (FILE also receives everything printed)
"""
import argparse
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import danbo_b200 as db  # noqa: E402
from danbo_b200 import kernels as K, mesh, skeleton as sk, synthetic as syn  # noqa: E402
from normals_bench import card, compare  # noqa: E402


def merge_ms(fn, calls):
    """Median over `calls` calls of fn of the time between the events around its merge_composite launch."""
    K.PROFILE = {"mlp": [], "launches": 0, "stages": []}
    try:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
        return statistics.median(e0.elapsed_time(e1) for name, e0, e1 in K.PROFILE["stages"] if name == "merge_composite")
    finally:
        K.PROFILE = None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=7)
    cli = ap.parse_args()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)
    dev = torch.device("cuda", 0)
    name, q = card()
    say(f"card: {name}; power.limit, clocks.max.sm: {q}")
    args = db.make_args("danbo_fast", no_reload=True)
    attrs = {"skel_type": sk.SMPLSkeleton, "near": syn.NEAR, "far": syn.FAR, "n_views": 8, "rest_pose": syn.rest_pose()}
    torch.manual_seed(0)
    _, kw_test, *_ = db.create_raycaster(args, attrs, device=dev)
    caster = kw_test["ray_caster"]
    caster.network.load_state_dict(syn.synthetic_params(0))
    caster.eval()
    pose = syn.make_pose(3)
    t = lambda a: torch.as_tensor(a)[None].to(dev)
    kps, skts, bones = t(pose["kps"]), t(pose["skts"]), t(pose["bones"])

    # ---- a 512x512 render with and without the part map (the bench's camera)
    H = W = 512
    c2w = syn.bullet_time_cameras(syn.camera(), 8)[0]
    b = syn.render_batch(pose, H, W, c2w=c2w, cam_idx=0)
    kw = dict(N_samples=args.N_samples, kp_batch=b["kp_batch"].to(dev), skts=b["skts"].to(dev), cyls=b["cyls"].to(dev),
              bones=b["bones"].to(dev), cams=b["cams"].to(dev), N_uniques=1, perturb=False,
              N_importance=args.N_importance, raw_noise_std=0., nanmean_chunk=args.chunk)
    rays = b["ray_batch"].to(dev)
    with torch.no_grad():
        parts = lambda: caster.render_rays(rays, want_parts=True, **kw)
        plain = lambda: caster.render_rays(rays, **kw)
        ms_w, ms_p = compare(parts, plain, 5, cli.reps)
        k_w, k_p = merge_ms(parts, 10), merge_ms(plain, 10)
        pm = parts()["part_map"]
    say(f"512x512 image ({rays.shape[0]} rays in the box): want_parts render {ms_w:.3f} ms, plain render {ms_p:.3f} ms, "
        f"overhead {ms_w - ms_p:+.3f} ms ({100 * (ms_w / ms_p - 1):+.1f} %)")
    say(f"  merge kernel alone: with part map {k_w * 1e3:.1f} us, plain {k_p * 1e3:.1f} us ({(k_w - k_p) * 1e3:+.1f} us)")
    say(f"  rays with a part weight >= 0.5: {int((pm.max(-1).values >= 0.5).sum())}")

    # ---- the res-255 mesh (radius 1.8, threshold a quarter of the lattice's max) with and without part colours
    res, radius = 255, 1.8
    with torch.no_grad():
        raw = caster(kps=kps, skts=skts, bones=bones, radius=radius, res=res, fwd_type="mesh")
        thr = float(torch.relu(raw).max()) * 0.25
        (v, tri), = mesh.render_mesh(caster, kps, skts, bones, radius=radius, res=res, threshold=thr)
    say(f"mesh res {res}: {v.shape[0]} vertices, {tri.shape[0]} triangles (threshold {thr:.3f})")
    ms_mp, ms_m = compare(lambda: mesh.render_mesh(caster, kps, skts, bones, radius=radius, res=res, threshold=thr,
                                                   parts=True),
                          lambda: mesh.render_mesh(caster, kps, skts, bones, radius=radius, res=res, threshold=thr),
                          1, cli.reps)
    say(f"render_mesh parts=True {ms_mp:.2f} ms, plain {ms_m:.2f} ms, overhead {ms_mp - ms_m:+.2f} ms "
        f"({100 * (ms_mp / ms_m - 1):+.1f} %)")
    pts = (kps[0, 0] + 2. * radius * v).contiguous()
    ms_q, ms_d = compare(lambda: caster.render_pts_parts(pts, kps, skts, bones),
                         lambda: caster.render_pts_density(pts, kps, skts, bones), 3, cli.reps)
    say(f"on its vertices: render_pts_parts {ms_q:.3f} ms, render_pts_density {ms_d:.3f} ms")
    say(f"peak memory allocated {torch.cuda.max_memory_allocated(dev) / 2 ** 30:.2f} GiB")
    if cli.out:
        os.makedirs(os.path.dirname(os.path.abspath(cli.out)), exist_ok=True)
        with open(cli.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
