"""Cost of the surface-normal paths against the plain calls they extend, on the bench pose with danbo_fast weights.

Prints, with the card's name, power limit and max SM clock read in the same run:
  - render_pts_gradient against render_pts_density on the vertex set of the res-255 mesh of the pose (points / s);
  - a 512x512 normal-map render (render_rays(want_normals=True)) against the plain eval render of the same rays.
Each pair is timed in alternating windows with CUDA events after a warm-up of both; the median window is reported.

    python scripts/normals_bench.py [--out FILE] [--reps N]      (FILE also receives everything printed)
"""
import argparse
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import danbo_b200 as db  # noqa: E402
from danbo_b200 import mesh, skeleton as sk, synthetic as syn  # noqa: E402


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return name, q


def window(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def compare(fa, fb, iters, reps):
    """Alternating windows of fa and fb -> (median ms of fa, median ms of fb)."""
    fa(), fb()
    torch.cuda.synchronize()
    ta, tb = [], []
    for _ in range(reps):
        ta.append(window(fa, iters))
        tb.append(window(fb, iters))
    return statistics.median(ta), statistics.median(tb)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
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

    # ---- points: the vertices of the res-255 mesh (radius 1.8, threshold a quarter of the lattice's max), in world
    res, radius = 255, 1.8
    with torch.no_grad():
        raw = caster(kps=kps, skts=skts, bones=bones, radius=radius, res=res, fwd_type="mesh")
        thr = float(torch.relu(raw).max()) * 0.25
        (v, tri), = mesh.render_mesh(caster, kps, skts, bones, radius=radius, res=res, threshold=thr)
    pts = (kps[0, 0] + 2. * radius * v).contiguous()
    say(f"mesh res {res}: {v.shape[0]} vertices, {tri.shape[0]} triangles (threshold {thr:.3f})")
    ms_g, ms_d = compare(lambda: caster.render_pts_gradient(pts, kps, skts, bones),
                         lambda: caster.render_pts_density(pts, kps, skts, bones), 3, cli.reps)
    P = pts.shape[0]
    say(f"render_pts_gradient {ms_g:.3f} ms ({P / ms_g / 1e3:.1f} M points/s); render_pts_density {ms_d:.3f} ms "
        f"({P / ms_d / 1e3:.1f} M points/s); ratio {ms_g / ms_d:.2f}")

    # ---- a 512x512 normal map against the plain render of the same rays (the bench's camera)
    H = W = 512
    c2w = syn.bullet_time_cameras(syn.camera(), 8)[0]
    b = syn.render_batch(pose, H, W, c2w=c2w, cam_idx=0)
    kw = dict(N_samples=args.N_samples, kp_batch=b["kp_batch"].to(dev), skts=b["skts"].to(dev), cyls=b["cyls"].to(dev),
              bones=b["bones"].to(dev), cams=b["cams"].to(dev), N_uniques=1, perturb=False,
              N_importance=args.N_importance, raw_noise_std=0., nanmean_chunk=args.chunk)
    rays = b["ray_batch"].to(dev)
    with torch.no_grad():
        ms_n, ms_p = compare(lambda: caster.render_rays(rays, want_normals=True, **kw),
                             lambda: caster.render_rays(rays, **kw), 2, cli.reps)
    say(f"512x512 image ({rays.shape[0]} rays in the box): normal-map render {ms_n:.2f} ms, plain render {ms_p:.2f} ms, "
        f"ratio {ms_n / ms_p:.2f}")
    say(f"peak memory allocated {torch.cuda.max_memory_allocated(dev) / 2 ** 30:.2f} GiB")
    if cli.out:
        os.makedirs(os.path.dirname(os.path.abspath(cli.out)), exist_ok=True)
        with open(cli.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
