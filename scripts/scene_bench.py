"""Cost of scenes of several bodies (raycaster.render_scene_rays) against the plain render, on the bench pose with
danbo_fast weights.

Prints, with the card's name, power limit and max SM clock read in the same run, for K = 1, 2 and 4 bodies (the bench
pose, each further body offset by (0.3, 0, -0.3) m from the last, so that they partly overlap in depth):
  - a 512x512 render_scene_images image in the bench camera against K plain render_images images of the bodies alone
    (each in its own box), alternating windows of CUDA events after a warm-up of both, median window;
  - on the scene's rays, the danbo_scene_composite launch against the danbo_merge_composite launch of the first body's
    plain render of the same rays (CUDA events around each launch, kernels.PROFILE stage timing, median of 10 calls).

    python scripts/scene_bench.py [--out FILE] [--reps N]      (FILE also receives everything printed)
"""
import argparse
import os
import statistics
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import danbo_b200 as db  # noqa: E402
from danbo_b200 import kernels as K, raycaster, render, skeleton as sk, synthetic as syn  # noqa: E402
from normals_bench import card, compare  # noqa: E402


def stage_ms(fn, stage, calls):
    """Median over `calls` calls of fn of the time between the events around its `stage` launch."""
    K.PROFILE = {"mlp": [], "launches": 0, "stages": []}
    try:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
        return statistics.median(e0.elapsed_time(e1) for name, e0, e1 in K.PROFILE["stages"] if name == stage)
    finally:
        K.PROFILE = None


def moved(pose, t):
    t = np.asarray(t, np.float32)
    skts = pose["skts"].copy()
    skts[:, :3, 3] -= skts[:, :3, :3] @ t
    cyl = pose["cyl"].copy()
    cyl[[0, 1, 3, 4]] += t[[0, 2, 1, 1]]
    return {"bones": pose["bones"], "kps": pose["kps"] + t, "skts": skts, "cyl": cyl}


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
    H = W = 512
    c2w = syn.bullet_time_cameras(syn.camera(), 8)[0]
    focal = 1.2 * H
    base = syn.make_pose(3)
    d = lambda a: torch.as_tensor(np.asarray(a, np.float32))[None].to(dev)
    for n_inst in (1, 2, 4):
        poses = [moved(base, (0.3 * k, 0., -0.3 * k)) for k in range(n_inst)]
        insts = [{"caster": caster, "kps": d(p["kps"]), "skts": d(p["skts"]), "bones": d(p["bones"]),
                  "cyls": d(p["cyl"]), "cams": 0} for p in poses]
        scene = lambda: render.render_scene_images(insts, args, [c2w], H, W)
        plain = lambda: [render.render_images(caster, args, [c2w], [p], H, W) for p in poses]
        ms_s, ms_p = compare(scene, plain, 3, cli.reps)
        n_rays = render.rays_in_box(H, W, focal, c2w, np.stack([p["cyl"] for p in poses]), dev)[2].numel()
        n_own = [render.rays_in_box(H, W, focal, c2w, p["cyl"], dev)[2].numel() for p in poses]
        say(f"K={n_inst}: scene image {ms_s:.3f} ms ({n_rays} rays in the union box), {n_inst} plain images "
            f"{ms_p:.3f} ms ({sum(n_own)} rays in their boxes): ratio {ms_s / ms_p:.3f}")
        ro, rd, _ = render.rays_in_box(H, W, focal, c2w, np.stack([p["cyl"] for p in poses]), dev)
        ones = torch.ones(ro.shape[0], 1, device=dev)
        rays = torch.cat([ro, rd, syn.NEAR * ones, syn.FAR * ones, rd / torch.norm(rd, dim=-1, keepdim=True)], -1)
        n = rays.shape[0]
        ex = lambda t: t.expand(n, *t.shape[1:])
        i0 = insts[0]
        with torch.no_grad():
            k_s = stage_ms(lambda: raycaster.render_scene_rays(rays, insts, args.N_samples, args.N_importance,
                                                               nanmean_chunk=args.chunk), "scene_composite", 10)
            k_m = stage_ms(lambda: caster.render_rays(rays, N_samples=args.N_samples, kp_batch=ex(i0["kps"]),
                                                      skts=ex(i0["skts"]), cyls=ex(i0["cyls"]), bones=ex(i0["bones"]),
                                                      cams=torch.zeros(n, 1, dtype=torch.long, device=dev), N_uniques=1,
                                                      perturb=False, N_importance=args.N_importance, raw_noise_std=0.,
                                                      nanmean_chunk=args.chunk), "merge_composite", 10)
            imap = raycaster.render_scene_rays(rays, insts, args.N_samples, args.N_importance,
                                               nanmean_chunk=args.chunk)["instance_map"]
        say(f"  on the {n} scene rays: scene kernel {k_s * 1e3:.1f} us, merge kernel of one body {k_m * 1e3:.1f} us "
            f"(x{n_inst} = {n_inst * k_m * 1e3:.1f} us); rays where two bodies each weigh > 0.05: "
            f"{int(((imap > 0.05).sum(-1) >= 2).sum())}")
    say(f"peak memory allocated {torch.cuda.max_memory_allocated(dev) / 2 ** 30:.2f} GiB")
    if cli.out:
        os.makedirs(os.path.dirname(os.path.abspath(cli.out)), exist_ok=True)
        with open(cli.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
