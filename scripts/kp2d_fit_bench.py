"""Cost of the 2D keypoint reprojection term in pose fitting: PoseFitStep(graph=True) with and without the term, at
training size on the GPU.

Prints, with the card's name, power limit and max SM clock read in the same run:
  - ms / iteration of h36m_zju danbo_fast at 16 poses x 192 rays (32 + 16 samples), both arms timed in alternating
    windows (CUDA events, the same batch every iteration).  The "with" arm's batch carries detections 5 px off the
    projections of the frames' joints through their cameras and kp2d_coef = 1; the "without" arm's batch has no 2D keys;
  - kernels per iteration of each arm, counted with torch.profiler on one eager execution of the function the graph
    captures, in a session after all timed windows, and the kernels by name that the term adds.

    python scripts/kp2d_fit_bench.py [--out FILE]      (FILE also receives everything printed)
"""
import argparse
import json
import os
import statistics
import sys
from collections import Counter

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
from danbo_b200 import feed as fd, render, synthetic as syn  # noqa: E402
from pose_fit_bench import card, kernel_count, make_step, timed  # noqa: E402


def detections(step, arrays, frames, H, W, noise=5.0):
    """The batch keys of the 2D term: the pose layer's joints of `frames` projected through the frames' cameras, plus
    seeded pixel noise, confidence 1."""
    with torch.no_grad():
        kps = step.popt["popt_layer"].calculate_kinematic(frames)[0].double().cpu()
    proj = torch.tensor(render.projection_matrix(arrays["c2ws"][frames], H, W, float(arrays["focals"][0])))
    h = torch.einsum("grc,gjc->gjr", proj, torch.cat([kps, torch.ones_like(kps[..., :1])], -1))
    uv = h[..., :2] / h[..., 2:] + noise * torch.randn(kps.shape[0], 24, 2, dtype=torch.float64,
                                                        generator=torch.Generator().manual_seed(0))
    kp2d = torch.cat([uv, torch.ones_like(uv[..., :1])], -1)
    dev = step.popt["popt_layer"].pelvis.device
    return {"kp2d": kp2d.float().to(dev), "kp2d_proj": proj.float().to(dev)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--windows", type=int, default=7)
    cli = ap.parse_args()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    dev = torch.device("cuda", 0)
    name, limits = card()
    say(f"card: {name}; power.limit, clocks.max.sm: {limits}")
    n_poses, rpp, H = 16, 192, 256
    arrays = fd.synthetic_arrays(n_images=32, H=H, W=H, seed=0)
    feed = fd.RayFeed.from_arrays(arrays, syn.NEAR, syn.FAR, N_rand=n_poses * rpp, N_sample_images=n_poses, device=dev,
                                  seed=0, cam_idxs=np.arange(32) % 8)
    plain = feed.next_batch(torch.Generator(device=dev).manual_seed(0))
    frames = feed.last_idxs[0].cpu().numpy()
    arms = {"without": make_step({}, arrays, dev, True), "with": make_step({}, arrays, dev, True)}
    arms["with"].args.kp2d_coef = 1.0
    batches = {"without": plain, "with": dict(plain, **detections(arms["with"], arrays, frames, H, H))}
    for k, step in arms.items():
        for _ in range(3):
            step(batches[k])
    torch.cuda.synchronize()
    px0 = float(arms["with"].last_stats["kp2d_px"])
    ms = {k: [] for k in arms}
    for _ in range(cli.windows):
        for k, step in arms.items():
            ms[k].append(timed(step, batches[k], cli.iters))
    med = {k: statistics.median(v) for k, v in ms.items()}
    del arms
    torch.cuda.empty_cache()
    counts = {}
    for k, coef in (("without", 0.0), ("with", 1.0)):
        step = make_step({}, arrays, dev, True)
        step.args.kp2d_coef = coef
        counts[k] = kernel_count(step, batches[k])
    say(f"h36m_zju danbo_fast PoseFitStep(graph=True), {n_poses} poses x {rpp} rays, 32+16 samples per ray, one CUDA graph "
        f"per iteration")
    for k in ("without", "with"):
        say(f"  {k + ' the 2D term':22s}: {med[k]:7.3f} ms / iteration; {counts[k][0]} kernels + {counts[k][1]} "
            f"memcpy/memset; windows {['%.3f' % v for v in ms[k]]}")
    say(f"  the term costs {med['with'] - med['without']:+.4f} ms / iteration ({med['with'] / med['without']:.3f}x); "
        f"kp2d_px at the 4th iteration {px0:.3f}")
    diff = Counter(n[:100] for n in counts["with"][2])
    diff.subtract(Counter(n[:100] for n in counts["without"][2]))
    say("  operations the term adds:")
    for n, c in sorted(diff.items(), key=lambda x: -x[1]):
        if c:
            say(f"    {c:+d} x {n}")
    say(json.dumps({"card": name, "limits": limits, "ms": med, "windows": ms,
                    "kernels": {k: v[:2] for k, v in counts.items()}}))
    if cli.out:
        os.makedirs(os.path.dirname(os.path.abspath(cli.out)), exist_ok=True)
        with open(cli.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
