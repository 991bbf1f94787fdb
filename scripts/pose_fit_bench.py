"""Pose fitting with a frozen field (PoseFitStep(graph=True)) against the captured --opt_pose training iteration
(TrainStep(graph=True) with a pose layer), at training size on the GPU.

Prints, with the card's name, power limit and max SM clock read in the same run:
  - ms / iteration of danbo_fast at 16 poses x 192 rays (32 + 16 samples) with h36m_zju and with perfcap flags, both
    arms timed in alternating windows (CUDA events, the same batch every iteration);
  - kernels per iteration of each arm, counted with torch.profiler on one eager execution of the function the graph
    captures (memcpy / memset operations listed apart), in a session after all timed windows (a profiler session slows
    the host for the rest of the process, DESIGN.md section 4), and the kernels by name that fitting drops.

    python scripts/pose_fit_bench.py [--out FILE]      (FILE also receives everything printed)
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
from collections import Counter

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import danbo_b200 as db  # noqa: E402
from danbo_b200 import feed as fd, pose_opt as po, skeleton as sk, synthetic as syn, training  # noqa: E402

PERFCAP = dict(view_type="relray", ray_tr_type="root_local", nerf_type="graph")   # configs/perfcap/danbo_*.txt


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return name, q


def make_step(flags, arrays, dev, fit):
    args = db.make_args("danbo_fast", no_reload=True, opt_pose=True, **flags)
    attrs = {"skel_type": sk.SMPLSkeleton, "near": syn.NEAR, "far": syn.FAR, "n_views": 8, "rest_pose": syn.rest_pose()}
    _, kw, *_ = db.create_raycaster(args, attrs, device=dev)
    caster = kw["ray_caster"]
    caster.network.load_state_dict(syn.synthetic_params(0))
    caster.train()
    pattrs = {"rest_pose": syn.rest_pose()[None], "betas": torch.zeros(1, 10).numpy(), "kp3d": arrays["kp3d"],
              "bones": arrays["bones"]}
    pose_optimizer, pkw = po.create_popt(args, pattrs, device=dev, flat=True)
    if fit:
        return training.PoseFitStep(caster, args, pkw, pose_optimizer, graph=True)
    return training.TrainStep(caster, args, graph=True, popt_kwargs=pkw, pose_optimizer=pose_optimizer)


def timed(step, batch, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        step(batch)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def kernel_count(step, batch):
    """Kernels (and memcpy / memset operations) of one eager run of what the step's graph captures (after one warm
    run, so that a first-call weight pack is not counted)."""
    from torch.profiler import profile, ProfilerActivity
    b = {k: v for k, v in batch.items() if k not in ("kp_batch", "skts", "bones")}
    step._step(b)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step._step(b)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    copies = sum(n.startswith("Memcpy") or n.startswith("Memset") for n in names)
    return len(names) - copies, copies, names


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
    n_poses, rpp = 16, 192
    arrays = fd.synthetic_arrays(n_images=32, H=256, W=256, seed=0)
    feed = fd.RayFeed.from_arrays(arrays, syn.NEAR, syn.FAR, N_rand=n_poses * rpp, N_sample_images=n_poses, device=dev,
                                  seed=0, cam_idxs=np.arange(32) % 8)
    batch = feed.next_batch(torch.Generator(device=dev).manual_seed(0))
    result = {"card": name, "limits": limits}
    cfgs = (("h36m_zju", {}), ("perfcap", PERFCAP))
    for cfg, flags in cfgs:
        arms = {"train": make_step(flags, arrays, dev, False), "fit": make_step(flags, arrays, dev, True)}
        for step in arms.values():
            for _ in range(3):
                step(batch)
        torch.cuda.synchronize()
        ms = {k: [] for k in arms}
        for _ in range(cli.windows):
            for k, step in arms.items():
                ms[k].append(timed(step, batch, cli.iters))
        result[cfg] = {"ms": {k: statistics.median(v) for k, v in ms.items()}, "windows": ms}
        del arms
        torch.cuda.empty_cache()
    for cfg, flags in cfgs:
        result[cfg]["kernels"] = {k: kernel_count(make_step(flags, arrays, dev, k == "fit"), batch)
                                  for k in ("train", "fit")}
    for cfg, _ in cfgs:
        med, ms, counts = (result[cfg][k] for k in ("ms", "windows", "kernels"))
        say(f"{cfg} danbo_fast, {n_poses} poses x {rpp} rays, 32+16 samples per ray, one CUDA graph per iteration")
        for k, label in (("train", "TrainStep, pose layer"), ("fit", "PoseFitStep")):
            say(f"  {label:22s}: {med[k]:7.3f} ms / iteration; {counts[k][0]} kernels + {counts[k][1]} memcpy/memset; "
                f"windows {['%.3f' % v for v in ms[k]]}")
        say(f"  training / fitting: {med['train'] / med['fit']:.2f}x ({med['train'] - med['fit']:+.3f} ms)")
        diff = Counter(n[:100] for n in counts["train"][2])
        diff.subtract(Counter(n[:100] for n in counts["fit"][2]))
        say("  operations of the training iteration that fitting does not run (negative: fitting runs more):")
        for n, c in sorted(diff.items(), key=lambda x: -x[1]):
            if c:
                say(f"    {c:+d} x {n}")
    for cfg, _ in cfgs:
        result[cfg]["kernels"] = {k: v[:2] for k, v in result[cfg]["kernels"].items()}
    say(json.dumps(result))
    if cli.out:
        os.makedirs(os.path.dirname(os.path.abspath(cli.out)), exist_ok=True)
        with open(cli.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
