"""A captured --opt_pose training iteration (TrainStep(graph=True) with a FlatAdam pose optimizer) at training size, on
the GPU.

Prints, with the card's name and power limit read in the same run:
  - ms / iteration of danbo_fast at 16 poses x 192 rays (32 + 16 samples) with h36m_zju and with perfcap flags, in
    three arms per config timed in alternating windows (CUDA events, the same batch every iteration): eager with a pose
    layer (the PyTorch pose ops), graphed with a pose layer (the pose kernels) and graphed without one;
  - kernels per iteration of each graphed arm, counted with torch.profiler on one eager execution of the function the
    graph captures (the capture's warm-up call; memcpy / memset operations listed apart), after the timed windows;
  - the new kernels and the pose layer's Adam alone, each captured 200 times in one CUDA graph and replayed.

    python scripts/pose_graph_bench.py [--out FILE]      (FILE also receives everything printed)
"""
import argparse
import json
import os
import statistics
from collections import Counter
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import danbo_b200 as db  # noqa: E402
from danbo_b200 import feed as fd, kernels as K, pose_opt as po, skeleton as sk, synthetic as syn  # noqa: E402
from danbo_b200 import training  # noqa: E402

PERFCAP = dict(view_type="relray", ray_tr_type="root_local", nerf_type="graph")   # configs/perfcap/danbo_*.txt


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return name, q


def make_step(flags, arrays, dev, pose, graph):
    args = db.make_args("danbo_fast", no_reload=True, opt_pose=pose, **flags)
    attrs = {"skel_type": sk.SMPLSkeleton, "near": syn.NEAR, "far": syn.FAR, "n_views": 8, "rest_pose": syn.rest_pose()}
    _, kw, *_ = db.create_raycaster(args, attrs, device=dev)
    caster = kw["ray_caster"]
    caster.network.load_state_dict(syn.synthetic_params(0))
    caster.train()
    if not pose:
        return training.TrainStep(caster, args, graph=graph)
    pattrs = {"rest_pose": syn.rest_pose()[None], "betas": torch.zeros(1, 10).numpy(), "kp3d": arrays["kp3d"],
              "bones": arrays["bones"]}
    pose_optimizer, pkw = po.create_popt(args, pattrs, device=dev, flat=graph)
    return training.TrainStep(caster, args, graph=graph, popt_kwargs=pkw, pose_optimizer=pose_optimizer)


def timed(step, batch, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        step(batch)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def kernel_count(step, batch):
    """Kernels (and memcpy / memset operations) of one eager run of what TrainStep(graph=True) captures."""
    from torch.profiler import profile, ProfilerActivity
    b = dict(batch)
    if step.popt is not None:
        b = {k: v for k, v in b.items() if k not in ("kp_batch", "skts", "bones")}
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step._step(b)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    copies = sum(n.startswith("Memcpy") or n.startswith("Memset") for n in names)
    return len(names) - copies, copies, names


def replayed_us(fn, n_rep=200):
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(n_rep):
            fn()
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / (5 * n_rep) * 1e3


def kernels_alone(step, batch, n_poses, rpp):
    """us / launch of the pose kernels and the pose Adam at the batch's size, replayed from a CUDA graph."""
    layer, opt = step.popt["popt_layer"], step.pose_optimizer
    idx = batch["kp_idx"].long()
    L = {n: p.detach() for n, p in layer.named_parameters()}
    L["rest_pose"] = layer.rest_pose
    anchors = step._pose_anchors
    d_skts = torch.randn(n_poses, 24, 4, 4, device=idx.device)
    d_bones = torch.randn(n_poses, 24, 3, device=idx.device)
    d_reg = torch.ones((), device=idx.device)
    grads = {n: torch.zeros_like(p) for n, p in layer.named_parameters()}
    out = {"danbo_pose_fwd": replayed_us(lambda: K.pose_fwd(L, idx, rpp, n_poses, anchors=anchors, tol=0.0, coef=1.0)),
           "danbo_pose_bwd": replayed_us(lambda: K.pose_bwd(L, idx, rpp, n_poses, d_skts, grads, d_bones=d_bones,
                                                           anchor_bones=anchors["bones"], d_reg=d_reg, coef=1.0))}
    net = step.caster.network
    aa = torch.randn(n_poses, 24, 3, device=idx.device) * 0.5
    gnp = dict(net.graph_net.named_parameters())
    gnp["layers.0.adj"], gnp["layers.1.adj"] = net.graph_net.layers[0].adj, net.graph_net.layers[1].adj
    vol, saved = K.graph_net_fwd(aa, [gnp[n].detach() for n in K.GN_PARAMS])
    work = K.graph_net_bwd(saved, torch.randn_like(vol), [torch.zeros_like(gnp[n]) for n in K.GN_GRADS])
    out["danbo_graph_net_bwd_pose"] = replayed_us(lambda: K.graph_net_bwd_pose(saved, work, aa))
    snap = [t.clone() for t in (opt.flat, opt.exp_avg, opt.exp_avg_sq, opt.step_dev)]
    out["pose danbo_adam_step (+ step counter)"] = replayed_us(opt.step)
    with torch.no_grad():
        for t, v in zip((opt.flat, opt.exp_avg, opt.exp_avg_sq, opt.step_dev), snap):
            t.copy_(v)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--windows", type=int, default=5)
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
                                  seed=0, cam_idxs=np.arange(32) % 8)        # the caster's 8 frame codes (n_views)
    batch = feed.next_batch(torch.Generator(device=dev).manual_seed(0))
    result = {"card": name, "limits": limits}
    cfgs = (("h36m_zju", {}), ("perfcap", PERFCAP))
    for cfg, flags in cfgs:
        arms = {"eager_pose": make_step(flags, arrays, dev, True, False),
                "graphed_pose": make_step(flags, arrays, dev, True, True),
                "graphed_plain": make_step(flags, arrays, dev, False, True)}
        torch.manual_seed(0)
        for step in arms.values():
            for _ in range(3):
                step(batch)
        torch.cuda.synchronize()
        ms = {k: [] for k in arms}
        for _ in range(cli.windows):
            for k, step in arms.items():
                ms[k].append(timed(step, batch, cli.iters))
        med = {k: statistics.median(v) for k, v in ms.items()}
        alone = kernels_alone(arms["graphed_pose"], batch, n_poses, rpp)
        result[cfg] = {"ms": med, "windows": ms, "alone_us": alone}
        del arms
        torch.cuda.empty_cache()
    # after every timed window: a profiler session slows the host's launches for the rest of the process, which the
    # eager arms would pay.  Fresh steps, so that the profiled run is what a capture's warm-up executes.
    for cfg, flags in cfgs:
        result[cfg]["kernels"] = {"graphed_pose": kernel_count(make_step(flags, arrays, dev, True, True), batch),
                                  "graphed_plain": kernel_count(make_step(flags, arrays, dev, False, True), batch)}
    for cfg, _ in cfgs:
        med, ms, counts, alone = (result[cfg][k] for k in ("ms", "windows", "kernels", "alone_us"))
        say(f"{cfg} danbo_fast training, {n_poses} poses x {rpp} rays, 32+16 samples per ray")
        for k, label in (("eager_pose", "eager, pose layer"), ("graphed_pose", "graphed, pose layer"),
                         ("graphed_plain", "graphed, no pose layer")):
            extra = f"; {counts[k][0]} kernels + {counts[k][1]} memcpy/memset per iteration" if k in counts else ""
            say(f"  {label:24s}: {med[k]:7.3f} ms / iteration{extra}; windows {['%.3f' % v for v in ms[k]]}")
        say(f"  graphed pose vs graphed plain: {med['graphed_pose'] - med['graphed_plain']:+.3f} ms; "
            f"eager pose / graphed pose: {med['eager_pose'] / med['graphed_pose']:.1f}x")
        for k, us in alone.items():
            say(f"  {k} alone ({n_poses} poses): {us:.2f} us / launch")
        # what the pose layer adds to the captured iteration, by kernel name (names shortened to 100 characters)
        extra = Counter(n[:100] for n in counts["graphed_pose"][2])
        extra.subtract(Counter(n[:100] for n in counts["graphed_plain"][2]))
        say(f"  operations of the graphed pose iteration that the plain one does not run:")
        for n, c in sorted(extra.items(), key=lambda x: -x[1]):
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
