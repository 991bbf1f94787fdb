"""Pose refinement on the perfcap configs (root-local view directions, --opt_pose) at training size, on the GPU.

Prints, with the card's name and power limit read in the same run:
  - ms / iteration of eager TrainStep at 16 poses x 192 rays (danbo_fast: 32 + 16 samples) in three arms, timed in
    alternating windows (CUDA events, the same batch every iteration):
      perfcap danbo_fast with a pose layer, perfcap danbo_fast without one, and h36m_zju danbo_fast with a pose layer.
    The last arm is the control: it differs from the first only in the view branch, so the difference of the two is
    what the root-local view directions and their pose gradient (`danbo_view_root_bwd`) cost;
  - kernel launches per iteration of each arm, and the CUDA-event time of `danbo_view_root_bwd` inside one iteration
    (events around the launch, so it includes the host's argument checks and enqueue);
  - `danbo_view_root_bwd` alone at 3 072 and 65 536 rays.  Its d_ray_bias inputs rotate through 256 MB of buffers,
    so every launch reads them from HBM rather than L2.

    python scripts/perfcap_pose_bench.py [--out FILE]      (FILE also receives everything printed)
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import danbo_b200 as db  # noqa: E402
from danbo_b200 import feed as fd, kernels as K, pose_opt as po, skeleton as sk, synthetic as syn, training  # noqa: E402

PERFCAP = dict(view_type="relray", ray_tr_type="root_local", nerf_type="graph")   # configs/perfcap/danbo_*.txt
FMA_PER_RAY = 128 * 27                                                               # g = W_v[:, 256:283]^T d_ray_bias


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return name, q


def make_step(flags, arrays, dev, pose):
    args = db.make_args("danbo_fast", no_reload=True, opt_pose=pose, **flags)
    attrs = {"skel_type": sk.SMPLSkeleton, "near": syn.NEAR, "far": syn.FAR, "n_views": 8, "rest_pose": syn.rest_pose()}
    _, kw, *_ = db.create_raycaster(args, attrs, device=dev)
    caster = kw["ray_caster"]
    caster.network.load_state_dict(syn.synthetic_params(0))
    caster.train()
    if not pose:
        return training.TrainStep(caster, args)
    pattrs = {"rest_pose": syn.rest_pose()[None], "betas": torch.zeros(1, 10).numpy(), "kp3d": arrays["kp3d"],
              "bones": arrays["bones"]}
    pose_optimizer, pkw = po.create_popt(args, pattrs, device=dev)
    return training.TrainStep(caster, args, popt_kwargs=pkw, pose_optimizer=pose_optimizer)


def timed(step, batch, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        step(batch)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def stage_times(step, batch):
    K.PROFILE = {"mlp": [], "launches": 0, "stages": []}
    try:
        step(batch)
        torch.cuda.synchronize()
        out = {}
        for name, a, b in K.PROFILE["stages"]:
            out.setdefault(name, []).append(a.elapsed_time(b))
        return out, K.PROFILE["launches"]
    finally:
        K.PROFILE = None


def kernel_alone(n, skts, rpp, w_view, dev):
    """-> (us per launch, bytes per launch) of danbo_view_root_bwd over n rays, d_ray_bias cycling through >= 256 MB.
    The launches are captured in one CUDA graph and replayed, so the time is the kernels', not the host's
    per-launch argument checks and enqueue."""
    per = n * 128 * 4
    k = max(2, -(-(256 << 20) // per))
    n_rep = max(64, k)                                  # every launch of a replay reads a different buffer
    pool = torch.randn(k, n, 128, device=dev)
    g = torch.Generator(device=dev).manual_seed(1)
    rays = torch.randn(n, 11, device=dev, generator=g)
    d_skts = torch.zeros_like(skts)
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        for i in range(3):
            K.view_root_bwd(rays, skts, rpp, w_view, pool[i % k], d_skts)
    torch.cuda.current_stream(dev).wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for i in range(n_rep):
            K.view_root_bwd(rays, skts, rpp, w_view, pool[i % k], d_skts)
    graph.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(3):
        graph.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / (3 * n_rep) * 1e3, per + n * 3 * 4


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--windows", type=int, default=3)
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
    arms = {"perfcap_pose": make_step(PERFCAP, arrays, dev, True),
            "perfcap_plain": make_step(PERFCAP, arrays, dev, False),
            "h36m_pose": make_step({}, arrays, dev, True)}
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
    launches, in_step = {}, {}
    for k, step in arms.items():
        st, launches[k] = stage_times(step, batch)
        in_step[k] = st.get("view_root_bwd", [])
    say(f"danbo_fast eager training, {n_poses} poses x {rpp} rays, 32+16 samples per ray")
    labels = {"perfcap_pose": "perfcap, pose layer", "perfcap_plain": "perfcap, no pose layer",
              "h36m_pose": "h36m_zju, pose layer (control)"}
    for k, label in labels.items():
        say(f"  {label:31s}: {med[k]:7.1f} ms / iteration; {launches[k]} launches; windows "
            f"{['%.1f' % v for v in ms[k]]}; danbo_view_root_bwd in the step {['%.4f ms' % v for v in in_step[k]]}")
    say(f"  perfcap pose layer vs none: {med['perfcap_pose'] - med['perfcap_plain']:+.1f} ms; "
        f"vs the h36m_zju control: {med['perfcap_pose'] - med['h36m_pose']:+.1f} ms")
    step = arms["perfcap_pose"]
    skts = batch["skts"][::rpp].float().contiguous()
    w_view = step.caster.network.views_linears[0].weight.detach()
    alone = {}
    for n in (3072, 65536):
        us, nbytes = kernel_alone(n, skts, n // n_poses, w_view, dev)
        alone[n] = us
        say(f"  danbo_view_root_bwd alone, {n} rays: {us:.2f} us / launch; {nbytes / 1e6:.2f} MB from HBM -> "
            f"{nbytes / us / 1e6:.2f} TB/s; {n * FMA_PER_RAY / 1e6:.1f} M FMA -> {n * FMA_PER_RAY / us / 1e6:.2f} TFMA/s")
    say(json.dumps({"card": name, "limits": limits, "ms": med, "windows": ms, "launches": launches,
                    "view_root_bwd_ms_in_step": in_step, "view_root_bwd_alone_us": alone}))
    if cli.out:
        os.makedirs(os.path.dirname(os.path.abspath(cli.out)), exist_ok=True)
        with open(cli.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
