"""A-NeRF training with and without the pose gradient (--opt_pose) at the config's own size (anerf_base: 16 poses x 192
rays, 96 + 48 samples), on the GPU.

Prints, with the card's name and power limit read in the same run:
  - ms / iteration of TrainStep without a pose layer and with one (pose layer, render gradient to the poses, kp_loss,
    both optimisers), in alternating timed windows (CUDA events, the same batch every iteration);
  - CUDA-event times, inside one iteration, of `danbo_anerf_embed_bwd` (coarse and fine pass) and of the three extra
    danbo_gemm_dgrad launches per pass that form the MLP's input gradient;
  - `danbo_anerf_embed_bwd` alone on the coarse pass's rows (20 launches, inputs far larger than L2): bytes it must move
    over its time, against the data sheet's 7.7 TB/s of HBM3e.

    python scripts/anerf_pose_bench.py [--out FILE]      (FILE also receives everything printed)
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
from danbo_b200 import feed as fd, kernels as K, params, pose_opt as po, skeleton as sk, synthetic as syn, training  # noqa: E402

HBM_BPS = 7.7e12


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return name, q


def make_caster(args, dev):
    attrs = {"skel_type": sk.SMPLSkeleton, "near": syn.NEAR, "far": syn.FAR, "n_views": 8, "rest_pose": syn.rest_pose()}
    _, kw, *_ = db.create_raycaster(args, attrs, device=dev)
    caster = kw["ray_caster"]
    caster.network.load_state_dict(syn.synth_state_dict(params.anerf_param_shapes(), 0), strict=False)
    return caster


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
    args = db.make_args("anerf_base", no_reload=True)
    n_poses, rpp = 16, 192
    S_c, S_f = args.N_samples, args.N_importance
    arrays = fd.synthetic_arrays(n_images=32, H=256, W=256, seed=0)
    feed = fd.RayFeed.from_arrays(arrays, syn.NEAR, syn.FAR, N_rand=n_poses * rpp, N_sample_images=n_poses, device=dev,
                                  seed=0, cam_idxs=np.arange(32) % 8)        # the caster's 8 frame codes (n_views)
    batch = feed.next_batch(torch.Generator(device=dev).manual_seed(0))
    plain = training.TrainStep(make_caster(args, dev), args)
    attrs = {"rest_pose": syn.rest_pose()[None], "betas": torch.zeros(1, 10).numpy(), "kp3d": arrays["kp3d"],
             "bones": arrays["bones"]}
    pose_optimizer, kw = po.create_popt(args, attrs, device=dev)
    posed = training.TrainStep(make_caster(args, dev), args, popt_kwargs=kw, pose_optimizer=pose_optimizer)
    torch.manual_seed(0)
    for step in (plain, posed):
        for _ in range(3):
            step(batch)
    torch.cuda.synchronize()
    ms = {"plain": [], "pose": []}
    for _ in range(cli.windows):
        ms["plain"].append(timed(plain, batch, cli.iters))
        ms["pose"].append(timed(posed, batch, cli.iters))
    med = {k: statistics.median(v) for k, v in ms.items()}
    say(f"anerf_base training, {n_poses} poses x {rpp} rays, {S_c}+{S_f} samples per ray")
    for k, label in (("plain", "without pose gradient"), ("pose", "with pose layer + pose gradient")):
        say(f"  {label:32s}: {med[k]:7.1f} ms / iteration ({1e3 / med[k]:.2f} it/s); windows {['%.1f' % v for v in ms[k]]}")
    say(f"  pose gradient costs {med['pose'] - med['plain']:+.1f} ms / iteration")
    st, launches = stage_times(posed, batch)
    st_plain, launches_plain = stage_times(plain, batch)
    eb, dx = st.get("anerf_embed_bwd", []), st.get("anerf_mlp_dx", [])
    say(f"  in one iteration: danbo_anerf_embed_bwd coarse {eb[0]:.3f} ms, fine {eb[1]:.3f} ms; extra dgrad launches "
        f"{len(dx)} totalling {sum(dx):.2f} ms ({', '.join('%.2f' % v for v in dx)}); launches {launches} vs {launches_plain}")
    # the kernel alone on the coarse pass's rows
    rows = n_poses * rpp * S_c
    caster = posed.caster
    rays = batch["ray_batch"].float().contiguous()
    skts = batch["skts"][::rpp].float().contiguous()
    cams = torch.zeros(rays.shape[0], device=dev, dtype=torch.int32)
    enc, _ = K.anerf_ray_encode(rays, skts, rpp, cams, caster._codes_with_mean(), caster._packed_mlp())
    z = torch.sort(torch.rand(rays.shape[0], S_c, device=dev) * (syn.FAR - syn.NEAR) + syn.NEAR, -1).values.contiguous()
    d_xd = torch.randn(rows, 432, device=dev)
    d_xv = torch.randn(rows, 648, device=dev)
    d_skts = torch.zeros_like(skts)
    for _ in range(3):
        K.anerf_embed_bwd(rays, S_c, z, skts, rpp, caster._align(), enc, 20., d_xd, d_xv, d_skts)
    n_rep = 20
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n_rep):
        K.anerf_embed_bwd(rays, S_c, z, skts, rpp, caster._align(), enc, 20., d_xd, d_xv, d_skts)
    e1.record()
    torch.cuda.synchronize()
    t = e0.elapsed_time(e1) / n_rep * 1e-3
    nbytes = rows * (432 + 648 + 1) * 4 + rays.shape[0] * (648 + 8) * 4      # d xd, d xv, z; per ray: enc, ray
    say(f"  danbo_anerf_embed_bwd alone, {rows} rows: {t * 1e3:.3f} ms, {nbytes / 1e9:.3f} GB -> {nbytes / t / 1e12:.2f} TB/s "
        f"= {100 * nbytes / t / HBM_BPS:.0f} % of 7.7 TB/s")
    say(json.dumps({"card": name, "limits": limits, "ms_plain": med["plain"], "ms_pose": med["pose"],
                    "embed_bwd_ms_in_step": eb, "dx_dgrad_ms_in_step": dx, "embed_bwd_alone_ms": t * 1e3,
                    "embed_bwd_bytes": nbytes, "windows": ms}))
    if cli.out:
        os.makedirs(os.path.dirname(os.path.abspath(cli.out)), exist_ok=True)
        with open(cli.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
