"""A-NeRF training with one network (anerf_base, single_net) and with a separate fine network (anerf_h,
single_net = False) at the config's own size, on the GPU: 16 poses x 192 rays, 96 + 48 samples, perturb 1,
raw_noise_std 1, L1 loss.  anerf_h evaluates its coarse network on the 96 coarse samples and its fine network on all
144 merged samples, so its MLPs run 240 rows per ray where anerf_base's run 144.

Prints, with the card's name, power limit and max SM clock read in the same run:
  - ms / iteration of `TrainStep` for each arm, in alternating timed windows (CUDA events, the same batch every
    iteration, after warm-up iterations of both arms);
  - the library's kernel launches per iteration (`kernels.PROFILE`) and `torch.cuda.max_memory_allocated` over one
    iteration of each arm (both arms' casters stay resident, so each figure includes the other arm's weights, Adam
    state and packed-weight workspaces);
  - for anerf_h, CUDA-event times of the stages of one iteration, split into the coarse and the fine network's pass;
  - with --profile DIR, a separate torch.profiler run of anerf_h iterations: its CUDA kernel table goes to DIR.

    python scripts/anerf_h_train_bench.py [--out FILE] [--profile DIR] [--arms anerf_base,anerf_h]
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
from danbo_b200 import feed as fd, kernels as K, params, skeleton as sk, synthetic as syn, training  # noqa: E402

N_POSES, RPP = 16, 192


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return name, q


def make_step(arm, dev):
    args = db.make_args("anerf_base", no_reload=True, single_net=(arm == "anerf_base"))
    attrs = {"skel_type": sk.SMPLSkeleton, "near": syn.NEAR, "far": syn.FAR, "n_views": 8, "rest_pose": syn.rest_pose()}
    _, kw, *_ = db.create_raycaster(args, attrs, device=dev)
    caster = kw["ray_caster"]
    caster.network.load_state_dict(syn.synth_state_dict(params.anerf_param_shapes(), 0), strict=False)
    if caster.network_fine is not caster.network:
        caster.network_fine.load_state_dict(syn.synth_state_dict(params.anerf_param_shapes(), 1), strict=False)
    return training.TrainStep(caster, args), args


def timed(step, batch, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        step(batch)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def launches_and_memory(step, batch):
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    K.PROFILE = {"mlp": [], "launches": 0}
    try:
        step(batch)
        torch.cuda.synchronize()
        return K.PROFILE["launches"], torch.cuda.max_memory_allocated()
    finally:
        K.PROFILE = None


def stage_times(step, batch):
    """One iteration with CUDA events around every stage the library times (forward) and around each compositing
    backward and MLP backward call -> [(name, ms)] in call order."""
    wrapped = ("composite_bwd", "anerf_mlp_backward")
    orig = {n: getattr(K, n) for n in wrapped}

    def timed_call(name, fn):
        def call(*a, **kw):
            with K._Timed(name):
                return fn(*a, **kw)
        return call

    K.PROFILE = {"mlp": [], "launches": 0, "stages": []}
    for n in wrapped:
        setattr(K, n, timed_call(n, orig[n]))
    try:
        step(batch)
        torch.cuda.synchronize()
        return [(name, a.elapsed_time(b)) for name, a, b in K.PROFILE["stages"]]
    finally:
        K.PROFILE = None
        for n in wrapped:
            setattr(K, n, orig[n])


def split_passes(stages):
    """anerf_h call order: forward coarse stages up to the coarse composite_resample, then the fine network's stages;
    backward: composite_bwd fine then coarse, anerf_mlp_backward coarse then fine."""
    coarse, fine, fwd_done = 0.0, 0.0, False
    seen = {}
    for name, ms in stages:
        i = seen[name] = seen.get(name, -1) + 1
        if name == "composite_bwd":
            is_fine = i == 0
        elif name == "anerf_mlp_backward":
            is_fine = i == 1
        elif name == "anerf_mlp_dx":                       # only with a pose gradient (not in this benchmark)
            continue
        else:
            is_fine = fwd_done
            fwd_done = fwd_done or name == "composite_resample"
        if is_fine:
            fine += ms
        else:
            coarse += ms
    return coarse, fine


def profile_run(step, batch, out_dir, iters=2):
    from torch.profiler import ProfilerActivity, profile
    os.makedirs(out_dir, exist_ok=True)
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            step(batch)
        torch.cuda.synchronize()
    table = prof.key_averages().table(sort_by="cuda_time_total", row_limit=40)
    with open(os.path.join(out_dir, "anerf_h_train_profile.txt"), "w") as f:
        f.write(f"# torch.profiler, {iters} anerf_h TrainStep iterations, {N_POSES} poses x {RPP} rays, 96+48 samples\n")
        f.write(table + "\n")
    return table


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write everything printed to this file")
    ap.add_argument("--profile", default=None, metavar="DIR", help="torch.profiler run of anerf_h, table into DIR")
    ap.add_argument("--arms", default="anerf_base,anerf_h")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--iters", type=int, default=5, help="iterations per timed window")
    ap.add_argument("--windows", type=int, default=3, help="alternating timed windows per arm")
    cli = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("needs a CUDA device")
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    dev = torch.device("cuda", 0)
    name, limits = card()
    say(f"card: {name}; power.limit, clocks.max.sm: {limits}")
    arms = cli.arms.split(",")
    arrays = fd.synthetic_arrays(n_images=32, H=256, W=256, seed=0)
    feed = fd.RayFeed.from_arrays(arrays, syn.NEAR, syn.FAR, N_rand=N_POSES * RPP, N_sample_images=N_POSES, device=dev,
                                  seed=0, cam_idxs=np.arange(32) % 8)        # the caster's 8 frame codes (n_views)
    batch = feed.next_batch(torch.Generator(device=dev).manual_seed(0))
    steps = {arm: make_step(arm, dev) for arm in arms}
    args = steps[arms[0]][1]
    say(f"{N_POSES} poses x {RPP} rays, {args.N_samples}+{args.N_importance} samples, perturb {args.perturb}, "
        f"raw_noise_std {args.raw_noise_std}, loss {args.loss_fn}; {cli.warmup} warm-up iterations per arm, then "
        f"{cli.windows} alternating windows of {cli.iters} iterations")
    torch.manual_seed(0)
    for arm in arms:
        for _ in range(cli.warmup):
            steps[arm][0](batch)
    torch.cuda.synchronize()
    ms = {arm: [] for arm in arms}
    for _ in range(cli.windows):
        for arm in arms:
            ms[arm].append(timed(steps[arm][0], batch, cli.iters))
    res = {"card": name, "limits": limits, "arms": {}}
    for arm in arms:
        med = statistics.median(ms[arm])
        n_launch, peak = launches_and_memory(steps[arm][0], batch)
        loss = float(steps[arm][0](batch)[0])
        res["arms"][arm] = {"ms_per_iter": med, "windows": ms[arm], "launches_per_iter": n_launch, "peak_bytes": peak,
                            "loss": loss}
        say(f"  {arm:10s}: {med:7.1f} ms / iteration ({1e3 / med:.2f} it/s); windows {['%.1f' % v for v in ms[arm]]}; "
            f"{n_launch} launches / iteration; peak memory {peak / 2 ** 30:.2f} GiB; loss {loss:.4f}")
    if "anerf_base" in res["arms"] and "anerf_h" in res["arms"]:
        a, h = res["arms"]["anerf_base"]["ms_per_iter"], res["arms"]["anerf_h"]["ms_per_iter"]
        say(f"  anerf_h / anerf_base: {h / a:.2f}x")
    if "anerf_h" in arms:
        st = stage_times(steps["anerf_h"][0], batch)
        coarse, fine = split_passes(st)
        res["anerf_h_stages"] = st
        say(f"  anerf_h, one iteration, CUDA events per stage: coarse network {coarse:.1f} ms, fine network {fine:.1f} ms "
            f"(stages: {', '.join('%s %.2f' % (n, t) for n, t in st)})")
        res["anerf_h_coarse_ms"], res["anerf_h_fine_ms"] = coarse, fine
        if cli.profile:
            profile_run(steps["anerf_h"][0], batch, cli.profile)
            say(f"  torch.profiler table: {os.path.join(cli.profile, 'anerf_h_train_profile.txt')}")
    say(json.dumps(res))
    if cli.out:
        os.makedirs(os.path.dirname(os.path.abspath(cli.out)), exist_ok=True)
        with open(cli.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
