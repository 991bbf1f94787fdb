#!/usr/bin/env python
"""Benchmark of the DANBO hot path on B200 (contract: see the task statement / DESIGN.md §Measurement).

    python bench.py --gpus 1 --steps 10 --warmup 3                 # this repo's CUDA path
    python bench.py --gpus 1 --steps 10 --warmup 3 --dump-outputs DIR   # ... and write what the last timed step returned
    python bench.py --impl reference --steps 2 --warmup 1           # the unmodified reference (baseline/_ref) on host cores
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[1]): DANBO `danbo_fast` (32 coarse + 16 fine samples, per-part volume near/far),
512x512 render of one synthetic 24-joint pose, random-init weights; rays restricted to the image box of the pose's
bounding cylinder exactly as the reference's render_path does.  One step = one image through the whole path
(near/far -> sampling -> bone transform/mask -> gather + aggregation net -> fused MLP -> composite -> resample ->
fine pass -> merged composite).  metric = rays/s.

  value : steps timed with CUDA events, inputs already resident in HBM.
  e2e   : the same call through the public `ray_caster(...)` API with pinned HOST inputs, H2D of the rays and D2H
          of the pixels inside the timed region.
At N > 1 every rank renders its own copy of the same image and the pixels are all-gathered (weak scaling).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

MLP_FLOP_PER_SAMPLE = 1354752          # SURVEY §8(a) row M1 (FlopCounter-verified): 677 376 MAC / sample
# dram__bytes_read.sum + dram__bytes_write.sum of one mlp_kernel launch from the ncu --set full capture under profiles/
# (profiles/r2_ncu_render_summary.txt: the 1.03 M-row fine-pass launch of the whole 261 121-ray image; 512 B/row of X tile
# read once - K padded 208 -> 256 - + 16 B/row of output).  A constant from that capture, not measured in the run.
MLP_DRAM_BYTES_PER_LAUNCH = 522275000 + 18544896
H = W = 512
PRESET = "danbo_fast"


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax = float(f[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


def build_scene(rank, device):
    import danbo_b200 as db
    from danbo_b200 import synthetic as syn, skeleton as sk
    args = db.make_args(PRESET, no_reload=True)
    data_attrs = {"skel_type": sk.SMPLSkeleton, "near": syn.NEAR, "far": syn.FAR, "n_views": 8,
                  "rest_pose": syn.rest_pose()}
    torch.manual_seed(0)
    _, kw_test, *_ = db.create_raycaster(args, data_attrs, device=device)
    caster = kw_test["ray_caster"]
    caster.network.load_state_dict(syn.synthetic_params(0))      # random-init weights, same on every rank
    caster.eval()
    pose = syn.make_pose(3)
    # weak scaling = the SAME work on every GPU: each rank renders its own copy of the configs[1] image (same pose, same
    # camera), so the per-N figures differ only by what N ranks cost (the pixel exchange, clocks), not by which view a
    # rank happened to get (bullet-time views of one pose differ by up to 15 % in rays inside the body's boxes)
    c2w = syn.bullet_time_cameras(syn.camera(), 8)[0]
    batch = syn.render_batch(pose, H, W, c2w=c2w, cam_idx=0)
    return caster, args, batch


def caster_kwargs(args, batch, device=None):
    mv = (lambda t: t.to(device)) if device is not None else (lambda t: t)
    return dict(N_samples=args.N_samples, kp_batch=mv(batch["kp_batch"]), skts=mv(batch["skts"]), cyls=mv(batch["cyls"]),
                bones=mv(batch["bones"]), cams=mv(batch["cams"]), N_uniques=1, perturb=False,
                N_importance=args.N_importance, raw_noise_std=0., nanmean_chunk=args.chunk)


DUMP_BYTES = 64 * 10 ** 6          # all files together, .npy headers included
NPY_HEADER_BYTES = 1024            # an upper bound for the header np.save writes for these arrays


def dump_outputs(ret, out_dir, budget=DUMP_BYTES, seed=0):
    """Writes every array of a render call's returned dict as `out_dir/<name>.npy` (float64 stays float64, other
    types become float32).  All arrays have one row per ray; when together they would exceed `budget` bytes, each keeps
    the same rays: a fixed, seeded random sample in ray order, as many as fit.  Equal inputs thus give files that can be
    compared one to one between two builds."""
    arrays = {k: v.detach().cpu() for k, v in ret.items()}
    arrays = {k: v if v.dtype == torch.float64 else v.float() for k, v in arrays.items()}
    n = {v.shape[0] for v in arrays.values()}
    assert len(n) == 1, {k: tuple(v.shape) for k, v in arrays.items()}
    n = n.pop()
    row_bytes = sum(v[:1].numel() * v.element_size() for v in arrays.values())
    keep = min(n, max(budget - NPY_HEADER_BYTES * len(arrays), 0) // max(row_bytes, 1))
    if keep < n:
        rows = torch.randperm(n, generator=torch.Generator().manual_seed(seed))[:keep].sort().values
        arrays = {k: v[rows] for k, v in arrays.items()}
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), v.numpy())


def _mark(msg):
    if os.environ.get("DANBO_BENCH_VERBOSE"):
        sys.stderr.write(f"[bench rank {os.environ.get('RANK', '0')} t={time.perf_counter():.1f}] {msg}\n")
        sys.stderr.flush()


def run_ours(opt):
    import torch.distributed as dist
    import danbo_b200 as db
    from danbo_b200 import parallel, kernels
    rank, world, local = parallel.init_distributed()
    if world != opt.gpus:
        opt.gpus = world
    device = torch.device("cuda", local)
    torch.cuda.set_device(device)
    _mark(f"init done world={world}")
    caster, args, batch = build_scene(rank, device)
    _mark("scene built")
    n_rays = batch["ray_batch"].shape[0]
    rays_dev = batch["ray_batch"].to(device)
    kw_dev = caster_kwargs(args, batch, device)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)       # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # every rank renders a fixed number of rays per step: exchange the shard sizes once, not per step
    shard_sizes = parallel.gather_sizes(n_rays, device) if world > 1 else None

    # N > 1: the pixel all-gather of step i runs on a communication stream while step i+1 renders (the exchange is
    # 5 MB per rank; issued on the render stream it is a per-step rendezvous of all ranks).  The timed region ends only
    # after the last gather has completed.
    main_stream = torch.cuda.current_stream()
    comm = torch.cuda.Stream() if world > 1 else None
    rendered = [torch.cuda.Event() for _ in range(2)]
    gathered = [None, None]

    def step_device(graphed=True, i=0):
        ret = caster.render_graphed(rays_dev, **kw_dev) if graphed else caster(rays_dev, **kw_dev)
        pix = parallel.pack_pixels(ret)                      # a fresh (n,5) tensor: the graph's static outputs are free again
        if world > 1:
            b = i & 1
            rendered[b].record(main_stream)
            with torch.cuda.stream(comm):
                comm.wait_event(rendered[b])
                gathered[b] = parallel.allgather_rows(pix, shard_sizes)
            pix.record_stream(comm)
        return ret

    def drain():
        if world > 1:
            main_stream.wait_stream(comm)

    # pinned host inputs for the end-to-end path
    rays_host = batch["ray_batch"].pin_memory()
    pix_host = torch.empty(n_rays, 5).pin_memory()
    kw_host = caster_kwargs(args, batch)

    def step_e2e():
        ret = caster.render_graphed(rays_host, **kw_host)   # H2D of the (n,11) ray batch happens inside
        pix = parallel.pack_pixels(ret)
        if world > 1:
            pix_all = parallel.allgather_rows(pix, shard_sizes)
        pix_host.copy_(pix, non_blocking=True)              # D2H of the 20 B / ray result
        torch.cuda.current_stream().synchronize()
        return pix_host

    for i in range(max(opt.warmup, 3)):
        step_device(i=i)
        flush.fill_(1)
    drain()
    _mark("warmup issued")
    barrier()
    _mark("warmup done")
    sampler = ClockSampler(local)
    sampler.start()
    kernels.PROFILE = {"mlp": [], "launches": 0}
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(opt.steps)]
    barrier()
    t_wall0 = time.perf_counter()
    tail0, tail1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for i in range(opt.steps):
        ev[i][0].record()
        ret = step_device(i=i)
        ev[i][1].record()
        flush.fill_(i)                                       # L2 flush between timed iterations (not timed)
    tail0.record()
    drain()                                                  # the last all-gather must have landed inside the timed region
    tail1.record()
    barrier()
    _mark("timed steps done")
    t_wall = time.perf_counter() - t_wall0
    # every rank renders the same whole image, so rank 0's outputs are the complete result; dumped before any later call
    # overwrites the graph's output buffers
    if opt.dump_outputs and rank == 0:
        dump_outputs(ret, opt.dump_outputs)
    dev_ms = sum(a.elapsed_time(b) for a, b in ev) + (tail0.elapsed_time(tail1) if world > 1 else 0.0)
    # the timed steps replay one CUDA graph; the same steps are run once more launch by launch with CUDA events around
    # the dominant kernel (and the launch counter on) for the roofline line
    for i in range(opt.steps):
        step_device(graphed=False, i=i)
        flush.fill_(i)
    drain()
    barrier()
    prof = kernels.PROFILE
    kernels.PROFILE = None
    mlp_ms = [a.elapsed_time(b) for a, b, _ in prof["mlp"]]
    mlp_rows = [int(c.item()) for _, _, c in prof["mlp"]]
    launches = prof["launches"] // max(opt.steps, 1) * opt.steps   # launches of the K timed steps (same sequence in the graph)
    # end-to-end (host buffers): every step copies its (n,11) ray batch from pinned host memory and reads its pixels back.
    # Steps are pipelined the way a serving loop runs them: a copy stream uploads the rays of step i+1 and downloads the
    # pixels of step i-1 while step i computes (double-buffered); the timed region is the whole K-step loop, L2 flush
    # writes included, closed by a wait on the last download.
    for _ in range(2):
        step_e2e()
    barrier()
    main, copy = torch.cuda.current_stream(), torch.cuda.Stream()
    rays_stage = [torch.empty_like(rays_dev) for _ in range(2)]
    # the pose tables (one pose: a few KB) and the per-ray camera indices are inputs of the call as well: they are uploaded
    # with the rays every step, from pinned host memory, and the call reads the uploaded copies
    pose_keys = ("kp_batch", "skts", "bones", "cyls")
    pose_host = {k: batch[k][:1].contiguous().pin_memory() for k in pose_keys}
    cams_host = batch["cams"].contiguous().pin_memory()
    pose_stage = [{k: torch.empty_like(v, device=device) for k, v in pose_host.items()} for _ in range(2)]
    cams_stage = [torch.empty_like(cams_host, device=device) for _ in range(2)]
    kw_stage = [dict(kw_dev, cams=cams_stage[b], **{k: pose_stage[b][k].expand(n_rays, *pose_stage[b][k].shape[1:])
                                                   for k in pose_keys}) for b in range(2)]
    h2d_bytes = int(rays_host.numel() * 4 + cams_host.numel() * 8 + sum(v.numel() * 4 for v in pose_host.values()))
    pix_stage = [torch.empty(n_rays, 5, device=device) for _ in range(2)]
    pix_hosts = [torch.empty(n_rays, 5).pin_memory() for _ in range(2)]
    up_done = [torch.cuda.Event() for _ in range(2)]
    used = [torch.cuda.Event() for _ in range(2)]          # compute of the step that read rays_stage[b] / wrote pix_stage[b]
    down_done = [torch.cuda.Event() for _ in range(2)]

    def upload(i):
        b = i & 1
        with torch.cuda.stream(copy):
            if i >= 2:
                copy.wait_event(used[b])
            rays_stage[b].copy_(rays_host, non_blocking=True)
            cams_stage[b].copy_(cams_host, non_blocking=True)
            for k in pose_keys:
                pose_stage[b][k].copy_(pose_host[k], non_blocking=True)
            up_done[b].record(copy)

    def run_pipelined(k):
        upload(0)
        for i in range(k):
            b = i & 1
            main.wait_event(up_done[b])
            if i >= 2:
                main.wait_event(down_done[b])                # pix_stage[b] has been read out
            ret = caster.render_graphed(rays_stage[b], **kw_stage[b])
            pix = parallel.pack_pixels(ret)
            pix_stage[b].copy_(pix)
            used[b].record(main)
            if world > 1:                                    # the exchange of step i overlaps step i+1, as in the device loop
                with torch.cuda.stream(comm):
                    comm.wait_event(used[b])
                    gathered[b] = parallel.allgather_rows(pix, shard_sizes)
                pix.record_stream(comm)
            if i + 1 < k:
                upload(i + 1)
            with torch.cuda.stream(copy):
                copy.wait_event(used[b])
                pix_hosts[b].copy_(pix_stage[b], non_blocking=True)
                down_done[b].record(copy)
            flush.fill_(i)
        main.wait_stream(copy)
        drain()

    run_pipelined(3)
    barrier()
    e2e0, e2e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2e0.record()
    run_pipelined(opt.steps)
    e2e1.record()
    barrier()
    _mark("e2e done")
    e2e_ms = e2e0.elapsed_time(e2e1)
    pix_host = pix_hosts[(opt.steps - 1) & 1]
    clocks = sampler.stop()
    t = torch.tensor([dev_ms, e2e_ms], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms = float(t[0]), float(t[1])
    del caster, rays_dev, kw_dev, flush
    torch.cuda.empty_cache()
    try:
        _mark("train start")
        train_info = ({"skipped": "DANBO_BENCH_SKIP_TRAIN=1"} if os.environ.get("DANBO_BENCH_SKIP_TRAIN", "") == "1" else
                      run_train(rank, world, device, max(opt.steps, 5), opt.warmup))
        _mark("train done")
    except Exception as exc:                                  # the headline render number must survive a training failure
        train_info = {"error": repr(exc)}
    configs = {}
    if os.environ.get("DANBO_BENCH_SKIP_CONFIGS", "") != "1":
        for key, fn in (("config4_anerf_1024", run_config4), ("config5_bullet_time_lattice", run_config5)):
            torch.cuda.empty_cache()
            try:
                _mark(key + " start")
                configs[key] = fn(rank, world, device)
            except Exception as exc:
                configs[key] = {"error": repr(exc)}
    if rank != 0:
        _finish(world)
        return
    peaks = measured_peaks()
    total_rays = (sum(shard_sizes) if world > 1 else n_rays) * opt.steps       # every rank renders its own view
    value = total_rays / (dev_ms / 1e3)
    flops = MLP_FLOP_PER_SAMPLE * float(sum(mlp_rows))
    mlp_s = sum(mlp_ms) / 1e3
    achieved = flops / mlp_s / 1e12 if mlp_s > 0 else 0.0
    # every MLP launch is timed alone by its own event pair (0.3-1 ms each, lighter kernels in between): the burst
    # figure is the comparable peak; the fraction of the sustained figure is reported next to it
    peak = peaks["bf16_tflops"]
    samples_per_ray = args.N_samples + args.N_importance
    line = {
        "metric": "DANBO render rays/s (fwd+composite)", "value": value, "unit": "rays/s", "n_gpus": world,
        "steps": opt.steps, "warmup": max(opt.warmup, 3), "ms_per_step": dev_ms / opt.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16 (tensor-core MLP, fp32 accumulate); fp32 elsewhere; fp64 box test",
        "data": "synthetic",
        "config": workload_config(args, n_rays),
        "run": {"parallelism": (f"1 image (the same view) per GPU x {world}; NCCL all-gather of every step's pixels on a "
                                "communication stream, overlapped with the next step's render") if world > 1 else "single GPU",
                "rays_this_view": n_rays,
                "l2": "256 MiB buffer written between timed steps (untimed)",
                "launch": "each step replays one CUDA graph of the call's fixed launch sequence",
                "wall_ms_per_step_incl_flush": t_wall * 1e3 / opt.steps},
        "e2e": {"value": total_rays / (e2e_ms / 1e3), "unit": "rays/s", "h2d_bytes_per_step": h2d_bytes,
                "d2h_bytes_per_step": int(pix_host.numel() * 4),
                "pipeline": "ray_caster call per step on rays, camera indices and pose tables uploaded from pinned host memory; uploads / downloads of "
                            "neighbouring steps overlap compute on a copy stream (double-buffered); timed over the whole loop"},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": {"bound": "tensor", "kernel": "danbo::mlp::mlp_kernel<true, true> (CTA pairs, cta_group::2)", "achieved": achieved,
                     "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak if peak else None, "traffic": MLP_DRAM_BYTES_PER_LAUNCH,
                     "traffic_source": "profiles/r2_ncu_render_summary.txt (ncu --set full, dram__bytes read + write of the fine-pass "
                                       "launch, 1.03 M rows = 525 B/row); not measured in this run",
                     "peak_source": f"MEASURED_PEAKS.json bf16_tflops, burst: each launch timed alone ({peaks['source']})",
                     "frac_of_sustained": achieved / peaks["bf16_tflops_sustained"],
                     "launches_timed": len(mlp_ms), "rows_per_step": float(sum(mlp_rows)) / max(opt.steps, 1),
                     "dense_samples_per_step": n_rays * samples_per_ray,
                     "note": "achieved = 1 354 752 FLOP x rows the launch processed / CUDA-event time of the launch; rows = "
                             "samples seen by at least one bone (+1 per ray); the rest reuse the ray's empty-sample output"},
    }
    line["train"] = train_info
    line["configs"] = configs
    if world == 1:
        line["cpu_baseline"] = cpu_baseline(sample_rays=REF_SAMPLE_RAYS, repeats=1)     # ~8 s on the box's 16 host cores
    print(json.dumps(line))
    _finish(world)


def _finish(world):
    """End of a rank.  At N > 1 the captured training graphs hold NCCL nodes; tearing the process group down (or letting the
    interpreter destroy those graphs) while they are alive deadlocks in NCCL's teardown - measured: the 8-rank job printed
    its line and then hung until the driver's limit.  So: rendezvous, flush, and leave without running destructors; the
    communicator and the graphs die with the process."""
    if world <= 1:
        return
    import torch.distributed as dist
    dist.barrier()
    torch.cuda.synchronize()
    sys.stdout.flush()
    sys.stderr.flush()
    os._exit(0)


_KEEP_ALIVE = []


def run_train(rank, world, device, steps, warmup):
    """BASELINE configs[2]: danbo_base with --N_samples 64 --N_importance 16, 3072 rays (16 poses x 192), forward +
    backward + Adam, data-parallel over the ray batch (each rank takes 16/world poses) with one all-reduce of the flat
    gradient bucket.  Returns iterations/s over the whole job."""
    import torch.distributed as dist
    import danbo_b200 as db
    from danbo_b200 import synthetic as syn, skeleton as sk, training
    args = db.make_args("danbo_cfg3", no_reload=True)
    data_attrs = {"skel_type": sk.SMPLSkeleton, "near": syn.NEAR, "far": syn.FAR, "n_views": 8, "rest_pose": syn.rest_pose()}
    _, kw_test, *_ = db.create_raycaster(args, data_attrs, device=device)
    caster = kw_test["ray_caster"]
    caster.network.load_state_dict(syn.synthetic_params(0))
    n_poses, rpp = 16, 192
    full = syn.training_batch(n_poses, rpp, seed=0)
    cfg = ("danbo_base --N_samples 64 --N_importance 16, 16 poses x 192 rays, perturb=1, raw_noise_std=1, L1 + "
           "soft-softmax + volume-scale losses, Adam 5e-4; whole iteration (fwd, losses, bwd, NCCL all-reduce of the flat "
           "9.8 MB gradient bucket, single-launch Adam) replayed as one CUDA graph")

    def measure(batch, tag):
        step = training.TrainStep(caster, args, world_size=world, graph=True)
        _KEEP_ALIVE.append(step)      # its captured graph holds NCCL nodes: never destroyed while collectives are in flight
        torch.manual_seed(1234 + rank)
        for _ in range(max(warmup, 3)):
            step(batch)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            loss, _ = step(batch)
        e1.record()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1), float(loss)], device=device, dtype=torch.float64)
        if world > 1:
            ms = t[:1].clone()
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            ls = t[1:].clone()
            dist.all_reduce(ls)                             # mean over ranks = the loss of the global batch
            t = torch.cat([ms, ls / world])
        return float(t[0]) / steps, float(t[1]), bool(step._graph_whole)

    # strong scaling: the 3072-ray batch of config #3 split over the ranks (16 / world poses each)
    per = max(n_poses // world, 1)
    lo = (rank % (n_poses // per)) * per * rpp
    batch = {k: (v[lo:lo + per * rpp].to(device) if torch.is_tensor(v) else v) for k, v in full.items()}
    batch["N_uniques"] = per
    ms, loss, whole = measure(batch, "strong")
    info = {"metric": "training iterations/s (fwd+bwd+Adam)", "value": 1e3 / ms, "unit": "it/s", "ms_per_iter": ms,
            "global_rays": per * rpp * world, "rays_per_gpu": per * rpp, "samples_per_ray": args.N_samples + args.N_importance,
            "scaling": "strong" if world <= n_poses else "weak", "loss": loss, "loss_note": "mean over ranks after the "
            "timed iterations, all starting from the same weights: equal across N up to the draws", "whole_iteration_graphed": whole,
            "config": cfg}
    if world > 1:
        # weak scaling: every rank keeps a full 3072-ray batch (its own poses), global batch = world x 3072 rays
        caster.network.load_state_dict(syn.synthetic_params(0))
        own = syn.training_batch(n_poses, rpp, seed=100 + rank)
        b2 = {k: (v.to(device) if torch.is_tensor(v) else v) for k, v in own.items()}
        b2["N_uniques"] = n_poses
        ms2, loss2, _ = measure(b2, "weak")
        info["weak"] = {"value": 1e3 / ms2, "unit": "it/s", "ms_per_iter": ms2, "rays_per_gpu": n_poses * rpp,
                        "global_rays": n_poses * rpp * world, "rays_per_s": n_poses * rpp * world * 1e3 / ms2, "loss": loss2}
    else:
        info["rays_per_s"] = n_poses * rpp * 1e3 / ms
    return info


def _max_over_ranks(ms, device, world):
    import torch.distributed as dist
    t = torch.tensor([ms], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t[0])


def run_config4(rank, world, device, reps=2, H4=1024):
    """BASELINE configs[3]: A-NeRF anerf_base (relative-encoding MLP, no GNN) 1024x1024 render of ONE image, 96+48
    samples, its rays sharded across the ranks in chunk-aligned ranges (`parallel.render_sharded`, the reference's
    4096-ray chunks of core/trainer.py:75-90 dealt to GPUs) + one all-gather of the pixels: strong scaling."""
    import torch.distributed as dist
    import danbo_b200 as db
    from danbo_b200 import synthetic as syn, skeleton as sk, params, parallel
    args = db.make_args("anerf_base", no_reload=True)
    attrs = {"skel_type": sk.SMPLSkeleton, "near": syn.NEAR, "far": syn.FAR, "n_views": 8, "rest_pose": syn.rest_pose()}
    _, kw_test, *_ = db.create_raycaster(args, attrs, device=device)
    caster = kw_test["ray_caster"]
    caster.network.load_state_dict(syn.synth_state_dict(params.anerf_param_shapes(), 0), strict=False)
    caster.eval()
    b = syn.render_batch(syn.make_pose(3), H4, H4)
    rays = b["ray_batch"].to(device)
    n = rays.shape[0]
    tkw = {k: b[k].to(device) for k in ("kp_batch", "skts", "cyls", "bones", "cams")}
    okw = dict(N_samples=args.N_samples, N_uniques=1, perturb=False, N_importance=args.N_importance, raw_noise_std=0.,
               nerf_type="nerf")
    lo, hi = parallel.shard_range(n, rank, world, align=args.chunk)
    sizes = [b_ - a_ for a_, b_ in (parallel.shard_range(n, r, world, align=args.chunk) for r in range(world))]

    def image():
        ret = caster(rays[lo:hi], nanmean_chunk=args.chunk, **{k: v[lo:hi] for k, v in tkw.items()}, **okw)
        pix = parallel.pack_pixels(ret)
        e_a, e_b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e_a.record()
        full = parallel.allgather_rows(pix, sizes) if world > 1 else pix
        e_b.record()
        return full, (e_a, e_b)
    image()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    gathers = []
    for _ in range(reps):
        full, ev = image()
        gathers.append(ev)
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ms = _max_over_ranks(e0.elapsed_time(e1) / reps, device, world)
    coll = _max_over_ranks(sum(a_.elapsed_time(b_) for a_, b_ in gathers) / reps, device, world)
    S_t = args.N_samples + args.N_importance
    return {"workload": f"anerf_base {H4}x{H4} render, one synthetic pose, {args.N_samples}+{args.N_importance} samples/ray, "
                        f"box-restricted rays ({n} rays), rays sharded across {world} GPU(s) in {args.chunk}-ray chunks",
            "n_gpus": world, "scaling": "strong", "rays": n, "rays_this_rank": hi - lo, "ms_per_image": ms,
            "value": n / (ms / 1e3), "unit": "rays/s", "allgather_ms_per_image": coll,
            "tensor_tflops_whole_job": 4536000.0 * n * S_t / (ms / 1e3) / 1e12,
            "pixels_finite": bool(torch.isfinite(full).all()), "reps": reps}


def run_config5(rank, world, device, n_poses=100, res=255):
    """BASELINE configs[4]: bullet-time render of 100 synthetic poses at 512x512 (danbo_fast; images dealt round robin to
    the ranks, one all-gather of the finished images) plus a 256^3 density lattice for mesh extraction (danbo_fast field;
    z-slabs of the lattice split across the ranks, one all-gather)."""
    import torch.distributed as dist
    import danbo_b200 as db
    from danbo_b200 import synthetic as syn, skeleton as sk, render
    args = db.make_args(PRESET, no_reload=True)
    attrs = {"skel_type": sk.SMPLSkeleton, "near": syn.NEAR, "far": syn.FAR, "n_views": 8, "rest_pose": syn.rest_pose()}
    _, kw_test, *_ = db.create_raycaster(args, attrs, device=device)
    caster = kw_test["ray_caster"]
    caster.network.load_state_dict(syn.synthetic_params(0))
    caster.eval()
    poses = [syn.make_pose(100 + k) for k in range(n_poses)]
    c2ws = list(syn.bullet_time_cameras(syn.camera(), n_poses))
    dist_on = world > 1

    def timed(fn):
        if dist_on:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = fn()
        e1.record()
        if dist_on:
            dist.barrier()
        torch.cuda.synchronize()
        return _max_over_ranks(e0.elapsed_time(e1), device, world), r
    render.render_images(caster, args, c2ws[:2 * world], poses[:2 * world], H, W, distributed=dist_on)        # warm-up
    ms_img, imgs = timed(lambda: render.render_images(caster, args, c2ws, poses, H, W, distributed=dist_on))
    n_rays = sum(int(np.prod(np.subtract(*syn.cylinder_image_box(p["cyl"], H, W, 1.2 * H, np.asarray(c))[::-1])))
                 for p, c in zip(poses, c2ws))
    t = lambda a: torch.as_tensor(a)[None].to(device)
    pose = poses[0]
    grid_fn = lambda r: render.density_grid(caster, t(pose["kps"]), t(pose["skts"]), t(pose["bones"]), radius=1.8, res=r,
                                            distributed=dist_on)
    grid_fn(63)                                                                                              # warm-up
    ms_grid, grid = timed(lambda: grid_fn(res))
    return {"workload": f"{n_poses} synthetic poses x {H}x{W} bullet-time views (danbo_fast, {args.N_samples}+"
                        f"{args.N_importance} samples/ray, box-restricted rays) + {(res + 1)}^3 density lattice, on {world} GPU(s)",
            "n_gpus": world, "scaling": "strong", "images": n_poses, "rays": n_rays, "ms_images": ms_img,
            "images_per_s": n_poses / (ms_img / 1e3), "rays_per_s": n_rays / (ms_img / 1e3),
            "ms_per_image_per_gpu": ms_img * world / n_poses,
            "lattice_points": (res + 1) ** 3, "ms_lattice": ms_grid, "points_per_s": (res + 1) ** 3 / (ms_grid / 1e3),
            "mean_pixel": float(imgs.mean()), "lattice_occupied_frac": float((grid > 10).float().mean())}


# the bounded sample of the 261 121-ray image both arms quote the CPU figure on (the env override is for the unit test)
REF_SAMPLE_RAYS = int(os.environ.get("DANBO_REF_SAMPLE_RAYS", "32768"))


def workload_config(args, n_rays=None):
    """`config` of the JSON line - identical for this repo's arm and the reference arm."""
    return {"workload": f"danbo_fast {H}x{W} render, 1 synthetic 24-joint pose, {args.N_samples}+{args.N_importance} "
                        "samples/ray, box-restricted rays (261121 rays/image), random-init weights",
            "rays_per_image": 261121, "samples_per_ray": args.N_samples + args.N_importance, "chunk": args.chunk}


def cpu_baseline(sample_rays=REF_SAMPLE_RAYS, repeats=1, threads=None):
    """The reference's CPU implementation of the path on the host cores, on a bounded sample of the same workload.

    kind "reference": the UNMODIFIED reference (baseline/_ref, copied by scripts/vendor_ref.sh, or $DANBO_REFERENCE)
    through its own `render` (core/trainer.py:96-162: ray assembly + `batchify_rays` in
    `args.chunk` = 4096-ray chunks, as `render_path` calls it per image, run_nerf.py:92-96) and its own GraphCaster, with
    this repo's synthetic weights.  kind "port": the oracle restatement, only if the reference copy is absent."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import danbo_b200 as db
    from danbo_b200 import synthetic as syn, skeleton as sk
    threads = threads or os.cpu_count()
    torch.set_num_threads(threads)
    args = db.make_args(PRESET)
    pose = syn.make_pose(3)
    b = syn.render_batch(pose, H, W)
    n = min(sample_rays, b["ray_batch"].shape[0])
    lo = (b["ray_batch"].shape[0] - n) // 2
    rays = b["ray_batch"][lo:lo + n].contiguous()
    cams = b["cams"][lo:lo + n]
    chunk = args.chunk
    import ref_harness as rh
    if rh.available():
        kind = "reference"
        render, kw_test, rargs = rh.reference_render_setup("h36m_zju/danbo_fast.txt")
        assert rargs.chunk == chunk and rargs.N_samples == args.N_samples and rargs.N_importance == args.N_importance

        def run(m):
            rh.reference_render_rays(render, kw_test, rargs, rays[:m, 0:3], rays[:m, 3:6], pose, cams[:m], H, W, 1.2 * H)
    else:
        kind = "port"
        sys.stderr.write("bench.py: no copy of the original DANBO-pytorch ($DANBO_REFERENCE or baseline/_ref, see "
                         "scripts/vendor_ref.sh): the CPU baseline runs the oracle port (kind \"port\")\n")
        import danbo_oracle as orc
        P = syn.synthetic_params(0)
        A = torch.from_numpy(sk.bone_align_transforms(syn.rest_pose())[0])
        t = lambda a: torch.as_tensor(a)[None]

        def run(m):
            for s0 in range(0, m, chunk):
                s1 = min(m, s0 + chunk)
                orc.render_rays(rays[s0:s1], t(pose["skts"]), t(pose["bones"]), t(pose["cyl"]), cams[s0:s1], A, P,
                                args.N_samples, args.N_importance, rays_per_pose=s1 - s0, use_volume_near_far=True)
    best = None
    with torch.no_grad():
        run(min(n, chunk))                                   # warm-up: one chunk
        for _ in range(repeats):
            t0 = time.perf_counter()
            run(n)
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
    return {"value": n / best, "unit": "rays/s", "cores": int(torch.get_num_threads()), "kind": kind,
            "sample": f"{n} consecutive rays from the middle of the same {H}x{W} danbo_fast image, rendered in chunks of "
                      f"{chunk} rays, fp32 torch CPU ops, best of {repeats} after a one-chunk warm-up ({best:.2f} s)"}


def run_reference(opt):
    """The reference arm: the reference's own CPU implementation on the host cores (rank 0 only), each step one bounded
    sample (REF_SAMPLE_RAYS rays) of the workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = REF_SAMPLE_RAYS
    res, base = [], None
    for i in range(opt.warmup + opt.steps):
        base = cpu_baseline(sample_rays=n, repeats=1)
        if i >= opt.warmup:
            res.append(base["value"])
    v = float(np.mean(res))
    import danbo_b200 as db
    args = db.make_args(PRESET)
    line = {"impl": "reference", "metric": "DANBO render rays/s (fwd+composite)", "value": v, "unit": "rays/s",
            "n_gpus": opt.gpus, "steps": opt.steps, "warmup": opt.warmup, "ms_per_step": n / v * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args),
            "run": {"parallelism": f"host CPU, {base['cores']} threads (rank 0 only)",
                    "sample": f"each step = {n} consecutive rays from the middle of the image (bounded sample of the same "
                              "workload); rays/s does not depend on the sample size beyond one 4096-ray chunk"},
            "cpu_baseline": dict(base, value=v),
            "e2e": {"value": v, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the arrays the last timed step returned as DIR/<name>.npy (at most 64 MB in all; at N > 1 "
                         "rank 0's: every rank renders the same whole image)")
    opt = ap.parse_args()
    if opt.steps < 1:
        ap.error("--steps must be at least 1")
    if opt.dump_outputs and opt.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if opt.impl == "reference":
        run_reference(opt)
    else:
        run_ours(opt)


if __name__ == "__main__":
    main()
