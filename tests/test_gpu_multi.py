"""Data-parallel training on 2 GPUs against the same iteration on 1 GPU (run with -m gpu; skipped below 2 devices).

Mirrors what nn.DataParallel gives the reference (core/raycasters.py:116, core/trainer.py:257-300): the gradient of the
mean loss over the whole ray batch, one Adam step on it.  Here every rank holds half of the poses, the flat gradient
bucket is all-reduced (averaged) over NCCL and every rank applies the same single-launch Adam - inside ONE captured CUDA
graph per iteration (forward, losses, backward, all-reduce, Adam; `TrainStep(graph=True)`).

Checked: (1) the all-reduced gradient equals the 1-GPU gradient of the concatenated batch; (2) 25 graphed iterations
on 2 ranks end at the same loss and the same parameters as 25 graphed iterations on 1 GPU (this is the test that
catches a replayed graph evaluating stale packed weights: its loss would stay at the untrained level); (3) the eager
2-rank iteration agrees as well.  Draws are switched off (perturb = 0, raw_noise_std = 0) so that both runs see the same
samples."""
import json
import os
import socket
import sys
import tempfile

import pytest
import torch

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600, method="thread")]

N_POSES, RPP, ITERS = 4, 96, 25


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _setup(device, world=1, graph=False):
    import danbo_b200 as db
    from danbo_b200 import synthetic as syn, skeleton as sk, training
    args = db.make_args("danbo_cfg3", no_reload=True, perturb=0., raw_noise_std=0.)
    attrs = {"skel_type": sk.SMPLSkeleton, "near": syn.NEAR, "far": syn.FAR, "n_views": 8, "rest_pose": syn.rest_pose()}
    _, kw_test, *_ = db.create_raycaster(args, attrs, device=device)
    caster = kw_test["ray_caster"]
    caster.network.load_state_dict(syn.synthetic_params(0))
    step = training.TrainStep(caster, args, world_size=world, graph=graph)
    return caster, args, step


def _batch(device, rank=0, world=1):
    from danbo_b200 import synthetic as syn
    full = syn.training_batch(N_POSES, RPP, seed=5)
    per = N_POSES // world
    lo, hi = rank * per * RPP, (rank + 1) * per * RPP
    b = {k: (v[lo:hi].to(device) if torch.is_tensor(v) else v) for k, v in full.items()}
    b["N_uniques"] = per
    return b


def _train(step, batch, iters):
    losses = []
    for _ in range(iters):
        loss, _ = step(batch)
        losses.append(loss.detach().float().reshape(1).clone())
    torch.cuda.synchronize()
    return torch.cat(losses).cpu()


def _single_gpu_reference(path):
    dev = torch.device("cuda", 0)
    caster, args, step = _setup(dev)
    b = _batch(dev)
    loss, _ = step._fwd_bwd(b)
    grad = step.bucket.flat.detach().cpu().clone()
    caster_g, _, step_g = _setup(dev, graph=True)
    losses = _train(step_g, b, ITERS)
    torch.save({"grad": grad, "loss0": float(loss), "losses": losses, "params": step_g.optimizer.flat.detach().cpu().clone()},
               path)


def _say(rank, msg):
    print(f"[multi rank {rank}] {msg}", flush=True)


def worker_main(ref_path, out_path):
    """Body of one rank (launched by torch.distributed.run, like bench.py at N > 1)."""
    import faulthandler
    import torch.distributed as dist
    from danbo_b200 import parallel
    faulthandler.dump_traceback_later(150, exit=True)       # a hang prints every thread's Python stack, then exits
    rank, world, local = parallel.init_distributed()
    dev = torch.device("cuda", local)
    _say(rank, f"init done, world {world}")
    ref = torch.load(ref_path)
    res = {}
    rel = lambda a, b: float((a - b).norm() / b.norm().clamp_min(1e-30))
    # (1) gradient after the all-reduce == gradient of the whole batch on one GPU
    caster, args, step = _setup(dev, world=world)
    b = _batch(dev, rank, world)
    loss, _ = step._fwd_bwd(b)
    step.bucket.allreduce(average=True)
    torch.cuda.synchronize()
    lt = loss.detach().float().reshape(1).clone()
    dist.all_reduce(lt)
    res["grad_rel"] = rel(step.bucket.flat.cpu(), ref["grad"])
    res["loss0"] = float(lt) / world
    res["loss0_ref"] = ref["loss0"]
    _say(rank, f"gradient check done: rel {res['grad_rel']:.3e}")
    # (2) graphed iterations: forward + backward + all-reduce + Adam in one captured graph; (3) the same, eager
    alive = [step]            # a CUDA graph holding NCCL nodes must not be destroyed while collectives are still being issued
    for tag, graph in (("graph", True), ("eager", False)):
        _, _, st = _setup(dev, world=world, graph=graph)
        alive.append(st)
        losses = _train(st, b, ITERS).to(dev)
        _say(rank, f"{tag}: {ITERS} iterations done")
        dist.all_reduce(losses)
        losses = (losses / world).cpu()
        res[tag + "_whole_graph"] = bool(st._graph_whole)
        res[tag + "_loss_first"], res[tag + "_loss_last"] = float(losses[0]), float(losses[-1])
        res[tag + "_loss_err"] = float((losses - ref["losses"]).abs().max())
        res[tag + "_param_rel"] = rel(st.optimizer.flat.cpu(), ref["params"])
        res[tag + "_adam_steps"] = float(st.optimizer.step_dev.item())
    res["ref_loss_first"], res["ref_loss_last"] = float(ref["losses"][0]), float(ref["losses"][-1])
    if rank == 0:
        with open(out_path, "w") as f:
            json.dump(res, f)
    dist.barrier()
    torch.cuda.synchronize()
    _say(rank, "done")
    sys.stdout.flush()
    os._exit(0)               # skip interpreter teardown: the captured graphs (NCCL nodes) die with the process


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_rank_training_equals_single_gpu():
    import signal
    import subprocess
    with tempfile.TemporaryDirectory() as d:
        ref_path, out_path = os.path.join(d, "ref.pt"), os.path.join(d, "out.json")
        _single_gpu_reference(ref_path)
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
               "127.0.0.1", "--master-port", str(_free_port()), os.path.abspath(__file__), ref_path, out_path]
        # own process group + a hard limit: a hung collective must not outlive the test
        log_path = os.path.join(d, "multi_worker.log")           # the worker's output is shown when the test fails
        with open(log_path, "w") as lf:
            proc = subprocess.Popen(cmd, stdout=lf, stderr=subprocess.STDOUT, start_new_session=True)
            try:
                proc.wait(timeout=240)
            except subprocess.TimeoutExpired:
                os.killpg(proc.pid, signal.SIGKILL)
                proc.wait(timeout=30)
                pytest.fail("2-rank worker hung:\n" + open(log_path).read()[-6000:])
        log = open(log_path).read()
        print(log[-3000:])
        assert proc.returncode == 0, log[-6000:]
        res = json.load(open(out_path))
    print("[multi]", json.dumps(res))
    assert res["grad_rel"] <= 2e-3, res                      # fp32 atomics order + per-shard near/far fill only
    assert abs(res["loss0"] - res["loss0_ref"]) <= 1e-4
    assert res["ref_loss_last"] < res["ref_loss_first"] - 0.02          # the single-GPU run itself trains
    for tag in ("graph", "eager"):
        assert res[tag + "_adam_steps"] == ITERS, res        # building the graph must not step the optimizer
        # 25 Adam steps amplify the fp32 atomics-order differences of the gradients (measured: loss 1.7e-3, parameters
        # 1.1e-3 of their norm); stale weights would leave the loss at its initial 0.649 instead of 0.500
        assert res[tag + "_loss_err"] <= 5e-3, res
        assert res[tag + "_param_rel"] <= 5e-3, res
        assert res[tag + "_loss_last"] < res[tag + "_loss_first"] - 0.1, res
    assert res["graph_whole_graph"]


def test_graph_build_has_no_side_effect_and_sees_new_weights():
    """1 GPU: (a) the first graphed iteration applies exactly ONE Adam step (warm-up and capture are rolled back), and
    equals the eager iteration; (b) a graphed eval render after a weight change uses the new weights."""
    from util import load_fixture, pose_tensors
    dev = torch.device("cuda", 0)
    _, _, eager = _setup(dev)
    _, _, graphed = _setup(dev, graph=True)
    b = _batch(dev)
    for _ in range(3):
        eager(b)
        graphed(b)
    torch.cuda.synchronize()
    assert float(graphed.optimizer.step_dev.item()) == 3.0
    d = float((eager.optimizer.flat - graphed.optimizer.flat).abs().max())
    print(f"[multi] params after 3 iterations, graphed vs eager: max diff {d:.3e}")
    assert d <= 2e-5            # Adam's first steps move every weight by ~lr = 5e-4: a double step would show as 5e-4
    # (b) render_graphed must follow the weights
    caster = graphed.caster
    caster.eval()
    fx = load_fixture("render_fast")
    skts, bones, cyl = pose_tensors(fx)
    N = fx["ray_batch"].shape[0]
    ex = lambda t: t.expand(N, *t.shape[1:])
    kw = dict(N_samples=64, kp_batch=ex(fx["pose_kps"][None]), skts=ex(skts), cyls=ex(cyl), bones=ex(bones),
              cams=fx["cams"], N_uniques=1, N_importance=16)
    g0 = {k: v.clone() for k, v in caster.render_graphed(fx["ray_batch"], **kw).items()}
    graphed.caster.train()
    graphed(b)                                              # one more optimizer step through raw pointers
    caster.eval()
    g1 = caster.render_graphed(fx["ray_batch"], **kw)
    e1 = caster(fx["ray_batch"], perturb=False, raw_noise_std=0., **kw)
    torch.cuda.synchronize()
    assert not torch.equal(g0["rgb_map"], g1["rgb_map"])
    for k in ("rgb_map", "acc_map", "rgb0"):
        assert torch.equal(g1[k], e1[k]), k


if __name__ == "__main__":                                  # one rank of test_two_rank_training_equals_single_gpu
    _root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for _p in (_root, os.path.join(_root, "tests")):
        if _p not in sys.path:
            sys.path.insert(0, _p)
    worker_main(sys.argv[1], sys.argv[2])
