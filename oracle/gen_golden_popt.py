"""Generates tests/golden/popt.npz by running the UNMODIFIED reference pose layer (see oracle/ref_harness.py).
TEST INFRASTRUCTURE.

    python oracle/gen_golden_popt.py       # needs the reference ($DANBO_REFERENCE or baseline/_ref)

Pins `danbo-pytorch_b200/pose_opt.py` (SURVEY §8f rank 2): core/pose_opt.py's `PoseOptLayer` is built on synthetic
poses (axis-angle and rot6d parameters, and the multi-view parameter split), its parameters are moved off their initial
values, and for a batch of repeated indices the fixture records the state dict, the five outputs, the gradients of a
fixed scalar of (kps, skts) with respect to the parameters, and the trainer's pose regulariser
(`Trainer._compute_kp_loss`, core/trainer.py:446-505) with the temporal term."""
import os
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import ref_harness                                   # noqa: E402
import danbo_b200                                    # noqa: E402,F401
from danbo_b200 import synthetic as syn              # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "popt.npz")
N_POSES = 7
IDXS = np.array([5, 5, 5, 0, 0, 0, 6, 6, 6, 2, 2, 2])


def poses():
    rest = syn.rest_pose()
    ps = [syn.make_pose(40 + i, rest, render_cylinder=False) for i in range(N_POSES)]
    kps = np.stack([p["kps"] for p in ps]) + np.linspace(-0.3, 0.3, N_POSES * 3).reshape(N_POSES, 1, 3).astype(np.float32)
    return rest[None], kps.astype(np.float32), np.stack([p["bones"] for p in ps])


def probe_weights(seed=0):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(len(IDXS), 24, 3, generator=g), torch.randn(len(IDXS), 24, 4, 4, generator=g)


def run_case(tag, out, use_rot6d=False, multiview=False):
    ref_harness._imports()
    import core.pose_opt as po
    import core.trainer as tr
    rest, kps, bones = poses()
    kw = {}
    if multiview:                                   # frames 0..6 are views of 4 distinct poses
        kw = dict(kp_map=np.array([0, 1, 1, 2, 3, 3, 0]), kp_uidxs=np.array([0, 1, 3, 4]))
    layer = po.PoseOptLayer(torch.tensor(kps), torch.tensor(bones), torch.tensor(rest), use_rot6d=use_rot6d, **kw)
    g = torch.Generator().manual_seed(7)
    with torch.no_grad():
        for p in layer.parameters():
            p.add_(0.05 * torch.randn(p.shape, generator=g))
    for k, v in layer.state_dict().items():
        out[f"{tag}.sd.{k}"] = v.detach().numpy().copy()
    k_, b_, s_, l_, r_ = layer(IDXS)
    for nm, t in zip(("kps", "bones", "skts", "l2ws", "rots"), (k_, b_, s_, l_, r_)):
        out[f"{tag}.out.{nm}"] = t.detach().numpy()
    wk, ws = probe_weights()
    ((k_ * wk).sum() + (s_ * ws).sum()).backward()
    for nm, p in layer.named_parameters():
        out[f"{tag}.grad.{nm}"] = p.grad.numpy().copy()
    if not multiview:
        # the trainer's regulariser on the same batch (anchors = the initial poses), with the temporal term
        args = types.SimpleNamespace(opt_rot6d=use_rot6d, opt_pose_tol=0.002, opt_pose_coef=2.0, use_temp_loss=True,
                                     temp_coef=0.05, ext_scale=0.001)
        from core.utils.skeleton_utils import axisang_to_rot
        anchors = {"kps": torch.tensor(kps), "bones": torch.tensor(bones),
                   "rots": axisang_to_rot(torch.tensor(bones).view(-1, 3)).view(N_POSES, 24, 3, 3)}
        fake = types.SimpleNamespace(args=args, popt_kwargs={"popt_anchors": anchors, "popt_layer": layer})
        temp_val = torch.tensor((IDXS % 2).astype(np.float32))
        k_, b_, s_, l_, r_ = layer(IDXS)
        losses, stats = tr.Trainer._compute_kp_loss(fake, {"kp_idx": torch.tensor(IDXS), "temp_val": temp_val},
                                                    {"kp_batch": k_, "bones": b_, "rots": r_})
        out[f"{tag}.loss.kp_loss"] = losses["kp_loss"].detach().numpy()
        out[f"{tag}.loss.temp_loss"] = losses["temp_loss"].detach().numpy()
        out[f"{tag}.loss.MPJPC"] = stats["MPJPC"].detach().numpy()
        out[f"{tag}.loss.temp_val"] = temp_val.numpy()


def main():
    if not ref_harness.available():
        raise SystemExit("needs the reference ($DANBO_REFERENCE or baseline/_ref)")
    out = {}
    rest, kps, bones = poses()
    out["rest_pose"], out["init_kps"], out["init_bones"], out["idxs"] = rest, kps, bones, IDXS
    run_case("axisang", out)
    run_case("rot6d", out, use_rot6d=True)
    run_case("multiview", out, multiview=True)
    np.savez_compressed(OUT, **out)
    print({k: v.shape for k, v in out.items()})


if __name__ == "__main__":
    main()
