"""anerf_h (a separate fine network, single_net=False) training without a GPU: `TrainStep` trains the parameters of
`create_raycaster`'s `grad_vars` in their order, so its gradient bucket, optimizer state and checkpoints index the same
tensors as the reference's Adam; the other configs keep their parameter lists; and a train-mode call on CPU tensors
raises (there is no CPU path).  Kernels are never launched here."""
import pytest
import torch

import danbo_b200 as db
from danbo_b200 import skeleton as sk, synthetic as syn, training


def _caster(preset, **overrides):
    args = db.make_args(preset, no_reload=True, **overrides)
    attrs = {"skel_type": sk.SMPLSkeleton, "near": syn.NEAR, "far": syn.FAR, "n_views": 8, "rest_pose": syn.rest_pose()}
    _, kw_test, _, grad_vars, _, _ = db.create_raycaster(args, attrs, device="cpu")
    return kw_test["ray_caster"], args, grad_vars


def _same(a, b):
    return len(a) == len(b) and all(x is y for x, y in zip(a, b))


def test_anerf_h_train_step_trains_grad_vars():
    caster, args, grad_vars = _caster("anerf_base", single_net=False)
    assert caster.network_fine is not caster.network
    step = training.TrainStep(caster, args)
    coarse = [p for p in caster.network.parameters() if p.requires_grad]
    fine = [p for p in caster.network_fine.parameters() if p.requires_grad]
    assert len(coarse) == len(fine) == 25
    assert _same(step.bucket.params, grad_vars) and len(grad_vars) == 50
    assert _same(step.bucket.params, coarse + fine)                       # coarse first
    assert isinstance(step.optimizer, torch.optim.Adam)                   # CPU tensors: the torch optimizer
    assert _same([p for g in step.optimizer.param_groups for p in g["params"]], grad_vars)
    # every parameter's gradient is a view of the one flat bucket (the all-reduce covers both networks)
    assert all(p.grad is not None and p.grad.untyped_storage().data_ptr() == step.bucket.flat.untyped_storage().data_ptr()
               for p in grad_vars)
    assert step.bucket.flat.numel() == sum(p.numel() for p in grad_vars)
    with pytest.raises(NotImplementedError, match="separate fine network"):
        training.TrainStep(caster, args, graph=True)


@pytest.mark.parametrize("preset", ["anerf_base", "danbo_fast"])
def test_single_network_parameter_lists_unchanged(preset):
    caster, args, grad_vars = _caster(preset)
    assert caster.network_fine is caster.network
    step = training.TrainStep(caster, args)
    before = [p for p in caster.network.parameters() if p.requires_grad]
    assert _same(step.bucket.params, before) and _same(step.bucket.params, grad_vars)
    if preset == "anerf_base":
        assert len(before) == 25


def test_anerf_h_train_mode_call_on_cpu_raises():
    caster, args, _ = _caster("anerf_base", single_net=False, N_samples=8, N_importance=4)
    caster.train()
    b = syn.training_batch(1, 8, seed=0)
    with pytest.raises(RuntimeError):
        out = caster(b["ray_batch"], N_samples=args.N_samples, kp_batch=b["kp_batch"], skts=b["skts"], cyls=b["cyls"],
                     bones=b["bones"], cams=b["cams"], N_uniques=1, perturb=1.0, N_importance=args.N_importance,
                     raw_noise_std=1.0, nerf_type="nerf")
        out["rgb_map"].sum().backward()
