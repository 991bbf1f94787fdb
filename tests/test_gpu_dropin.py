"""The reference's OWN callers on this repo's ray caster (run with -m gpu; needs the reference copy under baseline/_ref,
made by scripts/vendor_ref.sh, or $DANBO_REFERENCE).

`danbo_b200.install()` rebinds `create_raycaster` (core/raycasters.py:17) - nothing else of the reference is touched - and
then the unmodified `Trainer.train_batch` (core/trainer.py:257-300: render -> compute_loss -> backward -> Adam -> decay)
and `render_path` (run_nerf.py:29-147: kp_to_valid_rays -> render per image -> image assembly) run on the CUDA path.
Compared with (a) this repo's own TrainStep on the same batch and seed, (b) the same reference callers on the reference's
own CPU caster."""
import numpy as np
import pytest
import torch

import ref_harness as rh
from danbo_b200 import synthetic as syn, skeleton as sk

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600, method="thread")]
needs_reference = pytest.mark.skipif(not rh.available(), reason="no reference copy (run scripts/vendor_ref.sh)")
DEV = "cuda"
N_POSES, RPP = 4, 96


class _reference_cuda_defaults:
    """The reference runs under `torch.set_default_tensor_type('torch.cuda.FloatTensor')` (run_nerf.py:728,
    run_render.py:1353): its helpers build constants with the legacy `torch.Tensor([...])` constructor and bare factory
    calls and expect them on the GPU."""

    def __enter__(self):
        torch.set_default_tensor_type("torch.cuda.FloatTensor")

    def __exit__(self, *exc):
        torch.set_default_tensor_type("torch.FloatTensor")
        if torch.empty(0).device.type != "cpu":             # the legacy call does not always take the device back
            torch.set_default_device("cpu")


def _cpu_ray_generation(fn):
    """Compatibility shim (like F5 / F6 of oracle/ref_harness.py): under a CUDA default tensor type the reference's
    `kp_to_valid_rays` (ray_utils.py:84-138) indexes CPU ray tensors with `torch.arange` results that current torch puts
    on the GPU, which torch >= 2 rejects.  The wrapper runs that one function under the CPU default, unmodified."""
    def wrapped(*a, **k):
        torch.set_default_tensor_type("torch.FloatTensor")
        try:
            a = [x.cpu() if torch.is_tensor(x) else x for x in a]
            k = {n: (x.cpu() if torch.is_tensor(x) else x) for n, x in k.items()}
            return fn(*a, **k)
        finally:
            torch.set_default_tensor_type("torch.cuda.FloatTensor")
    return wrapped


class _Handle(torch.nn.Module):
    """`.module`, as nn.DataParallel gives the reference's trainer (DataParallel itself would scatter a CPU module)."""

    def __init__(self, m):
        super().__init__()
        self.module = m

    def forward(self, *a, **k):
        return self.module(*a, **k)


def _attrs(H=512):
    return {"skel_type": sk.SMPLSkeleton, "near": syn.NEAR, "far": syn.FAR, "n_views": 8, "rest_pose": syn.rest_pose(),
            "hwf": (H, H, 1.2 * H)}


def _ref_batch(device):
    b = syn.training_batch(N_POSES, RPP, seed=5)
    rays = torch.stack([b["ray_batch"][:, 0:3], b["ray_batch"][:, 3:6]], 0)            # (2, N, 3) like ray_collate_fn
    rb = {"rays": rays, "target_s": b["target_s"], "kp3d": b["kp_batch"], "skts": b["skts"], "bones": b["bones"],
          "cyls": b["cyls"], "cam_idxs": b["cams"], "bgs": b["bgs"]}
    return {k: v.contiguous().to(device) for k, v in rb.items()}, b


def test_install_rebinds_create_raycaster_only(tmp_path):
    """On the reference when a copy is given, else on the stand-in of its `core/` (tests/util.py `reference_core`)."""
    import danbo_b200 as db
    from util import reference_modules
    with reference_modules(tmp_path) as (rc, run_nerf):
        orig = rc.create_raycaster
        db.install()
        try:
            assert getattr(rc.create_raycaster, "__danbo_b200__", False) and run_nerf.create_raycaster is rc.create_raycaster
        finally:
            db.uninstall()
        assert rc.create_raycaster is orig and run_nerf.create_raycaster is orig


@needs_reference
@pytest.mark.parametrize("perturb", [0.0, 1.0])
def test_reference_trainer_train_batch_on_this_caster(perturb):
    import danbo_b200 as db
    from danbo_b200 import training
    rc, run_nerf = rh._imports()
    from core.trainer import Trainer
    extra = ["--N_rand", str(N_POSES * RPP), "--N_sample_images", str(N_POSES), "--perturb", str(perturb),
             "--raw_noise_std", str(perturb)]
    args = rh.parse_args("h36m_zju/danbo_fast.txt", extra)
    ref_losses = None
    if perturb == 0.0:
        # (b) the reference's own caster (CPU, fp32) under the same Trainer code, same batch - run first, before anything
        # touches the default tensor type
        ref_caster, kw_ref = rh.build(args, syn.rest_pose())
        rh.load_weights(ref_caster, syn.synthetic_params(0))
        ref_caster.train()
        kw_ref_train = dict(kw_ref, ray_caster=_Handle(ref_caster), perturb=args.perturb, raw_noise_std=args.raw_noise_std)
        opt_ref = torch.optim.Adam(ref_caster.network.parameters(), lr=args.lrate)
        tr_ref = Trainer(args, _attrs(), opt_ref, None, kw_ref_train, kw_ref, popt_kwargs=None, device=torch.device("cpu"))
        batch_cpu, _ = _ref_batch("cpu")
        ld_ref, _ = tr_ref.train_batch(batch_cpu, i=1, global_step=1)
        ref_losses = {k: float(v) for k, v in ld_ref.items()}
    db.install()
    try:
        kw_train, kw_test, start, grad_vars, optimizer, _ = run_nerf.create_raycaster(args, _attrs(), device=torch.device(DEV))
    finally:
        db.uninstall()
    caster = kw_test["ray_caster"]
    assert isinstance(caster, db.RayCaster)
    caster.network.load_state_dict(syn.synthetic_params(0))
    trainer = Trainer(args, _attrs(), optimizer, None, kw_train, kw_test, popt_kwargs=None, device=torch.device(DEV))
    batch, b = _ref_batch(DEV)
    torch.manual_seed(11)
    caster.train()
    with _reference_cuda_defaults():
        loss_dict, stats = trainer.train_batch(batch, i=1, global_step=1)
    torch.cuda.synchronize()
    got = {k: float(v) for k, v in loss_dict.items()}
    assert set(got) == {"rgb_loss", "rgb_loss0", "soft_softmax_loss", "vol_scale_loss", "total_loss"}
    p_after = torch.cat([p.detach().reshape(-1) for p in caster.network.parameters() if p.requires_grad]).cpu()

    # (a) this repo's own iteration (loss kernel + single-launch Adam) on the same batch, weights and seed
    args2 = db.make_args("danbo_fast", no_reload=True, perturb=perturb, raw_noise_std=perturb)
    _, kw2, *_ = db.create_raycaster(args2, _attrs(), device=DEV)
    caster2 = kw2["ray_caster"]
    caster2.network.load_state_dict(syn.synthetic_params(0))
    step = training.TrainStep(caster2, args2)
    b2 = {k: (v.to(DEV) if torch.is_tensor(v) else v) for k, v in b.items()}
    torch.manual_seed(11)
    loss2, _ = step(b2)
    torch.cuda.synchronize()
    p2 = torch.cat([p.detach().reshape(-1) for p in caster2.network.parameters() if p.requires_grad]).cpu()
    print(f"[dropin] perturb {perturb}: reference Trainer on this caster {got['total_loss']:.6f}  TrainStep {float(loss2):.6f}  "
          f"params max diff {float((p_after - p2).abs().max()):.3e}")
    assert abs(got["total_loss"] - float(loss2)) <= 2e-5 * max(abs(float(loss2)), 1.0)
    assert float((p_after - p2).abs().max()) <= 2e-4            # one Adam step moves weights by lr = 5e-4
    if ref_losses is not None:
        for k in got:
            print(f"[dropin] {k}: this caster {got[k]:.6f}  reference caster (CPU) {ref_losses[k]:.6f}")
            assert abs(got[k] - ref_losses[k]) <= 3e-3 * max(abs(ref_losses[k]), 1e-2), k



@needs_reference
def test_reference_render_path_on_this_caster():
    """BASELINE config #1 shape: danbo_base, one 64x64 image, through the reference's render_path on both casters."""
    import danbo_b200 as db
    rc, run_nerf = rh._imports()
    args = rh.parse_args("h36m_zju/danbo_base.txt")
    H = 64
    db.install()
    try:
        _, kw_test, *_ = run_nerf.create_raycaster(args, _attrs(H), device=torch.device(DEV))
    finally:
        db.uninstall()
    caster = kw_test["ray_caster"]
    caster.network.load_state_dict(syn.synthetic_params(0))
    caster.eval()
    pose = syn.make_pose(3, render_cylinder=False)
    c2w = torch.tensor(syn.camera())[None]
    t = lambda a: torch.tensor(np.asarray(a))[None]
    kw = dict(kp=t(pose["kps"]), skts=t(pose["skts"]), bones=t(pose["bones"]), cams=torch.zeros(1, 1, dtype=torch.long),
              ret_acc=True, ext_scale=args.ext_scale)
    # the reference's own caster on the CPU first (before the default tensor type is touched)
    ref_caster, kw_ref = rh.build(args, syn.rest_pose())
    rh.load_weights(ref_caster, syn.synthetic_params(0))
    ref_caster.eval()
    with torch.no_grad():
        out_ref = run_nerf.render_path(c2w, (H, H, 1.2 * H), args.chunk, kw_ref, **kw)
    orig_rays = run_nerf.kp_to_valid_rays
    run_nerf.kp_to_valid_rays = _cpu_ray_generation(orig_rays)
    try:
        with _reference_cuda_defaults(), torch.no_grad():
            out = run_nerf.render_path(c2w.to(DEV), (H, H, 1.2 * H), args.chunk, kw_test,
                                       **{k: (v.to(DEV) if torch.is_tensor(v) else v) for k, v in kw.items()})
    finally:
        run_nerf.kp_to_valid_rays = orig_rays
    rgbs, disps, accs = out[0], out[1], out[2]
    for name, a, r in (("rgb", rgbs, out_ref[0]), ("disp", disps, out_ref[1]), ("acc", accs, out_ref[2])):
        e = np.abs(np.asarray(a) - np.asarray(r))
        print(f"[dropin] render_path {name}: shape {np.asarray(a).shape} mean err {e.mean():.3e} max {e.max():.3e}")
        assert np.asarray(a).shape == np.asarray(r).shape
        assert e.mean() <= 4e-3
