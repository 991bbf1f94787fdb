"""The drop-in boundary of SURVEY §8(b) that does not need a GPU: what `create_raycaster` returns, the attribute surface
the reference's trainer / run scripts touch on the caster, the checkpoint key scheme and the parameter inventory
(SURVEY appendix A).  Kernels are never launched here."""
import os
import tempfile

import numpy as np
import pytest
import torch

import danbo_b200 as db
from danbo_b200 import params, skeleton as sk, synthetic as syn


def _attrs():
    return {"skel_type": sk.SMPLSkeleton, "near": syn.NEAR, "far": syn.FAR, "n_views": 8, "rest_pose": syn.rest_pose()}


def test_create_raycaster_return_contract():
    """core/raycasters.py:17-143: (render_kwargs_train, render_kwargs_test, start, grad_vars, optimizer, loaded_ckpt) and the
    keys of the two kwargs dicts (:115-137)."""
    args = db.make_args("danbo_base", no_reload=True)
    attrs = _attrs()
    kw_train, kw_test, start, grad_vars, optimizer, loaded = db.create_raycaster(args, attrs, device="cpu")
    keys = {"ray_caster", "perturb", "N_importance", "N_samples", "use_viewdirs", "raw_noise_std", "ray_noise_std",
            "ext_scale", "preproc_kwargs", "lindisp", "nerf_type"}
    assert set(kw_train) == keys and set(kw_test) == keys
    assert set(kw_train["preproc_kwargs"]) == {"density_scale", "density_fn"}
    assert kw_test["perturb"] is False and kw_test["raw_noise_std"] == 0. and kw_test["ray_noise_std"] == 0.
    assert start == 0 and loaded is None and "skel_profile" in attrs                      # added in place, :31-32
    caster = kw_test["ray_caster"]
    assert kw_train["ray_caster"].module is caster                                       # where the reference has DataParallel
    assert isinstance(optimizer, torch.optim.Adam) and optimizer.param_groups[0]["lr"] == args.lrate
    n_train = sum(p.numel() for p in grad_vars)
    assert n_train == 2455876, n_train                                                   # SURVEY appendix A


def test_attribute_surface_the_trainer_touches():
    """trainer.py:208-220,294-300,509-546,616; run_render.py:125-132; run_nerf.py:156,162."""
    args = db.make_args("danbo_fast", no_reload=True)
    _, kw_test, *_ = db.create_raycaster(args, _attrs(), device="cpu")
    c = kw_test["ray_caster"]
    net, fine = c.get_networks()
    assert net is c.network and fine is c.network_fine and fine is net
    assert tuple(c.transforms.shape) == (1, 24, 4, 4) and c.rest_poses.shape == (24, 3)
    assert isinstance(net.pe_fn.get_tau(), float)
    c.update_embed_fns(1000, args)
    gn = net.graph_net
    assert tuple(gn.axis_scale.shape) == (24, 3) and tuple(gn.init_scale.shape) == (24, 3)
    assert gn.get_axis_scale() is gn.axis_scale and gn.axis_scale.requires_grad
    confd, invalid = torch.randn(5, 7, 24), (torch.rand(5, 7, 24) > 0.5).float()
    p = net.sigmoid(confd, invalid, mask_invalid=False, clamp=False)                     # trainer.py:521
    assert torch.allclose(p, torch.sigmoid(confd) * 1.002 - 0.001)
    pm = net.sigmoid(confd.reshape(-1, 24), invalid)
    assert torch.equal(pm == 0, (invalid.reshape(-1, 24) == 1) | (pm == 0))
    assert len(net.get_adjw()) == 3
    c.train(); assert c.training and net.training
    c.eval(); assert not c.training
    assert all(p.grad is None for p in c.parameters())
    with pytest.raises(NotImplementedError):
        c(fwd_type="density_color")                                                      # broken in the reference itself


def test_checkpoint_key_scheme_and_parameter_inventory():
    """raycasters.py:601-637 (custom state_dict keys), trainer.py:610-617 (checkpoint dict), SURVEY appendix A (names and
    shapes): a checkpoint written in the reference's format reloads through create_raycaster."""
    args = db.make_args("danbo_base", no_reload=True)
    _, kw_test, _, _, optimizer, _ = db.create_raycaster(args, _attrs(), device="cpu")
    c = kw_test["ray_caster"]
    sd = c.state_dict()
    assert set(sd) == {"network_fn_state_dict", "network_fine_state_dict"}
    shapes = params.danbo_param_shapes()
    net_sd = sd["network_fn_state_dict"]
    for k, shp in shapes.items():
        assert k in net_sd and tuple(net_sd[k].shape) == tuple(shp), k
    c.network.load_state_dict(syn.synthetic_params(3))
    with tempfile.TemporaryDirectory() as d:
        os.makedirs(os.path.join(d, "exp"))
        ckpt = {"global_step": 1234, "network_fn_state_dict": c.state_dict()["network_fn_state_dict"],
                "network_fine_state_dict": c.state_dict()["network_fine_state_dict"],
                "optimizer_state_dict": optimizer.state_dict()}
        torch.save(ckpt, os.path.join(d, "exp", "001234.tar"))
        args2 = db.make_args("danbo_base", basedir=d, expname="exp")
        _, kw2, start, _, _, loaded = db.create_raycaster(args2, _attrs(), device="cpu")
        assert start == 1234 and loaded is not None
        got = kw2["ray_caster"].network.state_dict()
        for k in shapes:
            assert torch.equal(got[k], c.network.state_dict()[k]), k


def test_kernels_fail_loudly_without_a_gpu():
    """No CPU fallback: the ray caster raises on CPU tensors instead of computing anything."""
    args = db.make_args("danbo_fast", no_reload=True)
    _, kw_test, *_ = db.create_raycaster(args, _attrs(), device="cpu")
    c = kw_test["ray_caster"]
    b = syn.render_batch(syn.make_pose(0), 16, 16)
    with pytest.raises(RuntimeError):
        c(b["ray_batch"], N_samples=args.N_samples, kp_batch=b["kp_batch"], skts=b["skts"], cyls=b["cyls"], bones=b["bones"],
          cams=b["cams"], N_uniques=1, perturb=False, N_importance=args.N_importance, raw_noise_std=0.)


def test_flat_adam_state_is_interchangeable_with_torch_adam(tmp_path):
    """Checkpoints keep the reference's format (core/trainer.py:597-618): the flat moment arenas of the single-launch Adam
    serialise to torch.optim.Adam's own state dict and back, so either side resumes from the other's file."""
    import torch
    from danbo_b200 import training
    torch.manual_seed(0)
    net = torch.nn.Sequential(torch.nn.Linear(5, 4), torch.nn.Linear(4, 2))
    params = list(net.parameters())
    opt = torch.optim.Adam(params, lr=3e-4, betas=(0.9, 0.999))
    for _ in range(3):
        opt.zero_grad()
        net(torch.randn(7, 5)).pow(2).sum().backward()
        opt.step()
    sd = opt.state_dict()
    n = sum(p.numel() for p in params)
    m, v = torch.full((n,), 9.), torch.full((n,), 9.)
    step, lr = training.adam_state_from_dict(sd, params, m, v)
    assert step == 3.0 and lr == 3e-4
    off = 0
    for i, p in enumerate(params):
        assert torch.equal(m[off:off + p.numel()].view_as(p), sd["state"][i]["exp_avg"])
        assert torch.equal(v[off:off + p.numel()].view_as(p), sd["state"][i]["exp_avg_sq"])
        off += p.numel()
    back = training.adam_state_to_dict(params, m, v, step, {"lr": lr, "betas": (0.9, 0.999), "eps": 1e-8})
    # a fresh torch Adam resumed from the flat state continues exactly like the original
    import copy
    net2 = copy.deepcopy(net)
    opt2 = torch.optim.Adam(list(net2.parameters()), lr=1.0)
    opt2.load_state_dict(back)
    x = torch.randn(7, 5)
    for o, nn_ in ((opt, net), (opt2, net2)):
        o.zero_grad()
        nn_(x).pow(2).sum().backward()
        o.step()
    for a, b in zip(net.parameters(), net2.parameters()):
        assert torch.equal(a, b)
    # parameters that never stepped have no state: zeros
    opt3 = torch.optim.Adam(params, lr=1e-3)
    m.fill_(5.)
    assert training.adam_state_from_dict(opt3.state_dict(), params, m, v)[0] == 0.0 and float(m.abs().max()) == 0.0
    # the checkpoint file carries the reference's keys

    class Caster:
        def state_dict(self):
            return {"network_fn_state_dict": net.state_dict(), "network_fine_state_dict": net.state_dict()}
    path = os.path.join(tmp_path, "000010.tar")
    training.save_checkpoint(path, 10, Caster(), opt)
    ck = torch.load(path, weights_only=False)
    assert set(ck) == {"global_step", "optimizer_state_dict", "poseopt_layer_state_dict", "pose_optimizer_state_dict",
                       "poseopt_anchors", "network_fn_state_dict", "network_fine_state_dict"}
    assert ck["global_step"] == 10 and ck["poseopt_layer_state_dict"] is None


def test_train_step_learning_rate_schedule_and_resume(tmp_path):
    """Steps 4-5 of train_batch (core/trainer.py:286-294) on a stand-in caster: the rate follows decay_optimizer_lrate
    (:189-200) in units of decay_unit optimizer steps, the encoders' schedule hook is called, and a checkpoint written by
    `TrainStep.save` resumes at the same step count and rate."""
    import types
    import torch
    from danbo_b200 import training

    class Net(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.w = torch.nn.Parameter(torch.full((3,), 0.5))

    class Caster(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.network = Net()
            self.calls = []

        def update_embed_fns(self, step, args):
            self.calls.append(step)

        def state_dict(self, *a, **k):
            return {"network_fn_state_dict": self.network.state_dict(), "network_fine_state_dict": self.network.state_dict()}

        def forward(self, ray_batch, **kw):
            rgb = torch.sigmoid(ray_batch[:, :3] * self.network.w)
            return {"rgb_map": rgb, "acc_map": torch.sigmoid(ray_batch[:, 3])}

    args = types.SimpleNamespace(lrate=1e-2, lrate_decay=4, lrate_decay_rate=0.1, decay_unit=3, loss_fn="L1",
                                 agg_type="sigmoid", N_samples=8, N_importance=4, perturb=1.0, raw_noise_std=0.,
                                 use_background=False, opt_vol_scale=False)
    batch = {"ray_batch": torch.randn(6, 11), "kp_batch": None, "skts": None, "cyls": None, "bones": None, "cams": None,
             "N_uniques": 1, "target_s": torch.full((6, 3), 0.3)}
    caster = Caster()
    step = training.TrainStep(caster, args)
    rates = []
    for _ in range(7):
        step(batch)
        rates.append(step.optimizer.param_groups[0]["lr"])
    want = [1e-2 * 0.1 ** (((i + 1) // 3) / 4) for i in range(7)]          # rate in force after optimizer step i + 1
    assert all(abs(a - b) < 1e-12 for a, b in zip(rates, want)), (rates, want)
    assert caster.calls == list(range(1, 8))
    path = os.path.join(tmp_path, "ck.tar")
    step.save(path, 7)
    caster2 = Caster()
    caster2.network.load_state_dict(torch.load(path, weights_only=False)["network_fn_state_dict"])
    step2 = training.TrainStep(caster2, args)
    assert step2.resume(torch.load(path, weights_only=False)) == 7 and step2.n_steps == 7
    step(batch), step2(batch)
    assert torch.equal(caster.network.w, caster2.network.w)                 # same moments, same rate, same update
    assert step2.optimizer.param_groups[0]["lr"] == step.optimizer.param_groups[0]["lr"]


def test_internal_block_plan():
    """`RayCaster._plan_blocks`: how a call is cut into launch blocks (and, opt-in, streams)."""
    from danbo_b200.raycaster import RayCaster, MAX_RAYS_PER_LAUNCH
    plan = RayCaster._plan_blocks
    # one stream: the measured behaviour - one block per 262 144 rays, whole chunks when a fill chunk is given
    assert plan(261121, 1, 261121, 4096, 1) == (MAX_RAYS_PER_LAUNCH, 1)
    assert plan(261121, 1, 261121, None, 1) == (MAX_RAYS_PER_LAUNCH, 1)
    assert plan(1 << 20, 1, 1 << 20, 3000, 1) == ((MAX_RAYS_PER_LAUNCH // 3000) * 3000, 1)
    # several poses: whole poses per block, never more than one stream
    assert plan(16 * 192, 16, 192, None, 2) == ((MAX_RAYS_PER_LAUNCH // 192) * 192, 1)
    assert plan(400000, 4, 100000, 4096, 3) == (200000, 1)
    # streams: only with a fill chunk and a big single-pose call; blocks are whole chunks and cover the call
    assert plan(261121, 1, 261121, None, 2)[1] == 1 and plan(20000, 1, 20000, 4096, 2)[1] == 1
    for N in (32768, 40000, 261121, 1000000):
        for ns in (2, 3):
            for chunk in (1024, 4096):
                block, s = plan(N, 1, N, chunk, ns)
                assert s == ns and block % chunk == 0 and 0 < block <= MAX_RAYS_PER_LAUNCH
                n_blocks = -(-N // block)
                assert n_blocks >= min(ns, -(-N // chunk)) and (n_blocks - 1) * block < N


@pytest.mark.parametrize("name", ["train_fast", "train_cfg3", "train_fast_softmax", "train_surreal"])
def test_compute_loss_on_the_references_outputs(name):
    """`training.compute_loss` (the PyTorch-op restatement of core/trainer.py:396-422,507-553 the loss kernel is tested
    against on the GPU) on the reference's OWN render outputs must give the reference's own loss terms."""
    import numpy as np
    from danbo_b200 import networks, training
    from util import load_fixture, agg_type_of, preset_of, config_flags_of, params_for
    fx = load_fixture(name)
    agg = agg_type_of(fx)
    args = db.make_args(preset_of(fx), no_reload=True, agg_type=agg, **config_flags_of(fx))
    net = networks.DanboField(n_framecodes=8, skel_profile=sk.skeleton_profile(syn.rest_pose()), opt_scale=True,
                              agg_type=agg, mask_vol_prob=True, opt_framecode=bool(args.opt_framecode))
    net.load_state_dict(params_for(fx))
    b = syn.training_batch(int(fx["n_poses"]), int(fx["rays_per_pose"]), seed=int(fx["batch_seed"]))
    preds = {k[4:]: v for k, v in fx.items() if k.startswith("out.")}
    total, terms = training.compute_loss(args, preds, {"target_s": b["target_s"], "bgs": b["bgs"]}, net)
    assert abs(float(total) - float(fx["loss.total"])) <= 2e-6 * max(1.0, abs(float(fx["loss.total"])))
    for k, v in terms.items():
        assert ("loss." + k) in fx, k
        assert abs(float(v) - float(fx["loss." + k])) <= 2e-6 * max(1e-3, abs(float(fx["loss." + k]))), (k, float(v))
    ref_terms = {k[5:] for k in fx if k.startswith("loss.")} - {"total", "total_loss"}
    assert ref_terms == set(terms), (ref_terms, set(terms))


@pytest.mark.parametrize("name", ["render_fast", "render_base"])
def test_graph_net_module_matches_reference_volumes(name):
    """`DanboField.bone_volumes` as PyTorch ops (the parameter owner, the twin the graph-net kernels are tested against
    on the GPU, and the route a pose with a gradient takes) against the reference's own bone volumes; a rot6d pose
    (6 numbers per joint, as a rot6d pose layer hands it over, encoders.py:873-877) gives the same volumes."""
    from danbo_b200 import networks, pose_opt as po
    from util import load_fixture
    fx = load_fixture(name)
    net = networks.DanboField(n_framecodes=8, skel_profile=sk.skeleton_profile(syn.rest_pose()), opt_scale=True)
    net.load_state_dict(syn.synthetic_params(int(fx.get("weight_seed", 0))))
    bones = fx["pose_bones"].reshape(1, 24, 3)
    with torch.no_grad():
        vol = net.bone_volumes(bones)
        rot6d = po.rot_to_rot6d(po.axisang_to_rot(bones))
        vol6 = net.bone_volumes(rot6d)
    want = fx["st.vol.0"].reshape(1, 24, 240)
    assert float((vol - want).abs().max()) <= 2e-5 * float(want.abs().max())
    assert float((vol6 - vol).abs().max()) <= 1e-5 * float(want.abs().max())
    # and it is differentiable with respect to the pose
    b = bones.clone().requires_grad_(True)
    net.bone_volumes(b).square().sum().backward()
    assert b.grad is not None and float(b.grad.abs().max()) > 0


def test_field_without_frame_codes_and_view_modes():
    """configs/surreal (opt_framecode=False): no `framecodes.codes.weight`, a 283-input view layer - the reference's
    own parameter inventory for that config; configs/perfcap (relray + root_local) are accepted, mixed pairs are not."""
    from danbo_b200 import networks, raycaster
    net = networks.DanboField(n_framecodes=8, skel_profile=sk.skeleton_profile(syn.rest_pose()), opt_framecode=False)
    P = syn.synthetic_params(0, opt_framecode=False)
    net.load_state_dict(P, strict=True)
    assert net.framecodes is None and net.views_linears[0].weight.shape == (128, 283)
    full = syn.synthetic_params(0)
    assert torch.equal(P["views_linears.0.weight"], full["views_linears.0.weight"][:, :283])
    n = sum(p.numel() for p in net.parameters() if p.requires_grad)
    assert n == 2455876 - 8 * 128 - 128 * 128
    assert set(params.danbo_param_shapes(opt_framecode=False)) == set(params.danbo_param_shapes()) - {"framecodes.codes.weight"}
    raycaster.check_args(db.make_args("danbo_fast", opt_framecode=False, loss_fn="MSE"))
    raycaster.check_args(db.make_args("danbo_fast", view_type="relray", ray_tr_type="root_local", nerf_type="graph"))
    for bad in (dict(view_type="relray"), dict(ray_tr_type="root_local"), dict(view_type="world"), dict(ray_tr_type="local")):
        with pytest.raises(NotImplementedError):
            raycaster.check_args(db.make_args("danbo_fast", **bad))


def test_view_rays_root_local_matches_oracle():
    """`RayCaster._view_rays` (perfcap configs) against the oracle's `view_directions`, one pose and several."""
    import types
    sys_path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle")
    import sys
    sys.path.insert(0, sys_path)
    import danbo_oracle as orc
    from danbo_b200.raycaster import RayCaster
    g = torch.Generator().manual_seed(0)
    for G, skip in ((1, 12), (3, 4)):
        rays = torch.randn(12, 11, generator=g)
        skts = torch.stack([torch.as_tensor(syn.make_pose(30 + i)["skts"]) for i in range(G)])
        me = types.SimpleNamespace(view_mode="root_local")
        out = RayCaster._view_rays(me, rays, skts, skip)
        pose = torch.clamp(torch.arange(12) // skip, max=G - 1)
        want = orc.view_directions(rays[:, 3:6], skts[pose], "root_local")
        assert out.shape == (12, 8) and float((out[:, 3:6] - want).abs().max()) < 1e-6
        assert torch.equal(out[:, :3], rays[:, :3]) and torch.equal(out[:, 6:8], rays[:, 6:8])
        assert float((out[:, 3:6].norm(dim=-1) - 1).abs().max()) < 1e-6
        assert RayCaster._view_rays(types.SimpleNamespace(view_mode="world"), rays, skts, skip) is rays


def test_create_raycaster_for_the_other_shipped_configs(tmp_path):
    """configs/surreal (no frame codes) and configs/perfcap (root-local view directions) through the factory: module
    shapes, checkpoint keys, and a checkpoint round trip through the reference's file layout."""
    args = db.make_args("danbo_fast", no_reload=True, opt_framecode=False, loss_fn="MSE")
    _, kw, _, grad_vars, _, _ = db.create_raycaster(args, _attrs(), device="cpu")
    caster = kw["ray_caster"]
    sd = caster.state_dict()
    assert "framecodes.codes.weight" not in sd["network_fn_state_dict"]
    assert sd["network_fn_state_dict"]["views_linears.0.weight"].shape == (128, 283)
    assert sum(p.numel() for p in grad_vars) == 2455876 - 8 * 128 - 128 * 128
    assert caster.view_mode == "world" and not caster.network.opt_framecode
    caster.network.load_state_dict(syn.synthetic_params(1, opt_framecode=False))
    path = os.path.join(tmp_path, "000001.tar")
    torch.save({"global_step": 1, **caster.state_dict()}, path)
    args2 = db.make_args("danbo_fast", opt_framecode=False, ft_path=path)
    _, kw2, start, *_ = db.create_raycaster(args2, _attrs(), device="cpu")
    assert start == 1
    for k, v in kw2["ray_caster"].state_dict()["network_fn_state_dict"].items():
        assert torch.equal(v, caster.state_dict()["network_fn_state_dict"][k]), k
    with pytest.raises(ValueError):                                   # a field WITH frame codes needs cams
        c3 = db.create_raycaster(db.make_args("danbo_fast", no_reload=True), _attrs(), device="cpu")[1]["ray_caster"]
        c3.render_rays(torch.zeros(4, 11), 8, None, skts=torch.zeros(4, 24, 4, 4), cyls=torch.zeros(4, 5),
                       bones=torch.zeros(4, 24, 3), cams=None, N_importance=4)
    perf = db.make_args("danbo_fast", no_reload=True, view_type="relray", ray_tr_type="root_local", nerf_type="graph")
    assert db.create_raycaster(perf, _attrs(), device="cpu")[1]["ray_caster"].view_mode == "root_local"


def test_dropin_hook_rebinds_create_raycaster_only(tmp_path):
    """`danbo_b200.install()` (dropin.py): the reference's `create_raycaster` name - in core.raycasters and in the modules
    that copied it (run_nerf) - points at this repo's factory, nothing else changes, and `uninstall()` restores it.  Runs
    on the reference when a copy is given, else on a stand-in of its `core/` (tests/util.py `reference_core`)."""
    import ref_harness as rh                 # tests/conftest.py puts oracle/ and tests/ on sys.path
    from util import reference_modules
    with reference_modules(tmp_path) as (rc, run_nerf):
        args = (rh.parse_args("h36m_zju/danbo_fast.txt", ["--agg_type", "relu"]) if rh.available() else
                db.make_args("danbo_fast", agg_type="relu"))
        orig = rc.create_raycaster
        names_before = {k: id(v) for k, v in vars(rc).items() if not k.startswith("__")}
        db.install()
        try:
            assert getattr(rc.create_raycaster, "__danbo_b200__", False)
            assert run_nerf.create_raycaster is rc.create_raycaster
            changed = [k for k, v in vars(rc).items() if not k.startswith("__") and names_before.get(k) != id(v)]
            assert changed == ["create_raycaster"], changed
            # flags outside the supported subset raise through the hook as well (no fallback to the reference's caster)
            with pytest.raises(NotImplementedError):
                rc.create_raycaster(args, {"rest_pose": None, "n_views": 8})
        finally:
            db.uninstall()
        assert rc.create_raycaster is orig and run_nerf.create_raycaster is orig


def test_run_launcher_executes_a_reference_script_with_the_hook_installed(tmp_path):
    """`python -m danbo_b200.run <script> [args]`: the script runs as __main__ from the reference's root with
    `create_raycaster` already rebound and its own argv.  A stand-in script is placed beside the reference's `core/`
    (or beside its stand-in, tests/util.py `reference_core`)."""
    import shutil
    import subprocess
    import sys
    from util import reference_core
    root = tmp_path / "ref"
    shutil.copytree(os.path.join(reference_core(tmp_path), "core"), root / "core")
    (root / "probe_script.py").write_text(
        "import sys, os\n"
        "from core.raycasters import create_raycaster\n"
        "print('HOOKED', getattr(create_raycaster, '__danbo_b200__', False), sys.argv[1:], os.path.basename(os.getcwd()), __name__)\n")
    repo = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([repo, os.path.join(repo, "oracle", "ref_stubs")]))
    out = subprocess.run([sys.executable, "-m", "danbo_b200.run", str(root / "probe_script.py"), "--config", "x.txt"],
                         capture_output=True, text=True, timeout=300, env=env, cwd=str(tmp_path))
    assert out.returncode == 0, out.stderr[-2000:]
    assert "HOOKED True ['--config', 'x.txt'] ref __main__" in out.stdout, out.stdout[-500:]


def test_check_args_is_fail_closed_on_missing_flags():
    """A namespace that does not carry a flag is checked against the REFERENCE CLI's default for it (config.DEFAULTS =
    run_nerf.py:186-572), never against "whatever is supported": an empty namespace therefore selects the reference's
    default model (nerf_type = 'nerf', PoolPNGCN, ...), which the DANBO path must refuse."""
    import argparse
    from danbo_b200 import raycaster
    with pytest.raises(NotImplementedError):
        raycaster.check_args(argparse.Namespace())
    full = db.make_args("danbo_fast")
    raycaster.check_args(full)
    partial = argparse.Namespace(**{k: v for k, v in vars(full).items() if k not in ("agg_backbone", "voxel_res")})
    with pytest.raises(NotImplementedError):                    # reference defaults: agg_backbone='mlp', voxel_res=4
        raycaster.check_args(partial)


def test_train_step_refuses_trainer_flags_it_does_not_implement():
    """core/trainer.py honours opt_pose_step / opt_pose_stop / weight_decay / reg_fn / use_lpips_loss; TrainStep raises
    for any of them instead of silently training something else (checked before any device work)."""
    from danbo_b200 import training
    for flag, val in (("opt_pose_step", 4), ("opt_pose_stop", 1000), ("weight_decay", 0.01), ("reg_fn", "L1"),
                      ("use_lpips_loss", True)):
        args = db.make_args("danbo_fast", **{flag: val})
        with pytest.raises(NotImplementedError, match=flag):
            training.TrainStep(object(), args)


def test_both_bench_arms_quote_the_same_config():
    """The driver compares the `config` dict of `bench.py` and `bench.py --impl reference`: one function builds both."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    args = db.make_args(bench.PRESET)
    a, b = bench.workload_config(args, 261121), bench.workload_config(args)
    assert a == b and a["rays_per_image"] == 261121 and a["samples_per_ray"] == 48 and a["chunk"] == 4096
    src = open(bench.__file__).read()
    assert src.count('"config": workload_config(args') == 2            # both JSON lines


def test_bench_dump_outputs_writes_the_returned_arrays(tmp_path):
    """`bench.py --dump-outputs DIR`: every returned array as DIR/<name>.npy in float32 (float64 kept); above the byte
    budget every array keeps the same seeded sample of rays, in ray order, so that two runs write identical files."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    n = 1000
    rid = torch.arange(n, dtype=torch.float32)
    ret = {"rgb_map": rid[:, None].expand(n, 3).contiguous(), "acc_map": rid.to(torch.float64),
           "T_i": rid[:, None].expand(n, 48).to(torch.bfloat16)}
    bench.dump_outputs(ret, str(tmp_path / "all"))
    full = {k: np.load(tmp_path / "all" / f"{k}.npy") for k in ret}
    assert sorted(os.listdir(tmp_path / "all")) == ["T_i.npy", "acc_map.npy", "rgb_map.npy"]
    assert full["acc_map"].dtype == np.float64 and full["rgb_map"].dtype == full["T_i"].dtype == np.float32
    for k, v in ret.items():
        np.testing.assert_array_equal(full[k], v.double().numpy())
    budget = 100 * (3 * 4 + 8 + 48 * 4) + 3 * bench.NPY_HEADER_BYTES     # 100 rays' worth + the headers
    for d in ("a", "b"):
        bench.dump_outputs(ret, str(tmp_path / d), budget=budget)
    part = {k: np.load(tmp_path / "a" / f"{k}.npy") for k in ret}
    assert sum(os.path.getsize(tmp_path / "a" / f"{k}.npy") for k in ret) <= budget
    rows = part["acc_map"].astype(np.int64)
    assert len(rows) == 100 and np.all(np.diff(rows) > 0)
    for k in ret:
        np.testing.assert_array_equal(part[k], full[k][rows])
        np.testing.assert_array_equal(part[k], np.load(tmp_path / "b" / f"{k}.npy"))
