"""Generates tests/golden/*.npz by running the UNMODIFIED reference (see oracle/ref_harness.py).

    python oracle/gen_golden.py            # needs the reference ($DANBO_REFERENCE or baseline/_ref); writes tests/golden/

Every fixture holds the synthetic inputs (SURVEY §8d), the seed of the deterministic weights
(danbo_b200.synthetic.synth_state_dict, numpy RandomState -> reproducible anywhere) and the reference's own
tensors at each stage boundary of SURVEY §8(a), captured by wrapping the reference's functions in place.
The reference is never committed; the tests only need these vectors.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

import danbo_b200  # noqa: E402
from danbo_b200 import synthetic as syn, params  # noqa: E402
import ref_harness as rh  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
STAGE_RAYS = 16          # rays for which the big per-(sample,bone) tensors are kept


class Tap:
    """Wraps callables on the reference objects and records what flows through them."""

    def __init__(self):
        self.rec = {}
        self._undo = []

    def add(self, key, val):
        self.rec.setdefault(key, []).append(val.detach().clone() if torch.is_tensor(val) else val)

    def wrap(self, obj, name, fn):
        import types
        orig = getattr(obj, name)
        if isinstance(orig, torch.nn.Module):            # child module: observe through a forward hook
            h = orig.register_forward_hook(lambda m, a, out: fn(lambda *x, **y: out))
            self._undo.append(("hook", h, None, None))
            return
        is_module_global = isinstance(obj, types.ModuleType)
        setattr(obj, name, lambda *a, **k: fn(orig, *a, **k))
        self._undo.append(("global" if is_module_global else "inst", obj, name, orig))

    def undo(self):
        for kind, obj, name, orig in reversed(self._undo):
            if kind == "hook":
                obj.remove()
            elif kind == "global":
                setattr(obj, name, orig)
            else:
                obj.__dict__.pop(name, None)             # un-shadow the bound method
        self._undo = []


def tap_reference(caster, tap, rc):
    net = caster.network

    def cyl(orig, *a, **k):
        n, f = orig(*a, **k)
        tap.add("near_cyl", n), tap.add("far_cyl", f)
        return n, f
    tap.wrap(rc, "get_near_far_in_cylinder", cyl)

    def nf(orig, *a, **k):
        n, f = orig(*a, **k)
        tap.add("near", n), tap.add("far", f)
        return n, f
    tap.wrap(caster, "get_near_far", nf)

    def boxes(orig, *a, **k):
        pv, vv, seg = orig(*a, **k)
        tap.add("p_valid", pv), tap.add("v_valid", vv)
        return pv, vv, seg
    tap.wrap(rc, "get_ray_box_intersections", boxes)

    def spts(orig, *a, **k):
        pts, z = orig(*a, **k)
        tap.add("z", z)
        return pts, z
    tap.wrap(caster, "sample_pts", spts)

    def spts_is(orig, *a, **k):
        pts, z_all, zs, order = orig(*a, **k)
        tap.add("z_all", z_all), tap.add("z_samples", zs), tap.add("sorted_idxs", order)
        return pts, z_all, zs, order
    tap.wrap(caster, "sample_pts_is", spts_is)

    def emb(orig, *a, **k):
        enc = orig(*a, **k)
        tap.add("pts_t", enc["pts_t"][:STAGE_RAYS])
        return enc
    tap.wrap(net.pts_embedder, "encode_pts", emb)

    def gfwd(orig, *a, **k):
        v = orig(*a, **k)
        tap.add("vol", v)
        return v
    tap.wrap(net, "forward_graph", gfwd)

    def gpe(orig, *a, **k):
        w = orig(*a, **k)
        tap.add("graph_w", w[0])
        return w
    tap.wrap(net, "graph_pe_fn", gpe)

    def samp(orig, *a, **k):
        h, inv = orig(*a, **k)
        tap.add("h", h[:STAGE_RAYS]), tap.add("invalid", inv)
        return h, inv
    tap.wrap(net, "extract_graph_feat", samp)

    def enc_pts(orig, *a, **k):
        d, enc = orig(*a, **k)
        S = enc["confd"].shape[1]
        tap.add("density_inputs", d[:STAGE_RAYS * S]), tap.add("confd", enc["confd"]), tap.add("agg_p", enc["agg_p"])
        return d, enc
    tap.wrap(net, "encode_pts", enc_pts)

    def enc_views(orig, *a, **k):
        v, enc = orig(*a, **k)
        S = a[0]["pts"].shape[1] if a else k["inputs"]["pts"].shape[1]
        tap.add("view_inputs", v[::S])
        return v, enc
    tap.wrap(net, "encode_views", enc_views)

    def r2o(orig, raw, z, rays_d, *a, **k):
        out = orig(raw, z, rays_d, *a, **k)
        tap.add("raw", raw), tap.add("weights", out["weights"]), tap.add("alpha", out["alpha"])
        return out
    tap.wrap(net, "raw2outputs", r2o)

    def spdf(orig, *a, **k):
        return orig(*a, **k)
    tap.wrap(rc, "sample_pdf", spdf)


class RandTape:
    """Records torch.rand / torch.randn draws in call order (SURVEY §7 hard part 4)."""

    def __enter__(self):
        self.tape = []
        self._rand, self._randn = torch.rand, torch.randn

        def rand(*a, **k):
            t = self._rand(*a, **k)
            self.tape.append(("rand", t.clone()))
            return t

        def randn(*a, **k):
            t = self._randn(*a, **k)
            self.tape.append(("randn", t.clone()))
            return t
        torch.rand, torch.randn = rand, randn
        return self

    def __exit__(self, *exc):
        torch.rand, torch.randn = self._rand, self._randn


def npify(d):
    out = {}
    for k, v in d.items():
        if torch.is_tensor(v):
            v = v.detach().cpu().numpy()
        out[k] = v
    return out


def subsample_rays(batch, n, seed=0):
    tot = batch["ray_batch"].shape[0]
    pick = torch.as_tensor(np.sort(np.random.RandomState(seed).choice(tot, n, replace=False)))
    out = {}
    for k, v in batch.items():
        out[k] = v[pick].contiguous() if torch.is_tensor(v) and v.shape[0] == tot else v
    return out


def run_render_case(name, config, extra, pose_seed, H, n_rays, weight_seed=0, full_image=False):
    rc, _ = rh._imports()
    args = rh.parse_args(config, extra)
    rest = syn.rest_pose()
    caster, kw = rh.build(args, rest)
    caster.eval()
    # (opt_framecode=False, configs/surreal: the standard synthetic weights without the frame-code part)
    sd = {k: v for k, v in syn.synthetic_params(weight_seed, opt_framecode=bool(args.opt_framecode)).items()
          if k not in params.BUFFER_NAMES and k != "graph_net.axis_scale"}
    rh.load_weights(caster, sd)
    pose = syn.make_pose(pose_seed)
    b = subsample_rays(syn.render_batch(pose, H, H, full_image=full_image), n_rays, seed=pose_seed)
    cams = b["cams"] if args.opt_framecode else None           # trainer.py:310: no cams without frame codes
    tap = Tap()
    tap_reference(caster, tap, rc)
    kwargs = {k: v for k, v in kw.items() if k not in ("ray_caster", "N_samples", "use_viewdirs")}
    with torch.no_grad():
        ret = caster(b["ray_batch"], N_samples=args.N_samples, kp_batch=b["kp_batch"], skts=b["skts"],
                     cyls=b["cyls"], bones=b["bones"], cams=cams, N_uniques=1, **kwargs)
    tap.undo()
    fx = {"config": config, "extra": " ".join(extra), "pose_seed": pose_seed, "weight_seed": weight_seed, "H": H,
          "N_samples": args.N_samples, "N_importance": args.N_importance,
          "use_volume_near_far": int(bool(args.use_volume_near_far)), "opt_framecode": int(bool(args.opt_framecode)),
          "ray_batch": b["ray_batch"], "cams": b["cams"], "pose_bones": pose["bones"], "pose_kps": pose["kps"],
          "pose_skts": pose["skts"], "pose_cyl": pose["cyl"]}
    for k, v in ret.items():
        fx["out." + k] = v
    for k, lst in tap.rec.items():
        for i, v in enumerate(lst):
            fx[f"st.{k}.{i}"] = v
    path = os.path.join(OUT, name + ".npz")
    np.savez_compressed(path, **npify(fx))
    print(name, "->", path, f"{os.path.getsize(path) / 1e6:.2f} MB", {k: len(v) for k, v in tap.rec.items()})


def run_anerf_case(name, extra, pose_seed, H, n_rays, weight_seed=0, config="h36m_zju/anerf_base.txt"):
    """A-NeRF (BASELINE config #4): eval-mode render_rays of the reference's plain RayCaster + NeRF(W=448).
    With configs/h36m_zju/anerf_h.txt (single_net = False) the separate fine network gets the weights of seed + 1."""
    rc, _ = rh._imports()
    args = rh.parse_args(config, extra)
    rest = syn.rest_pose()
    caster, kw = rh.build(args, rest)
    caster.eval()
    sd = syn.synth_state_dict(params.anerf_param_shapes(), weight_seed)
    rh.load_weights(caster, sd)
    if caster.network_fine is not caster.network:
        fine = caster.network_fine
        own = fine.state_dict()
        for k, v in syn.synth_state_dict(params.anerf_param_shapes(), weight_seed + 1).items():
            assert k in own and tuple(own[k].shape) == tuple(v.shape), k
            own[k] = v.clone()
        fine.load_state_dict(own)
    pose = syn.make_pose(pose_seed)
    b = subsample_rays(syn.render_batch(pose, H, H), n_rays, seed=pose_seed)
    net = caster.network
    tap = Tap()

    def cyl(orig, *a, **k):
        n, f = orig(*a, **k)
        tap.add("near", n), tap.add("far", f)
        return n, f
    tap.wrap(rc, "get_near_far_in_cylinder", cyl)

    def spts(orig, *a, **k):
        pts, z = orig(*a, **k)
        tap.add("z", z)
        return pts, z
    tap.wrap(caster, "sample_pts", spts)

    def spts_is(orig, *a, **k):
        pts, z_all, zs, order = orig(*a, **k)
        tap.add("z_all", z_all), tap.add("z_samples", zs), tap.add("sorted_idxs", order)
        return pts, z_all, zs, order
    tap.wrap(caster, "sample_pts_is", spts_is)

    def enc_pts(orig, *a, **k):
        d, enc = orig(*a, **k)
        S = enc["v"].shape[1]
        tap.add("density_inputs", d[:STAGE_RAYS * S]), tap.add("v", enc["v"][:STAGE_RAYS])
        return d, enc
    tap.wrap(net, "encode_pts", enc_pts)

    def enc_views(orig, *a, **k):
        v, enc = orig(*a, **k)
        S = k["refs"].shape[1]
        tap.add("view_inputs", v[:STAGE_RAYS * S])
        return v, enc
    tap.wrap(net, "encode_views", enc_views)

    def r2o(orig, raw, z, rays_d, *a, **k):
        out = orig(raw, z, rays_d, *a, **k)
        tap.add("raw", raw), tap.add("weights", out["weights"]), tap.add("alpha", out["alpha"])
        return out
    tap.wrap(net, "raw2outputs", r2o)
    if caster.network_fine is not net:
        tap.wrap(caster.network_fine, "raw2outputs", r2o)

    kwargs = {k: v for k, v in kw.items() if k not in ("ray_caster", "N_samples", "use_viewdirs")}
    with torch.no_grad():
        ret = caster(b["ray_batch"], N_samples=args.N_samples, kp_batch=b["kp_batch"], skts=b["skts"],
                     cyls=b["cyls"], bones=b["bones"], cams=b["cams"], N_uniques=1, **kwargs)
    tap.undo()
    fx = {"config": config, "extra": " ".join(extra), "pose_seed": pose_seed, "weight_seed": weight_seed, "H": H,
          "single_net": int(bool(args.single_net)),
          "N_samples": args.N_samples, "N_importance": args.N_importance, "tau": float(net.pe_fn.get_tau()),
          "ray_batch": b["ray_batch"], "cams": b["cams"], "pose_bones": pose["bones"], "pose_kps": pose["kps"],
          "pose_skts": pose["skts"], "pose_cyl": pose["cyl"]}
    for k, v in ret.items():
        fx["out." + k] = v
    for k, lst in tap.rec.items():
        for i, v in enumerate(lst):
            fx[f"st.{k}.{i}"] = v
    path = os.path.join(OUT, name + ".npz")
    np.savez_compressed(path, **npify(fx))
    print(name, "->", path, f"{os.path.getsize(path) / 1e6:.2f} MB", {k: len(v) for k, v in tap.rec.items()})


def run_train_case(name, config, extra, n_poses, rays_per_pose, weight_seed=0, batch_seed=0, pose_grads=False):
    rc, _ = rh._imports()
    import core.trainer as trainer_mod
    args = rh.parse_args(config, extra)
    rest = syn.rest_pose()
    caster, kw = rh.build(args, rest)
    caster.train()
    anerf = args.nerf_type == "nerf"
    if anerf:
        sd = syn.synth_state_dict(params.anerf_param_shapes(), weight_seed)
    else:
        sd = {k: v for k, v in syn.synthetic_params(weight_seed, opt_framecode=bool(args.opt_framecode)).items()
              if k not in params.BUFFER_NAMES and k != "graph_net.axis_scale"}
    rh.load_weights(caster, sd)
    b = syn.training_batch(n_poses, rays_per_pose, seed=batch_seed)
    cams = b["cams"] if args.opt_framecode else None               # trainer.py:310
    if pose_grads:
        # the pose tensors as leaves: what the pose layer's outputs are to the ray caster under --opt_pose
        # (core/trainer.py:314-341); their gradients pin the oracle for the backward-to-poses kernels (SURVEY §8f rank 2)
        for k in ("skts", "bones", "kp_batch"):
            b[k] = b[k].clone().requires_grad_(True)
    tap = Tap()
    if not anerf:
        tap_reference(caster, tap, rc)
    torch.manual_seed(1234)
    with RandTape() as tape:
        ret = caster(b["ray_batch"], N_samples=args.N_samples, kp_batch=b["kp_batch"], skts=b["skts"],
                     cyls=b["cyls"], bones=b["bones"], cams=cams, N_uniques=n_poses,
                     perturb=args.perturb, N_importance=args.N_importance, raw_noise_std=args.raw_noise_std,
                     ray_noise_std=0., ext_scale=args.ext_scale, lindisp=False, nerf_type=args.nerf_type,
                     preproc_kwargs={"density_scale": args.density_scale, "density_fn": torch.nn.functional.relu})
    tap.undo()
    # the trainer's own loss code (core/trainer.py:348-553) on a minimal shim of its state
    class _Wrap:                                   # stands in for nn.DataParallel(...).module
        def __init__(self, m): self.module = m
    tr = trainer_mod.Trainer.__new__(trainer_mod.Trainer)
    tr.args = args
    tr.render_kwargs_train = {"ray_caster": _Wrap(caster)}
    batch = {"target_s": b["target_s"], "bgs": b["bgs"]}
    loss_dict, stats = tr.compute_loss(batch, ret, kp_opts=None, popt_detach=True, global_step=0)
    loss_dict["total_loss"].backward()
    fx = {"config": config, "extra": " ".join(extra), "weight_seed": weight_seed, "batch_seed": batch_seed,
          "n_poses": n_poses, "rays_per_pose": rays_per_pose,
          "N_samples": args.N_samples, "N_importance": args.N_importance,
          "use_volume_near_far": int(bool(args.use_volume_near_far)),
          "raw_noise_std": args.raw_noise_std, "opt_framecode": int(bool(args.opt_framecode)), "loss_fn": args.loss_fn,
          "loss.total": loss_dict["total_loss"].detach()}
    for k, v in loss_dict.items():
        fx["loss." + k] = v.detach()
    kinds = [k for k, _ in tape.tape]
    if args.raw_noise_std > 0:
        assert kinds == ["rand", "randn", "rand", "randn"], kinds
        names = ("t_rand", "noise0", "u", "noise1")
    else:                                                    # no density noise drawn (nerf.py:314-316)
        assert kinds == ["rand", "rand"], kinds
        names = ("t_rand", "u")
    for nm, (_, t) in zip(names, tape.tape):
        fx["rand." + nm] = t
    for k, v in ret.items():
        fx["out." + k] = v.detach()
    for k, lst in tap.rec.items():
        if k in ("h", "pts_t", "density_inputs", "agg_p"):
            continue
        for i, v in enumerate(lst):
            fx[f"st.{k}.{i}"] = v
    if pose_grads:
        for k in ("skts", "bones", "kp_batch"):
            g = b[k].grad
            fx["pose_grad." + k] = torch.zeros(n_poses, *b[k].shape[1:]) if g is None else \
                g.reshape(n_poses, rays_per_pose, *g.shape[1:]).sum(1)
            fx["pose_grad_none." + k] = int(g is None)
    rng = np.random.RandomState(7)
    for n, p in caster.network.named_parameters():
        g = p.grad
        if g is None:
            continue
        flat = g.detach().reshape(-1)
        idx = torch.as_tensor(rng.choice(flat.numel(), min(512, flat.numel()), replace=False))
        fx["grad_idx." + n] = idx
        fx["grad_val." + n] = flat[idx]
        fx["grad_norm." + n] = flat.norm()
        fx["grad_sum." + n] = flat.double().sum()
    path = os.path.join(OUT, name + ".npz")
    np.savez_compressed(path, **npify(fx))
    print(name, "->", path, f"{os.path.getsize(path) / 1e6:.2f} MB")


def run_grid_case(name, config, pose_seed, res, radius=0.9, weight_seed=0):
    rc, _ = rh._imports()
    args = rh.parse_args(config)
    rest = syn.rest_pose()
    caster, kw = rh.build(args, rest)
    caster.eval()
    shapes = params.anerf_param_shapes() if args.nerf_type == "nerf" else params.danbo_param_shapes()
    rh.load_weights(caster, syn.synth_state_dict(shapes, weight_seed))
    pose = syn.make_pose(pose_seed)
    t = lambda a: torch.as_tensor(a)[None]
    with torch.no_grad():
        sigma = caster(kps=t(pose["kps"]), skts=t(pose["skts"]), bones=t(pose["bones"]), radius=radius, res=res,
                       fwd_type="mesh")
    fx = {"config": config, "pose_seed": pose_seed, "weight_seed": weight_seed, "res": res, "radius": radius,
          "pose_bones": pose["bones"], "pose_kps": pose["kps"], "pose_skts": pose["skts"], "sigma": sigma}
    path = os.path.join(OUT, name + ".npz")
    np.savez_compressed(path, **npify(fx))
    print(name, "->", path, f"{os.path.getsize(path) / 1e6:.2f} MB")


def main():
    assert rh.available(), "needs the reference ($DANBO_REFERENCE or baseline/_ref)"
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(8)
    only = sys.argv[1] if len(sys.argv) > 1 else None       # `python oracle/gen_golden.py anerf` regenerates that case only
    if only == "anerf":
        run_anerf_case("render_anerf", ["--N_samples", "24", "--N_importance", "12"], pose_seed=4, H=64, n_rays=64)
        return
    if only == "variants":
        variants()
        return
    if only == "train_anerf":
        run_train_case("train_anerf", "h36m_zju/anerf_base.txt", ["--N_samples", "24", "--N_importance", "12"],
                       n_poses=2, rays_per_pose=24)
        return
    if only == "train_popt":
        run_train_case("train_fast_popt", "h36m_zju/danbo_fast.txt", [], n_poses=4, rays_per_pose=48, batch_seed=1,
                       pose_grads=True)
        return
    if only == "train_nonoise":
        nonoise()
        return
    if only == "train_perfcap":
        run_train_case("train_perfcap", "perfcap/danbo_fast.txt", [], n_poses=4, rays_per_pose=48, batch_seed=3)
        return
    if only == "train_surreal":
        run_train_case("train_surreal", "surreal/danbo_fast.txt", [], n_poses=4, rays_per_pose=48, batch_seed=2)
        return
    if only == "surreal":
        run_render_case("render_surreal", "surreal/danbo_fast.txt", [], pose_seed=5, H=64, n_rays=200)
        return
    if only == "perfcap":
        run_render_case("render_perfcap", "perfcap/danbo_fast.txt", [], pose_seed=6, H=64, n_rays=160)
        return
    if only == "anerf_h":
        run_anerf_case("render_anerf_h", ["--N_samples", "24", "--N_importance", "12"], pose_seed=4, H=64, n_rays=48,
                       config="h36m_zju/anerf_h.txt")
        return
    if only == "grid_anerf":
        run_grid_case("grid_anerf", "h36m_zju/anerf_base.txt", pose_seed=4, res=9)
        return
    run_render_case("render_fast", "h36m_zju/danbo_fast.txt", [], pose_seed=3, H=64, n_rays=256)
    run_render_case("render_base", "h36m_zju/danbo_base.txt", [], pose_seed=5, H=64, n_rays=96)
    run_render_case("render_fast_miss", "h36m_zju/danbo_fast.txt", [], pose_seed=7, H=48, n_rays=192, full_image=True)
    run_train_case("train_fast", "h36m_zju/danbo_fast.txt", [], n_poses=4, rays_per_pose=48)
    run_train_case("train_cfg3", "h36m_zju/danbo_base.txt", ["--N_samples", "64", "--N_importance", "16"],
                   n_poses=2, rays_per_pose=32)
    run_grid_case("grid_base", "h36m_zju/danbo_base.txt", pose_seed=3, res=11)
    run_anerf_case("render_anerf", ["--N_samples", "24", "--N_importance", "12"], pose_seed=4, H=64, n_rays=64)
    variants()
    run_grid_case("grid_anerf", "h36m_zju/anerf_base.txt", pose_seed=4, res=9)
    run_anerf_case("render_anerf_h", ["--N_samples", "24", "--N_importance", "12"], pose_seed=4, H=64, n_rays=48,
                   config="h36m_zju/anerf_h.txt")
    # train-mode A-NeRF step (loss + gradients): pins the oracle ahead of the A-NeRF backward kernels (DESIGN §8)
    run_train_case("train_anerf", "h36m_zju/anerf_base.txt", ["--N_samples", "24", "--N_importance", "12"],
                   n_poses=2, rays_per_pose=24)
    # configs/perfcap/danbo_*.txt: view directions in the root joint's frame (ray_tr_type=root_local, view_type=relray)
    run_render_case("render_perfcap", "perfcap/danbo_fast.txt", [], pose_seed=6, H=64, n_rays=160)
    # configs/surreal/danbo_*.txt: no per-frame code (opt_framecode=False)
    run_render_case("render_surreal", "surreal/danbo_fast.txt", [], pose_seed=5, H=64, n_rays=200)
    run_train_case("train_surreal", "surreal/danbo_fast.txt", [], n_poses=4, rays_per_pose=48, batch_seed=2)
    run_train_case("train_perfcap", "perfcap/danbo_fast.txt", [], n_poses=4, rays_per_pose=48, batch_seed=3)
    # gradients with respect to the pose tensors (skts, bones): pins the oracle ahead of the backward-to-poses kernels
    run_train_case("train_fast_popt", "h36m_zju/danbo_fast.txt", [], n_poses=4, rays_per_pose=48, batch_seed=1,
                   pose_grads=True)
    nonoise()


def nonoise():
    """The two training cases again with --raw_noise_std 0: without the reference's random density gate
    (relu(raw + noise)) the end-to-end gradient comparison measures the kernels, not which samples the noise kept."""
    run_train_case("train_fast_nonoise", "h36m_zju/danbo_fast.txt", ["--raw_noise_std", "0"], n_poses=4, rays_per_pose=48)
    run_train_case("train_cfg3_nonoise", "h36m_zju/danbo_base.txt",
                   ["--N_samples", "64", "--N_importance", "16", "--raw_noise_std", "0"], n_poses=2, rays_per_pose=32)


def variants():
    """Flag values outside the shipped configs that the path supports: agg_type=softmax (the CLI default,
    run_nerf.py:364; danbo.py:388-404) in eval and train mode, and lindisp (ray_utils.py:226-227)."""
    run_render_case("render_fast_softmax", "h36m_zju/danbo_fast.txt", ["--agg_type", "softmax"], pose_seed=3, H=64, n_rays=128)
    run_train_case("train_fast_softmax", "h36m_zju/danbo_fast.txt", ["--agg_type", "softmax"], n_poses=4, rays_per_pose=48)
    run_render_case("render_fast_lindisp", "h36m_zju/danbo_fast.txt", ["--lindisp"], pose_seed=3, H=64, n_rays=256)


if __name__ == "__main__":
    main()
