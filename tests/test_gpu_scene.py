"""Scenes of several posed bodies on the GPU (danbo_scene_composite, raycaster.render_scene_rays,
render.render_scene_images) with sigmoid and softmax casters: one instance against the plain render, several against
the fp64 restatement of test_scene_cpu built from each instance's own render, and the identities of the definition
(duplicates, unreached and occluded instances).  Measured numbers are printed."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)
from danbo_b200 import kernels as K, raycaster, render, synthetic as syn   # noqa: E402
from test_scene_cpu import scene_fp64                                      # noqa: E402
from util import agg_type_of, load_fixture, make_caster, pose_tensors, preset_of   # noqa: E402

pytestmark = pytest.mark.gpu
DEV = "cuda"
AGG = ["sigmoid", "softmax"]
FIXTURE = {"sigmoid": "render_fast", "softmax": "render_fast_softmax"}
PLAIN_EVAL_LAUNCHES = 24                 # one eval render_rays block of one pose (tests/test_gpu_parts.py)


@pytest.fixture(autouse=True)
def _keep_global_rng():
    """Building a caster draws from torch's global generators: restore them for the tests that run later."""
    cpu, cuda = torch.get_rng_state(), torch.cuda.get_rng_state_all()
    yield
    torch.set_rng_state(cpu)
    torch.cuda.set_rng_state_all(cuda)


def _caster(agg_type, density_gain=1.):
    caster, args, _ = make_caster("danbo_fast", agg_type=agg_type)
    caster.eval()
    if density_gain != 1.:                   # an opaque body: the random-init weights leave it translucent
        with torch.no_grad():
            caster.network.alpha_linear.weight.mul_(density_gain)
            caster.network.alpha_linear.bias.mul_(density_gain)
    return caster, args


def _moved(pose, t):
    """The pose translated by t (world): joints, world-to-bone transforms and the bounding cylinder (x, z, r, y, y)."""
    t = np.asarray(t, np.float32)
    skts = pose["skts"].copy()
    skts[:, :3, 3] -= skts[:, :3, :3] @ t
    cyl = pose["cyl"].copy()
    cyl[[0, 1, 3, 4]] += t[[0, 2, 1, 1]]
    return {"bones": pose["bones"], "kps": pose["kps"] + t, "skts": skts, "cyl": cyl}


def _instance(caster, pose, cams=0):
    d = lambda a: torch.as_tensor(np.asarray(a, np.float32))[None].to(DEV)
    return {"caster": caster, "kps": d(pose["kps"]), "skts": d(pose["skts"]), "bones": d(pose["bones"]),
            "cyls": d(pose["cyl"]), "cams": cams}


def _fx_pose(fx):
    skts, bones, cyl = pose_tensors(fx)
    return {"kps": fx["pose_kps"].numpy(), "skts": skts[0].numpy(), "bones": bones[0].numpy(), "cyl": cyl[0].numpy()}


def _rays(poses, H=64, stride=1):
    """Rays of the union of the poses' boxes in the synthetic camera (as render_scene_images makes them)."""
    cyls = np.stack([p["cyl"] for p in poses])
    ro, rd, _ = render.rays_in_box(H, H, 1.2 * H, syn.camera(), cyls, DEV)
    ones = torch.ones(ro.shape[0], 1, device=DEV)
    return torch.cat([ro, rd, syn.NEAR * ones, syn.FAR * ones, rd / torch.norm(rd, dim=-1, keepdim=True)], -1)[::stride]


def _alone(inst, rays, args, stages=None, chunk=None):
    """The instance's plain render_rays on the rays."""
    n = rays.shape[0]
    ex = lambda t: t.expand(n, *t.shape[1:])
    with torch.no_grad():
        return inst["caster"].render_rays(rays, N_samples=args.N_samples, kp_batch=ex(inst["kps"]),
                                          skts=ex(inst["skts"]), cyls=ex(inst["cyls"]), bones=ex(inst["bones"]),
                                          cams=torch.full((n, 1), inst["cams"], dtype=torch.long, device=DEV),
                                          N_uniques=1, perturb=False, N_importance=args.N_importance,
                                          raw_noise_std=0., nanmean_chunk=args.chunk if chunk is None else chunk,
                                          _stages=stages)


def _scene(insts, rays, args, chunk=None):
    with torch.no_grad():
        return raycaster.render_scene_rays(rays, insts, args.N_samples, args.N_importance,
                                           nanmean_chunk=args.chunk if chunk is None else chunk)


@pytest.mark.parametrize("agg_type", AGG)
def test_one_instance_is_the_plain_render(agg_type):
    """K = 1 on the fixture's rays: rgb, disp and acc are render_rays' bit for bit, instance_map[:, 0] is acc_map to
    fp32 rounding, and the call runs the plain call's launch count with the scene kernel in place of the merge."""
    fx = load_fixture(FIXTURE[agg_type])
    assert agg_type_of(fx) == agg_type and preset_of(fx) == "danbo_fast"
    caster, args = _caster(agg_type)
    inst = _instance(caster, _fx_pose(fx), cams=int(fx["cams"].reshape(-1)[0]))
    rays = fx["ray_batch"].to(DEV)
    _alone(inst, rays, args)                                              # packs the weights
    K.PROFILE = {"mlp": [], "launches": 0}
    try:
        plain = _alone(inst, rays, args)
        n_plain = K.PROFILE["launches"]
        K.PROFILE["launches"] = 0
        scene = _scene([inst], rays, args)
        n_scene = K.PROFILE["launches"]
    finally:
        K.PROFILE = None
    d_inst = float((scene["instance_map"][:, 0] - plain["acc_map"]).abs().max())
    print(f"[scene] {agg_type}: launches plain {n_plain}, scene {n_scene}; instance_map vs acc_map max |diff| "
          f"{d_inst:.3e}; max acc {float(plain['acc_map'].max()):.3f}")
    assert n_plain == PLAIN_EVAL_LAUNCHES and n_scene == n_plain
    assert set(scene) == {"rgb_map", "disp_map", "acc_map", "instance_map"} and scene["instance_map"].shape == (rays.shape[0], 1)
    for k in ("rgb_map", "disp_map", "acc_map"):
        assert torch.equal(scene[k], plain[k]), k
    assert d_inst <= 1e-6 and float(plain["acc_map"].max()) > 0.1


@pytest.mark.parametrize("n_inst", [2, 3])
def test_scene_against_fp64_restatement(n_inst):
    """K = 2 and 3 instances in different poses, sigmoid and softmax casters in one scene, partly overlapping in depth:
    the maps against scene_fp64 built from each instance's own render (its merged raw and z_all, `_stages`) on a fixed
    ray sample, max |diff| <= 1e-5 on rgb, acc and the instance map."""
    cs, args = _caster("sigmoid")
    cx, _ = _caster("softmax")
    poses = [syn.make_pose(3), _moved(syn.make_pose(5), (0.35, 0., -0.3)), _moved(syn.make_pose(7), (-0.3, 0.05, 0.4))]
    insts = [_instance(cs, poses[0]), _instance(cx, poses[1], cams=-1), _instance(cs, poses[2], cams=2)][:n_inst]
    rays = _rays(poses[:n_inst], stride=2)
    zs, raws = [], []
    for inst in insts:
        st = {}
        _alone(inst, rays, args, stages=st)
        zs.append(st["z_all"].cpu())
        raws.append(st["raw"].cpu())
    scene = _scene(insts, rays, args)
    rgb, disp, acc, imap = scene_fp64(zs, raws, rays[:, 3:6].cpu())
    e = {"rgb": float((scene["rgb_map"].cpu().double() - rgb).abs().max()),
         "acc": float((scene["acc_map"].cpu().double() - acc).abs().max()),
         "instance_map": float((scene["instance_map"].cpu().double() - imap).abs().max())}
    hit = imap > 0.05
    both = int((hit.sum(-1) >= 2).sum())
    print(f"[scene] K={n_inst} on {rays.shape[0]} rays: max |diff| vs fp64 " + ", ".join(f"{k} {v:.2e}" for k, v in e.items())
          + f"; rays where two instances each weigh > 0.05: {both}")
    assert max(e.values()) <= 1e-5
    assert both > 0                                                       # the bodies do overlap along rays


@pytest.mark.parametrize("agg_type", AGG)
def test_duplicate_instance(agg_type):
    """The same instance twice: acc = 1 - (1 - acc_1)^2 within 1e-6, acc_1 the instance's plain render."""
    fx = load_fixture(FIXTURE[agg_type])
    caster, args = _caster(agg_type)
    inst = _instance(caster, _fx_pose(fx))
    rays = fx["ray_batch"].to(DEV)
    acc1 = _alone(inst, rays, args)["acc_map"]
    scene = _scene([inst, inst], rays, args)
    err = float((scene["acc_map"] - (1. - (1. - acc1) ** 2)).abs().max())
    print(f"[scene] {agg_type}: duplicate instance, acc vs 1 - (1 - acc_1)^2 max |diff| {err:.2e} "
          f"(max acc_1 {float(acc1.max()):.3f})")
    assert err <= 1e-6 and float(acc1.max()) > 0.1
    assert bool((scene["instance_map"][:, 0] >= scene["instance_map"][:, 1]).all())


def test_separated_bodies():
    """B 3 m beside A: on the rays where B's own render has every alpha 0, the scene is A alone within 1e-6 and
    instance_map[:, B] is exactly 0."""
    cs, args = _caster("sigmoid")
    cx, _ = _caster("softmax")
    pa, pb = syn.make_pose(3), _moved(syn.make_pose(5), (3., 0., 0.))
    a, b = _instance(cs, pa), _instance(cx, pb)
    rays = _rays([pa])
    alone_a, alone_b = _alone(a, rays, args), _alone(b, rays, args)
    for order in ((a, b), (b, a)):
        scene = _scene(list(order), rays, args)
        ib = order.index(b)
        free = (alone_b["alpha"] == 0).all(-1)
        d = {k: float((scene[k][free] - alone_a[k][free]).abs().max()) for k in ("rgb_map", "disp_map", "acc_map")}
        d["instance_map[A]"] = float((scene["instance_map"][free, 1 - ib] - alone_a["acc_map"][free]).abs().max())
        print(f"[scene] separated, B at {ib}: {int(free.sum())} of {rays.shape[0]} rays B does not reach; max |diff| "
              f"vs A alone " + ", ".join(f"{k} {v:.2e}" for k, v in d.items()))
        assert int(free.sum()) > rays.shape[0] // 2 and float(alone_a["acc_map"][free].max()) > 0.1
        assert max(d.values()) <= 1e-6
        assert bool((scene["instance_map"][free, ib] == 0).all())


def test_occlusion():
    """A (an opaque field) 1.5 m in front of B along the camera axis: where A alone has acc > 0.99, the scene's rgb is
    A's within 1e-2 and B's weight is below 0.01."""
    ca, args = _caster("sigmoid", density_gain=20.)
    cb, _ = _caster("softmax", density_gain=20.)
    pa, pb = syn.make_pose(3), _moved(syn.make_pose(5), (0.1, 0., -1.5))
    a, b = _instance(ca, pa), _instance(cb, pb)
    rays = _rays([pa, pb])
    alone_a, alone_b = _alone(a, rays, args), _alone(b, rays, args)
    scene = _scene([b, a], rays, args)
    front = alone_a["acc_map"] > 0.99
    d = float((scene["rgb_map"][front] - alone_a["rgb_map"][front]).abs().max())
    wb = float(scene["instance_map"][front, 0].max())
    behind = front & (alone_b["acc_map"] > 0.5)
    print(f"[scene] occlusion: {int(front.sum())} of {rays.shape[0]} rays with A's acc > 0.99 ({int(behind.sum())} of "
          f"them with B's own acc > 0.5); rgb vs A alone max |diff| {d:.2e}, max weight of B {wb:.2e}")
    assert int(behind.sum()) > 20
    assert d <= 1e-2 and wb < 0.01


def test_blocks(monkeypatch):
    """A call of 2 instances cut into two launch blocks (MAX_RAYS_PER_LAUNCH lowered to 1024, nanmean_chunk 256)
    equals the one-block call bit for bit."""
    cs, args = _caster("sigmoid")
    cx, _ = _caster("softmax")
    poses = [syn.make_pose(3), _moved(syn.make_pose(5), (0.35, 0., -0.3))]
    insts = [_instance(cs, poses[0]), _instance(cx, poses[1])]
    rays = _rays(poses, H=96)[:2048]
    assert rays.shape[0] == 2048
    one = _scene(insts, rays, args, chunk=256)
    monkeypatch.setattr(raycaster, "MAX_RAYS_PER_LAUNCH", 1024)
    cut = _scene(insts, rays, args, chunk=256)
    assert raycaster.RayCaster._plan_blocks(2048, 1, 2048, 256, 1)[0] == 1024
    for k in one:
        assert torch.equal(one[k], cut[k]), k
    assert float(one["acc_map"].max()) > 0.1


@pytest.mark.parametrize("agg_type", AGG)
def test_scene_images(agg_type):
    """render_scene_images: one instance gives render_images' images bit for bit; with two bodies the instance maps
    are 0 off the boxes, and part_labels gives -1 there."""
    caster, args = _caster(agg_type)
    H = W = 64
    pa, pb = syn.make_pose(3), _moved(syn.make_pose(5), (0.6, 0., -0.3))
    c2ws = [syn.camera(), syn.bullet_time_cameras(syn.camera(), 8)[1]]
    imgs, imaps = render.render_scene_images([_instance(caster, pa)], args, c2ws, H, W)
    want = render.render_images(caster, args, c2ws, [pa], H, W)
    assert imgs.shape == (2, H, W, 3) and imaps.shape == (2, H, W, 1) and torch.equal(imgs, want)
    imgs2, imaps2 = render.render_scene_images([_instance(caster, pa), _instance(caster, pb)], args, c2ws, H, W)
    assert imaps2.shape == (2, H, W, 2)
    for k, c2w in enumerate(c2ws):
        _, _, idx = render.rays_in_box(H, W, 1.2 * H, c2w, np.stack([pa["cyl"], pb["cyl"]]), DEV)
        bg = torch.ones(H * W, dtype=torch.bool, device=DEV)
        bg[idx] = False
        m = imaps2[k].reshape(-1, 2)
        assert torch.equal(m[bg], torch.zeros(int(bg.sum()), 2, device=DEV))
        assert bool((imgs2[k].reshape(-1, 3)[bg] == 1.).all())                  # white background
        lab = render.part_labels(imaps2[k], min_weight=0.5 * float(imaps2[k].max())).reshape(-1)
        assert bool((lab[bg] == -1).all()) and int((lab >= 0).sum()) > 0
        print(f"[scene] {agg_type} image {k}: {int(bg.sum())} background pixels, labels A {int((lab == 0).sum())}, "
              f"B {int((lab == 1).sum())}")
