"""CPU checks of scenes of several posed bodies: an fp64 restatement of the scene composite's definition against the
oracle's `composite` (one instance) and against the identities the definition implies (a duplicated instance, an
instance no ray reaches), every refusal of render_scene_rays / render_scene_images (raised before any device work,
with no parameter, gradient or state touched), and the ctypes signature of danbo_scene_composite against the header.
`scene_fp64` is also the reference of tests/test_gpu_scene.py."""
import ctypes
import os
import re
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)
import danbo_b200 as db                              # noqa: E402
import danbo_oracle as orc                           # noqa: E402
from danbo_b200 import _lib, kernels as K, raycaster, render   # noqa: E402
from danbo_b200 import skeleton as sk, synthetic as syn        # noqa: E402
from util import load_fixture, pose_tensors          # noqa: E402


# ---------------------------------------------------------------------------------------------------- definition
def scene_fp64(z_lists, raw_lists, rays_d):
    """The scene composite restated in fp64.  z_lists[k] (n,S) is instance k's merged list (sorted by z), raw_lists[k]
    (n,S,4) its raw (rgb logits, sigma) in that order, rays_d (n,3).  Each sample's alpha is taken over the distance to
    the next sample of its OWN list (1e10 after the last) times |d|; the union of all lists is ordered by z with ties to
    the lower instance, then the list position (a stable sort of the lists concatenated in instance order); w = alpha T
    with T the product of (1 - alpha + 1e-10) before the sample in the union.
    -> rgb (n,3), disp (n), acc (n), instance map (n,K) = per instance, the sum of its samples' weights."""
    norm = torch.norm(rays_d.double(), dim=-1, keepdim=True)
    zs, als, cs, ids = [], [], [], []
    for k, (z, raw) in enumerate(zip(z_lists, raw_lists)):
        z, raw = z.double(), raw.double()
        d = torch.cat([z[:, 1:] - z[:, :-1], torch.full_like(z[:, :1], 1e10)], -1) * norm
        als.append(1. - torch.exp(-torch.relu(raw[..., 3]) * d))
        cs.append(torch.sigmoid(raw[..., :3]) * 1.002 - 0.001)
        zs.append(z)
        ids.append(torch.full(z.shape, k, dtype=torch.long))
    z, order = torch.sort(torch.cat(zs, 1), dim=-1, stable=True)
    a = torch.gather(torch.cat(als, 1), 1, order)
    c = torch.gather(torch.cat(cs, 1), 1, order[..., None].expand(-1, -1, 3))
    inst = torch.gather(torch.cat(ids, 1), 1, order)
    T = torch.cumprod(torch.cat([torch.ones_like(a[:, :1]), 1. - a + 1e-10], -1), -1)[:, :-1]
    w = a * T
    wsum = w.sum(-1)
    disp = 1. / torch.clamp((w * z).sum(-1) / (wsum + 1e-10), min=1e-10)
    disp = torch.where(torch.isclose(wsum, torch.zeros_like(wsum)), torch.zeros_like(disp), disp)
    imap = torch.zeros(z.shape[0], len(z_lists), dtype=torch.float64).scatter_add_(1, inst, w)
    return (w[..., None] * c).sum(1), disp, torch.clamp(wsum, max=1.), imap


def _lists(n=64, S=48, seed=0, sigma_shift=0., z0=2.):
    """A random merged list per ray: sorted z in [z0, z0 + 2] with some repeated values, raw with sigma partly <= 0."""
    g = torch.Generator().manual_seed(seed)
    z = torch.sort(z0 + 2. * torch.rand(n, S, generator=g, dtype=torch.float64), -1).values
    z[:, 10] = z[:, 9]                                                # a tie inside the list
    raw = torch.randn(n, S, 4, generator=g, dtype=torch.float64) * 2.
    raw[..., 3] = raw[..., 3] * 3. + sigma_shift
    d = torch.randn(n, 3, generator=g, dtype=torch.float64)
    return z, raw, d


def test_one_instance_is_the_oracle_composite():
    """One instance: raw2outputs as the oracle states it (in fp32, the precision it runs at), on the same values."""
    z, raw, d = (t.float() for t in _lists(sigma_shift=-4.))
    rgb, disp, acc, imap = scene_fp64([z], [raw], d)
    ref = orc.composite(raw, z, d)
    torch.testing.assert_close(rgb, ref["rgb_map"].double(), rtol=0, atol=2e-6)
    torch.testing.assert_close(acc, ref["acc_map"].double(), rtol=0, atol=2e-6)
    torch.testing.assert_close(disp, ref["disp_map"].double(), rtol=2e-6, atol=0)
    torch.testing.assert_close(imap[:, 0], ref["weights"].double().sum(-1), rtol=0, atol=2e-6)
    assert float(acc.max()) > 0.5 and float(acc.min()) < 0.5           # neither empty nor saturated rays only


def test_duplicate_instance_identity():
    """Two copies of one list: every pair of equal samples multiplies T by (1 - alpha)^2, so acc' = 1 - (1 - acc)^2 up
    to the 1e-10 terms; the two columns share acc' in order (the lower instance first at each tie)."""
    z, raw, d = _lists(sigma_shift=-4.)
    _, _, acc1, _ = scene_fp64([z], [raw], d)
    _, _, acc2, imap = scene_fp64([z, z], [raw, raw], d)
    assert float((acc1 < 0.99).float().mean()) > 0.5                  # the identity is not checked at saturation only
    torch.testing.assert_close(acc2, 1. - (1. - acc1) ** 2, rtol=0, atol=1e-8)
    torch.testing.assert_close(imap.sum(-1), acc2, rtol=0, atol=1e-8)          # acc = min(sum w, 1)
    assert bool((imap[:, 0] >= imap[:, 1]).all())


def test_unreached_instance_changes_nothing():
    """An instance whose alpha is 0 on every sample (sigma <= 0) gets a column of exact zeros, wherever its samples
    fall among the other instance's, and leaves the maps at rounding level (its samples multiply T by 1 + 1e-10)."""
    za, ra, d = _lists(seed=1)
    zb, rb, _ = _lists(seed=2, z0=1.5)
    rb[..., 3] = -rb[..., 3].abs()
    a_alone = scene_fp64([za], [ra], d)
    for lists in (([za, zb], [ra, rb]), ([zb, za], [rb, ra])):
        rgb, disp, acc, imap = scene_fp64(*lists, d)
        b = 1 if lists[0][0] is za else 0
        assert bool((imap[:, b] == 0).all())
        for got, want in zip((rgb, disp, acc, imap[:, 1 - b]), a_alone[:3] + (a_alone[3][:, 0],)):
            torch.testing.assert_close(got, want, rtol=1e-7, atol=1e-7)


# ---------------------------------------------------------------------------------------------------- refusals
def _cpu_caster(preset):
    args = db.make_args(preset, no_reload=True)
    attrs = {"skel_type": sk.SMPLSkeleton, "near": syn.NEAR, "far": syn.FAR, "n_views": 8, "rest_pose": syn.rest_pose()}
    _, kw_test, *_ = db.create_raycaster(args, attrs, device="cpu")
    caster = kw_test["ray_caster"]
    caster.eval()
    return caster, args


@pytest.fixture
def no_device(monkeypatch):
    """Any use of the kernel library (which every device launch goes through) fails the test."""
    def boom():
        raise AssertionError("device work started before the refusal")
    monkeypatch.setattr(_lib, "load", boom)


def _instance(caster, fx, n_poses=1):
    skts, bones, cyl = pose_tensors(fx)
    rep = lambda t: t.expand(n_poses, *t.shape[1:])
    return {"caster": caster, "kps": rep(fx["pose_kps"][None]), "skts": rep(skts), "bones": rep(bones),
            "cyls": rep(cyl), "cams": 0}


def _state(caster):
    return ({k: v.clone() for k, v in caster.network.state_dict().items()},
            [None if p.grad is None else p.grad.clone() for p in caster.parameters()], caster.training,
            caster._packed, caster._align_dev)


def _same_state(a, b):
    assert a[0].keys() == b[0].keys() and all(torch.equal(a[0][k], b[0][k]) for k in a[0])
    assert all((x is None and y is None) or torch.equal(x, y) for x, y in zip(a[1], b[1]))
    assert a[2:] == b[2:]


def test_scene_refusals(no_device):
    caster, args = _cpu_caster("danbo_fast")
    fx = load_fixture("render_fast")
    rays = fx["ray_batch"][:4]
    inst = _instance(caster, fx)
    before = _state(caster)
    images = lambda insts, a=args: render.render_scene_images(insts, a, [np.eye(4, dtype=np.float32)], 8, 8)
    with torch.no_grad():
        for insts, word in (([], "instances"), ([inst] * 9, "instances"), ([inst, _instance(caster, fx, 2)], "one pose")):
            with pytest.raises(NotImplementedError, match=word):
                raycaster.render_scene_rays(rays, insts, args.N_samples, args.N_importance)
            with pytest.raises(NotImplementedError, match=word):
                images(insts)
        # 8 instances of 96 + 64 samples pass the per-instance bound (160) and exceed the union's (8 x 144)
        for S_c, S_f in ((96, 64), (128, 48)):
            with pytest.raises(NotImplementedError, match="at most"):
                raycaster.render_scene_rays(rays, [inst] * (8 if S_c == 96 else 1), S_c, S_f)
        with pytest.raises(NotImplementedError, match="at most"):
            images([inst] * 8, db.make_args("danbo_base", no_reload=True, N_importance=64))
        with pytest.raises(NotImplementedError, match="N_importance"):
            raycaster.render_scene_rays(rays, [inst], args.N_samples, 0)
    with torch.enable_grad():
        with pytest.raises(NotImplementedError, match="without gradients"):
            raycaster.render_scene_rays(rays, [inst], args.N_samples, args.N_importance)
    caster.train()
    with torch.no_grad():
        with pytest.raises(NotImplementedError, match="eval mode"):
            raycaster.render_scene_rays(rays, [inst], args.N_samples, args.N_importance)
    with pytest.raises(NotImplementedError, match="eval mode"):                 # render_scene_images runs no_grad
        images([inst])
    caster.eval()
    _same_state(before, _state(caster))


def test_anerf_caster_refuses_scenes(no_device):
    caster, _ = _cpu_caster("danbo_fast")
    acaster, a_args = _cpu_caster("anerf_base")
    fx = load_fixture("render_fast")
    before = _state(acaster)
    with torch.no_grad():
        for insts in ([_instance(acaster, fx)], [_instance(caster, fx), _instance(acaster, fx)]):
            with pytest.raises(NotImplementedError, match="DANBO field only"):
                raycaster.render_scene_rays(fx["ray_batch"][:4], insts, 24, 12)
            with pytest.raises(NotImplementedError, match="DANBO field only"):
                render.render_scene_images(insts, a_args, [np.eye(4, dtype=np.float32)], 8, 8)
    _same_state(before, _state(acaster))


def test_scene_composite_wrapper_checks_counts():
    for n_inst, S_c, S_f in ((0, 32, 16), (9, 32, 16), (8, 96, 64)):
        with pytest.raises(ValueError, match="instances"):
            K.scene_composite(torch.zeros(4, 11), S_c, S_f, [{}] * n_inst)


def test_rays_in_box_union():
    """Two cylinders: the rays of the union of their boxes; one cylinder, given as (5,) or (1,5): its own box."""
    H = W = 96
    focal, c2w = 1.2 * H, syn.camera(8.)                               # far enough for boxes inside the image
    cyl_a = syn.make_pose(3)["cyl"]
    cyl_b = cyl_a.copy()
    cyl_b[0] += 1.5
    _, _, ia = render.rays_in_box(H, W, focal, c2w, cyl_a, "cpu")
    _, _, ia1 = render.rays_in_box(H, W, focal, c2w, cyl_a[None], "cpu")
    _, _, ib = render.rays_in_box(H, W, focal, c2w, cyl_b, "cpu")
    _, _, iab = render.rays_in_box(H, W, focal, c2w, np.stack([cyl_a, cyl_b]), "cpu")
    assert torch.equal(ia, ia1)
    box = lambda idx: (int((idx // W).min()), int((idx // W).max()), int((idx % W).min()), int((idx % W).max()))
    (a0, a1, a2, a3), (b0, b1, b2, b3) = box(ia), box(ib)
    assert box(iab) == (min(a0, b0), max(a1, b1), min(a2, b2), max(a3, b3))
    assert iab.numel() == (box(iab)[1] - box(iab)[0] + 1) * (box(iab)[3] - box(iab)[2] + 1) > ia.numel()


# ---------------------------------------------------------------------------------------------------- ABI
def _decl(name):
    text = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "danbo_b200.h")).read(), flags=re.S)
    m = re.search(r"\bint\s+" + name + r"\s*\(([^;]*?)\)\s*;", text, flags=re.S)
    return [" ".join(p.split()) for p in m.group(1).replace("\n", " ").split(",")]


def test_scene_composite_signature():
    """danbo_scene_composite: the rays and sizes, n_inst, six host arrays of per-instance device pointers (the inputs
    of danbo_merge_composite, in its order), the four maps and the stream; the ctypes table matches the header; the ABI
    version is unchanged."""
    decl = _decl("danbo_scene_composite")
    assert decl == ["const float* rays", "int ray_stride", "int n_rays", "int S_c", "int S_f", "int n_inst",
                    "const float* const* raw0", "const unsigned int* const* mask0", "const float* const* raw1",
                    "const unsigned int* const* mask1", "const float* const* z_all", "const int* const* order",
                    "float* rgb", "float* disp", "float* acc", "float* inst_map", "void* stream"]
    merge = _decl("danbo_merge_composite")
    assert [p.replace("* const*", "*") for p in decl[6:12]] == merge[5:11]
    sig = _lib._SIGNATURES["danbo_scene_composite"]
    assert len(sig) == len(decl)
    for p, t in zip(decl, sig):
        assert t is (ctypes.c_void_p if "*" in p else ctypes.c_int), p
    assert _lib.ABI_VERSION == 5
