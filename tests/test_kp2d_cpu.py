"""CPU checks of the 2D keypoint reprojection term: the closed-form d kps that danbo_pose_kp2d computes, restated in
torch, against fp64 autograd of pose_opt.kp2d_loss; render.projection_matrix against the rays of render.rays_in_box; the
batch checks of training.kp2d_batch, raised by PoseFitStep and TrainStep before any kernel call; and the ctypes
signature of danbo_pose_kp2d against the header."""
import ctypes
import os
import re
import sys
import types

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import danbo_b200 as db                              # noqa: E402
from danbo_b200 import _lib, pose_opt as po, render, synthetic as syn, training   # noqa: E402

FX = np.load(os.path.join(ROOT, "tests", "golden", "popt.npz"))


def closed_form(kps, kp2d, proj, sigma, coef):
    """danbo_pose_kp2d's arithmetic, joint by joint: (loss, kp2d_px, d loss / d kps)."""
    G, J = kps.shape[:2]
    s2, scale = sigma * sigma, coef / (G * J)
    X = torch.cat([kps, torch.ones_like(kps[..., :1])], -1)
    h = torch.einsum("grc,gjc->gjr", proj, X)
    d = torch.zeros_like(kps)
    loss, px, seen = 0., 0., 0
    for g in range(G):
        P = proj[g]
        for j in range(J):
            w = h[g, j, 2]
            if not w > 1e-6:
                continue
            u, v = h[g, j, 0] / w, h[g, j, 1] / w
            ru, rv = u - kp2d[g, j, 0], v - kp2d[g, j, 1]
            c = kp2d[g, j, 2]
            qu, qv = s2 + ru * ru, s2 + rv * rv
            loss = loss + c * (s2 * ru * ru / qu + s2 * rv * rv / qv)
            if c > 0:
                px, seen = px + torch.sqrt(ru * ru + rv * rv), seen + 1
            gu = scale * c * 2 * s2 * s2 * ru / (qu * qu) / w
            gv = scale * c * 2 * s2 * s2 * rv / (qv * qv) / w
            d[g, j] = gu * (P[0, :3] - u * P[2, :3]) + gv * (P[1, :3] - v * P[2, :3])
    return loss * scale, (px / seen if seen else torch.zeros(())), d


def _scene(G=4, seed=0, H=256, W=256, at_centre=True):
    """Joints of synthetic poses, the bullet-time cameras, and detections at the projections plus residuals of every
    scale: ~1e-3 px, ~sigma, far beyond sigma; some joints with c = 0 and, with G > 2, two behind their cameras (one of
    them at the camera centre with at_centre)."""
    rng = np.random.RandomState(seed)
    kps = np.stack([syn.make_pose(seed * G + g)["kps"] for g in range(G)]).astype(np.float64)
    c2ws = syn.bullet_time_cameras(syn.camera(), G)
    proj = render.projection_matrix(c2ws, H, W, 1.2 * H)
    c2w = c2ws.astype(np.float64)
    if G > 2:
        kps[1, 5] = c2w[1, :3, 3] + (0. if at_centre else c2w[1, :3, :3] @ np.array([0.0, 0.0, 0.3]))   # w = 0 or < 0
        kps[2, 9] = c2w[2, :3, 3] + c2w[2, :3, :3] @ np.array([0.1, 0.0, 1.0])        # behind the camera (+z)
    X = np.concatenate([kps, np.ones_like(kps[..., :1])], -1)
    h = np.einsum("grc,gjc->gjr", proj, X)
    uv = h[..., :2] / np.where(np.abs(h[..., 2:]) > 0, h[..., 2:], 1.)
    scale = rng.choice([1e-3, 5.0, 100.0, 3e3], size=(G, 24, 1))
    det = uv + rng.randn(G, 24, 2) * scale
    conf = rng.rand(G, 24, 1)
    conf[rng.rand(G, 24, 1) < 0.2] = 0.
    kp2d = np.concatenate([det, conf], -1)
    return torch.tensor(kps), torch.tensor(kp2d), torch.tensor(proj)


@pytest.mark.parametrize("sigma,coef", [(100., 1.0), (7.5, 0.3)])
def test_closed_form_gradient_equals_fp64_autograd(sigma, coef):
    kps, kp2d, proj = _scene()
    x = kps.clone().requires_grad_(True)
    loss, px = po.kp2d_loss(x, kp2d, proj, sigma, coef)
    loss.backward()
    c_loss, c_px, c_d = closed_form(kps, kp2d, proj, sigma, coef)
    assert abs(float(loss.detach()) - float(c_loss)) <= 1e-12 * abs(float(loss.detach()))
    assert abs(float(px) - float(c_px)) <= 1e-12 * abs(float(px))
    err = float((x.grad - c_d).norm() / x.grad.norm())
    assert err <= 1e-12, err
    # joints at and behind the camera, and joints with c = 0: exactly zero gradient, in both
    for g, j in ((1, 5), (2, 9)):
        assert torch.equal(x.grad[g, j], torch.zeros(3)) and torch.equal(c_d[g, j], torch.zeros(3))
    zero_c = kp2d[..., 2] == 0
    assert bool(zero_c.any()) and float(x.grad[zero_c].abs().max()) == 0.
    # every residual regime is present, and each joint's gradient matches on its own
    X = torch.cat([kps, torch.ones_like(kps[..., :1])], -1)
    h = torch.einsum("grc,gjc->gjr", proj, X)
    front = h[..., 2] > 1e-6
    r = (h[..., :2] / h[..., 2:] - kp2d[..., :2]).abs()[front]
    assert float(r.min()) < 1e-2 and float(r.max()) > 10 * sigma
    per = (x.grad - c_d).norm(dim=-1) <= 1e-10 * x.grad.norm(dim=-1)
    assert bool(per.all())


def test_pixel_error_counts_visible_confident_joints():
    kps, kp2d, proj = _scene(seed=1)
    _, px = po.kp2d_loss(kps, kp2d, proj, 100., 1.)
    X = torch.cat([kps, torch.ones_like(kps[..., :1])], -1)
    h = torch.einsum("grc,gjc->gjr", proj, X)
    keep = (h[..., 2] > 1e-6) & (kp2d[..., 2] > 0)
    r = (h[..., :2] / h[..., 2:] - kp2d[..., :2]).norm(dim=-1)
    assert abs(float(px) - float(r[keep].mean())) <= 1e-12 * float(px)
    # no confident joint in front of the camera: 0, and a loss of 0
    loss, px = po.kp2d_loss(kps, torch.cat([kp2d[..., :2], torch.zeros_like(kp2d[..., 2:])], -1), proj, 100., 1.)
    assert float(loss) == 0. and float(px) == 0.


@pytest.mark.parametrize("n_views", [3, 7])
def test_projection_matrix_matches_rays_in_box(n_views):
    H, W = 96, 80
    focal = 1.2 * H
    pose = syn.make_pose(3)
    for c2w in syn.bullet_time_cameras(syn.camera(), n_views):
        P = torch.tensor(render.projection_matrix(c2w, H, W, focal))
        ro, rd, idx = render.rays_in_box(H, W, focal, c2w, pose["cyl"], "cpu")
        assert ro.shape[0] > 100
        i, j = (idx % W).double(), (idx // W).double()
        for s in (0.5, 2.0, 3.7):
            X = ro.double() + s * rd.double()
            h = torch.cat([X, torch.ones_like(X[:, :1])], -1) @ P.T
            assert float(h[:, 2].min()) > 0
            err = torch.maximum((h[:, 0] / h[:, 2] - i).abs(), (h[:, 1] / h[:, 2] - j).abs())
            assert float(err.max()) <= 1e-3, float(err.max())
    # a batch of cameras gives the per-camera matrices
    c2ws = syn.bullet_time_cameras(syn.camera(), n_views)
    Ps = render.projection_matrix(c2ws, H, W, focal)
    assert Ps.shape == (n_views, 3, 4)
    assert np.array_equal(Ps[1], render.projection_matrix(c2ws[1], H, W, focal))


def test_package_flags():
    args = db.make_args("danbo_fast")
    assert args.kp2d_sigma == 100.0 and args.kp2d_coef == 0.0


@pytest.fixture
def no_device(monkeypatch):
    """Any use of the kernel library (which every device launch goes through) fails the test."""
    def boom():
        raise AssertionError("device work started before the refusal")
    monkeypatch.setattr(_lib, "load", boom)


def _batch(G=4, skip=3, **kw):
    b = {"kp_idx": torch.arange(G).repeat_interleave(skip), "N_uniques": G,
         "kp2d": torch.zeros(G, 24, 3), "kp2d_proj": torch.zeros(G, 3, 4)}
    b.update(kw)
    return {k: v for k, v in b.items() if v is not None}


BAD = [(dict(kp2d_proj=None), "both"), (dict(kp2d=None), "both"), (dict(kp2d=torch.zeros(4, 17, 3)), "24, 3"),
       (dict(kp2d=torch.zeros(3, 24, 3)), "24, 3"), (dict(kp2d_proj=torch.zeros(4, 4, 4)), "3, 4"),
       (dict(kp2d_proj=torch.zeros(4, 12)), "3, 4")]


def test_kp2d_batch():
    on = types.SimpleNamespace(kp2d_coef=1.0, kp2d_sigma=100.)
    assert training.kp2d_batch(on, {"kp_idx": torch.zeros(6), "N_uniques": 2}) is None          # no keys: off
    got = training.kp2d_batch(on, _batch())
    assert got is not None and got[0].shape == (4, 24, 3) and got[1].shape == (4, 3, 4)
    assert training.kp2d_batch(types.SimpleNamespace(kp2d_coef=0.0), _batch()) is None         # coef 0: off
    assert training.kp2d_batch(types.SimpleNamespace(), _batch()) is None                      # the default is off
    for kw, word in BAD:
        for args in (on, types.SimpleNamespace(kp2d_coef=0.0)):
            with pytest.raises(ValueError, match=re.escape(word)):
                training.kp2d_batch(args, _batch(**kw))
    with pytest.raises(ValueError, match="pose layer"):
        training.kp2d_batch(on, _batch(), pose_layer=False)
    with pytest.raises(ValueError, match="sigma"):
        training.kp2d_batch(types.SimpleNamespace(kp2d_coef=1.0, kp2d_sigma=0.), _batch())


def _popt():
    args = db.make_args("danbo_fast", no_reload=True, opt_pose=True, kp2d_coef=1.0, opt_pose_lrate=1e-2)
    attrs = {"rest_pose": FX["rest_pose"], "betas": np.zeros((1, 10), np.float32), "kp3d": FX["init_kps"],
             "bones": FX["init_bones"]}
    opt, popt = po.create_popt(args, attrs)
    return args, opt, popt


@pytest.mark.parametrize("kw,word", BAD)
def test_pose_fit_step_refuses_bad_kp2d_batches(no_device, kw, word):
    # PoseFitStep needs a CUDA FlatAdam to be built: the bare object stands in (a call that got past the checks would
    # fail on the missing attributes instead)
    step = training.PoseFitStep.__new__(training.PoseFitStep)
    step.args = _popt()[0]
    with pytest.raises(ValueError, match=re.escape(word)):
        step(_batch(**kw))


@pytest.mark.parametrize("kw,word", BAD)
def test_train_step_refuses_bad_kp2d_batches(no_device, kw, word):
    args, opt, popt = _popt()

    class Caster(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.network = torch.nn.Linear(2, 2)
    caster = Caster()
    step = training.TrainStep(caster, args, popt_kwargs=popt, pose_optimizer=opt)
    layer = {k: v.clone() for k, v in popt["popt_layer"].state_dict().items()}
    with pytest.raises(ValueError, match=re.escape(word)):
        step(_batch(**kw))
    assert all(p.grad is None for p in popt["popt_layer"].parameters())
    assert all(torch.equal(v, layer[k]) for k, v in popt["popt_layer"].state_dict().items())
    # and without a pose layer the term is refused too
    plain = training.TrainStep(caster, args)
    with pytest.raises(ValueError, match="pose layer"):
        plain(_batch())


def _header_args(name):
    text = open(os.path.join(ROOT, "include", "danbo_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    m = re.search(r"\bint\s+" + name + r"\s*\(([^)]*)\)", text)
    return [a.strip() for a in m.group(1).split(",")]


def test_pose_kp2d_signature_matches_the_header():
    args = _header_args("danbo_pose_kp2d")
    sig = _lib._SIGNATURES["danbo_pose_kp2d"]
    kinds = {"float": ctypes.c_float, "int": ctypes.c_int}
    assert len(sig) == len(args) == 9
    for a, t in zip(args, sig):
        if "*" in a:
            assert t is ctypes.c_void_p, (a, t)
        else:
            assert t is kinds[a.split()[-2]], (a, t)
    assert _lib.ABI_VERSION == 5
