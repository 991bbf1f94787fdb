"""CPU checks of the surface-normal feature: the fp64 reference gradient (`normals_ref.density_at_points`, the oracle's
density lattice body at points, with the feature window differentiated) against central differences and against the translation identity that the GPU tests use
on the kernel, the PLY writer / reader with and without vertex normals, every refusal (raised before any device work),
and the ctypes signature of danbo_field_agg_bwd_pts against the header."""
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
from danbo_b200 import _lib, mesh, render           # noqa: E402
from danbo_b200 import skeleton as sk, synthetic as syn   # noqa: E402
from normals_ref import density_at_points   # noqa: E402
from util import align_A, load_fixture, params_for, pose_tensors   # noqa: E402

RES = 16


def _f64(P):
    return {k: v.double() for k, v in P.items()}


def _pose64():
    fx = load_fixture("render_fast")
    skts, bones, _ = pose_tensors(fx)
    return fx, skts.double(), bones.double(), fx["pose_kps"].double()


def _interior_points(skts, A, axis_scale, n, seed, margin=2e-3):
    """Random points near the joints that lie inside at least one bone box and at least `margin` (in box units) away
    from every box face and every interpolation knot of every bone - the places where sigma is not differentiable."""
    g = torch.Generator().manual_seed(seed)
    kps = skts.new_tensor(np.linalg.inv(skts[0].numpy())[:, :3, 3])            # joint positions (the skts' inverses)
    out = []
    while sum(len(o) for o in out) < n:
        c = kps[torch.randint(0, 24, (4 * n,), generator=g)]
        pts = c + 0.12 * torch.randn(4 * n, 3, generator=g, dtype=torch.float64)
        x = orc.world_to_bone(pts.reshape(-1, 1, 3), skts.expand(pts.shape[0], -1, -1, -1), A)[:, 0]
        x = x / axis_scale.abs()
        iy = ((x + 1.) * RES - 1.) / 2.
        frac = iy - torch.floor(iy)
        knot = torch.minimum(frac, 1. - frac) * 2. / RES                          # distance to a knot in x units
        face = (x.abs() - 1.).abs()
        ok = (knot.min(-1).values > margin).all(-1) & (face.min(-1).values > margin).all(-1)
        ok &= (x.abs() <= 1.).all(-1).any(-1)                                     # some bone sees it
        out.append(pts[ok])
    return torch.cat(out, 0)[:n]


def _relu_states(pts, skts, bones, A, P, agg_type):
    """(M, units) bool: which relu that depends on the point (aggregation net, MLP trunk) is on, per point."""
    import torch.nn.functional as F
    M = pts.shape[0]
    seen = []

    class _Recording:
        def __getattr__(self, k):
            return getattr(F, k)

        @staticmethod
        def relu(x):
            if x.shape[0] == M:                       # the graph net's relus (one pose) do not depend on the point
                seen.append((x.detach() > 0).reshape(M, -1))
            return F.relu(x)
    saved, orc.F = orc.F, _Recording()
    try:
        density_at_points(pts, skts, bones, A, P, agg_type, detach_window=False)
    finally:
        orc.F = saved
    return torch.cat(seen, -1)


def _smooth_on_stencil(pts, h, skts, bones, A, P, agg_type):
    """Points whose relus all keep their state on the central-difference stencil p +- h e_a: sigma is smooth there."""
    s0 = _relu_states(pts, skts, bones, A, P, agg_type)
    ok = torch.ones(pts.shape[0], dtype=torch.bool)
    for a in range(3):
        for sgn in (1., -1.):
            e = torch.zeros(3, dtype=pts.dtype)
            e[a] = sgn * h
            ok &= (_relu_states(pts + e, skts, bones, A, P, agg_type) == s0).all(-1)
    return ok


@pytest.mark.parametrize("agg_type", ["sigmoid", "softmax"])
def test_oracle_gradient_matches_central_differences(agg_type):
    """d sigma / d p by fp64 autograd of the oracle with the window in the graph equals central differences with h = 1e-6
    to 1e-6 relative, at points away from the kinks of sigma (box faces, interpolation knots, relus): this is the
    reference the GPU tests compare the kernels with."""
    fx, skts, bones, _ = _pose64()
    P, A = _f64(params_for(fx)), align_A().double()
    h = 1e-6
    pts = _interior_points(skts, A, P["graph_net.axis_scale"], 96, seed=1)
    pts = pts[_smooth_on_stencil(pts, h, skts, bones, A, P, agg_type)]          # no relu kink inside the stencil
    assert pts.shape[0] >= 64
    p = pts.clone().requires_grad_(True)
    sig = density_at_points(p, skts, bones, A, P, agg_type, detach_window=False)
    grad, = torch.autograd.grad(sig.sum(), p)
    fd = torch.zeros_like(pts)
    with torch.no_grad():
        for a in range(3):
            e = torch.zeros(3, dtype=torch.float64)
            e[a] = h
            fd[:, a] = (density_at_points(pts + e, skts, bones, A, P, agg_type, detach_window=False)
                        - density_at_points(pts - e, skts, bones, A, P, agg_type, detach_window=False)) / (2 * h)
    nrm = grad.norm(dim=-1)
    assert float(nrm.min()) > 0
    rel = (fd - grad).norm(dim=-1) / nrm
    assert float(rel.max()) <= 1e-6, float(rel.max())
    # the detached window (training's gradient) is a different quantity: the test above is not vacuous
    p2 = pts.clone().requires_grad_(True)
    g_det, = torch.autograd.grad(density_at_points(p2, skts, bones, A, P, agg_type).sum(), p2)
    assert float(((g_det - grad).norm(dim=-1) / nrm).max()) > 1e-3


@pytest.mark.parametrize("agg_type", ["sigmoid", "softmax"])
def test_oracle_translation_identity(agg_type):
    """Moving the body and the points by the same delta leaves sigma unchanged (t_k' = t_k - R_k delta), so
    sum_i grad_i = sum_k R_k^T d(sum sigma)/d t_k, with t_k the translation column of skts[k]."""
    fx, skts, bones, _ = _pose64()
    P, A = _f64(params_for(fx)), align_A().double()
    pts = _interior_points(skts, A, P["graph_net.axis_scale"], 64, seed=2)
    p = pts.clone().requires_grad_(True)
    s = skts.clone().requires_grad_(True)
    sig = density_at_points(p, s, bones, A, P, agg_type, detach_window=False)
    gp, gs = torch.autograd.grad(sig.sum(), (p, s))
    lhs = gp.sum(0)
    terms = torch.einsum("kij,ki->kj", skts[0, :, :3, :3], gs[0, :, :3, 3])
    rhs = terms.sum(0)
    scale = float(terms.abs().sum() + gp.abs().sum())
    assert float((lhs - rhs).abs().max()) <= 1e-10 * scale, (lhs, rhs)
    assert float(lhs.norm()) > 1e-6 * scale                      # not a sum of zeros


def test_density_at_points_is_the_grid_body():
    """density_at_points evaluates what the oracle's density_grid evaluates, lattice point by lattice point (fp32; the rows go through
    the CPU matrix products in another order, so equality is to rounding)."""
    fx = load_fixture("render_fast")
    skts, bones, _ = pose_tensors(fx)
    P, A = params_for(fx), align_A()
    kps = fx["pose_kps"][None]
    radius, res = 1.1, 4
    grid = orc.density_grid(kps, skts, bones, A, P, radius, res)
    t = np.linspace(-radius, radius, res + 1)
    # the returned lattice is in xyz index order: grid[i, j, k] is the point root + (t[i], t[j], t[k])
    I, Jj, Kk = np.meshgrid(t, t, t, indexing="ij")
    pts = torch.tensor(np.stack([I, Jj, Kk], -1).reshape(-1, 3).astype(np.float32)) + kps[0, 0]
    got = density_at_points(pts, skts, bones, A, P)
    torch.testing.assert_close(got.reshape(res + 1, res + 1, res + 1), grid, rtol=1e-6, atol=1e-5)


# ---------------------------------------------------------------------------------------------------- PLY
def _plain_ply_bytes(v, t):
    """The bytes of a vertex + face PLY as the writer produced them before it took normals."""
    head = ("ply\nformat binary_little_endian 1.0\n"
            f"element vertex {len(v)}\nproperty float x\nproperty float y\nproperty float z\n"
            f"element face {len(t)}\nproperty list uchar int vertex_indices\nend_header\n").encode("ascii")
    rec = np.empty(len(t), dtype=[("n", "u1"), ("idx", "<i4", (3,))])
    rec["n"], rec["idx"] = 3, t
    return head + np.ascontiguousarray(v, dtype="<f4").tobytes() + rec.tobytes()


def test_ply_round_trip_with_and_without_normals(tmp_path):
    g = torch.Generator().manual_seed(0)
    v = torch.randn(37, 3, generator=g)
    t = torch.randint(0, 37, (51, 3), generator=g)
    n = torch.nn.functional.normalize(torch.randn(37, 3, generator=g), dim=-1)
    plain, with_n = str(tmp_path / "a.ply"), str(tmp_path / "b.ply")
    mesh.write_ply(plain, v, t)
    assert open(plain, "rb").read() == _plain_ply_bytes(v.numpy(), t.numpy())
    mesh.write_ply(plain, v, t, normals=None)
    assert open(plain, "rb").read() == _plain_ply_bytes(v.numpy(), t.numpy())
    rv, rt = mesh.read_ply(plain)
    assert np.array_equal(rv, v.numpy()) and np.array_equal(rt, t.numpy())
    with pytest.raises(ValueError):
        mesh.read_ply(plain, with_normals=True)
    mesh.write_ply(with_n, v, t, normals=n)
    head = open(with_n, "rb").read().split(b"end_header\n")[0].decode()
    assert "property float nx\nproperty float ny\nproperty float nz\n" in head
    rv, rt, rn = mesh.read_ply(with_n, with_normals=True)
    assert np.array_equal(rv, v.numpy()) and np.array_equal(rt, t.numpy()) and np.array_equal(rn, n.numpy())
    rv, rt = mesh.read_ply(with_n)                                 # the two-value return stays as it was
    assert np.array_equal(rv, v.numpy()) and np.array_equal(rt, t.numpy())
    with pytest.raises(ValueError):
        mesh.write_ply(with_n, v, t, normals=n[:5])


# ---------------------------------------------------------------------------------------------------- refusals
def _cpu_caster(preset):
    args = db.make_args(preset, no_reload=True)
    attrs = {"skel_type": sk.SMPLSkeleton, "near": syn.NEAR, "far": syn.FAR, "n_views": 8, "rest_pose": syn.rest_pose()}
    _, kw_test, *_ = db.create_raycaster(args, attrs, device="cpu")
    return kw_test["ray_caster"], args


@pytest.fixture
def no_device(monkeypatch):
    """Any use of the kernel library (which every device launch goes through) fails the test."""
    def boom():
        raise AssertionError("device work started before the refusal")
    monkeypatch.setattr(_lib, "load", boom)


def _ray_kwargs(n=4):
    fx = load_fixture("render_fast")
    skts, bones, cyl = pose_tensors(fx)
    ex = lambda t: t.expand(n, *t.shape[1:])
    return fx["ray_batch"][:n], dict(N_samples=8, kp_batch=ex(fx["pose_kps"][None]), skts=ex(skts), cyls=ex(cyl),
                                     bones=ex(bones), cams=fx["cams"][:n], N_importance=4), fx


def test_want_normals_refusals(no_device):
    caster, _ = _cpu_caster("danbo_fast")
    rays, kw, _ = _ray_kwargs()
    caster.train()
    with pytest.raises(NotImplementedError, match="eval mode"):
        caster.render_rays(rays, want_normals=True, **kw)
    with pytest.raises(NotImplementedError, match="eval mode"):          # forward() in training keeps gradients on
        caster(rays, want_normals=True, **kw)
    caster.eval()
    with torch.enable_grad():
        with pytest.raises(NotImplementedError, match="without gradients"):
            caster.render_rays(rays, want_normals=True, **kw)
    with torch.no_grad():
        with pytest.raises(NotImplementedError, match="render_graphed"):
            caster.render_graphed(rays, want_normals=True, **kw)


def test_render_images_normals_refusals(no_device):
    caster, args = _cpu_caster("danbo_fast")
    caster.eval()
    pose = None                                      # never read: the refusals come first
    c2ws = [np.eye(4, dtype=np.float32)]
    for kw, word in (({"distributed": True}, "distributed"), ({"graphed": True}, "graphed")):
        with pytest.raises(NotImplementedError, match=word):
            render.render_images(caster, args, c2ws, [pose], 8, 8, normals=True, **kw)
    caster.train()
    with pytest.raises(NotImplementedError, match="eval mode"):
        render.render_images(caster, args, c2ws, [pose], 8, 8, normals=True)


def test_several_poses_refused(no_device):
    caster, _ = _cpu_caster("danbo_fast")
    fx = load_fixture("render_fast")
    skts, bones, _ = pose_tensors(fx)
    kps = fx["pose_kps"][None]
    with pytest.raises(NotImplementedError, match="one pose"):
        caster.render_pts_gradient(torch.zeros(5, 3), kps.expand(2, -1, -1), skts.expand(2, -1, -1, -1),
                                   bones.expand(2, -1, -1))


def test_anerf_caster_refuses_normals(no_device):
    caster, args = _cpu_caster("anerf_base")
    caster.eval()
    rays, kw, fx = _ray_kwargs()
    skts, bones, _ = pose_tensors(fx)
    kps = fx["pose_kps"][None]
    with pytest.raises(NotImplementedError, match="A-NeRF"):
        caster.render_pts_gradient(torch.zeros(5, 3), kps, skts, bones)
    with torch.no_grad():
        with pytest.raises(NotImplementedError, match="A-NeRF"):
            caster.render_rays(rays, want_normals=True, nerf_type="nerf", **kw)
    with pytest.raises(NotImplementedError, match="A-NeRF"):
        mesh.render_mesh(caster, kps, skts, bones, res=4, normals=True)
    with pytest.raises(NotImplementedError, match="A-NeRF"):
        render.render_images(caster, args, [np.eye(4, dtype=np.float32)], [None], 8, 8, normals=True)


# ---------------------------------------------------------------------------------------------------- ABI
def _decl(name):
    text = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "danbo_b200.h")).read(), flags=re.S)
    m = re.search(r"\bint\s+" + name + r"\s*\(([^;]*?)\)\s*;", text, flags=re.S)
    return [p.strip() for p in m.group(1).replace("\n", " ").split(",")]


def test_field_agg_bwd_pts_signature():
    """danbo_field_agg_bwd_pts takes danbo_field_agg_bwd's arguments with the accumulator array replaced by d_pts,
    d_vol and d_skts; the ctypes table matches the header; the ABI version is unchanged."""
    import ctypes
    new, old = _decl("danbo_field_agg_bwd_pts"), _decl("danbo_field_agg_bwd")
    i = old.index("float* const* grads")
    assert new[:i] == old[:i] and new[i + 3:] == old[i + 1:]
    assert new[i:i + 3] == ["float* d_pts", "float* d_vol", "float* d_skts"]
    sig = _lib._SIGNATURES["danbo_field_agg_bwd_pts"]
    assert len(sig) == len(new)
    for p, t in zip(new, sig):
        assert (t is ctypes.c_void_p) == ("*" in p), p
        if "*" not in p:
            assert t is ctypes.c_int, p
    assert _lib.ABI_VERSION == 5
