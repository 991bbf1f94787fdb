"""CPU checks of the body-part feature: an fp64 restatement of the part-weight definition against the field module's
`get_agg` (both aggregation types), the PLY writer / reader with vertex colours, `render.part_labels`, every refusal
(raised before any device work), and the ctypes signature of danbo_merge_composite_parts against the header."""
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
from danbo_b200 import _lib, mesh, render           # noqa: E402
from danbo_b200 import networks, skeleton as sk, synthetic as syn   # noqa: E402
from util import load_fixture, pose_tensors          # noqa: E402


# ---------------------------------------------------------------------------------------------------- definition
def _parts_fp64(logits, visible, agg_type):
    """p = get_agg(l, 1 - v) of one sample, written out element by element in fp64 (danbo.py:388-415)."""
    l, v = np.asarray(logits, np.float64), np.asarray(visible, np.float64)
    if agg_type == "sigmoid":
        return np.array([(1. / (1. + np.exp(-l[j])) * 1.002 - 0.001) * v[j] for j in range(24)])
    m = max(l)                                       # over all 24 logits, visible or not
    e = [np.exp(l[j] - m) * v[j] for j in range(24)]
    den = max(sum(e[j] + 1e-7 for j in range(24)), 1e-7)
    return np.array([e[j] / den for j in range(24)])


def _rows(seed=0):
    """Logit rows with their visibility: random rows; rows whose invisible bones hold the row's max (by a wide margin,
    so that the softmax denominator is dominated by the 24 eps terms); a row with one visible bone; a row no bone
    sees."""
    g = torch.Generator().manual_seed(seed)
    l = torch.randn(64, 24, generator=g, dtype=torch.float64) * 3.
    v = (torch.rand(64, 24, generator=g, dtype=torch.float64) < 0.2).double()
    v[:, 5] = 1.
    l[8:16] = torch.where(v[8:16] > 0, l[8:16], l[8:16] + 25.)        # invisible maxima
    l[16:20] = torch.where(v[16:20] > 0, l[16:20] - 40., l[16:20])
    v[20] = 0.
    v[20, 11] = 1.
    v[21] = 0.                                                        # no bone sees it
    return l, v


@pytest.mark.parametrize("agg_type", ["sigmoid", "softmax"])
def test_definition_is_get_agg(agg_type):
    net = networks.DanboField(agg_type=agg_type)
    l, v = _rows()
    got = net.get_agg(l, 1. - v)
    want = torch.from_numpy(np.stack([_parts_fp64(l[i], v[i], agg_type) for i in range(l.shape[0])]))
    torch.testing.assert_close(got, want, rtol=1e-13, atol=1e-15)
    assert torch.equal(got[21], torch.zeros(24, dtype=torch.float64))          # no visible bone: p = 0
    assert bool((got[v == 0] == 0).all())                                      # invisible bones: exactly 0
    if agg_type == "softmax":
        # the max over invisible logits matters: with the max over the visible ones only the eps terms would weigh less
        vis_max = torch.where(v > 0, l, torch.full_like(l, -1e30)).max(-1, keepdim=True).values
        e = torch.exp(l - vis_max) * v
        other = e / (e + 1e-7).sum(-1, keepdim=True)
        assert float((other[8:16] - got[8:16]).abs().max()) > 1e-3
        assert bool((got.sum(-1) <= 1.).all())
    else:
        assert bool((got >= -0.001).all())


# ---------------------------------------------------------------------------------------------------- PLY
def _plain_ply_bytes(v, t):
    head = ("ply\nformat binary_little_endian 1.0\n"
            f"element vertex {len(v)}\nproperty float x\nproperty float y\nproperty float z\n"
            f"element face {len(t)}\nproperty list uchar int vertex_indices\nend_header\n").encode("ascii")
    rec = np.empty(len(t), dtype=[("n", "u1"), ("idx", "<i4", (3,))])
    rec["n"], rec["idx"] = 3, t
    return head + np.ascontiguousarray(v, dtype="<f4").tobytes() + rec.tobytes()


def test_ply_colour_round_trip(tmp_path):
    g = torch.Generator().manual_seed(0)
    v = torch.randn(37, 3, generator=g)
    t = torch.randint(0, 37, (51, 3), generator=g)
    n = torch.nn.functional.normalize(torch.randn(37, 3, generator=g), dim=-1)
    c = mesh.PART_COLORS[torch.randint(0, 24, (37,), generator=g).numpy()]
    path = str(tmp_path / "m.ply")
    mesh.write_ply(path, v, t, colors=None)
    assert open(path, "rb").read() == _plain_ply_bytes(v.numpy(), t.numpy())
    with pytest.raises(ValueError):
        mesh.read_ply(path, with_colors=True)
    mesh.write_ply(path, v, t, colors=c)
    head = open(path, "rb").read().split(b"end_header\n")[0].decode()
    assert "property uchar red\nproperty uchar green\nproperty uchar blue\n" in head
    rv, rt, rc = mesh.read_ply(path, with_colors=True)
    assert np.array_equal(rv, v.numpy()) and np.array_equal(rt, t.numpy()) and np.array_equal(rc, c)
    rv, rt = mesh.read_ply(path)                                   # the two-value return stays as it was
    assert np.array_equal(rv, v.numpy()) and np.array_equal(rt, t.numpy())
    with pytest.raises(ValueError):
        mesh.read_ply(path, with_normals=True)
    mesh.write_ply(path, v, t, normals=n, colors=c)                 # normals and colours together
    rv, rt, rn, rc = mesh.read_ply(path, with_normals=True, with_colors=True)
    assert np.array_equal(rv, v.numpy()) and np.array_equal(rt, t.numpy())
    assert np.array_equal(rn, n.numpy()) and np.array_equal(rc, c)
    for bad in (c[:5], c.astype(np.float32)):
        with pytest.raises(ValueError):
            mesh.write_ply(path, v, t, colors=bad)


def test_part_colors_table():
    assert mesh.PART_COLORS.shape == (24, 3) and mesh.PART_COLORS.dtype == np.uint8
    assert len({tuple(c) for c in mesh.PART_COLORS}) == 24


# ---------------------------------------------------------------------------------------------------- labels
def test_part_labels():
    m = torch.zeros(2, 3, 24)
    m[0, 0, 4] = 0.9                                      # clear winner
    m[0, 1, 7], m[0, 1, 8] = 0.45, 0.3                    # below the threshold
    m[0, 2, 3], m[0, 2, 9] = 0.5, 0.5                     # tie at the threshold: the first bone, as argmax
    m[1, 0, 23] = 0.51
    m[1, 1, 0] = 1.0                                      # bone 0 is a label, not background
    lab = render.part_labels(m)
    assert lab.dtype == torch.int64 and lab.shape == (2, 3)
    assert lab.tolist() == [[4, -1, 3], [23, 0, -1]]
    assert render.part_labels(m, min_weight=0.4).tolist() == [[4, 7, 3], [23, 0, -1]]
    assert render.part_labels(m, min_weight=0.).tolist()[1][2] == 0       # an all-zero pixel at threshold 0


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


def test_want_parts_refusals(no_device):
    caster, _ = _cpu_caster("danbo_fast")
    rays, kw, _ = _ray_kwargs()
    caster.train()
    with pytest.raises(NotImplementedError, match="eval mode"):
        caster.render_rays(rays, want_parts=True, **kw)
    with pytest.raises(NotImplementedError, match="eval mode"):          # forward() in training keeps gradients on
        caster(rays, want_parts=True, **kw)
    caster.eval()
    with torch.enable_grad():
        with pytest.raises(NotImplementedError, match="without gradients"):
            caster.render_rays(rays, want_parts=True, **kw)
    with torch.no_grad():
        with pytest.raises(NotImplementedError, match="want_normals"):
            caster.render_rays(rays, want_parts=True, want_normals=True, **kw)
        with pytest.raises(NotImplementedError, match="render_graphed"):
            caster.render_graphed(rays, want_parts=True, **kw)


def test_render_images_parts_refusals(no_device):
    caster, args = _cpu_caster("danbo_fast")
    caster.eval()
    pose = None                                      # never read: the refusals come first
    c2ws = [np.eye(4, dtype=np.float32)]
    for kw, word in (({"distributed": True}, "distributed"), ({"graphed": True}, "graphed"),
                     ({"normals": True}, "normals")):
        with pytest.raises(NotImplementedError, match=word):
            render.render_images(caster, args, c2ws, [pose], 8, 8, parts=True, **kw)
    caster.train()
    with pytest.raises(NotImplementedError, match="eval mode"):
        render.render_images(caster, args, c2ws, [pose], 8, 8, parts=True)


def test_render_pts_parts_takes_one_pose(no_device):
    caster, _ = _cpu_caster("danbo_fast")
    fx = load_fixture("render_fast")
    skts, bones, _ = pose_tensors(fx)
    kps = fx["pose_kps"][None]
    with pytest.raises(NotImplementedError, match="one pose"):
        caster.render_pts_parts(torch.zeros(5, 3), kps.expand(2, -1, -1), skts.expand(2, -1, -1, -1),
                                bones.expand(2, -1, -1))


def test_anerf_caster_refuses_parts(no_device):
    caster, args = _cpu_caster("anerf_base")
    caster.eval()
    rays, kw, fx = _ray_kwargs()
    skts, bones, _ = pose_tensors(fx)
    kps = fx["pose_kps"][None]
    with pytest.raises(NotImplementedError, match="A-NeRF"):
        caster.render_pts_parts(torch.zeros(5, 3), kps, skts, bones)
    with torch.no_grad():
        with pytest.raises(NotImplementedError, match="A-NeRF"):
            caster.render_rays(rays, want_parts=True, nerf_type="nerf", **kw)
    with pytest.raises(NotImplementedError, match="A-NeRF"):
        mesh.render_mesh(caster, kps, skts, bones, res=4, parts=True)
    with pytest.raises(NotImplementedError, match="A-NeRF"):
        render.render_images(caster, args, [np.eye(4, dtype=np.float32)], [None], 8, 8, parts=True)


# ---------------------------------------------------------------------------------------------------- ABI
def _decl(name):
    text = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "danbo_b200.h")).read(), flags=re.S)
    m = re.search(r"\bint\s+" + name + r"\s*\(([^;]*?)\)\s*;", text, flags=re.S)
    return [" ".join(p.split()) for p in m.group(1).replace("\n", " ").split(",")]


def test_merge_composite_parts_signature():
    """danbo_merge_composite_parts takes danbo_merge_composite's arguments without the two train-mode outputs, with
    agg_mode and part_map before the stream; the ctypes table matches the header; the ABI version is unchanged."""
    import ctypes
    new, old = _decl("danbo_merge_composite_parts"), _decl("danbo_merge_composite")
    kept = [p for p in old if p not in ("float* confd_merged", "float* invalid_merged")]
    assert len(kept) == len(old) - 2
    assert new == kept[:-1] + ["int agg_mode", "float* part_map"] + kept[-1:]
    sig = _lib._SIGNATURES["danbo_merge_composite_parts"]
    assert len(sig) == len(new)
    for p, t in zip(new, sig):
        if "*" in p:
            assert t is ctypes.c_void_p, p
        else:
            assert t is (ctypes.c_float if p.startswith("float") else ctypes.c_int), p
    assert _lib.ABI_VERSION == 5
