"""Mesh extraction after the density lattice (SURVEY §8f rank 4): marching cubes on the device + PLY / PNG writers.

Mirrors what run_render.py:1266-1281 does with `mcubes.marching_cubes(sigma, threshold)` and `trimesh.Trimesh(...).export`
(both absent from this image, un-vendored and unpinned in the reference): the 256^3 lattice of `fwd_type='mesh'` stays on
the GPU and comes back as (vertices, triangles) instead of 67 MB of sigma going to the host for a CPU extraction.

Vertices are where `mcubes` puts them - on every lattice edge whose end points lie on opposite sides of the threshold,
linearly interpolated, in index coordinates - so the vertex SET is pinned by definition.  The triangulation table is
generated here (PyMCubes' own table is not available to compare with): per cube case the crossing points are joined
face by face, ambiguous faces by a rule that depends only on the face's own corner pattern (segments cut off the inside
corners), which makes neighbouring cubes agree on their shared face and the surface watertight; loops are fanned into
triangles.  Parity of the triangle lists with mcubes is therefore UNPINNED; what the tests pin is the vertex set, closed
orientable surfaces (every edge shared by two triangles, once per direction), and enclosed volumes.

Everything is torch ops on the lattice's device (no custom kernel: 16.6 M cells are a few passes of elementwise work,
two prefix sums and gathers); nothing here is on the measured hot path.
"""
import functools
import struct
import zlib

import numpy as np
import torch

# corner c of a cell sits at offset (c & 1, (c >> 1) & 1, (c >> 2) & 1); an edge joins two corners that differ in one bit
_CORNERS = np.array([[c & 1, (c >> 1) & 1, (c >> 2) & 1] for c in range(8)])
_EDGES = [(a, b) for a in range(8) for b in range(a + 1, 8) if bin(a ^ b).count("1") == 1]          # 12 edges
_EDGE_ID = {e: i for i, e in enumerate(_EDGES)}


def _face_cycles():
    """The 6 faces as cyclic corner lists, counter-clockwise seen from outside the cube."""
    faces = []
    for axis in range(3):
        u, v = (axis + 1) % 3, (axis + 2) % 3
        for side in (0, 1):
            cyc = []
            for du, dv in ((0, 0), (1, 0), (1, 1), (0, 1)):
                p = [0, 0, 0]
                p[axis], p[u], p[v] = side, du, dv
                cyc.append(p[0] + 2 * p[1] + 4 * p[2])
            if side == 0:                              # u x v points along +axis: reverse for the face at axis = 0
                cyc = cyc[::-1]
            faces.append(cyc)
    return faces


@functools.lru_cache(maxsize=1)
def tables():
    """-> (n_tri (256,) int64, tri (256, T, 3) int64 of cube-edge ids, -1 padded)."""
    faces = _face_cycles()
    all_tris = []
    for case in range(256):
        inside = [(case >> c) & 1 for c in range(8)]
        nxt = {}                                        # directed segments between crossed cube edges
        for cyc in faces:
            # Walk the face counter-clockwise (seen from outside).  Every maximal run of inside corners is entered
            # across one crossed edge and left across another; one segment cuts the run off, directed from the edge
            # where the walk leaves the run to the edge where it entered it - boundary piece + segment then circle the
            # run counter-clockwise, so the inside lies on the segment's left.  With four crossings (two single inside
            # corners on a diagonal) that gives one segment per corner, a choice that depends only on the face's own
            # corner pattern, so the two cubes sharing the face agree.
            crossed = []
            for i in range(4):
                a, b = cyc[i], cyc[(i + 1) % 4]
                if inside[a] != inside[b]:
                    crossed.append((i, _EDGE_ID[(min(a, b), max(a, b))], inside[a]))
            pos = {e: i for (i, e, _) in crossed}
            leave = [e for (_, e, was_in) in crossed if was_in]            # inside -> outside along the walk
            enter = [e for (_, e, was_in) in crossed if not was_in]        # outside -> inside
            for e_in in enter:
                e_out = min(leave, key=lambda e: (pos[e] - pos[e_in]) % 4)  # the run entered at e_in ends here
                assert e_out not in nxt
                nxt[e_out] = e_in
        # every crossed edge is a `leave` edge on one of its two faces and an `enter` edge on the other (their walks pass
        # it in opposite directions), so the segments chain into closed loops
        assert sorted(nxt.keys()) == sorted(nxt.values())
        loops, seen = [], set()
        for start in list(nxt):
            if start in seen:
                continue
            loop, e = [], start
            while e not in seen:
                seen.add(e)
                loop.append(e)
                e = nxt[e]
            loops.append(loop)
        # fan triangulation; the loops run with the inside on their left seen from outside the cube, i.e. clockwise seen
        # from the outside of the SURFACE, so the fan is reversed to make the normals point out of the inside
        tris = [(lp[0], lp[i + 1], lp[i]) for lp in loops for i in range(1, len(lp) - 1)]
        all_tris.append(tris)
    T = max(len(t) for t in all_tris)
    tri = -np.ones((256, T, 3), dtype=np.int64)
    for c, t in enumerate(all_tris):
        if t:
            tri[c, :len(t)] = np.array(t)
    n_tri = np.array([len(t) for t in all_tris], dtype=np.int64)
    return torch.from_numpy(n_tri), torch.from_numpy(tri)


def marching_cubes(volume, threshold):
    """volume (X,Y,Z) float tensor -> vertices (V,3) float32 in index coordinates, triangles (T,3) int64.
    A lattice point is inside when its value exceeds the threshold; triangle normals point out of the inside."""
    vol = volume.float()
    dev = vol.device
    X, Y, Z = vol.shape
    inside = vol > threshold
    # ---- vertices: one per lattice edge with a sign change, numbered axis by axis in row-major order
    vid, verts, base = [], [], 0
    for axis in range(3):
        lo = [slice(None)] * 3
        hi = [slice(None)] * 3
        lo[axis], hi[axis] = slice(0, -1), slice(1, None)
        cross = inside[tuple(lo)] != inside[tuple(hi)]
        ids = torch.cumsum(cross.reshape(-1).long(), 0).reshape(cross.shape) - 1 + base
        vid.append(torch.where(cross, ids, torch.full_like(ids, -1)))
        idx = torch.nonzero(cross)
        v0, v1 = vol[tuple(lo)][cross], vol[tuple(hi)][cross]
        t = (threshold - v0) / (v1 - v0)
        p = idx.float()
        p[:, axis] += t
        verts.append(p)
        base += idx.shape[0]
    vertices = torch.cat(verts, 0)
    # ---- cells
    case = torch.zeros(X - 1, Y - 1, Z - 1, dtype=torch.long, device=dev)
    for c, (dx, dy, dz) in enumerate(_CORNERS):
        case |= inside[dx:X - 1 + dx, dy:Y - 1 + dy, dz:Z - 1 + dz].long() << c
    n_tri, tri = (t.to(dev) for t in tables())
    cells = torch.nonzero((case > 0) & (case < 255))
    if cells.shape[0] == 0:
        return vertices, torch.zeros(0, 3, dtype=torch.long, device=dev)
    ccase = case[cells[:, 0], cells[:, 1], cells[:, 2]]
    # global vertex id of each of the 12 cube edges of every surface cell
    edge_vid = torch.empty(cells.shape[0], 12, dtype=torch.long, device=dev)
    for e, (a, b) in enumerate(_EDGES):
        axis = int(np.log2(a ^ b))
        off = _CORNERS[a]
        edge_vid[:, e] = vid[axis][cells[:, 0] + int(off[0]), cells[:, 1] + int(off[1]), cells[:, 2] + int(off[2])]
    t_edges = tri[ccase]                                                   # (C, T, 3) cube-edge ids, -1 padded
    keep = t_edges[..., 0] >= 0
    t_vid = torch.gather(edge_vid[:, None, :].expand(-1, t_edges.shape[1], -1), 2, t_edges.clamp(min=0))
    return vertices, t_vid[keep]


def mesh_volume(vertices, triangles):
    """Signed volume enclosed by a closed triangle mesh (divergence theorem), float64."""
    v = vertices.double()
    a, b, c = v[triangles[:, 0]], v[triangles[:, 1]], v[triangles[:, 2]]
    return float((a * torch.cross(b, c, dim=-1)).sum() / 6.0)


# RGB of the part of each of the 24 SMPL joints (skeleton.JOINT_NAMES order) in part-labelled meshes: 24 distinct
# colours of a common categorical palette, fixed so that a part has the same colour in every file.
PART_COLORS = np.array([
    [128, 128, 128], [230, 25, 75], [0, 130, 200], [170, 255, 195],        # pelvis, l/r hip, spine1
    [245, 130, 48], [70, 240, 240], [60, 180, 75], [255, 225, 25],         # l/r knee, spine2, l ankle
    [0, 0, 128], [210, 245, 60], [128, 0, 0], [145, 30, 180],              # r ankle, spine3, l/r foot
    [255, 255, 255], [250, 190, 212], [220, 190, 255], [64, 64, 64],       # neck, l/r collar, head
    [240, 50, 230], [0, 128, 128], [170, 110, 40], [255, 215, 180],        # l/r shoulder, l/r elbow
    [128, 128, 0], [0, 0, 255], [255, 250, 200], [0, 255, 0]], np.uint8)   # l/r wrist, l/r hand


# ---- writers (trimesh.export / imageio.imwrite of run_render.py:1280,1343-1346) -----------------------------------
def write_ply(path, vertices, triangles, normals=None, colors=None):
    """Binary little-endian PLY with float32 vertices and int32 triangle indices; with `normals` (V,3) each vertex also
    carries float32 nx ny nz (viewers then shade the mesh smoothly), with `colors` (V,3) uint8 red green blue.  Without
    either the bytes are those of a plain vertex + face file."""
    v = np.ascontiguousarray(torch.as_tensor(vertices).detach().cpu().numpy(), dtype="<f4")
    f = np.ascontiguousarray(torch.as_tensor(triangles).detach().cpu().numpy(), dtype="<i4")
    props = "property float x\nproperty float y\nproperty float z\n"
    if normals is not None:
        nrm = np.ascontiguousarray(torch.as_tensor(normals).detach().cpu().numpy(), dtype="<f4")
        if nrm.shape != v.shape:
            raise ValueError(f"write_ply: normals {nrm.shape} must match vertices {v.shape}")
        v = np.ascontiguousarray(np.concatenate([v.reshape(-1, 3), nrm.reshape(-1, 3)], 1))
        props += "property float nx\nproperty float ny\nproperty float nz\n"
    if colors is not None:
        col = torch.as_tensor(colors).detach().cpu().numpy()
        if col.dtype != np.uint8 or col.shape != (len(v), 3):
            raise ValueError(f"write_ply: colors must be uint8 ({len(v)}, 3), got {col.dtype} {col.shape}")
        rec_v = np.empty(len(v), dtype=[("p", "<f4", (v.shape[1],)), ("c", "u1", (3,))])
        rec_v["p"], rec_v["c"] = v, col
        v = rec_v
        props += "property uchar red\nproperty uchar green\nproperty uchar blue\n"
    head = ("ply\nformat binary_little_endian 1.0\n"
            f"element vertex {len(v)}\n{props}"
            f"element face {len(f)}\nproperty list uchar int vertex_indices\nend_header\n").encode("ascii")
    rec = np.empty(len(f), dtype=[("n", "u1"), ("idx", "<i4", (3,))])
    rec["n"], rec["idx"] = 3, f
    with open(path, "wb") as fh:
        fh.write(head)
        fh.write(v.tobytes())
        fh.write(rec.tobytes())


def read_ply(path, with_normals=False, with_colors=False):
    """Inverse of write_ply (for tests and round trips) -> (vertices, triangles), followed by the normals with
    `with_normals` and the uint8 colours with `with_colors` (a file without nx ny nz / red green blue raises)."""
    with open(path, "rb") as fh:
        data = fh.read()
    end = data.index(b"end_header\n") + len(b"end_header\n")
    head = data[:end].decode("ascii").split("\n")
    nv = int([l for l in head if l.startswith("element vertex")][0].split()[-1])
    nf = int([l for l in head if l.startswith("element face")][0].split()[-1])
    has_n = "property float nx" in head
    has_c = "property uchar red" in head
    if with_normals and not has_n:
        raise ValueError(f"{path} has no vertex normals")
    if with_colors and not has_c:
        raise ValueError(f"{path} has no vertex colours")
    width = 6 if has_n else 3
    vrec = np.frombuffer(data, dtype=[("p", "<f4", (width,)), ("c", "u1", (3 if has_c else 0,))], count=nv, offset=end)
    vn = vrec["p"]
    rec = np.frombuffer(data, dtype=[("n", "u1"), ("idx", "<i4", (3,))], count=nf, offset=end + vrec.nbytes)
    out = (vn[:, :3].copy(), rec["idx"].copy())
    if with_normals:
        out += (vn[:, 3:].copy(),)
    if with_colors:
        out += (vrec["c"].copy(),)
    return out


def write_png(path, img):
    """8-bit RGB / grey PNG from a (H,W,3) or (H,W) uint8 array (zlib only)."""
    a = np.ascontiguousarray(torch.as_tensor(img).detach().cpu().numpy() if torch.is_tensor(img) else np.asarray(img))
    if a.dtype != np.uint8:
        raise ValueError("write_png takes uint8 pixels")
    if a.ndim == 2:
        a = a[..., None]
    H, W, C = a.shape
    if C not in (1, 3):
        raise ValueError("1 or 3 channels")
    raw = np.concatenate([np.zeros((H, 1), np.uint8), a.reshape(H, W * C)], 1).tobytes()       # filter type 0 per row

    def chunk(tag, payload):
        return struct.pack(">I", len(payload)) + tag + payload + struct.pack(">I", zlib.crc32(tag + payload) & 0xffffffff)
    with open(path, "wb") as fh:
        fh.write(b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", W, H, 8, 2 if C == 3 else 0, 0, 0, 0))
                 + chunk(b"IDAT", zlib.compress(raw, 6)) + chunk(b"IEND", b""))


def write_video(path, frames, fps=14):
    """(N,H,W,3) uint8 RGB frames -> mp4 (imageio.mimwrite of run_render.py:1348), through OpenCV's writer."""
    try:
        import cv2
    except ImportError as e:                               # no silent skip: the caller asked for a file
        raise RuntimeError("write_video needs OpenCV (cv2), the only video encoder in this image") from e
    a = torch.as_tensor(frames).detach().cpu().numpy() if torch.is_tensor(frames) else np.asarray(frames)
    if a.dtype != np.uint8 or a.ndim != 4 or a.shape[-1] != 3:
        raise ValueError("write_video takes (N,H,W,3) uint8 frames")
    w = cv2.VideoWriter(path, cv2.VideoWriter_fourcc(*"mp4v"), float(fps), (a.shape[2], a.shape[1]))
    if not w.isOpened():
        raise RuntimeError(f"cannot open {path} for writing")
    for f in a:
        w.write(np.ascontiguousarray(f[..., ::-1]))        # OpenCV takes BGR
    w.release()


def save_renders(basedir, rgbs, accs, fps=14):
    """run_render.py:1332-1348 without the skeleton overlay: float images in [0,1] -> image/{i:05d}.png,
    acc/{i:05d}.png and render_rgb.mp4."""
    import os
    to8 = lambda x: (torch.as_tensor(x).detach().float().cpu().clamp(0, 1) * 255).to(torch.uint8).numpy()
    rgbs, accs = to8(rgbs), to8(accs)
    for d in ("image", "acc"):
        os.makedirs(os.path.join(basedir, d), exist_ok=True)
    for i, (rgb, acc) in enumerate(zip(rgbs, accs)):
        write_png(os.path.join(basedir, "image", f"{i:05d}.png"), rgb)
        write_png(os.path.join(basedir, "acc", f"{i:05d}.png"), acc.reshape(acc.shape[0], acc.shape[1]))
    write_video(os.path.join(basedir, "render_rgb.mp4"), rgbs, fps=fps)


@torch.no_grad()
def render_mesh(ray_caster, kps, skts, bones, radius=1.80, res=255, threshold=10., out_dir=None, preproc_kwargs=None,
                normals=False, parts=False):
    """run_render.py:1266-1281: per pose, the (res+1)^3 raw-density lattice (`fwd_type='mesh'`), relu, marching cubes at
    `threshold`, vertices scaled to `v / res - 0.5`; written as `meshes/{i:03d}.ply` when out_dir is given.
    -> list of (vertices, triangles).

    normals=True: -> list of (vertices, triangles, normals), the same vertices and triangles, with the unit outward
    normal -grad sigma / |grad sigma| of the field at every vertex (0 where the gradient is 0), from
    `render_pts_gradient` at the vertex's world position root + 2 radius v (the lattice is in xyz index order around
    the root joint, `render_mesh_density`); the PLY files carry them as nx ny nz.

    parts=True: each entry also ends with the (V,24) aggregation weights of the bones at those vertex positions
    (`render_pts_parts`), after the normals when both are asked for; the PLY files carry the PART_COLORS entry of each
    vertex's arg-max bone as red green blue."""
    import os
    caster = getattr(ray_caster, "module", ray_caster)          # the training handle wraps the caster
    if normals:
        if not hasattr(caster, "render_pts_gradient"):
            raise NotImplementedError("render_mesh(normals=True) needs a caster with render_pts_gradient")
        caster._refuse_normals("render_mesh(normals=True)")
    if parts:
        if not hasattr(caster, "render_pts_parts"):
            raise NotImplementedError("render_mesh(parts=True) needs a caster with render_pts_parts")
        caster._refuse_parts("render_mesh(parts=True)")
    out = []
    if out_dir is not None:
        os.makedirs(os.path.join(out_dir, "meshes"), exist_ok=True)
    for i in range(len(kps)):
        raw = ray_caster(kps=kps[i:i + 1], skts=skts[i:i + 1], bones=bones[i:i + 1], radius=radius, res=res,
                         render_kwargs=preproc_kwargs, fwd_type="mesh")
        v, t = marching_cubes(torch.relu(raw.reshape(res + 1, res + 1, res + 1)), threshold)
        v = v / res - 0.5
        n = p = col = None
        if normals or parts:
            root = torch.as_tensor(kps[i:i + 1]).reshape(1, -1, 3)[0, 0].to(v.device).float()
        if normals:
            _, g = caster.render_pts_gradient(root + 2. * radius * v, kps[i:i + 1], skts[i:i + 1], bones[i:i + 1])
            n = caster._unit_normals(g).to(v.device)
        if parts:
            _, p = caster.render_pts_parts(root + 2. * radius * v, kps[i:i + 1], skts[i:i + 1], bones[i:i + 1])
            p = p.to(v.device)
        if out_dir is not None:
            if parts:
                col = PART_COLORS[p.argmax(-1).cpu().numpy()]
            write_ply(os.path.join(out_dir, "meshes", f"{i:03d}.ply"), v, t, normals=n, colors=col)
        out.append((v, t) + tuple(x for x in (n, p) if x is not None))
    return out
