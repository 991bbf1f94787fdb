"""Callers of the hot path (SURVEY §8f rank 1, §8e): image rendering and the density lattice, single- or multi-GPU.

Mirrors what the reference does around `ray_caster(...)`:
  * render()/batchify_rays  core/trainer.py:75-162   -> `render`
  * render_path             run_nerf.py:29-147       -> `render_images` (ray generation, cylinder box culling and image
                                                        assembly on the GPU instead of per-image numpy + .cpu() round trips)
  * render_mesh             run_render.py:1266-1281  -> `density_grid` (z-slabs of the lattice per rank + all-gather)
Work is sharded without any data-path collective: whole images (or lattice slabs) per rank, one all-gather at the end.
"""
import numpy as np
import torch
import torch.distributed as dist

from . import parallel
from . import synthetic as syn


def batchify_rays(rays_flat, chunk=1024 * 64, ray_caster=None, **kwargs):
    """trainer.py:75-90: slice every tensor kwarg per chunk, concatenate the returned dicts."""
    all_ret = {}
    for i in range(0, rays_flat.shape[0], chunk):
        kw = {k: (v[i:i + chunk] if torch.is_tensor(v) else v) for k, v in kwargs.items()}
        ret = ray_caster(rays_flat[i:i + chunk], **kw)
        for k, v in ret.items():
            all_ret.setdefault(k, []).append(v)
    return {k: torch.cat(v, 0) for k, v in all_ret.items()}


def render(H, W, focal, chunk=1024 * 64, rays=None, near=0., far=1., use_viewdirs=False, single_call=True, **kwargs):
    """trainer.py:96-162.  `rays` = (rays_o, rays_d).  With single_call (default) the whole batch goes to the caster in
    one call with nanmean_chunk=chunk, which reproduces the reference's per-chunk near/far fill (F8) without the
    per-chunk Python loop; single_call=False is the reference's loop."""
    rays_o, rays_d = rays
    sh = rays_d.shape
    rays_o = torch.reshape(rays_o, [-1, 3]).float()
    rays_d = torch.reshape(rays_d, [-1, 3]).float()
    parts = [rays_o, rays_d, near * torch.ones_like(rays_d[..., :1]), far * torch.ones_like(rays_d[..., :1])]
    if use_viewdirs:
        parts.append(rays_d / torch.norm(rays_d, dim=-1, keepdim=True))
    ray_batch = torch.cat(parts, -1)
    caster = kwargs.pop("ray_caster")
    if single_call:
        all_ret = caster(ray_batch, nanmean_chunk=chunk, **kwargs)
    else:
        all_ret = batchify_rays(ray_batch, chunk, ray_caster=caster, **kwargs)
    for k in all_ret:
        if all_ret[k].dim() < 4:
            all_ret[k] = torch.reshape(all_ret[k], list(sh[:-1]) + list(all_ret[k].shape[1:]))
    return all_ret


def rays_in_box(H, W, focal, c2w, cyl, device, c2w_dev=None):
    """Pinhole rays of the pixels inside the image box of a bounding cylinder, generated on the device
    (ray_utils.py:7-29,84-138; skeleton_utils.py:633-720).  -> rays_o, rays_d (n,3), flat pixel index (n).
    c2w / cyl: host arrays (the pixel box is a host-side computation over 100 projected points); c2w_dev: the same
    camera already on the device (saves the per-image upload)."""
    c2w_np = np.asarray(c2w, dtype=np.float32)
    tl, br = syn.cylinder_image_box(np.asarray(cyl, dtype=np.float32), H, W, float(focal), c2w_np)
    ys = torch.arange(int(tl[1]), int(br[1]), device=device, dtype=torch.float32)
    xs = torch.arange(int(tl[0]), int(br[0]), device=device, dtype=torch.float32)
    j, i = torch.meshgrid(ys, xs, indexing="ij")
    dirs = torch.stack([(i - W * 0.5) / focal, -(j - H * 0.5) / focal, -torch.ones_like(i)], -1).reshape(-1, 3)
    c2w_t = torch.as_tensor(c2w_np, device=device) if c2w_dev is None else c2w_dev
    rays_d = torch.sum(dirs[:, None, :] * c2w_t[:3, :3], -1)
    rays_o = c2w_t[:3, -1].expand(rays_d.shape)
    idx = (j * W + i).reshape(-1).long()
    return rays_o, rays_d, idx


def projection_matrix(c2w, H, W, focal):
    """The 3x4 projection P of the pinhole cameras of `rays_in_box` and `synthetic` (looking down -z; pixel (i, j) on
    the direction ((i - W/2)/f, -(j - H/2)/f, -1) in the camera frame): a world point X projects to pixel
    (P0 [X,1], P1 [X,1]) / P2 [X,1].  P = [[f, 0, -W/2], [0, -f, -H/2], [0, 0, -1]] [R^T | -R^T t] with c2w = [R | t].
    c2w: (4,4) or (3,4), or a batch (..., 3|4, 4), numpy or torch.  -> float64 numpy (..., 3, 4)."""
    c2w = np.asarray(c2w.detach().cpu() if torch.is_tensor(c2w) else c2w, dtype=np.float64)[..., :3, :4]
    R, t = c2w[..., :3, :3], c2w[..., :3, 3:]
    Rt = np.swapaxes(R, -1, -2)
    K = np.array([[focal, 0., -W * 0.5], [0., -focal, -H * 0.5], [0., 0., -1.]], dtype=np.float64)
    return K @ np.concatenate([Rt, -Rt @ t], -1)


@torch.no_grad()
def render_images(caster, args, c2ws, poses, H, W, focal=None, cam_idx=0, white_bkgd=True, near=syn.NEAR, far=syn.FAR,
                  graphed=False, distributed=False, normals=False, parts=False):
    """Render one image per (camera, pose) pair.  poses: list of dicts from synthetic.make_pose (kps, skts, bones, cyl);
    image k uses c2ws[k] and poses[k % len(poses)], like render_path.  With distributed=True images are dealt round
    robin to the ranks and the finished images all-gathered: every rank returns all images (n, H, W, 3) float32.
    normals=True (single process, not graphed): -> (images, normal_images), the second (n, H, W, 3) float32 world-frame
    normal maps (`render_rays(want_normals=True)`), 0 on the background.
    parts=True (single process, not graphed, not with normals): -> (images, part_maps), the second (n, H, W, 24) float32
    body-part maps (`render_rays(want_parts=True)`: the composited aggregation weight of every bone), 0 on the
    background; `part_labels` turns them into a segmentation."""
    if parts:
        if graphed:
            raise NotImplementedError("render_images(parts=True) with graphed=True: part maps are not captured")
        if distributed:
            raise NotImplementedError("render_images(parts=True) with distributed=True is not implemented")
        if normals:
            raise NotImplementedError("render_images(parts=True) together with normals=True is not implemented: make "
                                      "two calls")
        if hasattr(caster, "_refuse_parts"):
            caster._refuse_parts("render_images(parts=True)")
        if caster.training:
            raise NotImplementedError("render_images(parts=True) is for eval mode (caster.eval())")
    if normals:
        if graphed:
            raise NotImplementedError("render_images(normals=True) with graphed=True: normals are not captured")
        if distributed:
            raise NotImplementedError("render_images(normals=True) with distributed=True is not implemented")
        if hasattr(caster, "_refuse_normals"):
            caster._refuse_normals("render_images(normals=True)")
        if caster.training:
            raise NotImplementedError("render_images(normals=True) is for eval mode (caster.eval())")
    dev = next(caster.parameters()).device
    focal = 1.2 * H if focal is None else focal
    rank, world = parallel.world() if distributed else (0, 1)
    mine = list(range(rank, len(c2ws), world))
    out = torch.ones(len(mine), H * W, 3, device=dev) if white_bkgd else torch.zeros(len(mine), H * W, 3, device=dev)
    nmaps = torch.zeros(len(mine), H * W, 3, device=dev) if normals else None
    pmaps = torch.zeros(len(mine), H * W, 24, device=dev) if parts else None
    call = caster.render_graphed if graphed else caster
    # every pose table and camera of this rank's images goes to the device ONCE (5 copies), not per image: a pageable
    # host-to-device copy is synchronous, and one per tensor per image kept the GPU idle for half of each image
    mine_poses = sorted({k % len(poses) for k in mine})
    slot_of = {p: i for i, p in enumerate(mine_poses)}
    tab = {name: torch.as_tensor(np.stack([np.asarray(poses[p][name], dtype=np.float32) for p in mine_poses])).to(dev)
           for name in ("kps", "skts", "bones", "cyl")} if mine else {}
    c2w_dev = torch.as_tensor(np.stack([np.asarray(c2ws[k], dtype=np.float32) for k in mine])).to(dev) if mine else None
    for slot, k in enumerate(mine):
        pose = poses[k % len(poses)]
        ps = slot_of[k % len(poses)]
        ro, rd, idx = rays_in_box(H, W, focal, c2ws[k], pose["cyl"], dev, c2w_dev=c2w_dev[slot])
        n = ro.shape[0]
        ones = torch.ones(n, 1, device=dev)
        ray_batch = torch.cat([ro, rd, near * ones, far * ones, rd / torch.norm(rd, dim=-1, keepdim=True)], -1)
        ret = call(ray_batch, N_samples=args.N_samples, kp_batch=tab["kps"][ps:ps + 1].expand(n, -1, -1),
                   skts=tab["skts"][ps:ps + 1].expand(n, -1, -1, -1), cyls=tab["cyl"][ps:ps + 1].expand(n, -1),
                   bones=tab["bones"][ps:ps + 1].expand(n, -1, -1),
                   cams=torch.full((n, 1), cam_idx, dtype=torch.long, device=dev), N_uniques=1, perturb=False,
                   N_importance=args.N_importance, raw_noise_std=0., nanmean_chunk=args.chunk,
                   **({"want_normals": True} if normals else {}), **({"want_parts": True} if parts else {}))
        bg = 1.0 if white_bkgd else 0.0
        out[slot, idx] = ret["rgb_map"] + (1. - ret["acc_map"])[:, None] * bg         # run_nerf.py:103-133
        if normals:
            nmaps[slot, idx] = ret["normal_map"]
        if parts:
            pmaps[slot, idx] = ret["part_map"]
    out = out.reshape(len(mine), H, W, 3)
    if normals:
        return out, nmaps.reshape(len(mine), H, W, 3)
    if parts:
        return out, pmaps.reshape(len(mine), H, W, 24)
    if world == 1:
        return out
    counts = [len(range(r, len(c2ws), world)) for r in range(world)]
    gathered = parallel.allgather_rows(out, counts)
    # undo the round-robin deal
    order = [k for r in range(world) for k in range(r, len(c2ws), world)]
    inv = torch.empty(len(order), dtype=torch.long, device=dev)
    inv[torch.as_tensor(order, device=dev)] = torch.arange(len(order), device=dev)
    return gathered[inv]


def part_labels(part_maps, min_weight=0.5):
    """Body-part segmentation of part maps (..., 24) -> int64 (...): the bone of the largest weight, -1 where that
    weight is below `min_weight` (background, and pixels no part explains clearly)."""
    w, j = part_maps.max(-1)
    return torch.where(w >= min_weight, j, torch.full_like(j, -1))


@torch.no_grad()
def density_grid(caster, kps, skts, bones, radius=1.8, res=255, distributed=False, slab_points=1 << 22):
    """(res+1)^3 raw sigma lattice (raycasters.py:421-437), x/y swapped like the reference.  The lattice is cut into
    slabs along its first axis; with distributed=True the slabs are split across ranks and all-gathered."""
    dev = next(caster.parameters()).device
    t = np.linspace(-radius, radius, res + 1)
    R = res + 1
    rank, world = parallel.world() if distributed else (0, 1)
    lo, hi = parallel.shard_range(R, rank, world, align=1)
    tt = torch.as_tensor(t, device=dev)
    root = torch.as_tensor(kps, device=dev).reshape(-1, 24, 3)[0, 0].float()
    # np.meshgrid(t, t, t) default 'xy' indexing: grid[a, b, c] = (t[b], t[a], t[c])
    rows_per_call = max(1, slab_points // (R * R))
    parts = []
    for a0 in range(lo, hi, rows_per_call):
        a1 = min(hi, a0 + rows_per_call)
        A, B, C = torch.meshgrid(tt[a0:a1], tt, tt, indexing="ij")
        pts = torch.stack([B, A, C], -1).reshape(-1, 3).float() + root
        sig = caster.render_pts_density(pts.reshape(-1, 1, 3), kps, skts, bones)
        parts.append(sig.reshape(a1 - a0, R, R))
    local = torch.cat(parts, 0) if parts else torch.zeros(0, R, R, device=dev)
    if world > 1:
        sizes = [b - a for a, b in (parallel.shard_range(R, r, world, align=1) for r in range(world))]
        local = parallel.allgather_rows(local.contiguous(), sizes)
    return local.transpose(1, 0)
