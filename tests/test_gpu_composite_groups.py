"""The forward compositing kernels run several rays per warp (a group of lanes per ray).  These tests reach what the
fixture tests (small N, one layout) do not, at every sample count the launchers dispatch on: a ray count that is not a
multiple of the rays per warp, rays with all-empty masks next to active ones, train-mode random u with sorted and
unsorted rays side by side in one warp, tied fine samples, and u exactly on a cdf entry.

The reference is a plain-torch restatement: compositing in fp64 (weights, alpha, maps within fp32 rounding), and the
resampling and merge from the kernel's own weights in the kernel's fp32 / fp64 operation order, so that inds, z_samples,
z_all and the stable merge order must match exactly."""
import pytest
import torch

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(300, method="thread")]
DEV = "cuda"
J = 24
N_RAYS = 1003                       # odd: the last warp of every layout holds a partial set of rays
# (S, S_f): samples per lane 1..5 for the coarse launcher (S) and the merge launcher (S + S_f)
SHAPES = [(32, 16), (24, 8), (64, 16), (96, 48), (100, 20), (128, 0), (144, 0)]


def K():
    from danbo_b200 import kernels
    return kernels


def make_inputs(N, S, S_f, seed):
    g = torch.Generator().manual_seed(seed)
    rays = torch.randn(N, 8, generator=g)
    near = 1.0 + torch.rand(N, 1, generator=g)
    far = near + 2.0 + 2.0 * torch.rand(N, 1, generator=g)
    t = torch.sort(torch.rand(N, S, generator=g), -1).values
    z = (near + (far - near) * t).float()
    z[5, 3:6] = z[5, 3]                                         # repeated coarse z: zero-length bins and merge ties
    raw = torch.randn(N * S + N, 4, generator=g) * torch.tensor([2.0, 2.0, 2.0, 20.0]) + torch.tensor([0.0, 0.0, 0.0, 5.0])
    mask = torch.randint(1, 1 << 24, (N, S), generator=g, dtype=torch.int32)
    mask[torch.rand(N, S, generator=g) < 0.5] = 0
    empty = torch.zeros(N, dtype=torch.bool)
    empty[::7] = True                                           # all-empty rays between active ones
    mask[empty] = 0
    raw[N * S:][::2, 3] = -1.0                                  # half of those see sigma 0 everywhere: zero weights
    raw1 = torch.randn(N * max(S_f, 1), 4, generator=g) * torch.tensor([2.0, 2.0, 2.0, 20.0]) + 5.0
    mask1 = torch.randint(1, 1 << 24, (N, max(S_f, 1)), generator=g, dtype=torch.int32)
    mask1[torch.rand(N, max(S_f, 1), generator=g) < 0.5] = 0
    mask1[empty] = 0
    return dict(rays=rays, z=z, raw=raw, mask=mask, raw1=raw1[: N * S_f], mask1=mask1[:, :S_f].contiguous(), g=g)


def ref_composite(rays, z, raw, noise, inv_B):
    """raw2outputs in fp64: z (N,S), raw (N,S,4) with the empty entries already substituted."""
    z, raw = z.double(), raw.double()
    norm_d = rays[:, 3:6].double().norm(dim=-1, keepdim=True)
    dist = torch.cat([z[:, 1:] - z[:, :-1], torch.full_like(z[:, :1], 1e10)], -1) * norm_d
    rgb = torch.sigmoid(raw[..., :3]) * 1.002 - 0.001
    sg = raw[..., 3] * inv_B
    if noise is not None:
        sg = sg + noise.double()
    alpha = 1.0 - torch.exp(-torch.relu(sg) * dist)
    T = torch.cumprod(torch.cat([torch.ones_like(alpha[:, :1]), 1.0 - alpha + 1e-10], -1), -1)[:, :-1]
    w = alpha * T
    acc = w.sum(-1)
    disp = 1.0 / torch.clamp(((w * z).sum(-1)) / (acc + 1e-10), min=1e-10)
    disp[acc.abs() <= 1e-8] = 0.0
    return dict(weights=w, alpha=alpha, rgb_map=(w[..., None] * rgb).sum(-2), disp_map=disp, acc_map=acc.clamp(max=1.0))


def ref_cdf(w, smooth):
    """The kernel's cdf from its own fp32 weights: fp32 pdf terms, fp64 sums (exact for these terms), fp32 cdf."""
    if smooth:
        a, b = torch.maximum(w[:, :-2], w[:, 1:-1]), torch.maximum(w[:, 1:-1], w[:, 2:])
        dw = 0.5 * (a + b) + 0.01 + 1e-5
    else:
        dw = w[:, 1:-1] + 1e-5
    total = dw.double().sum(-1).float()
    pdf = dw / total[:, None]
    return torch.cat([torch.zeros_like(w[:, :1]), torch.cumsum(pdf.double(), -1).float()], -1)


def ref_resample(z, cdf, u):
    n_cdf = cdf.shape[1]
    ind = torch.searchsorted(cdf, u, right=True)
    below = torch.clamp(ind - 1, min=0)
    above = torch.clamp(ind, max=n_cdf - 1)
    bins = 0.5 * (z[:, 1:] + z[:, :-1])
    cb, ca = cdf.gather(1, below), cdf.gather(1, above)
    bb, ba = bins.gather(1, below), bins.gather(1, above)
    den = ca - cb
    den = torch.where(den < 1e-5, torch.ones_like(den), den)
    zs = bb + ((u - cb) / den) * (ba - bb)
    cat = torch.cat([z, zs], -1)
    order = torch.sort(cat, dim=-1, stable=True).indices
    return ind, zs, order, cat.gather(1, order)


def close(got, want, what, rtol=1e-5, atol=2e-6):
    got, want = got.cpu().double(), want.double()
    bad = ((got - want).abs() > atol + rtol * want.abs())
    assert not bool(bad.any()), f"{what}: {int(bad.sum())} elements off, max err {float((got - want).abs().max()):.3e}"


def check_composite(out, ref):
    for k in ("weights", "alpha", "rgb_map", "acc_map"):
        close(out[k], ref[k], k)
    # disparity = acc / depth, a ratio of two fp32 sums of up to 144 terms: 1e-4 relative; compared where acc > 1e-3,
    # since a near-transparent ray amplifies the rounding further
    lit = ref["acc_map"] > 1e-3
    close(out["disp_map"].cpu()[lit], ref["disp_map"][lit], "disp_map", rtol=1e-4)
    assert bool((out["disp_map"].cpu()[ref["acc_map"] == 0] == 0).all()), "disp_map of an empty ray"


@pytest.mark.parametrize("S,S_f", SHAPES)
@pytest.mark.parametrize("mode", ["eval", "train"])
def test_grouped_composite_resample_merge(S, S_f, mode):
    N = N_RAYS
    x = make_inputs(N, S, S_f, seed=S * 1000 + S_f + (mode == "train"))
    g = x["g"]
    train = mode == "train"
    smooth = not train
    noise0 = torch.randn(N, S, generator=g) if train else None
    inv_B = 0.5
    d = {k: x[k].to(DEV) for k in ("rays", "z", "raw", "mask", "raw1", "mask1")}
    u = None
    if train and S_f > 0:
        u = torch.rand(N, S_f, generator=g)
        u[::2] = torch.sort(u[::2], -1).values                 # sorted and unsorted rays side by side in every warp
        u[3::8, 1] = u[3::8, 0]                                 # tied fine samples: the merge keeps index order
    kw = dict(noise=noise0.to(DEV) if train else None, inv_B=inv_B, want_inds=True, smooth=smooth)
    out = K().composite_resample(d["rays"], S, S_f, d["raw"], d["mask"], d["z"],
                                 u_rand=u.to(DEV) if u is not None else None, **kw)
    torch.cuda.synchronize()
    raw0 = torch.where((x["mask"] != 0)[..., None], x["raw"][: N * S].view(N, S, 4), x["raw"][N * S:][:, None])
    ref = ref_composite(x["rays"], x["z"], raw0, noise0, inv_B)
    check_composite(out, ref)
    if not train:
        assert bool((out["weights"][::7][::2].cpu() == 0).all()), "an all-empty ray with sigma 0 has zero weights"
    if S_f == 0:
        return
    w = out["weights"].cpu()
    cdf = ref_cdf(w, smooth)
    if train:                                                   # u exactly on cdf entries, then render again
        rows = torch.arange(1, N, 4)
        k = torch.randint(0, S - 1, (rows.numel(), S_f), generator=g)
        u[rows] = cdf[rows].gather(1, k)
        u[rows[::2]] = torch.sort(u[rows[::2]], -1).values
        out = K().composite_resample(d["rays"], S, S_f, d["raw"], d["mask"], d["z"], u_rand=u.to(DEV), **kw)
        torch.cuda.synchronize()
        assert torch.equal(out["weights"].cpu(), w), "weights must not depend on u"
    else:
        u = torch.linspace(0., 1., S_f)[None].expand(N, -1).contiguous()
    ind, zs, order, z_all = ref_resample(x["z"], cdf, u)
    assert torch.equal(out["inds"].cpu().long(), ind), "inds"
    assert torch.equal(out["z_samples"].cpu(), zs), "z_samples"
    assert torch.equal(out["order"].cpu().long(), order), "merge order"
    assert torch.equal(out["z_all"].cpu(), z_all), "z_all"
    # ---- merge_composite on that order, with the train-mode outputs
    St = S + S_f
    noise1 = torch.randn(N, St, generator=g) if train else None
    confd0, confd1 = torch.randn(N * S, J, generator=g), torch.randn(N * S_f, J, generator=g)
    m = K().merge_composite(d["rays"], S, S_f, d["raw"], d["mask"], d["raw1"], d["mask1"], out["z_all"], out["order"],
                            noise=noise1.to(DEV) if train else None, inv_B=inv_B, want_raw=True,
                            confd0=confd0.to(DEV), confd1=confd1.to(DEV), want_invalid=True)
    torch.cuda.synchronize()
    raw1 = torch.where((x["mask1"] != 0)[..., None], x["raw1"].view(N, S_f, 4), x["raw"][N * S:][:, None])
    cat_raw = torch.cat([raw0, raw1], 1)
    merged = cat_raw.gather(1, order[..., None].expand(-1, -1, 4))
    assert torch.equal(m["raw"].cpu(), merged), "raw_merged"
    check_composite(m, ref_composite(x["rays"], z_all, merged, noise1, inv_B))
    bits = torch.cat([x["mask"], x["mask1"]], 1).gather(1, order).long()
    vis = ((bits[..., None] >> torch.arange(J)) & 1).bool()
    cat_conf = torch.cat([confd0.view(N, S, J), confd1.view(N, S_f, J)], 1)
    conf = torch.where(vis, cat_conf.gather(1, order[..., None].expand(-1, -1, J)), torch.zeros(()))
    assert torch.equal(m["part_invalid"].cpu(), (~vis).float()), "part_invalid"
    assert torch.equal(m["confd"].cpu(), conf), "confd"


def test_coarse_weights_row_is_optional():
    """want_weights=False skips the (n, S) weight row; every other output is unchanged."""
    N, S, S_f = N_RAYS, 32, 16
    x = make_inputs(N, S, S_f, seed=7)
    d = {k: x[k].to(DEV) for k in ("rays", "z", "raw", "mask")}
    a = K().composite_resample(d["rays"], S, S_f, d["raw"], d["mask"], d["z"])
    b = K().composite_resample(d["rays"], S, S_f, d["raw"], d["mask"], d["z"], want_weights=False)
    assert "weights" not in b and set(a) == set(b) | {"weights"}
    for k in b:
        assert torch.equal(a[k], b[k]), k
