"""The layer-local fp64 oracle and the error predicates of tests/test_gpu_mlp_tiles.py, proven on the CPU.

1. Chained, the layer-local references ARE the network: with straight-through bf16 rounding they reproduce fp64 autograd
   of util.mlp_bf16_reference (delta planes, dX, dW, db) to 1e-12.
2. The predicates accept what a correct kernel writes: bf16_rn(r), either neighbour of an exact tie, fp32 sums.
3. The predicates reject each structural error a tiled kernel can make: a dropped 64-row block of a K = 40 000
   reduction, rows shifted by one tile, swapped 128-column output halves, the relu gate of the neighbouring plane,
   a missing sigma-head term, and a consistent 1-ulp bias on 5 % of the entries."""
import pytest
import torch

from util import (BIAS_ITEMS, MIN_NEAREST_BF16, MLP_LAYERS, WGRAD_ITEMS, bf16_rn, check_bf16, check_fp32,
                  check_reduction, delta9_ref, dgrad_plane_ref, dx_ref, fwd_plane_ref, head_bwd_refs, mlp_bf16_reference,
                  mlp_bf16_weights, nearest_bf16_fraction, random_mlp_params, wgrad_refs)

N = 300          # rows: more than two 128-row tiles


def chain(P, x, rb, g_out):
    """The layer-local references composed: forward planes rounded to bf16 as the kernels store them, delta planes
    left unrounded (autograd does not round them) -> (acts, g, D, dX, wgrad, bias grads)."""
    W = mlp_bf16_weights(P)
    acts = []
    for L in range(9):
        acts.append(bf16_rn(fwd_plane_ref(L, x, acts, W)[0]))
    g = fwd_plane_ref(9, x, acts, W, rb)[0]
    D = [delta9_ref(g_out, g, W)[0]]
    for p in range(1, 10):
        D.append(dgrad_plane_ref(p, D, acts, g_out, W)[0])
    dw, db = wgrad_refs(D, acts, x)
    return acts, g, D, dx_ref(D, W)[0], dw, db


@pytest.fixture(scope="module")
def net():
    torch.manual_seed(0)
    P = {k: v.double() for k, v in random_mlp_params(0).items()}
    x = bf16_rn(torch.randn(N, 195, dtype=torch.float64) * 0.7)
    rb = torch.randn(N, 128, dtype=torch.float64) * 0.3
    g_out = torch.randn(N, 4, dtype=torch.float64)
    return P, x, rb, g_out, chain(P, x, rb, g_out)


def test_chain_reproduces_autograd(net):
    """Autograd of the bf16-emulating restatement (straight-through rounding, fp64) with per-row bias leaves, whose
    gradients are the delta planes: every delta plane, dX, dW and db of the chained oracle within 1e-12."""
    P, x, rb, g_out, (acts, g, D, dX, dw, db) = net
    ste = lambda t: t + (bf16_rn(t) - t).detach()
    Q = {k: v.clone().requires_grad_(True) for k, v in P.items()}
    rows = {n: Q[n + ".bias"].detach().expand(N, -1).clone().requires_grad_(True) for n in MLP_LAYERS[:9]}
    Qr = dict(Q, **{n + ".bias": rows[n] for n in rows})
    xl, rbl = x.clone().requires_grad_(True), rb.clone().requires_grad_(True)
    out = mlp_bf16_reference(xl, rbl, Qr, bf=ste)
    (out * g_out).sum().backward()

    def close(name, got, want):
        err = float((got - want).abs().max())
        scale = float(want.abs().max())
        assert scale > 0 and err <= 1e-12 * scale, (name, err, scale)

    close("delta plane 0", D[0], rbl.grad)
    for p in range(1, 10):
        close(f"delta plane {p}", D[p], rows[MLP_LAYERS[9 - p]].grad)
    close("dX", dX, xl.grad)
    for name, cols, (r, _, _) in dw:
        close(f"{name}[:, {cols}]", r, Q[name].grad[:, cols])
    for name, (r, _, _) in db:
        close(name, r, rows[name[:-len(".bias")]].grad.sum(0))
    assert [n for n, _, _, _ in WGRAD_ITEMS].count("pts_linears.5.weight") == 2 and len(BIAS_ITEMS) == 9


def test_predicates_accept_correct_rounding(net):
    P, x, rb, g_out, (acts, g, D, dX, dw, db) = net
    W = mlp_bf16_weights(P)
    for L in range(9):
        ref = fwd_plane_ref(L, x, acts, W)
        check_bf16(f"a{L}", bf16_rn(ref[0]), ref)
    for p in range(1, 10):
        ref = dgrad_plane_ref(p, [bf16_rn(d) for d in D], acts, g_out, W)
        check_bf16(f"delta {p}", bf16_rn(ref[0]), ref)
    ref = dx_ref([bf16_rn(d) for d in D], W)
    check_fp32("dX", ref[0].float(), ref)
    for name, cols, ref in dw:
        pre = torch.randn_like(ref[0]).float()
        check_reduction(name, (pre.double() + ref[0]).float(), ref, pre)
    hb = head_bwd_refs(g_out, bf16_rn(g), acts[7], torch.arange(N) % 7, 7, W)
    for name, ref in hb.items():
        pre = torch.randn_like(ref[0]).float()
        check_reduction(name, (pre.double() + ref[0]).float(), ref, pre)


def test_predicates_accept_either_neighbour_of_a_tie():
    lo = bf16_rn(torch.randn(4096, dtype=torch.float64) * 3)
    hi = (lo.to(torch.bfloat16).view(torch.int16) + 1).view(torch.bfloat16).double()     # next bf16 away from zero
    r = (lo + hi) / 2                                                                     # exact ties
    assert torch.equal(bf16_rn(r).abs() >= lo.abs(), torch.ones_like(lo, dtype=torch.bool))
    for got in (lo, hi, torch.where(torch.arange(4096) % 2 == 0, lo, hi)):
        check_bf16("tie", got, (r, r.abs(), 1))
        assert nearest_bf16_fraction(got, r) == 1.0


def test_rejects_dropped_block_of_a_long_reduction():
    """K = 40 000 rows, one 64-row block missing: inside the per-entry bound (it grows with K), caught by the norm."""
    g = torch.Generator().manual_seed(3)
    d = bf16_rn(torch.randn(40_000, 16, generator=g, dtype=torch.float64))
    a = bf16_rn(torch.randn(40_000, 32, generator=g, dtype=torch.float64).relu())
    ref = (d.t() @ a, d.t().abs() @ a.abs(), 40_000)
    pre = torch.randn(16, 32, generator=g)
    check_reduction("dW", (pre.double() + ref[0]).float(), ref, pre)
    dropped = d.clone()
    dropped[640:704] = 0
    with pytest.raises(AssertionError, match="relative error"):
        check_reduction("dW", (pre.double() + dropped.t() @ a).float(), ref, pre)


def test_rejects_rows_shifted_by_one_tile(net):
    P, x, rb, g_out, (acts, g, D, dX, dw, db) = net
    ref = fwd_plane_ref(3, x, acts, mlp_bf16_weights(P))
    got = bf16_rn(ref[0])
    with pytest.raises(AssertionError):
        check_bf16("a3", torch.cat([got[128:], got[:128]]), ref)


def test_rejects_swapped_output_halves(net):
    P, x, rb, g_out, (acts, g, D, dX, dw, db) = net
    ref = dgrad_plane_ref(6, [bf16_rn(d) for d in D], acts, g_out, mlp_bf16_weights(P))
    got = bf16_rn(ref[0])
    with pytest.raises(AssertionError):
        check_bf16("delta 6", torch.cat([got[:, 128:], got[:, :128]], 1), ref)


@pytest.mark.parametrize("p,wrong", [(3, 7), (3, 5), (9, 1)])
def test_rejects_relu_gate_of_the_neighbouring_plane(net, p, wrong):
    P, x, rb, g_out, (acts, g, D, dX, dw, db) = net
    W = mlp_bf16_weights(P)
    Db = [bf16_rn(d) for d in D]
    got = bf16_rn(dgrad_plane_ref(p, Db, acts, g_out, W, gate_plane=wrong)[0])
    with pytest.raises(AssertionError):
        check_bf16(f"delta {p}", got, dgrad_plane_ref(p, Db, acts, g_out, W))


def test_rejects_missing_sigma_term(net):
    P, x, rb, g_out, (acts, g, D, dX, dw, db) = net
    W = mlp_bf16_weights(P)
    Db = [bf16_rn(d) for d in D]
    got = bf16_rn(dgrad_plane_ref(2, Db, acts, g_out, W, sigma_term=False)[0])
    with pytest.raises(AssertionError):
        check_bf16("delta 2", got, dgrad_plane_ref(2, Db, acts, g_out, W))


def test_rejects_consistent_one_ulp_bias(net):
    """+1 ulp (away from zero) on 5 % of the non-zero entries of a correctly rounded plane."""
    P, x, rb, g_out, (acts, g, D, dX, dw, db) = net
    ref = fwd_plane_ref(6, x, acts, mlp_bf16_weights(P))
    got = bf16_rn(ref[0])
    nz = (got != 0).reshape(-1).nonzero().reshape(-1)
    pick = nz[torch.randperm(len(nz), generator=torch.Generator().manual_seed(5))[: len(nz) // 20]]
    bits = got.to(torch.bfloat16).view(torch.int16).reshape(-1).clone()
    bits[pick] += 1
    biased = bits.view(torch.bfloat16).double().reshape(got.shape)
    assert nearest_bf16_fraction(biased, ref[0]) < MIN_NEAREST_BF16
    with pytest.raises(AssertionError):
        check_bf16("a6", biased, ref)
