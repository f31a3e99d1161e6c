"""Every entry the device emits against the entrywise reference of oracle/exact_z.py (one B200):

    |Z_dev[r,c] − ref[r,c]| ≤ γ_N·abs[r,c] + N·2⁻¹⁰⁷⁴,   entries with abs = 0 exactly 0.

Z is rebuilt from the emitted clique blocks (overlapping blocks must agree bit for bit) and every entry is checked, on
queries whose entries span many binades (helpers.wide_range_net / wide_range_query) alternating with plain ones,
through reused ring slots.  Covered: every tile program of the emission plan and the band kernel, β ∈ {0, 1, 2, 4, 7},
both Gram tile sizes, the four output kinds, a layer narrower than β; the affine column on every product path of
nnsdp_batch_prepare; the interval bounds layer by layer on every propagation path; and one stress-size query
(W1000-D20, β = 2) on the rows around every tile edge and block boundary.

Which kernel (Gram tile, band kernel, affine product, interval path) a case takes is predicted on the host from the
library's dispatch rules, and each GPU case asserts that prediction against the kernels the device actually launched
(their names as torch.profiler records them); the host-side coverage tests assert that the predictions cover every
path."""
import re

import numpy as np
import pytest

import exact_z as ez
import nnsdp_oracle as o
from helpers import assert_meets, rand_query, to_numeric_batch, wide_range_net, wide_range_query

pytestmark = pytest.mark.gpu
EXACT_ZDIM = 150           # Fraction arithmetic up to here, long double beyond


def _launched(fn):
    """Names (with template arguments, e.g. "gram_kernel<64>") of the kernels fn launches on the device."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = set()
    for e in prof.key_averages():
        key = e.key.replace("(int)", "")
        names.update(m.group(0) for m in re.finditer(r"\w+_kernel(<[^>(]*>)?", key))
    return names


def _plain_query(net, beta, kind, rng):
    """A query of the parity suite (γ ~ U(0, 1)) on the same net, with its IBP bounds as the given bounds; a point
    box, so every stably active neuron is Gram-active."""
    q = rand_query(net, beta, rng, kind=kind, radius=0.0)
    info = o.intervals_worst_case(q.x1min, q.x1max, net)
    amin = np.concatenate([p[0] for p in info.acx_intvs])
    amax = np.concatenate([p[1] for p in info.acx_intvs])
    smin, smax = o.make_sector_min_max(amin, amax)
    ymin = np.concatenate([p[0] for p in info.x_intvs[1:-1]])
    ymax = np.concatenate([p[1] for p in info.x_intvs[1:-1]])
    return q, (ymin, ymax, smin, smax)


def _batch_inputs(nb, net, qs, bounds):
    b = to_numeric_batch(nb, net, qs)
    b.ymin, b.ymax, b.smin, b.smax = (np.stack([bd[i] for bd in bounds]) for i in range(4))
    return b


def _dense_from_blocks(flat, cliques, Zdim):
    import nnsdp_b200 as nb

    Z, seen = np.zeros((Zdim, Zdim)), np.zeros((Zdim, Zdim), dtype=bool)
    for B, (Ck, _, _) in zip(nb.split_blocks(flat, cliques), cliques):
        c = np.asarray(Ck) - 1
        both = seen[np.ix_(c, c)]
        assert np.array_equal(Z[np.ix_(c, c)][both], B[both]), "overlapping blocks differ"
        Z[np.ix_(c, c)] = B
        seen[np.ix_(c, c)] = True
    assert np.array_equal(Z, Z.T)
    return Z


def _reference(net, beta, q, bounds, rows=None):
    mode = "exact" if net.Zdim <= EXACT_ZDIM and rows is None else "extended"
    return ez.exact_z(net, beta, q, bounds, mode=mode, rows=rows)


# ---- coverage of the emitter -----------------------------------------------------------------------------------------

# (xdims, beta, output kind, queries, ring slots): queries alternate wide-range / plain.  Batch.run into host memory
# uses the ring as two halves (a pass is ring // 2 queries), so a pass after the second writes into reused slots.
CASES = [
    ([2, 4, 7, 3, 5, 2], 7, "safety", 6, 2),          # layers narrower than beta, band across two boundaries
    ([3, 3, 3, 3, 4, 3, 3], 2, "hplane", 6, 2),
    ([2] + [10] * 6 + [2], 1, "circle", 6, 4),
    ([2, 10, 10, 10, 2], 0, "ellipsoid", 3, 2),
    ([3, 150, 260, 140, 2], 4, "ellipsoid", 6, 2),     # 128 x 32 tiles, RC / CR window programs, band kernel
    ([3, 150, 260, 140, 2], 0, "safety", 6, 2),
    ([2, 129, 128, 127, 300, 4], 2, "hplane", 6, 2),
    ([6, 300, 33, 290, 3], 7, "circle", 6, 2),        # beta above the window-program limit, a narrow layer
    ([2, 384, 384, 384, 2], 1, "hplane", 30, 20),      # passes of 10 queries, 30 Gram-active pairs: 128 x 128 tiles
]
CHECKED = {30: (0, 1, 20, 21)}                         # the queries checked when a case has many (first / reused slots)
PROGRAMS = {"SAME", "DIAG", "AFF", "RC", "CR", "MIXED", "GENERAL", "BAND"}


def _gram_tile(max_n, npairs):
    """The Gram tile launch_gram (kernels_gram.cu) picks for one launch."""
    nt128, nt64 = (max_n + 127) // 128, (max_n + 63) // 64
    items128 = nt128 * (nt128 + 1) // 2 * npairs
    pad128, pad64 = nt128 * (nt128 + 1) // 2 * 4, nt64 * (nt64 + 1) // 2
    return 64 if (items128 < 148 or pad64 * 100 <= pad128 * 85) else 128


def _gram_pairs(net, q, bounds):
    """Gram-active (query, layer) pairs of one query: layers with a neuron whose d11 = -2 (smin smax λ) is not 0, as
    prep_neuron_kernel rounds it (a λ = 0 or an underflowing product is not Gram-active)."""
    ac = net.acdim
    d11 = -2.0 * ((bounds[2] * bounds[3]) * q.gsec[:ac])
    nst = np.concatenate([[0], np.cumsum(net.xdims[1:-1])])
    return sum(bool(np.any(d11[nst[L]:nst[L + 1]] != 0.0)) for L in range(net.K - 1))


def _queries(net, beta, kind, Q, seed):
    rng = np.random.default_rng(seed)
    qs, bounds = [], []
    for i in range(Q):
        q, bd = (wide_range_query if i % 2 == 0 else _plain_query)(net, beta, kind, rng)
        qs.append(q)
        bounds.append(bd)
    return qs, bounds


def _gram_tiles(net, Q, ring, qs, bounds):
    """The Gram tile of every pass of Batch.run(host buffer): passes of ring // 2 queries (ring >= 2), the tile width
    max_block = the widest block of a Gram side (n[b], b <= K - 2)."""
    chunk = ring // 2 if ring >= 2 else ring
    max_n = max(net.xdims[:-2])
    tiles = set()
    for q0 in range(0, Q, chunk):
        npairs = sum(_gram_pairs(net, qs[i], bounds[i]) for i in range(q0, min(Q, q0 + chunk)))
        if npairs:
            tiles.add(_gram_tile(max_n, npairs))
    return tiles


def _band_kernel(xdims):
    """The plan leaves the band of the DIAG ranges to emit_band_kernel when a Gram-side hidden block is >= 256 wide."""
    return any(x >= 256 for x in xdims[1:-2])


def case_features(net, beta, kind, Q, ring, qs, bounds):
    import nnsdp_b200 as nb
    from nnsdp_b200.core import PROGRAMS as NAMES

    xdims = net.xdims
    f = {NAMES[p] for p in nb.plan_tiles(xdims, beta)[:, 10]} - {"ZERO"}
    if _band_kernel(xdims):
        f.add("BAND")
    f |= {f"beta{beta}", kind} | {f"gram{t}" for t in _gram_tiles(net, Q, ring, qs, bounds)}
    if any(x < beta for x in xdims[1:-1]):
        f.add("narrow")
    return f


def test_cases_cover_every_program_beta_gram_tile_and_kind():
    got = set()
    for xdims, beta, kind, Q, ring in CASES:
        net = wide_range_net(xdims, seed=sum(xdims) + beta)
        qs, bounds = _queries(net, beta, kind, Q, seed=beta)
        got |= case_features(net, beta, kind, Q, ring, qs, bounds)
    want = PROGRAMS | {f"beta{b}" for b in (0, 1, 2, 4, 7)} | {"gram64", "gram128", "narrow"} | \
        {"safety", "hplane", "circle", "ellipsoid"}
    assert want <= got, want - got


@pytest.mark.parametrize("xdims,beta,kind,Q,ring", CASES)
def test_every_emitted_entry_meets_the_bound(ctx, xdims, beta, kind, Q, ring):
    import nnsdp_b200 as nb

    net = wide_range_net(xdims, seed=sum(xdims) + beta)
    qs, bounds = _queries(net, beta, kind, Q, seed=beta)
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    b = nb.Batch(dnet, beta, Qcap=Q, ring=ring)
    b.set_inputs(_batch_inputs(nb, net, qs, bounds))
    out = np.full((Q, b.per_query), np.nan)
    names = _launched(lambda: b.run(out))
    b.close()
    tiles = {int(t) for n in names for t in re.findall(r"gram_kernel<(\d+)>", n)}
    assert tiles == _gram_tiles(net, Q, ring, qs, bounds), names
    if _band_kernel(xdims):
        assert "emit_band_kernel" in names, names
    cliques = dnet.cliques(beta)
    for i in CHECKED.get(Q, range(Q)):
        Z = _dense_from_blocks(out[i], cliques, net.Zdim)
        assert_meets(_reference(net, beta, qs[i], bounds[i]), Z, f"query {i} (pass {i // max(1, ring // 2)})")


# ---- the affine column on every product path -----------------------------------------------------------------------

AFFINE_CASES = [([3, 70, 131, 9, 64, 257, 4], n) for n in (1, 2, 4, 5, 9, 17, 33)] + \
    [([2, 300, 260, 200, 2], 160), ([2, 960, 1000, 2], 128)]


def _affine_paths(xdims, Q):
    """The products nnsdp_batch_prepare launches for the affine column (api.cu, kernels_bounds.cu, kernels_dgemm.cu):
    affine_all_kernel<nqt> for few queries or narrow Gram sides; otherwise the longest run of >= 2 tensor-core-sized
    layers in one dgemm_dmma_affine_layers_kernel (Q >= 128), the other layers one by one as dgemm_dmma_kernel or the
    tiled gemm_nn_kernel."""
    K, ac = len(xdims) - 1, sum(xdims[1:-1])
    if not (Q > 32 and max(xdims[:K - 1]) > 256):
        return {f"all{1 if Q == 1 else 2 if Q == 2 else 4 if Q <= 4 else 8}"}
    noff = lambda blk: sum(xdims[1:blk + 1])
    fits = [xdims[b] >= 192 and xdims[b + 1] >= 128 and noff(b + 1) % 2 == 0 and ac % 2 == 0 for b in range(K - 1)]
    run, b = (0, 0), 0
    while b < K - 1:
        if not fits[b]:
            b += 1
            continue
        e = b
        while e < K - 1 and fits[e]:
            e += 1
        if e - b > run[1] - run[0]:
            run = (b, e)
        b = e
    paths, layers = set(), run[1] - run[0] >= 2 and Q >= 128
    if layers:
        paths.add("layers")
    for b in range(K - 1):
        if layers and run[0] <= b < run[1]:
            continue
        dmma = xdims[b] >= 192 and Q >= 128 and xdims[b + 1] >= 128 and ac % 2 == 0 and noff(b + 1) % 2 == 0
        paths.add("dmma" if dmma else "gemm")
    return paths


def _affine_observed(names):
    pats = {"affine_all_kernel<": None, "dgemm_dmma_affine_layers_kernel": "layers", "dgemm_dmma_kernel": "dmma",
            "gemm_nn_kernel<1>": "gemm", "gemv_small_kernel<1": "gemv"}
    out = set()
    for n in names:
        for p, tag in pats.items():
            if n.startswith(p):
                out.add(tag or "all" + re.findall(r"\d+", n)[0])
    return out


def test_affine_cases_cover_every_product_path():
    got = set().union(*(_affine_paths(x, q) for x, q in AFFINE_CASES))
    assert got == {"all1", "all2", "all4", "all8", "layers", "dmma", "gemm"}, got


@pytest.mark.parametrize("xdims,nq", AFFINE_CASES)
def test_affine_column_meets_the_bound(ctx, xdims, nq):
    """get_affine = Z[:, a] on every product path of nnsdp_batch_prepare: affine_all_kernel with 1, 2, 4 and 8 queries
    per CTA (Q <= 32, or Gram sides <= 256 wide, whatever Q), and for Q > 32 on wider layers the multi-layer FP64
    tensor-core kernel, the single-layer one and the tiled GEMM."""
    import nnsdp_b200 as nb

    beta = 2
    net = wide_range_net(xdims, seed=nq)
    rng = np.random.default_rng(nq)
    qs, bounds = zip(*[wide_range_query(net, beta, "hplane", rng) for _ in range(nq)])
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    b = nb.Batch(dnet, beta, Qcap=nq, ring=1)
    b.set_inputs(_batch_inputs(nb, net, list(qs), list(bounds)))
    names = _launched(b.prepare)
    assert _affine_observed(names) == _affine_paths(xdims, nq), names
    aff = b.get_affine()
    b.close()
    a = net.Zdim - 1
    for i in sorted({0, nq // 2, nq - 1}):
        R = ez.exact_z(net, beta, qs[i], bounds[i], mode="extended", rows=[a])
        assert_meets(R, aff[i][None, :], f"affine column of query {i}")


# ---- interval bounds, layer by layer -------------------------------------------------------------------------------

def _ibp_path(xdims, Q):
    if max(xdims) <= 256:
        return {"chain"}
    if Q <= 8:
        return {"all"}
    if Q <= 32:
        return {"gemv"}
    out = set()
    xtot = sum(xdims)
    off = np.concatenate([[0], np.cumsum(xdims)])
    for k in range(len(xdims) - 1):
        n_in, n_out = xdims[k], xdims[k + 1]
        dmma = n_out >= 192 and Q >= 128 and n_in >= 128 and n_out % 2 == 0 and xtot % 2 == 0 and off[k] % 2 == 0
        out.add("dmma" if dmma else "gemm")
    return out


def _ibp_observed(names):
    pats = {"ibp_chain_kernel": "chain", "ibp_all_kernel": "all", "gemv_small_kernel<0": "gemv", "gemm_nn_kernel<0>": "gemm",
            "ibp_dmma_kernel": "dmma"}
    return {tag for n in names for p, tag in pats.items() if n.startswith(p)}


IBP_CASES = [([3, 70, 131, 9, 64, 200, 4], 40), ([3, 70, 131, 9, 64, 257, 4], 5), ([3, 70, 131, 9, 64, 257, 4], 17),
             ([3, 70, 131, 9, 64, 257, 4], 33), ([2, 300, 260, 200, 2], 160)]


def test_ibp_cases_cover_every_path():
    got = set().union(*(_ibp_path(x, q) for x, q in IBP_CASES))
    assert got == {"chain", "all", "gemv", "gemm", "dmma"}, got


@pytest.mark.parametrize("xdims,nq", IBP_CASES)
def test_interval_bounds_meet_the_bound_layer_by_layer(ctx, xdims, nq):
    """The device's layer-k bounds are the exact inputs of layer k+1: |y_dev − y| ≤ γ_{n+3}(|W| max(|xmin|, |xmax|) + |b|)
    with y = W⁺xmin + W⁻xmax + b (and the W⁻xmin + W⁺xmax form for ymax).  The bound covers the W⁺/W⁻ form and the
    centre / radius form of the chain and tensor-core kernels (c and r each round once, |c| + |r| = max(|xmin|, |xmax|)).
    Post-activation bounds are max(pre, 0) exactly."""
    import nnsdp_b200 as nb

    net = wide_range_net(xdims, seed=nq)
    rng = np.random.default_rng(nq)
    c = rng.uniform(-1, 1, (nq, xdims[0]))
    r = 2.0 ** rng.uniform(-20, 0, (nq, 1)) * rng.random((nq, xdims[0]))
    r[0] = 0.0                                                                        # a point box
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    b = nb.Batch(dnet, 1, Qcap=nq, ring=0)                                           # bounds only
    b.set_inputs(nb.NumericBatch(x1min=c - r, x1max=c + r))
    names = _launched(b.bounds)
    assert _ibp_observed(names) == _ibp_path(xdims, nq), names
    bd = b.get_bounds()
    b.close()
    off = np.concatenate([[0], np.cumsum(xdims)])
    noff = np.concatenate([[0], np.cumsum(xdims[1:-1])])
    K = len(xdims) - 1
    for i in sorted({0, 1, nq // 2, nq - 1}):
        assert np.array_equal(bd["xmin"][i, :xdims[0]], c[i] - r[i]) and np.array_equal(bd["xmax"][i, :xdims[0]], c[i] + r[i])
        for k in range(K):
            M = net.Ms[k].astype(np.longdouble)
            W, bias = M[:, :-1], M[:, -1]
            lo = bd["xmin"][i, off[k]:off[k + 1]].astype(np.longdouble)
            hi = bd["xmax"][i, off[k]:off[k + 1]].astype(np.longdouble)
            Wp, Wn = np.maximum(W, 0), np.minimum(W, 0)
            ylo, yhi = Wp @ lo + Wn @ hi + bias, Wp @ hi + Wn @ lo + bias
            n = xdims[k]
            scale = np.abs(W) @ np.maximum(np.abs(lo), np.abs(hi)) + np.abs(bias)
            tol = (ez.gamma(n + 3) + 2 * ez.gamma(n + 2, ez.UEXT)) * scale.astype(np.float64) * (1 + 2.0 ** -50)
            if k < K - 1:
                dlo, dhi = bd["acxmin"][i, noff[k]:noff[k + 1]], bd["acxmax"][i, noff[k]:noff[k + 1]]
                assert np.array_equal(bd["xmin"][i, off[k + 1]:off[k + 2]], np.maximum(dlo, 0.0))
                assert np.array_equal(bd["xmax"][i, off[k + 1]:off[k + 2]], np.maximum(dhi, 0.0))
            else:
                dlo, dhi = bd["xmin"][i, off[k + 1]:off[k + 2]], bd["xmax"][i, off[k + 1]:off[k + 2]]
            for d, y in ((dlo, ylo), (dhi, yhi)):
                err = np.abs(d.astype(np.longdouble) - y).astype(np.float64)
                assert (err <= tol).all(), (i, k, float((err / np.where(tol > 0, tol, 1)).max()))


# ---- one stress-size query ------------------------------------------------------------------------------------------

def _edge_rows(cliques, xdims, nsample, rng):
    """Global rows within 2 of every 32 / 64 / 128 tile edge of every clique's local index (the two rows on either side of
    it), within ±2 of every block boundary, the last rows of every clique, plus a random sample."""
    rows = set()
    for Ck, _, _ in cliques:
        Ck = np.asarray(Ck) - 1
        loc = np.arange(len(Ck))
        near = (loc % 32 <= 1) | (loc % 32 >= 30) | (loc >= len(Ck) - 2)
        rows.update(Ck[near].tolist())
    off = np.concatenate([[0], np.cumsum(xdims[:-1]), [sum(xdims[:-1]) + 1]])
    for e in off:
        rows.update(range(max(0, e - 2), min(off[-1], e + 2)))
    Zdim = sum(xdims[:-1]) + 1
    rows.update(rng.choice(Zdim, nsample, replace=False).tolist())
    return np.array(sorted(r for r in rows if 0 <= r < Zdim))


def test_stress_query_rows_at_every_tile_edge(ctx):
    import nnsdp_b200 as nb

    xdims, beta = [2] + [1000] * 20 + [2], 2
    net = wide_range_net(xdims, seed=2024)
    rng = np.random.default_rng(2024)
    q, bounds = wide_range_query(net, beta, "ellipsoid", rng)
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    b = nb.Batch(dnet, beta, Qcap=1, ring=1)
    b.set_inputs(_batch_inputs(nb, net, [q], [bounds]))
    out = np.empty((1, b.per_query))
    b.run(out)
    b.close()
    cliques = dnet.cliques(beta)
    rows = _edge_rows(cliques, xdims, 64, rng)
    Zdim = net.Zdim
    pos = np.full(Zdim, -1)
    pos[rows] = np.arange(len(rows))
    Zr, seen = np.zeros((len(rows), Zdim)), np.zeros((len(rows), Zdim), dtype=bool)
    for B, (Ck, _, _) in zip(nb.split_blocks(out[0], cliques), cliques):
        c = np.asarray(Ck) - 1
        li = np.nonzero(pos[c] >= 0)[0]
        p = pos[c[li]]
        prev = Zr[np.ix_(p, c)][seen[np.ix_(p, c)]]
        assert np.array_equal(prev, B[li][seen[np.ix_(p, c)]]), "overlapping blocks differ"
        Zr[np.ix_(p, c)] = B[li]
        seen[np.ix_(p, c)] = True
    del out
    for part in np.array_split(np.arange(len(rows)), -(-len(rows) // 768)):     # bounded host memory
        R = ez.exact_z(net, beta, q, bounds, mode="extended", rows=rows[part])
        assert_meets(R, Zr[part], "stress query")
