"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle on seeded inputs.

Bars (BASELINE.json north_star): clique index sets and sparsity patterns bit-exact; sector slopes
(values in {0,1}) bit-exact; FP64 bounds and block entries within 1e-12 relative (normwise per
block: the Gram entries cancel, so an entrywise bound is not attainable -- SURVEY.md section 7).
"""
import os

import numpy as np
import pytest

import nnsdp_oracle as o
from helpers import rand_net, rand_query, relerr, to_numeric_batch

pytestmark = pytest.mark.gpu

TOL = 1e-12

NETS = [
    ([2, 3, 3, 2], 1),
    ([2, 3, 2], 0),
    ([2, 3, 2], 2),
    ([3, 3, 3, 3, 4, 3, 3], 2),          # xdims of experiments/plot_sparsity.ipynb
    ([2, 10, 10, 10, 10, 2], 3),
    ([2, 4, 7, 3, 5, 2], 5),              # beta wider than a layer: band crosses two boundaries
    ([5, 50, 50, 50, 50, 50, 50, 5], 2),  # ACAS-shaped (config 4)
    ([2] + [20] * 10 + [2], 1),
    ([2, 70, 130, 64, 3], 2),             # ragged widths, block-split tiles, 2 Gram tiles
]


def _oracle_bounds(net, q):
    info = o.intervals_worst_case(q.x1min, q.x1max, net)
    xmin = np.concatenate([p[0] for p in info.x_intvs])
    xmax = np.concatenate([p[1] for p in info.x_intvs])
    amin = np.concatenate([p[0] for p in info.acx_intvs])
    amax = np.concatenate([p[1] for p in info.acx_intvs])
    return info, xmin, xmax, amin, amax


@pytest.mark.parametrize("xdims,beta", NETS)
def test_bounds_and_sector(ctx, xdims, beta):
    import nnsdp_b200 as nb

    net = rand_net(xdims, seed=11)
    rng = np.random.default_rng(5)
    qs = [rand_query(net, beta, rng, radius=r) for r in (0.0, 0.01, 0.1, 0.5)]
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    r = nb.bounds_ibp(dnet, np.stack([q.x1min for q in qs]), np.stack([q.x1max for q in qs]))
    for i, q in enumerate(qs):
        _, xmin, xmax, amin, amax = _oracle_bounds(net, q)
        scale = max(np.abs(xmax).max(), np.abs(xmin).max(), 1.0)
        assert np.abs(r["xmin"][i] - xmin).max() <= TOL * scale
        assert np.abs(r["xmax"][i] - xmax).max() <= TOL * scale
        assert np.abs(r["acxmin"][i] - amin).max() <= TOL * scale
        assert np.abs(r["acxmax"][i] - amax).max() <= TOL * scale
        assert np.all(r["xmin"][i] <= r["xmax"][i])
        smin, smax = nb.sector_minmax(ctx, r["acxmin"][i], r["acxmax"][i])
        rmin, rmax = o.make_sector_min_max(r["acxmin"][i], r["acxmax"][i])
        assert np.array_equal(smin, rmin) and np.array_equal(smax, rmax)  # bit-exact on equal inputs
        # one-step pre-activation IBP from given x bounds (intervals_auto_lirpa.jl:55-62)
    amin_d, amax_d = nb.preact_from_x(dnet, r["xmin"], r["xmax"])
    for i, q in enumerate(qs):
        info, *_ = _oracle_bounds(net, q)
        ref = o.preact_from_x(info.x_intvs, net)
        scale = max(np.abs(np.concatenate([p[1] for p in ref])).max(), 1.0)
        assert np.abs(amin_d[i] - np.concatenate([p[0] for p in ref])).max() <= TOL * scale
        assert np.abs(amax_d[i] - np.concatenate([p[1] for p in ref])).max() <= TOL * scale


def test_preact_assert(ctx):
    """ykmin <= ykmax is asserted by the reference (intervals_auto_lirpa.jl:60)."""
    import nnsdp_b200 as nb

    net = rand_net([2, 5, 5, 2], seed=1)
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    xmin = np.ones((1, sum(net.xdims)))
    xmax = np.zeros((1, sum(net.xdims)))  # inverted box
    with pytest.raises(nb.NnsdpError) as e:
        nb.preact_from_x(dnet, xmin, xmax)
    assert e.value.code == -5


@pytest.mark.parametrize("kind", ["safety", "hplaneS", "hplane", "circle", "ellipsoid"])
@pytest.mark.parametrize("xdims,beta", NETS)
def test_dense_Z_and_blocks(ctx, xdims, beta, kind):
    import nnsdp_b200 as nb

    net = rand_net(xdims, seed=3)
    rng = np.random.default_rng(17)
    # tight boxes give stably-active neurons (Gram path), wide boxes give unstable ones
    qs = [rand_query(net, beta, rng, kind=kind, radius=r) for r in (0.001, 0.02, 0.3)]
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    batch = to_numeric_batch(nb, net, qs)
    Z = nb.assemble_dense(dnet, beta, batch)
    flat = nb.assemble_blocks(dnet, beta, batch)
    cliques = dnet.cliques(beta)
    ref_cliques = o.make_cliques(net, beta)
    assert len(cliques) == len(ref_cliques)
    for (a, pa, da), (b, pb, db) in zip(cliques, ref_cliques):
        assert a.dtype == np.int64 and np.array_equal(a, b)
        assert all(np.array_equal(x, y) for x, y in zip(pa, pb)) and len(pa) == len(pb)
        assert all(np.array_equal(x, y) for x, y in zip(da, db)) and len(da) == len(db)
    for i, q in enumerate(qs):
        ref = o.run_query(net, beta, q, form="closed")
        assert relerr(Z[i], ref["Z"]) <= TOL
        assert np.array_equal(Z[i], Z[i].T)  # bit-symmetric
        lit = o.run_query(net, beta, q, form="literal")
        assert relerr(Z[i], lit["Z"]) <= TOL
        # sparsity pattern: structural pattern of the notebook contains ours; mask equals the oracle's
        pat = o.structural_pattern_notebook(net.xdims, beta)
        assert not np.any((Z[i] != 0) & ~pat)
        blocks = nb.split_blocks(flat[i], cliques)
        for blk, rb in zip(blocks, ref["blocks"]):
            assert blk.shape == rb.shape
            assert relerr(blk, rb) <= TOL
            thr = 1e-13 * max(np.abs(rb).max(), 1e-300)
            assert np.array_equal(np.abs(blk) > thr, np.abs(rb) > thr)
        # blocks are exactly the restriction of the dense Z the same library produced
        for blk, (Ck, _, _) in zip(blocks, cliques):
            assert np.array_equal(blk, Z[i][np.ix_(Ck - 1, Ck - 1)])


def test_gram_active_path(ctx):
    """Degenerate box (xmin == xmax): every neuron is stably on or off, so the Gram term
    W' diag(-2 lambda) W is exercised on every layer, including multi-tile widths."""
    import nnsdp_b200 as nb

    xdims, beta = [3, 150, 260, 140, 2], 2
    net = rand_net(xdims, seed=9, sigma=0.3)
    rng = np.random.default_rng(2)
    qs = [rand_query(net, beta, rng, kind="safety", radius=0.0) for _ in range(2)]
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    b = nb.Batch(dnet, beta, Qcap=2, ring=2, dense=True)
    b.set_inputs(to_numeric_batch(nb, net, qs))
    b.run()
    ncon, nact = b.gram_stats()
    assert ncon == 2 * (len(xdims) - 2) and nact > 100
    for i, q in enumerate(qs):
        ref = o.run_query(net, beta, q, form="closed")
        Z = b.get_slot(i).reshape(ref["Z"].shape).T
        assert relerr(Z, ref["Z"]) <= TOL
        assert np.array_equal(Z, Z.T)


def test_supplied_bounds_and_shared_inputs(ctx):
    """Caller-supplied QC data (the CROWN route of the reference: bounds come from outside) and
    stride-0 sharing: a reach batch where only the hyperplane normal differs (NnSdp.jl:73-95)."""
    import nnsdp_b200 as nb

    xdims, beta, nq = [2, 20, 20, 20, 20, 2], 2, 16
    net = rand_net(xdims, seed=4)
    rng = np.random.default_rng(8)
    base = rand_query(net, beta, rng, kind="hplane", radius=0.1)
    ref0 = o.run_query(net, beta, base)
    # perturb the bounds so that they are NOT what IBP would give
    bnd, sec = ref0["qc_bounded"], ref0["qc_sector"]
    ymin = bnd.acymin - 0.01 * rng.random(net.acdim)
    ymax = bnd.acymax + 0.01 * rng.random(net.acdim)
    smin = (rng.random(net.acdim) < 0.3).astype(float)
    smax = np.maximum(smin, (rng.random(net.acdim) < 0.7).astype(float))
    thetas = 2 * np.pi * np.arange(nq) / nq
    normals = np.stack([np.cos(thetas), np.sin(thetas)], axis=1)
    gouts = rng.random((nq, 1))
    batch = nb.NumericBatch(
        x1min=base.x1min, x1max=base.x1max, gamma_in=base.gin, gamma_bnd=base.gbnd, gamma_sec=base.gsec,
        ymin=ymin, ymax=ymax, smin=smin, smax=smax, out_kind=nb.OUT_HPLANE, out_vec=normals, gamma_out=gouts)
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    flat = nb.assemble_blocks(dnet, beta, batch, Q=nq)
    cliques = o.make_cliques(net, beta)
    qb = o.QcActivBounded(net.acdim, ymin, ymax)
    qs_ = o.QcActivSector(net.acdim, beta, smin, smax)
    for i in range(nq):
        Zr = o.assemble_Z_closed_form(net, o.QcInputBox(base.x1min, base.x1max), o.QcReachHplane(normals[i]), qb, qs_,
                                      base.gin, base.gbnd, base.gsec, gouts[i])
        for blk, rb in zip(nb.split_blocks(flat[i], cliques), o.clique_blocks(Zr, cliques)):
            assert relerr(blk, rb) <= TOL


def test_tile_classes_do_not_change_results(ctx):
    """The host-side tile flags only skip terms that are structurally zero: evaluating every term
    in every tile (NNSDP_NO_TILE_CLASSES=1) must give bit-identical output."""
    import nnsdp_b200 as nb

    outs = []
    for flag in ("0", "1"):
        os.environ["NNSDP_NO_TILE_CLASSES"] = flag
        try:
            for xdims, beta in ([2, 70, 130, 64, 3], 3), ([2] + [12] * 6 + [2], 4):
                net = rand_net(xdims, seed=21)
                rng = np.random.default_rng(1)
                qs = [rand_query(net, beta, rng, kind="safety", radius=r) for r in (0.0, 0.2)]
                dnet = nb.Net(ctx, net.xdims, net.Ms)
                outs.append(nb.assemble_blocks(dnet, beta, to_numeric_batch(nb, net, qs)))
        finally:
            os.environ["NNSDP_NO_TILE_CLASSES"] = "0"
    assert np.array_equal(outs[0], outs[2]) and np.array_equal(outs[1], outs[3])


def test_batch_ring_and_chunking(ctx):
    """More queries than ring slots, odd ring, host gather through the two-half ring."""
    import nnsdp_b200 as nb

    xdims, beta, nq = [2, 16, 16, 16, 2], 1, 11
    net = rand_net(xdims, seed=5)
    rng = np.random.default_rng(3)
    qs = [rand_query(net, beta, rng, kind="circle", radius=0.05 * (i + 1)) for i in range(nq)]
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    b = nb.Batch(dnet, beta, Qcap=nq, ring=5)
    b.set_inputs(to_numeric_batch(nb, net, qs))
    out = np.zeros((nq, b.per_query))
    b.run(out)
    cliques = o.make_cliques(net, beta)
    for i, q in enumerate(qs):
        ref = o.run_query(net, beta, q)
        for blk, rb in zip(nb.split_blocks(out[i], cliques), ref["blocks"]):
            assert relerr(blk, rb) <= TOL
    ms, launches = b.stage_ms("emit")
    assert launches >= 3 and ms > 0


def test_reference_api_mirror(ctx):
    """makeZin / makeZac / makeZout / makeCliques through the reference-shaped host API."""
    from nnsdp_b200 import reference_api as R

    xdims, beta = [2, 6, 5, 7, 2], 2
    net = rand_net(xdims, seed=13)
    ff = R.FeedFwdNet(net.xdims, net.Ms)
    rng = np.random.default_rng(6)
    x1min, x1max = np.array([0.4, 0.6]), np.array([0.5, 0.9])
    qc_in = R.QcInputBox(x1min, x1max)
    qc_acts = R.makeQcActivs(ff, x1min=x1min, x1max=x1max, beta=beta)
    o_acts = o.make_qc_activs_intvs(net, x1min, x1max, beta)
    assert np.array_equal(qc_acts[1].smin, o_acts[1].smin) and np.array_equal(qc_acts[1].smax, o_acts[1].smax)
    gin, gb, gs = rng.random(2), rng.random(net.acdim), rng.random(qc_acts[1].vardim)
    assert relerr(R.makeZin(gin, qc_in, ff), o.makeZin(gin, o.QcInputBox(x1min, x1max), net).toarray()) <= TOL
    assert relerr(R.makeZac(gb, qc_acts[0], ff), o.makeZac(gb, o_acts[0], net).toarray()) <= TOL
    assert relerr(R.makeZac(gs, qc_acts[1], ff), o.makeZac(gs, o_acts[1], net).toarray()) <= TOL
    S = R.hplaneS([1.0, -0.5], 0.3, ff)
    assert relerr(R.makeZout(R.QcSafety(S), ff), o.makeZout(o.QcSafety(S), net).toarray()) <= TOL
    ell = R.QcReachEllipsoid(rng.standard_normal((2, 2)), rng.standard_normal(2))
    assert relerr(R.makeZout([0.4], ell, ff), o.makeZout(o.QcReachEllipsoid(ell.invP, ell.yc), net, [0.4]).toarray()) <= TOL
    query = R.SafetyQuery(ff, qc_in, R.QcSafety(S), qc_acts)
    cl = R.makeCliques(query.qcs, ff)
    for (a, _, _), (b, _, _) in zip(cl, o.make_cliques(net, beta)):
        assert np.array_equal(a, b)
    Z = R.assembleZ(query, gin, [gb, gs])
    Zr = o.assemble_Z_literal(net, o.QcInputBox(x1min, x1max), o.QcSafety(S), o_acts, gin, [gb, gs])
    assert relerr(Z, Zr) <= TOL
    cl2, blocks = R.assembleCliqueBlocks(query, gin, [gb, gs])
    for blk, (Ck, _, _) in zip(blocks, cl2):
        assert relerr(blk, Zr[np.ix_(Ck - 1, Ck - 1)]) <= TOL
    ev = np.linalg.eigvalsh(Zr)
    assert abs(R.eigmaxZ(query, gin, [gb, gs]) - ev[-1]) <= 1e-9 * max(abs(ev[0]), abs(ev[-1]))


def test_error_paths(ctx):
    import nnsdp_b200 as nb

    net = rand_net([2, 4, 4, 2], seed=1)
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    with pytest.raises(nb.NnsdpError):  # beta > acdim: _lambda_dim assert of the reference
        dnet.sizes(9)
    rng = np.random.default_rng(0)
    q = rand_query(net, 1, rng)
    batch = to_numeric_batch(nb, net, [q])
    batch.ymin = np.ones((1, net.acdim))
    batch.ymax = np.zeros((1, net.acdim))  # acymin <= acymax violated
    batch.smin = np.zeros((1, net.acdim))
    batch.smax = np.ones((1, net.acdim))
    with pytest.raises(nb.NnsdpError) as e:
        nb.assemble_blocks(dnet, 1, batch)
    assert e.value.code == -5
    b = nb.Batch(dnet, 1, Qcap=1, ring=1)
    with pytest.raises(nb.NnsdpError) as e:
        b.prepare()  # before set_inputs
    assert e.value.code == -4


# ---------------------------------------------------------------------------------------------
# committed golden fixtures (tests/golden/, made by tests/golden/make_golden.py)
# ---------------------------------------------------------------------------------------------
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _gold_net(d):
    xd = d["xdims"].tolist()
    return xd, [d[f"M{k}"] for k in range(len(xd) - 1)]


@pytest.mark.parametrize("tag", ["safety", "ellipsoid", "tight"])
def test_golden_config1(ctx, tag):
    """BASELINE.json configs[0]: the reference's shipped scale-I2-O2-W10-D10 net, beta = 1."""
    import nnsdp_b200 as nb

    d = np.load(os.path.join(GOLD, "config1_W10_D10_beta1.npz"))
    xd, Ms = _gold_net(d)
    beta = int(d["beta"])
    dnet = nb.Net(ctx, xd, Ms)
    kw = dict(out_kind=nb.OUT_SAFETY, out_S=d["S"][None]) if tag != "ellipsoid" else dict(
        out_kind=nb.OUT_ELLIPSOID, out_vec=d["yc"][None], out_invP=np.eye(2)[None], gamma_out=d["gout"][None])
    batch = nb.NumericBatch(x1min=d[f"{tag}_x1min"][None], x1max=d[f"{tag}_x1max"][None], gamma_in=d[f"{tag}_gin"][None],
                            gamma_bnd=d[f"{tag}_gbnd"][None], gamma_sec=d[f"{tag}_gsec"][None], **kw)
    r = nb.bounds_ibp(dnet, d[f"{tag}_x1min"][None], d[f"{tag}_x1max"][None])
    for k in ("xmin", "xmax", "acxmin", "acxmax"):
        ref = d[f"{tag}_{k}"]
        assert np.abs(r[k][0] - ref).max() <= TOL * max(np.abs(ref).max(), 1.0)
    smin, smax = nb.sector_minmax(ctx, r["acxmin"][0], r["acxmax"][0])
    assert np.array_equal(smin, d[f"{tag}_smin"]) and np.array_equal(smax, d[f"{tag}_smax"])
    Z = nb.assemble_dense(dnet, beta, batch)[0]
    assert relerr(Z, d[f"{tag}_Z"]) <= TOL
    cliques = dnet.cliques(beta)
    assert len(cliques) == int(d["ncliques"])
    flat = nb.assemble_blocks(dnet, beta, batch)[0]
    for k, (blk, (Ck, _, ds)) in enumerate(zip(nb.split_blocks(flat, cliques), cliques)):
        assert np.array_equal(Ck, d[f"Ck{k}"])
        for i, dd in enumerate(ds):
            assert np.array_equal(dd, d[f"Dk{k}_{i}"])
        rb = d[f"{tag}_Z"][np.ix_(Ck - 1, Ck - 1)]
        assert relerr(blk, rb) <= TOL


def test_golden_config3_reach_batch(ctx):
    """BASELINE.json configs[2]: 64 hyperplane directions on reach-I2-O2-W20-D10, shared bounds and
    multipliers (stride 0), per-direction normal and gamma_out."""
    import nnsdp_b200 as nb

    d = np.load(os.path.join(GOLD, "config3_reach_W20_D10_beta2.npz"))
    xd, Ms = _gold_net(d)
    beta = int(d["beta"])
    dnet = nb.Net(ctx, xd, Ms)
    batch = nb.NumericBatch(x1min=d["dir0_x1min"], x1max=d["dir0_x1max"], gamma_in=d["dir0_gin"], gamma_bnd=d["dir0_gbnd"],
                            gamma_sec=d["dir0_gsec"], out_kind=nb.OUT_HPLANE, out_vec=d["normals"], gamma_out=d["gout"][:, None])
    flat = nb.assemble_blocks(dnet, beta, batch, Q=64)
    cliques = dnet.cliques(beta)
    for i in range(64):
        blocks = nb.split_blocks(flat[i], cliques)
        fro = np.array([np.linalg.norm(b) for b in blocks])
        assert np.abs(fro - d["block_fro"][i]).max() <= TOL * d["block_fro"][i].max()
        # the affine column of Z restricted to each clique is the last column of its block
        for blk, (Ck, _, _) in zip(blocks, cliques):
            ref = d["affine_cols"][i][Ck - 1]
            assert np.abs(blk[:, -1] - ref).max() <= TOL * max(np.abs(d["affine_cols"][i]).max(), 1.0)
    for i in (0, 17):
        Zr = d[f"dir{i}_Z"]
        for blk, (Ck, _, _) in zip(nb.split_blocks(flat[i], cliques), cliques):
            assert relerr(blk, Zr[np.ix_(Ck - 1, Ck - 1)]) <= TOL


# ---------------------------------------------------------------------------------------------
# full-size configs through size-independent properties (the oracle would need minutes and GBs)
# ---------------------------------------------------------------------------------------------
def test_stress_config_properties(ctx):
    """BASELINE.json configs[4]: width 1000, depth 20, beta = 2.  Checked: (1) every block is
    bit-symmetric; (2) overlapping cliques agree bit-for-bit on their shared index range;
    (3) Z is affine in the multipliers: blocks(g1) + blocks(g2) - blocks(0) == blocks(g1 + g2) to
    1e-12; (4) bounds are ordered; (5) one clique block against the closed-form oracle restricted
    to that clique's rows (built without the dense Z)."""
    import bench
    import nnsdp_b200 as nb

    xdims, Ms, beta, inp = bench.make_workload("stress-W1000-D20-beta2-Q1024", 0, Q=2)
    dnet = nb.Net(ctx, xdims, Ms)
    sz = dnet.sizes(beta)
    assert sz["ncliques"] == 19 and sz["sum_ck_sq"] * 8 == 1330657432
    cliques = dnet.cliques(beta)
    # tight box on query 1 so that some layers carry stably-active neurons (Gram term)
    inp["x1min"][1] = inp["x1min"][1] * 0 + 1.0 - 1e-4
    inp["x1max"][1] = inp["x1min"][1] + 2e-4

    def run(scale1, scale2):
        g = {k: inp[k] * scale1 for k in ("gamma_in", "gamma_bnd", "gamma_sec")}
        g2 = {k: inp[k][::-1] * scale2 for k in ("gamma_in", "gamma_bnd", "gamma_sec")}
        batch = nb.NumericBatch(x1min=inp["x1min"], x1max=inp["x1max"], out_kind=nb.OUT_SAFETY, out_S=inp["out_S"],
                                **{k: g[k] + g2[k] for k in g})
        b = nb.Batch(dnet, beta, Qcap=2, ring=1)
        b.set_inputs(batch, Q=2)
        b.bounds()
        b.prepare()
        b.emit(1, 1)
        b.sync()
        out = b.get_slot(0)
        bounds = b.get_bounds()
        stats = b.gram_stats()
        b.close()
        return out, bounds, stats

    f1, bounds, stats = run(1.0, 0.0)
    assert stats[1] > 0  # the Gram path ran
    assert np.all(bounds["xmin"] <= bounds["xmax"]) and np.all(bounds["acxmin"] <= bounds["acxmax"])
    blocks = nb.split_blocks(f1, cliques)
    for blk in blocks:
        assert np.array_equal(blk, blk.T)
    for (Ca, _, _), (Cb, _, _), A, B in zip(cliques, cliques[1:], blocks, blocks[1:]):
        common = np.intersect1d(Ca, Cb)
        ia, ib = np.searchsorted(Ca, common), np.searchsorted(Cb, common)
        assert np.array_equal(A[np.ix_(ia, ia)], B[np.ix_(ib, ib)])
    f2, _, _ = run(0.0, 1.0)
    f0, _, _ = run(0.0, 0.0)
    f12, _, _ = run(1.0, 1.0)
    scale = np.abs(f12).max()
    assert np.abs((f1 - f0) + (f2 - f0) - (f12 - f0)).max() <= 1e-12 * scale
    del f2, f0, f12

    # (5) cliques against the oracle, assembled from the closed form on each clique's rows only: the first clique
    # (x_1 coupling, Z_in), one of the regular ones, a middle one and the last (W_K' S22 W_K, x_K against itself),
    # for BOTH queries -- the wide box (no Gram-active layer) and the tight one
    net = o.FeedFwdNet(xdims, Ms)
    b = nb.Batch(dnet, beta, Qcap=2, ring=1)
    b.set_inputs(nb.NumericBatch(x1min=inp["x1min"], x1max=inp["x1max"], out_kind=nb.OUT_SAFETY, out_S=inp["out_S"],
                                 **{k: inp[k] for k in ("gamma_in", "gamma_bnd", "gamma_sec")}), Q=2)
    b.bounds()
    b.prepare()
    for qi in (0, 1):
        b.emit(qi, 1)
        b.sync()
        blocks = nb.split_blocks(b.get_slot(0), cliques)
        q = o.NumericQuery(x1min=inp["x1min"][qi], x1max=inp["x1max"][qi], gin=inp["gamma_in"][qi], gbnd=inp["gamma_bnd"][qi],
                           gsec=inp["gamma_sec"][qi], qc_out=o.QcSafety(S=inp["out_S"][0]))
        for k in ((0, 3, 9, 18) if qi == 1 else (0, 18)):
            ref = clique_block_oracle(net, beta, q, cliques[k][0] - 1)
            assert relerr(blocks[k], ref) <= TOL, (qi, k)
        del blocks
    b.close()


@pytest.mark.parametrize("beta", [1, 2, 3])
def test_config2_top_W100_D50(ctx, beta):
    """Top of BASELINE.json configs[1] (experiments/scale.jl sweep: width 100, depth 50, beta in {1,2,3}) with the
    box of scale.jl:26-27 and a tight box -- the shapes the narrow-net kernels serve (ibp_chain_kernel, 100-row
    register-window tiles): bounds, dense Z, every clique block and the packed records against the oracle."""
    import nnsdp_b200 as nb

    xdims = [2] + [100] * 50 + [2]
    net = rand_net(xdims, seed=50100)               # sigma by the rule of scripts/make_networks.jl:44
    rng = np.random.default_rng(7)
    qs = [rand_query(net, beta, rng, kind="ellipsoid", radius=0.5, centre=[1.0, 1.0]),
          rand_query(net, beta, rng, kind="safety", radius=1e-4, centre=[1.0, 1.0])]
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    cliques = dnet.cliques(beta)
    ref_cliques = o.make_cliques(net, beta)
    assert all(np.array_equal(a[0], b[0]) for a, b in zip(cliques, ref_cliques)) and len(cliques) == len(ref_cliques)
    for q in qs:
        batch = to_numeric_batch(nb, net, [q])
        r = nb.bounds_ibp(dnet, q.x1min[None], q.x1max[None])
        _, xmin, xmax, amin, amax = _oracle_bounds(net, q)
        scale = max(np.abs(xmax).max(), np.abs(xmin).max(), 1.0)
        assert np.abs(r["xmin"][0] - xmin).max() <= TOL * scale and np.abs(r["acxmax"][0] - amax).max() <= TOL * scale
        ref = o.run_query(net, beta, q)
        Z = nb.assemble_dense(dnet, beta, batch)[0]
        assert relerr(Z, ref["Z"]) <= TOL and np.array_equal(Z, Z.T)
        flat = nb.assemble_blocks(dnet, beta, batch)[0]
        for blk, (Ck, _, _), rb in zip(nb.split_blocks(flat, cliques), cliques, ref["blocks"]):
            assert np.array_equal(blk, Z[np.ix_(Ck - 1, Ck - 1)])
            assert relerr(blk, rb) <= TOL
        rec, present, _ = nb.assemble_packed(dnet, beta, batch)
        assert np.array_equal(nb.packed_unpack(xdims, beta, rec[0], present[0]), flat)


def test_config2_reference_net_W20_D100(ctx):
    """The reference's largest recorded run (dump/scale/chordalsdp-scale-I2-O2-W20-D100.nnet.csv): its shipped
    bench/rand/scale-I2-O2-W20-D100.nnet read through nnsdp_nnet_read, beta = 2, box of scale.jl:26-27, 99 cliques."""
    import nnsdp_b200 as nb

    path = os.path.join(GOLD, "scale-I2-O2-W20-D100.nnet")
    xdims, Ms = nb.read_nnet(path)
    net = o.load_nnet(path)
    assert xdims == list(net.xdims) and all(np.array_equal(a, b) for a, b in zip(Ms, net.Ms))
    beta = 2
    rng = np.random.default_rng(3)
    qs = [rand_query(net, beta, rng, kind="ellipsoid", radius=0.5, centre=[1.0, 1.0]),
          rand_query(net, beta, rng, kind="hplane", radius=0.0, centre=[1.0, 1.0])]
    dnet = nb.Net(ctx, xdims, Ms)
    cliques = dnet.cliques(beta)
    assert len(cliques) == 99
    for q in qs:
        batch = to_numeric_batch(nb, net, [q])
        ref = o.run_query(net, beta, q)
        Z = nb.assemble_dense(dnet, beta, batch)[0]
        assert relerr(Z, ref["Z"]) <= TOL
        flat = nb.assemble_blocks(dnet, beta, batch)[0]
        for blk, (Ck, _, _), rb in zip(nb.split_blocks(flat, cliques), ref["cliques"], ref["blocks"]):
            assert relerr(blk, rb) <= TOL
        rec, present, _ = nb.assemble_packed(dnet, beta, batch)
        assert np.array_equal(nb.packed_unpack(xdims, beta, rec[0], present[0]), flat)
        # CROWN bounds (the reference's default) on the same net against the restatement
        rc = nb.bounds_crown(dnet, q.x1min[None], q.x1max[None])
        info = o.intervals_crown(q.x1min, q.x1max, net)
        xr = np.concatenate([p[1] for p in info.x_intvs])
        assert np.abs(rc["xmax"][0] - xr).max() <= 1e-9 * max(np.abs(xr).max(), 1.0)


def clique_block_oracle(net, beta, q, Ck):
    """Z[Ck, Ck] from the closed form (SURVEY.md 8a appendix) without materialising Z: only the
    terms with both indices in Ck are evaluated.  Independent of assemble_Z_closed_form's code path
    for the band (dense banded M here)."""
    info = o.intervals_worst_case(q.x1min, q.x1max, net)
    qb, qs = o.make_qc_activs_intvs(net, q.x1min, q.x1max, beta, info)
    xd, K, n1, ac, a = net.xdims, net.K, net.xdims[0], net.acdim, net.Zdim - 1
    s = o.split_sector_gamma(q.gsec, ac, beta)
    p, qq = qs.smin * qs.smax, qs.smin + qs.smax
    d11 = -2.0 * p * s.lam
    c13, c23 = -qs.smin * s.eta - qs.smax * s.nu, s.eta + s.nu
    Tb = o.band_T(s.v, ac, beta)
    pos = {g: i for i, g in enumerate(Ck)}
    n = len(Ck)
    out = np.zeros((n, n))
    off = np.concatenate([[0], np.cumsum(xd[:-1])])
    bias = o.makeb(net)
    S11, S12, S13, S22, S23, S33 = o.out_S_blocks(q.qc_out, net, q.gout)

    def loc(idx):
        return np.array([pos.get(int(g), -1) for g in idx])

    def Mcoef(j, c):  # M = diag(q lam) + T
        t = abs(j - c)
        if t > beta:
            return 0.0
        v = Tb[t, min(j, c)]
        return v + (qq[j] * s.lam[j] if t == 0 else 0.0)

    aff = np.zeros(net.Zdim)
    aff[:n1] += q.gin * (q.x1min + q.x1max) + S12 @ net.Ms[K - 1][:, -1] + S13
    aff[n1:a] += q.gbnd * (qb.acymin + qb.acymax) + c23
    aff[a] += -2.0 * np.sum(q.gin * q.x1min * q.x1max) - 2.0 * np.sum(q.gbnd * qb.acymin * qb.acymax)
    for j in range(ac):
        for c in range(max(0, j - beta), min(ac, j + beta + 1)):
            aff[n1 + c] += bias[j] * Mcoef(j, c)
    for k in range(1, K):  # W_k: block k-1 (0-based) -> neurons of layer k
        W, bk = net.Ms[k - 1][:, :-1], net.Ms[k - 1][:, -1]
        j0 = off[k] - n1
        rows = np.arange(off[k - 1], off[k - 1] + xd[k - 1])
        dj = d11[j0:j0 + xd[k]]
        u = dj * bk + c13[j0:j0 + xd[k]]
        aff[rows] += W.T @ u
        aff[a] += np.sum(dj * bk * bk) + 2.0 * np.sum(bk * c13[j0:j0 + xd[k]])
        lr = loc(rows)
        sel = lr >= 0
        if np.any(sel):
            lrs, Ws = lr[sel], W[:, sel]
            if np.any(dj != 0):
                out[np.ix_(lrs, lrs)] += Ws.T @ (dj[:, None] * Ws)
            for jl in range(xd[k]):
                j = j0 + jl
                for c in range(max(0, j - beta), min(ac, j + beta + 1)):
                    lc = pos.get(n1 + c, -1)
                    if lc >= 0:
                        m = Mcoef(j, c)
                        out[lrs, lc] += Ws[jl] * m
                        out[lc, lrs] += Ws[jl] * m
    for j in range(ac):
        lj = pos.get(n1 + j, -1)
        if lj < 0:
            continue
        out[lj, lj] += -2.0 * q.gbnd[j]
        for c in range(max(0, j - beta), min(ac, j + beta + 1)):
            lc = pos.get(n1 + c, -1)
            if lc >= 0:
                out[lj, lc] += -2.0 * Tb[abs(j - c), min(j, c)]
    WK, bK = net.Ms[K - 1][:, :-1], net.Ms[K - 1][:, -1]
    rK = np.arange(off[K - 1], off[K - 1] + xd[K - 1])
    aff[rK] += WK.T @ (S22 @ bK + S23)
    aff[a] += bK @ S22 @ bK + 2.0 * (bK @ S23) + S33
    lK, l1 = loc(rK), loc(np.arange(n1))
    sK, s1 = lK >= 0, l1 >= 0
    out[np.ix_(lK[sK], lK[sK])] += (WK.T @ S22 @ WK)[np.ix_(sK, sK)]
    out[np.ix_(l1[s1], l1[s1])] += (S11 - 2.0 * np.diag(q.gin))[np.ix_(s1, s1)]
    t = (S12 @ WK)[np.ix_(s1, sK)]
    out[np.ix_(l1[s1], lK[sK])] += t
    out[np.ix_(lK[sK], l1[s1])] += t.T
    la = pos[a]
    out[:, la] = aff[Ck]
    out[la, :] = aff[Ck]
    return out


# ---------------------------------------------------------------------------------------------
# sparse host gather (nnsdp_batch_run_ex): wide layers, so dense cells travel by strided DMA, thin
# entries packed, the rest zero-filled on the host
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["hplaneS", "ellipsoid"])
def test_sparse_host_gather_matches_dense_copy(ctx, kind):
    import nnsdp_b200 as nb

    xdims, beta, nq = [2, 300, 280, 320, 290, 2], 2, 5
    net = rand_net(xdims, seed=31, sigma=0.08)
    rng = np.random.default_rng(4)
    # radius 0 -> every layer Gram-active; large radius -> none; mixed in one batch
    qs = [rand_query(net, beta, rng, kind=kind, radius=r) for r in (0.0, 0.4, 1e-4, 0.05, 0.0)]
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    b = nb.Batch(dnet, beta, Qcap=nq, ring=3)      # odd ring: chunks of 1 query, staging buffers wrap
    b.set_inputs(to_numeric_batch(nb, net, qs))
    dense = np.full((nq, b.per_query), np.nan)
    b.run(dense, flags=nb.RUN_DENSE_COPY)
    assert not b.gather_stats()["sparse"] or b.gather_stats()["zeroed_bytes"] == 0
    sparse = np.full((nq, b.per_query), np.nan)     # garbage everywhere: every entry must be written
    b.run(sparse)
    st = b.gather_stats()
    assert st["sparse"] and st["zeroed_bytes"] > 0 and st["thin_bytes"] > 0
    assert st["dma_bytes"] < 0.8 * dense.nbytes
    assert np.array_equal(dense, sparse)
    pre = np.zeros((nq, b.per_query))               # structural zeros already in place
    pre[:, :] = 0.0
    # non-structural entries hold garbage: only ZERO tiles are promised to be zero
    tiles = nb.plan_tiles(xdims, beta)
    sz = dnet.sizes(beta)
    cl = dnet.cliques(beta)
    offs = np.concatenate([[0], np.cumsum([len(c[0]) ** 2 for c in cl])])
    mask = np.ones(b.per_query, dtype=bool)         # True = may hold garbage
    for t in tiles[tiles[:, 10] == 0]:
        n = len(cl[t[0]][0])
        blk = mask[offs[t[0]]:offs[t[0] + 1]].reshape(n, n)          # [col, row] view of the column-major block
        blk[t[3]:t[3] + t[4], t[1]:t[1] + t[2]] = False
    pre[:, mask] = np.nan
    b.run(pre, flags=nb.RUN_HOST_PREZEROED)
    st2 = b.gather_stats()
    assert st2["zeroed_bytes"] < st["zeroed_bytes"]
    assert np.array_equal(dense, pre)
    # and against the oracle
    cliques = o.make_cliques(net, beta)
    ref = o.run_query(net, beta, qs[0], form="closed")
    for blk, rb in zip(nb.split_blocks(sparse[0], cliques), ref["blocks"]):
        assert relerr(blk, rb) <= TOL
    assert sz["sum_ck_sq"] == b.per_query
    b.close()


def test_sparse_host_gather_dense_Z(ctx):
    """The same gather on the whole-Z output (one matrix, every block pair a cell)."""
    import nnsdp_b200 as nb

    xdims, beta, nq = [3, 270, 300, 260, 3], 1, 3
    net = rand_net(xdims, seed=8, sigma=0.08)
    rng = np.random.default_rng(9)
    qs = [rand_query(net, beta, rng, kind="circle", radius=r) for r in (0.0, 0.3, 1e-3)]
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    b = nb.Batch(dnet, beta, Qcap=nq, ring=2, dense=True)
    b.set_inputs(to_numeric_batch(nb, net, qs))
    a = np.full((nq, b.per_query), np.nan)
    c = np.full((nq, b.per_query), np.nan)
    b.run(a, flags=nb.RUN_DENSE_COPY)
    b.run(c)
    assert b.gather_stats()["sparse"]
    assert np.array_equal(a, c)
    Z = c[1].reshape(sum(xdims[:-1]) + 1, -1).T
    assert relerr(Z, o.run_query(net, beta, qs[1], form="closed")["Z"]) <= TOL
    b.close()


# ---------------------------------------------------------------------------------------------
# affine-coefficient mode (SURVEY.md 8f-1): Z(gamma) = Z0 + sum_v gamma_v Z_v as COO over the cover
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["safety", "hplane", "ellipsoid"])
@pytest.mark.parametrize("xdims,beta", [([2, 3, 2], 0), ([2, 3, 3, 2], 1), ([3, 3, 3, 3, 4, 3, 3], 2), ([2, 4, 7, 3, 5, 2], 5),
                                        ([2, 6, 5, 7, 4, 2], 2)])
def test_affine_form_against_oracle(ctx, xdims, beta, kind):
    import nnsdp_b200 as nb

    net = rand_net(xdims, seed=5, sigma=0.5)
    rng = np.random.default_rng(12)
    for radius in (0.0, 0.3):
        q = rand_query(net, beta, rng, kind=kind, radius=radius)
        dnet = nb.Net(ctx, net.xdims, net.Ms)
        batch = to_numeric_batch(nb, net, [q])
        A = nb.affine_form(dnet, beta, batch)
        Z0, Zv = o.affine_structure(net, beta, q.x1min, q.x1max, q.qc_out)
        cliques = o.make_cliques(net, beta)
        er, ec = o.cover_upper_entries(net, cliques)
        assert A["nent"] == len(er) and np.array_equal(A["ent_row"], er) and np.array_equal(A["ent_col"], ec)
        assert A["nvar"] == len(Zv)
        n1, ac = net.xdims[0], net.acdim
        assert A["var_out"] == n1 and A["var_sec"] - A["var_bnd"] == ac
        assert A["var_bnd"] - A["var_out"] == (0 if kind == "safety" else 1)
        scale = max(np.abs(Z0).max(), max(np.abs(z).max() for z in Zv), 1.0)
        # constant part
        assert np.abs(A["z0"] - Z0[er - 1, ec - 1]).max() <= TOL * scale
        # per-variable coefficient matrices (duplicates summed)
        dense = np.zeros((A["nvar"], A["nent"]))
        np.add.at(dense, (A["coo_var"] - 1, A["coo_ent"] - 1), A["coo_val"])
        for v in range(A["nvar"]):
            ref = Zv[v][er - 1, ec - 1]
            assert np.abs(dense[v] - ref).max() <= TOL * scale, (v, np.abs(dense[v] - ref).max())
            # nothing of Z_v lives outside the cover
            mask = np.zeros_like(Zv[v], dtype=bool)
            mask[er - 1, ec - 1] = True
            mask |= mask.T
            assert not np.any((Zv[v] != 0) & ~mask)
        # Z(gamma) from the affine form == the numeric device path at a random gamma
        g = np.concatenate([q.gin, q.gout if kind != "safety" else [], q.gbnd, q.gsec])
        zg = A["z0"] + g @ dense
        Znum = nb.assemble_dense(dnet, beta, batch)[0]
        assert np.abs(zg - Znum[er - 1, ec - 1]).max() <= TOL * max(np.abs(Znum).max(), 1.0)


def test_affine_form_mid_size_and_limit(ctx):
    """W = 40, D = 6: the Gram term dominates nnz; max_nnz is enforced."""
    import nnsdp_b200 as nb

    xdims, beta = [2] + [40] * 6 + [2], 2
    net = rand_net(xdims, seed=2, sigma=0.3)
    rng = np.random.default_rng(1)
    q = rand_query(net, beta, rng, kind="hplane", radius=0.0)   # every neuron stable: p_j in {0, 1}
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    batch = to_numeric_batch(nb, net, [q])
    A = nb.affine_form(dnet, beta, batch)
    info = o.intervals_worst_case(q.x1min, q.x1max, net)
    smin, smax = o.make_sector_min_max(np.concatenate([p[0] for p in info.acx_intvs]), np.concatenate([p[1] for p in info.acx_intvs]))
    nact = int((smin * smax != 0).sum())
    assert A["nnz"] >= nact * (40 * 41 // 2) or nact == 0
    g = np.concatenate([q.gin, q.gout, q.gbnd, q.gsec])
    zg = A["z0"].copy()
    np.add.at(zg, A["coo_ent"] - 1, A["coo_val"] * g[A["coo_var"] - 1])
    Znum = nb.assemble_dense(dnet, beta, batch)[0]
    assert np.abs(zg - Znum[A["ent_row"] - 1, A["ent_col"] - 1]).max() <= TOL * max(np.abs(Znum).max(), 1.0)
    with pytest.raises(nb.NnsdpError) as e:
        nb.affine_form(dnet, beta, batch, max_nnz=10)
    assert e.value.code == -3


# ---------------------------------------------------------------------------------------------
# wide layers (128-row tiles, strips, RC / CR window programs, sliver sub-tiles) x output kinds x beta
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["safety", "hplane", "ellipsoid"])
@pytest.mark.parametrize("xdims,beta", [
    ([3, 150, 260, 140, 2], 0), ([3, 150, 260, 140, 2], 1), ([3, 150, 260, 140, 2], 4),
    ([3, 150, 260, 140, 2], 6),            # beta > MAX_WINDOW_BETA: no register-window programs
    ([2, 129, 128, 127, 300, 4], 3),       # widths around the tile size, last block wide
    ([6, 520, 33, 520, 3], 2),             # a narrow layer between wide ones: slivers dominate
])
def test_wide_nets_all_programs(ctx, xdims, beta, kind):
    import nnsdp_b200 as nb

    net = rand_net(xdims, seed=17, sigma=0.1)
    rng = np.random.default_rng(23)
    qs = [rand_query(net, beta, rng, kind=kind, radius=r) for r in (0.0, 0.2)]
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    batch = to_numeric_batch(nb, net, qs)
    Z = nb.assemble_dense(dnet, beta, batch)
    flat = nb.assemble_blocks(dnet, beta, batch)
    cliques = dnet.cliques(beta)
    for i, q in enumerate(qs):
        ref = o.run_query(net, beta, q, form="closed")
        assert relerr(Z[i], ref["Z"]) <= TOL
        assert np.array_equal(Z[i], Z[i].T)
        for blk, (Ck, _, _), rb in zip(nb.split_blocks(flat[i], cliques), cliques, ref["blocks"]):
            assert np.array_equal(blk, Z[i][np.ix_(Ck - 1, Ck - 1)])
            assert relerr(blk, rb) <= TOL


_PANEL_SNIPPET = r"""
import hashlib, os, sys
import numpy as np
root = sys.argv[1]
for p in ("nn-sdp_b200", "oracle", "tests"):
    sys.path.insert(0, os.path.join(root, p))
import nnsdp_b200 as nb
from helpers import rand_net, rand_query, to_numeric_batch
ctx = nb.Context([0])
for xdims, beta in (([2, 300, 270, 280, 2], 2), ([3, 150, 260, 140, 2], 4), ([2, 129, 128, 127, 300, 4], 3)):
    net = rand_net(xdims, seed=3, sigma=0.1)
    rng = np.random.default_rng(5)
    qs = [rand_query(net, beta, rng, kind="ellipsoid", radius=0.004 * i) for i in range(7)]
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    for ring in (3, 7):
        b = nb.Batch(dnet, beta, Qcap=7, ring=ring)
        b.set_inputs(to_numeric_batch(nb, net, qs))
        out = np.full((7, b.per_query), np.nan)
        b.run(out)
        fill, window = b.stage_ms("emit_fill")[1], b.stage_ms("emit_window")[1]
        b.close()
        print(hashlib.sha256(out.tobytes()).hexdigest(), int(np.isnan(out).sum()), fill, window)
"""


def test_panel_ordered_launch_equals_the_separate_kernels(ctx, tmp_path):
    """Dense blocks of wide nets: the fill strips and the window tiles as one panel-ordered launch (the default) and as
    two kernels one after the other (NNSDP_PANEL=0) are the same programs on the same items -- the outputs must agree
    bit for bit, for whole and ragged passes.  The switch is read once per process, hence the two subprocesses."""
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    script = tmp_path / "panel_ab.py"
    script.write_text(_PANEL_SNIPPET)
    outs = {}
    for mode in ("1", "0"):
        env = dict(os.environ, NNSDP_PANEL=mode)
        r = subprocess.run([sys.executable, str(script), root], capture_output=True, text=True, env=env, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        outs[mode] = [ln.split() for ln in r.stdout.strip().splitlines()]
    assert len(outs["1"]) == 6 and len(outs["0"]) == 6
    for a, b_ in zip(outs["1"], outs["0"]):
        assert a[0] == b_[0] and a[1] == b_[1] == "0"          # same bytes, every entry written
        assert int(a[3]) == 0 and int(b_[3]) > 0               # one launch against two: the window span is empty / used


def test_ragged_batches_and_rings(ctx):
    """Q not a multiple of the ring, ring of 1, Q = 1, more ring slots than queries."""
    import nnsdp_b200 as nb

    xdims, beta = [2, 300, 270, 2], 2
    net = rand_net(xdims, seed=3, sigma=0.1)
    rng = np.random.default_rng(5)
    qs = [rand_query(net, beta, rng, kind="circle", radius=0.01 * i) for i in range(7)]
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    cliques = o.make_cliques(net, beta)
    refs = [o.run_query(net, beta, q)["blocks"] for q in qs]
    for nq, ring in ((7, 3), (7, 1), (1, 4), (5, 8), (7, 2)):
        b = nb.Batch(dnet, beta, Qcap=nq, ring=ring)
        b.set_inputs(to_numeric_batch(nb, net, qs[:nq]))
        out = np.full((nq, b.per_query), np.nan)
        b.run(out)
        for i in range(nq):
            for blk, rb in zip(nb.split_blocks(out[i], cliques), refs[i]):
                assert relerr(blk, rb) <= TOL
        b.close()


# ---------------------------------------------------------------------------------------------
# certificate check (SURVEY.md 8f-3): lambda_max(Z) matrix-free against numpy's dense eigvalsh
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["safety", "hplane", "ellipsoid"])
@pytest.mark.parametrize("xdims,beta", [([2, 3, 2], 0), ([3, 3, 3, 3, 4, 3, 3], 2), ([2, 4, 7, 3, 5, 2], 5), ([2] + [20] * 6 + [2], 2),
                                        ([5, 50, 50, 50, 5], 2), ([3, 150, 260, 140, 2], 3)])
def test_lambda_max_matrix_free(ctx, xdims, beta, kind):
    import nnsdp_b200 as nb

    net = rand_net(xdims, seed=4, sigma=0.2)
    rng = np.random.default_rng(6)
    qs = [rand_query(net, beta, rng, kind=kind, radius=r) for r in (0.0, 0.05, 0.4)]
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    b = nb.Batch(dnet, beta, Qcap=3, ring=1)
    b.set_inputs(to_numeric_batch(nb, net, qs))
    b.bounds()
    b.prepare()
    lam, its, resid, conv = b.lambda_max(max_iters=400, tol=1e-10, full=True)
    assert conv.all()
    for i, q in enumerate(qs):
        Z = o.run_query(net, beta, q, form="closed")["Z"]
        ev = np.linalg.eigvalsh(Z)
        scale = max(abs(ev[0]), abs(ev[-1]))
        assert abs(lam[i] - ev[-1]) <= 1e-9 * scale, (lam[i], ev[-1], its[i])
        assert lam[i] <= ev[-1] + 1e-12 * scale           # a Ritz value never exceeds lambda_max
        assert np.abs(ev - lam[i]).min() <= resid[i] + 1e-12 * scale   # an eigenvalue lies within the residual
        assert 1 <= its[i] <= min(400, Z.shape[0])
    b.close()


def test_lambda_max_reports_non_convergence(ctx):
    """Zdim >> max_iters with lambda_max near zero -- the regime of the acceptance gate eigmax(Z) <= 1e-4
    (experiments/acas.jl:76-79): a run that stops at max_iters must say so (converged = 0, NNSDP_ERR_NOCONV from the
    plain call) and its value must be a LOWER bound; with enough iterations the same batch converges."""
    import nnsdp_b200 as nb

    xdims, beta = [2, 300, 300, 2], 1
    net = rand_net(xdims, seed=1, sigma=0.0)       # zero weights: Z is (almost) diagonal, eigenvalues ~ -2 gamma
    rng = np.random.default_rng(0)
    q = rand_query(net, beta, rng, kind="hplane", radius=0.1)
    q.gsec[:] = 0.0
    q.gbnd[:] = rng.uniform(0.5, 2.0, q.gbnd.size)
    q.gbnd[17] = 1e-9                               # lambda_max = -2e-9 against a spectral scale of ~4
    q.qc_out = o.QcReachHplane(np.zeros(2))
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    b = nb.Batch(dnet, beta, Qcap=1, ring=1)
    b.set_inputs(to_numeric_batch(nb, net, [q]))
    b.bounds()
    b.prepare()
    ev = np.linalg.eigvalsh(o.run_query(net, beta, q, form="closed")["Z"])
    scale = max(abs(ev[0]), abs(ev[-1]))
    assert abs(ev[-1]) < 1e-6 * scale
    lam, its, resid, conv = b.lambda_max(max_iters=12, tol=1e-10, full=True)
    assert conv[0] == 0 and its[0] == 12 and resid[0] > 1e-10 * scale
    assert lam[0] <= ev[-1] + 1e-12 * scale and lam[0] < ev[-1] - 1e-6 * scale      # a lower bound, visibly short
    with pytest.raises(nb.NnsdpError) as e:
        b.lambda_max(max_iters=12, tol=1e-10)
    assert e.value.code == -6
    lam, its, resid, conv = b.lambda_max(max_iters=700, tol=1e-10, full=True)
    assert conv[0] == 1 and abs(lam[0] - ev[-1]) <= 1e-9 * scale
    b.close()


def test_lambda_max_negative_definite_certificate(ctx):
    """A Z that is negative definite by construction (only the -2 gamma diagonals): the check returns its
    largest (negative) eigenvalue, i.e. the certificate eigmax(Z) <= 0 of experiments/acas.jl:71-79."""
    import nnsdp_b200 as nb

    xdims, beta = [2, 30, 30, 2], 1
    net = rand_net(xdims, seed=1, sigma=0.0)       # zero weights and biases: no coupling at all
    rng = np.random.default_rng(0)
    q = rand_query(net, beta, rng, kind="hplane", radius=0.1)
    q.gsec[:] = 0.0
    q.qc_out = o.QcReachHplane(np.zeros(2))
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    b = nb.Batch(dnet, beta, Qcap=1, ring=1)
    b.set_inputs(to_numeric_batch(nb, net, [q]))
    b.bounds()
    b.prepare()
    lam, _ = b.lambda_max(max_iters=100, tol=1e-10)
    Z = o.run_query(net, beta, q, form="closed")["Z"]
    ev = np.linalg.eigvalsh(Z)
    assert ev[-1] < 0 and abs(lam[0] - ev[-1]) <= 1e-9 * abs(ev[0])
    b.close()


def test_multi_device_context_shards_queries(ctx):
    """One nnsdp_ctx over two devices: queries are split in contiguous ranges, one host thread per device, and
    gathered into the caller's buffer (SURVEY.md 8e, second form).  Needs >= 2 GPUs."""
    import nnsdp_b200 as nb

    if nb.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    xdims, beta, nq = [2, 300, 270, 2], 2, 7
    net = rand_net(xdims, seed=3, sigma=0.1)
    rng = np.random.default_rng(5)
    qs = [rand_query(net, beta, rng, kind="ellipsoid", radius=0.02 * i) for i in range(nq)]
    batch = to_numeric_batch(nb, net, qs)
    one = nb.assemble_blocks(nb.Net(ctx, net.xdims, net.Ms), beta, batch)
    ctx2 = nb.Context([0, 1])
    dnet2 = nb.Net(ctx2, net.xdims, net.Ms)
    two = nb.assemble_blocks(dnet2, beta, batch)
    assert np.array_equal(one, two)
    r1 = nb.bounds_ibp(nb.Net(ctx, net.xdims, net.Ms), np.stack([q.x1min for q in qs]), np.stack([q.x1max for q in qs]))
    r2 = nb.bounds_ibp(dnet2, np.stack([q.x1min for q in qs]), np.stack([q.x1max for q in qs]))
    assert all(np.array_equal(r1[k], r2[k]) for k in r1)


# ---------------------------------------------------------------------------------------------
# CROWN bounds (SURVEY.md 8f-2): the reference's default IntervalsAutoLirpa, sliced variant
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("xdims", [[2, 3, 2], [2, 6, 5, 7, 2], [2] + [10] * 10 + [2], [5, 50, 50, 50, 50, 50, 50, 5],
                                   [2] + [20] * 10 + [2], [3, 150, 260, 140, 2], [2, 4, 7, 3, 5, 2],
                                   [3, 131, 257, 193, 129, 2]])   # odd widths >= 192 x 128: every edge of the tensor-core GEMM tiles
def test_crown_bounds_against_oracle(ctx, xdims):
    import nnsdp_b200 as nb

    net = rand_net(xdims, seed=8)
    rng = np.random.default_rng(3)
    n1 = xdims[0]
    centres = rng.uniform(0.5, 1.5, (5, n1))
    radii = np.array([0.0, 1e-3, 0.05, 0.2, 0.5])[:, None]
    lo, hi = centres - radii, centres + radii
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    r = nb.bounds_crown(dnet, lo, hi)
    ibp = nb.bounds_ibp(dnet, lo, hi)
    for i in range(5):
        ref = o.intervals_crown(lo[i], hi[i], net)
        xmin = np.concatenate([p[0] for p in ref.x_intvs])
        xmax = np.concatenate([p[1] for p in ref.x_intvs])
        amin = np.concatenate([p[0] for p in ref.acx_intvs])
        amax = np.concatenate([p[1] for p in ref.acx_intvs])
        scale = max(np.abs(xmin).max(), np.abs(xmax).max(), 1.0)
        for got, want in ((r["xmin"][i], xmin), (r["xmax"][i], xmax), (r["acxmin"][i], amin), (r["acxmax"][i], amax)):
            assert np.abs(got - want).max() <= 1e-11 * scale
        assert np.all(r["xmin"][i] <= r["xmax"][i]) and np.all(r["acxmin"][i] <= r["acxmax"][i])
        # the first hidden layer is interval arithmetic in both methods
        n2 = xdims[1]
        assert np.abs(r["acxmin"][i][:n2] - ibp["acxmin"][i][:n2]).max() <= TOL * scale
        # soundness: sampled activations lie inside the bounds
        for _ in range(50):
            x = rng.uniform(lo[i], hi[i])
            xs = [x]
            for k, M in enumerate(net.Ms):
                y = M @ np.append(xs[-1], 1.0)
                xs.append(np.maximum(y, 0.0) if k < net.K - 1 else y)
            allx = np.concatenate(xs)
            assert np.all(allx >= r["xmin"][i] - 1e-9 * scale) and np.all(allx <= r["xmax"][i] + 1e-9 * scale)


@pytest.mark.parametrize("name", ["scale_W10_D10", "scale_W5_D5", "rand_acas_5x50", "rand_ragged"])
def test_crown_bounds_against_the_vendored_auto_lirpa(ctx, name):
    """The device CROWN against x_intvs computed by the reference's vendored auto_LiRPA itself
    (tests/golden/crown_autolirpa.npz, generator tests/golden/make_crown_golden.py): float64 run to 1e-11, float32
    run (what the reference executes) to float32 rounding."""
    import nnsdp_b200 as nb

    d = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "crown_autolirpa.npz"))
    xd = d[f"{name}.xdims"].tolist()
    Ms = [d[f"{name}.M{k}"] for k in range(len(xd) - 1)]
    dnet = nb.Net(ctx, xd, Ms)
    r = nb.bounds_crown(dnet, d[f"{name}.x1min"][None, :], d[f"{name}.x1max"][None, :])
    scale = max(np.abs(d[f"{name}.f64.lo"]).max(), np.abs(d[f"{name}.f64.hi"]).max())
    assert np.abs(r["xmin"][0] - d[f"{name}.f64.lo"]).max() <= 1e-11 * scale
    assert np.abs(r["xmax"][0] - d[f"{name}.f64.hi"]).max() <= 1e-11 * scale
    assert np.abs(r["xmin"][0] - d[f"{name}.f32.lo"]).max() <= 2e-6 * scale
    assert np.abs(r["xmax"][0] - d[f"{name}.f32.hi"]).max() <= 2e-6 * scale


def test_crown_in_the_batch_pipeline(ctx):
    """Blocks assembled with CROWN bounds computed on the device == blocks from the oracle with the oracle's
    CROWN intervals (makeQcActivsIntvs with the default method, src/Qc/activ.jl:45-67)."""
    import nnsdp_b200 as nb

    xdims, beta = [2] + [12] * 8 + [2], 2
    net = rand_net(xdims, seed=6)
    rng = np.random.default_rng(2)
    qs = [rand_query(net, beta, rng, kind="hplane", radius=r) for r in (0.02, 0.3)]
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    b = nb.Batch(dnet, beta, Qcap=2, ring=2)
    b.set_inputs(to_numeric_batch(nb, net, qs))
    b.set_bounds_method("crown")
    out = np.empty((2, b.per_query))
    b.run(out)
    cliques = o.make_cliques(net, beta)
    tighter = 0
    for i, q in enumerate(qs):
        info = o.intervals_crown(q.x1min, q.x1max, net)
        ref = o.run_query(net, beta, q, intv_info=info)
        for blk, rb in zip(nb.split_blocks(out[i], cliques), ref["blocks"]):
            assert relerr(blk, rb) <= 1e-11
        ibp = o.intervals_worst_case(q.x1min, q.x1max, net)
        tighter += sum((p[1] - p[0]).sum() for p in ibp.x_intvs) > sum((p[1] - p[0]).sum() for p in info.x_intvs)
    assert tighter == 2
    b.close()


def test_reach_batch_shares_the_gram_blocks(ctx):
    """A reach batch on a wide net (shared box and multipliers, per-direction normal and gamma_out): the Gram
    contraction runs once for the whole batch (src/NnSdp.jl:73-95 builds qc_input / qc_activs once)."""
    import nnsdp_b200 as nb

    xdims, beta, nq = [2, 150, 260, 140, 2], 2, 6
    net = rand_net(xdims, seed=9, sigma=0.3)
    rng = np.random.default_rng(2)
    base = rand_query(net, beta, rng, kind="hplane", radius=0.0)     # degenerate box: every layer Gram-active
    th = 2 * np.pi * np.arange(nq) / nq
    normals = np.stack([np.cos(th), np.sin(th)], axis=1)
    gouts = rng.random((nq, 1))
    batch = nb.NumericBatch(x1min=base.x1min, x1max=base.x1max, gamma_in=base.gin, gamma_bnd=base.gbnd,
                            gamma_sec=base.gsec, out_kind=nb.OUT_HPLANE, out_vec=normals, gamma_out=gouts)
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    b = nb.Batch(dnet, beta, Qcap=nq, ring=4)
    b.set_inputs(batch, Q=nq)
    out = np.full((nq, b.per_query), np.nan)
    b.run(out)
    ms, launches = b.stage_ms("gram")
    assert launches == 1                      # one contraction for 6 queries in 3 chunks
    ncon, nact = b.gram_stats()
    assert ncon == nq * (len(xdims) - 2)
    cliques = o.make_cliques(net, beta)
    for i in range(nq):
        q = o.NumericQuery(base.x1min, base.x1max, base.gin, base.gbnd, base.gsec, o.QcReachHplane(normals[i]), gouts[i])
        ref = o.run_query(net, beta, q)
        for blk, rb in zip(nb.split_blocks(out[i], cliques), ref["blocks"]):
            assert relerr(blk, rb) <= TOL
    b.close()


def test_crown_and_lambda_max_over_several_chunks(ctx):
    """More queries than one internal chunk holds (CROWN: 256, lambda_max: 64)."""
    import nnsdp_b200 as nb

    xdims, beta, Q = [2, 8, 9, 7, 2], 1, 300
    net = rand_net(xdims, seed=12)
    rng = np.random.default_rng(1)
    c = rng.uniform(0.5, 1.5, (Q, 2))
    rad = rng.uniform(0.0, 0.3, (Q, 1))
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    r = nb.bounds_crown(dnet, c - rad, c + rad)
    for i in (0, 127, 255, 256, 257, 299):
        ref = o.intervals_crown(c[i] - rad[i], c[i] + rad[i], net)
        xmin = np.concatenate([p[0] for p in ref.x_intvs])
        xmax = np.concatenate([p[1] for p in ref.x_intvs])
        scale = max(np.abs(xmax).max(), 1.0)
        assert np.abs(r["xmin"][i] - xmin).max() <= 1e-11 * scale and np.abs(r["xmax"][i] - xmax).max() <= 1e-11 * scale
    qs = [rand_query(net, beta, rng, kind="circle", radius=0.1) for _ in range(70)]
    b = nb.Batch(dnet, beta, Qcap=70, ring=1)
    b.set_inputs(to_numeric_batch(nb, net, qs))
    b.bounds()
    b.prepare()
    lam, its = b.lambda_max(max_iters=100, tol=1e-10)
    for i in (0, 63, 64, 69):
        ev = np.linalg.eigvalsh(o.run_query(net, beta, qs[i])["Z"])
        assert abs(lam[i] - ev[-1]) <= 1e-9 * max(abs(ev[0]), abs(ev[-1]))
    b.close()


# ---------------------------------------------------------------------------------------------
# randomised shapes around every threshold of the planner (block split at 48, tiles of 128 x 32, strips of 512,
# gather cells of 256, window programs up to beta = 4, fast band up to beta = 8)
# ---------------------------------------------------------------------------------------------
def _random_shapes():
    rng = np.random.default_rng(20241018)
    pool = [3, 7, 31, 33, 47, 48, 49, 63, 64, 65, 127, 128, 129, 200, 255, 256, 257, 300, 511, 513]
    shapes = []
    for i in range(24):
        depth = int(rng.integers(1, 5))
        hidden = [int(rng.choice(pool if i % 3 else pool[:12])) for _ in range(depth)]
        if sum(h * h for h in hidden) > 600_000:      # keep the oracle's dense Z small
            hidden = [min(h, 300) for h in hidden]
        xd = [int(rng.integers(1, 7))] + hidden + [int(rng.integers(1, 6))]
        beta = int(rng.choice([0, 1, 2, 3, 4, 5, 8, 9]))
        beta = min(beta, sum(hidden))
        kind = ["safety", "hplane", "circle", "ellipsoid", "hplaneS"][i % 5]
        shapes.append((xd, beta, kind))
    return shapes


@pytest.mark.parametrize("xdims,beta,kind", _random_shapes())
def test_random_shapes_around_planner_thresholds(ctx, xdims, beta, kind):
    import nnsdp_b200 as nb

    net = rand_net(xdims, seed=sum(xdims) + beta, sigma=0.15)
    rng = np.random.default_rng(beta + 7)
    qs = [rand_query(net, beta, rng, kind=kind, radius=r) for r in (0.0, 0.25)]
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    batch = to_numeric_batch(nb, net, qs)
    b = nb.Batch(dnet, beta, Qcap=2, ring=2)
    b.set_inputs(batch)
    out = np.full((2, b.per_query), np.nan)
    b.run(out)                                   # sparse gather where the net is wide enough
    Zd = nb.assemble_dense(dnet, beta, batch)
    cliques = dnet.cliques(beta)
    refc = o.make_cliques(net, beta)
    assert len(cliques) == len(refc) and all(np.array_equal(a[0], r[0]) for a, r in zip(cliques, refc))
    for i, q in enumerate(qs):
        ref = o.run_query(net, beta, q, form="closed")
        assert relerr(Zd[i], ref["Z"]) <= TOL
        assert np.array_equal(Zd[i], Zd[i].T)
        for blk, (Ck, _, _) in zip(nb.split_blocks(out[i], cliques), cliques):
            assert np.array_equal(blk, Zd[i][np.ix_(Ck - 1, Ck - 1)])
    lam, _, _, _ = b.lambda_max(max_iters=300, tol=1e-10, full=True)
    ev = np.linalg.eigvalsh(o.run_query(net, beta, qs[1], form="closed")["Z"])
    assert abs(lam[1] - ev[-1]) <= 1e-8 * max(abs(ev[0]), abs(ev[-1]))
    b.close()


@pytest.mark.parametrize("xdims,beta", [([3, 65, 49, 2], 2), ([4, 127, 48, 3], 3), ([2, 63, 63, 64, 4], 4), ([5, 47, 3, 3, 4], 3)])
def test_affine_form_and_crown_on_mid_shapes(ctx, xdims, beta):
    """Affine form: Z(gamma) rebuilt from the COO triplets == the numeric device path at a random gamma (no
    oracle needed at these sizes); CROWN == the oracle's restatement."""
    import nnsdp_b200 as nb

    net = rand_net(xdims, seed=3, sigma=0.2)
    rng = np.random.default_rng(4)
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    for kind, radius in (("ellipsoid", 0.0), ("safety", 0.2)):
        q = rand_query(net, beta, rng, kind=kind, radius=radius)
        batch = to_numeric_batch(nb, net, [q])
        A = nb.affine_form(dnet, beta, batch)
        g = np.concatenate([q.gin, q.gout if kind != "safety" else [], q.gbnd, q.gsec])
        zg = A["z0"].copy()
        np.add.at(zg, A["coo_ent"] - 1, A["coo_val"] * g[A["coo_var"] - 1])
        Z = nb.assemble_dense(dnet, beta, batch)[0]
        assert np.abs(zg - Z[A["ent_row"] - 1, A["ent_col"] - 1]).max() <= TOL * max(np.abs(Z).max(), 1.0)
        # nothing of Z lies outside the entries the affine form lists
        mask = np.zeros_like(Z, dtype=bool)
        mask[A["ent_row"] - 1, A["ent_col"] - 1] = True
        assert not np.any((Z != 0) & ~(mask | mask.T))
        r = nb.bounds_crown(dnet, q.x1min[None], q.x1max[None])
        ref = o.intervals_crown(q.x1min, q.x1max, net)
        xmax = np.concatenate([p[1] for p in ref.x_intvs])
        assert np.abs(r["xmax"][0] - xmax).max() <= 1e-11 * max(np.abs(xmax).max(), 1.0)


def test_crown_wavefront_deep_narrow_net(ctx):
    """K >= 16 and widths <= 64: the post-activation targets are bounded as one stack (wavefront); same numbers
    as the oracle's one-target-at-a-time restatement."""
    import nnsdp_b200 as nb

    xdims = [3] + [9, 12, 7, 10] * 5 + [2]      # K = 21, ragged widths
    net = rand_net(xdims, seed=21)
    rng = np.random.default_rng(5)
    c = rng.uniform(0.5, 1.5, (3, 3))
    rad = np.array([[0.0], [0.02], [0.3]])
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    r = nb.bounds_crown(dnet, c - rad, c + rad)
    for i in range(3):
        ref = o.intervals_crown(c[i] - rad[i], c[i] + rad[i], net)
        xmin = np.concatenate([p[0] for p in ref.x_intvs])
        xmax = np.concatenate([p[1] for p in ref.x_intvs])
        amax = np.concatenate([p[1] for p in ref.acx_intvs])
        scale = max(np.abs(xmax).max(), np.abs(xmin).max(), 1.0)
        assert np.abs(r["xmin"][i] - xmin).max() <= 1e-11 * scale
        assert np.abs(r["xmax"][i] - xmax).max() <= 1e-11 * scale
        assert np.abs(r["acxmax"][i] - amax).max() <= 1e-11 * scale


# ---------------------------------------------------------------------------------------------
# Few-query paths: one cooperative kernel for the interval propagation (Q <= 8), cluster split-K GEMVs per layer
# (Q <= 32), every affine-column GEMV in one launch, and the tiled GEMM beyond.  Same numbers on every path.
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nq", [1, 2, 3, 4, 5, 8, 9, 17, 32, 33])
def test_query_count_thresholds_of_the_bounds_and_affine_kernels(ctx, nq):
    import nnsdp_b200 as nb

    xdims, beta = [3, 70, 131, 9, 64, 257, 4], 2    # widths around the 8/16/64-row tiles, one narrow layer
    net = rand_net(xdims, seed=21, sigma=0.3)
    rng = np.random.default_rng(nq)
    qs = [rand_query(net, beta, rng, kind="hplane", radius=0.02 * (1 + i % 4)) for i in range(nq)]
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    b = nb.Batch(dnet, beta, Qcap=nq, ring=min(nq, 4))
    b.set_inputs(to_numeric_batch(nb, net, qs))
    out = np.full((nq, b.per_query), np.nan)
    b.run(out)
    bd = b.get_bounds()
    aff = b.get_affine()
    cliques = o.make_cliques(net, beta)
    for i in (0, nq // 2, nq - 1):
        _, xmin, xmax, amin, amax = _oracle_bounds(net, qs[i])
        scale = max(np.abs(xmax).max(), np.abs(xmin).max(), 1.0)
        assert np.abs(bd["xmin"][i] - xmin).max() <= TOL * scale
        assert np.abs(bd["xmax"][i] - xmax).max() <= TOL * scale
        assert np.abs(bd["acxmin"][i] - amin).max() <= TOL * scale
        assert np.abs(bd["acxmax"][i] - amax).max() <= TOL * scale
        rmin, rmax = o.make_sector_min_max(bd["acxmin"][i], bd["acxmax"][i])
        assert np.array_equal(bd["smin"][i], rmin) and np.array_equal(bd["smax"][i], rmax)
        ref = o.run_query(net, beta, qs[i])
        assert relerr(aff[i], ref["Z"][:, -1]) <= TOL
        for blk, rb in zip(nb.split_blocks(out[i], cliques), ref["blocks"]):
            assert relerr(blk, rb) <= TOL
    # a query's numbers do not depend on how many share the launch (within one path)
    if nq in (2, 5, 8):
        b1 = nb.Batch(dnet, beta, Qcap=1, ring=1)
        b1.set_inputs(to_numeric_batch(nb, net, qs[nq - 1:nq]))
        o1 = np.empty((1, b.per_query))
        b1.run(o1)
        assert np.array_equal(o1[0], out[nq - 1])
        b1.close()
    b.close()


@pytest.mark.parametrize("xdims,nq", [([2, 300, 260, 200, 2], 160), ([4, 194, 256, 131, 320, 3], 129),
                                      ([2, 256, 250, 256, 2], 200),
                                      ([2, 960, 1000, 2], 512),     # 64-neuron tiles (the three above: 32-neuron tiles)
                                      ([2, 640, 768, 2], 1536)])    # 64-neuron tiles, 24 column tiles
def test_many_queries_on_wide_layers_use_the_tensor_core_bounds_and_affine_paths(ctx, xdims, nq):
    """Q >= 128 on layers of >= 192 neurons: interval propagation as the two-accumulator FP64 tensor-core kernel
    (centre / radius form of intervals_easy.jl:23-24) and the affine-column products of all layers in one launch.
    Same bounds, sector slopes, affine column and blocks as the oracle; odd widths fall back layer by layer."""
    import nnsdp_b200 as nb

    beta = 2
    net = rand_net(xdims, seed=31, sigma=0.15)
    rng = np.random.default_rng(nq)
    qs = [rand_query(net, beta, rng, kind="safety", radius=0.01 * (1 + i % 5)) for i in range(nq)]
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    b = nb.Batch(dnet, beta, Qcap=nq, ring=4)
    b.set_inputs(to_numeric_batch(nb, net, qs))
    b.bounds()
    b.prepare()
    bd = b.get_bounds()
    aff = b.get_affine()
    for i in (0, 1, nq // 2, nq - 2, nq - 1):
        _, xmin, xmax, amin, amax = _oracle_bounds(net, qs[i])
        scale = max(np.abs(xmax).max(), np.abs(xmin).max(), 1.0)
        assert np.abs(bd["xmin"][i] - xmin).max() <= TOL * scale
        assert np.abs(bd["xmax"][i] - xmax).max() <= TOL * scale
        assert np.abs(bd["acxmin"][i] - amin).max() <= TOL * scale
        assert np.abs(bd["acxmax"][i] - amax).max() <= TOL * scale
        rmin, rmax = o.make_sector_min_max(bd["acxmin"][i], bd["acxmax"][i])
        assert np.array_equal(bd["smin"][i], rmin) and np.array_equal(bd["smax"][i], rmax)
        ref = o.run_query(net, beta, qs[i])
        assert relerr(aff[i], ref["Z"][:, -1]) <= TOL
    # the same queries a few at a time (GEMV paths): same numbers to rounding
    b8 = nb.Batch(dnet, beta, Qcap=8, ring=4)
    b8.set_inputs(to_numeric_batch(nb, net, qs[:8]))
    b8.bounds()
    b8.prepare()
    bd8, aff8 = b8.get_bounds(), b8.get_affine()
    for key in ("xmin", "xmax", "acxmin", "acxmax"):
        scale = max(np.abs(bd8[key]).max(), 1.0)
        assert np.abs(bd8[key] - bd[key][:8]).max() <= 1e-13 * scale
    assert np.array_equal(bd8["smin"], bd["smin"][:8]) and np.array_equal(bd8["smax"], bd["smax"][:8])
    assert np.abs(aff8 - aff[:8]).max() <= 1e-12 * max(np.abs(aff8).max(), 1.0)
    b.close()
    b8.close()


def test_recorded_optimum_minimiser_through_the_device_pipeline(ctx):
    """The reference's scale experiment on its shipped W10-D10 net (experiments/scale.jl: box [0.5, 1.5]^2,
    findEllipsoid), at the minimiser gamma* stored by oracle/sdp_crosscheck.py: the device pipeline -- CROWN bounds,
    QC data, blocks, matrix-free lambda_max -- must give the oracle's Z(gamma*) and its certificate value
    lambda_max(Z(gamma*)) ~ 0^- (the LMI is active at an optimum), for beta = 0, 2, 5."""
    import json
    import sys

    import nnsdp_b200 as nb

    gold = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    sys.path.insert(0, os.path.join(os.path.dirname(gold), "..", "oracle"))
    res = json.load(open(os.path.join(gold, "scale_W10_D10_optimum.json")))
    net = o.load_nnet(os.path.join(gold, "scale-I2-O2-W10-D10.nnet"))
    x1min, x1max = np.full(2, 0.5), np.full(2, 1.5)
    P, yc = np.asarray(res["P"]), np.asarray(res["yc"])
    invP = np.linalg.inv(P)
    invP = 0.5 * (invP + invP.T)
    info = o.intervals_crown(x1min, x1max, net)
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    n1, ac = net.xdims[0], net.acdim
    for beta in (0, 2, 5):
        g = np.asarray(res["oracle_optimum"][str(beta)]["gamma"])
        q = o.NumericQuery(x1min=x1min, x1max=x1max, qc_out=o.QcReachEllipsoid(invP=invP, yc=yc), gin=g[:n1],
                           gout=g[n1:n1 + 1], gbnd=g[n1 + 1:n1 + 1 + ac], gsec=g[n1 + 1 + ac:])
        ref = o.run_query(net, beta, q, intv_info=info)
        b = nb.Batch(dnet, beta, Qcap=1, ring=1)
        b.set_inputs(to_numeric_batch(nb, net, [q]))
        b.set_bounds_method("crown")
        out = np.empty((1, b.per_query))
        b.run(out)
        for blk, rb in zip(nb.split_blocks(out[0], ref["cliques"]), ref["blocks"]):
            assert relerr(blk, rb) <= 1e-10        # multipliers span 1e-9 .. 1e4: normwise per block
        lam, its = b.lambda_max(max_iters=400, tol=1e-10)
        want = np.linalg.eigvalsh(0.5 * (ref["Z"] + ref["Z"].T)).max()
        scale = np.abs(ref["Z"]).max()
        assert abs(lam[0] - want) <= 1e-8 * scale and lam[0] <= 1e-7 * scale
        b.close()


def test_vnnlib_property_as_one_batch(ctx, tmp_path):
    """SURVEY.md 8f-4: a vnnlib property read by the library (boxes x output half-spaces, the CNF of
    experiments/vnnlib_utils.jl:18-56) goes through nnsdp_assemble_blocks as ONE batch; every member equals the
    oracle's blocks for the (QcInputBox, QcSafety) pair of the restated reference parser."""
    import nnsdp_b200 as nb

    xdims, beta = [5] + [50] * 6 + [5], 2               # ACAS-shaped (the real nets are not shipped)
    net = rand_net(xdims, seed=12)
    text = "\n".join(f"(declare-const X_{i} Real)" for i in range(5)) + """
(assert (<= X_0 0.68))
(assert (>= X_0 0.6))
(assert (<= X_1 0.05))
(assert (>= X_1 -0.05))
(assert (<= X_2 0.05))
(assert (>= X_2 -0.05))
(assert (<= X_4 -0.45))
(assert (>= X_4 -0.5))
(assert (or (and (<= X_3 0.5)(>= X_3 0.45)) (and (<= X_3 0.3)(>= X_3 0.25))))
(assert (or (and (<= Y_0 Y_1)(<= Y_0 Y_2)(<= Y_0 Y_3)(<= Y_0 Y_4)) (and (>= Y_2 0.75))))
"""
    path = str(tmp_path / "prop.vnnlib")
    open(path, "w").write(text)
    r = nb.read_vnnlib(path, 5, 5)
    cnf = o.load_vnnlib_cnf(path, net)
    flat = [pair for clause in cnf for pair in clause]
    nq = len(flat)
    assert nq == 10 and r["nclauses"] == 4 and np.array_equal(r["clause"], [0, 0, 0, 0, 1, 2, 2, 2, 2, 3])
    rng = np.random.default_rng(4)
    sz = nb.sizes_from_xdims(xdims, beta)
    gin, gbnd, gsec = rng.random((nq, 5)), rng.random((nq, sz["acdim"])), rng.random((nq, sz["secdim"]))
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    batch = nb.NumericBatch(x1min=r["x1min"], x1max=r["x1max"], gamma_in=gin, gamma_bnd=gbnd, gamma_sec=gsec,
                            out_kind=nb.OUT_SAFETY, out_S=r["S"])
    out = nb.assemble_blocks(dnet, beta, batch)
    cliques = o.make_cliques(net, beta)
    for i, (qi, qs) in enumerate(flat):
        q = o.NumericQuery(x1min=qi.x1min, x1max=qi.x1max, qc_out=qs, gin=gin[i], gbnd=gbnd[i], gsec=gsec[i])
        ref = o.run_query(net, beta, q)
        for blk, rb in zip(nb.split_blocks(out[i], cliques), ref["blocks"]):
            assert relerr(blk, rb) <= TOL


# ---------------------------------------------------------------------------------------------
# the hand-off the decomposed SDP was solved from (tests/test_decomposed_cpu.py) is what the library computes
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["W10-D10_beta0", "W10-D10_beta2", "W10-D10_beta5", "W10-D20_beta2"])
def test_affine_handoff_equals_the_committed_fixture(ctx, name):
    """tests/golden/handoff_*.npz were dumped from nnsdp_affine_get / nnsdp_cliques on a B200
    (tests/golden/make_handoff.py); recomputing them must give the same index arrays exactly and the same values
    to 1e-12, and the cliques must be the oracle's makeCliques -- so the certificates of
    tests/test_decomposed_cpu.py are statements about THIS library's hand-off
    (/root/reference/src/Methods/chordal_sdp.jl:19-57,96-153)."""
    import importlib.util
    import nnsdp_b200 as nb

    spec = importlib.util.spec_from_file_location("make_handoff", os.path.join(GOLD, "make_handoff.py"))
    mh = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mh)
    net_name, beta = name.split("_beta")
    data, rec = mh.handoff(nb, ctx, net_name, int(beta), reps=1)
    fix = np.load(os.path.join(GOLD, f"handoff_{name}.npz"))
    for k in ("ent_row", "ent_col", "coo_ent", "coo_var", "ck_off", "ck_idx", "ck1_len", "d_off", "d_idx", "nvar", "nent", "nnz",
              "var_in", "var_out", "var_bnd", "var_sec"):
        assert np.array_equal(data[k], fix[k]), k
    for k in ("z0", "coo_val", "ymin", "ymax", "smin", "smax"):
        scale = max(np.abs(fix[k]).max(), 1e-300)
        assert np.abs(data[k] - fix[k]).max() <= 1e-12 * scale, k
    net = o.load_nnet(os.path.join(GOLD, f"scale-I2-O2-{net_name}.nnet"))
    import sdp_decomposed as sd

    for (Ck, parts, Ds), (Rk, rparts, rDs) in zip(sd.cliques_from_npz(fix), o.make_cliques(net, int(beta))):
        assert np.array_equal(Ck, Rk) and len(Ds) == len(rDs) and all(np.array_equal(a, b) for a, b in zip(Ds, rDs))


def test_bench_dump_outputs_holds_the_last_pass(ctx, tmp_path):
    """bench.py --dump-outputs: with 64 queries through a ring of 24 slots the last pass holds queries 48..63, and the
    dumped rows are their clique blocks (against the oracle); a dump over the size cap is the seeded entry sample of the
    same slots."""
    import subprocess
    import sys

    import torch

    import bench
    import nnsdp_b200 as nb

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    name = "tiny-W10-D10-beta1-Q64"
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--workload", name, "--ring", "24", "--steps", "2",
                        "--no-cpu", "--no-e2e", "--no-extras", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    dump = np.load(tmp_path / "dense_blocks.npy")
    xdims, Ms, beta, inp = bench.make_workload(name, 0)
    net = o.FeedFwdNet(xdims, Ms)
    cliques = o.make_cliques(net, beta)
    assert dump.dtype == np.float64 and dump.shape == (16, sum(len(Ck) ** 2 for Ck, _, _ in cliques))
    for i in range(16):
        q = 48 + i
        ref = o.run_query(net, beta, o.NumericQuery(
            x1min=inp["x1min"][q], x1max=inp["x1max"][q], gin=inp["gamma_in"][q], gbnd=inp["gamma_bnd"][q],
            gsec=inp["gamma_sec"][q], qc_out=o.QcSafety(S=inp["out_S"][0])))
        for blk, rb in zip(nb.split_blocks(dump[i], cliques), ref["blocks"]):
            assert relerr(blk, rb) <= TOL

    b = nb.Batch(nb.Net(ctx, xdims, Ms), beta, Qcap=64, ring=24)
    b.set_inputs(bench.numeric_batch(nb, name, inp), Q=64)
    b.run(None)
    whole = bench.last_pass_outputs(torch, b, 64, 24, bench.DUMP_BYTES)
    sample = bench.last_pass_outputs(torch, b, 64, 24, 16 * 8 * 1000)
    b.close()
    assert np.array_equal(whole, dump)
    idx = np.sort(np.random.default_rng(0).choice(whole.shape[1], size=1000, replace=False))
    assert np.array_equal(sample, whole[:, idx])
