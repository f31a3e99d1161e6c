"""The certificate for the exact Z(γ) (nnsdp_batch_assembly_error, nnsdp_batch_certify_gamma) on one B200:

- the device row sums s_q[r] of abs (every operation rounded up) against the exact row sums of oracle/exact_z.py:
  s ≥ Σ_c abs[r, c] and s ≤ (1 + 1e-12) Σ_c abs[r, c], on every row, for β = 0 … 7, layers narrower than β, the four
  output kinds, stride-0 reach batches, γ components 2^U(−40, 40), λ = 0 on stably active neurons, a subnormal λ on a
  layer whose weights exceed 1, several ring passes, and the rows of a W1000‑D20 query around every block boundary;
- soundness against the exact Z(γ) (Fractions, inertia counted by test_cpu_certify_gamma.count_above_exact): certified ⇒ no
  eigenvalue of Z(γ) above bound, failed with a finite lower ⇒ one at least above lower, at τ around the exact λmax and
  on Z scaled by 2^k;
- nnsdp_batch_certify_ex and lambda_max_bracket() unchanged by a certify_gamma call, and the argument checks."""
from fractions import Fraction

import numpy as np
import pytest

import exact_z as ez
import nnsdp_oracle as o
from helpers import rand_net, rand_query, to_numeric_batch, wide_range_net, wide_range_query
from test_cpu_certify_gamma import count_above_exact
from test_gpu_certify_exact import EDGE_SHAPES

pytestmark = pytest.mark.gpu
EXACT_ZDIM = 150
REL = Fraction(1, 10 ** 12)


def _ibp_bounds(net, q):
    info = o.intervals_worst_case(q.x1min, q.x1max, net)
    amin = np.concatenate([p[0] for p in info.acx_intvs])
    amax = np.concatenate([p[1] for p in info.acx_intvs])
    smin, smax = o.make_sector_min_max(amin, amax)
    ymin = np.concatenate([p[0] for p in info.x_intvs[1:-1]])
    ymax = np.concatenate([p[1] for p in info.x_intvs[1:-1]])
    return ymin, ymax, smin, smax


def _inputs(nb, net, qs, bounds):
    b = to_numeric_batch(nb, net, qs)
    b.ymin, b.ymax, b.smin, b.smax = (np.stack([bd[i] for bd in bounds]) for i in range(4))
    return b


def _batch(ctx, net, beta, qs, bounds, ring=1, nbq=None):
    import nnsdp_b200 as nb

    dnet = nb.Net(ctx, net.xdims, net.Ms)
    b = nb.Batch(dnet, beta, Qcap=len(qs) if nbq is None else nbq[1], ring=ring)
    if nbq is None:
        b.set_inputs(_inputs(nb, net, qs, bounds))
    else:
        b.set_inputs(nbq[0], Q=nbq[1])
    b.prepare()
    return dnet, b


def _check_rows(net, beta, q, bounds, rows, err, kind_code):
    """Every row sum of one query against exact_z (exact mode up to EXACT_ZDIM, extended beyond)."""
    import nnsdp_b200 as nb

    exact = net.Zdim <= EXACT_ZDIM
    R = ez.exact_z(net, beta, q, bounds, mode="exact" if exact else "extended")
    if exact:
        ref = [sum(R._abs_exact[i], Fraction(0)) for i in range(net.Zdim)]
        for r, (s, x) in enumerate(zip(rows, ref)):
            fs = Fraction(float(s))
            assert x <= fs <= x * (1 + REL), (r, float(s), float(x))
        smax = max(ref)
    else:
        _check_rows_extended(R, rows)
        smax = Fraction(float(R.abs.sum(1).max()))
    nmax = nb.assembly_error_nmax(net.xdims, beta, kind_code)
    assert nmax >= R.N.max()
    assert Fraction(float(err)) >= Fraction(float(ez.gamma(nmax))) * smax * (1 - REL)


def _check_rows_extended(R, rows):
    """R.abs is each entry's abs rounded up to FP64 after a long-double sum inflated by γ_N(2⁻⁶³) + 2⁻⁶²."""
    ref = R.abs.astype(np.longdouble).sum(1)
    slack = np.longdouble(float(ez.gamma(R.N.max(), ez.UEXT)) + 2.0 ** -50)
    got = np.asarray(rows, dtype=np.longdouble)
    assert (got >= ref * (1 - slack)).all(), np.nonzero(got < ref * (1 - slack))
    assert (got <= ref * (1 + np.longdouble(1e-12))).all(), np.nonzero(got > ref * (1 + np.longdouble(1e-12)))


KIND = {"safety": 0, "hplane": 1, "circle": 2, "ellipsoid": 3}


def _subnormal_on_heavy_layer(xdims, seed):
    """wide_range_case with the first layer scaled by 2^10: the subnormal λ of wide_range_query then sits on a layer
    whose weights exceed 1 (outside the precondition of exact_z's underflow term)."""
    net = wide_range_net(xdims, seed)
    net.Ms[0] = net.Ms[0] * 1024.0
    return net


# (xdims, beta, kind, Q, ring): queries alternate wide-range / plain (IBP bounds)
ROW_CASES = [([2] + [10] * 9 + [2], 2, "circle", 2, 1)] + \
    [(x, b, k, 2, 1) for (x, b), k in zip(EDGE_SHAPES, ["safety", "hplane", "circle", "ellipsoid", "safety", "hplane"])] + \
    [([2, 4, 7, 3, 5, 2], 7, "safety", 5, 2),       # layers narrower than β, band across two boundaries, 3 ring passes
     ([3, 3, 3, 3, 4, 3, 3], 4, "ellipsoid", 3, 2),
     ([2] + [10] * 6 + [2], 1, "hplane", 3, 1),
     ([2, 10, 10, 10, 2], 0, "circle", 3, 2)]


@pytest.mark.parametrize("xdims,beta,kind,Q,ring", ROW_CASES)
def test_row_sums_bound_the_exact_abs(ctx, xdims, beta, kind, Q, ring):
    net = wide_range_net(xdims, seed=sum(xdims) + beta)
    rng = np.random.default_rng(beta + 31)
    qs, bounds = [], []
    for i in range(Q):
        if i % 2 == 0:
            q, bd = wide_range_query(net, beta, kind, rng)
        else:
            q = rand_query(net, beta, rng, kind=kind, radius=0.0)
            bd = _ibp_bounds(net, q)
        qs.append(q)
        bounds.append(bd)
    _, b = _batch(ctx, net, beta, qs, bounds, ring=ring)
    err, rows = b.assembly_error(rowsums=True)
    b.close()
    assert np.isfinite(err).all()
    for i in range(Q):
        _check_rows(net, beta, qs[i], bounds[i], rows[i], err[i], KIND[kind])


def test_row_sums_with_a_subnormal_lambda_on_a_layer_above_one(ctx):
    xdims, beta = [2, 6, 5, 4, 2], 2
    net = _subnormal_on_heavy_layer(xdims, 77)
    assert np.abs(net.Ms[0][:, :-1]).max() > 1
    q, bd = wide_range_query(net, beta, "ellipsoid", np.random.default_rng(77))
    assert q.gsec[1] == 2.0 ** -1074 and q.gsec[0] == 2.0 ** -1070
    _, b = _batch(ctx, net, beta, [q], [bd])
    err, rows = b.assembly_error(rowsums=True)
    b.close()
    _check_rows(net, beta, q, bd, rows[0], err[0], KIND["ellipsoid"])


def test_row_sums_of_a_stride_zero_reach_batch(ctx):
    """One box, one set of multipliers and bounds for every query (stride 0), a different half-plane normal each."""
    import nnsdp_b200 as nb

    xdims, beta, Q = [2] + [10] * 9 + [2], 2, 4
    net = wide_range_net(xdims, seed=9)
    q0, bd = wide_range_query(net, beta, "hplane", np.random.default_rng(9))
    normals = np.random.default_rng(10).standard_normal((Q, xdims[-1]))
    nbq = nb.NumericBatch(x1min=q0.x1min, x1max=q0.x1max, gamma_in=q0.gin, gamma_bnd=q0.gbnd, gamma_sec=q0.gsec,
                          out_kind=nb.OUT_HPLANE, out_vec=normals, gamma_out=np.asarray(q0.gout).reshape(1, 1),
                          ymin=bd[0], ymax=bd[1], smin=bd[2], smax=bd[3])
    _, b = _batch(ctx, net, beta, None, None, ring=3, nbq=(nbq, Q))
    err, rows = b.assembly_error(rowsums=True)
    b.close()
    for i in range(Q):
        qi = o.NumericQuery(x1min=q0.x1min, x1max=q0.x1max, gin=q0.gin, gbnd=q0.gbnd, gsec=q0.gsec,
                            qc_out=o.QcReachHplane(normals[i]), gout=q0.gout)
        _check_rows(net, beta, qi, bd, rows[i], err[i], KIND["hplane"])


def test_stress_query_rows_around_every_block_boundary(ctx):
    """W1000-D20, β = 2: the rows within ±2 of every block boundary, the affine row and a random sample (extended
    mode), through the tiles of the |W|' G products (64 rows) and the 1000-wide layers."""
    xdims, beta = [2] + [1000] * 20 + [2], 2
    net = wide_range_net(xdims, seed=2024)
    rng = np.random.default_rng(2024)
    q, bd = wide_range_query(net, beta, "ellipsoid", rng)
    _, b = _batch(ctx, net, beta, [q], [bd])
    err, rows = b.assembly_error(rowsums=True)
    b.close()
    assert np.isfinite(err[0])
    off = np.concatenate([[0], np.cumsum(xdims[:-1]), [net.Zdim]])
    sel = set()
    for e in off:
        sel.update(range(max(0, e - 2), min(net.Zdim, e + 2)))
    sel.update(rng.choice(net.Zdim, 32, replace=False).tolist())
    sel.add(net.Zdim - 1)
    sel = np.array(sorted(sel))
    for part in np.array_split(sel, -(-len(sel) // 256)):
        R = ez.exact_z(net, beta, q, bd, mode="extended", rows=part)
        _check_rows_extended(R, rows[0][part])


def test_assembly_error_is_deterministic_and_independent_of_the_batch(ctx):
    """Two calls give the same bits, and a query's e_q does not depend on the queries beside it."""
    xdims, beta, Q = [2] + [10] * 9 + [2], 1, 3
    net = wide_range_net(xdims, seed=5)
    rng = np.random.default_rng(5)
    qs, bds = zip(*[wide_range_query(net, beta, "safety", rng) for _ in range(Q)])
    _, b = _batch(ctx, net, beta, list(qs), list(bds), ring=2)
    e1, r1 = b.assembly_error(rowsums=True)
    e2, r2 = b.assembly_error(rowsums=True)
    assert np.array_equal(e1, e2) and np.array_equal(r1, r2)
    assert np.array_equal(b.assembly_error(), e1)
    b.close()
    for i in range(Q):
        _, bi = _batch(ctx, net, beta, [qs[i]], [bds[i]])
        ei, ri = bi.assembly_error(rowsums=True)
        bi.close()
        assert ei[0] == e1[i] and np.array_equal(ri[0], r1[i])


# ---- soundness for the exact Z(γ) -----------------------------------------------------------------------------------

def _soundness_case(name):
    if name == "random_W10-D10":
        xdims, beta = [2] + [10] * 9 + [2], 2
        net = rand_net(xdims, seed=13)
        q = rand_query(net, beta, np.random.default_rng(13), kind="circle")
        return net, beta, q, _ibp_bounds(net, q)
    if name == "wide_range":
        xdims, beta = [2, 8, 9, 7, 2], 2
        net = wide_range_net(xdims, seed=21)
        q, bd = wide_range_query(net, beta, "safety", np.random.default_rng(21))
        return net, beta, q, bd
    xdims, beta = [2, 6, 5, 4, 2], 1                    # "subnormal_heavy"
    net = _subnormal_on_heavy_layer(xdims, 78)
    q, bd = wide_range_query(net, beta, "hplane", np.random.default_rng(78))
    return net, beta, q, bd


SOUND = ["random_W10-D10", "wide_range", "subnormal_heavy"]
_witness = {}


def _exact_lambda(Zg):
    """λmax of the exact Z(γ) to ~30 digits (eigvalsh of its FP64 rounding places the bracket)."""
    Zf = np.vectorize(float)(Zg)
    ev = np.linalg.eigvalsh(Zf)
    s = float(np.abs(ev).max())
    lo, hi = ev[-1] - 1e-9 * s, ev[-1] + 1e-9 * s
    assert count_above_exact(Zg, lo) >= 1 and count_above_exact(Zg, hi) == 0
    for _ in range(30):
        mid = 0.5 * (lo + hi)
        if mid in (lo, hi):
            break
        if count_above_exact(Zg, mid):
            lo = mid
        else:
            hi = mid
    return 0.5 * (lo + hi), s


def _check_gamma(Zg, cert, bound, lower):
    if cert:
        assert count_above_exact(Zg, bound) == 0, bound
    elif np.isfinite(lower):
        assert count_above_exact(Zg, lower) >= 1, lower


@pytest.mark.parametrize("name", SOUND)
def test_certify_gamma_is_sound_for_the_exact_z(ctx, name):
    import certify as oc

    net, beta, q, bd = _soundness_case(name)
    assert net.Zdim <= EXACT_ZDIM
    _, b = _batch(ctx, net, beta, [q], [bd])
    Zg = ez.exact_z(net, beta, q, bd, mode="exact").ref
    lam, s = _exact_lambda(Zg)
    e = float(b.assembly_error()[0])
    assert 0 < e < 1e-6 * s
    Zf = np.vectorize(float)(Zg)
    c = oc.certify_margin(lam, net.Zdim, float(np.trace(Zf)), float(np.abs(np.diag(Zf)).sum()),
                          float(np.abs(np.diag(Zf)).max()))
    offs = [d * x for x in (c, e, 10 * e) for d in (-1, 1)] + [c + e * f for f in (-1, 0.1, 0.25, 0.5, 0.75, 1.5, 2)]
    for off in offs:
        tau = lam + off
        cert, bound, fidx, _, lower, err = b.certify_gamma(tau, lower=True)
        assert err[0] == e
        _check_gamma(Zg, cert[0], bound[0], lower[0])
        if cert[0]:
            assert bound[0] <= tau and fidx[0] == -1
        if b.certify(tau)[0][0] and not cert[0]:
            _witness[name] = tau
    b.close()


def test_the_assembly_term_is_live():
    """At least one τ of the sweeps above (run before this test) is certified for Z_dev but not for Z(γ)."""
    assert _witness, "no τ was certified by certify but not by certify_gamma"


def _scaled(net, beta, q, bd, k):
    f = 2.0 ** k
    return o.NumericQuery(x1min=q.x1min, x1max=q.x1max, gin=q.gin * f, gbnd=q.gbnd * f, gsec=q.gsec * f,
                          qc_out=o.QcSafety(S=q.qc_out.S * f), gout=None)


@pytest.mark.parametrize("k", [100, -100, -1000, -1060, 1020])
def test_scaled_z_stays_sound(ctx, k):
    xdims, beta = [2] + [10] * 9 + [2], 2
    net = rand_net(xdims, seed=12)
    q0 = rand_query(net, beta, np.random.default_rng(12), kind="safety")
    bd = _ibp_bounds(net, q0)
    q = _scaled(net, beta, q0, bd, k)
    _, b = _batch(ctx, net, beta, [q], [bd])
    Zg0 = ez.exact_z(net, beta, q0, bd, mode="exact").ref
    lam0, s0 = _exact_lambda(Zg0)
    f = 2.0 ** k
    if k == 1020:
        cert, bound, _, _, lower, err = b.certify_gamma((lam0 + 1e-3 * s0) * f, lower=True)
        assert err[0] == np.inf and cert[0] == 0 and lower[0] == -np.inf and bound[0] == np.inf
        b.close()
        return
    Zg = ez.exact_z(net, beta, q, bd, mode="exact").ref          # of the scaled (possibly rounded) inputs
    e = float(b.assembly_error()[0])
    assert np.isfinite(e)
    for rel in (-1e-3, 1e-6, 1e-3, 1e-1, 1.0):
        tau = (lam0 + rel * s0) * f
        cert, bound, _, _, lower, _ = b.certify_gamma(tau, lower=True)
        _check_gamma(Zg, cert[0], bound[0], lower[0])
        if rel < 0:
            assert cert[0] == 0
        if abs(k) == 100 and rel >= 1e-3:
            assert cert[0] == 1
    b.close()


# ---- nothing moved and the argument checks --------------------------------------------------------------------------

def test_certify_ex_and_bracket_do_not_move(ctx):
    net, beta, q, bd = _soundness_case("random_W10-D10")
    _, b = _batch(ctx, net, beta, [q], [bd])
    lam = float(np.linalg.eigvalsh(np.vectorize(float)(ez.exact_z(net, beta, q, bd, mode="extended").ref)).max())
    taus = [lam - 1e-3, lam + 1e-9, lam + 1e-3]
    before = [b.certify(t, lower=True) for t in taus]
    br0 = b.lambda_max_bracket()
    for t in taus:
        b.certify_gamma(t, lower=True)
    after = [b.certify(t, lower=True) for t in taus]
    br1 = b.lambda_max_bracket()
    for x, y in zip(before, after):
        for u, v in zip(x, y):
            assert np.array_equal(u, v)
    for u, v in zip(br0, br1):
        assert np.array_equal(u, v)
    lo, hi, cert = b.lambda_max_bracket(of_gamma=True)
    Zg = ez.exact_z(net, beta, q, bd, mode="exact").ref
    assert cert[0] == 1
    assert count_above_exact(Zg, lo[0]) >= 1 and count_above_exact(Zg, hi[0]) == 0
    b.close()


def test_argument_checks(ctx):
    import nnsdp_b200 as nb
    from nnsdp_b200 import _lib as L

    xdims, beta = [2, 5, 4, 2], 1
    net = rand_net(xdims, seed=4)
    q = rand_query(net, beta, np.random.default_rng(4), kind="safety")
    dnet = nb.Net(ctx, net.xdims, net.Ms)

    def code(fn):
        with pytest.raises(nb.NnsdpError) as e:
            fn()
        return e.value.code

    for kw in ({"packed": True}, {"dense": True}):
        b = nb.Batch(dnet, beta, Qcap=1, ring=1, **kw)
        b.set_inputs(to_numeric_batch(nb, net, [q]))
        b.bounds()
        b.prepare()
        assert code(lambda: b.certify_gamma(0.0)) == L.ERR_ARG
        assert np.isfinite(b.assembly_error()).all()          # any output format: nothing is emitted
        b.close()
    b = nb.Batch(dnet, beta, Qcap=1, ring=0)                    # bounds only
    b.set_inputs(to_numeric_batch(nb, net, [q]))
    b.bounds()
    assert code(lambda: b.certify_gamma(0.0)) == L.ERR_ARG
    assert code(lambda: b.assembly_error()) == L.ERR_ARG
    b.close()
    b = nb.Batch(dnet, beta, Qcap=1, ring=1)
    b.set_inputs(to_numeric_batch(nb, net, [q]))
    b.bounds()
    assert code(lambda: b.certify_gamma(0.0)) == L.ERR_STATE
    assert code(lambda: b.assembly_error()) == L.ERR_STATE
    b.prepare()
    for bad in (np.nan, np.inf, -np.inf):
        assert code(lambda: b.certify_gamma(bad)) == L.ERR_ARG
    b.close()
