"""nnsdp_batch_certify and Batch.lambda_max_bracket against an exact reference: the FP64 Z the device factorises is
rebuilt from the blocks it emits (split_blocks of get_slot, scattered into a dense Z) and its inertia at the returned
bounds is counted in 256-bit arithmetic (oracle/exact_psd.py).  Covered: the edges of kernels_chol.cu (last panels of
width 1-3, npriv = 32 / 64, TRSM over more than one 128-row block, trailing sizes 0, 1, 63 mod 64, a layer narrower
than beta, a single clique), queries with different outcomes in one pass, stride-0 reach batches, Z scaled by 2^k down
to subnormal products and up to overflow, and a tau sweep within ulps of the exact lambda_max."""
import json
import os
import time

import numpy as np
import pytest

import certify as oc
import exact_psd as ex
import nnsdp_oracle as o
from helpers import rand_net, rand_query, to_numeric_batch
from test_cpu_certify_exact import _lambda_star, _stats, check_sweep

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
EXACT_ZDIM = 150          # exact inertia counts on larger Z cost seconds each


# ---- shapes chosen for the edges of kernels_chol.cu --------------------------------------------------------------

EDGE_SHAPES = [
    ([2, 29, 2], 2),              # one clique, npriv = 32: the last panel leaves nothing below
    ([2, 33, 1, 29, 2], 0),       # npriv = 64 in the last front, last panels of width 2, 63 rows below a panel
    ([2, 29, 4, 31, 2], 3),       # last panels of width 1 and 2, 64 and 65 rows below a panel
    ([3, 1, 4, 1, 2], 1),         # a last panel of width 3
    ([2, 1, 2, 2], 3),            # a layer narrower than beta, one clique
    ([3, 129, 2, 129, 2], 0),     # 3 TRSM row blocks (> 256 rows below a panel), a last panel of width 3
]
EDGES = {"single", "narrow", "w1", "w2", "w3", "npriv32", "npriv64", "N>128", "N>256", "N%64=0", "N%64=1", "N%64=63"}


def edge_features(xdims, beta):
    """The edges of the certify kernels one (xdims, beta) reaches, from the elimination plan."""
    import nnsdp_b200 as nb

    plan = nb.certify_plan(xdims, beta)
    f = {"single"} if len(plan) == 1 else set()
    if any(x < beta for x in xdims[1:-1]):
        f.add("narrow")
    for _, n, npriv, _, _, _ in plan.tolist():
        if npriv in (32, 64):
            f.add(f"npriv{npriv}")
        for j0 in range(0, npriv, 32):
            w = min(32, npriv - j0)
            below = n - j0 - w          # rows of the TRSM and side of the trailing update
            if w < 4:
                f.add(f"w{w}")
            if below > 128:
                f.add("N>128")
            if below > 256:
                f.add("N>256")
            if below > 0 and below % 64 in (0, 1, 63):
                f.add(f"N%64={below % 64}")
    return f


def test_edge_shapes_cover_every_edge():
    got = set().union(*(edge_features(x, b) for x, b in EDGE_SHAPES))
    assert got == EDGES, EDGES - got


# ---- helpers -------------------------------------------------------------------------------------------------------

def _batch(dnet, beta, nbq, Q, ring, crown=False):
    import nnsdp_b200 as nb

    b = nb.Batch(dnet, beta, Qcap=Q, ring=ring)
    b.set_inputs(nbq, Q=Q)
    if crown:
        b.set_bounds_method("crown")
        b.bounds_crown()
    else:
        b.bounds()
    b.prepare()
    return b


def _emitted(b, dnet, beta, q):
    """(dense Z, clique blocks) of query q exactly as certify reads them: the lower triangles of the emitted blocks."""
    import nnsdp_b200 as nb

    b.emit(q, 1)
    cl = dnet.cliques(beta)
    blocks = nb.split_blocks(b.get_slot(0), cl)
    n = b.sz["Zdim"]
    Z, seen = np.zeros((n, n)), np.zeros((n, n), dtype=bool)
    for B, (Ck, _, _) in zip(blocks, cl):
        c = np.asarray(Ck) - 1
        r, s = np.tril_indices(len(c))
        gi, gj = np.maximum(c[r], c[s]), np.minimum(c[r], c[s])
        both = seen[gi, gj]
        assert np.array_equal(Z[gi[both], gj[both]], B[r[both], s[both]]), "overlapping blocks differ"
        Z[gi, gj] = B[r, s]
        seen[gi, gj] = True
    Z = np.tril(Z) + np.tril(Z, -1).T
    return Z, blocks


def _cl0(dnet, beta):
    return [np.asarray(Ck) - 1 for Ck, _, _ in dnet.cliques(beta)]


def _scale(Z):
    return float(np.abs(np.linalg.eigvalsh(Z)).max())


def _check_exact(Z, cert, bound, lower):
    if cert:
        assert ex.count_above(Z, bound) == 0, bound
    elif np.isfinite(lower):
        assert ex.count_above(Z, lower) >= 1, lower


# ---- 1. edge shapes ------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("xdims,beta", EDGE_SHAPES)
def test_edge_shapes_match_restatement_and_are_sound(ctx, xdims, beta):
    import nnsdp_b200 as nb

    net = rand_net(xdims, seed=sum(xdims) + beta)
    rng = np.random.default_rng(beta)
    Q = 2
    qs = [rand_query(net, beta, rng, kind="safety") for _ in range(Q)]
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    b = _batch(dnet, beta, to_numeric_batch(nb, net, qs), Q, ring=1)
    cl = _cl0(dnet, beta)
    em = [_emitted(b, dnet, beta, q) for q in range(Q)]
    lam = np.array([np.linalg.eigvalsh(Z).max() for Z, _ in em])
    scale = np.array([_scale(Z) for Z, _ in em])
    for tau, want in ((lam - 1e-3 * scale, 0), (lam + 1e-6 * scale, 1)):
        cert, bound, fidx, minp, lower = b.certify(tau, lower=True)
        assert (cert == want).all(), (cert, want)
        for q, (Z, blocks) in enumerate(em):
            rc, rb, rf, rp = oc.certify_fronts(blocks, cl, tau[q])
            assert rc == want and fidx[q] == rf
            assert abs(minp[q] - rp) <= 1e-9 * scale[q], (minp[q], rp)
            assert abs(bound[q] - rb) <= 1e-12 * scale[q] + abs(tau[q]) * 1e-15
            assert bound[q] <= tau[q]
            assert (lower[q] == -np.inf) if want else (tau[q] - 1e-6 * scale[q] <= lower[q] <= tau[q])
            if Z.shape[0] <= EXACT_ZDIM:
                _check_exact(Z, cert[q], bound[q], lower[q])
    b.close()


# ---- 2. different outcomes in one pass -----------------------------------------------------------------------------

def _tau_failing_at(Z, lo, hi):
    """(tau, i): tau between lambda_max of the leading i and i+1 rows, at the i in [lo, hi) with the widest gap."""
    m = np.array([np.linalg.eigvalsh(Z[:i + 1, :i + 1]).max() for i in range(hi)])
    prev = np.concatenate([[m[0] - 1e-3 * _scale(Z)], m[:-1]])
    i = lo + int(np.argmax((m - prev)[lo:hi]))
    assert m[i] - prev[i] >= 1e-6 * _scale(Z), "no usable gap in this front"
    return 0.5 * (m[i] + prev[i]), i


def test_mixed_outcomes_in_one_pass_equal_single_query_batches(ctx):
    """Q = 5 through 2 ring slots (passes of 2, 2, 1): failures in the first, a middle and the last front next to
    certified queries; every query's results equal its results alone, bit for bit."""
    import nnsdp_b200 as nb

    xdims, beta, Q = [2] + [10] * 9 + [2], 1, 5
    net = rand_net(xdims, seed=8)
    rng = np.random.default_rng(8)
    qs = [rand_query(net, beta, rng, kind="safety") for _ in range(Q)]
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    plan = nb.certify_plan(xdims, beta)
    fronts = [(int(g0), int(g0 + npriv)) for _, _, npriv, g0, _, _ in plan]
    alone = [_batch(dnet, beta, to_numeric_batch(nb, net, [q]), 1, ring=1) for q in qs]
    Zs = [_emitted(a, dnet, beta, 0)[0] for a in alone]
    target = {0: fronts[0], 2: fronts[len(fronts) // 2], 3: fronts[-1]}
    tau, want_f = np.zeros(Q), {}
    for q in range(Q):
        if q in target:
            tau[q], want_f[q] = _tau_failing_at(Zs[q], *target[q])
        else:
            tau[q] = np.linalg.eigvalsh(Zs[q]).max() + 1e-6 * _scale(Zs[q])
    b = _batch(dnet, beta, to_numeric_batch(nb, net, qs), Q, ring=2)
    got = b.certify(tau, lower=True)
    for q in range(Q):
        one = alone[q].certify(tau[q], lower=True)
        for x, y in zip(got, one):
            assert np.array_equal(x[q:q + 1], y), (q, x[q], y)
        if q in want_f:
            assert got[0][q] == 0 and got[2][q] == want_f[q]
        else:
            assert got[0][q] == 1 and got[2][q] == -1
    b.close()
    for a in alone:
        a.close()


# ---- 3. reach batch with stride-0 inputs ---------------------------------------------------------------------------

def test_reach_batch_stride_zero_equals_single_queries(ctx):
    """One box and one set of multipliers (stride 0) for every query, a different half-plane normal each; the
    certificate of each query equals its own Q = 1 batch bit for bit."""
    import nnsdp_b200 as nb

    xdims, beta, Q = [2] + [10] * 9 + [2], 2, 4
    net = rand_net(xdims, seed=9)
    q0 = rand_query(net, beta, np.random.default_rng(9), kind="hplane")
    normals = np.random.default_rng(10).standard_normal((Q, xdims[-1]))

    def nbq(vec):
        return nb.NumericBatch(x1min=q0.x1min, x1max=q0.x1max, gamma_in=q0.gin, gamma_bnd=q0.gbnd, gamma_sec=q0.gsec,
                               out_kind=nb.OUT_HPLANE, out_vec=vec, gamma_out=np.asarray(q0.gout).reshape(1, 1))

    dnet = nb.Net(ctx, net.xdims, net.Ms)
    alone = [_batch(dnet, beta, nbq(normals[q:q + 1]), 1, ring=1) for q in range(Q)]
    Zs = [_emitted(a, dnet, beta, 0)[0] for a in alone]
    lam = np.array([np.linalg.eigvalsh(Z).max() for Z in Zs])
    scale = np.array([_scale(Z) for Z in Zs])
    tau = lam + np.where(np.arange(Q) % 2 == 0, 1e-6, -1e-3) * scale
    b = _batch(dnet, beta, nbq(normals), Q, ring=3)
    got = b.certify(tau, lower=True)
    assert list(got[0]) == [1, 0, 1, 0]
    for q in range(Q):
        one = alone[q].certify(tau[q], lower=True)
        for x, y in zip(got, one):
            assert np.array_equal(x[q:q + 1], y), (q, x[q], y)
        assert np.array_equal(_emitted(b, dnet, beta, q)[0], Zs[q])
    b.close()
    for a in alone:
        a.close()


# ---- 4. scaling by 2^k ---------------------------------------------------------------------------------------------

def _scaled_batch(dnet, net, beta, qs, k):
    import nnsdp_b200 as nb

    f = 2.0 ** k
    sq = [o.NumericQuery(x1min=q.x1min, x1max=q.x1max, gin=q.gin * f, gbnd=q.gbnd * f, gsec=q.gsec * f,
                         qc_out=o.QcSafety(S=q.qc_out.S * f), gout=None) for q in qs]
    return _batch(dnet, beta, to_numeric_batch(nb, net, sq), len(qs), ring=1)


@pytest.fixture(scope="module")
def scaled_case(ctx):
    import nnsdp_b200 as nb

    xdims, beta, Q = [2] + [10] * 9 + [2], 2, 2
    net = rand_net(xdims, seed=12)
    rng = np.random.default_rng(12)
    qs = [rand_query(net, beta, rng, kind="safety") for _ in range(Q)]
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    b = _scaled_batch(dnet, net, beta, qs, 0)
    em = [_emitted(b, dnet, beta, q) for q in range(Q)]
    lam = np.array([np.linalg.eigvalsh(Z).max() for Z, _ in em])
    scale = np.array([_scale(Z) for Z, _ in em])
    taus = [lam - 1e-3 * scale, lam + 1e-6 * scale]
    res = [b.certify(t) for t in taus]
    b.close()
    return dict(net=net, dnet=dnet, beta=beta, qs=qs, em=em, lam=lam, scale=scale, taus=taus, res=res)


@pytest.mark.parametrize("k", [100, -100, 200, -200])
def test_scaling_by_even_powers_of_two_is_exact(scaled_case, k):
    s = scaled_case
    f = 2.0 ** k
    b = _scaled_batch(s["dnet"], s["net"], s["beta"], s["qs"], k)
    for q, (Z, blocks) in enumerate(s["em"]):
        Zk, blocks_k = _emitted(b, s["dnet"], s["beta"], q)
        for B, Bk in zip(blocks, blocks_k):
            assert np.array_equal(np.tril(Bk), np.tril(B) * f)
    for tau, (cert, bound, fidx, minp) in zip(s["taus"], s["res"]):
        ck, bk, fk, mk = b.certify(tau * f)
        assert np.array_equal(ck, cert) and np.array_equal(fk, fidx)
        assert np.array_equal(bk, bound * f) and np.array_equal(mk, minp * f)
    b.close()


@pytest.mark.parametrize("k", [-1000, -1060])
def test_subnormal_products_stay_sound(scaled_case, k):
    """Entries near or below the normal range (products in the DMMA update are subnormal): every certified bound is
    above the exact lambda_max and every failure's lower bound below it."""
    s = scaled_case
    f = 2.0 ** k
    b = _scaled_batch(s["dnet"], s["net"], s["beta"], s["qs"], k)
    certified = 0
    for q in range(len(s["qs"])):
        Zk, _ = _emitted(b, s["dnet"], s["beta"], q)
        assert np.abs(Zk).max() > 0
        lam_k = np.linalg.eigvalsh(Zk / f).max() * f              # scaling up is exact
        for rel in (-1e-3, 1e-6, 1e-3, 1e-1, 1.0):
            tau = np.full(len(s["qs"]), lam_k + rel * s["scale"][q] * f)
            cert, bound, _, _, lower = b.certify(tau, lower=True)
            _check_exact(Zk, cert[q], bound[q], lower[q])
            certified += int(cert[q])
            if rel < 0:
                assert cert[q] == 0
    if k == -1000:
        assert certified > 0
    b.close()


@pytest.mark.parametrize("k", [1000, 1020])
def test_overflow_is_not_certified_and_returns(scaled_case, k):
    """At 2^1020 Z overflows to inf: no certificate, no lower bound, and the tau' descent ends at once.  At 2^1000 Z is
    finite and the results are the unscaled ones times 2^k."""
    s = scaled_case
    f = 2.0 ** k
    b = _scaled_batch(s["dnet"], s["net"], s["beta"], s["qs"], k)
    finite = all(np.isfinite(_emitted(b, s["dnet"], s["beta"], q)[0]).all() for q in range(len(s["qs"])))
    assert finite == (k == 1000)
    for tau, (cert, bound, fidx, minp) in zip(s["taus"], s["res"]):
        t0 = time.perf_counter()
        ck, bk, fk, mk, lk = b.certify(tau * f, lower=True)
        assert time.perf_counter() - t0 < 5.0
        if finite:
            assert np.array_equal(ck, cert) and np.array_equal(fk, fidx) and np.array_equal(bk, bound * f)
        else:
            assert (ck == 0).all() and (lk == -np.inf).all()
    b.close()


# ---- 5. device soundness sweep and 6. lambda_max_bracket -----------------------------------------------------------

def _random_w10(ctx):
    import nnsdp_b200 as nb

    xdims, beta = [2] + [10] * 9 + [2], 2
    net = rand_net(xdims, seed=13)
    q = rand_query(net, beta, np.random.default_rng(13), kind="circle")
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    return dnet, beta, _batch(dnet, beta, to_numeric_batch(nb, net, [q]), 1, ring=1)


def _gate_shaped(ctx):
    """The construction of the non-convergence query of test_gpu_parity at width 40: lambda_max ~ -1e-9 at scale ~4."""
    import nnsdp_b200 as nb

    xdims, beta = [2, 40, 40, 2], 1
    net = rand_net(xdims, seed=1, sigma=0.0)
    rng = np.random.default_rng(0)
    q = rand_query(net, beta, rng, kind="hplane", radius=0.1)
    q.gsec[:] = 0.0
    q.gbnd[:] = rng.uniform(0.5, 2.0, q.gbnd.size)
    q.gbnd[17] = 1e-9
    q.qc_out = o.QcReachHplane(np.zeros(2))
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    return dnet, beta, _batch(dnet, beta, to_numeric_batch(nb, net, [q]), 1, ring=1)


def _recorded_optimum(ctx):
    import nnsdp_b200 as nb

    res = json.load(open(os.path.join(GOLD, "scale_W10_D10_optimum.json")))
    net = o.load_nnet(os.path.join(GOLD, "scale-I2-O2-W10-D10.nnet"))
    P, yc = np.asarray(res["P"]), np.asarray(res["yc"])
    invP = np.linalg.inv(P)
    invP = 0.5 * (invP + invP.T)
    beta, n1, ac = 2, net.xdims[0], net.acdim
    g = np.asarray(res["oracle_optimum"][str(beta)]["gamma"])
    q = o.NumericQuery(x1min=np.full(2, 0.5), x1max=np.full(2, 1.5), qc_out=o.QcReachEllipsoid(invP=invP, yc=yc),
                       gin=g[:n1], gout=g[n1:n1 + 1], gbnd=g[n1 + 1:n1 + 1 + ac], gsec=g[n1 + 1 + ac:])
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    return dnet, beta, _batch(dnet, beta, to_numeric_batch(nb, net, [q]), 1, ring=1, crown=True)


CASES = {"random_W10-D10": _random_w10, "gate_shaped": _gate_shaped, "recorded_optimum": _recorded_optimum}


@pytest.fixture(scope="module", params=list(CASES))
def exact_case(request, ctx):
    dnet, beta, b = CASES[request.param](ctx)
    Z, blocks = _emitted(b, dnet, beta, 0)
    assert Z.shape[0] <= EXACT_ZDIM
    lam, lo, hi = _lambda_star(Z)
    c = oc.certify_margin(lam, Z.shape[0], *_stats(Z))
    yield dict(name=request.param, b=b, Z=Z, blocks=blocks, cl=_cl0(dnet, beta), lam=lam, lo=lo, hi=hi, c=c)
    b.close()


def test_device_sweep_is_sound(exact_case):
    """tau = lambda* + {+-1, +-4 ulps, +-c/10, +-c, +-10c, +100c}: certified => no eigenvalue above the bound; failed =>
    at least one above the lower bound; where |tau - lambda*| >= 10c the outcome is the restatement's."""
    s = exact_case

    def device(tau):
        cert, bound, _, _, lower = s["b"].certify(tau, lower=True)
        if abs(tau - s["lam"]) >= 10 * s["c"]:
            assert cert[0] == oc.certify_fronts(s["blocks"], s["cl"], tau)[0], tau
        return int(cert[0]), float(bound[0]), float(lower[0])

    check_sweep(s["Z"], s["lo"], s["hi"], s["lam"], s["c"], device)


@pytest.mark.parametrize("kw,want_cert", [({}, 1), ({"max_iters": 3}, 1), ({"max_tries": 1}, 0),
                                          ({"max_iters": 3, "max_tries": 1}, 0)])
def test_lambda_max_bracket_is_exact_interval(exact_case, kw, want_cert):
    s = exact_case
    lo, hi, cert = s["b"].lambda_max_bracket(**kw)
    assert cert[0] == want_cert and np.isfinite(hi[0]) == bool(want_cert)
    assert np.isfinite(lo[0]) and ex.count_above(s["Z"], lo[0]) >= 1          # lo < lambda*
    if want_cert:
        assert ex.count_above(s["Z"], hi[0]) == 0                               # lambda* <= hi
    if not kw:                                  # converged Lanczos: the interval is tight as well
        assert s["lam"] - 1e-6 * _scale(s["Z"]) <= lo[0] and hi[0] <= s["lam"] + 1e-6 * _scale(s["Z"])
