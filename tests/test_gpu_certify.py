"""nnsdp_batch_certify on the device: the sound certificate eigmax(Z) <= tau (multifrontal Cholesky of tau' I - Z with
a rounding-error margin) against numpy's eigenvalues of nnsdp_assemble_dense and against the CPU restatement
oracle/certify.py, the acceptance-gate cases, the stress size, the ring contract and the error codes."""
import os

import numpy as np
import pytest

import certify as oc
import nnsdp_oracle as o
from helpers import rand_net, rand_query, to_numeric_batch

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

CASES = [([2] + [10] * 9 + [2], b, "safety") for b in range(4)] + [
    ([2] + [10] * 9 + [2], 1, "hplane"),
    ([2] + [10] * 9 + [2], 2, "circle"),
    ([2] + [10] * 9 + [2], 3, "ellipsoid"),
    ([5] + [50] * 6 + [5], 2, "safety"),        # ACAS-shaped
    ([2, 10, 3, 10, 2], 4, "hplane"),           # a layer narrower than beta
    ("W20-D100", 2, "circle"),
]


def _dense_Z(dnet, beta, nbq, Q):
    import nnsdp_b200 as nb

    Z = nb.assemble_dense(dnet, beta, nbq, Q=Q)
    n = int(round(np.sqrt(Z[0].size)))
    return [Z[q].reshape(n, n, order="F") for q in range(Q)]


@pytest.mark.parametrize("xdims,beta,kind", CASES)
def test_certify_sound_tight_and_equal_to_restatement(ctx, xdims, beta, kind):
    import nnsdp_b200 as nb

    net = o.load_nnet(os.path.join(GOLD, "scale-I2-O2-W20-D100.nnet")) if xdims == "W20-D100" else rand_net(xdims, seed=3)
    rng = np.random.default_rng(7)
    Q = 2
    qs = [rand_query(net, beta, rng, kind=kind) for _ in range(Q)]
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    nbq = to_numeric_batch(nb, net, qs)
    Zs = _dense_Z(dnet, beta, nbq, Q)
    cl = [np.asarray(Ck) - 1 for Ck, _, _ in dnet.cliques(beta)]
    b = nb.Batch(dnet, beta, Qcap=Q, ring=1)                  # two passes through one slot
    b.set_inputs(nbq)
    b.bounds()
    b.prepare()
    lam = np.array([np.linalg.eigvalsh(Z).max() for Z in Zs])
    scale = np.array([np.abs(np.linalg.eigvalsh(Z)).max() for Z in Zs])
    for tau, want in ((lam - 1e-9 * scale, 0), (lam + 1e-8 * scale, 1)):
        cert, bound, fidx, minp = b.certify(tau)
        assert (cert == want).all(), (cert, want)
        for q in range(Q):
            rc, rb, rf, rp = oc.certify_multifrontal(Zs[q], cl, tau[q])
            assert rc == want and fidx[q] == rf
            assert abs(minp[q] - rp) <= 1e-9 * scale[q], (minp[q], rp)
            assert abs(bound[q] - rb) <= 1e-12 * scale[q] + abs(tau[q]) * 1e-15
            if want:
                assert lam[q] <= bound[q] <= tau[q] and fidx[q] == -1 and minp[q] > 0
            else:
                assert 0 <= fidx[q] < Zs[q].shape[0] and not minp[q] > 0
    b.close()


def test_gate_query_certifies_zero_without_iteration_cap(ctx):
    """The non-convergence query of test_gpu_parity (lambda_max = -2e-9 against a spectral scale of 4, where Lanczos
    needs ~700 iterations): the factorisation proves eigmax(Z) <= 0 in one call."""
    import nnsdp_b200 as nb

    xdims, beta = [2, 300, 300, 2], 1
    net = rand_net(xdims, seed=1, sigma=0.0)
    rng = np.random.default_rng(0)
    q = rand_query(net, beta, rng, kind="hplane", radius=0.1)
    q.gsec[:] = 0.0
    q.gbnd[:] = rng.uniform(0.5, 2.0, q.gbnd.size)
    q.gbnd[17] = 1e-9
    q.qc_out = o.QcReachHplane(np.zeros(2))
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    b = nb.Batch(dnet, beta, Qcap=1, ring=1)
    b.set_inputs(to_numeric_batch(nb, net, [q]))
    b.bounds()
    b.prepare()
    Z = o.run_query(net, beta, q, form="closed")["Z"]
    lam = np.linalg.eigvalsh(Z).max()
    cert, bound, fidx, minp = b.certify(0.0)
    assert cert[0] == 1 and lam <= bound[0] <= 0.0
    cert, _, fidx, _ = b.certify(lam - 1e-9 * 4)
    assert cert[0] == 0 and fidx[0] >= 0
    b.close()


def test_recorded_optimum_minimiser(ctx):
    """The minimiser gamma* of the reference's scale experiment (DESIGN.md section 1, CROWN bounds): the acceptance
    gate eigmax(Z) <= 1e-4 is certified; tau below lambda_max is not."""
    import json

    import nnsdp_b200 as nb

    res = json.load(open(os.path.join(GOLD, "scale_W10_D10_optimum.json")))
    net = o.load_nnet(os.path.join(GOLD, "scale-I2-O2-W10-D10.nnet"))
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
        Z = o.run_query(net, beta, q, intv_info=info)["Z"]
        ev = np.linalg.eigvalsh(0.5 * (Z + Z.T))
        lam, scale = ev[-1], np.abs(ev).max()
        b = nb.Batch(dnet, beta, Qcap=1, ring=1)
        b.set_inputs(to_numeric_batch(nb, net, [q]))
        b.set_bounds_method("crown")
        b.bounds_crown()
        b.prepare()
        cert, bound, _, _ = b.certify(1e-4)
        assert cert[0] == 1 and bound[0] <= 1e-4 and bound[0] >= lam - 1e-9 * scale
        cert, _, fidx, _ = b.certify(lam - 1e-9 * scale)
        assert cert[0] == 0 and fidx[0] >= 0
        b.close()


def test_ring_contract_repeatability_and_stride(ctx):
    """After certify the slots hold factors; run and get_slot must still equal a fresh batch bit for bit.  Two calls
    give the same bits; a scalar tau (stride 0) equals the same tau per query."""
    import nnsdp_b200 as nb

    xdims, beta, Q = [5] + [50] * 6 + [5], 2, 5
    net = rand_net(xdims, seed=4)
    rng = np.random.default_rng(4)
    qs = [rand_query(net, beta, rng, kind="safety") for _ in range(Q)]
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    nbq = to_numeric_batch(nb, net, qs)

    def fresh():
        b = nb.Batch(dnet, beta, Qcap=Q, ring=2)
        b.set_inputs(nbq)
        b.bounds()
        b.prepare()
        return b

    ref = fresh()
    want = np.zeros((Q, ref.per_query))
    ref.run(want)
    slots_want = [ref.get_slot(s) for s in range(2)]
    b = fresh()
    r1 = b.certify(0.0)
    r2 = b.certify(0.0)
    for x, y in zip(r1, r2):
        assert np.array_equal(x, y)
    r3 = b.certify(np.zeros(Q))
    for x, y in zip(r1, r3):
        assert np.array_equal(x, y)
    got = np.zeros_like(want)
    b.run(got)
    assert np.array_equal(got, want)
    for s in range(2):
        assert np.array_equal(b.get_slot(s), slots_want[s])
    b.close()
    ref.close()


def test_error_codes(ctx):
    import ctypes as C

    import nnsdp_b200 as nb
    import nnsdp_b200._lib as L

    xdims, beta = [2, 10, 10, 2], 1
    net = rand_net(xdims, seed=2)
    q = rand_query(net, beta, np.random.default_rng(2))
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    nbq = to_numeric_batch(nb, net, [q])
    b = nb.Batch(dnet, beta, Qcap=1, ring=1)
    b.set_inputs(nbq)
    with pytest.raises(nb.NnsdpError) as e:
        b.certify(0.0)
    assert e.value.code == L.ERR_STATE
    b.bounds()
    b.prepare()
    with pytest.raises(nb.NnsdpError) as e:
        b.certify(np.nan)
    assert e.value.code == L.ERR_ARG
    t = np.zeros(1)
    cert, fidx = np.zeros(1, dtype=np.int32), np.zeros(1, dtype=np.int64)
    st = L.lib.nnsdp_batch_certify(b._h, t.ctypes.data_as(L.c_dp), -1, cert.ctypes.data_as(C.POINTER(L.c_i32)),
                                   t.ctypes.data_as(L.c_dp), fidx.ctypes.data_as(L.c_i64p), None)
    assert st == L.ERR_ARG
    st = L.lib.nnsdp_batch_certify(b._h, t.ctypes.data_as(L.c_dp), 0, cert.ctypes.data_as(C.POINTER(L.c_i32)),
                                   t.ctypes.data_as(L.c_dp), fidx.ctypes.data_as(L.c_i64p), None)   # min_pivot NULL
    assert st == L.OK
    b.close()
    for kw in (dict(dense=True), dict(packed=True)):
        b = nb.Batch(dnet, beta, Qcap=1, ring=1, **kw)
        b.set_inputs(nbq)
        b.bounds()
        b.prepare()
        with pytest.raises(nb.NnsdpError) as e:
            b.certify(0.0)
        assert e.value.code == L.ERR_ARG
        b.close()
    b = nb.Batch(dnet, beta, Qcap=1, ring=0)
    b.set_inputs(nbq)
    b.bounds()
    with pytest.raises(nb.NnsdpError) as e:
        b.certify(0.0)
    assert e.value.code == L.ERR_ARG
    b.close()


def test_stress_size(ctx):
    """W1000-D20, beta = 2, Q = 4: tau below the Lanczos value (a lower bound of lambda_max) never certifies; tau a
    little above it does; query 0's smallest pivot equals the CPU restatement's on the blocks get_slot returns."""
    import nnsdp_b200 as nb

    xdims, beta, Q = [2] + [1000] * 19 + [2], 2, 4
    net = rand_net(xdims, seed=11)
    rng = np.random.default_rng(11)
    qs = [rand_query(net, beta, rng, kind="safety") for _ in range(Q)]
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    b = nb.Batch(dnet, beta, Qcap=Q, ring=Q)
    b.set_inputs(to_numeric_batch(nb, net, qs))
    b.bounds()
    b.prepare()
    lo, _, _, _ = b.lambda_max(max_iters=300, tol=1e-12, full=True)
    b.emit(0, 1)
    blocks = nb.split_blocks(b.get_slot(0), dnet.cliques(beta))
    # spectral scale: at least |lambda_max| (~1.7e16 here, a dominant direction) and the largest entry of query 0
    scale = np.maximum(np.abs(lo), max(np.abs(B).max() for B in blocks))
    cert, _, fidx, _ = b.certify(lo - 1e-6 * scale)
    assert (cert == 0).all() and (fidx >= 0).all()
    cert, bound, fidx, minp = b.certify(lo + 1e-6 * scale)
    assert (cert == 1).all() and (bound <= lo + 1e-6 * scale).all() and (bound >= lo).all()
    cl = [np.asarray(Ck) - 1 for Ck, _, _ in dnet.cliques(beta)]
    rc, rb, rf, rp = oc.certify_fronts(blocks, cl, lo[0] + 1e-6 * scale[0])
    assert rc == 1 and abs(minp[0] - rp) <= 1e-9 * scale[0]
    b.close()
