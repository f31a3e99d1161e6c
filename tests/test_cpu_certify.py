"""The certificate eigmax(Z) <= tau without a GPU: the elimination plan of nnsdp_batch_certify (host only) passes its
layout checks and agrees with the CPU restatement's, and the restatement (oracle/certify.py) is sound and tight on the
oracle's dense Z."""
import os

import numpy as np
import pytest

import certify as oc
import nnsdp_oracle as o
from helpers import rand_net, rand_query

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
KINDS = ("safety", "hplane", "circle", "ellipsoid")
SHAPES = [([2] + [10] * 9 + [2], b) for b in range(4)] + [
    ([5] + [50] * 6 + [5], 2),          # ACAS-shaped
    ([2, 10, 3, 10, 2], 4),             # a layer narrower than beta
    ([3, 6, 2, 1, 7, 3], 5),            # several of them, and a 1-neuron layer
    ([2, 8, 2], 1),                     # one hidden layer: a single clique
]


def _cliques0(xdims, beta):
    import nnsdp_b200 as nb

    return [np.asarray(Ck, dtype=np.int64) - 1 for Ck, _, _ in nb.cliques_from_xdims(xdims, beta)]


def _check_plan(xdims, beta):
    import nnsdp_b200 as nb

    plan = nb.certify_plan(xdims, beta)
    cl = _cliques0(xdims, beta)
    zdim = sum(xdims[:-1]) + 1
    assert len(plan) == len(cl)
    ref = oc.front_plan(cl, zdim)
    off = 0
    for (out_off, n, npriv, g0, lead, tail), c, (rp, rl, rt) in zip(plan, cl, ref):
        assert (out_off, n, npriv, g0, lead, tail) == (off, len(c), rp, c[0], rl, rt)
        off += n * n
    assert plan[-1][2] == plan[-1][1]                                    # the last front is all private
    assert sum(n - lead - tail for _, n, _, _, lead, tail in plan) == zdim   # every diagonal entry shifted once


@pytest.mark.parametrize("xdims,beta", SHAPES)
def test_plan_layout(xdims, beta):
    _check_plan(xdims, beta)


def test_plan_layout_w20_d100():
    net = o.load_nnet(os.path.join(GOLD, "scale-I2-O2-W20-D100.nnet"))
    for beta in (0, 2, 7):
        _check_plan(list(net.xdims), beta)


def _dense(xdims, beta, kind, seed):
    net = rand_net(xdims, seed=seed)
    q = rand_query(net, beta, np.random.default_rng(seed), kind=kind)
    ref = o.run_query(net, beta, q, form="closed")
    Z = 0.5 * (ref["Z"] + ref["Z"].T)
    return Z, [np.asarray(Ck) - 1 for Ck, _, _ in ref["cliques"]]


def _sound_and_tight(Z, cl):
    ev = np.linalg.eigvalsh(Z)
    lam, scale = ev[-1], max(abs(ev[0]), abs(ev[-1]))
    for rel in (1e-9, 1e-3):
        cert, bound, fidx, minp = oc.certify_multifrontal(Z, cl, lam - rel * scale)
        assert cert == 0 and 0 <= fidx < Z.shape[0] and not minp > 0
    tau = lam + 1e-8 * scale
    cert, bound, fidx, minp = oc.certify_multifrontal(Z, cl, tau)
    assert cert == 1 and fidx == -1 and minp > 0
    assert lam <= bound <= tau


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("xdims,beta", SHAPES[:6])
def test_restatement_sound_and_tight(xdims, beta, kind):
    Z, cl = _dense(xdims, beta, kind, seed=len(xdims) + beta)
    _sound_and_tight(Z, cl)


def test_restatement_w20_d100():
    net = o.load_nnet(os.path.join(GOLD, "scale-I2-O2-W20-D100.nnet"))
    q = rand_query(net, 2, np.random.default_rng(5), kind="circle")
    ref = o.run_query(net, 2, q, form="closed")
    _sound_and_tight(0.5 * (ref["Z"] + ref["Z"].T), [np.asarray(Ck) - 1 for Ck, _, _ in ref["cliques"]])


def test_margin_is_an_upper_rounding():
    """bound = tau' + c(tau') <= tau, and c grows with Zdim and with the trace of tau' I - Z."""
    tp, bound = oc.certify_shift(1e-4, 1000, -50.0, 50.0, 1.0)
    assert tp < 1e-4 and bound <= 1e-4 and bound > tp
    c1 = oc.certify_margin(0.0, 1000, -50.0, 50.0, 1.0)
    assert c1 < oc.certify_margin(0.0, 2000, -50.0, 50.0, 1.0) and c1 < oc.certify_margin(0.0, 1000, -100.0, 100.0, 1.0)
    # (Zdim + 1) u / (1 - ...) times the trace, to a few ulps
    assert abs(c1 / (50.0 * (1001 * 2.0 ** -52 + 2.0 ** -52)) - 1) < 1e-2


@pytest.mark.parametrize("name", [n for n in [f"W10-D10_beta{b}" for b in range(8)] + ["W10-D20_beta2"]
                                  if os.path.exists(os.path.join(GOLD, f"decomposed_{n}_single_from_dense.npz"))])
def test_stored_dense_optimum_certifies(name):
    """The point stored from the dense optimum (every decomposed block <= -2e-11) has eigmax(Z(gamma)) ~ -2e-9 against
    ||Z|| ~ 2e4: 1e-13 relative, below what a rounding-error-certified FP64 factorisation resolves (c(0) ~ 1e-8 here).
    What is provable is proven: Z(gamma) <= 1e-7 I, and the acceptance gate eigmax(Z) <= 1e-4 (experiments/acas.jl)."""
    import sdp_decomposed as sd

    h = np.load(os.path.join(GOLD, f"handoff_{name}.npz"))
    sol = np.load(os.path.join(GOLD, f"decomposed_{name}_single_from_dense.npz"))
    cliques = sd.cliques_from_npz(h)
    prob = sd.problem_from_handoff(h, cliques, "single")
    Z0, A = sd.dense_from_handoff(h, prob["keep"])
    Zg = Z0 + np.tensordot(sol["x"][:prob["ng"]], A, 1)
    lam = np.linalg.eigvalsh(Zg).max()
    assert lam < 0.0
    for tau in (1e-7, 1e-4):
        cert, bound, fidx, minp = oc.certify_multifrontal(Zg, [Ck - 1 for Ck, _, _ in cliques], tau)
        assert cert == 1 and lam <= bound <= tau and fidx == -1
