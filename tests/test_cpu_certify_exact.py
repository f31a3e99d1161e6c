"""The certificate eigmax(Z) <= tau of the CPU restatement (oracle/certify.py) against an independent 256-bit reference
(oracle/exact_psd.py: inertia of t I - Z by an LDL' in mpmath).  First the reference itself on matrices whose
eigenvalues are known exactly, then the restatement's claims at tau within a few ulps, c/10, c and 10c of the exact
lambda_max (c = the rounding-error margin): a certified bound is never below lambda_max, a failed factorisation's
lower bound is never above it, and tau >= lambda_max + 100 c always certifies."""
import math
import os

import numpy as np
import pytest
from mpmath import mp, mpf

import certify as oc
import exact_psd as ex
import nnsdp_oracle as o
from helpers import rand_net, rand_query

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


# ---- the reference on exact cases ---------------------------------------------------------------------------------

def _perm_similar(D, seed):
    """P D P' for a random signed permutation P: exact in FP64, same eigenvalues."""
    rng = np.random.default_rng(seed)
    n = D.shape[0]
    P = np.zeros((n, n))
    P[rng.permutation(n), np.arange(n)] = rng.choice([-1.0, 1.0], n)
    return P @ D @ P.T


@pytest.mark.parametrize("t", [1.0, -3.0, 2.0 ** -700, 1e300, -0.1])
def test_reference_counts_eigenvalues_one_ulp_either_side(t):
    up, dn = math.nextafter(t, math.inf), math.nextafter(t, -math.inf)
    ev = np.array([up, dn, t - 5 * abs(t), t + 7 * abs(t), up, dn])
    for Z in (np.diag(ev), _perm_similar(np.diag(ev), 1)):
        assert ex.count_above(Z, t) == 3
        assert ex.count_above(Z, math.nextafter(up, math.inf)) == 1
        assert ex.count_above(Z, math.nextafter(dn, -math.inf)) == 5
        with pytest.raises(ex.Inconclusive):
            ex.count_above(Z, up)                 # an eigenvalue exactly at t: a zero pivot
    # [[t + 3d, 4d], [4d, t - 3d]] has the eigenvalues t +- 5d exactly, and no zero pivot at t
    d = up - t
    R = np.zeros((6, 6))
    R[:2, :2] = [[t + 3 * d, 4 * d], [4 * d, t - 3 * d]]
    R[2:, 2:] = np.diag([t - 5 * abs(t), t - 6 * abs(t), t - 7 * abs(t), t - 8 * abs(t)])
    for Z in (R, _perm_similar(R, 2)):
        assert ex.count_above(Z, t) == 1
        assert ex.count_above(Z, math.nextafter(t + 5 * d, math.inf)) == 0
        assert ex.count_above(Z, math.nextafter(t - 5 * d, -math.inf)) == 2


def test_reference_exact_zero_eigenvalue_is_inconclusive():
    rng = np.random.default_rng(0)
    B = rng.integers(-4, 5, (7, 6)).astype(float)
    A = B @ B.T                                   # PSD, rank 6: an exact zero eigenvalue
    with pytest.raises(ex.Inconclusive):
        ex.count_above(A, 0.0)
    with pytest.raises(ex.Inconclusive):
        ex.count_above(-A, 0.0)
    assert ex.count_above(A, -1e-3) == 7 and ex.count_above(-A, 1e-3) == 0


def test_lambda_star_thirty_digits():
    with mp.workprec(256):
        phi = (1 + mp.sqrt(5)) / 2                # lambda_max of [[1, 1], [1, 0]]
        Z = np.array([[1.0, 1.0], [1.0, 0.0]])
        lo, hi = ex.lambda_star(Z, 1.5, 2.0)
        assert lo < phi <= hi and hi - lo <= mpf(10) ** -30 * phi
        s = 2.0 ** -600                           # 2 + sqrt(2) of the tridiagonal [1, 2, 1], scaled
        lam = (2 + mp.sqrt(2)) * s
        Z = s * (2 * np.eye(3) + np.eye(3, k=1) + np.eye(3, k=-1))
        lo, hi = ex.lambda_star(_perm_similar(Z, 3), 3.25 * s, 3.5 * s)
        assert lo < lam <= hi and hi - lo <= mpf(10) ** -30 * lam


# ---- the restatement against the reference -------------------------------------------------------------------------

def _random_case(kind, beta):
    net = rand_net([2] + [10] * 9 + [2], seed=20 + beta)
    q = rand_query(net, beta, np.random.default_rng(30 + beta), kind=kind)
    ref = o.run_query(net, beta, q, form="closed")
    return 0.5 * (ref["Z"] + ref["Z"].T), [np.asarray(Ck) - 1 for Ck, _, _ in ref["cliques"]]


def _stored_case(name):
    import sdp_decomposed as sd

    h = np.load(os.path.join(GOLD, f"handoff_{name}.npz"))
    sol = np.load(os.path.join(GOLD, f"decomposed_{name}_single_from_dense.npz"))
    cliques = sd.cliques_from_npz(h)
    prob = sd.problem_from_handoff(h, cliques, "single")
    Z0, A = sd.dense_from_handoff(h, prob["keep"])
    return Z0 + np.tensordot(sol["x"][:prob["ng"]], A, 1), [Ck - 1 for Ck, _, _ in cliques]


def _lambda_star(Z):
    """fl(lambda_max) with an exact bracket narrower than a tenth of an ulp around it."""
    ev = np.linalg.eigvalsh(Z)
    s = np.abs(ev).max()
    lo, hi = ex.lambda_star(Z, ev[-1] - 1e-10 * s, ev[-1] + 1e-10 * s, digits=30)
    lam = float(hi)
    assert hi - lo <= 0.1 * (math.nextafter(lam, math.inf) - lam)
    return lam, lo, hi


def sweep_taus(lam, c):
    """tau = lambda* + {+-1, +-4 ulps, +-c/10, +-c, +-10c, +100c}."""
    taus = []
    for k in (1, 4):
        up = dn = lam
        for _ in range(k):
            up, dn = math.nextafter(up, math.inf), math.nextafter(dn, -math.inf)
        taus += [up, dn]
    return taus + [lam + f * c for f in (0.1, -0.1, 1.0, -1.0, 10.0, -10.0, 100.0)]


def check_sweep(Z, lam_lo, lam_hi, lam, c, outcome):
    """outcome(tau) -> (certified, bound, lower or None).  Exact checks of every claim at every tau of the sweep."""
    seen = set()
    for tau in sweep_taus(lam, c):
        cert, bound, lower = outcome(tau)
        seen.add(cert)
        if cert:
            assert bound <= tau and ex.count_above(Z, bound) == 0, (tau, bound)
        elif lower is not None and np.isfinite(lower):
            assert ex.count_above(Z, lower) >= 1, (tau, lower)
            assert lower >= lam - 100 * c
        if tau >= lam_hi + 100 * c:
            assert cert == 1, tau
        if tau <= lam_lo:
            assert cert == 0, tau
    assert seen == {0, 1}


def _stats(Z):
    d = np.diag(Z)
    return float(np.sum(d)), float(np.sum(np.abs(d))), float(np.max(np.abs(d)))


def _restatement(Z, cl):
    trz, sabs, mabs = _stats(Z)

    def run(tau):
        cert, bound, _, _ = oc.certify_multifrontal(Z, cl, tau)
        tp, _ = oc.certify_shift(tau, Z.shape[0], trz, sabs, mabs)
        return cert, bound, None if cert else oc.certify_lower(tp, Z.shape[0], mabs)
    return run


@pytest.mark.parametrize("kind,beta", [("safety", 2), ("hplane", 1), ("circle", 3), ("ellipsoid", 0)])
def test_restatement_exact_sweep_random(kind, beta):
    Z, cl = _random_case(kind, beta)
    lam, lo, hi = _lambda_star(Z)
    c = oc.certify_margin(lam, Z.shape[0], *_stats(Z))
    check_sweep(Z, lo, hi, lam, c, _restatement(Z, cl))


@pytest.mark.parametrize("name", ["W10-D10_beta0", "W10-D10_beta2"])
def test_restatement_exact_sweep_stored_optimum(name):
    """lambda* ~ -8e-10 against ||Z|| ~ 2e4: numpy's eigvalsh is not a lower bound here, the exact bracket is."""
    Z, cl = _stored_case(name)
    lam, lo, hi = _lambda_star(Z)
    assert lam < 0
    c = oc.certify_margin(lam, Z.shape[0], *_stats(Z))
    check_sweep(Z, lo, hi, lam, c, _restatement(Z, cl))


def test_margin_lower_mirror_against_exact_diagonal():
    """certify_lower on a diagonal Z where the factorisation fails at the exact eigenvalue: the bound is below it."""
    t = 0.75
    Z = _perm_similar(np.diag([t, -1.0, 0.5, t - 2.0 ** -30]), 4)
    trz, sabs, mabs = _stats(Z)
    tp, _ = oc.certify_shift(t, 4, trz, sabs, mabs)
    cert, _, _, _ = oc.certify_multifrontal(Z, [np.arange(4)], t)
    assert cert == 0
    low = oc.certify_lower(tp, 4, mabs)
    assert low < tp and ex.count_above(Z, low) >= 1
    assert oc.certify_lower(0.0, 4, np.inf) == -math.inf
