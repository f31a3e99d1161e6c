"""The entrywise reference of Z (oracle/exact_z.py) and its rounding bound, on the CPU.

|Z_fp64[r,c] − ref[r,c]| ≤ γ_N·abs[r,c] + N·2⁻¹⁰⁷⁴ (entries with abs = 0 exactly 0) is checked for every entry.  Here:
the exact (Fraction) and extended (long double) modes agree; the oracle's independent FP64 closed form meets the bound
on every CPU shape and output kind, so the bound is not too tight; and four small bugs that the normwise criterion
(max |a − b| ≤ 1e-12 · max |b| per clique block) lets through are caught by it."""
from fractions import Fraction

import numpy as np
import pytest

import exact_z as ez
import nnsdp_oracle as o
from helpers import assert_meets, rand_net, rand_query, relerr, wide_range_case

KINDS = ["safety", "hplaneS", "hplane", "circle", "ellipsoid"]

# the shapes of the parity suite that the CPU can take in exact arithmetic, and a few more
SHAPES = [([2, 3, 2], 0), ([2, 3, 2], 2), ([2, 3, 3, 2], 1), ([3, 3, 3, 3, 4, 3, 3], 2), ([2, 10, 10, 10, 10, 2], 3),
          ([2, 4, 7, 3, 5, 2], 5), ([2, 1, 2, 2], 3), ([2] + [10] * 9 + [2], 7)]


def oracle_case(xdims, beta, kind, seed, radius=0.3):
    """(net, query, IBP bounds as the given QC bounds, the oracle's FP64 Z)."""
    net = rand_net(xdims, seed=seed)
    q = rand_query(net, beta, np.random.default_rng(seed), kind=kind, radius=radius)
    r = o.run_query(net, beta, q)
    bounds = (r["qc_bounded"].acymin, r["qc_bounded"].acymax, r["qc_sector"].smin, r["qc_sector"].smax)
    return net, q, bounds, r["Z"]


def oracle_Z(net, beta, q, bounds):
    ymin, ymax, smin, smax = bounds
    return o.assemble_Z_closed_form(net, o.QcInputBox(q.x1min, q.x1max), q.qc_out, o.QcActivBounded(net.acdim, ymin, ymax),
                                    o.QcActivSector(net.acdim, beta, smin, smax), q.gin, q.gbnd, q.gsec, q.gout)


# ---- the two arithmetic modes agree --------------------------------------------------------------------------------

@pytest.mark.parametrize("beta", range(8))
def test_exact_and_extended_modes_agree(beta):
    xdims = [2, 4, 7, 3, 5, 2] if beta % 2 else [3, 3, 3, 3, 4, 3, 3]
    for i, kind in enumerate(KINDS):
        net, q, bounds = wide_range_case(xdims, beta, kind, seed=10 * beta + i)
        X = ez.exact_z(net, beta, q, bounds, mode="exact")
        E = ez.exact_z(net, beta, q, bounds, mode="extended")
        assert np.array_equal(X.N, E.N) and np.array_equal(X.abs == 0, E.abs == 0)
        assert (E.abs >= X.abs).all()
        ext = np.frompyfunc(lambda v: Fraction(*v.as_integer_ratio()), 1, 1)(E.ref)
        err = np.abs(ext - X.ref)
        # in exact arithmetic: the subnormal entries (|ref| ~ 1e-325) would underflow a float64 tolerance
        u = Fraction(ez.UEXT)
        assert all(e <= (n * u / (1 - n * u)) * a for e, n, a in zip(err.ravel(), E.N.ravel().tolist(),
                                                                      X._abs_exact.ravel())), kind


def test_reference_on_a_hand_worked_entry():
    """[1, 1, 1] net, beta = 0: Z[x_1, x_1] = S11 − 2γin + w²·d11 with d11 = −2·smin·smax·λ, checked by hand."""
    w, bi, w2, b2 = 3.0, 0.5, 2.0, -1.0
    net = o.FeedFwdNet(xdims=[1, 1, 1], Ms=[np.array([[w, bi]]), np.array([[w2, b2]])])
    S = np.array([[1.0, 2.0, 3.0], [2.0, 5.0, 7.0], [3.0, 7.0, 11.0]])
    q = o.NumericQuery(x1min=np.array([-1.0]), x1max=np.array([2.0]), gin=np.array([0.25]), gbnd=np.array([0.5]),
                       gsec=np.array([0.125, 0.75, 1.5]), qc_out=o.QcSafety(S=S))
    bounds = (np.array([-2.0]), np.array([4.0]), np.array([0.5]), np.array([1.0]))
    R = ez.exact_z(net, 0, q, bounds)
    d11 = -2 * 0.5 * 1.0 * 0.125
    assert R.ref[0, 0] == 1.0 - 2 * 0.25 + w * w * d11
    assert R.N[0, 0] == 3 + ez.CHAIN + 2                      # S11, −2γin, the Gram term
    # Z[x_2, x_2] = −2γbnd + w2² S22;  Z[x_1, x_2] = w (smin + smax) λ + S12 w2
    assert R.ref[1, 1] == -2 * 0.5 + w2 * 5.0 * w2
    assert R.ref[0, 1] == w * (0.5 + 1.0) * 0.125 + 2.0 * w2
    assert R.abs[0, 1] == w * 1.5 * 0.125 + 2.0 * w2 and R.N[0, 1] == 3 + ez.CHAIN + 2
    assert np.array_equal(R.ref, R.ref.T)


# ---- the oracle's FP64 evaluation meets the bound ------------------------------------------------------------------

@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("xdims,beta", SHAPES)
def test_oracle_closed_form_meets_the_entrywise_bound(xdims, beta, kind):
    """An independent FP64 evaluation in another order (numpy, BLAS) is within the bound: the bound is not too tight."""
    net, q, bounds, Z = oracle_case(xdims, beta, kind, seed=len(xdims) + beta)
    assert_meets(ez.exact_z(net, beta, q, bounds), Z, "IBP bounds")
    net, q, bounds = wide_range_case(xdims, beta, kind, seed=len(xdims) + beta)
    assert_meets(ez.exact_z(net, beta, q, bounds), oracle_Z(net, beta, q, bounds), "wide range")


@pytest.mark.parametrize("kind", ["hplane", "circle", "ellipsoid", "hplaneS"])
def test_reach_kinds_and_hplaneS_meet_the_bound(kind):
    """S built from γout (hplane, circle, ellipsoid) and the safety S of o.hplaneS: the literal Julia restatement
    (R' Q R with sparse selectors, a third evaluation order) meets the bound as well."""
    xdims, beta = [2, 6, 5, 7, 3], 2
    net, q, bounds, _ = oracle_case(xdims, beta, kind, seed=3)
    R = ez.exact_z(net, beta, q, bounds)
    assert_meets(R, o.run_query(net, beta, q, form="literal")["Z"], "literal")
    assert_meets(R, oracle_Z(net, beta, q, bounds), "closed")


# ---- mutations the normwise criterion lets through -----------------------------------------------------------------

def _caught_only_entrywise(R, Z, Zmut, net, beta, entry):
    """The mutation breaks the entrywise bound at `entry` and nowhere else, but meets relerr ≤ 1e-12 per block."""
    assert_meets(R, Z, "unmutated")
    ok, ratio = R.check(Zmut)
    assert not ok[entry], ratio[entry]
    bad = set(zip(*np.nonzero(~ok)))
    assert bad <= {entry, entry[::-1]}, bad
    cl = o.make_cliques(net, beta)
    for Bm, B in zip(o.clique_blocks(Zmut, cl), o.clique_blocks(Z, cl)):
        assert relerr(Bm, B) <= 1e-12


def test_mutation_dropped_gram_term_of_a_small_d11():
    xdims, beta = [2, 5, 6, 2], 1
    net, q, bounds, _ = oracle_case(xdims, beta, "safety", seed=4, radius=0.0)
    smin, smax = bounds[2].copy(), bounds[3].copy()
    smin[:], smax[:] = 1.0, 1.0                         # every neuron Gram-active
    j = 2                                               # neuron 2 of layer 1: small λ
    q.gsec[j] = 1e-12
    bounds = (bounds[0], bounds[1], smin, smax)
    Z = oracle_Z(net, beta, q, bounds)
    R = ez.exact_z(net, beta, q, bounds)
    w = net.Ms[0][j, :-1]
    r, c = 0, 1
    Zm = Z.copy()
    Zm[r, c] -= w[r] * (-2.0 * q.gsec[j]) * w[c]
    Zm[c, r] = Zm[r, c]
    _caught_only_entrywise(R, Z, Zm, net, beta, (r, c))


def test_mutation_band_tap_shifted_across_a_layer_boundary():
    """The -2 T[i, j] tap of the last neuron i of layer 1 and the first neuron j = i + 1 of layer 2, taken from the
    pair (i - 1, j - 1) instead; the band multipliers near the boundary are small."""
    xdims, beta = [2, 4, 5, 2], 1
    net, q, bounds, Z = oracle_case(xdims, beta, "circle", seed=5)
    ac, n1 = net.acdim, xdims[0]
    pairs = o.sector_pairs(ac, beta) - 1
    i = xdims[1] - 1
    k_right = int(np.nonzero((pairs[:, 0] == i) & (pairs[:, 1] == i + 1))[0][0])
    k_wrong = int(np.nonzero((pairs[:, 0] == i - 1) & (pairs[:, 1] == i))[0][0])
    q.gsec[ac + k_right], q.gsec[ac + k_wrong] = 3e-13, 1e-13
    Z = oracle_Z(net, beta, q, bounds)
    R = ez.exact_z(net, beta, q, bounds)
    r, c = n1 + i, n1 + i + 1
    Zm = Z.copy()
    Zm[r, c] += 2.0 * (q.gsec[ac + k_wrong] - q.gsec[ac + k_right])
    Zm[c, r] = Zm[r, c]
    _caught_only_entrywise(R, Z, Zm, net, beta, (r, c))


def test_mutation_negated_small_S12_WK_entry():
    xdims, beta = [2, 4, 4, 4, 3], 1
    net, q, bounds, _ = oracle_case(xdims, beta, "safety", seed=6)
    n1, nK1 = xdims[0], xdims[-1]
    S = q.qc_out.S.copy()
    S[:n1, n1:n1 + nK1] *= 1e-13
    S[n1:n1 + nK1, :n1] = S[:n1, n1:n1 + nK1].T
    q.qc_out = o.QcSafety(S=S)
    Z = oracle_Z(net, beta, q, bounds)
    R = ez.exact_z(net, beta, q, bounds)
    r, c = 1, sum(xdims[:-2]) + 2                       # x_1[1] against x_K[2]: only S12 W_K there
    assert Z[r, c] != 0 and abs(Z[r, c]) < 1e-11 * np.abs(Z).max()
    Zm = Z.copy()
    Zm[r, c] = Zm[c, r] = -Z[r, c]
    _caught_only_entrywise(R, Z, Zm, net, beta, (r, c))


def test_mutation_Zaa_off_by_1e_13_of_the_block_scale():
    xdims, beta = [2, 3, 2], 0
    net, q, bounds, Z = oracle_case(xdims, beta, "hplane", seed=7)
    R = ez.exact_z(net, beta, q, bounds)
    a = net.Zdim - 1
    scale = np.abs(Z).max()
    Zm = Z.copy()
    Zm[a, a] += 1e-13 * scale
    _caught_only_entrywise(R, Z, Zm, net, beta, (a, a))
