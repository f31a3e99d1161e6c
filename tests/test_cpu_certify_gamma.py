"""Host side of the certificate for the exact Z(γ) (nnsdp_batch_certify_gamma): the monomial count Nmax of the
assembly-error bound against oracle/exact_z.py, and count_above_exact, the inertia of a matrix of Fractions (the exact
Z(γ) of exact_z) that the GPU tests check the certificate with."""
from fractions import Fraction

import numpy as np
import pytest
from mpmath import libmp, mpf

import exact_psd as ex
import exact_z as ez
import nnsdp_oracle as o
from helpers import rand_net, rand_query


def count_above_exact(Z, t):
    """Number of eigenvalues of the symmetric matrix Z of Fractions with power-of-two denominators (lower triangle)
    strictly above t: the LDL' of exact_psd.count_above, every entry of Z converted exactly (an mpf of as many bits as
    it needs), so that only the elimination rounds, as for an FP64 Z.  Raises exact_psd.Inconclusive like count_above
    (threshold 2^-120 max|Z|)."""
    Z = np.asarray(Z, dtype=object)
    if Z.ndim != 2 or Z.shape[0] != Z.shape[1]:
        raise ValueError("Z must be square")
    n = Z.shape[0]
    cols, zmax = [], libmp.fzero
    for j in range(n):
        col = {}
        for i in range(j, n):
            v = Fraction(Z[i, j])
            if v == 0:
                continue
            den = v.denominator
            if den & (den - 1):
                raise ValueError(f"Z[{i},{j}] = {v} is not dyadic")
            col[i] = libmp.from_man_exp(-v.numerator, -(den.bit_length() - 1))     # -z_ij, exact
            if libmp.mpf_cmp(libmp.mpf_abs(col[i]), zmax) > 0:
                zmax = libmp.mpf_abs(col[i])
        cols.append(col)
    scale = libmp.from_man_exp(1, -120)
    thr = scale if zmax == libmp.fzero else libmp.mpf_mul(zmax, scale, ex.PREC, libmp.round_nearest)
    tt = t._mpf_ if isinstance(t, mpf) else libmp.from_float(float(t))
    return ex._pivot_signs(cols, tt, thr)


KINDS = {"safety": 0, "hplane": 1, "circle": 2, "ellipsoid": 3}

# W10-D10, the edge shapes of the certify kernels, β = 0 .. 7 with layers narrower than β, a wide output layer
SHAPES = [
    ([2] + [10] * 9 + [2], 2),
    ([2, 29, 2], 2),
    ([2, 33, 1, 29, 2], 0),
    ([2, 29, 4, 31, 2], 3),
    ([3, 1, 4, 1, 2], 1),
    ([2, 1, 2, 2], 3),
    ([3, 129, 2, 129, 2], 0),
    ([2, 4, 7, 3, 5, 2], 7),
    ([3, 3, 3, 3, 4, 3, 3], 4),
    ([2, 6, 5, 9], 1),
]


@pytest.mark.parametrize("kind", list(KINDS))
@pytest.mark.parametrize("xdims,beta", SHAPES)
def test_nmax_bounds_the_monomial_count_and_is_not_vacuous(xdims, beta, kind):
    import nnsdp_b200 as nb

    net = rand_net(xdims, seed=sum(xdims) + beta)
    rng = np.random.default_rng(beta)
    q = rand_query(net, beta, rng, kind=kind)
    ac = net.acdim
    bounds = (-rng.random(ac), rng.random(ac), rng.random(ac) * 0.5, 0.5 + rng.random(ac) * 0.5)
    N = ez.exact_z(net, beta, q, bounds, mode="extended").N.max()
    nmax = nb.assembly_error_nmax(xdims, beta, KINDS[kind])
    assert N <= nmax <= 2 * N, (N, nmax)


def test_nmax_rejects_bad_arguments():
    import nnsdp_b200 as nb

    for args in (([2, 3, 2], 1, 4), ([2, 3, 2], -1, 0), ([2, 3], 1, 0)):
        with pytest.raises(nb.NnsdpError):
            nb.assembly_error_nmax(*args)


def test_exact_count_matches_the_fp64_count_on_fp64_matrices():
    rng = np.random.default_rng(5)
    for n in (1, 4, 9):
        A = rng.standard_normal((n, n))
        Z = A + A.T
        Zf = np.vectorize(Fraction, otypes=[object])(Z)
        ev = np.linalg.eigvalsh(Z)
        for t in np.concatenate([ev - 1e-9, ev + 1e-9]):
            assert count_above_exact(Zf, t) == ex.count_above(Z, t) == int((ev > t).sum())


def test_exact_count_takes_entries_beyond_fp64_exactly():
    """Entries that FP64 cannot hold (2^-1100, 1 + 2^-80) decide the count."""
    tiny = Fraction(1, 2 ** 1100)
    Z = np.array([[tiny]], dtype=object)
    assert count_above_exact(Z, 0.0) == 1 and count_above_exact(Z, 2.0 ** -1074) == 0
    Z = np.array([[1 + Fraction(1, 2 ** 80), 0], [0, -1]], dtype=object)
    assert count_above_exact(Z, 1.0) == 1
    with pytest.raises(ValueError):
        count_above_exact(np.array([[Fraction(1, 3)]], dtype=object), 0.0)


def test_exact_count_of_an_exact_z_of_the_oracle():
    """count_above_exact on exact_z's ref agrees with the eigenvalues of its FP64 rounding away from them."""
    xdims, beta = [2, 5, 4, 2], 1
    net = rand_net(xdims, seed=3)
    q = rand_query(net, beta, np.random.default_rng(3), kind="circle")
    info = o.intervals_worst_case(q.x1min, q.x1max, net)
    amin = np.concatenate([p[0] for p in info.acx_intvs])
    amax = np.concatenate([p[1] for p in info.acx_intvs])
    smin, smax = o.make_sector_min_max(amin, amax)
    ymin = np.concatenate([p[0] for p in info.x_intvs[1:-1]])
    ymax = np.concatenate([p[1] for p in info.x_intvs[1:-1]])
    R = ez.exact_z(net, beta, q, (ymin, ymax, smin, smax), mode="exact")
    Zf = np.vectorize(float)(R.ref)
    ev = np.linalg.eigvalsh(Zf)
    s = np.abs(ev).max()
    for t in np.concatenate([ev - 1e-6 * s, ev + 1e-6 * s]):
        assert count_above_exact(R.ref, t) == int((ev > t).sum())
