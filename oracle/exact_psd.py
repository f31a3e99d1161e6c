"""High-precision inertia of an FP64 symmetric matrix (test infrastructure only): an independent reference for the
certificate eigmax(Z) <= tau and for the interval of Batch.lambda_max_bracket.  It shares nothing with the device
plan or with oracle/certify.py: no panels, no margin, no clique layout.

    count_above(Z, t)          the number of eigenvalues of Z above t, from the signs of the pivots of an LDL' of
                               t I - Z in PREC-bit arithmetic (Sylvester's law of inertia)
    lambda_star(Z, lo, hi)     a bracket lo < lambda_max(Z) <= hi narrowed by bisection on count_above

Z is taken exactly as the FP64 matrix it is (only its lower triangle is read); t may be a float or an mpmath mpf.
Exact zeros of Z are skipped and fill is created where the elimination makes it, so a chordal Z eliminated in a
perfect elimination order costs only its clique blocks.  A pivot of magnitude below 2^-120 max|Z| raises
Inconclusive: the sign count is then not trusted.
"""
import numpy as np
from mpmath import libmp, mp, mpf

PREC = 256
_RND = libmp.round_nearest
_ZERO = libmp.fzero


class Inconclusive(ArithmeticError):
    """A pivot of the LDL' is too small for its sign to be trusted."""


def _columns(Z):
    """Lower triangle of -Z as sparse columns {row: mpf tuple}, exact (a double is exactly a 53-bit mpf)."""
    Z = np.asarray(Z, dtype=np.float64)
    if Z.ndim != 2 or Z.shape[0] != Z.shape[1]:
        raise ValueError("Z must be square")
    if not np.isfinite(Z).all():
        raise ValueError("Z has a non-finite entry")
    n = Z.shape[0]
    L = np.tril(Z)
    cols = []
    for j in range(n):
        rows = np.nonzero(L[:, j])[0]
        cols.append({int(i): libmp.from_float(-float(L[i, j])) for i in rows})
    return cols, float(np.abs(L).max()) if n else 0.0


def _pivot_signs(cols, t, thr):
    """(number of negative pivots) of the LDL' of t I - Z; cols is consumed."""
    prec = PREC
    neg = 0
    for j in range(len(cols)):
        cj = cols[j]
        d = libmp.mpf_add(t, cj.pop(j, _ZERO), prec, _RND)     # t - z_jj after the updates of earlier columns
        if d == _ZERO or libmp.mpf_cmp(libmp.mpf_abs(d), thr) < 0:
            raise Inconclusive(f"pivot {j} of t I - Z has magnitude {libmp.to_str(d, 5)}, below 2^-120 max|Z|")
        if libmp.mpf_sign(d) < 0:
            neg += 1
        items = sorted(cj.items())
        for a, (i, lij) in enumerate(items):
            f = libmp.mpf_div(lij, d, prec, _RND)
            ci = cols[i]
            for k, lkj in items[a:]:                        # rows k >= i of column i
                ci[k] = libmp.mpf_sub(ci.get(k, _ZERO), libmp.mpf_mul(f, lkj, prec, _RND), prec, _RND)
        cols[j] = None
    return neg


def count_above(Z, t):
    """Number of eigenvalues of the FP64 symmetric matrix Z (lower triangle) strictly above t."""
    cols, zmax = _columns(Z)
    thr = libmp.from_man_exp(1, -120) if zmax == 0.0 else libmp.mpf_mul(libmp.from_float(zmax),
                                                                        libmp.from_man_exp(1, -120))
    # the diagonal of t I - Z is t + (-z_jj): add t to the stored -z_jj as each pivot is formed
    tt = t._mpf_ if isinstance(t, mpf) else libmp.from_float(float(t))     # exact either way
    return _pivot_signs(cols, tt, thr)


def lambda_star(Z, lo, hi, digits=30, max_steps=400):
    """Bracket (lo, hi) of lambda_max(Z) as mpf: count_above(Z, lo) >= 1 and count_above(Z, hi) == 0, narrowed until
    hi - lo <= 10^-digits max(|lo|, |hi|).  A midpoint that is inconclusive is replaced by a few other points inside
    the bracket; when all are, bisection stops with the bracket it has (lambda_max lies within ~2^-120 max|Z| of
    them) and the caller checks the width it needs."""
    with mp.workprec(PREC):
        lo, hi = mpf(lo), mpf(hi)
        if count_above(Z, lo) < 1:
            raise ValueError("lambda_max(Z) <= lo")
        if count_above(Z, hi) != 0:
            raise ValueError("lambda_max(Z) > hi")
        tol = mpf(10) ** (-digits)
        for _ in range(max_steps):
            if hi - lo <= tol * max(abs(lo), abs(hi)):
                break
            for frac in (mpf(1) / 2, mpf(31) / 64, mpf(33) / 64, mpf(1) / 3, mpf(2) / 3):
                mid = lo + (hi - lo) * frac     # any point inside works; the middle may sit on a zero pivot
                try:
                    above = count_above(Z, mid)
                    break
                except Inconclusive:
                    pass
            else:
                break
            if above:
                lo = mid
            else:
                hi = mid
        return lo, hi
