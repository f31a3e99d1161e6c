"""CROWN bounds of one target with a proven rounding bound (test infrastructure only).

The device's CROWN (kernels_crown.cu) bounds every pre-activation y_t = W_t x_t + b_t, t >= 1, by a backward chain
over the relaxations of relu_{t-1}, ..., relu_0, each built from the FP64 bounds (l_k, u_k) of y_k the device computed
before.  This module restates that chain on its own (it does not call `intervals_crown` / `_crown_backward`):

1. The relaxation parameters of y_k come from (l_k, u_k) in float64 with exactly the operations of
   crown_params_kernel (`relax_params`): lb_r = min(l, 0), ub_r = max(u, 0), ub_r = max(ub_r, lb_r + 1e-8),
   d_u = ub_r / (ub_r - lb_r), b_u = -lb_r * d_u, d_l = (d_u > 0.5).  Each is one correctly rounded operation and no
   two can be contracted into an fma, so these are the device's d_u, b_u, d_l bit for bit: the `> 0.5` tie and the
   1e-8 are decided on identical numbers.
2. With those FP64 numbers taken as exact rationals, the chain of target row r runs in exact arithmetic
   (`fractions.Fraction`, mode "exact") or in the 64-bit-mantissa long double (mode "extended"):
       A <- W_t[r, :], beta <- b_t[r];  for k = t-1 .. 0:
           upper: s_c = d_u if A_c > 0 else d_l,  beta += sum_c max(A_c, 0) b_u,c   (lower: A_c < 0, min(A_c, 0))
           a = s o A;  beta += a . b_k;  A <- a W_k
       lower = A c - |A| r + beta,  upper = A c + |A| r + beta,  c = (lo + hi) / 2, r = (hi - lo) / 2 exactly.

Rounding bound.  Per bound the module also returns abs (the same chain with |W|, |b_k|, |b_u| and every slope
replaced by 1, concretised as |A|(|c| + |r|) + |beta|, |c| + |r| = max(|lo|, |hi|)) and the count N (`chain_count`).
Every device path (chain kernel, fused step, row kernel + GEMV / SIMT GEMM / DMMA GEMM, wavefront) computes the same
chain in FP64 with this structure: the relaxed row a = fl(s o A); the product a W_k as sums of n_{k+1} products in
some tree (fma or not); the 2 n_{k+1} bias terms of a level summed in some tree and added to the running beta; the
concretisation as a sum over the n_0 inputs of fl(A_i c'_i -/+ |A_i| r'_i), c' = fl(½(lo + hi)), r' = fl(½(hi - lo))
(×½ is exact), added to beta last.  Claim, with u = 2⁻⁵² (twice the unit roundoff, as in DESIGN §9):

    |dev − exact| ≤ γ_N · abs + N · 2⁻¹⁰⁷⁴,   γ_N = N u / (1 − N u).

Proof (no underflow first).  Let A' be the device's row at some level and m the number of roundings so far, and
assume |A'_c − A_c| ≤ γ_m Ā_c, Ā the abs row (true at the start: m = 0, A' = A).
- relax: the device applies relax_s(x) = x · (x > 0 ? d_u : d_l) (upper; lower with x < 0) to ITS value A'_c, with the
  SAME d_u, d_l.  relax_s is continuous and piecewise linear with slopes d_u, d_l ∈ [0, 1], so it is 1-Lipschitz even
  where A'_c and A_c differ in sign: |fl(relax(A'_c)) − relax(A_c)| ≤ u |A'_c| + |A'_c − A_c| ≤ γ_{m+1} Ā_c.  The bias
  factor max(x, 0) (min(x, 0)) is 1-Lipschitz as well, so the b_u term of c is off by ≤ γ_m Ā_c |b_u,c| before its own
  roundings.
- product: a sum of n = n_{k+1} products in any tree has ≤ n roundings on the path of each term (one product, at most
  n − 1 additions; an fma only merges two), so |fl(a' W) − a W|_i ≤ γ_n Σ|a'||W| + Σ|a' − a||W| ≤ γ_{m+1+n} Ā^{new}_i.
  Hence m grows by n_{k+1} + 1 per level.
- biases: a level's 2 n_{k+1} terms leave with ≤ m + 1 + 2 n_{k+1} roundings, then meet one `+=` per remaining level
  (k + 1 of them) and the final addition: m + 2 n_{k+1} + k + 3.  b_t itself meets t + 1 additions.
- concretisation: c' and r' each round once and |c'| + |r'| stays ≤ (1 + u) max(|lo|, |hi|); one product, the
  difference (or an fma) and n_0 − 1 additions, then beta: m + n_0 + 3 roundings for the A terms.
Every leaf of the final sum is a term of the exact value perturbed along a path of at most N roundings, N the largest
of these counts (`chain_count`); summing, |dev − exact| ≤ γ_N abs.  An operation that underflows commits an absolute
error ≤ 2⁻¹⁰⁷⁵ instead; with the factors applied after it at most 1 in magnitude this adds at most N · 2⁻¹⁰⁷⁴ (the
assumption of oracle/exact_z.py).  The extended mode is one more rounded evaluation of the same chain (u = 2⁻⁶³ covers
the long double), so its reference adds γ_N(2⁻⁶³) abs.

Post-activation targets x_{k+1} = relu(y_k), k <= K-2 ("identity o relu_k o prefix", what NNSDP_CROWN_POST_CHAINS=1
computes): the chain starts from A = d ∘ W_k (d = d_l for the lower, d_u for the upper bound), beta = d_l b_k or
b_u + d_u b_k, and runs on from level k-1; the device rounds the start once (A) and twice (beta), so m starts at 1 and
b_t's path at 2 (`chain_count(post=True)`), and abs starts from |W_k| and |b_u| + |b_k|.  Then lb = min(lb, ub),
ub = max(lb, ub) (intervals_auto_lirpa.jl:37-39), which is 1-Lipschitz in each argument: the criterion carries over.
The default device path forms the same x_{k+1} bounds as row scalings of y_k's (crown_post_kernel), reproduced bit for
bit by `post_rowscale`.
"""
from dataclasses import dataclass
from fractions import Fraction
from typing import Sequence

import numpy as np

U = 2.0 ** -52          # twice the unit roundoff of FP64 (DESIGN §9)
UEXT = 2.0 ** -63       # twice the unit roundoff of the 64-bit-mantissa long double
ETA = 2.0 ** -1074
EPS = 1e-8              # auto_LiRPA's ub_r = max(ub_r, lb_r + 1e-8)

assert np.finfo(np.longdouble).nmant >= 63, "extended mode needs an x87-style 64-bit-mantissa long double"


def gamma(n, u=U):
    n = np.asarray(n, dtype=np.float64)
    return n * u / (1.0 - n * u)


_frac = np.frompyfunc(Fraction, 1, 1)


def relax_params(l, u):
    """(d_u, b_u, d_l) of crown_params_kernel, in float64 with the kernel's operations (bit for bit)."""
    l, u = np.asarray(l, dtype=np.float64), np.asarray(u, dtype=np.float64)
    lb_r = np.minimum(l, 0.0)
    ub_r = np.maximum(u, 0.0)
    ub_r = np.maximum(ub_r, lb_r + EPS)
    d_u = ub_r / (ub_r - lb_r)
    return d_u, -lb_r * d_u, (d_u > 0.5).astype(np.float64)


def relax_params_exact(l, u):
    """The same relaxation from bounds given as Fractions, every operation exact (the 1e-8 is the double 1e-8)."""
    eps = Fraction(EPS)
    lb_r = np.array([min(v, 0) for v in l], dtype=object)
    ub_r = np.array([max(max(v, 0), lr + eps) for v, lr in zip(u, lb_r)], dtype=object)
    d_u = np.array([a / (a - b) for a, b in zip(ub_r, lb_r)], dtype=object)
    b_u = -lb_r * d_u
    d_l = np.array([Fraction(1) if v > Fraction(1, 2) else Fraction(0) for v in d_u], dtype=object)
    return d_u, b_u, d_l


def post_rowscale(l, u):
    """x_{k+1} bounds from y_k's as crown_post_kernel forms them (L = d_l l, U = d_u u + b_u, then the min/max of
    intervals_auto_lirpa.jl:37-39), float64 bit for bit."""
    d_u, b_u, d_l = relax_params(l, u)
    lo = d_l * np.asarray(l, dtype=np.float64)
    hi = d_u * np.asarray(u, dtype=np.float64) + b_u
    lo = np.minimum(lo, hi)
    return lo, np.maximum(lo, hi)


def chain_count(xdims: Sequence[int], k_first: int, post: bool = False) -> int:
    """N of a chain that starts linear in x_{k_first+1} and walks back through levels k_first .. 0 (see the module
    docstring): pre-activation target y_t has k_first = t - 1; post-activation target x_{k+1} has k_first = k - 1."""
    n = list(xdims)
    m = 1 if post else 0
    paths = [(2 if post else 0) + (k_first + 1) + 1]                 # the start bias
    for k in range(k_first, -1, -1):
        paths.append(m + 1 + 2 * n[k + 1] + (k + 1) + 1)             # the level's bias terms
        m += 1 + n[k + 1]
    paths.append(m + n[0] + 3)                                      # the concretisation terms
    return int(max(paths))


class _X:
    """Exact (Fraction objects) or extended (long double) arithmetic."""

    def __init__(self, exact: bool):
        self.exact = exact

    def x(self, a):
        a = np.asarray(a)
        if a.dtype == object:
            return a
        a = a.astype(np.float64)
        return np.asarray(_frac(a), dtype=object) if self.exact else a.astype(np.longdouble)

    def zeros(self, shape):
        if self.exact:
            z = np.empty(shape, dtype=object)
            z.fill(Fraction(0))
            return z
        return np.zeros(shape, dtype=np.longdouble)


def _backward(X: _X, net, params, A, beta, k_first, upper: bool):
    """Walk (A, beta), linear in x_{k_first+1}, back through relu_k and (W_k, b_k), k = k_first .. 0."""
    zero = X.zeros(())
    for k in range(k_first, -1, -1):
        d_u, b_u, d_l = (X.x(p) for p in params[k])
        W, b = X.x(net.Ms[k][:, :-1]), X.x(net.Ms[k][:, -1])
        take_u = (A > 0) if upper else (A < 0)
        beta = beta + np.where(take_u, A, zero) @ b_u
        a = A * np.where(take_u, d_u[None, :], d_l[None, :])
        beta = beta + a @ b
        A = a @ W
    return A, beta


def _concretise(X: _X, A, beta, x1min, x1max):
    lo, hi = X.x(x1min), X.x(x1max)
    two = 2 if X.exact else np.longdouble(2)
    c, r = (lo + hi) / two, (hi - lo) / two
    absA = np.abs(A)
    return A @ c - absA @ r + beta, A @ c + absA @ r + beta


def _abs_chain(net, k_first, Abar, bbar, x1min, x1max, params):
    """abs of every row: the chain with |W|, |b_k|, |b_u| and slopes 1, concretised on max(|lo|, |hi|)."""
    for k in range(k_first, -1, -1):
        _, b_u, _ = params[k]
        bbar = bbar + Abar @ np.abs(b_u) + Abar @ np.abs(net.Ms[k][:, -1])
        Abar = Abar @ np.abs(net.Ms[k][:, :-1])
    return Abar @ np.maximum(np.abs(x1min), np.abs(x1max)) + bbar


@dataclass
class ExactBounds:
    rows: np.ndarray
    lo: np.ndarray        # exact lower / upper bounds of the rows (Fraction objects or long doubles)
    hi: np.ndarray
    abs: np.ndarray       # float64, rounded up
    N: int
    exact: bool

    def bound(self):
        """γ_N abs + N 2⁻¹⁰⁷⁴ (+ γ_N(2⁻⁶³) abs in extended mode), rounded up a little."""
        g = gamma(self.N) + (0.0 if self.exact else gamma(self.N, UEXT))
        return (g * self.abs) * (1 + 2.0 ** -50) + self.N * ETA

    def error(self, dev, ref):
        dev = np.asarray(dev, dtype=np.float64)
        if self.exact:
            d = np.abs(np.asarray(_frac(dev), dtype=object) - ref)
            return np.array([float(v) for v in d]) * (1 + 2.0 ** -52)
        return (np.abs(dev.astype(np.longdouble) - ref) * (1 + np.longdouble(2.0 ** -62))).astype(np.float64)

    def check(self, lo_dev, hi_dev):
        """(ok, worst |err| / bound) of both halves; rows hold the bound's rows of the device's values."""
        b = self.bound()
        el, eh = self.error(lo_dev, self.lo), self.error(hi_dev, self.hi)
        ok = (el <= b) & (eh <= b)
        ratio = float(np.max(np.maximum(el, eh) / b)) if len(b) else 0.0
        return ok, ratio

    def postprocessed(self):
        """The same bounds after lb = min(lb, ub), ub = max(lb, ub) (the criterion carries over, see the docstring)."""
        lo = np.array([min(a, b) for a, b in zip(self.lo, self.hi)], dtype=self.lo.dtype)
        hi = np.array([max(a, b) for a, b in zip(self.lo, self.hi)], dtype=self.hi.dtype)
        return ExactBounds(self.rows, lo, hi, self.abs, self.N, self.exact)


def _up_abs(a, N):
    """float64 abs computed by numpy (a nonnegative expression, ≤ 2N roundings on a path) -> an upper bound."""
    return np.asarray(a, dtype=np.float64) * (1 + 2 * gamma(2 * N, 2.0 ** -53))


def crown_target(net, x1min, x1max, pre, t: int, rows=None, mode: str = "exact", params=None) -> ExactBounds:
    """Exact CROWN bounds of y_t (t >= 1), rows `rows` (default all), from the FP64 pre-activation bounds
    pre[k] = (l_k, u_k), k < t (the device's own, or any other FP64 bounds).  params overrides the relaxation (a list of
    (d_u, b_u, d_l) per layer, e.g. `relax_params_exact` of exact bounds for the soundness checks)."""
    assert t >= 1 and mode in ("exact", "extended")
    X = _X(mode == "exact")
    rows = np.arange(net.xdims[t + 1]) if rows is None else np.asarray(rows, dtype=np.int64)
    if params is None:
        params = [relax_params(*pre[k]) for k in range(t)]
    W, b = net.Ms[t][rows, :-1], net.Ms[t][rows, -1]
    lo_ref, _ = _concretise(X, *_backward(X, net, params, X.x(W), X.x(b), t - 1, False), x1min, x1max)
    _, hi_ref = _concretise(X, *_backward(X, net, params, X.x(W), X.x(b), t - 1, True), x1min, x1max)
    N = chain_count(net.xdims, t - 1)
    fparams = [tuple(np.asarray(p, dtype=np.float64) for p in pk) for pk in params]
    ab = _abs_chain(net, t - 1, np.abs(W), np.abs(b), x1min, x1max, fparams)
    return ExactBounds(rows, lo_ref, hi_ref, _up_abs(ab, N), N, X.exact)


def crown_post_target(net, x1min, x1max, pre, k: int, rows=None, mode: str = "exact", params=None) -> ExactBounds:
    """Exact bounds of x_{k+1} = relu(y_k), k <= K-2, as the output of identity o relu_k o prefix (before the min/max;
    see ExactBounds.postprocessed), from the FP64 bounds pre[j], j <= k."""
    assert 0 <= k <= net.K - 2 and mode in ("exact", "extended")
    X = _X(mode == "exact")
    rows = np.arange(net.xdims[k + 1]) if rows is None else np.asarray(rows, dtype=np.int64)
    if params is None:
        params = [relax_params(*pre[j]) for j in range(k + 1)]
    d_u, b_u, d_l = (X.x(p)[rows] for p in params[k])
    W, b = X.x(net.Ms[k][rows, :-1]), X.x(net.Ms[k][rows, -1])
    out = []
    for upper, d in ((False, d_l), (True, d_u)):
        A = d[:, None] * W
        beta = b_u + d_u * b if upper else d_l * b
        A, beta = _backward(X, net, params, A, beta, k - 1, upper)
        out.append(_concretise(X, A, beta, x1min, x1max)[1 if upper else 0])
    N = chain_count(net.xdims, k - 1, post=True)
    fparams = [tuple(np.asarray(p, dtype=np.float64) for p in pk) for pk in params]
    Wf, bf = net.Ms[k][rows, :-1], net.Ms[k][rows, -1]
    ab = _abs_chain(net, k - 1, np.abs(Wf), np.abs(fparams[k][1][rows]) + np.abs(bf), x1min, x1max, fparams)
    return ExactBounds(rows, out[0], out[1], _up_abs(ab, N), N, X.exact)


def ibp_exact(net, x1min, x1max):
    """y_0 by exact interval arithmetic (Fractions): W⁺ lo + W⁻ hi + b, W⁺ hi + W⁻ lo + b."""
    W, b = _frac(net.Ms[0][:, :-1]), _frac(net.Ms[0][:, -1])
    lo, hi = _frac(np.asarray(x1min, dtype=np.float64)), _frac(np.asarray(x1max, dtype=np.float64))
    pos = net.Ms[0][:, :-1] > 0
    Wp, Wn = np.where(pos, W, Fraction(0)), np.where(pos, Fraction(0), W)
    return Wp @ lo + Wn @ hi + b, Wp @ hi + Wn @ lo + b


def exact_crown(net, x1min, x1max):
    """CROWN in exact arithmetic with exact relaxations of exact earlier bounds: [(l_k, u_k)] for k = 0 .. K-1 and the
    relaxation parameters (Fractions).  Sound: every exact forward evaluation at a point of the box lies inside."""
    pre = [ibp_exact(net, x1min, x1max)]
    params = [relax_params_exact(*pre[0])]
    X = _X(True)
    for t in range(1, net.K):
        W, b = X.x(net.Ms[t][:, :-1]), X.x(net.Ms[t][:, -1])
        lo, _ = _concretise(X, *_backward(X, net, params, W, b, t - 1, False), x1min, x1max)
        _, hi = _concretise(X, *_backward(X, net, params, W, b, t - 1, True), x1min, x1max)
        pre.append((lo, hi))
        params.append(relax_params_exact(lo, hi))
    return pre, params


def ibp_tolerance(net, k, lo, hi):
    """The interval criterion of one layer given its FP64 inputs lo, hi: |dev − y| ≤ γ_{n+3}(|W| max(|lo|, |hi|) + |b|),
    plus the long double reference's own 2 γ_{n+2}(2⁻⁶³) (tests/test_gpu_z_exact.py::
    test_interval_bounds_meet_the_bound_layer_by_layer); returns (ylo, yhi) in long double and the tolerance."""
    M = net.Ms[k].astype(np.longdouble)
    W, bias = M[:, :-1], M[:, -1]
    lo, hi = np.asarray(lo).astype(np.longdouble), np.asarray(hi).astype(np.longdouble)
    Wp, Wn = np.maximum(W, 0), np.minimum(W, 0)
    n = net.xdims[k]
    scale = np.abs(W) @ np.maximum(np.abs(lo), np.abs(hi)) + np.abs(bias)
    tol = (gamma(n + 3) + 2 * gamma(n + 2, UEXT)) * scale.astype(np.float64) * (1 + 2.0 ** -50)
    return Wp @ lo + Wn @ hi + bias, Wp @ hi + Wn @ lo + bias, tol


def meets_ibp(net, k, lo, hi, dlo, dhi):
    ylo, yhi, tol = ibp_tolerance(net, k, lo, hi)
    el = np.abs(np.asarray(dlo).astype(np.longdouble) - ylo).astype(np.float64)
    eh = np.abs(np.asarray(dhi).astype(np.longdouble) - yhi).astype(np.float64)
    return bool(((el <= tol) & (eh <= tol)).all())
