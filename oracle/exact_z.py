"""Entrywise reference for Z(γ) with a proven rounding bound (test infrastructure only).

For one query (box, γin, γbnd, γsec, output QC, γout) and GIVEN QC bounds ymin / ymax / smin / smax, every entry of
Z is a sum of monomials in those inputs (the closed form of DESIGN §2, restated here from the Julia sources and
kernels_prep.cu; `assemble_Z_closed_form` is not used).  `exact_z` returns per entry
- ref: the value of that sum, exactly (`fractions.Fraction`, mode "exact") or in 64-bit-mantissa extended precision
  (`np.longdouble`, mode "extended");
- abs: the sum of the absolute values of the monomials, rounded up to FP64;
- N:   the number of monomials + CHAIN + 2, CHAIN = 4 being the longest chain of rounded multiplications inside one
  monomial (the degree-5 monomials smin·smax·λ·w·w of the Gram and smin·smax·λ·b·b of Z[a,a]; ×2 is exact).

Any evaluation of the entry with +, −, × and fma in FP64, in any order or tree, has at most N − 2 roundings on the
path of each monomial, so (Higham §3, with u = 2⁻⁵² as in DESIGN §9 to cover the rounding inside a DMMA step)

    |Z_fp64[r,c] − ref[r,c]| ≤ γ_N · abs[r,c] + N · 2⁻¹⁰⁷⁴,   γ_N = N u / (1 − N u),

and an entry whose abs is 0 is exactly 0.0.  The underflow term assumes that the factors applied after an operation
that underflows are at most 1 in magnitude (a subnormal λ on a layer whose weights and biases are ≤ 1).  The extended
mode adds γ_N(2⁻⁶³) · abs for its own rounding.

The three quantities come from ONE restatement evaluated in three arithmetics: exact / extended values; absolute
values of the inputs with every constant sign made positive (abs); all inputs set to 1 and the constant 2 to 1
(the monomial count, each −2·x being one monomial).  `rows` restricts the work to some rows of Z (all columns), for
stress-size queries.
"""
from dataclasses import dataclass
from fractions import Fraction
from typing import Optional

import numpy as np

from nnsdp_oracle import (QcReachCircle, QcReachEllipsoid, QcReachHplane, QcSafety, sector_pairs,
                          split_sector_gamma)

U = 2.0 ** -52          # twice the unit roundoff of FP64 (DESIGN §9)
UEXT = 2.0 ** -63       # twice the unit roundoff of the 64-bit-mantissa long double
ETA = Fraction(1, 2 ** 1074)
CHAIN = 4

assert np.finfo(np.longdouble).nmant >= 63, "extended mode needs an x87-style 64-bit-mantissa long double"


def gamma(n, u=U):
    n = np.asarray(n, dtype=np.float64)
    return n * u / (1.0 - n * u)


_frac = np.frompyfunc(Fraction, 1, 1)


class _Arith:
    """One of the three evaluations of the restatement."""

    def __init__(self, kind: str, exact: bool):
        self.kind, self.exact = kind, exact           # kind: "ref" | "abs" | "count"
        self.neg = -1 if kind == "ref" else 1         # a constant sign
        self.two = 1 if kind == "count" else 2        # the constant 2 (one monomial in the count)

    def x(self, a):
        a = np.asarray(a, dtype=np.float64)
        if self.kind == "count":
            return np.ones(a.shape)
        if self.kind == "abs":
            a = np.abs(a)
        if self.exact:
            return np.asarray(_frac(a), dtype=object) if a.ndim else Fraction(float(a))
        return a.astype(np.longdouble)

    def zeros(self, shape):
        if self.kind == "count":
            return np.zeros(shape)
        if self.exact:
            z = np.empty(shape, dtype=object)
            z.fill(Fraction(0))
            return z
        return np.zeros(shape, dtype=np.longdouble)

    def eye(self, n):
        z = self.zeros((n, n))
        z[np.arange(n), np.arange(n)] = 1
        return z


class _Rows:
    """Z restricted to the rows `rows` (all columns), written by additions of blocks and of single entries."""

    def __init__(self, ar: _Arith, rows, Zdim: int):
        self.rows = np.asarray(rows, dtype=np.int64)
        self.pos = np.full(Zdim, -1, dtype=np.int64)
        self.pos[self.rows] = np.arange(len(self.rows))
        self.out = ar.zeros((len(self.rows), Zdim))

    def add(self, grows, gcols, f):
        """Z[grows, gcols] += f(loc), f(loc) being the rows grows[loc] of the block (grows distinct, gcols distinct)."""
        p = self.pos[np.asarray(grows)]
        loc = np.nonzero(p >= 0)[0]
        if len(loc):
            self.out[np.ix_(p[loc], np.asarray(gcols))] += f(loc)

    def add_entries(self, gr, gc, vals):
        """Z[gr[i], gc[i]] += vals[i] (the pairs distinct)."""
        gr, gc = np.broadcast_arrays(np.asarray(gr), np.asarray(gc))
        vals = np.broadcast_to(np.asarray(vals, dtype=self.out.dtype), gr.shape)
        p = self.pos[gr]
        m = p >= 0
        if m.any():
            self.out[p[m], gc[m]] += vals[m]


def _out_S(ar: _Arith, qc_out, gout, n1: int, nK1: int):
    """(S11, S12, S13, S22, S23, S33) of src/Qc/output.jl:52-98 in the arithmetic ar."""
    m2 = ar.neg * ar.two
    if isinstance(qc_out, QcSafety):
        S = np.asarray(qc_out.S, dtype=np.float64)
        S = np.triu(S) + np.triu(S, 1).T           # Symmetric(S): the upper triangle is authoritative
        S = ar.x(S)
        i1, i2 = slice(0, n1), slice(n1, n1 + nK1)
        return S[i1, i1], S[i1, i2], S[i1, -1], S[i2, i2], S[i2, -1], S[-1, -1]
    g = ar.x(np.atleast_1d(np.asarray(gout, dtype=np.float64)).reshape(-1)[:1])[0]
    S11, S12, S13 = ar.zeros((n1, n1)), ar.zeros((n1, nK1)), ar.zeros(n1)
    if isinstance(qc_out, QcReachHplane):                                   # output.jl:74-75
        return S11, S12, S13, ar.zeros((nK1, nK1)), ar.x(qc_out.normal), m2 * g
    yc = ar.x(qc_out.yc)
    if isinstance(qc_out, QcReachCircle):                                   # output.jl:82-84
        return S11, S12, S13, ar.eye(nK1), ar.neg * yc, yc @ yc + ar.neg * g
    if isinstance(qc_out, QcReachEllipsoid):                                # output.jl:91-93
        P = ar.x(qc_out.invP)
        return S11, S12, S13, P.T @ P, ar.neg * (P.T @ yc), yc @ yc + ar.neg * g
    raise ValueError(qc_out)


def _restate(ar: _Arith, net, beta: int, q, bounds, rows):
    """Z[rows, :] of one query in the arithmetic ar (z = [x_1; ...; x_K; 1], a = Zdim - 1)."""
    xd, K = list(net.xdims), net.K
    n1, acdim, Zdim = xd[0], net.acdim, net.Zdim
    a = Zdim - 1
    off = np.concatenate([[0], np.cumsum(xd[:-1])]).astype(np.int64)      # first z index of block b = 0..K-1
    nst = np.concatenate([[0], np.cumsum(xd[1:-1])]).astype(np.int64)     # first neuron of layer L = 1..K-1 at nst[L-1]
    Z = _Rows(ar, rows, Zdim)
    m2 = ar.neg * ar.two                                                   # the constant -2
    W = [ar.x(M[:, :-1]) for M in net.Ms]
    bv = [ar.x(M[:, -1]) for M in net.Ms]
    ymin, ymax, smin, smax = (ar.x(v) for v in bounds)
    gin, x1min, x1max, gbnd = ar.x(q.gin), ar.x(q.x1min), ar.x(q.x1max), ar.x(q.gbnd)
    sp = split_sector_gamma(q.gsec, acdim, beta)
    lam, v, eta, nu = ar.x(sp.lam), ar.x(sp.v), ar.x(sp.eta), ar.x(sp.nu)
    bias = np.concatenate([bv[L - 1] for L in range(1, K)])
    layer_of = np.concatenate([np.full(xd[L], L) for L in range(1, K)])
    local_of = np.concatenate([np.arange(xd[L]) for L in range(1, K)])
    eps = n1 + np.arange(acdim)                                            # z index of neuron j

    # sector QC, activ_sector.jl:23-60: d11 = -2 smin smax λ, c13 = -smin η - smax ν
    d11 = m2 * (smin * smax * lam)
    c13 = ar.neg * (smin * eta) + ar.neg * (smax * nu)
    # band multipliers: Vb[t, i] = v of the pair (i, i+t) (activ_sector.jl:29), T[i,i] = Σ v of the pairs holding i
    Vb = ar.zeros((beta + 1, acdim))
    if beta > 0 and len(v):
        ij = sector_pairs(acdim, beta) - 1
        Vb[ij[:, 1] - ij[:, 0], ij[:, 0]] = v
    Tdiag = ar.zeros(acdim)
    for t in range(1, beta + 1):
        Tdiag[:acdim - t] += Vb[t, :acdim - t]
        Tdiag[t:] += Vb[t, :acdim - t]

    # Zin (input.jl:22-26) and S11
    i1 = np.arange(n1)
    Z.add_entries(i1, i1, m2 * gin)
    t1 = gin * x1min + gin * x1max
    Z.add_entries(i1, a, t1)
    Z.add_entries(a, i1, t1)
    # bounded QC (activ_bounded.jl:19-21): diagonal -2 γbnd, affine γbnd (ymin + ymax), the sector's η + ν
    Z.add_entries(eps, eps, m2 * gbnd)
    te = gbnd * ymin + gbnd * ymax + eta + nu
    Z.add_entries(eps, a, te)
    Z.add_entries(a, eps, te)
    zaa = m2 * np.sum(gin * x1min * x1max) + m2 * np.sum(gbnd * ymin * ymax)

    # per layer: Gram W_L' diag(d11) W_L on block L-1, affine rows W_L' (d11 b + c13), Z[a,a] terms
    for L in range(1, K):
        Wl, bl = W[L - 1], bv[L - 1]
        js = slice(nst[L - 1], nst[L - 1] + xd[L])
        rb = np.arange(off[L - 1], off[L - 1] + xd[L - 1])
        dj = d11[js]
        DW = dj[:, None] * Wl
        Z.add(rb, rb, lambda loc, Wl=Wl, DW=DW: Wl[:, loc].T @ DW)
        u = dj * bl + c13[js]
        tu = Wl.T @ u
        Z.add_entries(rb, a, tu)
        Z.add_entries(a, rb, tu)
        zaa = zaa + np.sum(dj * bl * bl) + ar.two * np.sum(bl * c13[js])

    # M = diag((smin + smax) λ) + T over the band: F(r, c) = Σ_j W[j, r] M[j, jc] on x rows, b_j M[j, jc] on row a,
    # and -2 T - 2 γbnd on the neuron-neuron band (the γbnd part above)
    for t in range(-beta, beta + 1):
        j = np.arange(max(0, -t), min(acdim, acdim - t))
        if len(j) == 0:
            continue
        c = j + t
        if t == 0:
            m = smin * lam + smax * lam + Tdiag
            Z.add_entries(eps, eps, m2 * Tdiag)
        else:
            m = ar.neg * (Vb[t, j] if t > 0 else Vb[-t, c])
            Z.add_entries(eps[j], eps[c], m2 * m)
        bm = bias[j] * m
        Z.add_entries(a, eps[c], bm)
        Z.add_entries(eps[c], a, bm)
        for L in range(1, K):
            sel = layer_of[j] == L
            if not sel.any():
                continue
            jj, cc, mm = j[sel], c[sel], m[sel]
            WM = W[L - 1][local_of[jj], :] * mm[:, None]                    # len(jj) x n_{L-1}
            rb = np.arange(off[L - 1], off[L - 1] + xd[L - 1])
            Z.add(rb, eps[cc], lambda loc, WM=WM: WM[:, loc].T)
            Z.add(eps[cc], rb, lambda loc, WM=WM: WM[loc, :])

    # Zout (output.jl:52-106): S11, S12 W_K, W_K' S22 W_K, the affine rows and Z[a,a]
    S11, S12, S13, S22, S23, S33 = _out_S(ar, q.qc_out, q.gout, n1, xd[-1])
    WK, bK = W[K - 1], bv[K - 1]
    rK = np.arange(off[K - 1], off[K - 1] + xd[K - 1])
    Z.add(i1, i1, lambda loc: S11[loc, :])
    Z.add(i1, rK, lambda loc: S12[loc, :] @ WK)
    Z.add(rK, i1, lambda loc: (S12 @ WK[:, loc]).T)
    t1 = S12 @ bK + S13
    Z.add_entries(i1, a, t1)
    Z.add_entries(a, i1, t1)
    S22W = S22 @ WK
    Z.add(rK, rK, lambda loc: WK[:, loc].T @ S22W)
    tK = WK.T @ (S22 @ bK + S23)
    Z.add_entries(rK, a, tK)
    Z.add_entries(a, rK, tK)
    zaa = zaa + bK @ (S22 @ bK) + bK @ S23 + bK @ S23 + S33           # b_K' (t2 + S23) + S33, t2 = S22 b_K + S23
    Z.add_entries(np.array([a]), np.array([a]), np.array([zaa], dtype=Z.out.dtype))
    return Z.out


def _up(x, exact):
    """float64 >= x (x: Fraction objects or long doubles)."""
    if exact:
        f = np.array([float(v) for v in x.ravel()])
        low = np.array([Fraction(fv) < v for fv, v in zip(f, x.ravel())], dtype=bool)
    else:
        f = x.astype(np.float64).ravel()
        low = f.astype(np.longdouble) < x.ravel()
    f[low] = np.nextafter(f[low], np.inf)
    return f.reshape(x.shape)


@dataclass
class ExactZ:
    rows: np.ndarray      # the rows of Z held (all columns)
    ref: np.ndarray       # Fraction objects (exact) or long doubles (extended)
    abs: np.ndarray       # float64, rounded up
    N: np.ndarray         # int64
    exact: bool

    def bound(self):
        """γ_N abs + N 2⁻¹⁰⁷⁴ (+ the extended term), float64 rounded up a little; 0 where abs = 0."""
        g = gamma(self.N) + (0.0 if self.exact else gamma(self.N, UEXT))
        b = (g * self.abs) * (1 + 2.0 ** -50) + self.N * 2.0 ** -1074
        return np.where(self.abs == 0, 0.0, b)

    def error(self, Zrows):
        """|Zrows − ref| (float64, rounded up) for FP64 values of the same rows."""
        Zrows = np.asarray(Zrows, dtype=np.float64)
        if self.exact:
            d = np.abs(np.asarray(_frac(Zrows), dtype=object) - self.ref)
            return _up(d, True)
        d = np.abs(Zrows.astype(np.longdouble) - self.ref)
        return _up(d * (1 + np.longdouble(2.0 ** -62)), False)

    def check(self, Zrows):
        """(ok mask, error / bound) of the entrywise criterion; ok is exact for the exact mode."""
        Zrows = np.asarray(Zrows, dtype=np.float64)
        err, bnd = self.error(Zrows), self.bound()
        ok = np.where(self.abs == 0, Zrows == 0.0, err <= bnd)
        if self.exact:                       # decide the entries close to the bound exactly
            close = ~ok | (err >= 0.5 * bnd)
            for i, k in zip(*np.nonzero(close & (self.abs != 0))):
                n = int(self.N[i, k])
                gN = Fraction(n) * Fraction(U) / (1 - Fraction(n) * Fraction(U))
                absx = self._abs_exact[i, k]
                ok[i, k] = abs(Fraction(float(Zrows[i, k])) - self.ref[i, k]) <= gN * absx + n * ETA
        with np.errstate(divide="ignore", invalid="ignore"):
            ratio = np.where(bnd > 0, err / bnd, np.where(Zrows == 0.0, 0.0, np.inf))
        return ok, ratio


def exact_z(net, beta: int, q, bounds, mode: str = "exact", rows: Optional[np.ndarray] = None) -> ExactZ:
    """The entrywise reference of Z (rows `rows`, default all) for one query q (an oracle NumericQuery) with the QC
    bounds `bounds` = (ymin, ymax, smin, smax) taken as given.  mode: "exact" (Fraction) or "extended" (long double)."""
    assert mode in ("exact", "extended")
    exact = mode == "exact"
    rows = np.arange(net.Zdim) if rows is None else np.asarray(rows, dtype=np.int64)
    bounds = tuple(np.asarray(b, dtype=np.float64) for b in bounds)
    ref = _restate(_Arith("ref", exact), net, beta, q, bounds, rows)
    ab = _restate(_Arith("abs", exact), net, beta, q, bounds, rows)
    cnt = _restate(_Arith("count", exact), net, beta, q, bounds, rows)
    N = cnt.astype(np.int64) + CHAIN + 2
    if exact:
        out = ExactZ(rows=rows, ref=ref, abs=_up(ab, True), N=N, exact=True)
        out._abs_exact = ab
        return out
    ab_up = _up(ab * (1 + np.longdouble(gamma(N.max(), UEXT)) + np.longdouble(2.0 ** -62)), False)
    return ExactZ(rows=rows, ref=ref, abs=ab_up, N=N, exact=False)
