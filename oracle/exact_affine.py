"""Entrywise reference for the affine-coefficient hand-off Z(γ) = Z₀ + Σ_v γ_v Z_v, with a proven rounding bound (test
infrastructure only).

For one query (box, output QC) and GIVEN QC bounds ymin / ymax / smin / smax, every coefficient Z_v[r, c] on the
upper triangle of the clique cover is a sum of monomials in those inputs.  The per-variable patterns are restated here
from the Julia sources (the Z_v of an AffExpr Z, src/Methods/chordal_sdp.jl:96-153), with ρ_j = row j of [W b]
placed in the block that feeds neuron j (bias at the affine index a), ε_j the neuron's own index and
sym(u, e) = u e' + e u':

    γin_i    −2 e_i e_i' + (xmin_i + xmax_i) sym(e_i, e_a) − 2 xmin_i xmax_i e_a e_a'          input.jl:22-26
    γout     −2 e_a e_a' (hyperplane), −e_a e_a' (circle, ellipsoid)                         output.jl:74-93
    γbnd_j   −2 ε ε' + (ymin_j + ymax_j) sym(ε, e_a) − 2 ymin_j ymax_j e_a e_a'                activ_bounded.jl:19-21
    λ_j      −2 smin_j smax_j ρ ρ' + (smin_j + smax_j) sym(ρ, ε)                               activ_sector.jl:23-60
    v_ij     sym(ρ_i − ρ_j, ε_i − ε_j) − 2 (ε_i − ε_j)(ε_i − ε_j)'                              activ_sector.jl:29-35
    η_j, ν_j −s_j sym(ρ, e_a) + sym(ε, e_a),  s = smin | smax                                  activ_sector.jl:51-56

The upper entry (r, c), r ≤ c, holds Z_v[r, c]: a term of sym(u, e_p) at support index k lands on (min(k, p),
max(k, p)), and on the diagonal k = p the two halves add (2·u[p]).  Variables are in the reference's creation order [γin; γout (reach kinds); γbnd;
λ; v pairs; η; ν] (split_sector_gamma, nnsdp_affine_sizes); entries are those of oracle.cover_upper_entries.
Z₀ needs no restatement: it is exact_z with every multiplier 0, γout included.

`exact_affine` lists every (variable, entry) pair the patterns touch, with
- ref: the exact value of the coefficient (`Fraction`, mode "exact") or its 64-bit-mantissa value (mode "extended");
- abs: the sum of the absolute values of its monomials, rounded up to FP64;
- N:   the number of its monomials + CHAIN + 2, CHAIN = 3.

Proof of the criterion.  Let a device evaluate one coefficient with +, −, × and fma in FP64, in any order, as the sum
of its monomials (Higham §3; u = 2⁻⁵², the convention of DESIGN §9).  A monomial has at most CHAIN = 3 rounded
products: −2·smin·smax·w_r·w_c forms smin·smax, w_r·w_c and their product (×2, ×(−1) and the doubling of a
diagonal term are exact away from overflow).  The sum of m monomials adds at most m − 1 roundings on any monomial's
path, and the device's sum of a duplicate pair in the CSC form (the v_ij entries where two sym terms meet) one more.
So each monomial carries at most m + CHAIN + 1 < N relative roundings, and without underflow

    |dev − ref| ≤ γ_N · abs,   γ_N = N u / (1 − N u).

An operation that underflows adds an absolute error ≤ 2⁻¹⁰⁷⁵ instead; if every factor applied after it is at most 1
in magnitude (the precondition of DESIGN §2: a subnormal smin·smax only on a layer whose weights and biases are ≤ 1),
that error stays ≤ 2⁻¹⁰⁷⁵ in the result, and at most N such errors occur on one coefficient, hence the term
N·2⁻¹⁰⁷⁴.  A product smin·smax that rounds to 0 makes the device skip the Gram terms of λ_j: that is the same
underflow error on each of them, with every later factor ≤ 1.  A coefficient whose abs is 0 has only zero monomials:
every operation on zeros gives 0.0, so it must be exactly 0.0, or absent.  The extended mode adds γ_N(2⁻⁶³)·abs for
its own rounding (exact_z); a device value summed from duplicates in long double adds its summation error as slack.

`vars` restricts the work to some variables (all their entries), for stress-size nets.
"""
from dataclasses import dataclass
from fractions import Fraction
from typing import Optional

import numpy as np

from exact_z import ExactZ, _Arith, _frac, _up, exact_z, gamma, UEXT
from nnsdp_oracle import (QcReachHplane, QcSafety, cover_upper_entries, make_cliques, sector_lambda_dim,
                          sector_pairs)

CHAIN = 3


@dataclass
class Layout:
    """Variable and entry layout of one (net, β, output kind)."""
    nvar: int
    var_out: int          # first variable after γin (= n_in)
    var_bnd: int
    var_sec: int
    lamdim: int
    ent_row: np.ndarray   # 0-based (row, column) of the cover's upper entries, column-major
    ent_col: np.ndarray
    ent_of: np.ndarray    # Zdim x Zdim: entry index of (r, c), r ≤ c; -1 off the cover

    @property
    def nent(self):
        return len(self.ent_row)


def layout(net, beta: int, qc_out) -> Layout:
    n1, ac = net.xdims[0], net.acdim
    er, ec = cover_upper_entries(net, make_cliques(net, beta))
    er, ec = er - 1, ec - 1
    ent_of = np.full((net.Zdim, net.Zdim), -1, dtype=np.int64)
    ent_of[er, ec] = np.arange(len(er))
    var_bnd = n1 + (0 if isinstance(qc_out, QcSafety) else 1)
    lamdim = sector_lambda_dim(ac, beta)
    return Layout(nvar=var_bnd + ac + lamdim + 2 * ac, var_out=n1, var_bnd=var_bnd, var_sec=var_bnd + ac,
                  lamdim=lamdim, ent_row=er, ent_col=ec, ent_of=ent_of)


class _Terms:
    """(variable, row, column, value) terms of the restatement, upper triangle, in one arithmetic."""

    def __init__(self, ar: _Arith):
        self.ar, self.v, self.r, self.c, self.x = ar, [], [], [], []
        self.dtype = ar.zeros(0).dtype

    def add(self, v, r, c, x):
        v, r, c = np.broadcast_arrays(np.asarray(v), np.asarray(r), np.asarray(c))
        x = np.broadcast_to(np.asarray(x, dtype=self.dtype), v.shape)
        assert (r <= c).all()
        for lst, y in ((self.v, v), (self.r, r), (self.c, c), (self.x, x)):
            lst.append(np.array(y, dtype=y.dtype).ravel())

    def sym(self, v, k, p, x):
        """sym(u, e_p) with u[k] = x: the term x on (min(k, p), max(k, p)), doubled where k = p."""
        v, k, p = np.broadcast_arrays(np.asarray(v), np.asarray(k), np.asarray(p))
        x = np.array(np.broadcast_to(np.asarray(x, dtype=self.dtype), v.shape))
        d = k == p
        if d.any():
            x[d] = x[d] * self.ar.two
        self.add(v, np.minimum(k, p), np.maximum(k, p), x)


def _restate(ar: _Arith, net, beta: int, q, bounds, lay: Layout, want):
    """All terms of the variables marked in `want` (bool, nvar) in the arithmetic ar."""
    xd, K = list(net.xdims), net.K
    n1, ac, a = xd[0], net.acdim, net.Zdim - 1
    off = np.concatenate([[0], np.cumsum(xd[:-1])]).astype(np.int64)      # first z index of block b
    nst = np.concatenate([[0], np.cumsum(xd[1:-1])]).astype(np.int64)     # first neuron of layer L at nst[L-1]
    layer_of = np.concatenate([np.full(xd[L], L) for L in range(1, K)])
    local_of = np.concatenate([np.arange(xd[L]) for L in range(1, K)])
    m2, neg, two = ar.neg * ar.two, ar.neg, ar.two
    T = _Terms(ar)
    x1min, x1max = ar.x(q.x1min), ar.x(q.x1max)
    ymin, ymax, smin, smax = (ar.x(b) for b in bounds)
    sminf, smaxf = (np.asarray(b, dtype=np.float64) for b in bounds[2:])
    W = [ar.x(M[:, :-1]) for M in net.Ms[:-1]]
    bv = [ar.x(M[:, -1]) for M in net.Ms[:-1]]
    eps = n1 + np.arange(ac)
    vl, vp0 = lay.var_sec, lay.var_sec + ac                                # λ_j, first pair
    ve, vn = lay.var_sec + lay.lamdim, lay.var_sec + lay.lamdim + ac       # η_j, ν_j

    # γin (input.jl:22-26)
    i = np.arange(n1)
    sel = want[i]
    if sel.any():
        i = i[sel]
        T.add(i, i, i, m2)
        T.add(i, i, a, x1min[i])
        T.add(i, i, a, x1max[i])
        T.add(i, a, a, m2 * x1min[i] * x1max[i])
    # γout (output.jl:74-93)
    if lay.var_bnd > lay.var_out and want[lay.var_out]:
        T.add(lay.var_out, a, a, m2 if isinstance(q.qc_out, QcReachHplane) else neg)
    # γbnd (activ_bounded.jl:19-21)
    j = np.arange(ac)
    sel = want[lay.var_bnd + j]
    if sel.any():
        jj, v = j[sel], lay.var_bnd + j[sel]
        T.add(v, eps[jj], eps[jj], m2)
        T.add(v, eps[jj], a, ymin[jj])
        T.add(v, eps[jj], a, ymax[jj])
        T.add(v, a, a, m2 * ymin[jj] * ymax[jj])

    # per layer L: the neurons J of L, their ρ (rows rb of block L-1, bias at a)
    for L in range(1, K):
        J = nst[L - 1] + np.arange(xd[L])
        Wl, bl = W[L - 1], bv[L - 1]
        rb = off[L - 1] + np.arange(xd[L - 1])

        # λ_j: -2 smin smax ρ ρ' (exactly zero when smin or smax is) and (smin + smax) sym(ρ, ε)
        s = want[vl + J] & (sminf[J] != 0) & (smaxf[J] != 0)
        if s.any():
            js = J[s]
            jl = local_of[js]
            p = m2 * (smin[js] * smax[js])
            iu, ic = np.triu_indices(xd[L - 1])
            T.add((vl + js)[:, None], rb[iu][None, :], rb[ic][None, :], p[:, None] * (Wl[jl][:, iu] * Wl[jl][:, ic]))
            T.add((vl + js)[:, None], rb[None, :], a, p[:, None] * (Wl[jl] * bl[jl][:, None]))
            T.add(vl + js, a, a, p * (bl[jl] * bl[jl]))
        s = want[vl + J] & (sminf[J] != -smaxf[J])
        if s.any():
            js = J[s]
            jl = local_of[js]
            for sv in (smin, smax):
                T.sym((vl + js)[:, None], rb[None, :], eps[js][:, None], sv[js][:, None] * Wl[jl])
                T.sym(vl + js, a, eps[js], sv[js] * bl[jl])

        # η_j, ν_j: -s sym(ρ, e_a) + sym(ε, e_a)
        for vbase, sv in ((ve, smin), (vn, smax)):
            s = want[vbase + J]
            if s.any():
                js = J[s]
                jl = local_of[js]
                v = vbase + js
                T.sym(v[:, None], rb[None, :], a, neg * (sv[js][:, None] * Wl[jl]))
                T.sym(v, a, a, neg * (sv[js] * bl[jl]))
                T.sym(v, eps[js], a, ar.x(np.ones(len(js))))

    # v_ij (activ_sector.jl:29-35): sym(ρ_i, ε_i) − sym(ρ_i, ε_j) − sym(ρ_j, ε_i) + sym(ρ_j, ε_j) − 2 (ε_i − ε_j)(ε_i − ε_j)'
    if beta > 0 and ac > 1:
        pr = sector_pairs(ac, beta) - 1
        vk = vp0 + np.arange(len(pr))
        s = want[vk]
        pr, vk = pr[s], vk[s]
        for x, y, sign in ((0, 0, 1), (0, 1, -1), (1, 0, -1), (1, 1, 1)):
            nx, ny = pr[:, x], pr[:, y]
            for L in range(1, K):
                m = layer_of[nx] == L
                if not m.any():
                    continue
                jl = local_of[nx[m]]
                rb = off[L - 1] + np.arange(xd[L - 1])
                sg = 1 if sign > 0 else neg
                T.sym(vk[m][:, None], rb[None, :], eps[ny[m]][:, None], sg * W[L - 1][jl])
                T.sym(vk[m], a, eps[ny[m]], sg * bv[L - 1][jl])
        ei, ej = eps[pr[:, 0]], eps[pr[:, 1]]
        T.add(vk, ei, ei, m2)
        T.add(vk, ei, ej, two)
        T.add(vk, ej, ej, m2)
    return T


def _combine(T: _Terms, lay: Layout):
    """Terms -> (sorted unique keys var * nent + entry, summed values)."""
    v, r, c, x = (np.concatenate(lst) if lst else np.zeros(0, dtype=T.dtype if k == 3 else np.int64)
                  for k, lst in enumerate((T.v, T.r, T.c, T.x)))
    e = lay.ent_of[r, c]
    assert (e >= 0).all(), "a coefficient off the clique cover"
    key = v.astype(np.int64) * lay.nent + e
    o = np.argsort(key, kind="stable")
    key, x = key[o], x[o]
    start = np.flatnonzero(np.r_[True, key[1:] != key[:-1]]) if len(key) else np.zeros(0, dtype=np.int64)
    return key[start], (np.add.reduceat(x, start) if len(key) else x)


@dataclass
class ExactAffine:
    lay: Layout
    key: np.ndarray       # var * nent + entry, ascending
    ref: np.ndarray       # Fraction objects (exact) or long doubles (extended)
    abs: np.ndarray       # float64, rounded up
    N: np.ndarray         # int64
    exact: bool
    abs_exact: Optional[np.ndarray] = None

    @property
    def var(self):
        return self.key // self.lay.nent

    @property
    def ent(self):
        return self.key % self.lay.nent

    def counts(self):
        """number of listed entries of every variable"""
        return np.bincount(self.var, minlength=self.lay.nvar)

    def dense(self):
        """Z_v as an nent x nvar array of the reference values (small nets)"""
        D = np.empty((self.lay.nent, self.lay.nvar), dtype=self.ref.dtype)
        D.fill(Fraction(0) if self.exact else 0)
        D[self.ent, self.var] = self.ref
        return D

    def check(self, dev, vars=None):
        """The criterion over the union of the listed pairs and the device's (var, ent, val) triplets, the device's
        duplicates summed exactly (exact mode) or in long double with their summation error as slack.  `vars`: check
        only these variables (the reference was built for them).  Returns (ok, ratio) over the union; `where(i, dev)`
        names union element i."""
        var, ent, val = (np.asarray(a) for a in dev)
        key = var.astype(np.int64) * self.lay.nent + ent.astype(np.int64)
        if vars is not None:
            m = np.isin(var, vars)
            key, val = key[m], val[m]
        o = np.argsort(key, kind="stable")
        key, val = key[o], np.asarray(val, dtype=np.float64)[o]
        start = np.flatnonzero(np.r_[True, key[1:] != key[:-1]]) if len(key) else np.zeros(0, dtype=np.int64)
        dkey = key[start]
        nterm = np.diff(np.r_[start, len(key)])
        slack = None
        if self.exact:
            dval = np.add.reduceat(np.asarray(_frac(val), dtype=object), start) if len(key) else np.zeros(0, object)
        else:
            dval = np.add.reduceat(val.astype(np.longdouble), start) if len(key) else np.zeros(0, np.longdouble)
            sabs = np.add.reduceat(np.abs(val), start) if len(key) else np.zeros(0)
            slack = np.where(nterm > 1, gamma(nterm, UEXT) * sabs * (1 + 2.0 ** -50), 0.0)
        u = np.union1d(self.key, dkey)
        self._union = u
        mine, theirs = np.searchsorted(self.key, u), np.searchsorted(dkey, u)
        have = (mine < len(self.key)) & (self.key[np.minimum(mine, len(self.key) - 1)] == u) if len(self.key) else \
            np.zeros(len(u), bool)
        got = (theirs < len(dkey)) & (dkey[np.minimum(theirs, len(dkey) - 1)] == u) if len(dkey) else \
            np.zeros(len(u), bool)
        zero = Fraction(0) if self.exact else np.longdouble(0)
        R = ExactZ(rows=u, ref=np.full(len(u), zero, dtype=self.ref.dtype), abs=np.zeros(len(u)),
                   N=np.full(len(u), CHAIN + 2, dtype=np.int64), exact=self.exact)
        R.ref[have], R.abs[have], R.N[have] = self.ref[mine[have]], self.abs[mine[have]], self.N[mine[have]]
        if self.exact:
            R._abs_exact = np.full(len(u), Fraction(0), dtype=object)
            R._abs_exact[have] = self.abs_exact[mine[have]]
        D = np.full(len(u), zero, dtype=dval.dtype)
        D[got] = dval[theirs[got]]
        sl = None
        if slack is not None:
            sl = np.zeros(len(u))
            sl[got] = slack[theirs[got]]
        self._udev, self._uR = D, R
        return R.check(D, sl)

    def where(self, i):
        """(variable, row, column) and the numbers of union element i of the last check"""
        k = int(self._union[i])
        v, e = divmod(k, self.lay.nent)
        R = self._uR
        return (f"variable {v}, Z[{self.lay.ent_row[e]},{self.lay.ent_col[e]}]: dev {float(self._udev[i])!r}, "
                f"ref {float(R.ref[i])!r}, abs = {R.abs[i]:.3g}, N = {R.N[i]}")


def exact_affine(net, beta: int, q, bounds, mode: str = "exact", vars=None, lay: Optional[Layout] = None) -> ExactAffine:
    """The entrywise reference of every coefficient Z_v[r, c] of one query q (an oracle NumericQuery: its box and
    output QC are used, its multipliers are not) with the QC bounds `bounds` = (ymin, ymax, smin, smax) taken as given.
    mode: "exact" (Fraction) or "extended" (long double); vars: only these variables (default all); lay: the
    layout(net, beta, q.qc_out) of an earlier call, to save its work."""
    assert mode in ("exact", "extended")
    exact = mode == "exact"
    lay = layout(net, beta, q.qc_out) if lay is None else lay
    want = np.zeros(lay.nvar, dtype=bool)
    want[np.arange(lay.nvar) if vars is None else np.asarray(vars, dtype=np.int64)] = True
    bounds = tuple(np.asarray(b, dtype=np.float64) for b in bounds)
    key, ref = _combine(_restate(_Arith("ref", exact), net, beta, q, bounds, lay, want), lay)
    k2, ab = _combine(_restate(_Arith("abs", exact), net, beta, q, bounds, lay, want), lay)
    k3, cnt = _combine(_restate(_Arith("count", exact), net, beta, q, bounds, lay, want), lay)
    assert np.array_equal(key, k2) and np.array_equal(key, k3)
    N = cnt.astype(np.int64) + CHAIN + 2
    if exact:
        return ExactAffine(lay=lay, key=key, ref=ref, abs=_up(ab, True), N=N, exact=True, abs_exact=ab)
    ab_up = _up(ab * (1 + np.longdouble(gamma(N.max() if len(N) else 0, UEXT)) + np.longdouble(2.0 ** -62)), False)
    return ExactAffine(lay=lay, key=key, ref=ref, abs=ab_up, N=N, exact=False)


def exact_z0(net, beta: int, q, bounds, mode: str = "exact", rows=None):
    """Z₀: exact_z of q with every multiplier 0, γout included."""
    z = type(q)(**{**q.__dict__})
    z.gin, z.gbnd, z.gsec = np.zeros_like(q.gin), np.zeros_like(q.gbnd), np.zeros_like(q.gsec)
    if q.gout is not None:
        z.gout = np.zeros_like(np.atleast_1d(q.gout))
    return exact_z(net, beta, z, bounds, mode=mode, rows=rows)
