"""Shared builders for the parity tests: seeded random nets / queries in oracle and ABI form."""
import numpy as np

import nnsdp_oracle as o


def rand_net(xdims, seed, sigma=None):
    rng = np.random.default_rng(seed)
    W = max(xdims[1:-1])
    if sigma is None:
        sigma = 2.0 / np.sqrt(W * np.log(max(W, 3)))  # scripts/make_networks.jl:44 rule
    return o.random_network(xdims, sigma, rng)


def rand_out(net, kind, rng):
    n1, nK1 = net.xdims[0], net.xdims[-1]
    if kind == "safety":
        A = rng.standard_normal((n1 + nK1 + 1, n1 + nK1 + 1))
        return o.QcSafety(S=A + A.T), None
    if kind == "hplaneS":
        return o.QcSafety(S=o.hplaneS(rng.standard_normal(nK1), 0.7, net)), None
    if kind == "hplane":
        return o.QcReachHplane(rng.standard_normal(nK1)), rng.random(1)
    if kind == "circle":
        return o.QcReachCircle(rng.standard_normal(nK1)), rng.random(1)
    if kind == "ellipsoid":
        return o.QcReachEllipsoid(rng.standard_normal((nK1, nK1)), rng.standard_normal(nK1)), rng.random(1)
    raise ValueError(kind)


def rand_query(net, beta, rng, kind="safety", radius=0.05, centre=None):
    n1, ac = net.xdims[0], net.acdim
    c = rng.uniform(0.5, 1.5, n1) if centre is None else np.asarray(centre, dtype=float)
    qc_out, gout = rand_out(net, kind, rng)
    return o.NumericQuery(
        x1min=c - radius, x1max=c + radius, gin=rng.random(n1), gbnd=rng.random(ac),
        gsec=rng.random(o.sector_lambda_dim(ac, beta) + 2 * ac), qc_out=qc_out, gout=gout)


def to_numeric_batch(nb, net, queries, with_bounds=None):
    """oracle NumericQuery list -> nnsdp_b200.NumericBatch (all queries share one output kind)."""
    q0 = queries[0].qc_out
    kw = {}
    if isinstance(q0, o.QcSafety):
        kw = dict(out_kind=nb.OUT_SAFETY, out_S=np.stack([q.qc_out.S for q in queries]))
    elif isinstance(q0, o.QcReachHplane):
        kw = dict(out_kind=nb.OUT_HPLANE, out_vec=np.stack([q.qc_out.normal for q in queries]),
                  gamma_out=np.stack([q.gout for q in queries]))
    elif isinstance(q0, o.QcReachCircle):
        kw = dict(out_kind=nb.OUT_CIRCLE, out_vec=np.stack([q.qc_out.yc for q in queries]),
                  gamma_out=np.stack([q.gout for q in queries]))
    elif isinstance(q0, o.QcReachEllipsoid):
        kw = dict(out_kind=nb.OUT_ELLIPSOID, out_vec=np.stack([q.qc_out.yc for q in queries]),
                  out_invP=np.stack([q.qc_out.invP for q in queries]),
                  gamma_out=np.stack([q.gout for q in queries]))
    if with_bounds is not None:
        kw.update(ymin=np.stack([b.acymin for b, _ in with_bounds]), ymax=np.stack([b.acymax for b, _ in with_bounds]),
                  smin=np.stack([s.smin for _, s in with_bounds]), smax=np.stack([s.smax for _, s in with_bounds]))
    return nb.NumericBatch(
        x1min=np.stack([q.x1min for q in queries]), x1max=np.stack([q.x1max for q in queries]),
        gamma_in=np.stack([q.gin for q in queries]), gamma_bnd=np.stack([q.gbnd for q in queries]),
        gamma_sec=np.stack([q.gsec for q in queries]), **kw)


def relerr(a, b):
    """normwise relative error (Frobenius / max-abs scale), the 1e-12 criterion for FP64 blocks."""
    a = np.asarray(a)
    b = np.asarray(b)
    scale = max(np.abs(b).max(), 1e-300)
    return np.abs(a - b).max() / scale


# ---- queries for the entrywise checks (oracle/exact_z.py) ---------------------------------------------------------

def wide_range_net(xdims, seed):
    """A net whose Gram blocks mix huge and tiny entries: the weight rows of layer k scaled by 2^U{-k_max..k_max}
    (k_max grows with the layer); the first layer keeps |w|, |b| ≤ 1 (the layer of the subnormal λ of
    wide_range_query, see the underflow term of exact_z).  Rows 0 and 1 of the last hidden layer are equal up to the
    sign of the second half of their inputs (the exact cancellation of wide_range_query)."""
    rng = np.random.default_rng(seed)
    Ms = []
    for k, M in enumerate(rand_net(xdims, seed=seed).Ms):
        M = M.copy()
        if k == 0:
            M /= max(1.0, np.abs(M).max())
            M[:, :-1] *= 2.0 ** -rng.integers(0, 6, M.shape[0])[:, None]
        else:
            km = min(4 + 4 * k, 24)
            M *= 2.0 ** rng.integers(-km, km + 1, M.shape[0])[:, None]
        Ms.append(M)
    K = len(xdims) - 1
    if K >= 3 and xdims[K - 1] >= 2:
        M, n_in = Ms[K - 2], xdims[K - 2]
        M[1, :-1] = M[0, :-1] * np.where(np.arange(n_in) < (n_in + 1) // 2, 1.0, -1.0)
    return o.FeedFwdNet(xdims=list(xdims), Ms=Ms)


def wide_range_query(net, beta, kind, rng):
    """A query (and its QC bounds) whose entries span many binades:
    - every γ component 2^U(-40, 40); fractional slopes 0 < smin ≤ smax < 1, some neurons stably active (1, 1) with
      λ = 0 on some of them, some with smin = 0 (d11 = 0: not Gram-active);
    - on layer 1 a λ = 2⁻¹⁰⁷⁰ (d11 subnormal, Gram-active) and a λ = 2⁻¹⁰⁷⁴ with smin·smax < 1/2 (d11 rounds to 0);
    - neurons 0 and 1 of the last hidden layer (rows equal up to sign, wide_range_net) with the same d11 are the only
      Gram-active neurons of their layer: their Gram terms cancel exactly on the mixed entries."""
    xdims, K = net.xdims, net.K
    ac, n1 = net.acdim, xdims[0]
    p2 = lambda n: 2.0 ** rng.uniform(-40, 40, n)
    ymin = -(2.0 ** rng.uniform(-6, 6, ac))
    ymax = ymin + 2.0 ** rng.uniform(-6, 6, ac)
    smin = rng.uniform(0.05, 0.95, ac)
    smax = np.minimum(smin + rng.uniform(0.0, 0.5, ac), 0.97)
    state = rng.random(ac)
    smin[state < 0.15], smax[state < 0.15] = 1.0, 1.0            # stably active
    smin[state > 0.85] = 0.0                                      # d11 = 0
    gsec = p2(o.sector_lambda_dim(ac, beta) + 2 * ac)
    lam = gsec[:ac]
    lam[(state < 0.15) & (rng.random(ac) < 0.5)] = 0.0           # λ = 0 on stably active neurons
    if xdims[1] >= 2:
        smin[0], smax[0], lam[0] = 0.5, 0.5, 2.0 ** -1070         # d11 = -2^-1071
        smin[1], smax[1], lam[1] = 0.5, 0.75, 2.0 ** -1074        # p λ = 0.375 · 2^-1074 rounds to 0
    if K >= 3 and xdims[K - 1] >= 2:
        j1 = ac - xdims[K - 1]
        smin[j1:] = 0.0
        smin[j1:j1 + 2], smax[j1:j1 + 2], lam[j1:j1 + 2] = 0.25, 0.5, p2(1)[0]
    q = rand_query(net, beta, rng, kind=kind, centre=rng.uniform(-1, 1, n1), radius=0.5)
    q.gin, q.gbnd, q.gsec = p2(n1), p2(ac), gsec
    if q.gout is not None:
        q.gout = p2(1)
    return q, (ymin, ymax, smin, smax)


def wide_range_case(xdims, beta, kind, seed):
    net = wide_range_net(xdims, seed)
    q, bounds = wide_range_query(net, beta, kind, np.random.default_rng(seed + 1000))
    return net, q, bounds


def assert_meets(R, Z, what=""):
    ok, ratio = R.check(Z)
    if not ok.all():
        i, c = np.unravel_index(np.argmax(np.where(ok, 0, ratio)), ok.shape)
        raise AssertionError(f"{what}: {int((~ok).sum())} entries break the bound; worst Z[{R.rows[i]},{c}] = "
                             f"{Z[i, c]!r}, |err| / bound = {ratio[i, c]:.3g}, abs = {R.abs[i, c]:.3g}, N = {R.N[i, c]}")
