"""CPU restatement of nnsdp_batch_certify (test infrastructure only): the sound certificate lambda_max(Z) <= tau by a
multifrontal Cholesky of tau' I - Z along the path of cliques, with the same elimination order, panel width, margin and
outputs as the device (DESIGN.md section 9).

    certify_multifrontal(Z, cliques, tau)     Z dense (Zdim x Zdim), cliques = 0-based index arrays in clique-local order
    certify_fronts(blocks, cliques, tau)      the same from the clique blocks Z[C_k, C_k] alone (large nets)

both return (certified, bound, fail_index, min_pivot) like Batch.certify for one query.
"""
import math

import numpy as np

NB = 32     # panel width of the device factorisation
U = 2.0 ** -52
ETA = 2.0 ** -1074


def _up(x):
    return math.nextafter(x, math.inf)


def _dn(x):
    return math.nextafter(x, -math.inf)


def certify_margin(tp, zdim, trz, sabs, mabs):
    """c(tau'): the rounding-error margin of a successful factorisation of fl(tau' I - Z), every operation rounded up."""
    n = float(zdim)
    nu = _up((n + 1) * U)
    gam = _up(nu / _dn(1.0 - nu))
    coef = _up(_up(gam / _dn(1.0 - gam)) + U)
    err = _up(_up(2.0 * (n + 2) * U) * _up(_up(abs(tp) * n) + sabs))
    tr = max(0.0, _up(_up(_up(tp * n) - trz) + err))
    uf = _up(_up(2.0 * n * (n + 2)) * _up(_up(2.0 + _up(abs(tp) + mabs)) * 2.0) * ETA)
    return _up(_up(coef * tr) + uf)


def certify_shift(tau, zdim, trz, sabs, mabs):
    """(tau', bound): the largest tau' found whose bound tau' + c(tau') rounds up to at most tau."""
    tp = float(tau)
    for _ in range(200):
        bnd = _up(tp + certify_margin(tp, zdim, trz, sabs, mabs))
        if bnd <= tau:
            return tp, bnd
        tp = _dn(tp - max(bnd - tau, abs(tp) * 2.0 ** -50))
    return -math.inf, math.inf


def certify_lower(tp, zdim, mabs):
    """Proven lower bound of lambda_max(Z) after the factorisation of fl(tau' I - Z) failed (Demmel's success condition,
    Higham Thm 10.7; nnsdp_batch_certify_ex).  -inf where the factorisation may have overflowed."""
    n = float(zdim)
    nu = _up((n + 1) * U)
    gam = _up(nu / _dn(1.0 - nu))
    ng = _up(n * gam)
    if not ng < 0.5:
        return -math.inf
    rho = _up(ng / _dn(1.0 - ng))
    amax = _up(_up(abs(tp) + mabs) * _up(1.0 + 2.0 * U))
    if not (math.isfinite(amax) and math.isfinite(_up(_up(4.0 * n) * amax)) and math.isfinite(tp)):
        return -math.inf
    uf = _up(_up(2.0 * n * (n + 2)) * _up(_up(2.0 + amax) * 2.0) * ETA)
    return _dn(tp - _up(_up(_up(rho * amax) + _up(U * amax)) + uf))


def front_plan(cliques, zdim):
    """Per front: (npriv, lead, tail) with the layout checks of the device plan."""
    p = len(cliques)
    owner = -np.ones(zdim, dtype=np.int64)
    for k, c in enumerate(cliques):
        owner[np.asarray(c)] = k
    assert (owner >= 0).all(), "an index lies in no clique"
    plan, shifted = [], np.zeros(zdim, dtype=np.int64)
    for k, c in enumerate(cliques):
        c = np.asarray(c)
        priv = owner[c] == k
        npriv = int(priv.sum())
        assert npriv >= 1 and priv[:npriv].all(), f"private indices of clique {k} are not a leading range"
        assert (c[:npriv] == c[0] + np.arange(npriv)).all(), f"private indices of clique {k} are not contiguous"
        lead = tail = 0
        if k > 0:
            pc, pn = np.asarray(cliques[k - 1]), plan[-1][0]
            sep = pc[pn:]
            pos = {g: i for i, g in enumerate(c)}
            loc = np.array([pos[g] for g in sep])
            lead = int(np.sum(loc == np.arange(len(sep))))
            tail = len(sep) - lead
            assert (loc[:lead] == np.arange(lead)).all() and (loc[lead:] == len(c) - tail + np.arange(tail)).all(), \
                f"the separator of cliques {k - 1}, {k} is not leading + tail in clique {k}"
        shifted[c[lead:len(c) - tail]] += 1
        plan.append((npriv, lead, tail))
    assert plan[-1][0] == len(cliques[-1]), "the last clique is not all private"
    assert (shifted == 1).all(), "a diagonal entry is not shifted exactly once"
    return plan


def certify_fronts(blocks, cliques, tau):
    cliques = [np.asarray(c, dtype=np.int64) for c in cliques]
    zdim = int(max(int(c.max()) for c in cliques)) + 1
    plan = front_plan(cliques, zdim)
    diag = np.concatenate([np.diag(B)[lead:len(c) - tail] for B, c, (_, lead, tail) in zip(blocks, cliques, plan)])
    tp, bound = certify_shift(float(tau), zdim, float(np.sum(diag)), float(np.sum(np.abs(diag))),
                              float(np.max(np.abs(diag))))
    min_piv, S = math.inf, None
    for k, (B, c, (npriv, lead, tail)) in enumerate(zip(blocks, cliques, plan)):
        n = len(c)
        F = -np.array(B, dtype=np.float64)
        F[np.diag_indices(n)] = tp - np.diag(B)
        if k > 0:
            loc = np.concatenate([np.arange(lead), n - tail + np.arange(tail)])
            F[np.ix_(loc, loc)] = S
        for j0 in range(0, npriv, NB):
            w = min(NB, npriv - j0)
            D = np.tril(F[j0:j0 + w, j0:j0 + w]).copy()
            for jj in range(w):
                d = D[jj, jj]
                if not d > 0.0:
                    return 0, bound, int(c[0] + j0 + jj), float(d)
                min_piv = min(min_piv, d)
                r = math.sqrt(d)
                D[jj, jj] = r
                D[jj + 1:, jj] /= r
                D[jj + 1:, jj + 1:] -= np.tril(np.outer(D[jj + 1:, jj], D[jj + 1:, jj]))
            X = F[j0 + w:, j0:j0 + w].copy()
            for l in range(w):
                X[:, l] = (X[:, l] - X[:, :l] @ D[l, :l]) / D[l, l]
            F[j0 + w:, j0:j0 + w] = X
            F[j0 + w:, j0 + w:] -= X @ X.T
        S = F[npriv:, npriv:].copy()
    return 1, bound, -1, float(min_piv)


def certify_multifrontal(Z, cliques, tau):
    Z = np.asarray(Z, dtype=np.float64)
    return certify_fronts([Z[np.ix_(np.asarray(c), np.asarray(c))] for c in cliques], cliques, tau)
