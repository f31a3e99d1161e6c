"""The exact CROWN reference of oracle/exact_crown.py checked on its own (no GPU):

- the exact (Fraction) and extended (long double) modes agree, and one target is worked by hand;
- the oracle's FP64 `intervals_crown` (another summation order than the device) meets the layer-by-layer criterion
  |dev − exact| ≤ γ_N abs + N 2⁻¹⁰⁷⁴, so the bound is not too tight;
- the restatement is sound: with exact relaxations of exact earlier bounds, exact forward evaluations at sampled points
  and at the box's vertices lie inside its exact bounds;
- four small bugs planted in an FP64 CROWN pass the old normwise criterion (max |x bound − oracle| ≤ 1e-11 · the largest
  |bound| of the net, tests/test_gpu_parity.py) and fail the new one."""
import itertools
from fractions import Fraction

import numpy as np
import pytest

import exact_crown as ec
import nnsdp_oracle as o
from helpers import rand_net, wide_range_net


def oracle_pre(net, lo, hi):
    """The pre-activation bounds y_0 .. y_{K-1} the oracle's intervals_crown builds its relaxations from."""
    pre = {1: o._ibp_layer(net.Ms[0], lo, hi)}
    for i in range(2, net.K + 1):
        W, b = net.Ms[i - 1][:, :-1], net.Ms[i - 1][:, -1]
        pre[i] = o._crown_backward(net, pre, W.copy(), W.copy(), b.copy(), b.copy(), i - 1, lo, hi)
    return [pre[k + 1] for k in range(net.K)]


def meets_new(net, lo, hi, pre, mode="exact"):
    """Every target t >= 1 of `pre` against the exact chain built from pre's own earlier bounds; worst ratio."""
    worst = 0.0
    for t in range(1, net.K):
        ok, r = ec.crown_target(net, lo, hi, pre, t, mode=mode).check(*pre[t])
        if not ok.all():
            return False, r
        worst = max(worst, r)
    return True, worst


def meets_old(net, lo, hi, x_lo, x_hi):
    ref = o.intervals_crown(lo, hi, net)
    xmin = np.concatenate([p[0] for p in ref.x_intvs])
    xmax = np.concatenate([p[1] for p in ref.x_intvs])
    scale = max(np.abs(xmin).max(), np.abs(xmax).max(), 1.0)
    return max(np.abs(x_lo - xmin).max(), np.abs(x_hi - xmax).max()) <= 1e-11 * scale


CPU_SHAPES = [[2, 3, 2], [2, 6, 5, 7, 2], [2, 4, 7, 3, 5, 2], [2] + [10] * 10 + [2], [5, 20, 20, 20, 5]]


def _box(n, seed, radius):
    c = np.random.default_rng(seed).uniform(-1, 1, n)
    return c - radius, c + radius


def _ext_error(ld, ex):
    """|long double − Fraction|, exactly, as floats."""
    return np.array([float(abs(Fraction(*v.as_integer_ratio()) - e)) for v, e in zip(ld, ex)])


def test_exact_and_extended_modes_agree():
    """The long double chain is within its own γ_N(2⁻⁶³) abs of the exact one, on every pre- and post-activation
    target of two wide-range nets; both modes give the same abs and N."""
    for xd in ([2, 6, 5, 7, 2], [3, 9, 8, 10, 2]):
        net = wide_range_net(xd, seed=7)
        lo, hi = _box(xd[0], 1, 0.3)
        pre = oracle_pre(net, lo, hi)
        pairs = [(ec.crown_target(net, lo, hi, pre, t, mode=m) for m in ("exact", "extended")) for t in range(1, net.K)]
        pairs += [(ec.crown_post_target(net, lo, hi, pre, k, mode=m) for m in ("exact", "extended"))
                  for k in range(net.K - 1)]
        for A, B in pairs:
            assert A.N == B.N and np.array_equal(A.abs, B.abs)
            tol = ec.gamma(A.N, ec.UEXT) * A.abs
            assert (_ext_error(B.lo, A.lo) <= tol).all() and (_ext_error(B.hi, A.hi) <= tol).all()


def test_one_target_by_hand():
    """x ∈ [-1, 1]; y_0 = (x, x - 1/2): l = (-1, -3/2), u = (1, 1/2), so d_u = (1/2, 1/4), b_u = (1/2, 3/8) and
    d_l = (0, 0) (neuron 0 is the l = -u tie: 1/2 is not > 1/2).  y_1 = x_1 - 2 x_2 + 1/4:
    upper: A = (1, -2) -> slopes (d_u, d_l) = (1/2, 0), beta = 1/4 + 1/2; A W_0 = 1/2: 1/2 · 0 + 1/2 · 1 + 3/4 = 5/4;
    lower: slopes (d_l, d_u) = (0, 1/4), beta = 1/4 - 2 · 3/8 + (-1/2)(-1/2) = -1/4; A W_0 = -1/2: -1/2 - 1/4 = -3/4.
    abs: |A| = (1, 2), beta 1/4 + (1 · 1/2 + 2 · 3/8) + (0 + 2 · 1/2) = 5/2, |A| |W_0| = 3: 3 · 1 + 5/2 = 11/2.
    N: the level's bias terms 0 + 1 + 2·2 + 1 + 1 = 7, the concretisation (1 + 2) + 1 + 3 = 7, b_1 1 + 1 = 2."""
    net = o.FeedFwdNet(xdims=[1, 2, 1], Ms=[np.array([[1.0, 0.0], [1.0, -0.5]]), np.array([[1.0, -2.0, 0.25]])])
    lo, hi = np.array([-1.0]), np.array([1.0])
    pre = oracle_pre(net, lo, hi)
    assert np.array_equal(pre[0][0], [-1.0, -1.5]) and np.array_equal(pre[0][1], [1.0, 0.5])
    d_u, b_u, d_l = ec.relax_params(*pre[0])
    assert np.array_equal(d_u, [0.5, 0.25]) and np.array_equal(b_u, [0.5, 0.375]) and np.array_equal(d_l, [0.0, 0.0])
    R = ec.crown_target(net, lo, hi, pre, 1, mode="exact")
    assert R.lo[0] == Fraction(-3, 4) and R.hi[0] == Fraction(5, 4)
    assert R.N == 7 and ec.chain_count([1, 2, 1], 0) == 7
    assert 5.5 <= R.abs[0] <= 5.5 * (1 + 1e-14)
    # the reference's numbers are sound for this target: y_1(x) over a fine grid
    xs = np.linspace(-1, 1, 401)
    y = np.maximum(xs, 0) - 2 * np.maximum(xs - 0.5, 0) + 0.25
    assert y.min() >= -0.75 and y.max() <= 1.25


@pytest.mark.parametrize("xdims", CPU_SHAPES + [[2, 4, 7, 3, 5, 2], [3, 9, 12, 7, 10, 2]])
@pytest.mark.parametrize("wide", [False, True])
def test_oracle_fp64_crown_meets_the_bound(xdims, wide):
    """The oracle's intervals_crown (numpy's summation order, not the device's) meets the criterion on every target,
    pre-activation and post-activation (identity-slice chains, after the min/max), at radii 0 .. 0.5."""
    net = (wide_range_net if wide else rand_net)(xdims, 8)
    for radius in (0.0, 2.0 ** -20, 0.05, 0.5):
        lo, hi = _box(xdims[0], len(xdims), radius)
        pre = oracle_pre(net, lo, hi)
        mode = "exact" if sum(xdims) <= 60 else "extended"
        ok, worst = meets_new(net, lo, hi, pre, mode)
        assert ok, (radius, worst)
        info = o.intervals_crown(lo, hi, net)
        for k in range(net.K - 1):
            R = ec.crown_post_target(net, lo, hi, pre, k, mode=mode).postprocessed()
            ok, r = R.check(*info.x_intvs[k + 1])
            assert ok.all(), (radius, k, r)
        assert np.array_equal(info.x_intvs[-1][0], np.minimum(*pre[-1]))


def _forward_exact(net, x):
    xs, ys = [np.array([Fraction(v) for v in x], dtype=object)], []
    for k, M in enumerate(net.Ms):
        W, b = np.array([[Fraction(v) for v in r] for r in M[:, :-1]], dtype=object), \
            np.array([Fraction(v) for v in M[:, -1]], dtype=object)
        y = W @ xs[-1] + b
        ys.append(y)
        xs.append(np.array([max(v, 0) for v in y], dtype=object))
    return ys, xs


@pytest.mark.parametrize("xdims", [[2, 6, 5, 7, 2], [3, 4, 7, 3, 5, 2]])
def test_exact_restatement_is_sound(xdims):
    net = wide_range_net(xdims, seed=3)
    rng = np.random.default_rng(0)
    lo, hi = _box(xdims[0], 9, 0.4)
    pre, params = ec.exact_crown(net, lo, hi)
    post = [ec.crown_post_target(net, lo, hi, None, k, params=params).postprocessed() for k in range(net.K - 1)]
    points = [np.array(v) for v in itertools.product(*zip(lo, hi))] + [rng.uniform(lo, hi) for _ in range(30)]
    tighter = 0
    for x in points:
        ys, xs = _forward_exact(net, x)
        for k in range(net.K):
            assert all(a <= v <= b for a, v, b in zip(pre[k][0], ys[k], pre[k][1])), k
        for k in range(net.K - 1):
            assert all(a <= v <= b for a, v, b in zip(post[k].lo, xs[k + 1], post[k].hi)), k
    ibp = o.intervals_worst_case(lo, hi, net)
    for k in range(1, net.K - 1):
        tighter += sum(float(b - a) for a, b in zip(*pre[k])) < float(np.sum(ibp.acx_intvs[k][1] - ibp.acx_intvs[k][0]))
    assert tighter >= 1                     # CROWN, not interval arithmetic


# ---- planted bugs -------------------------------------------------------------------------------------------------

def _params(l, u, bug):
    if bug == "eps":                                               # ub_r = max(ub_r, lb_r + 1e-8) dropped
        lb_r, ub_r = np.minimum(l, 0.0), np.maximum(u, 0.0)
        with np.errstate(invalid="ignore"):
            d_u = np.where(ub_r - lb_r > 0, ub_r / np.where(ub_r - lb_r > 0, ub_r - lb_r, 1.0), 0.0)
        return d_u, -lb_r * d_u, (d_u > 0.5).astype(float)
    d_u, b_u, d_l = ec.relax_params(l, u)
    if bug == "tie":                                               # d_l = (d_u >= 0.5)
        d_l = (d_u >= 0.5).astype(float)
    return d_u, b_u, d_l


def fp64_crown(net, lo, hi, bug=None):
    """An FP64 CROWN with the device's structure (pre-activation chains, x bounds as row scalings) and one planted
    bug; returns (pre, x_lo, x_hi)."""
    pre = [o._ibp_layer(net.Ms[0], lo, hi)]
    c, r = 0.5 * (lo + hi), 0.5 * (hi - lo)
    for t in range(1, net.K):
        out = []
        for upper in (False, True):
            A, beta = net.Ms[t][:, :-1].copy(), net.Ms[t][:, -1].copy()
            for k in range(t - 1, -1, -1):
                d_u, b_u, d_l = _params(*pre[k], bug)
                take_u = A > 0 if upper else A < 0
                side = np.where(take_u, A, 0.0)
                if bug == "lbias" and not upper and k == 0:        # entry 0 of layer 0 takes lA+ instead of lA-
                    side[:, 0] = np.maximum(A[:, 0], 0.0)
                beta = beta + side @ b_u
                a = A * np.where(take_u, d_u, d_l)
                bk = net.Ms[k][:, -1].copy()
                if bug == "bias0" and k == 0:                      # first-layer bias b_0[0] dropped
                    bk[0] = 0.0
                beta = beta + a @ bk
                A = a @ net.Ms[k][:, :-1]
            out.append(A @ c + (np.abs(A) @ r if upper else -(np.abs(A) @ r)) + beta)
        pre.append(tuple(out))
    x_lo, x_hi = [lo], [hi]
    for k in range(net.K - 1):
        d_u, b_u, d_l = _params(*pre[k], bug)
        L, Uu = d_l * pre[k][0], d_u * pre[k][1] + b_u
        L = np.minimum(L, Uu)
        x_lo.append(L)
        x_hi.append(np.maximum(L, Uu))
    x_lo.append(np.minimum(*pre[-1]))
    x_hi.append(np.maximum(np.minimum(*pre[-1]), pre[-1][1]))
    return pre, np.concatenate(x_lo), np.concatenate(x_hi)


def _mutation_case(point):
    """A deep net (K = 6) whose last layer is 10⁴ × larger than the others.  Neuron 0 of y_0 is the bug's site: a point
    box with y_0[0] = -4e-9 (W_0 row 0 = 0; the ε alone makes d_u = 0.6 > 1/2 there, so the lower slope is 1, where
    without it d_u = d_l = 0), or y_0[0] = x_0 + 2⁻²⁵ ∈ [-2⁻²⁷, 2⁻²⁷] exactly (an l = -u tie, wide enough that the ε
    does not apply, with a small b_u = 2⁻²⁸ and a small first-layer bias).  It feeds only y_1[0], whose own outgoing weights are 2⁻¹⁰ × the
    others: a bug there moves the early bounds by ~1e-9 and the last layer's by less than 1e-11 of its scale."""
    xd = [2, 6, 6, 6, 6, 6, 2]
    net = rand_net(xd, seed=5)
    Ms = [M.copy() for M in net.Ms]
    Ms[0][0] = [0.0, 0.0, -4e-9] if point else [1.0, 0.0, 2.0 ** -25]
    Ms[1][:, 0] = 0.0
    Ms[1][0, 0], Ms[1][0, -1] = 1.0, 1.0                          # y_1[0] stably active: the bug shows in x_2[0]
    Ms[2][:, 0] *= 2.0 ** -10
    Ms[-1] *= 1e4
    net = o.FeedFwdNet(xdims=xd, Ms=Ms)
    if point:
        lo = hi = np.array([0.25, 0.5])
    else:
        lo = np.array([-2.0 ** -25 - 2.0 ** -27, 0.3])
        hi = np.array([-2.0 ** -25 + 2.0 ** -27, 0.7])
    return net, lo, hi


@pytest.mark.parametrize("bug", ["eps", "tie", "lbias", "bias0"])
def test_planted_bug_passes_the_old_criterion_and_fails_the_new_one(bug):
    net, lo, hi = _mutation_case(point=(bug == "eps"))
    pre0, xl0, xh0 = fp64_crown(net, lo, hi)
    if bug == "eps":
        assert pre0[0][0][0] == pre0[0][1][0] == -4e-9 and ec.relax_params(*pre0[0])[2][0] == 1.0
    else:
        assert pre0[0][0][0] == -pre0[0][1][0] == -2.0 ** -27 and ec.relax_params(*pre0[0])[0][0] == 0.5
    # the unplanted restatement meets both criteria
    assert meets_old(net, lo, hi, xl0, xh0)
    assert meets_new(net, lo, hi, pre0)[0]
    pre, xl, xh = fp64_crown(net, lo, hi, bug)
    assert not (np.array_equal(xl, xl0) and np.array_equal(xh, xh0))           # the bug shows in the x bounds
    assert meets_old(net, lo, hi, xl, xh), "the planted bug should pass the old criterion"
    ok, ratio = meets_new(net, lo, hi, pre)
    assert not ok, f"the planted bug {bug} meets the new criterion (ratio {ratio:.3g})"
