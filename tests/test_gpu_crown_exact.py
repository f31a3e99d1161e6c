"""The device's CROWN bounds against the exact reference of oracle/exact_crown.py, layer by layer (one B200).

Each case runs Batch.bounds_crown() with the pre-activation bounds kept (Batch.keep_crown_preact) and checks, for every
checked query:
- y_0 (interval arithmetic) within γ_{n+3}(|W| max(|lo|, |hi|) + |b|) of the exact interval bounds;
- every y_t, t >= 1: |dev − exact| ≤ γ_N abs + N 2⁻¹⁰⁷⁴, the exact chain built from the device's OWN bounds of
  y_0 .. y_{t-1} (the relaxation parameters reproduced bit for bit);
- hidden x_{k+1}: bit for bit the row-scaling form of crown_post_kernel (default), or the exact criterion of the
  identity-slice chain (NNSDP_CROWN_POST_CHAINS=1); x_K the min/max of y_{K-1}; x_0 the box;
- acxmin / acxmax within the interval criterion from the CROWN x bounds; smin / smax = make_sector_min_max exactly.

The kernels a case takes (the one-launch chain kernel, the fused step, the row kernel + GEMV / SIMT GEMM / DMMA GEMM,
the row-scaling post kernel, the chain kernel's post targets, the wavefront and the per-target post chains) are predicted
on the host from the dispatch rules of api.cu / kernels_crown.cu / kernels_bounds.cu / kernels_dgemm.cu, and every
GPU case asserts the prediction against the kernels torch.profiler records and the launch count of the bounds stage.
The device runs happen in subprocesses: the A/B switches are read once per process, and the profiling stays out of the
test process."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import exact_crown as ec
import nnsdp_oracle as o
from helpers import rand_net, rand_query, wide_range_net

pytestmark = pytest.mark.gpu
EXACT_SUM = 40             # Fraction arithmetic up to this sum of widths, long double beyond
NAMES = {"crown_chain_kernel": "chain", "crown_step_kernel": "fused", "crown_row_kernel": "row",
         "gemv_small_kernel<2": "gemv", "gemm_nn_kernel<2>": "simt", "dgemm_dmma_kernel<0>": "dmma",
         "crown_post_kernel": "post", "crown_init_post_kernel": "init_post"}


# ---- the dispatch rules ----------------------------------------------------------------------------------------------

def _chain_fits(maxw, post, ntargets, nq, env):
    """launch_crown_chain: widths <= 128 whose two W buffers and row buffers fit 220 KiB of shared memory."""
    if env.get("NNSDP_NO_CROWN_CHAIN", "0") != "0" or maxw > 128 or ntargets < 1:
        return False
    ctas = nq * (ntargets if post else 1)
    rg = min(8, -(-128 // ctas)) if ctas < 128 else 1
    size = lambda rg: (2 * maxw * ((maxw + 1) & ~1) + 4 * (-(-maxw // rg)) * (maxw + 1) + 2 * (-(-maxw // rg))) * 8
    while size(rg) > 220 * 1024 and rg < 32:
        rg *= 2
    return size(rg) <= 220 * 1024


def plan(xdims, Q, env=None):
    """(kernel tags, launches of the bounds stage, queries per chunk) of Batch.bounds_crown()."""
    env = env or {}
    n, K = list(xdims), len(xdims) - 1
    acdim, maxn = sum(n[1:-1]), max(n)
    ld = (maxn + 1) & ~1
    wave = env.get("NNSDP_CROWN_NO_WAVEFRONT", "0") != "1" and K >= 16 and max(n[:K - 1]) <= 64
    rows_cap = max(maxn, acdim) if wave else maxn
    Qc = min(256, max(1, min(Q, (3 << 26) // max(1, 4 * rows_cap * ld))))
    fused_env = env.get("NNSDP_CROWN_FUSED")
    gemv_on, dmma_on = env.get("NNSDP_NO_GEMV", "0") == "0", env.get("NNSDP_NO_DMMA_GEMM", "0") == "0"
    post_chains = env.get("NNSDP_CROWN_POST_CHAINS") == "1"
    tags, launches = set(), 1                                               # place_x1

    def levels(k_first, nrows, nq):
        nonlocal launches
        for k in range(k_first, -1, -1):
            if (int(fused_env) != 0) if fused_env is not None else n[k] <= 64:
                tags.add("fused")
                launches += 1
                continue
            M, Kd, N = n[k], n[k + 1], 2 * nq * nrows
            tags.add("row")
            tags.add("gemv" if N <= 32 and gemv_on else
                     "dmma" if dmma_on and M >= 192 and N >= 128 and Kd >= 128 else "simt")
            launches += 2

    for q0 in range(0, Q, Qc):
        nq = min(Qc, Q - q0)
        launches += 2                                                       # y_0 by IBP, its relaxation
        for t in range(1, K):
            if _chain_fits(maxn, False, 1, nq, env):
                tags.add("chain")
                launches += 1
            else:
                launches += 2                                               # bias start, concretisation
                levels(t - 1, n[t + 1], nq)
            launches += t <= K - 2                                          # the relaxation of y_t
        if not post_chains:
            tags.add("post")
            launches += 1
        elif _chain_fits(maxn, True, K - 1, nq, env):
            tags |= {"chain", "chain_post"}
            launches += 1
        elif wave:
            tags |= {"wavefront", "init_post", "fused"}
            launches += (K - 1) + (K - 2) + (K - 1)
        else:
            tags |= {"per_target", "init_post"}
            for k in range(K - 1):
                launches += 2
                levels(k - 1, n[k + 1], nq)
        launches += 2                                                       # x_K
    launches += (K - 1) + 1                                                 # acx_intvs, sector slopes
    return tags, launches, Qc


def _launched(fn):
    import torch
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = set()
    for e in prof.key_averages():
        key = e.key.replace("(int)", "")
        names.update(m.group(0) for m in re.finditer(r"\w+_kernel(<[^>(]*>)?", key))
    return names


def observed(names):
    return {tag for nm in names for p, tag in NAMES.items() if nm.startswith(p)}


def name_level(tags):
    """The predicted tags as kernel names can show them."""
    return {t for t in tags if t in NAMES.values()}


# ---- the cases ---------------------------------------------------------------------------------------------------------

def _edge_net(seed):
    """First layer on the box [-1, 1]² with dyadic weights: y_0 ∈ [-1/2, 1/2] (l = -u), [0, 1/2] (l = 0), [-1/2, 0]
    (u = 0), [-2⁻³⁰, 2⁻³⁰] (|l|, |u| < 1e-8: the ε sets the slope), [-3·2⁻³⁰, -2⁻³⁰] (stably inactive, l > -1e-8), the
    point -4e-9 (the ε makes d_u = 0.6 > 1/2), [-1, 1] (another tie) and one generic neuron."""
    xd = [2, 8, 6, 5, 2]
    net = rand_net(xd, seed)
    M0 = np.array([[0.5, 0, 0], [0.25, 0, 0.25], [0.25, 0, -0.25], [2.0 ** -30, 0, 0], [2.0 ** -30, 0, -2.0 ** -29],
                   [0, 0, -4e-9], [-0.5, 0.5, 0], [0.5, 0.25, 0.125]])
    return o.FeedFwdNet(xdims=xd, Ms=[M0] + [M.copy() for M in net.Ms[1:]])


def _boxes(n0, Q, seed, radii=(0.0, 2.0 ** -20, 1e-3, 0.05, 0.5)):
    rng = np.random.default_rng(seed)
    c = rng.uniform(-1, 1, (Q, n0))
    r = np.array([radii[i % len(radii)] for i in range(Q)])[:, None] * rng.uniform(0.5, 1.0, (Q, n0))
    r[0] = 0.0
    return c - r, c + r


def case(name):
    """(net, x1min, x1max (Q x n0), checked queries, rows of y_t to check (a function of t; None = all))."""
    if name == "chain":                        # one-launch chain kernel, wide-range weights
        net = wide_range_net([2, 4, 7, 3, 5, 2], seed=11)
        lo, hi = _boxes(2, 6, 1)
        return net, lo, hi, range(6), None
    if name == "edge":
        net = _edge_net(4)
        lo = np.array([[-1.0, -1.0], [0.0, 0.5], [-2.0 ** -20, 0.25 - 2.0 ** -20]])
        hi = np.array([[1.0, 1.0], [0.0, 0.5], [2.0 ** -20, 0.25 + 2.0 ** -20]])
        return net, lo, hi, range(3), None
    if name == "deep":                         # K = 21, widths <= 64: the wavefront's shape
        net = wide_range_net([3] + [9, 12, 7, 10] * 5 + [2], seed=21)
        lo, hi = _boxes(3, 3, 2, radii=(0.0, 0.02, 0.3))
        return net, lo, hi, range(3), None
    if name == "gemm":                         # odd widths >= 192 x 128: every edge of the GEMM tiles
        net = wide_range_net([3, 131, 257, 193, 129, 2], seed=9)
        lo, hi = _boxes(3, 5, 3)
        return net, lo, hi, range(5), None
    if name == "narrow_chunks":                # Q > 256: two chunks of the chain kernel
        net = wide_range_net([2, 8, 9, 7, 2], seed=12)
        lo, hi = _boxes(2, 300, 4)
        return net, lo, hi, (0, 1, 255, 256, 299), None
    if name == "wide_chunks":                  # width 1000: 50 queries per chunk, queries on both sides, sampled rows
        net = rand_net([2, 1000, 1000, 2], seed=13)
        lo, hi = _boxes(2, 52, 5, radii=(0.0, 1e-3, 0.05))
        rows = lambda t: np.unique(np.r_[0, 1, 62, 63, 64, 127, 128, 998, 999,
                                         np.random.default_rng(t).choice(net.xdims[t + 1], 12)]) \
            if net.xdims[t + 1] > 64 else None
        return net, lo, hi, (0, 49, 50, 51), rows
    raise ValueError(name)


DEFAULT = ["chain", "edge", "deep", "gemm", "narrow_chunks", "wide_chunks"]
AB_RUNS = [
    ({"NNSDP_NO_CROWN_CHAIN": "1"}, ["edge", "deep"]),
    ({"NNSDP_NO_CROWN_CHAIN": "1", "NNSDP_CROWN_FUSED": "0"}, ["edge"]),
    ({"NNSDP_CROWN_FUSED": "1"}, ["gemm"]),
    ({"NNSDP_CROWN_FUSED": "0"}, ["gemm"]),
    ({"NNSDP_CROWN_POST_CHAINS": "1"}, ["deep", "gemm"]),
    ({"NNSDP_CROWN_POST_CHAINS": "1", "NNSDP_NO_CROWN_CHAIN": "1"}, ["deep", "edge"]),
    ({"NNSDP_CROWN_POST_CHAINS": "1", "NNSDP_NO_CROWN_CHAIN": "1", "NNSDP_CROWN_NO_WAVEFRONT": "1"}, ["deep"]),
    ({"NNSDP_NO_DMMA_GEMM": "1"}, ["gemm", "wide_chunks"]),
    ({"NNSDP_NO_GEMV": "1"}, ["gemm"]),
]
PATHS = {"chain", "fused", "row", "gemv", "simt", "dmma", "post"}
AB_PATHS = {"chain_post", "wavefront", "per_target"}


def device_run(ctx, name):
    """Run one case on the device: (prel, preu, bounds, kernel tags, bounds-stage launches)."""
    import nnsdp_b200 as nb

    net, lo, hi, _, _ = case(name)
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    b = nb.Batch(dnet, 1, Qcap=lo.shape[0], ring=0)
    b.set_inputs(nb.NumericBatch(x1min=lo, x1max=hi))
    b.keep_crown_preact(True)
    names = _launched(b.bounds_crown)
    launches = b.stage_ms("bounds")[1]
    prel, preu = b.get_crown_preact()
    bd = b.get_bounds()
    b.close()
    return prel, preu, bd, observed(names), launches


def check_query(net, lo, hi, prel, preu, bd, post_chains=False, rows=None):
    """Every criterion of the module docstring for one query."""
    xd, K, n0 = net.xdims, net.K, net.xdims[0]
    mode = "exact" if sum(xd) <= EXACT_SUM else "extended"
    xoff = np.concatenate([[0], np.cumsum(xd)])
    noff = np.concatenate([[0], np.cumsum(xd[1:-1])])
    pre = [(prel[xoff[k + 1] - n0:xoff[k + 2] - n0], preu[xoff[k + 1] - n0:xoff[k + 2] - n0]) for k in range(K)]
    xmin, xmax = bd["xmin"], bd["xmax"]
    assert np.array_equal(xmin[:n0], lo) and np.array_equal(xmax[:n0], hi)
    assert ec.meets_ibp(net, 0, lo, hi, *pre[0]), "y_0"
    for t in range(1, K):
        sel = rows(t) if rows else None
        R = ec.crown_target(net, lo, hi, pre, t, rows=sel, mode=mode)
        idx = R.rows
        ok, ratio = R.check(pre[t][0][idx], pre[t][1][idx])
        assert ok.all(), f"y_{t}: rows {idx[~ok][:8]} break the bound, worst |err| / bound = {ratio:.3g}"
    for k in range(K - 1):
        dlo, dhi = xmin[xoff[k + 1]:xoff[k + 2]], xmax[xoff[k + 1]:xoff[k + 2]]
        if post_chains:
            R = ec.crown_post_target(net, lo, hi, pre, k, mode=mode).postprocessed()
            ok, ratio = R.check(dlo, dhi)
            assert ok.all(), f"x_{k + 1}: worst |err| / bound = {ratio:.3g}"
        else:
            plo, phi = ec.post_rowscale(*pre[k])
            assert np.array_equal(dlo, plo) and np.array_equal(dhi, phi), f"x_{k + 1}"
    lK = np.minimum(*pre[K - 1])
    assert np.array_equal(xmin[xoff[K]:], lK) and np.array_equal(xmax[xoff[K]:], np.maximum(lK, pre[K - 1][1]))
    for k in range(K - 1):
        alo, ahi = bd["acxmin"][noff[k]:noff[k + 1]], bd["acxmax"][noff[k]:noff[k + 1]]
        assert ec.meets_ibp(net, k, xmin[xoff[k]:xoff[k + 1]], xmax[xoff[k]:xoff[k + 1]], alo, ahi), f"acx_{k}"
    smin, smax = o.make_sector_min_max(bd["acxmin"], bd["acxmax"])
    assert np.array_equal(bd["smin"], smin) and np.array_equal(bd["smax"], smax)


def check_case(name, prel, preu, bd, tags, launches, env=None):
    net, lo, hi, checked, rows = case(name)
    want, nlaunch, _ = plan(net.xdims, lo.shape[0], env)
    assert tags == name_level(want), (name, env, tags, want)
    assert launches == nlaunch, (name, env, launches, nlaunch)
    post_chains = (env or {}).get("NNSDP_CROWN_POST_CHAINS") == "1"
    for i in checked:
        try:
            check_query(net, lo[i], hi[i], prel[i], preu[i], {k: v[i] for k, v in bd.items()}, post_chains, rows)
        except AssertionError as e:
            raise AssertionError(f"case {name}, query {i}, env {env}: {e}") from None


# ---- host-side coverage -----------------------------------------------------------------------------------------------

def _case_shape(name):
    net, lo, _, _, _ = case(name)
    return net.xdims, lo.shape[0]


def test_cases_cover_every_default_path():
    got = set().union(*(plan(*_case_shape(c))[0] for c in DEFAULT))
    assert PATHS <= got, PATHS - got
    assert plan(*_case_shape("narrow_chunks"))[2] == 256 and plan(*_case_shape("wide_chunks"))[2] == 50


def test_ab_runs_cover_every_switch_and_post_path():
    got = set()
    for env, names in AB_RUNS:
        for c in names:
            tags = plan(*_case_shape(c), env)[0]
            assert tags != plan(*_case_shape(c))[0], (env, c)        # every run leaves the default path
            got |= tags
    assert (PATHS | AB_PATHS) <= got, (PATHS | AB_PATHS) - got
    switches = {"NNSDP_NO_CROWN_CHAIN", "NNSDP_CROWN_FUSED", "NNSDP_CROWN_POST_CHAINS", "NNSDP_CROWN_NO_WAVEFRONT",
                "NNSDP_NO_DMMA_GEMM", "NNSDP_NO_GEMV"}
    assert switches == set().union(*(env.keys() for env, _ in AB_RUNS))


# ---- the GPU cases ----------------------------------------------------------------------------------------------------

_RUN_SNIPPET = r"""
import os, sys
import numpy as np
root, out, names = sys.argv[1], sys.argv[2], sys.argv[3:]
for p in ("nn-sdp_b200", "oracle", "tests"):
    sys.path.insert(0, os.path.join(root, p))
import nnsdp_b200 as nb
import test_gpu_crown_exact as T
ctx = nb.Context([0])
for name in names:
    prel, preu, bd, tags, launches = T.device_run(ctx, name)
    np.savez(os.path.join(out, name + ".npz"), prel=prel, preu=preu, tags=np.array(sorted(tags)),
             launches=launches, **bd)
"""


def _run_in_subprocess(env, names, out):
    """device_run of the cases `names` in a fresh process with the switches `env`; (prel, preu, bounds, tags, launches)
    per case.  The profiling stays out of the test process, whose other files profile their own launches."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    script = out / "run.py"
    script.write_text(_RUN_SNIPPET)
    r = subprocess.run([sys.executable, str(script), root, str(out)] + names, capture_output=True, text=True,
                       env=dict(os.environ, **env), timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    runs = {}
    for name in names:
        d = np.load(out / f"{name}.npz")
        bd = {k: d[k] for k in ("xmin", "xmax", "acxmin", "acxmax", "smin", "smax")}
        runs[name] = (d["prel"], d["preu"], bd, set(d["tags"].tolist()), int(d["launches"]))
    return runs


@pytest.fixture(scope="module")
def default_runs(ctx, tmp_path_factory):
    return _run_in_subprocess({}, DEFAULT, tmp_path_factory.mktemp("crown_default"))


@pytest.mark.parametrize("name", DEFAULT)
def test_default_paths_meet_the_exact_criterion(default_runs, name):
    check_case(name, *default_runs[name])


@pytest.mark.parametrize("env,names", AB_RUNS, ids=["+".join(f"{k}={v}" for k, v in e.items()) for e, _ in AB_RUNS])
def test_ab_paths_meet_the_exact_criterion(ctx, env, names, tmp_path):
    runs = _run_in_subprocess(env, names, tmp_path)
    for name in names:
        check_case(name, *runs[name], env)


def test_shared_box_reach_batch_over_two_chunks(ctx):
    """A reach batch with one (stride-0) box for 300 directions, CROWN bounds through set_bounds_method + run: two
    chunks of 256 + 44 queries, every query the same bounds, which meet the criterion."""
    import nnsdp_b200 as nb

    net = wide_range_net([2, 8, 9, 7, 2], seed=31)
    Q, beta = 300, 1
    base = rand_query(net, beta, np.random.default_rng(3), kind="hplane", radius=0.2)
    th = 2 * np.pi * np.arange(Q) / Q
    batch = nb.NumericBatch(x1min=base.x1min, x1max=base.x1max, gamma_in=base.gin, gamma_bnd=base.gbnd,
                            gamma_sec=base.gsec, out_kind=nb.OUT_HPLANE,
                            out_vec=np.stack([np.cos(th), np.sin(th)], axis=1), gamma_out=np.full((Q, 1), 0.5))
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    b = nb.Batch(dnet, beta, Qcap=Q, ring=4)
    b.set_inputs(batch, Q=Q)
    b.set_bounds_method("crown")
    with pytest.raises(nb.NnsdpError):
        b.get_crown_preact()                              # keeping is off
    b.keep_crown_preact(True)
    with pytest.raises(nb.NnsdpError):
        b.get_crown_preact()                              # no CROWN pass yet
    out = np.empty((Q, b.per_query))
    b.run(out)
    prel, preu = b.get_crown_preact()
    bd = b.get_bounds()
    b.bounds()                                            # an IBP pass: the kept CROWN bounds are stale
    with pytest.raises(nb.NnsdpError):
        b.get_crown_preact()
    b.close()
    for a in (prel, preu, bd["xmin"], bd["xmax"], bd["acxmin"]):
        assert (a == a[0]).all()
    for i in (0, 256, 299):
        check_query(net, base.x1min, base.x1max, prel[i], preu[i], {k: v[i] for k, v in bd.items()})
