"""Every coefficient of the affine-coefficient hand-off (nnsdp_affine_create, nnsdp_affine_create_batch) against the
entrywise reference of oracle/exact_affine.py (one B200):

    |dev − ref| ≤ γ_N·abs + N·2⁻¹⁰⁷⁴ per (variable, cover entry), coefficients with abs = 0 exactly 0 or absent.

The device's COO duplicates are summed in exact arithmetic by the test; the criterion is required over the union of
the device-listed and the exactly non-zero pairs (a missing pair counts as 0).  z0 is held to exact_z at γ = 0.  Each
batched group is checked against the reference of its own first query's bounds, and its var_ptr against the exclusive
scan of the exact per-variable counts.

Cases: the parity shapes and the narrow-layer shapes with all five output kinds; caller-supplied wide-range bounds
(fractional slopes, smin = 0, stably active, a subnormal smin·smax and one that rounds to 0), CROWN bounds and bounds
the library computes from the box; layers past the fill kernels' stride of 256 (300, 520 and 1000 wide); the grouping
edges of the batched form; and batches whose device scan runs in one tile, in several and in more than 256 (the carry
loop of scan_sums_kernel).  Which launch path each case takes is predicted from the dispatch rules (predicted_paths), and a
host-side test asserts that the cases cover every path."""
import math

import numpy as np
import pytest

import exact_affine as ea
import nnsdp_oracle as o
from helpers import assert_meets, rand_net, rand_out, rand_query, to_numeric_batch, wide_range_net, wide_range_query

EXACT_ZDIM = 150           # Fraction arithmetic up to here, long double beyond
KINDS = ["safety", "hplaneS", "hplane", "circle", "ellipsoid"]
SCAN_TILE, SCAN_THREADS = 1024, 256   # kernels_affine.cu: items per scan tile, tile sums per pass of scan_sums_kernel
AFF_THREADS = 256                     # kernels_affine.cu: stride of the fill loops

# the parity NETS, β ≥ acdim − 1, β > a layer's width, β = 0 and a deep narrow net with β = 7
SHAPES = [([2, 3, 3, 2], 1), ([2, 3, 2], 0), ([2, 3, 2], 2), ([3, 3, 3, 3, 4, 3, 3], 2), ([2, 10, 10, 10, 10, 2], 3),
          ([2, 4, 7, 3, 5, 2], 5), ([5, 50, 50, 50, 50, 50, 50, 5], 2), ([2] + [20] * 10 + [2], 1),
          ([2, 70, 130, 64, 3], 2), ([2, 1, 2, 2], 3), ([2, 6, 5, 4, 2], 0), ([2] + [10] * 9 + [2], 7)]
SOURCES = ["wide", "crown", "computed"]
WIDE = [([2, 300, 257, 2], 1), ([2, 1000, 520, 2], 1)]
SCAN_NET, SCAN_BETA = [2, 10, 10, 2], 1


def nvar_of(xdims, beta, kind):
    n1, ac = xdims[0], sum(xdims[1:-1])
    return n1 + (0 if kind in ("safety", "hplaneS") else 1) + ac + o.sector_lambda_dim(ac, beta) + 2 * ac


SCAN_GROUPS = [11, 2700]   # 11 · 101 + 1 = 1112 counts: two tiles; 2700 · 101 + 1: 267 tiles, two carry passes


def _cases():
    """(xdims, β, kinds, form, groups, bounds source) of every GPU case below"""
    out = [(x, b, KINDS, "single", 1, s) for x, b in SHAPES for s in SOURCES]
    out += [(x, b, ["hplane"], form, 2 if form == "batch" else 1, "supplied") for x, b in WIDE
            for form in ("single", "batch")]
    out += [([2, 4, 7, 3, 5, 2], 3, ["safety"], "batch", 14, "supplied")]
    out += [([2, 6, 5, 7, 5], 2, [k], "batch", 3, "computed") for k in KINDS]
    out += [(SCAN_NET, SCAN_BETA, ["safety"], "batch", G, "supplied") for G in SCAN_GROUPS]
    return out


def predicted_paths(xdims, beta, kinds, form, groups, source):
    """the launch paths of one case, from the dispatch rules: the single call scans the counts on the host, the
    batched form on the device in ceil((groups · nvar + 1) / 1024) tiles, with a carry loop past 256 tiles; bounds
    the caller does not supply are computed by the interval kernels; the fill loops stride by 256 rows and columns"""
    paths = {f"kind:{k}" for k in kinds}
    if form == "single":
        paths.add("host scan")
    else:
        tiles = math.ceil((groups * nvar_of(xdims, beta, kinds[0]) + 1) / SCAN_TILE)
        paths.add("device scan, 1 tile" if tiles == 1 else
                  "device scan, several tiles" if tiles <= SCAN_THREADS else "device scan, carry loop")
    if source == "computed":
        paths.add("computed bounds")
    strides = math.ceil(max(xdims[1:-1]) / AFF_THREADS)
    paths.add(f"fill strides: {min(strides, 3)}")
    return paths


def test_cases_cover_every_path():
    """host-side: the cases reach every scan path, the computed bounds, widths past two fill strides, all kinds"""
    seen = set()
    for case in _cases():
        seen |= predicted_paths(*case)
    want = {"host scan", "device scan, 1 tile", "device scan, several tiles", "device scan, carry loop",
            "computed bounds", "fill strides: 1", "fill strides: 2", "fill strides: 3"} | {f"kind:{k}" for k in KINDS}
    assert want <= seen, want - seen
    # the scan batches: just above one tile, and past 256 tiles (SCAN_NET, β = 1, safety: 101 variables)
    assert nvar_of(SCAN_NET, SCAN_BETA, "safety") == 101
    tiles = [math.ceil((G * 101 + 1) / SCAN_TILE) for G in SCAN_GROUPS]
    assert tiles[0] == 2 and tiles[1] > SCAN_THREADS


# ---- helpers --------------------------------------------------------------------------------------------------------

def _mode(net):
    return "exact" if net.Zdim <= EXACT_ZDIM else "extended"


def _special_slopes(net, bounds):
    """on layer 1 (|w|, |b| ≤ 1 in wide_range_net): smin = smax = 2⁻⁵²⁰ (smin·smax = 2⁻¹⁰⁴⁰ subnormal) and 2⁻⁶⁰⁰
    (smin·smax rounds to 0: the device skips the Gram terms on the rounded product)"""
    if net.xdims[1] >= 4:
        for j, e in ((2, -520), (3, -600)):
            bounds[2][j] = bounds[3][j] = 2.0 ** e
    return bounds


def _query(xdims, beta, kind, source, seed):
    """(net, query, bounds or None)"""
    rng = np.random.default_rng(seed)
    if source == "wide":
        net = wide_range_net(xdims, seed)
        q, bounds = wide_range_query(net, beta, kind, rng)
        return net, q, _special_slopes(net, list(bounds))
    net = rand_net(xdims, seed=seed)
    return net, rand_query(net, beta, rng, kind=kind, radius=0.2), None


def _bounds_of_box(nb, dnet, net, source, x1min, x1max, Q=1, beta=0):
    """QC bounds of Q boxes: CROWN (the reference's path), or those the library computes in a batch of Q (IBP)"""
    n1, ac = net.xdims[0], net.acdim
    if source == "crown":
        r = nb.bounds_crown(dnet, x1min, x1max)
        smin, smax = nb.sector_minmax(dnet.ctx, r["acxmin"], r["acxmax"])
        return r["xmin"][:, n1:n1 + ac], r["xmax"][:, n1:n1 + ac], smin, smax
    secdim = nb.sizes_from_xdims(net.xdims, beta)["secdim"]
    b = nb.Batch(dnet, beta, Qcap=Q, ring=1)
    b.set_inputs(nb.NumericBatch(x1min=x1min, x1max=x1max, gamma_in=np.zeros(n1), gamma_bnd=np.zeros(ac),
                                 gamma_sec=np.zeros(secdim), out_kind=nb.OUT_HPLANE, out_vec=np.ones(net.xdims[-1]),
                                 gamma_out=np.zeros(1)), Q)
    b.bounds()
    bd = b.get_bounds()
    b.close()
    return bd["xmin"][:, n1:n1 + ac], bd["xmax"][:, n1:n1 + ac], bd["smin"], bd["smax"]


def _check_z0(net, beta, q, bounds, z0, er, ec, what, rows=None):
    Zd = np.zeros((net.Zdim, net.Zdim))
    Zd[er, ec] = Zd[ec, er] = z0
    R = ea.exact_z0(net, beta, q, bounds, mode=_mode(net) if rows is None else "extended", rows=rows)
    assert_meets(R, Zd if rows is None else Zd[rows], f"{what} z0")


def _check_sizes(D, lay):
    assert np.array_equal(D["ent_row"] - 1, lay.ent_row) and np.array_equal(D["ent_col"] - 1, lay.ent_col)
    assert (D["nvar"], D["nent"]) == (lay.nvar, lay.nent)
    assert (D["var_in"], D["var_out"], D["var_bnd"], D["var_sec"]) == (0, lay.var_out, lay.var_bnd, lay.var_sec)


def _csc_triplets(grp):
    vp = grp["var_ptr"] - 1
    var = np.repeat(np.arange(len(vp) - 1), np.diff(vp))
    return var, grp["ent_idx"] - 1, grp["val"]


def _check_group(grp, R, what, vars=None, counts=True):
    """one group's CSC: strictly ascending entries per variable, var_ptr = exclusive scan of the exact counts, values"""
    var, ent, val = _csc_triplets(grp)
    key = var * R.lay.nent + ent
    assert np.all(np.diff(key) > 0), f"{what}: entries not strictly ascending"
    if counts:
        assert np.array_equal(grp["var_ptr"], np.r_[0, np.cumsum(R.counts())] + 1), f"{what}: var_ptr"
    assert_meets(R, (var, ent, val), what, vars=vars)


def _underflows(bounds):
    smin, smax = bounds[2], bounds[3]
    return bool(np.any((smin * smax == 0) & (smin != 0) & (smax != 0)))


# ---- single calls: shapes, kinds and bound sources ------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("source", SOURCES)
@pytest.mark.parametrize("xdims,beta", SHAPES)
def test_single_call_every_coefficient(ctx, xdims, beta, source):
    import nnsdp_b200 as nb

    for i, kind in enumerate(KINDS):
        net, q, bounds = _query(xdims, beta, kind, source, seed=100 * beta + 7 * i + len(xdims))
        dnet = nb.Net(ctx, net.xdims, net.Ms)
        batch = to_numeric_batch(nb, net, [q])
        if source == "crown":
            bounds = [b[0] for b in _bounds_of_box(nb, dnet, net, "crown", q.x1min[None], q.x1max[None])]
        if source != "computed":
            batch.ymin, batch.ymax, batch.smin, batch.smax = (np.asarray(b)[None] for b in bounds)
        D = nb.affine_form(dnet, beta, batch)
        if source == "computed":
            bounds = [b[0] for b in _bounds_of_box(nb, dnet, net, "computed", q.x1min[None], q.x1max[None], 1, beta)]
        R = ea.exact_affine(net, beta, q, bounds, mode=_mode(net))
        _check_sizes(D, R.lay)
        what = f"{xdims} β={beta} {kind} {source}"
        assert_meets(R, (D["coo_var"] - 1, D["coo_ent"] - 1, D["coo_val"]), what)
        listed = len(np.unique((D["coo_var"] - 1) * R.lay.nent + D["coo_ent"] - 1))
        if _underflows(bounds):   # smin·smax rounded to 0: the Gram terms are absent, and within the bound
            assert listed < len(R.key), what
        else:
            assert listed == len(R.key), what
        _check_z0(net, beta, q, bounds, D["z0"], R.lay.ent_row, R.lay.ent_col, what)


# ---- widths past the fill kernels' stride --------------------------------------------------------------------------

def _wide_case(xdims, beta, seed=3):
    """hplane, caller bounds with at most two Gram-active neurons per layer (neuron 1 and the last)"""
    net = rand_net(xdims, seed=seed)
    rng = np.random.default_rng(seed)
    q = rand_query(net, beta, rng, kind="hplane", radius=0.2)
    ac = net.acdim
    ymin = -rng.uniform(0.1, 2.0, ac)
    ymax = ymin + rng.uniform(0.1, 2.0, ac)
    smin, smax = np.zeros(ac), rng.uniform(0.2, 1.0, ac)
    st = np.r_[0, np.cumsum(xdims[1:-1])]
    for L in range(len(xdims) - 2):
        for j in (st[L] + 1, st[L + 1] - 1):
            smin[j] = rng.uniform(0.05, 0.2)
    return net, q, (ymin, ymax, smin, smax)


def _wide_vars(net, beta, lay, seed=0):
    """λ, η, ν of neurons 0, 1, 255, 256, 257, 511, 512 and the last of each layer, every pair holding one of them, all
    γin, γout, γbnd, and a seeded sample of the rest"""
    ac = net.acdim
    st = np.r_[0, np.cumsum(net.xdims[1:-1])]
    J = np.unique(np.concatenate([st[L] + np.array([j for j in (0, 1, 255, 256, 257, 511, 512, n - 1) if j < n])
                                  for L, n in enumerate(net.xdims[1:-1])]))
    pairs = o.sector_pairs(ac, beta) - 1
    pk = np.flatnonzero(np.isin(pairs[:, 0], J) | np.isin(pairs[:, 1], J))
    vs = [np.arange(lay.var_sec), lay.var_sec + J, lay.var_sec + ac + pk, lay.var_sec + lay.lamdim + J,
          lay.var_sec + lay.lamdim + ac + J, np.random.default_rng(seed).integers(0, lay.nvar, 40)]
    return np.unique(np.concatenate(vs))


@pytest.mark.gpu
@pytest.mark.parametrize("xdims,beta", WIDE)
def test_wide_layers_single_and_batched(ctx, xdims, beta):
    import nnsdp_b200 as nb

    net, q, bounds = _wide_case(xdims, beta)
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    lay = ea.layout(net, beta, q.qc_out)
    vars = None if max(xdims) <= 512 else _wide_vars(net, beta, lay)
    R = ea.exact_affine(net, beta, q, bounds, mode="extended", vars=vars, lay=lay)
    batch = to_numeric_batch(nb, net, [q])
    batch.ymin, batch.ymax, batch.smin, batch.smax = (np.asarray(b)[None] for b in bounds)
    D = nb.affine_form(dnet, beta, batch)
    _check_sizes(D, lay)
    assert_meets(R, (D["coo_var"] - 1, D["coo_ent"] - 1, D["coo_val"]), f"{xdims} single", vars=vars)
    rows = np.unique(np.r_[0:3, np.cumsum(xdims[:-1]) - 1, np.cumsum(xdims[:-1]), 255, 256, 257, 511, 512, 513,
                           net.Zdim - 1])
    rows = rows[rows < net.Zdim]
    _check_z0(net, beta, q, bounds, D["z0"], lay.ent_row, lay.ent_col, f"{xdims} single", rows=rows)
    del D
    # two groups: the box and the bounds of q, and a second query whose last (Gram-active) neuron has another smax
    b2 = [np.stack([b, b]) for b in bounds]
    b2[3][1, -1] = 0.5
    batch = nb.NumericBatch(x1min=np.stack([q.x1min] * 2), x1max=np.stack([q.x1max] * 2), out_kind=nb.OUT_HPLANE,
                            out_vec=np.stack([q.qc_out.normal] * 2), ymin=b2[0], ymax=b2[1], smin=b2[2], smax=b2[3])
    B = nb.affine_form_batch(dnet, beta, batch)
    assert B["ngroups"] == 2 and list(B["group_of"]) == [0, 1]
    _check_sizes(B, lay)
    _check_group(B["groups"][0], R, f"{xdims} group 0", vars=vars, counts=vars is None)
    R1 = ea.exact_affine(net, beta, q, [b[1] for b in b2], mode="extended", vars=vars, lay=lay)
    _check_group(B["groups"][1], R1, f"{xdims} group 1", vars=vars, counts=vars is None)
    if vars is not None:   # the listed variables' counts, against the device's var_ptr
        for grp, RR in zip(B["groups"], (R, R1)):
            assert np.array_equal(np.diff(grp["var_ptr"])[vars], RR.counts()[vars])
    for i in range(2):
        _check_z0(net, beta, q, [b[i] for b in b2], B["z0"][i], lay.ent_row, lay.ent_col, f"{xdims} batch {i}", rows)


# ---- batched form: grouping edges, output kinds, computed bounds ---------------------------------------------------

@pytest.mark.gpu
def test_grouping_edges_each_group_exact(ctx):
    """A base query and, for each key column (x1min, x1max, ymin, ymax, smin, smax), a query differing at its last
    element by one ulp and one by a large amount: 12 groups of their own.  smin = −0.0 against +0.0: a 14th group.
    Queries that differ only in the output QC share the base's group.  Safety S with junk in its strict lower
    triangle (the upper triangle is authoritative)."""
    import nnsdp_b200 as nb

    xdims, beta = [2, 4, 7, 3, 5, 2], 3
    net = wide_range_net(xdims, 9)
    rng = np.random.default_rng(9)
    q0, bounds = wide_range_query(net, beta, "safety", rng)
    bounds = [np.asarray(b, dtype=np.float64).copy() for b in bounds]
    bounds[2][-1], bounds[3][-1] = 0.25, 0.5
    bounds[2][-2] = 0.0
    base = dict(x1min=q0.x1min, x1max=q0.x1max, ymin=bounds[0], ymax=bounds[1], smin=bounds[2], smax=bounds[3])
    big = dict(x1min=-0.25, x1max=0.25, ymin=-1.0, ymax=1.0, smin=-0.125, smax=0.25)
    rows = [base]
    for k in ("x1min", "x1max", "ymin", "ymax", "smin", "smax"):
        for step in ("ulp", "big"):
            r = {kk: v.copy() for kk, v in base.items()}
            x = r[k][-1]
            r[k][-1] = (np.nextafter(x, -np.inf if k in ("x1min", "ymin") else np.inf) if step == "ulp"
                        else x + big[k])
            rows.append(r)
    r = {kk: v.copy() for kk, v in base.items()}
    r["smin"][-2] = -0.0
    rows.append(r)
    rows += [base, base]
    Q = len(rows)
    S = []
    for i in range(Q):
        s = rand_out(net, "safety", rng)[0].S
        S.append(np.triu(s) + np.tril(rng.standard_normal(s.shape), -1))        # junk below the diagonal
    batch = nb.NumericBatch(out_kind=nb.OUT_SAFETY, out_S=np.stack(S),
                            **{k: np.stack([r[k] for r in rows]) for k in base})
    B = nb.affine_form_batch(nb.Net(ctx, net.xdims, net.Ms), beta, batch)
    assert B["ngroups"] == 14 and list(B["group_of"]) == list(range(14)) + [0, 0]
    lay = ea.layout(net, beta, o.QcSafety(S=S[0]))
    _check_sizes(B, lay)
    for g, grp in enumerate(B["groups"]):
        r = rows[grp["first"]]
        q = o.NumericQuery(x1min=r["x1min"], x1max=r["x1max"], gin=q0.gin, gbnd=q0.gbnd, gsec=q0.gsec,
                           qc_out=o.QcSafety(S=S[grp["first"]]))
        bnd = (r["ymin"], r["ymax"], r["smin"], r["smax"])
        _check_group(grp, ea.exact_affine(net, beta, q, bnd, lay=lay), f"group {g}")
    for i in range(Q):
        r = rows[i]
        q = o.NumericQuery(x1min=r["x1min"], x1max=r["x1max"], gin=q0.gin, gbnd=q0.gbnd, gsec=q0.gsec,
                           qc_out=o.QcSafety(S=S[i]))
        _check_z0(net, beta, q, (r["ymin"], r["ymax"], r["smin"], r["smax"]), B["z0"][i], lay.ent_row, lay.ent_col,
                  f"query {i}")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_batch_computed_bounds_every_kind(ctx, kind):
    """Q = 7 over 3 boxes, bounds computed by the library (IBP); the reference bounds from an nb.Batch over the same
    boxes at the same Q, where equal boxes give bit-identical bounds.  n_out = 5: the ellipsoid's U loop in z0."""
    import nnsdp_b200 as nb

    xdims, beta, box_of = [2, 6, 5, 7, 5], 2, [0, 1, 0, 2, 1, 0, 2]
    net = rand_net(xdims, seed=4)
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    rng = np.random.default_rng(4)
    boxes = [(c - r, c + r) for c, r in ((rng.uniform(0.5, 1.5, 2), r) for r in (0.3, 0.0, 0.1))]
    qs = []
    for b in box_of:
        q = rand_query(net, beta, rng, kind=kind, radius=0.0)
        q.x1min, q.x1max = boxes[b][0].copy(), boxes[b][1].copy()
        qs.append(q)
    B = nb.affine_form_batch(dnet, beta, to_numeric_batch(nb, net, qs))
    assert B["ngroups"] == 3 and list(B["group_of"]) == box_of
    x1min, x1max = np.stack([q.x1min for q in qs]), np.stack([q.x1max for q in qs])
    bd = _bounds_of_box(nb, dnet, net, "computed", x1min, x1max, Q=7, beta=beta)
    for i, b in enumerate(box_of):
        j = box_of.index(b)
        assert all(np.array_equal(x[i], x[j]) for x in bd), i
    lay = ea.layout(net, beta, qs[0].qc_out)
    _check_sizes(B, lay)
    for g, grp in enumerate(B["groups"]):
        f = grp["first"]
        _check_group(grp, ea.exact_affine(net, beta, qs[f], [x[f] for x in bd], lay=lay), f"{kind} group {g}")
    for i, q in enumerate(qs):
        _check_z0(net, beta, q, [x[i] for x in bd], B["z0"][i], lay.ent_row, lay.ent_col, f"{kind} query {i}")


# ---- the device scan: one tile, several, and more than 256 ---------------------------------------------------------

PATTERNS = 7


@pytest.mark.gpu
@pytest.mark.parametrize("G", SCAN_GROUPS)
def test_device_scan_every_group(ctx, G):
    """G groups on SCAN_NET: group g has its own box (x1min[1] moved by g · 2⁻⁴⁰) and one of PATTERNS slope patterns
    with different Gram-active sets, so the per-group counts differ.  Every group's var_ptr against the exclusive
    scan of its exact counts, and every coefficient: the γin ones against the group's own reference, the rest against
    its pattern's.  One shared safety S: every z0 against the one exact Z₀."""
    import nnsdp_b200 as nb

    xdims, beta = SCAN_NET, SCAN_BETA
    net = rand_net(xdims, seed=13)
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    rng = np.random.default_rng(13)
    ac = net.acdim
    q0 = rand_query(net, beta, rng, kind="safety", radius=0.25)
    ymin = -rng.uniform(0.1, 2.0, ac)
    ymax = ymin + rng.uniform(0.1, 2.0, ac)
    pats = []
    for p in range(PATTERNS):
        smin, smax = np.zeros(ac), rng.uniform(0.3, 1.0, ac)
        act = rng.random(ac) < (p + 1) / (PATTERNS + 1)
        smin[act] = rng.uniform(0.05, 0.3, act.sum())
        pats.append((ymin, ymax, smin, smax))
    pat = np.arange(G) % PATTERNS
    x1min = np.stack([q0.x1min] * G)
    x1min[:, 1] -= np.arange(G) * 2.0 ** -40
    batch = nb.NumericBatch(x1min=x1min, x1max=q0.x1max[None], ymin=ymin[None], ymax=ymax[None],
                            smin=np.stack([pats[p][2] for p in pat]), smax=np.stack([pats[p][3] for p in pat]),
                            out_kind=nb.OUT_SAFETY, out_S=q0.qc_out.S[None])
    B = nb.affine_form_batch(dnet, beta, batch, Q=G)
    assert B["ngroups"] == G and np.array_equal(B["group_of"], np.arange(G))
    lay = ea.layout(net, beta, q0.qc_out)
    _check_sizes(B, lay)
    nvar = lay.nvar
    tiles = math.ceil((G * nvar + 1) / SCAN_TILE)
    assert tiles == 2 if G == SCAN_GROUPS[0] else tiles > SCAN_THREADS
    rest = np.arange(lay.var_out, nvar)
    Rpat = [ea.exact_affine(net, beta, q0, pats[p], vars=rest, lay=lay) for p in range(PATTERNS)]
    cpat = [np.r_[np.full(lay.var_out, 3), R.counts()[rest]] for R in Rpat]
    assert len({tuple(c) for c in cpat}) == PATTERNS
    total = 0
    for g, grp in enumerate(B["groups"]):
        assert np.array_equal(grp["var_ptr"], np.r_[0, np.cumsum(cpat[pat[g]])] + 1), g
        total += len(grp["val"])
        var, ent, val = _csc_triplets(grp)
        assert np.all(np.diff(var * lay.nent + ent) > 0), g
        assert_meets(Rpat[pat[g]], (var, ent, val), f"group {g}", vars=rest)
        q = o.NumericQuery(x1min=x1min[g], x1max=q0.x1max, gin=q0.gin, gbnd=q0.gbnd, gsec=q0.gsec, qc_out=q0.qc_out)
        Rin = ea.exact_affine(net, beta, q, pats[pat[g]], vars=np.arange(lay.var_out), lay=lay)
        assert_meets(Rin, (var, ent, val), f"group {g} γin", vars=np.arange(lay.var_out))
    assert B["nnz_total"] == total
    for i, z0 in enumerate(np.unique(B["z0"], axis=0)):
        _check_z0(net, beta, q0, pats[0], z0, lay.ent_row, lay.ent_col, f"z0 class {i}")
