"""Batched affine-coefficient hand-off (nnsdp_affine_create_batch): one call for the queries of a reach polytope or a
vnnlib property.  Queries with equal bounds share one canonical CSC coefficient matrix; z0 is per query.  The
reference is nnsdp_affine_create on each query alone, its COO canonicalised here: stable sort by (variable, entry),
duplicates summed in order."""
import ctypes as C

import numpy as np
import pytest

import nnsdp_oracle as o
from helpers import rand_net, rand_query, relerr, to_numeric_batch

TOL = 1e-12


def canonical(A):
    """COO of nnsdp_affine_get -> (var_ptr, ent_idx, val), 1-based, as the batched call returns them."""
    var, ent, val = A["coo_var"] - 1, A["coo_ent"] - 1, A["coo_val"]
    order = np.lexsort((ent, var))  # stable: duplicates keep the order the single call lists them in
    var, ent, val = var[order], ent[order], val[order]
    key = var * A["nent"] + ent
    start = np.flatnonzero(np.r_[True, key[1:] != key[:-1]])
    sums = np.add.reduceat(val, start) if len(key) else val  # at most two terms per entry: order-free
    var_ptr = np.searchsorted(var[start], np.arange(A["nvar"] + 1)) + 1
    return var_ptr, ent[start] + 1, sums


def same_csc(grp, ref):
    var_ptr, ent_idx, val = ref
    return (np.array_equal(grp["var_ptr"], var_ptr) and np.array_equal(grp["ent_idx"], ent_idx)
            and np.array_equal(grp["val"], val))


def strictly_ascending(grp):
    vp = grp["var_ptr"] - 1
    return all(np.all(np.diff(grp["ent_idx"][vp[v]:vp[v + 1]]) > 0) for v in range(len(vp) - 1))


def csc_dense(grp, nent, nvar):
    A = np.zeros((nent, nvar))
    for v in range(nvar):
        s, e = grp["var_ptr"][v] - 1, grp["var_ptr"][v + 1] - 1
        A[grp["ent_idx"][s:e] - 1, v] = grp["val"][s:e]
    return A


def single(nb, dnet, beta, batch, q):
    """query q of a NumericBatch alone, through nnsdp_affine_create"""
    one = {}
    for f in ("x1min", "x1max", "out_S", "out_vec", "out_invP", "gamma_out", "ymin", "ymax", "smin", "smax"):
        a = getattr(batch, f)
        if a is not None:
            a = np.asarray(a)
            one[f] = a[q:q + 1] if a.ndim >= 2 and a.shape[0] > 1 else a
    return nb.affine_form(dnet, beta, nb.NumericBatch(out_kind=batch.out_kind, **one))


def box_bounds(nb, dnet, boxes):
    """caller-supplied bounds (post-activation intervals and sector slopes) of each box, computed once per box"""
    lo = np.stack([b[0] for b in boxes])
    hi = np.stack([b[1] for b in boxes])
    r = nb.bounds_ibp(dnet, lo, hi)
    n1, ac = lo.shape[1], r["acxmin"].shape[1]
    smin, smax = nb.sector_minmax(dnet.ctx, r["acxmin"], r["acxmax"])
    return r["xmin"][:, n1:n1 + ac], r["xmax"][:, n1:n1 + ac], smin, smax


NETS = [([2, 3, 2], 0), ([2, 3, 3, 2], 1), ([3, 3, 3, 3, 4, 3, 3], 2), ([2, 4, 7, 3, 5, 2], 5), ([2, 6, 5, 7, 4, 2], 2)]
BOX_OF = [0, 1, 0, 2, 1, 0, 2]  # Q = 7 over 3 boxes


def seven_queries(nb, net, dnet, beta, kind, supplied, seed=3):
    rng = np.random.default_rng(seed)
    n1 = net.xdims[0]
    centres = [rng.uniform(0.5, 1.5, n1) for _ in range(3)]
    boxes = [(c - r, c + r) for c, r in zip(centres, (0.3, 0.0, 0.1))]
    qs = []
    for b in BOX_OF:
        q = rand_query(net, beta, rng, kind=kind, radius=0.0)  # its own S / normal / ellipsoid
        q.x1min, q.x1max = boxes[b][0].copy(), boxes[b][1].copy()
        qs.append(q)
    batch = to_numeric_batch(nb, net, qs)
    if supplied:
        ymin, ymax, smin, smax = box_bounds(nb, dnet, boxes)
        idx = np.array(BOX_OF)
        batch.ymin, batch.ymax, batch.smin, batch.smax = ymin[idx], ymax[idx], smin[idx], smax[idx]
    return qs, batch


@pytest.mark.gpu
@pytest.mark.parametrize("supplied", [False, True], ids=["ibp", "caller_bounds"])
@pytest.mark.parametrize("kind", ["safety", "hplane", "ellipsoid"])
@pytest.mark.parametrize("xdims,beta", NETS)
def test_batch_equals_single_calls(ctx, xdims, beta, kind, supplied):
    import nnsdp_b200 as nb

    net = rand_net(xdims, seed=5, sigma=0.5)
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    qs, batch = seven_queries(nb, net, dnet, beta, kind, supplied)
    B = nb.affine_form_batch(dnet, beta, batch)
    assert B["Q"] == 7 and B["ngroups"] == 3
    assert np.array_equal(B["group_of"], BOX_OF)
    assert [g["first"] for g in B["groups"]] == [0, 1, 3]
    assert B["nnz_total"] == sum(len(g["val"]) for g in B["groups"])
    assert B["nnz_max"] == max(len(g["val"]) for g in B["groups"])
    for q in range(7):
        A = single(nb, dnet, beta, batch, q)
        assert np.array_equal(B["ent_row"], A["ent_row"]) and np.array_equal(B["ent_col"], A["ent_col"])
        for k in ("nvar", "nent", "var_in", "var_out", "var_bnd", "var_sec"):
            assert B[k] == A[k], k
        assert np.array_equal(B["z0"][q], A["z0"]), q
        grp = B["groups"][B["group_of"][q]]
        assert same_csc(grp, canonical(A)), q
        assert grp["var_ptr"][0] == 1 and grp["var_ptr"][-1] == len(grp["val"]) + 1
        assert strictly_ascending(grp)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["safety", "hplane", "ellipsoid"])
@pytest.mark.parametrize("xdims,beta", [([2, 4, 7, 3, 5, 2], 5), ([2, 6, 5, 7, 4, 2], 2)])
def test_batch_reproduces_numeric_assembly(ctx, xdims, beta, kind):
    """z0_q + A_g gamma_q == Z_q(gamma_q) of the numeric path on the cover entries, at random multipliers"""
    import nnsdp_b200 as nb

    net = rand_net(xdims, seed=7, sigma=0.5)
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    qs, batch = seven_queries(nb, net, dnet, beta, kind, False, seed=11)
    rng = np.random.default_rng(2)
    for q in qs:
        q.gsec = rng.random(len(q.gsec))
    num = to_numeric_batch(nb, net, qs)
    B = nb.affine_form_batch(dnet, beta, batch)
    Z = nb.assemble_dense(dnet, beta, num)
    er, ec = B["ent_row"] - 1, B["ent_col"] - 1
    for i, q in enumerate(qs):
        g = np.concatenate([q.gin, q.gout if kind != "safety" else [], q.gbnd, q.gsec])
        A = csc_dense(B["groups"][B["group_of"][i]], B["nent"], B["nvar"])
        assert relerr(B["z0"][i] + A @ g, Z[i][er, ec]) <= TOL


@pytest.mark.gpu
def test_batch_against_oracle(ctx):
    """two groups, every variable's matrix and Z0 against oracle.affine_structure"""
    import nnsdp_b200 as nb

    xdims, beta, kind = [2, 4, 7, 3, 5, 2], 3, "hplane"
    net = rand_net(xdims, seed=5, sigma=0.5)
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    rng = np.random.default_rng(8)
    qs = [rand_query(net, beta, rng, kind=kind, radius=r, centre=c)
          for r, c in ((0.3, [1.0, 0.8]), (0.3, [1.0, 0.8]), (0.05, [0.7, 1.2]))]
    B = nb.affine_form_batch(dnet, beta, to_numeric_batch(nb, net, qs))
    assert B["ngroups"] == 2 and np.array_equal(B["group_of"], [0, 0, 1])
    cliques = o.make_cliques(net, beta)
    er, ec = o.cover_upper_entries(net, cliques)
    assert np.array_equal(B["ent_row"], er) and np.array_equal(B["ent_col"], ec)
    for i, q in enumerate(qs):
        Z0, Zv = o.affine_structure(net, beta, q.x1min, q.x1max, q.qc_out)
        assert B["nvar"] == len(Zv)
        scale = max(np.abs(Z0).max(), max(np.abs(z).max() for z in Zv), 1.0)
        assert np.abs(B["z0"][i] - Z0[er - 1, ec - 1]).max() <= TOL * scale
        A = csc_dense(B["groups"][B["group_of"][i]], B["nent"], B["nvar"])
        for v in range(B["nvar"]):
            assert np.abs(A[:, v] - Zv[v][er - 1, ec - 1]).max() <= TOL * scale, v


@pytest.mark.gpu
def test_reach_polytope_is_one_group(ctx):
    """findReach2Dpoly (src/NnSdp.jl:73-95): box and bounds shared (stride 0), 64 hyperplane normals"""
    import nnsdp_b200 as nb

    xdims, beta = [2, 10, 10, 10, 2], 2
    net = rand_net(xdims, seed=4)
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    lo, hi = np.full(2, 0.5), np.full(2, 1.5)
    ymin, ymax, smin, smax = box_bounds(nb, dnet, [(lo, hi)])
    th = 2 * np.pi * np.arange(64) / 64
    normals = np.stack([np.cos(th), np.sin(th)], axis=1)
    batch = nb.NumericBatch(x1min=lo, x1max=hi, ymin=ymin[0], ymax=ymax[0], smin=smin[0], smax=smax[0],
                            out_kind=nb.OUT_HPLANE, out_vec=normals)
    B = nb.affine_form_batch(dnet, beta, batch, Q=64)
    assert B["ngroups"] == 1 and not B["group_of"].any()
    for q in (0, 17, 63):
        one = nb.NumericBatch(x1min=lo, x1max=hi, ymin=ymin, ymax=ymax, smin=smin, smax=smax, out_kind=nb.OUT_HPLANE,
                              out_vec=normals[q:q + 1])
        A = nb.affine_form(dnet, beta, one)
        ref = canonical(A)
        assert B["nnz_total"] == len(ref[2]) and same_csc(B["groups"][0], ref)
        assert np.array_equal(B["z0"][q], A["z0"])


@pytest.mark.gpu
def test_vnnlib_property_groups(ctx, tmp_path):
    """the ACAS-shaped property of test_vnnlib_property_as_one_batch: 10 queries over 2 boxes"""
    import nnsdp_b200 as nb

    xdims, beta = [5] + [50] * 6 + [5], 2
    net = rand_net(xdims, seed=12)
    text = "\n".join(f"(declare-const X_{i} Real)" for i in range(5)) + """
(assert (<= X_0 0.68))
(assert (>= X_0 0.6))
(assert (<= X_1 0.05))
(assert (>= X_1 -0.05))
(assert (<= X_2 0.05))
(assert (>= X_2 -0.05))
(assert (<= X_4 -0.45))
(assert (>= X_4 -0.5))
(assert (or (and (<= X_3 0.5)(>= X_3 0.45)) (and (<= X_3 0.3)(>= X_3 0.25))))
(assert (or (and (<= Y_0 Y_1)(<= Y_0 Y_2)(<= Y_0 Y_3)(<= Y_0 Y_4)) (and (>= Y_2 0.75))))
"""
    path = str(tmp_path / "prop.vnnlib")
    open(path, "w").write(text)
    r = nb.read_vnnlib(path, 5, 5)
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    batch = nb.NumericBatch(x1min=r["x1min"], x1max=r["x1max"], out_kind=nb.OUT_SAFETY, out_S=r["S"])
    B = nb.affine_form_batch(dnet, beta, batch)
    assert B["Q"] == 10 and B["ngroups"] == 2
    for q in range(10):
        g = B["group_of"][q]
        assert np.array_equal(r["x1min"][q], r["x1min"][B["groups"][g]["first"]])
        A = single(nb, dnet, beta, batch, q)
        assert np.array_equal(B["z0"][q], A["z0"])
        assert same_csc(B["groups"][g], canonical(A))


@pytest.mark.gpu
@pytest.mark.parametrize("supplied", [False, True], ids=["ibp", "caller_bounds"])
def test_wide_layers_many_queries(ctx, supplied):
    """260-wide layers, Q = 128: the batch's interval bounds run on the tensor cores, the single call's do not"""
    import nnsdp_b200 as nb

    xdims, beta, Q = [2, 260, 260, 2], 1, 128
    net = rand_net(xdims, seed=21)
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    rng = np.random.default_rng(6)
    centres = [rng.uniform(0.5, 1.5, 2) for _ in range(4)]
    boxes = [(c - r, c + r) for c, r in zip(centres, (0.3, 0.6, 1.0, 0.4))]
    box_of = np.arange(Q) % 4
    kw = dict(x1min=np.stack([boxes[b][0] for b in box_of]), x1max=np.stack([boxes[b][1] for b in box_of]),
              out_kind=nb.OUT_HPLANE, out_vec=rng.standard_normal((Q, 2)))
    if supplied:
        ymin, ymax, smin, smax = box_bounds(nb, dnet, boxes)
        kw.update(ymin=ymin[box_of], ymax=ymax[box_of], smin=smin[box_of], smax=smax[box_of])
    batch = nb.NumericBatch(**kw)
    B = nb.affine_form_batch(dnet, beta, batch)
    assert B["ngroups"] == 4 and np.array_equal(B["group_of"], box_of)
    if not supplied:  # the premise of grouping by input bytes: equal boxes get bit-identical bounds at this Q
        b = nb.Batch(dnet, beta, Qcap=Q, ring=1)
        b.set_inputs(nb.NumericBatch(x1min=kw["x1min"], x1max=kw["x1max"], gamma_in=np.zeros(2),
                                     gamma_bnd=np.zeros(520), gamma_sec=np.zeros(nb.sizes_from_xdims(xdims, beta)["secdim"]),
                                     out_kind=nb.OUT_HPLANE, out_vec=kw["out_vec"], gamma_out=np.zeros(1)), Q)
        b.bounds()
        bd = b.get_bounds()
        b.close()
        for q in range(Q):
            for k in bd:
                assert np.array_equal(bd[k][q], bd[k][box_of[q]]), (k, q)
    for g, grp in enumerate(B["groups"]):
        A = single(nb, dnet, beta, batch, grp["first"])
        ref = canonical(A)
        if supplied:
            assert same_csc(grp, ref)
        else:
            assert np.array_equal(grp["var_ptr"], ref[0]) and np.array_equal(grp["ent_idx"], ref[1])
            assert relerr(grp["val"], ref[2]) <= TOL
        assert strictly_ascending(grp)
        for q in np.flatnonzero(box_of == g)[:3]:
            Aq = single(nb, dnet, beta, batch, q)
            assert relerr(B["z0"][q], Aq["z0"]) <= TOL


@pytest.mark.gpu
def test_errors_and_lifetime(ctx):
    import nnsdp_b200 as nb
    from nnsdp_b200 import _lib as L

    xdims, beta = [2, 6, 5, 7, 4, 2], 2
    net = rand_net(xdims, seed=5, sigma=0.5)
    dnet = nb.Net(ctx, net.xdims, net.Ms)
    qs, batch = seven_queries(nb, net, dnet, beta, "hplane", False)
    qi, keep = batch.pack(7)
    h, sz = L.c_vp(), L.AffineBatchSizes()
    assert L.lib.nnsdp_affine_create_batch(ctx._h, dnet._h, beta, 0, C.byref(qi), 0, C.byref(h), C.byref(sz)) == -1
    B = nb.affine_form_batch(dnet, beta, batch)
    assert L.lib.nnsdp_affine_create_batch(ctx._h, dnet._h, beta, 7, C.byref(qi), B["nnz_max"] - 1, C.byref(h),
                                           C.byref(sz)) == -3
    assert "group" in L.lib.nnsdp_last_error().decode()
    # two live handles, destroyed in reverse order; numeric work on the same net between create and get
    h1, h2, s1, s2 = L.c_vp(), L.c_vp(), L.AffineBatchSizes(), L.AffineBatchSizes()
    L.check(L.lib.nnsdp_affine_create_batch(ctx._h, dnet._h, beta, 7, C.byref(qi), 0, C.byref(h1), C.byref(s1)))
    L.check(L.lib.nnsdp_affine_create_batch(ctx._h, dnet._h, beta, 7, C.byref(qi), 0, C.byref(h2), C.byref(s2)))
    rng = np.random.default_rng(0)
    for q in qs:
        q.gsec = rng.random(len(q.gsec))
    nb.assemble_blocks(dnet, beta, to_numeric_batch(nb, net, qs))
    ip = lambda a: a.ctypes.data_as(L.c_i64p)
    assert L.lib.nnsdp_affine_batch_get_group(h1, s1.ngroups, None, None, None) == -1
    assert L.lib.nnsdp_affine_batch_get_group(h1, -1, None, None, None) == -1
    assert L.lib.nnsdp_affine_batch_get_group(None, 0, None, None, None) == -1
    assert L.lib.nnsdp_affine_batch_get(None, None, None, None) == -1
    for h in (h2, h1):
        z0 = np.zeros((7, s1.nent))
        L.check(L.lib.nnsdp_affine_batch_get(h, None, None, z0.ctypes.data_as(L.c_dp)))
        assert np.array_equal(z0, B["z0"])
        for g, grp in enumerate(B["groups"]):
            vp, ei, v = np.zeros(s1.nvar + 1, dtype=np.int64), np.zeros(len(grp["val"]), dtype=np.int64), np.zeros(len(grp["val"]))
            L.check(L.lib.nnsdp_affine_batch_get_group(h, g, ip(vp), ip(ei), v.ctypes.data_as(L.c_dp)))
            assert np.array_equal(vp, grp["var_ptr"]) and np.array_equal(ei, grp["ent_idx"]) and np.array_equal(v, grp["val"])
        L.check(L.lib.nnsdp_affine_batch_destroy(h))
    assert L.lib.nnsdp_affine_batch_destroy(None) == 0


def test_affine_batch_sizes_layout():
    from nnsdp_b200 import _lib as L

    assert C.sizeof(L.AffineBatchSizes) == 80
    assert [n for n, _ in L.AffineBatchSizes._fields_] == ["Q", "ngroups", "nvar", "nent", "var_in", "var_out", "var_bnd",
                                                           "var_sec", "nnz_total", "nnz_max"]
    assert all(t is L.c_i64 for _, t in L.AffineBatchSizes._fields_)
