"""Thin object layer over the C ABI: Context, Net, Batch and the batched one-shot calls.

Array convention: a per-query vector of length n for Q queries is a C-contiguous float64 numpy
array of shape (Q, n) (row q = query q, i.e. the ABI's "n x Q, column q contiguous").  A leading
dimension of 1 means "shared by every query of the batch" (ABI stride 0).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import List, Optional, Sequence

import numpy as np

from . import _lib as L

STAGES = {"bounds": 0, "prepare": 1, "gram": 2, "emit": 3, "d2h": 4, "emit_fill": 5, "emit_window": 6, "emit_edge": 7}


def _dp(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(L.c_dp)


def _f64(a, shape_tail=None) -> np.ndarray:
    a = np.ascontiguousarray(np.asarray(a, dtype=np.float64))
    return a


class Context:
    """Devices + streams (nnsdp_ctx).  devices: list of CUDA ordinals, or an int count."""

    def __init__(self, devices=None):
        if devices is None:
            devices = [0]
        if isinstance(devices, int):
            devices = list(range(devices))
        ids = (L.c_i32 * len(devices))(*devices)
        self._h = L.c_vp()
        L.check(L.lib.nnsdp_ctx_create(len(devices), ids, C.byref(self._h)))
        self.devices = list(devices)

    def close(self):
        if getattr(self, "_h", None):
            L.lib.nnsdp_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Net:
    """A FeedFwdNet uploaded to every device of a Context (nnsdp_net)."""

    def __init__(self, ctx: Context, xdims: Sequence[int], Ms: Sequence[np.ndarray]):
        self.ctx = ctx
        self.xdims = [int(x) for x in xdims]
        self.K = len(self.xdims) - 1
        if len(Ms) != self.K:
            raise ValueError("length(Ms) must be length(xdims) - 1")
        # the ABI wants column-major [W_k b_k]
        self._Ms = []
        for k, M in enumerate(Ms):
            M = np.asarray(M, dtype=np.float64)
            if M.shape != (self.xdims[k + 1], self.xdims[k] + 1):
                raise ValueError(f"Ms[{k}] has shape {M.shape}")
            self._Ms.append(np.asfortranarray(M))
        xd = (L.c_i64 * (self.K + 1))(*self.xdims)
        ptrs = (L.c_dp * self.K)(*[m.ctypes.data_as(L.c_dp) for m in self._Ms])
        self._h = L.c_vp()
        L.check(L.lib.nnsdp_net_upload(ctx._h, self.K, xd, ptrs, C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None):
            L.lib.nnsdp_net_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def sizes(self, beta: int) -> dict:
        s = L.Sizes()
        L.check(L.lib.nnsdp_query_sizes(self._h, beta, C.byref(s)))
        return s.as_dict()

    def cliques(self, beta: int):
        return _cliques_call(lambda *a: L.lib.nnsdp_cliques(self._h, beta, *a), self.sizes(beta))


def read_vnnlib(path: str, n_in: int, n_out: int) -> dict:
    """Safety queries of a vnnlib property file (host only): x1min / x1max (nq x n_in), S (nq x sdim x sdim, each
    symmetric: hplaneS(-A_i, -b_i - 1e-4)) and clause (nq,), the disjunctive clause of the CNF each query belongs
    to -- read_vnnlib_simple + loadVnnlibCnf of the reference.  The arrays feed NumericBatch(out_S=...) as is."""
    nq, nc = L.c_i64(0), L.c_i64(0)
    L.check(L.lib.nnsdp_vnnlib_read(path.encode(), n_in, n_out, 0, C.byref(nq), C.byref(nc), None, None, None, None))
    sdim = n_in + n_out + 1
    lo, hi = np.zeros((nq.value, n_in)), np.zeros((nq.value, n_in))
    S = np.zeros((nq.value, sdim, sdim))
    cl = np.zeros(nq.value, dtype=np.int64)
    if nq.value:
        L.check(L.lib.nnsdp_vnnlib_read(path.encode(), n_in, n_out, nq.value, C.byref(nq), C.byref(nc), _dp(lo), _dp(hi),
                                        _dp(S), cl.ctypes.data_as(L.c_i64p)))
    return {"x1min": lo, "x1max": hi, "S": S, "clause": cl, "nclauses": int(nc.value)}


def read_nnet(path: str):
    """(xdims, Ms) of a .nnet file through the library's reader (host only); Ms[k] = [W_k b_k]."""
    K, need = L.c_i64(0), L.c_i64(0)
    L.check(L.lib.nnsdp_nnet_read(path.encode(), 0, C.byref(K), None, 0, None, C.byref(need)))
    xd = np.zeros(K.value + 1, dtype=np.int64)
    buf = np.zeros(need.value)
    L.check(L.lib.nnsdp_nnet_read(path.encode(), K.value, C.byref(K), xd.ctypes.data_as(L.c_i64p), need.value, _dp(buf),
                                  C.byref(need)))
    Ms, o = [], 0
    for k in range(K.value):
        n = int(xd[k + 1] * (xd[k] + 1))
        Ms.append(buf[o:o + n].reshape(int(xd[k] + 1), int(xd[k + 1])).T.copy())
        o += n
    return xd.tolist(), Ms


def sizes_from_xdims(xdims: Sequence[int], beta: int) -> dict:
    """nnsdp_sizes_from_xdims: host-only (no device needed)."""
    K = len(xdims) - 1
    xd = (L.c_i64 * (K + 1))(*[int(x) for x in xdims])
    s = L.Sizes()
    L.check(L.lib.nnsdp_sizes_from_xdims(K, xd, beta, C.byref(s)))
    return s.as_dict()


def cliques_from_xdims(xdims: Sequence[int], beta: int):
    """nnsdp_cliques_from_xdims: host-only makeCliques; returns [(Ck, [Ck1, Ck2], [Dk1, Dk2])], 1-based int64."""
    K = len(xdims) - 1
    xd = (L.c_i64 * (K + 1))(*[int(x) for x in xdims])
    sz = sizes_from_xdims(xdims, beta)
    return _cliques_call(lambda *a: L.lib.nnsdp_cliques_from_xdims(K, xd, beta, *a), sz)


PROGRAMS = ("ZERO", "SAME", "RC", "CR", "MIXED", "GENERAL", "DIAG", "AFF")


def plan_stats(xdims: Sequence[int], beta: int, dense: bool = False) -> dict:
    """Tiles / output entries per tile program of the emission plan (host only)."""
    K = len(xdims) - 1
    xd = (L.c_i64 * (K + 1))(*[int(x) for x in xdims])
    tiles = np.zeros(8, dtype=np.int64)
    entries = np.zeros(8, dtype=np.int64)
    tr, tc = L.c_i64(0), L.c_i64(0)
    L.check(L.lib.nnsdp_plan_stats(K, xd, beta, int(dense), tiles.ctypes.data_as(L.c_i64p),
                                   entries.ctypes.data_as(L.c_i64p), C.byref(tr), C.byref(tc)))
    return {"tile_rows": int(tr.value), "tile_cols": int(tc.value),
            "tiles": dict(zip(PROGRAMS, tiles.tolist())), "entries": dict(zip(PROGRAMS, entries.tolist()))}


TILE_FIELDS = ("mat", "row0", "nrows", "col0", "ncols", "grow0", "gcol0", "flags", "rblk", "cblk", "prog")


PANEL_FIELDS = ("out_off", "ld", "row0", "nrows", "col0", "ncols", "grow0", "gcol0", "prog", "rblk")


def plan_panel(xdims: Sequence[int], beta: int, dense: int = 0) -> np.ndarray:
    """The panel-ordered work list of the emitter (fill strips + window tiles of the dense formats of wide nets) as an
    (nitems, 10) int64 array (columns: PANEL_FIELDS); empty when the plan keeps the separate kernels.  Host only."""
    K = len(xdims) - 1
    xd = (L.c_i64 * (K + 1))(*[int(x) for x in xdims])
    n = L.c_i64(0)
    L.check(L.lib.nnsdp_plan_panel(K, xd, beta, int(dense), 0, None, C.byref(n)))
    out = np.zeros((int(n.value), 10), dtype=np.int64)
    if n.value:
        L.check(L.lib.nnsdp_plan_panel(K, xd, beta, int(dense), int(n.value), out.ctypes.data_as(L.c_i64p), C.byref(n)))
    return out


def plan_tiles(xdims: Sequence[int], beta: int, dense: bool = False) -> np.ndarray:
    """The emission plan's tile list as an (ntiles, 11) int32 array (columns: TILE_FIELDS); host only."""
    K = len(xdims) - 1
    xd = (L.c_i64 * (K + 1))(*[int(x) for x in xdims])
    n = L.c_i64(0)
    L.check(L.lib.nnsdp_plan_tiles(K, xd, beta, int(dense), 0, None, C.byref(n)))
    out = np.zeros((int(n.value), 11), dtype=np.int32)
    L.check(L.lib.nnsdp_plan_tiles(K, xd, beta, int(dense), int(n.value), out.ctypes.data_as(C.POINTER(L.c_i32)), C.byref(n)))
    return out


def gather_plan(xdims: Sequence[int], beta: int, dense: bool = False) -> dict:
    """Cells (ncells, 8) [mat, row0, nrows, col0, ncols, kind, blk, pure_zero] and thin-entry offsets of the
    host-gather plan (host only)."""
    K = len(xdims) - 1
    xd = (L.c_i64 * (K + 1))(*[int(x) for x in xdims])
    nc, nt, us = L.c_i64(0), L.c_i64(0), L.c_i32(0)
    L.check(L.lib.nnsdp_gather_plan(K, xd, beta, int(dense), 0, None, C.byref(nc), 0, None, C.byref(nt), C.byref(us)))
    cells = np.zeros((int(nc.value), 8), dtype=np.int32)
    thin = np.zeros(int(nt.value), dtype=np.int64)
    L.check(L.lib.nnsdp_gather_plan(K, xd, beta, int(dense), int(nc.value), cells.ctypes.data_as(C.POINTER(L.c_i32)),
                                    C.byref(nc), int(nt.value), thin.ctypes.data_as(L.c_i64p), C.byref(nt), C.byref(us)))
    return {"cells": cells, "thin": thin, "usable": bool(us.value)}


CELL_DTYPE = np.dtype([("kind", "<i4"), ("blk", "<i4"), ("row0", "<i8"), ("col0", "<i8"), ("nrows", "<i8"),
                       ("ncols", "<i8"), ("offset", "<i8"), ("always", "<i4"), ("reserved", "<i4")])


def packed_layout(xdims: Sequence[int], beta: int) -> dict:
    """Cell table of the packed records of (xdims, beta) (nnsdp_packed_layout, host only): a structured array
    `cells` (fields of nnsdp_packed_cell, row0 / col0 / blk 1-based) and the record sizes in doubles."""
    K = len(xdims) - 1
    xd = (L.c_i64 * (K + 1))(*[int(x) for x in xdims])
    n, rec, alw = L.c_i64(0), L.c_i64(0), L.c_i64(0)
    L.check(L.lib.nnsdp_packed_layout(K, xd, beta, 0, None, C.byref(n), C.byref(rec), C.byref(alw)))
    cells = np.zeros(int(n.value), dtype=CELL_DTYPE)
    assert CELL_DTYPE.itemsize == C.sizeof(L.PackedCell)
    L.check(L.lib.nnsdp_packed_layout(K, xd, beta, int(n.value), cells.ctypes.data_as(C.POINTER(L.PackedCell)),
                                      C.byref(n), C.byref(rec), C.byref(alw)))
    return {"cells": cells, "record_doubles": int(rec.value), "always_doubles": int(alw.value)}


def packed_unpack(xdims: Sequence[int], beta: int, record: np.ndarray, present: np.ndarray, dense_Z: bool = False,
                  out: Optional[np.ndarray] = None) -> np.ndarray:
    """One packed record -> the flat dense clique blocks (or the dense Z, column-major) through nnsdp_packed_unpack.
    `out` (float64, C-contiguous, the right size) is reused when given: a fresh 1.33 GB array costs more in page faults
    than the expansion itself."""
    K = len(xdims) - 1
    xd = (L.c_i64 * (K + 1))(*[int(x) for x in xdims])
    sz = sizes_from_xdims(xdims, beta)
    need = sz["Zdim"] ** 2 if dense_Z else sz["sum_ck_sq"]
    if out is None:
        out = np.empty(need)
    if out.dtype != np.float64 or out.size != need or not out.flags["C_CONTIGUOUS"]:
        raise ValueError(f"out must be a C-contiguous float64 array of {need} entries")
    record = np.ascontiguousarray(record, dtype=np.float64)
    present = np.ascontiguousarray(present, dtype=np.uint8)
    L.check(L.lib.nnsdp_packed_unpack(K, xd, beta, _dp(record), present.ctypes.data_as(C.POINTER(C.c_uint8)),
                                      L.FORMAT_DENSE_Z if dense_Z else L.FORMAT_BLOCKS, _dp(out)))
    return out


def assemble_packed(net: "Net", beta: int, batch: "NumericBatch", Q: Optional[int] = None):
    """Packed records of every query: (records (Q, record_doubles), present (Q, ncells) uint8, layout)."""
    Q = Q or _infer_Q(batch)
    lay = packed_layout(net.xdims, beta)
    rec = np.zeros((Q, lay["record_doubles"]))
    present = np.zeros((Q, len(lay["cells"])), dtype=np.uint8)
    qi, keep = batch.pack(Q)
    L.check(L.lib.nnsdp_assemble_packed(net.ctx._h, net._h, beta, Q, C.byref(qi), _dp(rec),
                                        present.ctypes.data_as(C.POINTER(C.c_uint8))))
    return rec, present, lay


def _cliques_call(fn, sz):
    p = sz["ncliques"]
    ck_off = np.zeros(p + 1, dtype=np.int64)
    ck_idx = np.zeros(sz["sum_ck"], dtype=np.int64)
    ck1 = np.zeros(p, dtype=np.int64)
    d_off = np.zeros(2 * p + 1, dtype=np.int64)
    d_idx = np.zeros(sz["sum_dk"], dtype=np.int64)
    ip = lambda a: a.ctypes.data_as(L.c_i64p)
    L.check(fn(ip(ck_off), ip(ck_idx), ip(ck1), ip(d_off), ip(d_idx)))
    out = []
    for k in range(p):
        Ck = ck_idx[ck_off[k]:ck_off[k + 1]].copy()
        parts = [Ck[: ck1[k]].copy()]
        if ck1[k] < len(Ck):
            parts.append(Ck[ck1[k]:].copy())
        ds = [d_idx[d_off[2 * k]:d_off[2 * k + 1]].copy()]
        if d_off[2 * k + 2] > d_off[2 * k + 1]:
            ds.append(d_idx[d_off[2 * k + 1]:d_off[2 * k + 2]].copy())
        out.append((Ck, parts, ds))
    return out


@dataclass
class NumericBatch:
    """Q numeric-gamma queries on one network (the ABI's nnsdp_query_inputs)."""

    x1min: np.ndarray
    x1max: np.ndarray
    gamma_in: Optional[np.ndarray] = None
    gamma_bnd: Optional[np.ndarray] = None
    gamma_sec: Optional[np.ndarray] = None
    out_kind: int = L.OUT_SAFETY
    out_S: Optional[np.ndarray] = None      # (Q|1, sdim, sdim), symmetric
    out_vec: Optional[np.ndarray] = None    # (Q|1, n_out)
    out_invP: Optional[np.ndarray] = None   # (Q|1, n_out, n_out)
    gamma_out: Optional[np.ndarray] = None  # (Q|1,) or (Q|1, 1)
    ymin: Optional[np.ndarray] = None       # caller-supplied bounds (all four or none)
    ymax: Optional[np.ndarray] = None
    smin: Optional[np.ndarray] = None
    smax: Optional[np.ndarray] = None

    def pack(self, Q: int):
        """Returns (QueryInputs, keepalive list)."""
        qi = L.QueryInputs()
        keep = []

        def put(name, arr, colmajor_matrix=False):
            if arr is None:
                return
            a = np.asarray(arr, dtype=np.float64)
            if colmajor_matrix:  # (q, r, c) -> per query column-major
                if a.ndim == 2:
                    a = a[None]
                a = np.ascontiguousarray(np.transpose(a, (0, 2, 1)))
                a = a.reshape(a.shape[0], -1)
            if a.ndim == 1:
                a = a[None, :] if name not in ("gamma_out",) else a[:, None]
            a = np.ascontiguousarray(a)
            if a.shape[0] not in (1, Q):
                raise ValueError(f"{name}: leading dimension {a.shape[0]} is neither 1 nor Q={Q}")
            keep.append(a)
            setattr(qi, name, _dp(a))
            setattr(qi, name + "_stride", 0 if (a.shape[0] == 1 and Q > 1) else a.shape[1])

        put("x1min", self.x1min)
        put("x1max", self.x1max)
        put("ymin", self.ymin)
        put("ymax", self.ymax)
        put("smin", self.smin)
        put("smax", self.smax)
        put("gamma_in", self.gamma_in)
        put("gamma_bnd", self.gamma_bnd)
        put("gamma_sec", self.gamma_sec)
        qi.out_kind = int(self.out_kind)
        put("out_S", self.out_S, colmajor_matrix=True)
        put("out_vec", self.out_vec)
        put("out_invP", self.out_invP, colmajor_matrix=True)
        put("gamma_out", self.gamma_out)
        return qi, keep


def bounds_ibp(net: Net, x1min, x1max):
    """intervalsWorstCase for Q boxes on the device.  Returns dict of (Q, .) arrays."""
    x1min = np.atleast_2d(_f64(x1min))
    x1max = np.atleast_2d(_f64(x1max))
    Q = x1min.shape[0]
    sz = net.sizes(0)
    xmin = np.empty((Q, sz["xtot"]))
    xmax = np.empty((Q, sz["xtot"]))
    acxmin = np.empty((Q, sz["acdim"]))
    acxmax = np.empty((Q, sz["acdim"]))
    L.check(L.lib.nnsdp_bounds_ibp(net.ctx._h, net._h, Q, _dp(x1min), _dp(x1max), _dp(xmin), _dp(xmax),
                                   _dp(acxmin), _dp(acxmax)))
    return {"xmin": xmin, "xmax": xmax, "acxmin": acxmin, "acxmax": acxmax}


def bounds_crown(net: Net, x1min, x1max):
    """CROWN bounds (the reference's default IntervalsAutoLirpa, sliced variant) for Q boxes on the device."""
    x1min = np.atleast_2d(_f64(x1min))
    x1max = np.atleast_2d(_f64(x1max))
    Q = x1min.shape[0]
    sz = net.sizes(0)
    out = {k: np.empty((Q, sz[d])) for k, d in (("xmin", "xtot"), ("xmax", "xtot"), ("acxmin", "acdim"), ("acxmax", "acdim"))}
    L.check(L.lib.nnsdp_bounds_crown(net.ctx._h, net._h, Q, _dp(x1min), _dp(x1max), _dp(out["xmin"]), _dp(out["xmax"]),
                                     _dp(out["acxmin"]), _dp(out["acxmax"])))
    return out


def preact_from_x(net: Net, xmin, xmax):
    xmin = np.atleast_2d(_f64(xmin))
    xmax = np.atleast_2d(_f64(xmax))
    Q = xmin.shape[0]
    sz = net.sizes(0)
    acxmin = np.empty((Q, sz["acdim"]))
    acxmax = np.empty((Q, sz["acdim"]))
    L.check(L.lib.nnsdp_preact_from_x(net.ctx._h, net._h, Q, _dp(xmin), _dp(xmax), _dp(acxmin), _dp(acxmax)))
    return acxmin, acxmax


def sector_minmax(ctx: Context, acxmin, acxmax):
    lo = _f64(acxmin)
    hi = _f64(acxmax)
    smin = np.empty_like(lo)
    smax = np.empty_like(hi)
    L.check(L.lib.nnsdp_sector_minmax(ctx._h, lo.size, _dp(lo), _dp(hi), _dp(smin), _dp(smax)))
    return smin, smax


def assemble_blocks(net: Net, beta: int, batch: NumericBatch, Q: Optional[int] = None, out: Optional[np.ndarray] = None):
    """Dense clique blocks of every query: returns (Q, sum_ck_sq) float64."""
    Q = Q or _infer_Q(batch)
    sz = net.sizes(beta)
    if out is None:
        out = np.empty((Q, sz["sum_ck_sq"]))
    qi, keep = batch.pack(Q)
    L.check(L.lib.nnsdp_assemble_blocks(net.ctx._h, net._h, beta, Q, C.byref(qi), _dp(out)))
    return out


def assemble_dense(net: Net, beta: int, batch: NumericBatch, Q: Optional[int] = None):
    """The whole Z of every query: returns (Q, Zdim, Zdim) with [q, r, c] = Z_q[r, c]."""
    Q = Q or _infer_Q(batch)
    sz = net.sizes(beta)
    out = np.empty((Q, sz["Zdim"], sz["Zdim"]))
    qi, keep = batch.pack(Q)
    L.check(L.lib.nnsdp_assemble_dense(net.ctx._h, net._h, beta, Q, C.byref(qi), _dp(out)))
    return np.transpose(out, (0, 2, 1))  # per-query column-major -> [q, r, c]


def affine_form(net: Net, beta: int, batch: NumericBatch, max_nnz: int = 0) -> dict:
    """Z(gamma) = Z0 + sum_v gamma_v Z_v of ONE query over the upper triangle of the clique cover
    (nnsdp_affine_create / nnsdp_affine_get).  Multipliers in `batch` are ignored.  Returns the sizes,
    the 1-based entry positions, z0 and the COO triplets (1-based entry / variable indices)."""
    qi, keep = batch.pack(1)
    h, sz = L.c_vp(), L.AffineSizes()
    L.check(L.lib.nnsdp_affine_create(net.ctx._h, net._h, beta, C.byref(qi), max_nnz, C.byref(h), C.byref(sz)))
    try:
        d = sz.as_dict()
        out = {"ent_row": np.zeros(d["nent"], dtype=np.int64), "ent_col": np.zeros(d["nent"], dtype=np.int64),
               "z0": np.zeros(d["nent"]), "coo_ent": np.zeros(d["nnz"], dtype=np.int64),
               "coo_var": np.zeros(d["nnz"], dtype=np.int64), "coo_val": np.zeros(d["nnz"])}
        ip = lambda a: a.ctypes.data_as(L.c_i64p)
        L.check(L.lib.nnsdp_affine_get(h, ip(out["ent_row"]), ip(out["ent_col"]), _dp(out["z0"]), ip(out["coo_ent"]),
                                       ip(out["coo_var"]), _dp(out["coo_val"])))
        out.update(d)
        return out
    finally:
        L.lib.nnsdp_affine_destroy(h)


def split_blocks(flat: np.ndarray, cliques) -> List[np.ndarray]:
    """One query's flat output -> list of |Ck| x |Ck| matrices ([r, c] indexing)."""
    out, o = [], 0
    for Ck, _, _ in cliques:
        n = len(Ck)
        out.append(flat[o:o + n * n].reshape(n, n).T)
        o += n * n
    return out


def _infer_Q(batch: NumericBatch) -> int:
    Q = 1
    for name in ("x1min", "x1max", "gamma_in", "gamma_bnd", "gamma_sec", "out_vec", "gamma_out", "ymin", "smin"):
        a = getattr(batch, name)
        if a is not None:
            a = np.asarray(a)
            if a.ndim >= 2:
                Q = max(Q, a.shape[0])
    for name in ("out_S", "out_invP"):
        a = getattr(batch, name)
        if a is not None and np.asarray(a).ndim == 3:
            Q = max(Q, np.asarray(a).shape[0])
    return Q


class Batch:
    """Device-resident batch (nnsdp_batch): what bench.py times with inputs already in HBM."""

    def __init__(self, net: Net, beta: int, Qcap: int, ring: int, dense: bool = False, dev_index: int = 0,
                 packed: bool = False):
        self.net, self.beta, self.Qcap, self.ring, self.dense, self.packed = net, beta, Qcap, ring, dense, packed
        fmt = L.FORMAT_PACKED if packed else (L.FORMAT_DENSE_Z if dense else L.FORMAT_BLOCKS)
        self._h = L.c_vp()
        L.check(L.lib.nnsdp_batch_create(net.ctx._h, dev_index, net._h, beta, Qcap, ring, fmt, C.byref(self._h)))
        self.sz = net.sizes(beta)
        self.per_query = self.sz["Zdim"] ** 2 if dense else self.sz["sum_ck_sq"]
        if packed:
            st = self.packed_stats()
            self.per_query, self.ncells = st["record_doubles"], st["ncells"]
        self.Q = 0

    def close(self):
        if getattr(self, "_h", None):
            L.lib.nnsdp_batch_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_inputs(self, batch: NumericBatch, Q: Optional[int] = None):
        Q = Q or _infer_Q(batch)
        qi, keep = batch.pack(Q)
        L.check(L.lib.nnsdp_batch_set_inputs(self._h, Q, C.byref(qi)))
        self.Q = Q

    def set_inputs_raw(self, qi: "L.QueryInputs", Q: int):
        L.check(L.lib.nnsdp_batch_set_inputs(self._h, Q, C.byref(qi)))
        self.Q = Q

    def bounds(self):
        L.check(L.lib.nnsdp_batch_bounds(self._h))

    def bounds_crown(self):
        L.check(L.lib.nnsdp_batch_bounds_crown(self._h))

    def set_bounds_method(self, method: str):
        L.check(L.lib.nnsdp_batch_set_bounds_method(self._h, {"ibp": 0, "crown": 1}[method]))

    def prepare(self):
        L.check(L.lib.nnsdp_batch_prepare(self._h))

    def emit(self, q0: int, nq: int):
        L.check(L.lib.nnsdp_batch_emit(self._h, q0, nq))

    def run(self, host_out: Optional[np.ndarray] = None, host_ptr: Optional[int] = None, flags: int = 0):
        if host_ptr is not None:
            p = C.cast(C.c_void_p(host_ptr), L.c_dp)
        else:
            p = _dp(host_out)
        L.check(L.lib.nnsdp_batch_run_ex(self._h, p, flags))

    def run_packed(self, host_records: Optional[np.ndarray] = None, present: Optional[np.ndarray] = None,
                   host_ptr: Optional[int] = None, flags: int = 0):
        """nnsdp_batch_run_packed: records into host memory (Q x record_doubles), present flags (Q x ncells uint8)."""
        p = C.cast(C.c_void_p(host_ptr), L.c_dp) if host_ptr is not None else _dp(host_records)
        pp = None if present is None else present.ctypes.data_as(C.POINTER(C.c_uint8))
        L.check(L.lib.nnsdp_batch_run_packed(self._h, p, pp, flags))

    def packed_stats(self) -> dict:
        v = [L.c_i64(0) for _ in range(5)]
        L.check(L.lib.nnsdp_batch_packed_stats(self._h, *[C.byref(x) for x in v]))
        return dict(zip(("record_doubles", "ncells", "emitted_bytes", "d2h_bytes", "present_optional_cells"),
                        [int(x.value) for x in v]))

    def lambda_max(self, max_iters: int = 200, tol: float = 1e-10, full: bool = False):
        """lambda_max(Z(gamma)) of every query (matrix-free Lanczos on the device); needs bounds + prepare.
        full=True returns (lam, iters, resid, converged) and does not raise when a query stops at max_iters (its
        value is then only a lower bound); otherwise non-convergence raises NnsdpError(ERR_NOCONV)."""
        lam = np.zeros(self.Q)
        its = np.zeros(self.Q, dtype=np.int32)
        resid = np.zeros(self.Q)
        conv = np.zeros(self.Q, dtype=np.int32)
        st = L.lib.nnsdp_batch_lambda_max_ex(self._h, max_iters, tol, _dp(lam), its.ctypes.data_as(C.POINTER(L.c_i32)),
                                             _dp(resid), conv.ctypes.data_as(C.POINTER(L.c_i32)))
        if full:
            if st not in (L.OK, L.ERR_NOCONV):
                L.check(st)
            return lam, its, resid, conv
        L.check(st)
        return lam, its

    def gather_stats(self) -> dict:
        a, t, z, u = L.c_i64(0), L.c_i64(0), L.c_i64(0), L.c_i32(0)
        L.check(L.lib.nnsdp_batch_gather_stats(self._h, C.byref(a), C.byref(t), C.byref(z), C.byref(u)))
        return {"dma_bytes": int(a.value), "thin_bytes": int(t.value), "zeroed_bytes": int(z.value),
                "sparse": bool(u.value)}

    def sync(self):
        L.check(L.lib.nnsdp_batch_sync(self._h))

    def get_bounds(self):
        Q, sz = self.Q, self.sz
        o = {k: np.empty((Q, sz[d])) for k, d in (("xmin", "xtot"), ("xmax", "xtot"), ("acxmin", "acdim"),
                                                  ("acxmax", "acdim"), ("smin", "acdim"), ("smax", "acdim"))}
        L.check(L.lib.nnsdp_batch_get_bounds(self._h, *[_dp(o[k]) for k in ("xmin", "xmax", "acxmin", "acxmax", "smin", "smax")]))
        return o

    def get_slot(self, slot: int) -> np.ndarray:
        out = np.empty(self.per_query)
        L.check(L.lib.nnsdp_batch_get_slot(self._h, slot, _dp(out)))
        return out

    def get_affine(self) -> np.ndarray:
        out = np.empty((self.Q, self.sz["Zdim"]))
        L.check(L.lib.nnsdp_batch_get_affine(self._h, _dp(out)))
        return out

    def ring_ptr(self):
        p, n = L.c_u64(0), L.c_i64(0)
        L.check(L.lib.nnsdp_batch_ring_ptr(self._h, C.byref(p), C.byref(n)))
        return int(p.value), int(n.value)

    def emitted_bytes(self) -> int:
        """nnsdp_batch_emit_stats: bytes the emitter stored in the last run (+ emit calls since), every format."""
        v = L.c_i64(0)
        L.check(L.lib.nnsdp_batch_emit_stats(self._h, C.byref(v)))
        return int(v.value)

    def ring_reset(self):
        """nnsdp_batch_ring_reset: zero every ring slot again on its next use (after writing into the ring)."""
        L.check(L.lib.nnsdp_batch_ring_reset(self._h))

    def event_record(self, which: int):
        L.check(L.lib.nnsdp_batch_event_record(self._h, which))

    def elapsed_ms(self) -> float:
        ms = C.c_float(0)
        L.check(L.lib.nnsdp_batch_elapsed_ms(self._h, C.byref(ms)))
        return float(ms.value)

    def stage_ms(self, stage: str):
        ms, n = C.c_float(0), L.c_i64(0)
        L.check(L.lib.nnsdp_batch_stage_ms(self._h, STAGES[stage], C.byref(ms), C.byref(n)))
        return float(ms.value), int(n.value)

    def stage_reset(self):
        L.check(L.lib.nnsdp_batch_stage_reset(self._h))

    def gram_stats(self):
        a, b = L.c_i64(0), L.c_i64(0)
        L.check(L.lib.nnsdp_batch_gram_stats(self._h, C.byref(a), C.byref(b)))
        return int(a.value), int(b.value)


class PinnedBuffer:
    """Page-locked host memory from nnsdp_host_alloc, viewed as a float64 numpy array."""

    def __init__(self, n_doubles: int):
        self._p = L.c_vp()
        L.check(L.lib.nnsdp_host_alloc(int(n_doubles) * 8, C.byref(self._p)))
        self.array = np.ctypeslib.as_array(C.cast(self._p, L.c_dp), shape=(int(n_doubles),))

    def close(self):
        if getattr(self, "_p", None):
            self.array = None
            L.lib.nnsdp_host_free(self._p)
            self._p = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
