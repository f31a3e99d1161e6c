"""ctypes binding of libnnsdp_b200.so (the C ABI in include/nnsdp_b200.h).

The library is the product; this module only loads it and declares the prototypes.  There is
no Python/CPU fallback: if the shared library is missing, importing this module raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("NNSDP_B200_LIB", os.path.join(_HERE, "..", "lib", "libnnsdp_b200.so"))

OK, ERR_ARG, ERR_CUDA, ERR_NOMEM, ERR_STATE, ERR_ASSERT, ERR_NOCONV = 0, -1, -2, -3, -4, -5, -6
OUT_SAFETY, OUT_HPLANE, OUT_CIRCLE, OUT_ELLIPSOID = 0, 1, 2, 3
RUN_HOST_PREZEROED, RUN_DENSE_COPY = 1, 2
FORMAT_BLOCKS, FORMAT_DENSE_Z, FORMAT_PACKED = 0, 1, 2
CELL_WINDOW, CELL_DIAG, CELL_BAND, CELL_RECT = 1, 2, 3, 4

c_i32, c_i64, c_u64 = C.c_int32, C.c_int64, C.c_uint64
c_dp = C.POINTER(C.c_double)
c_i64p = C.POINTER(C.c_int64)
c_vp = C.c_void_p


class Sizes(C.Structure):
    _fields_ = [(n, c_i64) for n in (
        "K", "Zdim", "acdim", "xtot", "lamdim", "secdim", "n_in", "n_out", "sdim", "ncliques",
        "sum_ck", "sum_ck_sq", "sum_dk", "max_ck")]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


class AffineSizes(C.Structure):
    _fields_ = [(n, c_i64) for n in ("nvar", "nent", "nnz", "var_in", "var_out", "var_bnd", "var_sec")]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


class AffineBatchSizes(C.Structure):
    _fields_ = [(n, c_i64) for n in ("Q", "ngroups", "nvar", "nent", "var_in", "var_out", "var_bnd", "var_sec",
                                     "nnz_total", "nnz_max")]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


class PackedCell(C.Structure):
    _fields_ = [("kind", C.c_int32), ("blk", C.c_int32), ("row0", C.c_int64), ("col0", C.c_int64), ("nrows", C.c_int64),
                ("ncols", C.c_int64), ("offset", C.c_int64), ("always", C.c_int32), ("reserved", C.c_int32)]


class QueryInputs(C.Structure):
    _fields_ = [
        ("x1min", c_dp), ("x1min_stride", c_i64),
        ("x1max", c_dp), ("x1max_stride", c_i64),
        ("ymin", c_dp), ("ymin_stride", c_i64),
        ("ymax", c_dp), ("ymax_stride", c_i64),
        ("smin", c_dp), ("smin_stride", c_i64),
        ("smax", c_dp), ("smax_stride", c_i64),
        ("gamma_in", c_dp), ("gamma_in_stride", c_i64),
        ("gamma_bnd", c_dp), ("gamma_bnd_stride", c_i64),
        ("gamma_sec", c_dp), ("gamma_sec_stride", c_i64),
        ("out_kind", c_i32), ("reserved", c_i32),
        ("out_S", c_dp), ("out_S_stride", c_i64),
        ("out_vec", c_dp), ("out_vec_stride", c_i64),
        ("out_invP", c_dp), ("out_invP_stride", c_i64),
        ("gamma_out", c_dp), ("gamma_out_stride", c_i64),
    ]


# name -> (restype, argtypes); every symbol include/nnsdp_b200.h declares
PROTOTYPES = {
    "nnsdp_last_error": (C.c_char_p, []),
    "nnsdp_version": (c_i32, []),
    "nnsdp_device_count": (c_i32, [C.POINTER(c_i32)]),
    "nnsdp_ctx_create": (c_i32, [c_i32, C.POINTER(c_i32), C.POINTER(c_vp)]),
    "nnsdp_ctx_destroy": (c_i32, [c_vp]),
    "nnsdp_ctx_num_devices": (c_i32, [c_vp, C.POINTER(c_i32)]),
    "nnsdp_host_alloc": (c_i32, [c_u64, C.POINTER(c_vp)]),
    "nnsdp_host_free": (c_i32, [c_vp]),
    "nnsdp_net_upload": (c_i32, [c_vp, c_i64, c_i64p, C.POINTER(c_dp), C.POINTER(c_vp)]),
    "nnsdp_net_destroy": (c_i32, [c_vp]),
    "nnsdp_nnet_read": (c_i32, [C.c_char_p, c_i64, c_i64p, c_i64p, c_i64, c_dp, c_i64p]),
    "nnsdp_vnnlib_read": (c_i32, [C.c_char_p, c_i64, c_i64, c_i64, c_i64p, c_i64p, c_dp, c_dp, c_dp, c_i64p]),
    "nnsdp_query_sizes": (c_i32, [c_vp, c_i64, C.POINTER(Sizes)]),
    "nnsdp_cliques": (c_i32, [c_vp, c_i64, c_i64p, c_i64p, c_i64p, c_i64p, c_i64p]),
    "nnsdp_sizes_from_xdims": (c_i32, [c_i64, c_i64p, c_i64, C.POINTER(Sizes)]),
    "nnsdp_cliques_from_xdims": (c_i32, [c_i64, c_i64p, c_i64, c_i64p, c_i64p, c_i64p, c_i64p, c_i64p]),
    "nnsdp_plan_stats": (c_i32, [c_i64, c_i64p, c_i64, c_i32, c_i64p, c_i64p, c_i64p, c_i64p]),
    "nnsdp_plan_tiles": (c_i32, [c_i64, c_i64p, c_i64, c_i32, c_i64, C.POINTER(c_i32), c_i64p]),
    "nnsdp_plan_panel": (c_i32, [c_i64, c_i64p, c_i64, c_i32, c_i64, c_i64p, c_i64p]),
    "nnsdp_gather_plan": (c_i32, [c_i64, c_i64p, c_i64, c_i32, c_i64, C.POINTER(c_i32), c_i64p, c_i64, c_i64p, c_i64p, C.POINTER(c_i32)]),
    "nnsdp_bounds_ibp": (c_i32, [c_vp, c_vp, c_i64, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp]),
    "nnsdp_bounds_crown": (c_i32, [c_vp, c_vp, c_i64, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp]),
    "nnsdp_batch_bounds_crown": (c_i32, [c_vp]),
    "nnsdp_batch_set_bounds_method": (c_i32, [c_vp, c_i32]),
    "nnsdp_batch_keep_crown_preact": (c_i32, [c_vp, c_i32]),
    "nnsdp_batch_get_crown_preact": (c_i32, [c_vp, c_dp, c_dp]),
    "nnsdp_preact_from_x": (c_i32, [c_vp, c_vp, c_i64, c_dp, c_dp, c_dp, c_dp]),
    "nnsdp_sector_minmax": (c_i32, [c_vp, c_i64, c_dp, c_dp, c_dp, c_dp]),
    "nnsdp_assemble_blocks": (c_i32, [c_vp, c_vp, c_i64, c_i64, C.POINTER(QueryInputs), c_dp]),
    "nnsdp_assemble_dense": (c_i32, [c_vp, c_vp, c_i64, c_i64, C.POINTER(QueryInputs), c_dp]),
    "nnsdp_batch_lambda_max": (c_i32, [c_vp, c_i32, C.c_double, c_dp, C.POINTER(c_i32)]),
    "nnsdp_batch_lambda_max_ex": (c_i32, [c_vp, c_i32, C.c_double, c_dp, C.POINTER(c_i32), c_dp, C.POINTER(c_i32)]),
    "nnsdp_batch_certify": (c_i32, [c_vp, c_dp, c_i64, C.POINTER(c_i32), c_dp, c_i64p, c_dp]),
    "nnsdp_batch_certify_ex": (c_i32, [c_vp, c_dp, c_i64, C.POINTER(c_i32), c_dp, c_i64p, c_dp, c_dp]),
    "nnsdp_certify_plan": (c_i32, [c_i64, c_i64p, c_i64, c_i64, c_i64p, c_i64p]),
    "nnsdp_batch_assembly_error": (c_i32, [c_vp, c_dp, c_dp]),
    "nnsdp_assembly_error_nmax": (c_i32, [c_i64, c_i64p, c_i64, c_i32, c_i64p]),
    "nnsdp_batch_certify_gamma": (c_i32, [c_vp, c_dp, c_i64, C.POINTER(c_i32), c_dp, c_i64p, c_dp, c_dp, c_dp]),
    "nnsdp_affine_create": (c_i32, [c_vp, c_vp, c_i64, C.POINTER(QueryInputs), c_i64, C.POINTER(c_vp), C.POINTER(AffineSizes)]),
    "nnsdp_affine_get": (c_i32, [c_vp, c_i64p, c_i64p, c_dp, c_i64p, c_i64p, c_dp]),
    "nnsdp_affine_destroy": (c_i32, [c_vp]),
    "nnsdp_affine_create_batch": (c_i32, [c_vp, c_vp, c_i64, c_i64, C.POINTER(QueryInputs), c_i64, C.POINTER(c_vp),
                                          C.POINTER(AffineBatchSizes)]),
    "nnsdp_affine_batch_groups": (c_i32, [c_vp, c_i64p, c_i64p, c_i64p]),
    "nnsdp_affine_batch_get": (c_i32, [c_vp, c_i64p, c_i64p, c_dp]),
    "nnsdp_affine_batch_get_group": (c_i32, [c_vp, c_i64, c_i64p, c_i64p, c_dp]),
    "nnsdp_affine_batch_destroy": (c_i32, [c_vp]),
    "nnsdp_batch_create": (c_i32, [c_vp, c_i32, c_vp, c_i64, c_i64, c_i64, c_i32, C.POINTER(c_vp)]),
    "nnsdp_batch_destroy": (c_i32, [c_vp]),
    "nnsdp_batch_set_inputs": (c_i32, [c_vp, c_i64, C.POINTER(QueryInputs)]),
    "nnsdp_batch_bounds": (c_i32, [c_vp]),
    "nnsdp_batch_prepare": (c_i32, [c_vp]),
    "nnsdp_batch_emit": (c_i32, [c_vp, c_i64, c_i64]),
    "nnsdp_batch_run": (c_i32, [c_vp, c_dp]),
    "nnsdp_batch_run_ex": (c_i32, [c_vp, c_dp, c_i32]),
    "nnsdp_batch_run_packed": (c_i32, [c_vp, c_dp, C.POINTER(C.c_uint8), c_i32]),
    "nnsdp_batch_packed_stats": (c_i32, [c_vp, c_i64p, c_i64p, c_i64p, c_i64p, c_i64p]),
    "nnsdp_packed_layout": (c_i32, [c_i64, c_i64p, c_i64, c_i64, C.POINTER(PackedCell), c_i64p, c_i64p, c_i64p]),
    "nnsdp_packed_unpack": (c_i32, [c_i64, c_i64p, c_i64, c_dp, C.POINTER(C.c_uint8), c_i32, c_dp]),
    "nnsdp_assemble_packed": (c_i32, [c_vp, c_vp, c_i64, c_i64, C.POINTER(QueryInputs), c_dp, C.POINTER(C.c_uint8)]),
    "nnsdp_batch_gather_stats": (c_i32, [c_vp, c_i64p, c_i64p, c_i64p, C.POINTER(c_i32)]),
    "nnsdp_batch_sync": (c_i32, [c_vp]),
    "nnsdp_batch_get_bounds": (c_i32, [c_vp, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp]),
    "nnsdp_batch_get_slot": (c_i32, [c_vp, c_i64, c_dp]),
    "nnsdp_batch_get_affine": (c_i32, [c_vp, c_dp]),
    "nnsdp_batch_ring_ptr": (c_i32, [c_vp, C.POINTER(c_u64), C.POINTER(c_i64)]),
    "nnsdp_batch_ring_reset": (c_i32, [c_vp]),
    "nnsdp_batch_emit_stats": (c_i32, [c_vp, c_i64p]),
    "nnsdp_batch_event_record": (c_i32, [c_vp, c_i32]),
    "nnsdp_batch_elapsed_ms": (c_i32, [c_vp, C.POINTER(C.c_float)]),
    "nnsdp_batch_stage_ms": (c_i32, [c_vp, c_i32, C.POINTER(C.c_float), C.POINTER(c_i64)]),
    "nnsdp_batch_stage_reset": (c_i32, [c_vp]),
    "nnsdp_batch_gram_stats": (c_i32, [c_vp, C.POINTER(c_i64), C.POINTER(c_i64)]),
}


class NnsdpError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"nnsdp_b200 error {code}: {msg}")
        self.code = code


def _load():
    path = os.path.abspath(LIB_PATH)
    if not os.path.exists(path):
        raise ImportError(
            f"{path} not found: build it with `make -C nn-sdp_b200` (or __graft_entry__.build()); "
            "nnsdp_b200 has no CPU fallback")
    lib = C.CDLL(path)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export it
        fn.restype = res
        fn.argtypes = args
    return lib


lib = _load()


def check(status: int):
    if status != OK:
        raise NnsdpError(status, lib.nnsdp_last_error().decode("utf-8", "replace"))


def device_count() -> int:
    n = c_i32(0)
    check(lib.nnsdp_device_count(C.byref(n)))
    return int(n.value)
