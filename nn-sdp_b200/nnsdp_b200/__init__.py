"""nnsdp_b200: B200-native constraint construction for Chordal-DeepSDP (host-side Python mirror).

The compute lives in lib/libnnsdp_b200.so (hand-written sm_100a CUDA, C ABI in
include/nnsdp_b200.h).  Importing this package loads that library and fails if it is missing.
"""
from . import _lib
from ._lib import NnsdpError, device_count, OUT_SAFETY, OUT_HPLANE, OUT_CIRCLE, OUT_ELLIPSOID, RUN_HOST_PREZEROED, RUN_DENSE_COPY, FORMAT_BLOCKS, FORMAT_DENSE_Z, FORMAT_PACKED, CELL_WINDOW, CELL_DIAG, CELL_BAND, CELL_RECT
from .core import (Context, Net, Batch, NumericBatch, PinnedBuffer, assemble_blocks, assemble_dense,
                   bounds_ibp, bounds_crown, preact_from_x, sector_minmax, split_blocks, sizes_from_xdims,
                   cliques_from_xdims, plan_stats, plan_tiles, plan_panel, certify_plan, assembly_error_nmax, affine_form, affine_form_batch, gather_plan, read_nnet, read_vnnlib, packed_layout, packed_unpack,
                   assemble_packed)
from . import reference_api
