/*
 * nnsdp_b200.h -- C ABI of libnnsdp_b200.so
 *
 * B200-native (sm_100a) implementation of the Chordal-DeepSDP constraint-construction
 * hot path of AntonXue/nn-sdp: interval bounds -> ReLU QC blocks -> per-clique LMI
 * assembly, batched over queries.  This is the drop-in boundary: Julia `ccall`s it
 * (see INTEGRATION.md), Python `ctypes` loads it in this repository's tests.
 *
 * The reference has no FFI for this path; each entry point cites the reference
 * function(s) it replaces (paths relative to the reference repository root).
 *
 * Conventions
 *  - every function returns int32 status: 0 = OK, < 0 = error; the message is
 *    available (thread-local) from nnsdp_last_error().  No C++ exception crosses.
 *  - all matrices are column-major FP64; all index arrays are Int64 and 1-BASED on
 *    the wire (Julia-native) so clique sets compare bit-exactly with makeCliques.
 *  - per-query arrays are stored query-major: column q of an (n x Q) array is the
 *    contiguous vector of query q.  A `*_stride` of 0 in nnsdp_query_inputs shares
 *    one column between all queries (reach batches, src/NnSdp.jl:73-95).
 *  - the caller owns every host buffer; the library owns device memory behind the
 *    opaque handles.  Calls are blocking unless stated otherwise.
 *  - there is NO CPU fallback: without a CUDA device every compute entry point
 *    returns NNSDP_ERR_CUDA.
 */
#ifndef NNSDP_B200_H
#define NNSDP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NNSDP_OK 0
#define NNSDP_ERR_ARG (-1)    /* bad argument / shape                                  */
#define NNSDP_ERR_CUDA (-2)   /* CUDA runtime failure, or no device                     */
#define NNSDP_ERR_NOMEM (-3)  /* host or device allocation failed                       */
#define NNSDP_ERR_STATE (-4)  /* call sequence error (e.g. emit before prepare)         */
#define NNSDP_ERR_ASSERT (-5) /* an @assert of the reference would have failed          */
#define NNSDP_ERR_NOCONV (-6) /* an iteration stopped at its cap (results are still written) */

/* Output QC kinds, src/Qc/output.jl:3-31 */
#define NNSDP_OUT_SAFETY 0    /* QcSafety(S)                                            */
#define NNSDP_OUT_HPLANE 1    /* QcReachHplane(normal)                                  */
#define NNSDP_OUT_CIRCLE 2    /* QcReachCircle(yc)                                      */
#define NNSDP_OUT_ELLIPSOID 3 /* QcReachEllipsoid(invP, yc)                             */

/* Output formats of a batch (the `dense_Z` argument of nnsdp_batch_create and of the plan introspection calls) */
#define NNSDP_FORMAT_BLOCKS 0   /* every clique block Z[C_k, C_k] dense, back to back                       */
#define NNSDP_FORMAT_DENSE_Z 1  /* the whole Z, dense                                                        */
#define NNSDP_FORMAT_PACKED 2   /* packed records: the block-sparse upper triangle of Z (see below)          */

typedef struct nnsdp_ctx nnsdp_ctx;     /* devices + streams                             */
typedef struct nnsdp_net nnsdp_net;     /* FeedFwdNet uploaded (replicated per device)   */
typedef struct nnsdp_batch nnsdp_batch; /* device-resident state of a batch of queries   */

/* Sizes derived from (net, beta).  Mirrors: FeedFwdNet.zdims (MyNeuralNetwork.jl:17),
 * QcActivSector._lambda_dim / vardim (src/Qc/activ_sector.jl:18-19), makeCliques. */
typedef struct {
  int64_t K;         /* number of affine layers, length(Ms)                              */
  int64_t Zdim;      /* sum(zdims) = sum(xdims[1:K]) + 1                                 */
  int64_t acdim;     /* sum(xdims[2:K]) : stacked hidden activations                     */
  int64_t xtot;      /* sum(xdims[1:K+1]) : stacked x_intvs length                       */
  int64_t lamdim;    /* _lambda_dim = sum((acdim-beta):acdim)                            */
  int64_t secdim;    /* sector vardim = lamdim + 2*acdim                                 */
  int64_t n_in;      /* xdims[1]                                                         */
  int64_t n_out;     /* xdims[K+1]                                                       */
  int64_t sdim;      /* n_in + n_out + 1 : side of the output matrix S                   */
  int64_t ncliques;  /* p                                                                */
  int64_t sum_ck;    /* sum_k |C_k|                                                      */
  int64_t sum_ck_sq; /* sum_k |C_k|^2 : doubles per query of dense block output          */
  int64_t sum_dk;    /* sum_k (|D_k1| + |D_k2|)                                          */
  int64_t max_ck;    /* max_k |C_k|                                                      */
} nnsdp_sizes;

/* One batch of Q numeric-gamma queries.  Pointers are HOST pointers for the one-shot
 * entry points and for nnsdp_batch_set_inputs.  stride = doubles between consecutive
 * queries (0 = shared by all queries; otherwise must be >= the vector length).
 *
 * Bounds: if ymin == NULL the library computes interval bounds on the device from
 * (x1min, x1max) with IBP (IntervalsWorstCase, src/Intervals/intervals_easy.jl:2-37)
 * and derives smin/smax with makeSectorMinMax (src/Qc/activ_sector.jl:63-72); this is
 * makeQcActivsIntvs (src/Qc/activ.jl:45-67) with method = IntervalsWorstCase.
 * Otherwise the caller supplies what the two activation QCs hold:
 *   ymin/ymax : QcActivBounded.acymin/acymax (POST-activation bounds of x_2..x_K)
 *   smin/smax : QcActivSector.smin/smax.
 */
typedef struct {
  const double* x1min;     int64_t x1min_stride;     /* n_in   QcInputBox.x1min (src/Qc/input.jl:3-8) */
  const double* x1max;     int64_t x1max_stride;     /* n_in   QcInputBox.x1max                       */
  const double* ymin;      int64_t ymin_stride;      /* acdim  or NULL                                */
  const double* ymax;      int64_t ymax_stride;      /* acdim                                          */
  const double* smin;      int64_t smin_stride;      /* acdim                                          */
  const double* smax;      int64_t smax_stride;      /* acdim                                          */
  const double* gamma_in;  int64_t gamma_in_stride;  /* n_in   gamma of makeZin                        */
  const double* gamma_bnd; int64_t gamma_bnd_stride; /* acdim  gamma of makeZac(QcActivBounded)        */
  const double* gamma_sec; int64_t gamma_sec_stride; /* secdim gamma of makeZac(QcActivSector):
                                                        [lambda(acdim); v(pairs i<j<=i+beta, i asc, j asc);
                                                         eta(acdim); nu(acdim)]  activ_sector.jl:26-54 */
  int32_t out_kind;        int32_t reserved;
  const double* out_S;     int64_t out_S_stride;     /* SAFETY: sdim*sdim col-major; like Julia's
                                                        Symmetric(S) the UPPER triangle is read        */
  const double* out_vec;   int64_t out_vec_stride;   /* HPLANE: normal(n_out); CIRCLE/ELLIPSOID: yc    */
  const double* out_invP;  int64_t out_invP_stride;  /* ELLIPSOID: n_out*n_out col-major               */
  const double* gamma_out; int64_t gamma_out_stride; /* reach kinds: 1 per query                       */
} nnsdp_query_inputs;

/* ---- error / environment ------------------------------------------------------------ */
const char* nnsdp_last_error(void);
int32_t nnsdp_version(void);
int32_t nnsdp_device_count(int32_t* count);

/* ---- context ------------------------------------------------------------------------
 * ndev devices (CUDA ordinals in dev_ids; NULL = 0..ndev-1).  One non-blocking stream
 * per device.  Queries of the one-shot entry points are sharded over the devices in
 * contiguous ranges with one host thread per device; no collective is used. */
int32_t nnsdp_ctx_create(int32_t ndev, const int32_t* dev_ids, nnsdp_ctx** ctx);
int32_t nnsdp_ctx_destroy(nnsdp_ctx* ctx);
int32_t nnsdp_ctx_num_devices(const nnsdp_ctx* ctx, int32_t* ndev);
/* Pinned host memory for fast host<->device copies (optional; any host memory works). */
int32_t nnsdp_host_alloc(uint64_t bytes, void** ptr);
int32_t nnsdp_host_free(void* ptr);

/* ---- network: FeedFwdNet (src/MyNeuralNetwork/MyNeuralNetwork.jl:12-27) ---------------
 * xdims has K+1 entries; Ms[k] is the column-major xdims[k+1] x (xdims[k]+1) matrix
 * [W_k b_k].  ReLU activations.  Weights are copied to every device of ctx. */
int32_t nnsdp_net_upload(nnsdp_ctx* ctx, int64_t K, const int64_t* xdims, const double* const* Ms,
                         nnsdp_net** net);
int32_t nnsdp_net_destroy(nnsdp_net* net);

/* .nnet reader, host only (SURVEY.md 8f-4): the format of the reference's fixtures bench/rand/*.nnet as read
 * by exts/nnet_parser.jl:35-131 and loadFromNnet (src/MyNeuralNetwork/network_files.jl).  Two calls: the first
 * with Ms_out == NULL returns K, xdims (K+1 entries, if xdims_out != NULL and max_layers >= K) and the number
 * of doubles needed; the second fills Ms_out with the matrices [W_k b_k] back to back, each column-major
 * xdims[k+1] x (xdims[k]+1) -- what nnsdp_net_upload takes (Ms[k] = Ms_out + sum_{k'<k} xdims[k'+1](xdims[k']+1)). */
int32_t nnsdp_nnet_read(const char* path, int64_t max_layers, int64_t* K, int64_t* xdims_out,
                        int64_t max_doubles, double* Ms_out, int64_t* doubles_needed);

/* vnnlib reader, host only (SURVEY.md 8f-4): the "simple" vnnlib subset of read_vnnlib_simple
 * (exts/vnnlib_parser.jl:99-216), flattened the way loadVnnlibCnf does (experiments/vnnlib_utils.jl:18-56) into
 * safety queries that nnsdp_assemble_blocks takes directly: the file states NOT phi as
 * OR_box OR_(A,b) (x in box AND A y <= b); every (box, (A, b)) is one disjunctive clause whose members are, per row
 * i, the query (box, S = hplaneS(-A_i, -b_i - 1e-4)).  Two calls: with x1min == NULL only nqueries / nclauses are
 * returned; then x1min, x1max (nqueries x n_in), out_S (nqueries x sdim x sdim, sdim = n_in + n_out + 1) and
 * clause_of (nqueries, 0-based clause index) are filled.  Boxes keep their order of first appearance (the
 * reference iterates a Dict there).  Unsupported statements are NNSDP_ERR_ARG, the reader's asserts
 * NNSDP_ERR_ASSERT. */
int32_t nnsdp_vnnlib_read(const char* path, int64_t n_in, int64_t n_out, int64_t max_queries, int64_t* nqueries,
                          int64_t* nclauses, double* x1min, double* x1max, double* out_S, int64_t* clause_of);

/* ---- integer work on the host, bit-exact --------------------------------------------- */
int32_t nnsdp_query_sizes(const nnsdp_net* net, int64_t beta, nnsdp_sizes* sizes);
/* makeCliques (src/Methods/chordal_cliques.jl:13-59).  Outputs (1-based):
 *   ck_off[ncliques+1]  offsets (0-based) into ck_idx;  ck_idx[sum_ck] = C_k concatenated
 *   ck1_len[ncliques]   |C_k1| (= |C_k| for the last clique, which has one part)
 *   d_off[2*ncliques+1] offsets into d_idx of D_k1, D_k2 (empty D_k2 for k = 1 and k = p)
 *   d_idx[sum_dk]       local indices into C_k */
int32_t nnsdp_cliques(const nnsdp_net* net, int64_t beta, int64_t* ck_off, int64_t* ck_idx,
                      int64_t* ck1_len, int64_t* d_off, int64_t* d_idx);
/* The same two functions from xdims alone (K+1 entries): no device, no uploaded network. */
int32_t nnsdp_sizes_from_xdims(int64_t K, const int64_t* xdims, int64_t beta, nnsdp_sizes* sizes);
int32_t nnsdp_cliques_from_xdims(int64_t K, const int64_t* xdims, int64_t beta, int64_t* ck_off,
                                 int64_t* ck_idx, int64_t* ck1_len, int64_t* d_off, int64_t* d_idx);

/* Introspection of the emission plan (host only): tiles and output entries per tile program
 * (8 slots: ZERO, SAME, RC, CR, MIXED, GENERAL, DIAG, AFF; see DESIGN.md, "emitter"). */
int32_t nnsdp_plan_stats(int64_t K, const int64_t* xdims, int64_t beta, int32_t dense_Z,
                         int64_t* tiles_per_prog, int64_t* entries_per_prog, int64_t* tile_rows,
                         int64_t* tile_cols);

/* The tile list itself: 11 int32 per tile {mat, row0, nrows, col0, ncols, grow0, gcol0, flags, rblk,
 * cblk, prog} (rows/cols local to output matrix `mat`, grow0/gcol0 global 0-based z indices).
 * tiles_out == NULL queries the count. */
int32_t nnsdp_plan_tiles(int64_t K, const int64_t* xdims, int64_t beta, int32_t dense_Z,
                         int64_t max_tiles, int32_t* tiles_out, int64_t* ntiles);

/* The panel-ordered work list of the dense formats of wide nets (host only): the items of the fill and the window
 * program classes as ONE list sorted by (output matrix, 32-column panel, first column, first row), so that all pieces
 * of a column of a clique block are written by consecutive CTAs of one launch.  10 int64 per item {out_off, ld, row0,
 * nrows, col0, ncols, grow0, gcol0, prog, rblk} (out_off = offset in doubles of the item's matrix inside one query's
 * output; rows / columns local to that matrix).  *nitems == 0: this plan keeps the separate kernels (packed records,
 * narrow layers, beta above the window programs).  items_out == NULL queries the count. */
int32_t nnsdp_plan_panel(int64_t K, const int64_t* xdims, int64_t beta, int32_t dense_Z, int64_t max_items,
                         int64_t* items_out, int64_t* nitems);

/* The host-gather plan of nnsdp_batch_run_ex (host only, for inspection and tests): every output matrix cut at
 * block boundaries into cells, 8 int32 each {mat, row0, nrows, col0, ncols, kind, blk, pure_zero} with kind
 * 0 = never copied as a whole, 1 = always dense, 2 = dense when layer blk has a stably-active neuron,
 * 3 = dense when the output QC has an S22 part; and the offsets (doubles inside one query's output) of the thin
 * entries that travel packed.  *usable = 0 means the dense copy is used for this network. */
int32_t nnsdp_gather_plan(int64_t K, const int64_t* xdims, int64_t beta, int32_t dense_Z, int64_t max_cells,
                          int32_t* cells_out, int64_t* ncells, int64_t max_thin, int64_t* thin_out,
                          int64_t* nthin, int32_t* usable);

/* ---- one-shot entry points with HOST buffers ------------------------------------------
 * intervalsWorstCase (src/Intervals/intervals_easy.jl:2-37), batched over Q boxes.
 *   x1min,x1max : n_in x Q;  xmin,xmax : xtot x Q (x_intvs stacked, x_1 first);
 *   acxmin,acxmax : acdim x Q (acx_intvs stacked).  Any output may be NULL. */
int32_t nnsdp_bounds_ibp(nnsdp_ctx* ctx, const nnsdp_net* net, int64_t Q, const double* x1min,
                         const double* x1max, double* xmin, double* xmax, double* acxmin,
                         double* acxmax);
/* CROWN bounds, the reference's DEFAULT interval method: makeIntervalsInfo(x1min, x1max, ffnet,
 * IntervalsAutoLirpa()) -> intervalsAutoLirpaSliced (src/Intervals/Intervals.jl:38,44-45;
 * src/Intervals/intervals_auto_lirpa.jl:44-63; exts/auto_lirpa_bridge.py:97-112 -> vendored auto_LiRPA,
 * compute_bounds(method="CROWN"), float32, one ONNX file + Python call per layer).  Same layout as
 * nnsdp_bounds_ibp: xmin/xmax are the x_intvs of the sliced method (x_{k+1} bounded as the output of the
 * k-layer prefix followed by an identity layer, then lb = min(lb, ub), ub = max(lb, ub)); acxmin/acxmax the
 * one-step IBP of intervals_auto_lirpa.jl:55-62.  FP64 on the device; the reference's values carry float32
 * precision.  Fails with NNSDP_ERR_ASSERT where the reference asserts ykmin <= ykmax (:60). */
int32_t nnsdp_bounds_crown(nnsdp_ctx* ctx, const nnsdp_net* net, int64_t Q, const double* x1min,
                           const double* x1max, double* xmin, double* xmax, double* acxmin, double* acxmax);
/* One-step pre-activation IBP from given x_intvs
 * (src/Intervals/intervals_auto_lirpa.jl:55-62): reads xmin/xmax (xtot x Q), writes
 * acxmin/acxmax (acdim x Q).  Fails with NNSDP_ERR_ASSERT if some ymin > ymax (:60). */
int32_t nnsdp_preact_from_x(nnsdp_ctx* ctx, const nnsdp_net* net, int64_t Q, const double* xmin,
                            const double* xmax, double* acxmin, double* acxmax);
/* makeSectorMinMax, ReLU branch (src/Qc/activ_sector.jl:63-72). n = acdim * Q entries. */
int32_t nnsdp_sector_minmax(nnsdp_ctx* ctx, int64_t n, const double* acxmin, const double* acxmax,
                            double* smin, double* smax);
/* Z[C_k, C_k] for every clique and query, dense column-major, for numeric gamma:
 * blocks_out[q * sum_ck_sq + off_k + i + j*|C_k|], off_k = sum_{k'<k} |C_k'|^2.
 * Z = makeZin + makeZout + makeZac(bounded) + makeZac(sector)
 * (src/Qc/input.jl:19-42, output.jl:52-106, activ.jl:30-41; summed as in
 * src/Methods/chordal_sdp.jl:114,145) restricted to the cliques of makeCliques. */
int32_t nnsdp_assemble_blocks(nnsdp_ctx* ctx, const nnsdp_net* net, int64_t beta, int64_t Q,
                              const nnsdp_query_inputs* in, double* blocks_out);
/* The full dense Z (Zdim x Zdim per query), i.e. Zin + Zout + sum(Zacs) of
 * src/Methods/chordal_sdp.jl:114 / scripts/test_acas.jl:81-85.  For moderate Zdim. */
int32_t nnsdp_assemble_dense(nnsdp_ctx* ctx, const nnsdp_net* net, int64_t beta, int64_t Q,
                             const nnsdp_query_inputs* in, double* Z_out);

/* ---- packed records (NNSDP_FORMAT_PACKED) ---------------------------------------------------
 * 78 % of the entries of the dense clique blocks of a wide net are structural zeros, every diagonal block is held
 * by two cliques and the x_K block by all of them.  Every clique block is a principal submatrix Z[C_k, C_k] and the
 * cliques cover the non-zeros of Z (the scatter structure of setupZksum!, src/Methods/chordal_sdp.jl:60-93,
 * chordal_cliques.jl:31-57), so a packed record stores each region of Z that can be non-zero ONCE, as column-major
 * cells (ld = nrows) at fixed offsets, upper triangle only (cells that straddle the diagonal are stored as
 * rectangles; only their entries with row <= column are defined, like Julia's Symmetric(A, :U)):
 *   NNSDP_CELL_WINDOW  rows x_b against x_{b+1}: the W' M window sums (and the band corner)            always
 *   NNSDP_CELL_DIAG    interior of the diagonal block of x_b (Gram W_b' diag(.) W_b | W_K' S22 W_K, band included);
 *                      written only for a query whose layer has a stably-active neuron / whose output QC has an S22
 *                      part -- present[] says which; an absent cell is all zero apart from its BAND cell and its
 *                      bytes in the record are not touched
 *   NNSDP_CELL_BAND    (beta+1) x m: band[t + (beta+1) i] = Z[row0+i, row0+i+t], the band inside the DIAG range  always
 *   NNSDP_CELL_RECT    everything else (affine column, slivers of width beta, x_1 block, x_1 / x_K coupling)     always
 * Where cells overlap they hold bit-identical values.  Small nets (a hidden layer under 48 neurons) have one RECT
 * cell, the whole Z.  Z[C_k, C_k] of any clique is a set of sub-rectangles of the cells (nnsdp_packed_unpack does
 * exactly that; Julia: views into the record, or sparse(...) from the cell table). */
#define NNSDP_CELL_WINDOW 1
#define NNSDP_CELL_DIAG 2
#define NNSDP_CELL_BAND 3
#define NNSDP_CELL_RECT 4
typedef struct {
  int32_t kind;          /* NNSDP_CELL_*                                                                  */
  int32_t blk;           /* b of WINDOW (x_b, x_{b+1}) / DIAG / BAND (1-based block); 0 for RECT           */
  int64_t row0, col0;    /* 1-based index in Z of the cell's first row / column                            */
  int64_t nrows, ncols;
  int64_t offset;        /* doubles from the start of a query's record                                     */
  int32_t always;        /* 1: written for every query; 0: only when present                               */
  int32_t reserved;
} nnsdp_packed_cell;
/* Cell table of (xdims, beta), host only.  cells == NULL queries the count.  A record is record_doubles long; the
 * always-written cells occupy its first always_doubles. */
int32_t nnsdp_packed_layout(int64_t K, const int64_t* xdims, int64_t beta, int64_t max_cells, nnsdp_packed_cell* cells,
                            int64_t* ncells, int64_t* record_doubles, int64_t* always_doubles);
/* One record -> the dense output of NNSDP_FORMAT_BLOCKS (every Z[C_k, C_k], sum_ck_sq doubles) or
 * NNSDP_FORMAT_DENSE_Z (Zdim^2), both triangles filled; present = the record's ncells bytes.  Host only. */
int32_t nnsdp_packed_unpack(int64_t K, const int64_t* xdims, int64_t beta, const double* record, const uint8_t* present,
                            int32_t format, double* out);
/* One-shot: packed records of Q queries into records_out[q * record_doubles], present_out[q * ncells] (may be NULL). */
int32_t nnsdp_assemble_packed(nnsdp_ctx* ctx, const nnsdp_net* net, int64_t beta, int64_t Q,
                              const nnsdp_query_inputs* in, double* records_out, uint8_t* present_out);

/* ---- device-resident batch (what bench.py times with inputs already in HBM) -----------
 * A batch lives on ONE device of the ctx (dev_index into the ctx's device list).
 * Limits: n_in + n_out + 1 <= 160 for batches that assemble (ring_queries > 0; the output-QC matrix S is held in
 * shared memory) -- bounds-only batches (ring_queries = 0: IBP / CROWN on image-sized inputs) have no such limit;
 * hidden widths up to ~46,000 (tile pairs of the Gram kernel); any Qcap < 2^30.
 * ring_queries = number of per-query output slots kept on the device; 0 = bounds only
 * (no gamma inputs are read and nothing can be emitted).  dense_Z is the output format of a query:
 * NNSDP_FORMAT_BLOCKS (0) the clique blocks, NNSDP_FORMAT_DENSE_Z (1) the whole Zdim x Zdim matrix,
 * NNSDP_FORMAT_PACKED (2) a packed record. */
int32_t nnsdp_batch_create(nnsdp_ctx* ctx, int32_t dev_index, const nnsdp_net* net, int64_t beta,
                           int64_t Qcap, int64_t ring_queries, int32_t dense_Z, nnsdp_batch** batch);
int32_t nnsdp_batch_destroy(nnsdp_batch* batch);
/* Host -> device copy of the inputs of Q <= Qcap queries (async on the batch stream). */
int32_t nnsdp_batch_set_inputs(nnsdp_batch* batch, int64_t Q, const nnsdp_query_inputs* in);
/* K1 + K2: IBP from the boxes and sector slopes, all on the device. */
int32_t nnsdp_batch_bounds(nnsdp_batch* batch);
/* The same with CROWN bounds (see nnsdp_bounds_crown), and the choice nnsdp_batch_run makes when the batch
 * carries no caller-supplied bounds (default NNSDP_BOUNDS_IBP). */
#define NNSDP_BOUNDS_IBP 0
#define NNSDP_BOUNDS_CROWN 1
int32_t nnsdp_batch_bounds_crown(nnsdp_batch* batch);
int32_t nnsdp_batch_set_bounds_method(nnsdp_batch* batch, int32_t method);
/* QC diagonals, band multipliers, affine column (all queries of the batch). */
int32_t nnsdp_batch_prepare(nnsdp_batch* batch);
/* Gram contractions + block emission of queries [q0, q0+nq) into ring slots
 * (q - q0) % ring_queries ... ; nq <= ring_queries.  Asynchronous.
 * Ring slots are read-only to consumers.  A slot is zeroed when a pass first uses it; after that the emitter stores
 * only the entries that can differ from what the slot already holds (structural zeros are never stored again, the
 * diagonal block of a layer only while this query or the slot's previous one has a non-zero bulk there), and every
 * slot still holds the complete dense output of its query after each pass.  A value written into a slot by anything
 * but the library may therefore survive into later queries of that slot: call nnsdp_batch_ring_reset after writing
 * into the ring. */
int32_t nnsdp_batch_emit(nnsdp_batch* batch, int64_t q0, int64_t nq);
/* Full pass: bounds (if the batch has no caller-supplied bounds) + prepare + emit of all
 * Q queries through the ring, chunk by chunk.  If host_out != NULL every chunk is copied
 * to host_out[q * per_query_doubles] (device -> host inside the call).  Blocking. */
int32_t nnsdp_batch_run(nnsdp_batch* batch, double* host_out);
/* The same with flags.  The host gather never moves structural zeros over PCIe when the network is
 * wide enough: dense cells of every block (the W' M windows, Gram-active diagonal blocks) are copied
 * by strided DMA, the few other non-zeros (band, slivers, affine row / column) travel packed and are
 * scattered by host threads, and everything else is zero-filled by host threads -- host_out ends up
 * holding the complete dense blocks either way.
 *   NNSDP_RUN_HOST_PREZEROED  the caller guarantees that every entry of host_out that is structurally
 *                             zero for this (network, beta) -- the ZERO tiles of nnsdp_plan_tiles --
 *                             already holds 0.0 (a fresh calloc / zeros(), or a buffer a previous run
 *                             of the same batch filled); those bytes are then not touched at all.
 *   NNSDP_RUN_DENSE_COPY      copy the dense ring contents (one contiguous DMA per chunk). */
#define NNSDP_RUN_HOST_PREZEROED 1
#define NNSDP_RUN_DENSE_COPY 2
int32_t nnsdp_batch_run_ex(nnsdp_batch* batch, double* host_out, int32_t flags);
/* A batch created with NNSDP_FORMAT_PACKED: the same pass with packed records in the ring.  host_records
 * (Q * record_doubles, may be NULL) receives the always-written part of every record and the DIAG cells that are
 * present; present (Q * ncells bytes, may be NULL) says which cells of each record were written.  Nothing is
 * zero-filled or scattered on the host.  flags: NNSDP_RUN_DENSE_COPY copies whole records. */
int32_t nnsdp_batch_run_packed(nnsdp_batch* batch, double* host_records, uint8_t* present, int32_t flags);
/* Sizes of a packed batch and, for its last run: bytes the emitter stored (as nnsdp_batch_emit_stats), bytes moved to
 * the host, number of optional (DIAG) cells present over all queries. */
int32_t nnsdp_batch_packed_stats(nnsdp_batch* batch, int64_t* record_doubles, int64_t* ncells, int64_t* emitted_bytes,
                                 int64_t* d2h_bytes, int64_t* present_optional_cells);
/* Bytes the emitter stored into the ring in the last nnsdp_batch_run* (every format), plus those of the
 * nnsdp_batch_emit calls since.  Structural zeros are stored once per slot, by a memset outside this count. */
int32_t nnsdp_batch_emit_stats(nnsdp_batch* batch, int64_t* emitted_bytes);
/* Bytes the host gather of the last run moved: DMA (strided cells or dense), packed thin entries, and
 * bytes zero-filled by host threads; *sparse_usable = 1 if the sparse gather applies to this batch. */
int32_t nnsdp_batch_gather_stats(nnsdp_batch* batch, int64_t* dma_bytes, int64_t* thin_bytes,
                                 int64_t* zeroed_bytes, int32_t* sparse_usable);
int32_t nnsdp_batch_sync(nnsdp_batch* batch);
/* Copy results back (any pointer may be NULL). Blocking. */
int32_t nnsdp_batch_get_bounds(nnsdp_batch* batch, double* xmin, double* xmax, double* acxmin,
                               double* acxmax, double* smin, double* smax);
/* Copy of ring slot `slot` (read-only to consumers, see nnsdp_batch_emit). */
int32_t nnsdp_batch_get_slot(nnsdp_batch* batch, int64_t slot, double* host_out);
/* The affine column Z[:, a] of every query (Zdim x Q) after nnsdp_batch_prepare. */
int32_t nnsdp_batch_get_affine(nnsdp_batch* batch, double* aff_out);
/* Device pointer of the ring (for zero-copy consumers, e.g. torch.from_blob / CuArray).  The slots are read-only to
 * consumers (see nnsdp_batch_emit). */
int32_t nnsdp_batch_ring_ptr(nnsdp_batch* batch, uint64_t* dev_ptr, int64_t* slot_doubles);
/* Forget what the ring slots hold: each slot is zeroed again on its next use and its next pass stores every entry.
 * Needed only after something other than the library wrote into the ring. */
int32_t nnsdp_batch_ring_reset(nnsdp_batch* batch);
/* CUDA-event timing on the batch stream.  which: 0 = start, 1 = stop. */
int32_t nnsdp_batch_event_record(nnsdp_batch* batch, int32_t which);
int32_t nnsdp_batch_elapsed_ms(nnsdp_batch* batch, float* ms);
/* Per-stage device time (ms, CUDA events on the launching stream) accumulated since the last reset:
 * stage 0 bounds, 1 prepare, 2 gram, 3 emit (= 5 + 6 + 7), 4 d2h, and the three kernels of an emitter
 * pass: 5 emit_fill_kernel, 6 emit_window_kernel, 7 emit_edge_kernel.  Also counts kernel launches. */
int32_t nnsdp_batch_stage_ms(nnsdp_batch* batch, int32_t stage, float* ms, int64_t* launches);
int32_t nnsdp_batch_stage_reset(nnsdp_batch* batch);
/* Executed Gram work of the last prepare: number of (query, layer) contractions with a
 * non-empty active set and the sum over them of |active|. */
int32_t nnsdp_batch_gram_stats(nnsdp_batch* batch, int64_t* n_contractions, int64_t* sum_active);

/* ---- certificate check (SURVEY.md 8f-3) -----------------------------------------------------
 * lambda_max of Z(gamma) for every query of a prepared batch, without forming Z: Z x is evaluated from the
 * factored form R' Q R + Zin + Zout (one GEMM per layer over the batch) inside a Lanczos iteration with full
 * re-orthogonalisation, at most max_iters steps.  A query stops when the residual ||Z v - theta v|| of its largest
 * Ritz pair is below tol * (largest |Ritz value|) -- a tolerance relative to the spectral scale, so it also
 * triggers when lambda_max is near zero, the regime of the acceptance gate eigmax(Z) <= 1e-4 -- or when the Krylov
 * space is invariant.  Replaces eigmax(Symmetric(Matrix(value.(Z)))) (src/Methods/Methods.jl:116-117; acceptance
 * test experiments/acas.jl:71-79, scale.jl:76).
 * The Ritz value is a LOWER bound of lambda_max and converges from below: a query that stopped at max_iters is NOT
 * a certificate.  Outputs: lam_max[Q]; iters[Q], resid[Q] (the residual norm: an eigenvalue of Z lies within resid of
 * lam_max) and converged[Q] (1 / 0) may be NULL.  Returns NNSDP_ERR_NOCONV -- with every output written -- when
 * some query did not converge.  nnsdp_batch_lambda_max is the same call without the last two outputs. */
int32_t nnsdp_batch_lambda_max_ex(nnsdp_batch* batch, int32_t max_iters, double tol, double* lam_max, int32_t* iters,
                                  double* resid, int32_t* converged);
int32_t nnsdp_batch_lambda_max(nnsdp_batch* batch, int32_t max_iters, double tol, double* lam_max,
                               int32_t* iters);

/* ---- affine-coefficient mode (SURVEY.md 8f-1) ---------------------------------------------
 * Z(gamma) = Z0 + sum_v gamma_v Z_v for ONE query, restricted to the upper triangle of the clique
 * cover, as COO triplets -- the data from which `@constraint(model, Z .== Zksum)`
 * (src/Methods/chordal_sdp.jl:119,150) can be added without building AffExpr matrices
 * (src/Methods/Methods.jl:69-78, chordal_sdp.jl:96-153).  No multipliers are read from `in`.
 *   variables (1-based, the reference's creation order):
 *     [gamma_in (n_in); gamma_out (reach kinds only: 1); gamma_ac1 = bounded (acdim); gamma_ac2 = sector (secdim)]
 *     -- var_in / var_out / var_bnd / var_sec are the 0-based offsets of the four groups
 *   entries e = 1..nent: the positions (ent_row[e] <= ent_col[e]) of the cover's upper triangle,
 *     column-major; Z is structurally zero outside the cover (and Zksum has no variable there)
 *   Z[ent_row[e], ent_col[e]](gamma) = z0[e] + sum over triplets t with coo_ent[t] = e of
 *     coo_val[t] * gamma[coo_var[t]].   Duplicate (entry, variable) pairs occur and are to be summed
 *     (Julia: sparse(coo_ent, coo_var, coo_val, nent, nvar)).
 * nnsdp_affine_create computes everything on the device and reports the sizes; it fails with
 * NNSDP_ERR_NOMEM if max_nnz > 0 and nnz > max_nnz (the Gram term costs n_k(n_k+1)/2 coefficients per
 * stably-active neuron).  nnsdp_affine_get copies into caller buffers (any pointer may be NULL). */
typedef struct nnsdp_affine nnsdp_affine;
typedef struct {
  int64_t nvar, nent, nnz;
  int64_t var_in, var_out, var_bnd, var_sec;
} nnsdp_affine_sizes;
int32_t nnsdp_affine_create(nnsdp_ctx* ctx, const nnsdp_net* net, int64_t beta,
                            const nnsdp_query_inputs* in, int64_t max_nnz, nnsdp_affine** affine,
                            nnsdp_affine_sizes* sizes);
int32_t nnsdp_affine_get(nnsdp_affine* affine, int64_t* ent_row, int64_t* ent_col, double* z0,
                         int64_t* coo_ent, int64_t* coo_var, double* coo_val);
int32_t nnsdp_affine_destroy(nnsdp_affine* affine);

#ifdef __cplusplus
}
#endif
#endif /* NNSDP_B200_H */
