// Internal declarations shared by the host runtime and the sm_100a kernels.
// Nothing in here is part of the C ABI (see include/nnsdp_b200.h).
//
// Index conventions (0-based internally, 1-based only on the C ABI):
//   block b = 0..K-1 holds x_{b+1} (size n[b]); index a = off[K] = Zdim-1 is the affine entry.
//   layer matrix M[k] = [W_k b_k] (k = 0..K-1) maps block k to the n[k+1] rows it produces.
//   hidden neuron j = 0..acdim-1 is z-index n[0]+j; the neurons of block b (1 <= b <= K-1)
//   are [noff(b), noff(b)+n[b]) with noff(b) = off[b]-n[0]; they are the rows of M[b-1].
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/nnsdp_b200.h"

namespace nnsdp {

// ---------------------------------------------------------------------------------
// error plumbing
// ---------------------------------------------------------------------------------
void set_error(const char* fmt, ...);
int32_t cuda_fail(cudaError_t e, const char* what, const char* file, int line);

#define NN_CUDA(call)                                                                \
  do {                                                                               \
    cudaError_t _e = (call);                                                         \
    if (_e != cudaSuccess) return ::nnsdp::cuda_fail(_e, #call, __FILE__, __LINE__); \
  } while (0)

#define NN_CHECK(cond, code, ...)      \
  do {                                 \
    if (!(cond)) {                     \
      ::nnsdp::set_error(__VA_ARGS__); \
      return (code);                   \
    }                                  \
  } while (0)

#define NN_TRY(expr)               \
  do {                             \
    int32_t _s = (expr);           \
    if (_s != NNSDP_OK) return _s; \
  } while (0)

// ---------------------------------------------------------------------------------
// host-side shape bookkeeping
// ---------------------------------------------------------------------------------
struct Shape {
  int K = 0;
  std::vector<int64_t> n;     // K+1 : xdims
  std::vector<int64_t> off;   // K+1 : off[b] = sum n[0..b-1]; off[K] = a = Zdim-1
  std::vector<int64_t> xoff;  // K+2 : offsets into stacked x_intvs
  int64_t Zdim = 0, acdim = 0, xtot = 0;
  int64_t n_in() const { return n[0]; }
  int64_t n_out() const { return n[K]; }
  int64_t noff(int b) const { return off[b] - n[0]; }
  int block_of(int64_t z) const {  // z in [0, Zdim)
    int b = 0;
    while (b < K && z >= off[b + 1]) ++b;
    return b;
  }
};

// A clique = one or two contiguous global index ranges [lo, hi] (0-based, inclusive).
struct CliqueRanges {
  int nseg = 0;
  int64_t lo[2] = {0, 0}, hi[2] = {0, 0};
  int64_t size() const {
    int64_t s = 0;
    for (int i = 0; i < nseg; ++i) s += hi[i] - lo[i] + 1;
    return s;
  }
};

struct CliqueInfoHost {
  std::vector<CliqueRanges> ck;              // p cliques
  std::vector<std::vector<int64_t>> d1, d2;  // 1-based local indices (Dk1, Dk2)
};

int32_t make_cliques_host(const Shape& sh, int64_t beta, CliqueInfoHost* out);
int64_t lambda_dim(int64_t acdim, int64_t beta);
// Gram scratch layout of one query: block b (b <= K-2) at goff[b], leading dimension ldG[b].
long long gram_layout(const Shape& sh, std::vector<long long>* goff, std::vector<int>* ldG);
int32_t fill_sizes(const Shape& sh, int64_t beta, nnsdp_sizes* out);

// ---------------------------------------------------------------------------------
// emission plan: every output matrix (a clique block, or the dense Z) is cut into
// rectangular tiles; each tile carries the set of terms of Z that can be non-zero in it.
// ---------------------------------------------------------------------------------
enum TileFlags : uint32_t {
  TF_AFF = 1u << 0,    // contains the affine row and/or column
  TF_SAME = 1u << 1,   // rows and columns share a block: Gram / Zin / S11 / W_K' S22 W_K
  TF_1K = 1u << 2,     // x_1 against x_K coupling S12 W_K (either orientation)
  TF_RC = 1u << 3,     // F(r,c) = sum_j W_b[j,r] M[j,c] with r in block b, c a neuron near layer b+1
  TF_CR = 1u << 4,     // F(c,r), the transposed term
  TF_BAND = 1u << 5,   // neuron-neuron band: -2 T and the -2 gamma_bnd diagonal
  TF_ALL = 0x3Fu,
  TF_UNIFORM = 1u << 8,  // rows lie in one block and columns lie in one block (rblk, cblk valid)
};

// Tile programs of the emitter (kernels_emit.cu).  RC / CR need 128 x 32 tiles and beta <= 4.
enum TileProg : int32_t {
  PROG_ZERO = 0, PROG_SAME = 1, PROG_RC = 2, PROG_CR = 3, PROG_MIXED = 4, PROG_GENERAL = 5,
  PROG_DIAG = 6, PROG_AFF = 7,
};

struct TileDev {
  int32_t mat;          // index of the output matrix (clique) this tile belongs to
  int32_t row0, nrows;  // local row range
  int32_t col0, ncols;  // local column range
  int32_t grow0;        // global z index of the first row
  int32_t gcol0;        // global z index of the first column
  uint32_t flags;
  int32_t rblk, cblk;   // block of the rows / columns when TF_UNIFORM
  int32_t prog;         // TileProg
};

// A strip of the fill kernel, self-contained (one 64 B load, no dependent look-ups at CTA start).
struct alignas(16) StripDev {
  long long out_off;  // offset (doubles) of the output matrix inside one query's output
  long long goff;     // offset of block rblk's Gram inside one query's Gram scratch (SAME / DIAG)
  int32_t ld, row0, nrows, col0;
  int32_t ncols, grow0, gcol0, prog;
  int32_t rblk, rl0, cl0, ldG;  // block-local index of output row r is rl0 + r, of column col0 + c is cl0 + c
};
static_assert(sizeof(StripDev) == 64, "StripDev must be 64 bytes");

struct MatDev {
  int64_t out_off;  // offset (doubles) of this matrix inside one query's output
  int32_t n;        // side
  int32_t ld;       // leading dimension (= n)
};

// ---------------------------------------------------------------------------------
// packed output (NNSDP_FORMAT_PACKED): the block-sparse upper triangle of Z.  Every clique block is a principal
// submatrix of Z and the cliques cover its non-zeros, so one query's record holds each structurally non-zero
// region of Z ONCE, as a list of column-major cells (ld = nrows) at fixed offsets:
//   WINDOW  rows of block b against block b+1 (the W' M window and the band corner)        always written
//   DIAG    the interior of the diagonal block of a hidden layer (Gram | W_K' S22 W_K, with its band); written
//           only for a query whose layer has a stably-active neuron (b <= K-2) / whose output QC has an S22 part
//   BAND    (beta+1) x m: band[t + (beta+1) i] = Z[g0+i, g0+i+t] inside the DIAG cell's range              always
//   RECT    everything else that can be non-zero (affine column, slivers, x_1 block, x_1/x_K coupling)    always
// Cells that are always written come first in the record; the DIAG cells follow.
// ---------------------------------------------------------------------------------
enum PackedKind : int32_t { PK_WINDOW = 1, PK_DIAG = 2, PK_BAND = 3, PK_RECT = 4 };
struct PackedCell {
  int32_t kind, blk;       // blk: b of WINDOW(b, b+1) / DIAG(b) / BAND(b); -1 for RECT
  int64_t grow0, gcol0;    // global 0-based z index of the first row / column (BAND: of Z[g0, g0])
  int64_t nrows, ncols;
  int64_t offset;          // doubles from the start of the record
  int32_t always;
};
struct PackedLayout {
  std::vector<PackedCell> cells;
  int64_t record_doubles = 0;   // size of one query's record
  int64_t always_doubles = 0;   // the always-written cells occupy [0, always_doubles)
  int64_t always_entries = 0;   // output entries the emitter writes for every query
  std::vector<int32_t> diag_cell;     // per block (K entries): index of its DIAG cell or -1
  std::vector<int64_t> diag_entries;  // per block: entries the fill strips of its DIAG cell write when present
};
// One job of the band kernel: the band |jr - jc| <= beta inside the square range of a diagonal block that the fill
// strips of one output matrix cover.  Two ways to get the band right, chosen per plan (PlanHost::band_inline):
//   inline    (narrow layers) the DIAG strips add the band term to the entries they store; jobs exist only for
//             the BAND cells of packed records;
//   separate  (wide layers) the strips store the bulk only and the band kernel, which runs after the fill kernel,
//             re-writes the band entries in place (ld > 0) -- the strips then need no per-entry test.
struct BandDev {
  long long out_off;    // offset of the output matrix (dense formats) / of the DIAG cell (packed) inside one query
  long long band_off;   // packed records: offset of the BAND cell; -1 in the dense formats
  int ld, row0, col0;   // in-place patch: leading dimension (0 = none) and local position of the range's first entry
  int g0, m, blk;       // first z index of the range, its side, the block
  int optional;         // packed records: the matrix is a DIAG cell, patched only when present for the query
  int upper_only;       // packed records: entries with row <= column only
};

struct PlanHost {
  std::vector<StripDev> strips;  // fill class, built from tiles[0 .. n_fill)
  std::vector<TileDev> tiles;
  std::vector<MatDev> mats;
  int64_t per_query_doubles = 0;
  int tile_rows = 0, tile_cols = 0;
  std::vector<BandDev> bands;    // jobs of the band kernel
  bool band_inline = true;       // see BandDev
  int n_fill = 0, n_window = 0, n_edge = 0;  // tiles are sorted by kernel class
  bool skip_absent = false;  // packed plans of wide nets: the fill strips of an absent DIAG cell are not written
  // Dense formats of wide nets (separate band handling, window programs available): the work items of the fill and the
  // window kernel as one list sorted by (matrix, 32-column panel, first column, first row) -- fill strips as they are,
  // window tiles re-packed into the strip layout (prog = PROG_RC / PROG_CR, rl0 = cblk, cl0 = flags, ldG = matrix order).
  // Empty when the plan keeps the two kernels.
  std::vector<StripDev> panel;
};

// ---------------------------------------------------------------------------------
// host gather plan: how one query's dense output reaches caller-owned host memory without moving
// structural zeros over PCIe.  Every output matrix is cut at block boundaries into cells; a cell is
//   DENSE_ALWAYS  W' M windows (rows of block b against the neurons of layer b+1, and the transpose),
//   DENSE_GRAM    diagonal block of a layer whose Gram is non-zero for this query (value dependent),
//   DENSE_S22     the x_K block when the output QC has an S22 part,
// (copied as one strided DMA each) or it is not dense: then it is zero-filled by host threads and its
// few possibly non-zero entries (band, slivers, affine row / column: the "thin" list) are packed on the
// device, copied contiguously and scattered by the host.
// ---------------------------------------------------------------------------------
enum GatherKind : int32_t { GK_NONE = 0, GK_ALWAYS = 1, GK_GRAM = 2, GK_S22 = 3 };
constexpr int GATHER_MIN_RECT = 256;  // smaller cells are never worth a strided DMA of their own

struct GatherCell {
  int32_t row0, nrows;  // local rows
  int32_t kind, blk;    // GatherKind; block of a GK_GRAM cell
  int32_t pure_zero;    // no term of Z can be non-zero in the cell (and no thin entry lies in it)
  int32_t ncols_hint, col0_hint;  // copy of the owning column segment's extent
};
struct GatherColSeg {   // a block-aligned range of columns of one matrix and its cells top to bottom
  int32_t mat, col0, ncols;
  std::vector<GatherCell> cells;
};
struct GatherPlan {
  bool usable = false;                 // false: copy the dense output (small nets)
  std::vector<GatherColSeg> colsegs;   // ordered by matrix
  std::vector<int32_t> colseg_begin;   // per matrix: first colseg (size nmats + 1)
  std::vector<int64_t> thin_idx;       // offsets (doubles) inside one query's output, ascending per matrix
  std::vector<int64_t> thin_begin;     // per matrix: first thin entry (size nmats + 1)
  int64_t dense_always_doubles = 0;    // statistics
};

// tile_rows in {32, 64, 128}; classify = false marks every tile TF_ALL (validation mode).
// packed != nullptr: mats must be the single matrix 1:Zdim; the plan then keeps only the tiles of the upper
// triangle that can be non-zero and addresses them inside the cells of *packed (PlanHost::mats = the cells).
int32_t build_plan(const Shape& sh, int64_t beta, const std::vector<CliqueRanges>& mats,
                   bool classify, PlanHost* plan, PackedLayout* packed = nullptr);
// Expands one packed record into dense matrices Z[C, C] (both triangles) for the index sets in mats, back to
// back (the dense formats of the ABI).  present: one byte per cell of the layout.
void unpack_record(const Shape& sh, int64_t beta, const PackedLayout& lay, const std::vector<CliqueRanges>& mats,
                   const double* record, const uint8_t* present, double* out);
int32_t build_gather_plan(const Shape& sh, int64_t beta, const std::vector<CliqueRanges>& mats,
                          const PlanHost& plan, GatherPlan* gp);

// ---------------------------------------------------------------------------------
// device-side descriptors (passed by value to kernels)
// ---------------------------------------------------------------------------------
struct NetDev {
  int K, n_in, n_out, Zdim, acdim, xtot;
  const int* n;               // K+1
  const int* off;             // K+1
  const int* xoff;            // K+2
  const int* blk_of;          // Zdim : block of every z index (K for the affine index)
  const double* const* M;     // K   : [W_k b_k], ld = n[k+1]              (neuron-contiguous)
  const double* const* Wt;    // K   : W_k' (n[k] x n[k+1]), ld = ldT[k]   (input-contiguous, zero padded)
  const int* ldT;             // K   : n[k] rounded up to 128
  const double* bias_all;     // acdim : b_1..b_{K-1} stacked
};

// Per-batch device arrays.  Strides are in doubles between queries (0 = shared).
struct BatchDev {
  int Q, beta;
  int out_kind, has_s22, has_s12;
  int sdim;
  long long lamdim;
  // inputs
  const double* x1min;   long long s_x1min;
  const double* x1max;   long long s_x1max;
  const double* ymin;    long long s_ymin;
  const double* ymax;    long long s_ymax;
  const double* smin;    long long s_smin;
  const double* smax;    long long s_smax;
  const double* gin;     long long s_gin;
  const double* gbnd;    long long s_gbnd;
  const double* gsec;    long long s_gsec;
  const double* outS;    long long s_outS;
  const double* outvec;  long long s_outvec;
  const double* outinvP; long long s_outinvP;
  const double* gout;    long long s_gout;
  // prepared per-query vectors (stride = natural size)
  double* d11;     // acdim                 -2 smin smax lambda
  double* Md;      // acdim                 (smin+smax) lambda + T[j,j]
  double* T0;      // acdim                 T[j,j]
  double* Bt;      // beta * acdim          Bt[(t-1)*acdim + i] = T[i, i+t]
  double* u;       // acdim                 d11 b + c13
  double* aff;     // Zdim                  the affine column Z[:, a]
  double* part;    // npart                 per-CTA partial sums of Z[a, a]
  int npart;
  int* act;        // acdim                 compacted local indices of Gram-active neurons, per layer
  int* cnt;        // K                     cnt[b] = active neurons among the rows of M[b]
  double* Z11;     // n_in * n_in           S11 - 2 diag(gamma_in)
  double* Z1K;     // n_in * n[K-1]         S12 W_K
  double* U;       // n_out * n[K-1]        S22 W_K
};

struct GramDev {
  double* scratch;           // nslots * per_query
  long long per_query;       // doubles
  const long long* goff;     // K : offset of block b's Gram inside one query's scratch (b <= K-2)
  const int* ldG;            // K : leading dimension of block b's Gram
  int mirror;                // write G[c, r] as well as G[r, c] (dense formats; packed records read the upper triangle only)
};

struct PlanDev {
  const StripDev* strips;    // n_strips fill strips stored for every query of a pass (no ZERO strips, no bulk strips)
  const StripDev* bulk;      // dense formats: the SAME / DIAG strips that only the (slot, block) pairs of a pass store
  int n_strips;
  const TileDev* tiles;
  const MatDev* mats;
  const StripDev* panel_desc;  // n_panel work items of the panel-ordered launch: AFF strips as they are; window tiles re-packed
                             // (prog = PROG_RC / PROG_CR, rblk, rl0 = cblk, cl0 = flags, ldG = matrix order)
  int n_panel;               // 0: fill and window kernels run one after the other
  int ntiles;                // tiles are sorted: [fill | window | edge]
  int n_fill, n_window, n_edge;
  int tile_rows;
  long long per_query;       // doubles per query in the output
  const void* tmaps;         // K tensor maps (CUtensorMap, 128 B each) of the W matrices for the CR window program, or null
  const int* tmap_ok;        // K : layer k has a usable tensor map
  int packed;                // packed records: fill strips of an absent DIAG cell are skipped
  int band_inline;           // DIAG strips add the band term themselves (else the band kernel patches it in)
};

// ---------------------------------------------------------------------------------
// kernel launchers (each returns the number of kernels it launched, < 0 on error)
// ---------------------------------------------------------------------------------
// K1: one IBP layer for Q boxes: y = W+ x- + W- x+ + b (and the mirrored bound); optional ReLU.
int ibp_layer_launch(const double* Mk, int n_out_k, int n_in_k, const double* xin_min,
                     const double* xin_max, long long x_stride, double* xout_min, double* xout_max,
                     double* acx_min, double* acx_max, long long acx_stride, int Q, int relu,
                     int write_x, int* flag_bad, cudaStream_t st);
// affine column: aff[r] += sum_j Wt[r, j] u[j]  (batched over queries)
int affine_layer_launch(const double* Wt, int ldT, int n_rows, int n_neurons, const double* u,
                        long long u_stride, double* aff, long long aff_stride, int Q,
                        cudaStream_t st);
// Few queries: every affine-column GEMV of the net in one launch / the whole interval propagation (+ sector
// slopes) as one cooperative kernel.  Return 0 when not applicable (the caller falls back to per-layer launches).
int affine_all_launch(const NetDev& nd, int K, int max_rows, const double* u, long long u_stride, double* aff,
                      long long aff_stride, int Q, cudaStream_t st);
int ibp_all_launch(const NetDev& nd, int max_out, const double* x1min, long long s_min, const double* x1max,
                   long long s_max, double* xmin, double* xmax, long long x_stride, double* acxmin, double* acxmax,
                   double* smin, double* smax, long long acx_stride, int Q, int* flag_bad, cudaStream_t st);
// C (+)= A B on the FP64 tensor cores (kernels_dgemm.cu); 0 = operands not suitable, the caller falls back.
int dgemm_dmma_launch(const double* A, int lda, int M, int K, const double* B, long long ldb, double* C, long long ldc,
                      int N, int accumulate, cudaStream_t st);
// interval propagation of one wide layer for many boxes on the FP64 tensor cores; 0 = not applicable
int ibp_dmma_launch(const double* Mk, int n_out_k, int n_in_k, const double* xin_min, const double* xin_max,
                    long long x_stride, double* xout_min, double* xout_max, double* acx_min, double* acx_max,
                    long long acx_stride, int Q, int relu, int write_x, int* flag_bad, cudaStream_t st);
// the affine-column products of all layers in one tensor-core launch (wide layers, many queries); 0 = not applicable
int dgemm_dmma_affine_layers_launch(const NetDev& nd, int b0, int nb, int max_rows, const double* u, long long u_stride,
                                    double* aff, long long aff_stride, int Q, cudaStream_t st);
int ibp_chain_launch(const NetDev& nd, int max_w, const double* x1min, long long s_min, const double* x1max,
                     long long s_max, double* xmin, double* xmax, long long x_stride, double* acxmin, double* acxmax,
                     double* smin, double* smax, long long acx_stride, int Q, int* flag_bad, cudaStream_t st);
// K2: smin/smax from acx bounds.
int launch_sector_minmax(long long n, const double* acxmin, const double* acxmax, double* smin,
                         double* smax, cudaStream_t st);
int launch_place_x1(const double* x1min, long long s_min, const double* x1max, long long s_max,
                    double* xmin, double* xmax, long long xtot, int n_in, int Q, cudaStream_t st);
// transposed, zero-padded copy of W_k out of [W_k b_k]
int launch_transpose_w(const double* Mk, int n_out_k, int n_in_k, double* Wt, int ldT,
                       cudaStream_t st);
// K2b: per-query QC diagonals, band multipliers, affine column, Gram active sets.
int launch_prep(const NetDev& net, const BatchDev& b, int* err_flag, cudaStream_t st);
// K3: Gram contractions (DMMA) for queries [q0, q0+nq) into scratch slots 0..nq-1.
// pairs: npairs active (query, block) pairs (two ints each) with q0 <= query < q0 + ring slots; scratch slot = query - q0
int launch_gram(const NetDev& net, const BatchDev& b, const GramDev& g, int max_n, int q0, const int* pairs,
                int npairs, cudaStream_t st);
// One (slot, diagonal block) pair of a pass whose SAME / DIAG strips are stored: bulk strips [first, first + count).
struct BulkItem {
  int32_t slot, first, count;
};
constexpr int BULK_PER_LAUNCH = 512;  // pairs per launch, passed by value (6 KB of kernel parameters)
struct BulkSel {
  int32_t n;
  BulkItem item[BULK_PER_LAUNCH];
};
// K4+K5: emit the tiles of queries [q0, q0+nq) to out + slot * per_query, slot = q - q0: every launched strip and tile
// for every query, the bulk strips for the nsel pairs of sel.  Structural zeros are never stored.
// which: -1 = the whole pass (fill, window, edge kernels back to back); 0 / 1 / 2 = one of them (0 holds the bulk strips).
int launch_emit(const NetDev& net, const BatchDev& b, const GramDev& g, const PlanDev& plan,
                int q0, int nq, double* out, cudaStream_t st, int which, const BulkItem* sel, int nsel);

// affine-coefficient mode (kernels_affine.cu): device view of one query's QC data and of the cover
struct AffineDev {
  long long nvar, var_out, var_bnd, var_sec;  // variable layout: [gin | gout | gbnd | gsec]
  long long acdim, lamdim, beta;
  int out_kind;
  const double *x1min, *x1max, *ymin, *ymax, *smin, *smax;  // one query
  const long long* col_ptr;  // Zdim + 1 : first cover entry of every column (upper triangle, column-major)
  const int* lo;             // Zdim     : first row of column c inside the cover
};
int launch_affine_count(const NetDev& net, const AffineDev& A, long long* counts, cudaStream_t st);
int launch_affine_fill(const NetDev& net, const AffineDev& A, const long long* offs, long long* ent,
                       long long* var, double* val, cudaStream_t st);
int launch_affine_z0(const NetDev& net, const BatchDev& b, const AffineDev& A, double* z0,
                     cudaStream_t st);

// matrix-free lambda_max (kernels_eig.cu); Qc = queries of the current chunk, first one is q_first
int launch_eig_init(double* v, int Zdim, int Qc, int q_first, cudaStream_t st);
int launch_eig_mid(const NetDev& net, const BatchDev& b, int q_first, int Qc, const double* x,
                   const double* t, double* s1, double* y, cudaStream_t st);
int launch_eig_io(const NetDev& net, const BatchDev& b, int q_first, int Qc, const double* x, double* y,
                  cudaStream_t st);
int launch_eig_multidot(const double* V, const double* w, int n, int Qc, int nv, double* c, int c_ld,
                        cudaStream_t st);
int launch_eig_project(const double* V, double* w, int n, int Qc, int nv, const double* c, int c_ld,
                       cudaStream_t st);
int launch_eig_normalize(const double* w, double* dst, int n, int Qc, double* nrm, cudaStream_t st);
// C (M x N, column q at C + q * ldc) += A (M x Kdim, column-major, lda) * B (column q at B + q * ldb)
int gemm_acc_launch(const double* A, int lda, int M, int Kdim, const double* B, long long ldb,
                    double* C, long long ldc, int N, cudaStream_t st);
// the same with C = A * B
int gemm_set_launch(const double* A, int lda, int M, int Kdim, const double* B, long long ldb,
                    double* C, long long ldc, int N, cudaStream_t st);

// CROWN bounds (kernels_crown.cu): rows of lA / uA of a chunk of Qc queries are stacked [2][Qc][Rs][ld]; a kernel
// works on nrows rows starting at row slot row0 of every (half, query) group (Rs = nrows, row0 = 0 for one target)
int launch_crown_params(const double* l, const double* u, long long stride, int n, int Qc, double* d_u,
                        double* b_u, double* d_l, cudaStream_t st);
// x_intvs of the hidden layers from the finished pre-activation bounds and relaxations (n stacked neurons per query)
int launch_crown_post(const double* prel, const double* preu, const double* d_u, const double* b_u, const double* d_l,
                      long long par_stride, int n, int Qc, double* out_lo, double* out_hi, long long out_stride,
                      cudaStream_t st);
int launch_crown_row(const double* srcL, const double* srcU, long long src_row_stride, long long src_q_stride,
                     double* dst, long long dst_row_stride, int nrows, int Qc, int n, const double* d_u,
                     const double* b_u, const double* d_l, long long par_stride, const double* bias_k,
                     double* bias, cudaStream_t st);
// relaxation through relu_k + bias updates + product with W_k in one launch (replaces launch_crown_row + GEMM)
int launch_crown_step(const double* Wt, int ldT, int M, int Kdim, const double* srcL, const double* srcU,
                      long long src_row_stride, long long src_q_stride, double* dst, long long ld, int nrows, int Rs,
                      int Qc, const double* d_u, const double* b_u, const double* d_l, long long par_stride,
                      const double* bias_k, double* bias, cudaStream_t st);
int launch_crown_init_bias(const double* bt, int nrows, int Qc, double* bias, cudaStream_t st);
int launch_crown_init_post(const double* Wt, int ldT, int n_in_k, const double* bias_k, const double* d_u,
                           const double* b_u, const double* d_l, long long par_stride, double* dst,
                           long long dst_row_stride, int nrows, int Rs, int row0, int Qc, double* bias,
                           cudaStream_t st);
int launch_crown_chain(const NetDev& net, int t, int post, int ntargets, int maxw, int Qc, const double* d_u,
                       const double* b_u, const double* d_l, long long par_stride, const double* x1min, long long s_min,
                       const double* x1max, long long s_max, int q_first, double* out_lo, double* out_hi,
                       long long out_stride, cudaStream_t st);
int launch_crown_concretize(const double* rowsL, const double* rowsU, long long row_stride, long long q_stride,
                            int nrows, int Rs, int row0, int Qc, int n0, const double* x1min, long long s_min,
                            const double* x1max, long long s_max, int q_first, const double* bias, double* out_lo,
                            double* out_hi, long long out_stride, int postprocess, cudaStream_t st);

// band jobs (in-place band of the DIAG ranges, BAND cells of packed records) for queries [q0, q0+nq); after the fill kernel
int launch_emit_band(const NetDev& net, const BatchDev& b, const GramDev& g, const BandDev* bands, int nbands,
                     int max_m, long long per_query, int q0, int nq, double* out, cudaStream_t st);
// thin-entry pack: packed[s * nthin + i] = ring[s * per_query + idx[i]] for the nq slots of a chunk
int launch_pack_thin(const double* ring, long long per_query, const long long* idx, long long nthin,
                     double* packed, int nq, cudaStream_t st);

constexpr int PREP_THREADS = 256;
constexpr int STRIP_ROWS = 512, STRIP_COLS = 8;  // fill-class strips (plan.cpp, emit_fill_kernel)
constexpr int AFFROW_COLS = 1024;                // columns of one affine-row job
constexpr int MAX_WINDOW_BETA = 4;  // RC / CR register-window programs are instantiated for beta <= 4
constexpr int MAX_FAST_BETA = 8;  // uniform-tile fast path of the emitter stages 2*beta+1 <= 17 band taps

}  // namespace nnsdp
