// K4 + K5: emission of the dense FP64 output matrices -- the clique blocks Z[C_k, C_k] of the
// chordal decomposition (reference: Ec(Ck) Z Ec(Ck)' for the cliques of
// src/Methods/chordal_cliques.jl:13-59, the blocks setupZksum! scatters at
// src/Methods/chordal_sdp.jl:60-93) or the whole Z (src/Methods/chordal_sdp.jl:114,145).
//
// Z is never materialised: every output entry is evaluated from the closed form
//   Z[r,c] = [same block] (G_b[r,c] | Z11 | W_K' S22 W_K)  +  [x_1 / x_K] S12 W_K
//          + F(r,c) + F(c,r)  +  [band] (-2 T[jr,jc] - 2 gamma_bnd [jr == jc])
//   F(r,c) = sum_{j in layer(blk(r)+1), |j - jc| <= beta} W[j, r] M[j, jc],   M = diag(q lambda) + T
// (see DESIGN.md) and written once, column-major, with consecutive threads on consecutive rows.
// The kernel is HBM-write bound: 8 |C_k|^2 bytes per block.
//
// Every output matrix is cut into tiles (128 x 32 for wide nets); the host plan gives each tile a
// PROGRAM.  One CTA runs its tile for a whole group of queries (ring slots), so whatever depends
// on the network only -- the W tile of a window sum -- is loaded once and reused from registers /
// shared memory for every query of the group:
//   ZERO     structurally zero                                   -> not stored (the ring slot is zeroed once)
//   SAME     interior of a diagonal block (no band, no sliver)   -> copy of the Gram scratch, or fill
//   RC       rows x_b against neurons of layer b+1               -> (2 beta+1)-tap sliding window over
//                                                                   columns of W' held in registers
//   CR       the transposed case                                 -> window over rows of a W tile in smem
//   MIXED    any combination, rows/cols each inside one block    -> per-entry evaluation, hoisted tests
//   GENERAL  anything (small nets, affine row/column)            -> per-entry evaluation with block lookup
// All programs produce bit-identical values (same fma sequences, ascending neuron index).
#include <stdlib.h>

#include <algorithm>

#include "internal.h"

namespace nnsdp {

namespace {

constexpr int ETHREADS = 256;
constexpr int SLOT_GROUP = 8;   // queries handled by one CTA (edge kernel; default of the RC kernel)
constexpr int FAST_TR = 128, FAST_TC = 32, FAST_NCOL = 16;
constexpr int MAX_TAPS = 2 * MAX_FAST_BETA + 1;
constexpr int MAX_TC = 32;

struct QView {  // per-query pointers
  const double* Md;
  const double* T0;
  const double* Bt;
  const double* gbnd;
  const double* aff;
  const double* Z11;
  const double* Z1K;
  const double* U;
  const int* cnt;
  const double* G;
};

__device__ __forceinline__ QView make_view(const NetDev& net, const BatchDev& b, const GramDev& g,
                                           int q, int slot) {
  const long long acdim = net.acdim;
  const int K = net.K, n0 = net.n_in;
  QView v;
  v.Md = b.Md + (long long)q * acdim;
  v.T0 = b.T0 + (long long)q * acdim;
  v.Bt = b.Bt + (long long)q * b.beta * acdim;
  v.gbnd = b.gbnd + q * b.s_gbnd;
  v.aff = b.aff + (long long)q * net.Zdim;
  v.Z11 = b.Z11 + (long long)q * n0 * n0;
  v.Z1K = b.Z1K + (long long)q * n0 * net.n[K - 1];
  v.U = b.U + (long long)q * net.n_out * net.n[K - 1];
  v.cnt = b.cnt + (long long)q * K;
  v.G = g.scratch + (long long)slot * g.per_query;
  return v;
}

// M[j, c] = delta_jc q_j lambda_j + T[j, c],  |j - c| <= beta
__device__ __forceinline__ double m_coef(const double* Md, const double* Bt, long long acdim, int j,
                                         int c) {
  if (j == c) return Md[j];
  const int t = j > c ? j - c : c - j;
  return Bt[(long long)(t - 1) * acdim + (j < c ? j : c)];
}

// Band term of neuron pair (jr, jc), |jr - jc| <= beta: -2 T[jr,jc] - 2 gamma_bnd [jr == jc].
// Written with non-contractible intrinsics so every program rounds it identically.
__device__ __forceinline__ double band_term(const double* T0, const double* gbnd, const double* Bt,
                                            long long acdim, int jr, int jc) {
  if (jr == jc) return __dadd_rn(__dmul_rn(-2.0, T0[jr]), __dmul_rn(-2.0, gbnd[jr]));
  const int d = jr > jc ? jr - jc : jc - jr;
  return __dmul_rn(-2.0, Bt[(long long)(d - 1) * acdim + (jr < jc ? jr : jc)]);
}

// ---------------------------------------------------------------------------------------------
// MIXED: uniform tile, every block-level decision hoisted, band coefficients staged in smem
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void emit_mixed(const NetDev& net, const BatchDev& b, const GramDev& g,
                                           const TileDev& t, const MatDev& mat, const QView& v,
                                           double* __restrict__ o, int tr, int cg, int ncg,
                                           double* smem) {
  const int K = net.K, n0 = net.n_in, beta = b.beta, ntap = 2 * beta + 1;
  const long long acdim = net.acdim;
  const uint32_t flags = t.flags;
  const int Br = t.rblk, Bc = t.cblk;
  const int rl0 = t.grow0 - net.off[Br], cl0 = t.gcol0 - net.off[Bc];
  const int jr0 = t.grow0 - n0, jc0 = t.gcol0 - n0;  // neuron index of the first row / column
  const bool same = (Br == Bc) && (flags & TF_SAME);
  const bool gram = same && Br <= K - 2 && v.cnt[Br] > 0;
  const bool z11 = same && Br == 0;
  const bool s22 = same && Br == K - 1 && b.has_s22;
  const bool k1a = (flags & TF_1K) && b.has_s12 && Br == 0 && Bc == K - 1;
  const bool k1b = (flags & TF_1K) && b.has_s12 && Bc == 0 && Br == K - 1;
  const bool rc = (flags & TF_RC) && Br <= K - 2 && Bc >= 1;
  const bool cr = (flags & TF_CR) && Bc <= K - 2 && Br >= 1;
  const bool band = (flags & TF_BAND) && Br >= 1 && Bc >= 1;
  const int Lr0 = rc ? net.off[Br + 1] - n0 : 0, nLr = rc ? net.n[Br + 1] : 0;
  const int Lc0 = cr ? net.off[Bc + 1] - n0 : 0, nLc = cr ? net.n[Bc + 1] : 0;
  double* coefRC = smem;
  double* coefCR = smem + MAX_TC * MAX_TAPS;

  __syncthreads();  // smem may still be read by the previous query of the group
  if (rc)
    for (int i = threadIdx.x; i < t.ncols * ntap; i += ETHREADS) {
      const int c = i / ntap, jc = jc0 + c, j = jc - beta + i % ntap;
      coefRC[i] = (j >= Lr0 && j < Lr0 + nLr) ? m_coef(v.Md, v.Bt, acdim, j, jc) : 0.0;
    }
  if (cr)
    for (int i = threadIdx.x; i < t.nrows * ntap; i += ETHREADS) {
      const int r = i / ntap, jr = jr0 + r, j = jr - beta + i % ntap;
      coefCR[i] = (j >= Lc0 && j < Lc0 + nLc) ? m_coef(v.Md, v.Bt, acdim, j, jr) : 0.0;
    }
  __syncthreads();
  if (tr >= t.nrows) return;

  const int rl = rl0 + tr, jr = jr0 + tr;
  const double* Gp = gram ? v.G + g.goff[Br] + rl : nullptr;
  const int ldG = gram ? g.ldG[Br] : 0;
  const double* WtR = rc ? net.Wt[Br] + rl : nullptr;
  const int ldTR = rc ? net.ldT[Br] : 0;
  const double* Wc0 = cr ? net.M[Bc] : nullptr;
  const double* WK = net.M[K - 1];
  const int n_out = net.n_out;
  // valid taps of the transposed term depend on the row only
  const int cr_lo = cr ? max(0, Lc0 - (jr - beta)) : 0;
  const int cr_hi = cr ? min(ntap - 1, Lc0 + nLc - 1 - (jr - beta)) : -1;
  const double* myCR = coefCR + tr * ntap;

  for (int c = cg; c < t.ncols; c += ncg) {
    const int cl = cl0 + c, jc = jc0 + c;
    double val = 0.0;
    if (gram) val += Gp[(long long)cl * ldG];
    if (z11) val += v.Z11[rl + cl * n0];
    if (s22) {
      // evaluated as (min, max) so that Z[r,c] and Z[c,r] are bit-identical
      const int lo = rl < cl ? rl : cl, hi = rl < cl ? cl : rl;
      double s = 0.0;
      for (int m = 0; m < n_out; ++m)
        s = fma(WK[m + (long long)lo * n_out], v.U[m + (long long)hi * n_out], s);
      val += s;
    }
    if (k1a) val += v.Z1K[rl + (long long)cl * n0];
    if (k1b) val += v.Z1K[cl + (long long)rl * n0];
    double f1 = 0.0, f2 = 0.0;
    if (rc) {
      const int jb = jc - beta;  // tap tt <-> neuron jb + tt
      const int lo = max(0, Lr0 - jb), hi = min(ntap - 1, Lr0 + nLr - 1 - jb);
      const double* w = WtR + (long long)(jb - Lr0) * ldTR;
      const double* cf = coefRC + c * ntap;
      for (int tt = lo; tt <= hi; ++tt) f1 = fma(w[(long long)tt * ldTR], cf[tt], f1);
    }
    if (cr) {
      const double* w = Wc0 + (long long)cl * nLc + (jr - beta - Lc0);
      for (int tt = cr_lo; tt <= cr_hi; ++tt) f2 = fma(w[tt], myCR[tt], f2);
    }
    val += f1 + f2;  // commutative: Z[r,c] and Z[c,r] come out bit-identical
    if (band) {
      const int d = jr > jc ? jr - jc : jc - jr;
      if (d <= beta) val = __dadd_rn(val, band_term(v.T0, v.gbnd, v.Bt, acdim, jr, jc));
    }
    o[(long long)c * mat.ld] = val;
  }
}

// ---------------------------------------------------------------------------------------------
// GENERAL: per-entry block lookup, every term tested per entry
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void emit_general(const NetDev& net, const BatchDev& b, const GramDev& g,
                                             const TileDev& t, const MatDev& mat, const QView& v,
                                             double* __restrict__ o, int tr, int cg, int ncg) {
  if (tr >= t.nrows) return;
  const int K = net.K, n0 = net.n_in, a = net.Zdim - 1, beta = b.beta;
  const long long acdim = net.acdim;
  const uint32_t flags = t.flags;
  const int gr = t.grow0 + tr;
  const int Br = net.blk_of[gr];
  const int rl = gr - (Br < K ? net.off[Br] : a);
  const int jr = (gr >= n0 && gr < a) ? gr - n0 : -1;
  // F(r,c): rows of block Br feed the neurons [Lr0, Lr0 + nLr) through M[Br]
  const bool r_feeds = (Br <= K - 2);
  const int Lr0 = r_feeds ? net.off[Br + 1] - n0 : 0;
  const int nLr = r_feeds ? net.n[Br + 1] : 0;
  const double* WtR = r_feeds ? net.Wt[Br] + rl : nullptr;
  const int ldTR = r_feeds ? net.ldT[Br] : 0;
  const double* WK = net.M[K - 1];
  const int n_out = net.n_out;

  for (int c = cg; c < t.ncols; c += ncg) {
    const int gc = t.gcol0 + c;
    double val = 0.0;
    if (gr == a || gc == a) {
      val = v.aff[gr == a ? gc : gr];
    } else {
      const int Bc = net.blk_of[gc];
      const int cl = gc - net.off[Bc];
      const int jc = gc >= n0 ? gc - n0 : -1;
      if ((flags & TF_SAME) && Br == Bc) {
        if (Br <= K - 2 && v.cnt[Br] > 0) val += v.G[g.goff[Br] + rl + (long long)cl * g.ldG[Br]];
        if (Br == 0) val += v.Z11[rl + cl * n0];
        if (Br == K - 1 && b.has_s22) {
          const int lo = rl < cl ? rl : cl, hi = rl < cl ? cl : rl;
          double s = 0.0;
          for (int m = 0; m < n_out; ++m)
            s = fma(WK[m + (long long)lo * n_out], v.U[m + (long long)hi * n_out], s);
          val += s;
        }
      }
      if ((flags & TF_1K) && b.has_s12) {
        if (Br == 0 && Bc == K - 1) val += v.Z1K[rl + (long long)cl * n0];
        if (Bc == 0 && Br == K - 1) val += v.Z1K[cl + (long long)rl * n0];
      }
      double f1 = 0.0, f2 = 0.0;
      if ((flags & TF_RC) && r_feeds && jc >= 0) {
        const int jlo = max(Lr0, jc - beta), jhi = min(Lr0 + nLr - 1, jc + beta);
        for (int j = jlo; j <= jhi; ++j)
          f1 = fma(WtR[(long long)(j - Lr0) * ldTR], m_coef(v.Md, v.Bt, acdim, j, jc), f1);
      }
      if ((flags & TF_CR) && Bc <= K - 2 && jr >= 0) {
        const int Lc0 = net.off[Bc + 1] - n0, nLc = net.n[Bc + 1];
        const double* Wc = net.M[Bc] + (long long)cl * nLc;  // column cl of W_Bc: neuron-contiguous
        const int jlo = max(Lc0, jr - beta), jhi = min(Lc0 + nLc - 1, jr + beta);
        for (int j = jlo; j <= jhi; ++j)
          f2 = fma(Wc[j - Lc0], m_coef(v.Md, v.Bt, acdim, j, jr), f2);
      }
      val += f1 + f2;
      if ((flags & TF_BAND) && jr >= 0 && jc >= 0) {
        const int d = jr > jc ? jr - jc : jc - jr;
        if (d <= beta) val = __dadd_rn(val, band_term(v.T0, v.gbnd, v.Bt, acdim, jr, jc));
      }
    }
    o[(long long)c * mat.ld] = val;
  }
}

// ---------------------------------------------------------------------------------------------
// RC: out[r, c] = sum_t Wt[r, jc - beta + t] * M[jc - beta + t, jc].  Thread = (row, 16 contiguous
// columns); the 16 + 2 beta values of W' it needs are loaded once (coalesced over rows) and reused
// for every query of the group.  M is a symmetric band, so the taps of a column are shifted reads of beta + 1
// vectors (value_0(i) = M[i, i], value_d(i) = M[i, i + d] = T[i, i + d]): they are staged per query as beta + 1
// rows in shared memory, read two columns at a time with 16-byte broadcast loads, and the values a later column
// needs again stay in registers -- (beta + 1) / 2 shared-memory loads per output instead of 2 beta + 1.
// The output pointer advances by one column per store (no per-entry address arithmetic); FULL = all 32 columns
// of the tile exist (no column predicate).
// ---------------------------------------------------------------------------------------------
template <int BETA, bool FULL>
__device__ __forceinline__ void emit_rc(const NetDev& net, const BatchDev& b, const PlanDev& plan,
                                        const TileDev& t, const MatDev& mat, int q0, int slot0,
                                        int nslots, double* __restrict__ out, double* smem) {
  constexpr int NTAP = 2 * BETA + 1;
  constexpr int PB = BETA + (BETA & 1);     // even, so that 16-byte loads stay aligned
  constexpr int RS = FAST_TC + PB;          // staged entries per vector: neurons jc0 - PB .. jc0 + 31
  constexpr int QS = (BETA + 1) * RS;       // doubles per query
  const int n0 = net.n_in;
  const long long acdim = net.acdim;
  const int Br = t.rblk;
  const int tr = threadIdx.x & (FAST_TR - 1), cg = threadIdx.x / FAST_TR;
  const int rl = t.grow0 - net.off[Br] + tr;
  const int jc0 = t.gcol0 - n0;
  const int Lr0 = net.off[Br + 1] - n0, nLr = net.n[Br + 1];

  for (int i = threadIdx.x; i < nslots * QS; i += ETHREADS) {
    const int s = i / QS, rem = i - s * QS, d = rem / RS, e = rem - d * RS;
    const long long idx = (long long)jc0 - PB + e;
    double v = 0.0;
    if (idx >= 0 && idx < acdim) {
      const long long q = q0 + slot0 + s;
      v = d == 0 ? b.Md[q * acdim + idx] : b.Bt[q * BETA * acdim + (long long)(d - 1) * acdim + idx];
    }
    smem[i] = v;
  }
  __syncthreads();
  if (tr >= t.nrows) return;

  const int cbase = cg * FAST_NCOL;
  // w[i] = W'[r, jc0 + cbase - beta + i]; zero outside the layer, which is what restricts the sum to the layer
  double w[FAST_NCOL + NTAP - 1];
  {
    const double* WtR = net.Wt[Br] + rl;
    const int ldTR = net.ldT[Br];
    const int jb = jc0 + cbase - BETA;
#pragma unroll
    for (int i = 0; i < FAST_NCOL + NTAP - 1; ++i) {
      const int j = jb + i;
      w[i] = (j >= Lr0 && j < Lr0 + nLr) ? WtR[(long long)(j - Lr0) * ldTR] : 0.0;
    }
  }
  const long long ld = mat.ld;
  double* o0 = out + (long long)slot0 * plan.per_query + mat.out_off + (t.row0 + tr) + (long long)(t.col0 + cbase) * ld;
  const int ncl = t.ncols - cbase;  // columns of this thread's strip that exist
  for (int s = 0; s < nslots; ++s, o0 += plan.per_query) {
    const double* cf = smem + s * QS + cbase;  // cf[d * RS + PB + c] = value_d(jc0 + cbase + c)
    double h[BETA + 1][BETA > 0 ? BETA : 1];   // h[d][k] = value_d(jc - d + k) of the current column, k < d
#pragma unroll
    for (int d = 1; d <= BETA; ++d)
#pragma unroll
      for (int k = 0; k < d; ++k) h[d][k] = cf[d * RS + PB - d + k];
    double* o = o0;
#pragma unroll
    for (int c = 0; c < FAST_NCOL; c += 2) {
      double x[BETA + 1], y[BETA + 1];
#pragma unroll
      for (int d = 0; d <= BETA; ++d) {
        const double2 v = *reinterpret_cast<const double2*>(cf + d * RS + PB + c);
        x[d] = v.x;
        y[d] = v.y;
      }
      double f = 0.0, g = 0.0;  // columns c and c + 1, taps in ascending neuron order
#pragma unroll
      for (int tt = 0; tt < BETA; ++tt) {
        f = fma(w[c + tt], h[BETA - tt][0], f);
        g = fma(w[c + 1 + tt], (BETA - tt >= 2) ? h[BETA - tt][1] : x[BETA - tt], g);
      }
      f = fma(w[c + BETA], x[0], f);
      g = fma(w[c + 1 + BETA], y[0], g);
#pragma unroll
      for (int d = 1; d <= BETA; ++d) {
        f = fma(w[c + BETA + d], x[d], f);
        g = fma(w[c + 1 + BETA + d], y[d], g);
      }
      if (FULL || c < ncl) o[0] = f;
      if (FULL || c + 1 < ncl) o[ld] = g;
      o += 2 * ld;
#pragma unroll
      for (int d = 1; d <= BETA; ++d)
#pragma unroll
        for (int k = 0; k < d; ++k) h[d][k] = (k + 2 < d) ? h[d][k + 2] : (k + 2 == d ? x[d] : y[d]);
    }
  }
}

__host__ __device__ constexpr int CR_LDW(int beta) { return FAST_TR + 2 * beta + 2; }

// ---- TMA (cp.async.bulk.tensor) staging of a W tile: one thread arms an mbarrier with the byte count and issues the
// 2-D bulk tensor copy; rows / columns outside the matrix arrive as zeros (out-of-bounds fill of the tensor map)
__device__ __forceinline__ void tma_load_tile_2d(double* smem_dst, unsigned long long* mbar, const void* tmap, int c0,
                                                 int c1, unsigned bytes) {
  const unsigned bar = (unsigned)__cvta_generic_to_shared(mbar);
  const unsigned dst = (unsigned)__cvta_generic_to_shared(smem_dst);
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;\n" ::"r"(bar));
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(bar), "r"(bytes) : "memory");
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];\n" ::"r"(dst),
        "l"(tmap), "r"(c0), "r"(c1), "r"(bar)
        : "memory");
  }
  __syncthreads();  // the barrier is initialised before anybody polls it
  unsigned done = 0, spins = 0;
  while (!done) {
    asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\nselp.u32 %0, 1, 0, p;\n}\n"
                 : "=r"(done)
                 : "r"(bar)
                 : "memory");
    if (!done && ++spins > (1u << 24)) __trap();  // a copy that never completes must fail the launch, not hang the device
  }
}

// ---------------------------------------------------------------------------------------------
// CR: out[jr, c] = sum_t W[jr - beta + t, c] * M[jr - beta + t, jr].  The (128 + 2 beta) x 32 tile of
// W (neuron-contiguous) is staged once in shared memory; the taps depend on the row only and live
// in registers per query.
// ---------------------------------------------------------------------------------------------
template <int BETA>
__device__ __forceinline__ void emit_cr(const NetDev& net, const BatchDev& b, const PlanDev& plan,
                                        const TileDev& t, const MatDev& mat, int q0, int slot0,
                                        int nslots, double* __restrict__ out, double* smem, unsigned long long* mbar) {
  constexpr int NTAP = 2 * BETA + 1;
  constexpr int LDW = CR_LDW(BETA);  // rows per staged column: 128 + 2 beta, + 2 so that a box can start on an even row
  const int n0 = net.n_in;
  const long long acdim = net.acdim;
  const int Bc = t.cblk;
  const int tr = threadIdx.x & (FAST_TR - 1), cg = threadIdx.x / FAST_TR;
  const int jr0 = t.grow0 - n0, jr = jr0 + tr;
  const int cl0 = t.gcol0 - net.off[Bc];
  const int Lc0 = net.off[Bc + 1] - n0, nLc = net.n[Bc + 1];
  int adj = 0;  // staged row ii holds neuron jr0 - BETA - adj + ii
  if (plan.tmaps && plan.tmap_ok[Bc]) {
    // The (128 + 2 beta + 2) x 32 box of W_Bc by TMA.  The start address of a box must be a multiple of 16 bytes
    // (an odd start row of doubles faults with "illegal instruction", tools/probe_tma.cu), so the box starts one row
    // early when jr0 - beta is odd; rows / columns outside the matrix arrive as zeros.
    const int c0 = jr0 - BETA - Lc0;
    adj = c0 & 1;
    tma_load_tile_2d(smem, mbar, (const char*)plan.tmaps + 128 * Bc, c0 - adj, cl0, (unsigned)(FAST_TC * LDW * 8));
  } else {
    const double* Wc0 = net.M[Bc] + (long long)cl0 * nLc;
    for (int i = threadIdx.x; i < t.ncols * LDW; i += ETHREADS) {
      const int c = i / LDW, ii = i - c * LDW;
      const int j = jr0 - BETA + ii;
      smem[i] = (j >= Lc0 && j < Lc0 + nLc) ? Wc0[(long long)c * nLc + (j - Lc0)] : 0.0;
    }
    __syncthreads();
  }
  if (tr >= t.nrows) return;
  const int cbase = cg * FAST_NCOL;
  const long long ld = mat.ld;
  double* o0 = out + (long long)slot0 * plan.per_query + mat.out_off + (t.row0 + tr) + (long long)(t.col0 + cbase) * ld;
  const int ncl = min(FAST_NCOL, t.ncols - cbase);
  const double* ws0 = smem + cbase * LDW + tr + adj;
  const double* Md = b.Md + (long long)(q0 + slot0) * acdim;
  const double* Bt = b.Bt + (long long)(q0 + slot0) * BETA * acdim;
  // two queries per trip: the 2 beta + 1 values of W a column needs are read from shared memory once for both
  const long long pq = plan.per_query;
  int s = 0;
  for (; s + 2 <= nslots; s += 2, o0 += 2 * pq, Md += 2 * acdim, Bt += 2 * BETA * acdim) {
    double cf0[NTAP], cf1[NTAP];
#pragma unroll
    for (int tt = 0; tt < NTAP; ++tt) {
      const int j = jr - BETA + tt;
      const bool in = j >= Lc0 && j < Lc0 + nLc;
      cf0[tt] = in ? m_coef(Md, Bt, acdim, j, jr) : 0.0;
      cf1[tt] = in ? m_coef(Md + acdim, Bt + BETA * acdim, acdim, j, jr) : 0.0;
    }
    double* o = o0;
    const double* ws = ws0;
    // (not fully unrolled on purpose: the W values do not depend on the query, and a fully unrolled column loop lets
    // the compiler hoist all of them out of the query loop -- spills)
#pragma unroll 4
    for (int c = 0; c < ncl; ++c, o += ld, ws += LDW) {
      double f0 = 0.0, f1 = 0.0;
#pragma unroll
      for (int tt = 0; tt < NTAP; ++tt) {
        const double w = ws[tt];
        f0 = fma(w, cf0[tt], f0);
        f1 = fma(w, cf1[tt], f1);
      }
      o[0] = f0;
      o[pq] = f1;
    }
  }
  if (s < nslots) {
    double cf[NTAP];
#pragma unroll
    for (int tt = 0; tt < NTAP; ++tt) {
      const int j = jr - BETA + tt;
      cf[tt] = (j >= Lc0 && j < Lc0 + nLc) ? m_coef(Md, Bt, acdim, j, jr) : 0.0;
    }
    double* o = o0;
    const double* ws = ws0;
#pragma unroll 4
    for (int c = 0; c < ncl; ++c, o += ld, ws += LDW) {
      double f = 0.0;
#pragma unroll
      for (int tt = 0; tt < NTAP; ++tt) f = fma(ws[tt], cf[tt], f);
      *o = f;
    }
  }
}

// ---- kernel 1: tiles whose bulk is a plain store stream; one (tile, query) per CTA -----------------
//   SAME  Gram copy | S22 Gram | fill
//   DIAG  SAME + the band term added to the entries with |jr - jc| <= beta as they are stored
//   AFF   the affine row / column Z[a, :], Z[:, a]
__device__ __forceinline__ double s22_entry(const double* WK, const double* U, int n_out, int rl, int cl) {
  const int lo = rl < cl ? rl : cl, hi = rl < cl ? cl : rl;  // (min, max): bit-symmetric
  double acc = 0.0;
  for (int m = 0; m < n_out; ++m)
    acc = fma(WK[m + (long long)lo * n_out], U[m + (long long)hi * n_out], acc);
  return acc;
}

// One strip (<= STRIP_ROWS x STRIP_COLS, or one wide affine-row job) for one query.  The 64 B descriptor is
// fetched with independent 16 B loads.  Structurally zero strips are never launched: a ring slot is zeroed once
// when it is first used and nothing else writes there (api.cu, prepare_slots).  Thread = row inside a TR-row
// chunk (x column group when the strip is short); for every column the chunks start on a 32 B sector boundary of the output (rows before the strip
// are masked), so each warp store covers whole sectors although ld is odd.  TR is a power of two.
#ifndef NNSDP_FILL_MINB
#define NNSDP_FILL_MINB 6
#endif
template <bool BAND_INLINE>  // DIAG strips add the band term themselves (narrow layers) or leave it to the band kernel
__device__ __forceinline__ void fill_strip(const NetDev& net, const BatchDev& b, const GramDev& g, const PlanDev& plan,
                                           const StripDev* desc, int slot, int q0, double* __restrict__ out) {
  const int4* dp = reinterpret_cast<const int4*>(desc);
  const int4 d0 = __ldg(dp), d1 = __ldg(dp + 1), d2 = __ldg(dp + 2);
  const int tid = threadIdx.x;
  const long long out_off = ((long long)(unsigned)d0.x) | ((long long)d0.y << 32);
  const long long ld = d1.x;
  const int row0 = d1.y, nrows = d1.z, col0 = d1.w, ncols = d2.x, prog = d2.w;
  const int row_end = row0 + nrows;
  double* o = out + (long long)slot * plan.per_query + out_off;  // base of the output matrix
  int lg = 5;
  while ((1 << lg) < ETHREADS && (1 << lg) < nrows + 3) ++lg;
  const int TR = 1 << lg;
  const int tr = tid & (TR - 1), cg = tid >> lg, ncg = ETHREADS >> lg;
  double* col = o + (col0 + cg) * ld;  // column cg of the strip; advanced by ncg columns per trip
  const long long cstep = (long long)ncg * ld;
#define NNSDP_STRIP_LOOP(VALUE)                                                     \
  for (int c = cg; c < ncols; c += ncg, col += cstep) {                               \
    int r = row0 - (int)(((size_t)(col + row0) >> 3) & 3) + tr;                       \
    if (r >= row0 && r < row_end) col[r] = (VALUE);                                   \
    for (r += TR; r < row_end; r += TR) col[r] = (VALUE);                             \
  }
  const int q = q0 + slot, K = net.K;
  const int grow0 = d2.y, gcol0 = d2.z;
  if (prog == PROG_AFF) {
    const double* aff = b.aff + (long long)q * net.Zdim;
    if (nrows == 1 && grow0 == net.Zdim - 1) {  // affine row Z[a, :], thread = column
      for (int c = tid; c < ncols; c += ETHREADS) o[row0 + (col0 + c) * ld] = aff[gcol0 + c];
    } else {  // affine column Z[:, a]
      aff += grow0 - row0;
      NNSDP_STRIP_LOOP(aff[r])
    }
    return;
  }
  // SAME / DIAG: rows and columns in block Br, 1 <= Br <= K-1
  const int4 d3 = __ldg(dp + 3);
  const int Br = d3.x, rl0 = d3.y, cl0 = d3.z, ldG = d3.w;  // block-local index of output row r is rl0 + r
  const long long goff = ((long long)(unsigned)d0.z) | ((long long)d0.w << 32);
  const bool copy = Br <= K - 2 && b.cnt[(long long)q * K + Br] > 0;  // Gram of an active layer
  const bool s22 = Br == K - 1 && b.has_s22;                           // W_K' S22 W_K of the output QC
  if (plan.packed && !copy && !s22) return;  // packed record: the DIAG cell of this block is absent for this query
  const double* WK = net.M[K - 1];
  const double* U = b.U + (long long)q * net.n_out * net.n[K - 1];
  const double* G = g.scratch + (long long)slot * g.per_query + goff + rl0;  // G[r + cl*ldG]
  if (BAND_INLINE && prog == PROG_DIAG) {
    // The strip crosses the band |jr - jc| <= beta: the entry is  (bulk) + (absent window terms) + band term, in the
    // operation order of the general programs; everywhere else the bulk value is stored as it is.
    const int beta = b.beta;
    const long long acdim = net.acdim;
    const int jr_base = grow0 - net.n_in - row0, jc0 = gcol0 - net.n_in;  // neuron of local row r: jr_base + r
    const double* T0 = b.T0 + (long long)q * acdim;
    const double* Bt = b.Bt + (long long)q * beta * acdim;
    const double* gbnd = b.gbnd + q * b.s_gbnd;
    const double* Gc = G + (long long)(cl0 + cg) * ldG;
    const long long gstep = (long long)ncg * ldG;
    for (int c = cg; c < ncols; c += ncg, col += cstep, Gc += gstep) {
      const int jc = jc0 + c;
      int r = row0 - (int)(((size_t)(col + row0) >> 3) & 3) + tr;
      for (; r < row_end; r += TR) {
        if (r < row0) continue;
        double v = copy ? Gc[r] : (s22 ? s22_entry(WK, U, net.n_out, rl0 + r, cl0 + c) : 0.0);
        const int d = jr_base + r - jc;
        if (d >= -beta && d <= beta) {
          v = 0.0 + v;
          v += 0.0;
          v = __dadd_rn(v, band_term(T0, gbnd, Bt, acdim, jc + d, jc));
        }
        col[r] = v;
      }
    }
  } else if (copy) {
    const double* Gc = G + (long long)(cl0 + cg) * ldG;
    const long long gstep = (long long)ncg * ldG;
    for (int c = cg; c < ncols; c += ncg, col += cstep, Gc += gstep) {
      int r = row0 - (int)(((size_t)(col + row0) >> 3) & 3) + tr;
      if (r >= row0 && r < row_end) col[r] = Gc[r];
      for (r += TR; r < row_end; r += TR) col[r] = Gc[r];
    }
  } else if (s22) {
    NNSDP_STRIP_LOOP(s22_entry(WK, U, net.n_out, rl0 + r, cl0 + c))
  } else {
    NNSDP_STRIP_LOOP(0.0)
  }
#undef NNSDP_STRIP_LOOP
}

template <bool BAND_INLINE>
__global__ void __launch_bounds__(ETHREADS, NNSDP_FILL_MINB)
emit_fill_kernel(NetDev net, BatchDev b, GramDev g, PlanDev plan, int q0, int nq,
                 double* __restrict__ out) {
  fill_strip<BAND_INLINE>(net, b, g, plan, plan.strips + blockIdx.x, blockIdx.y, q0, out);
}

// The SAME / DIAG strips of the (slot, block) pairs of `sel`: grid = (most strips of a block, pairs)
template <bool BAND_INLINE>
__global__ void __launch_bounds__(ETHREADS, NNSDP_FILL_MINB)
emit_fill_kernel(NetDev net, BatchDev b, GramDev g, PlanDev plan, int q0, BulkSel sel, double* __restrict__ out) {
  const BulkItem it = sel.item[blockIdx.y];
  if ((int)blockIdx.x >= it.count) return;
  fill_strip<BAND_INLINE>(net, b, g, plan, plan.bulk + it.first + blockIdx.x, it.slot, q0, out);
}

// ---- kernel 2: RC / CR window sums (128 x 32 tiles, beta <= 4) ------------------------------------
// One kernel for both programs: their CTAs interleave in plan order, so the rows a CR tile writes and the rows the
// RC tile of the same columns writes reach DRAM close in time (dense formats: a column of a clique block is
// written by several programs, and the write bandwidth depends on how soon its pieces follow each other).
template <int BETA>
__global__ void __launch_bounds__(ETHREADS, 4)
emit_window_kernel(NetDev net, BatchDev b, PlanDev plan, int tile0, int q0, int nq, int group, int group_major,
                   double* __restrict__ out) {
  constexpr int RC_DOUBLES = SLOT_GROUP * (BETA + 1) * (FAST_TC + BETA + 1), CR_DOUBLES = FAST_TC * CR_LDW(BETA);
  __shared__ __align__(128) double smem[RC_DOUBLES > CR_DOUBLES ? RC_DOUBLES : CR_DOUBLES];
  __shared__ __align__(8) unsigned long long mbar;
  // slot group is the fastest grid index: CTAs that share a W tile run back to back (L2 reuse)
  const int ngroups = (nq + group - 1) / group;
  const int ti = group_major ? blockIdx.x % plan.n_window : blockIdx.x / ngroups;
  const int gi = group_major ? blockIdx.x / plan.n_window : blockIdx.x % ngroups;
  const TileDev t = plan.tiles[tile0 + ti];
  const MatDev mat = plan.mats[t.mat];
  const int slot0 = gi * group;
  const int nslots = min(group, nq - slot0);
  if (t.prog == PROG_RC) {
    if (t.ncols == FAST_TC) emit_rc<BETA, true>(net, b, plan, t, mat, q0, slot0, nslots, out, smem);
    else emit_rc<BETA, false>(net, b, plan, t, mat, q0, slot0, nslots, out, smem);
  } else {
    emit_cr<BETA>(net, b, plan, t, mat, q0, slot0, nslots, out, smem, &mbar);
  }
}

// ---- kernel 3: everything else (band / sliver / corner tiles, affine row and column, small nets) -
constexpr int EDGE_DOUBLES = MAX_TC * MAX_TAPS + 128 * MAX_TAPS;  // shared memory of emit_mixed

// One MIXED / GENERAL tile for the queries (ring slots) [slot0, slot0 + nslots)
__device__ __forceinline__ void emit_edge_tile(const NetDev& net, const BatchDev& b, const GramDev& g,
                                               const PlanDev& plan, const TileDev& t, const MatDev& mat, int q0,
                                               int slot0, int nslots, double* __restrict__ out, double* smem) {
  // thread = (row, column group); thin sliver tiles (2 x 32, 128 x 2, ...) spread their few entries over
  // as many threads as possible: rows per column group = smallest power of two covering the tile's rows
  int TR = 1;
  while (TR < t.nrows) TR <<= 1;
  if (TR > ETHREADS) TR = ETHREADS;
  const int tr = threadIdx.x % TR, cg = threadIdx.x / TR, ncg = ETHREADS / TR;
  const long long tile_off = mat.out_off + (t.row0 + tr) + (long long)t.col0 * mat.ld;
  // thin sliver tiles (a few hundred entries) skip the shared-memory staging and its barriers: the per-entry
  // evaluator with direct loads is cheaper there (same bits), and since it has no barrier the threads a thin
  // tile leaves idle work on other queries of the group at the same time
  const bool uniform = (t.flags & TF_UNIFORM) != 0 && t.nrows * t.ncols > 512;
  if (uniform) {
    for (int s = 0; s < nslots; ++s) {
      const QView v = make_view(net, b, g, q0 + slot0 + s, slot0 + s);
      double* o = out + (long long)(slot0 + s) * plan.per_query + tile_off;
      emit_mixed(net, b, g, t, mat, v, o, tr, cg, ncg, smem);
    }
    return;
  }
  int TC = 1;
  while (TC < t.ncols && TC < ncg) TC <<= 1;  // column groups one query needs
  const int per = TR * TC;                     // threads per query
  const int spar = ETHREADS / per;             // queries in flight
  const int sub = threadIdx.x / per, cg2 = (threadIdx.x % per) / TR;
  for (int s = sub; s < nslots; s += spar) {
    const QView v = make_view(net, b, g, q0 + slot0 + s, slot0 + s);
    double* o = out + (long long)(slot0 + s) * plan.per_query + tile_off;
    emit_general(net, b, g, t, mat, v, o, tr, cg2, TC);
  }
}

__global__ void __launch_bounds__(ETHREADS, 4)
emit_edge_kernel(NetDev net, BatchDev b, GramDev g, PlanDev plan, int tile0, int q0, int nq,
                 int group, double* __restrict__ out) {
  __shared__ double smem[EDGE_DOUBLES];
  const TileDev t = plan.tiles[tile0 + blockIdx.x];
  const MatDev mat = plan.mats[t.mat];
  const int slot0 = blockIdx.y * group;
  emit_edge_tile(net, b, g, plan, t, mat, q0, slot0, min(group, nq - slot0), out, smem);
}

// ---- kernels 1 + 2 (+ 3) as one launch in PANEL order (dense formats of wide nets) -----------------------------
// A column of a clique block is written by several programs: fill strips (affine pieces; the Gram pieces go out in
// their own launch, for the (slot, block) pairs that need them), window tiles and edge tiles (slivers, corners).  Launched one kernel after the
// other, the pieces of a column reach DRAM milliseconds apart and each launch covers only part of every DRAM page it
// touches (tools/probe_write_bw.cu: two launches 5.7 TB/s, one launch with the items ordered by 32-column panel
// 7.0 TB/s on pure stores).  Here the work items of both kernels are sorted by
// (matrix, 32-column panel, row) and consecutive CTAs take consecutive items, so whole columns are written within
// microseconds.  Inside a sub-batch of queries (see below) a window CTA writes its tile for `group` consecutive queries and
// a strip CTA its strip for every (batch / group)-th query.  FOLD: the list holds the edge tiles too, and the first CTA
// of an edge item writes its tile for every query of the sub-batch (the others have nothing to do): a stress pass takes
// 2.90 ms this way, 2.94 ms with the queries spread over the item's CTAs like a strip's, 3.00 ms with the separate edge
// launch (one B200).  Both forms store the same bits.
template <int BETA, bool FOLD>
__global__ void __launch_bounds__(ETHREADS, 4)
emit_panel_kernel(NetDev net, BatchDev b, GramDev g, PlanDev plan, int q0, int nq, int group, double* __restrict__ out) {
  constexpr int RC_DOUBLES = SLOT_GROUP * (BETA + 1) * (FAST_TC + BETA + 1), CR_DOUBLES = FAST_TC * CR_LDW(BETA);
  constexpr int WIN_DOUBLES = RC_DOUBLES > CR_DOUBLES ? RC_DOUBLES : CR_DOUBLES;
  static_assert(WIN_DOUBLES >= EDGE_DOUBLES, "the edge tiles stage their band coefficients in the same buffer");
  __shared__ __align__(128) double smem[WIN_DOUBLES];
  __shared__ __align__(8) unsigned long long mbar;
  // CTA order: the queries of a pass go in sub-batches of `batch` (a multiple of group): all items for the first
  // sub-batch, then all items for the next one.  Fewer queries in flight at a time = fewer DRAM pages open at a time:
  // a 16-query pass runs at 5.75 TB/s and an 8-query pass at 5.83 TB/s where a 32-query pass reaches 5.58 TB/s.
  const int batch = group >> 8;
  group &= 255;
  const int gb = batch / group;                         // CTAs per item and full sub-batch
  const int per_batch = plan.n_panel * gb;
  const int sb = blockIdx.x / per_batch, rem = blockIdx.x - sb * per_batch;
  const int slot_lo = sb * batch, slot_hi = min(nq, slot_lo + batch);
  const int item = rem / gb, g0 = rem - item * gb;
  // one self-contained 64 B descriptor per item, in panel order: a fill strip as it is, a window tile re-packed into
  // the same layout (no index -> tile -> matrix chain of dependent loads at the start of a short CTA)
  const StripDev* desc = plan.panel_desc + item;
  const int4* dp = reinterpret_cast<const int4*>(desc);
  const int4 d2 = __ldg(dp + 2);
  if (d2.w != PROG_RC && d2.w != PROG_CR && !(FOLD && (d2.w == PROG_MIXED || d2.w == PROG_GENERAL))) {
    for (int slot = slot_lo + g0; slot < slot_hi; slot += gb) fill_strip<false>(net, b, g, plan, desc, slot, q0, out);
    return;
  }
  if (FOLD && (d2.w == PROG_MIXED || d2.w == PROG_GENERAL) && g0 != 0) return;
  const int4 d0 = __ldg(dp), d1 = __ldg(dp + 1), d3 = __ldg(dp + 3);
  TileDev t;
  t.mat = 0;
  t.row0 = d1.y, t.nrows = d1.z, t.col0 = d1.w, t.ncols = d2.x, t.grow0 = d2.y, t.gcol0 = d2.z, t.prog = d2.w;
  t.rblk = d3.x, t.cblk = d3.y, t.flags = (uint32_t)d3.z;
  MatDev mat;
  mat.out_off = ((long long)(unsigned)d0.x) | ((long long)d0.y << 32);
  mat.ld = d1.x;
  mat.n = d3.w;
  if (FOLD && t.prog != PROG_RC && t.prog != PROG_CR) {
    emit_edge_tile(net, b, g, plan, t, mat, q0, slot_lo, slot_hi - slot_lo, out, smem);
    return;
  }
  const int slot0 = slot_lo + g0 * group;
  const int nslots = min(group, slot_hi - slot0);
  if (nslots <= 0) return;
  if (t.prog == PROG_RC) {
    if (t.ncols == FAST_TC) emit_rc<BETA, true>(net, b, plan, t, mat, q0, slot0, nslots, out, smem);
    else emit_rc<BETA, false>(net, b, plan, t, mat, q0, slot0, nslots, out, smem);
  } else {
    emit_cr<BETA>(net, b, plan, t, mat, q0, slot0, nslots, out, smem, &mbar);
  }
}

}  // namespace

// ---- the band |jr - jc| <= beta of the DIAG ranges: Z[r, c] = (Gram | S22 Gram | 0) + (absent window terms) +
// (-2 T[jr, jc] - 2 gamma_bnd [jr = jc]), the operation sequence of the general programs.  In place over what the
// fill strips stored (plans with separate band handling; stream order makes this kernel the last writer; packed
// records: only when the DIAG cell is present, upper triangle) and / or into the BAND cell of a packed record.
namespace {
__device__ __forceinline__ void band_entry(const NetDev& net, const BatchDev& b, const GramDev& g, const BandDev& bd,
                                           long long per_query, int q0, int slot, int idx, double* __restrict__ out) {
  const int q = q0 + slot, K = net.K, beta = b.beta, nt = 2 * beta + 1;
  if (idx >= bd.m * nt) return;
  const int i = idx / nt, t = idx - i * nt - beta, c = i + t;  // entry (i, c) of the range, |t| <= beta
  if (bd.upper_only && t < 0) return;
  double* o = out + (long long)slot * per_query;
  if (c < 0 || c >= bd.m) {  // outside the range: the BAND cell holds a zero there
    if (bd.band_off >= 0 && t >= 0) o[bd.band_off + t + (long long)(beta + 1) * i] = 0.0;
    return;
  }
  const int Br = bd.blk, n0 = net.n_in;
  const long long acdim = net.acdim;
  const int rl = bd.g0 - net.off[Br] + i, cl = rl + t;
  const int jr = bd.g0 + i - n0, jc = jr + t;
  const bool copy = Br <= K - 2 && b.cnt[(long long)q * K + Br] > 0;
  const bool s22 = Br == K - 1 && b.has_s22;
  double val = 0.0;
  if (copy) val += g.scratch[(long long)slot * g.per_query + g.goff[Br] + rl + (long long)cl * g.ldG[Br]];
  if (s22) val += s22_entry(net.M[K - 1], b.U + (long long)q * net.n_out * net.n[K - 1], net.n_out, rl, cl);
  val += 0.0;
  val = __dadd_rn(val, band_term(b.T0 + (long long)q * acdim, b.gbnd + q * b.s_gbnd, b.Bt + (long long)q * beta * acdim,
                                 acdim, jr, jc));
  if (bd.ld > 0 && (!bd.optional || copy || s22)) o[bd.out_off + (bd.row0 + i) + (long long)(bd.col0 + c) * bd.ld] = val;
  if (bd.band_off >= 0 && t >= 0) o[bd.band_off + t + (long long)(beta + 1) * i] = val;
}

__global__ void __launch_bounds__(ETHREADS)
emit_band_kernel(NetDev net, BatchDev b, GramDev g, const BandDev* __restrict__ bands, long long per_query, int q0,
                 int nq, int spc, double* __restrict__ out) {
  const BandDev bd = bands[blockIdx.y];
  const int idx = blockIdx.x * ETHREADS + threadIdx.x;
  // spc queries per CTA (one entry per thread and query): a 32-query stress pass is 47,360 CTAs of one query each
  for (int slot = blockIdx.z * spc; slot < min(nq, (blockIdx.z + 1) * spc); ++slot)
    band_entry(net, b, g, bd, per_query, q0, slot, idx, out);
}
}  // namespace

int launch_emit_band(const NetDev& net, const BatchDev& b, const GramDev& g, const BandDev* bands, int nbands,
                     int max_m, long long per_query, int q0, int nq, double* out, cudaStream_t st) {
  if (nbands <= 0 || nq <= 0 || max_m <= 0) return 0;
  const int nx = (max_m * (2 * b.beta + 1) + ETHREADS - 1) / ETHREADS;
  static const int spc_env = [] { const char* e = getenv("NNSDP_BAND_GROUP"); return e ? atoi(e) : 0; }();
  const int spc = spc_env > 0 ? spc_env : (nq >= 16 ? 4 : 1);
  emit_band_kernel<<<dim3(nx, nbands, (nq + spc - 1) / spc), ETHREADS, 0, st>>>(net, b, g, bands, per_query, q0, nq, spc, out);
  return 1;
}

namespace {
__global__ void pack_thin_kernel(const double* __restrict__ ring, long long per_query,
                                 const long long* __restrict__ idx, long long nthin,
                                 double* __restrict__ packed, int nq) {
  const long long total = nthin * nq;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long s = i / nthin, k = i - s * nthin;
    packed[i] = ring[s * per_query + idx[k]];
  }
}
}  // namespace

int launch_pack_thin(const double* ring, long long per_query, const long long* idx, long long nthin,
                     double* packed, int nq, cudaStream_t st) {
  if (nthin <= 0 || nq <= 0) return 0;
  long long blocks = (nthin * nq + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  pack_thin_kernel<<<(int)blocks, 256, 0, st>>>(ring, per_query, idx, nthin, packed, nq);
  return 1;
}

// The bulk strips of the (slot, block) pairs of one pass, BULK_PER_LAUNCH pairs per launch (kernel parameter space)
static int launch_bulk(const NetDev& net, const BatchDev& b, const GramDev& g, const PlanDev& plan, int q0,
                       const BulkItem* sel, int nsel, double* out, cudaStream_t st) {
  int launches = 0;
  for (int i0 = 0; i0 < nsel; i0 += BULK_PER_LAUNCH) {
    BulkSel s;
    s.n = std::min(BULK_PER_LAUNCH, nsel - i0);
    int most = 0;
    for (int i = 0; i < s.n; ++i) {
      s.item[i] = sel[i0 + i];
      most = std::max(most, s.item[i].count);
    }
    if (most == 0) continue;
    const dim3 grid((unsigned)most, (unsigned)s.n);
    if (plan.band_inline) emit_fill_kernel<true><<<grid, ETHREADS, 0, st>>>(net, b, g, plan, q0, s, out);
    else emit_fill_kernel<false><<<grid, ETHREADS, 0, st>>>(net, b, g, plan, q0, s, out);
    ++launches;
  }
  return launches;
}

int launch_emit(const NetDev& net, const BatchDev& b, const GramDev& g, const PlanDev& plan,
                int q0, int nq, double* out, cudaStream_t st, int which, const BulkItem* sel, int nsel) {
  if (nq <= 0) return 0;
  static const int wgroup = [] { const char* e = getenv("NNSDP_WINDOW_GROUP"); int v = e ? atoi(e) : 4; return v < 1 ? 1 : (v > SLOT_GROUP ? SLOT_GROUP : v); }();
  // queries per edge CTA: one when a pass holds few queries (wide nets, 8 ring slots), eight when it holds many
  static const int egroup_env = [] { const char* e = getenv("NNSDP_EDGE_GROUP"); int v = e ? atoi(e) : 0; return v < 0 ? 0 : (v > SLOT_GROUP ? SLOT_GROUP : v); }();
  const int egroup = egroup_env > 0 ? egroup_env : (nq >= 64 ? SLOT_GROUP : (nq >= 16 ? 4 : 1));  // 32-query stress pass: 0.168 / 0.129 / 0.115 / 0.110 ms with 1 / 2 / 4 / 8
  int launches = 0;
  if (plan.n_panel > 0 && b.beta <= MAX_WINDOW_BETA) {   // fill strips and window tiles as one launch in panel order
    if (which < 0 || which == 0) {
      // queries per window CTA (a strip CTA then writes its strip for every ngroups-th query): 2 is the measured best
      // (W1000-D20, 32-query pass: 7.57 ms against 7.75 ms with 4, 8.63 ms with 1; fill + window kernels 7.88 ms)
      static const int pgroup = [] { const char* e = getenv("NNSDP_PANEL_GROUP"); int v = e ? atoi(e) : 2; return v < 1 ? 1 : (v > SLOT_GROUP ? SLOT_GROUP : v); }();
      // queries per sub-batch of the launch (a multiple of pgroup)
      static const int pbatch_env = [] { const char* e = getenv("NNSDP_PANEL_BATCH"); return e ? atoi(e) : 8; }();
      int pbatch = std::max(pgroup, (pbatch_env / pgroup) * pgroup);
      if (pbatch > 255) pbatch = (255 / pgroup) * pgroup;
      const int nbatches = (nq + pbatch - 1) / pbatch;
      const dim3 grid((unsigned)plan.n_panel * (pbatch / pgroup) * nbatches);
      const int gp = pgroup | (pbatch << 8);
#define NNSDP_PANEL_LAUNCH(B)                                                                                  \
  if (plan.fold) emit_panel_kernel<B, true><<<grid, ETHREADS, 0, st>>>(net, b, g, plan, q0, nq, gp, out);      \
  else emit_panel_kernel<B, false><<<grid, ETHREADS, 0, st>>>(net, b, g, plan, q0, nq, gp, out);
      switch (b.beta) {
        case 0: NNSDP_PANEL_LAUNCH(0) break;
        case 1: NNSDP_PANEL_LAUNCH(1) break;
        case 2: NNSDP_PANEL_LAUNCH(2) break;
        case 3: NNSDP_PANEL_LAUNCH(3) break;
        default: NNSDP_PANEL_LAUNCH(4) break;
      }
#undef NNSDP_PANEL_LAUNCH
      ++launches;
    }
  } else {
  if (plan.n_strips > 0 && (which < 0 || which == 0)) {
    if (plan.band_inline) emit_fill_kernel<true><<<dim3(plan.n_strips, nq), ETHREADS, 0, st>>>(net, b, g, plan, q0, nq, out);
    else emit_fill_kernel<false><<<dim3(plan.n_strips, nq), ETHREADS, 0, st>>>(net, b, g, plan, q0, nq, out);
    ++launches;
  }
  if (plan.n_window > 0 && (which < 0 || which == 1)) {
    const dim3 grid(plan.n_window * ((nq + wgroup - 1) / wgroup));
    const int t0 = plan.n_fill;
    // CTA order: wide layers -- the query groups of a tile back to back (its W tile stays in L2); narrow layers (all
    // weights L2-resident) -- the tiles of a query group back to back (vertically adjacent tiles are contiguous in
    // memory): W100-D50 1.05 -> 0.96 ms per pass, W1000-D20 2.43 -> 2.67 ms the other way round
    static const int gm_env = [] { const char* e = getenv("NNSDP_WINDOW_GROUP_MAJOR"); return e ? atoi(e) : -1; }();
    const int gm = gm_env >= 0 ? gm_env : plan.band_inline;
    switch (b.beta) {
      case 0: emit_window_kernel<0><<<grid, ETHREADS, 0, st>>>(net, b, plan, t0, q0, nq, wgroup, gm, out); break;
      case 1: emit_window_kernel<1><<<grid, ETHREADS, 0, st>>>(net, b, plan, t0, q0, nq, wgroup, gm, out); break;
      case 2: emit_window_kernel<2><<<grid, ETHREADS, 0, st>>>(net, b, plan, t0, q0, nq, wgroup, gm, out); break;
      case 3: emit_window_kernel<3><<<grid, ETHREADS, 0, st>>>(net, b, plan, t0, q0, nq, wgroup, gm, out); break;
      case 4: emit_window_kernel<4><<<grid, ETHREADS, 0, st>>>(net, b, plan, t0, q0, nq, wgroup, gm, out); break;
      default: return -1;  // the plan never emits window tiles for beta > MAX_WINDOW_BETA
    }
    ++launches;
  }
  }
  if (which < 0 || which == 0) launches += launch_bulk(net, b, g, plan, q0, sel, nsel, out, st);
  if (!plan.fold && plan.n_edge > 0 && (which < 0 || which == 2)) {
    emit_edge_kernel<<<dim3(plan.n_edge, (nq + egroup - 1) / egroup), ETHREADS, 0, st>>>(
        net, b, g, plan, plan.n_fill + plan.n_window, q0, nq, egroup, out);
    ++launches;
  }
  return launches;
}

}  // namespace nnsdp
