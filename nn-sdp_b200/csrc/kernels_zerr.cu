// Bound on the rounding error of the assembly of Z (nnsdp_batch_assembly_error, DESIGN.md section 9).
//
// Every entry Z[r,c] is a sum of monomials in the raw inputs (weights, biases, box, QC bounds, gamma, output QC).  With
// abs[r,c] the sum of the monomials' absolute values (oracle/exact_z.py), the FP64 Z the library emits satisfies
// |Z_dev[r,c] - Z(gamma)[r,c]| <= gamma_N abs[r,c] + N 2^-1074 entrywise (DESIGN.md section 2).  These kernels compute,
// for every query, s[r] >= sum_c abs[r,c] matrix free: the structure of the Lanczos matvec (kernels_eig.cu) applied to
// the all-ones vector, every factor replaced by its monomial-wise absolute value, built from the raw inputs (never
// from the rounded composite vectors d11, Md, aff, ... of kernels_prep.cu).  Every operand is non-negative and every
// operation rounds up (__dadd_ru, __dmul_ru, __fma_ru), so each s[r] is an upper bound by construction.
//
// Notation (all absolute values): for neuron j of layer L, rho_j = sum_c |W_L[j, c]| (the x block of layer L's inputs),
// D_j = 2 smin smax lambda, C_j = smin eta + smax nu, Td_j = sum of |v| of the pairs holding j, V_t[i] = |v| of the pair
// (i, i+t), Mrow_j = (smin + smax) lambda + 2 Td_j (= row sum of |M| = diag(smin lambda + smax lambda + Td) + |T_off|),
// uabs_j = D_j b_j + C_j.  Then
//   x row r of block L-1:   sum_j |W[j,r]| (D_j rho_j + Mrow_j + uabs_j)        Gram + F(r, .) + affine entry
//   neuron row j:           sum_{|j'-j|<=beta} m(j', j) (rho_j' + b_j') + 4 Td_j + 2 gbnd_j + te_j
//                           (F(c, r) transposed, the band, the affine entry te_j + sum b_j' m(j', j))
//   x_1 rows, x_K rows:     Zin, S11, S12 W_K, W_K' S22 W_K and their affine entries (zerr_io_kernel)
//   row a:                  the sum of the affine column plus Z[a, a].
#include <float.h>

#include "internal.h"

namespace nnsdp {

namespace {

constexpr int ZE_THREADS = ZERR_THREADS;
constexpr int ZE_TR = 64, ZE_TQ = 64, ZE_TK = 16;  // tile of the |W|' G products: rows x queries x neurons

__device__ __forceinline__ double add_up(double a, double b) { return __dadd_ru(a, b); }
__device__ __forceinline__ double mul_up(double a, double b) { return __dmul_ru(a, b); }
__device__ __forceinline__ double fma_up(double a, double b, double c) { return __fma_ru(a, b, c); }
// max that keeps a NaN (fmax would drop it): a non-finite class maximum must make the bound infinite
__device__ __forceinline__ double max_nan(double a, double b) { return (a != a || b != b) ? NAN : fmax(a, b); }

// same pair ordering as kernels_prep.cu (activ_sector.jl:29)
__device__ __forceinline__ long long pair_base_ze(long long i, long long acdim, long long beta) {
  long long m = acdim - beta;
  if (m < 0) m = 0;
  if (i <= m) return i * beta;
  return m * beta + (i - m) * (acdim - 1) - ((m + i - 1) * (i - m)) / 2;
}

// Per row of every layer (the acdim hidden neurons, then the n_out output rows): rho = sum_c |W[row, c]| and the
// largest |W[row, c]|, |b_row|.  netv = [rho (acdim + n_out) | rowmax (acdim + n_out) | wmax (1)].
__global__ void __launch_bounds__(ZE_THREADS) zerr_net_kernel(NetDev net, double* __restrict__ netv) {
  const long long nr = (long long)net.acdim + net.n_out;
  const long long i = (long long)blockIdx.x * ZE_THREADS + threadIdx.x;
  if (i >= nr) return;
  int L, l;
  if (i < net.acdim) {
    L = net.blk_of[net.n_in + i];
    l = (int)(net.n_in + i - net.off[L]);
  } else {
    L = net.K;
    l = (int)(i - net.acdim);
  }
  const int nrow = net.n[L], ncol = net.n[L - 1];
  const double* M = net.M[L - 1];
  double s = 0.0, mx = fabs(M[l + (long long)ncol * nrow]);
  for (int c = 0; c < ncol; ++c) {
    const double w = fabs(M[l + (long long)c * nrow]);
    s = add_up(s, w);
    mx = max_nan(mx, w);
  }
  netv[i] = s;
  netv[nr + i] = mx;
}

__global__ void __launch_bounds__(ZE_THREADS) zerr_wmax_kernel(long long nr, double* __restrict__ netv) {
  __shared__ double red[ZE_THREADS];
  double m = 0.0;
  for (long long i = threadIdx.x; i < nr; i += ZE_THREADS) m = max_nan(m, netv[nr + i]);
  red[threadIdx.x] = m;
  __syncthreads();
  for (int s = ZE_THREADS / 2; s > 0; s >>= 1) {
    if (threadIdx.x < s) red[threadIdx.x] = max_nan(red[threadIdx.x], red[threadIdx.x + s]);
    __syncthreads();
  }
  if (threadIdx.x == 0) netv[2 * nr] = red[0];
}

// One thread per neuron j of query q: the neuron row's sum (=: rows), the vector g_j = D_j rho_j + Mrow_j + uabs_j of
// the x-row products, and per CTA (fixed tree) the neuron terms of row a and the class maxima of the underflow factor:
// part[4 (q npart + blk) + {0, 1, 2, 3}] = {row a, max gamma, max |ymin|, |ymax|, max smin, smax}.
__global__ void __launch_bounds__(ZE_THREADS)
zerr_neuron_kernel(NetDev net, BatchDev b, const double* __restrict__ netv, double* __restrict__ g,
                   double* __restrict__ rows, double* __restrict__ part, int npart, int q_base) {
  const int q = q_base + blockIdx.y;
  const long long acdim = net.acdim, beta = b.beta;
  const long long j = (long long)blockIdx.x * ZE_THREADS + threadIdx.x;
  double ra = 0.0, mg = 0.0, my = 0.0, ms = 0.0;
  if (j < acdim) {
    const double* gsec = b.gsec + q * b.s_gsec;
    const double* v = gsec + acdim;
    const double* bias = net.bias_all;
    const double* rho = netv;
    const double sm = fabs(b.smin[q * b.s_smin + j]), sx = fabs(b.smax[q * b.s_smax + j]);
    const double y0 = fabs(b.ymin[q * b.s_ymin + j]), y1 = fabs(b.ymax[q * b.s_ymax + j]);
    const double gb = fabs(b.gbnd[q * b.s_gbnd + j]);
    const double lam = fabs(gsec[j]);
    const double eta = fabs(gsec[b.lamdim + j]), nu = fabs(gsec[b.lamdim + acdim + j]);
    const double bj = fabs(bias[j]), rj = rho[j];
    mg = max_nan(max_nan(max_nan(lam, eta), max_nan(nu, gb)), 0.0);
    my = max_nan(y0, y1);
    ms = max_nan(sm, sx);
    // the band: Td_j and the neighbours' terms m(j', j) (rho_j' + b_j') of the neuron row
    double td = 0.0, nb = 0.0;
    const long long base_j = pair_base_ze(j, acdim, beta);
    for (long long t = 1; t <= beta; ++t) {
      if (j + t < acdim) {
        const double vv = fabs(v[base_j + t - 1]);
        mg = max_nan(mg, vv);
        td = add_up(td, vv);
        nb = fma_up(vv, add_up(rho[j + t], fabs(bias[j + t])), nb);
      }
      if (j - t >= 0) {
        const double vv = fabs(v[pair_base_ze(j - t, acdim, beta) + t - 1]);
        td = add_up(td, vv);
        nb = fma_up(vv, add_up(rho[j - t], fabs(bias[j - t])), nb);
      }
    }
    const double d = mul_up(2.0, mul_up(mul_up(sm, sx), lam));                       // |d11| = 2 smin smax lambda
    const double c = add_up(mul_up(sm, eta), mul_up(sx, nu));                        // |c13|
    const double mdiag = add_up(add_up(mul_up(sm, lam), mul_up(sx, lam)), td);      // |M[j, j]|
    const double mrow = add_up(mdiag, td);                                           // sum_c |M[j, c]|
    const double ua = fma_up(d, bj, c);                                              // |u_j|
    const double te = add_up(add_up(mul_up(gb, y0), mul_up(gb, y1)), add_up(eta, nu));
    // neuron row: F(c, r) transposed + affine entry (te + sum_j' b_j' m(j', j)) + band (4 Td + 2 gbnd)
    double nr = fma_up(mdiag, add_up(rj, bj), nb);
    nr = add_up(nr, add_up(te, add_up(mul_up(4.0, td), mul_up(2.0, gb))));
    rows[(long long)q * net.Zdim + net.n_in + j] = nr;
    g[(long long)q * acdim + j] = add_up(fma_up(d, rj, mrow), ua);
    // row a: the affine entries of this neuron's row (te_j + b_j Mrow_j), of the x rows it feeds (rho_j uabs_j), and
    // its monomials of Z[a, a]: 2 gbnd ymin ymax + D b b + 2 b C
    ra = add_up(fma_up(bj, mrow, te), mul_up(rj, ua));
    ra = add_up(ra, mul_up(2.0, mul_up(mul_up(gb, y0), y1)));
    ra = add_up(ra, mul_up(mul_up(d, bj), bj));
    ra = add_up(ra, mul_up(2.0, mul_up(bj, c)));
  }
  __shared__ double red[4][ZE_THREADS];
  red[0][threadIdx.x] = ra;
  red[1][threadIdx.x] = mg;
  red[2][threadIdx.x] = my;
  red[3][threadIdx.x] = ms;
  __syncthreads();
  for (int s = ZE_THREADS / 2; s > 0; s >>= 1) {
    if (threadIdx.x < s) {
      red[0][threadIdx.x] = add_up(red[0][threadIdx.x], red[0][threadIdx.x + s]);
      for (int k = 1; k < 4; ++k) red[k][threadIdx.x] = max_nan(red[k][threadIdx.x], red[k][threadIdx.x + s]);
    }
    __syncthreads();
  }
  if (threadIdx.x < 4) part[4 * ((long long)q * npart + blockIdx.x) + threadIdx.x] = red[threadIdx.x][0];
}

// rows[q][roff + r] += sum_k |Wt[r + k ldT]| g[q][goff + k] for the n_rows x rows of one block: a SIMT product tiled over
// (rows, queries), every fma rounded up (the FP64 tensor cores have no directed rounding).
__global__ void __launch_bounds__(ZE_THREADS)
zerr_gemv_kernel(const double* __restrict__ Wt, int ldT, int n_rows, int nk, const double* __restrict__ g,
                 long long g_ld, long long goff, double* __restrict__ rows, long long rows_ld, long long roff, int Q,
                 int q_base) {
  __shared__ double Ws[ZE_TK][ZE_TR];
  __shared__ double Gs[ZE_TK][ZE_TQ];
  const int tid = threadIdx.x, tr = tid & 15, tq = tid >> 4;
  const int r0 = blockIdx.x * ZE_TR;
  const int q0 = q_base + blockIdx.y * ZE_TQ;
  double acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int k = 0; k < 4; ++k) acc[i][k] = 0.0;
  for (int k0 = 0; k0 < nk; k0 += ZE_TK) {
#pragma unroll
    for (int i = 0; i < ZE_TK * ZE_TR / ZE_THREADS; ++i) {
      const int e = tid + i * ZE_THREADS, kk = e / ZE_TR, r = e % ZE_TR;
      // Wt is zero padded to ldT >= every tile's last row
      Ws[kk][r] = (k0 + kk < nk) ? fabs(Wt[(r0 + r) + (long long)(k0 + kk) * ldT]) : 0.0;
    }
#pragma unroll
    for (int i = 0; i < ZE_TK * ZE_TQ / ZE_THREADS; ++i) {
      const int e = tid + i * ZE_THREADS, kk = e % ZE_TK, qq = e / ZE_TK;
      Gs[kk][qq] = (k0 + kk < nk && q0 + qq < Q) ? g[(long long)(q0 + qq) * g_ld + goff + k0 + kk] : 0.0;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < ZE_TK; ++kk) {
      double w[4], x[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) w[i] = Ws[kk][tr + 16 * i];
#pragma unroll
      for (int k = 0; k < 4; ++k) x[k] = Gs[kk][tq + 16 * k];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int k = 0; k < 4; ++k) acc[i][k] = fma_up(w[i], x[k], acc[i][k]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int q = q0 + tq + 16 * k;
    if (q >= Q) continue;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int r = r0 + tr + 16 * i;
      if (r < n_rows) {
        double* p = rows + (long long)q * rows_ld + roff + r;
        *p = add_up(*p, acc[i][k]);
      }
    }
  }
}

// One CTA per query: |S| of the output QC in the restatement's monomials (src/Qc/output.jl:52-98), the x_1 rows (=),
// the output terms of the x_K rows (+=), their share of row a and of Z[a, a].  io[4 q + {0, 1, 2, 3}] = {row a,
// max gamma (gamma_in, gamma_out), max |x1min|, |x1max|, max |output QC data|}.
__global__ void __launch_bounds__(ZE_THREADS)
zerr_io_kernel(NetDev net, BatchDev b, const double* __restrict__ netv, double* __restrict__ rows,
               double* __restrict__ io) {
  extern __shared__ double sh[];
  const int q = blockIdx.x, tid = threadIdx.x;
  const int K = net.K, n_in = net.n_in, n_out = net.n_out, sdim = b.sdim, nK = net.n[K - 1], oK = net.off[K - 1];
  double* S = sh;                  // sdim * sdim |S|, column-major
  double* w = S + sdim * sdim;     // n_out: colsum |S12| + |S22| (rhoK + |bK|) + |S23|
  double* t = w + n_out;           // n_out: |S22| |bK| + |S23|
  double* red = t + n_out;         // ZE_THREADS
  const double* rhoK = netv + net.acdim;
  const double* MK = net.M[K - 1];
  const double* bK = MK + (long long)nK * n_out;
  const int i2 = n_in, i3 = n_in + n_out;
  double mo = 0.0, mg = 0.0;
  for (int i = tid; i < sdim * sdim; i += ZE_THREADS) S[i] = 0.0;
  __syncthreads();
  if (b.out_kind == NNSDP_OUT_SAFETY) {
    const double* Sq = b.outS + q * b.s_outS;
    for (int i = tid; i < sdim * sdim; i += ZE_THREADS) {
      const int r = i % sdim, c = i / sdim;
      S[i] = fabs((r <= c) ? Sq[r + c * sdim] : Sq[c + r * sdim]);
      mo = max_nan(mo, S[i]);
    }
  } else {
    const double* vec = b.outvec + q * b.s_outvec;
    const double gout = fabs(b.gout[q * b.s_gout]);
    mg = gout;
    for (int o = tid; o < n_out; o += ZE_THREADS) mo = max_nan(mo, fabs(vec[o]));
    if (b.out_kind == NNSDP_OUT_HPLANE) {
      for (int o = tid; o < n_out; o += ZE_THREADS) S[(i2 + o) + i3 * sdim] = S[i3 + (i2 + o) * sdim] = fabs(vec[o]);
      if (tid == 0) S[i3 + i3 * sdim] = mul_up(2.0, gout);
    } else {
      const double* invP = b.outinvP + q * b.s_outinvP;
      const bool ell = (b.out_kind == NNSDP_OUT_ELLIPSOID);
      if (ell)
        for (int i = tid; i < n_out * n_out; i += ZE_THREADS) mo = max_nan(mo, fabs(invP[i]));
      for (int i = tid; i < n_out * n_out; i += ZE_THREADS) {
        const int r = i % n_out, c = i / n_out;
        double s22 = (r == c) ? 1.0 : 0.0;  // circle: I
        if (ell) {                         // |invP|' |invP|
          s22 = 0.0;
          for (int m = 0; m < n_out; ++m) s22 = fma_up(fabs(invP[m + r * n_out]), fabs(invP[m + c * n_out]), s22);
        }
        S[(i2 + r) + (i2 + c) * sdim] = s22;
      }
      for (int o = tid; o < n_out; o += ZE_THREADS) {
        double s23 = fabs(vec[o]);  // circle: |yc|
        if (ell) {                  // |invP|' |yc|
          s23 = 0.0;
          for (int m = 0; m < n_out; ++m) s23 = fma_up(fabs(invP[m + o * n_out]), fabs(vec[m]), s23);
        }
        S[(i2 + o) + i3 * sdim] = S[i3 + (i2 + o) * sdim] = s23;
      }
      if (tid == 0) {
        double yy = gout;  // yc'yc + gamma_out
        for (int m = 0; m < n_out; ++m) yy = fma_up(fabs(vec[m]), fabs(vec[m]), yy);
        S[i3 + i3 * sdim] = yy;
      }
    }
  }
  __syncthreads();
  for (int m = tid; m < n_out; m += ZE_THREADS) {
    double cs = 0.0, tm = S[(i2 + m) + i3 * sdim];
    for (int i = 0; i < n_in; ++i) cs = add_up(cs, S[i + (i2 + m) * sdim]);
    double sr = 0.0;
    for (int o = 0; o < n_out; ++o) {
      const double s22 = S[(i2 + m) + (i2 + o) * sdim];
      sr = fma_up(s22, rhoK[o], sr);
      tm = fma_up(s22, fabs(bK[o]), tm);
    }
    t[m] = tm;
    w[m] = add_up(add_up(cs, sr), tm);
  }
  __syncthreads();
  const double* gin = b.gin + q * b.s_gin;
  const double* x1min = b.x1min + q * b.s_x1min;
  const double* x1max = b.x1max + q * b.s_x1max;
  double* rq = rows + (long long)q * net.Zdim;
  double ra = 0.0, mx = 0.0;
  // x_1 rows: 2 gamma_in + S11 + S12 W_K, and the affine entry gamma_in (|x1min| + |x1max|) + S12 b_K + S13
  for (int i = tid; i < n_in; i += ZE_THREADS) {
    const double gi = fabs(gin[i]), lo = fabs(x1min[i]), hi = fabs(x1max[i]);
    mg = max_nan(mg, gi);
    mx = max_nan(mx, max_nan(lo, hi));
    double aff = add_up(add_up(mul_up(gi, lo), mul_up(gi, hi)), S[i + i3 * sdim]);
    double s = mul_up(2.0, gi);
    for (int c = 0; c < n_in; ++c) s = add_up(s, S[i + c * sdim]);
    for (int m = 0; m < n_out; ++m) {
      const double s12 = S[i + (i2 + m) * sdim];
      s = fma_up(s12, rhoK[m], s);
      aff = fma_up(s12, fabs(bK[m]), aff);
    }
    rq[i] = add_up(s, aff);
    ra = add_up(ra, add_up(aff, mul_up(2.0, mul_up(mul_up(gi, lo), hi))));  // + its monomial of Z[a, a]
  }
  // x_K rows: += sum_m |W_K[m, c]| w_m
  for (int c = tid; c < nK; c += ZE_THREADS) {
    const double* wc = MK + (long long)c * n_out;
    double s = 0.0;
    for (int m = 0; m < n_out; ++m) s = fma_up(fabs(wc[m]), w[m], s);
    rq[oK + c] = add_up(rq[oK + c], s);
  }
  // row a: sum_c of the x_K affine entries = sum_m rhoK_m t_m; Z[a, a] output part b_K' |S22| b_K + 2 b_K' |S23| + S33
  if (tid == 0) {
    double s = S[i3 + i3 * sdim];
    for (int m = 0; m < n_out; ++m) {
      double sb = 0.0;
      for (int o = 0; o < n_out; ++o) sb = fma_up(S[(i2 + m) + (i2 + o) * sdim], fabs(bK[o]), sb);
      s = fma_up(rhoK[m], t[m], s);
      s = fma_up(fabs(bK[m]), add_up(sb, mul_up(2.0, S[(i2 + m) + i3 * sdim])), s);
    }
    ra = add_up(ra, s);
  }
  const double vals[4] = {ra, mg, mx, mo};
  for (int k = 0; k < 4; ++k) {
    red[tid] = vals[k];
    __syncthreads();
    for (int s = ZE_THREADS / 2; s > 0; s >>= 1) {
      if (tid < s) red[tid] = k == 0 ? add_up(red[tid], red[tid + s]) : max_nan(red[tid], red[tid + s]);
      __syncthreads();
    }
    if (tid == 0) io[4 * q + k] = red[0];
    __syncthreads();
  }
}

// One CTA per query: row a, the largest row sum and e_q = up(gN max_r s[r]) + up(uf F_q) (+inf if anything is not finite).
// F_q = 4 max(1, W)^2 max(1, s)^2 max(1, gamma) max(1, box)^2 max(1, O)^2 bounds the factors a monomial applies after an
// underflow (DESIGN.md section 9).
__global__ void __launch_bounds__(ZE_THREADS)
zerr_final_kernel(int Zdim, const double* __restrict__ netv, long long nr, const double* __restrict__ part, int npart,
                  const double* __restrict__ io, double gN, double uf, double* __restrict__ rows,
                  double* __restrict__ err) {
  __shared__ double red[ZE_THREADS];
  __shared__ int bad_any;
  const int q = blockIdx.x, tid = threadIdx.x;
  double* rq = rows + (long long)q * Zdim;
  const int a = Zdim - 1;
  if (tid == 0) bad_any = 0;
  __syncthreads();
  double m = 0.0;
  int bad = 0;
  for (int r = tid; r < a; r += ZE_THREADS) {
    const double s = rq[r];
    bad |= !(s <= DBL_MAX);
    m = fmax(m, s);
  }
  if (bad) atomicOr(&bad_any, 1);
  red[tid] = m;
  __syncthreads();
  for (int s = ZE_THREADS / 2; s > 0; s >>= 1) {
    if (tid < s) red[tid] = fmax(red[tid], red[tid + s]);
    __syncthreads();
  }
  if (tid == 0) {
    const double* p = part + 4 * (long long)q * npart;
    const double* iq = io + 4 * (long long)q;
    double ra = iq[0], mg = iq[1], mb = iq[2], mo = iq[3], ms = 0.0;
    for (int i = 0; i < npart; ++i) {
      ra = add_up(ra, p[4 * i]);
      mg = max_nan(mg, p[4 * i + 1]);
      mb = max_nan(mb, p[4 * i + 2]);
      ms = max_nan(ms, p[4 * i + 3]);
    }
    rq[a] = ra;
    const double mrow = fmax(red[0], ra);
    const double fw = max_nan(1.0, netv[2 * nr]), fs = max_nan(1.0, ms), fg = max_nan(1.0, mg);
    const double fb = max_nan(1.0, mb), fo = max_nan(1.0, mo);
    double F = mul_up(4.0, mul_up(fw, fw));
    F = mul_up(F, mul_up(fs, fs));
    F = mul_up(F, fg);
    F = mul_up(F, mul_up(fb, fb));
    F = mul_up(F, mul_up(fo, fo));
    const double e = add_up(mul_up(gN, mrow), mul_up(uf, F));
    err[q] = (bad_any || !(ra <= DBL_MAX) || !(e <= DBL_MAX)) ? INFINITY : e;
  }
}

}  // namespace

int launch_zerr_net(const NetDev& net, double* netv, cudaStream_t st) {
  const long long nr = (long long)net.acdim + net.n_out;
  zerr_net_kernel<<<(unsigned)((nr + ZE_THREADS - 1) / ZE_THREADS), ZE_THREADS, 0, st>>>(net, netv);
  zerr_wmax_kernel<<<1, ZE_THREADS, 0, st>>>(nr, netv);
  return 2;
}

int launch_zerr_query(const NetDev& net, const BatchDev& b, const Shape& sh, const double* const* Wt, const int* ldT,
                      const double* netv, double* g, double* rows, double* part, double* io, double gN, double uf,
                      double* err, cudaStream_t st) {
  int launches = 0;
  const int npart = (int)((sh.acdim + ZE_THREADS - 1) / ZE_THREADS);
  for (int q_base = 0; q_base < b.Q; q_base += 65535) {
    zerr_neuron_kernel<<<dim3(npart, std::min(65535, b.Q - q_base)), ZE_THREADS, 0, st>>>(net, b, netv, g, rows, part,
                                                                                          npart, q_base);
    ++launches;
  }
  const size_t shbytes = (size_t)(b.sdim * b.sdim + 2 * sh.n_out() + ZE_THREADS) * sizeof(double);
  if (shbytes > 40000)  // the host checks sdim <= 160 (nnsdp_batch_create)
    cudaFuncSetAttribute(zerr_io_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)shbytes);
  zerr_io_kernel<<<b.Q, ZE_THREADS, shbytes, st>>>(net, b, netv, rows, io);
  ++launches;
  // the x rows of blocks 0 .. K-2 (after zerr_io_kernel has written the x_1 rows)
  for (int blk = 0; blk <= sh.K - 2; ++blk)
    for (int q_base = 0; q_base < b.Q; q_base += 65535 * ZE_TQ) {
      const int nq = std::min(65535 * ZE_TQ, b.Q - q_base);
      zerr_gemv_kernel<<<dim3((unsigned)((sh.n[blk] + ZE_TR - 1) / ZE_TR), (nq + ZE_TQ - 1) / ZE_TQ), ZE_THREADS, 0, st>>>(
          Wt[blk], ldT[blk], (int)sh.n[blk], (int)sh.n[blk + 1], g, sh.acdim, sh.noff(blk + 1), rows, sh.Zdim, sh.off[blk],
          b.Q, q_base);
      ++launches;
    }
  zerr_final_kernel<<<b.Q, ZE_THREADS, 0, st>>>((int)sh.Zdim, netv, sh.acdim + sh.n_out(), part, npart, io, gN, uf,
                                                rows, err);
  return launches + 1;
}

}  // namespace nnsdp
