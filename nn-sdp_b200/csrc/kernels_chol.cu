// Certificate eigmax(Z) <= tau (nnsdp_batch_certify): multifrontal Cholesky of tau' I - Z, in place in the ring slots
// of one emitter pass, batched over the queries of the pass (DESIGN.md section 9).  Per front (a clique block):
//   chol_front_init_kernel   tau' I - Z on the entries the front brings in, the previous front's Schur complement on
//                            the overlap (replacing, not adding: both fronts hold the same Z entries there)
// and per panel of CHOL_NB private columns:
//   chol_panel_kernel        Cholesky of the diagonal block in shared memory with the pivot check, then the TRSM of
//                            the rows below (one row per thread; every CTA of a query factorises the same small block)
//   chol_update_kernel       trailing lower triangle -= L21 L21' on the FP64 tensor cores (mma.sync.m8n8k4.f64, the
//                            fragment layout of kernels_dgemm.cu), 64 x 64 tiles on and below the diagonal
// Only the lower triangle is read or written.  A query whose pivot is not positive (or NaN) is marked failed and every
// later kernel skips it.  Nothing here uses atomics, so repeated calls give the same bits.
#include "internal.h"

#include <math.h>

namespace nnsdp {

namespace {

constexpr int NB = CHOL_NB;
constexpr int UT = 64;        // update tile side
constexpr int ULD = UT + 4;   // 4 (mod 16): a half warp's (k, m) fragment addresses fall in distinct banks
constexpr int PANEL_ROWS = 128;

__device__ __forceinline__ void dmma(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

__global__ void __launch_bounds__(256) chol_trace_kernel(const double* __restrict__ ring, long long per,
                                                         const CholFront* __restrict__ fronts, int nfronts,
                                                         double* __restrict__ stats) {
  const int s = blockIdx.x;
  const double* base = ring + (long long)s * per;
  double sum = 0.0, sabs = 0.0, mabs = 0.0;
  for (int k = 0; k < nfronts; ++k) {
    const CholFront f = fronts[k];
    for (int i = f.lead + threadIdx.x; i < f.n - f.tail; i += blockDim.x) {
      const double z = base[f.out_off + i + (long long)i * f.n];
      sum += z;
      sabs += fabs(z);
      mabs = fmax(mabs, fabs(z));
    }
  }
  __shared__ double r0[256], r1[256], r2[256];
  r0[threadIdx.x] = sum;
  r1[threadIdx.x] = sabs;
  r2[threadIdx.x] = mabs;
  __syncthreads();
  for (int h = 128; h > 0; h >>= 1) {
    if ((int)threadIdx.x < h) {
      r0[threadIdx.x] += r0[threadIdx.x + h];
      r1[threadIdx.x] += r1[threadIdx.x + h];
      r2[threadIdx.x] = fmax(r2[threadIdx.x], r2[threadIdx.x + h]);
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    stats[3 * s] = r0[0];
    stats[3 * s + 1] = r1[0];
    stats[3 * s + 2] = r2[0];
  }
}

// CTA = (column j, query): rows i >= j of column j
__global__ void __launch_bounds__(128) chol_front_init_kernel(double* __restrict__ ring, long long per, CholFront f,
                                                              CholFront pf, int has_prev, const double* __restrict__ taup,
                                                              const int* __restrict__ failed) {
  const int s = blockIdx.y, j = blockIdx.x;
  if (failed[s]) return;
  double* A = ring + (long long)s * per + f.out_off;
  const double* P = ring + (long long)s * per + pf.out_off;
  const double tp = taup[s];
  const bool jsep = has_prev && (j < f.lead || j >= f.n - f.tail);
  const int jp = j < f.lead ? j + pf.npriv : j - f.n + pf.n;
  for (int i = j + threadIdx.x; i < f.n; i += blockDim.x) {
    double* a = A + i + (long long)j * f.n;
    const bool isep = has_prev && (i < f.lead || i >= f.n - f.tail);
    if (jsep && isep) {
      const int ip = i < f.lead ? i + pf.npriv : i - f.n + pf.n;
      *a = P[ip + (long long)jp * pf.n];
    } else {
      *a = (i == j) ? tp - *a : -*a;
    }
  }
}

// grid (row blocks below the panel (>= 1), queries)
__global__ void __launch_bounds__(PANEL_ROWS) chol_panel_kernel(double* __restrict__ ring, long long per, CholFront f,
                                                                int j0, int w, int* __restrict__ failed,
                                                                long long* __restrict__ fail_index,
                                                                double* __restrict__ min_pivot) {
  const int s = blockIdx.y, tid = threadIdx.x;
  if (failed[s]) return;
  double* A = ring + (long long)s * per + f.out_off;
  const int n = f.n;
  __shared__ double D[NB][NB + 1];
  for (int e = tid; e < w * w; e += PANEL_ROWS) {
    const int r = e % w, c = e / w;
    D[r][c] = r >= c ? A[(j0 + r) + (long long)(j0 + c) * n] : 0.0;
  }
  __syncthreads();
  double pmin = INFINITY;
  for (int jj = 0; jj < w; ++jj) {
    const double d = D[jj][jj];
    if (!(d > 0.0)) {  // every thread reads the same value: the whole CTA leaves
      if (blockIdx.x == 0 && tid == 0) {
        failed[s] = 1;
        fail_index[s] = f.g0 + j0 + jj;
        min_pivot[s] = d;  // not above any earlier (positive) pivot
      }
      return;
    }
    pmin = fmin(pmin, d);
    const double r = sqrt(d);
    __syncthreads();
    if (tid == 0) D[jj][jj] = r;
    for (int i = jj + 1 + tid; i < w; i += PANEL_ROWS) D[i][jj] /= r;
    __syncthreads();
    const int m = w - jj - 1;
    for (int e = tid; e < m * m; e += PANEL_ROWS) {
      const int r2 = e % m, c2 = e / m;
      if (r2 >= c2) D[jj + 1 + r2][jj + 1 + c2] -= D[jj + 1 + r2][jj] * D[jj + 1 + c2][jj];
    }
    __syncthreads();
  }
  if (blockIdx.x == 0 && tid == 0) min_pivot[s] = fmin(min_pivot[s], pmin);
  // TRSM: row x of L21 solves x L11' = a (forward substitution).  The factorised diagonal block itself is not stored:
  // nothing reads it again, and other CTAs of this launch still read the original.
  const int i = j0 + w + blockIdx.x * PANEL_ROWS + tid;
  if (i >= n) return;
  double x[NB];
#pragma unroll
  for (int l = 0; l < NB; ++l)
    if (l < w) x[l] = A[i + (long long)(j0 + l) * n];
#pragma unroll
  for (int l = 0; l < NB; ++l) {
    if (l < w) {
      double v = x[l];
#pragma unroll
      for (int t = 0; t < l; ++t) v -= x[t] * D[l][t];
      x[l] = v / D[l][l];
      A[i + (long long)(j0 + l) * n] = x[l];
    }
  }
}

// grid (tiles, tiles, queries); tiles above the diagonal return at once
__global__ void __launch_bounds__(128) chol_update_kernel(double* __restrict__ ring, long long per, CholFront f, int j0,
                                                          int w, const int* __restrict__ failed) {
  const int ti = blockIdx.x, tj = blockIdx.y, s = blockIdx.z;
  if (tj > ti || failed[s]) return;
  double* A = ring + (long long)s * per + f.out_off;
  const int n = f.n, base = j0 + w, N = n - base;
  const int i0 = ti * UT, c0 = tj * UT;
  __shared__ double Pi[NB][ULD], Pj[NB][ULD];  // [k][row]: rows i0.. and c0.. of L21
  const int tid = threadIdx.x;
  for (int e = tid; e < NB * UT; e += 128) {
    const int r = e % UT, k = e / UT;
    const bool ok = k < w;
    Pi[k][r] = (ok && i0 + r < N) ? A[(base + i0 + r) + (long long)(j0 + k) * n] : 0.0;
    Pj[k][r] = (ok && c0 + r < N) ? A[(base + c0 + r) + (long long)(j0 + k) * n] : 0.0;
  }
  __syncthreads();
  const int lane = tid & 31, warp = tid >> 5;
  const int wm = (warp & 1) * 32, wn = (warp >> 1) * 32;
  double acc[4][4][2];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
  const int kend = (w + 3) & ~3;
  for (int k4 = 0; k4 < kend; k4 += 4) {
    const int k = k4 + (lane & 3);
    double af[4], bf[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) af[i] = Pi[k][wm + i * 8 + (lane >> 2)];
#pragma unroll
    for (int j = 0; j < 4; ++j) bf[j] = Pj[k][wn + j * 8 + (lane >> 2)];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) dmma(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = i0 + wm + i * 8 + (lane >> 2);
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int c = c0 + wn + j * 8 + (lane & 3) * 2 + e;
        if (r < N && c <= r) A[(base + r) + (long long)(base + c) * n] -= acc[i][j][e];
      }
  }
}

}  // namespace

int launch_chol_trace(const double* ring, long long per, const CholFront* fronts, int nfronts, int nq, double* stats,
                      cudaStream_t st) {
  chol_trace_kernel<<<nq, 256, 0, st>>>(ring, per, fronts, nfronts, stats);
  return 1;
}

int launch_chol_front_init(double* ring, long long per, const CholFront& f, const CholFront* prev, int nq,
                           const double* taup, const int* failed, cudaStream_t st) {
  chol_front_init_kernel<<<dim3(f.n, nq), 128, 0, st>>>(ring, per, f, prev ? *prev : f, prev ? 1 : 0, taup, failed);
  return 1;
}

int launch_chol_panel(double* ring, long long per, const CholFront& f, int j0, int w, int nq, int* failed,
                      long long* fail_index, double* min_pivot, cudaStream_t st) {
  const int below = f.n - j0 - w;
  const int rb = below > 0 ? (below + PANEL_ROWS - 1) / PANEL_ROWS : 1;
  chol_panel_kernel<<<dim3(rb, nq), PANEL_ROWS, 0, st>>>(ring, per, f, j0, w, failed, fail_index, min_pivot);
  if (below <= 0) return 1;
  const int t = (below + UT - 1) / UT;
  chol_update_kernel<<<dim3(t, t, nq), 128, 0, st>>>(ring, per, f, j0, w, failed);
  return 2;
}

}  // namespace nnsdp
