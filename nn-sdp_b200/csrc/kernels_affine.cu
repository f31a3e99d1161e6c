// Affine-coefficient ("symbolic") mode: Z(gamma) = Z0 + sum_v gamma_v Z_v as COO triplets over the upper
// triangle of the clique cover, for the hand-off that replaces the reference's AffExpr algebra
//   Z = Zin + Zout + sum(Zacs);  @constraint(model, Z .== Zksum)      src/Methods/chordal_sdp.jl:96-153
// (SURVEY.md section 8f-1).  Variables are stacked in the reference's creation order
//   [gamma_in (n_in); gamma_out (reach kinds: 1); gamma_ac1 = bounded (acdim); gamma_ac2 = sector (secdim)]
// and the coefficient patterns follow the closed form of DESIGN.md section 2:
//   gamma_in_i : -2 e_i e_i' + (xmin_i + xmax_i)(e_i e_a' + e_a e_i') - 2 xmin_i xmax_i e_a e_a'          input.jl:22-26
//   gamma_bnd_j: -2 eps eps' + (ymin_j + ymax_j)(eps e_a' + e_a eps') - 2 ymin_j ymax_j e_a e_a'          activ_bounded.jl:19-21
//   lambda_j   : -2 p_j rho rho' + q_j (rho eps' + eps rho')                                               activ_sector.jl:42-43
//   v_ij       : (rho_i - rho_j)(eps_i - eps_j)' + transpose - 2 (eps_i - eps_j)(eps_i - eps_j)'           activ_sector.jl:29-35,43,45
//   eta_j, nu_j: -s_j (rho e_a' + e_a rho') + (eps e_a' + e_a eps'),  s = smin | smax                      activ_sector.jl:55-56
//   gamma_out  : -2 e_a e_a' (hyperplane) | -e_a e_a' (circle, ellipsoid)                                  output.jl:76,84,93
// with rho_j = row j of [W b] placed in the block that feeds neuron j (bias at the affine index a) and
// eps_j the neuron's own index.  One CTA per variable; duplicate (entry, variable) pairs are allowed
// (consumers sum them, like Julia's sparse()).  All indices are 0-based here; the host adds 1.
//
// The batched form (nnsdp_affine_create_batch) writes the same coefficients as a canonical CSC per group of
// queries with equal bounds: one CTA per (variable, group), entries of a variable in ascending entry order,
// duplicates summed in the order the COO form lists them.  Only the band pairs v_ij have duplicates; every
// other variable's entries are a few ascending runs, so every output position is computed directly.
#include <algorithm>

#include "internal.h"

namespace nnsdp {

namespace {

constexpr int AFF_THREADS = 256;

struct VarInfo {
  int kind;       // 0 gin, 1 gout, 2 gbnd, 3 lambda, 4 v pair, 5 eta, 6 nu
  long long j;    // neuron (or input index); for pairs the smaller neuron i
  int t;          // pair distance j2 - i
};

__device__ __forceinline__ long long pair_base_dev(long long i, long long acdim, long long beta) {
  long long m = acdim - beta;
  if (m < 0) m = 0;
  if (i <= m) return i * beta;
  return m * beta + (i - m) * (acdim - 1) - ((m + i - 1) * (i - m)) / 2;
}

// variable index -> what it is.  Sector layout: [lambda(acdim); v(pairs); eta(acdim); nu(acdim)].
__device__ VarInfo decode_var(const AffineDev& A, long long v) {
  VarInfo r{0, 0, 0};
  if (v < A.var_out) { r.kind = 0; r.j = v; return r; }
  if (v < A.var_bnd) { r.kind = 1; return r; }
  if (v < A.var_sec) { r.kind = 2; r.j = v - A.var_bnd; return r; }
  long long s = v - A.var_sec;
  if (s < A.acdim) { r.kind = 3; r.j = s; return r; }
  if (s < A.lamdim) {
    // pair index -> (i, t): pairs of i start at pair_base(i); binary search on i
    const long long pidx = s - A.acdim;
    long long lo = 0, hi = A.acdim - 1;
    while (lo < hi) {
      const long long mid = (lo + hi + 1) >> 1;
      if (pair_base_dev(mid, A.acdim, A.beta) <= pidx) lo = mid; else hi = mid - 1;
    }
    r.kind = 4; r.j = lo; r.t = (int)(pidx - pair_base_dev(lo, A.acdim, A.beta)) + 1;
    return r;
  }
  s -= A.lamdim;
  if (s < A.acdim) { r.kind = 5; r.j = s; return r; }
  r.kind = 6; r.j = s - A.acdim;
  return r;
}

// block (0-based, >= 1) that holds neuron j, i.e. eps_j = n_in + j lies in block blk_of[n_in + j]
__device__ __forceinline__ int nblk(const NetDev& net, long long j) { return net.blk_of[net.n_in + j]; }

// coefficients of lambda_j: the Gram part -2 p rho rho' (when p != 0) and q (rho eps' + eps rho') (when q != 0)
__device__ __forceinline__ long long lambda_count(const NetDev& net, const AffineDev& A, long long j) {
  const long long nk = net.n[nblk(net, j) - 1];
  const double p = A.smin[j] * A.smax[j], q = A.smin[j] + A.smax[j];
  long long n = 0;
  if (p != 0.0) n += nk * (nk + 1) / 2 + nk + 1;
  if (q != 0.0) n += nk + 1;
  return n;
}

__global__ void affine_count_kernel(NetDev net, AffineDev A, long long* __restrict__ counts) {
  const long long v = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (v >= A.nvar) return;
  const VarInfo vi = decode_var(A, v);
  long long n = 0;
  switch (vi.kind) {
    case 0: n = 3; break;
    case 1: n = 1; break;
    case 2: n = 3; break;
    case 3: n = lambda_count(net, A, vi.j); break;
    case 4: {
      const long long ni = net.n[nblk(net, vi.j) - 1], nj = net.n[nblk(net, vi.j + vi.t) - 1];
      n = 2 * (ni + 1) + 2 * (nj + 1) + 3;
    } break;
    default: n = net.n[nblk(net, vi.j) - 1] + 2; break;
  }
  counts[v] = n;
}

struct Writer {
  long long* ent;
  long long* var;
  double* val;
  const long long* col_ptr;
  const int* lo;
  long long v;
  __device__ __forceinline__ void put(long long at, int r, int c, double x) const {
    // upper triangle: r <= c; entry index inside column c of the cover
    ent[at] = col_ptr[c] + (r - lo[c]);
    if (var) var[at] = v;  // NULL in the batched form (CSC: the variable is the column)
    val[at] = x;
  }
  // (u e_pos' + e_pos u')[.,.] for one support index r of u with value x
  __device__ __forceinline__ void put_sym(long long at, int r, int pos, double x) const {
    if (r < pos) put(at, r, pos, x);
    else if (r > pos) put(at, pos, r, x);
    else put(at, pos, pos, 2.0 * x);
  }
};

// rho_j (e_pos)' + transpose, scaled: support = block rows (n_k entries) and the affine index
__device__ void emit_rho_sym(const NetDev& net, const Writer& w, long long at, long long j, int pos,
                             double scale) {
  const int B = nblk(net, j), kb = B - 1;        // rows of M[kb] produce block B; inputs are block kb
  const int nk = net.n[kb], nout = net.n[B];
  const int jl = (int)(net.n_in + j - net.off[B]);
  const double* M = net.M[kb];
  const int a = net.Zdim - 1;
  for (int r = threadIdx.x; r < nk; r += AFF_THREADS)
    w.put_sym(at + r, net.off[kb] + r, pos, scale * M[jl + (long long)r * nout]);
  if (threadIdx.x == 0) w.put_sym(at + nk, a, pos, scale * M[jl + (long long)nk * nout]);
}

__global__ void __launch_bounds__(AFF_THREADS)
affine_fill_kernel(NetDev net, AffineDev A, const long long* __restrict__ offs, long long* ent,
                   long long* var, double* val) {
  const long long v = blockIdx.x;
  const VarInfo vi = decode_var(A, v);
  const Writer w{ent, var, val, A.col_ptr, A.lo, v};
  long long at = offs[v];
  const int a = net.Zdim - 1, n0 = net.n_in, tid = threadIdx.x;
  switch (vi.kind) {
    case 0: {
      if (tid == 0) {
        const int i = (int)vi.j;
        w.put(at, i, i, -2.0);
        w.put(at + 1, i, a, A.x1min[i] + A.x1max[i]);
        w.put(at + 2, a, a, -2.0 * (A.x1min[i] * A.x1max[i]));
      }
    } break;
    case 1: {
      if (tid == 0) w.put(at, a, a, A.out_kind == NNSDP_OUT_HPLANE ? -2.0 : -1.0);
    } break;
    case 2: {
      if (tid == 0) {
        const int e = n0 + (int)vi.j;
        w.put(at, e, e, -2.0);
        w.put(at + 1, e, a, A.ymin[vi.j] + A.ymax[vi.j]);
        w.put(at + 2, a, a, -2.0 * (A.ymin[vi.j] * A.ymax[vi.j]));
      }
    } break;
    case 3: {
      const long long j = vi.j;
      const int B = nblk(net, j), kb = B - 1, nk = net.n[kb], nout = net.n[B];
      const int jl = (int)(n0 + j - net.off[B]), r0 = net.off[kb];
      const double* M = net.M[kb];
      const double p = A.smin[j] * A.smax[j], q = A.smin[j] + A.smax[j];
      const double bj = M[jl + (long long)nk * nout];
      if (p != 0.0) {
        const double m2p = -2.0 * p;
        for (int c = tid; c < nk; c += AFF_THREADS) {  // column c of the upper triangle: rows 0..c
          const double wc = M[jl + (long long)c * nout];
          const long long base = at + (long long)c * (c + 1) / 2;
          for (int r = 0; r <= c; ++r) w.put(base + r, r0 + r, r0 + c, m2p * (M[jl + (long long)r * nout] * wc));
        }
        at += (long long)nk * (nk + 1) / 2;
        for (int r = tid; r < nk; r += AFF_THREADS) w.put(at + r, r0 + r, a, m2p * (M[jl + (long long)r * nout] * bj));
        if (tid == 0) w.put(at + nk, a, a, m2p * (bj * bj));
        at += nk + 1;
      }
      if (q != 0.0) emit_rho_sym(net, w, at, j, n0 + (int)j, q);
    } break;
    case 4: {
      const long long i = vi.j, j = vi.j + vi.t;
      const int ei = n0 + (int)i, ej = n0 + (int)j;
      const long long ni = net.n[nblk(net, i) - 1], nj = net.n[nblk(net, j) - 1];
      emit_rho_sym(net, w, at, i, ei, 1.0);   at += ni + 1;
      emit_rho_sym(net, w, at, i, ej, -1.0);  at += ni + 1;
      emit_rho_sym(net, w, at, j, ei, -1.0);  at += nj + 1;
      emit_rho_sym(net, w, at, j, ej, 1.0);   at += nj + 1;
      if (tid == 0) {
        w.put(at, ei, ei, -2.0);
        w.put(at + 1, ei, ej, 2.0);
        w.put(at + 2, ej, ej, -2.0);
      }
    } break;
    default: {
      const long long j = vi.j;
      const double s = (vi.kind == 5) ? A.smin[j] : A.smax[j];
      emit_rho_sym(net, w, at, j, a, -s);  // -s (rho e_a' + e_a rho'): (r, a) -s w_r and (a, a) -2 s b_j
      const long long nk = net.n[nblk(net, j) - 1];
      if (tid == 0) w.put(at + nk + 1, n0 + (int)j, a, 1.0);
    } break;
  }
}

// constant part Z0 at the cover entries: Zout with gamma_out = 0 (and every other multiplier 0), taken
// from what prep_final_kernel left for a batch whose multipliers are all zero.  Grid (Zdim, <= Q): query q
// writes z0[q * nent + e].
__global__ void affine_z0_kernel(NetDev net, BatchDev b, AffineDev A, long long nent, int Q, double* __restrict__ z0) {
  const int c = blockIdx.x;  // column of Z
  const int K = net.K, n0 = net.n_in, a = net.Zdim - 1, nK = net.n[K - 1];
  const int lo = A.lo[c];
  const long long base = A.col_ptr[c];
  const int Bc = net.blk_of[c];
  const double* WK = net.M[K - 1];
  for (int q = blockIdx.y; q < Q; q += gridDim.y) {
    const double* aff = b.aff + (long long)q * net.Zdim;
    const double* Z11 = b.Z11 + (long long)q * n0 * n0;
    const double* Z1K = b.Z1K + (long long)q * n0 * nK;
    const double* U = b.U + (long long)q * net.n_out * nK;
    double* zq = z0 + (long long)q * nent;
    for (int r = lo + threadIdx.x; r <= c; r += blockDim.x) {
      double val = 0.0;
      if (c == a) {
        val = aff[r];
      } else {
        const int Br = net.blk_of[r];
        if (Br == 0 && Bc == 0) val = Z11[r + c * n0];
        else if (Br == 0 && Bc == K - 1 && b.has_s12) val = Z1K[r + (long long)(c - net.off[K - 1]) * n0];
        else if (Br == K - 1 && Bc == K - 1 && b.has_s22) {
          const int rl = r - net.off[K - 1], cl = c - net.off[K - 1];
          double s = 0.0;
          for (int m = 0; m < net.n_out; ++m)
            s = fma(WK[m + (long long)rl * net.n_out], U[m + (long long)cl * net.n_out], s);
          val = s;
        }
      }
      zq[base + (r - lo)] = val;
    }
  }
}

// ---- batched form ------------------------------------------------------------------------------------------

// the bounds of query q (the first query of a group)
__device__ __forceinline__ AffineDev at_query(AffineDev A, long long q) {
  A.x1min += q * A.s_x1min;
  A.x1max += q * A.s_x1max;
  A.ymin += q * A.s_ymin;
  A.ymax += q * A.s_ymax;
  A.smin += q * A.s_smin;
  A.smax += q * A.s_smax;
  return A;
}

// Merged (entry, variable) count.  The pair v_ij, i < j, writes rho_i and rho_j into the columns e_i and e_j:
//   same layer          rho_i and rho_j share their rows (all above e_i):        2 n + 5
//   adjacent layers     rho_j's rows are the layer of e_i and reach (e_i, e_j):  2 n_i + 2 n_j + 3
//   further apart       (a layer narrower than beta in between):                 2 n_i + 2 n_j + 5
// In every case the two affine-row entries (e_i, a) and (e_j, a) each receive two terms.
__device__ long long merged_count(const NetDev& net, const AffineDev& A, long long v) {
  const VarInfo vi = decode_var(A, v);
  switch (vi.kind) {
    case 0: return 3;
    case 1: return 1;
    case 2: return 3;
    case 3: return lambda_count(net, A, vi.j);
    case 4: {
      const int Bi = nblk(net, vi.j), Bj = nblk(net, vi.j + vi.t);
      const long long ni = net.n[Bi - 1], nj = net.n[Bj - 1];
      if (Bj == Bi) return 2 * ni + 5;
      return 2 * (ni + nj) + (Bj == Bi + 1 ? 3 : 5);
    }
    default: return net.n[nblk(net, vi.j) - 1] + 2;
  }
}

// counts[g * nvar + v] for every (variable, group); the bounds of group g are those of query first[g]
__global__ void affine_csc_count_kernel(NetDev net, AffineDev A, const long long* __restrict__ first, long long ngroups,
                                        long long* __restrict__ counts) {
  const long long v = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (v >= A.nvar) return;
  for (long long g = blockIdx.y; g < ngroups; g += gridDim.y)
    counts[g * A.nvar + v] = merged_count(net, at_query(A, first[g]), v);
}

// One CTA per (variable, group): the variable's column of A_g at offs[g * nvar + v], rows (entries) ascending.
__global__ void __launch_bounds__(AFF_THREADS)
affine_csc_fill_kernel(NetDev net, AffineDev A0, const long long* __restrict__ first, long long ngroups,
                       const long long* __restrict__ offs, long long* ent, double* val) {
  const long long v = blockIdx.x;
  const VarInfo vi = decode_var(A0, v);
  const int a = net.Zdim - 1, n0 = net.n_in, tid = threadIdx.x;
  for (long long g = blockIdx.y; g < ngroups; g += gridDim.y) {
    const AffineDev A = at_query(A0, first[g]);
    const Writer w{ent, nullptr, val, A.col_ptr, A.lo, v};
    const long long at = offs[g * A.nvar + v];
    switch (vi.kind) {
      case 0: {  // (i, i), (i, a), (a, a): already ascending
        if (tid == 0) {
          const int i = (int)vi.j;
          w.put(at, i, i, -2.0);
          w.put(at + 1, i, a, A.x1min[i] + A.x1max[i]);
          w.put(at + 2, a, a, -2.0 * (A.x1min[i] * A.x1max[i]));
        }
      } break;
      case 1: {
        if (tid == 0) w.put(at, a, a, A.out_kind == NNSDP_OUT_HPLANE ? -2.0 : -1.0);
      } break;
      case 2: {
        if (tid == 0) {
          const int e = n0 + (int)vi.j;
          w.put(at, e, e, -2.0);
          w.put(at + 1, e, a, A.ymin[vi.j] + A.ymax[vi.j]);
          w.put(at + 2, a, a, -2.0 * (A.ymin[vi.j] * A.ymax[vi.j]));
        }
      } break;
      case 3: {  // [Gram triangle | q rho in column e_j | column a: Gram row, (e_j, a), (a, a)]
        const long long j = vi.j;
        const int B = nblk(net, j), kb = B - 1, nk = net.n[kb], nout = net.n[B];
        const int jl = (int)(n0 + j - net.off[B]), r0 = net.off[kb], pos = n0 + (int)j;
        const double* M = net.M[kb];
        const double p = A.smin[j] * A.smax[j], q = A.smin[j] + A.smax[j];
        const double bj = M[jl + (long long)nk * nout];
        const long long tri = p != 0.0 ? (long long)nk * (nk + 1) / 2 : 0, nq = q != 0.0 ? nk : 0;
        const long long colA = at + tri + nq, np = p != 0.0 ? nk : 0;
        const double m2p = -2.0 * p;
        if (p != 0.0) {
          for (int c = tid; c < nk; c += AFF_THREADS) {
            const double wc = M[jl + (long long)c * nout];
            const long long base = at + (long long)c * (c + 1) / 2;
            for (int r = 0; r <= c; ++r) w.put(base + r, r0 + r, r0 + c, m2p * (M[jl + (long long)r * nout] * wc));
          }
          for (int r = tid; r < nk; r += AFF_THREADS) w.put(colA + r, r0 + r, a, m2p * (M[jl + (long long)r * nout] * bj));
        }
        if (q != 0.0)
          for (int r = tid; r < nk; r += AFF_THREADS) w.put(at + tri + r, r0 + r, pos, q * M[jl + (long long)r * nout]);
        if (tid == 0) {
          if (q != 0.0) w.put(colA + np, pos, a, q * bj);
          if (p != 0.0) w.put(colA + np + (q != 0.0 ? 1 : 0), a, a, m2p * (bj * bj));
        }
      } break;
      case 4: {
        const long long i = vi.j, j = vi.j + vi.t;
        const int ei = n0 + (int)i, ej = n0 + (int)j;
        const int Bi = nblk(net, i), Bj = nblk(net, j);
        const int ni = net.n[Bi - 1], nj = net.n[Bj - 1], oi = net.off[Bi - 1], oj = net.off[Bj - 1];
        const int ldi = net.n[Bi], ldj = net.n[Bj];
        const double* Mi = net.M[Bi - 1] + (n0 + i - net.off[Bi]);  // rho_i[r] = Mi[r * ldi], bias at r = ni
        const double* Mj = net.M[Bj - 1] + (n0 + j - net.off[Bj]);
        const double bi = Mi[(long long)ni * ldi], bj = Mj[(long long)nj * ldj];
        long long tail;  // position of (e_j, e_j)
        if (Bj == Bi) {
          // column e_i: rows of rho, (e_i, e_i); column e_j: rows of rho, (e_i, e_j), (e_j, e_j)
          for (int r = tid; r < ni; r += AFF_THREADS) {
            const double xi = Mi[(long long)r * ldi], xj = Mj[(long long)r * ldj];
            w.put(at + r, oi + r, ei, xi + -xj);
            w.put(at + ni + 1 + r, oi + r, ej, -xi + xj);
          }
          if (tid == 0) {
            w.put(at + ni, ei, ei, -2.0);
            w.put(at + 2 * ni + 1, ei, ej, 2.0);
          }
          tail = at + 2 * ni + 2;
        } else if (Bj == Bi + 1) {
          // rho_j's rows are the layer of e_i (local index d): above e_i they join column e_i, at e_i they meet the
          // diagonal, below it they are row e_i of the columns up to that layer's end; column e_j: rho_i, rho_j
          const int d = ei - oj;
          const long long c2 = at + ni + nj;
          for (int r = tid; r < ni; r += AFF_THREADS) {
            const double xi = Mi[(long long)r * ldi];
            w.put(at + r, oi + r, ei, xi);
            w.put(c2 + r, oi + r, ej, -xi);
          }
          for (int s = tid; s < nj; s += AFF_THREADS) {
            const double xj = Mj[(long long)s * ldj];
            if (s < d) w.put(at + ni + s, oj + s, ei, -xj);
            else if (s == d) w.put(at + ni + s, ei, ei, 2.0 * -xj + -2.0);
            else w.put(at + ni + s, ei, oj + s, -xj);
            w.put(c2 + ni + s, oj + s, ej, s == d ? xj + 2.0 : xj);
          }
          tail = c2 + ni + nj;
        } else {
          // rho_j's rows lie strictly between e_i and e_j: row e_i of their columns, and in column e_j below e_i
          const long long c2 = at + ni + 1 + nj;
          for (int r = tid; r < ni; r += AFF_THREADS) {
            const double xi = Mi[(long long)r * ldi];
            w.put(at + r, oi + r, ei, xi);
            w.put(c2 + r, oi + r, ej, -xi);
          }
          for (int s = tid; s < nj; s += AFF_THREADS) {
            const double xj = Mj[(long long)s * ldj];
            w.put(at + ni + 1 + s, ei, oj + s, -xj);
            w.put(c2 + ni + 1 + s, oj + s, ej, xj);
          }
          if (tid == 0) {
            w.put(at + ni, ei, ei, -2.0);
            w.put(c2 + ni, ei, ej, 2.0);
          }
          tail = c2 + ni + 1 + nj;
        }
        if (tid == 0) {
          w.put(tail, ej, ej, -2.0);
          w.put(tail + 1, ei, a, bi + -bj);
          w.put(tail + 2, ej, a, -bi + bj);
        }
      } break;
      default: {  // -s (rho e_a' + e_a rho') + (eps e_a' + e_a eps'): column a holds rho's rows, e_j, a
        const long long j = vi.j;
        const double ms = -((vi.kind == 5) ? A.smin[j] : A.smax[j]);
        const int B = nblk(net, j), kb = B - 1, nk = net.n[kb], nout = net.n[B];
        const int jl = (int)(n0 + j - net.off[B]), r0 = net.off[kb];
        const double* M = net.M[kb];
        for (int r = tid; r < nk; r += AFF_THREADS) w.put(at + r, r0 + r, a, ms * M[jl + (long long)r * nout]);
        if (tid == 0) {
          w.put(at + nk, n0 + (int)j, a, 1.0);
          w.put(at + nk + 1, a, a, 2.0 * (ms * M[jl + (long long)nk * nout]));
        }
      } break;
    }
  }
}

// Exclusive scan of n int64 counts in place: tile sums, one CTA scanning the tile sums, tiles with their carry.
constexpr int SCAN_THREADS = 256, SCAN_ITEMS = 4, SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

// exclusive scan of one value per thread over the CTA; *total = the CTA's sum
__device__ long long block_exclusive_scan(long long x, long long* total) {
  __shared__ long long warp_incl[SCAN_THREADS / 32];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  long long inc = x;
  for (int d = 1; d < 32; d <<= 1) {
    const long long y = __shfl_up_sync(0xffffffffu, inc, d);
    if (lane >= d) inc += y;
  }
  if (lane == 31) warp_incl[wid] = inc;
  __syncthreads();
  if (wid == 0) {
    long long s = lane < SCAN_THREADS / 32 ? warp_incl[lane] : 0;
    for (int d = 1; d < 32; d <<= 1) {
      const long long y = __shfl_up_sync(0xffffffffu, s, d);
      if (lane >= d) s += y;
    }
    if (lane < SCAN_THREADS / 32) warp_incl[lane] = s;
  }
  __syncthreads();
  const long long ex = (wid > 0 ? warp_incl[wid - 1] : 0) + inc - x;
  *total = warp_incl[SCAN_THREADS / 32 - 1];
  __syncthreads();  // warp_incl is reused by the next call
  return ex;
}

__global__ void __launch_bounds__(SCAN_THREADS) scan_tile_sum_kernel(const long long* __restrict__ x, long long n,
                                                                      long long* __restrict__ sums) {
  const long long base = blockIdx.x * (long long)SCAN_TILE + threadIdx.x * SCAN_ITEMS;
  long long s = 0;
  for (int k = 0; k < SCAN_ITEMS; ++k)
    if (base + k < n) s += x[base + k];
  long long total;
  block_exclusive_scan(s, &total);
  if (threadIdx.x == 0) sums[blockIdx.x] = total;
}

__global__ void __launch_bounds__(SCAN_THREADS) scan_sums_kernel(long long* sums, long long nt) {
  long long carry = 0;
  for (long long t0 = 0; t0 < nt; t0 += SCAN_THREADS) {
    const long long t = t0 + threadIdx.x;
    const long long x = t < nt ? sums[t] : 0;
    long long total;
    const long long ex = block_exclusive_scan(x, &total);
    if (t < nt) sums[t] = carry + ex;
    carry += total;
  }
}

__global__ void __launch_bounds__(SCAN_THREADS) scan_tile_kernel(long long* x, long long n,
                                                                  const long long* __restrict__ sums) {
  const long long base = blockIdx.x * (long long)SCAN_TILE + threadIdx.x * SCAN_ITEMS;
  long long v[SCAN_ITEMS], s = 0;
  for (int k = 0; k < SCAN_ITEMS; ++k) {
    v[k] = base + k < n ? x[base + k] : 0;
    s += v[k];
  }
  long long total;
  long long run = sums[blockIdx.x] + block_exclusive_scan(s, &total);
  for (int k = 0; k < SCAN_ITEMS; ++k)
    if (base + k < n) {
      x[base + k] = run;
      run += v[k];
    }
}

// starts[g] = offs[g * nvar] for g = 0..ngroups (the last one is the total)
__global__ void affine_group_starts_kernel(const long long* __restrict__ offs, long long nvar, long long ngroups,
                                           long long* __restrict__ starts) {
  const long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (g <= ngroups) starts[g] = offs[g * nvar];
}

}  // namespace

int launch_affine_count(const NetDev& net, const AffineDev& A, long long* counts, cudaStream_t st) {
  const long long blocks = (A.nvar + 255) / 256;
  affine_count_kernel<<<(int)blocks, 256, 0, st>>>(net, A, counts);
  return 1;
}

int launch_affine_fill(const NetDev& net, const AffineDev& A, const long long* offs, long long* ent,
                       long long* var, double* val, cudaStream_t st) {
  affine_fill_kernel<<<(int)A.nvar, AFF_THREADS, 0, st>>>(net, A, offs, ent, var, val);
  return 1;
}

int launch_affine_z0(const NetDev& net, const BatchDev& b, const AffineDev& A, long long nent, int Q, double* z0,
                     cudaStream_t st) {
  affine_z0_kernel<<<dim3(net.Zdim, std::min(Q, 65535)), 128, 0, st>>>(net, b, A, nent, Q, z0);
  return 1;
}

int launch_affine_csc_count(const NetDev& net, const AffineDev& A, const long long* first, long long ngroups,
                            long long* counts, cudaStream_t st) {
  const dim3 grid((unsigned)((A.nvar + 255) / 256), (unsigned)std::min<long long>(ngroups, 65535));
  affine_csc_count_kernel<<<grid, 256, 0, st>>>(net, A, first, ngroups, counts);
  return 1;
}

int launch_affine_csc_fill(const NetDev& net, const AffineDev& A, const long long* first, long long ngroups,
                           const long long* offs, long long* ent, double* val, cudaStream_t st) {
  const dim3 grid((unsigned)A.nvar, (unsigned)std::min<long long>(ngroups, 65535));
  affine_csc_fill_kernel<<<grid, AFF_THREADS, 0, st>>>(net, A, first, ngroups, offs, ent, val);
  return 1;
}

long long scan_scratch_len(long long n) { return (n + SCAN_TILE - 1) / SCAN_TILE; }

int launch_scan_exclusive(long long* x, long long n, long long* sums, cudaStream_t st) {
  const long long nt = scan_scratch_len(n);
  scan_tile_sum_kernel<<<(unsigned)nt, SCAN_THREADS, 0, st>>>(x, n, sums);
  scan_sums_kernel<<<1, SCAN_THREADS, 0, st>>>(sums, nt);
  scan_tile_kernel<<<(unsigned)nt, SCAN_THREADS, 0, st>>>(x, n, sums);
  return 3;
}

int launch_affine_group_starts(const long long* offs, long long nvar, long long ngroups, long long* starts,
                               cudaStream_t st) {
  affine_group_starts_kernel<<<(unsigned)((ngroups + 256) / 256), 256, 0, st>>>(offs, nvar, ngroups, starts);
  return 1;
}

}  // namespace nnsdp
