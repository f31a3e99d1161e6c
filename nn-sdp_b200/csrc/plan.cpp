// Host-side integer work: sizes, clique index sets and the emission plan.
//
// make_cliques_host restates makeCliques (reference: src/Methods/chordal_cliques.jl:13-59)
// with index arithmetic only; nothing is materialised as a selector matrix (the reference
// builds Ec(Ck, Zdim) at src/Methods/chordal_sdp.jl:54 and then discards it).
#include <stdint.h>
#include <stdlib.h>

#include <algorithm>

#include "internal.h"
#include <atomic>
#include <cstring>
#include <thread>

namespace nnsdp {

int64_t lambda_dim(int64_t acdim, int64_t beta) {
  // _lambda_dim = sum((acxdim - beta):acxdim), src/Qc/activ_sector.jl:18
  int64_t s = 0;
  for (int64_t t = acdim - beta; t <= acdim; ++t) s += t;
  return s;
}

long long gram_layout(const Shape& sh, std::vector<long long>* goff, std::vector<int>* ldG) {
  goff->assign(sh.K, 0);
  ldG->assign(sh.K, 0);
  long long go = 0;
  for (int blk = 0; blk <= sh.K - 2; ++blk) {
    (*ldG)[blk] = (int)(((sh.n[blk] + 15) / 16) * 16);
    (*goff)[blk] = go;
    go += (long long)(*ldG)[blk] * sh.n[blk];
  }
  return go;
}

static int64_t Sfun(const Shape& sh, int64_t k) {  // S(k) = sum(xdims[1:k]), k = 0..K+1
  int64_t s = 0;
  for (int64_t i = 0; i < k; ++i) s += sh.n[i];
  return s;
}

int32_t make_cliques_host(const Shape& sh, int64_t beta, CliqueInfoHost* out) {
  const int K = sh.K;
  out->ck.clear();
  out->d1.clear();
  out->d2.clear();
  int64_t p = 1;
  for (int64_t i = 1; i <= K; ++i) {  // chordal_cliques.jl:22-27
    if (Sfun(sh, i + 1) + beta >= Sfun(sh, K - 1)) {
      p = i;
      break;
    }
  }
  for (int64_t k = 1; k <= p - 1; ++k) {  // :31-52
    CliqueRanges c;
    c.nseg = 2;
    c.lo[0] = Sfun(sh, k - 1);             // 0-based of S(k-1)+1
    c.hi[0] = Sfun(sh, k + 1) + beta - 1;  // 0-based of S(k+1)+beta
    c.lo[1] = Sfun(sh, K - 1);
    c.hi[1] = Sfun(sh, K);                 // 0-based of S(K)+1 (the affine index)
    NN_CHECK(c.hi[0] <= c.lo[1], NNSDP_ERR_ASSERT,
             "makeCliques: Ck1[end] <= Ck2[1] violated (chordal_cliques.jl:35)");
    // Ck = [Ck1; Ck2] must be sorted-unique for Ec (MyMath.jl:46); k < p guarantees it.
    NN_CHECK(c.hi[0] < c.lo[1], NNSDP_ERR_ASSERT, "makeCliques: Ck1 and Ck2 overlap");
    const int64_t ckdim = c.size();
    std::vector<int64_t> d1, d2;
    if (k == 1) {
      for (int64_t i = 1; i <= ckdim; ++i) d1.push_back(i);
    } else {
      const int64_t nk = sh.n[k - 1], nk1 = sh.n[k];  // zdims[k], zdims[k+1] (1-based)
      for (int64_t i = 1; i <= nk + nk1 + beta; ++i) d1.push_back(i);
      d1.push_back(ckdim);
      for (int64_t i = nk + nk1 + 1; i <= ckdim; ++i) d2.push_back(i);
    }
    out->ck.push_back(c);
    out->d1.push_back(d1);
    out->d2.push_back(d2);
  }
  CliqueRanges c;  // :55-57
  c.nseg = 1;
  c.lo[0] = Sfun(sh, p - 1);
  c.hi[0] = Sfun(sh, K);
  std::vector<int64_t> d1;
  for (int64_t i = 1; i <= c.size(); ++i) d1.push_back(i);
  out->ck.push_back(c);
  out->d1.push_back(d1);
  out->d2.push_back({});
  return NNSDP_OK;
}

int32_t fill_sizes(const Shape& sh, int64_t beta, nnsdp_sizes* s) {
  NN_CHECK(beta >= 0, NNSDP_ERR_ASSERT, "QcActivSector: 0 <= beta violated (activ_sector.jl:12)");
  NN_CHECK(beta <= sh.acdim, NNSDP_ERR_ASSERT,
           "QcActivSector: acxdim + length(ijs) == _lambda_dim needs beta <= acxdim "
           "(activ_sector.jl:18,32)");
  CliqueInfoHost ci;
  NN_TRY(make_cliques_host(sh, beta, &ci));
  s->K = sh.K;
  s->Zdim = sh.Zdim;
  s->acdim = sh.acdim;
  s->xtot = sh.xtot;
  s->lamdim = lambda_dim(sh.acdim, beta);
  s->secdim = s->lamdim + 2 * sh.acdim;
  s->n_in = sh.n_in();
  s->n_out = sh.n_out();
  s->sdim = sh.n_in() + sh.n_out() + 1;
  s->ncliques = (int64_t)ci.ck.size();
  s->sum_ck = s->sum_ck_sq = s->sum_dk = s->max_ck = 0;
  for (size_t k = 0; k < ci.ck.size(); ++k) {
    const int64_t n = ci.ck[k].size();
    s->sum_ck += n;
    s->sum_ck_sq += n * n;
    s->sum_dk += (int64_t)(ci.d1[k].size() + ci.d2[k].size());
    s->max_ck = std::max(s->max_ck, n);
  }
  return NNSDP_OK;
}

// The layout facts are checked, not assumed: every index lies in some clique; the private indices of clique k (whose
// last clique is k) are a leading, globally contiguous range of its local order; everything else of clique k lies in
// clique k+1, at local [0, lead) in order and at the tail [n_{k+1} - tail, n_{k+1}); the last clique is all private; and
// the indices a front does not take over (where its diagonal is shifted) cover 0 .. Zdim-1 exactly once.
int32_t build_chol_plan(const Shape& sh, const std::vector<CliqueRanges>& mats, std::vector<CholFront>* fronts) {
  const int p = (int)mats.size();
  NN_CHECK(p >= 1, NNSDP_ERR_ASSERT, "certify plan: no clique");
  std::vector<std::vector<int64_t>> idx(p);
  std::vector<int> owner(sh.Zdim, -1);
  for (int k = 0; k < p; ++k) {
    for (int s = 0; s < mats[k].nseg; ++s)
      for (int64_t g = mats[k].lo[s]; g <= mats[k].hi[s]; ++g) idx[k].push_back(g);
    for (int64_t g : idx[k]) {
      NN_CHECK(g >= 0 && g < sh.Zdim, NNSDP_ERR_ASSERT, "certify plan: index %lld outside Z", (long long)g);
      owner[g] = k;
    }
  }
  for (int64_t g = 0; g < sh.Zdim; ++g)
    NN_CHECK(owner[g] >= 0, NNSDP_ERR_ASSERT, "certify plan: index %lld lies in no clique", (long long)g);
  fronts->assign(p, CholFront{});
  std::vector<uint8_t> shifted(sh.Zdim, 0);
  long long off = 0;
  for (int k = 0; k < p; ++k) {
    CholFront& f = (*fronts)[k];
    const std::vector<int64_t>& c = idx[k];
    f.out_off = off;
    f.n = (int)c.size();
    off += (long long)f.n * f.n;
    int np = 0;
    while (np < f.n && owner[c[np]] == k) ++np;
    f.npriv = np;
    f.g0 = c[0];
    for (int i = 0; i < f.n; ++i) {
      NN_CHECK((owner[c[i]] == k) == (i < np), NNSDP_ERR_ASSERT,
               "certify plan: the private indices of clique %d are not a leading range", k + 1);
      if (i < np)
        NN_CHECK(c[i] == f.g0 + i, NNSDP_ERR_ASSERT, "certify plan: private indices of clique %d not contiguous", k + 1);
    }
    NN_CHECK(np >= 1, NNSDP_ERR_ASSERT, "certify plan: clique %d has no private index", k + 1);
    NN_CHECK(k + 1 < p || np == f.n, NNSDP_ERR_ASSERT, "certify plan: the last clique is not all private");
    if (k > 0) {  // map front k-1's Schur complement into this front
      const CholFront& pf = (*fronts)[k - 1];
      const std::vector<int64_t>& pc = idx[k - 1];
      const int ns = pf.n - pf.npriv;
      const int seg1 = (int)(mats[k - 1].hi[0] - mats[k - 1].lo[0] + 1);
      f.lead = seg1 - pf.npriv;
      f.tail = ns - f.lead;
      NN_CHECK(f.lead >= 0 && f.tail >= 0 && f.lead + f.tail <= f.n, NNSDP_ERR_ASSERT,
               "certify plan: separator of cliques %d, %d does not fit", k, k + 1);
      for (int s = 0; s < ns; ++s) {
        const int li = s < f.lead ? s : f.n - (ns - s);
        NN_CHECK(c[li] == pc[pf.npriv + s], NNSDP_ERR_ASSERT,
                 "certify plan: index %lld of clique %d is not at its place in clique %d", (long long)pc[pf.npriv + s], k,
                 k + 1);
      }
    }
    for (int i = f.lead; i < f.n - f.tail; ++i) {
      NN_CHECK(!shifted[c[i]], NNSDP_ERR_ASSERT, "certify plan: diagonal entry %lld shifted twice", (long long)c[i]);
      shifted[c[i]] = 1;
    }
  }
  for (int64_t g = 0; g < sh.Zdim; ++g)
    NN_CHECK(shifted[g], NNSDP_ERR_ASSERT, "certify plan: diagonal entry %lld never shifted", (long long)g);
  return NNSDP_OK;
}

namespace {

struct Piece {
  int64_t g0, g1;  // global range (inclusive)
  int64_t l0;      // local index of g0 inside the output matrix
};

bool intersects(int64_t a0, int64_t a1, int64_t b0, int64_t b1) {
  return a0 <= a1 && b0 <= b1 && std::max(a0, b0) <= std::min(a1, b1);
}

// Terms of Z that can be non-zero for rows [r0,r1] of block Bi against columns [c0,c1] of
// block Bj (global z indices).  Must be a superset of what the device evaluator tests per entry.
uint32_t pair_flags(const Shape& sh, int64_t beta, int Bi, int64_t r0, int64_t r1, int Bj,
                    int64_t c0, int64_t c1) {
  const int K = sh.K;
  if (Bi == K || Bj == K) return TF_AFF;
  uint32_t f = 0;
  const int64_t n0 = sh.n[0], a = sh.off[K];
  if (Bi == Bj) f |= TF_SAME;
  if ((Bi == 0 && Bj == K - 1) || (Bi == K - 1 && Bj == 0)) f |= TF_1K;
  if (Bi <= K - 2) {  // rows feed layer Bi+1: columns must be neurons within beta of that layer
    const int64_t lo = sh.off[Bi + 1] - beta, hi = sh.off[Bi + 2] - 1 + beta;
    if (intersects(std::max(c0, n0), std::min(c1, a - 1), lo, hi)) f |= TF_RC;
  }
  if (Bj <= K - 2) {
    const int64_t lo = sh.off[Bj + 1] - beta, hi = sh.off[Bj + 2] - 1 + beta;
    if (intersects(std::max(r0, n0), std::min(r1, a - 1), lo, hi)) f |= TF_CR;
  }
  if (r1 >= n0 && c1 >= n0) {
    const int64_t rr0 = std::max(r0, n0), cc0 = std::max(c0, n0);
    const int64_t dist = std::max<int64_t>(0, std::max(cc0 - r1, rr0 - c1));
    if (dist <= beta) f |= TF_BAND;
  }
  return f;
}

void cut(const Shape& sh, const CliqueRanges& c, bool split_blocks, int64_t step,
         std::vector<Piece>* out) {
  int64_t local = 0;
  for (int s = 0; s < c.nseg; ++s) {
    std::vector<std::pair<int64_t, int64_t>> ranges;
    if (split_blocks) {
      for (int b = 0; b <= sh.K; ++b) {
        const int64_t b0 = sh.off[b], b1 = (b == sh.K) ? sh.off[sh.K] : sh.off[b + 1] - 1;
        const int64_t g0 = std::max(c.lo[s], b0), g1 = std::min(c.hi[s], b1);
        if (g0 <= g1) ranges.push_back({g0, g1});
      }
    } else {
      ranges.push_back({c.lo[s], c.hi[s]});
    }
    for (auto& rg : ranges)
      for (int64_t g = rg.first; g <= rg.second; g += step)
        out->push_back({g, std::min(rg.second, g + step - 1), local + (g - c.lo[s])});
    local += c.hi[s] - c.lo[s] + 1;
  }
}

}  // namespace

int32_t build_plan(const Shape& sh, int64_t beta, const std::vector<CliqueRanges>& mats,
                   bool classify, PlanHost* plan, PackedLayout* packed) {
  const int K = sh.K;
  if (packed)
    NN_CHECK(mats.size() == 1 && mats[0].nseg == 1 && mats[0].lo[0] == 0 && mats[0].hi[0] == sh.Zdim - 1, NNSDP_ERR_ARG,
             "packed plans are built over the whole Z");
  // packed records hold the upper triangle: a tile strictly below the diagonal is never written
  auto strictly_lower = [](const TileDev& t) { return t.grow0 > t.gcol0 + t.ncols - 1; };
  plan->tiles.clear();
  plan->mats.clear();
  plan->skip_absent = false;
  int64_t max_n = 0;
  for (auto& c : mats) max_n = std::max(max_n, c.size());
  int64_t min_hidden = sh.n[1];
  for (int b = 1; b <= K - 1; ++b) min_hidden = std::min(min_hidden, sh.n[b]);
  const bool split_blocks = min_hidden >= 48;
  // 128-row tiles whenever rows are cut at block boundaries (a block of 50..127 rows is then one row piece and
  // the register-window programs apply); small nets get smaller tiles evaluated entry by entry
  plan->tile_rows = (split_blocks || max_n >= 512) ? 128 : (max_n >= 48 ? 64 : 32);
  plan->tile_cols = 32;
  int64_t out_off = 0;
  for (size_t ci = 0; ci < mats.size(); ++ci) {
    const CliqueRanges& c = mats[ci];
    const int64_t n = c.size();
    NN_CHECK(n < (int64_t(1) << 30), NNSDP_ERR_ARG, "output matrix too large");
    std::vector<Piece> rows, cols;
    cut(sh, c, split_blocks, plan->tile_rows, &rows);
    cut(sh, c, split_blocks, plan->tile_cols, &cols);
    // classification of one rectangular tile (global ranges inclusive, l0 = local index of g0)
    auto make_tile = [&](int64_t rg0, int64_t rg1, int64_t rl0, int64_t cg0, int64_t cg1, int64_t cl0) {
      TileDev t{};
      t.mat = (int32_t)ci;
      t.row0 = (int32_t)rl0;
      t.nrows = (int32_t)(rg1 - rg0 + 1);
      t.grow0 = (int32_t)rg0;
      t.col0 = (int32_t)cl0;
      t.ncols = (int32_t)(cg1 - cg0 + 1);
      t.gcol0 = (int32_t)cg0;
      const int rb0 = sh.block_of(rg0), rb1 = sh.block_of(rg1);
      const int cb0 = sh.block_of(cg0), cb1 = sh.block_of(cg1);
      uint32_t f = 0;
      for (int Bi = rb0; Bi <= rb1; ++Bi) {
        const int64_t br0 = std::max<int64_t>(rg0, sh.off[Bi]);
        const int64_t br1 = std::min<int64_t>(rg1, Bi == K ? sh.off[K] : sh.off[Bi + 1] - 1);
        for (int Bj = cb0; Bj <= cb1; ++Bj) {
          const int64_t bc0 = std::max<int64_t>(cg0, sh.off[Bj]);
          const int64_t bc1 = std::min<int64_t>(cg1, Bj == K ? sh.off[K] : sh.off[Bj + 1] - 1);
          f |= pair_flags(sh, beta, Bi, br0, br1, Bj, bc0, bc1);
        }
      }
      if (!classify) f = TF_ALL;
      t.rblk = t.cblk = -1;
      if (rb0 == rb1 && cb0 == cb1 && rb0 < K && cb0 < K && beta <= MAX_FAST_BETA) {
        f |= TF_UNIFORM;
        t.rblk = rb0;
        t.cblk = cb0;
      }
      t.flags = f;
      const uint32_t terms = f & TF_ALL;
      const bool fast = (f & TF_UNIFORM) && plan->tile_rows == 128 && plan->tile_cols == 32 &&
                        beta <= MAX_WINDOW_BETA;
      // SAME tiles of x_1 (Zin / S11) go to the edge kernel
      const bool aff_only = (rg0 == sh.off[K] && rg1 == sh.off[K]) || (cg0 == sh.off[K] && cg1 == sh.off[K]);
      if (terms == 0) t.prog = PROG_ZERO;
      else if (aff_only && classify) t.prog = PROG_AFF;
      else if (!(f & TF_UNIFORM)) t.prog = PROG_GENERAL;
      else if (terms == (TF_SAME | TF_BAND) && t.rblk >= 1) t.prog = PROG_DIAG;
      else if (terms == TF_SAME && t.rblk >= 1) t.prog = PROG_SAME;
      else if (terms == TF_RC && fast) t.prog = PROG_RC;
      else if (terms == TF_CR && fast) t.prog = PROG_CR;
      else t.prog = PROG_MIXED;
      return t;
    };
    // Cut points that isolate the beta-thin slivers of a block: the last beta indices of a hidden block
    // are the neurons within beta of the next layer (F(r,c) / F(c,r) slivers inside the diagonal block and
    // the band corner), the first beta those within beta of the previous layer.
    auto sliver_cuts = [&](int blk, int64_t g0, int64_t g1, std::vector<int64_t>* pts) {
      pts->clear();
      pts->push_back(g0);
      if (blk >= 1 && blk < K && beta > 0) {
        const int64_t a0 = sh.off[blk] + beta, a1 = sh.off[blk + 1] - beta;  // first index of mid / of tail
        if (a0 > g0 && a0 <= g1) pts->push_back(a0);
        if (a1 > g0 && a1 <= g1 && a1 > a0) pts->push_back(a1);
      }
      pts->push_back(g1 + 1);
    };
    for (const Piece& cp : cols) {
      for (const Piece& rp : rows) {
        TileDev t = make_tile(rp.g0, rp.g1, rp.l0, cp.g0, cp.g1, cp.l0);
        // (the same for a window tile over the block pair (b, b+2) / (b+2, b): only its beta columns / rows next to
        // layer b+1 carry a window sum, the rest of the 32-column tile is structurally zero)
        const bool thin_window = (t.prog == PROG_RC && t.cblk == t.rblk + 2) || (t.prog == PROG_CR && t.rblk == t.cblk + 2);
        if (classify && (t.prog == PROG_MIXED || thin_window) && plan->tile_rows == 128) {
          // A tile is MIXED when several terms meet in it.  Often that is one thin sliver inside a tile
          // whose bulk is a plain copy / fill / window: split at the sliver boundaries and classify the
          // pieces separately, so that only the slivers are evaluated entry by entry.
          std::vector<int64_t> rc, cc;
          sliver_cuts(t.rblk, rp.g0, rp.g1, &rc);
          sliver_cuts(t.cblk, cp.g0, cp.g1, &cc);
          if (rc.size() > 2 || cc.size() > 2) {
            std::vector<TileDev> sub;
            bool gain = false;
            for (size_t j = 0; j + 1 < cc.size(); ++j)
              for (size_t i = 0; i + 1 < rc.size(); ++i) {
                TileDev u = make_tile(rc[i], rc[i + 1] - 1, rp.l0 + (rc[i] - rp.g0), cc[j], cc[j + 1] - 1,
                                      cp.l0 + (cc[j] - cp.g0));
                gain |= thin_window ? (u.prog == PROG_ZERO) : (u.prog != PROG_MIXED);
                sub.push_back(u);
              }
            if (gain) {
              for (const TileDev& u : sub) plan->tiles.push_back(u);
              continue;
            }
          }
        }
        plan->tiles.push_back(t);
      }
    }
    MatDev md{};
    md.out_off = out_off;
    md.n = (int32_t)n;
    md.ld = (int32_t)n;
    plan->mats.push_back(md);
    out_off += n * n;
  }
  plan->per_query_doubles = out_off;
  if (packed) {
    std::vector<TileDev> keep;
    for (const TileDev& t : plan->tiles)
      if (!(split_blocks && t.prog == PROG_ZERO) && !strictly_lower(t)) keep.push_back(t);
    plan->tiles.swap(keep);
    // small nets keep one cell, the whole Z, with every tile of its upper triangle (zeros included)
    plan->skip_absent = split_blocks;
  }
  auto cls = [](const TileDev& t) {
    return (t.prog == PROG_ZERO || t.prog == PROG_SAME || t.prog == PROG_DIAG || t.prog == PROG_AFF) ? 0 : (t.prog == PROG_RC || t.prog == PROG_CR) ? 1 : 2;
  };
  // ---- fill class -> tall strips -----------------------------------------------------------------
  // The fill programs are plain store streams, and a store stream into a column-major matrix with an
  // odd leading dimension runs fastest as tall narrow strips whose 256-row chunks start on a 32 B
  // sector boundary (tools/probe_write_bw.cu: 7.4 TB/s against 5.7 TB/s for 128 x 32 tiles at
  // ld = 3003).  Vertically adjacent tiles of one kind are merged and re-cut into strips of at most
  // STRIP_ROWS x STRIP_COLS; SAME and DIAG tiles of a diagonal block merge into DIAG strips (the band
  // patch is a no-op where the strip holds no band entry); the affine row becomes wide 1-row jobs.
  {
    std::vector<TileDev> fillv, rest;
    for (const TileDev& t : plan->tiles) (cls(t) == 0 ? fillv : rest).push_back(t);
    const int32_t a = (int32_t)sh.off[K];
    auto is_affrow = [&](const TileDev& t) { return t.prog == PROG_AFF && t.grow0 == a && t.nrows == 1; };
    auto kind = [&](const TileDev& t) -> int {  // merge key
      if (t.prog == PROG_ZERO) return 0;
      if (t.prog == PROG_AFF) return 1;
      return 2 + t.rblk;  // SAME / DIAG of diagonal block rblk
    };
    std::vector<TileDev> rowjobs, colv;
    for (const TileDev& t : fillv) (is_affrow(t) ? rowjobs : colv).push_back(t);
    std::stable_sort(colv.begin(), colv.end(), [&](const TileDev& x, const TileDev& y) {
      if (x.mat != y.mat) return x.mat < y.mat;
      if (x.col0 != y.col0) return x.col0 < y.col0;
      if (x.ncols != y.ncols) return x.ncols < y.ncols;
      if (kind(x) != kind(y)) return kind(x) < kind(y);
      return x.row0 < y.row0;
    });
    std::vector<TileDev> strips;
    static const int strip_rows = [] { const char* e = getenv("NNSDP_STRIP_ROWS"); int v = e ? atoi(e) : STRIP_ROWS; return v < 32 ? 32 : v; }();
    static const int strip_cols_min = [] { const char* e = getenv("NNSDP_STRIP_COLS"); int v = e ? atoi(e) : STRIP_COLS; return v < 1 ? 1 : v; }();
    auto flush = [&](const TileDev& m) {
      const int nchunk = (m.nrows + strip_rows - 1) / strip_rows;
      const int h = (m.nrows + nchunk - 1) / nchunk;
      // short strips are made wider so that a CTA still has ~32 KB to write (tall ones: at most a tile's 32 columns;
      // strips of at most 128 rows -- narrow layers -- up to 128 columns, in equal parts)
      int strip_cols = std::max(strip_cols_min, std::min(32, 4096 / std::max(h, 1)));
      if (h <= 128) {
        const int limit = std::max(strip_cols_min, std::min(128, 8192 / std::max(h, 1)));
        const int nparts = (m.ncols + limit - 1) / limit;
        strip_cols = (m.ncols + nparts - 1) / nparts;
      }
      for (int c0 = 0; c0 < m.ncols; c0 += strip_cols)
        for (int r0 = 0; r0 < m.nrows; r0 += h) {
          TileDev u = m;
          u.row0 = m.row0 + r0;
          u.grow0 = m.grow0 + r0;
          u.nrows = std::min(h, m.nrows - r0);
          u.col0 = m.col0 + c0;
          u.gcol0 = m.gcol0 + c0;
          u.ncols = std::min(strip_cols, m.ncols - c0);
          strips.push_back(u);
        }
    };
    // vertical merge of equal column ranges, then horizontal merge of equal row ranges
    std::vector<TileDev> vm;
    for (size_t i = 0; i < colv.size();) {
      TileDev m = colv[i];
      size_t j = i + 1;
      for (; j < colv.size(); ++j) {
        const TileDev& n = colv[j];
        if (n.mat != m.mat || n.col0 != m.col0 || n.ncols != m.ncols || kind(n) != kind(m)) break;
        if (n.row0 != m.row0 + m.nrows) break;
        if (m.prog != PROG_ZERO && n.grow0 != m.grow0 + m.nrows) break;  // value depends on the global row
        m.nrows += n.nrows;
        if (n.prog == PROG_DIAG) m.prog = PROG_DIAG;
        m.flags |= n.flags;
      }
      vm.push_back(m);
      i = j;
    }
    std::stable_sort(vm.begin(), vm.end(), [&](const TileDev& x, const TileDev& y) {
      if (x.mat != y.mat) return x.mat < y.mat;
      if (x.row0 != y.row0) return x.row0 < y.row0;
      if (x.nrows != y.nrows) return x.nrows < y.nrows;
      if (kind(x) != kind(y)) return kind(x) < kind(y);
      return x.col0 < y.col0;
    });
    for (size_t i = 0; i < vm.size();) {
      TileDev m = vm[i];
      size_t j = i + 1;
      for (; j < vm.size(); ++j) {
        const TileDev& n = vm[j];
        if (n.mat != m.mat || n.row0 != m.row0 || n.nrows != m.nrows || kind(n) != kind(m) || n.grow0 != m.grow0) break;
        if (n.col0 != m.col0 + m.ncols) break;
        if (m.prog != PROG_ZERO && n.gcol0 != m.gcol0 + m.ncols) break;  // value depends on the global column
        if (m.prog == PROG_AFF) break;                                    // the affine column stays one column wide
        m.ncols += n.ncols;
        if (n.prog == PROG_DIAG) m.prog = PROG_DIAG;
        m.flags |= n.flags;
      }
      flush(m);
      i = j;
    }
    // CTA order = memory order: strips of one column range back to back, top to bottom (consecutive CTAs then write
    // vertically adjacent, i.e. contiguous, pieces of the same columns)
    std::stable_sort(strips.begin(), strips.end(), [](const TileDev& x, const TileDev& y) {
      if (x.mat != y.mat) return x.mat < y.mat;
      if (x.col0 != y.col0) return x.col0 < y.col0;
      return x.row0 < y.row0;
    });
    std::stable_sort(rowjobs.begin(), rowjobs.end(), [](const TileDev& x, const TileDev& y) {
      if (x.mat != y.mat) return x.mat < y.mat;
      return x.col0 < y.col0;
    });
    for (size_t i = 0; i < rowjobs.size();) {
      TileDev m = rowjobs[i];
      size_t j = i + 1;
      for (; j < rowjobs.size(); ++j) {
        const TileDev& n = rowjobs[j];
        if (n.mat != m.mat || n.row0 != m.row0 || n.col0 != m.col0 + m.ncols || n.gcol0 != m.gcol0 + m.ncols ||
            m.ncols + n.ncols > AFFROW_COLS)
          break;
        m.ncols += n.ncols;
      }
      strips.push_back(m);
      i = j;
    }
    plan->tiles = strips;
    plan->tiles.insert(plan->tiles.end(), rest.begin(), rest.end());
  }
  if (packed) {
    // ---- cells of the packed record, and every tile re-addressed inside its cell -------------------------
    std::vector<TileDev> keep;
    for (const TileDev& t : plan->tiles)
      if (!strictly_lower(t)) keep.push_back(t);  // strips cut out of a tile that straddled the diagonal
    plan->tiles.swap(keep);
    PackedLayout& L = *packed;
    L = PackedLayout();
    L.diag_cell.assign(K, -1);
    L.diag_entries.assign(K, 0);
    std::vector<PackedCell> rect, band, window, diag;
    auto is_diag_strip = [&](const TileDev& t) {
      return (t.prog == PROG_SAME || t.prog == PROG_DIAG) && cls(t) == 0 && t.rblk >= 1 && t.rblk == t.cblk;
    };
    auto inside = [](const TileDev& t, const PackedCell& c) {
      return t.grow0 >= c.grow0 && t.grow0 + t.nrows <= c.grow0 + c.nrows && t.gcol0 >= c.gcol0 &&
             t.gcol0 + t.ncols <= c.gcol0 + c.ncols;
    };
    if (split_blocks) {
      for (int b = 0; b <= K - 2; ++b)
        window.push_back({PK_WINDOW, b, sh.off[b], sh.off[b + 1], sh.n[b], sh.n[b + 1], 0, 1});
      std::vector<int64_t> lo(K, sh.Zdim), hi(K, -1);
      for (const TileDev& t : plan->tiles)
        if (is_diag_strip(t)) {
          lo[t.rblk] = std::min<int64_t>(lo[t.rblk], std::min(t.grow0, t.gcol0));
          hi[t.rblk] = std::max<int64_t>(hi[t.rblk], std::max(t.grow0 + t.nrows, t.gcol0 + t.ncols) - 1);
        }
      for (int b = 1; b <= K - 1; ++b)
        if (hi[b] >= lo[b]) {
          const int64_t m = hi[b] - lo[b] + 1;
          diag.push_back({PK_DIAG, b, lo[b], lo[b], m, m, 0, 0});
          band.push_back({PK_BAND, b, lo[b], lo[b], beta + 1, m, 0, 1});
        }
    }
    // which cell a tile is written into: -1 = none of the explicit ones
    auto find_cell = [&](const TileDev& t, int* which) -> int {
      if (is_diag_strip(t)) {
        for (size_t i = 0; i < diag.size(); ++i)
          if (diag[i].blk == t.rblk && inside(t, diag[i])) { *which = PK_DIAG; return (int)i; }
      } else {
        for (size_t i = 0; i < window.size(); ++i)
          if (inside(t, window[i])) { *which = PK_WINDOW; return (int)i; }
      }
      return -1;
    };
    // leftover tiles: vertically adjacent ones of equal column range merge into one RECT cell
    std::vector<int> left;
    for (size_t i = 0; i < plan->tiles.size(); ++i) {
      int which = 0;
      if (find_cell(plan->tiles[i], &which) < 0) left.push_back((int)i);
    }
    if (!split_blocks) {  // small nets: one cell, the whole Z
      rect.push_back({PK_RECT, -1, 0, 0, sh.Zdim, sh.Zdim, 0, 1});
    } else {
      std::sort(left.begin(), left.end(), [&](int x, int y) {
        const TileDev &a = plan->tiles[x], &b2 = plan->tiles[y];
        if (a.gcol0 != b2.gcol0) return a.gcol0 < b2.gcol0;
        if (a.ncols != b2.ncols) return a.ncols < b2.ncols;
        return a.grow0 < b2.grow0;
      });
      for (int i : left) {
        const TileDev& t = plan->tiles[i];
        if (!rect.empty()) {
          PackedCell& c = rect.back();
          if (c.gcol0 == t.gcol0 && c.ncols == t.ncols && c.grow0 + c.nrows == t.grow0) {
            c.nrows += t.nrows;
            continue;
          }
        }
        rect.push_back({PK_RECT, -1, t.grow0, t.gcol0, t.nrows, t.ncols, 0, 1});
      }
      // ... and horizontally adjacent ones of equal row range (the x_1 / x_K coupling, cut into 32-column tiles)
      std::sort(rect.begin(), rect.end(), [](const PackedCell& a, const PackedCell& b2) {
        if (a.grow0 != b2.grow0) return a.grow0 < b2.grow0;
        if (a.nrows != b2.nrows) return a.nrows < b2.nrows;
        return a.gcol0 < b2.gcol0;
      });
      std::vector<PackedCell> merged;
      for (const PackedCell& c : rect) {
        if (!merged.empty()) {
          PackedCell& m = merged.back();
          if (m.grow0 == c.grow0 && m.nrows == c.nrows && m.gcol0 + m.ncols == c.gcol0) {
            m.ncols += c.ncols;
            continue;
          }
        }
        merged.push_back(c);
      }
      rect.swap(merged);
    }
    // record: [RECT | BAND | WINDOW | DIAG], every cell on a 128 B boundary
    int64_t off = 0;
    auto place = [&](std::vector<PackedCell>& v) {
      for (PackedCell& c : v) {
        c.offset = off;
        off += ((c.nrows * c.ncols + 15) / 16) * 16;
        L.cells.push_back(c);
      }
    };
    place(rect);
    place(band);
    place(window);
    L.always_doubles = off;
    const size_t first_diag = L.cells.size();
    place(diag);
    L.record_doubles = off;
    for (size_t i = first_diag; i < L.cells.size(); ++i) L.diag_cell[L.cells[i].blk] = (int32_t)i;
    const size_t first_window = rect.size() + band.size();
    plan->mats.clear();
    for (const PackedCell& c : L.cells) plan->mats.push_back({c.offset, (int32_t)c.nrows, (int32_t)c.nrows});
    for (TileDev& t : plan->tiles) {
      int which = 0, ci = find_cell(t, &which), cell = -1;
      if (ci >= 0) {
        cell = (int)((which == PK_DIAG ? first_diag : first_window) + ci);
      } else {
        for (size_t i = 0; i < rect.size() && cell < 0; ++i)
          if (inside(t, L.cells[i])) cell = (int)i;
      }
      NN_CHECK(cell >= 0, NNSDP_ERR_STATE, "packed plan: a tile lies in no cell");
      const PackedCell& c = L.cells[cell];
      t.mat = cell;
      t.row0 = (int32_t)(t.grow0 - c.grow0);
      t.col0 = (int32_t)(t.gcol0 - c.gcol0);
      if (c.kind == PK_DIAG) L.diag_entries[c.blk] += (int64_t)t.nrows * t.ncols;
      else L.always_entries += (int64_t)t.nrows * t.ncols;
    }
    for (const PackedCell& c : band) L.always_entries += c.nrows * c.ncols;
    plan->per_query_doubles = L.record_doubles;
  }
  // sort by kernel class: fill (ZERO, SAME, DIAG, AFF strips) | window (RC, CR) | edge (MIXED, GENERAL)
  std::stable_sort(plan->tiles.begin(), plan->tiles.end(),
                   [&](const TileDev& x, const TileDev& y) { return cls(x) < cls(y); });
  {  // self-contained descriptors of the fill strips
    std::vector<long long> goff;
    std::vector<int> ldG;
    gram_layout(sh, &goff, &ldG);
    plan->strips.clear();
    for (const TileDev& t : plan->tiles) {
      if (cls(t) != 0) break;
      StripDev d{};
      d.out_off = plan->mats[t.mat].out_off;
      d.ld = plan->mats[t.mat].ld;
      d.row0 = t.row0; d.nrows = t.nrows; d.col0 = t.col0; d.ncols = t.ncols;
      d.grow0 = t.grow0; d.gcol0 = t.gcol0; d.prog = t.prog; d.rblk = t.rblk;
      if ((t.prog == PROG_SAME || t.prog == PROG_DIAG) && t.rblk >= 0) {
        d.rl0 = (int32_t)(t.grow0 - sh.off[t.rblk] - t.row0);
        d.cl0 = (int32_t)(t.gcol0 - sh.off[t.rblk]);
        if (t.rblk <= K - 2) {
          d.goff = goff[t.rblk];
          d.ldG = ldG[t.rblk];
        }
      }
      plan->strips.push_back(d);
    }
  }
  {  // band jobs: per (matrix, diagonal block), the square range its SAME / DIAG strips cover
    plan->bands.clear();
    struct Box { int64_t lo = INT64_MAX, hi = -1, l0 = 0; bool band = false; };
    std::vector<std::vector<Box>> box(plan->mats.size(), std::vector<Box>(K));
    int64_t widest = 0;
    for (const TileDev& t : plan->tiles) {
      if (cls(t) != 0 || !(t.prog == PROG_SAME || t.prog == PROG_DIAG) || t.rblk < 1 || t.rblk != t.cblk) continue;
      Box& bx = box[t.mat][t.rblk];
      const int64_t lo = std::min<int64_t>(t.grow0, t.gcol0);
      if (lo < bx.lo) {
        bx.lo = lo;
        bx.l0 = (t.grow0 <= t.gcol0) ? t.row0 : t.col0;  // local index of z index lo (rows and columns index alike)
      }
      bx.hi = std::max<int64_t>(bx.hi, std::max<int64_t>(t.grow0 + t.nrows, t.gcol0 + t.ncols) - 1);
      bx.band |= (t.prog == PROG_DIAG);
      widest = std::max<int64_t>(widest, bx.hi - bx.lo + 1);
    }
    // wide layers: tall strips of which a few rows per column lie in the band -> bulk-only strips + the band kernel
    plan->band_inline = widest < 256;
    for (size_t m = 0; m < plan->mats.size(); ++m)
      for (int blk = 1; blk < K; ++blk) {
        const Box& bx = box[m][blk];
        if (bx.hi < bx.lo || !bx.band) continue;
        BandDev j{};
        j.out_off = plan->mats[m].out_off;
        j.band_off = -1;
        j.ld = plan->band_inline ? 0 : plan->mats[m].ld;
        j.row0 = j.col0 = (int)bx.l0;
        j.g0 = (int)bx.lo;
        j.m = (int)(bx.hi - bx.lo + 1);
        j.blk = blk;
        if (packed) {  // the matrix is the DIAG cell of the block; its BAND cell holds the band for every query
          const PackedCell& c = packed->cells[m];
          j.optional = (c.kind == PK_DIAG);
          j.upper_only = 1;
          for (const PackedCell& bc : packed->cells)
            if (bc.kind == PK_BAND && bc.blk == blk) j.band_off = bc.offset;
        }
        if (j.ld > 0 || j.band_off >= 0) plan->bands.push_back(j);
      }
  }
  plan->n_fill = plan->n_window = plan->n_edge = 0;
  for (const TileDev& t : plan->tiles) {
    const int c = cls(t);
    (c == 0 ? plan->n_fill : c == 1 ? plan->n_window : plan->n_edge)++;
  }
  // ---- panel order (emit_panel_kernel): a column of a clique block is written by several programs; with the items of
  // the fill and the window kernel in ONE list sorted by 32-column panel, all pieces of a column are written by
  // consecutive CTAs of one launch.  Dense formats of wide nets only: packed cells are contiguous per program, and
  // narrow layers are issue-bound, not locality-bound (profiles/r2_experiments.txt).
  plan->panel.clear();
  plan->panel_fold.clear();
  if (!packed && !plan->band_inline && plan->n_window > 0 && beta <= MAX_WINDOW_BETA) {
    struct Key { long long off; int panel, row0, col0; StripDev d; };
    std::vector<Key> keys;
    auto sorted = [](std::vector<Key> k) {
      std::stable_sort(k.begin(), k.end(), [](const Key& x, const Key& y) {
        if (x.off != y.off) return x.off < y.off;
        if (x.panel != y.panel) return x.panel < y.panel;
        if (x.col0 != y.col0) return x.col0 < y.col0;
        return x.row0 < y.row0;
      });
      std::vector<StripDev> v(k.size());
      for (size_t i = 0; i < k.size(); ++i) v[i] = k[i].d;
      return v;
    };
    auto add_tile = [&](const TileDev& t) {  // window / edge tile re-packed into the strip layout
      const MatDev& m = plan->mats[t.mat];
      StripDev d{};
      d.out_off = m.out_off;
      d.ld = m.ld;
      d.row0 = t.row0; d.nrows = t.nrows; d.col0 = t.col0; d.ncols = t.ncols;
      d.grow0 = t.grow0; d.gcol0 = t.gcol0; d.prog = t.prog;
      d.rblk = t.rblk; d.rl0 = t.cblk; d.cl0 = (int32_t)t.flags; d.ldG = m.n;
      keys.push_back({d.out_off, d.col0 / 32, d.row0, d.col0, d});
    };
    for (int i = 0; i < plan->n_fill; ++i) {
      const StripDev& d = plan->strips[i];
      keys.push_back({d.out_off, d.col0 / 32, d.row0, d.col0, d});
    }
    for (int i = 0; i < plan->n_window; ++i) add_tile(plan->tiles[plan->n_fill + i]);
    plan->panel = sorted(keys);
    for (int i = 0; i < plan->n_edge; ++i) add_tile(plan->tiles[plan->n_fill + plan->n_window + i]);
    plan->panel_fold = sorted(keys);
  }
  return NNSDP_OK;
}


// Expands one record into the dense matrices of `mats` (clique blocks or the dense Z), both triangles.  Host work at
// memory speed: the upper-triangle part of a cell is copied column run by column run (contiguous on both sides), its
// mirror image in 64 x 64 tiles (contiguous writes, cache-resident strided reads); the matrices are independent and are
// expanded by several threads.  Cells are applied in the order DIAG, WINDOW, BAND, RECT (later ones are authoritative
// where cells overlap), so the result does not depend on the number of threads.
static void unpack_one(int64_t beta, const PackedLayout& lay, const CliqueRanges& ck, const double* record,
                       const uint8_t* present, double* o) {
  const int64_t n = ck.size();
  std::memset(o, 0, (size_t)n * n * sizeof(double));
  constexpr int64_t TB = 64;
  // rows [r0, r1] x columns [c0, c1] of a cell (global, inclusive) restricted to the index set
  auto copy_rect = [&](const PackedCell& c) {
    const double* src = record + c.offset;
    int64_t rbase = 0;
    for (int sr = 0; sr < ck.nseg; rbase += ck.hi[sr] - ck.lo[sr] + 1, ++sr) {
      const int64_t r0 = std::max(c.grow0, ck.lo[sr]), r1 = std::min(c.grow0 + c.nrows - 1, ck.hi[sr]);
      if (r0 > r1) continue;
      int64_t cbase = 0;
      for (int sc = 0; sc < ck.nseg; cbase += ck.hi[sc] - ck.lo[sc] + 1, ++sc) {
        const int64_t c0 = std::max(c.gcol0, ck.lo[sc]), c1 = std::min(c.gcol0 + c.ncols - 1, ck.hi[sc]);
        if (c0 > c1 || r0 > c1) continue;               // nothing on or above the diagonal
        const int64_t lr_of = rbase - ck.lo[sr], lc_of = cbase - ck.lo[sc];   // local = global + offset
        for (int64_t gcb = std::max(c0, r0); gcb <= c1; gcb += TB) {
          const int64_t gce = std::min(gcb + TB - 1, c1);
          for (int64_t grb = r0; grb <= std::min(r1, gce); grb += TB) {
            const int64_t gre = std::min(grb + TB - 1, r1);
            // as stored: column runs of the upper triangle
            for (int64_t gc = gcb; gc <= gce; ++gc) {
              const int64_t rhi = std::min(gre, gc);
              if (grb > rhi) continue;
              const double* col = src + (gc - c.gcol0) * c.nrows - c.grow0;
              std::memcpy(o + (lr_of + grb) + (lc_of + gc) * n, col + grb, (size_t)(rhi - grb + 1) * sizeof(double));
            }
            // mirrored: entry (gr, gc), gr <= gc, also at (gc, gr); row by row, so the writes are contiguous
            for (int64_t gr = grb; gr <= gre; ++gr) {
              const int64_t glo = std::max(gcb, gr);
              if (glo > gce) continue;
              double* dst = o + (lr_of + gr) * n + lc_of;             // o[lc + lr * n], lc = lc_of + gc
              const double* s0 = src - c.grow0 + gr - c.gcol0 * c.nrows;
              for (int64_t gc = glo; gc <= gce; ++gc) dst[gc] = s0[gc * c.nrows];
            }
          }
        }
      }
    }
  };
  auto local = [&](int64_t g) -> int64_t {
    int64_t base = 0;
    for (int s = 0; s < ck.nseg; base += ck.hi[s] - ck.lo[s] + 1, ++s)
      if (g >= ck.lo[s] && g <= ck.hi[s]) return base + g - ck.lo[s];
    return -1;
  };
  for (int pass : {PK_DIAG, PK_WINDOW, PK_BAND, PK_RECT})  // later passes are authoritative where cells overlap
    for (size_t i = 0; i < lay.cells.size(); ++i) {
      const PackedCell& c = lay.cells[i];
      if (c.kind != pass || !present[i]) continue;
      if (c.kind != PK_BAND) {
        copy_rect(c);
        continue;
      }
      const double* src = record + c.offset;
      for (int64_t j = 0; j < c.ncols; ++j) {
        const int64_t lr = local(c.grow0 + j);
        if (lr < 0) continue;
        for (int64_t t = 0; t <= beta && j + t < c.ncols; ++t) {
          const int64_t lc = local(c.grow0 + j + t);
          if (lc < 0) continue;
          const double v = src[t + (beta + 1) * j];
          o[lr + lc * n] = v;
          o[lc + lr * n] = v;
        }
      }
    }
}

void unpack_record(const Shape& sh, int64_t beta, const PackedLayout& lay, const std::vector<CliqueRanges>& mats,
                   const double* record, const uint8_t* present, double* out) {
  (void)sh;
  std::vector<int64_t> off(mats.size() + 1, 0);
  for (size_t m = 0; m < mats.size(); ++m) off[m + 1] = off[m] + mats[m].size() * mats[m].size();
  int nthreads = 1;
  if (mats.size() > 1 && off.back() >= (int64_t(1) << 20)) {     // small outputs: a thread start costs more than the copy
    const char* e = getenv("NNSDP_HOST_THREADS");
    const unsigned hw = std::thread::hardware_concurrency();
    nthreads = e ? atoi(e) : (int)std::min<unsigned>(hw ? hw : 1, 16);
    nthreads = std::max(1, std::min<int>(nthreads, (int)mats.size()));
  }
  if (nthreads == 1) {
    for (size_t m = 0; m < mats.size(); ++m) unpack_one(beta, lay, mats[m], record, present, out + off[m]);
    return;
  }
  std::atomic<size_t> next{0};
  auto work = [&] {
    for (size_t m = next.fetch_add(1); m < mats.size(); m = next.fetch_add(1))
      unpack_one(beta, lay, mats[m], record, present, out + off[m]);
  };
  std::vector<std::thread> th;
  for (int t = 1; t < nthreads; ++t) th.emplace_back(work);
  work();
  for (auto& t : th) t.join();
}

int32_t build_gather_plan(const Shape& sh, int64_t beta, const std::vector<CliqueRanges>& mats,
                          const PlanHost& plan, GatherPlan* gp) {
  const int K = sh.K;
  gp->usable = false;
  gp->colsegs.clear();
  gp->thin_idx.clear();
  gp->colseg_begin.assign(mats.size() + 1, 0);
  gp->thin_begin.assign(mats.size() + 1, 0);
  gp->dense_always_doubles = 0;
  // cells
  std::vector<std::vector<Piece>> segs(mats.size());
  for (size_t m = 0; m < mats.size(); ++m) {
    cut(sh, mats[m], true, int64_t(1) << 40, &segs[m]);
    gp->colseg_begin[m] = (int32_t)gp->colsegs.size();
    for (const Piece& sc : segs[m]) {
      GatherColSeg cs;
      cs.mat = (int32_t)m;
      cs.col0 = (int32_t)sc.l0;
      cs.ncols = (int32_t)(sc.g1 - sc.g0 + 1);
      const int Bj = sh.block_of(sc.g0);
      for (const Piece& sr : segs[m]) {
        GatherCell c{};
        c.row0 = (int32_t)sr.l0;
        c.nrows = (int32_t)(sr.g1 - sr.g0 + 1);
        c.ncols_hint = cs.ncols;
        c.col0_hint = cs.col0;
        const int Bi = sh.block_of(sr.g0);
        c.kind = GK_NONE;
        c.blk = -1;
        if (std::min(c.nrows, cs.ncols) >= GATHER_MIN_RECT && Bi < K && Bj < K) {
          if (Bj == Bi + 1 || Bi == Bj + 1) c.kind = GK_ALWAYS;
          else if (Bi == Bj && Bi >= 1 && Bi <= K - 2) c.kind = GK_GRAM, c.blk = Bi;
          else if (Bi == Bj && Bi == K - 1) c.kind = GK_S22;
        }
        c.pure_zero = pair_flags(sh, beta, Bi, sr.g0, sr.g1, Bj, sc.g0, sc.g1) == 0;
        if (c.kind == GK_ALWAYS) gp->dense_always_doubles += (int64_t)c.nrows * cs.ncols;
        cs.cells.push_back(c);
      }
      gp->colsegs.push_back(cs);
    }
  }
  gp->colseg_begin[mats.size()] = (int32_t)gp->colsegs.size();
  // thin entries, from the tiles of the emission plan
  auto cell_of = [&](int mat, int row, int col, int nrows, int ncols) -> const GatherCell* {
    for (int s = gp->colseg_begin[mat]; s < gp->colseg_begin[mat + 1]; ++s) {
      const GatherColSeg& cs = gp->colsegs[s];
      if (col < cs.col0 || col + ncols > cs.col0 + cs.ncols) continue;
      for (const GatherCell& c : cs.cells)
        if (row >= c.row0 && row + nrows <= c.row0 + c.nrows) return &c;
    }
    return nullptr;  // the tile straddles cells
  };
  std::vector<std::vector<int64_t>> per_mat(mats.size());
  const int64_t n0 = sh.n[0];
  for (const TileDev& t : plan.tiles) {
    if (t.prog == PROG_ZERO) continue;
    const MatDev& md = plan.mats[t.mat];
    std::vector<int64_t>& out = per_mat[t.mat];
    bool band_only = false;
    if (t.prog != PROG_AFF) {
      const GatherCell* c = cell_of(t.mat, t.row0, t.col0, t.nrows, t.ncols);
      if (c && c->kind == GK_ALWAYS) continue;
      if (c && (c->kind == GK_GRAM || c->kind == GK_S22)) {
        if (t.prog == PROG_SAME) continue;
        band_only = (t.prog == PROG_DIAG);
      }
    }
    for (int c = 0; c < t.ncols; ++c) {
      int r_lo = 0, r_hi = t.nrows - 1;
      if (band_only) {
        const int64_t jc = t.gcol0 - n0 + c, jr0 = t.grow0 - n0;
        r_lo = (int)std::max<int64_t>(0, jc - beta - jr0);
        r_hi = (int)std::min<int64_t>(t.nrows - 1, jc + beta - jr0);
      }
      for (int r = r_lo; r <= r_hi; ++r)
        out.push_back(md.out_off + (t.row0 + r) + (int64_t)(t.col0 + c) * md.ld);
    }
  }
  for (size_t m = 0; m < mats.size(); ++m) {
    std::sort(per_mat[m].begin(), per_mat[m].end());
    per_mat[m].erase(std::unique(per_mat[m].begin(), per_mat[m].end()), per_mat[m].end());
    gp->thin_begin[m] = (int64_t)gp->thin_idx.size();
    gp->thin_idx.insert(gp->thin_idx.end(), per_mat[m].begin(), per_mat[m].end());
  }
  gp->thin_begin[mats.size()] = (int64_t)gp->thin_idx.size();
  // worth it only when most of the output is either dense cells or zeros
  gp->usable = gp->dense_always_doubles > 0 &&
               (int64_t)gp->thin_idx.size() * 8 <= plan.per_query_doubles;
  return NNSDP_OK;
}

}  // namespace nnsdp
