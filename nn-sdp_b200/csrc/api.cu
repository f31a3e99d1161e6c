// Host runtime behind the C ABI of include/nnsdp_b200.h: contexts (devices + streams), uploaded
// networks, device-resident batches of queries, and the one-shot entry points that shard queries
// over the devices of a context (one host thread per device, no collective).
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <condition_variable>
#include <deque>
#include <functional>
#include <memory>
#include <mutex>
#include <thread>

#include <cuda.h>  // CUtensorMap and its enums; cuTensorMapEncodeTiled is obtained through cudaGetDriverEntryPoint

#include "internal.h"

namespace nnsdp {

static thread_local std::string g_err;

void set_error(const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_err = buf;
}

int32_t cuda_fail(cudaError_t e, const char* what, const char* file, int line) {
  set_error("CUDA error %d (%s) in %s at %s:%d", (int)e, cudaGetErrorString(e), what, file, line);
  return e == cudaErrorMemoryAllocation ? NNSDP_ERR_NOMEM : NNSDP_ERR_CUDA;
}

}  // namespace nnsdp

using namespace nnsdp;

// -----------------------------------------------------------------------------------------
// handles
// -----------------------------------------------------------------------------------------
struct nnsdp_ctx {
  std::vector<int> devs;
  std::vector<cudaStream_t> streams;
};

namespace {

struct DevBuf {  // growable device allocation bound to one device
  void* p = nullptr;
  size_t cap = 0;
  int32_t ensure(size_t bytes) {
    if (bytes <= cap && p) return NNSDP_OK;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    if (bytes == 0) bytes = 8;
    NN_CUDA(cudaMalloc(&p, bytes));
    cap = bytes;
    return NNSDP_OK;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  template <class T>
  T* as() const {
    return reinterpret_cast<T*>(p);
  }
};

struct NetPerDev {
  int dev = -1;
  std::vector<DevBuf> M, Wt;
  DevBuf n, off, xoff, blk_of, Mptr, Wtptr, ldT, bias;
  NetDev nd{};
  void release() {
    for (auto& x : M) x.release();
    for (auto& x : Wt) x.release();
    n.release(); off.release(); xoff.release(); blk_of.release();
    Mptr.release(); Wtptr.release(); ldT.release(); bias.release();
  }
};

int round_up(int64_t v, int64_t m) { return (int)(((v + m - 1) / m) * m); }

}  // namespace

struct nnsdp_net {
  nnsdp_ctx* ctx = nullptr;
  Shape sh;
  std::vector<int> ldT;
  std::vector<NetPerDev> per;
  int64_t max_block = 0;  // max_b n[b], b <= K-2 (Gram side)
  // batches kept alive between one-shot calls (plan, buffers, streams): creating and destroying a batch
  // costs milliseconds to a hundred milliseconds (cudaMalloc / cudaFree), more than the work of a small query
  struct Cached {
    int dev_index;
    int64_t beta, Qcap, ring;
    int dense;
    nnsdp_batch* b;
  };
  mutable std::mutex cache_mu;
  mutable std::vector<Cached> cache;
};

namespace {

enum Stage {
  ST_BOUNDS = 0, ST_PREP = 1, ST_GRAM = 2, ST_EMIT = 3, ST_D2H = 4,
  ST_EMIT_FILL = 5, ST_EMIT_WINDOW = 6, ST_EMIT_EDGE = 7,  // the three kernels of an emitter pass (sub-spans of ST_EMIT)
  ST_COUNT = 8
};

struct StageSpan {
  int stage;
  cudaEvent_t e0, e1;
};

}  // namespace

namespace {

// Host worker threads of a batch: zero-fill and scatter of the sparse host gather.
class WorkerPool {
 public:
  explicit WorkerPool(int n) {
    for (int i = 0; i < n; ++i) th_.emplace_back([this] { loop(); });
  }
  ~WorkerPool() {
    {
      std::lock_guard<std::mutex> l(m_);
      stop_ = true;
    }
    cv_.notify_all();
    for (auto& t : th_) t.join();
  }
  // tasks are tagged with a group id (the chunk); wait_group blocks until that group has drained
  void submit(int group, std::function<void()> fn) {
    {
      std::lock_guard<std::mutex> l(m_);
      if ((int)pending_.size() <= group) pending_.resize(group + 1, 0);
      ++pending_[group];
      q_.emplace_back(group, std::move(fn));
    }
    cv_.notify_one();
  }
  void wait_group(int group) {
    std::unique_lock<std::mutex> l(m_);
    done_cv_.wait(l, [&] { return (int)pending_.size() <= group || pending_[group] == 0; });
  }
  void wait_all() {
    std::unique_lock<std::mutex> l(m_);
    done_cv_.wait(l, [&] {
      for (int p : pending_)
        if (p) return false;
      return true;
    });
    pending_.clear();
  }
  int size() const { return (int)th_.size(); }

 private:
  void loop() {
    for (;;) {
      std::pair<int, std::function<void()>> job;
      {
        std::unique_lock<std::mutex> l(m_);
        cv_.wait(l, [&] { return stop_ || !q_.empty(); });
        if (stop_ && q_.empty()) return;
        job = std::move(q_.front());
        q_.pop_front();
      }
      job.second();
      {
        std::lock_guard<std::mutex> l(m_);
        --pending_[job.first];
      }
      done_cv_.notify_all();
    }
  }
  std::vector<std::thread> th_;
  std::deque<std::pair<int, std::function<void()>>> q_;
  std::vector<int> pending_;
  std::mutex m_;
  std::condition_variable cv_, done_cv_;
  bool stop_ = false;
};

constexpr int GATHER_STAGES = 4;  // packed thin-entry staging buffers in flight

}  // namespace

struct nnsdp_batch {
  // sparse host gather (DESIGN.md "end to end")
  GatherPlan gp;
  std::vector<CliqueRanges> mats_host;
  DevBuf d_thin_idx, d_packed;
  double* h_packed = nullptr;  // pinned, GATHER_STAGES * chunk * nthin doubles
  size_t h_packed_doubles = 0;
  cudaEvent_t ev_packed[GATHER_STAGES] = {nullptr, nullptr, nullptr, nullptr};
  std::unique_ptr<WorkerPool> pool;
  std::vector<int> h_cnt;      // Gram-active neuron counts per (query, block), host copy
  std::vector<int> h_pairs;    // active (query, block) pairs (two ints each) in query order; pair_begin[q] = first pair of query q
  std::vector<int64_t> pair_begin;
  DevBuf d_pairs;
  int64_t gather_bytes_dma = 0, gather_bytes_zeroed = 0, gather_bytes_thin = 0;  // of the last run
  nnsdp_ctx* ctx = nullptr;
  int dev_index = 0, dev = 0;
  const nnsdp_net* net = nullptr;
  const NetPerDev* nd = nullptr;
  int64_t beta = 0, Qcap = 0, ring = 0, Q = 0;
  bool dense = false;
  bool packed = false;   // output = packed records (the block-sparse upper triangle of Z), see PackedLayout
  PackedLayout lay;
  DevBuf d_bands;
  DevBuf d_tmaps, d_tmap_ok;  // tensor maps of the W matrices for the TMA staging of the CR window program
  int nbands = 0, band_max_m = 0;
  int64_t emitted_bytes = 0, packed_present_cells = 0;  // of the last run (emitted_bytes: what the emitter stored)
  // Ring slot state (DESIGN.md section 4).  Slots [0, ring_zeroed) have been zeroed since creation or the last
  // nnsdp_batch_ring_reset; structural zeros are never stored again.  slot_bulk[s * K + Br] = physical slot s holds a
  // non-zero bulk (Gram copy, S22 Gram) in the SAME / DIAG strips of block Br.
  int64_t ring_zeroed = 0;
  std::vector<uint8_t> slot_bulk;
  std::vector<int> bulk_begin;           // K + 1: the bulk strips of block Br are [bulk_begin[Br], bulk_begin[Br + 1])
  std::vector<int64_t> bulk_entries;     // K: output entries of those strips
  int64_t pass_entries = 0;              // entries every query of a pass stores (strips, windows, edges, band)
  std::vector<BulkItem> sel;             // the (slot, block) pairs of the current pass
  nnsdp_sizes sz{};
  PlanHost plan;
  DevBuf d_tiles, d_strips, d_bulk, d_mats, d_panel, d_goff, d_ldG;
  std::vector<long long> goff;
  std::vector<int> ldG;
  long long gram_per_query = 0;
  // inputs
  DevBuf x1min, x1max, ymin, ymax, smin, smax, gin, gbnd, gsec, outS, outvec, outinvP, gout;
  // bounds
  DevBuf xmin, xmax, acxmin, acxmax, smin_c, smax_c;
  // prepared
  DevBuf d11, Md, T0, Bt, u, aff, part, act, cnt, Z11, Z1K, U;
  DevBuf gram, ringbuf, flags;
  DevBuf cr_rowsA, cr_rowsB, cr_bias, cr_prel, cr_preu, cr_du, cr_bu, cr_dl;  // CROWN work buffers (kept when small)
  BatchDev bd{};
  GramDev gd{};
  PlanDev pd{};
  bool have_inputs = false, bounds_supplied = false, bounds_done = false, prepared = false;
  bool shared_gram = false;  // all queries of the batch have the same Gram blocks (set by prepare)
  int bounds_method = 0;  // 0 = IBP (intervalsWorstCase), 1 = CROWN (the reference's default, IntervalsAutoLirpa)
  cudaStream_t st = nullptr, st_copy = nullptr;
  cudaEvent_t ev_start = nullptr, ev_stop = nullptr;
  cudaEvent_t ev_done[2] = {nullptr, nullptr}, ev_free[2] = {nullptr, nullptr};
  std::vector<StageSpan> spans;
  std::vector<cudaEvent_t> ev_pool;
  float stage_ms[ST_COUNT] = {};
  int64_t stage_launches[ST_COUNT] = {};

  cudaEvent_t get_event() {
    if (!ev_pool.empty()) {
      cudaEvent_t e = ev_pool.back();
      ev_pool.pop_back();
      return e;
    }
    cudaEvent_t e = nullptr;
    cudaEventCreate(&e);
    return e;
  }
  bool span_open = false;
  void span_begin(int stage, cudaStream_t s) {
    span_open = spans.size() < 16384;  // spans are resolved at every sync; beyond the cap they are dropped
    if (!span_open) return;
    StageSpan sp{stage, get_event(), get_event()};
    cudaEventRecord(sp.e0, s);
    spans.push_back(sp);
  }
  void span_end(cudaStream_t s, int launches) {
    if (!span_open) return;
    span_open = false;
    cudaEventRecord(spans.back().e1, s);
    stage_launches[spans.back().stage] += launches;
  }
  void resolve_spans() {  // requires the streams to be idle
    for (auto& sp : spans) {
      float ms = 0.f;
      if (cudaEventElapsedTime(&ms, sp.e0, sp.e1) == cudaSuccess) {
        stage_ms[sp.stage] += ms;
        if (sp.stage >= 5 && sp.stage <= 7) stage_ms[3] += ms;  // ST_EMIT = sum of its three kernels
      }
      ev_pool.push_back(sp.e0);
      ev_pool.push_back(sp.e1);
    }
    spans.clear();
  }
  std::vector<DevBuf*> all_bufs() {
    return {&d_bands, &d_tmaps, &d_tmap_ok, &d_tiles, &d_strips, &d_bulk, &d_mats, &d_panel, &d_goff, &d_ldG, &x1min, &x1max, &ymin, &ymax, &smin, &smax,
            &gin, &gbnd, &gsec, &outS, &outvec, &outinvP, &gout, &xmin, &xmax, &acxmin, &acxmax,
            &smin_c, &smax_c, &d11, &Md, &T0, &Bt, &u, &aff, &part, &act, &cnt, &Z11, &Z1K, &U,
            &gram, &ringbuf, &flags, &cr_rowsA, &cr_rowsB, &cr_bias, &cr_prel, &cr_preu, &cr_du, &cr_bu, &cr_dl};
  }
};

namespace {

int32_t require_device() {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n <= 0) {
    cudaGetLastError();
    set_error("no CUDA device available (%s); this library has no CPU fallback",
              e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    return NNSDP_ERR_CUDA;
  }
  return NNSDP_OK;
}

int32_t upload(DevBuf& buf, const void* src, size_t bytes, cudaStream_t st) {
  NN_TRY(buf.ensure(bytes));
  if (bytes) NN_CUDA(cudaMemcpyAsync(buf.p, src, bytes, cudaMemcpyHostToDevice, st));
  return NNSDP_OK;
}

// host (len x Q, given stride) -> device; returns the device stride through *dstride
int32_t upload_cols(DevBuf& buf, const double* src, int64_t stride, int64_t len, int64_t Q,
                    cudaStream_t st, long long* dstride, const char* name) {
  NN_CHECK(src != nullptr, NNSDP_ERR_ARG, "query input '%s' is NULL", name);
  NN_CHECK(stride == 0 || stride >= len, NNSDP_ERR_ARG,
           "query input '%s': stride %lld < length %lld", name, (long long)stride, (long long)len);
  if (stride == 0 || Q == 1) {
    NN_TRY(buf.ensure((size_t)len * 8));
    if (len) NN_CUDA(cudaMemcpyAsync(buf.p, src, (size_t)len * 8, cudaMemcpyHostToDevice, st));
    *dstride = (stride == 0) ? 0 : len;
    return NNSDP_OK;
  }
  NN_TRY(buf.ensure((size_t)len * Q * 8));
  if (len == 0) {
    *dstride = 0;
    return NNSDP_OK;
  }
  if (stride == len)
    NN_CUDA(cudaMemcpyAsync(buf.p, src, (size_t)len * Q * 8, cudaMemcpyHostToDevice, st));
  else
    NN_CUDA(cudaMemcpy2DAsync(buf.p, (size_t)len * 8, src, (size_t)stride * 8, (size_t)len * 8,
                              (size_t)Q, cudaMemcpyHostToDevice, st));
  *dstride = len;
  return NNSDP_OK;
}

int32_t check_flags(nnsdp_batch* b, const char* where) {
  int h[4] = {0, 0, 0, 0};
  NN_CUDA(cudaMemcpyAsync(h, b->flags.p, sizeof(h), cudaMemcpyDeviceToHost, b->st));
  NN_CUDA(cudaStreamSynchronize(b->st));
  if (h[0] | h[1]) {
    NN_CUDA(cudaMemsetAsync(b->flags.p, 0, sizeof(h), b->st));
    if (h[0] & 1)
      NN_CHECK(false, NNSDP_ERR_ASSERT, "%s: acymin <= acymax violated (src/Qc/activ_bounded.jl:8)",
               where);
    if (h[0] & 2)
      NN_CHECK(false, NNSDP_ERR_ASSERT,
               "%s: 0 <= smin <= smax <= 1 violated (src/Qc/activ_sector.jl:14-16)", where);
    NN_CHECK(false, NNSDP_ERR_ASSERT,
             "%s: ykmin <= ykmax violated (src/Intervals/intervals_auto_lirpa.jl:60)", where);
  }
  return NNSDP_OK;
}

}  // namespace

// -----------------------------------------------------------------------------------------
// C ABI
// -----------------------------------------------------------------------------------------
extern "C" {

const char* nnsdp_last_error(void) { return g_err.c_str(); }
int32_t nnsdp_version(void) { return 100; }

int32_t nnsdp_device_count(int32_t* count) {
  NN_CHECK(count != nullptr, NNSDP_ERR_ARG, "count is NULL");
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess) {
    cudaGetLastError();
    n = 0;
  }
  *count = n;
  return NNSDP_OK;
}

int32_t nnsdp_ctx_create(int32_t ndev, const int32_t* dev_ids, nnsdp_ctx** out) {
  NN_CHECK(out != nullptr, NNSDP_ERR_ARG, "ctx output pointer is NULL");
  *out = nullptr;
  NN_CHECK(ndev >= 1, NNSDP_ERR_ARG, "ndev must be >= 1");
  NN_TRY(require_device());
  int avail = 0;
  NN_CUDA(cudaGetDeviceCount(&avail));
  std::unique_ptr<nnsdp_ctx> ctx(new nnsdp_ctx());
  for (int i = 0; i < ndev; ++i) {
    const int d = dev_ids ? dev_ids[i] : i;
    NN_CHECK(d >= 0 && d < avail, NNSDP_ERR_ARG, "device ordinal %d out of range (have %d)", d, avail);
    ctx->devs.push_back(d);
  }
  for (int d : ctx->devs) {
    NN_CUDA(cudaSetDevice(d));
    cudaStream_t s = nullptr;
    NN_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    ctx->streams.push_back(s);
  }
  *out = ctx.release();
  return NNSDP_OK;
}

int32_t nnsdp_ctx_destroy(nnsdp_ctx* ctx) {
  if (!ctx) return NNSDP_OK;
  for (size_t i = 0; i < ctx->streams.size(); ++i) {
    cudaSetDevice(ctx->devs[i]);
    cudaStreamSynchronize(ctx->streams[i]);
    cudaStreamDestroy(ctx->streams[i]);
  }
  delete ctx;
  return NNSDP_OK;
}

int32_t nnsdp_ctx_num_devices(const nnsdp_ctx* ctx, int32_t* ndev) {
  NN_CHECK(ctx && ndev, NNSDP_ERR_ARG, "NULL argument");
  *ndev = (int32_t)ctx->devs.size();
  return NNSDP_OK;
}

int32_t nnsdp_host_alloc(uint64_t bytes, void** ptr) {
  NN_CHECK(ptr != nullptr, NNSDP_ERR_ARG, "ptr is NULL");
  *ptr = nullptr;
  NN_TRY(require_device());
  NN_CUDA(cudaHostAlloc(ptr, bytes ? bytes : 8, cudaHostAllocPortable));
  return NNSDP_OK;
}

int32_t nnsdp_host_free(void* ptr) {
  if (ptr) NN_CUDA(cudaFreeHost(ptr));
  return NNSDP_OK;
}

// ---- network -----------------------------------------------------------------------------
static int32_t shape_from_xdims(int64_t K, const int64_t* xdims, Shape* sh) {
  NN_CHECK(xdims != nullptr, NNSDP_ERR_ARG, "xdims is NULL");
  // FeedFwdNet: length(xdims) >= 3 (MyNeuralNetwork.jl:18), K = length(Ms) = length(xdims)-1 (:22-23)
  NN_CHECK(K >= 2, NNSDP_ERR_ASSERT, "FeedFwdNet needs length(xdims) >= 3 (K >= 2)");
  NN_CHECK(K < 32768, NNSDP_ERR_ARG, "K too large");
  sh->K = (int)K;
  sh->n.assign(xdims, xdims + K + 1);
  for (auto v : sh->n) NN_CHECK(v >= 1 && v < (1 << 24), NNSDP_ERR_ARG, "bad layer width %lld", (long long)v);
  sh->off.assign(K + 1, 0);
  for (int b = 1; b <= K; ++b) sh->off[b] = sh->off[b - 1] + sh->n[b - 1];
  sh->xoff.assign(K + 2, 0);
  for (int b = 1; b <= K + 1; ++b) sh->xoff[b] = sh->xoff[b - 1] + sh->n[b - 1];
  sh->Zdim = sh->off[K] + 1;
  sh->acdim = sh->off[K] - sh->n[0];
  sh->xtot = sh->xoff[K + 1];
  NN_CHECK(sh->Zdim < (int64_t(1) << 30), NNSDP_ERR_ARG, "Zdim too large");
  return NNSDP_OK;
}

int32_t nnsdp_net_upload(nnsdp_ctx* ctx, int64_t K, const int64_t* xdims, const double* const* Ms,
                         nnsdp_net** out) {
  NN_CHECK(out != nullptr, NNSDP_ERR_ARG, "net output pointer is NULL");
  *out = nullptr;
  NN_CHECK(ctx != nullptr && Ms != nullptr, NNSDP_ERR_ARG, "NULL argument");
  std::unique_ptr<nnsdp_net> net(new nnsdp_net());
  net->ctx = ctx;
  NN_TRY(shape_from_xdims(K, xdims, &net->sh));
  const Shape& sh = net->sh;
  for (int k = 0; k < sh.K; ++k) NN_CHECK(Ms[k] != nullptr, NNSDP_ERR_ARG, "Ms[%d] is NULL", k);
  net->ldT.resize(sh.K);
  for (int k = 0; k < sh.K; ++k) net->ldT[k] = round_up(sh.n[k], 128);
  for (int b = 0; b <= sh.K - 2; ++b) net->max_block = std::max(net->max_block, sh.n[b]);

  std::vector<int> n32(sh.n.begin(), sh.n.end()), off32(sh.off.begin(), sh.off.end()),
      xoff32(sh.xoff.begin(), sh.xoff.end()), blk((size_t)sh.Zdim);
  for (int64_t z = 0; z < sh.Zdim; ++z) blk[z] = sh.block_of(z);
  std::vector<double> bias((size_t)sh.acdim);
  for (int k = 0; k <= sh.K - 2; ++k)
    for (int64_t i = 0; i < sh.n[k + 1]; ++i)
      bias[sh.noff(k + 1) + i] = Ms[k][i + sh.n[k] * sh.n[k + 1]];

  net->per.resize(ctx->devs.size());
  for (size_t di = 0; di < ctx->devs.size(); ++di) {
    NetPerDev& pd = net->per[di];
    pd.dev = ctx->devs[di];
    cudaStream_t st = ctx->streams[di];
    NN_CUDA(cudaSetDevice(pd.dev));
    pd.M.resize(sh.K);
    pd.Wt.resize(sh.K);
    std::vector<const double*> mp(sh.K), wp(sh.K);
    for (int k = 0; k < sh.K; ++k) {
      const size_t mbytes = (size_t)sh.n[k + 1] * (sh.n[k] + 1) * 8;
      NN_TRY(upload(pd.M[k], Ms[k], mbytes, st));
      const size_t wbytes = (size_t)net->ldT[k] * sh.n[k + 1] * 8;
      NN_TRY(pd.Wt[k].ensure(wbytes));
      NN_CUDA(cudaMemsetAsync(pd.Wt[k].p, 0, wbytes, st));
      launch_transpose_w(pd.M[k].as<double>(), (int)sh.n[k + 1], (int)sh.n[k], pd.Wt[k].as<double>(),
                         net->ldT[k], st);
      mp[k] = pd.M[k].as<double>();
      wp[k] = pd.Wt[k].as<double>();
    }
    NN_TRY(upload(pd.n, n32.data(), n32.size() * 4, st));
    NN_TRY(upload(pd.off, off32.data(), off32.size() * 4, st));
    NN_TRY(upload(pd.xoff, xoff32.data(), xoff32.size() * 4, st));
    NN_TRY(upload(pd.blk_of, blk.data(), blk.size() * 4, st));
    NN_TRY(upload(pd.Mptr, mp.data(), mp.size() * sizeof(double*), st));
    NN_TRY(upload(pd.Wtptr, wp.data(), wp.size() * sizeof(double*), st));
    NN_TRY(upload(pd.ldT, net->ldT.data(), net->ldT.size() * 4, st));
    NN_TRY(upload(pd.bias, bias.data(), bias.size() * 8, st));
    NN_CUDA(cudaStreamSynchronize(st));  // host staging vectors go out of scope below
    NN_CUDA(cudaGetLastError());
    NetDev& nd = pd.nd;
    nd.K = sh.K;
    nd.n_in = (int)sh.n_in();
    nd.n_out = (int)sh.n_out();
    nd.Zdim = (int)sh.Zdim;
    nd.acdim = (int)sh.acdim;
    nd.xtot = (int)sh.xtot;
    nd.n = pd.n.as<int>();
    nd.off = pd.off.as<int>();
    nd.xoff = pd.xoff.as<int>();
    nd.blk_of = pd.blk_of.as<int>();
    nd.M = pd.Mptr.as<const double*>();
    nd.Wt = pd.Wtptr.as<const double*>();
    nd.ldT = pd.ldT.as<int>();
    nd.bias_all = pd.bias.as<double>();
  }
  *out = net.release();
  return NNSDP_OK;
}

int32_t nnsdp_batch_destroy(nnsdp_batch* b);

int32_t nnsdp_net_destroy(nnsdp_net* net) {
  if (!net) return NNSDP_OK;
  for (auto& c : net->cache) nnsdp_batch_destroy(c.b);
  net->cache.clear();
  for (auto& pd : net->per) {
    cudaSetDevice(pd.dev);
    pd.release();
  }
  delete net;
  return NNSDP_OK;
}

// ---- integer work on the host ---------------------------------------------------------------
int32_t nnsdp_query_sizes(const nnsdp_net* net, int64_t beta, nnsdp_sizes* sizes) {
  NN_CHECK(net && sizes, NNSDP_ERR_ARG, "NULL argument");
  return fill_sizes(net->sh, beta, sizes);
}

int32_t nnsdp_sizes_from_xdims(int64_t K, const int64_t* xdims, int64_t beta, nnsdp_sizes* sizes) {
  NN_CHECK(sizes != nullptr, NNSDP_ERR_ARG, "NULL argument");
  Shape sh;
  NN_TRY(shape_from_xdims(K, xdims, &sh));
  return fill_sizes(sh, beta, sizes);
}

static int32_t cliques_out(const Shape& sh, int64_t beta, int64_t* ck_off, int64_t* ck_idx,
                           int64_t* ck1_len, int64_t* d_off, int64_t* d_idx) {
  NN_CHECK(beta >= 0, NNSDP_ERR_ASSERT, "0 <= beta violated (activ_sector.jl:12)");
  CliqueInfoHost ci;
  NN_TRY(make_cliques_host(sh, beta, &ci));
  int64_t o = 0, od = 0;
  for (size_t k = 0; k < ci.ck.size(); ++k) {
    const CliqueRanges& c = ci.ck[k];
    if (ck_off) ck_off[k] = o;
    if (ck1_len) ck1_len[k] = c.hi[0] - c.lo[0] + 1;
    for (int s = 0; s < c.nseg; ++s)
      for (int64_t g = c.lo[s]; g <= c.hi[s]; ++g, ++o)
        if (ck_idx) ck_idx[o] = g + 1;  // 1-based on the wire
    if (d_off) d_off[2 * k] = od;
    for (int64_t v : ci.d1[k]) {
      if (d_idx) d_idx[od] = v;
      ++od;
    }
    if (d_off) d_off[2 * k + 1] = od;
    for (int64_t v : ci.d2[k]) {
      if (d_idx) d_idx[od] = v;
      ++od;
    }
  }
  if (ck_off) ck_off[ci.ck.size()] = o;
  if (d_off) d_off[2 * ci.ck.size()] = od;
  return NNSDP_OK;
}

int32_t nnsdp_cliques(const nnsdp_net* net, int64_t beta, int64_t* ck_off, int64_t* ck_idx,
                      int64_t* ck1_len, int64_t* d_off, int64_t* d_idx) {
  NN_CHECK(net != nullptr, NNSDP_ERR_ARG, "net is NULL");
  return cliques_out(net->sh, beta, ck_off, ck_idx, ck1_len, d_off, d_idx);
}

int32_t nnsdp_cliques_from_xdims(int64_t K, const int64_t* xdims, int64_t beta, int64_t* ck_off,
                                 int64_t* ck_idx, int64_t* ck1_len, int64_t* d_off, int64_t* d_idx) {
  Shape sh;
  NN_TRY(shape_from_xdims(K, xdims, &sh));
  return cliques_out(sh, beta, ck_off, ck_idx, ck1_len, d_off, d_idx);
}

/* The output matrices of a format: 0 = clique blocks, 1 / 2 = the whole Z (dense / packed). */
static int32_t format_mats(const Shape& sh, int64_t beta, int32_t format, std::vector<CliqueRanges>* mats) {
  NN_CHECK(format >= 0 && format <= 2, NNSDP_ERR_ARG, "format must be NNSDP_FORMAT_BLOCKS, _DENSE_Z or _PACKED");
  mats->clear();
  if (format != NNSDP_FORMAT_BLOCKS) {
    CliqueRanges c;
    c.nseg = 1;
    c.lo[0] = 0;
    c.hi[0] = sh.Zdim - 1;
    mats->push_back(c);
  } else {
    CliqueInfoHost ci;
    NN_TRY(make_cliques_host(sh, beta, &ci));
    *mats = ci.ck;
  }
  return NNSDP_OK;
}

/* Host-only introspection of the emission plan: number of tiles and of output entries per tile
 * program (index = TileProg, 8 entries each) and per flag combination is not exposed. */
int32_t nnsdp_plan_stats(int64_t K, const int64_t* xdims, int64_t beta, int32_t dense_Z,
                         int64_t* tiles_per_prog, int64_t* entries_per_prog, int64_t* tile_rows,
                         int64_t* tile_cols) {
  NN_CHECK(tiles_per_prog && entries_per_prog, NNSDP_ERR_ARG, "NULL argument");
  Shape sh;
  NN_TRY(shape_from_xdims(K, xdims, &sh));
  nnsdp_sizes sz;
  NN_TRY(fill_sizes(sh, beta, &sz));
  std::vector<CliqueRanges> mats;
  NN_TRY(format_mats(sh, beta, dense_Z, &mats));
  PlanHost plan;
  PackedLayout lay;
  NN_TRY(build_plan(sh, beta, mats, true, &plan, dense_Z == NNSDP_FORMAT_PACKED ? &lay : nullptr));
  for (int i = 0; i < 8; ++i) tiles_per_prog[i] = entries_per_prog[i] = 0;
  for (const TileDev& t : plan.tiles) {
    tiles_per_prog[t.prog] += 1;
    entries_per_prog[t.prog] += (int64_t)t.nrows * t.ncols;
  }
  if (tile_rows) *tile_rows = plan.tile_rows;
  if (tile_cols) *tile_cols = plan.tile_cols;
  return NNSDP_OK;
}

/* The tile list of the emission plan (host only): 11 int32 per tile
 * {mat, row0, nrows, col0, ncols, grow0, gcol0, flags, rblk, cblk, prog}.  tiles_out may be NULL to
 * query the count. */
int32_t nnsdp_plan_tiles(int64_t K, const int64_t* xdims, int64_t beta, int32_t dense_Z,
                         int64_t max_tiles, int32_t* tiles_out, int64_t* ntiles) {
  NN_CHECK(ntiles != nullptr, NNSDP_ERR_ARG, "NULL argument");
  Shape sh;
  NN_TRY(shape_from_xdims(K, xdims, &sh));
  nnsdp_sizes sz;
  NN_TRY(fill_sizes(sh, beta, &sz));
  std::vector<CliqueRanges> mats;
  NN_TRY(format_mats(sh, beta, dense_Z, &mats));
  PlanHost plan;
  PackedLayout lay;
  NN_TRY(build_plan(sh, beta, mats, true, &plan, dense_Z == NNSDP_FORMAT_PACKED ? &lay : nullptr));
  *ntiles = (int64_t)plan.tiles.size();
  if (tiles_out) {
    NN_CHECK(max_tiles >= *ntiles, NNSDP_ERR_ARG, "tiles_out too small");
    static_assert(sizeof(TileDev) == 11 * sizeof(int32_t), "TileDev layout");
    memcpy(tiles_out, plan.tiles.data(), plan.tiles.size() * sizeof(TileDev));
  }
  return NNSDP_OK;
}

int32_t nnsdp_plan_panel(int64_t K, const int64_t* xdims, int64_t beta, int32_t dense_Z, int64_t max_items,
                         int64_t* items_out, int64_t* nitems) {
  NN_CHECK(nitems != nullptr, NNSDP_ERR_ARG, "NULL argument");
  Shape sh;
  NN_TRY(shape_from_xdims(K, xdims, &sh));
  nnsdp_sizes sz;
  NN_TRY(fill_sizes(sh, beta, &sz));
  std::vector<CliqueRanges> mats;
  NN_TRY(format_mats(sh, beta, dense_Z, &mats));
  PlanHost plan;
  PackedLayout lay;
  NN_TRY(build_plan(sh, beta, mats, true, &plan, dense_Z == NNSDP_FORMAT_PACKED ? &lay : nullptr));
  *nitems = (int64_t)plan.panel.size();
  if (items_out) {
    NN_CHECK(max_items >= *nitems, NNSDP_ERR_ARG, "items_out too small");
    for (size_t i = 0; i < plan.panel.size(); ++i) {
      const StripDev& d = plan.panel[i];
      int64_t* o = items_out + 10 * i;
      o[0] = d.out_off; o[1] = d.ld; o[2] = d.row0; o[3] = d.nrows; o[4] = d.col0; o[5] = d.ncols;
      o[6] = d.grow0; o[7] = d.gcol0; o[8] = d.prog; o[9] = d.rblk;
    }
  }
  return NNSDP_OK;
}

/* The host-gather plan (host only): cells {mat, row0, nrows, col0, ncols, kind, blk, pure_zero} (8 int32 each;
 * kind 0 = never dense, 1 = always, 2 = Gram-active layers only, 3 = S22 only) and the thin-entry offsets
 * (doubles inside one query's output).  Either output may be NULL to query the counts. */
int32_t nnsdp_gather_plan(int64_t K, const int64_t* xdims, int64_t beta, int32_t dense_Z, int64_t max_cells,
                          int32_t* cells_out, int64_t* ncells, int64_t max_thin, int64_t* thin_out,
                          int64_t* nthin, int32_t* usable) {
  NN_CHECK(ncells && nthin, NNSDP_ERR_ARG, "NULL argument");
  Shape sh;
  NN_TRY(shape_from_xdims(K, xdims, &sh));
  nnsdp_sizes sz;
  NN_TRY(fill_sizes(sh, beta, &sz));
  std::vector<CliqueRanges> mats;
  NN_CHECK(dense_Z == 0 || dense_Z == 1, NNSDP_ERR_ARG, "the host-gather plan exists for the dense formats only");
  NN_TRY(format_mats(sh, beta, dense_Z, &mats));
  PlanHost plan;
  NN_TRY(build_plan(sh, beta, mats, true, &plan));
  GatherPlan gp;
  NN_TRY(build_gather_plan(sh, beta, mats, plan, &gp));
  int64_t nc = 0;
  for (const GatherColSeg& cs : gp.colsegs) nc += (int64_t)cs.cells.size();
  *ncells = nc;
  *nthin = (int64_t)gp.thin_idx.size();
  if (usable) *usable = gp.usable ? 1 : 0;
  if (cells_out) {
    NN_CHECK(max_cells >= nc, NNSDP_ERR_ARG, "cells_out too small");
    int64_t i = 0;
    for (const GatherColSeg& cs : gp.colsegs)
      for (const GatherCell& c : cs.cells) {
        int32_t* o = cells_out + 8 * i++;
        o[0] = cs.mat; o[1] = c.row0; o[2] = c.nrows; o[3] = cs.col0; o[4] = cs.ncols;
        o[5] = c.kind; o[6] = c.blk; o[7] = c.pure_zero;
      }
  }
  if (thin_out) {
    NN_CHECK(max_thin >= *nthin, NNSDP_ERR_ARG, "thin_out too small");
    memcpy(thin_out, gp.thin_idx.data(), gp.thin_idx.size() * 8);
  }
  return NNSDP_OK;
}

// ---- batch ----------------------------------------------------------------------------------
int32_t nnsdp_batch_destroy(nnsdp_batch* b) {
  if (!b) return NNSDP_OK;
  cudaSetDevice(b->dev);
  if (b->st) cudaStreamSynchronize(b->st);
  if (b->st_copy) cudaStreamSynchronize(b->st_copy);
  b->resolve_spans();
  b->pool.reset();
  for (DevBuf* x : b->all_bufs()) x->release();
  b->d_thin_idx.release();
  b->d_packed.release();
  b->d_pairs.release();
  if (b->h_packed) cudaFreeHost(b->h_packed);
  for (cudaEvent_t e : b->ev_packed)
    if (e) cudaEventDestroy(e);
  for (cudaEvent_t e : b->ev_pool) cudaEventDestroy(e);
  for (cudaEvent_t e : {b->ev_start, b->ev_stop, b->ev_done[0], b->ev_done[1], b->ev_free[0], b->ev_free[1]})
    if (e) cudaEventDestroy(e);
  if (b->st) cudaStreamDestroy(b->st);
  if (b->st_copy) cudaStreamDestroy(b->st_copy);
  delete b;
  return NNSDP_OK;
}

int32_t nnsdp_batch_create(nnsdp_ctx* ctx, int32_t dev_index, const nnsdp_net* net, int64_t beta,
                           int64_t Qcap, int64_t ring_queries, int32_t dense_Z, nnsdp_batch** out) {
  NN_CHECK(out != nullptr, NNSDP_ERR_ARG, "batch output pointer is NULL");
  *out = nullptr;
  NN_CHECK(ctx && net, NNSDP_ERR_ARG, "NULL argument");
  NN_CHECK(net->ctx == ctx, NNSDP_ERR_ARG, "net was uploaded through a different ctx");
  NN_CHECK(dev_index >= 0 && dev_index < (int)ctx->devs.size(), NNSDP_ERR_ARG, "bad dev_index");
  NN_CHECK(Qcap >= 1 && Qcap < (1 << 30), NNSDP_ERR_ARG, "bad Qcap");
  NN_CHECK(ring_queries >= 0 && ring_queries <= 65535, NNSDP_ERR_ARG, "ring_queries must be in [0, 65535]");
  const Shape& sh = net->sh;
  nnsdp_batch* b = new nnsdp_batch();
  struct Guard {
    nnsdp_batch* b;
    ~Guard() { if (b) nnsdp_batch_destroy(b); }
  } guard{b};
  b->ctx = ctx;
  b->dev_index = dev_index;
  b->dev = ctx->devs[dev_index];
  b->net = net;
  b->nd = &net->per[dev_index];
  b->beta = beta;
  b->Qcap = Qcap;
  b->ring = std::min<int64_t>(ring_queries, Qcap);
  NN_CHECK(dense_Z >= 0 && dense_Z <= 2, NNSDP_ERR_ARG, "format must be NNSDP_FORMAT_BLOCKS, _DENSE_Z or _PACKED");
  b->dense = dense_Z == NNSDP_FORMAT_DENSE_Z;
  b->packed = dense_Z == NNSDP_FORMAT_PACKED;
  NN_TRY(fill_sizes(sh, beta, &b->sz));
  // the output-QC kernel keeps S (sdim^2 doubles) in shared memory: sdim = n_in + n_out + 1 <= 160.  Bounds-only
  // batches (ring_queries == 0) never run it.
  NN_CHECK(ring_queries == 0 || b->sz.sdim * b->sz.sdim * 8 + b->sz.n_out * 8 <= 200 * 1024, NNSDP_ERR_ARG,
           "n_in + n_out + 1 = %lld too large for the output-QC kernel (limit 160); bounds-only batches "
           "(ring_queries = 0) have no such limit", (long long)b->sz.sdim);
  NN_CUDA(cudaSetDevice(b->dev));
  NN_CUDA(cudaStreamCreateWithFlags(&b->st, cudaStreamNonBlocking));
  NN_CUDA(cudaStreamCreateWithFlags(&b->st_copy, cudaStreamNonBlocking));
  NN_CUDA(cudaEventCreate(&b->ev_start));
  NN_CUDA(cudaEventCreate(&b->ev_stop));
  for (int i = 0; i < 2; ++i) {
    NN_CUDA(cudaEventCreateWithFlags(&b->ev_done[i], cudaEventDisableTiming));
    NN_CUDA(cudaEventCreateWithFlags(&b->ev_free[i], cudaEventDisableTiming));
  }
  NN_TRY(b->flags.ensure(16));
  NN_CUDA(cudaMemsetAsync(b->flags.p, 0, 16, b->st));

  const int64_t Q = Qcap, ac = sh.acdim;
  // bounds + prepared vectors
  NN_TRY(b->xmin.ensure((size_t)sh.xtot * Q * 8));
  NN_TRY(b->xmax.ensure((size_t)sh.xtot * Q * 8));
  NN_TRY(b->acxmin.ensure((size_t)ac * Q * 8));
  NN_TRY(b->acxmax.ensure((size_t)ac * Q * 8));
  NN_TRY(b->smin_c.ensure((size_t)ac * Q * 8));
  NN_TRY(b->smax_c.ensure((size_t)ac * Q * 8));
  if (b->ring > 0) {
    const int npart = (int)((ac + PREP_THREADS - 1) / PREP_THREADS);
    NN_TRY(b->d11.ensure((size_t)ac * Q * 8));
    NN_TRY(b->Md.ensure((size_t)ac * Q * 8));
    NN_TRY(b->T0.ensure((size_t)ac * Q * 8));
    NN_TRY(b->Bt.ensure((size_t)ac * Q * 8 * std::max<int64_t>(beta, 1)));
    NN_TRY(b->u.ensure((size_t)ac * Q * 8));
    NN_TRY(b->aff.ensure((size_t)sh.Zdim * Q * 8));
    NN_TRY(b->part.ensure((size_t)npart * Q * 8));
    NN_TRY(b->act.ensure((size_t)ac * Q * 4));
    NN_TRY(b->cnt.ensure((size_t)sh.K * Q * 4));
    NN_TRY(b->Z11.ensure((size_t)sh.n_in() * sh.n_in() * Q * 8));
    NN_TRY(b->Z1K.ensure((size_t)sh.n_in() * sh.n[sh.K - 1] * Q * 8));
    NN_TRY(b->U.ensure((size_t)sh.n_out() * sh.n[sh.K - 1] * Q * 8));
    b->bd.npart = npart;
    // Gram scratch layout (one slot per ring entry)
    const long long go = gram_layout(sh, &b->goff, &b->ldG);
    b->gram_per_query = go;
    NN_TRY(upload(b->d_goff, b->goff.data(), b->goff.size() * 8, b->st));
    NN_TRY(upload(b->d_ldG, b->ldG.data(), b->ldG.size() * 4, b->st));
    NN_TRY(b->gram.ensure((size_t)go * b->ring * 8));
    // plan
    std::vector<CliqueRanges> mats;
    NN_TRY(format_mats(sh, beta, dense_Z, &mats));
    const char* noclass = getenv("NNSDP_NO_TILE_CLASSES");  // validation aid: evaluate every term everywhere
    NN_TRY(build_plan(sh, beta, mats, b->packed || !(noclass && noclass[0] == '1'), &b->plan,
                      b->packed ? &b->lay : nullptr));
    b->mats_host = mats;
    for (const BandDev& j : b->plan.bands) b->band_max_m = std::max(b->band_max_m, j.m);
    b->nbands = (int)b->plan.bands.size();
    NN_TRY(upload(b->d_bands, b->plan.bands.data(), b->plan.bands.size() * sizeof(BandDev), b->st));
    if (!b->packed) NN_TRY(build_gather_plan(sh, beta, mats, b->plan, &b->gp));
    if (const char* e = getenv("NNSDP_DENSE_GATHER"))  // developer aid: always copy the dense output
      if (e[0] == '1') b->gp.usable = false;
    if (b->gp.usable) {
      NN_TRY(upload(b->d_thin_idx, b->gp.thin_idx.data(), b->gp.thin_idx.size() * 8, b->st));
      for (int i = 0; i < GATHER_STAGES; ++i)
        NN_CUDA(cudaEventCreateWithFlags(&b->ev_packed[i], cudaEventDisableTiming));
    }
    NN_TRY(upload(b->d_tiles, b->plan.tiles.data(), b->plan.tiles.size() * sizeof(TileDev), b->st));
    NN_TRY(upload(b->d_mats, b->plan.mats.data(), b->plan.mats.size() * sizeof(MatDev), b->st));
    NN_TRY(b->ringbuf.ensure((size_t)b->plan.per_query_doubles * b->ring * 8));
    b->slot_bulk.assign((size_t)b->ring * sh.K, 0);
    // What a pass launches (the plan itself keeps every tile, ZERO included): structurally zero strips never, since a
    // ring slot is zeroed once; in the dense formats the SAME / DIAG strips whose band is written elsewhere (every SAME
    // strip, and the DIAG strips of wide layers) go to a per-block list, stored only for the (slot, block) pairs that
    // need them (prepare_slots)
    auto is_bulk = [&](const StripDev& d) {
      return !b->packed && d.rblk >= 1 && d.rblk <= sh.K - 1 &&
             (d.prog == PROG_SAME || (d.prog == PROG_DIAG && !b->plan.band_inline));
    };
    std::vector<StripDev> strips, bulk;
    std::vector<std::vector<StripDev>> per_blk(sh.K);
    b->pass_entries = 0;
    b->bulk_entries.assign(sh.K, 0);
    for (const StripDev& d : b->plan.strips) {
      if (d.prog == PROG_ZERO) continue;
      if (is_bulk(d)) {
        per_blk[d.rblk].push_back(d);
        b->bulk_entries[d.rblk] += (int64_t)d.nrows * d.ncols;
      } else {
        strips.push_back(d);
        b->pass_entries += (int64_t)d.nrows * d.ncols;
      }
    }
    b->bulk_begin.assign(sh.K + 1, 0);
    for (int blk = 0; blk < sh.K; ++blk) {
      b->bulk_begin[blk] = (int)bulk.size();
      bulk.insert(bulk.end(), per_blk[blk].begin(), per_blk[blk].end());
    }
    b->bulk_begin[sh.K] = (int)bulk.size();
    for (int i = b->plan.n_fill; i < (int)b->plan.tiles.size(); ++i)
      b->pass_entries += (int64_t)b->plan.tiles[i].nrows * b->plan.tiles[i].ncols;
    for (const BandDev& j : b->plan.bands)  // in-place band of the DIAG ranges: (2 beta + 1) m entries less the corners
      if (j.ld > 0) b->pass_entries += (int64_t)j.m * (2 * beta + 1) - beta * (beta + 1);
    NN_TRY(upload(b->d_strips, strips.data(), strips.size() * sizeof(StripDev), b->st));
    NN_TRY(upload(b->d_bulk, bulk.data(), bulk.size() * sizeof(StripDev), b->st));
    b->pd.strips = b->d_strips.as<StripDev>();
    b->pd.bulk = b->d_bulk.as<StripDev>();
    b->pd.n_strips = (int)strips.size();
    b->pd.tiles = b->d_tiles.as<TileDev>();
    b->pd.mats = b->d_mats.as<MatDev>();
    b->pd.panel_desc = nullptr;
    b->pd.n_panel = 0;
    {
      // dense formats of wide nets: fill strips and window tiles in one launch in panel order (plan.cpp build_panel,
      // emit_panel_kernel).  NNSDP_PANEL=0 keeps the two kernels.
      static const int panel_env = [] { const char* e = getenv("NNSDP_PANEL"); return e ? atoi(e) : 1; }();
      if (panel_env && !b->packed && !b->plan.panel.empty()) {
        std::vector<StripDev> panel;
        for (const StripDev& d : b->plan.panel)
          if (d.prog != PROG_ZERO && (d.prog == PROG_RC || d.prog == PROG_CR || !is_bulk(d))) panel.push_back(d);
        NN_TRY(upload(b->d_panel, panel.data(), panel.size() * sizeof(StripDev), b->st));
        b->pd.panel_desc = b->d_panel.as<StripDev>();
        b->pd.n_panel = (int)panel.size();
      }
    }
    b->pd.ntiles = (int)b->plan.tiles.size();
    b->pd.n_fill = b->plan.n_fill;
    b->pd.n_window = b->plan.n_window;
    b->pd.n_edge = b->plan.n_edge;
    b->pd.tile_rows = b->plan.tile_rows;
    b->pd.per_query = b->plan.per_query_doubles;
    b->pd.tmaps = nullptr;
    b->pd.tmap_ok = nullptr;
    if (b->plan.n_window > 0 && beta <= MAX_WINDOW_BETA) {
      // One tensor map per layer: W_k as a 2-D tensor (neurons contiguous, then inputs), box (128 + 2 beta) x 32, zero
      // fill outside.  A layer qualifies when its column pitch is a multiple of 16 bytes (an even number of neurons);
      // boxes may stick out of the matrix on every side (tools/probe_tma.cu, profiles/r2_probe_tma.txt).
      typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                   const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
      void* fn = nullptr;
      cudaDriverEntryPointQueryResult qres;
      static const bool no_tma = [] { const char* e = getenv("NNSDP_NO_TMA"); return e && e[0] == '1'; }();
      if (!no_tma && cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) == cudaSuccess && fn &&
          qres == cudaDriverEntryPointSuccess) {
        std::vector<CUtensorMap> maps(sh.K);
        std::vector<int> ok(sh.K, 0);
        bool any = false;
        for (int k = 0; k < sh.K; ++k) {
          if (sh.n[k + 1] % 2 != 0) continue;
          const cuuint64_t dims[2] = {(cuuint64_t)sh.n[k + 1], (cuuint64_t)sh.n[k]};
          const cuuint64_t strides[1] = {(cuuint64_t)sh.n[k + 1] * 8};
          const cuuint32_t box[2] = {(cuuint32_t)(128 + 2 * beta + 2), 32};  // CR_LDW(beta) of kernels_emit.cu
          const cuuint32_t estr[2] = {1, 1};
          const CUresult r = ((EncodeFn)fn)(&maps[k], CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, b->nd->M[k].p, dims, strides, box, estr,
                                            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                            CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
          ok[k] = (r == CUDA_SUCCESS);
          any |= ok[k] != 0;
        }
        if (any) {
          static_assert(sizeof(CUtensorMap) == 128, "CUtensorMap is 128 bytes");
          NN_TRY(upload(b->d_tmaps, maps.data(), maps.size() * sizeof(CUtensorMap), b->st));
          NN_TRY(upload(b->d_tmap_ok, ok.data(), ok.size() * 4, b->st));
          NN_CUDA(cudaStreamSynchronize(b->st));
          b->pd.tmaps = b->d_tmaps.p;
          b->pd.tmap_ok = b->d_tmap_ok.as<int>();
        }
      } else {
        cudaGetLastError();
      }
    }
    b->pd.packed = b->plan.skip_absent ? 1 : 0;
    b->pd.band_inline = b->plan.band_inline ? 1 : 0;
    b->gd.scratch = b->gram.as<double>();
    b->gd.per_query = go;
    b->gd.goff = b->d_goff.as<long long>();
    b->gd.ldG = b->d_ldG.as<int>();
    b->gd.mirror = b->packed && b->plan.skip_absent ? 0 : 1;  // packed records of wide nets hold the upper triangle only
  }
  NN_CUDA(cudaStreamSynchronize(b->st));
  guard.b = nullptr;
  *out = b;
  return NNSDP_OK;
}

int32_t nnsdp_batch_set_inputs(nnsdp_batch* b, int64_t Q, const nnsdp_query_inputs* in) {
  NN_CHECK(b && in, NNSDP_ERR_ARG, "NULL argument");
  NN_CHECK(Q >= 1 && Q <= b->Qcap, NNSDP_ERR_ARG, "Q = %lld outside [1, Qcap = %lld]", (long long)Q,
           (long long)b->Qcap);
  NN_CUDA(cudaSetDevice(b->dev));
  const Shape& sh = b->net->sh;
  const nnsdp_sizes& sz = b->sz;
  BatchDev& bd = b->bd;
  cudaStream_t st = b->st;
  b->have_inputs = false;
  b->bounds_done = b->prepared = false;
  b->Q = Q;
  bd.Q = (int)Q;
  bd.beta = (int)b->beta;
  bd.lamdim = sz.lamdim;
  bd.sdim = (int)sz.sdim;
  NN_TRY(upload_cols(b->x1min, in->x1min, in->x1min_stride, sz.n_in, Q, st, &bd.s_x1min, "x1min"));
  NN_TRY(upload_cols(b->x1max, in->x1max, in->x1max_stride, sz.n_in, Q, st, &bd.s_x1max, "x1max"));
  bd.x1min = b->x1min.as<double>();
  bd.x1max = b->x1max.as<double>();
  b->bounds_supplied = (in->ymin != nullptr);
  if (b->bounds_supplied) {
    NN_TRY(upload_cols(b->ymin, in->ymin, in->ymin_stride, sz.acdim, Q, st, &bd.s_ymin, "ymin"));
    NN_TRY(upload_cols(b->ymax, in->ymax, in->ymax_stride, sz.acdim, Q, st, &bd.s_ymax, "ymax"));
    NN_TRY(upload_cols(b->smin, in->smin, in->smin_stride, sz.acdim, Q, st, &bd.s_smin, "smin"));
    NN_TRY(upload_cols(b->smax, in->smax, in->smax_stride, sz.acdim, Q, st, &bd.s_smax, "smax"));
    bd.ymin = b->ymin.as<double>();
    bd.ymax = b->ymax.as<double>();
    bd.smin = b->smin.as<double>();
    bd.smax = b->smax.as<double>();
  } else {  // device IBP: post-activation bounds of x_2..x_K live inside the stacked x bounds
    bd.ymin = b->xmin.as<double>() + sh.n_in();
    bd.ymax = b->xmax.as<double>() + sh.n_in();
    bd.s_ymin = bd.s_ymax = sh.xtot;
    bd.smin = b->smin_c.as<double>();
    bd.smax = b->smax_c.as<double>();
    bd.s_smin = bd.s_smax = sh.acdim;
  }
  if (b->ring > 0) {
    NN_TRY(upload_cols(b->gin, in->gamma_in, in->gamma_in_stride, sz.n_in, Q, st, &bd.s_gin, "gamma_in"));
    NN_TRY(upload_cols(b->gbnd, in->gamma_bnd, in->gamma_bnd_stride, sz.acdim, Q, st, &bd.s_gbnd, "gamma_bnd"));
    NN_TRY(upload_cols(b->gsec, in->gamma_sec, in->gamma_sec_stride, sz.secdim, Q, st, &bd.s_gsec, "gamma_sec"));
    bd.gin = b->gin.as<double>();
    bd.gbnd = b->gbnd.as<double>();
    bd.gsec = b->gsec.as<double>();
    bd.out_kind = in->out_kind;
    bd.outS = bd.outvec = bd.outinvP = bd.gout = nullptr;
    bd.s_outS = bd.s_outvec = bd.s_outinvP = bd.s_gout = 0;
    bd.has_s12 = bd.has_s22 = 0;
    switch (in->out_kind) {
      case NNSDP_OUT_SAFETY: {
        NN_TRY(upload_cols(b->outS, in->out_S, in->out_S_stride, sz.sdim * sz.sdim, Q, st, &bd.s_outS, "out_S"));
        bd.outS = b->outS.as<double>();
        // does any query carry S12 / S22 ?  (upper triangle is authoritative, Symmetric(S))
        const int64_t nq = in->out_S_stride == 0 ? 1 : Q, sd = sz.sdim, ni = sz.n_in, no = sz.n_out;
        for (int64_t q = 0; q < nq && !(bd.has_s12 && bd.has_s22); ++q) {
          const double* S = in->out_S + q * in->out_S_stride;
          for (int64_t c = ni; c < ni + no; ++c) {
            for (int64_t r = 0; r < ni; ++r) bd.has_s12 |= (S[r + c * sd] != 0.0);
            for (int64_t r = ni; r <= c; ++r) bd.has_s22 |= (S[r + c * sd] != 0.0);
          }
        }
        break;
      }
      case NNSDP_OUT_ELLIPSOID:
        NN_TRY(upload_cols(b->outinvP, in->out_invP, in->out_invP_stride, sz.n_out * sz.n_out, Q, st, &bd.s_outinvP, "out_invP"));
        bd.outinvP = b->outinvP.as<double>();
        // fallthrough
      case NNSDP_OUT_CIRCLE:
        bd.has_s22 = 1;
        // fallthrough
      case NNSDP_OUT_HPLANE:
        NN_TRY(upload_cols(b->outvec, in->out_vec, in->out_vec_stride, sz.n_out, Q, st, &bd.s_outvec, "out_vec"));
        NN_TRY(upload_cols(b->gout, in->gamma_out, in->gamma_out_stride, 1, Q, st, &bd.s_gout, "gamma_out"));
        bd.outvec = b->outvec.as<double>();
        bd.gout = b->gout.as<double>();
        break;
      default:
        NN_CHECK(false, NNSDP_ERR_ARG, "unrecognized out_kind %d (src/Qc/output.jl:95)", in->out_kind);
    }
    bd.d11 = b->d11.as<double>();
    bd.Md = b->Md.as<double>();
    bd.T0 = b->T0.as<double>();
    bd.Bt = b->Bt.as<double>();
    bd.u = b->u.as<double>();
    bd.aff = b->aff.as<double>();
    bd.part = b->part.as<double>();
    bd.act = b->act.as<int>();
    bd.cnt = b->cnt.as<int>();
    bd.Z11 = b->Z11.as<double>();
    bd.Z1K = b->Z1K.as<double>();
    bd.U = b->U.as<double>();
  }
  NN_CUDA(cudaStreamSynchronize(st));  // caller may reuse its host buffers after return
  b->have_inputs = true;
  return NNSDP_OK;
}

int32_t nnsdp_batch_bounds(nnsdp_batch* b) {
  NN_CHECK(b != nullptr, NNSDP_ERR_ARG, "batch is NULL");
  NN_CHECK(b->have_inputs, NNSDP_ERR_STATE, "nnsdp_batch_bounds before nnsdp_batch_set_inputs");
  NN_CUDA(cudaSetDevice(b->dev));
  const Shape& sh = b->net->sh;
  const NetPerDev& nd = *b->nd;
  const int Q = (int)b->Q;
  double* xmin = b->xmin.as<double>();
  double* xmax = b->xmax.as<double>();
  b->span_begin(ST_BOUNDS, b->st);
  int launches = 0;
  int max_out = 0;
  for (int k = 1; k <= sh.K; ++k) max_out = std::max(max_out, (int)sh.n[k]);
  const int max_w = std::max(max_out, (int)sh.n[0]);
  int whole = ibp_chain_launch(nd.nd, max_w, b->bd.x1min, b->bd.s_x1min, b->bd.x1max, b->bd.s_x1max, xmin, xmax, sh.xtot,
                               b->acxmin.as<double>(), b->acxmax.as<double>(), b->smin_c.as<double>(),
                               b->smax_c.as<double>(), sh.acdim, Q, nullptr, b->st);
  if (whole == 0)
    whole = ibp_all_launch(nd.nd, max_out, b->bd.x1min, b->bd.s_x1min, b->bd.x1max, b->bd.s_x1max, xmin, xmax,
                           sh.xtot, b->acxmin.as<double>(), b->acxmax.as<double>(), b->smin_c.as<double>(),
                           b->smax_c.as<double>(), sh.acdim, Q, nullptr, b->st);
  NN_CHECK(whole >= 0, NNSDP_ERR_CUDA, "cooperative launch of the interval propagation failed: %s",
           cudaGetErrorString(cudaGetLastError()));
  launches += whole;
  if (whole == 0) {
    launches += launch_place_x1(b->bd.x1min, b->bd.s_x1min, b->bd.x1max, b->bd.s_x1max, xmin, xmax,
                                sh.xtot, (int)sh.n_in(), Q, b->st);
    for (int k = 0; k < sh.K; ++k) {
      const bool last = (k == sh.K - 1);
      launches += ibp_layer_launch(
          nd.M[k].as<double>(), (int)sh.n[k + 1], (int)sh.n[k], xmin + sh.xoff[k], xmax + sh.xoff[k],
          sh.xtot, xmin + sh.xoff[k + 1], xmax + sh.xoff[k + 1],
          last ? nullptr : b->acxmin.as<double>() + sh.noff(k + 1),
          last ? nullptr : b->acxmax.as<double>() + sh.noff(k + 1), sh.acdim, Q, last ? 0 : 1, 1,
          nullptr, b->st);
    }
    launches += launch_sector_minmax(sh.acdim * (long long)Q, b->acxmin.as<double>(),
                                     b->acxmax.as<double>(), b->smin_c.as<double>(),
                                     b->smax_c.as<double>(), b->st);
  }
  b->span_end(b->st, launches);
  NN_CUDA(cudaGetLastError());
  b->bounds_done = true;
  return NNSDP_OK;
}

int32_t nnsdp_batch_prepare(nnsdp_batch* b) {
  NN_CHECK(b != nullptr, NNSDP_ERR_ARG, "batch is NULL");
  NN_CHECK(b->have_inputs, NNSDP_ERR_STATE, "nnsdp_batch_prepare before nnsdp_batch_set_inputs");
  NN_CHECK(b->ring > 0, NNSDP_ERR_STATE, "batch was created without an output ring");
  NN_CHECK(b->bounds_supplied || b->bounds_done, NNSDP_ERR_STATE,
           "nnsdp_batch_prepare needs bounds: supply ymin/ymax/smin/smax or call nnsdp_batch_bounds");
  NN_CUDA(cudaSetDevice(b->dev));
  const Shape& sh = b->net->sh;
  const NetPerDev& nd = *b->nd;
  b->span_begin(ST_PREP, b->st);
  int launches = launch_prep(nd.nd, b->bd, b->flags.as<int>(), b->st);
  int max_rows = 0;
  for (int blk = 0; blk <= sh.K - 2; ++blk) max_rows = std::max(max_rows, (int)sh.n[blk]);
  const int all = affine_all_launch(nd.nd, sh.K, max_rows, b->bd.u, sh.acdim, b->bd.aff, sh.Zdim, (int)b->Q, b->st);
  launches += all;
  // wide layers, many queries: the products of a run of layers [lb0, lb1) in ONE tensor-core launch (a single layer
  // is 64 tiles at width 1000 and Q = 1024, under half of the SMs); the others one by one
  int lb0 = 0, lb1 = 0;
  if (all == 0) {
    auto fits = [&](int blk) {
      return sh.n[blk] >= 192 && sh.n[blk + 1] >= 128 && (sh.noff(blk + 1) & 1) == 0 && (sh.acdim & 1) == 0 &&
             (((uintptr_t)b->bd.u) & 15) == 0;
    };
    int best0 = 0, best1 = 0;
    for (int s = 0; s <= sh.K - 2;) {
      if (!fits(s)) { ++s; continue; }
      int e = s;
      while (e <= sh.K - 2 && fits(e)) ++e;
      if (e - s > best1 - best0) best0 = s, best1 = e;
      s = e;
    }
    int rows = 0;
    for (int blk = best0; blk < best1; ++blk) rows = std::max(rows, (int)sh.n[blk]);
    if (best1 - best0 >= 2 && dgemm_dmma_affine_layers_launch(nd.nd, best0, best1 - best0, rows, b->bd.u, sh.acdim, b->bd.aff,
                                                              sh.Zdim, (int)b->Q, b->st)) {
      lb0 = best0, lb1 = best1;
      ++launches;
    }
  }
  if (all == 0)
    for (int blk = 0; blk <= sh.K - 2; ++blk)
      if (blk < lb0 || blk >= lb1)
        launches += affine_layer_launch(nd.Wt[blk].as<double>(), b->net->ldT[blk], (int)sh.n[blk],
                                      (int)sh.n[blk + 1], b->bd.u + sh.noff(blk + 1), sh.acdim,
                                      b->bd.aff + sh.off[blk], sh.Zdim, (int)b->Q, b->st);
  b->span_end(b->st, launches);
  NN_CUDA(cudaGetLastError());
  // Gram-active neuron counts per (query, block): the host builds the work list of the Gram kernel from them
  // (most (query, layer) pairs have no stably-active neuron) and the host gather needs them as well
  b->h_cnt.resize((size_t)sh.K * b->Q);
  NN_CUDA(cudaMemcpyAsync(b->h_cnt.data(), b->cnt.p, b->h_cnt.size() * 4, cudaMemcpyDeviceToHost, b->st));
  NN_TRY(check_flags(b, "nnsdp_batch_prepare"));  // synchronises the stream
  b->h_pairs.clear();
  b->pair_begin.assign((size_t)b->Q + 1, 0);
  for (int64_t q = 0; q < b->Q; ++q) {
    for (int blk = 0; blk <= sh.K - 2; ++blk)
      if (b->h_cnt[(size_t)q * sh.K + blk] > 0) {
        b->h_pairs.push_back((int)q);
        b->h_pairs.push_back(blk);
      }
    b->pair_begin[q + 1] = (int64_t)b->h_pairs.size() / 2;
  }
  NN_TRY(upload(b->d_pairs, b->h_pairs.data(), b->h_pairs.size() * 4, b->st));
  // A reach batch (src/NnSdp.jl:73-95) shares the box, the bounds and every multiplier but gamma_out between
  // its queries: the Gram blocks are then the same for all of them and are contracted once, into slot 0.
  const BatchDev& bd = b->bd;
  b->shared_gram = b->Q > 1 && bd.s_gsec == 0 &&
                   (b->bounds_supplied ? (bd.s_smin == 0 && bd.s_smax == 0) : (bd.s_x1min == 0 && bd.s_x1max == 0));
  b->prepared = true;
  return NNSDP_OK;
}

// Ring slots keep what earlier passes stored in them.  A slot is zeroed the first time a pass uses it; after that the
// SAME / DIAG strips of block Br are stored into slot s only when the query of this pass or the slot's previous query
// has a non-zero bulk there (the Gram of a layer with a stably-active neuron; W_K' S22 W_K for Br = K-1).  Everything
// else a pass launches is stored for every query.  The pairs to store go to b->sel; slots are physical positions in
// the ring (dst = ring + p0 slots), queries [q0, q0 + nq) go to slots p0 .. p0 + nq - 1.
static int32_t prepare_slots(nnsdp_batch* b, int64_t q0, int64_t nq, int64_t p0) {
  const int64_t per = b->plan.per_query_doubles;
  const int K = b->net->sh.K;
  if (p0 + nq > b->ring_zeroed) {
    NN_CUDA(cudaMemsetAsync(b->ringbuf.as<double>() + b->ring_zeroed * per, 0, (size_t)(p0 + nq - b->ring_zeroed) * per * 8,
                            b->st));
    std::fill(b->slot_bulk.begin() + b->ring_zeroed * K, b->slot_bulk.begin() + (p0 + nq) * K, 0);
    b->ring_zeroed = p0 + nq;
  }
  b->sel.clear();
  int64_t entries = b->pass_entries * nq;
  for (int64_t i = 0; i < nq; ++i) {
    const int64_t q = q0 + i;
    uint8_t* held = &b->slot_bulk[(size_t)(p0 + i) * K];
    for (int blk = 1; blk < K; ++blk) {
      const int first = b->bulk_begin[blk], count = b->bulk_begin[blk + 1] - first;
      if (count == 0) continue;
      const bool now = blk <= K - 2 ? b->h_cnt[(size_t)q * K + blk] > 0 : b->bd.has_s22 != 0;
      if (now || held[blk]) {
        b->sel.push_back({(int32_t)i, first, count});
        entries += b->bulk_entries[blk];
      }
      held[blk] = now;
    }
  }
  if (!b->packed) b->emitted_bytes += entries * 8;
  return NNSDP_OK;
}

// One emitter pass = fill, window and edge kernels back to back, each inside its own CUDA-event span
// (ST_EMIT_FILL / _WINDOW / _EDGE) so that the per-kernel launch durations can be read back.
static int32_t emit_pass(nnsdp_batch* b, const GramDev& gd, int q0, int nq, double* dst) {
  const NetPerDev& nd = *b->nd;
  NN_TRY(prepare_slots(b, q0, nq, (dst - b->ringbuf.as<double>()) / b->plan.per_query_doubles));
  int total = 0;
  for (int which = 0; which < 3; ++which) {
    b->span_begin(ST_EMIT_FILL + which, b->st);
    const int l = launch_emit(nd.nd, b->bd, gd, b->pd, q0, nq, dst, b->st, which, b->sel.data(), (int)b->sel.size());
    b->span_end(b->st, l);
    total += l;
  }
  if (b->nbands > 0) {  // after the fill kernel: in-place band of the DIAG ranges (wide layers), BAND cells (packed)
    b->span_begin(ST_EMIT_EDGE, b->st);
    const int l = launch_emit_band(nd.nd, b->bd, gd, b->d_bands.as<BandDev>(), b->nbands, b->band_max_m, b->pd.per_query,
                                   q0, nq, dst, b->st);
    b->span_end(b->st, l);
    total += l;
  }
  b->stage_launches[ST_EMIT] += total;
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    b->ring_zeroed = 0;  // the slots may not hold what the state says: zero them again on next use
    return cuda_fail(e, "emitter pass", __FILE__, __LINE__);
  }
  return NNSDP_OK;
}

int32_t nnsdp_batch_emit(nnsdp_batch* b, int64_t q0, int64_t nq) {
  NN_CHECK(b != nullptr, NNSDP_ERR_ARG, "batch is NULL");
  NN_CHECK(b->prepared, NNSDP_ERR_STATE, "nnsdp_batch_emit before nnsdp_batch_prepare");
  NN_CHECK(q0 >= 0 && nq >= 1 && q0 + nq <= b->Q && nq <= b->ring, NNSDP_ERR_ARG,
           "bad query range [%lld, %lld) for Q = %lld, ring = %lld", (long long)q0,
           (long long)(q0 + nq), (long long)b->Q, (long long)b->ring);
  NN_CUDA(cudaSetDevice(b->dev));
  const NetPerDev& nd = *b->nd;
  GramDev gd = b->gd;
  b->span_begin(ST_GRAM, b->st);
  int l;
  if (b->shared_gram) {  // query 0's Gram blocks serve every query: every slot reads slot 0
    l = launch_gram(nd.nd, b->bd, gd, (int)b->net->max_block, 0, b->d_pairs.as<int>(), (int)b->pair_begin[1], b->st);
    gd.per_query = 0;
  } else {
    l = launch_gram(nd.nd, b->bd, gd, (int)b->net->max_block, (int)q0, b->d_pairs.as<int>() + 2 * b->pair_begin[q0],
                    (int)(b->pair_begin[q0 + nq] - b->pair_begin[q0]), b->st);
  }
  b->span_end(b->st, l > 0 ? l : 0);
  NN_CHECK(l >= 0, NNSDP_ERR_ARG, "a hidden layer of %lld neurons is too wide for the Gram kernel's grid", (long long)b->net->max_block);
  NN_CUDA(cudaGetLastError());
  NN_TRY(emit_pass(b, gd, (int)q0, (int)nq, b->ringbuf.as<double>()));
  return NNSDP_OK;
}

int32_t nnsdp_batch_sync(nnsdp_batch* b) {
  NN_CHECK(b != nullptr, NNSDP_ERR_ARG, "batch is NULL");
  NN_CUDA(cudaSetDevice(b->dev));
  NN_CUDA(cudaStreamSynchronize(b->st));
  NN_CUDA(cudaStreamSynchronize(b->st_copy));
  b->resolve_spans();
  return NNSDP_OK;
}

// Sparse host gather of the queries [q0, q0 + nq) of chunk `ci` whose blocks sit in ring slots starting
// at `dst`: strided DMA of the dense cells, packed copy of the thin entries, host-side zero fill +
// scatter on the worker threads.  Everything is asynchronous; the caller drains pool and streams.
static int32_t gather_chunk(nnsdp_batch* b, int ci, int64_t q0, int64_t nq, int h, const double* dst,
                            double* host_out, int32_t flags) {
  const GatherPlan& gp = b->gp;
  const int64_t per = b->plan.per_query_doubles;
  const int64_t nthin = (int64_t)gp.thin_idx.size();
  const int sb = ci % GATHER_STAGES;
  const int K = b->net->sh.K;
  const bool prezeroed = (flags & NNSDP_RUN_HOST_PREZEROED) != 0;
  const int64_t chunk_cap = std::max<int64_t>(1, b->ring / 2);
  double* d_pk = b->d_packed.as<double>() + (int64_t)sb * chunk_cap * nthin;
  double* h_pk = b->h_packed + (int64_t)sb * chunk_cap * nthin;
  launch_pack_thin(dst, per, b->d_thin_idx.as<long long>(), nthin, d_pk, (int)nq, b->st);
  NN_CUDA(cudaEventRecord(b->ev_done[h], b->st));
  NN_CUDA(cudaStreamWaitEvent(b->st_copy, b->ev_done[h], 0));
  b->span_begin(ST_D2H, b->st_copy);
  if (nthin) NN_CUDA(cudaMemcpyAsync(h_pk, d_pk, (size_t)nq * nthin * 8, cudaMemcpyDeviceToHost, b->st_copy));
  NN_CUDA(cudaEventRecord(b->ev_packed[sb], b->st_copy));
  // Large cells that are NOT dense for this query hold zeros in the ring (plus thin entries, which are
  // scattered afterwards in any case).  The copy engine idles most of the time while the host threads
  // zero-fill, so a share of those cells is copied as well: both then finish at about the same time.
  static const int dma_zero_pct = [] {
    const char* e = getenv("NNSDP_GATHER_DMA_ZERO_PCT");
    const int v = e ? atoi(e) : 20;
    return v < 0 ? 0 : (v > 100 ? 100 : v);
  }();
  auto dense_now = [&](const GatherCell& c, int64_t q) {
    return c.kind == GK_ALWAYS || (c.kind == GK_GRAM && b->h_cnt[q * K + c.blk] > 0) ||
           (c.kind == GK_S22 && b->bd.has_s22);
  };
  auto active = [&](const GatherCell& c, int64_t q) {
    if (dense_now(c, q)) return true;
    if (std::min<int64_t>(c.nrows, c.ncols_hint) < GATHER_MIN_RECT) return false;
    if (prezeroed) return false;  // little is left to zero-fill: the host threads keep up without help
    // deterministic pseudo-random share, independent of the order of evaluation
    const uint64_t hsh = ((uint64_t)q * 1315423911u) ^ ((uint64_t)c.row0 * 2654435761u) ^ ((uint64_t)c.col0_hint * 97u);
    return (int)((hsh >> 7) % 100) < dma_zero_pct;
  };
  for (int64_t q = q0; q < q0 + nq; ++q) {
    const double* src = dst + (q - q0) * per;
    double* out = host_out + q * per;
    for (const GatherColSeg& cs : gp.colsegs) {
      const MatDev& md = b->plan.mats[cs.mat];
      for (const GatherCell& c : cs.cells) {
        if (!active(c, q)) continue;
        const int64_t off = md.out_off + c.row0 + (int64_t)cs.col0 * md.ld;
        NN_CUDA(cudaMemcpy2DAsync(out + off, (size_t)md.ld * 8, src + off, (size_t)md.ld * 8,
                                  (size_t)c.nrows * 8, (size_t)cs.ncols, cudaMemcpyDeviceToHost, b->st_copy));
        b->gather_bytes_dma += (int64_t)c.nrows * cs.ncols * 8;
      }
    }
  }
  b->span_end(b->st_copy, 0);
  NN_CUDA(cudaEventRecord(b->ev_free[h], b->st_copy));
  b->gather_bytes_thin += nq * nthin * 8;
  // host side: one task per (query, matrix)
  const int nm = (int)b->plan.mats.size();
  cudaEvent_t ev = b->ev_packed[sb];
  const int dev = b->dev;
  for (int64_t q = q0; q < q0 + nq; ++q) {
    for (int m = 0; m < nm; ++m) {
      double* out = host_out + q * per;
      const double* pk = h_pk + (q - q0) * nthin;
      // what to zero is decided here (cheap) so the task needs no access to mutable batch state
      struct Run { int64_t off; int32_t nrows, ncols, ld; };
      std::vector<Run> runs;
      const MatDev& md = b->plan.mats[m];
      for (int s = gp.colseg_begin[m]; s < gp.colseg_begin[m + 1]; ++s) {
        const GatherColSeg& cs = gp.colsegs[s];
        int32_t run0 = -1, runlen = 0;
        auto flush = [&] {
          if (runlen > 0) {
            runs.push_back({md.out_off + run0 + (int64_t)cs.col0 * md.ld, runlen, cs.ncols, md.ld});
            b->gather_bytes_zeroed += (int64_t)runlen * cs.ncols * 8;
          }
          run0 = -1;
          runlen = 0;
        };
        for (const GatherCell& c : cs.cells) {
          const bool skip = active(c, q) || (prezeroed && c.pure_zero);
          if (skip) {
            flush();
            continue;
          }
          if (runlen > 0 && run0 + runlen == c.row0) {
            runlen += c.nrows;
          } else {
            flush();
            run0 = c.row0;
            runlen = c.nrows;
          }
        }
        flush();
      }
      const int64_t t0 = gp.thin_begin[m], t1 = gp.thin_begin[m + 1];
      const int64_t* idx = gp.thin_idx.data();
      b->pool->submit(ci, [=, runs = std::move(runs)] {
        for (const Run& r : runs)
          for (int32_t c = 0; c < r.ncols; ++c) memset(out + r.off + (int64_t)c * r.ld, 0, (size_t)r.nrows * 8);
        if (t1 > t0) {
          cudaSetDevice(dev);
          cudaEventSynchronize(ev);
          for (int64_t i = t0; i < t1; ++i) out[idx[i]] = pk[i];
        }
      });
    }
  }
  return NNSDP_OK;
}

extern "C" int32_t nnsdp_batch_bounds_crown(nnsdp_batch* b);

static int32_t run_impl(nnsdp_batch* b, double* host_out, uint8_t* present, int32_t flags) {
  NN_CHECK(b != nullptr, NNSDP_ERR_ARG, "batch is NULL");
  NN_CHECK(b->have_inputs, NNSDP_ERR_STATE, "nnsdp_batch_run before nnsdp_batch_set_inputs");
  NN_CHECK(b->ring > 0, NNSDP_ERR_STATE, "batch was created without an output ring");
  NN_CUDA(cudaSetDevice(b->dev));
  if (!b->bounds_supplied) NN_TRY(b->bounds_method == 1 ? nnsdp_batch_bounds_crown(b) : nnsdp_batch_bounds(b));
  NN_TRY(nnsdp_batch_prepare(b));
  const NetPerDev& nd = *b->nd;
  const int64_t per = b->plan.per_query_doubles;
  // the ring is used as two halves so the device->host copy of one half overlaps the
  // emission of the other
  const int nhalf = (host_out && b->ring >= 2) ? 2 : 1;
  const int64_t chunk = (nhalf == 2) ? b->ring / 2 : b->ring;
  const bool sparse = host_out && !b->packed && b->gp.usable && !(flags & NNSDP_RUN_DENSE_COPY);
  b->gather_bytes_dma = b->gather_bytes_zeroed = b->gather_bytes_thin = 0;
  b->emitted_bytes = b->packed_present_cells = 0;
  const int K = b->net->sh.K;
  const size_t ncells = b->lay.cells.size();
  // packed records: which DIAG cells a query carries is known from the Gram-active counts of prepare
  auto cell_present = [&](int64_t q, const PackedCell& c) {
    if (c.always) return true;
    return c.blk <= K - 2 ? b->h_cnt[(size_t)q * K + c.blk] > 0 : b->bd.has_s22 != 0;
  };
  int64_t zero_entries = 0;  // structurally zero tiles of the record: zeroed once with the ring slot, never stored
  if (b->packed)
    for (int i = 0; i < b->plan.n_fill; ++i)
      if (b->plan.tiles[i].prog == PROG_ZERO) zero_entries += (int64_t)b->plan.tiles[i].nrows * b->plan.tiles[i].ncols;
  if (b->packed)
    for (int64_t q = 0; q < b->Q; ++q) {
      int64_t ent = b->lay.always_entries - zero_entries;
      for (size_t i = 0; i < ncells; ++i) {
        const PackedCell& c = b->lay.cells[i];
        const bool p = cell_present(q, c);
        if (present) present[(size_t)q * ncells + i] = p ? 1 : 0;
        if (!c.always && p) ent += b->plan.skip_absent ? b->lay.diag_entries[c.blk] : 0, ++b->packed_present_cells;
      }
      b->emitted_bytes += ent * 8;
    }
  if (sparse) {
    const size_t need = (size_t)GATHER_STAGES * chunk * b->gp.thin_idx.size();
    if (need > b->h_packed_doubles) {
      if (b->h_packed) cudaFreeHost(b->h_packed);
      b->h_packed = nullptr;
      b->h_packed_doubles = 0;
      NN_CUDA(cudaHostAlloc((void**)&b->h_packed, std::max<size_t>(need, 1) * 8, cudaHostAllocPortable));
      b->h_packed_doubles = need;
      NN_TRY(b->d_packed.ensure(std::max<size_t>(need, 1) * 8));
    }
    if (!b->pool) {
      int nt = (int)std::min<unsigned>(16u, std::max(1u, std::thread::hardware_concurrency()));
      if (const char* e = getenv("NNSDP_HOST_THREADS")) nt = std::max(1, atoi(e));
      b->pool.reset(new WorkerPool(nt));
    }
  }
  bool used[2] = {false, false};
  int h = 0, ci = 0;
  int32_t status = NNSDP_OK;
  for (int64_t q0 = 0; q0 < b->Q && status == NNSDP_OK; q0 += chunk, h = (h + 1) % nhalf, ++ci) {
    const int64_t nq = std::min(chunk, b->Q - q0);
    double* dst = b->ringbuf.as<double>() + (int64_t)h * chunk * per;
    GramDev gd = b->gd;
    if (b->shared_gram) gd.per_query = 0;  // every slot reads the Gram blocks of query 0 (contracted once, below)
    else gd.scratch += (int64_t)h * chunk * gd.per_query;
    if (sparse && ci >= GATHER_STAGES) b->pool->wait_group(ci - GATHER_STAGES);  // staging buffer reuse
    if (host_out && used[h]) NN_CUDA(cudaStreamWaitEvent(b->st, b->ev_free[h], 0));
    if (!b->shared_gram || ci == 0) {
      b->span_begin(ST_GRAM, b->st);
      int l = b->shared_gram
                  ? launch_gram(nd.nd, b->bd, b->gd, (int)b->net->max_block, 0, b->d_pairs.as<int>(), (int)b->pair_begin[1], b->st)
                  : launch_gram(nd.nd, b->bd, gd, (int)b->net->max_block, (int)q0, b->d_pairs.as<int>() + 2 * b->pair_begin[q0],
                                (int)(b->pair_begin[q0 + nq] - b->pair_begin[q0]), b->st);
      b->span_end(b->st, l > 0 ? l : 0);
      NN_CHECK(l >= 0, NNSDP_ERR_ARG, "a hidden layer of %lld neurons is too wide for the Gram kernel's grid",
               (long long)b->net->max_block);
      NN_CUDA(cudaGetLastError());  // a failed Gram launch must not go unnoticed until the emitter has read its scratch
    }
    status = emit_pass(b, gd, (int)q0, (int)nq, dst);
    if (status != NNSDP_OK) break;
    if (sparse) {
      status = gather_chunk(b, ci, q0, nq, h, dst, host_out, flags);
      used[h] = true;
    } else if (host_out && b->packed && !(flags & NNSDP_RUN_DENSE_COPY)) {
      // packed records: the always-written part of all records of the chunk is one strided copy, every DIAG
      // cell a query carries one contiguous copy; absent cells are not moved (and the host bytes not touched)
      NN_CUDA(cudaEventRecord(b->ev_done[h], b->st));
      NN_CUDA(cudaStreamWaitEvent(b->st_copy, b->ev_done[h], 0));
      b->span_begin(ST_D2H, b->st_copy);
      const int64_t alw = b->lay.always_doubles;
      if (alw == per)
        NN_CUDA(cudaMemcpyAsync(host_out + q0 * per, dst, (size_t)nq * per * 8, cudaMemcpyDeviceToHost, b->st_copy));
      else
        NN_CUDA(cudaMemcpy2DAsync(host_out + q0 * per, (size_t)per * 8, dst, (size_t)per * 8, (size_t)alw * 8, (size_t)nq,
                                  cudaMemcpyDeviceToHost, b->st_copy));
      b->gather_bytes_dma += nq * alw * 8;
      for (int64_t q = q0; q < q0 + nq; ++q)
        for (size_t i = 0; i < ncells; ++i) {
          const PackedCell& c = b->lay.cells[i];
          if (c.always || !cell_present(q, c)) continue;
          const int64_t cells_doubles = c.nrows * c.ncols;
          NN_CUDA(cudaMemcpyAsync(host_out + q * per + c.offset, dst + (q - q0) * per + c.offset, (size_t)cells_doubles * 8,
                                  cudaMemcpyDeviceToHost, b->st_copy));
          b->gather_bytes_dma += cells_doubles * 8;
        }
      b->span_end(b->st_copy, 0);
      NN_CUDA(cudaEventRecord(b->ev_free[h], b->st_copy));
      used[h] = true;
    } else if (host_out) {
      NN_CUDA(cudaEventRecord(b->ev_done[h], b->st));
      NN_CUDA(cudaStreamWaitEvent(b->st_copy, b->ev_done[h], 0));
      b->span_begin(ST_D2H, b->st_copy);
      NN_CUDA(cudaMemcpyAsync(host_out + q0 * per, dst, (size_t)nq * per * 8, cudaMemcpyDeviceToHost,
                              b->st_copy));
      b->span_end(b->st_copy, 0);
      NN_CUDA(cudaEventRecord(b->ev_free[h], b->st_copy));
      used[h] = true;
      b->gather_bytes_dma += nq * per * 8;
    }
  }
  if (b->pool) b->pool->wait_all();
  if (status != NNSDP_OK) {
    cudaStreamSynchronize(b->st);
    cudaStreamSynchronize(b->st_copy);
    return status;
  }
  NN_CUDA(cudaGetLastError());
  NN_CUDA(cudaStreamSynchronize(b->st));
  NN_CUDA(cudaStreamSynchronize(b->st_copy));
  b->resolve_spans();
  return NNSDP_OK;
}

int32_t nnsdp_batch_run_ex(nnsdp_batch* b, double* host_out, int32_t flags) { return run_impl(b, host_out, nullptr, flags); }

int32_t nnsdp_batch_run(nnsdp_batch* b, double* host_out) { return run_impl(b, host_out, nullptr, 0); }

int32_t nnsdp_batch_run_packed(nnsdp_batch* b, double* host_records, uint8_t* present, int32_t flags) {
  NN_CHECK(b != nullptr, NNSDP_ERR_ARG, "batch is NULL");
  NN_CHECK(b->packed, NNSDP_ERR_STATE, "the batch was not created with NNSDP_FORMAT_PACKED");
  return run_impl(b, host_records, present, flags);
}

int32_t nnsdp_batch_packed_stats(nnsdp_batch* b, int64_t* record_doubles, int64_t* ncells, int64_t* emitted_bytes,
                                 int64_t* d2h_bytes, int64_t* present_optional_cells) {
  NN_CHECK(b != nullptr, NNSDP_ERR_ARG, "batch is NULL");
  NN_CHECK(b->packed, NNSDP_ERR_STATE, "the batch was not created with NNSDP_FORMAT_PACKED");
  if (record_doubles) *record_doubles = b->lay.record_doubles;
  if (ncells) *ncells = (int64_t)b->lay.cells.size();
  if (emitted_bytes) *emitted_bytes = b->emitted_bytes;
  if (d2h_bytes) *d2h_bytes = b->gather_bytes_dma;
  if (present_optional_cells) *present_optional_cells = b->packed_present_cells;
  return NNSDP_OK;
}

int32_t nnsdp_batch_emit_stats(nnsdp_batch* b, int64_t* emitted_bytes) {
  NN_CHECK(b && emitted_bytes, NNSDP_ERR_ARG, "NULL argument");
  *emitted_bytes = b->emitted_bytes;
  return NNSDP_OK;
}

/* Bytes moved by the host gather of the last nnsdp_batch_run*: strided / dense DMA, packed thin
 * entries, and bytes zero-filled by host threads. */
int32_t nnsdp_batch_gather_stats(nnsdp_batch* b, int64_t* dma_bytes, int64_t* thin_bytes,
                                 int64_t* zeroed_bytes, int32_t* sparse_usable) {
  NN_CHECK(b != nullptr, NNSDP_ERR_ARG, "batch is NULL");
  if (dma_bytes) *dma_bytes = b->gather_bytes_dma;
  if (thin_bytes) *thin_bytes = b->gather_bytes_thin;
  if (zeroed_bytes) *zeroed_bytes = b->gather_bytes_zeroed;
  if (sparse_usable) *sparse_usable = b->gp.usable ? 1 : 0;
  return NNSDP_OK;
}

int32_t nnsdp_batch_get_bounds(nnsdp_batch* b, double* xmin, double* xmax, double* acxmin,
                               double* acxmax, double* smin, double* smax) {
  NN_CHECK(b != nullptr, NNSDP_ERR_ARG, "batch is NULL");
  NN_CHECK(b->bounds_done, NNSDP_ERR_STATE, "bounds have not been computed on the device");
  NN_CUDA(cudaSetDevice(b->dev));
  const Shape& sh = b->net->sh;
  const size_t Q = (size_t)b->Q;
  auto get = [&](double* dst, const DevBuf& src, size_t len) -> int32_t {
    if (dst) NN_CUDA(cudaMemcpyAsync(dst, src.p, len * Q * 8, cudaMemcpyDeviceToHost, b->st));
    return NNSDP_OK;
  };
  NN_TRY(get(xmin, b->xmin, sh.xtot));
  NN_TRY(get(xmax, b->xmax, sh.xtot));
  NN_TRY(get(acxmin, b->acxmin, sh.acdim));
  NN_TRY(get(acxmax, b->acxmax, sh.acdim));
  NN_TRY(get(smin, b->smin_c, sh.acdim));
  NN_TRY(get(smax, b->smax_c, sh.acdim));
  NN_CUDA(cudaStreamSynchronize(b->st));
  return NNSDP_OK;
}

int32_t nnsdp_batch_get_slot(nnsdp_batch* b, int64_t slot, double* host_out) {
  NN_CHECK(b && host_out, NNSDP_ERR_ARG, "NULL argument");
  NN_CHECK(slot >= 0 && slot < b->ring, NNSDP_ERR_ARG, "slot out of range");
  NN_CUDA(cudaSetDevice(b->dev));
  const int64_t per = b->plan.per_query_doubles;
  NN_CUDA(cudaMemcpyAsync(host_out, b->ringbuf.as<double>() + slot * per, (size_t)per * 8,
                          cudaMemcpyDeviceToHost, b->st));
  NN_CUDA(cudaStreamSynchronize(b->st));
  return NNSDP_OK;
}

int32_t nnsdp_batch_get_affine(nnsdp_batch* b, double* aff_out) {
  NN_CHECK(b && aff_out, NNSDP_ERR_ARG, "NULL argument");
  NN_CHECK(b->prepared, NNSDP_ERR_STATE, "batch is not prepared");
  NN_CUDA(cudaSetDevice(b->dev));
  NN_CUDA(cudaMemcpyAsync(aff_out, b->aff.p, (size_t)b->net->sh.Zdim * b->Q * 8,
                          cudaMemcpyDeviceToHost, b->st));
  NN_CUDA(cudaStreamSynchronize(b->st));
  return NNSDP_OK;
}

int32_t nnsdp_batch_ring_ptr(nnsdp_batch* b, uint64_t* dev_ptr, int64_t* slot_doubles) {
  NN_CHECK(b != nullptr, NNSDP_ERR_ARG, "batch is NULL");
  if (dev_ptr) *dev_ptr = (uint64_t)(uintptr_t)b->ringbuf.p;
  if (slot_doubles) *slot_doubles = b->plan.per_query_doubles;
  return NNSDP_OK;
}

int32_t nnsdp_batch_ring_reset(nnsdp_batch* b) {
  NN_CHECK(b != nullptr, NNSDP_ERR_ARG, "batch is NULL");
  b->ring_zeroed = 0;
  return NNSDP_OK;
}

int32_t nnsdp_batch_event_record(nnsdp_batch* b, int32_t which) {
  NN_CHECK(b != nullptr, NNSDP_ERR_ARG, "batch is NULL");
  NN_CUDA(cudaSetDevice(b->dev));
  NN_CUDA(cudaEventRecord(which == 0 ? b->ev_start : b->ev_stop, b->st));
  return NNSDP_OK;
}

int32_t nnsdp_batch_elapsed_ms(nnsdp_batch* b, float* ms) {
  NN_CHECK(b && ms, NNSDP_ERR_ARG, "NULL argument");
  NN_CUDA(cudaSetDevice(b->dev));
  NN_CUDA(cudaEventSynchronize(b->ev_stop));
  NN_CUDA(cudaEventElapsedTime(ms, b->ev_start, b->ev_stop));
  return NNSDP_OK;
}

int32_t nnsdp_batch_stage_ms(nnsdp_batch* b, int32_t stage, float* ms, int64_t* launches) {
  NN_CHECK(b != nullptr, NNSDP_ERR_ARG, "batch is NULL");
  NN_CHECK(stage >= 0 && stage < ST_COUNT, NNSDP_ERR_ARG, "bad stage");
  NN_TRY(nnsdp_batch_sync(b));
  if (ms) *ms = b->stage_ms[stage];
  if (launches) *launches = b->stage_launches[stage];
  return NNSDP_OK;
}

int32_t nnsdp_batch_stage_reset(nnsdp_batch* b) {
  NN_CHECK(b != nullptr, NNSDP_ERR_ARG, "batch is NULL");
  NN_TRY(nnsdp_batch_sync(b));
  for (int i = 0; i < ST_COUNT; ++i) b->stage_ms[i] = 0.f, b->stage_launches[i] = 0;
  return NNSDP_OK;
}

int32_t nnsdp_batch_gram_stats(nnsdp_batch* b, int64_t* n_contractions, int64_t* sum_active) {
  NN_CHECK(b != nullptr, NNSDP_ERR_ARG, "batch is NULL");
  NN_CHECK(b->prepared, NNSDP_ERR_STATE, "batch is not prepared");
  NN_CUDA(cudaSetDevice(b->dev));
  const int K = b->net->sh.K;
  std::vector<int> cnt((size_t)K * b->Q);
  NN_CUDA(cudaMemcpyAsync(cnt.data(), b->cnt.p, cnt.size() * 4, cudaMemcpyDeviceToHost, b->st));
  NN_CUDA(cudaStreamSynchronize(b->st));
  int64_t nc = 0, sa = 0;
  for (int64_t q = 0; q < b->Q; ++q)
    for (int blk = 0; blk <= K - 2; ++blk) {
      const int c = cnt[q * K + blk];
      if (c > 0) ++nc, sa += c;
    }
  if (n_contractions) *n_contractions = nc;
  if (sum_active) *sum_active = sa;
  return NNSDP_OK;
}

}  // extern "C"

// ---- one-shot entry points --------------------------------------------------------------------
namespace {

// Split Q queries over the devices of ctx in contiguous ranges and run fn(dev_index, q0, nq) with
// one host thread per device.  Errors of worker threads are forwarded to the caller's thread.
template <class F>
int32_t shard_queries(nnsdp_ctx* ctx, int64_t Q, F fn) {
  const int nd = (int)ctx->devs.size();
  if (nd == 1 || Q < nd) return fn(0, (int64_t)0, Q);
  std::vector<int32_t> status(nd, NNSDP_OK);
  std::vector<std::string> errs(nd);
  std::vector<std::thread> th;
  const int64_t base = Q / nd, rem = Q % nd;
  int64_t q0 = 0;
  for (int d = 0; d < nd; ++d) {
    const int64_t nq = base + (d < rem ? 1 : 0);
    th.emplace_back([&, d, q0, nq]() {
      status[d] = fn(d, q0, nq);
      if (status[d] != NNSDP_OK) errs[d] = nnsdp_last_error();
    });
    q0 += nq;
  }
  for (auto& t : th) t.join();
  for (int d = 0; d < nd; ++d)
    if (status[d] != NNSDP_OK) {
      set_error("device %d: %s", ctx->devs[d], errs[d].c_str());
      return status[d];
    }
  return NNSDP_OK;
}

// A batch for a one-shot call: taken from the network's cache when one with the same (device, beta, kind)
// and enough capacity is idle, created otherwise; handed back on release if it is small enough to keep.
struct BatchHolder {
  nnsdp_batch* b = nullptr;
  const nnsdp_net* net = nullptr;
  nnsdp_net::Cached key{};
  bool keep = false;
  int32_t acquire(nnsdp_ctx* ctx, int d, const nnsdp_net* n, int64_t beta, int64_t Q, int64_t ring, int dense) {
    net = n;
    key = {d, beta, Q, ring, dense, nullptr};
    {
      std::lock_guard<std::mutex> l(n->cache_mu);
      for (size_t i = 0; i < n->cache.size(); ++i) {
        const auto& c = n->cache[i];
        if (c.dev_index == d && c.beta == beta && c.dense == dense && c.Qcap >= Q && c.ring >= std::min(ring, Q) &&
            (ring > 0) == (c.ring > 0)) {
          b = c.b;
          key = c;
          n->cache.erase(n->cache.begin() + i);
          keep = true;
          return NNSDP_OK;
        }
      }
    }
    NN_TRY(nnsdp_batch_create(ctx, d, n, beta, Q, ring, dense, &b));
    key.b = b;
    // keep only batches whose device footprint is modest (the ring of a wide net is gigabytes)
    keep = (b->plan.per_query_doubles * std::max<int64_t>(b->ring, 1) + (int64_t)n->sh.Zdim * Q * 16) * 8 <= (int64_t(512) << 20);
    return NNSDP_OK;
  }
  ~BatchHolder() {
    if (!b) return;
    if (keep) {
      std::lock_guard<std::mutex> l(net->cache_mu);
      if (net->cache.size() >= 6) {  // drop the oldest
        nnsdp_batch_destroy(net->cache.front().b);
        net->cache.erase(net->cache.begin());
      }
      key.b = b;
      net->cache.push_back(key);
    } else {
      nnsdp_batch_destroy(b);
    }
  }
};

const double* col(const double* p, int64_t stride, int64_t q0) { return p ? p + stride * q0 : p; }

nnsdp_query_inputs shift_inputs(const nnsdp_query_inputs& in, int64_t q0) {
  nnsdp_query_inputs o = in;
  o.x1min = col(in.x1min, in.x1min_stride, q0);
  o.x1max = col(in.x1max, in.x1max_stride, q0);
  o.ymin = col(in.ymin, in.ymin_stride, q0);
  o.ymax = col(in.ymax, in.ymax_stride, q0);
  o.smin = col(in.smin, in.smin_stride, q0);
  o.smax = col(in.smax, in.smax_stride, q0);
  o.gamma_in = col(in.gamma_in, in.gamma_in_stride, q0);
  o.gamma_bnd = col(in.gamma_bnd, in.gamma_bnd_stride, q0);
  o.gamma_sec = col(in.gamma_sec, in.gamma_sec_stride, q0);
  o.out_S = col(in.out_S, in.out_S_stride, q0);
  o.out_vec = col(in.out_vec, in.out_vec_stride, q0);
  o.out_invP = col(in.out_invP, in.out_invP_stride, q0);
  o.gamma_out = col(in.gamma_out, in.gamma_out_stride, q0);
  return o;
}

int32_t assemble_impl(nnsdp_ctx* ctx, const nnsdp_net* net, int64_t beta, int64_t Q,
                      const nnsdp_query_inputs* in, double* out, int dense) {
  NN_CHECK(ctx && net && in && out, NNSDP_ERR_ARG, "NULL argument");
  NN_CHECK(Q >= 1, NNSDP_ERR_ARG, "Q must be >= 1");
  nnsdp_sizes sz;
  NN_TRY(fill_sizes(net->sh, beta, &sz));
  const int64_t per = dense ? sz.Zdim * sz.Zdim : sz.sum_ck_sq;
  return shard_queries(ctx, Q, [&](int d, int64_t q0, int64_t nq) -> int32_t {
    // ring: two halves of up to ~2 GiB each, at least one query per half
    int64_t ring = std::max<int64_t>(2, (int64_t)((4ll << 30) / (per * 8)));
    ring = std::min<int64_t>(std::min<int64_t>(ring, nq), 4096);
    BatchHolder h;
    NN_TRY(h.acquire(ctx, d, net, beta, nq, ring, dense));
    nnsdp_query_inputs sub = shift_inputs(*in, q0);
    NN_TRY(nnsdp_batch_set_inputs(h.b, nq, &sub));
    return nnsdp_batch_run(h.b, out + q0 * per);
  });
}

}  // namespace

extern "C" {

int32_t nnsdp_bounds_ibp(nnsdp_ctx* ctx, const nnsdp_net* net, int64_t Q, const double* x1min,
                         const double* x1max, double* xmin, double* xmax, double* acxmin,
                         double* acxmax) {
  NN_CHECK(ctx && net && x1min && x1max, NNSDP_ERR_ARG, "NULL argument");
  NN_CHECK(Q >= 1, NNSDP_ERR_ARG, "Q must be >= 1");
  const Shape& sh = net->sh;
  return shard_queries(ctx, Q, [&](int d, int64_t q0, int64_t nq) -> int32_t {
    BatchHolder h;
    NN_TRY(h.acquire(ctx, d, net, 0, nq, 0, 0));
    nnsdp_query_inputs in;
    memset(&in, 0, sizeof(in));
    in.x1min = x1min + q0 * sh.n_in();
    in.x1max = x1max + q0 * sh.n_in();
    in.x1min_stride = in.x1max_stride = sh.n_in();
    NN_TRY(nnsdp_batch_set_inputs(h.b, nq, &in));
    NN_TRY(nnsdp_batch_bounds(h.b));
    return nnsdp_batch_get_bounds(h.b, xmin ? xmin + q0 * sh.xtot : nullptr,
                                  xmax ? xmax + q0 * sh.xtot : nullptr,
                                  acxmin ? acxmin + q0 * sh.acdim : nullptr,
                                  acxmax ? acxmax + q0 * sh.acdim : nullptr, nullptr, nullptr);
  });
}

int32_t nnsdp_preact_from_x(nnsdp_ctx* ctx, const nnsdp_net* net, int64_t Q, const double* xmin,
                            const double* xmax, double* acxmin, double* acxmax) {
  NN_CHECK(ctx && net && xmin && xmax && acxmin && acxmax, NNSDP_ERR_ARG, "NULL argument");
  NN_CHECK(Q >= 1, NNSDP_ERR_ARG, "Q must be >= 1");
  const Shape& sh = net->sh;
  return shard_queries(ctx, Q, [&](int d, int64_t q0, int64_t nq) -> int32_t {
    BatchHolder h;
    NN_TRY(h.acquire(ctx, d, net, 0, nq, 0, 0));
    nnsdp_batch* b = h.b;
    NN_CUDA(cudaSetDevice(b->dev));
    const NetPerDev& nd = *b->nd;
    NN_CUDA(cudaMemcpyAsync(b->xmin.p, xmin + q0 * sh.xtot, (size_t)sh.xtot * nq * 8,
                            cudaMemcpyHostToDevice, b->st));
    NN_CUDA(cudaMemcpyAsync(b->xmax.p, xmax + q0 * sh.xtot, (size_t)sh.xtot * nq * 8,
                            cudaMemcpyHostToDevice, b->st));
    for (int k = 0; k <= sh.K - 2; ++k)
      ibp_layer_launch(nd.M[k].as<double>(), (int)sh.n[k + 1], (int)sh.n[k],
                       b->xmin.as<double>() + sh.xoff[k], b->xmax.as<double>() + sh.xoff[k], sh.xtot,
                       nullptr, nullptr, b->acxmin.as<double>() + sh.noff(k + 1),
                       b->acxmax.as<double>() + sh.noff(k + 1), sh.acdim, (int)nq, 0, 0,
                       b->flags.as<int>() + 1, b->st);
    NN_CUDA(cudaGetLastError());
    NN_CUDA(cudaMemcpyAsync(acxmin + q0 * sh.acdim, b->acxmin.p, (size_t)sh.acdim * nq * 8,
                            cudaMemcpyDeviceToHost, b->st));
    NN_CUDA(cudaMemcpyAsync(acxmax + q0 * sh.acdim, b->acxmax.p, (size_t)sh.acdim * nq * 8,
                            cudaMemcpyDeviceToHost, b->st));
    return check_flags(b, "nnsdp_preact_from_x");
  });
}

int32_t nnsdp_sector_minmax(nnsdp_ctx* ctx, int64_t n, const double* acxmin, const double* acxmax,
                            double* smin, double* smax) {
  NN_CHECK(ctx && acxmin && acxmax && smin && smax, NNSDP_ERR_ARG, "NULL argument");
  NN_CHECK(n >= 0, NNSDP_ERR_ARG, "n must be >= 0");
  if (n == 0) return NNSDP_OK;
  NN_CUDA(cudaSetDevice(ctx->devs[0]));
  cudaStream_t st = ctx->streams[0];
  DevBuf lo, hi, a, b;
  struct Rel {
    DevBuf *w, *x, *y, *z;
    ~Rel() { w->release(); x->release(); y->release(); z->release(); }
  } rel{&lo, &hi, &a, &b};
  NN_TRY(upload(lo, acxmin, (size_t)n * 8, st));
  NN_TRY(upload(hi, acxmax, (size_t)n * 8, st));
  NN_TRY(a.ensure((size_t)n * 8));
  NN_TRY(b.ensure((size_t)n * 8));
  launch_sector_minmax(n, lo.as<double>(), hi.as<double>(), a.as<double>(), b.as<double>(), st);
  NN_CUDA(cudaGetLastError());
  NN_CUDA(cudaMemcpyAsync(smin, a.p, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
  NN_CUDA(cudaMemcpyAsync(smax, b.p, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
  NN_CUDA(cudaStreamSynchronize(st));
  return NNSDP_OK;
}

int32_t nnsdp_assemble_blocks(nnsdp_ctx* ctx, const nnsdp_net* net, int64_t beta, int64_t Q,
                              const nnsdp_query_inputs* in, double* blocks_out) {
  return assemble_impl(ctx, net, beta, Q, in, blocks_out, 0);
}

int32_t nnsdp_assemble_dense(nnsdp_ctx* ctx, const nnsdp_net* net, int64_t beta, int64_t Q,
                             const nnsdp_query_inputs* in, double* Z_out) {
  return assemble_impl(ctx, net, beta, Q, in, Z_out, 1);
}

int32_t nnsdp_assemble_packed(nnsdp_ctx* ctx, const nnsdp_net* net, int64_t beta, int64_t Q,
                              const nnsdp_query_inputs* in, double* records_out, uint8_t* present_out) {
  NN_CHECK(ctx && net && in && records_out, NNSDP_ERR_ARG, "NULL argument");
  NN_CHECK(Q >= 1, NNSDP_ERR_ARG, "Q must be >= 1");
  return shard_queries(ctx, Q, [&](int d, int64_t q0, int64_t nq) -> int32_t {
    // the record size is known once a batch (and with it the plan) exists: probe with the smallest ring first
    BatchHolder h;
    NN_TRY(h.acquire(ctx, d, net, beta, nq, std::min<int64_t>(nq, 2), NNSDP_FORMAT_PACKED));
    const int64_t per = h.b->lay.record_doubles;
    const int64_t want = std::min<int64_t>(std::min<int64_t>(std::max<int64_t>(2, (int64_t)((4ll << 30) / (per * 8))), nq), 4096);
    if (h.b->ring < want) {  // worth a larger ring: re-acquire (the small batch goes back to the cache)
      BatchHolder big;
      NN_TRY(big.acquire(ctx, d, net, beta, nq, want, NNSDP_FORMAT_PACKED));
      nnsdp_query_inputs sub = shift_inputs(*in, q0);
      NN_TRY(nnsdp_batch_set_inputs(big.b, nq, &sub));
      return run_impl(big.b, records_out + q0 * per, present_out ? present_out + q0 * big.b->lay.cells.size() : nullptr, 0);
    }
    nnsdp_query_inputs sub = shift_inputs(*in, q0);
    NN_TRY(nnsdp_batch_set_inputs(h.b, nq, &sub));
    return run_impl(h.b, records_out + q0 * per, present_out ? present_out + q0 * h.b->lay.cells.size() : nullptr, 0);
  });
}

/* Layout of a packed record (host only). */
int32_t nnsdp_packed_layout(int64_t K, const int64_t* xdims, int64_t beta, int64_t max_cells, nnsdp_packed_cell* cells,
                            int64_t* ncells, int64_t* record_doubles, int64_t* always_doubles) {
  NN_CHECK(ncells != nullptr, NNSDP_ERR_ARG, "NULL argument");
  Shape sh;
  NN_TRY(shape_from_xdims(K, xdims, &sh));
  nnsdp_sizes sz;
  NN_TRY(fill_sizes(sh, beta, &sz));
  std::vector<CliqueRanges> mats;
  NN_TRY(format_mats(sh, beta, NNSDP_FORMAT_PACKED, &mats));
  PlanHost plan;
  PackedLayout lay;
  NN_TRY(build_plan(sh, beta, mats, true, &plan, &lay));
  *ncells = (int64_t)lay.cells.size();
  if (record_doubles) *record_doubles = lay.record_doubles;
  if (always_doubles) *always_doubles = lay.always_doubles;
  if (cells) {
    NN_CHECK(max_cells >= *ncells, NNSDP_ERR_ARG, "cells too small");
    for (size_t i = 0; i < lay.cells.size(); ++i) {
      const PackedCell& c = lay.cells[i];
      nnsdp_packed_cell& o = cells[i];
      o.kind = c.kind;
      o.blk = c.blk < 0 ? 0 : c.blk + 1;  // 1-based block (x_blk), 0 = none
      o.row0 = c.grow0 + 1;               // 1-based on the wire
      o.col0 = c.gcol0 + 1;
      o.nrows = c.nrows;
      o.ncols = c.ncols;
      o.offset = c.offset;
      o.always = c.always;
      o.reserved = 0;
    }
  }
  return NNSDP_OK;
}

/* One packed record -> the dense matrices of NNSDP_FORMAT_BLOCKS (all clique blocks back to back) or
 * NNSDP_FORMAT_DENSE_Z, both triangles filled (host only). */
int32_t nnsdp_packed_unpack(int64_t K, const int64_t* xdims, int64_t beta, const double* record, const uint8_t* present,
                            int32_t format, double* out) {
  NN_CHECK(record && present && out, NNSDP_ERR_ARG, "NULL argument");
  NN_CHECK(format == NNSDP_FORMAT_BLOCKS || format == NNSDP_FORMAT_DENSE_Z, NNSDP_ERR_ARG, "format must be _BLOCKS or _DENSE_Z");
  NN_CHECK(K >= 1 && xdims != nullptr, NNSDP_ERR_ARG, "bad xdims");
  // the cell table of the last (xdims, beta, format) is kept: building it costs 37 ms at the stress size, a third of
  // the expansion itself, and records are unpacked one after the other for the same network
  struct Cached {
    std::vector<int64_t> key;
    Shape sh;
    PackedLayout lay;
    std::vector<CliqueRanges> mats;
  };
  static std::mutex mu;
  static std::shared_ptr<const Cached> last;
  std::vector<int64_t> key(xdims, xdims + K + 1);
  key.push_back(beta);
  key.push_back(format);
  std::shared_ptr<const Cached> c;
  {
    std::lock_guard<std::mutex> lk(mu);
    if (last && last->key == key) c = last;
  }
  if (!c) {
    auto fresh = std::make_shared<Cached>();
    fresh->key = key;
    NN_TRY(shape_from_xdims(K, xdims, &fresh->sh));
    nnsdp_sizes sz;
    NN_TRY(fill_sizes(fresh->sh, beta, &sz));
    std::vector<CliqueRanges> whole;
    NN_TRY(format_mats(fresh->sh, beta, NNSDP_FORMAT_PACKED, &whole));
    NN_TRY(format_mats(fresh->sh, beta, format, &fresh->mats));
    PlanHost plan;
    NN_TRY(build_plan(fresh->sh, beta, whole, true, &plan, &fresh->lay));
    c = fresh;
    std::lock_guard<std::mutex> lk(mu);
    last = c;
  }
  unpack_record(c->sh, beta, c->lay, c->mats, record, present, out);
  return NNSDP_OK;
}

}  // extern "C"

// -----------------------------------------------------------------------------------------
// CROWN bounds (SURVEY.md section 8f-2), see kernels_crown.cu
// -----------------------------------------------------------------------------------------
namespace {

// x_intvs of intervalsAutoLirpaSliced (post-activation bounds through the relaxation of relu_k, min/max
// post-processed) into b->xmin / b->xmax, then acx_intvs by one IBP step and the sector slopes.
int32_t crown_bounds_device(nnsdp_batch* b) {
  NN_CUDA(cudaSetDevice(b->dev));
  const Shape& sh = b->net->sh;
  const NetPerDev& npd = *b->nd;
  const int K = sh.K, n0 = (int)sh.n_in();
  const int64_t P = sh.xtot - n0;  // stacked pre-activations y_0 .. y_{K-1}
  int64_t maxn = 0;
  for (int k = 0; k <= K; ++k) maxn = std::max(maxn, sh.n[k]);
  const int64_t ld = (maxn + 1) & ~(int64_t)1;   // even: 16 B copies in the tensor-core GEMM
  // narrow nets (every step is the fused kernel): the post-activation targets walk back together, stacked
  static const bool no_wave = [] { const char* e = getenv("NNSDP_CROWN_NO_WAVEFRONT"); return e && e[0] == '1'; }();
  int64_t max_hidden_in = 0;
  for (int k = 0; k <= K - 2; ++k) max_hidden_in = std::max(max_hidden_in, sh.n[k]);
  const bool wavefront = !no_wave && K >= 16 && max_hidden_in <= 64;  // shallow nets: too few steps to save
  const int64_t rows_cap = wavefront ? std::max<int64_t>(maxn, sh.acdim) : maxn;  // row slots per (half, query)
  // queries per chunk: two row buffers of 2 * Qc * rows_cap * ld doubles, kept under ~1.5 GiB together
  int Qc = (int)std::max<int64_t>(1, std::min<int64_t>(b->Q, (int64_t(3) << 26) / std::max<int64_t>(1, 4 * rows_cap * ld)));
  Qc = std::min(Qc, 256);
  // work buffers live in the batch and are kept between calls (cudaMalloc + cudaFree of the ~0.5 GB row buffers of a
  // wide net cost 50 .. 570 ms per call depending on the box, more than the 440 ms of kernels for 16 queries at width
  // 1000); the chunk size above bounds them at ~1.5 GiB.  NNSDP_CROWN_KEEP_MB lowers the limit above which they are
  // given back on return.
  DevBuf &rowsA = b->cr_rowsA, &rowsB = b->cr_rowsB, &bias = b->cr_bias, &prel = b->cr_prel, &preu = b->cr_preu,
         &du = b->cr_du, &bu = b->cr_bu, &dl = b->cr_dl;
  static const size_t keep_cap = [] {
    const char* e = getenv("NNSDP_CROWN_KEEP_MB");
    return (size_t)(e ? std::max(0, atoi(e)) : 2048) << 20;
  }();
  const size_t work_bytes = ((size_t)4 * Qc * rows_cap * ld + (size_t)2 * Qc * rows_cap + (size_t)5 * Qc * P) * 8;
  struct Rel {
    std::vector<DevBuf*> v;
    bool keep;
    ~Rel() { if (!keep) for (DevBuf* x : v) x->release(); }
  } rel{{&rowsA, &rowsB, &bias, &prel, &preu, &du, &bu, &dl}, work_bytes <= keep_cap};
  NN_TRY(rowsA.ensure((size_t)2 * Qc * rows_cap * ld * 8));
  NN_TRY(rowsB.ensure((size_t)2 * Qc * rows_cap * ld * 8));
  NN_TRY(bias.ensure((size_t)2 * Qc * rows_cap * 8));
  for (DevBuf* x : {&prel, &preu, &du, &bu, &dl}) NN_TRY(x->ensure((size_t)Qc * P * 8));
  cudaStream_t st = b->st;
  double* xmin = b->xmin.as<double>();
  double* xmax = b->xmax.as<double>();
  auto poff = [&](int k) { return sh.xoff[k + 1] - n0; };  // offset of y_k inside the stacked pre-activations
  auto bias_of = [&](int k) { return npd.M[k].as<double>() + (size_t)sh.n[k] * sh.n[k + 1]; };
  b->span_begin(ST_BOUNDS, st);
  int launches = 0;
  launches += launch_place_x1(b->bd.x1min, b->bd.s_x1min, b->bd.x1max, b->bd.s_x1max, xmin, xmax, sh.xtot, n0,
                              (int)b->Q, st);
  for (int64_t q0 = 0; q0 < b->Q; q0 += Qc) {
    const int nq = (int)std::min<int64_t>(Qc, b->Q - q0);
    // pushes the current rows (in `cur`, nrows x n[k+1], functions of x_{k+1}) back through relu_k, W_k, ...,
    // relu_0, W_0 and concretises on the input box
    auto chain = [&](const double* srcL, const double* srcU, long long src_row_stride, long long src_q_stride,
                     int k_first, int nrows, double* out_lo, double* out_hi, long long out_stride, int post) {
      // Per step either one fused launch (relaxation + biases + product; fewer launches) or a row kernel followed
      // by a plain GEMM (less work per GEMM tile: the relaxation parameters are read once per row, not once per
      // row and GEMM row-tile).  The output alternates between the two row buffers; the source of the first step
      // is either the shared W rows or rowsB, so the first output goes to rowsA.
      static const int fused_env = [] { const char* e = getenv("NNSDP_CROWN_FUSED"); return e ? atoi(e) : -1; }();
      double* nxt = rowsA.as<double>();
      double* other = rowsB.as<double>();
      for (int k = k_first; k >= 0; --k) {
        const int n = (int)sh.n[k + 1];
        const bool fused = fused_env >= 0 ? fused_env != 0 : (sh.n[k] <= 64);  // one GEMM row-tile: nothing is re-read
        if (fused) {
          launches += launch_crown_step(npd.Wt[k].as<double>(), b->net->ldT[k], (int)sh.n[k], n, srcL, srcU,
                                        src_row_stride, src_q_stride, nxt, ld, nrows, nrows, nq, du.as<double>() + poff(k),
                                        bu.as<double>() + poff(k), dl.as<double>() + poff(k), P, bias_of(k),
                                        bias.as<double>(), st);
        } else {
          // the row kernel may work in place when its source is one of the two row buffers
          double* scaled = (srcL == other) ? other : nxt;
          double* prod = (scaled == nxt) ? other : nxt;
          launches += launch_crown_row(srcL, srcU, src_row_stride, src_q_stride, scaled, ld, nrows, nq, n,
                                       du.as<double>() + poff(k), bu.as<double>() + poff(k), dl.as<double>() + poff(k),
                                       P, bias_of(k), bias.as<double>(), st);
          launches += gemm_set_launch(npd.Wt[k].as<double>(), b->net->ldT[k], (int)sh.n[k], n, scaled, ld, prod, ld,
                                      2 * nq * nrows, st);
          if (prod != nxt) std::swap(nxt, other);
        }
        srcL = nxt;
        srcU = nxt + (size_t)nq * nrows * ld;
        src_row_stride = ld;
        src_q_stride = (long long)nrows * ld;
        std::swap(nxt, other);
      }
      launches += launch_crown_concretize(srcL, srcU, src_row_stride, src_q_stride, nrows, nrows, 0, nq, n0, b->bd.x1min,
                                          b->bd.s_x1min, b->bd.x1max, b->bd.s_x1max, (int)q0, bias.as<double>(),
                                          out_lo, out_hi, out_stride, post, st);
    };
    // y_0 by interval arithmetic (exact for the first layer; auto_LiRPA bound_general.py:1257-1262)
    launches += ibp_layer_launch(npd.M[0].as<double>(), (int)sh.n[1], n0, xmin + q0 * sh.xtot, xmax + q0 * sh.xtot,
                                 sh.xtot, nullptr, nullptr, prel.as<double>(), preu.as<double>(), P, nq, 0, 0, nullptr,
                                 st);
    launches += launch_crown_params(prel.as<double>(), preu.as<double>(), P, (int)sh.n[1], nq, du.as<double>(),
                                    bu.as<double>(), dl.as<double>(), st);
    // y_t, t = 1 .. K-1: backward from A = W_t
    for (int t = 1; t <= K - 1; ++t) {
      const int nrows = (int)sh.n[t + 1];
      // narrow nets: the whole chain of this target in one launch
      const int fusedc = launch_crown_chain(npd.nd, t, 0, 1, (int)maxn, nq, du.as<double>(), bu.as<double>(), dl.as<double>(), P,
                                            b->bd.x1min, b->bd.s_x1min, b->bd.x1max, b->bd.s_x1max, (int)q0,
                                            prel.as<double>() + poff(t), preu.as<double>() + poff(t), P, st);
      launches += fusedc;
      if (!fusedc) {
        launches += launch_crown_init_bias(bias_of(t), nrows, nq, bias.as<double>(), st);
        const double* wrows = npd.Wt[t].as<double>();  // row r of W_t = column r of Wt_t
        chain(wrows, wrows, b->net->ldT[t], 0, t - 1, nrows, prel.as<double>() + poff(t), preu.as<double>() + poff(t),
              P, 0);
      }
      if (t <= K - 2)
        launches += launch_crown_params(prel.as<double>() + poff(t), preu.as<double>() + poff(t), P, nrows, nq,
                                        du.as<double>() + poff(t), bu.as<double>() + poff(t),
                                        dl.as<double>() + poff(t), st);
    }
    // x_{k+1} = relu(y_k), k = 0 .. K-2: the output of the (k+1)-layer prefix followed by an identity layer.  Its
    // chains are row scalings of the chains of y_k that are already finished (see crown_post_kernel): one launch.
    // NNSDP_CROWN_POST_CHAINS=1 walks the K-1 chains instead (the first implementation, kept for A/B runs).
    static const bool post_chains = [] { const char* e = getenv("NNSDP_CROWN_POST_CHAINS"); return e && e[0] == '1'; }();
    if (!post_chains) {
      launches += launch_crown_post(prel.as<double>(), preu.as<double>(), du.as<double>(), bu.as<double>(), dl.as<double>(),
                                    P, (int)sh.acdim, nq, xmin + q0 * sh.xtot + n0, xmax + q0 * sh.xtot + n0, sh.xtot, st);
    }
    const int post_fused = !post_chains ? 1 : launch_crown_chain(npd.nd, 0, 1, K - 1, (int)maxn, nq, du.as<double>(), bu.as<double>(),
                                              dl.as<double>(), P, b->bd.x1min, b->bd.s_x1min, b->bd.x1max, b->bd.s_x1max,
                                              (int)q0, xmin + q0 * sh.xtot, xmax + q0 * sh.xtot, sh.xtot, st);
    if (post_chains) launches += post_fused;
    if (post_fused) {
      // done above, or (narrow nets, A/B path) every target was a CTA of one launch
    } else if (wavefront) {
      // Narrow nets: all K-1 targets walk back together.  Their rows are stacked (target K-2 first); the step
      // through (relu_j, W_j) handles the rows of every target k > j in one fused launch, after which target j
      // joins the stack: 2 (K-1) launches instead of (K-1)(K-2)/2 chain steps.
      const int Rs = (int)sh.acdim;
      std::vector<int> roff(K, 0);
      for (int k = K - 3; k >= 0; --k) roff[k] = roff[k + 1] + (int)sh.n[k + 2];
      double* cur = rowsA.as<double>();
      double* nxt = rowsB.as<double>();
      auto join = [&](int k) {  // rows of target k, functions of x_k, into `cur`
        launches += launch_crown_init_post(npd.Wt[k].as<double>(), b->net->ldT[k], (int)sh.n[k], bias_of(k),
                                           du.as<double>() + poff(k), bu.as<double>() + poff(k),
                                           dl.as<double>() + poff(k), P, cur, ld, (int)sh.n[k + 1], Rs, roff[k], nq,
                                           bias.as<double>(), st);
      };
      join(K - 2);
      for (int j = K - 3; j >= 0; --j) {
        launches += launch_crown_step(npd.Wt[j].as<double>(), b->net->ldT[j], (int)sh.n[j], (int)sh.n[j + 1], cur,
                                      cur + (size_t)nq * Rs * ld, ld, (long long)Rs * ld, nxt, ld, roff[j], Rs, nq,
                                      du.as<double>() + poff(j), bu.as<double>() + poff(j), dl.as<double>() + poff(j),
                                      P, bias_of(j), bias.as<double>(), st);
        std::swap(cur, nxt);
        join(j);
      }
      for (int k = 0; k <= K - 2; ++k)
        launches += launch_crown_concretize(cur + (size_t)roff[k] * ld, cur + ((size_t)nq * Rs + roff[k]) * ld, ld,
                                            (long long)Rs * ld, (int)sh.n[k + 1], Rs, roff[k], nq, n0, b->bd.x1min,
                                            b->bd.s_x1min, b->bd.x1max, b->bd.s_x1max, (int)q0, bias.as<double>(),
                                            xmin + q0 * sh.xtot + sh.xoff[k + 1], xmax + q0 * sh.xtot + sh.xoff[k + 1],
                                            sh.xtot, 1, st);
    } else {
      for (int k = 0; k <= K - 2; ++k) {
        const int nrows = (int)sh.n[k + 1];
        double* src = rowsB.as<double>();  // chain() writes its first step into rowsA
        launches += launch_crown_init_post(npd.Wt[k].as<double>(), b->net->ldT[k], (int)sh.n[k], bias_of(k),
                                           du.as<double>() + poff(k), bu.as<double>() + poff(k),
                                           dl.as<double>() + poff(k), P, src, ld, nrows, nrows, 0, nq,
                                           bias.as<double>(), st);
        // rows are now functions of x_k: continue with relu_{k-1}, W_{k-1}, ... (k = 0: concretise at once)
        chain(src, src + (size_t)nq * nrows * ld, ld, (long long)nrows * ld, k - 1, nrows,
              xmin + q0 * sh.xtot + sh.xoff[k + 1], xmax + q0 * sh.xtot + sh.xoff[k + 1], sh.xtot, 1);
      }
    }
    // x_K = y_{K-1} with the same post-processing: copy through a concretisation-free path
    {
      const int nrows = (int)sh.n[K];
      // rows = identity is not needed: min/max of the already computed bounds
      launches += launch_crown_init_bias(nullptr, nrows, nq, bias.as<double>(), st);
      // reuse the concretize kernel with zero-length rows: L = lbias, U = ubias -- so load the bounds as biases
      cudaMemcpy2DAsync(bias.as<double>(), (size_t)nrows * 8, prel.as<double>() + poff(K - 1), (size_t)P * 8,
                        (size_t)nrows * 8, nq, cudaMemcpyDeviceToDevice, st);
      cudaMemcpy2DAsync(bias.as<double>() + (size_t)nq * nrows, (size_t)nrows * 8, preu.as<double>() + poff(K - 1),
                        (size_t)P * 8, (size_t)nrows * 8, nq, cudaMemcpyDeviceToDevice, st);
      launches += launch_crown_concretize(rowsA.as<double>(), rowsA.as<double>(), ld, 0, nrows, nrows, 0, nq, 0, b->bd.x1min,
                                          b->bd.s_x1min, b->bd.x1max, b->bd.s_x1max, (int)q0, bias.as<double>(),
                                          xmin + q0 * sh.xtot + sh.xoff[K], xmax + q0 * sh.xtot + sh.xoff[K], sh.xtot,
                                          1, st);
    }
  }
  // acx_intvs: one IBP step from x_intvs (intervals_auto_lirpa.jl:55-62), then makeSectorMinMax
  for (int k = 0; k <= K - 2; ++k)
    launches += ibp_layer_launch(npd.M[k].as<double>(), (int)sh.n[k + 1], (int)sh.n[k], xmin + sh.xoff[k],
                                 xmax + sh.xoff[k], sh.xtot, nullptr, nullptr, b->acxmin.as<double>() + sh.noff(k + 1),
                                 b->acxmax.as<double>() + sh.noff(k + 1), sh.acdim, (int)b->Q, 0, 0,
                                 b->flags.as<int>() + 1, st);
  launches += launch_sector_minmax(sh.acdim * (long long)b->Q, b->acxmin.as<double>(), b->acxmax.as<double>(),
                                   b->smin_c.as<double>(), b->smax_c.as<double>(), st);
  b->span_end(st, launches);
  NN_CUDA(cudaGetLastError());
  NN_CUDA(cudaStreamSynchronize(st));  // the temporary buffers are released on return
  b->bounds_done = true;
  return NNSDP_OK;
}

}  // namespace

extern "C" int32_t nnsdp_batch_bounds_crown(nnsdp_batch* b) {
  NN_CHECK(b != nullptr, NNSDP_ERR_ARG, "batch is NULL");
  NN_CHECK(b->have_inputs, NNSDP_ERR_STATE, "nnsdp_batch_bounds_crown before nnsdp_batch_set_inputs");
  NN_TRY(crown_bounds_device(b));
  return check_flags(b, "nnsdp_batch_bounds_crown");
}

// -----------------------------------------------------------------------------------------
// lambda_max of Z(gamma), matrix-free (SURVEY.md section 8f-3)
// -----------------------------------------------------------------------------------------
namespace {

// extreme eigenvalue of the symmetric tridiagonal (alpha[0..m), beta[0..m-1)) by Sturm bisection:
// the largest (which = +1) or the smallest (which = -1)
double tridiag_extreme(const double* alpha, const double* beta, int m, int which) {
  if (m <= 0) return 0.0;
  double lo = alpha[0], hi = alpha[0];
  for (int i = 0; i < m; ++i) {
    const double r = (i > 0 ? fabs(beta[i - 1]) : 0.0) + (i + 1 < m ? fabs(beta[i]) : 0.0);
    lo = std::min(lo, alpha[i] - r);
    hi = std::max(hi, alpha[i] + r);
  }
  auto count_below = [&](double x) {  // number of eigenvalues < x
    int cnt = 0;
    double d = 1.0;
    for (int i = 0; i < m; ++i) {
      const double b2 = i > 0 ? beta[i - 1] * beta[i - 1] : 0.0;
      d = (alpha[i] - x) - (i > 0 ? b2 / d : 0.0);
      if (d == 0.0) d = -1e-300;
      if (d < 0.0) ++cnt;
    }
    return cnt;
  };
  const int target = which > 0 ? m : 1;  // smallest x with count_below(x) >= target brackets the wanted eigenvalue
  for (int it = 0; it < 200 && hi - lo > 4e-16 * std::max(fabs(lo), fabs(hi)); ++it) {
    const double mid = 0.5 * (lo + hi);
    if (count_below(mid) >= target) hi = mid; else lo = mid;
  }
  return 0.5 * (lo + hi);
}

double tridiag_lambda_max(const double* alpha, const double* beta, int m) { return tridiag_extreme(alpha, beta, m, +1); }

// |last component| of the unit eigenvector of the tridiagonal for its eigenvalue theta: two steps of inverse
// iteration with (T - theta' I), theta' nudged off the eigenvalue, solved by Gaussian elimination with partial
// pivoting.  beta_m * |s_last| is the residual norm ||Z v - theta v|| of the Ritz pair.
double tridiag_last_component(const double* alpha, const double* beta, int m, double theta, double scale) {
  if (m <= 1) return 1.0;
  const double shift = theta + 1e-13 * std::max(scale, 1e-300);
  std::vector<double> x(m, 1.0), dl(m), d(m), du(m), du2(m);
  for (int rep = 0; rep < 2; ++rep) {
    for (int i = 0; i < m; ++i) {
      d[i] = alpha[i] - shift;
      dl[i] = i > 0 ? beta[i - 1] : 0.0;   // sub-diagonal entry in row i
      du[i] = i + 1 < m ? beta[i] : 0.0;   // super-diagonal entry in row i
      du2[i] = 0.0;
    }
    for (int i = 0; i + 1 < m; ++i) {      // eliminate row i+1's sub-diagonal
      if (fabs(d[i]) >= fabs(dl[i + 1])) {
        const double piv = d[i] != 0.0 ? d[i] : 1e-300;
        const double f = dl[i + 1] / piv;
        d[i + 1] -= f * du[i];
        x[i + 1] -= f * x[i];
        d[i] = piv;
      } else {                              // swap rows i and i+1
        const double f = d[i] / dl[i + 1];
        const double nd = dl[i + 1], ndu = d[i + 1], ndu2 = du[i + 1];
        d[i + 1] = du[i] - f * ndu;
        du[i + 1] = -f * ndu2;
        d[i] = nd;
        du[i] = ndu;
        du2[i] = ndu2;
        const double t = x[i];
        x[i] = x[i + 1];
        x[i + 1] = t - f * x[i + 1];
      }
    }
    if (d[m - 1] == 0.0) d[m - 1] = 1e-300;
    x[m - 1] /= d[m - 1];
    if (m >= 2) x[m - 2] = (x[m - 2] - du[m - 2] * x[m - 1]) / d[m - 2];
    for (int i = m - 3; i >= 0; --i) x[i] = (x[i] - du[i] * x[i + 1] - du2[i] * x[i + 2]) / d[i];
    double nrm = 0.0, mx = 0.0;
    for (double v : x) mx = std::max(mx, fabs(v));
    if (!(mx > 0.0) || !std::isfinite(mx)) return 1.0;
    for (double& v : x) { v /= mx; nrm += v * v; }
    nrm = sqrt(nrm);
    for (double& v : x) v /= nrm;
  }
  return fabs(x[m - 1]);
}

}  // namespace

extern "C" int32_t nnsdp_batch_lambda_max_ex(nnsdp_batch* b, int32_t max_iters, double tol, double* lam_max,
                                             int32_t* iters_out, double* resid_out, int32_t* converged_out) {
  NN_CHECK(b && lam_max, NNSDP_ERR_ARG, "NULL argument");
  NN_CHECK(b->prepared, NNSDP_ERR_STATE, "nnsdp_batch_lambda_max before nnsdp_batch_prepare");
  NN_CHECK(max_iters >= 1, NNSDP_ERR_ARG, "max_iters must be >= 1");
  NN_CUDA(cudaSetDevice(b->dev));
  const Shape& sh = b->net->sh;
  const NetPerDev& npd = *b->nd;
  const NetDev& nd = npd.nd;
  const int n = (int)sh.Zdim, ac = (int)sh.acdim, K = sh.K;
  const int m = (int)std::min<int64_t>(max_iters, sh.Zdim);
  // queries per chunk: the Krylov basis is (m + 1) x Qc x Zdim doubles; keep it under ~2 GiB
  int Qc = (int)std::max<int64_t>(1, std::min<int64_t>(b->Q, (int64_t(1) << 28) / ((int64_t)(m + 1) * n)));
  Qc = std::min(Qc, 64);
  DevBuf dV, dw, dt, ds1, dc, dnrm, dalpha, dbeta;
  struct Rel {
    std::vector<DevBuf*> v;
    ~Rel() { for (DevBuf* x : v) x->release(); }
  } rel{{&dV, &dw, &dt, &ds1, &dc, &dnrm, &dalpha, &dbeta}};
  NN_TRY(dV.ensure((size_t)(m + 1) * Qc * n * 8));
  NN_TRY(dw.ensure((size_t)Qc * n * 8));
  NN_TRY(dt.ensure((size_t)Qc * ac * 8));
  NN_TRY(ds1.ensure((size_t)Qc * ac * 8));
  NN_TRY(dc.ensure((size_t)Qc * (m + 1) * 8));
  NN_TRY(dnrm.ensure((size_t)Qc * 8));
  cudaStream_t st = b->st;
  std::vector<double> hc((size_t)Qc * (m + 1)), hn((size_t)Qc);
  bool all_converged = true;
  for (int64_t q0 = 0; q0 < b->Q; q0 += Qc) {
    const int nq = (int)std::min<int64_t>(Qc, b->Q - q0);
    double* V = dV.as<double>();
    double* w = dw.as<double>();
    auto Vj = [&](int j) { return V + (size_t)j * Qc * n; };
    launch_eig_init(w, n, nq, (int)q0, st);
    launch_eig_normalize(w, Vj(0), n, nq, dnrm.as<double>(), st);
    std::vector<std::vector<double>> alpha(nq), beta(nq);
    std::vector<double> theta(nq, 0.0), resid(nq, 0.0);
    std::vector<int> done(nq, 0), its(nq, 0), conv(nq, 0);
    int j = 0;
    for (; j < m; ++j) {
      // ---- w = Z v_j ----
      const double* x = Vj(j);
      NN_CUDA(cudaMemsetAsync(dt.p, 0, (size_t)nq * ac * 8, st));
      for (int k = 0; k <= K - 2; ++k)  // t_{k+1} = W_k x_k
        gemm_acc_launch(npd.M[k].as<double>(), (int)sh.n[k + 1], (int)sh.n[k + 1], (int)sh.n[k], x + sh.off[k], n,
                        dt.as<double>() + sh.noff(k + 1), ac, nq, st);
      launch_eig_mid(nd, b->bd, (int)q0, nq, x, dt.as<double>(), ds1.as<double>(), w, st);
      launch_eig_io(nd, b->bd, (int)q0, nq, x, w, st);
      for (int k = 0; k <= K - 2; ++k)  // y_k += W_k' s1_{k+1}
        gemm_acc_launch(npd.Wt[k].as<double>(), b->net->ldT[k], (int)sh.n[k], (int)sh.n[k + 1],
                        ds1.as<double>() + sh.noff(k + 1), ac, w + sh.off[k], n, nq, st);
      // ---- alpha_j and full re-orthogonalisation against v_0..v_j (classical Gram-Schmidt, twice) ----
      launch_eig_multidot(V, w, n, Qc, j + 1, dc.as<double>(), m + 1, st);
      launch_eig_project(V, w, n, Qc, j + 1, dc.as<double>(), m + 1, st);
      NN_CUDA(cudaMemcpyAsync(hc.data(), dc.p, (size_t)nq * (m + 1) * 8, cudaMemcpyDeviceToHost, st));
      NN_CUDA(cudaStreamSynchronize(st));
      for (int q = 0; q < nq; ++q) alpha[q].push_back(hc[(size_t)q * (m + 1) + j]);
      launch_eig_multidot(V, w, n, Qc, j + 1, dc.as<double>(), m + 1, st);
      launch_eig_project(V, w, n, Qc, j + 1, dc.as<double>(), m + 1, st);
      NN_CUDA(cudaMemcpyAsync(hc.data(), dc.p, (size_t)nq * (m + 1) * 8, cudaMemcpyDeviceToHost, st));
      launch_eig_normalize(w, Vj(j + 1), n, nq, dnrm.as<double>(), st);
      NN_CUDA(cudaMemcpyAsync(hn.data(), dnrm.p, (size_t)nq * 8, cudaMemcpyDeviceToHost, st));
      NN_CUDA(cudaStreamSynchronize(st));
      bool all_done = true;
      for (int q = 0; q < nq; ++q) {
        alpha[q][j] += hc[(size_t)q * (m + 1) + j];  // second-pass correction of alpha_j
        if (done[q]) continue;
        its[q] = j + 1;
        theta[q] = tridiag_extreme(alpha[q].data(), beta[q].data(), j + 1, +1);
        // The tolerance is relative to the SPECTRAL SCALE (the largest |Ritz value|), not to |theta|: the acceptance
        // gate eigmax(Z) <= 1e-4 (experiments/acas.jl:76-79) asks about a lambda_max near zero, where a test relative
        // to theta itself can never trigger.  ||Z v - theta v|| = beta_j |s_last| for the Ritz pair (theta, v).
        const double tmin = tridiag_extreme(alpha[q].data(), beta[q].data(), j + 1, -1);
        const double scale = std::max(std::max(fabs(theta[q]), fabs(tmin)), 1e-300);
        resid[q] = hn[q] * tridiag_last_component(alpha[q].data(), beta[q].data(), j + 1, theta[q], scale);
        // stop on an invariant subspace (beta_j ~ 0: the Ritz values are eigenvalues) or on a small residual
        if (hn[q] <= 1e-13 * scale || resid[q] <= tol * scale || j + 1 == n) done[q] = conv[q] = 1;
        beta[q].push_back(hn[q]);
        if (!done[q]) all_done = false;
      }
      if (all_done) {
        ++j;
        break;
      }
    }
    for (int q = 0; q < nq; ++q) {
      lam_max[q0 + q] = theta[q];
      if (iters_out) iters_out[q0 + q] = its[q];
      if (resid_out) resid_out[q0 + q] = resid[q];
      if (converged_out) converged_out[q0 + q] = conv[q];
      all_converged &= conv[q] != 0;
    }
  }
  NN_CUDA(cudaGetLastError());
  if (!all_converged) {
    set_error("nnsdp_batch_lambda_max: some query did not reach the residual tolerance within max_iters = %d "
              "(its value is a LOWER bound of lambda_max; see the residual)", (int)max_iters);
    return NNSDP_ERR_NOCONV;
  }
  return NNSDP_OK;
}

extern "C" int32_t nnsdp_batch_lambda_max(nnsdp_batch* b, int32_t max_iters, double tol, double* lam_max,
                                          int32_t* iters_out) {
  return nnsdp_batch_lambda_max_ex(b, max_iters, tol, lam_max, iters_out, nullptr, nullptr);
}

// -----------------------------------------------------------------------------------------
// affine-coefficient mode (SURVEY.md section 8f-1): Z(gamma) = Z0 + sum_v gamma_v Z_v over the cover
// -----------------------------------------------------------------------------------------
struct nnsdp_affine {
  nnsdp_batch* batch = nullptr;  // Q = 1, all multipliers zero: bounds, slopes, constant part
  nnsdp_affine_sizes sz{};
  std::vector<int> lo;           // first cover row of every column (0-based)
  std::vector<long long> col_ptr;
  DevBuf d_lo, d_colptr, d_counts, d_offs, d_ent, d_var, d_val, d_z0;
};

extern "C" {

int32_t nnsdp_affine_destroy(nnsdp_affine* h) {
  if (!h) return NNSDP_OK;
  if (h->batch) cudaSetDevice(h->batch->dev);
  for (DevBuf* x : {&h->d_lo, &h->d_colptr, &h->d_counts, &h->d_offs, &h->d_ent, &h->d_var, &h->d_val, &h->d_z0})
    x->release();
  nnsdp_batch_destroy(h->batch);
  delete h;
  return NNSDP_OK;
}

int32_t nnsdp_affine_create(nnsdp_ctx* ctx, const nnsdp_net* net, int64_t beta,
                            const nnsdp_query_inputs* in, int64_t max_nnz, nnsdp_affine** out,
                            nnsdp_affine_sizes* sizes) {
  NN_CHECK(out != nullptr, NNSDP_ERR_ARG, "affine output pointer is NULL");
  *out = nullptr;
  NN_CHECK(ctx && net && in && sizes, NNSDP_ERR_ARG, "NULL argument");
  const Shape& sh = net->sh;
  nnsdp_affine* h = new nnsdp_affine();
  struct Guard {
    nnsdp_affine* h;
    ~Guard() { if (h) nnsdp_affine_destroy(h); }
  } guard{h};
  NN_TRY(nnsdp_batch_create(ctx, 0, net, beta, 1, 1, 0, &h->batch));
  nnsdp_batch* b = h->batch;
  // one query with every multiplier zero: the prepared vectors then hold the constant part of Z
  nnsdp_query_inputs q = *in;
  std::vector<double> zeros((size_t)std::max<int64_t>(b->sz.secdim, 1), 0.0);
  const double zero1 = 0.0;
  q.gamma_in = zeros.data();
  q.gamma_bnd = zeros.data();
  q.gamma_sec = zeros.data();
  q.gamma_in_stride = q.gamma_bnd_stride = q.gamma_sec_stride = 0;
  if (q.out_kind != NNSDP_OUT_SAFETY) {
    q.gamma_out = &zero1;
    q.gamma_out_stride = 0;
  }
  NN_TRY(nnsdp_batch_set_inputs(b, 1, &q));
  if (!b->bounds_supplied) NN_TRY(nnsdp_batch_bounds(b));
  NN_TRY(nnsdp_batch_prepare(b));
  NN_CUDA(cudaSetDevice(b->dev));
  // cover: column c holds rows [lo(c), c]; lo(c) = smallest index sharing a clique with c
  CliqueInfoHost ci;
  NN_TRY(make_cliques_host(sh, beta, &ci));
  h->lo.assign((size_t)sh.Zdim, 0);
  for (int64_t c = 0; c < sh.Zdim; ++c) {
    int64_t lo = c;
    for (const CliqueRanges& ck : ci.ck) {
      bool has = false;
      for (int s = 0; s < ck.nseg; ++s) has |= (c >= ck.lo[s] && c <= ck.hi[s]);
      if (has) lo = std::min(lo, ck.lo[0]);
    }
    h->lo[c] = (int)lo;
  }
  h->col_ptr.assign((size_t)sh.Zdim + 1, 0);
  for (int64_t c = 0; c < sh.Zdim; ++c) h->col_ptr[c + 1] = h->col_ptr[c] + (c - h->lo[c] + 1);
  nnsdp_affine_sizes& sz = h->sz;
  sz.var_in = 0;
  sz.var_out = sh.n_in();
  sz.var_bnd = sz.var_out + (in->out_kind == NNSDP_OUT_SAFETY ? 0 : 1);
  sz.var_sec = sz.var_bnd + sh.acdim;
  sz.nvar = sz.var_sec + b->sz.secdim;
  sz.nent = h->col_ptr[sh.Zdim];
  NN_TRY(upload(h->d_lo, h->lo.data(), h->lo.size() * 4, b->st));
  NN_TRY(upload(h->d_colptr, h->col_ptr.data(), h->col_ptr.size() * 8, b->st));
  AffineDev A{};
  A.nvar = sz.nvar;
  A.var_out = sz.var_out;
  A.var_bnd = sz.var_bnd;
  A.var_sec = sz.var_sec;
  A.acdim = sh.acdim;
  A.lamdim = b->sz.lamdim;
  A.beta = beta;
  A.out_kind = in->out_kind;
  A.x1min = b->bd.x1min;
  A.x1max = b->bd.x1max;
  A.ymin = b->bd.ymin;
  A.ymax = b->bd.ymax;
  A.smin = b->bd.smin;
  A.smax = b->bd.smax;
  A.col_ptr = h->d_colptr.as<long long>();
  A.lo = h->d_lo.as<int>();
  const NetDev& nd = b->nd->nd;
  NN_TRY(h->d_counts.ensure((size_t)sz.nvar * 8));
  launch_affine_count(nd, A, h->d_counts.as<long long>(), b->st);
  std::vector<long long> counts((size_t)sz.nvar), offs((size_t)sz.nvar + 1, 0);
  NN_CUDA(cudaMemcpyAsync(counts.data(), h->d_counts.p, counts.size() * 8, cudaMemcpyDeviceToHost, b->st));
  NN_CUDA(cudaStreamSynchronize(b->st));
  for (int64_t v = 0; v < sz.nvar; ++v) offs[v + 1] = offs[v] + counts[v];
  sz.nnz = offs[sz.nvar];
  *sizes = sz;
  NN_CHECK(max_nnz <= 0 || sz.nnz <= max_nnz, NNSDP_ERR_NOMEM,
           "affine form has %lld coefficients, more than max_nnz = %lld (the Gram term is n_k^2 per "
           "stably-active neuron: wide layers need the factored form)", (long long)sz.nnz, (long long)max_nnz);
  NN_TRY(upload(h->d_offs, offs.data(), offs.size() * 8, b->st));
  NN_TRY(h->d_ent.ensure((size_t)std::max<int64_t>(sz.nnz, 1) * 8));
  NN_TRY(h->d_var.ensure((size_t)std::max<int64_t>(sz.nnz, 1) * 8));
  NN_TRY(h->d_val.ensure((size_t)std::max<int64_t>(sz.nnz, 1) * 8));
  NN_TRY(h->d_z0.ensure((size_t)std::max<int64_t>(sz.nent, 1) * 8));
  launch_affine_fill(nd, A, h->d_offs.as<long long>(), h->d_ent.as<long long>(), h->d_var.as<long long>(),
                     h->d_val.as<double>(), b->st);
  launch_affine_z0(nd, b->bd, A, h->d_z0.as<double>(), b->st);
  NN_CUDA(cudaGetLastError());
  NN_CUDA(cudaStreamSynchronize(b->st));
  guard.h = nullptr;
  *out = h;
  return NNSDP_OK;
}

int32_t nnsdp_affine_get(nnsdp_affine* h, int64_t* ent_row, int64_t* ent_col, double* z0,
                         int64_t* coo_ent, int64_t* coo_var, double* coo_val) {
  NN_CHECK(h != nullptr, NNSDP_ERR_ARG, "affine handle is NULL");
  nnsdp_batch* b = h->batch;
  NN_CUDA(cudaSetDevice(b->dev));
  const int64_t Zdim = b->net->sh.Zdim, nnz = h->sz.nnz;
  if (ent_row || ent_col)
    for (int64_t c = 0; c < Zdim; ++c)
      for (int64_t r = h->lo[c]; r <= c; ++r) {
        const int64_t e = h->col_ptr[c] + (r - h->lo[c]);
        if (ent_row) ent_row[e] = r + 1;  // 1-based on the wire
        if (ent_col) ent_col[e] = c + 1;
      }
  if (z0) NN_CUDA(cudaMemcpyAsync(z0, h->d_z0.p, (size_t)h->sz.nent * 8, cudaMemcpyDeviceToHost, b->st));
  if (coo_ent && nnz) NN_CUDA(cudaMemcpyAsync(coo_ent, h->d_ent.p, (size_t)nnz * 8, cudaMemcpyDeviceToHost, b->st));
  if (coo_var && nnz) NN_CUDA(cudaMemcpyAsync(coo_var, h->d_var.p, (size_t)nnz * 8, cudaMemcpyDeviceToHost, b->st));
  if (coo_val && nnz) NN_CUDA(cudaMemcpyAsync(coo_val, h->d_val.p, (size_t)nnz * 8, cudaMemcpyDeviceToHost, b->st));
  NN_CUDA(cudaStreamSynchronize(b->st));
  if (coo_ent)
    for (int64_t i = 0; i < nnz; ++i) coo_ent[i] += 1;
  if (coo_var)
    for (int64_t i = 0; i < nnz; ++i) coo_var[i] += 1;
  return NNSDP_OK;
}

}  // extern "C"

extern "C" {

int32_t nnsdp_batch_set_bounds_method(nnsdp_batch* b, int32_t method) {
  NN_CHECK(b != nullptr, NNSDP_ERR_ARG, "batch is NULL");
  NN_CHECK(method == NNSDP_BOUNDS_IBP || method == NNSDP_BOUNDS_CROWN, NNSDP_ERR_ARG, "unrecognized method: %d", method);
  b->bounds_method = method;
  return NNSDP_OK;
}

int32_t nnsdp_bounds_crown(nnsdp_ctx* ctx, const nnsdp_net* net, int64_t Q, const double* x1min,
                           const double* x1max, double* xmin, double* xmax, double* acxmin, double* acxmax) {
  NN_CHECK(ctx && net && x1min && x1max, NNSDP_ERR_ARG, "NULL argument");
  NN_CHECK(Q >= 1, NNSDP_ERR_ARG, "Q must be >= 1");
  const Shape& sh = net->sh;
  return shard_queries(ctx, Q, [&](int d, int64_t q0, int64_t nq) -> int32_t {
    BatchHolder h;
    NN_TRY(h.acquire(ctx, d, net, 0, nq, 0, 0));
    nnsdp_query_inputs in;
    memset(&in, 0, sizeof(in));
    in.x1min = x1min + q0 * sh.n_in();
    in.x1max = x1max + q0 * sh.n_in();
    in.x1min_stride = in.x1max_stride = sh.n_in();
    NN_TRY(nnsdp_batch_set_inputs(h.b, nq, &in));
    NN_TRY(nnsdp_batch_bounds_crown(h.b));
    return nnsdp_batch_get_bounds(h.b, xmin ? xmin + q0 * sh.xtot : nullptr, xmax ? xmax + q0 * sh.xtot : nullptr,
                                  acxmin ? acxmin + q0 * sh.acdim : nullptr,
                                  acxmax ? acxmax + q0 * sh.acdim : nullptr, nullptr, nullptr);
  });
}

}  // extern "C"

