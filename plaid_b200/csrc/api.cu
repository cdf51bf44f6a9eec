// C ABI of libplaidgpu (include/plaidgpu.h): context, gene-set plan, the score pipeline
// (rank -> score product -> median normalisation -> epilogue) and the stand-alone entry points.
// Host-side orchestration only; the arithmetic is in score_kernels.cu / stats_kernels.cu /
// rank_kernels.cu.  There is no CPU fallback: every entry point fails with PLAIDGPU_ERR_CUDA
// when the GPU is unusable.
#include <math.h>
#include <stdio.h>
#include <string.h>
#include <stdlib.h>
#include <time.h>
#if defined(__x86_64__)
#include <immintrin.h>
#endif

#include <algorithm>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <new>
#include <thread>

#include "common.cuh"

using namespace plaidgpu;

namespace {

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t reserve(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    if (bytes == 0) return cudaSuccess;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e == cudaSuccess) cap = bytes;
    return e;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  template <typename T>
  T* as() const { return reinterpret_cast<T*>(p); }
};

// Large host copies into a destination that will not be read again soon (the caller's result matrix): streaming
// (non-temporal) stores skip the read-for-ownership of every destination line, which otherwise doubles the write
// traffic; glibc's memcpy only switches to them far above the 5 MB a copy thread handles at a time.
#if defined(__x86_64__)
__attribute__((target("avx2"))) static void copy_stream_avx2(char* d, const char* s, size_t n) {
  while (n && ((uintptr_t)d & 31)) {
    *d++ = *s++;
    --n;
  }
  size_t v = n / 128;
  for (; v; --v) {
    const __m256i a = _mm256_loadu_si256((const __m256i*)s), b = _mm256_loadu_si256((const __m256i*)(s + 32));
    const __m256i c2 = _mm256_loadu_si256((const __m256i*)(s + 64)), e = _mm256_loadu_si256((const __m256i*)(s + 96));
    _mm256_stream_si256((__m256i*)d, a);
    _mm256_stream_si256((__m256i*)(d + 32), b);
    _mm256_stream_si256((__m256i*)(d + 64), c2);
    _mm256_stream_si256((__m256i*)(d + 96), e);
    s += 128;
    d += 128;
  }
  _mm_sfence();
  n &= 127;
  if (n) memcpy(d, s, n);
}
static void copy_streaming(void* d, const void* s, size_t n) {
  static const bool avx2 = __builtin_cpu_supports("avx2") && !getenv("PLAIDGPU_NO_NT_COPY");
  if (avx2 && n >= 4096) copy_stream_avx2(static_cast<char*>(d), static_cast<const char*>(s), n);
  else memcpy(d, s, n);
}
#else
static void copy_streaming(void* d, const void* s, size_t n) { memcpy(d, s, n); }
#endif

// Blocking memcpy split over a few persistent host threads: moves finished column blocks from the pinned ring
// into a PAGEABLE caller buffer (what an R caller hands in: Rf_allocMatrix memory) at memory speed, while the
// next block is still crossing PCIe.
class CopyPool {
 public:
  explicit CopyPool(int n) {
    for (int i = 0; i < n; ++i) th_.emplace_back([this, i] { run(i); });
  }
  ~CopyPool() {
    {
      std::lock_guard<std::mutex> lk(m_);
      stop_ = true;
    }
    cv_work_.notify_all();
    for (auto& t : th_) t.join();
  }
  void copy(void* dst, const void* src, size_t bytes) {
    if (bytes < (size_t)(1 << 20) || th_.empty()) {
      memcpy(dst, src, bytes);
      return;
    }
    std::unique_lock<std::mutex> lk(m_);
    d_ = static_cast<char*>(dst);
    s_ = static_cast<const char*>(src);
    n_ = bytes;
    fn_ = nullptr;
    pending_ = (int)th_.size();
    ++gen_;
    cv_work_.notify_all();
    cv_done_.wait(lk, [this] { return pending_ == 0; });
  }
  // fn(part, parts) on every worker thread, blocking
  void run(const std::function<void(int, int)>& fn) {
    if (th_.empty()) {
      fn(0, 1);
      return;
    }
    std::unique_lock<std::mutex> lk(m_);
    fn_ = &fn;
    pending_ = (int)th_.size();
    ++gen_;
    cv_work_.notify_all();
    cv_done_.wait(lk, [this] { return pending_ == 0; });
    fn_ = nullptr;
  }
  int threads() const { return (int)th_.size(); }

 private:
  void run(int i) {
    int seen = 0;
    for (;;) {
      std::unique_lock<std::mutex> lk(m_);
      cv_work_.wait(lk, [&] { return stop_ || gen_ != seen; });
      if (stop_) return;
      seen = gen_;
      const size_t parts = th_.size();
      const size_t per = ((n_ / parts) + 4095) & ~(size_t)4095;
      const size_t lo = std::min(n_, per * (size_t)i), hi = std::min(n_, lo + per);
      char* d = d_;
      const char* s = s_;
      const std::function<void(int, int)>* fn = fn_;
      lk.unlock();
      if (fn) (*fn)(i, (int)parts);
      else if (hi > lo) copy_streaming(d + lo, s + lo, hi - lo);
      lk.lock();
      if (--pending_ == 0) cv_done_.notify_all();
    }
  }
  std::vector<std::thread> th_;
  std::mutex m_;
  std::condition_variable cv_work_, cv_done_;
  char* d_ = nullptr;
  const char* s_ = nullptr;
  size_t n_ = 0;
  const std::function<void(int, int)>* fn_ = nullptr;
  int gen_ = 0, pending_ = 0;
  bool stop_ = false;
};

bool is_pageable(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return true;
  }
  return a.type == cudaMemoryTypeUnregistered;
}

}  // namespace

struct plaidgpu_ctx {
  int device = 0;
  cudaStream_t stream = nullptr, copy_stream = nullptr;
  cudaEvent_t ev[8] = {};
  cudaEvent_t ev_chunk[2] = {};
  // pageable host output: pinned ring + copy threads (plaidgpu_score_finish)
  static constexpr int RING = 3;
  void* ring[RING] = {};
  size_t ring_bytes = 0;
  cudaEvent_t ev_ring[RING] = {};
  CopyPool* pool = nullptr;
  // early shipping (pinned host output): column chunks of the RAW scores cross PCIe while later chunks are still
  // being scored; plaidgpu_score_finish fixes those columns up on the host (same arithmetic as k_fixup)
  double* early_out = nullptr;
  int64_t early_cols = 0;
  cudaEvent_t ev_early = nullptr, ev_d2h[2] = {};
  // the early copies are enqueued by a helper thread: cudaMemcpyAsync blocks its caller once a few GB are queued on
  // the copy engine, and the thread that launches the scoring kernels must never wait for PCIe
  static constexpr int SHIP_EV = 64;
  cudaEvent_t ev_ship[SHIP_EV] = {};
  std::thread shipper;
  std::mutex ship_m;
  std::condition_variable ship_cv;
  std::vector<std::pair<int64_t, int64_t>> ship_q;  // (first column, columns) of the chunks to ship, in order
  bool ship_done = true;
  double d2h_ms_per_col = 0.0, comp_ms_per_col = 0.0;  // measured by the previous call: sizes the early part
  double t_begin = 0.0, t_known = 0.0;  // wall clock: call started / scores and medians known
  // host CSC input of plaid(): i / x cross PCIe in pieces on their own stream; a column chunk waits only for the
  // piece that holds its last entry, so scoring (and the first D2H) starts after ~1/50 of the upload
  static constexpr int H2D_EV = 64;
  cudaStream_t h2d_stream = nullptr;
  cudaEvent_t ev_h2d[H2D_EV] = {};
  int h2d_pieces = 0;
  int64_t h2d_piece = 0;
  bool h2d_pending = false;
  const int32_t* xp_host = nullptr;
  // mailbox: pinned, device-mapped host memory the GPU writes small results into (launch_copy_words)
  void* mbox = nullptr;
  void* mbox_dev = nullptr;
  size_t mbox_cap = 0;
  std::string err;
  int64_t launches = 0;
  double ms[4] = {0, 0, 0, 0};  // 0 score, 1 colstats, 2 fixup, 3 rank

  // gene sets (host copy of the binary pattern)
  bool have_g = false;
  int32_t PG = 0, S = 0;
  std::vector<int32_t> Gp, Gi;
  std::vector<double> g_colsums;  // colSums(matG != 0) over all rows

  // plan: adjacency of X rows, tiled by set range (depends on rowmap)
  bool plan_ok = false;
  int32_t plan_P = 0, plan_hint = 0;
  std::vector<int32_t> plan_rowmap;
  int32_t Ts = 0, T = 0;
  LaunchCfg cfg{};
  int64_t nnz_mapped = 0;
  int32_t n_overlap = 0;
  DevBuf d_ptr, d_idx, d_inv_mean, d_inv_one, d_ns, d_custom_inv, d_beta;
  // gather blocks: sparse X -> one block of the K highest-degree rows (d_dmap) + scatter for the rest;
  // dense X -> every row, in nblocks blocks of K consecutive rows, no scatter at all
  bool plan_dense = false;
  int32_t gK = 0, gblocks = 0;
  int64_t g_entries = 0;
  DevBuf d_dmap, d_dptr, d_didx, d_colscale;
  // tensor-core pass over the block (tc_kernels.cu): tcK = block rows padded to a multiple of 128 (0 = off)
  int32_t tcK = 0, tc_rows = 0, tc_slices = 4;
  DevBuf d_abits, b_tcB, b_colinv, b_tcflag;
  // tail pass over every other row of a sparse X (tail_kernels.cu): Pt rows with a tail id, set-major member lists
  bool tail_on = false;
  int32_t Pt = 0;
  DevBuf d_tmap, d_tptr, d_tidx, d_sorder, b_colfb, b_tcnt, b_trowptr, b_ttotal, b_tent, b_ttmp, b_tcounter;

  // current scoring call
  bool in_call = false, computed = false;
  plaidgpu_opts opts{};
  bool dense = false;
  int32_t P = 0;
  int64_t N = 0, nnz = 0;
  const int32_t* xp = nullptr;
  const int32_t* xi = nullptr;
  const double* xx = nullptr;
  DevBuf b_xp, b_xi, b_xx, b_rank, b_r0, b_colmax, b_raw, b_med_all, b_med_nz, b_colmin, b_scal, b_i32, b_dense, b_rowa, b_rowb, b_fail, b_list, b_ci, b_cx, b_ce;
  double* raw = nullptr;  // device S x N raw scores (caller's buffer or b_raw)
  bool need_norm = false, need_norm_hint = false;
  // which column medians of the raw scores are known (the statistics pass computes only the one the
  // shard's own minimum says normalize_medians will use; the other is computed on demand)
  bool have_all = false, have_nz = false, raw_valid = false, want_both = false;
  double local_min = INFINITY;
  DevBuf b_smin;
  DevBuf b_design;  // this call's rows of the design basis (plaidgpu_design_stats)
  std::vector<double> h_med_all, h_med_nz, h_colmin;
  const double* score_vals = nullptr;  // what the score kernel reads as values
  const double* score_r0 = nullptr;
};

namespace {

// PLAIDGPU_TRACE=1: wall-clock marks of the host path on stderr (development)
double trace_now() {
  struct timespec ts;
  clock_gettime(CLOCK_MONOTONIC, &ts);
  return (double)ts.tv_sec * 1e3 + (double)ts.tv_nsec * 1e-6;
}
void trace(const char* what) {
  static const bool on = getenv("PLAIDGPU_TRACE") != nullptr;
  static double t0 = 0.0;
  if (!on) return;
  const double t = trace_now();
  if (strcmp(what, "begin") == 0) t0 = t;
  fprintf(stderr, "[plaidgpu trace] %8.2f ms  %s\n", t - t0, what);
}

int fail(plaidgpu_ctx* c, int code, const std::string& msg) {
  if (c) c->err = msg;
  return code;
}
int fail_cuda(plaidgpu_ctx* c, cudaError_t e, const char* where) {
  if (c) c->err = std::string(where) + ": " + cudaGetErrorString(e);
  return PLAIDGPU_ERR_CUDA;
}
#define CK(call)                                              \
  do {                                                        \
    cudaError_t _e = (call);                                  \
    if (_e != cudaSuccess) return fail_cuda(c, _e, #call);    \
  } while (0)

// ---- plan ------------------------------------------------------------------------------
int build_plan(plaidgpu_ctx* c, int32_t P, const int32_t* rowmap, int32_t tile_hint, bool dense) {
  if (c->plan_ok && c->plan_P == P && c->plan_hint == tile_hint && c->plan_dense == dense &&
      memcmp(c->plan_rowmap.data(), rowmap, sizeof(int32_t) * (size_t)P) == 0)
    return PLAIDGPU_OK;
  c->plan_ok = false;
  const int32_t S = c->S, PG = c->PG;
  std::vector<int32_t> g2x((size_t)PG, -1);
  int32_t n_overlap = 0;
  for (int32_t r = 0; r < P; ++r) {
    const int32_t g = rowmap[r];
    if (g < 0) continue;
    if (g >= PG) return fail(c, PLAIDGPU_ERR_ARG, "rowmap entry out of range");
    if (g2x[g] != -1) return fail(c, PLAIDGPU_ERR_ARG, "two rows of X map to the same gene-set row");
    g2x[g] = r;
    ++n_overlap;
  }
  c->n_overlap = n_overlap;
  if (n_overlap == 0) return fail(c, PLAIDGPU_ERR_NOOVERLAP, "[plaid] ERROR. No overlapping features.");

  int32_t Ts = 0, T = 0;
  cudaError_t e = score_configure(c->device, S, tile_hint, &Ts, &T, &c->cfg);
  if (e != cudaSuccess) return fail_cuda(c, e, "score_configure");

  // degrees of the X rows and set sizes n_s = |set s ∩ rows(X)|
  std::vector<uint32_t> deg((size_t)P, 0);
  std::vector<double> ns((size_t)S, 0.0);
  int64_t nnzm = 0;
  for (int32_t s = 0; s < S; ++s)
    for (int32_t q = c->Gp[s]; q < c->Gp[s + 1]; ++q) {
      const int32_t r = g2x[c->Gi[q]];
      if (r >= 0) {
        ++deg[r];
        ns[s] += 1.0;
        ++nnzm;
      }
    }

  // ---- the block: rows of X that leave the scatter pass ---------------------------------------
  // sparse X: the highest-degree rows (in single-cell data the ubiquitous genes: nearly dense rows of X that
  // sit in thousands of sets and carry most of the adds); dense X: every row.  The block is scored on the
  // tensor cores (tc_kernels.cu) from bit masks of t(G); the fp64 gather passes (blocks of gK local ids,
  // gather_kernels.cu) cover the same rows when the tensor-core path is off or meets a non-finite entry.
  const int Kmax = gather_max_block(c->device);
  bool tc_on = true;
  if (const char* e = getenv("PLAIDGPU_TC")) tc_on = atoi(e) != 0;
  std::vector<uint16_t> dmap;          // sparse mode: row -> local id in the block, 0xFFFF otherwise
  std::vector<int32_t> blk_of_row;     // sparse mode: row -> gather block or -1
  std::vector<int32_t> local_of_row;   // row -> local id in the block or -1 (both modes)
  int32_t gK = 0, gblocks = 0, tcK = 0, tc_rows = 0;
  if (dense) {
    gK = std::min<int32_t>(Kmax, ((P + 31) / 32) * 32);
    if (gK <= 0) return fail(c, PLAIDGPU_ERR_CUDA, "no shared memory for the gather tile");
    gblocks = (P + gK - 1) / gK;
    if (tc_on && S >= 128 && P >= 128 && P <= 32768) {  // 128 * Kp must stay below 2^22 (tc epilogue)
      tc_rows = P;
      tcK = ((P + 127) / 128) * 128;
      local_of_row.resize((size_t)P);
      for (int32_t r = 0; r < P; ++r) local_of_row[r] = r;
    }
  } else if (Kmax > 0 && S >= 1024 && nnzm >= 100000) {
    std::vector<int32_t> order((size_t)P);
    for (int32_t r = 0; r < P; ++r) order[r] = r;
    std::sort(order.begin(), order.end(),
              [&](int32_t x, int32_t y) { return deg[x] != deg[y] ? deg[x] > deg[y] : x < y; });
    int32_t k = 0;
    if (tc_on) {
      // a row costs the tensor-core pass the same whatever its degree, the tail pass in proportion to it (degree x
      // ceil(entries per 1,056-cell tile / 32)): rows in at least ~0.75 % of the sets go to the block (about 1,800
      // rows on the 30k-set benchmark collection; measured optimum 1,536 - 2,048)
      double frac = 0.0075;
      if (const char* e = getenv("PLAIDGPU_TC_DEGFRAC")) frac = atof(e);
      const uint32_t thr = (uint32_t)std::max(32.0, ceil(frac * (double)S));
      while (k < P && deg[order[k]] >= thr) ++k;
      k = std::min<int32_t>(k, 8192);
      if (const char* e = getenv("PLAIDGPU_TC_K")) k = std::max(0, std::min<int32_t>({atoi(e), P, 8192}));
      k = (k / 128) * 128;  // whole K blocks: the padding of a partial one would be paid for like real rows
      while (k > 0 && deg[order[k - 1]] == 0) --k;
      if (k >= 128) {
        tc_rows = k;
        tcK = ((k + 127) / 128) * 128;
      } else {
        k = 0;
      }
    }
    if (k == 0) {  // legacy: one gather block of the Kmax highest-degree rows
      int want_blocks = 1;  // measured on C4: a 2nd / 3rd block costs more (extra pass over the output) than it saves
      if (const char* e = getenv("PLAIDGPU_GATHER_BLOCKS")) want_blocks = std::max(0, std::min(8, atoi(e)));
      const int32_t want = (int32_t)std::min<int64_t>((int64_t)Kmax * want_blocks, P);
      while (k < want && deg[order[k]] > 0) ++k;
      if (k >= Kmax) k = (k / Kmax) * Kmax;      // full blocks only, except that a single partial block of
      else if (k < 32) k = 0;                    // >= 32 rows is still worth a gather pass
    }
    if (k > 0) {
      gK = std::min(Kmax, ((k + 31) / 32) * 32);
      gblocks = (k + gK - 1) / gK;
      std::vector<int32_t> sel(order.begin(), order.begin() + k);
      std::sort(sel.begin(), sel.end());  // local ids ascend with the row index (reference sum order)
      blk_of_row.assign((size_t)P, -1);
      local_of_row.assign((size_t)P, -1);
      dmap.assign((size_t)P, 0xFFFFu);
      for (size_t i = 0; i < sel.size(); ++i) {
        dmap[sel[i]] = (uint16_t)i;
        local_of_row[sel[i]] = (int32_t)i;
        blk_of_row[sel[i]] = (int32_t)(i / (size_t)gK);
      }
    }
  }
  // set-major member lists per block, 16-bit local ids, padded to multiples of 4 with gK (a zero row)
  std::vector<uint32_t> dptr;
  std::vector<uint32_t> didx;  // local id * 256 = byte offset of the row in the [K+1][32] fp64 tile
  if (gblocks > 0) {
    dptr.assign((size_t)gblocks * (S + 1), 0);
    // count
    std::vector<uint32_t> cnt((size_t)gblocks * S, 0);
    for (int32_t s = 0; s < S; ++s)
      for (int32_t q = c->Gp[s]; q < c->Gp[s + 1]; ++q) {
        const int32_t r = g2x[c->Gi[q]];
        if (r < 0) continue;
        if (dense) ++cnt[(size_t)(r / gK) * S + s];
        else if (blk_of_row[r] >= 0) ++cnt[(size_t)blk_of_row[r] * S + s];
      }
    uint64_t off = 0;
    for (int32_t b = 0; b < gblocks; ++b) {
      for (int32_t s = 0; s < S; ++s) {
        dptr[(size_t)b * (S + 1) + s] = (uint32_t)off;
        off += (cnt[(size_t)b * S + s] + 3u) & ~3u;
      }
      dptr[(size_t)b * (S + 1) + S] = (uint32_t)off;
    }
    if (off >= 0xFFFFFFFFull) return fail(c, PLAIDGPU_ERR_ARG, "gene-set matrix too large for 32-bit offsets");
    didx.assign((size_t)std::max<uint64_t>(off, 4), (uint32_t)gK * 256u);
    std::vector<uint32_t> pos((size_t)gblocks * S);
    for (int32_t b = 0; b < gblocks; ++b)
      for (int32_t s = 0; s < S; ++s) pos[(size_t)b * S + s] = dptr[(size_t)b * (S + 1) + s];
    // members of a set arrive in the order of matG's rows; sort each list so sums run in ascending X row
    for (int32_t s = 0; s < S; ++s)
      for (int32_t q = c->Gp[s]; q < c->Gp[s + 1]; ++q) {
        const int32_t r = g2x[c->Gi[q]];
        if (r < 0) continue;
        if (dense) didx[pos[(size_t)(r / gK) * S + s]++] = (uint32_t)(r % gK) * 256u;
        else if (blk_of_row[r] >= 0)
          didx[pos[(size_t)blk_of_row[r] * S + s]++] = (uint32_t)(local_of_row[r] % gK) * 256u;
      }
    for (int32_t b = 0; b < gblocks; ++b)
      for (int32_t s = 0; s < S; ++s) {
        const uint32_t lo = dptr[(size_t)b * (S + 1) + s];
        std::sort(didx.begin() + lo, didx.begin() + pos[(size_t)b * S + s]);
      }
    c->g_entries = (int64_t)off;
  }

  // ---- scatter adjacency (sparse X only): CSR by X row without the gather-block rows ----------
  std::vector<uint32_t> ptr;
  std::vector<uint16_t> idx(1);
  int64_t nnz_scatter = 0;
  if (!dense) {
    auto in_block = [&](int32_t r) { return !blk_of_row.empty() && blk_of_row[r] >= 0; };
    std::vector<uint32_t> rowcnt((size_t)P + 1, 0);
    for (int32_t r = 0; r < P; ++r) rowcnt[r + 1] = rowcnt[r] + (in_block(r) ? 0u : deg[r]);
    nnz_scatter = rowcnt[P];
    std::vector<uint32_t> fill(rowcnt.begin(), rowcnt.end() - 1);
    std::vector<int32_t> setof((size_t)std::max<int64_t>(nnz_scatter, 1));
    // walking the sets in ascending order leaves every row's list sorted by set
    for (int32_t s = 0; s < S; ++s)
      for (int32_t q = c->Gp[s]; q < c->Gp[s + 1]; ++q) {
        const int32_t r = g2x[c->Gi[q]];
        if (r >= 0 && !in_block(r)) setof[fill[r]++] = s;
      }
    // one 32-byte record per (row, tile): {u32 overflow offset, u16 length, u16 0, u16 entry[12]}; entries
    // are byte offsets (tile-local set id * 8); lists longer than 12 continue in the overflow array in
    // chunks of 4 padded with 0xFFFF
    idx.clear();
    idx.reserve((size_t)nnz_scatter / 4 + 16);
    ptr.assign((size_t)P * T * 8, 0);
    for (int32_t r = 0; r < P; ++r) {
      uint32_t e0 = rowcnt[r];
      const uint32_t e1 = rowcnt[r + 1];
      for (int32_t t = 0; t < T; ++t) {
        uint32_t* rc = ptr.data() + ((size_t)r * T + t) * 8;
        const int32_t hi = (t + 1) * Ts;
        uint16_t in12[12];
        for (int k = 0; k < 12; ++k) in12[k] = 0xFFFFu;
        uint32_t n = 0;
        rc[0] = (uint32_t)idx.size();
        while (e0 < e1 && setof[e0] < hi) {
          const uint16_t off = (uint16_t)((setof[e0] - t * Ts) * 8);
          if (n < 12) in12[n] = off; else idx.push_back(off);
          ++n;
          ++e0;
        }
        while (idx.size() & 3) idx.push_back((uint16_t)0xFFFFu);
        if (n > 0xFFFFu) return fail(c, PLAIDGPU_ERR_ARG, "gene-set list too long for one tile");
        rc[1] = n;
        for (int k = 0; k < 6; ++k) rc[2 + k] = (uint32_t)in12[2 * k] | ((uint32_t)in12[2 * k + 1] << 16);
      }
    }
    for (int k = 0; k < 8; ++k) idx.push_back((uint16_t)0xFFFFu);
  }
  // bit masks of t(G) over the block for the tensor-core pass: [set tile][K block][128 set rows] x 128 bits
  std::vector<uint32_t> abits;
  if (tcK > 0) {
    const size_t tiles_m = ((size_t)S + 127) / 128, kbn = (size_t)tcK / 128;
    abits.assign(tiles_m * kbn * 128 * 4, 0u);
    for (int32_t s = 0; s < S; ++s)
      for (int32_t q = c->Gp[s]; q < c->Gp[s + 1]; ++q) {
        const int32_t r = g2x[c->Gi[q]];
        if (r < 0) continue;
        const int32_t l = local_of_row[r];
        if (l < 0) continue;
        // gene t of a 32-gene word sits at bit 8 (t mod 4) + t / 4: the expander's (w >> k) & 0x01010101 then
        // yields TMEM column k = genes 4k .. 4k+3 as four 0/1 bytes
        const size_t m = (size_t)s >> 7, i = (size_t)s & 127, kb = (size_t)l >> 7, b = (size_t)l & 127, t = b & 31;
        abits[((m * kbn + kb) * 128 + i) * 4 + (b >> 5)] |= 1u << (8 * (t & 3) + (t >> 2));
      }
  }
  // tail pass (sparse X with a tensor-core block): every other row that is in at least one set gets a tail id
  // (ascending with the row index = the reference's summation order); member lists per set; sets by tail size
  std::vector<int32_t> tmap, sorder;
  std::vector<uint32_t> tptr;
  std::vector<uint16_t> tidx;
  int32_t Pt = 0;
  bool tail_on = !dense && tcK > 0;
  if (const char* e = getenv("PLAIDGPU_TAIL")) tail_on = tail_on && atoi(e) != 0;
  if (tail_on) {
    tmap.assign((size_t)P, -1);
    for (int32_t r = 0; r < P; ++r)
      if (deg[r] > 0 && local_of_row[r] < 0) tmap[r] = Pt++;
    if (Pt > 65535) tail_on = false;  // 16-bit member ids
  }
  if (tail_on) {
    tptr.assign((size_t)S + 1, 0);
    tidx.reserve((size_t)nnzm);
    std::vector<uint16_t> one;
    for (int32_t s = 0; s < S; ++s) {
      one.clear();
      for (int32_t q = c->Gp[s]; q < c->Gp[s + 1]; ++q) {
        const int32_t r = g2x[c->Gi[q]];
        if (r >= 0 && tmap[r] >= 0) one.push_back((uint16_t)tmap[r]);
      }
      std::sort(one.begin(), one.end());
      tidx.insert(tidx.end(), one.begin(), one.end());
      tptr[s + 1] = (uint32_t)tidx.size();
    }
    if (tidx.empty()) tidx.push_back(0);
    sorder.resize((size_t)S);
    for (int32_t s = 0; s < S; ++s) sorder[s] = s;
    std::stable_sort(sorder.begin(), sorder.end(), [&](int32_t a, int32_t b) {
      return tptr[a + 1] - tptr[a] > tptr[b + 1] - tptr[b];
    });
  }
  std::vector<double> inv_mean((size_t)S), inv_one((size_t)S, 1.0);
  for (int32_t s = 0; s < S; ++s) inv_mean[s] = 1.0 / (1e-8 + ns[s]);  // R/plaid.R:75-76

  auto up = [&](DevBuf& b, const void* src, size_t bytes) -> cudaError_t {
    cudaError_t e2 = b.reserve(std::max<size_t>(bytes, 16));
    if (e2 != cudaSuccess || bytes == 0) return e2;
    return cudaMemcpyAsync(b.p, src, bytes, cudaMemcpyHostToDevice, c->stream);
  };
  CK(up(c->d_ptr, ptr.data(), ptr.size() * sizeof(uint32_t)));
  CK(up(c->d_idx, idx.data(), idx.size() * sizeof(uint16_t)));
  CK(up(c->d_inv_mean, inv_mean.data(), (size_t)S * sizeof(double)));
  CK(up(c->d_inv_one, inv_one.data(), (size_t)S * sizeof(double)));
  CK(up(c->d_ns, ns.data(), (size_t)S * sizeof(double)));
  CK(up(c->d_dmap, dmap.data(), dmap.size() * sizeof(uint16_t)));
  CK(up(c->d_dptr, dptr.data(), dptr.size() * sizeof(uint32_t)));
  CK(up(c->d_didx, didx.data(), didx.size() * sizeof(uint32_t)));
  CK(up(c->d_abits, abits.data(), abits.size() * sizeof(uint32_t)));
  CK(up(c->d_tmap, tmap.data(), tmap.size() * sizeof(int32_t)));
  CK(up(c->d_tptr, tptr.data(), tptr.size() * sizeof(uint32_t)));
  CK(up(c->d_tidx, tidx.data(), tidx.size() * sizeof(uint16_t)));
  CK(up(c->d_sorder, sorder.data(), sorder.size() * sizeof(int32_t)));
  CK(cudaStreamSynchronize(c->stream));  // the host vectors die with this scope
  c->tail_on = tail_on;
  c->Pt = Pt;
  c->Ts = Ts;
  c->T = T;
  c->gK = gK;
  c->gblocks = gblocks;
  c->tcK = tcK;
  c->tc_rows = tc_rows;
  c->tc_slices = 4;
  if (const char* e = getenv("PLAIDGPU_TC_SLICES")) c->tc_slices = (atoi(e) == 2) ? 2 : 4;
  c->nnz_mapped = nnzm;
  c->plan_P = P;
  c->plan_hint = tile_hint;
  c->plan_dense = dense;
  c->plan_rowmap.assign(rowmap, rowmap + P);
  c->plan_ok = true;
  return PLAIDGPU_OK;
}

// bring a caller buffer onto the device (or alias it when it already is there)
template <typename T>
int to_device(plaidgpu_ctx* c, const T* src, size_t n, int location, DevBuf& buf, const T** out) {
  if (location == PLAIDGPU_DEVICE) {
    *out = src;
    return PLAIDGPU_OK;
  }
  CK(buf.reserve(std::max<size_t>(n, 1) * sizeof(T)));
  if (n) CK(cudaMemcpyAsync(buf.p, src, n * sizeof(T), cudaMemcpyHostToDevice, c->stream));
  *out = buf.as<T>();
  return PLAIDGPU_OK;
}

int device_minmax(plaidgpu_ctx* c, const double* d, int64_t n, double* mn, double* mx) {
  CK(c->b_scal.reserve(4 * sizeof(double)));
  CK(launch_minmax(d, n, c->b_scal.as<double>(), c->stream));
  c->launches += (n > 0) ? 3 : 2;
  double h[2];
  CK(cudaMemcpyAsync(h, c->b_scal.p, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  *mn = h[0];
  *mx = h[1];
  return PLAIDGPU_OK;
}

// pinned ring + copy threads shared by the pageable upload (load_matrix) and the pageable result path (finish)
int ensure_ring(plaidgpu_ctx* c) {
  const size_t want = (size_t)256 << 20;
  if (!c->ring[0] || c->ring_bytes < want) {
    for (int i = 0; i < plaidgpu_ctx::RING; ++i) {
      if (c->ring[i]) cudaFreeHost(c->ring[i]);
      c->ring[i] = nullptr;
      CK(cudaMallocHost(&c->ring[i], want));
      if (!c->ev_ring[i]) CK(cudaEventCreateWithFlags(&c->ev_ring[i], cudaEventDisableTiming));
    }
    c->ring_bytes = want;
  }
  if (!c->pool) {
    int nt = (int)std::min<unsigned>(12, std::max(2u, std::thread::hardware_concurrency() * 3 / 4));
    if (const char* e = getenv("PLAIDGPU_COPY_THREADS")) nt = std::max(1, std::min(64, atoi(e)));
    c->pool = new CopyPool(nt);
  }
  return PLAIDGPU_OK;
}

// pageable host array -> device through the pinned ring: the copy threads fill slot k + 1 while slot k crosses PCIe
// (the driver's own staging of a pageable cudaMemcpyAsync is single-threaded: ~11 GB/s measured)
int upload_pageable(plaidgpu_ctx* c, void* dev, const void* host, size_t bytes, cudaStream_t st) {
  int rc = ensure_ring(c);
  if (rc) return rc;
  const char* src = static_cast<const char*>(host);
  char* dst = static_cast<char*>(dev);
  int k = 0;
  for (size_t off = 0; off < bytes; off += c->ring_bytes, ++k) {
    const size_t n = std::min(c->ring_bytes, bytes - off);
    const int slot = k % plaidgpu_ctx::RING;
    if (k >= plaidgpu_ctx::RING) CK(cudaEventSynchronize(c->ev_ring[slot]));
    c->pool->copy(c->ring[slot], src + off, n);
    CK(cudaMemcpyAsync(dst + off, c->ring[slot], n, cudaMemcpyHostToDevice, st));
    CK(cudaEventRecord(c->ev_ring[slot], st));
  }
  for (int i = 0; i < std::min(k, (int)plaidgpu_ctx::RING); ++i) CK(cudaEventSynchronize(c->ev_ring[i]));  // slots are free again
  return PLAIDGPU_OK;
}

int load_matrix(plaidgpu_ctx* c, const plaidgpu_matrix* X, bool piecewise = false) {
  c->dense = (X->kind == PLAIDGPU_DENSE);
  c->P = X->P;
  c->N = X->N;
  if (X->P <= 0 || X->N < 0) return fail(c, PLAIDGPU_ERR_ARG, "bad matrix dimensions");
  if (c->dense) {
    if (!X->x && X->N > 0) return fail(c, PLAIDGPU_ERR_ARG, "dense X without values");
    c->nnz = (int64_t)X->P * X->N;
    c->xp = nullptr;
    c->xi = nullptr;
    int rc = to_device<double>(c, X->x, (size_t)c->nnz, X->location, c->b_xx, &c->xx);
    if (rc) return rc;
  } else if (X->kind == PLAIDGPU_CSC) {
    if (!X->p) return fail(c, PLAIDGPU_ERR_ARG, "CSC X without column pointers");
    int32_t last = 0;
    if (X->location == PLAIDGPU_HOST) {
      last = X->p[X->N];
    } else {
      CK(cudaMemcpyAsync(&last, X->p + X->N, sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
      CK(cudaStreamSynchronize(c->stream));
    }
    c->nnz = last;
    int rc = to_device<int32_t>(c, X->p, (size_t)X->N + 1, X->location, c->b_xp, &c->xp);
    if (rc) return rc;
    c->h2d_pending = false;
    c->xp_host = nullptr;
    int64_t piece_min = (int64_t)4 << 20;  // entries per piece (48 MB); test knob: PLAIDGPU_H2D_PIECE
    if (const char* e = getenv("PLAIDGPU_H2D_PIECE")) piece_min = std::max<int64_t>(1024, atoll(e));
    const bool big_pageable = X->location == PLAIDGPU_HOST && c->nnz > ((int64_t)4 << 20) && is_pageable(X->x) &&
                              !getenv("PLAIDGPU_NO_RING");
    if (big_pageable) {
      // a pageable X (an R dgCMatrix): staged through the pinned ring by the copy threads
      CK(c->b_xi.reserve((size_t)c->nnz * sizeof(int32_t)));
      CK(c->b_xx.reserve((size_t)c->nnz * sizeof(double)));
      CK(cudaStreamSynchronize(c->stream));  // the buffers may still be read by the previous call's kernels
      rc = upload_pageable(c, c->b_xi.p, X->i, (size_t)c->nnz * sizeof(int32_t), c->stream);
      if (rc) return rc;
      rc = upload_pageable(c, c->b_xx.p, X->x, (size_t)c->nnz * sizeof(double), c->stream);
      if (rc) return rc;
      c->xi = c->b_xi.as<int32_t>();
      c->xx = c->b_xx.as<double>();
    } else if (piecewise && X->location == PLAIDGPU_HOST && c->nnz > 2 * piece_min && !getenv("PLAIDGPU_NO_H2D_PIPE")) {
      // pieces of i and x on the upload stream, one event each (see plaidgpu_ctx::ev_h2d)
      CK(c->b_xi.reserve((size_t)c->nnz * sizeof(int32_t)));
      CK(c->b_xx.reserve((size_t)c->nnz * sizeof(double)));
      c->h2d_piece = std::max<int64_t>(piece_min, (c->nnz + plaidgpu_ctx::H2D_EV - 1) / plaidgpu_ctx::H2D_EV);
      c->h2d_pieces = (int)((c->nnz + c->h2d_piece - 1) / c->h2d_piece);
      CK(cudaEventRecord(c->ev_chunk[1], c->stream));  // buffers may still be read by the previous call's kernels
      CK(cudaStreamWaitEvent(c->h2d_stream, c->ev_chunk[1], 0));
      for (int k = 0; k < c->h2d_pieces; ++k) {
        const int64_t e0 = (int64_t)k * c->h2d_piece, n = std::min<int64_t>(c->h2d_piece, c->nnz - e0);
        CK(cudaMemcpyAsync(c->b_xi.as<int32_t>() + e0, X->i + e0, (size_t)n * sizeof(int32_t), cudaMemcpyHostToDevice, c->h2d_stream));
        CK(cudaMemcpyAsync(c->b_xx.as<double>() + e0, X->x + e0, (size_t)n * sizeof(double), cudaMemcpyHostToDevice, c->h2d_stream));
        CK(cudaEventRecord(c->ev_h2d[k], c->h2d_stream));
      }
      c->xi = c->b_xi.as<int32_t>();
      c->xx = c->b_xx.as<double>();
      c->h2d_pending = true;
      c->xp_host = X->p;
    } else {
      rc = to_device<int32_t>(c, X->i, (size_t)c->nnz, X->location, c->b_xi, &c->xi);
      if (rc) return rc;
      rc = to_device<double>(c, X->x, (size_t)c->nnz, X->location, c->b_xx, &c->xx);
      if (rc) return rc;
    }
  } else {
    return fail(c, PLAIDGPU_ERR_ARG, "unknown matrix kind");
  }
  return PLAIDGPU_OK;
}

// the compute stream waits for the upload pieces up to entry `upto` (exclusive); upto < 0: all of X
int h2d_wait(plaidgpu_ctx* c, int64_t upto) {
  if (!c->h2d_pending) return PLAIDGPU_OK;
  int k = c->h2d_pieces - 1;
  if (upto >= 0 && upto < c->nnz) k = (int)(std::max<int64_t>(upto - 1, 0) / c->h2d_piece);
  CK(cudaStreamWaitEvent(c->stream, c->ev_h2d[k], 0));
  if (k == c->h2d_pieces - 1) c->h2d_pending = false;
  return PLAIDGPU_OK;
}

// gsva works on a dense matrix: expand a CSC shard on the device (zeros filled)
int make_dense(plaidgpu_ctx* c) {
  if (c->dense) return PLAIDGPU_OK;
  const int64_t total = (int64_t)c->P * c->N;
  CK(c->b_dense.reserve((size_t)std::max<int64_t>(total, 1) * sizeof(double)));
  CK(launch_densify(c->xp, c->xi, c->xx, c->P, c->N, c->b_dense.as<double>(), c->stream));
  c->launches += 1;
  c->dense = true;
  c->xp = nullptr;
  c->xi = nullptr;
  c->xx = c->b_dense.as<double>();
  c->nnz = total;
  return PLAIDGPU_OK;
}

// out_host[r] = sum_j x[r,j] or sum_j (x[r,j] - mean[r])^2 of the (dense) loaded matrix
int row_moments(plaidgpu_ctx* c, const double* mean_host, double* out_host) {
  CK(c->b_rowa.reserve((size_t)c->P * sizeof(double)));
  CK(c->b_rowb.reserve((size_t)c->P * sizeof(double)));
  const double* dmean = nullptr;
  if (mean_host) {
    CK(cudaMemcpyAsync(c->b_rowb.p, mean_host, (size_t)c->P * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    dmean = c->b_rowb.as<double>();
  }
  CK(launch_row_moments(c->xx, c->P, c->N, dmean, c->b_rowa.as<double>(), c->stream));
  c->launches += 1;
  CK(cudaMemcpyAsync(out_host, c->b_rowa.p, (size_t)c->P * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return PLAIDGPU_OK;
}

bool is_rank_scorer(int s) {
  return s == PLAIDGPU_SING || s == PLAIDGPU_SSGSEA || s == PLAIDGPU_UCELL || s == PLAIDGPU_AUCELL;
}

// the scores of the call are median-normalised (normalize_medians, R/plaid.R)
bool needs_norm(const plaidgpu_opts& o) {
  return (o.scorer == PLAIDGPU_PLAID && o.normalize) || o.scorer == PLAIDGPU_SSGSEA || o.scorer == PLAIDGPU_UCELL ||
         o.scorer == PLAIDGPU_AUCELL || o.scorer == PLAIDGPU_GSVA;
}

// order-preserving key -> double on the host (inverse of key_of in common.cuh)
double host_value_of(unsigned long long k) {
  const unsigned long long b = (k & 0x8000000000000000ull) ? (k & 0x7fffffffffffffffull) : ~k;
  double d;
  memcpy(&d, &b, sizeof(d));
  return d;
}

// the statistics pass over the raw scores of the current call
int run_colstats(plaidgpu_ctx* c, int which) {
  CK(c->b_med_all.reserve(std::max<int64_t>(c->N, 1) * sizeof(double)));
  CK(c->b_med_nz.reserve(std::max<int64_t>(c->N, 1) * sizeof(double)));
  CK(c->b_colmin.reserve(std::max<int64_t>(c->N, 1) * sizeof(double)));
  CK(c->b_fail.reserve(sizeof(int)));
  CK(c->b_list.reserve(std::max<int64_t>(c->N, 1) * sizeof(int64_t)));
  CK(launch_colstats(c->raw, c->S, c->S, c->N, c->b_med_all.as<double>(), c->b_med_nz.as<double>(),
                     c->b_colmin.as<double>(), c->b_fail.as<int>(), c->b_list.as<int64_t>(), which, c->stream));
  c->launches += 1;
  if (which != COLSTATS_NZ) c->have_all = true;
  if (which != COLSTATS_ALL) c->have_nz = true;
  return PLAIDGPU_OK;
}

// ---- helper thread that enqueues the early result blocks (see plaidgpu_ctx::shipper) ----
void ship_join(plaidgpu_ctx* c) {
  if (!c->shipper.joinable()) return;
  {
    std::lock_guard<std::mutex> lk(c->ship_m);
    c->ship_done = true;
  }
  c->ship_cv.notify_all();
  c->shipper.join();
}
void ship_body(plaidgpu_ctx* c) {
  cudaSetDevice(c->device);
  size_t next = 0;
  for (;;) {
    std::pair<int64_t, int64_t> job;
    {
      std::unique_lock<std::mutex> lk(c->ship_m);
      c->ship_cv.wait(lk, [&] { return next < c->ship_q.size() || c->ship_done; });
      if (next >= c->ship_q.size()) return;
      job = c->ship_q[next];
    }
    cudaStreamWaitEvent(c->copy_stream, c->ev_ship[next], 0);
    cudaMemcpyAsync(c->early_out + job.first * (int64_t)c->S, c->raw + job.first * (int64_t)c->S,
                    (size_t)job.second * c->S * sizeof(double), cudaMemcpyDeviceToHost, c->copy_stream);
    cudaEventRecord(c->ev_early, c->copy_stream);
    ++next;
  }
}
// forget the result blocks that left early: wait until their copies have landed, so that nothing overwrites the
// raw scores under them, and let plaidgpu_score_finish ship every column
int drop_early(plaidgpu_ctx* c) {
  ship_join(c);
  CK(cudaStreamSynchronize(c->copy_stream));
  c->early_cols = 0;
  return PLAIDGPU_OK;
}
// called by the scoring thread right after the kernels of a chunk were launched
int ship_chunk(plaidgpu_ctx* c, int64_t j0, int64_t nj) {
  size_t k;
  {
    std::lock_guard<std::mutex> lk(c->ship_m);
    k = c->ship_q.size();
  }
  if (k >= (size_t)plaidgpu_ctx::SHIP_EV) return 1;  // out of events: the rest leaves after the fix-up
  CK(cudaEventRecord(c->ev_ship[k], c->stream));
  {
    std::lock_guard<std::mutex> lk(c->ship_m);
    c->ship_q.emplace_back(j0, nj);
  }
  if (!c->shipper.joinable()) {
    c->ship_done = false;
    c->shipper = std::thread(ship_body, c);
  }
  c->ship_cv.notify_all();
  return PLAIDGPU_OK;
}

// Small device -> host reads (8-byte words) through the mailbox: a kernel stores into mapped host memory, so the
// read does not wait behind result blocks queued in the copy engine.  items: {host dst, device src, words}
struct SmallRead {
  void* host;
  const void* dev;
  int64_t words;
};
int read_small(plaidgpu_ctx* c, const SmallRead* it, int n) {
  int64_t total = 0;
  for (int k = 0; k < n; ++k) total += it[k].words;
  if (total <= 0) {
    CK(cudaStreamSynchronize(c->stream));
    return PLAIDGPU_OK;
  }
  if (c->mbox_cap < (size_t)total * 8) {
    if (c->mbox) cudaFreeHost(c->mbox);
    c->mbox = nullptr;
    c->mbox_cap = 0;
    const size_t want = std::max<size_t>((size_t)total * 8, (size_t)1 << 20);
    CK(cudaHostAlloc(&c->mbox, want, cudaHostAllocMapped));
    CK(cudaHostGetDevicePointer(&c->mbox_dev, c->mbox, 0));
    c->mbox_cap = want;
  }
  int64_t off = 0;
  for (int k = 0; k < n; ++k) {
    CK(launch_copy_words(it[k].dev, static_cast<char*>(c->mbox_dev) + off * 8, it[k].words, c->stream));
    off += it[k].words;
  }
  CK(cudaStreamSynchronize(c->stream));
  off = 0;
  for (int k = 0; k < n; ++k) {
    if (it[k].words > 0) memcpy(it[k].host, static_cast<char*>(c->mbox) + off * 8, (size_t)it[k].words * 8);
    off += it[k].words;
  }
  return PLAIDGPU_OK;
}

int fetch_medians(plaidgpu_ctx* c) {
  c->h_med_all.resize((size_t)c->N);
  c->h_med_nz.resize((size_t)c->N);
  c->h_colmin.resize((size_t)c->N);
  const SmallRead it[3] = {{c->h_med_all.data(), c->b_med_all.p, c->have_all ? c->N : 0},
                           {c->h_med_nz.data(), c->b_med_nz.p, c->have_nz ? c->N : 0},
                           {c->h_colmin.data(), c->b_colmin.p, c->N}};
  return read_small(c, it, 3);
}

// make the plain (want_nz = false) or the non-zero median of every column available on device and host
int ensure_median(plaidgpu_ctx* c, bool want_nz) {
  if (want_nz ? c->have_nz : c->have_all) return PLAIDGPU_OK;
  if (!c->raw_valid) return fail(c, PLAIDGPU_ERR_STATE, "the raw scores are gone (plaidgpu_score_finish already ran)");
  CK(cudaSetDevice(c->device));
  int rc = run_colstats(c, want_nz ? COLSTATS_NZ : COLSTATS_ALL);
  if (rc) return rc;
  return fetch_medians(c);
}

int max_col_nnz(plaidgpu_ctx* c, int32_t* out) {
  CK(c->b_i32.reserve(sizeof(int32_t)));
  CK(launch_max_col_nnz(c->xp, c->N, c->b_i32.as<int32_t>(), c->stream));
  c->launches += 1;
  CK(cudaMemcpyAsync(out, c->b_i32.p, sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return PLAIDGPU_OK;
}

// one column of the fix-up on the host: out = alpha * (x + ((-med) + c)) [+ beta_s], every operation rounded on its own
// like the device kernels (k_fixup / k_fixup_flat are written with __dadd_rn / __dmul_rn, this file is compiled
// without FMA contraction for the host)
#pragma GCC push_options
#pragma GCC optimize("fp-contract=off")
void host_fixup_column(double* col, int32_t S, double med, bool has_med, double c, double alpha, const double* beta) {
  const double shift = (has_med ? -med : 0.0) + c;
  if (beta) {
    for (int32_t s = 0; s < S; ++s) {
      const double t = alpha * (col[s] + shift);
      col[s] = t + beta[s];
    }
  } else {
    for (int32_t s = 0; s < S; ++s) col[s] = alpha * (col[s] + shift);
  }
}
#pragma GCC pop_options

double r_mean(const double* v, int64_t n) {  // base::mean(na.rm = TRUE): long double, one refinement
  long double s = 0.0L;
  int64_t m = 0;
  for (int64_t i = 0; i < n; ++i)
    if (v[i] == v[i]) {
      s += v[i];
      ++m;
    }
  if (m == 0) return NAN;
  s /= (long double)m;
  long double t = 0.0L;
  for (int64_t i = 0; i < n; ++i)
    if (v[i] == v[i]) t += (v[i] - s);
  return (double)(s + t / (long double)m);
}

// ---- per-group moments (plaid.test "lm" for K groups) ---------------------------------------
// labels: int32[N] in [-1, K); -1 = the column belongs to no group
int check_groups(plaidgpu_ctx* c, const int32_t* labels, int64_t N, int K) {
  if (K < 1) return fail(c, PLAIDGPU_ERR_ARG, "the number of groups K must be at least 1");
  if (N > 0 && !labels) return fail(c, PLAIDGPU_ERR_ARG, "null argument");
  if (N >= INT32_MAX) return fail(c, PLAIDGPU_ERR_ARG, "group statistics take fewer than 2^31 columns per call");
  for (int64_t j = 0; j < N; ++j)
    if (labels[j] < -1 || labels[j] >= K)
      return fail(c, PLAIDGPU_ERR_ARG, "label " + std::to_string(labels[j]) + " of column " + std::to_string(j) +
                                           " is outside [-1, " + std::to_string(K) + ")");
  return PLAIDGPU_OK;
}

// Column chunks of a reduction whose result is `width` doubles: up to 64 (and at least 64 columns each), fewer when
// the per-chunk partials would exceed 1 GiB.  K <= 2 groups (width 2 K S) keep min(64, N / 64) for any S below two
// million sets.
int reduce_nchunk(int64_t N, int64_t width) {
  const double partial_budget = 1073741824.0;
  int64_t n = std::min<int64_t>(64, N / 64);
  n = std::min<int64_t>(n, (int64_t)(partial_budget / ((double)width * 8.0)));
  return (int)std::max<int64_t>(1, n);
}

// Per-group sums / sums of squares of the S x N device matrix dx (ld = S) into host out[K][2][S] (checked labels).
// The host counting-sorts the labelled columns by (chunk, group), keeping column order inside a group, so each
// group's values are added in column order within a chunk and the chunks in chunk order: for K = 2 and labels
// y != 0 these are the additions of the two-group reduction this replaced, operation by operation.
// fix / med / cc / alpha / beta: the fix-up of plaidgpu_score_finish, applied in registers to raw scores.
int group_stats_device(plaidgpu_ctx* c, const double* dx, int32_t S, int64_t N, const int32_t* labels, int K, double* out,
                       bool fix = false, const double* med = nullptr, double cc = 0.0, double alpha = 1.0,
                       const double* beta = nullptr) {
  const int nchunk = reduce_nchunk(N, (int64_t)K * 2 * S);
  const int64_t nseg = (int64_t)nchunk * K;
  std::vector<int32_t> plan((size_t)(nseg + 1 + N));  // seg[nseg + 1], then cols
  int32_t* seg = plan.data();
  int32_t* cols = seg + nseg + 1;
  for (int ch = 0; ch < nchunk; ++ch)
    for (int64_t j = (N * ch) / nchunk, j1 = (N * (ch + 1)) / nchunk; j < j1; ++j)
      if (labels[j] >= 0) ++seg[(int64_t)ch * K + labels[j] + 1];
  for (int64_t g = 0; g < nseg; ++g) seg[g + 1] += seg[g];
  std::vector<int32_t> pos(seg, seg + nseg);
  for (int ch = 0; ch < nchunk; ++ch)
    for (int64_t j = (N * ch) / nchunk, j1 = (N * (ch + 1)) / nchunk; j < j1; ++j)
      if (labels[j] >= 0) cols[pos[(size_t)((int64_t)ch * K + labels[j])]++] = (int32_t)j;
  const int64_t words = nseg + 1 + seg[nseg];
  CK(c->b_i32.reserve((size_t)words * sizeof(int32_t)));
  CK(cudaMemcpyAsync(c->b_i32.p, plan.data(), (size_t)words * sizeof(int32_t), cudaMemcpyHostToDevice, c->stream));
  const int64_t width = (int64_t)K * 2 * S;
  CK(c->b_rowa.reserve((size_t)(nseg * 2 * S) * sizeof(double)));
  CK(c->b_rowb.reserve((size_t)width * sizeof(double)));
  CK(cudaEventRecord(c->ev[4], c->stream));
  const int32_t* dseg = c->b_i32.as<int32_t>();
  CK(launch_group_stats(dx, S, S, K, dseg + nseg + 1, dseg, nchunk, c->b_rowa.as<double>(), c->b_rowb.as<double>(),
                        c->stream, fix, med, cc, alpha, beta));
  c->launches += 2;
  CK(cudaEventRecord(c->ev[5], c->stream));
  const SmallRead it[1] = {{out, c->b_rowb.p, width}};
  int rc = read_small(c, it, 1);  // synchronises the stream: `plan` may go
  if (rc) return rc;
  float ms = 0.f;
  cudaEventElapsedTime(&ms, c->ev[4], c->ev[5]);
  c->ms[2] = ms;
  return PLAIDGPU_OK;
}

// ---- per-set products with a design (plaid.lm) -------------------------------------------------
// B: host double, column-major N x Q with leading dimension ldb >= N; 1 <= Q <= 64, every entry finite
int check_design(plaidgpu_ctx* c, const double* B, int64_t N, int64_t ldb, int Q) {
  if (Q < 1 || Q > DESIGN_Q_MAX)
    return fail(c, PLAIDGPU_ERR_ARG, "the design has Q = " + std::to_string(Q) + " columns, outside [1, " +
                                         std::to_string(DESIGN_Q_MAX) + "]");
  if (N > 0 && !B) return fail(c, PLAIDGPU_ERR_ARG, "null argument");
  for (int q = 0; q < Q; ++q)
    for (int64_t j = 0; j < N; ++j)
      if (!std::isfinite(B[j + q * ldb]))
        return fail(c, PLAIDGPU_ERR_ARG, "design entry (" + std::to_string(j) + ", " + std::to_string(q) +
                                             ") is not finite");
  return PLAIDGPU_OK;
}

// {x B, row sums, row sums of squares} of the S x N device matrix dx (ld = S) into host out[(Q + 2) * S] (checked B,
// host, ld = ldb).  Only the N rows of B this call needs go to the device.  The columns are split into chunks like
// group_stats_device, added in column order within a chunk and the chunks in chunk order.  Kernel time in ms[2].
// fix / med / cc / alpha / beta: the fix-up of plaidgpu_score_finish, applied in registers to raw scores.
int design_stats_device(plaidgpu_ctx* c, const double* dx, int32_t S, int64_t N, const double* B, int64_t ldb, int Q,
                        double* out, bool fix = false, const double* med = nullptr, double cc = 0.0,
                        double alpha = 1.0, const double* beta = nullptr) {
  const int64_t width = (int64_t)(Q + 2) * S;
  const int nchunk = reduce_nchunk(N, width);
  CK(c->b_design.reserve((size_t)std::max<int64_t>(N * Q, 1) * sizeof(double)));
  if (N > 0)
    CK(cudaMemcpy2DAsync(c->b_design.p, (size_t)N * sizeof(double), B, (size_t)ldb * sizeof(double),
                         (size_t)N * sizeof(double), (size_t)Q, cudaMemcpyHostToDevice, c->stream));
  CK(c->b_rowa.reserve((size_t)nchunk * (size_t)width * sizeof(double)));
  CK(c->b_rowb.reserve((size_t)width * sizeof(double)));
  CK(cudaEventRecord(c->ev[4], c->stream));
  CK(launch_design_stats(dx, S, S, N, c->b_design.as<double>(), N, Q, nchunk, c->b_rowa.as<double>(),
                         c->b_rowb.as<double>(), c->stream, fix, med, cc, alpha, beta));
  c->launches += 2;
  CK(cudaEventRecord(c->ev[5], c->stream));
  const SmallRead it[1] = {{out, c->b_rowb.p, width}};
  int rc = read_small(c, it, 1);  // synchronises the stream: B may go
  if (rc) return rc;
  float ms = 0.f;
  cudaEventElapsedTime(&ms, c->ev[4], c->ev[5]);
  c->ms[2] = ms;
  return PLAIDGPU_OK;
}

// ---- per-column top k (plaid.topsets) -------------------------------------------------------
int check_topk(plaidgpu_ctx* c, int32_t S, int k) {
  if (k < 1 || k > TOPK_MAX || k > S)
    return fail(c, PLAIDGPU_ERR_ARG, "k = " + std::to_string(k) + " is outside [1, min(S = " + std::to_string(S) +
                                         ", " + std::to_string(TOPK_MAX) + ")]");
  return PLAIDGPU_OK;
}

// Each column's top k of the S x N device matrix dx (ld = S) into host idx / val[k * N] (checked k).  Kernel time in
// ms[2].  fix / med / cc / alpha / beta: the fix-up of plaidgpu_score_finish, applied in registers to raw scores.
int topk_device(plaidgpu_ctx* c, const double* dx, int32_t S, int64_t N, int k, int decreasing, int32_t* idx,
                double* val, bool fix = false, const double* med = nullptr, double cc = 0.0, double alpha = 1.0,
                const double* beta = nullptr) {
  const size_t n = (size_t)k * (size_t)N;
  CK(c->b_i32.reserve(std::max<size_t>(n, 1) * sizeof(int32_t)));
  CK(c->b_rowb.reserve(std::max<size_t>(n, 1) * sizeof(double)));
  CK(cudaEventRecord(c->ev[4], c->stream));
  CK(launch_col_topk(dx, S, S, N, k, decreasing, c->b_i32.as<int32_t>(), c->b_rowb.as<double>(), c->stream, fix, med,
                     cc, alpha, beta));
  c->launches += 1;
  CK(cudaEventRecord(c->ev[5], c->stream));
  if (n) {
    CK(cudaMemcpyAsync(idx, c->b_i32.p, n * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(val, c->b_rowb.p, n * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  }
  CK(cudaStreamSynchronize(c->stream));
  float ms = 0.f;
  cudaEventElapsedTime(&ms, c->ev[4], c->ev[5]);
  c->ms[2] = ms;
  return PLAIDGPU_OK;
}

// ---- per-row top k (plaid.topcells) ---------------------------------------------------------
// k over the N columns of the whole call
int check_row_topk(plaidgpu_ctx* c, int64_t N, int k) {
  if (k < 1 || k > TOPK_MAX || k > N)
    return fail(c, PLAIDGPU_ERR_ARG, "k = " + std::to_string(k) + " is outside [1, min(N = " + std::to_string(N) +
                                         ", " + std::to_string(TOPK_MAX) + ")]");
  return PLAIDGPU_OK;
}

// Each row's top k of the S x N device matrix dx (ld = S) into host idx / val[k * S], idx = col0 + column (checked
// k; when N < k the last entries are empty: idx -1, val NaN).  The column chunks follow reduce_nchunk with the
// partial lists (16 bytes an entry) as the width.  Kernel time in ms[2].  fix / med / cc / alpha / beta: the fix-up
// of plaidgpu_score_finish, applied in registers to raw scores.
int row_topk_device(plaidgpu_ctx* c, const double* dx, int32_t S, int64_t N, int k, int decreasing, int64_t col0,
                    int64_t* idx, double* val, bool fix = false, const double* med = nullptr, double cc = 0.0,
                    double alpha = 1.0, const double* beta = nullptr) {
  const size_t n = (size_t)k * (size_t)S;
  const int nchunk = reduce_nchunk(N, 2 * (int64_t)n);
  CK(c->b_rowa.reserve(2 * (size_t)nchunk * n * sizeof(uint64_t)));
  CK(c->b_rowb.reserve(n * (sizeof(int64_t) + sizeof(double))));
  int64_t* didx = c->b_rowb.as<int64_t>();
  double* dval = reinterpret_cast<double*>(didx + n);
  CK(cudaEventRecord(c->ev[4], c->stream));
  CK(launch_row_topk(dx, S, S, N, k, decreasing, nchunk, c->b_rowa.as<uint64_t>(), col0, didx, dval, c->stream, fix,
                     med, cc, alpha, beta));
  c->launches += 2;
  CK(cudaEventRecord(c->ev[5], c->stream));
  CK(cudaMemcpyAsync(idx, didx, n * sizeof(int64_t), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaMemcpyAsync(val, dval, n * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  float ms = 0.f;
  cudaEventElapsedTime(&ms, c->ev[4], c->ev[5]);
  c->ms[2] = ms;
  return PLAIDGPU_OK;
}

// The order of the device's selection key (topk_select.cuh) on final values: larger first (smaller when
// !decreasing), -0 == +0, NaN after every number, equal values by ascending column.  An empty entry (column -1,
// value NaN) compares as the largest column, after every NaN.
uint64_t host_order_key(double v, bool decreasing) {
  if (v != v) return 0;
  uint64_t b = 0;
  if (v != 0.0) memcpy(&b, &v, sizeof(b));
  b = (b >> 63) ? ~b : (b | 0x8000000000000000ull);
  return decreasing ? b : ~b;
}

// Merges the row top-k lists b into a (k * S each, sorted, with distinct columns): a becomes each row's k best of
// both.  The order is total, so merging tiles or shards in any grouping gives the same lists.
void merge_row_topk(int32_t S, int k, bool decreasing, int64_t* ai, double* av, const int64_t* bi, const double* bv) {
  std::vector<int64_t> ti((size_t)k);
  std::vector<double> tv((size_t)k);
  for (int32_t s = 0; s < S; ++s) {
    int64_t* ri = ai + (size_t)k * s;
    double* rv = av + (size_t)k * s;
    const int64_t* qi = bi + (size_t)k * s;
    const double* qv = bv + (size_t)k * s;
    int x = 0, y = 0;
    for (int t = 0; t < k; ++t) {
      const uint64_t kx = host_order_key(rv[x], decreasing), ky = host_order_key(qv[y], decreasing);
      const bool take_b = ky > kx || (ky == kx && (uint64_t)qi[y] < (uint64_t)ri[x]);
      ti[t] = take_b ? qi[y] : ri[x];
      tv[t] = take_b ? qv[y] : rv[x];
      take_b ? ++y : ++x;
    }
    std::copy(ti.begin(), ti.end(), ri);
    std::copy(tv.begin(), tv.end(), rv);
  }
}

// Host X and host output larger than the device can hold: the column tile width score_chunked should use, or 0
// when one pass fits (the raw scores get 45 % of the free memory; X, ranks and slack share the rest)
int host_chunk_cols(plaidgpu_ctx* c, const plaidgpu_matrix* X, int64_t* chunk) {
  *chunk = 0;
  if (!c->have_g || X->location != PLAIDGPU_HOST || X->N <= 1) return PLAIDGPU_OK;
  CK(cudaSetDevice(c->device));
  size_t free_b = 0, total_b = 0;
  CK(cudaMemGetInfo(&free_b, &total_b));
  double budget = 0.45 * (double)free_b + (double)c->b_raw.cap;
  if (const char* e = getenv("PLAIDGPU_MAX_OUT_BYTES")) budget = atof(e);  // test knob
  if ((double)c->S * (double)X->N * 8.0 <= budget) return PLAIDGPU_OK;
  int64_t ch = (int64_t)(budget / ((double)c->S * 8.0));
  if (ch < 1) ch = 1;
  if (ch > 32) ch = (ch / 32) * 32;
  *chunk = ch;
  return PLAIDGPU_OK;
}

// columns [j0, j1) of the host matrix X; a CSC slice's rebased column pointers live in pbuf
plaidgpu_matrix column_slice(const plaidgpu_matrix* X, int64_t j0, int64_t j1, std::vector<int32_t>& pbuf) {
  plaidgpu_matrix M = *X;
  M.N = j1 - j0;
  if (X->kind == PLAIDGPU_CSC) {
    const int32_t base = X->p[j0];
    pbuf.resize((size_t)(j1 - j0 + 1));
    for (int64_t j = j0; j <= j1; ++j) pbuf[(size_t)(j - j0)] = X->p[j] - base;
    M.p = pbuf.data();
    M.i = X->i + base;
    M.x = X->x + base;
  } else {
    M.x = X->x + j0 * (int64_t)X->P;
  }
  return M;
}

// A column tile's or a shard's share of a result the whole call reduces: its group or design moments, or each row's
// top-k list.  Target::from sizes it and Target::combine folds it into the call's result.
struct Partial {
  std::vector<double> moments;
  std::vector<int64_t> cols;
  std::vector<double> val;
};

// What the finish step of a scoring call makes of the raw S x N scores.  Every kind but SCORES keeps the raw scores
// in the library's device buffer (out_location = PLAIDGPU_HOST) and applies the fix-up in registers.
struct Target {
  enum Kind { SCORES, GROUP_STATS, DESIGN_STATS, TOPK, ROW_TOPK, FILE_TILES } kind = SCORES;
  double* out = nullptr;            // SCORES: the S x N scores at opts.out_location; GROUP_STATS: K * 2 * S moments;
                                    // DESIGN_STATS: (Q + 2) * S moments
  const int32_t* labels = nullptr;  // GROUP_STATS: int32[N] in [-1, K)
  int K = 0;
  const double* B = nullptr;        // DESIGN_STATS: host, column-major N x Q, leading dimension ldb
  int64_t ldb = 0;
  int Q = 0;
  int k = 0, decreasing = 0;        // TOPK: idx / val hold k * N entries; ROW_TOPK: cols / val hold k * S entries
  int32_t* idx = nullptr;
  int64_t* cols = nullptr;          // ROW_TOPK: columns of the call; this target's column 0 is column col0
  int64_t col0 = 0;
  double* val = nullptr;
  FILE* file = nullptr;             // FILE_TILES (score_chunked): tile t is staged in stage[t & 1] (stage[0] when
  double* stage[2] = {};            // stage[1] is null) and written to `file` by a helper thread

  static Target scores(double* out) { Target t; t.out = out; return t; }
  static Target group_stats(const int32_t* labels, int K, double* out) {
    Target t; t.kind = GROUP_STATS; t.labels = labels; t.K = K; t.out = out; return t;
  }
  static Target design_stats(const double* B, int64_t ldb, int Q, double* out) {
    Target t; t.kind = DESIGN_STATS; t.B = B; t.ldb = ldb; t.Q = Q; t.out = out; return t;
  }
  static Target topk(int k, int decreasing, int32_t* idx, double* val) {
    Target t; t.kind = TOPK; t.k = k; t.decreasing = decreasing != 0; t.idx = idx; t.val = val; return t;
  }
  static Target row_topk(int k, int decreasing, int64_t* cols, double* val) {
    Target t; t.kind = ROW_TOPK; t.k = k; t.decreasing = decreasing != 0; t.cols = cols; t.val = val; return t;
  }
  static Target to_file(FILE* file, double* stage0, double* stage1) {
    Target t; t.kind = FILE_TILES; t.file = file; t.stage[0] = stage0; t.stage[1] = stage1; return t;
  }
  // the result before any tile or shard is combined into it: zero moments, empty row lists
  void clear(int32_t S) const {
    if (kind == GROUP_STATS) std::fill(out, out + (size_t)K * 2 * (size_t)S, 0.0);
    if (kind == DESIGN_STATS) std::fill(out, out + (size_t)(Q + 2) * (size_t)S, 0.0);
    if (kind == ROW_TOPK) {
      std::fill(cols, cols + (size_t)k * (size_t)S, (int64_t)-1);
      std::fill(val, val + (size_t)k * (size_t)S, NAN);
    }
  }
  // the same target for the columns from j0 on: their columns of the scores or of idx / val; the group or design
  // moments or row lists of a reduced kind go to p, for combine
  Target from(int64_t j0, int32_t S, Partial& p) const {
    Target t = *this;
    if (kind == SCORES) t.out = out + j0 * (int64_t)S;
    if (kind == GROUP_STATS) {
      p.moments.resize((size_t)K * 2 * (size_t)S);
      t.labels = labels + j0;
      t.out = p.moments.data();
    }
    if (kind == DESIGN_STATS) {
      p.moments.resize((size_t)(Q + 2) * (size_t)S);
      t.B = B + j0;  // rows j0.. of B, same leading dimension
      t.out = p.moments.data();
    }
    if (kind == TOPK) {
      t.idx = idx + j0 * k;
      t.val = val + j0 * k;
    }
    if (kind == ROW_TOPK) {
      p.cols.resize((size_t)k * (size_t)S);
      p.val.resize((size_t)k * (size_t)S);
      t.cols = p.cols.data();
      t.val = p.val.data();
      t.col0 = col0 + j0;
    }
    return t;
  }
  // folds the partial result of a tile or shard into the call's result: moments are added (in the order of the
  // calls), row lists merged by the selection order
  void combine(const Partial& p, int32_t S) const {
    for (size_t i = 0; i < p.moments.size(); ++i) out[i] += p.moments[i];
    if (kind == ROW_TOPK) merge_row_topk(S, k, decreasing != 0, cols, val, p.cols.data(), p.val.data());
  }
};

}  // namespace

// =========================================================================================
extern "C" {

int plaidgpu_version(void) { return PLAIDGPU_VERSION; }

void plaidgpu_default_opts(plaidgpu_opts* o) {
  if (!o) return;
  memset(o, 0, sizeof(*o));
  o->scorer = PLAIDGPU_PLAID;
  o->stats_mean = 1;
  o->normalize = 1;
  o->ignore_zero = -1;
  o->remove_log2 = -1;
  o->score_mean = 0;
  o->out_location = PLAIDGPU_HOST;
  o->tile_sets = 0;
  o->alpha = 0.0;
  o->rmax = 1500.0;
  o->auc_max_rank = 0.0;
  o->tau = 0.0;
  o->nrow_x = 0;
  o->matg_full_colsums = nullptr;
}

int plaidgpu_init(int device, plaidgpu_ctx** out) try {
  if (!out) return PLAIDGPU_ERR_ARG;
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n <= 0 || device < 0 || device >= n) return PLAIDGPU_ERR_CUDA;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return PLAIDGPU_ERR_CUDA;
  if (prop.major < 10) return PLAIDGPU_ERR_CUDA;  // sm_100a code only
  plaidgpu_ctx* c = new (std::nothrow) plaidgpu_ctx();
  if (!c) return PLAIDGPU_ERR_NOMEM;
  c->device = device;
  if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&c->h2d_stream, cudaStreamNonBlocking) != cudaSuccess) {
    delete c;
    return PLAIDGPU_ERR_CUDA;
  }
  for (auto& ev : c->ev) cudaEventCreate(&ev);
  for (auto& ev : c->ev_chunk) cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
  cudaEventCreateWithFlags(&c->ev_early, cudaEventDisableTiming);
  for (auto& ev : c->ev_ship) cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
  for (auto& ev : c->ev_h2d) cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
  for (auto& ev : c->ev_d2h) cudaEventCreate(&ev);
  *out = c;
  return PLAIDGPU_OK;
} catch (const std::bad_alloc&) {
  return PLAIDGPU_ERR_NOMEM;
} catch (...) {
  return PLAIDGPU_ERR_ARG;
}

void plaidgpu_destroy(plaidgpu_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  cudaStreamSynchronize(c->copy_stream);
  DevBuf* bufs[] = {&c->d_ptr, &c->d_idx, &c->d_inv_mean, &c->d_inv_one, &c->d_ns, &c->d_custom_inv, &c->d_beta,
                    &c->d_dmap, &c->d_dptr, &c->d_didx, &c->d_colscale, &c->d_abits, &c->b_tcB, &c->b_colinv, &c->b_tcflag, &c->d_tmap, &c->d_tptr, &c->d_tidx, &c->d_sorder, &c->b_colfb, &c->b_tcnt, &c->b_trowptr, &c->b_ttotal, &c->b_tent, &c->b_ttmp, &c->b_tcounter, &c->b_xp, &c->b_xi, &c->b_xx, &c->b_rank, &c->b_r0, &c->b_colmax, &c->b_raw,
                    &c->b_med_all, &c->b_med_nz, &c->b_colmin, &c->b_scal, &c->b_i32, &c->b_dense, &c->b_rowa, &c->b_rowb, &c->b_fail, &c->b_list, &c->b_ci, &c->b_cx, &c->b_ce};
  for (DevBuf* b : bufs) b->release();
  for (auto& ev : c->ev) if (ev) cudaEventDestroy(ev);
  for (auto& ev : c->ev_chunk) if (ev) cudaEventDestroy(ev);
  for (auto& ev : c->ev_ring) if (ev) cudaEventDestroy(ev);
  ship_join(c);
  if (c->ev_early) cudaEventDestroy(c->ev_early);
  for (auto& ev : c->ev_ship) if (ev) cudaEventDestroy(ev);
  if (c->mbox) cudaFreeHost(c->mbox);
  for (auto& ev : c->ev_h2d) if (ev) cudaEventDestroy(ev);
  if (c->h2d_stream) cudaStreamDestroy(c->h2d_stream);
  for (auto& ev : c->ev_d2h) if (ev) cudaEventDestroy(ev);
  for (auto& r : c->ring) if (r) cudaFreeHost(r);
  delete c->pool;
  cudaStreamDestroy(c->stream);
  cudaStreamDestroy(c->copy_stream);
  delete c;
}

const char* plaidgpu_last_error(const plaidgpu_ctx* c) { return c ? c->err.c_str() : "null context"; }
int64_t plaidgpu_launch_count(const plaidgpu_ctx* c) { return c ? c->launches : 0; }
void plaidgpu_reset_launch_count(plaidgpu_ctx* c) { if (c) c->launches = 0; }
double plaidgpu_last_kernel_ms(const plaidgpu_ctx* c, int which) {
  return (c && which >= 0 && which < 4) ? c->ms[which] : -1.0;
}
void* plaidgpu_stream(const plaidgpu_ctx* c) { return c ? (void*)c->stream : nullptr; }

int plaidgpu_plan_info(const plaidgpu_ctx* c, int32_t* tile_sets, int32_t* n_tiles, int64_t* nnz_mapped,
                       int32_t* warps_per_cta, int32_t* ctas, int32_t* gather_block, int32_t* gather_blocks) try {
  if (!c || !c->plan_ok) return PLAIDGPU_ERR_STATE;
  if (tile_sets) *tile_sets = c->Ts;
  if (n_tiles) *n_tiles = c->T;
  if (nnz_mapped) *nnz_mapped = c->nnz_mapped;
  if (warps_per_cta) *warps_per_cta = c->cfg.warps;
  if (ctas) *ctas = c->cfg.ctas;
  if (gather_block) *gather_block = c->gK;
  if (gather_blocks) *gather_blocks = c->gblocks;
  return PLAIDGPU_OK;
} catch (const std::bad_alloc&) {
  return PLAIDGPU_ERR_NOMEM;
} catch (...) {
  return PLAIDGPU_ERR_ARG;
}

int plaidgpu_tc_info(const plaidgpu_ctx* c, int32_t* block_rows, int32_t* padded_rows, int32_t* slices) try {
  if (!c || !c->plan_ok) return PLAIDGPU_ERR_STATE;
  if (block_rows) *block_rows = c->tcK > 0 ? c->tc_rows : 0;
  if (padded_rows) *padded_rows = c->tcK;
  if (slices) *slices = c->tc_slices;
  return PLAIDGPU_OK;
} catch (const std::bad_alloc&) {
  return PLAIDGPU_ERR_NOMEM;
} catch (...) {
  return PLAIDGPU_ERR_ARG;
}

int plaidgpu_tail_info(const plaidgpu_ctx* c, int32_t* tail_rows, int32_t* tile_cells) try {
  if (!c || !c->plan_ok) return PLAIDGPU_ERR_STATE;
  if (tail_rows) *tail_rows = c->tail_on ? c->Pt : 0;
  if (tile_cells) *tile_cells = tail_tile_cells();
  return PLAIDGPU_OK;
} catch (const std::bad_alloc&) {
  return PLAIDGPU_ERR_NOMEM;
} catch (...) {
  return PLAIDGPU_ERR_ARG;
}

int plaidgpu_set_genesets(plaidgpu_ctx* c, int32_t P_G, int32_t S, const int32_t* Gp, const int32_t* Gi,
                          const double* Gx) try {
  if (!c) return PLAIDGPU_ERR_ARG;
  if (P_G <= 0 || S <= 0 || !Gp || (!Gi && Gp[S] > 0)) return fail(c, PLAIDGPU_ERR_ARG, "bad gene-set matrix");
  // the same pattern again (an R caller re-registers matG on every call): keep the plan
  if (c->have_g && !Gx && c->PG == P_G && c->S == S && Gp[0] == 0 && (size_t)Gp[S] == c->Gi.size() &&
      memcmp(c->Gp.data(), Gp, sizeof(int32_t) * ((size_t)S + 1)) == 0 &&
      (c->Gi.empty() || memcmp(c->Gi.data(), Gi, sizeof(int32_t) * c->Gi.size()) == 0))
    return PLAIDGPU_OK;
  c->have_g = false;
  c->plan_ok = false;
  c->PG = P_G;
  c->S = S;
  c->Gp.assign((size_t)S + 1, 0);
  c->Gi.clear();
  c->Gi.reserve((size_t)Gp[S]);
  c->g_colsums.assign((size_t)S, 0.0);
  for (int32_t s = 0; s < S; ++s) {
    if (Gp[s + 1] < Gp[s]) return fail(c, PLAIDGPU_ERR_ARG, "gene-set column pointers not monotone");
    for (int32_t q = Gp[s]; q < Gp[s + 1]; ++q) {
      if (Gx && !(Gx[q] != 0.0)) continue;  // 1 * (matG != 0): explicit zeros drop out (R/plaid.R:73)
      if (Gi[q] < 0 || Gi[q] >= P_G) return fail(c, PLAIDGPU_ERR_ARG, "gene-set row index out of range");
      c->Gi.push_back(Gi[q]);
      c->g_colsums[s] += 1.0;
    }
    c->Gp[s + 1] = (int32_t)c->Gi.size();
  }
  c->have_g = true;
  return PLAIDGPU_OK;
} catch (const std::bad_alloc&) {
  return PLAIDGPU_ERR_NOMEM;
} catch (...) {
  return PLAIDGPU_ERR_ARG;
}

// -----------------------------------------------------------------------------------------
int plaidgpu_score_begin(plaidgpu_ctx* c, const plaidgpu_matrix* X, const int32_t* rowmap,
                         const plaidgpu_opts* opts, plaidgpu_scalars* local) try {
  if (!c) return PLAIDGPU_ERR_ARG;
  if (!X || !rowmap || !opts || !local) return fail(c, PLAIDGPU_ERR_ARG, "null argument");
  if (!c->have_g) return fail(c, PLAIDGPU_ERR_STATE, "plaidgpu_set_genesets has not been called");
  trace("begin");
  CK(cudaSetDevice(c->device));
  if (c->early_cols > 0) {  // the last call was computed but not finished (a shard or tile scored again in fp64 after
    // another fell back): its early copies may still be reading the raw scores this call is about to overwrite
    int rcd = drop_early(c);
    if (rcd) return rcd;
  }
  c->in_call = false;
  c->computed = false;
  c->opts = *opts;
  if (opts->scorer < PLAIDGPU_PLAID || opts->scorer > PLAIDGPU_GSVA) return fail(c, PLAIDGPU_ERR_ARG, "unknown scorer");
  if (opts->scorer == PLAIDGPU_SSGSEA && !(1.0 + opts->alpha > 0.0)) return fail(c, PLAIDGPU_ERR_ARG, "ssgsea needs alpha > -1");
  // gsva scores a dense z-matrix whatever the storage of X
  int rc = build_plan(c, X->P, rowmap, opts->tile_sets, X->kind == PLAIDGPU_DENSE || opts->scorer == PLAIDGPU_GSVA);
  if (rc) return rc;
  rc = load_matrix(c, X, opts->scorer == PLAIDGPU_PLAID);  // plaid(): the upload runs under the scoring of earlier chunks
  if (rc) return rc;

  if (opts->scorer != PLAIDGPU_PLAID) {  // ranks / column sums / row moments read all of X in this call
    rc = h2d_wait(c, -1);
    if (rc) return rc;
  }
  c->t_begin = trace_now();
  memset(local, 0, sizeof(*local));
  local->x_min = INFINITY;
  local->x_max = -INFINITY;
  local->score_min = INFINITY;
  local->ignore_zero = -1;
  c->score_vals = c->xx;
  c->score_r0 = nullptr;

  if (opts->scorer == PLAIDGPU_SCSE && opts->remove_log2 < 0) {  // R/plaid.R:160-161
    double mn, mx;
    rc = device_minmax(c, c->xx, c->nnz, &mn, &mx);
    if (rc) return rc;
    if (!c->dense && c->nnz < (int64_t)c->P * c->N) {  // implicit zeros take part in min / max
      mn = fmin(mn, 0.0);
      mx = fmax(mx, 0.0);
    }
    local->x_min = mn;
    local->x_max = mx;
  }

  if (opts->scorer == PLAIDGPU_GSVA) {
    // zX <- (X - rowMeans(X)) / (1e-8 + rowSds(X)); rX <- sign(zX) * colRanks(|zX|)   (R/plaid.R:343,351)
    rc = make_dense(c);
    if (rc) return rc;
    CK(c->b_rank.reserve(std::max<int64_t>(c->nnz, 1) * sizeof(double)));
    CK(c->b_colmax.reserve(std::max<int64_t>(c->N, 1) * sizeof(double)));
    std::vector<double> mean((size_t)c->P), sd((size_t)c->P);
    if (opts->gsva_ecdf == PLAIDGPU_ROWTF_DONE) {
      // the caller applied the row transform across all shards (plaidgpu_row_ecdf after the
      // column -> row exchange, or its own z): rank the columns of X as they are
      CK(cudaEventRecord(c->ev[6], c->stream));
      CK(cudaMemcpyAsync(c->b_rank.p, c->xx, (size_t)c->nnz * sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
    } else if (opts->gsva_ecdf) {
      // zX[g, j] = ecdf(X[g, ])(X[g, j]) = #{samples with X[g, .] <= X[g, j]} / N = max-rank across the
      // samples / N: transpose, rank every gene's row as a column (ties = max), transpose back  (R/plaid.R:346)
      const int64_t total = (int64_t)c->P * c->N;
      CK(c->b_raw.reserve((size_t)std::max<int64_t>(total, 1) * sizeof(double)));
      CK(cudaEventRecord(c->ev[6], c->stream));
      CK(launch_transpose(c->xx, c->P, c->N, 1.0, c->b_raw.as<double>(), c->stream));  // N x P
      if (c->N > 0x7fffffff) return fail(c, PLAIDGPU_ERR_ARG, "too many samples for rowtf = ecdf");
      CK(launch_rank_dense(c->b_raw.as<double>(), (int32_t)c->N, c->P, PLAIDGPU_TIES_MAX, 0, c->b_raw.as<double>(),
                           nullptr, c->stream));
      CK(launch_transpose(c->b_raw.as<double>(), c->N, c->P, 1.0 / (double)c->N, c->b_rank.as<double>(), c->stream));
      c->launches += 3;
    } else if (opts->row_mean && opts->row_sd) {
      memcpy(mean.data(), opts->row_mean, (size_t)c->P * sizeof(double));
      memcpy(sd.data(), opts->row_sd, (size_t)c->P * sizeof(double));
    } else {  // single shard: both passes locally
      rc = row_moments(c, nullptr, mean.data());
      if (rc) return rc;
      for (int32_t r = 0; r < c->P; ++r) mean[r] /= (double)c->N;
      rc = row_moments(c, mean.data(), sd.data());
      if (rc) return rc;
      for (int32_t r = 0; r < c->P; ++r) sd[r] = c->N > 1 ? sqrt(sd[r] / (double)(c->N - 1)) : NAN;
    }
    if (opts->gsva_ecdf == PLAIDGPU_ROWTF_Z) {
      CK(c->b_rowa.reserve((size_t)c->P * sizeof(double)));
      CK(c->b_rowb.reserve((size_t)c->P * sizeof(double)));
      CK(cudaMemcpyAsync(c->b_rowa.p, mean.data(), (size_t)c->P * sizeof(double), cudaMemcpyHostToDevice, c->stream));
      CK(cudaMemcpyAsync(c->b_rowb.p, sd.data(), (size_t)c->P * sizeof(double), cudaMemcpyHostToDevice, c->stream));
      CK(cudaEventRecord(c->ev[6], c->stream));
      CK(launch_ztransform(c->xx, c->P, c->N, c->b_rowa.as<double>(), c->b_rowb.as<double>(), c->b_rank.as<double>(), c->stream));
    }
    CK(cudaStreamSynchronize(c->stream));  // mean / sd host vectors die with this scope
    // signed average ranks of the dense z columns, in place (each position is read, then written, by one thread)
    CK(launch_rank_dense(c->b_rank.as<double>(), c->P, c->N, PLAIDGPU_TIES_AVERAGE, 1, c->b_rank.as<double>(),
                         c->b_colmax.as<double>(), c->stream));
    c->launches += 2;
    CK(cudaEventRecord(c->ev[7], c->stream));
    double mn, mx;
    rc = device_minmax(c, c->b_colmax.as<double>(), c->N, &mn, &mx);
    if (rc) return rc;
    float ms = 0.f;
    cudaEventElapsedTime(&ms, c->ev[6], c->ev[7]);
    c->ms[3] = ms;
    local->rank_max = mx;  // max(abs(rX))   (R/plaid.R:352)
    c->score_vals = c->b_rank.as<double>();
  }

  if (is_rank_scorer(opts->scorer)) {
    const int ties = (opts->scorer == PLAIDGPU_SING) ? PLAIDGPU_TIES_MIN : PLAIDGPU_TIES_AVERAGE;
    CK(cudaEventRecord(c->ev[6], c->stream));
    CK(c->b_rank.reserve(std::max<int64_t>(c->nnz, 1) * sizeof(double)));
    CK(c->b_colmax.reserve(std::max<int64_t>(c->N, 1) * sizeof(double)));
    if (c->dense) {
      // colranks() dense branch for every rank scorer (R/plaid.R:617)
      CK(launch_rank_dense(c->xx, c->P, c->N, ties, 0, c->b_rank.as<double>(), c->b_colmax.as<double>(), c->stream));
    } else {
      int32_t mcn = 0;
      rc = max_col_nnz(c, &mcn);
      if (rc) return rc;
      CK(c->b_r0.reserve(std::max<int64_t>(c->N, 1) * sizeof(double)));
      // ssgsea: sparse_colranks (keep.zero = TRUE) ranks the stored entries only (R/plaid.R:245, 601);
      // sing / ucell / aucell: dense-semantics ranks with the zero group (R/plaid.R:608)
      const int dense_sem = (opts->scorer == PLAIDGPU_SSGSEA) ? 0 : 1;
      CK(launch_rank_csc(c->xp, c->xx, c->P, c->N, ties, 0, dense_sem, c->b_rank.as<double>(),
                         c->b_r0.as<double>(), c->b_colmax.as<double>(), mcn, c->stream));
      c->score_r0 = c->b_r0.as<double>();
    }
    c->launches += 1;
    CK(cudaEventRecord(c->ev[7], c->stream));
    double mn, mx;
    rc = device_minmax(c, c->b_colmax.as<double>(), c->N, &mn, &mx);
    if (rc) return rc;
    float ms = 0.f;
    cudaEventElapsedTime(&ms, c->ev[6], c->ev[7]);
    c->ms[3] = ms;
    local->rank_max = mx;
    c->score_vals = c->b_rank.as<double>();
  }
  trace("begin done (X uploaded / ranked)");
  c->in_call = true;
  return PLAIDGPU_OK;
} catch (const std::bad_alloc&) {
  return PLAIDGPU_ERR_NOMEM;
} catch (...) {
  return PLAIDGPU_ERR_ARG;
}

int plaidgpu_score_compute(plaidgpu_ctx* c, plaidgpu_scalars* scal, double* out) try {
  if (!c) return PLAIDGPU_ERR_ARG;
  if (!scal) return fail(c, PLAIDGPU_ERR_ARG, "null argument");
  if (!c->in_call) return fail(c, PLAIDGPU_ERR_STATE, "plaidgpu_score_begin has not been called");
  CK(cudaSetDevice(c->device));
  const plaidgpu_opts& o = c->opts;

  ScoreParams p{};
  p.xp = c->xp;
  p.xi = c->xi;
  p.xx = c->score_vals;
  p.r0 = nullptr;
  p.P = c->P;
  p.N = c->N;
  p.ptr = c->d_ptr.as<uint32_t>();
  p.idx = c->d_idx.as<uint16_t>();
  p.ns = c->d_ns.as<double>();
  p.S = c->S;
  p.T = c->T;
  p.Ts = c->Ts;
  p.mode = XF_IDENT;
  p.a0 = p.a1 = 0.0;
  p.colscale = nullptr;
  p.accumulate = 0;
  p.final = 1;
  p.ld = c->S;
  int colnorm = 0;
  bool mean = true;
  c->need_norm = needs_norm(o);
  switch (o.scorer) {
    case PLAIDGPU_PLAID:
      mean = o.stats_mean != 0;
      break;
    case PLAIDGPU_SCSE: {
      const bool rl = o.remove_log2 < 0 ? (scal->x_min == 0.0 && scal->x_max < 20.0) : (o.remove_log2 != 0);
      if (rl) p.mode = c->dense ? XF_EXP2_POS : XF_EXP2;
      mean = o.score_mean != 0;
      colnorm = o.score_mean ? 2 : 1;
      break;
    }
    case PLAIDGPU_SING:
      p.mode = XF_SING;
      p.a0 = (double)(o.nrow_x > 0 ? o.nrow_x : c->P);
      break;
    case PLAIDGPU_SSGSEA:
      p.mode = XF_SSGSEA;
      p.a1 = o.alpha;
      p.a0 = (o.alpha != 0.0) ? pow(scal->rank_max, 1.0 + o.alpha) : scal->rank_max;
      break;
    case PLAIDGPU_UCELL:
      p.mode = XF_UCELL;
      p.a0 = scal->rank_max;
      p.a1 = o.rmax + 1.0;
      break;
    case PLAIDGPU_AUCELL:
      p.mode = XF_AUCELL;
      p.a0 = scal->rank_max;
      p.a1 = o.auc_max_rank > 0.0 ? o.auc_max_rank : ceil(0.05 * (double)c->P);
      break;
    case PLAIDGPU_GSVA:
      p.mode = XF_GSVA;
      p.a0 = scal->rank_max;
      p.a1 = o.tau;
      break;
    default:
      return fail(c, PLAIDGPU_ERR_ARG, "unknown scorer");
  }
  p.inv = mean ? c->d_inv_mean.as<double>() : c->d_inv_one.as<double>();
  c->need_norm_hint = c->need_norm || o.scorer == PLAIDGPU_UCELL;
  if (is_rank_scorer(o.scorer) || o.scorer == PLAIDGPU_GSVA) {
    if (c->dense) {
      // dense input: transform the dense rank matrix in place, then plain product
      CK(launch_xform_dense(c->b_rank.as<double>(), c->b_rank.as<double>(), c->nnz, p.mode, p.a0, p.a1, c->stream));
      c->launches += 1;
      p.mode = XF_IDENT;
    } else {
      p.r0 = c->score_r0;  // nullptr for ssgsea: zeros rank 0
      if (o.scorer == PLAIDGPU_SSGSEA) p.r0 = nullptr;
    }
  }

  // where the raw scores go
  const int64_t total = (int64_t)c->S * c->N;
  if (o.out_location == PLAIDGPU_DEVICE) {
    if (!out && total > 0) return fail(c, PLAIDGPU_ERR_ARG, "device output buffer required by plaidgpu_score_compute");
    c->raw = out;  // raw scores land in the caller's buffer; finish fixes them up in place
  } else {
    CK(c->b_raw.reserve((size_t)std::max<int64_t>(total, 1) * sizeof(double)));
    c->raw = c->b_raw.as<double>();
  }
  p.out = c->raw;
  // early shipping: with a pinned host destination, finished column chunks start crossing PCIe at once
  ship_join(c);
  c->ship_q.clear();
  c->early_out = nullptr;
  c->early_cols = 0;
  int64_t early_limit = 0;
  if (o.out_location == PLAIDGPU_HOST && out && total > 0 && !getenv("PLAIDGPU_NO_EARLY") && !is_pageable(out)) {
    c->early_out = out;
    double frac = 1.0;  // no normalisation: every chunk is final as soon as it is scored
    if (c->need_norm_hint) {
      // normalised scores need mean(medians) of ALL columns: only as many chunks go out raw as PCIe can move
      // while the rest is scored (rates of the previous call; a conservative guess for the first one)
      frac = (c->d2h_ms_per_col > 0.0 && c->comp_ms_per_col > 0.0) ? 1.1 * c->comp_ms_per_col / c->d2h_ms_per_col : 0.15;
      if (const char* e = getenv("PLAIDGPU_EARLY_FRAC")) frac = atof(e);
      frac = std::min(0.6, std::max(0.0, frac));
    }
    early_limit = (int64_t)(frac * (double)c->N);
  }

  if (colnorm) {  // replaid.scse: column sums / means of |X| over ALL rows of X (R/plaid.R:176,181)
    CK(c->d_colscale.reserve(std::max<int64_t>(c->N, 1) * sizeof(double)));
    CK(launch_colabs(c->xp, c->xx, c->P, c->N, p.mode, p.a0, p.a1, colnorm, c->d_colscale.as<double>(), c->stream));
    c->launches += 1;
    p.colscale = c->d_colscale.as<double>();
  }

  unsigned long long* smin = nullptr;
  if (c->need_norm) {  // the score kernels report their smallest final score (see ensure_median)
    CK(c->b_smin.reserve(sizeof(unsigned long long)));
    CK(launch_fill_u32(c->b_smin.p, 0xFFFFFFFFu, 2, c->stream));
    smin = c->b_smin.as<unsigned long long>();
  }
  p.smin = smin;
  CK(cudaEventRecord(c->ev[0], c->stream));
  // ---- the block (high-degree rows of sparse X / every row of dense X) ----------------------------
  const bool use_tc = c->tcK > 0 && !o.exact_fp64 && c->N > 0;
  const int* tc_flag = nullptr;
  bool compacted = false;
  if (!(use_tc && !c->dense)) {  // only the chunk loop below waits piece by piece
    int rcw = h2d_wait(c, -1);
    if (rcw) return rcw;
  }
  if (use_tc) {
    // tensor cores: fixed-point digit rows of the block (k_tc_prep_*), then t(G) bits x digits (k_tc_score).
    // A non-finite block entry cannot be quantised: it raises a device flag, the tensor-core kernel returns at
    // once and the fp64 gather passes below (otherwise no-ops) redo the block.
    const int sl = c->tc_slices;
    const int ct = tc_cells_per_tile(sl);
    CK(c->b_tcflag.reserve(8));
    CK(launch_fill_u32(c->b_tcflag.p, 0u, 2, c->stream));
    CK(c->b_colinv.reserve((size_t)c->N * sizeof(double)));
    // column chunks keep the digit-row operand within ~4 GiB whatever N is; with a tail pass a chunk is a whole
    // number of tail tiles and its int64 tail sums (S x chunk) stay within ~4 GB too
    const bool tail = c->tail_on && !c->dense;
    const int TC_ = tail_tile_cells();
    int64_t chunk = std::max<int64_t>(ct, ((int64_t)(4ll << 30) / ((int64_t)c->tcK * sl)) / ct * ct);
    if (tail) {
      int64_t tiles = std::max<int64_t>(1, (int64_t)(4ll << 30) / ((int64_t)c->S * TC_ * 8));
      if (const char* e = getenv("PLAIDGPU_TAIL_TILES")) tiles = std::max(1, atoi(e));
      chunk = std::max<int64_t>(TC_, std::min<int64_t>(chunk / TC_, tiles) * TC_);
      if (chunk > c->N) chunk = (c->N + TC_ - 1) / TC_ * TC_;
    } else if (chunk > c->N) {
      chunk = c->N;
    }
    CK(c->b_tcB.reserve(tc_operand_bytes(chunk, c->tcK, sl)));
    if (!c->dense && c->nnz > 0) {
      CK(c->b_ci.reserve((size_t)c->nnz * sizeof(int32_t)));
      CK(c->b_cx.reserve((size_t)c->nnz * sizeof(double)));
      CK(c->b_ce.reserve((size_t)c->N * sizeof(int32_t)));
    }
    const int64_t ctiles = tail ? chunk / TC_ : 0;
    if (tail) {
      CK(c->b_tcnt.reserve((size_t)ctiles * c->Pt * sizeof(uint32_t) + 16));
      CK(c->b_trowptr.reserve((size_t)ctiles * (c->Pt + 1) * sizeof(uint32_t)));
      CK(c->b_ttotal.reserve((size_t)ctiles * sizeof(uint32_t)));
      CK(c->b_tent.reserve((size_t)std::max<int64_t>(c->nnz, 1) * sizeof(uint2)));
      CK(c->b_ttmp.reserve((size_t)c->S * (size_t)chunk * sizeof(long long)));
      CK(c->b_tcounter.reserve(sizeof(unsigned int)));
      CK(c->b_colfb.reserve((size_t)c->N * sizeof(double)));
    }
    tc_flag = c->b_tcflag.as<int>();
    int64_t nj = 0;
    for (int64_t j0 = 0; j0 < c->N; j0 += nj) {
      nj = std::min<int64_t>(chunk, c->N - j0);
      // while chunks leave early for the host (pinned output), keep them small: PCIe starts sooner and the early
      // part is sized in finer steps; full-size chunks (fewer launches, fuller waves) afterwards
      if (tail && c->early_out && c->need_norm_hint && j0 < early_limit && !getenv("PLAIDGPU_TAIL_TILES"))
        nj = std::min<int64_t>(nj, 4 * (int64_t)TC_);
      const int tiles = tail ? (int)((nj + TC_ - 1) / TC_) : 0;
      if (c->h2d_pending) {  // this chunk's entries (and everything before them) must have landed
        int rcw = h2d_wait(c, c->xp_host ? (int64_t)c->xp_host[j0 + nj] : -1);
        if (rcw) return rcw;
      }
      if (c->dense) {
        CK(launch_tc_prep_dense(p.xx + j0 * (int64_t)c->P, c->P, nj, p.mode, p.a0, p.a1, c->tcK, sl,
                                c->b_tcB.as<signed char>(), c->b_colinv.as<double>() + j0, c->b_tcflag.as<int>(), c->stream));
      } else {
        if (tail) CK(launch_fill_u32(c->b_tcnt.p, 0u, (int64_t)tiles * c->Pt, c->stream));
        CK(launch_tc_prep_csc(c->xp + j0, c->xi, p.xx, p.r0 ? p.r0 + j0 : nullptr, c->d_dmap.as<uint16_t>(), nj, p.mode,
                              p.a0, p.a1, c->tcK, sl, c->b_tcB.as<signed char>(), c->b_colinv.as<double>() + j0,
                              c->b_ci.as<int32_t>(), c->b_cx.as<double>(), c->b_ce.as<int32_t>() + j0,
                              c->b_tcflag.as<int>(), tail ? c->d_tmap.as<int32_t>() : nullptr, c->b_tcnt.as<uint32_t>(),
                              c->Pt, TC_, tail ? c->b_colfb.as<double>() + j0 : nullptr, c->stream));
      }
      if (tail) {
        // regroup the tail entries of the chunk gene-major per cell tile, then one warp per (tile, set)
        CK(launch_tile_scan(c->b_tcnt.as<uint32_t>(), c->Pt, tiles, c->b_trowptr.as<uint32_t>(), c->b_ttotal.as<uint32_t>(), c->stream));
        CK(launch_tile_place(c->xp + j0, c->b_ce.as<int32_t>() + j0, c->b_ci.as<int32_t>(), c->b_cx.as<double>(),
                             p.r0 ? p.r0 + j0 : nullptr, c->d_tmap.as<int32_t>(), c->b_colinv.as<double>() + j0, nj, p.mode,
                             p.a0, p.a1, c->Pt, c->b_trowptr.as<uint32_t>(), c->b_ttotal.as<uint32_t>(),
                             c->b_tcnt.as<uint32_t>(), c->b_tent.as<uint2>(), tc_flag, c->stream));
        CK(launch_tail(c->d_tptr.as<uint32_t>(), c->d_tidx.as<uint16_t>(), c->d_sorder.as<int32_t>(),
                       c->b_trowptr.as<uint32_t>(), c->b_ttotal.as<uint32_t>(), c->b_tent.as<uint2>(), c->S, c->Pt, tiles, c->b_ttmp.as<long long>(),
                       c->b_tcounter.as<unsigned int>(), tc_flag, c->stream));
        c->launches += 3;
      }
      TcParams t{};
      t.abits = c->d_abits.as<uint4>();
      t.S = c->S;
      t.N = nj;
      t.colinv = c->b_colinv.as<double>() + j0;
      t.skip_if = tc_flag;
      t.final = (c->dense || tail) ? 1 : 0;
      t.mode = p.mode;
      t.a0 = p.a0;
      t.a1 = p.a1;
      t.r0 = p.r0 ? p.r0 + j0 : nullptr;
      t.inv = p.inv;
      t.ns = p.ns;
      t.colscale = p.colscale ? p.colscale + j0 : nullptr;
      t.out = c->raw + j0 * (int64_t)c->S;
      t.ld = c->S;
      t.smin = smin;
      t.tail = tail ? c->b_ttmp.as<long long>() : nullptr;
      t.tail_ld = (int64_t)tiles * TC_;
      t.colfb = (tail && p.mode >= XF_SING) ? c->b_colfb.as<double>() + j0 : nullptr;
      t.small_sums = c->P <= (1 << 20) ? 1 : 0;
      CK(launch_tc_score(t, c->b_tcB.as<signed char>(), c->tcK, sl, c->stream));
      c->launches += 2;
      if (c->early_out && t.final && j0 + nj <= early_limit) {
        const int rcs = ship_chunk(c, j0, nj);
        if (rcs == PLAIDGPU_OK) c->early_cols = j0 + nj;
        else if (rcs < 0) return rcs;
        else early_limit = 0;
      }
    }
    {  // no more early blocks: the helper drains its list and exits (joined in plaidgpu_score_finish)
      std::lock_guard<std::mutex> lk(c->ship_m);
      c->ship_done = true;
    }
    c->ship_cv.notify_all();
    compacted = !c->dense && c->nnz > 0;
    {
      int rcw = h2d_wait(c, -1);
      if (rcw) return rcw;
    }
  }
  if (c->gblocks > 0) {
    GatherParams g{};
    g.smin = smin;
    g.xp = c->xp;
    g.xi = c->xi;
    g.xx = p.xx;
    g.r0 = p.r0;
    g.P = c->P;
    g.N = c->N;
    g.K = c->gK;
    g.didx = c->d_didx.as<uint32_t>();
    g.inv = p.inv;
    g.ns = p.ns;
    g.colscale = p.colscale;
    g.S = c->S;
    g.mode = p.mode;
    g.a0 = p.a0;
    g.a1 = p.a1;
    g.out = c->raw;
    g.ld = c->S;
    g.run_if = tc_flag;  // after a tensor-core pass: only when it had to give up
    g.dmap = c->dense ? nullptr : c->d_dmap.as<uint16_t>();
    for (int32_t b = 0; b < c->gblocks; ++b) {
      g.g0 = b * c->gK;
      g.dlo = b * c->gK;
      g.dptr = c->d_dptr.as<uint32_t>() + (size_t)b * (c->S + 1);
      g.accumulate = b > 0;
      g.final = c->dense && (b == c->gblocks - 1);  // sparse X: the scatter pass finishes the scores
      CK(launch_gather(g, c->stream));
      c->launches += 1;
    }
    p.accumulate = 1;
  }
  if (!c->dense) {
    if (!compacted && c->gblocks > 0 && c->nnz > 0) {
      // the scatter pass never needs the block's entries: compact the columns once
      CK(c->b_ci.reserve((size_t)c->nnz * sizeof(int32_t)));
      CK(c->b_cx.reserve((size_t)c->nnz * sizeof(double)));
      CK(c->b_ce.reserve((size_t)std::max<int64_t>(c->N, 1) * sizeof(int32_t)));
      CK(launch_compact(c->xp, c->xi, p.xx, c->d_dmap.as<uint16_t>(), c->N, c->b_ci.as<int32_t>(), c->b_cx.as<double>(),
                        c->b_ce.as<int32_t>(), c->stream));
      c->launches += 1;
      compacted = true;
    }
    if (compacted) {
      p.xi = c->b_ci.as<int32_t>();
      p.xx = c->b_cx.as<double>();
      p.xe = c->b_ce.as<int32_t>();
    }
    p.run_if = (use_tc && c->tail_on) ? tc_flag : nullptr;  // with a tail pass the scatter pass is the fallback only
    CK(launch_score(p, false, c->cfg, c->stream));
    c->launches += 1;
  }
  CK(cudaEventRecord(c->ev[1], c->stream));
  trace("compute: score kernels enqueued");

  scal->score_min = INFINITY;
  c->have_all = c->have_nz = false;
  c->raw_valid = true;
  // did the fixed-point route give up (b_tcflag)?  Read with the score minimum when there is one, else in place of
  // the stream synchronisation below.  b_tcflag is reserved with 8 bytes: the int flag sits in the low half.
  unsigned long long flag = 0;
  if (c->need_norm) {
    // normalize_medians uses ONE of the two medians, chosen by min(x) == 0 over all shards (R/plaid.R:556-557).
    // The shard's own minimum (tracked by the score kernels) settles which: > 0 -> no zeros here, both medians
    // coincide; < 0 -> the global minimum is negative too, the plain median is used; == 0 -> the non-zero
    // median, unless another shard holds a negative score (then the plain one is computed on demand).
    unsigned long long key = ~0ull;
    {
      const SmallRead it[2] = {{&key, c->b_smin.p, 1}, {&flag, c->b_tcflag.p, use_tc ? 1 : 0}};
      int rcs = read_small(c, it, 2);
      if (rcs) return rcs;
    }
    c->local_min = (key == ~0ull) ? INFINITY : host_value_of(key);
    int which = COLSTATS_BOTH;
    if (!c->want_both && !colstats_small(c->S)) {
      if (o.ignore_zero >= 0) which = o.ignore_zero ? COLSTATS_NZ : COLSTATS_ALL;
      else which = (c->local_min == 0.0) ? COLSTATS_NZ : COLSTATS_ALL;
    }
    CK(cudaEventRecord(c->ev[2], c->stream));
    int rc = run_colstats(c, which);
    if (rc) return rc;
    CK(cudaEventRecord(c->ev[3], c->stream));
    if (which == COLSTATS_ALL && c->local_min > 0.0 && c->N) {  // no zeros: the two medians are the same numbers
      CK(launch_med_nz_from_all(c->b_med_all.as<double>(), c->b_med_nz.as<double>(), c->N, c->stream));
      c->have_nz = true;
    }
    rc = fetch_medians(c);
    if (rc) return rc;
  }
  if (use_tc && !c->need_norm) {
    const SmallRead it[1] = {{&flag, c->b_tcflag.p, 1}};
    int rcs = read_small(c, it, 1);
    if (rcs) return rcs;
  } else {
    CK(cudaStreamSynchronize(c->stream));
  }
  scal->fp64 = (int32_t)(flag & 0xFFFFFFFFull) != 0;
  if (scal->fp64) {  // the fp64 passes redid the scores AFTER chunks had left: ship everything again
    int rcd = drop_early(c);
    if (rcd) return rcd;
  }
  float ms = 0.f;
  cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]);
  c->ms[0] = ms;
  if (c->need_norm) {
    cudaEventElapsedTime(&ms, c->ev[2], c->ev[3]);
    c->ms[1] = ms;
    double mn = INFINITY;
    for (int64_t j = 0; j < c->N; ++j) mn = fmin(mn, c->h_colmin[j]);
    scal->score_min = mn;
  }
  c->t_known = trace_now();
  trace("compute done (scores + medians)");
  c->computed = true;
  return PLAIDGPU_OK;
} catch (const std::bad_alloc&) {
  return PLAIDGPU_ERR_NOMEM;
} catch (...) {
  return PLAIDGPU_ERR_ARG;
}

int plaidgpu_get_col_medians(plaidgpu_ctx* c, double* med_all, double* med_nz) try {
  if (!c) return PLAIDGPU_ERR_ARG;
  if (!c->computed || !c->need_norm) return fail(c, PLAIDGPU_ERR_STATE, "no medians: run plaidgpu_score_compute with normalisation");
  if (med_all) {
    int rc = ensure_median(c, false);
    if (rc) return rc;
    memcpy(med_all, c->h_med_all.data(), (size_t)c->N * sizeof(double));
  }
  if (med_nz) {
    int rc = ensure_median(c, true);
    if (rc) return rc;
    memcpy(med_nz, c->h_med_nz.data(), (size_t)c->N * sizeof(double));
  }
  return PLAIDGPU_OK;
} catch (const std::bad_alloc&) {
  return PLAIDGPU_ERR_NOMEM;
} catch (...) {
  return PLAIDGPU_ERR_ARG;
}

int plaidgpu_get_col_medians_for(plaidgpu_ctx* c, int ignore_zero, double* med) try {
  if (!c) return PLAIDGPU_ERR_ARG;
  if (!med && c->N > 0) return fail(c, PLAIDGPU_ERR_ARG, "null argument");
  return ignore_zero ? plaidgpu_get_col_medians(c, nullptr, med) : plaidgpu_get_col_medians(c, med, nullptr);
} catch (const std::bad_alloc&) {
  return PLAIDGPU_ERR_NOMEM;
} catch (...) {
  return PLAIDGPU_ERR_ARG;
}

int plaidgpu_combine_medians(int ignore_zero_opt, double score_min, const double* med_all, const double* med_nz,
                             int64_t N_total, plaidgpu_scalars* scal) try {
  if (!scal || !med_all || !med_nz || N_total < 0) return PLAIDGPU_ERR_ARG;
  const int iz = ignore_zero_opt < 0 ? (score_min == 0.0 ? 1 : 0) : (ignore_zero_opt != 0);  // R/plaid.R:556-557
  scal->ignore_zero = iz;
  scal->score_min = score_min;
  scal->med_mean = r_mean(iz ? med_nz : med_all, N_total);  // R/plaid.R:572
  return PLAIDGPU_OK;
} catch (const std::bad_alloc&) {
  return PLAIDGPU_ERR_NOMEM;
} catch (...) {
  return PLAIDGPU_ERR_ARG;
}

// plaidgpu_score_finish into target t (SCORES, GROUP_STATS, DESIGN_STATS, TOPK or ROW_TOPK)
static int score_finish(plaidgpu_ctx* c, const plaidgpu_scalars* scal, const Target& t) try {
  if (t.kind == Target::SCORES && !t.out && c->N > 0) return fail(c, PLAIDGPU_ERR_ARG, "null argument");
  if (!c->computed) return fail(c, PLAIDGPU_ERR_STATE, "plaidgpu_score_compute has not been called");
  CK(cudaSetDevice(c->device));
  const plaidgpu_opts& o = c->opts;
  const int32_t S = c->S;
  const int64_t N = c->N;

  double alpha = 1.0, cc = 0.0;
  const double* med = nullptr;
  const double* beta = nullptr;
  std::vector<double> hbeta;  // host copy of beta (outlives the early-column patcher below)
  bool fix = false;
  if (c->need_norm) {
    int rc = ensure_median(c, scal->ignore_zero != 0);
    if (rc) return rc;
    med = scal->ignore_zero ? c->b_med_nz.as<double>() : c->b_med_all.as<double>();
    cc = scal->med_mean;
    fix = true;
  }
  if (o.scorer == PLAIDGPU_UCELL) {  // 1 - S/rmax + (colSums(matG != 0) + 1) / (2 rmax)   (R/plaid.R:280)
    hbeta.resize((size_t)S);
    const double* gs = o.matg_full_colsums ? o.matg_full_colsums : c->g_colsums.data();
    for (int32_t s = 0; s < S; ++s) hbeta[s] = 1.0 + (gs[s] + 1.0) / (2.0 * o.rmax);
    CK(c->d_beta.reserve((size_t)S * sizeof(double)));
    CK(cudaMemcpyAsync(c->d_beta.p, hbeta.data(), (size_t)S * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    beta = c->d_beta.as<double>();
    alpha = -1.0 / o.rmax;
    fix = true;
  }

  // the reductions read the raw scores with the fix-up applied in registers: the S x N matrix stays on the device
  // and only K * 2 * S or (Q + 2) * S moments, or k * N or k * S indices and values, go back
  if (t.kind == Target::GROUP_STATS) return group_stats_device(c, c->raw, S, N, t.labels, t.K, t.out, fix, med, cc, alpha, beta);
  if (t.kind == Target::DESIGN_STATS)
    return design_stats_device(c, c->raw, S, N, t.B, t.ldb, t.Q, t.out, fix, med, cc, alpha, beta);
  if (t.kind == Target::TOPK) return topk_device(c, c->raw, S, N, t.k, t.decreasing, t.idx, t.val, fix, med, cc, alpha, beta);
  if (t.kind == Target::ROW_TOPK)
    return row_topk_device(c, c->raw, S, N, t.k, t.decreasing, t.col0, t.cols, t.val, fix, med, cc, alpha, beta);
  double* out = t.out;
  c->raw_valid = false;  // the fix-up below rewrites the raw scores in place
  CK(cudaEventRecord(c->ev[4], c->stream));
  if (o.out_location == PLAIDGPU_DEVICE) {
    if (out != c->raw) return fail(c, PLAIDGPU_ERR_ARG, "plaidgpu_score_finish: device `out` differs from the buffer given to compute");
    if (fix) {
      CK(launch_fixup(c->raw, out, S, S, 0, N, med, cc, alpha, beta, c->stream));
      c->launches += 1;
    }
    CK(cudaEventRecord(c->ev[5], c->stream));
    CK(cudaStreamSynchronize(c->stream));
  } else {
    // host output: fix up a block of columns, then stream it out while the next block is fixed
    const bool pageable = N > 0 && is_pageable(out) && !getenv("PLAIDGPU_NO_RING");
    if (pageable) {
      // A pageable destination (an R matrix) would make every cudaMemcpyAsync a staged, synchronous copy at a
      // fraction of the PCIe rate.  Blocks go through a pinned ring instead and the copy threads move block
      // k - 1 into the caller's matrix while block k crosses PCIe and block k + 1 is fixed up.
      {
        int rcr = ensure_ring(c);
        if (rcr) return rcr;
      }
      const int64_t chunk = std::max<int64_t>(1, (int64_t)(c->ring_bytes / ((size_t)S * 8)));
      const int64_t nchunks = (N + chunk - 1) / chunk;
      auto drain = [&](int64_t k) {  // block k: wait for its DMA, then pinned slot -> caller matrix
        const int64_t j0 = k * chunk, j1 = std::min<int64_t>(N, j0 + chunk);
        cudaEventSynchronize(c->ev_ring[k % plaidgpu_ctx::RING]);
        c->pool->copy(out + j0 * S, c->ring[k % plaidgpu_ctx::RING], (size_t)(j1 - j0) * S * sizeof(double));
      };
      for (int64_t k = 0; k < nchunks; ++k) {
        const int64_t j0 = k * chunk, j1 = std::min<int64_t>(N, j0 + chunk);
        if (fix) {
          CK(launch_fixup(c->raw, c->raw, S, S, j0, j1, med, cc, alpha, beta, c->stream));
          c->launches += 1;
        }
        CK(cudaEventRecord(c->ev_chunk[k & 1], c->stream));
        CK(cudaStreamWaitEvent(c->copy_stream, c->ev_chunk[k & 1], 0));
        CK(cudaMemcpyAsync(c->ring[k % plaidgpu_ctx::RING], c->raw + j0 * S, (size_t)(j1 - j0) * S * sizeof(double),
                           cudaMemcpyDeviceToHost, c->copy_stream));
        CK(cudaEventRecord(c->ev_ring[k % plaidgpu_ctx::RING], c->copy_stream));
        if (k >= 1) drain(k - 1);
      }
      CK(cudaEventRecord(c->ev[5], c->stream));
      if (nchunks > 0) drain(nchunks - 1);
      CK(cudaStreamSynchronize(c->stream));
      CK(cudaStreamSynchronize(c->copy_stream));
      float msr = 0.f;
      cudaEventElapsedTime(&msr, c->ev[4], c->ev[5]);
      c->ms[2] = msr;
      return PLAIDGPU_OK;
    }
    // columns [0, E) already left as RAW scores while the rest was being scored (plaidgpu_score_compute): a helper
    // thread fixes them up in the caller's matrix — the arithmetic of k_fixup, operation by operation — while the
    // remaining blocks are fixed up on the device and follow over PCIe
    ship_join(c);  // every early block is enqueued on the copy stream from here on
    const int64_t E = (c->early_out == out) ? std::min<int64_t>(c->early_cols, N) : 0;
    c->early_out = nullptr;
    c->early_cols = 0;
    std::thread patcher;
    struct Joiner {
      std::thread& t;
      ~Joiner() {
        if (t.joinable()) t.join();
      }
    } joiner{patcher};  // also on the error returns below
    if (E > 0 && fix) {
      if (!c->pool) {
        int nt = (int)std::min<unsigned>(8, std::max(2u, std::thread::hardware_concurrency() / 2));
        if (const char* e = getenv("PLAIDGPU_COPY_THREADS")) nt = std::max(1, std::min(64, atoi(e)));
        c->pool = new CopyPool(nt);
      }
      const double* hm = med ? (scal->ignore_zero ? c->h_med_nz.data() : c->h_med_all.data()) : nullptr;
      const double* hb = beta ? hbeta.data() : nullptr;
      cudaEvent_t evE = c->ev_early;
      CopyPool* pool = c->pool;
      const int dev = c->device;
      patcher = std::thread([=] {
        cudaSetDevice(dev);
        cudaEventSynchronize(evE);
        trace("patcher: early D2H landed");
        pool->run([=](int part, int parts) {
          const int64_t lo = E * part / parts, hi = E * (part + 1) / parts;
          for (int64_t j = lo; j < hi; ++j) host_fixup_column(out + j * (int64_t)S, S, hm ? hm[j] : 0.0, hm != nullptr, cc, alpha, hb);
        });
      });
    }
    int64_t chunk = std::max<int64_t>(1, (int64_t)(256ll << 20) / ((int64_t)S * 8));
    int k = 0;
    bool first = true;
    for (int64_t j0 = E; j0 < N; j0 += chunk, ++k) {
      const int64_t j1 = std::min<int64_t>(N, j0 + chunk);
      if (fix) {
        CK(launch_fixup(c->raw, c->raw, S, S, j0, j1, med, cc, alpha, beta, c->stream));
        c->launches += 1;
      }
      CK(cudaEventRecord(c->ev_chunk[k & 1], c->stream));
      CK(cudaStreamWaitEvent(c->copy_stream, c->ev_chunk[k & 1], 0));
      if (first) CK(cudaEventRecord(c->ev_d2h[0], c->copy_stream));
      first = false;
      CK(cudaMemcpyAsync(out + j0 * S, c->raw + j0 * S, (size_t)(j1 - j0) * S * sizeof(double),
                         cudaMemcpyDeviceToHost, c->copy_stream));
    }
    if (!first) CK(cudaEventRecord(c->ev_d2h[1], c->copy_stream));
    trace("finish: late blocks enqueued");
    CK(cudaEventRecord(c->ev[5], c->stream));
    cudaError_t e1 = cudaStreamSynchronize(c->stream);
    cudaError_t e2 = cudaStreamSynchronize(c->copy_stream);
    trace("finish: D2H done");
    if (patcher.joinable()) patcher.join();
    trace("finish: host fix-up of the early part done");
    CK(e1);
    CK(e2);
    if (!first && N - E >= 64) {  // rates for the next call's early part
      float dms = 0.f;
      if (cudaEventElapsedTime(&dms, c->ev_d2h[0], c->ev_d2h[1]) == cudaSuccess && dms > 0.f) {
        c->d2h_ms_per_col = (double)dms / (double)(N - E);
        c->comp_ms_per_col = (c->ms[0] + c->ms[1]) / (double)N;  // kernel time: the wall clock of compute also counts the early copies it overlaps
      }
    }
  }
  float ms = 0.f;
  cudaEventElapsedTime(&ms, c->ev[4], c->ev[5]);
  c->ms[2] = ms;
  return PLAIDGPU_OK;
} catch (const std::bad_alloc&) {
  return PLAIDGPU_ERR_NOMEM;
} catch (...) {
  return PLAIDGPU_ERR_ARG;
}

int plaidgpu_score_finish(plaidgpu_ctx* c, const plaidgpu_scalars* scal, double* out) try {
  if (!c) return PLAIDGPU_ERR_ARG;
  if (!scal) return fail(c, PLAIDGPU_ERR_ARG, "null argument");
  return score_finish(c, scal, Target::scores(out));
} catch (const std::bad_alloc&) {
  return PLAIDGPU_ERR_NOMEM;
} catch (...) {
  return PLAIDGPU_ERR_ARG;
}

// Column-chunked scoring for host input / host output when the S x N result does not fit the device
// (e.g. 30k sets x 1M cells = 240 GB): the same begin / compute / finish pipeline runs per chunk of
// columns (the axis chunked_crossprod splits on, R/plaid.R:110-119).  The global scalars need all
// columns, so a normalised call recomputes the scores: pass 1 keeps only the per-column medians,
// pass 2 recomputes, fixes up and streams each chunk out (recomputing costs less than moving the raw
// scores over PCIe twice).  Results are bit-identical to the un-chunked path.
// The tile of columns [j0, j1) finishes into t.from(j0): its columns of the scores or of idx / val, or its group or
// design moments or row top-k lists, which t.combine folds into the result (cleared here) in tile order.  FILE_TILES stages every finished tile in a pinned
// buffer and writes it to the file: tiled egress for results larger than host memory (scope row f4).
// One pass over the tiles; it stops with *fell_back set as soon as a tile leaves the fixed-point route.
static int score_chunked_pass(plaidgpu_ctx* c, const plaidgpu_matrix* X, const int32_t* rowmap, const plaidgpu_opts* opts,
                              const Target& t, int64_t chunk, bool* fell_back) {
  const int64_t N = X->N;
  const int32_t S = c->S;
  Partial part;  // one tile's moments or row lists
  t.clear(S);     // a pass scored again after a fallback starts over
  if (opts->scorer == PLAIDGPU_GSVA && opts->gsva_ecdf != PLAIDGPU_ROWTF_DONE &&
      (opts->gsva_ecdf || !(opts->row_mean && opts->row_sd)))
    return fail(c, PLAIDGPU_ERR_ARG, "replaid.gsva: matrix too large for one device pass (rowtf ecdf needs all samples; rowtf z needs row_mean / row_sd)");
  std::vector<int32_t> pbuf;
  plaidgpu_scalars g;
  memset(&g, 0, sizeof(g));
  g.x_min = INFINITY;
  g.x_max = -INFINITY;
  g.score_min = INFINITY;
  g.ignore_zero = -1;
  const bool need_pre = is_rank_scorer(opts->scorer) || opts->scorer == PLAIDGPU_GSVA ||
                        (opts->scorer == PLAIDGPU_SCSE && opts->remove_log2 < 0);
  plaidgpu_matrix M;
  plaidgpu_scalars loc;
  int rc;
  if (need_pre) {
    for (int64_t j0 = 0; j0 < N; j0 += chunk) {
      M = column_slice(X, j0, std::min(N, j0 + chunk), pbuf);
      rc = plaidgpu_score_begin(c, &M, rowmap, opts, &loc);
      if (rc) return rc;
      g.x_min = fmin(g.x_min, loc.x_min);
      g.x_max = fmax(g.x_max, loc.x_max);
      g.rank_max = fmax(g.rank_max, loc.rank_max);
    }
  }
  const bool norm = needs_norm(*opts);
  if (norm) {
    std::vector<double> ma((size_t)N), mz((size_t)N);
    double smin = INFINITY;
    // the raw scores of a chunk are gone when the global min(x) == 0 flag is known: keep both medians
    struct BothGuard {
      plaidgpu_ctx* c;
      ~BothGuard() { c->want_both = false; }
    } guard{c};
    c->want_both = opts->ignore_zero < 0;
    for (int64_t j0 = 0; j0 < N; j0 += chunk) {
      const int64_t j1 = std::min(N, j0 + chunk);
      M = column_slice(X, j0, j1, pbuf);
      rc = plaidgpu_score_begin(c, &M, rowmap, opts, &loc);
      if (rc) return rc;
      plaidgpu_scalars s = g;
      rc = plaidgpu_score_compute(c, &s, nullptr);
      if (rc) return rc;
      if (s.fp64) {
        *fell_back = true;
        return PLAIDGPU_OK;
      }
      memcpy(ma.data() + j0, c->h_med_all.data(), (size_t)(j1 - j0) * sizeof(double));
      memcpy(mz.data() + j0, c->h_med_nz.data(), (size_t)(j1 - j0) * sizeof(double));
      smin = fmin(smin, s.score_min);
    }
    rc = plaidgpu_combine_medians(opts->ignore_zero, smin, ma.data(), mz.data(), N, &g);
    if (rc) return fail(c, rc, "combine_medians failed");
  }
  plaidgpu_opts o2 = *opts;
  if (norm) o2.ignore_zero = g.ignore_zero;  // decided: the second pass needs only that median
  // file sink: tile k is written by a helper thread from one staging buffer while tile k + 1 is scored into the other
  std::thread writer;
  bool short_write = false;
  struct WriterJoin {
    std::thread& t;
    ~WriterJoin() {
      if (t.joinable()) t.join();
    }
  } writer_join{writer};  // also on the error returns below
  int64_t tile = 0;
  for (int64_t j0 = 0; j0 < N; j0 += chunk, ++tile) {
    const int64_t j1 = std::min(N, j0 + chunk);
    M = column_slice(X, j0, j1, pbuf);
    rc = plaidgpu_score_begin(c, &M, rowmap, &o2, &loc);
    if (rc) return rc;
    plaidgpu_scalars s = g;
    rc = plaidgpu_score_compute(c, &s, nullptr);
    if (rc) return rc;
    if (s.fp64) {
      *fell_back = true;
      return PLAIDGPU_OK;
    }
    s.ignore_zero = g.ignore_zero;
    s.med_mean = g.med_mean;
    if (t.kind != Target::FILE_TILES) {
      rc = score_finish(c, &s, t.from(j0, S, part));
      if (rc) return rc;
      t.combine(part, S);
      continue;
    }
    double* dst = (t.stage[1] && (tile & 1)) ? t.stage[1] : t.stage[0];
    if (!t.stage[1] && writer.joinable()) writer.join();  // one buffer only: it must be free again
    rc = score_finish(c, &s, Target::scores(dst));
    if (rc) return rc;
    if (writer.joinable()) writer.join();  // tile k - 1 on disk (its buffer is the one tile k + 1 will use)
    if (short_write) return fail(c, PLAIDGPU_ERR_ARG, "short write to the output file");
    const size_t cnt = (size_t)(j1 - j0) * (size_t)S;
    FILE* f = t.file;
    writer = std::thread([dst, cnt, f, &short_write] {
      if (fwrite(dst, sizeof(double), cnt, f) != cnt) short_write = true;
    });
  }
  if (writer.joinable()) writer.join();
  if (short_write) return fail(c, PLAIDGPU_ERR_ARG, "short write to the output file");
  return PLAIDGPU_OK;
}

// The tiles of one call all take the same route: when one of them falls back to the fp64 passes, the whole call is
// scored again from tile 0 with exact_fp64 (a file is rewritten from its first tile), so the result does not depend
// on the tiling.
static int score_chunked(plaidgpu_ctx* c, const plaidgpu_matrix* X, const int32_t* rowmap, const plaidgpu_opts* opts,
                         const Target& t, int64_t chunk) {
  const off_t start = t.file ? ftello(t.file) : 0;
  bool fell_back = false;
  int rc = score_chunked_pass(c, X, rowmap, opts, t, chunk, &fell_back);
  if (rc || !fell_back) return rc;
  plaidgpu_opts o = *opts;
  o.exact_fp64 = 1;
  if (t.file && fseeko(t.file, start, SEEK_SET) != 0) return fail(c, PLAIDGPU_ERR_ARG, "cannot rewind the output file");
  return score_chunked_pass(c, X, rowmap, &o, t, chunk, &fell_back);
}

int plaidgpu_score_to_file(plaidgpu_ctx* c, const plaidgpu_matrix* X, const int32_t* rowmap, const plaidgpu_opts* opts,
                           const char* path, int format) try {
  if (!c) return PLAIDGPU_ERR_ARG;
  if (!X || !opts || !path) return fail(c, PLAIDGPU_ERR_ARG, "null argument");
  if (!c->have_g) return fail(c, PLAIDGPU_ERR_STATE, "no gene sets registered");
  if (X->location != PLAIDGPU_HOST) return fail(c, PLAIDGPU_ERR_ARG, "plaidgpu_score_to_file: X must be in host memory");
  if (format != PLAIDGPU_FILE_RAW && format != PLAIDGPU_FILE_NPY) return fail(c, PLAIDGPU_ERR_ARG, "unknown file format");
  CK(cudaSetDevice(c->device));
  const int32_t S = c->S;
  const int64_t N = X->N;
  // column tile: what the device can hold next to X and the ranks, capped at 1 GiB of pinned staging
  size_t free_b = 0, total_b = 0;
  CK(cudaMemGetInfo(&free_b, &total_b));
  // (two staging buffers of half that when the result takes several tiles: tile k is written while k + 1 is scored)
  double budget = std::min(0.45 * (double)free_b + (double)c->b_raw.cap, (double)(1ull << 30));
  if ((double)S * 8.0 * (double)N > budget) budget *= 0.5;
  if (const char* e = getenv("PLAIDGPU_MAX_OUT_BYTES")) budget = atof(e);  // test knob
  int64_t chunk = (int64_t)(budget / ((double)S * 8.0));
  if (chunk < 1) chunk = 1;
  if (chunk > 32) chunk = (chunk / 32) * 32;
  if (chunk > N) chunk = std::max<int64_t>(N, 1);
  FILE* f = fopen(path, "wb");
  if (!f) return fail(c, PLAIDGPU_ERR_ARG, std::string("cannot create ") + path);
  if (format == PLAIDGPU_FILE_NPY) {  // NumPy format 1.0: magic, version, u16 header length, dict, padded to 64
    std::string dict = "{'descr': '<f8', 'fortran_order': True, 'shape': (" + std::to_string(S) + ", " + std::to_string(N) + "), }";
    const size_t unpadded = 10 + dict.size() + 1;
    dict.append((64 - unpadded % 64) % 64, ' ');
    dict.push_back('\n');
    const unsigned char head[10] = {0x93, 'N', 'U', 'M', 'P', 'Y', 1, 0, (unsigned char)(dict.size() & 0xff),
                                    (unsigned char)(dict.size() >> 8)};
    fwrite(head, 1, sizeof(head), f);
    fwrite(dict.data(), 1, dict.size(), f);
  }
  double* stage = nullptr;
  const size_t stage_elems = std::max<size_t>((size_t)chunk * (size_t)S, 1);
  const bool tiled = N > chunk;
  cudaError_t e = cudaMallocHost(&stage, stage_elems * sizeof(double) * (tiled ? 2 : 1));
  if (e != cudaSuccess) {
    fclose(f);
    return fail_cuda(c, e, "cudaMallocHost (file staging)");
  }
  plaidgpu_opts o = *opts;
  o.out_location = PLAIDGPU_HOST;
  int rc = PLAIDGPU_OK;
  if (N <= chunk) {  // one pass: nothing to recompute
    rc = plaidgpu_score(c, X, rowmap, &o, stage);
    const size_t cnt = (size_t)N * (size_t)S;
    if (!rc && cnt && fwrite(stage, sizeof(double), cnt, f) != cnt) rc = fail(c, PLAIDGPU_ERR_ARG, "short write to the output file");
  } else {
    rc = score_chunked(c, X, rowmap, &o, Target::to_file(f, stage, stage + stage_elems), chunk);
  }
  cudaFreeHost(stage);
  if (fclose(f) != 0 && !rc) rc = fail(c, PLAIDGPU_ERR_ARG, "closing the output file failed");
  return rc;
} catch (const std::bad_alloc&) {
  return PLAIDGPU_ERR_NOMEM;
} catch (...) {
  return PLAIDGPU_ERR_ARG;
}

// One device: begin -> compute -> the single shard's median combine -> finish into t.  Host X whose S x N scores
// exceed the device goes through score_chunked.
static int score_one(plaidgpu_ctx* c, const plaidgpu_matrix* X, const int32_t* rowmap, const plaidgpu_opts* opts,
                     const Target& t) {
  plaidgpu_opts o = *opts;
  if (t.kind != Target::SCORES) o.out_location = PLAIDGPU_HOST;  // raw scores in the library's device buffer
  if (o.out_location == PLAIDGPU_HOST) {  // host in / host out larger than the device can hold -> column chunks
    int64_t chunk = 0;
    int rc = host_chunk_cols(c, X, &chunk);
    if (rc) return rc;
    if (chunk > 0) return score_chunked(c, X, rowmap, &o, t, chunk);
  }
  plaidgpu_scalars s;
  int rc = plaidgpu_score_begin(c, X, rowmap, &o, &s);
  if (rc) return rc;
  rc = plaidgpu_score_compute(c, &s, t.kind == Target::SCORES ? t.out : nullptr);
  if (rc) return rc;
  if (c->need_norm) {
    // one shard holds every column: its own minimum decides, and only that median was computed
    const bool iz = o.ignore_zero < 0 ? (s.score_min == 0.0) : (o.ignore_zero != 0);
    rc = ensure_median(c, iz);
    if (rc) return rc;
    const double* m = iz ? c->h_med_nz.data() : c->h_med_all.data();
    rc = plaidgpu_combine_medians(o.ignore_zero, s.score_min, m, m, c->N, &s);
    if (rc) return fail(c, rc, "combine_medians failed");
  }
  return score_finish(c, &s, t);
}

int plaidgpu_score(plaidgpu_ctx* c, const plaidgpu_matrix* X, const int32_t* rowmap, const plaidgpu_opts* opts,
                   double* out) try {
  if (!c) return PLAIDGPU_ERR_ARG;
  if (!X || !opts) return fail(c, PLAIDGPU_ERR_ARG, "null argument");
  return score_one(c, X, rowmap, opts, Target::scores(out));
} catch (const std::bad_alloc&) {
  return PLAIDGPU_ERR_NOMEM;
} catch (...) {
  return PLAIDGPU_ERR_ARG;
}

// score -> test fused ("next" row f1 as specified): plaid() / a replaid.* scorer followed by the per-set group moments of
// plaid.test(tests = "lm") (R/plaid.R:426-431) without the S x N matrix ever leaving the device or being written in
// its normalised form.  Bit-identical to plaidgpu_score + plaidgpu_group_stats.  Host X whose S x N scores exceed
// the device goes through score_chunked (two passes when normalised) and adds the tiles' moments in tile order.
int plaidgpu_score_group_stats(plaidgpu_ctx* c, const plaidgpu_matrix* X, const int32_t* rowmap, const plaidgpu_opts* opts,
                               const int32_t* labels, int K, double* out) try {
  if (!c) return PLAIDGPU_ERR_ARG;
  if (!X || !rowmap || !opts || !out) return fail(c, PLAIDGPU_ERR_ARG, "null argument");
  int rc = check_groups(c, labels, X->N, K);
  if (rc) return rc;
  return score_one(c, X, rowmap, opts, Target::group_stats(labels, K, out));
} catch (const std::bad_alloc&) {
  return PLAIDGPU_ERR_NOMEM;
} catch (...) {
  return PLAIDGPU_ERR_ARG;
}

// score -> linear model fused: plaid() / a replaid.* scorer followed by the per-set products with the design basis B
// (plaid.lm) without the S x N matrix leaving the device or being written in its normalised form.  Bit-identical to
// plaidgpu_score + plaidgpu_design_stats.  Host X whose S x N scores exceed the device goes through score_chunked
// (two passes when normalised) and adds the tiles' moments in tile order.
int plaidgpu_score_design_stats(plaidgpu_ctx* c, const plaidgpu_matrix* X, const int32_t* rowmap,
                                const plaidgpu_opts* opts, const double* B, int Q, double* out) try {
  if (!c) return PLAIDGPU_ERR_ARG;
  if (!X || !rowmap || !opts || !out) return fail(c, PLAIDGPU_ERR_ARG, "null argument");
  int rc = check_design(c, B, X->N, X->N, Q);
  if (rc) return rc;
  return score_one(c, X, rowmap, opts, Target::design_stats(B, X->N, Q, out));
} catch (const std::bad_alloc&) {
  return PLAIDGPU_ERR_NOMEM;
} catch (...) {
  return PLAIDGPU_ERR_ARG;
}

// score -> top sets fused: plaid() / a replaid.* scorer followed by each column's top k (plaid.topsets) without the
// S x N matrix leaving the device or being written in its normalised form.  Bit-identical to plaidgpu_score +
// plaidgpu_col_topk.  Host X whose S x N scores exceed the device is scored in column tiles, each writing its own
// columns of idx / val.
int plaidgpu_score_topk(plaidgpu_ctx* c, const plaidgpu_matrix* X, const int32_t* rowmap, const plaidgpu_opts* opts,
                        int k, int decreasing, int32_t* idx, double* val) try {
  if (!c) return PLAIDGPU_ERR_ARG;
  if (!X || !rowmap || !opts || !idx || !val) return fail(c, PLAIDGPU_ERR_ARG, "null argument");
  if (!c->have_g) return fail(c, PLAIDGPU_ERR_STATE, "plaidgpu_set_genesets has not been called");
  int rc = check_topk(c, c->S, k);
  if (rc) return rc;
  if (X->N == 0) return PLAIDGPU_OK;
  return score_one(c, X, rowmap, opts, Target::topk(k, decreasing, idx, val));
} catch (const std::bad_alloc&) {
  return PLAIDGPU_ERR_NOMEM;
} catch (...) {
  return PLAIDGPU_ERR_ARG;
}

// score -> top cells fused: plaid() / a replaid.* scorer followed by each set's top k columns (plaid.topcells) without
// the S x N matrix leaving the device or being written in its normalised form.  Bit-identical to plaidgpu_score +
// plaidgpu_row_topk.  Host X whose S x N scores exceed the device is scored in column tiles whose lists are merged in
// tile order.
int plaidgpu_score_row_topk(plaidgpu_ctx* c, const plaidgpu_matrix* X, const int32_t* rowmap, const plaidgpu_opts* opts,
                            int k, int decreasing, int64_t* idx, double* val) try {
  if (!c) return PLAIDGPU_ERR_ARG;
  if (!X || !rowmap || !opts || !idx || !val) return fail(c, PLAIDGPU_ERR_ARG, "null argument");
  if (!c->have_g) return fail(c, PLAIDGPU_ERR_STATE, "plaidgpu_set_genesets has not been called");
  int rc = check_row_topk(c, X->N, k);
  if (rc) return rc;
  return score_one(c, X, rowmap, opts, Target::row_topk(k, decreasing, idx, val));
} catch (const std::bad_alloc&) {
  return PLAIDGPU_ERR_NOMEM;
} catch (...) {
  return PLAIDGPU_ERR_ARG;
}

// two groups y != 0 / y == 0: the labels of plaidgpu_score_group_stats with K = 2
int plaidgpu_score_group_moments(plaidgpu_ctx* c, const plaidgpu_matrix* X, const int32_t* rowmap, const plaidgpu_opts* opts,
                                 const int32_t* y, double* out) try {
  if (!c) return PLAIDGPU_ERR_ARG;
  if (!X || !opts || !y || !out) return fail(c, PLAIDGPU_ERR_ARG, "null argument");
  std::vector<int32_t> lab((size_t)std::max<int64_t>(X->N, 0));
  for (size_t j = 0; j < lab.size(); ++j) lab[j] = y[j] != 0;
  return plaidgpu_score_group_stats(c, X, rowmap, opts, lab.data(), 2, out);
} catch (const std::bad_alloc&) {
  return PLAIDGPU_ERR_NOMEM;
} catch (...) {
  return PLAIDGPU_ERR_ARG;
}

// -----------------------------------------------------------------------------------------
// Several devices from ONE host process (what an R session has): contiguous column shards, one host thread and
// one context per device, every shard's block written straight into the caller's S x N matrix, the cross-shard
// scalars combined on the host in column order (bit-identical to the single-context result).  The axis is the
// column loop of chunked_crossprod (R/plaid.R:110-119).
namespace {
struct ShardBarrier {
  std::mutex m;
  std::condition_variable cv;
  int n, count = 0, gen = 0;
  explicit ShardBarrier(int n_) : n(n_) {}
  void wait() {
    std::unique_lock<std::mutex> lk(m);
    const int g = gen;
    if (++count == n) {
      count = 0;
      ++gen;
      cv.notify_all();
    } else {
      cv.wait(lk, [&] { return gen != g; });
    }
  }
};
}  // namespace

// the contexts of a multi-device call: distinct, each holding the same gene sets, and no scorer that ranks across
// samples
static int check_shard_ctxs(plaidgpu_ctx* const* ctxs, int n, const plaidgpu_opts* opts, const std::string& who) {
  plaidgpu_ctx* c = ctxs[0];
  for (int r = 0; r < n; ++r) {
    if (!ctxs[r] || !ctxs[r]->have_g) return fail(c, PLAIDGPU_ERR_STATE, who + ": every context needs plaidgpu_set_genesets");
    if (ctxs[r]->S != c->S) return fail(c, PLAIDGPU_ERR_ARG, who + ": contexts hold different gene sets");
    for (int q = 0; q < r; ++q)
      if (ctxs[q] == ctxs[r]) return fail(c, PLAIDGPU_ERR_ARG, who + ": the same context twice");
  }
  if (opts->scorer == PLAIDGPU_GSVA && opts->gsva_ecdf == PLAIDGPU_ROWTF_ECDF)
    return fail(c, PLAIDGPU_ERR_ARG, who + ": gsva rowtf = ecdf ranks across samples (use one context, or the row exchange of plaid_b200/sharded.py)");
  return PLAIDGPU_OK;
}

// Shard r (columns [lo_r, lo_{r+1})) finishes on ctxs[r] into t.from(lo_r): its block of the scores, its columns of
// idx / val, or its own group or design moments or row top-k lists, which t.combine folds into the result in shard
// order.  After a fallback only the lists of the fp64 route exist: finish runs once per shard, after the rerun.
static int score_multi_impl(plaidgpu_ctx* const* ctxs, int n, const plaidgpu_matrix* X, const int32_t* rowmap,
                            const plaidgpu_opts* opts, const Target& t, const std::string& who) {
  plaidgpu_ctx* c = ctxs[0];
  try {
    const int64_t N = X->N;
    const int32_t S = c->S, P = X->P;
    const bool norm = needs_norm(*opts);
    const bool gsva_z = opts->scorer == PLAIDGPU_GSVA && opts->gsva_ecdf == PLAIDGPU_ROWTF_Z && !(opts->row_mean && opts->row_sd);
    std::vector<int64_t> lo((size_t)n + 1);
    for (int r = 0; r <= n; ++r) lo[r] = N * r / n;
    std::vector<std::vector<int32_t>> pbuf((size_t)n);
    std::vector<plaidgpu_matrix> M((size_t)n);
    for (int r = 0; r < n; ++r) M[r] = column_slice(X, lo[r], lo[r + 1], pbuf[r]);
    std::vector<plaidgpu_scalars> loc((size_t)n);
    std::vector<int> rc((size_t)n, PLAIDGPU_OK);
    std::vector<Partial> parts((size_t)n);
    std::vector<double> med((size_t)std::max<int64_t>(N, 1));
    std::vector<std::vector<double>> part(gsva_z ? (size_t)n : 0, std::vector<double>((size_t)P));
    std::vector<double> rmean(gsva_z ? (size_t)P : 0), rsd(gsva_z ? (size_t)P : 0);
    plaidgpu_scalars g;
    memset(&g, 0, sizeof(g));
    ShardBarrier bar(n);
    auto failed = [&] {
      for (int r = 0; r < n; ++r)
        if (rc[r]) return true;
      return false;
    };
    auto body = [&](int r) {
      plaidgpu_ctx* cr = ctxs[r];
      plaidgpu_opts o = *opts;
      if (t.kind != Target::SCORES) o.out_location = PLAIDGPU_HOST;  // raw scores stay in the context's device buffer
      const Target tr = t.from(lo[r], S, parts[r]);
      double* dst = t.kind == Target::SCORES ? tr.out : nullptr;
      if (gsva_z) {  // rowMeans / rowSds over ALL shards, summed in shard order (R/plaid.R:343)
        rc[r] = plaidgpu_row_moments(cr, &M[r], nullptr, part[r].data());
        bar.wait();
        if (failed()) return;
        if (r == 0)
          for (int32_t q = 0; q < P; ++q) {
            double a = 0.0;
            for (int k = 0; k < n; ++k) a += part[k][q];
            rmean[q] = a / (double)N;
          }
        bar.wait();
        rc[r] = plaidgpu_row_moments(cr, &M[r], rmean.data(), part[r].data());
        bar.wait();
        if (failed()) return;
        if (r == 0)
          for (int32_t q = 0; q < P; ++q) {
            double a = 0.0;
            for (int k = 0; k < n; ++k) a += part[k][q];
            rsd[q] = N > 1 ? sqrt(a / (double)(N - 1)) : NAN;
          }
        bar.wait();
        o.row_mean = rmean.data();
        o.row_sd = rsd.data();
      }
      rc[r] = plaidgpu_score_begin(cr, &M[r], rowmap, &o, &loc[r]);
      bar.wait();
      if (failed()) return;
      plaidgpu_scalars s = loc[0];
      for (int k = 1; k < n; ++k) {
        s.x_min = fmin(s.x_min, loc[k].x_min);
        s.x_max = fmax(s.x_max, loc[k].x_max);
        s.rank_max = fmax(s.rank_max, loc[k].rank_max);
      }
      const plaidgpu_scalars s_in = s;
      rc[r] = plaidgpu_score_compute(cr, &s, dst);
      loc[r].score_min = s.score_min;
      loc[r].fp64 = s.fp64;
      bar.wait();
      if (failed()) return;
      bool fell_back = false;
      for (int k = 0; k < n; ++k) fell_back |= loc[k].fp64 != 0;
      if (fell_back) {  // one shard left the fixed-point route: every shard scores in fp64, as one context would
        if (!s.fp64) {
          plaidgpu_scalars again;
          o.exact_fp64 = 1;
          rc[r] = plaidgpu_score_begin(cr, &M[r], rowmap, &o, &again);
          s = s_in;
          if (!rc[r]) rc[r] = plaidgpu_score_compute(cr, &s, dst);
          loc[r].score_min = s.score_min;
        }
        bar.wait();
        if (failed()) return;
      }
      if (norm) {
        double smin = INFINITY;
        for (int k = 0; k < n; ++k) smin = fmin(smin, loc[k].score_min);
        const int iz = opts->ignore_zero < 0 ? (smin == 0.0 ? 1 : 0) : (opts->ignore_zero != 0);  // R/plaid.R:556-557
        rc[r] = plaidgpu_get_col_medians_for(cr, iz, med.data() + lo[r]);
        bar.wait();
        if (failed()) return;
        if (r == 0) rc[0] = plaidgpu_combine_medians(iz, smin, med.data(), med.data(), N, &g);
        bar.wait();
        if (failed()) return;
        s.ignore_zero = g.ignore_zero;
        s.med_mean = g.med_mean;
        s.score_min = smin;
      }
      rc[r] = score_finish(cr, &s, tr);
    };
    std::vector<std::thread> th;
    for (int r = 1; r < n; ++r) th.emplace_back(body, r);
    body(0);
    for (auto& t : th) t.join();
    for (int r = 0; r < n; ++r)
      if (rc[r]) {
        if (r > 0) c->err = "shard " + std::to_string(r) + ": " + ctxs[r]->err;
        return rc[r];
      }
    t.clear(S);
    for (int r = 0; r < n; ++r) t.combine(parts[r], S);
    return PLAIDGPU_OK;
  } catch (const std::bad_alloc&) {
    return fail(c, PLAIDGPU_ERR_NOMEM, "out of host memory");
  } catch (...) {
    return fail(c, PLAIDGPU_ERR_ARG, "unexpected failure in " + who);
  }
}

// The multi-context entry points after their own argument checks: X in host memory, then the contexts (n > 1, so bad
// contexts fail whatever N is), then the single-device entry point on ctxs[0] (n == 1 or N < 2n) or the shards
static int score_multi(plaidgpu_ctx* const* ctxs, int n, const plaidgpu_matrix* X, const int32_t* rowmap,
                       const plaidgpu_opts* opts, const Target& t, const char* name) {
  plaidgpu_ctx* c = ctxs[0];
  const std::string who(name);
  if (t.kind == Target::SCORES && (X->location != PLAIDGPU_HOST || opts->out_location != PLAIDGPU_HOST))
    return fail(c, PLAIDGPU_ERR_ARG, who + ": X and out must be in host memory");
  if (X->location != PLAIDGPU_HOST) return fail(c, PLAIDGPU_ERR_ARG, who + ": X must be in host memory");
  int rc = n > 1 ? check_shard_ctxs(ctxs, n, opts, who) : PLAIDGPU_OK;
  if (rc) return rc;
  if (n == 1 || X->N < 2 * (int64_t)n) {
    if (t.kind == Target::GROUP_STATS) return plaidgpu_score_group_stats(c, X, rowmap, opts, t.labels, t.K, t.out);
    if (t.kind == Target::DESIGN_STATS) return plaidgpu_score_design_stats(c, X, rowmap, opts, t.B, t.Q, t.out);
    if (t.kind == Target::TOPK) return plaidgpu_score_topk(c, X, rowmap, opts, t.k, t.decreasing, t.idx, t.val);
    if (t.kind == Target::ROW_TOPK) return plaidgpu_score_row_topk(c, X, rowmap, opts, t.k, t.decreasing, t.cols, t.val);
    return plaidgpu_score(c, X, rowmap, opts, t.out);
  }
  if (t.kind == Target::GROUP_STATS) rc = check_groups(c, t.labels, X->N, t.K);
  if (t.kind == Target::DESIGN_STATS) rc = check_design(c, t.B, X->N, t.ldb, t.Q);
  if (t.kind == Target::TOPK) rc = check_topk(c, c->S, t.k);
  if (t.kind == Target::ROW_TOPK) rc = check_row_topk(c, X->N, t.k);
  if (rc) return rc;
  return score_multi_impl(ctxs, n, X, rowmap, opts, t, who);
}

int plaidgpu_score_multi(plaidgpu_ctx* const* ctxs, int n, const plaidgpu_matrix* X, const int32_t* rowmap,
                         const plaidgpu_opts* opts, double* out) try {
  if (!ctxs || n <= 0 || !ctxs[0]) return PLAIDGPU_ERR_ARG;
  if (!X || !rowmap || !opts) return fail(ctxs[0], PLAIDGPU_ERR_ARG, "null argument");
  return score_multi(ctxs, n, X, rowmap, opts, Target::scores(out), "plaidgpu_score_multi");
} catch (const std::bad_alloc&) {
  return PLAIDGPU_ERR_NOMEM;
} catch (...) {
  return PLAIDGPU_ERR_ARG;
}

int plaidgpu_score_group_stats_multi(plaidgpu_ctx* const* ctxs, int n, const plaidgpu_matrix* X, const int32_t* rowmap,
                                     const plaidgpu_opts* opts, const int32_t* labels, int K, double* out) try {
  if (!ctxs || n <= 0 || !ctxs[0]) return PLAIDGPU_ERR_ARG;
  if (!X || !rowmap || !opts || !out) return fail(ctxs[0], PLAIDGPU_ERR_ARG, "null argument");
  return score_multi(ctxs, n, X, rowmap, opts, Target::group_stats(labels, K, out), "plaidgpu_score_group_stats_multi");
} catch (const std::bad_alloc&) {
  return PLAIDGPU_ERR_NOMEM;
} catch (...) {
  return PLAIDGPU_ERR_ARG;
}

int plaidgpu_score_design_stats_multi(plaidgpu_ctx* const* ctxs, int n, const plaidgpu_matrix* X, const int32_t* rowmap,
                                      const plaidgpu_opts* opts, const double* B, int Q, double* out) try {
  if (!ctxs || n <= 0 || !ctxs[0]) return PLAIDGPU_ERR_ARG;
  if (!X || !rowmap || !opts || !out) return fail(ctxs[0], PLAIDGPU_ERR_ARG, "null argument");
  return score_multi(ctxs, n, X, rowmap, opts, Target::design_stats(B, X->N, Q, out), "plaidgpu_score_design_stats_multi");
} catch (const std::bad_alloc&) {
  return PLAIDGPU_ERR_NOMEM;
} catch (...) {
  return PLAIDGPU_ERR_ARG;
}

int plaidgpu_score_topk_multi(plaidgpu_ctx* const* ctxs, int n, const plaidgpu_matrix* X, const int32_t* rowmap,
                              const plaidgpu_opts* opts, int k, int decreasing, int32_t* idx, double* val) try {
  if (!ctxs || n <= 0 || !ctxs[0]) return PLAIDGPU_ERR_ARG;
  if (!X || !rowmap || !opts || !idx || !val) return fail(ctxs[0], PLAIDGPU_ERR_ARG, "null argument");
  return score_multi(ctxs, n, X, rowmap, opts, Target::topk(k, decreasing, idx, val), "plaidgpu_score_topk_multi");
} catch (const std::bad_alloc&) {
  return PLAIDGPU_ERR_NOMEM;
} catch (...) {
  return PLAIDGPU_ERR_ARG;
}

int plaidgpu_score_row_topk_multi(plaidgpu_ctx* const* ctxs, int n, const plaidgpu_matrix* X, const int32_t* rowmap,
                                  const plaidgpu_opts* opts, int k, int decreasing, int64_t* idx, double* val) try {
  if (!ctxs || n <= 0 || !ctxs[0]) return PLAIDGPU_ERR_ARG;
  if (!X || !rowmap || !opts || !idx || !val) return fail(ctxs[0], PLAIDGPU_ERR_ARG, "null argument");
  return score_multi(ctxs, n, X, rowmap, opts, Target::row_topk(k, decreasing, idx, val), "plaidgpu_score_row_topk_multi");
} catch (const std::bad_alloc&) {
  return PLAIDGPU_ERR_NOMEM;
} catch (...) {
  return PLAIDGPU_ERR_ARG;
}

int plaidgpu_crossprod(plaidgpu_ctx* c, const plaidgpu_matrix* Y, const int32_t* rowmap, const double* colscale,
                       int out_location, double* out) try {
  if (!c) return PLAIDGPU_ERR_ARG;
  if (!Y || !rowmap) return fail(c, PLAIDGPU_ERR_ARG, "null argument");
  if (!c->have_g) return fail(c, PLAIDGPU_ERR_STATE, "plaidgpu_set_genesets has not been called");
  plaidgpu_opts o;
  plaidgpu_default_opts(&o);
  o.stats_mean = 0;
  o.normalize = 0;
  o.out_location = out_location;
  plaidgpu_scalars s;
  int rc = plaidgpu_score_begin(c, Y, rowmap, &o, &s);
  if (rc) return rc;
  if (colscale) {  // swap the per-set scale for the caller's column scale of x
    CK(c->d_custom_inv.reserve((size_t)c->S * sizeof(double)));
    CK(cudaMemcpyAsync(c->d_custom_inv.p, colscale, (size_t)c->S * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    std::swap(c->d_inv_one.p, c->d_custom_inv.p);
    std::swap(c->d_inv_one.cap, c->d_custom_inv.cap);
  }
  rc = plaidgpu_score_compute(c, &s, out);
  if (colscale) {
    std::swap(c->d_inv_one.p, c->d_custom_inv.p);
    std::swap(c->d_inv_one.cap, c->d_custom_inv.cap);
  }
  if (rc) return rc;
  return plaidgpu_score_finish(c, &s, out);
} catch (const std::bad_alloc&) {
  return PLAIDGPU_ERR_NOMEM;
} catch (...) {
  return PLAIDGPU_ERR_ARG;
}

int plaidgpu_row_moments(plaidgpu_ctx* c, const plaidgpu_matrix* X, const double* mean, double* out) try {
  if (!c) return PLAIDGPU_ERR_ARG;
  if (!X || !out) return fail(c, PLAIDGPU_ERR_ARG, "null argument");
  trace("begin");
  CK(cudaSetDevice(c->device));
  c->in_call = false;
  c->computed = false;
  int rc = load_matrix(c, X);
  if (rc) return rc;
  rc = make_dense(c);
  if (rc) return rc;
  return row_moments(c, mean, out);
} catch (const std::bad_alloc&) {
  return PLAIDGPU_ERR_NOMEM;
} catch (...) {
  return PLAIDGPU_ERR_ARG;
}

int plaidgpu_row_ecdf(plaidgpu_ctx* c, double* x, int64_t N, int32_t rows, int location) try {
  if (!c) return PLAIDGPU_ERR_ARG;
  if (!x && N > 0 && rows > 0) return fail(c, PLAIDGPU_ERR_ARG, "null argument");
  if (N < 0 || rows < 0 || N > 0x7fffffff) return fail(c, PLAIDGPU_ERR_ARG, "bad dimensions for row ecdf");
  trace("begin");
  CK(cudaSetDevice(c->device));
  c->in_call = false;
  c->computed = false;
  const int64_t total = N * (int64_t)rows;
  if (total == 0) return PLAIDGPU_OK;
  const double* src = nullptr;
  int rc = to_device<double>(c, x, (size_t)total, location, c->b_xx, &src);
  if (rc) return rc;
  double* d = const_cast<double*>(src);
  // every gene's samples are one column of the N x rows matrix: max-rank / N  (R/plaid.R:346)
  CK(cudaEventRecord(c->ev[6], c->stream));
  CK(launch_rank_dense(d, (int32_t)N, rows, PLAIDGPU_TIES_MAX, 0, d, nullptr, c->stream));
  CK(launch_xform_dense(d, d, total, XF_SCALE, 1.0 / (double)N, 0.0, c->stream));
  c->launches += 2;
  CK(cudaEventRecord(c->ev[7], c->stream));
  if (location == PLAIDGPU_HOST)
    CK(cudaMemcpyAsync(x, d, (size_t)total * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  float ms = 0.f;
  cudaEventElapsedTime(&ms, c->ev[6], c->ev[7]);
  c->ms[3] = ms;
  return PLAIDGPU_OK;
} catch (const std::bad_alloc&) {
  return PLAIDGPU_ERR_NOMEM;
} catch (...) {
  return PLAIDGPU_ERR_ARG;
}

// -----------------------------------------------------------------------------------------
int plaidgpu_colranks(plaidgpu_ctx* c, const plaidgpu_matrix* X, int ties, int is_signed, int keep_zero,
                      int out_location, double* out) try {
  if (!c) return PLAIDGPU_ERR_ARG;
  if (!X || !out) return fail(c, PLAIDGPU_ERR_ARG, "null argument");
  if (ties < PLAIDGPU_TIES_AVERAGE || ties > PLAIDGPU_TIES_DENSE) return fail(c, PLAIDGPU_ERR_ARG, "unsupported ties.method");
  if (ties > PLAIDGPU_TIES_MAX && X->kind == PLAIDGPU_CSC && !keep_zero)
    return fail(c, PLAIDGPU_ERR_ARG, "ties.method first / last / dense: not available for sparse input without keep.zero "
                                     "(sparseMatrixStats::colRanks knows max, average, min)");
  trace("begin");
  CK(cudaSetDevice(c->device));
  c->in_call = false;
  c->computed = false;
  int rc = load_matrix(c, X);
  if (rc) return rc;
  CK(cudaEventRecord(c->ev[6], c->stream));
  if (c->dense) {
    double* dst = out;
    if (out_location == PLAIDGPU_HOST) {
      CK(c->b_rank.reserve(std::max<int64_t>(c->nnz, 1) * sizeof(double)));
      dst = c->b_rank.as<double>();
    }
    CK(launch_rank_dense(c->xx, c->P, c->N, ties, is_signed, dst, nullptr, c->stream));
    c->launches += 1;
    CK(cudaEventRecord(c->ev[7], c->stream));
    if (out_location == PLAIDGPU_HOST && c->nnz)
      CK(cudaMemcpyAsync(out, dst, (size_t)c->nnz * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  } else {
    int32_t mcn = 0;
    rc = max_col_nnz(c, &mcn);
    if (rc) return rc;
    if (keep_zero) {  // sparse_colranks: nnz ranks
      double* dst = out;
      if (out_location == PLAIDGPU_HOST) {
        CK(c->b_rank.reserve(std::max<int64_t>(c->nnz, 1) * sizeof(double)));
        dst = c->b_rank.as<double>();
      }
      CK(launch_rank_csc(c->xp, c->xx, c->P, c->N, ties, is_signed, 0, dst, nullptr, nullptr, mcn, c->stream));
      c->launches += 1;
      CK(cudaEventRecord(c->ev[7], c->stream));
      if (out_location == PLAIDGPU_HOST && c->nnz)
        CK(cudaMemcpyAsync(out, dst, (size_t)c->nnz * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    } else {  // dense P x N ranks with the zero group
      CK(c->b_rank.reserve(std::max<int64_t>(c->nnz, 1) * sizeof(double)));
      CK(c->b_r0.reserve(std::max<int64_t>(c->N, 1) * sizeof(double)));
      CK(launch_rank_csc(c->xp, c->xx, c->P, c->N, ties, is_signed, 1, c->b_rank.as<double>(),
                         c->b_r0.as<double>(), nullptr, mcn, c->stream));
      const int64_t total = (int64_t)c->P * c->N;
      double* dst = out;
      if (out_location == PLAIDGPU_HOST) {
        CK(c->b_raw.reserve((size_t)std::max<int64_t>(total, 1) * sizeof(double)));
        dst = c->b_raw.as<double>();
      }
      CK(launch_expand_ranks(c->xp, c->xi, c->b_rank.as<double>(), c->b_r0.as<double>(), c->P, c->N, dst, c->stream));
      c->launches += 2;
      CK(cudaEventRecord(c->ev[7], c->stream));
      if (out_location == PLAIDGPU_HOST && total)
        CK(cudaMemcpyAsync(out, dst, (size_t)total * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    }
  }
  CK(cudaStreamSynchronize(c->stream));
  float ms = 0.f;
  cudaEventElapsedTime(&ms, c->ev[6], c->ev[7]);
  c->ms[3] = ms;
  return PLAIDGPU_OK;
} catch (const std::bad_alloc&) {
  return PLAIDGPU_ERR_NOMEM;
} catch (...) {
  return PLAIDGPU_ERR_ARG;
}

int plaidgpu_group_stats(plaidgpu_ctx* c, const double* x, int32_t S, int64_t N, const int32_t* labels, int K, int location,
                         double* out) try {
  if (!c) return PLAIDGPU_ERR_ARG;
  if (S <= 0 || N < 0) return fail(c, PLAIDGPU_ERR_ARG, "bad argument");
  if (!out || (N > 0 && !x)) return fail(c, PLAIDGPU_ERR_ARG, "null argument");
  int rc = check_groups(c, labels, N, K);
  if (rc) return rc;
  CK(cudaSetDevice(c->device));
  const int64_t total = (int64_t)S * N;
  const double* dx = x;
  if (location == PLAIDGPU_HOST) {
    CK(c->b_raw.reserve((size_t)std::max<int64_t>(total, 1) * sizeof(double)));
    if (total) CK(cudaMemcpyAsync(c->b_raw.p, x, (size_t)total * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    dx = c->b_raw.as<double>();
  }
  return group_stats_device(c, dx, S, N, labels, K, out);
} catch (const std::bad_alloc&) {
  return PLAIDGPU_ERR_NOMEM;
} catch (...) {
  return PLAIDGPU_ERR_ARG;
}

int plaidgpu_design_stats(plaidgpu_ctx* c, const double* x, int32_t S, int64_t N, const double* B, int Q, int location,
                          double* out) try {
  if (!c) return PLAIDGPU_ERR_ARG;
  if (S <= 0 || N < 0) return fail(c, PLAIDGPU_ERR_ARG, "bad argument");
  if (!out || (N > 0 && !x)) return fail(c, PLAIDGPU_ERR_ARG, "null argument");
  if (location != PLAIDGPU_HOST && location != PLAIDGPU_DEVICE) return fail(c, PLAIDGPU_ERR_ARG, "unknown location");
  int rc = check_design(c, B, N, N, Q);
  if (rc) return rc;
  CK(cudaSetDevice(c->device));
  const int64_t total = (int64_t)S * N;
  const double* dx = x;
  if (location == PLAIDGPU_HOST) {
    CK(c->b_raw.reserve((size_t)std::max<int64_t>(total, 1) * sizeof(double)));
    if (total) CK(cudaMemcpyAsync(c->b_raw.p, x, (size_t)total * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    dx = c->b_raw.as<double>();
  }
  return design_stats_device(c, dx, S, N, B, N, Q, out);
} catch (const std::bad_alloc&) {
  return PLAIDGPU_ERR_NOMEM;
} catch (...) {
  return PLAIDGPU_ERR_ARG;
}

// two groups y != 0 / y == 0: the labels of plaidgpu_group_stats with K = 2
int plaidgpu_group_moments(plaidgpu_ctx* c, const double* x, int32_t S, int64_t N, const int32_t* y, int location,
                           double* out) try {
  if (!c) return PLAIDGPU_ERR_ARG;
  if (S <= 0 || N < 0 || !out || (N > 0 && (!x || !y))) return fail(c, PLAIDGPU_ERR_ARG, "bad argument");
  std::vector<int32_t> lab((size_t)N);
  for (int64_t j = 0; j < N; ++j) lab[(size_t)j] = y[j] != 0;
  return plaidgpu_group_stats(c, x, S, N, lab.data(), 2, location, out);
} catch (const std::bad_alloc&) {
  return PLAIDGPU_ERR_NOMEM;
} catch (...) {
  return PLAIDGPU_ERR_ARG;
}

int plaidgpu_col_topk(plaidgpu_ctx* c, const double* x, int32_t S, int64_t N, int k, int decreasing, int location,
                      int32_t* idx, double* val) try {
  if (!c) return PLAIDGPU_ERR_ARG;
  if (S <= 0 || N < 0) return fail(c, PLAIDGPU_ERR_ARG, "bad argument");
  if (!idx || !val || (N > 0 && !x)) return fail(c, PLAIDGPU_ERR_ARG, "null argument");
  if (location != PLAIDGPU_HOST && location != PLAIDGPU_DEVICE) return fail(c, PLAIDGPU_ERR_ARG, "unknown location");
  int rc = check_topk(c, S, k);
  if (rc) return rc;
  if (N == 0) return PLAIDGPU_OK;
  CK(cudaSetDevice(c->device));
  const double* dx = x;
  if (location == PLAIDGPU_HOST) {
    const size_t total = (size_t)S * (size_t)N;
    CK(c->b_raw.reserve(total * sizeof(double)));
    CK(cudaMemcpyAsync(c->b_raw.p, x, total * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    dx = c->b_raw.as<double>();
  }
  return topk_device(c, dx, S, N, k, decreasing != 0, idx, val);
} catch (const std::bad_alloc&) {
  return PLAIDGPU_ERR_NOMEM;
} catch (...) {
  return PLAIDGPU_ERR_ARG;
}

int plaidgpu_row_topk(plaidgpu_ctx* c, const double* x, int32_t S, int64_t N, int k, int decreasing, int location,
                      int64_t* idx, double* val) try {
  if (!c) return PLAIDGPU_ERR_ARG;
  if (S <= 0 || N < 0) return fail(c, PLAIDGPU_ERR_ARG, "bad argument");
  if (!x || !idx || !val) return fail(c, PLAIDGPU_ERR_ARG, "null argument");
  if (location != PLAIDGPU_HOST && location != PLAIDGPU_DEVICE) return fail(c, PLAIDGPU_ERR_ARG, "unknown location");
  int rc = check_row_topk(c, N, k);
  if (rc) return rc;
  CK(cudaSetDevice(c->device));
  const double* dx = x;
  if (location == PLAIDGPU_HOST) {
    const size_t total = (size_t)S * (size_t)N;
    CK(c->b_raw.reserve(total * sizeof(double)));
    CK(cudaMemcpyAsync(c->b_raw.p, x, total * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    dx = c->b_raw.as<double>();
  }
  return row_topk_device(c, dx, S, N, k, decreasing != 0, 0, idx, val);
} catch (const std::bad_alloc&) {
  return PLAIDGPU_ERR_NOMEM;
} catch (...) {
  return PLAIDGPU_ERR_ARG;
}

// -----------------------------------------------------------------------------------------
int plaidgpu_normalize_medians(plaidgpu_ctx* c, const double* x, int32_t S, int64_t N, int ignore_zero,
                               int location, double* out) try {
  if (!c) return PLAIDGPU_ERR_ARG;
  if (S <= 0 || N < 0 || (N > 0 && (!x || !out))) return fail(c, PLAIDGPU_ERR_ARG, "bad argument");
  trace("begin");
  CK(cudaSetDevice(c->device));
  c->in_call = false;
  c->computed = false;
  const int64_t total = (int64_t)S * N;
  const double* dx = x;
  if (location == PLAIDGPU_HOST) {
    CK(c->b_raw.reserve((size_t)std::max<int64_t>(total, 1) * sizeof(double)));
    if (total) CK(cudaMemcpyAsync(c->b_raw.p, x, (size_t)total * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    dx = c->b_raw.as<double>();
  }
  CK(c->b_med_all.reserve(std::max<int64_t>(N, 1) * sizeof(double)));
  CK(c->b_med_nz.reserve(std::max<int64_t>(N, 1) * sizeof(double)));
  CK(c->b_colmin.reserve(std::max<int64_t>(N, 1) * sizeof(double)));
  CK(cudaEventRecord(c->ev[2], c->stream));
  CK(c->b_fail.reserve(sizeof(int)));
  CK(c->b_list.reserve(std::max<int64_t>(N, 1) * sizeof(int64_t)));
  // ignore.zero given: one median; auto: the flag needs min(x) first, so both come out of the same pass
  const int which = ignore_zero < 0 ? COLSTATS_BOTH : (ignore_zero ? COLSTATS_NZ : COLSTATS_ALL);
  CK(launch_colstats(dx, S, S, N, c->b_med_all.as<double>(), c->b_med_nz.as<double>(), c->b_colmin.as<double>(),
                     c->b_fail.as<int>(), c->b_list.as<int64_t>(), which, c->stream));
  c->launches += 1;
  CK(cudaEventRecord(c->ev[3], c->stream));
  c->h_med_all.resize((size_t)N);
  c->h_med_nz.resize((size_t)N);
  c->h_colmin.resize((size_t)N);
  if (N) {
    CK(cudaMemcpyAsync(c->h_med_all.data(), c->b_med_all.p, (size_t)N * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(c->h_med_nz.data(), c->b_med_nz.p, (size_t)N * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(c->h_colmin.data(), c->b_colmin.p, (size_t)N * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  }
  CK(cudaStreamSynchronize(c->stream));
  float ms = 0.f;
  cudaEventElapsedTime(&ms, c->ev[2], c->ev[3]);
  c->ms[1] = ms;
  double mn = INFINITY;
  for (int64_t j = 0; j < N; ++j) mn = fmin(mn, c->h_colmin[j]);
  plaidgpu_scalars s{};
  plaidgpu_combine_medians(ignore_zero, mn, c->h_med_all.data(), c->h_med_nz.data(), N, &s);
  const double* med = s.ignore_zero ? c->b_med_nz.as<double>() : c->b_med_all.as<double>();
  CK(cudaEventRecord(c->ev[4], c->stream));
  if (location == PLAIDGPU_DEVICE) {
    CK(launch_fixup(dx, out, S, S, 0, N, med, s.med_mean, 1.0, nullptr, c->stream));
    c->launches += 1;
    CK(cudaEventRecord(c->ev[5], c->stream));
  } else {
    CK(launch_fixup(dx, c->b_raw.as<double>(), S, S, 0, N, med, s.med_mean, 1.0, nullptr, c->stream));
    c->launches += 1;
    CK(cudaEventRecord(c->ev[5], c->stream));
    if (total) CK(cudaMemcpyAsync(out, c->b_raw.p, (size_t)total * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  }
  CK(cudaStreamSynchronize(c->stream));
  cudaEventElapsedTime(&ms, c->ev[4], c->ev[5]);
  c->ms[2] = ms;
  return PLAIDGPU_OK;
} catch (const std::bad_alloc&) {
  return PLAIDGPU_ERR_NOMEM;
} catch (...) {
  return PLAIDGPU_ERR_ARG;
}

}  // extern "C"
