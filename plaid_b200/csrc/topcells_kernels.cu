// Per-row top-k selection with column indices (plaid.topcells: each gene set's best cells).
//
// The scores are column-major, so the sets of one cell are contiguous and a set's row is strided by 8 * S bytes:
// reading it directly would use 8 bytes of every 32-byte sector.  k_row_topk_partial stages tiles of
// (32 sets x ROW_COLS columns) through shared memory instead, each warp loading 32 consecutive sets of one column
// (256 bytes), and then runs the warp selection of topk_select.cuh over each set's contiguous row segment.
// The grid is (set block, column chunk): chunk c writes a sorted partial list of k (key, column) entries per set,
// padded with an explicit "no entry" (key 0 and the largest column: after every NaN) when the chunk has fewer than k
// columns.  k_row_topk_merge then selects each set's k best from its chunks' lists with the same warp selection.
// The composite key decides the order, so the result does not depend on the chunking or the launch geometry.
// FIX: the values are RAW scores and the fix-up of plaidgpu_score_finish (fixup_value, k_fixup's operations in its
// order, the column's median shift changing along the stream) is applied in registers as the tile is loaded.  The
// returned values are recomputed from x at the selected columns, so they are bit for bit the ones plaid() returns.
#include "topk_select.cuh"

namespace plaidgpu {
namespace {

constexpr int ROW_WARPS = 8;                         // warps per block
constexpr int ROW_SETS = 32;                         // sets per block: one 256-byte load of a column per warp
constexpr int ROW_SETS_PER_WARP = ROW_SETS / ROW_WARPS;
constexpr int ROW_COLS = 64;                         // columns per staged tile: two 32-column batches per set
constexpr int ROW_LOADS = ROW_COLS / ROW_WARPS;      // columns each warp loads per tile
constexpr uint32_t NO_COL = 0xffffffffu;             // "no entry" in a chunk (chunk-relative columns)
constexpr uint64_t NO_COL64 = ~0ull;                 // "no entry" in a partial list (columns of the launch)

using topk::better;
using topk::order_key;

template <bool FIX>
__device__ __forceinline__ double fixed_at(const double* __restrict__ x, int64_t ld, int32_t s, int64_t j,
                                           const double* __restrict__ med, double c, double alpha,
                                           const double* __restrict__ beta) {
  const double v = x[j * ld + s];
  return FIX ? fixup_value(v, j, med, c, alpha, beta, beta ? beta[s] : 0.0) : v;
}

// Chunk blockIdx.y of the columns (the N * c / nchunk split) for sets [32 * blockIdx.x, + 32): each set's k best
// into partial key / column lists pkey / pcol[(chunk * S + s) * k + t], sorted best first.
// SMALL: k <= 32, lists in registers; otherwise k <= 256 with 2 * k entries of shared memory per set.
template <bool FIX, bool SMALL>
__global__ void __launch_bounds__(ROW_WARPS * 32) k_row_topk_partial(
    const double* __restrict__ x, int64_t ld, int32_t S, int64_t N, int nchunk, int k, int decreasing,
    uint64_t* __restrict__ pkey, uint64_t* __restrict__ pcol, const double* __restrict__ med, double c, double alpha,
    const double* __restrict__ beta) {
  extern __shared__ __align__(16) unsigned char row_smem[];
  double(*tile)[ROW_SETS + 1] = reinterpret_cast<double(*)[ROW_SETS + 1]>(row_smem);  // [ROW_COLS][ROW_SETS + 1]
  const int lane = threadIdx.x & 31;
  const int w = threadIdx.x >> 5;
  const int32_t s0 = (int32_t)blockIdx.x * ROW_SETS;
  const int64_t j0 = N * (int64_t)blockIdx.y / nchunk, j1 = N * ((int64_t)blockIdx.y + 1) / nchunk;
  const bool dec = decreasing != 0;
  using Entry = topk::Entry<uint32_t>;
  const Entry none{0ull, NO_COL};  // worse than every real entry, NaN included

  // loads: lane = set s0 + lane of columns w, w + ROW_WARPS, ... of the tile
  const int32_t ls = s0 + lane;
  const bool lrow = ls < S;
  const double lb = FIX && beta && lrow ? beta[ls] : 0.0;
  double v[ROW_LOADS];
  auto load = [&](int64_t jt) {
#pragma unroll
    for (int u = 0; u < ROW_LOADS; ++u) {
      const int64_t j = jt + w + ROW_WARPS * u;
      v[u] = 0.0;
      if (lrow && j < j1) {
        v[u] = __ldcs(x + j * ld + ls);
        if (FIX) v[u] = fixup_value(v[u], j, med, c, alpha, beta, lb);
      }
    }
  };

  // selection: warp w owns the sets s0 + ROW_SETS_PER_WARP * w + i (tile row r_i); their lists and thresholds
  Entry list[ROW_SETS_PER_WARP], thr[ROW_SETS_PER_WARP];
  int cur[ROW_SETS_PER_WARP];
  topk::SharedList<uint32_t> L[ROW_SETS_PER_WARP];
#pragma unroll
  for (int i = 0; i < ROW_SETS_PER_WARP; ++i) {
    list[i] = none;
    thr[i] = none;
    cur[i] = 0;
    if (!SMALL) {
      // per set: lists of 2 k entries; the 32-entry batch is the warp's, shared by its sets (they take turns)
      unsigned char* lists = row_smem + sizeof(double) * ROW_COLS * (ROW_SETS + 1);
      const int r = ROW_SETS_PER_WARP * w + i;
      uint64_t* key = reinterpret_cast<uint64_t*>(lists) + (size_t)r * 2 * k;
      uint32_t* idx = reinterpret_cast<uint32_t*>(lists + (size_t)ROW_SETS * 2 * k * 8) + (size_t)r * 2 * k;
      unsigned char* batch = lists + (size_t)ROW_SETS * 2 * k * 12 + (size_t)w * 32 * 12;
      L[i].key = key;
      L[i].idx = idx;
      L[i].bkey = reinterpret_cast<uint64_t*>(batch);
      L[i].bidx = reinterpret_cast<uint32_t*>(batch + 32 * 8);
      for (int t = lane; t < k; t += 32) {
        key[t] = none.key;
        idx[t] = none.idx;
      }
    }
  }
  __syncwarp();

  load(j0);
  for (int64_t jt = j0; jt < j1; jt += ROW_COLS) {
    __syncthreads();  // every warp is done with the previous tile
#pragma unroll
    for (int u = 0; u < ROW_LOADS; ++u) tile[w + ROW_WARPS * u][lane] = v[u];
    __syncthreads();
    if (jt + ROW_COLS < j1) load(jt + ROW_COLS);  // the next tile's loads are in flight while this one is selected
#pragma unroll
    for (int i = 0; i < ROW_SETS_PER_WARP; ++i) {
      const int r = ROW_SETS_PER_WARP * w + i;
      if (s0 + r >= S) continue;  // whole warps
#pragma unroll
      for (int b = 0; b < ROW_COLS / 32; ++b) {
        const int64_t j = jt + 32 * b + lane;
        Entry e = none;
        if (j < j1) {
          e.key = order_key(tile[32 * b + lane][r], dec);
          e.idx = (uint32_t)(j - j0);
        }
        const unsigned pass = __ballot_sync(FULL, better(e, thr[i]));
        if (!pass) continue;
        if (SMALL) topk::offer_small(e, pass, list[i], thr[i], k, lane);
        else topk::offer_large(e, L[i], cur[i], thr[i], k, lane);
      }
    }
  }

#pragma unroll
  for (int i = 0; i < ROW_SETS_PER_WARP; ++i) {
    const int32_t s = s0 + ROW_SETS_PER_WARP * w + i;
    if (s >= S) continue;
    const size_t o = ((size_t)blockIdx.y * (size_t)S + (size_t)s) * (size_t)k;
    if (SMALL) {
      if (lane < k) {
        pkey[o + lane] = list[i].key;
        pcol[o + lane] = list[i].idx == NO_COL ? NO_COL64 : (uint64_t)j0 + list[i].idx;
      }
    } else {
      const uint64_t* ck = L[i].key + cur[i] * k;
      const uint32_t* cr = L[i].idx + cur[i] * k;
      for (int t = lane; t < k; t += 32) {
        pkey[o + t] = ck[t];
        pcol[o + t] = cr[t] == NO_COL ? NO_COL64 : (uint64_t)j0 + cr[t];
      }
    }
  }
}

// One warp per set: the k best of its nchunk partial lists into idx[t + k * s] = col0 + column (-1 for no entry)
// and val[t + k * s] = the value at that column (NaN for no entry).
template <bool FIX, bool SMALL>
__global__ void __launch_bounds__(ROW_WARPS * 32) k_row_topk_merge(
    const uint64_t* __restrict__ pkey, const uint64_t* __restrict__ pcol, int32_t S, int nchunk, int k,
    const double* __restrict__ x, int64_t ld, int64_t col0, int64_t* __restrict__ idx, double* __restrict__ val,
    const double* __restrict__ med, double c, double alpha, const double* __restrict__ beta) {
  extern __shared__ __align__(16) unsigned char merge_smem[];
  const int lane = threadIdx.x & 31;
  const int w = threadIdx.x >> 5;
  const int32_t s = (int32_t)blockIdx.x * ROW_WARPS + w;
  if (s >= S) return;  // whole warps leave together
  using Entry = topk::Entry<uint64_t>;
  const Entry none{0ull, NO_COL64};
  topk::SharedList<uint64_t> L;
  int cur = 0;
  Entry list = none, thr = none;
  if (!SMALL) L.init(merge_smem + (size_t)w * topk::SharedList<uint64_t>::bytes(k), k, lane, none);
  const int n = nchunk * k;
  for (int i0 = 0; i0 < n; i0 += 32) {
    const int i = i0 + lane;
    Entry e = none;
    if (i < n) {
      const size_t o = ((size_t)(i / k) * (size_t)S + (size_t)s) * (size_t)k + (size_t)(i % k);
      e.key = pkey[o];
      e.idx = pcol[o];
    }
    const unsigned pass = __ballot_sync(FULL, better(e, thr));
    if (!pass) continue;
    if (SMALL) topk::offer_small(e, pass, list, thr, k, lane);
    else topk::offer_large(e, L, cur, thr, k, lane);
  }
  int64_t* is = idx + (int64_t)k * s;
  double* vs = val + (int64_t)k * s;
  auto put = [&](int t, uint64_t j) {
    if (j == NO_COL64) {
      is[t] = -1;
      vs[t] = __longlong_as_double(0x7ff8000000000000ll);
    } else {
      is[t] = col0 + (int64_t)j;
      vs[t] = fixed_at<FIX>(x, ld, s, (int64_t)j, med, c, alpha, beta);
    }
  };
  if (SMALL) {
    if (lane < k) put(lane, list.idx);
  } else {
    const uint64_t* cr = L.idx + cur * k;
    for (int t = lane; t < k; t += 32) put(t, cr[t]);
  }
}

size_t partial_smem(bool small, int k) {
  return sizeof(double) * ROW_COLS * (ROW_SETS + 1) + (small ? 0 : (size_t)ROW_SETS * 2 * k * 12 + ROW_WARPS * 32 * 12);
}

template <bool FIX, bool SMALL>
cudaError_t launch_both(const double* x, int64_t ld, int32_t S, int64_t N, int k, int decreasing, int nchunk,
                        uint64_t* partial, int64_t col0, int64_t* idx, double* val, cudaStream_t st,
                        const double* med, double c, double alpha, const double* beta) {
  const size_t psmem = partial_smem(SMALL, k);
  const size_t msmem = SMALL ? 0 : ROW_WARPS * topk::SharedList<uint64_t>::bytes(k);
  cudaError_t e = cudaFuncSetAttribute(k_row_topk_partial<FIX, SMALL>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)psmem);
  if (e == cudaSuccess && !SMALL)
    e = cudaFuncSetAttribute(k_row_topk_merge<FIX, SMALL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)msmem);
  if (e != cudaSuccess) return e;
  uint64_t* pkey = partial;
  uint64_t* pcol = partial + (size_t)nchunk * (size_t)S * (size_t)k;
  const dim3 grid((unsigned)((S + ROW_SETS - 1) / ROW_SETS), (unsigned)nchunk);
  k_row_topk_partial<FIX, SMALL><<<grid, ROW_WARPS * 32, psmem, st>>>(x, ld, S, N, nchunk, k, decreasing, pkey, pcol,
                                                                      med, c, alpha, beta);
  e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  k_row_topk_merge<FIX, SMALL><<<(unsigned)((S + ROW_WARPS - 1) / ROW_WARPS), ROW_WARPS * 32, msmem, st>>>(
      pkey, pcol, S, nchunk, k, x, ld, col0, idx, val, med, c, alpha, beta);
  return cudaGetLastError();
}

}  // namespace

cudaError_t launch_row_topk(const double* x, int64_t ld, int32_t S, int64_t N, int k, int decreasing, int nchunk,
                            uint64_t* partial, int64_t col0, int64_t* idx, double* val, cudaStream_t st, bool fix,
                            const double* med, double c, double alpha, const double* beta) {
  if (S <= 0 || N <= 0) return cudaSuccess;
  if (k < 1 || k > TOPK_MAX || nchunk < 1 || nchunk > 65535) return cudaErrorInvalidValue;
  if ((N + nchunk - 1) / nchunk >= (int64_t)NO_COL) return cudaErrorInvalidValue;  // chunk-relative columns are u32
  if (fix) {
    return k <= 32 ? launch_both<true, true>(x, ld, S, N, k, decreasing, nchunk, partial, col0, idx, val, st, med, c, alpha, beta)
                   : launch_both<true, false>(x, ld, S, N, k, decreasing, nchunk, partial, col0, idx, val, st, med, c, alpha, beta);
  }
  return k <= 32
             ? launch_both<false, true>(x, ld, S, N, k, decreasing, nchunk, partial, col0, idx, val, st, nullptr, 0.0, 1.0, nullptr)
             : launch_both<false, false>(x, ld, S, N, k, decreasing, nchunk, partial, col0, idx, val, st, nullptr, 0.0, 1.0, nullptr);
}

}  // namespace plaidgpu
