// Per-column top-k selection with set indices (plaid.topsets: each cell's best gene sets).
//
// One warp per column streams the column once.  Every value becomes a composite key (order-preserving u64 of the
// value, then the row index) in which "larger" means "comes first" in R's order(v, decreasing = ...):
//   key = 0 for NaN (after every number, in both directions); otherwise the order-preserving bits of v with -0 mapped
//   to +0, complemented when decreasing = 0.  Equal keys are ordered by ascending row.
// The key alone decides the order, so the result does not depend on the scan order or the launch geometry.
// The warp keeps its current best list and tests every key against the list's k-th entry; only when a lane of a
// 32-row batch beats it (ballot) is the batch sorted (bitonic, by shuffles) and merged into the list:
//   k <= 32: the list is 32 entries in registers, one per lane, merged by a bitonic merge;
//   k > 32:  the list is k entries in shared memory, merged by a parallel merge (binary search of each entry's rank).
// With scores in random order about k ln(S / k) rows of a column pass the test; a column already sorted in the
// selection order merges every batch and stays correct, only slower.
// FIX: the values are RAW scores and the fix-up of plaidgpu_score_finish (k_fixup: alpha * (x + (c - med_j))
// [+ beta_s], the same operations in the same order) is applied in registers, so the selected values are the ones
// plaid() returns.  They are recomputed from x at the selected rows when the list is written out.
#include "common.cuh"

namespace plaidgpu {
namespace {

constexpr int TOPK_WARPS = 8;   // warps (columns) per block
constexpr int TOPK_UNROLL = 8;  // 32-row batches loaded together per warp step
constexpr int TOPK_INSERT_MAX = 8;  // k <= 32: up to this many survivors of a batch are inserted one by one
constexpr uint32_t NO_ROW = 0xffffffffu;

struct Entry {
  uint64_t key;
  uint32_t row;
};

__device__ __forceinline__ bool better(const Entry& a, const Entry& b) {
  return a.key > b.key || (a.key == b.key && a.row < b.row);
}

__device__ __forceinline__ uint64_t order_key(double v, bool decreasing) {
  if (v != v) return 0ull;                                  // NaN: last in both directions
  uint64_t b = v == 0.0 ? 0ull : (uint64_t)__double_as_longlong(v);  // -0 ties with +0
  b = (b >> 63) ? ~b : (b | 0x8000000000000000ull);  // ascending in v, and >= 0x000fffffffffffff (-Inf) > 0
  return decreasing ? b : ~b;                        // ~b <= 0xfff0000000000000 and > 0 as well
}

__device__ __forceinline__ Entry shfl_xor(const Entry& e, int m) {
  Entry p;
  p.key = __shfl_xor_sync(FULL, e.key, m);
  p.row = __shfl_xor_sync(FULL, e.row, m);
  return p;
}

// the 32 entries of a warp, one per lane, sorted best first (lane 0 best)
__device__ __forceinline__ Entry warp_sort(Entry e, int lane) {
#pragma unroll
  for (int size = 2; size <= 32; size <<= 1) {
    const bool first_best = (lane & size) == 0;  // direction of this lane's bitonic block
#pragma unroll
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      const Entry p = shfl_xor(e, stride);
      const bool keep_better = ((lane & stride) == 0) == first_best;
      if (keep_better ? better(p, e) : better(e, p)) e = p;
    }
  }
  return e;
}

// a bitonic sequence of 32 entries -> sorted best first
__device__ __forceinline__ Entry warp_clean(Entry e, int lane) {
#pragma unroll
  for (int stride = 16; stride > 0; stride >>= 1) {
    const Entry p = shfl_xor(e, stride);
    if (((lane & stride) == 0) ? better(p, e) : better(e, p)) e = p;
  }
  return e;
}

template <bool FIX>
__device__ __forceinline__ double fixed(const double* __restrict__ xj, uint32_t r, double shift, double alpha,
                                        const double* __restrict__ beta) {
  double v = xj[r];
  if (FIX) {
    v = __dmul_rn(alpha, __dadd_rn(v, shift));
    if (beta) v = __dadd_rn(v, beta[r]);
  }
  return v;
}

// SMALL: k <= 32, list in registers; otherwise k <= 256 with 2 * k + 32 entries of shared memory per warp
template <bool FIX, bool SMALL>
__global__ void __launch_bounds__(TOPK_WARPS * 32) k_col_topk(const double* __restrict__ x, int64_t ld, int32_t S,
                                                              int64_t N, int k, int decreasing, int32_t* __restrict__ idx,
                                                              double* __restrict__ val, const double* __restrict__ med,
                                                              double c, double alpha, const double* __restrict__ beta) {
  extern __shared__ unsigned char topk_smem[];
  const int lane = threadIdx.x & 31;
  const int w = threadIdx.x >> 5;
  const int64_t j = (int64_t)blockIdx.x * TOPK_WARPS + w;
  if (j >= N) return;  // whole warps leave together
  const bool dec = decreasing != 0;
  const double* __restrict__ xj = x + j * ld;
  const double shift = FIX ? (med ? -med[j] : 0.0) + c : 0.0;
  const Entry none{0ull, NO_ROW};  // worse than every real entry, NaN included

  // k > 32: two lists of k entries (current, next) and the 32 entries of the batch being merged
  uint64_t* lkey = nullptr;
  uint32_t* lrow = nullptr;
  uint64_t* bkey = nullptr;
  uint32_t* brow = nullptr;
  int cur = 0;
  Entry list = none;  // k <= 32: lane l holds entry l
  if (!SMALL) {
    unsigned char* base = topk_smem + (size_t)w * (2 * k + 32) * 12;
    lkey = reinterpret_cast<uint64_t*>(base);
    bkey = lkey + 2 * k;
    lrow = reinterpret_cast<uint32_t*>(bkey + 32);
    brow = lrow + 2 * k;
    for (int i = lane; i < k; i += 32) {
      lkey[i] = none.key;
      lrow[i] = none.row;
    }
    __syncwarp();
  }
  Entry thr = none;  // the list's k-th entry: a row must beat it to enter

  for (int32_t r0 = 0; r0 < S; r0 += 32 * TOPK_UNROLL) {
    double v[TOPK_UNROLL];
#pragma unroll
    for (int u = 0; u < TOPK_UNROLL; ++u) {
      const int32_t r = r0 + u * 32 + lane;
      v[u] = r < S ? __ldcs(xj + r) : 0.0;
    }
#pragma unroll
    for (int u = 0; u < TOPK_UNROLL; ++u) {
      const int32_t r = r0 + u * 32 + lane;
      Entry e = none;
      if (r < S) {
        double t = v[u];
        if (FIX) {
          t = __dmul_rn(alpha, __dadd_rn(t, shift));
          if (beta) t = __dadd_rn(t, beta[r]);
        }
        e.key = order_key(t, dec);
        e.row = (uint32_t)r;
      }
      unsigned pass = __ballot_sync(FULL, better(e, thr));
      if (!pass) continue;
      if (SMALL && __popc(pass) <= TOPK_INSERT_MAX) {
        // a few survivors (the common case once the list has filled): insert them one by one, each a broadcast and a
        // shift of the list by one lane, instead of sorting and merging the whole batch
        do {
          const int src = __ffs(pass) - 1;
          pass &= pass - 1;
          const Entry s{__shfl_sync(FULL, e.key, src), __shfl_sync(FULL, e.row, src)};
          const unsigned worse = __ballot_sync(FULL, better(s, list));  // a suffix of the sorted list
          const int pos = __ffs(worse) - 1;
          const Entry up{__shfl_up_sync(FULL, list.key, 1), __shfl_up_sync(FULL, list.row, 1)};
          if (worse && lane >= pos) list = lane == pos ? s : up;
        } while (pass);
        thr.key = __shfl_sync(FULL, list.key, k - 1);
        thr.row = __shfl_sync(FULL, list.row, k - 1);
        continue;
      }
      e = warp_sort(e, lane);
      if (SMALL) {
        const Entry o = shfl_xor(e, 31);  // batch reversed: list + reversed batch is bitonic after the max below
        list = warp_clean(better(list, o) ? list : o, lane);
        thr.key = __shfl_sync(FULL, list.key, k - 1);
        thr.row = __shfl_sync(FULL, list.row, k - 1);
      } else {
        const uint64_t* ck = lkey + cur * k;
        const uint32_t* cr = lrow + cur * k;
        uint64_t* nk = lkey + (cur ^ 1) * k;
        uint32_t* nr = lrow + (cur ^ 1) * k;
        bkey[lane] = e.key;
        brow[lane] = e.row;
        __syncwarp();
        // batch entry `lane`: its rank in the batch plus the list entries that are better or equal (list first on
        // ties; only the shared placeholder rows can tie)
        int lo = 0, hi = k;
        while (lo < hi) {
          const int mid = (lo + hi) >> 1;
          const Entry m{ck[mid], cr[mid]};
          if (!better(e, m)) lo = mid + 1;
          else hi = mid;
        }
        if (lane + lo < k) {
          nk[lane + lo] = e.key;
          nr[lane + lo] = e.row;
        }
        // list entry i: its rank in the list plus the batch entries strictly better
        for (int i = lane; i < k; i += 32) {
          const Entry m{ck[i], cr[i]};
          int a = 0, b = 32;
          while (a < b) {
            const int mid = (a + b) >> 1;
            if (better(Entry{bkey[mid], brow[mid]}, m)) a = mid + 1;
            else b = mid;
          }
          if (i + a < k) {
            nk[i + a] = m.key;
            nr[i + a] = m.row;
          }
        }
        __syncwarp();
        cur ^= 1;
        thr.key = nk[k - 1];
        thr.row = nr[k - 1];
      }
    }
  }

  int32_t* ij = idx + j * k;
  double* vj = val + j * k;
  if (SMALL) {
    if (lane < k) {
      ij[lane] = (int32_t)list.row;
      vj[lane] = fixed<FIX>(xj, list.row, shift, alpha, beta);
    }
  } else {
    const uint32_t* cr = lrow + cur * k;
    for (int i = lane; i < k; i += 32) {
      const uint32_t r = cr[i];
      ij[i] = (int32_t)r;
      vj[i] = fixed<FIX>(xj, r, shift, alpha, beta);
    }
  }
}

template <bool FIX, bool SMALL>
cudaError_t launch_one(const double* x, int64_t ld, int32_t S, int64_t N, int k, int decreasing, int32_t* idx,
                       double* val, cudaStream_t st, const double* med, double c, double alpha, const double* beta) {
  const size_t smem = SMALL ? 0 : (size_t)TOPK_WARPS * (2 * k + 32) * 12;
  if (!SMALL) {
    cudaError_t e = cudaFuncSetAttribute(k_col_topk<FIX, SMALL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  const unsigned grid = (unsigned)((N + TOPK_WARPS - 1) / TOPK_WARPS);
  k_col_topk<FIX, SMALL><<<grid, TOPK_WARPS * 32, smem, st>>>(x, ld, S, N, k, decreasing, idx, val, med, c, alpha, beta);
  return cudaGetLastError();
}

}  // namespace

cudaError_t launch_col_topk(const double* x, int64_t ld, int32_t S, int64_t N, int k, int decreasing, int32_t* idx,
                            double* val, cudaStream_t st, bool fix, const double* med, double c, double alpha,
                            const double* beta) {
  if (N <= 0) return cudaSuccess;
  if (k < 1 || k > TOPK_MAX || k > S) return cudaErrorInvalidValue;
  if (fix) {
    return k <= 32 ? launch_one<true, true>(x, ld, S, N, k, decreasing, idx, val, st, med, c, alpha, beta)
                   : launch_one<true, false>(x, ld, S, N, k, decreasing, idx, val, st, med, c, alpha, beta);
  }
  return k <= 32 ? launch_one<false, true>(x, ld, S, N, k, decreasing, idx, val, st, nullptr, 0.0, 1.0, nullptr)
                 : launch_one<false, false>(x, ld, S, N, k, decreasing, idx, val, st, nullptr, 0.0, 1.0, nullptr);
}

}  // namespace plaidgpu
