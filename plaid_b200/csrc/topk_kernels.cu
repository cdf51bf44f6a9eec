// Per-column top-k selection with set indices (plaid.topsets: each cell's best gene sets).
//
// One warp per column streams the column once through the warp selection of topk_select.cuh (composite key of the
// value and the row, register list for k <= 32, shared-memory list for k > 32).
// With scores in random order about k ln(S / k) rows of a column pass the test; a column already sorted in the
// selection order merges every batch and stays correct, only slower.
// FIX: the values are RAW scores and the fix-up of plaidgpu_score_finish (k_fixup: alpha * (x + (c - med_j))
// [+ beta_s], the same operations in the same order) is applied in registers, so the selected values are the ones
// plaid() returns.  They are recomputed from x at the selected rows when the list is written out.
#include "topk_select.cuh"

namespace plaidgpu {
namespace {

constexpr int TOPK_WARPS = 8;   // warps (columns) per block
constexpr int TOPK_UNROLL = 8;  // 32-row batches loaded together per warp step
constexpr uint32_t NO_ROW = 0xffffffffu;

using topk::better;
using topk::order_key;
using Entry = topk::Entry<uint32_t>;

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
  topk::SharedList<uint32_t> L;
  int cur = 0;
  Entry list = none;  // k <= 32: lane l holds entry l
  if (!SMALL) L.init(topk_smem + (size_t)w * topk::SharedList<uint32_t>::bytes(k), k, lane, none);
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
        e.idx = (uint32_t)r;
      }
      const unsigned pass = __ballot_sync(FULL, better(e, thr));
      if (!pass) continue;
      if (SMALL) topk::offer_small(e, pass, list, thr, k, lane);
      else topk::offer_large(e, L, cur, thr, k, lane);
    }
  }

  int32_t* ij = idx + j * k;
  double* vj = val + j * k;
  if (SMALL) {
    if (lane < k) {
      ij[lane] = (int32_t)list.idx;
      vj[lane] = fixed<FIX>(xj, list.idx, shift, alpha, beta);
    }
  } else {
    const uint32_t* cr = L.idx + cur * k;
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
  const size_t smem = SMALL ? 0 : (size_t)TOPK_WARPS * topk::SharedList<uint32_t>::bytes(k);
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
