// Shared declarations of libplaidgpu (sm_100a only; no CPU fallback anywhere).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/plaidgpu.h"

namespace plaidgpu {

constexpr unsigned FULL = 0xffffffffu;

// ---- value transforms applied when a stored entry of X is loaded -----------------------
// (per stored entry, not per accumulate: the scatter loop only ever sees the result)
enum XformMode : int {
  XF_IDENT = 0,     // plaid(): x
  XF_EXP2 = 1,      // replaid.scse sparse: 2^x on every stored entry (R/plaid.R:165-166)
  XF_EXP2_POS = 2,  // replaid.scse dense: 2^x where x > 0 (R/plaid.R:168-169)
  XF_SING = 3,      // r / a0 - 0.5, a0 = nrow(X)                         (R/plaid.R:216)
  XF_SSGSEA = 4,    // r^(1+a1) / a0 - 0.5, a0 = max(r^(1+a1))            (R/plaid.R:246-251)
  XF_UCELL = 5,     // min(a0 - r, a1), a0 = max(r), a1 = rmax + 1         (R/plaid.R:278)
  XF_AUCELL = 6,    // 1.08 * max((r - (a0 - a1)) / a1, 0), a1 = aucMaxRank (R/plaid.R:306)
  XF_GSVA = 7,      // r / a0, then sign * |.|^(1 + a1) when a1 > 0 (dense only)  (R/plaid.R:352-357)
  XF_SCALE = 8      // v * a0: max-rank -> ecdf value, a0 = 1 / N                 (R/plaid.R:346)
};

struct ScoreParams {
  // X shard (device): CSC (xp/xi/xx) or dense column-major (xx only)
  const int32_t* xp;
  const int32_t* xe;   // optional: end of column j (compacted columns), nullptr -> xp[j + 1]
  const int32_t* xi;
  const double* xx;   // values; for rank scorers the per-entry rank array instead
  const double* r0;   // rank scorers: rank of the zero group per column [N] (else nullptr)
  int32_t P;
  int64_t N;
  // gene-set plan (device): adjacency of every X row, tiled by set range
  const uint32_t* ptr;  // [P * T] 32-byte tile records {u32 overflow offset, u16 length, u16 0, u16 entry[12]}
  const uint16_t* idx;  // overflow entries (lists longer than 12), chunks of 4, padded with 0xFFFF;
                        // an entry is the byte offset (tile-local set id * 8) of the accumulator
  const double* inv;    // [S] epilogue scale per set: 1/(n_s + 1e-8) ("mean") or 1 ("sum")
  const double* ns;     // [S] n_s as double
  int32_t S, T, Ts;
  // transform
  int32_t mode;
  double a0, a1;
  // per-column scale applied in the epilogue (replaid.scse), or nullptr
  const double* colscale;
  // accumulate != 0: add to what `out` already holds (partial sums of an earlier pass);
  // final != 0: apply the epilogue (set scale, zero-group term, column scale); else store raw sums
  int32_t accumulate, final;
  // output, column-major S x N, leading dimension ld
  double* out;
  int64_t ld;
  // optional: order-preserving key (key_of) of the smallest FINAL score written, atomicMin'ed per warp;
  // tells the host which median normalize_medians will need before the statistics pass runs
  unsigned long long* smin;
  const int* run_if;  // optional device flag: the kernel runs only when it is non-zero (fallback after a fixed-point pass)
};

// Gather pass over one block of K genes (the dense-ish part of the product):
//   out[s, j] (+)= sum over members g of set s inside the block of X[g, j]
// with the block's X rows staged DENSE in shared memory for 32 columns at a time and one warp
// per set (lanes = columns), accumulating in registers.
struct GatherParams {
  const int32_t* xp;     // CSC (sparse mode) or nullptr (dense mode)
  const int32_t* xi;
  const double* xx;
  const double* r0;      // rank scorers: zero-group rank per column, else nullptr
  int32_t P;
  int64_t N;
  const uint16_t* dmap;  // sparse mode: X row -> local id in the whole block, 0xFFFF = not in block
  int32_t dlo;           // sparse mode: this pass covers local ids [dlo, dlo + K)
  const int* run_if;     // optional device flag: the pass runs only when it is non-zero
  int32_t g0;            // dense mode: block = rows [g0, g0 + K)
  int32_t K;
  const uint32_t* dptr;  // [S + 1] offsets into didx (multiples of 4)
  const uint32_t* didx;  // byte offsets (local id * 256) of the members' rows in the shared-memory tile; each
                         // set's list is padded to a multiple of 4 with row K (zeros)
  const double* inv;
  const double* ns;
  const double* colscale;
  int32_t S;
  int32_t mode;
  double a0, a1;
  int32_t accumulate, final;
  int32_t nsplit;        // CTAs per column batch (set range split), set by launch_gather
  double* out;
  int64_t ld;
  unsigned long long* smin;  // as in ScoreParams
};

// Tensor-core pass over the block (tc_kernels.cu): out[s, j] = 2^-e_j * sum_g A[s, g] * q[g, j], see there.
struct TcParams {
  const uint4* abits;    // [ceil(S / 128)][Kp / 128][128] membership masks: bit b of row i = gene (kb*128 + b) in set (m*128 + i)
  int32_t kblocks;       // Kp / 128 (set by launch_tc_score)
  int32_t ncell_tiles;   // set by launch_tc_score
  int32_t S;
  int64_t N;
  const double* colinv;  // [N] 2^-e_j: fixed point -> value
  const int* skip_if;    // device flag: non-zero -> the kernel returns at once (non-finite block entries)
  // final != 0 (dense X, no scatter pass follows): apply the score epilogue; else store the partial set sums
  int32_t final, mode;
  double a0, a1;
  const double* r0;
  const double* inv;
  const double* ns;
  const double* colscale;
  double* out;
  int64_t ld;
  unsigned long long* smin;
  // optional (sparse X): int64 fixed-point sums of the rows outside the block, [S][tail_ld] (tail_kernels.cu),
  // added to the block's integer sums before the conversion to fp64; column 0 = the first column of this launch
  const long long* tail;
  int64_t tail_ld;
  const double* colfb;   // [N] f(rank of the zero group) per column (rank scorers on sparse X), or nullptr
  int32_t dbg;           // development switches (PLAIDGPU_TC_DBG): 1 no tail loads, 2 no wait for A, 4 no wait for B
  int32_t small_sums;    // every integer set sum is below 2^51 in magnitude (rows <= 2^20, |q| < 2^30): the fast epilogue's
                         // int64 -> fp64 conversion is an integer add + one DADD instead of I2F.F64.S64
};

struct LaunchCfg {
  int warps;       // warps per CTA
  int ctas;        // persistent grid size
  size_t smem;     // dynamic shared memory per CTA
};

// score_kernels.cu
cudaError_t score_configure(int device, int32_t S, int32_t tile_sets_hint, int32_t* Ts, int32_t* T,
                            LaunchCfg* cfg);
cudaError_t launch_score(const ScoreParams& p, bool dense, const LaunchCfg& cfg, cudaStream_t st);
cudaError_t launch_compact(const int32_t* xp, const int32_t* xi, const double* xx, const uint16_t* dmap, int64_t N,
                           int32_t* oi, double* ox, int32_t* xe, cudaStream_t st);

// gather_kernels.cu
int gather_max_block(int device);  // largest K (genes per block) the shared-memory tile allows
cudaError_t launch_gather(const GatherParams& p, cudaStream_t st);
// colscale[j] = 100 / (sum_i |f(x_ij)| + 1e-8) (kind 1) or 1 / (mean_i |f(x_ij)| + 1e-8) (kind 2)
cudaError_t launch_colabs(const int32_t* xp, const double* xx, int32_t P, int64_t N, int mode, double a0,
                          double a1, int kind, double* colscale, cudaStream_t st);

// tc_kernels.cu — tensor-core (tcgen05, int8 fixed point) pass over the block of high-degree rows / dense X
int tc_cells_per_tile(int slices);
size_t tc_operand_bytes(int64_t N, int Kp, int slices);  // bytes of the digit-row operand Bd
// quantise the block rows of a CSC shard into Bd (+ colinv), compact every other entry for the scatter pass
cudaError_t launch_tc_prep_csc(const int32_t* xp, const int32_t* xi, const double* xx, const double* r0,
                               const uint16_t* dmap, int64_t N, int mode, double a0, double a1, int Kp, int slices,
                               signed char* Bd, double* colinv, int32_t* oi, double* ox, int32_t* xe, int* flag,
                               const int32_t* tmap, uint32_t* tcnt, int32_t Pt, int tileC, double* colfb, cudaStream_t st);
cudaError_t launch_tc_prep_dense(const double* x, int32_t P, int64_t N, int mode, double a0, double a1, int Kp,
                                 int slices, signed char* Bd, double* colinv, int* flag, cudaStream_t st);
cudaError_t launch_tc_score(const TcParams& p, const signed char* Bd, int Kp, int slices, cudaStream_t st);

// tail_kernels.cu — rows of a sparse X outside the tensor-core block: gene-major cell tiles, one warp per (tile, set)
int tail_tile_cells();
cudaError_t launch_fill_u32(void* p, uint32_t v, int64_t n32, cudaStream_t st);  // n32 32-bit words := v, by a kernel
cudaError_t launch_tile_scan(uint32_t* cnt, int32_t Pt, int tiles, uint32_t* rowptr, uint32_t* total, cudaStream_t st);
cudaError_t launch_tile_place(const int32_t* xp, const int32_t* xe, const int32_t* oi, const double* ox, const double* r0,
                              const int32_t* tmap, const double* colinv, int64_t N, int mode, double a0, double a1,
                              int32_t Pt, const uint32_t* rowptr, const uint32_t* total, uint32_t* cnt, uint2* ent,
                              const int* skip_if, cudaStream_t st);
cudaError_t launch_tail(const uint32_t* tptr, const uint16_t* tidx, const int32_t* sorder, const uint32_t* rowptr,
                        const uint32_t* total, const uint2* ent, int32_t S, int32_t Pt, int tiles,
                        long long* tmp, unsigned int* counter, const int* skip_if, cudaStream_t st);

// stats_kernels.cu
// per-column statistics of a dense S x N matrix (ld = leading dimension):
//   med_all[j]: median over non-NaN values (NaN when none)
//   med_nz[j] : median over non-NaN, non-zero values (0 when none)        (R/plaid.R:561-566)
//   colmin[j] : min over non-NaN values (+inf when none)
// d_fail: 1 int, d_list: N int64 of device scratch (columns the single-pass kernel hands to the exact one)
// which: COLSTATS_BOTH, or only one of the medians when the caller already knows which one
// normalize_medians will use (the other array is then left untouched, except for columns that fall back
// to the exact kernel, which always writes both)
enum { COLSTATS_BOTH = 0, COLSTATS_ALL = 1, COLSTATS_NZ = 2 };
bool colstats_small(int32_t S);  // short columns go to the exact kernel, which always yields both medians
cudaError_t launch_colstats(const double* x, int64_t ld, int32_t S, int64_t N, double* med_all,
                            double* med_nz, double* colmin, int* d_fail, int64_t* d_list, int which, cudaStream_t st);
// out[s,j] = alpha * (x[s,j] - med[j] + c) + (beta ? beta[s] : 0); med may be nullptr (then 0)
cudaError_t launch_fixup(const double* x, double* out, int64_t ld, int32_t S, int64_t j0, int64_t j1,
                         const double* med, double c, double alpha, const double* beta,
                         cudaStream_t st);
// per-row sums / sums of squares by column group (plaid.test "lm" for K groups).  cols / seg: the labelled columns
// sorted by (chunk, group), column order kept inside a group; segment g = chunk * K + group is cols[seg[g], seg[g+1])
// (group_stats_plan in api.cu builds them).  partial = nchunk * K * 2 * S doubles of scratch, out = K * 2 * S doubles
// {sum_k[S], sumsq_k[S]} per group; fixed summation order.
// fix: x holds RAW scores and out = moments of alpha * (x - med_j + c) + beta_s, applied on the fly (k_fixup's arithmetic)
cudaError_t launch_group_stats(const double* x, int64_t ld, int32_t S, int K, const int32_t* cols, const int32_t* seg,
                               int nchunk, double* partial, double* out, cudaStream_t st, bool fix = false,
                               const double* med = nullptr, double c = 0.0, double alpha = 1.0, const double* beta = nullptr);
// per-row products with a dense design (plaid.lm): out[(Q + 2) * S] = {sum_j x[s,j] * B[j,q] for q < Q [S each],
// sum_j x[s,j] [S], sum_j x[s,j]^2 [S]}; B is device, column-major N x Q with leading dimension ldb.  Columns are
// split into nchunk chunks as in launch_group_stats (partial = nchunk * (Q + 2) * S doubles of scratch), added in
// ascending order inside a chunk and the chunks in chunk order; one pass over x for every Q (two launches).
// fix: as for launch_group_stats
constexpr int DESIGN_Q_MAX = 64;
cudaError_t launch_design_stats(const double* x, int64_t ld, int32_t S, int64_t N, const double* B, int64_t ldb, int Q,
                                int nchunk, double* partial, double* out, cudaStream_t st, bool fix = false,
                                const double* med = nullptr, double c = 0.0, double alpha = 1.0,
                                const double* beta = nullptr);
// per column of a column-major S x N matrix: the k (1 <= k <= min(S, TOPK_MAX)) rows first in R's
// order(v, decreasing = decreasing) (ties by ascending row, NaN last) into idx / val[k * N] (device, column-major).
// fix: x holds RAW scores and the selection is over alpha * (x - med_j + c) + beta_s (k_fixup's arithmetic)
constexpr int TOPK_MAX = 256;
cudaError_t launch_col_topk(const double* x, int64_t ld, int32_t S, int64_t N, int k, int decreasing, int32_t* idx,
                            double* val, cudaStream_t st, bool fix = false, const double* med = nullptr, double c = 0.0,
                            double alpha = 1.0, const double* beta = nullptr);
// nwords 8-byte words device -> host-mapped (cudaHostAllocMapped) memory by a kernel, bypassing the copy engine
cudaError_t launch_copy_words(const void* src, void* dst_mapped, int64_t nwords, cudaStream_t st);
// global min / max of a device array of n doubles, NaN ignored (na.rm = TRUE); res[0]=min res[1]=max
cudaError_t launch_minmax(const double* x, int64_t n, double* res2, cudaStream_t st);

// rank_kernels.cu
// Column ranks of the stored entries of a CSC matrix.
//   dense_semantics = 0: rank among stored entries only (sparse_colranks, R/plaid.R:631-650)
//   dense_semantics = 1: rank among all P entries of the column with the implicit zeros taking
//                        part as the value 0 (sparseMatrixStats::colRanks, R/plaid.R:605,608);
//                        r0[j] receives the rank of the zero group (also for columns without
//                        implicit zeros: the rank an additional zero would tie into is not
//                        needed then and r0 is set from the stored zeros or 0).
//   is_signed: rank abs(x), multiply by sign(x)                          (R/plaid.R:603-606,637-640)
// rank[nnz] out (may alias nothing), colmax[N] = max |rank| of the column incl. zero group.
cudaError_t launch_rank_csc(const int32_t* xp, const double* xx, int32_t P, int64_t N, int ties,
                            int is_signed, int dense_semantics, double* rank, double* r0,
                            double* colmax, int32_t max_col_nnz, cudaStream_t st);
// Dense column ranks (matrixStats::colRanks, R/plaid.R:614,617): x, rank: P x N column-major.
cudaError_t launch_rank_dense(const double* x, int32_t P, int64_t N, int ties, int is_signed,
                              double* rank, double* colmax, cudaStream_t st);
// expand CSC ranks to a dense P x N matrix, implicit zeros -> r0[j] (or 0 when r0 == nullptr)
cudaError_t launch_expand_ranks(const int32_t* xp, const int32_t* xi, const double* rank,
                                const double* r0, int32_t P, int64_t N, double* dense,
                                cudaStream_t st);
// elementwise transform of a dense matrix with an XformMode (rank scorers on dense input)
cudaError_t launch_xform_dense(const double* in, double* out, int64_t n, int mode, double a0,
                               double a1, cudaStream_t st);
// gsva row z-transform (dense P x N, column-major):
//   launch_row_moments: out[r] = sum_j x[r,j]  (mean == nullptr)  or  sum_j (x[r,j] - mean[r])^2, compensated sums
//   launch_ztransform : z[r,j] = (x[r,j] - mean[r]) / (1e-8 + sd[r])
//   launch_densify    : CSC -> dense (zeros filled)
cudaError_t launch_row_moments(const double* x, int32_t P, int64_t N, const double* mean, double* out, cudaStream_t st);
cudaError_t launch_ztransform(const double* x, int32_t P, int64_t N, const double* mean, const double* sd, double* z,
                              cudaStream_t st);
cudaError_t launch_densify(const int32_t* xp, const int32_t* xi, const double* xx, int32_t P, int64_t N, double* dense,
                           cudaStream_t st);
// out (cols x rows, column-major) = scale * transpose(in (rows x cols, column-major))
cudaError_t launch_transpose(const double* in, int64_t rows, int64_t cols, double scale, double* out, cudaStream_t st);
// max nnz of any column of a device CSC pointer array
cudaError_t launch_max_col_nnz(const int32_t* xp, int64_t N, int32_t* d_res, cudaStream_t st);

// shared device helpers ------------------------------------------------------------------
__device__ __forceinline__ double xform_value(int mode, double v, double a0, double a1) {
  switch (mode) {
    case XF_EXP2: return exp2(v);
    case XF_EXP2_POS: return v > 0.0 ? exp2(v) : v;
    case XF_SING: return v / a0 - 0.5;
    case XF_SSGSEA: return (a1 != 0.0 ? pow(v, 1.0 + a1) : v) / a0 - 0.5;
    case XF_UCELL: return fmin(a0 - v, a1);
    case XF_AUCELL: return 1.08 * fmax((v - (a0 - a1)) / a1, 0.0);
    case XF_SCALE: return v * a0;
    case XF_GSVA: {
      const double r = v / a0;
      return a1 > 0.0 ? copysign(pow(fabs(r), 1.0 + a1), r) * (r == 0.0 ? 0.0 : 1.0) : r;
    }
    default: return v;
  }
}

// epilogue shared by the scatter and gather kernels: raw set sum -> score
__device__ __forceinline__ double score_epilogue(double v, int s, int64_t j, double fb, int mode,
                                                 const double* __restrict__ inv, const double* __restrict__ ns,
                                                 const double* __restrict__ colscale) {
  if (mode >= XF_SING) v += fb * ns[s];
  v *= inv[s];
  if (colscale) v *= colscale[j];
  return v;
}

// order-preserving 64-bit key of a double; -0 and +0 share one key
__device__ __forceinline__ unsigned long long key_of(double v) {
  if (v == 0.0) v = 0.0;
  unsigned long long b = (unsigned long long)__double_as_longlong(v);
  return (b & 0x8000000000000000ull) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double value_of(unsigned long long k) {
  unsigned long long b = (k & 0x8000000000000000ull) ? (k & 0x7fffffffffffffffull) : ~k;
  return __longlong_as_double((long long)b);
}

}  // namespace plaidgpu
