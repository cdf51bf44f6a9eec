/*
 * plaidgpu.h — C ABI of libplaidgpu.so, the B200 (sm_100a) implementation of the
 * bigomics/plaid gene-set scoring hot path.
 *
 * This is the drop-in boundary.  The reference (a pure-R package) has NO native
 * boundary of its own (no src/, no .Call, no useDynLib — reference NAMESPACE:1-16); its
 * hot path runs inside Matrix / matrixStats / sparseMatrixStats.  Each entry point
 * below therefore cites the reference R function (file:line under the reference
 * repository) whose arithmetic it replaces; the R `.Call` shim that binds them is in
 * rpkg/src/shim.c and is shown in INTEGRATION.md.
 *
 * Conventions
 *   - plain C types only; no C++ exceptions cross this boundary;
 *   - every function returns PLAIDGPU_OK (0) or a negative status; the message is
 *     available from plaidgpu_last_error(ctx);
 *   - the caller owns every input and output buffer; inputs are never written;
 *   - matrices follow R: CSC = dgCMatrix slots (p int32[N+1], i int32[nnz] 0-based rows
 *     sorted within a column, x double[nnz]); dense = column-major double;
 *   - a buffer may live in host memory (PLAIDGPU_HOST) or in device memory of the
 *     context's GPU (PLAIDGPU_DEVICE); the latter is what device-resident pipelines and
 *     the roofline benchmark use;
 *   - one context drives ONE GPU.  Samples (columns) shard across GPUs with one
 *     context (and normally one process) per GPU; the handful of cross-shard scalars are
 *     exchanged through the *_begin / *_finish pair (see plaidgpu_score_begin).
 */
#ifndef PLAIDGPU_H
#define PLAIDGPU_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PLAIDGPU_VERSION 100

/* status codes */
#define PLAIDGPU_OK 0
#define PLAIDGPU_ERR_ARG (-1)      /* bad argument */
#define PLAIDGPU_ERR_CUDA (-2)     /* CUDA runtime failure (no usable GPU, OOM, launch error) */
#define PLAIDGPU_ERR_NOOVERLAP (-3)/* no row of X maps to a gene-set row (reference: message + NULL, R/plaid.R:66-69) */
#define PLAIDGPU_ERR_STATE (-4)    /* call order violated (e.g. score before set_genesets) */
#define PLAIDGPU_ERR_NOMEM (-5)    /* host allocation failure */

/* memory location of a caller buffer */
#define PLAIDGPU_HOST 0
#define PLAIDGPU_DEVICE 1

/* matrix kinds */
#define PLAIDGPU_CSC 0
#define PLAIDGPU_DENSE 1

/* scorers: which reference function the call reproduces */
#define PLAIDGPU_PLAID 0   /* plaid()            R/plaid.R:60-87   */
#define PLAIDGPU_SCSE 1    /* replaid.scse()     R/plaid.R:155-190 */
#define PLAIDGPU_SING 2    /* replaid.sing()     R/plaid.R:213-219 */
#define PLAIDGPU_SSGSEA 3  /* replaid.ssgsea()   R/plaid.R:244-255 */
#define PLAIDGPU_UCELL 4   /* replaid.ucell()    R/plaid.R:276-282 */
#define PLAIDGPU_AUCELL 5  /* replaid.aucell()   R/plaid.R:304-309 */
#define PLAIDGPU_GSVA 6    /* replaid.gsva()     R/plaid.R:338-363 */

#define PLAIDGPU_ROWTF_Z 0
#define PLAIDGPU_ROWTF_ECDF 1
#define PLAIDGPU_ROWTF_DONE 2

/* ties.method of base::rank / colRanks (R/plaid.R:589-650) */
#define PLAIDGPU_TIES_AVERAGE 0
#define PLAIDGPU_TIES_MIN 1
#define PLAIDGPU_TIES_MAX 2
/* order-of-appearance methods of base::rank / matrixStats::colRanks: stored-entry ranks (keep_zero = 1) and dense input
 * only — sparseMatrixStats::colRanks (sparse input, keep_zero = 0) knows max / average / min alone.  "random" draws from
 * R's RNG and stays an error. */
#define PLAIDGPU_TIES_FIRST 3
#define PLAIDGPU_TIES_LAST 4
#define PLAIDGPU_TIES_DENSE 5 /* matrixStats only: consecutive ranks of the distinct values */

typedef struct plaidgpu_ctx plaidgpu_ctx;

/* gene x sample input matrix (X of plaid(X, matG)) */
typedef struct plaidgpu_matrix {
  int32_t kind;      /* PLAIDGPU_CSC or PLAIDGPU_DENSE */
  int32_t location;  /* PLAIDGPU_HOST or PLAIDGPU_DEVICE (applies to p, i, x alike) */
  int32_t P;         /* rows (genes) */
  int32_t _pad;
  int64_t N;         /* columns (samples / cells) */
  const int32_t* p;  /* CSC: column pointers [N+1]; DENSE: NULL */
  const int32_t* i;  /* CSC: row indices [nnz];     DENSE: NULL */
  const double* x;   /* CSC: values [nnz];          DENSE: column-major [P*N] */
} plaidgpu_matrix;

/* options of one scoring call; zero-initialise, then plaidgpu_default_opts() */
typedef struct plaidgpu_opts {
  int32_t scorer;        /* PLAIDGPU_PLAID ... */
  int32_t stats_mean;    /* plaid(stats=): 1 "mean" (default), 0 "sum"            R/plaid.R:74-77 */
  int32_t normalize;     /* plaid(normalize=): median-normalise the scores       R/plaid.R:83   */
  int32_t ignore_zero;   /* normalize_medians(ignore.zero=): -1 auto (min==0), 0, 1  R/plaid.R:556-557 */
  int32_t remove_log2;   /* replaid.scse(removeLog2=): -1 auto, 0, 1             R/plaid.R:160-161 */
  int32_t score_mean;    /* replaid.scse(scoreMean=)                             R/plaid.R:172-182 */
  int32_t out_location;  /* where `out` lives: PLAIDGPU_HOST / PLAIDGPU_DEVICE */
  int32_t tile_sets;     /* 0 = auto; gene sets per shared-memory accumulator tile (tuning) */
  double alpha;          /* replaid.ssgsea(alpha=)                               R/plaid.R:246-250 */
  double rmax;           /* replaid.ucell(rmax=), default 1500                   R/plaid.R:276    */
  double auc_max_rank;   /* replaid.aucell(aucMaxRank=); <=0 -> ceiling(0.05*P)  R/plaid.R:304    */
  double tau;            /* replaid.gsva(tau=)                                   R/plaid.R:354-357 */
  /* (gsva_ecdf below selects rowtf = "ecdf") */
  int64_t nrow_x;        /* nrow(X) used by replaid.sing (rX / nrow(X)); 0 -> X.P  R/plaid.R:216 */
  const double* matg_full_colsums; /* ucell: colSums(matG != 0) over ALL rows of matG [S] (host);
                                      NULL -> taken from plaidgpu_set_genesets      R/plaid.R:280 */
  const double* row_mean;  /* gsva: rowMeans(X) over ALL samples of ALL shards [P] (host); NULL -> this shard only */
  const double* row_sd;    /* gsva: rowSds(X) (sample SD, n-1) [P] (host); NULL -> this shard only  R/plaid.R:343 */
  int32_t gsva_ecdf;       /* gsva row transform: PLAIDGPU_ROWTF_Z (0) = rowtf "z"; PLAIDGPU_ROWTF_ECDF (1) = rowtf
                              "ecdf", per-gene ECDF across the samples of THIS call (one shard holds all
                              samples, R/plaid.R:344-346); PLAIDGPU_ROWTF_DONE (2) = X already holds the
                              row-transformed values (column shards: plaidgpu_row_ecdf after the
                              column -> row exchange, see plaid_b200/sharded.py gsva_shard) */
  int32_t exact_fp64;      /* 0 (default): the block of high-degree rows (sparse X) / every row (dense X) is scored on
                              the tensor cores in per-column 30-bit fixed point with exact integer accumulation
                              (|error| <= 2^-31 * max|x_gj| per term, see plaid_b200/csrc/tc_kernels.cu);
                              1: every add in fp64 (gather + scatter passes only) */
} plaidgpu_opts;

/* cross-shard scalars.  Produced per shard by *_begin (local values), combined by the
 * caller over all shards (min / max / sum as named), and handed back to *_finish.
 * With a single shard pass the struct through unchanged (plaidgpu_score does). */
typedef struct plaidgpu_scalars {
  double x_min;        /* min(X) incl. implicit zeros   (combine: min)  scse auto removeLog2 */
  double x_max;        /* max(X) incl. implicit zeros   (combine: max) */
  double rank_max;     /* max(rX) / max(abs(rX))        (combine: max)  R/plaid.R:251,278,306,352 */
  double score_min;    /* min(raw scores, na.rm)        (combine: min)  R/plaid.R:557 */
  double med_mean;     /* mean(medx): OUTPUT of the combine step, see plaidgpu_combine_medians */
  int32_t ignore_zero; /* resolved flag (0/1) after combine */
  int32_t _pad;
} plaidgpu_scalars;

/* ---- lifecycle ---------------------------------------------------------------- */

/* Create a context on CUDA device `device`.  Fails (PLAIDGPU_ERR_CUDA) when no usable
 * sm_100 GPU is present: there is NO CPU fallback. */
int plaidgpu_init(int device, plaidgpu_ctx** ctx);
void plaidgpu_destroy(plaidgpu_ctx* ctx);
const char* plaidgpu_last_error(const plaidgpu_ctx* ctx);
int plaidgpu_version(void);
void plaidgpu_default_opts(plaidgpu_opts* o);

/* ---- gene sets ------------------------------------------------------------------ */

/* matG as a CSC pattern (P_G genes x S sets): Gp int32[S+1], Gi int32[nnzG] (host).  Gx may
 * be NULL (all stored entries count) or the stored values, in which case exact zeros are
 * dropped like `1*(matG != 0)` (R/plaid.R:73).  The library keeps its own copy. */
int plaidgpu_set_genesets(plaidgpu_ctx* ctx, int32_t P_G, int32_t S, const int32_t* Gp,
                          const int32_t* Gi, const double* Gx);

/* ---- scoring (the hot path) ----------------------------------------------------- */

/* One-shot, single shard.  rowmap: int32[X.P] (host), rowmap[r] = row of matG that X row r
 * aligns with, or -1 (the result of R's intersect/match on rownames, R/plaid.R:65-72;
 * at most one X row may map to a given matG row).  out: S x N column-major doubles.
 * Replaces, per opts.scorer: plaid / replaid.* (R/plaid.R:60-87,155-363) including
 * chunked_crossprod (R/plaid.R:100-123), normalize_medians (:554-575) and the ranking
 * (:589-650) those call. */
int plaidgpu_score(plaidgpu_ctx* ctx, const plaidgpu_matrix* X, const int32_t* rowmap,
                   const plaidgpu_opts* opts, double* out);

/* The same call over n devices from ONE host process (an R session): ctxs[0..n) are contexts on
 * different devices, each with the same gene sets registered.  X and out are HOST buffers; the
 * columns are split into n contiguous shards (the loop axis of chunked_crossprod, R/plaid.R:110-119),
 * one host thread drives each context, every shard's block lands directly in `out`, and the
 * cross-shard scalars (min / max of X, max rank, min score, the column medians and their mean,
 * gsva row means / SDs) are combined on the host in column order, so the result equals the
 * single-context one bit for bit.  gsva rowtf = "ecdf" needs one context. */
int plaidgpu_score_multi(plaidgpu_ctx* const* ctxs, int n, const plaidgpu_matrix* X,
                         const int32_t* rowmap, const plaidgpu_opts* opts, double* out);

/* Sharded protocol (columns of X split over several contexts / GPUs / processes):
 *   1. every shard: plaidgpu_score_begin(ctx, X_shard, rowmap, opts, &local)
 *        uploads / ranks the shard and reports x_min, x_max, rank_max;
 *   2. caller combines x_min (min), x_max (max), rank_max (max) over shards;
 *   3. every shard: plaidgpu_score_compute(ctx, &combined, out)
 *        runs the score kernel; reports score_min and leaves per-column medians in the
 *        context (plaidgpu_get_col_medians).  `out` is the buffer later given to
 *        plaidgpu_score_finish: with out_location == PLAIDGPU_DEVICE the raw scores are written
 *        straight into it (no second copy of the S x N matrix exists); with PLAIDGPU_HOST it
 *        may be NULL here;
 *   4. if opts.normalize: caller combines score_min (min), gathers the medians of all shards
 *        in column order and calls plaidgpu_combine_medians() once to get med_mean /
 *        ignore_zero (bit-identical for any shard count);
 *   5. every shard: plaidgpu_score_finish(ctx, &combined, out) applies the normalisation
 *        and scorer epilogue and delivers `out` (S x N_shard, host or device). */
int plaidgpu_score_begin(plaidgpu_ctx* ctx, const plaidgpu_matrix* X, const int32_t* rowmap,
                         const plaidgpu_opts* opts, plaidgpu_scalars* local);
int plaidgpu_score_compute(plaidgpu_ctx* ctx, plaidgpu_scalars* scal, double* out);
/* per-column medians of the raw scores of this shard: med_all (NaN dropped) and med_nz
 * (NaN and zeros dropped, all-dropped -> 0); each double[N_shard] (host). */
int plaidgpu_get_col_medians(plaidgpu_ctx* ctx, double* med_all, double* med_nz);
/* The one median vector normalize_medians will use once the global flag is known: ignore_zero != 0 ->
 * medians over the non-zero scores, else over all scores; med: host double[N of this shard].  The library
 * computes up front only the median its own shard's minimum predicts (min > 0: no zeros, both coincide;
 * min < 0: plain; min == 0: non-zero) and computes the other one here on demand — which only happens when
 * this shard's minimum is 0 and another shard holds a negative score.  plaidgpu_get_col_medians (both
 * vectors) stays available and fills in whatever is missing the same way.  Call before *_finish. */
int plaidgpu_get_col_medians_for(plaidgpu_ctx* ctx, int ignore_zero, double* med);

/* ignore_zero_opt: -1 auto from score_min; med_* over ALL columns of ALL shards in order.
 * Writes scal->ignore_zero and scal->med_mean (= R mean(medx, na.rm=TRUE)). */
int plaidgpu_combine_medians(int ignore_zero_opt, double score_min, const double* med_all,
                             const double* med_nz, int64_t N_total, plaidgpu_scalars* scal);
int plaidgpu_score_finish(plaidgpu_ctx* ctx, const plaidgpu_scalars* scal, double* out);

/* Tiled egress (scope row f4): the same scores, written to `path` column tile by column tile so that the
 * S x N result never has to fit in host memory (30k sets x 1M cells = 240 GB).  X must be in host
 * memory; a normalised call makes two passes over X (medians, then scores) exactly like the chunked
 * plaidgpu_score path, and the bytes written equal what plaidgpu_score returns.
 *   PLAIDGPU_FILE_RAW: S*N doubles, column-major;  PLAIDGPU_FILE_NPY: NumPy .npy (fortran_order). */
#define PLAIDGPU_FILE_RAW 0
#define PLAIDGPU_FILE_NPY 1
int plaidgpu_score_to_file(plaidgpu_ctx* ctx, const plaidgpu_matrix* X, const int32_t* rowmap,
                           const plaidgpu_opts* opts, const char* path, int format);

/* t(x) %*% y with x = the gene sets registered by plaidgpu_set_genesets, optionally
 * column-scaled (colscale double[S] or NULL): chunked_crossprod(x, y) (R/plaid.R:100-123).
 * y is X restricted/ordered by rowmap as in plaidgpu_score.  out: S x N dense. */
int plaidgpu_crossprod(plaidgpu_ctx* ctx, const plaidgpu_matrix* Y, const int32_t* rowmap,
                       const double* colscale, int out_location, double* out);

/* Per-row sums across the columns of this shard, for replaid.gsva's row z-transform
 * (rowMeans / rowSds, R/plaid.R:343,365-370) when X is column-sharded:
 *   mean == NULL : out[r] = sum_j X[r, j]
 *   mean != NULL : out[r] = sum_j (X[r, j] - mean[r])^2     (mean: host double[P])
 * The caller adds the shards' vectors, divides by N_total (resp. N_total - 1, sqrt) and passes the
 * results as opts.row_mean / opts.row_sd.  out: host double[P]. */
int plaidgpu_row_moments(plaidgpu_ctx* ctx, const plaidgpu_matrix* X, const double* mean, double* out);

/* replaid.gsva(rowtf = "ecdf") on column shards (R/plaid.R:346: apply(X, 1, function(x) ecdf(x)(x))).
 * The ECDF of a gene runs ACROSS samples, the one axis the path is sharded on, so the shards exchange
 * (all-to-all) their dense blocks into row blocks first.  x: N x rows col-major, i.e. the N samples of
 * every gene of this rank's row block are contiguous; replaced in place by
 * #{samples with value <= x} / N.  The caller exchanges the result back and scores the shard with
 * opts.gsva_ecdf = PLAIDGPU_ROWTF_DONE.  location: where x lives. */
int plaidgpu_row_ecdf(plaidgpu_ctx* ctx, double* x, int64_t N, int32_t rows, int location);

/* ---- ranking ---------------------------------------------------------------------- */

/* colranks(X, signed, keep.zero, ties.method) (R/plaid.R:589-623).
 *   CSC input, keep_zero=1: sparse_colranks (R/plaid.R:631-650) — out double[nnz], ranks of the
 *     stored entries in storage order (pattern unchanged);
 *   CSC input, keep_zero=0: dense P x N ranks over all entries incl. implicit zeros
 *     (t(sparseMatrixStats::colRanks), :605,608) — out double[P*N];
 *   DENSE input: t(matrixStats::colRanks) (:614,617) — out double[P*N].
 * NaN -> NaN.  out lives where out_location says. */
int plaidgpu_colranks(plaidgpu_ctx* ctx, const plaidgpu_matrix* X, int ties, int is_signed,
                      int keep_zero, int out_location, double* out);

/* ---- median normalisation --------------------------------------------------------- */

/* normalize_medians(x, ignore.zero) (R/plaid.R:554-575) on a dense S x N matrix, in place
 * semantics expressed as in -> out (may alias).  ignore_zero: -1 auto, 0, 1. */
int plaidgpu_normalize_medians(plaidgpu_ctx* ctx, const double* x, int32_t S, int64_t N,
                               int ignore_zero, int location, double* out);

/* ---- differential enrichment on the scores ("next" row f1 of the scope table) ------------- */

/* Per gene set (row of the S x N score matrix) the sums and sums of squares over the samples of each
 * group y[j] in {0, 1}: the reductions behind plaid.test(tests = "lm") (Rfast::ttests on t(gsetX),
 * reference R/plaid.R:429-431).  x: S x N column-major doubles at `location`; y: host int32[N];
 * out: host double[4 * S] = {sum0[S], sumsq0[S], sum1[S], sumsq1[S]}.  Columns are added in a fixed
 * order, so results are bit-reproducible.  The t statistics / p-values stay on the host (stats::pt). */
int plaidgpu_group_moments(plaidgpu_ctx* ctx, const double* x, int32_t S, int64_t N, const int32_t* y,
                           int location, double* out);

/* The same reductions FUSED onto the scoring call (row f1 as SURVEY.md states it): scores X like plaidgpu_score
 * (HOST or DEVICE X), then reduces the (median-normalised) scores per set and sample group in one pass over the raw
 * scores still on the device — the normalisation is applied in registers, the S x N matrix is neither written in
 * its final form nor copied to the host; 4 * S doubles come back (layout as above).  Equal, bit for bit, to
 * plaidgpu_score followed by plaidgpu_group_moments.  Replaces R/plaid.R:423-431 (plaid() + Rfast::ttests). */
int plaidgpu_score_group_moments(plaidgpu_ctx* ctx, const plaidgpu_matrix* X, const int32_t* rowmap,
                                 const plaidgpu_opts* opts, const int32_t* y, double* out);

/* Per gene set the sums and sums of squares over the samples of each of K groups: the reductions behind
 * plaid.test(tests = "lm") when every cluster is compared with the rest (one pass over the scores, whatever K is).
 * x: S x N column-major doubles at `location`; labels: host int32[N], labels[j] in [0, K) is the group of sample j and
 * -1 leaves it out; out: host double[K * 2 * S] = {sum_k[S], sumsq_k[S]} for k = 0 .. K-1 (an empty group gives
 * zeros).  Columns are added in a fixed order, so results are bit-reproducible; with K = 2 and labels y != 0 they
 * equal plaidgpu_group_moments bit for bit.  K < 1 or a label outside [-1, K) is PLAIDGPU_ERR_ARG. */
int plaidgpu_group_stats(plaidgpu_ctx* ctx, const double* x, int32_t S, int64_t N, const int32_t* labels, int K,
                         int location, double* out);

/* The same reductions fused onto the scoring call, for any scorer and option plaidgpu_score accepts: the scores stay
 * on the device as raw scores and are normalised in registers while reducing; K * 2 * S doubles come back (layout as
 * above).  Equal, bit for bit, to plaidgpu_score followed by plaidgpu_group_stats.  When X is in host memory and the
 * S x N scores exceed the device, the columns are scored in tiles (a normalised call makes two passes over X like
 * plaidgpu_score: medians first, then scores reduced tile by tile) and the tiles' moments are added in tile order.
 * plaidgpu_score_group_moments is this call with K = 2. */
int plaidgpu_score_group_stats(plaidgpu_ctx* ctx, const plaidgpu_matrix* X, const int32_t* rowmap,
                               const plaidgpu_opts* opts, const int32_t* labels, int K, double* out);

/* plaidgpu_score_group_stats over n devices from ONE host process, split like plaidgpu_score_multi (X in host memory,
 * one host thread per context, scalars and medians combined on the host in column order); every shard reduces its
 * own scores and the shards' moments are added in shard order.  Each shard's scores must fit its device. */
int plaidgpu_score_group_stats_multi(plaidgpu_ctx* const* ctxs, int n, const plaidgpu_matrix* X, const int32_t* rowmap,
                                     const plaidgpu_opts* opts, const int32_t* labels, int K, double* out);

/* Per gene set the products of its scores with the columns of a dense design basis, and its sum and sum of squares:
 * the reductions behind plaid.lm (ordinary least squares of every set's scores on a design; the host takes a thin
 * QR D = U R of the design and passes B = U).  x: S x N column-major doubles at `location`; B: host double,
 * column-major N x Q (ld = N); 1 <= Q <= 64, every entry finite.  out: host double[(Q + 2) * S] =
 * {sum_j x[s,j]*B[j,q] for q < Q [S each], sum_j x[s,j] [S], sum_j x[s,j]^2 [S]}.  Columns are added in a fixed
 * order: bit-reproducible.  Q outside [1, 64], a null pointer or a non-finite entry of B is PLAIDGPU_ERR_ARG.
 * Kernel time: plaidgpu_last_kernel_ms(ctx, 2). */
int plaidgpu_design_stats(plaidgpu_ctx* ctx, const double* x, int32_t S, int64_t N, const double* B, int Q,
                          int location, double* out);

/* The same reductions fused onto the scoring call, for any scorer and option plaidgpu_score accepts: the scores stay
 * on the device as raw scores and are normalised in registers while reducing; (Q + 2) * S doubles come back (layout
 * as above, B has X->N rows).  Equal, bit for bit, to plaidgpu_score followed by plaidgpu_design_stats.  When X is in
 * host memory and the S x N scores exceed the device, the columns are scored in tiles (two passes over X when
 * normalised, like plaidgpu_score), each tile uploads only its own rows of B, and the tiles' moments are added in
 * tile order. */
int plaidgpu_score_design_stats(plaidgpu_ctx* ctx, const plaidgpu_matrix* X, const int32_t* rowmap,
                                const plaidgpu_opts* opts, const double* B, int Q, double* out);

/* plaidgpu_score_design_stats over n devices from ONE host process, split like plaidgpu_score_multi: shard r reduces
 * its own scores with rows [lo_r, hi_r) of B and the shards' moments are added in shard order.  Each shard's scores
 * must fit its device.  The same context twice, or gsva rowtf = "ecdf" with n > 1, is PLAIDGPU_ERR_ARG. */
int plaidgpu_score_design_stats_multi(plaidgpu_ctx* const* ctxs, int n, const plaidgpu_matrix* X,
                                      const int32_t* rowmap, const plaidgpu_opts* opts, const double* B, int Q,
                                      double* out);

/* Per column of a dense S x N matrix at `location`: the k largest (decreasing = 1) or smallest values and their row
 * indices, i.e. the first k entries of R's order(v, decreasing = decreasing): ties (fp64 ==, so -0 == +0) by
 * ascending row, NaN last in both directions and by ascending row.  idx int32[k * N] (0-based rows) and val
 * double[k * N] (val = v[idx] bit for bit), host, column-major: entry t of column j at t + k * j.
 * 1 <= k <= min(S, 256), otherwise PLAIDGPU_ERR_ARG; N = 0 does nothing.  Kernel time: plaidgpu_last_kernel_ms(, 2). */
int plaidgpu_col_topk(plaidgpu_ctx* ctx, const double* x, int32_t S, int64_t N, int k, int decreasing,
                      int location, int32_t* idx, double* val);

/* The same fused onto the scoring call, for any scorer and option plaidgpu_score accepts: the scores stay on the
 * device as raw scores and are normalised in registers while selecting; k * N indices and values come back.  Equal,
 * bit for bit, to plaidgpu_score followed by plaidgpu_col_topk.  When X is in host memory and the S x N scores exceed
 * the device, the columns are scored in tiles (two passes over X when normalised, like plaidgpu_score), each tile
 * writing its own columns of idx / val. */
int plaidgpu_score_topk(plaidgpu_ctx* ctx, const plaidgpu_matrix* X, const int32_t* rowmap, const plaidgpu_opts* opts,
                        int k, int decreasing, int32_t* idx, double* val);

/* plaidgpu_score_topk over n devices from ONE host process, split like plaidgpu_score_multi: shard r writes columns
 * [lo_r, hi_r) of idx / val, and nothing is combined.  Each shard's scores must fit its device.  The same context
 * twice, or gsva rowtf = "ecdf" with n > 1, is PLAIDGPU_ERR_ARG. */
int plaidgpu_score_topk_multi(plaidgpu_ctx* const* ctxs, int n, const plaidgpu_matrix* X, const int32_t* rowmap,
                              const plaidgpu_opts* opts, int k, int decreasing, int32_t* idx, double* val);

/* ---- gene-set ingestion ("next" row f2): host-side, no GPU needed -------------------------- */

/* read.gmt() + gmt2mat() with default arguments (reference R/gmt-utils.R:99-125, 19-66): a GMT text
 * (name <tab> source <tab> genes...) becomes the genes x sets incidence matrix in gmt2mat's order (sets by
 * decreasing size, duplicated set names dropped; genes by decreasing membership count, ties by name in
 * byte order - R uses the session collation, which only permutes rows and never changes a score). */
typedef struct plaidgpu_gmt plaidgpu_gmt;
int plaidgpu_gmt_read(const char* path, plaidgpu_gmt** out);
int plaidgpu_gmt_from_buffer(const char* text, int64_t len, plaidgpu_gmt** out);
void plaidgpu_gmt_free(plaidgpu_gmt* g);
int64_t plaidgpu_gmt_num_sets(const plaidgpu_gmt* g);
int64_t plaidgpu_gmt_num_genes(const plaidgpu_gmt* g);
int64_t plaidgpu_gmt_nnz(const plaidgpu_gmt* g);
const char* plaidgpu_gmt_set_name(const plaidgpu_gmt* g, int64_t k);   /* colnames(matG)[k] */
const char* plaidgpu_gmt_gene_name(const plaidgpu_gmt* g, int64_t k);  /* rownames(matG)[k] */
/* CSC pattern of matG: Gp int32[num_sets + 1], Gi int32[nnz] (rows ascending within a column) */
int plaidgpu_gmt_csc(const plaidgpu_gmt* g, int32_t* Gp, int32_t* Gi);
/* rowmap for plaidgpu_score: intersect(rownames(X), rownames(matG)) + match (R/plaid.R:65-72) */
int plaidgpu_gmt_rowmap(const plaidgpu_gmt* g, const char* const* x_rownames, int32_t P, int32_t* rowmap);

/* ---- introspection (bench / tests) ------------------------------------------------ */

/* number of kernels launched by this context since creation (or since reset) */
int64_t plaidgpu_launch_count(const plaidgpu_ctx* ctx);
void plaidgpu_reset_launch_count(plaidgpu_ctx* ctx);
/* device time (ms, CUDA events on the context's stream) spent in the dominant score
 * kernel during the last plaidgpu_score_compute / plaidgpu_score call, and its launches */
double plaidgpu_last_kernel_ms(const plaidgpu_ctx* ctx, int which);
/* cudaStream_t of the context, as void* (so callers can order their own work) */
void* plaidgpu_stream(const plaidgpu_ctx* ctx);
/* plan facts after a score call: scatter tile size / count, mapped memberships, launch shape, and the
 * gather blocks (genes per block, number of blocks; 0 blocks = scatter only) */
int plaidgpu_plan_info(const plaidgpu_ctx* ctx, int32_t* tile_sets, int32_t* n_tiles,
                       int64_t* nnz_mapped, int32_t* warps_per_cta, int32_t* ctas,
                       int32_t* gather_block, int32_t* gather_blocks);
/* the tensor-core block of the current plan: rows of X scored by tcgen05 (0 = the pass is off), the same
 * padded to whole K blocks of 128, and the number of 8-bit fixed-point digits per value */
int plaidgpu_tc_info(const plaidgpu_ctx* ctx, int32_t* block_rows, int32_t* padded_rows, int32_t* slices);
/* the tail pass of the current plan (sparse X): rows of X outside the block that are in at least one set
 * (0 = the pass is off and the fp64 scatter pass finishes the scores), cells per gene-major tile */
int plaidgpu_tail_info(const plaidgpu_ctx* ctx, int32_t* tail_rows, int32_t* tile_cells);

/* ---- expression-matrix files (scope row f4) -------------------------------------------
 * The on-disk formats on the input side of the path, decoded on the host into the CSC arrays of a
 * dgCMatrix (SURVEY.md §8 a1):
 *   read_rda : R save() / saveRDS() file (gzip or plain XDR serialisation, version 2 / 3) holding a
 *              dgCMatrix — the reference's fixture format, inst/extdata/pbmc3k-50cells.rda written by
 *              dev/extdata.R:15.  `object` = name of the saved object, NULL / "" = the first dgCMatrix.
 *   read_mtx : Matrix Market coordinate file (real / integer / pattern; general / symmetric), plain
 *              or .gz; entries in any order, duplicates summed (as(readMM(f), "CsparseMatrix")).
 *   read_10x : directory with matrix.mtx[.gz], features.tsv[.gz] | genes.tsv[.gz] (rownames = column 2,
 *              the gene symbols, as Seurat::Read10X(gene.column = 2)) and barcodes.tsv[.gz].
 * All return PLAIDGPU_OK or PLAIDGPU_ERR_ARG with a message in plaidgpu_io_error() (thread-local). */
typedef struct plaidgpu_spmat plaidgpu_spmat;
int plaidgpu_spmat_read_rda(const char* path, const char* object, plaidgpu_spmat** out);
int plaidgpu_spmat_read_mtx(const char* path, plaidgpu_spmat** out);
int plaidgpu_spmat_read_10x(const char* dir, plaidgpu_spmat** out);
void plaidgpu_spmat_free(plaidgpu_spmat* m);
/* host CSC view of the matrix; the pointers stay valid until plaidgpu_spmat_free */
int plaidgpu_spmat_view(const plaidgpu_spmat* m, plaidgpu_matrix* M);
int64_t plaidgpu_spmat_nnz(const plaidgpu_spmat* m);
int64_t plaidgpu_spmat_num_rownames(const plaidgpu_spmat* m); /* 0 when the file carries no names */
int64_t plaidgpu_spmat_num_colnames(const plaidgpu_spmat* m);
const char* plaidgpu_spmat_rowname(const plaidgpu_spmat* m, int64_t k);
const char* plaidgpu_spmat_colname(const plaidgpu_spmat* m, int64_t k);
const char* plaidgpu_io_error(void);

#ifdef __cplusplus
}
#endif
#endif /* PLAIDGPU_H */
