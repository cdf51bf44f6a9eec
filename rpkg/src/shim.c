/*
 * .Call shim between R and libplaidgpu (include/plaidgpu.h).  Thin by design: it only unpacks
 * SEXPs into plain pointers, allocates the result, and maps status codes to R conditions.
 * No arithmetic happens here.  R's API is single-threaded: SEXPs are touched on the calling
 * thread only; the library joins its streams before it returns.
 *
 * Replaces nothing in the reference (it has no src/); it is the binding a maintainer adds to
 * route R/plaid.R:60-87,100-123,155-309,554-650 to the GPU.
 */
#include <R.h>
#include <Rinternals.h>
#include <R_ext/Rdynload.h>
#include <limits.h>
#include <string.h>

#include "plaidgpu.h"

static void ctx_finalizer(SEXP ptr) {
  plaidgpu_ctx* c = (plaidgpu_ctx*)R_ExternalPtrAddr(ptr);
  if (c) {
    plaidgpu_destroy(c);
    R_ClearExternalPtr(ptr);
  }
}

static plaidgpu_ctx* get_ctx(SEXP s) {
  plaidgpu_ctx* c = (plaidgpu_ctx*)R_ExternalPtrAddr(s);
  if (!c) Rf_error("plaidgpu: context has been released");
  return c;
}

SEXP C_plaidgpu_ctx(SEXP device) {
  plaidgpu_ctx* c = NULL;
  int rc = plaidgpu_init(Rf_asInteger(device), &c);
  if (rc != PLAIDGPU_OK) Rf_error("plaidgpu_init failed (%d): no usable B200; this package has no CPU fallback", rc);
  SEXP p = PROTECT(R_MakeExternalPtr(c, R_NilValue, R_NilValue));
  R_RegisterCFinalizerEx(p, ctx_finalizer, TRUE);
  UNPROTECT(1);
  return p;
}

static SEXP list_get(SEXP lst, const char* name) {
  SEXP names = Rf_getAttrib(lst, R_NamesSymbol);
  for (R_xlen_t k = 0; k < XLENGTH(lst); ++k)
    if (strcmp(CHAR(STRING_ELT(names, k)), name) == 0) return VECTOR_ELT(lst, k);
  return R_NilValue;
}
static int opt_int(SEXP lst, const char* n, int def) { SEXP v = list_get(lst, n); return v == R_NilValue ? def : Rf_asInteger(v); }
static double opt_dbl(SEXP lst, const char* n, double def) { SEXP v = list_get(lst, n); return v == R_NilValue ? def : Rf_asReal(v); }

static void fill_matrix(plaidgpu_matrix* M, int kind, SEXP p, SEXP i, SEXP x, SEXP dim) {
  memset(M, 0, sizeof(*M));
  M->kind = kind;
  M->location = PLAIDGPU_HOST;
  M->P = INTEGER(dim)[0];
  M->N = INTEGER(dim)[1];
  M->p = kind == PLAIDGPU_CSC ? INTEGER(p) : NULL;
  M->i = kind == PLAIDGPU_CSC ? INTEGER(i) : NULL;
  M->x = REAL(x);
}

/* named list of options from R -> plaidgpu_opts (defaults for whatever is absent) */
static void fill_opts(plaidgpu_opts* op, SEXP opts) {
  plaidgpu_opts o;
  plaidgpu_default_opts(&o);
  o.scorer = opt_int(opts, "scorer", o.scorer);
  o.stats_mean = opt_int(opts, "stats_mean", o.stats_mean);
  o.normalize = opt_int(opts, "normalize", o.normalize);
  o.remove_log2 = opt_int(opts, "remove_log2", o.remove_log2);
  o.score_mean = opt_int(opts, "score_mean", o.score_mean);
  o.alpha = opt_dbl(opts, "alpha", o.alpha);
  o.rmax = opt_dbl(opts, "rmax", o.rmax);
  o.auc_max_rank = opt_dbl(opts, "auc_max_rank", o.auc_max_rank);
  o.tau = opt_dbl(opts, "tau", o.tau);
  o.gsva_ecdf = opt_int(opts, "gsva_ecdf", 0);
  o.nrow_x = (int64_t)opt_dbl(opts, "nrow_x", 0.0);
  SEXP csums = list_get(opts, "matg_full_colsums");
  o.matg_full_colsums = csums == R_NilValue ? NULL : REAL(csums);
  *op = o;
}

/* plaid() and the replaid.* scorers.  `ctx` is one context (external pointer) or a list of contexts on different
 * devices (options(plaid.gpus = n) in R/plaid.R): the columns are then split over them by plaidgpu_score_multi, one
 * host thread per device inside the library, the shards landing directly in the result matrix. */
SEXP C_plaidgpu_score(SEXP ctx, SEXP kind, SEXP Xp, SEXP Xi, SEXP Xx, SEXP Xdim, SEXP Gp, SEXP Gi, SEXP Gx,
                      SEXP Gdim, SEXP rowmap, SEXP opts) {
  plaidgpu_ctx* cs[16];
  int nctx = 1;
  if (TYPEOF(ctx) == VECSXP) {
    nctx = (int)XLENGTH(ctx);
    if (nctx < 1 || nctx > 16) Rf_error("plaidgpu: between 1 and 16 contexts expected");
    for (int k = 0; k < nctx; ++k) cs[k] = get_ctx(VECTOR_ELT(ctx, k));
  } else {
    cs[0] = get_ctx(ctx);
  }
  plaidgpu_ctx* c = cs[0];
  const int PG = INTEGER(Gdim)[0], S = INTEGER(Gdim)[1];
  /* re-registering the same pattern is a memcmp inside the library: the plan is kept across calls */
  for (int k = 0; k < nctx; ++k) {
    int rc0 = plaidgpu_set_genesets(cs[k], PG, S, INTEGER(Gp), INTEGER(Gi), REAL(Gx));
    if (rc0 != PLAIDGPU_OK) Rf_error("plaidgpu_set_genesets: %s", plaidgpu_last_error(cs[k]));
  }
  int rc;
  plaidgpu_matrix M;
  fill_matrix(&M, Rf_asInteger(kind), Xp, Xi, Xx, Xdim);
  plaidgpu_opts o;
  fill_opts(&o, opts);
  o.out_location = PLAIDGPU_HOST;
  R_CheckUserInterrupt(); /* before the (blocking) device call; the library itself never touches the R API */
  /* S x N may exceed 2^31 elements: Rf_allocMatrix takes ints for the dims, the product is R_xlen_t */
  SEXP out = PROTECT(Rf_allocMatrix(REALSXP, S, (int)M.N));
  if (nctx > 1 && !(o.scorer == PLAIDGPU_GSVA && o.gsva_ecdf == PLAIDGPU_ROWTF_ECDF))
    rc = plaidgpu_score_multi(cs, nctx, &M, INTEGER(rowmap), &o, REAL(out));
  else
    rc = plaidgpu_score(c, &M, INTEGER(rowmap), &o, REAL(out));
  if (rc != PLAIDGPU_OK) {
    UNPROTECT(1);
    Rf_error("plaidgpu_score: %s", plaidgpu_last_error(c)); /* longjmp: nothing left to release */
  }
  UNPROTECT(1);
  return out;
}

/* chunked_crossprod(x, y): t(x) %*% y for a column-scaled binary sparse x */
SEXP C_plaidgpu_crossprod(SEXP ctx, SEXP kind, SEXP Yp, SEXP Yi, SEXP Yx, SEXP Ydim, SEXP Gp, SEXP Gi, SEXP Gx,
                          SEXP Gdim, SEXP colscale) {
  plaidgpu_ctx* c = get_ctx(ctx);
  const int PG = INTEGER(Gdim)[0], S = INTEGER(Gdim)[1];
  int rc = plaidgpu_set_genesets(c, PG, S, INTEGER(Gp), INTEGER(Gi), REAL(Gx));
  if (rc != PLAIDGPU_OK) Rf_error("plaidgpu_set_genesets: %s", plaidgpu_last_error(c));
  plaidgpu_matrix M;
  fill_matrix(&M, Rf_asInteger(kind), Yp, Yi, Yx, Ydim);
  if (M.P != PG) Rf_error("non-conformable arguments");
  int* rowmap = (int*)R_alloc((size_t)PG, sizeof(int)); /* identity: same rows on both sides */
  for (int r = 0; r < PG; ++r) rowmap[r] = r;
  SEXP out = PROTECT(Rf_allocMatrix(REALSXP, S, (int)M.N));
  rc = plaidgpu_crossprod(c, &M, rowmap, REAL(colscale), PLAIDGPU_HOST, REAL(out));
  if (rc != PLAIDGPU_OK) {
    UNPROTECT(1);
    Rf_error("plaidgpu_crossprod: %s", plaidgpu_last_error(c));
  }
  UNPROTECT(1);
  return out;
}

/* normalize_medians(x, ignore.zero) */
SEXP C_plaidgpu_normalize_medians(SEXP ctx, SEXP x, SEXP ignore_zero) {
  plaidgpu_ctx* c = get_ctx(ctx);
  SEXP dim = Rf_getAttrib(x, R_DimSymbol);
  const int S = INTEGER(dim)[0], N = INTEGER(dim)[1];
  SEXP out = PROTECT(Rf_allocMatrix(REALSXP, S, N));
  int rc = plaidgpu_normalize_medians(c, REAL(x), S, N, Rf_asInteger(ignore_zero), PLAIDGPU_HOST, REAL(out));
  if (rc != PLAIDGPU_OK) {
    UNPROTECT(1);
    Rf_error("plaidgpu_normalize_medians: %s", plaidgpu_last_error(c));
  }
  UNPROTECT(1);
  return out;
}

/* colranks() / sparse_colranks(): returns nnz ranks (keep_zero) or P*N ranks */
SEXP C_plaidgpu_colranks(SEXP ctx, SEXP kind, SEXP Xp, SEXP Xi, SEXP Xx, SEXP Xdim, SEXP ties, SEXP is_signed,
                         SEXP keep_zero) {
  plaidgpu_ctx* c = get_ctx(ctx);
  plaidgpu_matrix M;
  fill_matrix(&M, Rf_asInteger(kind), Xp, Xi, Xx, Xdim);
  const int kz = Rf_asInteger(keep_zero);
  const R_xlen_t n = (M.kind == PLAIDGPU_CSC && kz) ? XLENGTH(Xx) : (R_xlen_t)M.P * (R_xlen_t)M.N;
  SEXP out = PROTECT(Rf_allocVector(REALSXP, n));
  int rc = plaidgpu_colranks(c, &M, Rf_asInteger(ties), Rf_asInteger(is_signed), kz, PLAIDGPU_HOST, REAL(out));
  if (rc != PLAIDGPU_OK) {
    UNPROTECT(1);
    Rf_error("plaidgpu_colranks: %s", plaidgpu_last_error(c));
  }
  UNPROTECT(1);
  return out;
}

/* per-set sums / sums of squares of gsetX by group (plaid.test "lm"): labels in [-1, K), -1 = no group.  An S x 2K
 * matrix: columns 2k + 1, 2k + 2 (1-based) hold sum_k, sumsq_k */
SEXP C_plaidgpu_group_stats(SEXP ctx, SEXP x, SEXP labels, SEXP K) {
  plaidgpu_ctx* c = get_ctx(ctx);
  SEXP dim = Rf_getAttrib(x, R_DimSymbol);
  const int S = INTEGER(dim)[0], N = INTEGER(dim)[1], k = Rf_asInteger(K);
  if (XLENGTH(labels) != N) Rf_error("plaidgpu: length(labels) must equal ncol(x)");
  if (k < 1 || k > INT_MAX / 2) Rf_error("plaidgpu: K must be at least 1");
  SEXP out = PROTECT(Rf_allocMatrix(REALSXP, S, 2 * k));
  int rc = plaidgpu_group_stats(c, REAL(x), S, N, INTEGER(labels), k, PLAIDGPU_HOST, REAL(out));
  if (rc != PLAIDGPU_OK) {
    UNPROTECT(1);
    Rf_error("plaidgpu_group_stats: %s", plaidgpu_last_error(c));
  }
  UNPROTECT(1);
  return out;
}

/* plaid.test(tests = "lm") without gsetX (R/plaid.R:423-431), for K sample groups: plaid() fused with the per-set group
 * reductions — the S x N scores stay on the device, an S x 2K matrix (sum_k, sumsq_k per group) comes back.  A list of
 * contexts (options(plaid.gpus = n)) splits the columns over the devices (plaidgpu_score_group_stats_multi). */
SEXP C_plaidgpu_score_group_stats(SEXP ctx, SEXP kind, SEXP Xp, SEXP Xi, SEXP Xx, SEXP Xdim, SEXP Gp, SEXP Gi, SEXP Gx,
                                  SEXP Gdim, SEXP rowmap, SEXP opts, SEXP labels, SEXP K) {
  plaidgpu_ctx* cs[16];
  int nctx = 1;
  if (TYPEOF(ctx) == VECSXP) {
    nctx = (int)XLENGTH(ctx);
    if (nctx < 1 || nctx > 16) Rf_error("plaidgpu: between 1 and 16 contexts expected");
    for (int j = 0; j < nctx; ++j) cs[j] = get_ctx(VECTOR_ELT(ctx, j));
  } else {
    cs[0] = get_ctx(ctx);
  }
  plaidgpu_ctx* c = cs[0];
  const int PG = INTEGER(Gdim)[0], S = INTEGER(Gdim)[1], k = Rf_asInteger(K);
  for (int j = 0; j < nctx; ++j)
    if (plaidgpu_set_genesets(cs[j], PG, S, INTEGER(Gp), INTEGER(Gi), REAL(Gx)) != PLAIDGPU_OK)
      Rf_error("plaidgpu_set_genesets: %s", plaidgpu_last_error(cs[j]));
  plaidgpu_matrix M;
  fill_matrix(&M, Rf_asInteger(kind), Xp, Xi, Xx, Xdim);
  if ((int64_t)XLENGTH(labels) != M.N) Rf_error("plaidgpu: length(labels) must equal ncol(X)");
  if (k < 1 || k > INT_MAX / 2) Rf_error("plaidgpu: K must be at least 1");
  plaidgpu_opts o;
  fill_opts(&o, opts);
  R_CheckUserInterrupt();
  SEXP out = PROTECT(Rf_allocMatrix(REALSXP, S, 2 * k));
  int rc = nctx > 1 ? plaidgpu_score_group_stats_multi(cs, nctx, &M, INTEGER(rowmap), &o, INTEGER(labels), k, REAL(out))
                    : plaidgpu_score_group_stats(c, &M, INTEGER(rowmap), &o, INTEGER(labels), k, REAL(out));
  if (rc != PLAIDGPU_OK) {
    UNPROTECT(1);
    Rf_error("plaidgpu_score_group_stats: %s", plaidgpu_last_error(c));
  }
  UNPROTECT(1);
  return out;
}

/* plaid.lm(gsetX = ): per set of gsetX (S x N) the products with the N x Q design basis B, the sum and the sum of
 * squares as an S x (Q + 2) matrix */
SEXP C_plaidgpu_design_stats(SEXP ctx, SEXP x, SEXP B) {
  plaidgpu_ctx* c = get_ctx(ctx);
  SEXP dim = Rf_getAttrib(x, R_DimSymbol), bdim = Rf_getAttrib(B, R_DimSymbol);
  const int S = INTEGER(dim)[0], N = INTEGER(dim)[1];
  if (bdim == R_NilValue || INTEGER(bdim)[0] != N) Rf_error("plaidgpu: nrow(design) must equal ncol(gsetX)");
  const int Q = INTEGER(bdim)[1];
  if (Q < 1 || Q > 64) Rf_error("plaidgpu: the design must have 1 to 64 columns");
  SEXP out = PROTECT(Rf_allocMatrix(REALSXP, S, Q + 2));
  int rc = plaidgpu_design_stats(c, REAL(x), S, N, REAL(B), Q, PLAIDGPU_HOST, REAL(out));
  if (rc != PLAIDGPU_OK) {
    UNPROTECT(1);
    Rf_error("plaidgpu_design_stats: %s", plaidgpu_last_error(c));
  }
  UNPROTECT(1);
  return out;
}

/* plaid.lm(): plaid() fused with the per-set products with the design basis B (N x Q) — the S x N scores stay on the
 * device, an S x (Q + 2) matrix comes back.  A list of contexts (options(plaid.gpus = n)) splits the columns over the
 * devices (plaidgpu_score_design_stats_multi). */
SEXP C_plaidgpu_score_design_stats(SEXP ctx, SEXP kind, SEXP Xp, SEXP Xi, SEXP Xx, SEXP Xdim, SEXP Gp, SEXP Gi,
                                   SEXP Gx, SEXP Gdim, SEXP rowmap, SEXP opts, SEXP B) {
  plaidgpu_ctx* cs[16];
  int nctx = 1;
  if (TYPEOF(ctx) == VECSXP) {
    nctx = (int)XLENGTH(ctx);
    if (nctx < 1 || nctx > 16) Rf_error("plaidgpu: between 1 and 16 contexts expected");
    for (int j = 0; j < nctx; ++j) cs[j] = get_ctx(VECTOR_ELT(ctx, j));
  } else {
    cs[0] = get_ctx(ctx);
  }
  plaidgpu_ctx* c = cs[0];
  const int PG = INTEGER(Gdim)[0], S = INTEGER(Gdim)[1];
  for (int j = 0; j < nctx; ++j)
    if (plaidgpu_set_genesets(cs[j], PG, S, INTEGER(Gp), INTEGER(Gi), REAL(Gx)) != PLAIDGPU_OK)
      Rf_error("plaidgpu_set_genesets: %s", plaidgpu_last_error(cs[j]));
  plaidgpu_matrix M;
  fill_matrix(&M, Rf_asInteger(kind), Xp, Xi, Xx, Xdim);
  SEXP bdim = Rf_getAttrib(B, R_DimSymbol);
  if (bdim == R_NilValue || (int64_t)INTEGER(bdim)[0] != M.N) Rf_error("plaidgpu: nrow(design) must equal ncol(X)");
  const int Q = INTEGER(bdim)[1];
  if (Q < 1 || Q > 64) Rf_error("plaidgpu: the design must have 1 to 64 columns");
  plaidgpu_opts o;
  fill_opts(&o, opts);
  R_CheckUserInterrupt();
  SEXP out = PROTECT(Rf_allocMatrix(REALSXP, S, Q + 2));
  int rc = nctx > 1 ? plaidgpu_score_design_stats_multi(cs, nctx, &M, INTEGER(rowmap), &o, REAL(B), Q, REAL(out))
                    : plaidgpu_score_design_stats(c, &M, INTEGER(rowmap), &o, REAL(B), Q, REAL(out));
  if (rc != PLAIDGPU_OK) {
    UNPROTECT(1);
    Rf_error("plaidgpu_score_design_stats: %s", plaidgpu_last_error(c));
  }
  UNPROTECT(1);
  return out;
}

/* per-column top k as one k x 2N matrix: columns 1..N the 1-based row indices (exact in a double), N+1..2N the values;
 * idx / val are what plaidgpu_col_topk / plaidgpu_score_topk wrote, val already in place */
static void topk_indices_to_r(SEXP out, const int32_t* idx, int k, int N) {
  double* o = REAL(out);
  for (R_xlen_t t = 0, n = (R_xlen_t)k * N; t < n; ++t) o[t] = (double)idx[t] + 1.0;
}

/* plaid.topsets(gsetX = ): each column's k first rows of order(x[, j], decreasing = decreasing) */
SEXP C_plaidgpu_col_topk(SEXP ctx, SEXP x, SEXP k, SEXP decreasing) {
  plaidgpu_ctx* c = get_ctx(ctx);
  SEXP dim = Rf_getAttrib(x, R_DimSymbol);
  const int S = INTEGER(dim)[0], N = INTEGER(dim)[1], kk = Rf_asInteger(k);
  if (kk < 1 || kk > 256 || kk > S) Rf_error("plaidgpu: k must be in [1, min(nrow(x), 256)]");
  int32_t* idx = (int32_t*)R_alloc((size_t)kk * (size_t)N + 1, sizeof(int32_t));
  SEXP out = PROTECT(Rf_allocMatrix(REALSXP, kk, 2 * N));
  int rc = plaidgpu_col_topk(c, REAL(x), S, N, kk, Rf_asInteger(decreasing), PLAIDGPU_HOST, idx,
                             REAL(out) + (R_xlen_t)kk * N);
  if (rc != PLAIDGPU_OK) {
    UNPROTECT(1);
    Rf_error("plaidgpu_col_topk: %s", plaidgpu_last_error(c));
  }
  topk_indices_to_r(out, idx, kk, N);
  UNPROTECT(1);
  return out;
}

/* plaid.topsets(): plaid() fused with each cell's top k sets — the S x N scores stay on the device, a k x 2N matrix
 * (indices, then scores) comes back.  A list of contexts (options(plaid.gpus = n)) splits the columns over the
 * devices (plaidgpu_score_topk_multi). */
SEXP C_plaidgpu_score_topk(SEXP ctx, SEXP kind, SEXP Xp, SEXP Xi, SEXP Xx, SEXP Xdim, SEXP Gp, SEXP Gi, SEXP Gx,
                           SEXP Gdim, SEXP rowmap, SEXP opts, SEXP k, SEXP decreasing) {
  plaidgpu_ctx* cs[16];
  int nctx = 1;
  if (TYPEOF(ctx) == VECSXP) {
    nctx = (int)XLENGTH(ctx);
    if (nctx < 1 || nctx > 16) Rf_error("plaidgpu: between 1 and 16 contexts expected");
    for (int j = 0; j < nctx; ++j) cs[j] = get_ctx(VECTOR_ELT(ctx, j));
  } else {
    cs[0] = get_ctx(ctx);
  }
  plaidgpu_ctx* c = cs[0];
  const int PG = INTEGER(Gdim)[0], S = INTEGER(Gdim)[1], kk = Rf_asInteger(k);
  if (kk < 1 || kk > 256 || kk > S) Rf_error("plaidgpu: k must be in [1, min(ncol(matG), 256)]");
  for (int j = 0; j < nctx; ++j)
    if (plaidgpu_set_genesets(cs[j], PG, S, INTEGER(Gp), INTEGER(Gi), REAL(Gx)) != PLAIDGPU_OK)
      Rf_error("plaidgpu_set_genesets: %s", plaidgpu_last_error(cs[j]));
  plaidgpu_matrix M;
  fill_matrix(&M, Rf_asInteger(kind), Xp, Xi, Xx, Xdim);
  if (M.N > INT_MAX / 2) Rf_error("plaidgpu: too many columns for one k x 2N result");
  const int N = (int)M.N;
  plaidgpu_opts o;
  fill_opts(&o, opts);
  R_CheckUserInterrupt();
  int32_t* idx = (int32_t*)R_alloc((size_t)kk * (size_t)N + 1, sizeof(int32_t));
  SEXP out = PROTECT(Rf_allocMatrix(REALSXP, kk, 2 * N));
  double* val = REAL(out) + (R_xlen_t)kk * N;
  const int dec = Rf_asInteger(decreasing);
  int rc = nctx > 1 ? plaidgpu_score_topk_multi(cs, nctx, &M, INTEGER(rowmap), &o, kk, dec, idx, val)
                    : plaidgpu_score_topk(c, &M, INTEGER(rowmap), &o, kk, dec, idx, val);
  if (rc != PLAIDGPU_OK) {
    UNPROTECT(1);
    Rf_error("plaidgpu_score_topk: %s", plaidgpu_last_error(c));
  }
  topk_indices_to_r(out, idx, kk, N);
  UNPROTECT(1);
  return out;
}

static const R_CallMethodDef call_methods[] = {
    {"C_plaidgpu_ctx", (DL_FUNC)&C_plaidgpu_ctx, 1},
    {"C_plaidgpu_score", (DL_FUNC)&C_plaidgpu_score, 12},
    {"C_plaidgpu_normalize_medians", (DL_FUNC)&C_plaidgpu_normalize_medians, 3},
    {"C_plaidgpu_colranks", (DL_FUNC)&C_plaidgpu_colranks, 9},
    {"C_plaidgpu_group_stats", (DL_FUNC)&C_plaidgpu_group_stats, 4},
    {"C_plaidgpu_score_group_stats", (DL_FUNC)&C_plaidgpu_score_group_stats, 14},
    {"C_plaidgpu_design_stats", (DL_FUNC)&C_plaidgpu_design_stats, 3},
    {"C_plaidgpu_score_design_stats", (DL_FUNC)&C_plaidgpu_score_design_stats, 13},
    {"C_plaidgpu_col_topk", (DL_FUNC)&C_plaidgpu_col_topk, 4},
    {"C_plaidgpu_score_topk", (DL_FUNC)&C_plaidgpu_score_topk, 14},
    {"C_plaidgpu_crossprod", (DL_FUNC)&C_plaidgpu_crossprod, 11},
    {NULL, NULL, 0}};

void R_init_plaid(DllInfo* dll) {
  R_registerRoutines(dll, NULL, call_methods, NULL, NULL);
  R_useDynamicSymbols(dll, FALSE);
}
