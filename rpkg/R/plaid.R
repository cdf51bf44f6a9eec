## Drop-in R wrappers: same signatures, defaults, messages and return types as the reference
## (R/plaid.R of bigomics/plaid; line numbers cited per function).  Only name matching,
## dimnames and argument defaults stay in R; all arithmetic runs in libplaidgpu through .Call.

.plaid_env <- new.env(parent = emptyenv())

.ctx <- function() {
  if (is.null(.plaid_env$ctx)) .plaid_env$ctx <- .Call(C_plaidgpu_ctx, 0L)
  .plaid_env$ctx
}

## options(plaid.gpus = n): the scorers split the columns of X over n devices (one context each; the axis of
## chunked_crossprod's column loop, R/plaid.R:110-119).  Results are identical for any n.
.ctxs <- function() {
  n <- as.integer(getOption("plaid.gpus", 1L))
  if (is.na(n) || n <= 1L) return(.ctx())
  have <- length(.plaid_env$ctxs)
  if (have < n) {
    if (have == 0L) .plaid_env$ctxs <- list(.ctx())
    for (d in seq.int(length(.plaid_env$ctxs), n - 1L))
      .plaid_env$ctxs[[d + 1L]] <- .Call(C_plaidgpu_ctx, as.integer(d))
  }
  .plaid_env$ctxs[seq_len(n)]
}

## X -> list(kind, p, i, x, dim): dgCMatrix slots are passed as they are (no copy)
.as_x <- function(X) {
  if (is.null(dim(X))) X <- cbind(X)                                  # R/plaid.R:63
  if (inherits(X, "CsparseMatrix")) {
    X <- methods::as(X, "CsparseMatrix")
    if (!inherits(X, "dgCMatrix")) X <- methods::as(X, "generalMatrix")
    list(kind = 0L, p = X@p, i = X@i, x = X@x, dim = dim(X), dimnames = dimnames(X))
  } else {
    X <- as.matrix(X)
    storage.mode(X) <- "double"
    list(kind = 1L, p = NULL, i = NULL, x = X, dim = dim(X), dimnames = dimnames(X))
  }
}

.score <- function(X, matG, opts, labels = NULL, K = NULL, topk = NULL, decreasing = TRUE, design = NULL) {
  x <- .as_x(X)
  rn <- x$dimnames[[1]]
  gg <- intersect(rn, rownames(matG))                                 # R/plaid.R:65
  if (length(gg) == 0) {
    message("[plaid] ERROR. No overlapping features.")               # R/plaid.R:66-69
    return(NULL)
  }
  ## rowmap[r] = 0-based row of matG aligned with X row r, or -1; first occurrences only,
  ## exactly what X[gg,] / matG[gg,] select (R/plaid.R:71-72)
  rowmap <- match(rn, rownames(matG)) - 1L
  rowmap[is.na(rowmap) | duplicated(rn)] <- -1L
  G <- methods::as(matG, "CsparseMatrix")
  if (!inherits(G, "dgCMatrix")) G <- methods::as(methods::as(G, "dMatrix"), "generalMatrix")
  if (!is.null(labels)) {  # plaid.test("lm"): scores reduced per set and sample group on the device, S x 2K back
    out <- .Call(C_plaidgpu_score_group_stats, .ctxs(), x$kind, x$p, x$i, x$x, as.integer(x$dim),
                 G@p, G@i, G@x, as.integer(dim(G)), as.integer(rowmap), opts, as.integer(labels), as.integer(K))
    rownames(out) <- colnames(matG)
    return(out)
  }
  if (!is.null(design)) {  # plaid.lm: scores times the design basis, reduced per set on the device, S x (Q + 2) back
    out <- .Call(C_plaidgpu_score_design_stats, .ctxs(), x$kind, x$p, x$i, x$x, as.integer(x$dim),
                 G@p, G@i, G@x, as.integer(dim(G)), as.integer(rowmap), opts, design)
    rownames(out) <- colnames(matG)
    return(out)
  }
  if (!is.null(topk)) {  # plaid.topsets: each column's top k sets selected on the device, k x 2N back
    out <- .Call(C_plaidgpu_score_topk, .ctxs(), x$kind, x$p, x$i, x$x, as.integer(x$dim),
                 G@p, G@i, G@x, as.integer(dim(G)), as.integer(rowmap), opts, as.integer(topk),
                 as.integer(isTRUE(decreasing)))
    return(.topsets(out, topk, x$dimnames[[2]]))
  }
  out <- .Call(C_plaidgpu_score, .ctxs(), x$kind, x$p, x$i, x$x, as.integer(x$dim),
               G@p, G@i, G@x, as.integer(dim(G)), as.integer(rowmap), opts)
  dimnames(out) <- list(colnames(matG), x$dimnames[[2]])
  out
}

## the k x 2N matrix of the top-k shim entries (1-based indices, then scores) -> list(index, score)
.topsets <- function(out, k, cn) {
  N <- ncol(out) %/% 2L
  index <- matrix(as.integer(out[, seq_len(N)]), k, N)
  score <- out[, N + seq_len(N), drop = FALSE]
  colnames(index) <- cn
  colnames(score) <- cn
  list(index = index, score = score)
}

## Each cell's k best gene sets: the first k entries of order(v, decreasing = decreasing) for every column v of
## plaid(X, matG) (ties by set order, NA last), i.e. apply(plaid(X, matG), 2, order, decreasing = TRUE)[1:k, ] and
## the scores at those sets, without the S x N score matrix ever reaching R: plaid() and the selection run as one
## device call (options(plaid.gpus) applies).  With gsetX (the scores of any scorer, sets x cells) the selection
## runs on that matrix instead.  1 <= k <= min(ncol(matG), 256).  Returns list(index = integer k x N (rows of matG,
## 1-based), score = double k x N), both with colnames(X); colnames(matG)[index] names the sets.
plaid.topsets <- function(X, matG, k = 10, decreasing = TRUE, gsetX = NULL) {
  if (is.null(gsetX))
    return(.score(X, matG, list(scorer = 0L, stats_mean = 1L, normalize = 1L), topk = k, decreasing = decreasing))
  gsetX <- as.matrix(gsetX)
  storage.mode(gsetX) <- "double"
  out <- .Call(C_plaidgpu_col_topk, .ctx(), gsetX, as.integer(k), as.integer(isTRUE(decreasing)))
  cn <- colnames(X)
  if (is.null(cn)) cn <- colnames(gsetX)
  .topsets(out, k, cn)
}

plaid <- function(X, matG, stats = c("mean", "sum"), chunk = NULL, normalize = TRUE) {
  stats <- stats[1]                                                   # R/plaid.R:62
  ## `chunk` is accepted and ignored exactly like the reference (R/plaid.R:80 passes NULL)
  .score(X, matG, list(scorer = 0L, stats_mean = as.integer(stats == "mean"),
                       normalize = as.integer(isTRUE(normalize))))
}

normalize_medians <- function(x, ignore.zero = NULL) {                # R/plaid.R:554-575
  x <- as.matrix(x)
  storage.mode(x) <- "double"
  iz <- if (is.null(ignore.zero)) -1L else as.integer(isTRUE(ignore.zero))
  out <- .Call(C_plaidgpu_normalize_medians, .ctx(), x, iz)
  dimnames(out) <- dimnames(x)
  out
}

sparse_colranks <- function(X, signed = FALSE, ties.method = "average") {   # R/plaid.R:631-650
  X <- methods::as(X, "CsparseMatrix")
  rX <- X
  rX@x <- .Call(C_plaidgpu_colranks, .ctx(), 0L, X@p, X@i, X@x, as.integer(dim(X)),
                .ties(ties.method), as.integer(signed), 1L)
  rX
}

## ties.method -> PLAIDGPU_TIES_*: "first" / "last" (base::rank, matrixStats) and "dense" (matrixStats) are ranked in
## order of appearance on the device; "random" draws from R's RNG and is not available
.ties <- function(m) {
  k <- match(m, c("average", "min", "max", "first", "last", "dense"))
  if (is.na(k)) stop("ties.method '", m, "' is not available on the GPU path (average, min, max, first, last, dense)")
  k - 1L
}

colranks <- function(X, sparse = NULL, signed = FALSE, keep.zero = FALSE,   # R/plaid.R:589-623
                     ties.method = "average") {
  if (is.null(sparse)) sparse <- inherits(X, "CsparseMatrix")
  if (sparse) {
    X <- methods::as(X, "CsparseMatrix")
    if (keep.zero) return(sparse_colranks(X, signed = signed, ties.method = ties.method))
    r <- .Call(C_plaidgpu_colranks, .ctx(), 0L, X@p, X@i, X@x, as.integer(dim(X)),
               .ties(ties.method), as.integer(signed), 0L)
  } else {
    M <- as.matrix(X)
    storage.mode(M) <- "double"
    r <- .Call(C_plaidgpu_colranks, .ctx(), 1L, NULL, NULL, M, as.integer(dim(M)),
               .ties(ties.method), as.integer(signed), 0L)
  }
  r <- matrix(r, nrow = nrow(X), ncol = ncol(X), dimnames = dimnames(X))
  r
}

replaid.scse <- function(X, matG, removeLog2 = NULL, scoreMean = FALSE) {   # R/plaid.R:155-190
  rl <- if (is.null(removeLog2)) -1L else as.integer(isTRUE(removeLog2))
  if (isTRUE(removeLog2)) message("[replaid.scse] Converting data to linear scale (removing log2)...")
  .score(X, matG, list(scorer = 1L, remove_log2 = rl, score_mean = as.integer(isTRUE(scoreMean))))
}

replaid.sing <- function(X, matG) {                                         # R/plaid.R:213-219
  .score(X, matG, list(scorer = 2L, nrow_x = NROW(X)))
}

replaid.ssgsea <- function(X, matG, alpha = 0) {                            # R/plaid.R:244-255
  .score(X, matG, list(scorer = 3L, alpha = as.numeric(alpha)))
}

replaid.ucell <- function(X, matG, rmax = 1500) {                           # R/plaid.R:276-282
  .score(X, matG, list(scorer = 4L, rmax = as.numeric(rmax),
                       matg_full_colsums = as.numeric(Matrix::colSums(matG != 0))))
}

replaid.aucell <- function(X, matG, aucMaxRank = ceiling(0.05 * nrow(X))) { # R/plaid.R:304-309
  .score(X, matG, list(scorer = 5L, auc_max_rank = as.numeric(aucMaxRank)))
}

replaid.gsva <- function(X, matG, tau = 0, rowtf = c("z", "ecdf")[1]) {      # R/plaid.R:338-363
  rowtf <- rowtf[1]
  if (!rowtf %in% c("z", "ecdf")) stop("Error: unknown row transform", rowtf) # R/plaid.R:348
  .score(X, matG, list(scorer = 6L, tau = as.numeric(tau), gsva_ecdf = as.integer(rowtf == "ecdf")))
}

## the "one" and "two" tests of plaid.test from crossprod(G != 0, [fc, fc^2]) = [s1, q1] (R/plaid.R:476-520)
.set_tests <- function(tests, s1, q1, sumG, ngenes, fc) {
  pv <- list(); ff <- list()
  if ("one" %in% tests) {
    mx <- s1 / (1e-8 + sumG)
    sdx <- sqrt((q1 - mx^2 * sumG) / (sumG - 1))
    tt <- mx / (1e-8 + sdx) * sqrt(sumG)
    pv$one <- 2 * stats::pt(abs(tt), df = pmax(sumG - 1, 1), lower.tail = FALSE); ff$one <- mx
  }
  if ("two" %in% tests) {
    sum0 <- ngenes - sumG
    mean1 <- s1 / (1e-8 + sumG); mean0 <- (sum(fc) - s1) / (1e-8 + sum0)
    var0 <- ((sum(fc^2) - q1) - mean0^2 * sum0) / (sum0 - 1)
    var1 <- (q1 - mean1^2 * sumG) / (sumG - 1)
    vs <- var0 / sum0 + var1 / sumG
    dof <- vs^2 / (var0 / sum0 * (sum0 - 1) + var1 / sumG * (sumG - 1))
    pv$two <- 2 * stats::pt(abs((mean1 - mean0) / sqrt(vs)), df = pmax(dof, 1), lower.tail = FALSE)
    ff$two <- mean1 - mean0
  }
  list(pv = pv, ff = ff)
}

## Rfast::ttests(t(gsetX), ina = y + 1) (R/plaid.R:429-431) from the group sums / sums of squares: group 1 vs group 0
.lm_test <- function(s0, q0, n0, s1, q1, n1) {
  m0 <- s0 / n0; m1 <- s1 / n1
  v0 <- (q0 - n0 * m0^2) / (n0 - 1); v1 <- (q1 - n1 * m1^2) / (n1 - 1)
  fac <- v0 / n0 + v1 / n1
  dof <- fac^2 / ((v0 / n0)^2 / (n0 - 1) + (v1 / n1)^2 / (n1 - 1))
  list(p = 2 * stats::pt(abs((m0 - m1) / sqrt(fac)), df = dof, lower.tail = FALSE), f = m1 - m0)
}

## p-value clamp, meta p-value, FDR and the sorted result table of plaid.test (R/plaid.R:440-474)
.test_table <- function(pv, ff, G, metap.method, sort.by) {
  pv <- lapply(pv, function(p) { p[is.na(p)] <- 1; pmin(pmax(p, 1e-99), 1 - 1e-99) })
  gsetFC <- rowMeans(do.call(cbind, ff))
  if (length(pv) > 1) {
    if (metap.method %in% c("fisher", "sumlog")) {
      pmeta <- stats::pchisq(-2 * Reduce(`+`, lapply(pv, log)), 2 * length(pv), lower.tail = FALSE)
    } else if (metap.method %in% c("stouffer", "sumz")) {
      pmeta <- stats::pnorm(Reduce(`+`, lapply(pv, stats::qnorm, lower.tail = FALSE)) / sqrt(length(pv)), lower.tail = FALSE)
    } else stop("Invalid method: ", metap.method)
  } else pmeta <- pv[[1]]
  P <- do.call(cbind, pv); colnames(P) <- paste0("p.", names(pv))
  res <- cbind(gsetFC = gsetFC, P, p.meta = pmeta, q.meta = stats::p.adjust(pmeta, method = "fdr"))
  rownames(res) <- colnames(G)
  if (sort.by %in% colnames(res)) res <- res[order(res[, sort.by]), ]
  res
}

## plaid.test (R/plaid.R:392-474): same arguments and result table; the score matrix, the set-wise sums of
## logFC / logFC^2 and the per-set group moments come from the GPU, pt / pchisq / p.adjust stay in R.
plaid.test <- function(X, y, G, gsetX, tests = c("one", "two", "lm"),
                       metap.method = "fisher", sort.by = "p.meta") {
  if (!all(unique(y) %in% c(0, 1))) stop("elements of y must be 0 or 1")
  if (is.list(G)) G <- gmt2mat(G)                                      # R/plaid.R: a GMT list is converted first
  gg <- intersect(rownames(G), rownames(X))
  X <- X[gg, , drop = FALSE]
  G <- G[gg, , drop = FALSE]
  n1 <- sum(y == 1); n0 <- sum(y == 0)
  fc <- Matrix::rowMeans(X[, y == 1, drop = FALSE]) - Matrix::rowMeans(X[, y == 0, drop = FALSE])
  B <- 1 * (G != 0)
  pv <- list(); ff <- list()
  if (any(c("one", "two") %in% tests)) {
    sq <- chunked_crossprod(B, cbind(fc, fc^2))           # GPU: t(G != 0) %*% [F, F^2]
    r <- .set_tests(tests, sq[, 1], sq[, 2], Matrix::colSums(B), nrow(B), fc)
    pv <- r$pv; ff <- r$ff
  }
  if ("lm" %in% tests) {
    lab <- as.integer(y != 0)  # groups 0 / 1: columns sum0, sumsq0, sum1, sumsq1
    if (missing(gsetX) || is.null(gsetX)) {
      ## the S x N score matrix is never materialised for the host: plaid() and the group sums run as one device call
      message("[plaid.test] computing plaid scores...")
      gm <- .score(X, G, list(scorer = 0L, stats_mean = 1L, normalize = 1L), labels = lab, K = 2L)
    } else {
      gm <- .Call(C_plaidgpu_group_stats, .ctx(), as.matrix(gsetX), lab, 2L)
    }
    r <- .lm_test(gm[, 1], gm[, 2], n0, gm[, 3], gm[, 4], n1)
    pv$lm <- r$p; ff$lm <- r$f
  }
  .test_table(pv, ff, G, metap.method, sort.by)
}

## plaid.test for every sample group against all other labelled cells, from ONE scoring pass: a named list with one
## result per level of factor(groups), each what plaid.test(X[, keep], groups[keep] == level, G, gsetX[, keep])
## returns (keep = !is.na(groups)).  The per-group gene means are one sparse product on the host; the scores, their
## per-group moments and crossprod(G != 0, [F_1..F_K, F_1^2..F_K^2]) run on the GPU (options(plaid.gpus) applies).
plaid.test.groups <- function(X, groups, G, gsetX, tests = c("one", "two", "lm"),
                              metap.method = "fisher", sort.by = "p.meta") {
  if (length(groups) != ncol(X)) stop("length(groups) must equal ncol(X)")
  keep <- !is.na(groups)
  f <- factor(groups[keep])
  lev <- levels(f); K <- length(lev)
  if (K == 0) stop("no cell has a group label")
  lab <- as.integer(f) - 1L
  if (is.list(G)) G <- gmt2mat(G)
  gg <- intersect(rownames(G), rownames(X))
  X <- X[gg, keep, drop = FALSE]
  G <- G[gg, , drop = FALSE]
  n <- length(lab); nk <- tabulate(lab + 1L, K)
  B <- 1 * (G != 0)
  if (any(c("one", "two") %in% tests)) {
    onehot <- Matrix::sparseMatrix(i = seq_len(n), j = lab + 1L, x = 1, dims = c(n, K))
    gsum <- as.matrix(X %*% onehot)
    tot <- Matrix::rowSums(X)
    Fk <- sweep(gsum, 2, nk, "/") - sweep(tot - gsum, 2, n - nk, "/")   # mean(group) - mean(other labelled cells)
    alone <- nk == n                                                   # no other cell: every statistic is NA
    Fz <- Fk; Fz[, alone] <- 0
    sq <- chunked_crossprod(B, cbind(Fz, Fz^2))
    sq[, c(alone, alone)] <- NA
  }
  if ("lm" %in% tests) {
    if (missing(gsetX) || is.null(gsetX)) {
      message("[plaid.test] computing plaid scores...")
      gm <- .score(X, G, list(scorer = 0L, stats_mean = 1L, normalize = 1L), labels = lab, K = K)
    } else {
      labs <- rep(-1L, length(groups)); labs[keep] <- lab
      gm <- .Call(C_plaidgpu_group_stats, .ctx(), as.matrix(gsetX), labs, as.integer(K))
    }
    s_all <- rowSums(gm[, 2L * seq_len(K) - 1L, drop = FALSE]); q_all <- rowSums(gm[, 2L * seq_len(K), drop = FALSE])
  }
  res <- lapply(seq_len(K), function(k) {
    pv <- list(); ff <- list()
    if (any(c("one", "two") %in% tests)) {
      r <- .set_tests(tests, sq[, k], sq[, K + k], Matrix::colSums(B), nrow(B), Fk[, k])
      pv <- r$pv; ff <- r$ff
    }
    if ("lm" %in% tests) {
      s1 <- gm[, 2L * k - 1L]; q1 <- gm[, 2L * k]
      r <- .lm_test(s_all - s1, q_all - q1, n - nk[k], s1, q1, nk[k])
      pv$lm <- r$p; ff$lm <- r$f
    }
    .test_table(pv, ff, G, metap.method, sort.by)
  })
  names(res) <- lev
  res
}

## Ordinary least squares of every gene set's plaid scores on a design: lm(gsetX[s, ] ~ design - 1) for every set s,
## or limma's lmFit + contrasts.fit without eBayes.  design: N x Q (one row per column of X), finite, of full column
## rank, 1 <= Q <= 64; contrasts: NULL (one result per column of the design) or a Q x L matrix.  qr() of the design
## runs in R; without gsetX, plaid() runs fused with the reduction U^T s, sum s, sum s^2 per set, so the S x N scores
## never reach R (options(plaid.gpus) applies); with gsetX (the scores of any scorer, sets x cells) the reduction runs
## on that matrix.  A named list (colnames of the design or the contrasts) of tables with rows = colnames(matG) and
## columns logFC, SE, AveExpr, t, P.Value, adj.P.Val (BH over sets).  With N = Q or a perfect fit, SE, t and P.Value
## are NA.  A NaN score makes that set's statistics NaN (lm would drop the sample instead).
plaid.lm <- function(X, matG, design, contrasts = NULL, gsetX = NULL, sort.by = "none") {
  design <- as.matrix(design)
  storage.mode(design) <- "double"
  if (nrow(design) != ncol(X)) stop("nrow(design) must equal ncol(X)")
  if (anyNA(design) || any(!is.finite(design))) stop("the design must be finite (no NA)")
  Q <- ncol(design); N <- nrow(design)
  if (Q < 1 || Q > 64) stop("the design must have 1 to 64 columns")
  qd <- qr(design)
  if (qd$rank < Q || N < Q) stop("the design is not of full column rank")
  U <- qr.Q(qd); R <- qr.R(qd)                             # full rank: no column was pivoted
  cn <- colnames(design)
  if (is.null(cn)) cn <- paste0("coef", seq_len(Q))
  if (is.null(contrasts)) {
    contrasts <- diag(Q); colnames(contrasts) <- cn
  } else {
    contrasts <- as.matrix(contrasts)
    if (nrow(contrasts) != Q) stop("nrow(contrasts) must equal ncol(design)")
    if (is.null(colnames(contrasts))) colnames(contrasts) <- paste0("contrast", seq_len(ncol(contrasts)))
  }
  if (is.null(gsetX)) {
    mom <- .score(X, matG, list(scorer = 0L, stats_mean = 1L, normalize = 1L), design = U)
    if (is.null(mom)) return(NULL)
  } else {
    gsetX <- as.matrix(gsetX)
    storage.mode(gsetX) <- "double"
    mom <- .Call(C_plaidgpu_design_stats, .ctx(), gsetX, U)
  }
  z <- t(mom[, seq_len(Q), drop = FALSE])
  beta <- backsolve(R, z)
  rss <- pmax(mom[, Q + 2L] - colSums(z^2), 0)
  df <- N - Q
  sigma <- if (df > 0) sqrt(rss / df) else rep(NA_real_, nrow(mom))
  sigma[!is.na(sigma) & sigma == 0] <- NA_real_
  sefac <- sqrt(colSums(backsolve(R, contrasts, transpose = TRUE)^2))
  res <- lapply(seq_len(ncol(contrasts)), function(l) {
    logFC <- drop(crossprod(contrasts[, l], beta))
    SE <- sigma * sefac[l]
    tt <- logFC / SE
    p <- if (df > 0) 2 * stats::pt(-abs(tt), df) else rep(NA_real_, length(tt))
    tab <- cbind(logFC = logFC, SE = SE, AveExpr = mom[, Q + 1L] / N, t = tt, P.Value = p,
                 adj.P.Val = stats::p.adjust(p, method = "BH"))
    rownames(tab) <- colnames(matG)
    if (sort.by %in% colnames(tab)) tab <- tab[order(tab[, sort.by]), , drop = FALSE]
    tab
  })
  names(res) <- colnames(contrasts)
  res
}

chunked_crossprod <- function(x, y, chunk = NULL) {                         # R/plaid.R:100-123
  x <- methods::as(x, "CsparseMatrix")
  sc <- rep(1, ncol(x))                      # x must be column-scaled binary (what plaid() builds)
  nz <- diff(x@p) > 0
  sc[nz] <- x@x[x@p[-length(x@p)][nz] + 1L]
  if (is.null(chunk) || chunk < 0) chunk <- round(0.8 * .Machine$integer.max / ncol(x))
  if (NCOL(y) >= chunk) message("[chunked_crossprod] chunked compute: chunk = ", chunk)
  yy <- .as_x(y)
  out <- .Call(C_plaidgpu_crossprod, .ctx(), yy$kind, yy$p, yy$i, yy$x, as.integer(yy$dim),
               x@p, x@i, x@x, as.integer(dim(x)), as.numeric(sc))
  dimnames(out) <- list(colnames(x), yy$dimnames[[2]])
  out
}
