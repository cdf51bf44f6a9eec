# Runs wherever R + the built package + a B200 exist (not in the build container: no R there).
test_that("plaid.lm matches summary(lm(gsetX[s, ] ~ design - 1)) on the bundled fixture", {
  load(system.file("extdata", "pbmc3k-50cells.rda", package = "plaid"))
  matG <- gmt2mat(read.gmt(system.file("extdata", "hallmarks.gmt", package = "plaid")))
  set.seed(3)
  design <- cbind(intercept = 1, y = rnorm(ncol(X)), batch = rep(0:1, length.out = ncol(X)))
  gsetX <- plaid(X, matG)
  fused <- plaid.lm(X, matG, design)
  given <- plaid.lm(X, matG, design, gsetX = gsetX)
  expect_equal(names(fused), colnames(design))
  for (s in colnames(matG)[c(1, 7, 20, 33)]) {
    cf <- summary(lm(gsetX[s, ] ~ design - 1))$coefficients
    for (k in seq_len(ncol(design))) {
      for (res in list(fused, given)) {
        tab <- res[[colnames(design)[k]]]
        expect_equal(unname(tab[s, c("logFC", "SE", "t", "P.Value")]), unname(cf[k, ]), tolerance = 1e-9)
      }
    }
  }
  ## a contrast of the two last coefficients, and the errors
  cm <- matrix(c(0, 1, -1), 3, 1, dimnames = list(NULL, "y-batch"))
  r <- plaid.lm(X, matG, design, contrasts = cm)
  expect_equal(unname(r[["y-batch"]][, "logFC"]), unname(fused$y[, "logFC"] - fused$batch[, "logFC"]), tolerance = 1e-9)
  expect_error(plaid.lm(X, matG, design[-1, ]))
  expect_error(plaid.lm(X, matG, cbind(design, 2 * design[, "y"])))
  d2 <- design; d2[3, 2] <- NA
  expect_error(plaid.lm(X, matG, d2))
})
