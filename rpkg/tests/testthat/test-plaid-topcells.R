# Runs wherever R + the built package + a B200 exist (not in the build container: no R there).
test_that("plaid.topcells matches apply(plaid(X, matG), 1, order, decreasing = ...)[1:k, ]", {
  load(system.file("extdata", "pbmc3k-50cells.rda", package = "plaid"))
  matG <- gmt2mat(read.gmt(system.file("extdata", "hallmarks.gmt", package = "plaid")))
  gsetX <- plaid(X, matG)
  for (dec in c(TRUE, FALSE)) {
    for (k in c(1, 10, ncol(X))) {
      want <- apply(gsetX, 1, order, decreasing = dec)[seq_len(k), , drop = FALSE]
      for (res in list(plaid.topcells(X, matG, k, dec), plaid.topcells(X, matG, k, dec, gsetX = gsetX))) {
        expect_identical(unname(res$index), matrix(as.integer(want), k))
        expect_identical(colnames(res$index), colnames(matG))
        expect_identical(unname(res$score), matrix(gsetX[cbind(rep(seq_len(nrow(gsetX)), each = k), as.vector(want))], k))
      }
    }
  }
  top <- plaid.topcells(X, matG, 3)
  expect_identical(colnames(X)[top$index[, 1]], colnames(X)[order(gsetX[1, ], decreasing = TRUE)[1:3]])
  old <- options(plaid.gpus = 2)
  two <- plaid.topcells(X, matG, 5)
  options(old)
  expect_identical(two, plaid.topcells(X, matG, 5))
  expect_error(plaid.topcells(X, matG, 0))
  expect_error(plaid.topcells(X, matG, 257))
})
