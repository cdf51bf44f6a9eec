"""The R package exports plaid.topcells and binds the row top-k entry points of include/plaidgpu.h."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_plaid_topcells_is_defined_and_exported():
    ns = open(os.path.join(ROOT, "rpkg", "NAMESPACE")).read()
    code = open(os.path.join(ROOT, "rpkg", "R", "plaid.R")).read()
    assert "export(plaid.topcells)" in ns
    assert "\nplaid.topcells <- function(X, matG, k = 10, decreasing = TRUE, gsetX = NULL)" in "\n" + code
    shim = open(os.path.join(ROOT, "rpkg", "src", "shim.c")).read()
    registered = dict(re.findall(r'\{"(C_plaidgpu_[a-z_]+)", \(DL_FUNC\)&C_plaidgpu_[a-z_]+, (\d+)\}', shim))
    assert registered.get("C_plaidgpu_row_topk") == "4"
    assert registered.get("C_plaidgpu_score_row_topk") == "14"
    assert "plaidgpu_score_row_topk_multi(" in shim  # several contexts (options(plaid.gpus)) take the multi-device call
    for name in re.findall(r"\.Call\((C_plaidgpu_[a-z_]+)", code):
        assert name in registered, name
