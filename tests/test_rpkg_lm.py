"""The R package exports plaid.lm and binds the design-statistics entry points of include/plaidgpu.h."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_plaid_lm_is_defined_and_exported():
    ns = open(os.path.join(ROOT, "rpkg", "NAMESPACE")).read()
    code = open(os.path.join(ROOT, "rpkg", "R", "plaid.R")).read()
    assert "export(plaid.lm)" in ns
    assert "\nplaid.lm <- function(X, matG, design, contrasts = NULL, gsetX = NULL, sort.by = \"none\")" in "\n" + code
    shim = open(os.path.join(ROOT, "rpkg", "src", "shim.c")).read()
    registered = dict(re.findall(r'\{"(C_plaidgpu_[a-z_]+)", \(DL_FUNC\)&C_plaidgpu_[a-z_]+, (\d+)\}', shim))
    assert registered.get("C_plaidgpu_design_stats") == "3"
    assert registered.get("C_plaidgpu_score_design_stats") == "13"
    assert "plaidgpu_score_design_stats_multi(" in shim  # several contexts (options(plaid.gpus)) take the multi-device call
    for name in re.findall(r"\.Call\((C_plaidgpu_[a-z_]+)", code):
        assert name in registered, name
