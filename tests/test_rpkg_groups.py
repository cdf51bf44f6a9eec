"""The R package exports plaid.test.groups and binds the K-group entry points of include/plaidgpu.h."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_plaid_test_groups_is_defined_and_exported():
    ns = open(os.path.join(ROOT, "rpkg", "NAMESPACE")).read()
    code = open(os.path.join(ROOT, "rpkg", "R", "plaid.R")).read()
    assert "export(plaid.test.groups)" in ns
    assert ('\nplaid.test.groups <- function(X, groups, G, gsetX, tests = c("one", "two", "lm"),\n'
            '                              metap.method = "fisher", sort.by = "p.meta")') in "\n" + code
    shim = open(os.path.join(ROOT, "rpkg", "src", "shim.c")).read()
    registered = set(re.findall(r'\{"(C_plaidgpu_[a-z_]+)"', shim))
    assert {"C_plaidgpu_group_stats", "C_plaidgpu_score_group_stats"} <= registered
    assert "plaidgpu_score_group_stats_multi" in shim
    for name in re.findall(r"\.Call\((C_plaidgpu_[a-z_]+)", code):
        assert name in registered, name
