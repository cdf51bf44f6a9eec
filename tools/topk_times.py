"""Times of plaidgpu_score_topk (a scorer fused with each cell's top k gene sets) on the C4 shard: 125,000 cells x
20,000 genes x 30,000 sets, sparse X in pinned host memory, idx / val back in host memory.

  * ms per call of plaid() fused with the selection for k = 1, 10, 32, 256 (decreasing), and of replaid.ucell for
    k = 10 with decreasing = FALSE (ucell scores trend downward along the set index: the streaming worst case);
  * the selection kernel's device time (plaidgpu_last_kernel_ms(ctx, 2)) against the least time one read of the
    S x N raw scores can take (30.0 GB at --read-gbs);
  * for comparison in the same process: plaidgpu_score_group_stats with K = 16, and plaid() with the scores shipped
    to host memory;
  * the kernel alone (plaidgpu_col_topk on a device matrix) on columns already sorted in the selection order, where
    every 32-row batch is merged.
Prints one JSON object (also written to --out when given) with the card's name and power limit."""
import argparse
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import plaid_b200 as pb  # noqa: E402
from plaid_b200 import _lib as L, synth  # noqa: E402
from plaid_b200.api import _opts  # noqa: E402
from group_stats_times import CELLS, P, S, card, host_shard, timed  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--read-gbs", type=float, default=6553.0, help="device copy rate of the card (GB/s) for the read floor")
    ap.add_argument("--sorted-cols", type=int, default=20000, help="columns of the sorted-column kernel run (0 = skip)")
    ap.add_argument("--out", default="", help="also write the JSON object to this file")
    a = ap.parse_args()
    if a.steps < 1:
        raise SystemExit("--steps must be at least 1")
    if not torch.cuda.is_available():
        raise SystemExit("needs a GPU")
    res = {"card": card(), "shape": f"{CELLS} cells x {P} genes x {S} sets (sparse, ~7% nnz), host X -> host idx / val",
           "steps": a.steps}
    Gp, Gi = synth.genesets_torch(P, S, seed=synth.SEED0 + 3, device="cuda")
    Gp, Gi = np.ascontiguousarray(Gp, dtype=np.int32), np.ascontiguousarray(Gi, dtype=np.int32)
    ctx = pb.Context(0)
    lib = ctx.lib
    ctx.check(lib.plaidgpu_set_genesets(ctx.h, P, S, Gp.ctypes.data, Gi.ctypes.data, None))
    rowmap = np.arange(P, dtype=np.int32)
    o_plaid = _opts(lib, scorer=L.PLAID, stats_mean=1, normalize=1, out_location=L.HOST)
    o_ucell = _opts(lib, scorer=L.UCELL, rmax=1500.0, out_location=L.HOST)
    M, keep = host_shard(CELLS, synth.SEED0 + 3 + 1000)
    floor_ms = S * CELLS * 8 / (a.read_gbs * 1e9) * 1e3
    res["read_floor_ms"] = round(floor_ms, 2)

    def fused(o, k, dec):
        idx = np.empty((k, CELLS), dtype=np.int32)
        val = np.empty((k, CELLS))
        return lambda: ctx.check(lib.plaidgpu_score_topk(ctx.h, C.byref(M), rowmap.ctypes.data, C.byref(o), k, dec,
                                                         idx.ctypes.data, val.ctypes.data))

    def with_kernel(t):
        t["select_kernel_ms"] = round(ctx.kernel_ms(2), 2)
        t["select_over_read_floor"] = round(ctx.kernel_ms(2) / floor_ms, 2)
        return t

    res["plaid_topk"] = {str(k): with_kernel(timed(fused(o_plaid, k, 1), a.steps)) for k in (1, 10, 32, 256)}
    res["ucell_topk10_increasing"] = with_kernel(timed(fused(o_ucell, 10, 0), a.steps))

    labels = (np.arange(CELLS) % 16).astype(np.int32)
    mom = np.empty((16, 2, S))
    res["group_stats_k16"] = timed(lambda: ctx.check(lib.plaidgpu_score_group_stats(
        ctx.h, C.byref(M), rowmap.ctypes.data, C.byref(o_plaid), labels.ctypes.data, 16, mom.ctypes.data)), a.steps)
    res["group_stats_k16"]["reduction_kernel_ms"] = round(ctx.kernel_ms(2), 2)
    scores = np.empty((S, CELLS), order="F")  # 30 GB of pageable host memory, as plaid() returns it
    res["plaid_to_host"] = timed(lambda: ctx.check(lib.plaidgpu_score(ctx.h, C.byref(M), rowmap.ctypes.data,
                                                                      C.byref(o_plaid), scores.ctypes.data)),
                                 max(1, a.steps // 2))
    del scores, keep, M
    res["topk10_vs_group_stats_ms"] = round(res["plaid_topk"]["10"]["ms_mean"] - res["group_stats_k16"]["ms_mean"], 2)
    res["plaid_to_host_over_topk10"] = round(res["plaid_to_host"]["ms_mean"] / res["plaid_topk"]["10"]["ms_mean"], 2)

    if a.sorted_cols > 0:  # every column already in the selection order: each batch beats the k-th entry
        n = a.sorted_cols
        x = torch.arange(S, 0, -1, dtype=torch.float64, device="cuda").repeat(n)  # descending: worst for increasing
        idx = np.empty((256, n), dtype=np.int32)
        val = np.empty((256, n))
        floor_n = S * n * 8 / (a.read_gbs * 1e9) * 1e3
        out = {"cols": n, "read_floor_ms": round(floor_n, 2)}
        for k, dec, name in ((10, 0, "k10_worst"), (256, 0, "k256_worst"), (10, 1, "k10_best"), (256, 1, "k256_best")):
            ks = []
            for _ in range(a.steps + 1):
                ctx.check(lib.plaidgpu_col_topk(ctx.h, x.data_ptr(), S, n, k, dec, L.DEVICE, idx.ctypes.data,
                                                val.ctypes.data))
                ks.append(ctx.kernel_ms(2))
            out[name] = {"kernel_ms_mean": round(float(np.mean(ks[1:])), 2), "kernel_ms_min": round(float(np.min(ks[1:])), 2),
                         "over_read_floor": round(float(np.mean(ks[1:])) / floor_n, 2)}
        res["sorted_columns_kernel"] = out
        del x
    txt = json.dumps(res)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")
    print(txt)


if __name__ == "__main__":
    main()
