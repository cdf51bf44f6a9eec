"""Times of plaidgpu_score_row_topk (a scorer fused with each gene set's top k cells) on the C4 shard: 125,000 cells x
20,000 genes x 30,000 sets, sparse X in pinned host memory, idx / val back in host memory.

  * ms per call of plaid() fused with the row selection for k = 1, 10, 32, 100, 256 (decreasing);
  * the selection kernels' device time (plaidgpu_last_kernel_ms(ctx, 2): the chunk pass and the merge) against the
    least time one read of the S x N raw scores can take (30.0 GB at --read-gbs);
  * for comparison in the same process: plaidgpu_score_topk (each cell's top k sets) at k = 10;
  * the kernels alone (plaidgpu_row_topk on a device matrix) on rows ascending along the columns, where with
    decreasing = TRUE every column beats the current list (the worst case), and with decreasing = FALSE none does.
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
    ap.add_argument("--sorted-cols", type=int, default=CELLS, help="columns of the ascending-row kernel run (0 = skip)")
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
    M, keep = host_shard(CELLS, synth.SEED0 + 3 + 1000)
    floor_ms = S * CELLS * 8 / (a.read_gbs * 1e9) * 1e3
    res["read_floor_ms"] = round(floor_ms, 2)

    def fused(k):
        idx = np.empty((k, S), dtype=np.int64)
        val = np.empty((k, S))
        return lambda: ctx.check(lib.plaidgpu_score_row_topk(ctx.h, C.byref(M), rowmap.ctypes.data, C.byref(o_plaid), k,
                                                             1, idx.ctypes.data, val.ctypes.data))

    def with_kernel(t):
        t["select_kernel_ms"] = round(ctx.kernel_ms(2), 2)
        t["select_over_read_floor"] = round(ctx.kernel_ms(2) / floor_ms, 2)
        return t

    res["plaid_topcells"] = {str(k): with_kernel(timed(fused(k), a.steps)) for k in (1, 10, 32, 100, 256)}
    ti = np.empty((10, CELLS), dtype=np.int32)
    tv = np.empty((10, CELLS))
    res["plaid_topsets_k10"] = with_kernel(timed(lambda: ctx.check(lib.plaidgpu_score_topk(
        ctx.h, C.byref(M), rowmap.ctypes.data, C.byref(o_plaid), 10, 1, ti.ctypes.data, tv.ctypes.data)), a.steps))
    del keep, M

    if a.sorted_cols > 0:  # x[s, j] = j: with decreasing = TRUE every column beats the current list
        n = a.sorted_cols
        x = torch.arange(n, dtype=torch.float64, device="cuda").repeat_interleave(S)  # column-major S x n
        idx = np.empty((256, S), dtype=np.int64)
        val = np.empty((256, S))
        floor_n = S * n * 8 / (a.read_gbs * 1e9) * 1e3
        out = {"cols": n, "read_floor_ms": round(floor_n, 2)}
        for k, dec, name in ((10, 1, "k10_worst"), (32, 1, "k32_worst"), (256, 1, "k256_worst"), (10, 0, "k10_best"),
                             (256, 0, "k256_best")):
            ks = []
            for _ in range(a.steps + 1):
                ctx.check(lib.plaidgpu_row_topk(ctx.h, x.data_ptr(), S, n, k, dec, L.DEVICE, idx.ctypes.data,
                                                val.ctypes.data))
                ks.append(ctx.kernel_ms(2))
            out[name] = {"kernel_ms_mean": round(float(np.mean(ks[1:])), 2), "kernel_ms_min": round(float(np.min(ks[1:])), 2),
                         "over_read_floor": round(float(np.mean(ks[1:])) / floor_n, 2)}
        res["ascending_rows_kernel"] = out
        del x
    txt = json.dumps(res)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")
    print(txt)


if __name__ == "__main__":
    main()
