"""Times of plaidgpu_score_design_stats (plaid(), normalised, fused with the per-set products with an N x Q design
basis) on the C4 shard: 125,000 cells x 20,000 genes x 30,000 sets, sparse X in pinned host memory, moments back in
host memory.

  * ms per call for each Q of --qs, and the reduction kernels' device time (plaidgpu_last_kernel_ms(ctx, 2)) against
    the least time one read of the S x N raw scores can take (30.0 GB at --read-gbs);
  * plaidgpu_score_group_stats with K = 16 in the same run, for reference;
  * --big-cells N (0 = skip): one GPU and N cells with Q = 16, where the S x N scores exceed the device and the call
    takes the two-pass column-tiled route.
Prints one JSON object with the card's name and power limit; writes it to a file only when --out names one."""
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
    ap.add_argument("--qs", default="1,2,8,16,32,64")
    ap.add_argument("--big-cells", type=int, default=375000)
    ap.add_argument("--read-gbs", type=float, default=6553.0, help="device copy rate of the card (GB/s) for the read floor")
    ap.add_argument("--out", default="", help="also write the JSON object to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a GPU")
    res = {"card": card(), "shape": f"{CELLS} cells x {P} genes x {S} sets (sparse, ~7% nnz), host X -> host moments",
           "steps": a.steps, "library": os.environ.get("PLAIDGPU_LIB", L.lib_path())}
    Gp, Gi = synth.genesets_torch(P, S, seed=synth.SEED0 + 3, device="cuda")
    Gp, Gi = np.ascontiguousarray(Gp, dtype=np.int32), np.ascontiguousarray(Gi, dtype=np.int32)
    ctx = pb.Context(0)
    lib = ctx.lib
    ctx.check(lib.plaidgpu_set_genesets(ctx.h, P, S, Gp.ctypes.data, Gi.ctypes.data, None))
    rowmap = np.arange(P, dtype=np.int32)
    o = _opts(lib, scorer=L.PLAID, stats_mean=1, normalize=1, out_location=L.HOST)
    M, keep = host_shard(CELLS, synth.SEED0 + 3 + 1000)
    floor_ms = S * CELLS * 8 / (a.read_gbs * 1e9) * 1e3
    res["read_floor_ms"] = round(floor_ms, 2)
    rng = np.random.default_rng(5)

    def fused(Mx, B, out):
        return lambda: ctx.check(lib.plaidgpu_score_design_stats(ctx.h, C.byref(Mx), rowmap.ctypes.data, C.byref(o),
                                                                 B.ctypes.data, B.shape[1], out.ctypes.data))

    per_q = {}
    for Q in (int(v) for v in a.qs.split(",")):
        B = np.asfortranarray(rng.normal(size=(CELLS, Q)))
        out = np.empty((Q + 2, S))
        t = timed(fused(M, B, out), a.steps)
        t["kernel_ms"] = round(ctx.kernel_ms(2), 2)
        t["kernel_over_read_floor"] = round(ctx.kernel_ms(2) / floor_ms, 2)
        per_q[str(Q)] = t
    res["design"] = per_q

    labels = (np.arange(CELLS) % 16).astype(np.int32)
    gout = np.empty((16, 2, S))
    t = timed(lambda: ctx.check(lib.plaidgpu_score_group_stats(ctx.h, C.byref(M), rowmap.ctypes.data, C.byref(o),
                                                               labels.ctypes.data, 16, gout.ctypes.data)), a.steps)
    t["kernel_ms"] = round(ctx.kernel_ms(2), 2)
    res["group_stats_k16"] = t

    del keep, M
    torch.cuda.empty_cache()
    if a.big_cells > 0:
        Mb, kb = host_shard(a.big_cells, synth.SEED0 + 3 + 2000)
        B = np.asfortranarray(rng.normal(size=(a.big_cells, 16)))
        out = np.empty((18, S))
        t = timed(fused(Mb, B, out), max(1, a.steps // 2))
        t.update(cells=a.big_cells, scores_gb=round(S * a.big_cells * 8 / 1e9, 1), Q=16)
        res["beyond_device_memory"] = t
        del kb
    txt = json.dumps(res)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")
    print(txt)


if __name__ == "__main__":
    main()
