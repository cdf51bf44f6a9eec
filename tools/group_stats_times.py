"""Times of plaidgpu_score_group_stats (plaid(), normalised, fused with the per-set moments of K sample groups) on the
C4 shard: 125,000 cells x 20,000 genes x 30,000 sets, sparse X in pinned host memory, moments back in host memory.

  * ms per call for K = 2, 16, 128, and the reduction kernels' device time (plaidgpu_last_kernel_ms(ctx, 2)) against
    the least time one read of the S x N raw scores can take (30.0 GB at --read-gbs);
  * K = 16 fused against 16 consecutive plaidgpu_score_group_moments calls (one per cluster vs rest);
  * with --parent-lib: the K = 2 call (plaidgpu_score_group_moments) of another build of the library and of this one,
    alternating in the same process, and whether their results agree bit for bit;
  * --big-cells N (0 = skip): one GPU and N cells, where the S x N scores exceed the device and the call takes the
    two-pass column-tiled route.
Prints one JSON object (also written to --out when given) with the card's name and power limit."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import plaid_b200 as pb  # noqa: E402
from plaid_b200 import _lib as L, synth  # noqa: E402
from plaid_b200.api import _opts  # noqa: E402

P, S, CELLS = 20000, 30000, 125000


def host_shard(n, seed):
    """the bench's sparse C4 shard generator, copied to pinned host memory"""
    p, i, x = synth.sparse_x_torch(P, n, seed=seed, device="cuda")
    keep = [t.cpu().pin_memory() for t in (p, i, x)]
    del p, i, x
    torch.cuda.empty_cache()
    M = L.Matrix()
    M.kind, M.location, M.P, M.N = L.CSC, L.HOST, P, n
    M.p, M.i, M.x = (t.data_ptr() for t in keep)
    return M, keep


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power, clock = (v.strip() for v in q.split(","))
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # the numbers stand without it, but say so
        return {"error": str(e)[:100]}


def timed(fn, steps):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return {"ms_mean": round(float(np.mean(ts)), 2), "ms_min": round(float(np.min(ts)), 2),
            "ms_max": round(float(np.max(ts)), 2), "steps": steps}


def parent_context(path, Gp, Gi):
    lib = C.CDLL(path)
    for name in ("plaidgpu_init", "plaidgpu_set_genesets", "plaidgpu_score_group_moments", "plaidgpu_default_opts",
                 "plaidgpu_last_error"):
        res, args = L.SYMBOLS[name]
        getattr(lib, name).restype, getattr(lib, name).argtypes = res, args
    h = C.c_void_p()
    assert lib.plaidgpu_init(0, C.byref(h)) == L.OK, "parent library: plaidgpu_init failed"
    assert lib.plaidgpu_set_genesets(h, P, S, Gp.ctypes.data, Gi.ctypes.data, None) == L.OK
    return lib, h


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--parent-lib", default="")
    ap.add_argument("--big-cells", type=int, default=375000)
    ap.add_argument("--read-gbs", type=float, default=6553.0, help="device copy rate of the card (GB/s) for the read floor")
    ap.add_argument("--out", default="", help="also write the JSON object to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a GPU")
    res = {"card": card(), "shape": f"{CELLS} cells x {P} genes x {S} sets (sparse, ~7% nnz), host X -> host moments",
           "steps": a.steps}
    Gp, Gi = synth.genesets_torch(P, S, seed=synth.SEED0 + 3, device="cuda")
    Gp, Gi = np.ascontiguousarray(Gp, dtype=np.int32), np.ascontiguousarray(Gi, dtype=np.int32)
    ctx = pb.Context(0)
    ctx.check(ctx.lib.plaidgpu_set_genesets(ctx.h, P, S, Gp.ctypes.data, Gi.ctypes.data, None))
    rowmap = np.arange(P, dtype=np.int32)
    o = _opts(ctx.lib, scorer=L.PLAID, stats_mean=1, normalize=1, out_location=L.HOST)
    M, keep = host_shard(CELLS, synth.SEED0 + 3 + 1000)
    lib = ctx.lib
    floor_ms = S * CELLS * 8 / (a.read_gbs * 1e9) * 1e3
    res["read_floor_ms"] = round(floor_ms, 2)

    def fused(K, labels, out):
        return lambda: ctx.check(lib.plaidgpu_score_group_stats(ctx.h, C.byref(M), rowmap.ctypes.data, C.byref(o),
                                                                labels.ctypes.data, K, out.ctypes.data))

    per_k = {}
    for K in (2, 16, 128):
        labels = (np.arange(CELLS) % K).astype(np.int32)
        out = np.empty((K, 2, S))
        t = timed(fused(K, labels, out), a.steps)
        t["reduction_kernel_ms"] = round(ctx.kernel_ms(2), 2)
        t["reduction_over_read_floor"] = round(ctx.kernel_ms(2) / floor_ms, 2)
        per_k[str(K)] = t
    res["fused"] = per_k
    res["k128_over_k2"] = round(per_k["128"]["ms_mean"] / per_k["2"]["ms_mean"], 3)

    # one cluster against the rest, 16 times, with the two-group call
    labels = (np.arange(CELLS) % 16).astype(np.int32)
    y = [(labels == k).astype(np.int32) for k in range(16)]
    mo = np.empty(4 * S)
    loop = timed(lambda: [ctx.check(lib.plaidgpu_score_group_moments(ctx.h, C.byref(M), rowmap.ctypes.data, C.byref(o),
                                                                     yk.ctypes.data, mo.ctypes.data)) for yk in y],
                 max(1, a.steps // 2))
    res["loop_16_group_moments"] = loop
    res["fused16_speedup_over_loop"] = round(loop["ms_mean"] / per_k["16"]["ms_mean"], 2)

    if a.parent_lib:
        plib, ph = parent_context(a.parent_lib, Gp, Gi)
        y2 = (np.arange(CELLS) % 2).astype(np.int32)
        new, old = np.empty(4 * S), np.empty(4 * S)
        fn_new = lambda: ctx.check(lib.plaidgpu_score_group_moments(ctx.h, C.byref(M), rowmap.ctypes.data, C.byref(o),
                                                                    y2.ctypes.data, new.ctypes.data))

        def fn_old():
            if plib.plaidgpu_score_group_moments(ph, C.byref(M), rowmap.ctypes.data, C.byref(o), y2.ctypes.data,
                                                 old.ctypes.data) != L.OK:
                raise RuntimeError(plib.plaidgpu_last_error(ph).decode())
        fn_new()
        fn_old()
        torch.cuda.synchronize()
        tn, to = [], []
        for _ in range(a.steps):
            for fn, acc in ((fn_old, to), (fn_new, tn)):
                t0 = time.perf_counter()
                fn()
                acc.append((time.perf_counter() - t0) * 1e3)
        res["k2_parent_vs_this"] = {"parent_ms": [round(v, 2) for v in to], "this_ms": [round(v, 2) for v in tn],
                                    "parent_ms_mean": round(float(np.mean(to)), 2), "this_ms_mean": round(float(np.mean(tn)), 2),
                                    "bitwise_equal": bool(np.array_equal(new, old))}
        plib.plaidgpu_destroy.argtypes = [C.c_void_p]
        plib.plaidgpu_destroy(ph)  # its device buffers would shrink the budget of the run below

    del keep, M
    torch.cuda.empty_cache()
    if a.big_cells > 0:
        Mb, kb = host_shard(a.big_cells, synth.SEED0 + 3 + 2000)
        labels = (np.arange(a.big_cells) % 16).astype(np.int32)
        out = np.empty((16, 2, S))
        M = Mb
        t = timed(fused(16, labels, out), max(1, a.steps // 2))
        t["cells"] = a.big_cells
        t["scores_gb"] = round(S * a.big_cells * 8 / 1e9, 1)
        t["K"] = 16
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
