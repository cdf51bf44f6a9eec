"""Where the time of the score product goes on the C4 shard (125,000 cells x 20,000 genes x 30,000 sets, X and the
scores resident on the device, the default plaid() call of bench.py).

  * per kernel of the fixed-point product (k_tc_prep_csc, k_tile_scan, k_tile_place, k_tail, k_tc_score): device time
    per step and per column chunk, from torch.profiler with CUDA activities over --prof-steps steps of their own;
  * the whole product per step from the library's device events (plaidgpu_last_kernel_ms(ctx, 0)) over --steps
    steps with the profiler off.

Prints one JSON line with the card's name and power limit.  PLAIDGPU_TC_K (block rows) applies as it does to any call,
so the same command sweeps the block / tail split.  Writes nothing unless --trace names a file for the Chrome trace."""
import argparse
import json
import os
import re
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
import plaid_b200 as pb  # noqa: E402
from plaid_b200 import _lib as L, sharded, synth  # noqa: E402
from plaid_b200.api import _matrix_struct, _opts  # noqa: E402
from group_stats_times import card  # noqa: E402

KERNELS = ("k_tc_prep_csc", "k_tile_scan", "k_tile_place", "k_tail", "k_tc_score")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cells", type=int, default=bench.CELLS_PER_GPU)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--prof-steps", type=int, default=3)
    ap.add_argument("--trace", default="", help="also write the profiler's Chrome trace here")
    a = ap.parse_args()
    if min(a.steps, a.prof_steps) < 1:
        raise SystemExit("--steps and --prof-steps must be at least 1")
    if not torch.cuda.is_available():
        raise SystemExit("needs a GPU")
    Nc = a.cells
    G, xp, xi, xx = bench.make_inputs("cuda:0", 0, Nc)
    names = synth.gene_names(bench.P_GENES)
    rowmap = pb.make_rowmap(names, names)
    ctx = pb.Context(0)
    ctx.set_genesets(G)
    out = torch.empty(bench.S_SETS * Nc, dtype=torch.float64, device="cuda:0")
    keep = []
    M = _matrix_struct(pb.DeviceCSC(xp, xi, xx, (bench.P_GENES, Nc)), keep)
    opts = _opts(ctx.lib, scorer=L.PLAID, stats_mean=1, normalize=1, out_location=L.DEVICE)
    comm = sharded.LocalComm()

    def step():
        sharded.score_shard(ctx, comm, M, rowmap, opts, out.data_ptr(), Nc)

    for _ in range(a.warmup):
        step()
    torch.cuda.synchronize()
    prod = []
    for _ in range(a.steps):
        step()
        prod.append(ctx.kernel_ms(0))
    torch.cuda.synchronize()

    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(a.prof_steps):
            step()
        torch.cuda.synchronize()
    if a.trace:
        prof.export_chrome_trace(a.trace)
    per = {k: [0.0, 0] for k in KERNELS}
    for ev in prof.events():
        if ev.device_type != torch.autograd.DeviceType.CUDA:
            continue
        m = re.search(r"\b(k_\w+)[(<]", ev.name)  # demangled: plaidgpu::(anonymous namespace)::k_tail(...)
        if m and m.group(1) in per:
            per[m.group(1)][0] += ev.device_time / 1e3  # us -> ms
            per[m.group(1)][1] += 1
    chunks = per["k_tc_score"][1] / a.prof_steps
    res = {
        "card": card(),
        "shape": f"{Nc} cells x {bench.P_GENES} genes x {bench.S_SETS} sets, device-resident, plaid() default",
        "tc_k": os.environ.get("PLAIDGPU_TC_K", "default"),
        "product_ms_per_step": {"median": round(float(np.median(prod)), 3), "min": round(min(prod), 3),
                                "max": round(max(prod), 3), "steps": a.steps},
        "chunks_per_step": chunks,
        "kernels": {k: {"ms_per_step": round(v[0] / a.prof_steps, 3),
                        "ms_per_chunk": round(v[0] / v[1], 3) if v[1] else None,
                        "launches_per_step": v[1] / a.prof_steps} for k, v in per.items()},
    }
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
