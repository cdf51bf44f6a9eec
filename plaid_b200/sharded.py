"""Column-sharded scoring: one process (rank) per GPU, samples split across ranks.

The product, the ranking and the per-column medians are column-independent (the axis
`chunked_crossprod` already splits on, R/plaid.R:115-119), so there is NO data-path
collective.  What does couple the shards are a handful of scalars (SURVEY.md §8e):
  * min / max of X                      (replaid.scse auto removeLog2, R/plaid.R:160-161)
  * max(rX)                             (ssgsea / ucell / aucell, R/plaid.R:251,278,306)
  * min(scores) and mean(col medians)   (normalize_medians, R/plaid.R:557,572)
replaid.gsva is the exception (SURVEY.md §8e, f3): its row transform runs ACROSS samples.  rowtf "z"
needs per-gene sums (all-reduce of P doubles, twice); rowtf "ecdf" needs every gene's values over all
samples, so the dense shards are re-partitioned column blocks -> row blocks with an all-to-all, ranked
(plaidgpu_row_ecdf) and sent back — `gsva_shard` below.
The scalars are exchanged with torch.distributed (NCCL on GPUs, gloo in the CPU tests): one
all-reduce(max) of (-x_min, x_max, rank_max), one all-reduce(min) of the score minimum and one
all-gather of both per-column median vectors, which every rank then combines in GLOBAL COLUMN
ORDER (plaidgpu_combine_medians), so results are bit-identical for any number of shards.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np

from . import _lib as L


class LocalComm:
    """world_size == 1."""
    rank, world = 0, 1

    def allreduce_min(self, v: float) -> float:
        return v

    def allreduce_max(self, v: float) -> float:
        return v

    def allreduce_max_vec(self, v: np.ndarray) -> np.ndarray:
        return v

    def allgather_vec(self, v: np.ndarray) -> np.ndarray:
        return v

    def allgather_vecs(self, vs):
        return list(vs)

    def allreduce_sum_vec(self, v: np.ndarray) -> np.ndarray:
        return v

    def alltoall(self, parts):
        return list(parts)


class ThreadComm:
    """Shards driven by threads of ONE process (one context each; ctypes calls release the GIL).
    `ThreadComm.group(world)` returns the `world` endpoints; every collective is a rendezvous on a
    shared slot table, combined in rank order."""

    def __init__(self, shared, rank):
        self._s, self.rank, self.world = shared, rank, shared["world"]

    @classmethod
    def group(cls, world: int):
        import threading
        shared = {"world": world, "slots": [None] * world, "barrier": threading.Barrier(world)}
        return [cls(shared, r) for r in range(world)]

    def _exchange(self, v):
        s = self._s
        s["slots"][self.rank] = v
        s["barrier"].wait()
        # copy before the release: a rank may overwrite the array it contributed (gsva_shard reuses `part`)
        # as soon as the second barrier lets it go, while a slower rank is still summing the references
        vals = [x.copy() if isinstance(x, np.ndarray) else x for x in s["slots"]]
        s["barrier"].wait()
        return vals

    def allreduce_min(self, v: float) -> float:
        return min(self._exchange(v))

    def allreduce_max(self, v: float) -> float:
        return max(self._exchange(v))

    def allreduce_max_vec(self, v: np.ndarray) -> np.ndarray:
        return np.max(np.stack(self._exchange(np.asarray(v, dtype=np.float64))), axis=0)

    def allgather_vec(self, v: np.ndarray) -> np.ndarray:
        return np.concatenate(self._exchange(np.asarray(v, dtype=np.float64)))

    def allgather_vecs(self, vs):
        return [self.allgather_vec(v) for v in vs]

    def allreduce_sum_vec(self, v: np.ndarray) -> np.ndarray:
        vals = self._exchange(np.asarray(v, dtype=np.float64))
        acc = vals[0].copy()
        for w in vals[1:]:
            acc += w
        return acc

    def alltoall(self, parts):
        """parts[q] goes to rank q; returns what every rank r sent to this rank, in rank order"""
        table = self._exchange(list(parts))
        return [table[r][self.rank] for r in range(self.world)]


class TorchComm:
    """torch.distributed adapter (backend nccl -> tensors on the rank's GPU; gloo -> CPU)."""

    def __init__(self, device=None, group=None):
        import torch
        import torch.distributed as dist
        self.torch, self.dist, self.group = torch, dist, group
        self.rank = dist.get_rank(group)
        self.world = dist.get_world_size(group)
        self.device = device if device is not None else "cpu"
        self._pin = {}

    def _red(self, v: float, op):
        t = self.torch.tensor([v], dtype=self.torch.float64, device=self.device)
        self.dist.all_reduce(t, op=op, group=self.group)
        return float(t.item())

    def allreduce_min(self, v: float) -> float:
        return self._red(v, self.dist.ReduceOp.MIN)

    def allreduce_max(self, v: float) -> float:
        return self._red(v, self.dist.ReduceOp.MAX)

    def allreduce_max_vec(self, v: np.ndarray) -> np.ndarray:
        t = self.torch.from_numpy(np.ascontiguousarray(v, dtype=np.float64)).to(self.device)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX, group=self.group)
        return t.cpu().numpy()

    def allgather_vecs(self, vs):
        """several float64 vectors of one common (per-rank) length: ONE size exchange, ONE all-gather of the
        stacked vectors and ONE copy back; returns the list of rank-order concatenations"""
        torch, dist = self.torch, self.dist
        k, n = len(vs), int(vs[0].size)
        sz = torch.tensor([n], dtype=torch.int64, device=self.device)
        sizes = [torch.zeros_like(sz) for _ in range(self.world)]
        dist.all_gather(sizes, sz, group=self.group)
        sizes = [int(t.item()) for t in sizes]
        m = max(max(sizes), 1)
        buf = torch.zeros((k, m), dtype=torch.float64, device=self.device)
        if n:
            buf[:, :n] = torch.from_numpy(np.ascontiguousarray(np.stack([np.asarray(v, dtype=np.float64) for v in vs]))).to(self.device)
        out = torch.empty((self.world, k, m), dtype=torch.float64, device=self.device)
        dist.all_gather([out[r] for r in range(self.world)], buf, group=self.group)
        if out.is_cuda:  # pinned staging (cached): a pageable 16 MB copy costs ~3 ms per step at 8 ranks
            key = tuple(out.shape)
            pin = self._pin.get(key)
            if pin is None:
                pin = self._pin[key] = torch.empty(key, dtype=torch.float64, pin_memory=True)
            pin.copy_(out, non_blocking=True)
            torch.cuda.current_stream(out.device).synchronize()
            host = pin.numpy()
        else:
            host = out.numpy()
        return [np.concatenate([host[r, i, :sizes[r]] for r in range(self.world)]) for i in range(k)]

    def allgather_vec(self, v: np.ndarray) -> np.ndarray:
        """concatenate variable-length float64 vectors of all ranks in rank order"""
        return self.allgather_vecs([np.asarray(v, dtype=np.float64)])[0]

    def allreduce_sum_vec(self, v: np.ndarray) -> np.ndarray:
        """element-wise sum over ranks, added in RANK ORDER on every rank (not a tree all-reduce), so
        all ranks hold the same bits"""
        v = np.ascontiguousarray(v, dtype=np.float64)
        flat = self.allgather_vec(v).reshape(self.world, v.size)
        acc = flat[0].copy()
        for r in range(1, self.world):
            acc += flat[r]
        return acc.reshape(v.shape)

    def alltoall(self, parts):
        """parts[q] (2-D float64, rows fixed by the receiver's row block) goes to rank q.  NCCL: one
        all_to_all over NVLink; gloo (CPU tests) has no all-to-all, so pairwise send / recv."""
        torch, dist = self.torch, self.dist
        shapes = np.array([[p.shape[0], p.shape[1]] for p in parts], dtype=np.float64).ravel()
        allshapes = self.allgather_vec(shapes).reshape(self.world, self.world, 2).astype(np.int64)
        ins = [torch.from_numpy(np.ascontiguousarray(p, dtype=np.float64)).to(self.device) for p in parts]
        outs = [torch.empty((int(allshapes[r, self.rank, 0]), int(allshapes[r, self.rank, 1])), dtype=torch.float64,
                            device=self.device) for r in range(self.world)]
        if dist.get_backend(self.group) == "nccl":
            dist.all_to_all(outs, ins, group=self.group)
        else:
            outs[self.rank].copy_(ins[self.rank])
            reqs = []
            for r in range(self.world):
                if r == self.rank:
                    continue
                if ins[r].numel():
                    reqs.append(dist.isend(ins[r], dst=dist.get_global_rank(self.group, r) if self.group else r, group=self.group))
                if outs[r].numel():
                    reqs.append(dist.irecv(outs[r], src=dist.get_global_rank(self.group, r) if self.group else r, group=self.group))
            for q in reqs:
                q.wait()
        return [o.cpu().numpy() for o in outs]


def combine_scalars(comm, local: L.Scalars) -> L.Scalars:
    """step 2 of the protocol in include/plaidgpu.h: x_min (min), x_max (max), rank_max (max)."""
    g = L.Scalars()
    C.memmove(C.byref(g), C.byref(local), C.sizeof(L.Scalars))
    # one all-reduce(max) of (-x_min, x_max, rank_max): min(a) == -max(-a), exact in fp64
    r = comm.allreduce_max_vec(np.array([-local.x_min, local.x_max, local.rank_max], dtype=np.float64))
    g.x_min, g.x_max, g.rank_max = -float(r[0]), float(r[1]), float(r[2])
    return g


def combine_medians(lib, comm, ignore_zero_opt: int, scal: L.Scalars, med_all: np.ndarray, med_nz: np.ndarray):
    """step 4: global score_min, all medians in column order -> ignore_zero flag + mean(medx)."""
    smin = comm.allreduce_min(scal.score_min)
    ga, gz = (np.ascontiguousarray(v, dtype=np.float64) for v in comm.allgather_vecs([med_all, med_nz]))
    rc = lib.plaidgpu_combine_medians(int(ignore_zero_opt), smin, ga.ctypes.data, gz.ctypes.data, ga.size, C.byref(scal))
    if rc != L.OK:
        raise L.PlaidGpuError(rc, "plaidgpu_combine_medians failed")
    return scal


def combine_medians_of(ctx, comm, ignore_zero_opt: int, scal: L.Scalars, n_cols: int):
    """step 4 for a live context: the global score minimum settles ignore.zero first, so only THAT median vector
    is fetched (plaidgpu_get_col_medians_for: already computed unless this shard's minimum is 0 while another
    shard holds a negative score) and all-gathered; every rank then takes mean(medx) in global column order."""
    lib = ctx.lib
    smin = comm.allreduce_min(scal.score_min)
    iz = (smin == 0.0) if ignore_zero_opt < 0 else bool(ignore_zero_opt)
    med = np.empty(max(n_cols, 0), dtype=np.float64)
    ctx.check(lib.plaidgpu_get_col_medians_for(ctx.h, int(iz), med.ctypes.data))
    g = np.ascontiguousarray(comm.allgather_vec(med), dtype=np.float64)
    rc = lib.plaidgpu_combine_medians(int(ignore_zero_opt), smin, g.ctypes.data, g.ctypes.data, g.size, C.byref(scal))
    if rc != L.OK:
        raise L.PlaidGpuError(rc, "plaidgpu_combine_medians failed")
    return scal


def score_shard(ctx, comm, M: L.Matrix, rowmap: np.ndarray, opts: L.Opts, out_ptr: int, n_cols: int):
    """Run the begin / compute / finish protocol for this rank's column shard."""
    lib = ctx.lib
    local = L.Scalars()
    ctx.check(lib.plaidgpu_score_begin(ctx.h, C.byref(M), rowmap.ctypes.data, C.byref(opts), C.byref(local)))
    # plaid() itself has no cross-shard scalar before the scores exist (x_min / x_max feed scse's removeLog2 switch,
    # rank_max the rank scorers): no collective, no host sync on its critical path
    scal = local if opts.scorer == L.PLAID else combine_scalars(comm, local)
    ctx.check(lib.plaidgpu_score_compute(ctx.h, C.byref(scal), out_ptr))
    needs_norm = (opts.scorer in (L.SSGSEA, L.UCELL, L.AUCELL, L.GSVA)) or (opts.scorer == L.PLAID and opts.normalize)
    if needs_norm:
        combine_medians_of(ctx, comm, opts.ignore_zero, scal, n_cols)
    ctx.check(lib.plaidgpu_score_finish(ctx.h, C.byref(scal), out_ptr))
    return scal


def score_group_stats_shard(ctx, comm, M: L.Matrix, rowmap: np.ndarray, opts: L.Opts, labels, K: int, n_cols: int):
    """Per-group sums / sums of squares of this rank's scores, summed over all ranks (in rank order): score_shard into
    a device buffer, plaidgpu_group_stats on it, then one all-reduce of K * 2 * S doubles.  labels: int32[n_cols] of
    this shard's columns in [-1, K).  `ctx` must hold the gene sets (Context.set_genesets).  Returns (K, 2, S)."""
    import torch
    S = ctx.n_sets
    lab = np.ascontiguousarray(labels, dtype=np.int32)
    if lab.size != n_cols:
        raise ValueError("length(labels) must equal the shard's column count")
    buf = torch.empty(max(S * n_cols, 1), dtype=torch.float64, device=f"cuda:{ctx.device}")
    opts.out_location = L.DEVICE
    score_shard(ctx, comm, M, rowmap, opts, buf.data_ptr(), n_cols)
    out = np.empty((int(K), 2, S), dtype=np.float64)
    ctx.check(ctx.lib.plaidgpu_group_stats(ctx.h, buf.data_ptr(), S, n_cols, lab.ctypes.data, int(K), L.DEVICE,
                                           out.ctypes.data))
    return comm.allreduce_sum_vec(out.ravel()).reshape(out.shape)


def score_design_stats_shard(ctx, comm, M: L.Matrix, rowmap: np.ndarray, opts: L.Opts, B_rows, n_cols: int):
    """design_stats of this rank's scores, summed over all ranks (in rank order): score_shard into a device buffer,
    plaidgpu_design_stats on it, then one all-reduce of (Q + 2) * S doubles.  B_rows: this rank's n_cols rows of the
    global design basis U (N x Q).  `ctx` must hold the gene sets (Context.set_genesets).  Returns (Q + 2, S)."""
    import torch
    S = ctx.n_sets
    b = np.asfortranarray(np.asarray(B_rows, dtype=np.float64).reshape(n_cols, -1))
    buf = torch.empty(max(S * n_cols, 1), dtype=torch.float64, device=f"cuda:{ctx.device}")
    opts.out_location = L.DEVICE
    score_shard(ctx, comm, M, rowmap, opts, buf.data_ptr(), n_cols)
    out = np.empty((b.shape[1] + 2, S), dtype=np.float64)
    ctx.check(ctx.lib.plaidgpu_design_stats(ctx.h, buf.data_ptr(), S, n_cols, b.ctypes.data, b.shape[1], L.DEVICE,
                                            out.ctypes.data))
    return comm.allreduce_sum_vec(out.ravel()).reshape(out.shape)


def score_topk_shard(ctx, comm, M: L.Matrix, rowmap: np.ndarray, opts: L.Opts, k: int, decreasing: bool, n_cols: int):
    """Each of this rank's cells' k best gene sets: score_shard into a device buffer, then plaidgpu_col_topk on it.
    The selection is column-local, so nothing is exchanged beyond what scoring needs.  `ctx` must hold the gene sets
    (Context.set_genesets).  Returns (idx, val) of shape (k, n_cols) for this shard's columns."""
    import torch
    S = ctx.n_sets
    buf = torch.empty(max(S * n_cols, 1), dtype=torch.float64, device=f"cuda:{ctx.device}")
    opts.out_location = L.DEVICE
    score_shard(ctx, comm, M, rowmap, opts, buf.data_ptr(), n_cols)
    idx = np.empty((max(int(k), 0), n_cols), dtype=np.int32, order="F")
    val = np.empty((max(int(k), 0), n_cols), dtype=np.float64, order="F")
    ctx.check(ctx.lib.plaidgpu_col_topk(ctx.h, buf.data_ptr(), S, n_cols, int(k), 1 if decreasing else 0, L.DEVICE,
                                        idx.ctypes.data, val.ctypes.data))
    return idx, val


def shard_columns(n_total: int, world: int, rank: int):
    """contiguous, equal-count column ranges (equal output bytes, the dominant cost)"""
    base, rem = divmod(n_total, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


# ---------------------------------------------------------------------------------------
# replaid.gsva on column shards
# ---------------------------------------------------------------------------------------
def exchange_to_rows(comm, Xd: np.ndarray):
    """Column shard (P x n_r) -> this rank's row block over ALL samples.  Returns (block, counts):
    block is (P_q, N) C-contiguous — the memory layout of an N x P_q column-major matrix, every gene's
    samples contiguous in global column order — and counts[r] = n_r."""
    P = Xd.shape[0]
    parts = []
    for q in range(comm.world):
        g0, g1 = shard_columns(P, comm.world, q)
        parts.append(np.ascontiguousarray(Xd[g0:g1, :], dtype=np.float64))
    recv = comm.alltoall(parts)
    return np.ascontiguousarray(np.concatenate(recv, axis=1)), [int(p.shape[1]) for p in recv]


def exchange_to_columns(comm, block: np.ndarray, counts):
    """inverse of exchange_to_rows: row block (P_q, N) -> column shard (P, n_r), Fortran order"""
    offs = np.concatenate([[0], np.cumsum(counts)])
    parts = [np.ascontiguousarray(block[:, offs[r]:offs[r + 1]]) for r in range(comm.world)]
    recv = comm.alltoall(parts)
    return np.asfortranarray(np.concatenate(recv, axis=0))


def gsva_shard(ctx, comm, Xd: np.ndarray, rowmap: np.ndarray, opts: L.Opts, out_ptr: int, rowtf: str = "z"):
    """replaid.gsva(X, matG, tau, rowtf) (R/plaid.R:338-363) for this rank's dense column shard Xd (P x n_r).
      rowtf "z":    rowMeans / rowSds over all shards = two all-reduces of P doubles around
                    plaidgpu_row_moments (two-pass SD like mat.rowsds, R/plaid.R:365-370);
      rowtf "ecdf": all-to-all into row blocks, plaidgpu_row_ecdf, all-to-all back (SURVEY.md §8 f3).
    Then the ordinary sharded protocol (score_shard) ranks and scores the columns."""
    lib = ctx.lib
    Xd = np.asfortranarray(Xd, dtype=np.float64)
    P, n = Xd.shape
    keep = []
    if rowtf == "ecdf":
        block, counts = exchange_to_rows(comm, Xd)
        rows, N = block.shape
        ctx.check(lib.plaidgpu_row_ecdf(ctx.h, block.ctypes.data, N, rows, L.HOST))
        Xd = exchange_to_columns(comm, block, counts)
        opts.gsva_ecdf = L.ROWTF_DONE
    elif rowtf == "z":
        M = L.Matrix()
        M.kind, M.location, M.P, M.N, M.x = L.DENSE, L.HOST, P, n, Xd.ctypes.data
        N = int(round(comm.allgather_vec(np.array([float(n)])).sum()))
        part = np.empty(P)
        ctx.check(lib.plaidgpu_row_moments(ctx.h, C.byref(M), None, part.ctypes.data))
        mean = comm.allreduce_sum_vec(part) / N
        ctx.check(lib.plaidgpu_row_moments(ctx.h, C.byref(M), mean.ctypes.data, part.ctypes.data))
        with np.errstate(invalid="ignore", divide="ignore"):
            sd = np.sqrt(comm.allreduce_sum_vec(part) / (N - 1)) if N > 1 else np.full(P, np.nan)
        keep += [mean, sd]
        opts.row_mean, opts.row_sd = mean.ctypes.data, sd.ctypes.data
        opts.gsva_ecdf = L.ROWTF_Z
    else:
        raise ValueError('rowtf must be "z" or "ecdf"')
    M = L.Matrix()
    M.kind, M.location, M.P, M.N, M.x = L.DENSE, L.HOST, P, n, Xd.ctypes.data
    opts.scorer = L.GSVA
    return score_shard(ctx, comm, M, rowmap, opts, out_ptr, n)


def score_multi(ctxs, mats, rowmap: np.ndarray, opts_list, out_ptrs, n_cols):
    """The same protocol with several contexts driven by ONE process (one context per GPU, or several
    on one GPU): shards in column order.  This is how a single R process would use more than one GPU."""
    lib = ctxs[0].lib
    k = len(ctxs)
    locs = [L.Scalars() for _ in range(k)]
    for c, M, o, loc in zip(ctxs, mats, opts_list, locs):
        c.check(lib.plaidgpu_score_begin(c.h, C.byref(M), rowmap.ctypes.data, C.byref(o), C.byref(loc)))
    g = L.Scalars()
    C.memmove(C.byref(g), C.byref(locs[0]), C.sizeof(L.Scalars))
    g.x_min = min(l.x_min for l in locs)
    g.x_max = max(l.x_max for l in locs)
    g.rank_max = max(l.rank_max for l in locs)
    scal = []
    for c, outp in zip(ctxs, out_ptrs):
        s = L.Scalars()
        C.memmove(C.byref(s), C.byref(g), C.sizeof(L.Scalars))
        c.check(lib.plaidgpu_score_compute(c.h, C.byref(s), outp))
        scal.append(s)
    o0 = opts_list[0]
    if (o0.scorer in (L.SSGSEA, L.UCELL, L.AUCELL, L.GSVA)) or (o0.scorer == L.PLAID and o0.normalize):
        smin = min(s.score_min for s in scal)
        iz = (smin == 0.0) if o0.ignore_zero < 0 else bool(o0.ignore_zero)
        meds = []
        for c, n in zip(ctxs, n_cols):
            m = np.empty(n)
            c.check(lib.plaidgpu_get_col_medians_for(c.h, int(iz), m.ctypes.data))
            meds.append(m)
        g = np.ascontiguousarray(np.concatenate(meds))
        for s in scal:
            rc = lib.plaidgpu_combine_medians(int(o0.ignore_zero), smin, g.ctypes.data, g.ctypes.data, g.size, C.byref(s))
            if rc != L.OK:
                raise L.PlaidGpuError(rc, "plaidgpu_combine_medians failed")
    for c, s, outp in zip(ctxs, scal, out_ptrs):
        c.check(lib.plaidgpu_score_finish(c.h, C.byref(s), outp))
    return scal
