// K3 — the sparse remainder of the gene-set score product (reference R/plaid.R:100-123, Matrix::crossprod ->
// CHOLMOD): every row of a sparse X that is NOT in the tensor-core block (tc_kernels.cu), i.e. the many genes
// that are expressed in a few per cent of the cells and sit in ~100 sets each.
//
// Formulation (replaces the lanes = genes scatter of score_kernels.cu on the fixed-point path):
//   * the cells are cut into tiles of TAIL_C columns; per tile the tail entries of X are regrouped GENE-major
//     (k_tile_scan / k_tile_place: counting sort by tail row -> `rowptr` and 8-byte records `ent` = {value in the
//     column's fixed point (the same 2^e_j the tensor-core pass uses, int32), cell inside the tile});
//   * one warp owns one (tile, set) item at a time: it walks the set's tail members 32 at a time, concatenates
//     their sparse rows of the tile into one stream and adds it 32 entries per step (LANES = ENTRIES, whatever
//     row each belongs to) into TAIL_C accumulators in shared memory;
//   * accumulators are 64-bit integers split into a u32 low word (a shared-memory atomic on every add) and a
//     16-bit high counter (a second atomic only on carry / borrow, see acc_add): lanes of one step may hit the
//     same cell, and integer sums are exact and order-independent;
//   * the finished row (TAIL_C sums of one set) is written as int64 to `tmp[set][cell]` with coalesced stores;
//     the tensor-core kernel fetches its 128 sets x 48 cells by TMA and adds it to its own integer sums
//     before the one conversion to fp64 (so tail + block is exact, then scaled by 2^-e_j).
// Items are dealt dynamically (one atomic per item) in decreasing order of the set's tail size.
#include "common.cuh"

namespace plaidgpu {

namespace {

constexpr int TAIL_WARPS = 32;

// block-wide exclusive scan of the per-(tile, tail row) entry counts -> tile-local row pointers; the counters
// are zeroed again (k_tile_place re-uses them as cursors).  grid = tiles, 1024 threads.
__global__ void __launch_bounds__(1024) k_tile_scan(uint32_t* __restrict__ cnt, int32_t Pt, uint32_t* __restrict__ rowptr,
                                                    uint32_t* __restrict__ total) {
  __shared__ uint32_t wsum[32];
  const int t = blockIdx.x, tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  uint32_t* __restrict__ c = cnt + (size_t)t * Pt;
  uint32_t* __restrict__ rp = rowptr + (size_t)t * (Pt + 1);
  const int per = (Pt + 1023) / 1024;
  const int lo = min(Pt, tid * per), hi = min(Pt, lo + per);
  uint32_t s = 0;
  for (int i = lo; i < hi; ++i) s += c[i];
  uint32_t incl = s;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t v = __shfl_up_sync(FULL, incl, o);
    if (lane >= o) incl += v;
  }
  if (lane == 31) wsum[w] = incl;
  __syncthreads();
  if (w == 0) {
    uint32_t v = wsum[lane], a = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t u = __shfl_up_sync(FULL, a, o);
      if (lane >= o) a += u;
    }
    wsum[lane] = a - v;  // exclusive
    if (lane == 31) {
      total[t] = a;
      rp[Pt] = a;
    }
  }
  __syncthreads();
  uint32_t run = wsum[w] + incl - s;
  for (int i = lo; i < hi; ++i) {
    const uint32_t v = c[i];
    rp[i] = run;
    run += v;
    c[i] = 0;
  }
}

// one warp per column: tail entries of the (compacted) column -> their slot in the tile's gene-major arrays
__global__ void __launch_bounds__(256) k_tile_place(const int32_t* __restrict__ xp, const int32_t* __restrict__ xe,
                                                    const int32_t* __restrict__ oi, const double* __restrict__ ox,
                                                    const double* __restrict__ r0, const int32_t* __restrict__ tmap,
                                                    const double* __restrict__ colinv, int64_t N, int mode, double a0,
                                                    double a1, int32_t Pt, int C, const uint32_t* __restrict__ rowptr,
                                                    const uint32_t* __restrict__ total, uint32_t* __restrict__ cnt,
                                                    uint2* __restrict__ ent, const int* __restrict__ skip_if) {
  if (skip_if && *skip_if != 0) return;
  const int lane = threadIdx.x & 31;
  const int64_t w0 = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t j = w0; j < N; j += nw) {
    const int t = (int)(j / C);
    const uint32_t cell = (uint32_t)(j - (int64_t)t * C);
    uint32_t base = 0;  // entries of the tiles before this one
    for (int u = lane; u < t; u += 32) base += total[u];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) base += __shfl_xor_sync(FULL, base, o);
    const uint32_t* __restrict__ rp = rowptr + (size_t)t * (Pt + 1);
    uint32_t* __restrict__ cur = cnt + (size_t)t * Pt;
    double fb = 0.0;
    if (mode >= XF_SING) fb = xform_value(mode, r0 ? r0[j] : 0.0, a0, a1);
    const double sc = 1.0 / colinv[j];  // 2^e_j, exact
    // four iterations at a time, each dependent level (index -> tail row -> row pointer + cursor) issued for all four
    // before the next: one warp per column has no other way of overlapping the chain
    const int32_t e1 = xe[j];
    for (int32_t e0 = xp[j]; e0 < e1; e0 += 128) {
      int32_t rr[4], gg[4];
      double xv[4];
      uint32_t pos[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int32_t e = e0 + 32 * u + lane;
        const bool in = e < e1;
        rr[u] = in ? __ldg(oi + e) : -1;
        xv[u] = in ? __ldg(ox + e) : 0.0;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) gg[u] = rr[u] >= 0 ? __ldg(tmap + rr[u]) : -1;
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (gg[u] >= 0) pos[u] = base + rp[gg[u]] + atomicAdd(cur + gg[u], 1u);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        if (gg[u] < 0) continue;
        double v = xform_value(mode, xv[u], a0, a1);
        if (mode >= XF_SING) v -= fb;
        const int32_t q = (int32_t)__double2ll_rn(v * sc);
        // a non-zero tail entry that the column's fixed point would flush to zero: the call is redone in fp64
        // (tc_kernels.cu, k_tc_prep_dense); every kernel after this one looks at the flag before it starts
        if (q == 0 && v != 0.0 && skip_if) atomicExch(const_cast<int*>(skip_if), 1);
        ent[pos[u]] = make_uint2((uint32_t)q, cell);
      }
    }
  }
}

// fills by kernel, not cudaMemsetAsync: a memset may be scheduled on a copy engine and then waits behind the
// gigabyte result blocks that are leaving for the host on another stream
__global__ void __launch_bounds__(256) k_fill_u32(uint32_t* __restrict__ p, uint32_t v, int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) p[i] = v;
}

// One addend {q, cell} into a 64-bit accumulator kept as a u32 low word and a 16-bit high counter.  The low word
// takes a shared-memory atomic that returns the old value; the high counter moves by d = carry out of the low word
// minus the sign extension of q (-1, 0 or +1), through a no-return atomic on the lane's own predicate.  Every
// atomic sees a consistent old value, so (hi << 32) + lo is the exact int64 sum whatever order the adds land in,
// and lanes of one step may share a cell.
// There are no 16-bit atomics: the counters of cells 2i and 2i + 1 are the two halves of hiw[i], each biased by
// 2^15 so that a borrow never reaches the other half.  A set has fewer than 2^16 tail members (tail ids are u16)
// and each adds at most one entry to a cell, |q| < 2^30, so every partial sum of a cell lies in (-2^46, 2^46) and
// its high word in [-2^14, 2^14); the counter runs ahead of or behind that by the few adds of one warp whose
// second atomic has not landed yet, far inside the 2^15 either side that the bias allows.
constexpr uint32_t HI_BIAS = 0x8000u, HI_BIAS2 = 0x80008000u;

__device__ __forceinline__ void acc_add(uint32_t lo_sa, uint32_t hi_sa, const uint2 rec) {
  const uint32_t q = rec.x, c = rec.y;
  uint32_t old, d;
  asm volatile("atom.shared.add.u32 %0, [%1], %2;" : "=r"(old) : "r"(lo_sa + c * 4u), "r"(q) : "memory");
  asm("{\n\t.reg .u32 t;\n\tadd.cc.u32 t, %1, %2;\n\taddc.u32 %0, %3, 0;\n\t}"  // d = carry + (q >> 31)
      : "=r"(d) : "r"(old), "r"(q), "r"((uint32_t)((int32_t)q >> 31)));
  // d << 16 * (c & 1): the funnel shift takes its amount modulo 32
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %1, 0;\n\t@p red.shared.add.u32 [%0], %2;\n\t}"
               ::"r"(hi_sa + (c & ~1u) * 2u), "r"(d), "r"(__funnelshift_l(0u, d, c << 4)) : "memory");
}

struct TailParams {
  const uint32_t* tptr;    // [S + 1] set -> its tail members
  const uint16_t* tidx;    // tail ids, ascending inside a set
  const int32_t* sorder;   // [S] sets in decreasing order of their tail size
  const uint32_t* rowptr;  // [tiles][Pt + 1]
  const uint32_t* total;   // [tiles]
  const uint2* ent;        // {fixed-point value, cell inside the tile}, gene-major per tile
  int32_t S, Pt, C, tiles;
  long long* tmp;          // [S][ld] int64 sums
  int64_t ld;              // = tiles * C
  unsigned int* counter;   // work counter (zeroed before the launch)
  const int* skip_if;
};

__global__ void __launch_bounds__(TAIL_WARPS * 32, 1) k_tail(const TailParams p) {
  if (p.skip_if && *p.skip_if != 0) return;
  extern __shared__ uint32_t tail_sm[];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int C = p.C;
  // cell c: low word lo[c], high counter in half c & 1 of hiw[c >> 1], biased by 2^15 (see acc_add); scr: the
  // non-empty rows of a member batch
  uint32_t* __restrict__ lo = tail_sm + (size_t)w * C;
  uint32_t* __restrict__ hiw = tail_sm + (size_t)TAIL_WARPS * C + (size_t)w * (C / 2);
  uint2* __restrict__ scr = reinterpret_cast<uint2*>(tail_sm + (size_t)TAIL_WARPS * C * 3 / 2) + w * 32;
  for (int c = lane; c < C / 2; c += 32) {
    lo[2 * c] = 0u;
    lo[2 * c + 1] = 0u;
    hiw[c] = HI_BIAS2;
  }
  __syncwarp();
  const uint32_t lo_sa = (uint32_t)__cvta_generic_to_shared(lo), hi_sa = (uint32_t)__cvta_generic_to_shared(hiw);
  uint32_t le, lt;
  asm("mov.u32 %0, %%lanemask_le;" : "=r"(le));
  asm("mov.u32 %0, %%lanemask_lt;" : "=r"(lt));
  const unsigned nitems = (unsigned)p.tiles * (unsigned)p.S;
  for (;;) {
    unsigned item = 0;
    if (lane == 0) item = atomicAdd(p.counter, 1u);
    item = __shfl_sync(FULL, item, 0);
    if (item >= nitems) break;
    const int t = (int)(item / (unsigned)p.S);
    const int s = p.sorder[item - (unsigned)t * (unsigned)p.S];
    const uint32_t* __restrict__ rp = p.rowptr + (size_t)t * (p.Pt + 1);
    uint32_t base = 0;
    for (int u = lane; u < t; u += 32) base += p.total[u];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) base += __shfl_xor_sync(FULL, base, o);
    const uint2* ent = p.ent + base + lane;
    asm("mov.b64 %0, %0;" : "+l"(ent));  // keeps the lane's base address in a register: one IMAD.WIDE per load
    const uint32_t m0 = p.tptr[s], m1 = p.tptr[s + 1];
    for (uint32_t mb = m0; mb < m1; mb += 32) {
      // lane i looks up the row of member mb + i in this tile
      uint32_t r0 = 0, rn = 0;
      if (mb + lane < m1) {
        const uint32_t g = p.tidx[mb + lane];
        r0 = rp[g];
        rn = rp[g + 1] - r0;
      }
      // the rows of the 32 members, concatenated, form one stream of `total` entries cut into 32-entry segments:
      // lane l of a segment starting at stream position P0 adds entry P0 + l, whatever row it belongs to
      uint32_t incl = rn;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t v = __shfl_up_sync(FULL, incl, o);
        if (lane >= o) incl += v;
      }
      const uint32_t total = __shfl_sync(FULL, incl, 31);
      if (total == 0u) continue;
      // compact the non-empty rows (an empty row would share its start with the next one): lane k holds the k-th
      // non-empty row's start in the stream and its offset in `ent` relative to that start
      const uint32_t ne = __ballot_sync(FULL, rn != 0u);
      __syncwarp();  // the previous batch has read scr
      if (rn != 0u) scr[__popc(ne & lt)] = make_uint2(incl - rn, r0 - (incl - rn));
      __syncwarp();
      const uint2 so = scr[lane];
      const uint32_t start = (uint32_t)lane < (uint32_t)__popc(ne) ? so.x : 0xFFFFFFFFu, off = so.y;
      // rows that start before the current segment, minus one
      int before = -1;
      // the row of each lane's entry: the rows starting inside the segment (one OR over the lanes), counted up to
      // the lane, after the `before` rows that started earlier
      auto fetch = [&](uint32_t P0) {
        uint32_t bit;  // PTX shl yields 0 for a shift of 32 or more
        asm("shl.b32 %0, 1, %1;" : "=r"(bit) : "r"(start - P0));
        const uint32_t m = __reduce_or_sync(FULL, bit);
        const uint32_t o = __shfl_sync(FULL, off, before + __popc(m & le));
        before += __popc(m);
        uint2 rec = make_uint2(0u, (uint32_t)lane);  // padding: adds 0, each lane at its own cell
        if (P0 + lane < total) rec = __ldg(ent + (o + P0));
        return rec;
      };
      // three segments in flight while one is added: entries come from L2, ~350 clocks away
      uint2 q0 = fetch(0u), q1 = fetch(32u), q2 = fetch(64u);
      for (uint32_t P0 = 0;; P0 += 96u) {
        acc_add(lo_sa, hi_sa, q0);
        q0 = fetch(P0 + 96u);
        if (P0 + 32u >= total) break;
        acc_add(lo_sa, hi_sa, q1);
        q1 = fetch(P0 + 128u);
        if (P0 + 64u >= total) break;
        acc_add(lo_sa, hi_sa, q2);
        q2 = fetch(P0 + 160u);
        if (P0 + 96u >= total) break;
      }
    }
    // flush: int64 sums of set s over the tile's cells, two cells per lane, coalesced; re-zero
    __syncwarp();
    long long* __restrict__ o = p.tmp + (size_t)s * p.ld + (size_t)t * C;
    for (int c = lane; c < C / 2; c += 32) {
      const uint2 l = *reinterpret_cast<const uint2*>(lo + 2 * c);
      const uint32_t h = hiw[c];
      const long long v0 = (long long)(((uint64_t)(h & 0xFFFFu) - HI_BIAS) << 32) + l.x;
      const long long v1 = (long long)(((uint64_t)(h >> 16) - HI_BIAS) << 32) + l.y;
      *reinterpret_cast<uint2*>(lo + 2 * c) = make_uint2(0u, 0u);
      hiw[c] = HI_BIAS2;
      __stcs(reinterpret_cast<longlong2*>(o + 2 * c), make_longlong2(v0, v1));
    }
    __syncwarp();
  }
}

}  // namespace

cudaError_t launch_fill_u32(void* p, uint32_t v, int64_t n, cudaStream_t st) {
  if (n <= 0) return cudaSuccess;
  int64_t grid = (n + 255) / 256;
  if (grid > 148 * 8) grid = 148 * 8;
  k_fill_u32<<<(unsigned)grid, 256, 0, st>>>(static_cast<uint32_t*>(p), v, n);
  return cudaGetLastError();
}

int tail_tile_cells() { return 1056; }  // 22 tensor-core cell tiles of 48

size_t tail_smem_bytes() { return (size_t)TAIL_WARPS * (tail_tile_cells() * 6 + 32 * sizeof(uint2)); }

cudaError_t launch_tile_scan(uint32_t* cnt, int32_t Pt, int tiles, uint32_t* rowptr, uint32_t* total, cudaStream_t st) {
  if (tiles <= 0) return cudaSuccess;
  k_tile_scan<<<(unsigned)tiles, 1024, 0, st>>>(cnt, Pt, rowptr, total);
  return cudaGetLastError();
}

cudaError_t launch_tile_place(const int32_t* xp, const int32_t* xe, const int32_t* oi, const double* ox, const double* r0,
                              const int32_t* tmap, const double* colinv, int64_t N, int mode, double a0, double a1,
                              int32_t Pt, const uint32_t* rowptr, const uint32_t* total, uint32_t* cnt, uint2* ent,
                              const int* skip_if, cudaStream_t st) {
  if (N <= 0) return cudaSuccess;
  int64_t grid = (N + 7) / 8;
  if (grid > 148 * 16) grid = 148 * 16;
  k_tile_place<<<(unsigned)grid, 256, 0, st>>>(xp, xe, oi, ox, r0, tmap, colinv, N, mode, a0, a1, Pt, tail_tile_cells(),
                                               rowptr, total, cnt, ent, skip_if);
  return cudaGetLastError();
}

cudaError_t launch_tail(const uint32_t* tptr, const uint16_t* tidx, const int32_t* sorder, const uint32_t* rowptr,
                        const uint32_t* total, const uint2* ent, int32_t S, int32_t Pt, int tiles,
                        long long* tmp, unsigned int* counter, const int* skip_if, cudaStream_t st) {
  if (tiles <= 0 || S <= 0) return cudaSuccess;
  TailParams p{};
  p.tptr = tptr;
  p.tidx = tidx;
  p.sorder = sorder;
  p.rowptr = rowptr;
  p.total = total;
  p.ent = ent;
  p.S = S;
  p.Pt = Pt;
  p.C = tail_tile_cells();
  p.tiles = tiles;
  p.tmp = tmp;
  p.ld = (int64_t)tiles * p.C;
  p.counter = counter;
  p.skip_if = skip_if;
  const size_t smem = tail_smem_bytes();
  cudaError_t e = cudaFuncSetAttribute(k_tail, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  e = launch_fill_u32(counter, 0u, 1, st);
  if (e != cudaSuccess) return e;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  k_tail<<<(unsigned)sms, TAIL_WARPS * 32, smem, st>>>(p);
  return cudaGetLastError();
}

}  // namespace plaidgpu
