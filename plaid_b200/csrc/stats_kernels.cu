// K5 — normalize_medians() (reference R/plaid.R:554-575): per-column medians of the S x N score
// matrix (matrixStats::colMedians(na.rm=TRUE), with and without the zeros), the column minima
// that decide the global `ignore.zero` switch, and the fused fix-up
//   out = alpha * (x - med_j + mean(med)) + beta_s.
//
// Medians are exact order statistics: an MSD radix select on order-preserving 64-bit keys
// (11-bit digits, shared-memory histograms), which stops as soon as the bucket holding the
// wanted rank is small and finishes by ranking the few candidates directly.  Up to four ranks
// are selected together (two middles x {all values, non-zero values}); removing the zeros only
// shifts ranks because the zeros are one contiguous block of the sorted column.
#include "common.cuh"

#include <math.h>
#include <stdio.h>
#include <stdlib.h>

namespace plaidgpu {

namespace {

constexpr int NT = 256;     // threads per column CTA
constexpr int NBIN = 2048;  // 11-bit digits
constexpr int NTGT = 4;     // simultaneous order statistics
constexpr int CAND = 256;   // finish by direct ranking below this bucket size
constexpr int NDIG = 6;     // 11+11+11+11+11+9 bits
constexpr unsigned long long ZERO_KEY = 0x8000000000000000ull;

__device__ __forceinline__ int digit_shift(int d) { return d < 5 ? 53 - 11 * d : 0; }
__device__ __forceinline__ int digit_bits(int d) { return d < 5 ? 11 : 9; }


// Cooperative search of the histogram bin that holds rank k: every thread sums nb/NT consecutive
// bins, warp 0 scans the NT partial sums and walks the winning group.  All NT threads must call.
struct BinHit { int bin; unsigned before, count; };
__device__ BinHit find_bin(const unsigned* __restrict__ hist, int nb, unsigned k, unsigned* __restrict__ part,
                           BinHit* __restrict__ slot) {
  const int tid = threadIdx.x, lane = tid & 31;
  const int per = nb / NT;  // 8 (2048 bins) or 2 (512 bins)
  unsigned sum = 0;
  for (int i = 0; i < per; ++i) sum += hist[tid * per + i];
  part[tid] = sum;
  __syncthreads();
  if (tid < 32) {
    unsigned loc = 0;
#pragma unroll
    for (int i = 0; i < NT / 32; ++i) loc += part[lane * (NT / 32) + i];
    unsigned incl = loc;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned v = __shfl_up_sync(FULL, incl, o);
      if (lane >= o) incl += v;
    }
    const unsigned hit = __ballot_sync(FULL, k < incl);
    const int l = hit ? __ffs(hit) - 1 : 31;
    if (lane == l) {
      unsigned before = incl - loc;
      int g = lane * (NT / 32);
      while (g < lane * (NT / 32) + NT / 32 - 1 && k >= before + part[g]) before += part[g++];
      int b = g * per;
      while (b < g * per + per - 1 && k >= before + hist[b]) before += hist[b++];
      slot->bin = b;
      slot->before = before;
      slot->count = hist[b];
    }
  }
  __syncthreads();
  return *slot;
}

struct StatsSmem {
  unsigned hist[NTGT][NBIN];
  unsigned long long cand[NTGT][CAND];
  unsigned long long prefix[NTGT];  // key bits decided so far (high digits)
  unsigned long long result[NTGT];
  unsigned k[NTGT];      // remaining 0-based rank inside the current bucket
  unsigned cnt[NTGT];    // size of the current bucket
  unsigned ncand[NTGT];
  int active[NTGT];
  int depth[NTGT];       // digits decided
  unsigned red_u[NT / 32][3];
  unsigned long long red_k[NT / 32];
  unsigned nnan, nzero, nneg;
  unsigned long long minkey;
  unsigned part[NT];
  BinHit hit;
};

// All threads: the bin of hist[g] (digit d) that holds rank k[g]; updates prefix / k / cnt / depth.
__device__ void pick_bin(StatsSmem& s, int g, int d) {
  const BinHit h = find_bin(s.hist[g], 1 << digit_bits(d), s.k[g], s.part, &s.hit);
  __syncthreads();
  if (threadIdx.x == 0) {
    s.prefix[g] |= (unsigned long long)h.bin << digit_shift(d);
    s.k[g] -= h.before;
    s.cnt[g] = h.count;
    s.depth[g] = d + 1;
  }
  __syncthreads();
}

// cols == nullptr: columns 0..N-1; else the N columns listed in cols (the fast path's rejects)
__global__ void __launch_bounds__(NT) k_colstats(const double* __restrict__ x, int64_t ld, int32_t S,
                                                 int64_t N, const int64_t* __restrict__ cols,
                                                 double* __restrict__ med_all,
                                                 double* __restrict__ med_nz,
                                                 double* __restrict__ colmin) {
  extern __shared__ unsigned char smem_raw[];
  StatsSmem& s = *reinterpret_cast<StatsSmem*>(smem_raw);
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;

  for (int64_t it = blockIdx.x; it < N; it += gridDim.x) {
    const int64_t j = cols ? cols[it] : it;
    const double* __restrict__ c = x + j * ld;

    // ---- pass 1: top-digit histogram + NaN / zero counts + min -------------------------
    for (int i = tid; i < NBIN; i += NT) s.hist[0][i] = 0;
    __syncthreads();
    unsigned nnan = 0, nzero = 0;
    unsigned long long mink = ~0ull;
    int runbin = -1;
    unsigned runcnt = 0;
    for (int l = tid; l < S; l += NT) {
      const double v = c[l];
      if (v != v) {
        ++nnan;
        continue;
      }
      const unsigned long long key = key_of(v);
      nzero += (key == ZERO_KEY);
      mink = key < mink ? key : mink;
      const int bin = (int)(key >> 53);
      if (bin != runbin) {  // run-length aggregation: the scores of a column share 1-3 binades
        if (runcnt) atomicAdd(&s.hist[0][runbin], runcnt);
        runbin = bin;
        runcnt = 0;
      }
      ++runcnt;
    }
    if (runcnt) atomicAdd(&s.hist[0][runbin], runcnt);
    __syncthreads();
    // negatives = keys with the top bit clear = bins [0, NBIN/2)
    unsigned nneg = 0;
    for (int i = tid; i < NBIN / 2; i += NT) nneg += s.hist[0][i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      nnan += __shfl_xor_sync(FULL, nnan, o);
      nzero += __shfl_xor_sync(FULL, nzero, o);
      nneg += __shfl_xor_sync(FULL, nneg, o);
      const unsigned long long mk = __shfl_xor_sync(FULL, mink, o);
      mink = mk < mink ? mk : mink;
    }
    if (lane == 0) {
      s.red_u[wid][0] = nnan;
      s.red_u[wid][1] = nzero;
      s.red_u[wid][2] = nneg;
      s.red_k[wid] = mink;
    }
    __syncthreads();
    if (tid == 0) {
      unsigned a = 0, z = 0, ng = 0;
      unsigned long long mk = ~0ull;
      for (int i = 0; i < NT / 32; ++i) {
        a += s.red_u[i][0];
        z += s.red_u[i][1];
        ng += s.red_u[i][2];
        mk = s.red_k[i] < mk ? s.red_k[i] : mk;
      }
      s.nnan = a;
      s.nzero = z;
      s.nneg = ng;
      s.minkey = mk;
      const unsigned nvalid = (unsigned)S - a;
      for (int g = 0; g < NTGT; ++g) {
        s.active[g] = 0;
        s.prefix[g] = 0;
        s.ncand[g] = 0;
        s.cnt[g] = nvalid;
        s.depth[g] = 0;
        s.k[g] = 0;
        s.result[g] = 0;
      }
      // targets: overall 0-based ranks among the sorted non-NaN values
      if (nvalid > 0) {
        s.active[0] = 1;
        s.k[0] = (nvalid - 1) / 2;
        s.active[1] = 1;
        s.k[1] = nvalid / 2;  // == k[0] when the count is odd
      }
      const unsigned m2 = nvalid - z;
      if (m2 > 0) {
        const unsigned r0 = (m2 - 1) / 2, r1 = m2 / 2;
        s.active[2] = 1;
        s.k[2] = r0 < ng ? r0 : r0 + z;
        s.active[3] = 1;
        s.k[3] = r1 < ng ? r1 : r1 + z;
      }
    }
    __syncthreads();
    // digit 0 was histogrammed once for all targets
    for (int g = 1; g < NTGT; ++g)
      if (s.active[g])
        for (int i = tid; i < NBIN; i += NT) s.hist[g][i] = s.hist[0][i];
    __syncthreads();
    for (int g = 0; g < NTGT; ++g)
      if (s.active[g]) pick_bin(s, g, 0);

    // ---- refine digit by digit while a bucket is large (a target that stops never resumes) --
    for (int d = 1; d < NDIG; ++d) {
      bool need = false;
#pragma unroll
      for (int g = 0; g < NTGT; ++g) need |= (s.active[g] && s.cnt[g] > CAND);
      if (!need) break;
      const int sh = digit_shift(d), nb = 1 << digit_bits(d);
      const int psh = digit_shift(d - 1);  // bits >= psh are decided for refining targets
      bool ref[NTGT];
      unsigned long long pf[NTGT];
#pragma unroll
      for (int g = 0; g < NTGT; ++g) {
        ref[g] = s.active[g] && s.cnt[g] > CAND;
        pf[g] = s.prefix[g] >> psh;
        if (ref[g])
          for (int i = tid; i < nb; i += NT) s.hist[g][i] = 0;
      }
      __syncthreads();
      for (int l = tid; l < S; l += NT) {
        const double v = c[l];
        if (v != v) continue;
        const unsigned long long key = key_of(v);
        const unsigned long long hi = key >> psh;
        const unsigned bin = (unsigned)(key >> sh) & (unsigned)(nb - 1);
#pragma unroll
        for (int g = 0; g < NTGT; ++g)
          if (ref[g] && hi == pf[g]) atomicAdd(&s.hist[g][bin], 1u);
      }
      __syncthreads();
      for (int g = 0; g < NTGT; ++g)
        if (ref[g]) pick_bin(s, g, d);
    }

    // ---- collect the candidates of every unfinished target and rank them directly ---------
    bool collect = false;
    bool col[NTGT];
    unsigned long long pf[NTGT];
    int psh_g[NTGT];
#pragma unroll
    for (int g = 0; g < NTGT; ++g) {
      col[g] = s.active[g] && s.depth[g] < NDIG;
      psh_g[g] = digit_shift(s.depth[g] > 0 ? s.depth[g] - 1 : 0);
      pf[g] = s.prefix[g] >> psh_g[g];
      collect |= col[g];
      if (s.active[g] && s.depth[g] == NDIG && tid == 0) s.result[g] = s.prefix[g];
    }
    if (collect) {
      for (int l = tid; l < S; l += NT) {
        const double v = c[l];
        if (v != v) continue;
        const unsigned long long key = key_of(v);
#pragma unroll
        for (int g = 0; g < NTGT; ++g)
          if (col[g] && (key >> psh_g[g]) == pf[g]) {
            const unsigned pos = atomicAdd(&s.ncand[g], 1u);
            if (pos < CAND) s.cand[g][pos] = key;
          }
      }
      __syncthreads();
#pragma unroll
      for (int g = 0; g < NTGT; ++g) {
        if (!col[g]) continue;
        const unsigned n = min(s.ncand[g], (unsigned)CAND);
        if ((unsigned)tid < n) {
          const unsigned long long mine = s.cand[g][tid];
          unsigned r = 0;
          for (unsigned u = 0; u < n; ++u) {
            const unsigned long long o = s.cand[g][u];
            r += (o < mine) || (o == mine && u < (unsigned)tid);
          }
          if (r == s.k[g]) s.result[g] = mine;
        }
      }
    }
    __syncthreads();
    if (tid == 0) {
      const unsigned nvalid = (unsigned)S - s.nnan;
      double ma = nan(""), mz = 0.0;
      if (nvalid > 0) {
        const double a = value_of(s.result[0]), b = value_of(s.result[1]);
        ma = (nvalid & 1u) ? a : (a + b) / 2.0;
      }
      const unsigned m2 = nvalid - s.nzero;
      if (m2 > 0) {
        const double a = value_of(s.result[2]), b = value_of(s.result[3]);
        mz = (m2 & 1u) ? a : (a + b) / 2.0;
        if (mz != mz) mz = 0.0;  // middles -inf and +inf: NA -> 0 like an empty column (R/plaid.R:561-566)
      }
      med_all[j] = ma;
      med_nz[j] = mz;
      colmin[j] = nvalid > 0 ? value_of(s.minkey) : INFINITY;
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------
// Fast path: ONE pass over the column.  A strided sample of 1024 keys is sorted in shared memory and
// gives, for each of the two medians, a bracket [lo, hi] of sample order statistics +-2.5 sigma around
// the wanted quantile.  The single full pass counts keys below lo / equal to lo / equal to hi and
// collects the keys strictly inside (lo, hi) in shared memory (a few % of the column); once the exact
// counts are known the wanted ranks are located in {==lo | inside | ==hi} and selected exactly by a
// radix select over the collected keys.  Any column whose ranks fall outside the bracket (p ~ 1 %)
// or whose candidates overflow is flagged and redone by the three-pass kernel above: exactness never
// depends on the sample.
constexpr int SAMP = 1024;
constexpr int WCAP = 416;             // candidate slots per warp and bracket (expected ~300)
constexpr int CCAP = WCAP * (NT / 32); // candidate slots per bracket

struct Stats2Smem {
  union {  // the sorted sample is dead once the brackets are known
    unsigned long long samp[SAMP];
    unsigned hist[2][NBIN];
  };
  unsigned wcnt[2][NT / 32];
  unsigned long long lo[2], hi[2];
  unsigned below[2], eqlo[2], eqhi[2], ncand[2];
  unsigned nnan, nzero, nneg;
  unsigned long long minkey;
  unsigned long long res[2][2];
  int ok[2];
  // scratch of the list select
  unsigned long long prefix[2];
  unsigned k[2], cnt[2];
  int depth[2];
  unsigned nsmall;
  unsigned long long small[64];
  unsigned part[NT];
  BinHit hit;
  // [bracket][warp][WCAP]: every warp appends to its own segment.  LAST member: a launch that wants one
  // median only allocates cand[0] (and uses it for whichever bracket is live) -> more CTAs per SM
  unsigned long long cand[2][CCAP];
};
constexpr size_t STATS2_SMEM_ONE = sizeof(Stats2Smem) - sizeof(unsigned long long) * CCAP;

__device__ void sort_sample(unsigned long long* k, int n) {  // n = power of two, all threads
  for (int size = 2; size <= n; size <<= 1) {
    const int hs = size >> 1;
    for (int q = threadIdx.x; q < n / 2; q += blockDim.x) {
      const int o = q & (hs - 1), base = (q & ~(hs - 1)) << 1;
      const int i = base + o, l = base + size - 1 - o;
      const unsigned long long a = k[i], b = k[l];
      if (a > b) { k[i] = b; k[l] = a; }
    }
    __syncthreads();
    for (int stride = size >> 2; stride >= 1; stride >>= 1) {
      for (int q = threadIdx.x; q < n / 2; q += blockDim.x) {
        const int i = ((q & ~(stride - 1)) << 1) | (q & (stride - 1)), l = i + stride;
        const unsigned long long a = k[i], b = k[l];
        if (a > b) { k[i] = b; k[l] = a; }
      }
      __syncthreads();
    }
  }
}

// exact selection of ranks ka <= kb (kb - ka <= 1) among n keys in shared memory (radix, 11-bit digits);
// every key lies in (klo, khi), so the digits klo and khi share are decided up front
__device__ void select_from_list(Stats2Smem& s, const unsigned long long* list, const unsigned* wcnt, unsigned ntot,
                                 unsigned ka, unsigned kb, unsigned long long klo, unsigned long long khi,
                                 unsigned long long* out2) {
  const int tid = threadIdx.x;
  const unsigned n = CCAP;  // slots; slot i is live iff (i % WCAP) < wcnt[i / WCAP]
  auto live = [&](unsigned i) { return (i % WCAP) < wcnt[i / WCAP]; };
  int d0 = 0;
  while (d0 < NDIG && (klo >> digit_shift(d0)) == (khi >> digit_shift(d0))) ++d0;
  if (tid == 0) {
    const unsigned long long common = d0 > 0 ? (klo >> digit_shift(d0 - 1)) << digit_shift(d0 - 1) : 0ull;
    s.prefix[0] = s.prefix[1] = common;
    s.k[0] = ka; s.k[1] = kb;
    s.cnt[0] = s.cnt[1] = ntot;
    s.depth[0] = s.depth[1] = d0;
  }
  __syncthreads();
  for (int d = d0; d < NDIG; ++d) {
    const bool r0 = s.cnt[0] > 32, r1 = s.cnt[1] > 32;
    if (!r0 && !r1) break;
    const int sh = digit_shift(d), nb = 1 << digit_bits(d);
    const int psh = d > 0 ? digit_shift(d - 1) : 63;
    const unsigned long long p0 = d > 0 ? s.prefix[0] >> psh : 0, p1 = d > 0 ? s.prefix[1] >> psh : 0;
    __syncthreads();
    for (int i = tid; i < nb; i += NT) { s.hist[0][i] = 0; s.hist[1][i] = 0; }
    __syncthreads();
    for (unsigned i = tid; i < n; i += NT) {
      if (!live(i)) continue;
      const unsigned long long key = list[i];
      const unsigned long long hi = d > 0 ? key >> psh : 0;
      const unsigned bin = (unsigned)(key >> sh) & (unsigned)(nb - 1);
      if (r0 && hi == p0) atomicAdd(&s.hist[0][bin], 1u);
      if (r1 && hi == p1) atomicAdd(&s.hist[1][bin], 1u);
    }
    __syncthreads();
    for (int g = 0; g < 2; ++g) {
      if (!(g == 0 ? r0 : r1)) continue;
      const BinHit h = find_bin(s.hist[g], nb, s.k[g], s.part, &s.hit);
      __syncthreads();
      if (tid == 0) {
        s.prefix[g] |= (unsigned long long)h.bin << sh;
        s.k[g] -= h.before;
        s.cnt[g] = h.count;
        s.depth[g] = d + 1;
      }
      __syncthreads();
    }
  }
  // finish each target by direct ranking inside its bucket (<= 32 keys, or a fully decided key)
  for (int g = 0; g < 2; ++g) {
    if (s.depth[g] == NDIG) {
      if (tid == 0) out2[g] = s.prefix[g];
      __syncthreads();
      continue;
    }
    const int psh = s.depth[g] > 0 ? digit_shift(s.depth[g] - 1) : 63;
    const unsigned long long pf = s.depth[g] > 0 ? s.prefix[g] >> psh : 0;
    if (tid == 0) s.nsmall = 0;
    __syncthreads();
    for (unsigned i = tid; i < n; i += NT) {
      if (!live(i)) continue;
      const unsigned long long mine = list[i];
      if ((s.depth[g] > 0 ? mine >> psh : 0) != pf) continue;
      const unsigned q = atomicAdd(&s.nsmall, 1u);
      if (q < 64) s.small[q] = mine;
    }
    __syncthreads();
    const unsigned m = min(s.nsmall, 64u);
    if ((unsigned)tid < m) {
      const unsigned long long mine = s.small[tid];
      unsigned r = 0;
      for (unsigned u = 0; u < m; ++u) {
        const unsigned long long o = s.small[u];
        r += (o < mine) || (o == mine && u < (unsigned)tid);
      }
      if (r == s.k[g]) out2[g] = mine;
    }
    __syncthreads();
  }
}

// DO0 / DO1: which medians are wanted (all valid values / the non-zero values).  The caller usually knows
// which one normalize_medians will use (R/plaid.R:556-557) before this pass; the unused bracket is compiled out.
template <bool DO0, bool DO1>
__global__ void __launch_bounds__(NT) k_colstats_fast(const double* __restrict__ x, int64_t ld, int32_t S, int64_t N,
                                                      double* __restrict__ med_all, double* __restrict__ med_nz,
                                                      double* __restrict__ colmin, int* __restrict__ fail_count,
                                                      int64_t* __restrict__ fail_list) {
  extern __shared__ unsigned char smem_raw2[];
  Stats2Smem& s = *reinterpret_cast<Stats2Smem*>(smem_raw2);
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const unsigned lt = (1u << lane) - 1u;

  for (int64_t j = blockIdx.x; j < N; j += gridDim.x) {
    const double* __restrict__ c = x + j * ld;
    // ---- sample ----
    for (int i = tid; i < SAMP; i += NT) {
      const int pos = (int)(((int64_t)i * S) / SAMP);
      const double v = c[pos];
      s.samp[i] = (v != v) ? ~0ull : key_of(v);
    }
    if (tid == 0) {
      s.nnan = s.nzero = s.nneg = 0;
      s.minkey = ~0ull;
      for (int g = 0; g < 2; ++g) { s.below[g] = s.eqlo[g] = s.eqhi[g] = s.ncand[g] = 0; s.ok[g] = 1; }
    }
    __syncthreads();
    sort_sample(s.samp, SAMP);
    if (tid == 0) {
      // valid sample entries [0, mv); zero block [zs, ze)
      int mv = SAMP;
      {  // NaN keys (~0) sorted last
        int lo = 0, hi = SAMP;
        while (lo < hi) { const int mid = (lo + hi) >> 1; if (s.samp[mid] != ~0ull) lo = mid + 1; else hi = mid; }
        mv = lo;
      }
      int zs, ze;
      {
        int lo = 0, hi = mv;
        while (lo < hi) { const int mid = (lo + hi) >> 1; if (s.samp[mid] < ZERO_KEY) lo = mid + 1; else hi = mid; }
        zs = lo;
        hi = mv;
        while (lo < hi) { const int mid = (lo + hi) >> 1; if (s.samp[mid] <= ZERO_KEY) lo = mid + 1; else hi = mid; }
        ze = lo;
      }
      // bracket g = 0: median of all valid values; g = 1: median of the non-zero values
      for (int g = 0; g < 2; ++g) {
        if (!(g == 0 ? DO0 : DO1)) {
          s.lo[g] = s.hi[g] = 0ull;
          continue;
        }
        const int mcount = g == 0 ? mv : mv - (ze - zs);
        if (mcount < 48) {  // too few sample points: take everything (the candidate cap decides)
          s.lo[g] = key_of(-INFINITY);
          s.hi[g] = key_of(INFINITY);
          continue;
        }
        const double mid = 0.5 * (double)(mcount - 1);
        const double delta = 1.25 * sqrt((double)mcount) + 2.0;  // 2.5 sigma of a binomial(m, 1/2) rank
        int a = (int)floor(mid - delta), b = (int)ceil(mid + delta);
        unsigned long long klo = key_of(-INFINITY), khi = key_of(INFINITY);
        if (a >= 0) {
          if (g == 1 && a >= zs) a += ze - zs;
          klo = s.samp[a];
        }
        if (b <= mcount - 1) {
          if (g == 1 && b >= zs) b += ze - zs;
          khi = s.samp[b];
        }
        s.lo[g] = klo;
        s.hi[g] = khi;
      }
    }
    __syncthreads();
    // brackets as doubles: one DSETP per test instead of a 64-bit key compare; keys are only built
    // for the few rows that land inside a bracket
    const double lo0 = value_of(s.lo[0]), hi0 = value_of(s.hi[0]), lo1 = value_of(s.lo[1]), hi1 = value_of(s.hi[1]);
    const float lo0f = __double2float_rd(lo0), hi0f = __double2float_ru(hi0);
    const float lo1f = __double2float_rd(lo1), hi1f = __double2float_ru(hi1);
    // ---- the one full pass ----
    unsigned nnan = 0, nzero = 0, nneg = 0, bel0 = 0, bel1 = 0, el0 = 0, el1 = 0, eh0 = 0, eh1 = 0;
    double minv = INFINITY;
    unsigned wc0 = 0, wc1 = 0;  // this warp's candidate counts (warp-uniform)
    unsigned long long* __restrict__ seg0 = s.cand[0] + wid * WCAP;
    unsigned long long* __restrict__ seg1 = s.cand[(DO0 && DO1) ? 1 : 0] + wid * WCAP;
    constexpr int UNR = 8;  // loads of 8 rows are issued before any of them is consumed
    for (int l0 = 0; l0 < S; l0 += NT * UNR) {
      double vv[UNR];
#pragma unroll
      for (int u = 0; u < UNR; ++u) {
        const int l = l0 + u * NT + tid;
        vv[u] = (l < S) ? __ldcs(c + l) : INFINITY;  // +inf padding is subtracted below
      }
#pragma unroll
      for (int u = 0; u < UNR; ++u) {
        const double v = vv[u];
        // fp32 filter (fp64 compares run on the slow pipe): rn(v) < rd(lo) implies v < lo, rn(v) > ru(hi)
        // implies v > hi; whatever the filter cannot decide goes to the exact path below
        const float f = __double2float_rn(v);
        const bool isnan_ = f != f;
        const unsigned long long bits = (unsigned long long)__double_as_longlong(v);
        const bool isz = (bits << 1) == 0ull;
        nnan += isnan_;
        nzero += isz;
        minv = fmin(minv, v);
        const bool lt0 = DO0 && f < lo0f, gt0 = DO0 && f > hi0f;
        const bool lt1 = DO1 && f < lo1f, gt1 = DO1 && f > hi1f;
        if (DO0) bel0 += lt0;
        if (DO1) bel1 += lt1 && !isz;
        const bool mid0 = DO0 && !(lt0 || gt0 || isnan_);
        const bool mid1 = DO1 && !(lt1 || gt1 || isnan_ || isz);
        const unsigned mm = __ballot_sync(FULL, mid0 || mid1);
        if (mm) {
          // exact tests for the undecided rows; every warp appends to its own segment (no atomics)
          const bool live = (l0 + u * NT + tid) < S;
          const bool b0 = live && mid0 && v < lo0, b1 = live && mid1 && v < lo1;  // filter inconclusive, exact says below
          bel0 += b0;
          bel1 += b1;
          el0 += live && mid0 && v == lo0;
          eh0 += live && mid0 && v == hi0 && hi0 != lo0;
          el1 += live && mid1 && v == lo1;
          eh1 += live && mid1 && v == hi1 && hi1 != lo1;
          const bool in0 = live && mid0 && v > lo0 && v < hi0;
          const bool in1 = live && mid1 && v > lo1 && v < hi1;
          const unsigned m0 = __ballot_sync(FULL, in0), m1 = __ballot_sync(FULL, in1);
          if (m0 | m1) {
            const unsigned long long key = key_of(v);
            const unsigned p0 = wc0 + __popc(m0 & lt), p1 = wc1 + __popc(m1 & lt);
            if (in0 && p0 < WCAP) seg0[p0] = key;
            if (in1 && p1 < WCAP) seg1[p1] = key;
            wc0 += __popc(m0);
            wc1 += __popc(m1);
          }
        }
      }
    }
    if (lane == 0) {
      s.wcnt[0][wid] = wc0;
      s.wcnt[1][wid] = wc1;
      atomicAdd(&s.ncand[0], min(wc0, (unsigned)WCAP));
      atomicAdd(&s.ncand[1], min(wc1, (unsigned)WCAP));
      if (wc0 > WCAP || wc1 > WCAP) s.ok[0] = 0;  // segment overflow: exact fallback
    }
    // rows past the end were loaded as +inf: they are neither NaN, zero nor negative, never below a bracket,
    // and only count as "== hi" when hi is +inf, which the `live` test above already excludes
    unsigned long long mink = minv == INFINITY ? ~0ull : key_of(minv);
    // block totals
    auto wsum = [&](unsigned v) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
      return v;
    };
    nnan = wsum(nnan); nzero = wsum(nzero); nneg = wsum(nneg);
    bel0 = wsum(bel0); bel1 = wsum(bel1); el0 = wsum(el0); el1 = wsum(el1); eh0 = wsum(eh0); eh1 = wsum(eh1);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const unsigned long long mk = __shfl_xor_sync(FULL, mink, o);
      mink = mk < mink ? mk : mink;
    }
    if (lane == 0) {
      atomicAdd(&s.nnan, nnan); atomicAdd(&s.nzero, nzero); atomicAdd(&s.nneg, nneg);
      atomicAdd(&s.below[0], bel0); atomicAdd(&s.below[1], bel1);
      atomicAdd(&s.eqlo[0], el0); atomicAdd(&s.eqlo[1], el1);
      atomicAdd(&s.eqhi[0], eh0); atomicAdd(&s.eqhi[1], eh1);
      atomicMin(&s.minkey, mink);
    }
    __syncthreads();
    // ---- locate the wanted ranks ----
    const unsigned nvalid = (unsigned)S - s.nnan;
    const unsigned cnt[2] = {nvalid, nvalid - s.nzero};
    bool good = true;
    for (int g = 0; g < 2; ++g) {
      if (!(g == 0 ? DO0 : DO1)) continue;
      if (cnt[g] == 0) continue;
      const unsigned ka = (cnt[g] - 1) / 2, kb = cnt[g] / 2;
      const unsigned b = s.below[g], e1 = b + s.eqlo[g], nin = s.ncand[g], e2 = e1 + nin, e3 = e2 + s.eqhi[g];
      if (!s.ok[0] || nin > CCAP || ka < b || kb >= e3) {
        good = false;
        continue;
      }
      // both ranks inside {==lo | inside | ==hi}
      const bool a_in = ka >= e1 && ka < e2, b_in = kb >= e1 && kb < e2;
      if (a_in || b_in) {
        const unsigned qa = a_in ? ka - e1 : kb - e1, qb = b_in ? kb - e1 : ka - e1;
        select_from_list(s, s.cand[(DO0 && DO1) ? g : 0], s.wcnt[g], nin, qa < qb ? qa : qb, qa < qb ? qb : qa, s.lo[g], s.hi[g], s.res[g]);
        // res[g][0] = smaller requested rank, res[g][1] = larger
      }
      __syncthreads();
      if (tid == 0) {
        unsigned long long ra, rb;
        if (ka < e1) ra = s.lo[g]; else if (ka < e2) ra = s.res[g][0]; else ra = s.hi[g];
        if (kb < e1) rb = s.lo[g]; else if (kb < e2) rb = (a_in ? s.res[g][1] : s.res[g][0]); else rb = s.hi[g];
        s.res[g][0] = ra;
        s.res[g][1] = rb;
      }
      __syncthreads();
    }
    if (tid == 0) {
      if (!good) {
        const int slot = atomicAdd(fail_count, 1);
        fail_list[slot] = j;
      } else {
        double ma = nan(""), mz = 0.0;
        if (DO0 && cnt[0] > 0) {
          const double a = value_of(s.res[0][0]), b = value_of(s.res[0][1]);
          ma = (cnt[0] & 1u) ? a : (a + b) / 2.0;
        }
        if (DO1 && cnt[1] > 0) {
          const double a = value_of(s.res[1][0]), b = value_of(s.res[1][1]);
          mz = (cnt[1] & 1u) ? a : (a + b) / 2.0;
          if (mz != mz) mz = 0.0;  // middles -inf and +inf (see k_colstats)
        }
        if (DO0) med_all[j] = ma;
        if (DO1) med_nz[j] = mz;
        colmin[j] = nvalid > 0 ? value_of(s.minkey) : INFINITY;
      }
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------
// Single-median variant of the one-pass kernel (the launch normalize_medians needs once the median flavour is
// known — every scoring call).  The bracket lives entirely in FP32: rn(.) is monotone, so f(v1) < f(v2) implies
// v1 < v2 and the three classes {f < lo}, {lo <= f <= hi}, {f > hi} are ordered by exact value — the full pass
// needs no fp64 test at all: one F2F, two FSETP, a predicated count and (for ~8 % of the rows) a predicated
// store of the raw bits into the thread's PRIVATE candidate slots (slot k of thread t = cand[k * NT + t]: no
// ballots, no atomics, conflict-free).  The bracket ends need not be sample values either: a two-digit radix
// select over the 1024 float keys of the sample (22 of 32 bits) replaces the bitonic sort; the ends are the bin
// edges around the wanted sample ranks.  The wanted ranks are then selected exactly among the candidates
// (doubles) by a radix select that starts at the first bit in which the bracket ends differ.  Rejects (rank
// outside the bracket, slot overflow, any NaN in the column) go to the three-pass kernel as before.
constexpr int TCAP = 20;   // private candidate slots per thread (expected ~7-10; moved out beyond 16)
constexpr int OVF = 512;   // shared overflow slots (threads whose private slots are full: ~2 % of the threads; 256 slots
                           // overflowed in 0.8 % of the C4 columns, 512 in none: rejects 1.7 % -> 0.9 %)

struct Stats3Smem {
  // sampling phase scratch lives in cand (not yet in use): samp[SAMP] | h1[NBIN] | h2a[NBIN] | h2b[NBIN] (28 KB)
  unsigned long long cand[TCAP * NT + OVF];
  unsigned hist[NBIN];
  unsigned part[NT];
  BinHit hit;
  float lof, hif;
  unsigned mcount, novf, below, nzero, ncand, nsmall, cle;
  int bad;
  unsigned long long minkey, nxt, resA;
  unsigned long long small[64];
};

__device__ __forceinline__ unsigned fkey_of(float f) {
  const unsigned b = __float_as_uint(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float fvalue_of(unsigned k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

template <bool NZ>
__global__ void __launch_bounds__(NT) k_colstats_one(const double* __restrict__ x, int64_t ld, int32_t S, int64_t N,
                                                     double* __restrict__ med, double* __restrict__ colmin,
                                                     int* __restrict__ fail_count, int64_t* __restrict__ fail_list) {
  extern __shared__ unsigned char smem_raw3[];
  Stats3Smem& s = *reinterpret_cast<Stats3Smem*>(smem_raw3);
  const int tid = threadIdx.x, lane = tid & 31;
  unsigned* const samp = reinterpret_cast<unsigned*>(s.cand);
  unsigned* const h1 = samp + SAMP;
  unsigned* const h2a = h1 + NBIN;
  unsigned* const h2b = h2a + NBIN;

  for (int64_t j = blockIdx.x; j < N; j += gridDim.x) {
    const double* __restrict__ c = x + j * ld;
    // ---- sample: float keys, invalid (NaN, or zero when the zeros are dropped) = ~0 ----
    for (int i = tid; i < 3 * NBIN; i += NT) h1[i] = 0;
    if (tid == 0) {
      s.mcount = s.novf = s.below = s.nzero = s.ncand = 0;
      s.bad = 0;
      s.minkey = ~0ull;
    }
    __syncthreads();
    {
      unsigned mv = 0;
      for (int i = tid; i < SAMP; i += NT) {
        const int pos = (int)(((int64_t)i * S) / SAMP);
        const double v = c[pos];
        const bool valid = (v == v) && !(NZ && v == 0.0);
        const unsigned k = valid ? fkey_of(__double2float_rn(v)) : ~0u;
        samp[i] = k;
        if (valid) {
          atomicAdd(&h1[k >> 21], 1u);
          ++mv;
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) mv += __shfl_xor_sync(FULL, mv, o);
      if (lane == 0 && mv) atomicAdd(&s.mcount, mv);
    }
    __syncthreads();
    const unsigned mcount = s.mcount;
    int ra = -1, rb = -1;  // wanted sample ranks; -1 = open end
    if (mcount >= 48) {
      const double mid = 0.5 * (double)(mcount - 1);
      const double delta = 1.25 * sqrt((double)mcount) + 2.0;  // 2.5 sigma of a binomial(m, 1/2) rank
      const int a = (int)floor(mid - delta), b = (int)ceil(mid + delta);
      if (a >= 0) ra = a;
      if (b <= (int)mcount - 1) rb = b;
    }
    // second digit of the two ends (block-uniform control flow: ra / rb / mcount are uniform)
    BinHit ha{0, 0, 0}, hb{0, 0, 0};
    if (ra >= 0) ha = find_bin(h1, NBIN, (unsigned)ra, s.part, &s.hit);
    __syncthreads();
    if (rb >= 0) hb = find_bin(h1, NBIN, (unsigned)rb, s.part, &s.hit);
    __syncthreads();
    if (ra >= 0 || rb >= 0) {
      for (int i = tid; i < SAMP; i += NT) {
        const unsigned k = samp[i];
        if (k == ~0u) continue;
        const unsigned top = k >> 21, d2 = (k >> 10) & 2047u;
        if (ra >= 0 && top == (unsigned)ha.bin) atomicAdd(&h2a[d2], 1u);
        if (rb >= 0 && top == (unsigned)hb.bin) atomicAdd(&h2b[d2], 1u);
      }
    }
    __syncthreads();
    BinHit ga{0, 0, 0}, gb{0, 0, 0};
    if (ra >= 0) ga = find_bin(h2a, NBIN, (unsigned)ra - ha.before, s.part, &s.hit);
    __syncthreads();
    if (rb >= 0) gb = find_bin(h2b, NBIN, (unsigned)rb - hb.before, s.part, &s.hit);
    __syncthreads();
    if (tid == 0) {
      // bin edges as floats: low edge of the bin holding sample rank a, high edge of the one holding rank b
      float lof = -INFINITY, hif = INFINITY;
      if (ra >= 0) {
        const unsigned klo = ((unsigned)ha.bin << 21) | ((unsigned)ga.bin << 10);
        const float f = fvalue_of(klo);
        if (f == f) lof = f;
      }
      if (rb >= 0) {
        const unsigned khi = ((unsigned)hb.bin << 21) | ((unsigned)gb.bin << 10) | 1023u;
        const float f = fvalue_of(khi);
        if (f == f) hif = f;
      }
      s.lof = lof;
      s.hif = hif;
    }
    __syncthreads();
    const float lof = s.lof, hif = s.hif;
    __syncthreads();  // the sampling scratch (inside cand) is dead from here on

    // ---- the one full pass ----
    unsigned bel = 0, nz = 0, cnt = 0, flushed = 0;
    double minv = INFINITY;
    unsigned long long* const mine = s.cand + tid;
    // a thread whose private slots are nearly full (~2 % of the threads) moves them to the shared overflow area;
    // checked once per 4 rows so the per-row path has no capacity test
    auto flush = [&]() {
      const unsigned base = atomicAdd(&s.novf, cnt);
      for (unsigned k = 0; k < cnt; ++k)
        if (base + k < (unsigned)OVF) s.cand[TCAP * NT + base + k] = mine[k * NT];
      flushed += cnt;
      cnt = 0;
    };
    // zeros (dropped when NZ) have f = +-0: they are "below" iff lo > 0 and inside the bracket iff lo <= 0 <= hi —
    // both uniform per column, so the per-row path only counts them
    const bool zin = NZ && lof <= 0.f && hif >= 0.f;
    auto visit = [&](double v, bool ZIN) {
      const float f = __double2float_rn(v);
      minv = v < minv ? v : minv;             // NaN never selected
      const bool lt = f < lof;
      bool cd = !(lt || f > hif);             // NaN: neither -> candidate, rejects the column after the pass
      if (NZ) {
        const unsigned hi = (unsigned)__double2hiint(v), lo = (unsigned)__double2loint(v);
        const bool isz = ((hi + hi) | lo) == 0u;
        nz += isz;
        if (ZIN) cd = cd && !isz;
      }
      bel += lt;
      if (cd) mine[cnt * NT] = (unsigned long long)__double_as_longlong(v);
      cnt += cd;
    };
    constexpr int UNR = 8;  // loads of 8 rows are issued before any of them is consumed
    int l0 = 0;
    for (; l0 + NT * UNR <= S; l0 += NT * UNR) {
      double vv[UNR];
#pragma unroll
      for (int u = 0; u < UNR; ++u) vv[u] = __ldcs(c + l0 + u * NT + tid);
#pragma unroll
      for (int h = 0; h < UNR; h += 4) {
        if (cnt > (unsigned)(TCAP - 4)) flush();
        if (zin) {
#pragma unroll
          for (int u = 0; u < 4; ++u) visit(vv[h + u], true);
        } else {
#pragma unroll
          for (int u = 0; u < 4; ++u) visit(vv[h + u], false);
        }
      }
    }
    for (int l = l0 + tid; l < S; l += NT) {
      if (cnt >= (unsigned)TCAP) flush();
      visit(__ldcs(c + l), zin);
    }
    if (NZ && lof > 0.f) bel -= nz;  // the zeros were counted as below

    // ---- block totals ----
    {
      unsigned tot = cnt + flushed;
      unsigned long long mink = minv == INFINITY ? ~0ull : key_of(minv);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        bel += __shfl_xor_sync(FULL, bel, o);
        nz += __shfl_xor_sync(FULL, nz, o);
        tot += __shfl_xor_sync(FULL, tot, o);
        const unsigned long long mk = __shfl_xor_sync(FULL, mink, o);
        mink = mk < mink ? mk : mink;
      }
      if (lane == 0) {
        atomicAdd(&s.below, bel);
        if (NZ) atomicAdd(&s.nzero, nz);
        atomicAdd(&s.ncand, tot);
        atomicMin(&s.minkey, mink);
      }
    }
    // raw bits -> order-preserving keys in place; any NaN rejects the column
    const unsigned own = cnt < (unsigned)TCAP ? cnt : (unsigned)TCAP;
    {
      bool nan_seen = false;
      for (unsigned k = 0; k < own; ++k) {
        const double v = __longlong_as_double((long long)mine[k * NT]);
        nan_seen |= (v != v);
        mine[k * NT] = key_of(v);
      }
      __syncthreads();  // novf final
      const unsigned novf = s.novf < (unsigned)OVF ? s.novf : (unsigned)OVF;
      for (unsigned i = tid; i < novf; i += NT) {
        const double v = __longlong_as_double((long long)s.cand[TCAP * NT + i]);
        nan_seen |= (v != v);
        s.cand[TCAP * NT + i] = key_of(v);
      }
      if (nan_seen) s.bad = 1;
    }
    __syncthreads();
    const unsigned novf = s.novf;
    const unsigned count = (unsigned)S - (NZ ? s.nzero : 0u);  // valid values the median runs over (no NaN if !bad)
    const unsigned ka = count ? (count - 1) / 2 : 0, kb = count / 2;
    const unsigned below = s.below, ncand = s.ncand;
    bool good = !s.bad && novf <= (unsigned)OVF;
    if (count > 0 && (ka < below || kb >= below + ncand)) good = false;
    unsigned long long A = 0, B = 0;
    if (good && count > 0) {  // block-uniform
      // ---- exact selection of rank qa among the candidates (and its successor if the count is even) ----
      const unsigned qa = ka - below, qb = kb - below;
      // every candidate lies in [lo - 1 ulp(float), hi + 1 ulp(float)]: the bits above the first differing one are shared
      const unsigned long long klo = key_of((double)nextafterf(lof, -INFINITY)), khi = key_of((double)nextafterf(hif, INFINITY));
      int top = 63 - __clzll((long long)((klo ^ khi) | 1ull));  // highest bit that may differ
      unsigned long long pref = 0, pmask = 0;                    // decided bits / which bits are decided (below `top`)
      unsigned k = qa, bucket = ncand;
      int hi_bit = top;  // undecided bits: [0, hi_bit]
      while (bucket > 64 && hi_bit >= 0) {
        const int nb = hi_bit + 1 < 11 ? hi_bit + 1 : 11;
        const int sh = hi_bit + 1 - nb;
        for (int i = tid; i < NBIN; i += NT) s.hist[i] = 0;
        __syncthreads();
        for (unsigned q = 0; q < own; ++q) {
          const unsigned long long key = mine[q * NT];
          if ((key & pmask) == pref) atomicAdd(&s.hist[(unsigned)(key >> sh) & ((1u << nb) - 1u)], 1u);
        }
        for (unsigned i = tid; i < novf; i += NT) {
          const unsigned long long key = s.cand[TCAP * NT + i];
          if ((key & pmask) == pref) atomicAdd(&s.hist[(unsigned)(key >> sh) & ((1u << nb) - 1u)], 1u);
        }
        __syncthreads();
        const BinHit h = find_bin(s.hist, NBIN, k, s.part, &s.hit);
        __syncthreads();
        pref |= (unsigned long long)h.bin << sh;
        pmask |= (unsigned long long)((1u << nb) - 1u) << sh;
        k -= h.before;
        bucket = h.count;
        hi_bit = sh - 1;
      }
      if (hi_bit < 0) {
        A = 0;  // every remaining bit decided: the bucket holds copies of one key; shared high bits added below
        if (tid == 0) s.resA = pref;
      } else {
        if (tid == 0) s.nsmall = 0;
        __syncthreads();
        for (unsigned q = 0; q < own; ++q) {
          const unsigned long long key = mine[q * NT];
          if ((key & pmask) == pref) {
            const unsigned w = atomicAdd(&s.nsmall, 1u);
            if (w < 64) s.small[w] = key;
          }
        }
        for (unsigned i = tid; i < novf; i += NT) {
          const unsigned long long key = s.cand[TCAP * NT + i];
          if ((key & pmask) == pref) {
            const unsigned w = atomicAdd(&s.nsmall, 1u);
            if (w < 64) s.small[w] = key;
          }
        }
        __syncthreads();
        const unsigned m = s.nsmall < 64u ? s.nsmall : 64u;
        if ((unsigned)tid < m) {
          const unsigned long long me = s.small[tid];
          unsigned r = 0;
          for (unsigned u = 0; u < m; ++u) {
            const unsigned long long o = s.small[u];
            r += (o < me) || (o == me && u < (unsigned)tid);
          }
          if (r == k) s.resA = me;
        }
      }
      __syncthreads();
      A = s.resA;
      if (hi_bit < 0) A |= klo & ~((top >= 63) ? ~0ull : ((2ull << top) - 1ull));  // bits above `top` (shared by all)
      B = A;
      if (qb != qa) {  // successor of A in sorted order: A again if copies of A reach rank qb, else the next key
        if (tid == 0) {
          s.cle = 0;
          s.nxt = ~0ull;
        }
        __syncthreads();
        unsigned le = 0;
        unsigned long long nx = ~0ull;
        for (unsigned q = 0; q < own; ++q) {
          const unsigned long long key = mine[q * NT];
          le += key <= A;
          if (key > A && key < nx) nx = key;
        }
        for (unsigned i = tid; i < novf; i += NT) {
          const unsigned long long key = s.cand[TCAP * NT + i];
          le += key <= A;
          if (key > A && key < nx) nx = key;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          le += __shfl_xor_sync(FULL, le, o);
          const unsigned long long t = __shfl_xor_sync(FULL, nx, o);
          nx = t < nx ? t : nx;
        }
        if (lane == 0) {
          atomicAdd(&s.cle, le);
          atomicMin(&s.nxt, nx);
        }
        __syncthreads();
        B = (qb < s.cle) ? A : s.nxt;
      }
    }
    if (tid == 0) {
      if (!good) {
        const int slot = atomicAdd(fail_count, 1);
        fail_list[slot] = j;
      } else {
        double m = NZ ? 0.0 : nan("");
        if (count > 0) {
          const double a = value_of(A), b = value_of(B);
          m = (count & 1u) ? a : (a + b) / 2.0;
          if (NZ && m != m) m = 0.0;  // middles -inf and +inf (see k_colstats)
        }
        med[j] = m;
        colmin[j] = s.minkey != ~0ull ? value_of(s.minkey) : INFINITY;
      }
    }
    __syncthreads();
  }
}

// out[s, j] = alpha * (x[s, j] - med[j] + c) + beta[s]   for columns j0 <= j < j1
__global__ void __launch_bounds__(256) k_fixup(const double* __restrict__ x, double* __restrict__ out,
                                               int64_t ld, int32_t S, int64_t j0, int64_t j1,
                                               const double* __restrict__ med, double c, double alpha,
                                               const double* __restrict__ beta) {
  for (int64_t j = j0 + blockIdx.x; j < j1; j += gridDim.x) {
    const double shift = (med ? -med[j] : 0.0) + c;
    const double* __restrict__ xi = x + j * ld;
    double* __restrict__ oi = out + j * ld;
    const bool vec = ((((uintptr_t)xi) | ((uintptr_t)oi)) & 15) == 0;
    if (vec) {
      const int S2 = S >> 1;
      const double2* __restrict__ x2 = reinterpret_cast<const double2*>(xi);
      double2* __restrict__ o2 = reinterpret_cast<double2*>(oi);
      for (int l = threadIdx.x; l < S2; l += blockDim.x) {
        double2 v = __ldcs(x2 + l);
        v.x = __dmul_rn(alpha, __dadd_rn(v.x, shift));  // no FMA: the host applies the same fix-up to early-shipped columns
        v.y = __dmul_rn(alpha, __dadd_rn(v.y, shift));
        if (beta) {
          v.x = __dadd_rn(v.x, beta[2 * l]);
          v.y = __dadd_rn(v.y, beta[2 * l + 1]);
        }
        __stcs(o2 + l, v);
      }
      if ((S & 1) && threadIdx.x == 0) {
        double v = __dmul_rn(alpha, __dadd_rn(xi[S - 1], shift));
        if (beta) v = __dadd_rn(v, beta[S - 1]);
        oi[S - 1] = v;
      }
    } else {
      for (int l = threadIdx.x; l < S; l += blockDim.x) {
        double v = __dmul_rn(alpha, __dadd_rn(xi[l], shift));
        if (beta) v = __dadd_rn(v, beta[l]);
        oi[l] = v;
      }
    }
  }
}

// The same fix-up for a contiguous block of columns (ld == S, S even, 16-byte aligned): the grid walks the
// block as ONE flat array, consecutive CTAs on consecutive 32 KB pieces, so DRAM sees a single sequential
// read stream and a single write stream (like a copy) instead of one stream per CTA-owned column.
constexpr int FIX_CHUNK = 4096;  // elements per CTA iteration (<= S is required: at most one column boundary)
__global__ void __launch_bounds__(256) k_fixup_flat(const double* __restrict__ x, double* __restrict__ out, int32_t S,
                                                    int64_t j0, int64_t j1, const double* __restrict__ med, double c,
                                                    double alpha, const double* __restrict__ beta) {
  const int64_t total = (j1 - j0) * S;
  const double2* __restrict__ x2 = reinterpret_cast<const double2*>(x + j0 * S);
  double2* __restrict__ o2 = reinterpret_cast<double2*>(out + j0 * S);
  for (int64_t start = (int64_t)blockIdx.x * FIX_CHUNK; start < total; start += (int64_t)gridDim.x * FIX_CHUNK) {
    const int64_t ja = start / S;                 // column of the first element of this chunk
    const int64_t bound = (ja + 1) * S;           // first element of the next column
    const double sa = (med ? -med[j0 + ja] : 0.0) + c;
    const double sb = (bound < total) ? (med ? -med[j0 + ja + 1] : 0.0) + c : sa;
    const int32_t ra = (int32_t)(start - ja * S);  // row of the first element
#pragma unroll
    for (int u = 0; u < FIX_CHUNK / 2 / 256; ++u) {
      const int64_t e = start + 2 * (int64_t)(u * 256 + threadIdx.x);
      if (e >= total) break;
      double2 v = __ldcs(x2 + (e >> 1));
      const bool second = e >= bound;             // S is even: both halves of a pair lie in one column
      const double shift = second ? sb : sa;
      v.x = __dmul_rn(alpha, __dadd_rn(v.x, shift));
      v.y = __dmul_rn(alpha, __dadd_rn(v.y, shift));
      if (beta) {
        const int32_t r = (int32_t)(e - start) + ra - (second ? S : 0);
        v.x = __dadd_rn(v.x, beta[r]);
        v.y = __dadd_rn(v.y, beta[r + 1]);
      }
      __stcs(o2 + (e >> 1), v);
    }
  }
}

__global__ void __launch_bounds__(256) k_minmax(const double* __restrict__ x, int64_t n,
                                                unsigned long long* __restrict__ res) {
  unsigned long long lo = ~0ull, hi = 0ull;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x) {
    const double v = x[i];
    if (v != v) continue;
    const unsigned long long k = key_of(v);
    lo = k < lo ? k : lo;
    hi = k > hi ? k : hi;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long a = __shfl_xor_sync(FULL, lo, o), b = __shfl_xor_sync(FULL, hi, o);
    lo = a < lo ? a : lo;
    hi = b > hi ? b : hi;
  }
  if ((threadIdx.x & 31) == 0) {
    atomicMin(res, lo);
    atomicMax(res + 1, hi);
  }
}

// row sums / sums of squares of a column-major S x N matrix by column group (labels in [0, K); unlabelled columns
// take no part).  The host sorts the labelled columns by (chunk, group), ascending inside each group, into `cols`;
// segment g = chunk * K + group is cols[seg[g] .. seg[g + 1]).  grid = (segments, row blocks): each thread owns one
// set row and adds the segment's columns in ascending order, so every score is read once whatever K is, and
// partial[g][2][S] = {sum, sumsq} of that segment; k_group_combine adds the segments of one group in chunk order.
// FIX: the values are RAW scores and the fix-up of normalize_medians / replaid.ucell (k_fixup: alpha * (x + (c - med_j))
// [+ beta_s], the same operations in the same order) is applied in registers — the normalised matrix is never
// written (plaidgpu_score_group_stats: score -> test without materialising S x N for the host).
template <bool FIX>
__global__ void __launch_bounds__(256) k_group_partial(const double* __restrict__ x, int64_t ld, int32_t S,
                                                       const int32_t* __restrict__ cols, const int32_t* __restrict__ seg,
                                                       double* __restrict__ partial, const double* __restrict__ med,
                                                       double c, double alpha, const double* __restrict__ beta) {
  const int r = blockIdx.y * blockDim.x + threadIdx.x;
  const int64_t g = blockIdx.x;
  if (r >= S) return;
  const int32_t i0 = seg[g], i1 = seg[g + 1];
  const double b = (FIX && beta) ? beta[r] : 0.0;
  double s = 0.0, q = 0.0;
#pragma unroll 4
  for (int32_t i = i0; i < i1; ++i) {
    const int64_t j = cols[i];
    double v = __ldcs(x + j * ld + r);
    if (FIX) v = fixup_value(v, j, med, c, alpha, beta, b);
    s += v;
    q += v * v;
  }
  double* p = partial + (size_t)g * 2 * S;
  p[r] = s;
  p[S + r] = q;
}
// out[i] = sum over chunks, in chunk order, of partial[chunk][i]; i < width = K * 2 * S
__global__ void __launch_bounds__(256) k_group_combine(const double* __restrict__ partial, int64_t width, int nchunk,
                                                       double* __restrict__ out) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= width) return;
  double a = 0.0;
  for (int ch = 0; ch < nchunk; ++ch) a += partial[(size_t)ch * width + i];
  out[i] = a;
}

// Per set row of a column-major S x N matrix and one chunk of columns (chunk ch is [N ch / nchunk, N (ch + 1) / nchunk),
// the split of group_stats_device): sum_j x[s, j] * B[j, q] for the Q <= QB columns of B, sum_j x[s, j] and
// sum_j x[s, j]^2.  grid = (set blocks, chunks): each thread owns one set and adds its chunk's columns in ascending
// order, so every raw score is read once; the CTAs that run together share a chunk, so its rows of B come from DRAM
// about once.  The chunk's rows of B are staged DESIGN_TJ at a time in shared memory, zero-padded to QB columns, and
// read as 16-byte broadcasts (the row stride QB + 2 keeps them aligned).  partial[ch][(Q + 2) * S] = {row q of the moments at q * S, the sums at Q * S, the sums of squares at
// (Q + 1) * S}; k_group_combine adds the chunks in chunk order.  FIX: as in k_group_partial.
constexpr int DESIGN_TJ = 32;
template <bool FIX, int QB>
__global__ void __launch_bounds__(256) k_design_partial(const double* __restrict__ x, int64_t ld, int32_t S, int64_t N,
                                                        int nchunk, const double* __restrict__ B, int64_t ldb, int Q,
                                                        double* __restrict__ partial,
                                                        const double* __restrict__ med, double c, double alpha,
                                                        const double* __restrict__ beta) {
  __shared__ __align__(16) double Bs[DESIGN_TJ][QB + 2];
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  const int ch = blockIdx.y;
  const int64_t j0 = (N * ch) / nchunk, j1 = (N * (ch + 1)) / nchunk;
  const bool live = r < S;
  const double b = (FIX && beta && live) ? beta[r] : 0.0;
  double acc[QB];
#pragma unroll
  for (int q = 0; q < QB; ++q) acc[q] = 0.0;
  double s = 0.0, t = 0.0;
  for (int64_t jt = j0; jt < j1; jt += DESIGN_TJ) {
    const int nj = (int)min((int64_t)DESIGN_TJ, j1 - jt);
    __syncthreads();  // every thread is done with the previous tile
    for (int i = threadIdx.x; i < DESIGN_TJ * QB; i += blockDim.x) {
      const int jj = i % DESIGN_TJ, q = i / DESIGN_TJ;  // a warp reads 32 consecutive rows of one column of B
      Bs[jj][q] = (jj < nj && q < Q) ? B[(jt + jj) + (int64_t)q * ldb] : 0.0;
    }
    __syncthreads();
    if (!live) continue;
#pragma unroll 4
    for (int jj = 0; jj < nj; ++jj) {
      const int64_t j = jt + jj;
      double v = __ldcs(x + j * ld + r);
      if (FIX) v = fixup_value(v, j, med, c, alpha, beta, b);
      s += v;
      t += v * v;
#pragma unroll
      for (int q = 0; q < QB; q += 2) {
        const double2 w = *reinterpret_cast<const double2*>(&Bs[jj][q]);
        acc[q] += v * w.x;
        acc[q + 1] += v * w.y;
      }
    }
  }
  if (!live) return;
  double* p = partial + (size_t)ch * (size_t)(Q + 2) * S;
#pragma unroll
  for (int q = 0; q < QB; ++q)
    if (q < Q) p[(size_t)q * S + r] = acc[q];
  p[(size_t)Q * S + r] = s;
  p[(size_t)(Q + 1) * S + r] = t;
}

template <bool FIX>
void design_partial(dim3 g, cudaStream_t st, int qb, const double* x, int64_t ld, int32_t S, int64_t N, int nchunk,
                    const double* B, int64_t ldb, int Q, double* partial, const double* med, double c,
                    double alpha, const double* beta) {
#define PLAIDGPU_DESIGN_CASE(W)                                                                                   \
  case W:                                                                                                         \
    k_design_partial<FIX, W><<<g, 256, 0, st>>>(x, ld, S, N, nchunk, B, ldb, Q, partial, med, c, alpha, beta);     \
    break;
  switch (qb) {
    PLAIDGPU_DESIGN_CASE(2)
    PLAIDGPU_DESIGN_CASE(4)
    PLAIDGPU_DESIGN_CASE(8)
    PLAIDGPU_DESIGN_CASE(16)
    PLAIDGPU_DESIGN_CASE(32)
    PLAIDGPU_DESIGN_CASE(64)
  }
#undef PLAIDGPU_DESIGN_CASE
}

// device -> host-mapped memory by SM stores: small control values (minimum key, flags, medians) must not queue
// behind gigabytes of result blocks in the copy engine
__global__ void __launch_bounds__(256) k_copy_words(const unsigned long long* __restrict__ src, unsigned long long* __restrict__ dst,
                                                    int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) dst[i] = src[i];
}

// by a kernel, not a copy engine: those may be busy with result blocks.  A NaN median of a column without zeros or
// -inf comes from a column without any valid value, whose non-zero median is 0 (R/plaid.R:561-566)
__global__ void __launch_bounds__(256) k_med_nz_from_all(const double* __restrict__ med_all, double* __restrict__ med_nz,
                                                         int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const double m = med_all[i];
    med_nz[i] = m == m ? m : 0.0;
  }
}

__global__ void k_minmax_init(unsigned long long* res) {
  res[0] = ~0ull;
  res[1] = 0ull;
}
__global__ void k_minmax_fin(const unsigned long long* res, double* out) {
  out[0] = res[0] == ~0ull ? INFINITY : value_of(res[0]);
  out[1] = res[1] == 0ull ? -INFINITY : value_of(res[1]);
}

}  // namespace

bool colstats_small(int32_t S) { return S < 4 * SAMP; }

cudaError_t launch_colstats(const double* x, int64_t ld, int32_t S, int64_t N, double* med_all,
                            double* med_nz, double* colmin, int* d_fail, int64_t* d_list, int which, cudaStream_t st) {
  if (N <= 0) return cudaSuccess;
  {  // per device (a process may drive several GPUs): cheap, so set on every launch
    cudaError_t e = cudaFuncSetAttribute(k_colstats, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)sizeof(StatsSmem));
    if (e != cudaSuccess) return e;
    const void* fast[3] = {(const void*)k_colstats_fast<true, true>, (const void*)k_colstats_fast<true, false>,
                           (const void*)k_colstats_fast<false, true>};
    for (int i = 0; i < 3; ++i) {
      e = cudaFuncSetAttribute(fast[i], cudaFuncAttributeMaxDynamicSharedMemorySize,
                               (int)(i == 0 ? sizeof(Stats2Smem) : STATS2_SMEM_ONE));
      if (e != cudaSuccess) return e;
    }
    e = cudaFuncSetAttribute(k_colstats_one<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Stats3Smem));
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(k_colstats_one<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Stats3Smem));
    if (e != cudaSuccess) return e;
  }
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (S < 4 * SAMP) {  // short columns: the three-pass kernel is as cheap as sampling
    int64_t grid = (int64_t)sms * 4;
    if (grid > N) grid = N;
    k_colstats<<<(unsigned)grid, NT, sizeof(StatsSmem), st>>>(x, ld, S, N, nullptr, med_all, med_nz, colmin);
    return cudaGetLastError();
  }
  // single-pass kernel, then the exact three-pass kernel on whatever it rejected
  // d_fail (1 int) and d_list (N int64) are caller-owned scratch: no allocation on the hot path
  cudaError_t e = launch_fill_u32(d_fail, 0u, 1, st);
  if (e != cudaSuccess) return e;
  int per_sm = 1;
  static const bool old_one = getenv("PLAIDGPU_COLSTATS_OLD") != nullptr;  // A/B switch: two-bracket kernel for one median
  if (which != COLSTATS_BOTH && !old_one) {
    const size_t sm3 = sizeof(Stats3Smem);
    if (which == COLSTATS_ALL) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_colstats_one<false>, NT, sm3);
    else cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_colstats_one<true>, NT, sm3);
    if (per_sm < 1) per_sm = 1;
    int64_t grid = (int64_t)sms * per_sm;
    if (grid > N) grid = N;
    if (which == COLSTATS_ALL)
      k_colstats_one<false><<<(unsigned)grid, NT, sm3, st>>>(x, ld, S, N, med_all, colmin, d_fail, d_list);
    else
      k_colstats_one<true><<<(unsigned)grid, NT, sm3, st>>>(x, ld, S, N, med_nz, colmin, d_fail, d_list);
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
  } else {
  const size_t smem = which == COLSTATS_BOTH ? sizeof(Stats2Smem) : STATS2_SMEM_ONE;
  if (which == COLSTATS_ALL)
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_colstats_fast<true, false>, NT, smem);
  else if (which == COLSTATS_NZ)
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_colstats_fast<false, true>, NT, smem);
  else
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_colstats_fast<true, true>, NT, smem);
  if (per_sm < 1) per_sm = 1;
  int64_t grid = (int64_t)sms * per_sm;
  if (grid > N) grid = N;
  if (which == COLSTATS_ALL)
    k_colstats_fast<true, false><<<(unsigned)grid, NT, smem, st>>>(x, ld, S, N, med_all, med_nz, colmin, d_fail, d_list);
  else if (which == COLSTATS_NZ)
    k_colstats_fast<false, true><<<(unsigned)grid, NT, smem, st>>>(x, ld, S, N, med_all, med_nz, colmin, d_fail, d_list);
  else
    k_colstats_fast<true, true><<<(unsigned)grid, NT, smem, st>>>(x, ld, S, N, med_all, med_nz, colmin, d_fail, d_list);
  e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  }
  int nfail = 0;
  e = cudaMemcpyAsync(&nfail, d_fail, sizeof(int), cudaMemcpyDeviceToHost, st);
  if (e != cudaSuccess) return e;
  e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) return e;
  if (getenv("PLAIDGPU_TRACE_COLSTATS"))
    fprintf(stderr, "[plaidgpu] colstats: %d of %lld columns redone by the three-pass kernel\n", nfail, (long long)N);
  if (nfail > 0) {
    int64_t g2 = (int64_t)sms * 4;
    if (g2 > nfail) g2 = nfail;
    k_colstats<<<(unsigned)g2, NT, sizeof(StatsSmem), st>>>(x, ld, S, nfail, d_list, med_all, med_nz, colmin);
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
  }
  return cudaSuccess;
}

cudaError_t launch_fixup(const double* x, double* out, int64_t ld, int32_t S, int64_t j0, int64_t j1,
                         const double* med, double c, double alpha, const double* beta,
                         cudaStream_t st) {
  if (j1 <= j0) return cudaSuccess;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (ld == S && (S & 1) == 0 && S >= FIX_CHUNK && ((((uintptr_t)(x + j0 * ld)) | ((uintptr_t)(out + j0 * ld))) & 15) == 0) {
    const int64_t chunks = ((j1 - j0) * (int64_t)S + FIX_CHUNK - 1) / FIX_CHUNK;
    int64_t grid = (int64_t)sms * 8;
    if (grid > chunks) grid = chunks;
    k_fixup_flat<<<(unsigned)grid, 256, 0, st>>>(x, out, S, j0, j1, med, c, alpha, beta);
    return cudaGetLastError();
  }
  int64_t grid = (int64_t)sms * 8;
  if (grid > j1 - j0) grid = j1 - j0;
  k_fixup<<<(unsigned)grid, 256, 0, st>>>(x, out, ld, S, j0, j1, med, c, alpha, beta);
  return cudaGetLastError();
}

cudaError_t launch_group_stats(const double* x, int64_t ld, int32_t S, int K, const int32_t* cols, const int32_t* seg,
                               int nchunk, double* partial, double* out, cudaStream_t st, bool fix, const double* med,
                               double c, double alpha, const double* beta) {
  if (S <= 0 || K <= 0) return cudaSuccess;
  dim3 g((unsigned)((int64_t)nchunk * K), (unsigned)((S + 255) / 256));
  if (fix) k_group_partial<true><<<g, 256, 0, st>>>(x, ld, S, cols, seg, partial, med, c, alpha, beta);
  else k_group_partial<false><<<g, 256, 0, st>>>(x, ld, S, cols, seg, partial, nullptr, 0.0, 1.0, nullptr);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  const int64_t width = (int64_t)K * 2 * S;
  k_group_combine<<<(unsigned)((width + 255) / 256), 256, 0, st>>>(partial, width, nchunk, out);
  return cudaGetLastError();
}

cudaError_t launch_design_stats(const double* x, int64_t ld, int32_t S, int64_t N, const double* B, int64_t ldb, int Q,
                                int nchunk, double* partial, double* out, cudaStream_t st, bool fix, const double* med,
                                double c, double alpha, const double* beta) {
  if (S <= 0 || Q < 1 || Q > DESIGN_Q_MAX) return cudaErrorInvalidValue;
  const dim3 g((unsigned)((S + 255) / 256), (unsigned)nchunk);
  int qb = 2;  // the narrowest instantiation that holds Q: one pass over x for every Q
  while (qb < Q) qb *= 2;
  if (fix) design_partial<true>(g, st, qb, x, ld, S, N, nchunk, B, ldb, Q, partial, med, c, alpha, beta);
  else design_partial<false>(g, st, qb, x, ld, S, N, nchunk, B, ldb, Q, partial, nullptr, 0.0, 1.0, nullptr);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  const int64_t width = (int64_t)(Q + 2) * S;
  k_group_combine<<<(unsigned)((width + 255) / 256), 256, 0, st>>>(partial, width, nchunk, out);
  return cudaGetLastError();
}

cudaError_t launch_copy_words(const void* src, void* dst_mapped, int64_t nwords, cudaStream_t st) {
  if (nwords <= 0) return cudaSuccess;
  int64_t grid = (nwords + 255) / 256;
  if (grid > 148 * 4) grid = 148 * 4;
  k_copy_words<<<(unsigned)grid, 256, 0, st>>>(static_cast<const unsigned long long*>(src), static_cast<unsigned long long*>(dst_mapped), nwords);
  return cudaGetLastError();
}

cudaError_t launch_med_nz_from_all(const double* med_all, double* med_nz, int64_t n, cudaStream_t st) {
  if (n <= 0) return cudaSuccess;
  int64_t grid = (n + 255) / 256;
  if (grid > 148 * 4) grid = 148 * 4;
  k_med_nz_from_all<<<(unsigned)grid, 256, 0, st>>>(med_all, med_nz, n);
  return cudaGetLastError();
}

// res2: device double[2]; uses 16 bytes right after it as scratch -> caller passes double[4]
cudaError_t launch_minmax(const double* x, int64_t n, double* res4, cudaStream_t st) {
  unsigned long long* scratch = reinterpret_cast<unsigned long long*>(res4 + 2);
  k_minmax_init<<<1, 1, 0, st>>>(scratch);
  if (n > 0) {
    int64_t grid = (n + 255) / 256;
    if (grid > 148 * 16) grid = 148 * 16;
    k_minmax<<<(unsigned)grid, 256, 0, st>>>(x, n, scratch);
  }
  k_minmax_fin<<<1, 1, 0, st>>>(scratch, res4);
  return cudaGetLastError();
}

}  // namespace plaidgpu
