// Warp-wide top-k selection over a stream of composite keys, shared by k_col_topk (topk_kernels.cu: each column's
// best rows) and the row kernels of topcells_kernels.cu (each row's best columns).
//
// Every candidate is an Entry: the order-preserving u64 key of its value, then its index, in which "larger" means
// "comes first" in R's order(v, decreasing = ...):
//   key = 0 for NaN (after every number, in both directions); otherwise the order-preserving bits of v with -0 mapped
//   to +0, complemented when decreasing = 0.  Equal keys are ordered by ascending index.
// The key alone decides the order, so a selection does not depend on the scan order or the launch geometry.
// A warp keeps its current best list and tests every candidate against the list's k-th entry; only when a lane of a
// 32-candidate batch beats it (ballot) is the batch offered to the list:
//   k <= 32 (offer_small): the list is 32 entries in registers, one per lane; a few survivors are inserted one by one,
//           more are sorted (bitonic, by shuffles) and merged by a bitonic merge;
//   k > 32 (offer_large):  the list is k entries in shared memory, the sorted batch is merged by a parallel merge
//           (binary search of each entry's rank).
#pragma once
#include "common.cuh"

namespace plaidgpu {
namespace topk {

constexpr int INSERT_MAX = 8;  // k <= 32: up to this many survivors of a batch are inserted one by one

// I: the index type (uint32_t for a row or a chunk-relative column, uint64_t for a column of the whole launch)
template <typename I>
struct Entry {
  uint64_t key;
  I idx;
};

template <typename I>
__device__ __forceinline__ bool better(const Entry<I>& a, const Entry<I>& b) {
  return a.key > b.key || (a.key == b.key && a.idx < b.idx);
}

__device__ __forceinline__ uint64_t order_key(double v, bool decreasing) {
  if (v != v) return 0ull;                                  // NaN: last in both directions
  uint64_t b = v == 0.0 ? 0ull : (uint64_t)__double_as_longlong(v);  // -0 ties with +0
  b = (b >> 63) ? ~b : (b | 0x8000000000000000ull);  // ascending in v, and >= 0x000fffffffffffff (-Inf) > 0
  return decreasing ? b : ~b;                        // ~b <= 0xfff0000000000000 and > 0 as well
}

template <typename I>
__device__ __forceinline__ Entry<I> shfl_xor(const Entry<I>& e, int m) {
  Entry<I> p;
  p.key = __shfl_xor_sync(FULL, e.key, m);
  p.idx = __shfl_xor_sync(FULL, e.idx, m);
  return p;
}

template <typename I>
__device__ __forceinline__ Entry<I> shfl(const Entry<I>& e, int src) {
  return Entry<I>{__shfl_sync(FULL, e.key, src), __shfl_sync(FULL, e.idx, src)};
}

// the 32 entries of a warp, one per lane, sorted best first (lane 0 best)
template <typename I>
__device__ __forceinline__ Entry<I> warp_sort(Entry<I> e, int lane) {
#pragma unroll
  for (int size = 2; size <= 32; size <<= 1) {
    const bool first_best = (lane & size) == 0;  // direction of this lane's bitonic block
#pragma unroll
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      const Entry<I> p = shfl_xor(e, stride);
      const bool keep_better = ((lane & stride) == 0) == first_best;
      if (keep_better ? better(p, e) : better(e, p)) e = p;
    }
  }
  return e;
}

// a bitonic sequence of 32 entries -> sorted best first
template <typename I>
__device__ __forceinline__ Entry<I> warp_clean(Entry<I> e, int lane) {
#pragma unroll
  for (int stride = 16; stride > 0; stride >>= 1) {
    const Entry<I> p = shfl_xor(e, stride);
    if (((lane & stride) == 0) ? better(p, e) : better(e, p)) e = p;
  }
  return e;
}

// k <= 32: offer this lane's candidate e to the register list (lane l holds entry l, best first).  pass: the ballot
// of the lanes whose candidate beats thr, not zero.  thr becomes the list's new k-th entry.
template <typename I>
__device__ __forceinline__ void offer_small(Entry<I> e, unsigned pass, Entry<I>& list, Entry<I>& thr, int k, int lane) {
  if (__popc(pass) <= INSERT_MAX) {
    // a few survivors (the common case once the list has filled): insert them one by one, each a broadcast and a
    // shift of the list by one lane, instead of sorting and merging the whole batch
    do {
      const int src = __ffs(pass) - 1;
      pass &= pass - 1;
      const Entry<I> s = shfl(e, src);
      const unsigned worse = __ballot_sync(FULL, better(s, list));  // a suffix of the sorted list
      const int pos = __ffs(worse) - 1;
      const Entry<I> up{__shfl_up_sync(FULL, list.key, 1), __shfl_up_sync(FULL, list.idx, 1)};
      if (worse && lane >= pos) list = lane == pos ? s : up;
    } while (pass);
    thr = shfl(list, k - 1);
    return;
  }
  e = warp_sort(e, lane);
  const Entry<I> o = shfl_xor(e, 31);  // batch reversed: list + reversed batch is bitonic after the max below
  list = warp_clean(better(list, o) ? list : o, lane);
  thr = shfl(list, k - 1);
}

// k > 32: one warp's lists in shared memory: two lists of k entries (current and next, `cur` selects) and the batch
// being merged.  bytes(k) per list; init lays one out at `base` and fills the current list with `none`.
template <typename I>
struct SharedList {
  uint64_t* key;   // [2 * k]
  uint64_t* bkey;  // [32]
  I* idx;          // [2 * k]
  I* bidx;         // [32]
  __host__ __device__ static constexpr size_t bytes(int k) { return (size_t)(2 * k + 32) * (8 + sizeof(I)); }
  __device__ __forceinline__ void init(unsigned char* base, int k, int lane, const Entry<I>& none) {
    key = reinterpret_cast<uint64_t*>(base);
    bkey = key + 2 * k;
    idx = reinterpret_cast<I*>(bkey + 32);
    bidx = idx + 2 * k;
    for (int i = lane; i < k; i += 32) {
      key[i] = none.key;
      idx[i] = none.idx;
    }
    __syncwarp();
  }
};

// k > 32: offer this lane's candidate e to the shared list L (current list `cur`, flipped); thr becomes its new k-th
// entry
template <typename I>
__device__ __forceinline__ void offer_large(Entry<I> e, const SharedList<I>& L, int& cur, Entry<I>& thr, int k, int lane) {
  e = warp_sort(e, lane);
  const uint64_t* ck = L.key + cur * k;
  const I* cr = L.idx + cur * k;
  uint64_t* nk = L.key + (cur ^ 1) * k;
  I* nr = L.idx + (cur ^ 1) * k;
  L.bkey[lane] = e.key;
  L.bidx[lane] = e.idx;
  __syncwarp();
  // batch entry `lane`: its rank in the batch plus the list entries that are better or equal (list first on ties;
  // only the shared placeholder entries can tie)
  int lo = 0, hi = k;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    const Entry<I> m{ck[mid], cr[mid]};
    if (!better(e, m)) lo = mid + 1;
    else hi = mid;
  }
  if (lane + lo < k) {
    nk[lane + lo] = e.key;
    nr[lane + lo] = e.idx;
  }
  // list entry i: its rank in the list plus the batch entries strictly better
  for (int i = lane; i < k; i += 32) {
    const Entry<I> m{ck[i], cr[i]};
    int a = 0, b = 32;
    while (a < b) {
      const int mid = (a + b) >> 1;
      if (better(Entry<I>{L.bkey[mid], L.bidx[mid]}, m)) a = mid + 1;
      else b = mid;
    }
    if (i + a < k) {
      nk[i + a] = m.key;
      nr[i + a] = m.idx;
    }
  }
  __syncwarp();
  cur ^= 1;
  thr.key = nk[k - 1];
  thr.idx = nr[k - 1];
}

}  // namespace topk
}  // namespace plaidgpu
