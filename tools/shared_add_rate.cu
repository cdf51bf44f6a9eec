// Microbenchmark (development): cost of one warp step of the tail pass's shared-memory accumulation (tail_kernels.cu,
// k_tail) with the ways of adding that the kernel could use.  One CTA per SM with 32 warps, each warp owning a
// private row of 1,056 u32 accumulators (plus 528 words of packed 16-bit high counters), as in k_tail.  Every warp
// step adds one addend per lane at the cell the lane reads from a table of random steps (16 KB, stays in L1):
//   distinct: 32 distinct cells per step;  dup4: the same, then up to 4 lanes of each step moved onto another
//   lane's cell (duplicate addresses inside a step).
// Variants, per lane and step:
//   load      the table read alone (the common overhead of every variant below)
//   a         ld.shared.u32 + add + st.shared.u32, then __syncwarp (the 32-bit half of the old k_tail step)
//   a+hi      a, plus the old carry branch: ld/st.shared.s16 of the high word where the carry differs from the sign
//   b         atom.shared.add.u32 returning the old value
//   c         b, plus a no-return atomic add on a second word for ~10 % of the lanes (predicated on a table bit)
//   b+hi      b, plus the carry rule of the new k_tail (d = carry - sign, no-return add of d << 16 * (c & 1))
// Prints SM clocks per warp step: (clock64 at the end - at the start of the CTA) / (steps of all 32 warps).
// Duplicate cells make `a` / `a+hi` lose adds; only their time is measured here.
//   nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a tools/shared_add_rate.cu -o /tmp/sar && /tmp/sar
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include <algorithm>
#include <random>
#include <vector>

constexpr int WARPS = 32, C = 1056, TSTEPS = 256, REPS = 64;

#define CK(x)                                                                              \
  do {                                                                                     \
    cudaError_t e_ = (x);                                                                  \
    if (e_ != cudaSuccess) {                                                               \
      fprintf(stderr, "%s:%d %s\n", __FILE__, __LINE__, cudaGetErrorString(e_));           \
      exit(1);                                                                             \
    }                                                                                      \
  } while (0)

enum { V_LOAD, V_A, V_AHI, V_B, V_C, V_BHI, NV };
static const char* NAMES[NV] = {"load", "a", "a+hi", "b", "c", "b+hi"};

// table entry: cell (bits 0-15) | flag for variant c (bit 16); the addend is derived from the entry
template <int V>
__global__ void __launch_bounds__(WARPS * 32, 1) k_rate(const uint32_t* __restrict__ tab, unsigned long long* clk,
                                                        uint32_t* sink) {
  extern __shared__ uint32_t sm[];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  uint32_t* lo = sm + w * C;
  uint32_t* hiw = sm + WARPS * C + w * (C / 2);
  for (int c = lane; c < C; c += 32) lo[c] = 0u;
  for (int c = lane; c < C / 2; c += 32) hiw[c] = 0x80008000u;
  __syncthreads();
  const uint32_t lo_sa = (uint32_t)__cvta_generic_to_shared(lo), hi_sa = (uint32_t)__cvta_generic_to_shared(hiw);
  uint32_t acc = 0;
  const unsigned long long t0 = clock64();
  for (int r = 0; r < REPS; ++r) {
#pragma unroll 4
    for (int i = 0; i < TSTEPS; ++i) {
      const uint32_t e = __ldg(tab + ((i + w * 8) & (TSTEPS - 1)) * 32 + lane);
      const uint32_t c = e & 0xFFFFu;
      uint32_t q = (e * 2654435761u) >> 2;  // |q| < 2^30, either sign
      if (e & 0x20000u) q = 0u - q;
      if (V == V_LOAD) {
        acc += c;
      } else if (V == V_A || V == V_AHI) {
        uint32_t old;
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(old) : "r"(lo_sa + c * 4u) : "memory");
        const uint32_t nv = old + q;
        asm volatile("st.shared.u32 [%0], %1;" ::"r"(lo_sa + c * 4u), "r"(nv) : "memory");
        if (V == V_AHI && (nv < q) != ((int32_t)q < 0)) {
          const uint32_t ah = hi_sa + c * 2u;
          short hv;
          asm volatile("ld.shared.s16 %0, [%1];" : "=h"(hv) : "r"(ah) : "memory");
          hv = (short)(hv + ((nv < q) ? 1 : -1));
          asm volatile("st.shared.s16 [%0], %1;" ::"r"(ah), "h"(hv) : "memory");
        }
        __syncwarp();
      } else {
        uint32_t old;
        asm volatile("atom.shared.add.u32 %0, [%1], %2;" : "=r"(old) : "r"(lo_sa + c * 4u), "r"(q) : "memory");
        if (V == V_B) acc += old;
        if (V == V_C) {
          acc += old;
          asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %2, 0;\n\t@p red.shared.add.u32 [%0], %1;\n\t}"
                       ::"r"(hi_sa + (c >> 1) * 4u), "r"(1u), "r"(e & 0x10000u) : "memory");
        }
        if (V == V_BHI) {
          const uint32_t d = (uint32_t)(old + q < old) + (uint32_t)((int32_t)q >> 31);
          asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %1, 0;\n\t@p red.shared.add.u32 [%0], %1;\n\t}"
                       ::"r"(hi_sa + (c >> 1) * 4u), "r"(d << ((c & 1u) * 16u)) : "memory");
        }
      }
    }
  }
  __syncthreads();
  const unsigned long long t1 = clock64();
  if (threadIdx.x == 0) clk[blockIdx.x] = t1 - t0;
  uint32_t x = acc;
  for (int c = lane; c < C; c += 32) x ^= lo[c];
  for (int c = lane; c < C / 2; c += 32) x ^= hiw[c];
  if (x == 0x12345678u) sink[threadIdx.x] = x;  // keeps the work alive
}

template <int V>
static double run(const uint32_t* tab, unsigned long long* clk, uint32_t* sink, int sms, size_t smem) {
  CK(cudaFuncSetAttribute(k_rate<V>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_rate<V><<<sms, WARPS * 32, smem>>>(tab, clk, sink);  // warm-up
  k_rate<V><<<sms, WARPS * 32, smem>>>(tab, clk, sink);
  CK(cudaDeviceSynchronize());
  std::vector<unsigned long long> h(sms);
  CK(cudaMemcpy(h.data(), clk, sms * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  std::sort(h.begin(), h.end());
  return (double)h[sms / 2] / ((double)WARPS * REPS * TSTEPS);  // median over the SMs
}

int main() {
  int dev = 0, sms = 0;
  CK(cudaGetDevice(&dev));
  CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, dev));
  const size_t smem = (size_t)WARPS * C * 6;
  std::mt19937 rng(7);
  uint32_t *tab, *sink;
  unsigned long long* clk;
  CK(cudaMalloc(&tab, TSTEPS * 32 * sizeof(uint32_t)));
  CK(cudaMalloc(&sink, WARPS * 32 * sizeof(uint32_t)));
  CK(cudaMalloc(&clk, sms * sizeof(unsigned long long)));
  printf("%s, %d SMs; SM clocks per warp step (32 warps per SM, 1,056 cells per warp)\n", prop.name, sms);
  printf("%-10s %10s %10s\n", "variant", "distinct", "dup4");
  double t[2][NV];
  for (int dup = 0; dup < 2; ++dup) {
    std::vector<uint32_t> h(TSTEPS * 32);
    std::vector<uint32_t> cells(C);
    for (int c = 0; c < C; ++c) cells[c] = c;
    for (int i = 0; i < TSTEPS; ++i) {
      std::shuffle(cells.begin(), cells.end(), rng);  // first 32: distinct cells
      for (int l = 0; l < 32; ++l) {
        uint32_t c = cells[l];
        h[i * 32 + l] = c | ((rng() % 10 == 0) ? 0x10000u : 0u) | ((rng() & 1) ? 0x20000u : 0u);
      }
      if (dup) {
        const int nd = 1 + (int)(rng() % 4);
        for (int k = 0; k < nd; ++k) {
          const int a = (int)(rng() % 32), b = (int)(rng() % 32);
          h[i * 32 + a] = (h[i * 32 + a] & ~0xFFFFu) | (h[i * 32 + b] & 0xFFFFu);
        }
      }
    }
    CK(cudaMemcpy(tab, h.data(), h.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
    t[dup][V_LOAD] = run<V_LOAD>(tab, clk, sink, sms, smem);
    t[dup][V_A] = run<V_A>(tab, clk, sink, sms, smem);
    t[dup][V_AHI] = run<V_AHI>(tab, clk, sink, sms, smem);
    t[dup][V_B] = run<V_B>(tab, clk, sink, sms, smem);
    t[dup][V_C] = run<V_C>(tab, clk, sink, sms, smem);
    t[dup][V_BHI] = run<V_BHI>(tab, clk, sink, sms, smem);
  }
  for (int v = 0; v < NV; ++v) printf("%-10s %10.2f %10.2f\n", NAMES[v], t[0][v], t[1][v]);
  CK(cudaFree(tab));
  CK(cudaFree(sink));
  CK(cudaFree(clk));
  return 0;
}
