// Micro-benchmark: cycles per tcgen05.mma (K=16, fp16) issued back to back from shared-memory
// operands in the no-swizzle K-major layout, with optional competing shared-memory store
// traffic, for cta_group::1 (M=128 per SM) and cta_group::2 (M=256 over an SM pair, each SM
// holding half of B).  Answers: what bounds the MMA rate inside conv.cu?
// usage: umma_bench N a_rows b_rows [grid] [iters] [writer_warps 0..3] [two_cta 0|1] [data 0=zeros|1=random] [spinner_warps 0..8]
#include <cstdio>
#include <cstdlib>
#include <cuda_runtime.h>
#include "../muzero_b200/csrc/umma.cuh"

using namespace mz::umma;

__device__ __forceinline__ void mma2(uint32_t d, uint64_t a, uint64_t b, uint32_t idesc, uint32_t acc) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
               "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d), "l"(a), "l"(b), "r"(idesc), "r"(acc)
               : "memory");
}

template <bool kTwo>
__global__ void __launch_bounds__(384) bench(int N, int a_rows, int b_rows, int iters, long long* out, int writer, int data) {
  extern __shared__ __align__(1024) unsigned char smem[];
  __shared__ __align__(8) uint64_t bar;
  __shared__ __align__(8) uint64_t bar2;   // never completes: spinner warps poll it like idle pipeline roles do
  __shared__ uint32_t tmem_base;
  __shared__ volatile int stop;
  const int tid = threadIdx.x, warp = tid >> 5;
  uint32_t rank = 0;
  if (kTwo) asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));
  unsigned char* sA = smem;
  unsigned char* sB = smem + 16 * a_rows * 16;
  // operand data: zeros (data == 0) or pseudo-random fp16 in [-1, 1) (data == 1): tensor-core power depends on it
  for (int i = tid; i < (16 * a_rows + 8 * b_rows) * 4; i += blockDim.x) {
    uint32_t v = 0;
    if (data) {
      uint32_t h = (uint32_t)i * 2654435761u + blockIdx.x * 40503u;
      h ^= h >> 15; h *= 2246822519u; h ^= h >> 13;
      const uint32_t lo = 0x3800u | (h & 0x83ffu), hi = 0x3800u | ((h >> 16) & 0x83ffu);   // +-[0.5, 1)
      v = lo | (hi << 16);
    }
    reinterpret_cast<uint32_t*>(smem)[i] = v;
  }
  if (tid == 0) { mbar_init(&bar, 1); mbar_init(&bar2, 1); fence_mbar_init(); stop = 0; }
  if (warp == 0) {
    if (kTwo) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base)), "r"(512) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      tmem_alloc(&tmem_base, 512);
    }
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  if (kTwo) cluster_sync();
  tc_fence_after();
  const uint32_t tm = tmem_base;
  if (tid == 0) {
    long long t0 = 0, t1 = 0;
    if (!kTwo || rank == 0) {
      const uint32_t idesc = instr_desc_f16(kTwo ? 256 : 128, N);
      const uint64_t at = smem_desc(smem_u32(sA) + 11 * 16, a_rows * 16, 128);
      const uint64_t bt = smem_desc(smem_u32(sB), b_rows * 16, 128);
      t0 = clock64();
      for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
          const uint64_t a = at + (uint64_t)(2 * ks * a_rows), b = bt + (uint64_t)(2 * ks * b_rows);
          if (kTwo) { mma2(tm, a, b, idesc, 1); mma2(tm + 256, a + 128, b, idesc, 1); }
          else { mma_f16(tm, a, b, idesc, 1); mma_f16(tm + 256, a + 128, b, idesc, 1); }
        }
      }
      if (kTwo)
        asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                         smem_u32(&bar)), "h"((unsigned short)3) : "memory");
      else
        commit(&bar);
    }
    mbar_wait(&bar, 0);
    t1 = clock64();
    out[blockIdx.x] = t1 - t0;
    stop = 1;
  } else if (warp >= 1 && warp <= writer) {
    // competing shared-memory store traffic (what the TMA weight fills / cp.async tile fills do)
    const uint32_t w = smem_u32(sB + 8 * b_rows * 16) + (uint32_t)(tid - 32) * 16;
    int it = 0;
    while (!stop) {
#pragma unroll
      for (int u = 0; u < 8; ++u)
        asm volatile("st.shared.v4.b32 [%0], {%1, %1, %1, %1};" ::"r"(w + (uint32_t)(((it + u) & 7) * 96 * 16)), "r"(it) : "memory");
      it += 8;
    }
    if (tid == 32) out[gridDim.x + blockIdx.x] = (long long)it * 16 * 32 * writer;   // bytes stored by this CTA
  } else if (warp >= 4) {
    while (!stop) { if (mbar_try_wait(&bar2, 0)) break; }
  }
  tc_fence_before();
  __syncthreads();
  if (kTwo) cluster_sync();
  if (warp == 0) {
    if (kTwo) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tm), "r"(512) : "memory");
    else tmem_dealloc(tm, 512);
  }
}

int main(int argc, char** argv) {
  const int N = argc > 1 ? atoi(argv[1]) : 128, a_rows = argc > 2 ? atoi(argv[2]) : 279, b_rows = argc > 3 ? atoi(argv[3]) : N;
  const int grid = argc > 4 ? atoi(argv[4]) : 1, iters = argc > 5 ? atoi(argv[5]) : 2000, writer = argc > 6 ? atoi(argv[6]) : 0;
  const int two = argc > 7 ? atoi(argv[7]) : 0;
  const int data = argc > 8 ? atoi(argv[8]) : 0;
  const int spin = argc > 9 ? atoi(argv[9]) : 0;
  const int threads = 128 + 32 * spin;
  long long* d;
  cudaMalloc(&d, 2 * grid * sizeof(long long));
  cudaMemset(d, 0, 2 * grid * sizeof(long long));
  const int smem = 16 * a_rows * 16 + 8 * b_rows * 16 + 8 * 96 * 16 + 1024;
  cudaError_t e;
  if (two) {
    cudaFuncSetAttribute(bench<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(threads); cfg.dynamicSmemBytes = smem;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    e = cudaLaunchKernelEx(&cfg, bench<true>, N, a_rows, b_rows, iters, d, writer, data);
    if (e != cudaSuccess) { printf("launch error %s\n", cudaGetErrorString(e)); return 1; }
  } else {
    cudaFuncSetAttribute(bench<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    bench<false><<<grid, threads, smem>>>(N, a_rows, b_rows, iters, d, writer, data);
  }
  e = cudaDeviceSynchronize();
  if (e != cudaSuccess) { printf("error %s\n", cudaGetErrorString(e)); return 1; }
  long long h[1024];
  cudaMemcpy(h, d, 2 * grid * sizeof(long long), cudaMemcpyDeviceToHost);
  double mx = 0, wbytes = 0;
  for (int i = 0; i < grid; ++i) { if (two && (i & 1)) continue; mx = h[i] > mx ? h[i] : mx; }
  for (int i = 0; i < grid; ++i) wbytes += (double)h[grid + i] / grid;
  const double cyc = mx / ((double)iters * 8);
  const double flop = 2.0 * 128 * N * 16;     // per SM per MMA (a 2-SM MMA does this much on each SM)
  printf("spin=%d data=%s cta_group::%d N=%d A-LBO %d B b_rows=%d grid=%d writer_warps=%d: %.1f cycles/MMA, %.0f flop/cycle/SM (ideal 8192), "
         "competing stores %.1f B/cycle/SM\n", spin, data ? "random" : "zeros", two ? 2 : 1, N, a_rows * 16, b_rows, grid, writer, cyc, flop / cyc, wbytes / mx);
  return 0;
}
