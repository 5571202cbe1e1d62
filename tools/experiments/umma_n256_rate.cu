// Does one M128 x N256 x K16 tcgen05 MMA issue faster than the same FLOPs as two M128 x N128 x K16 MMAs?
// The N=128 pair is how the streamed-weight 3x3 convs ran before (two 16x8-pixel halves sharing one weight stage); N=256 is
// the swapped formulation (weights as M, 256 pixels as N).  Per SM an M128 x N x K16 bf16 MMA reads 4 KB of A and N*32 B of B
// from shared memory, so the pair reads 16 KB per 2 x 64 cycles and the N=256 MMA 12 KB per 128 cycles.
// One CTA per SM on every SM; both operands resident in shared memory (K-major, SWIZZLE_128B); one thread issues a long loop
// of K=64 chunks (4 K steps each, the conv kernel's inline-PTX issue pattern) into a TMEM accumulator.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O2 -o umma_n256_rate umma_n256_rate.cu && ./umma_n256_rate
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t desc_lo(uint32_t a) { return ((a & 0x3FFFFu) >> 4) | (1u << 16); }
constexpr uint32_t DESC_HI = (1024u >> 4) | (1u << 14) | (2u << 29);   // SBO = 1024 B | version 1 | SWIZZLE_128B

// four K=16 steps (+32 B per step on both operands) in one asm block, as in the conv kernel
__device__ __forceinline__ void mma_k4(uint32_t td, uint32_t al, uint32_t bl, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p, e, t;\n\t.reg .b64 da, db;\n\t.reg .b32 a1, b1;\n\t"
      "elect.sync _|e, 0xffffffff;\n\tsetp.ne.b32 p, %4, 0;\n\tsetp.eq.b32 t, 0, 0;\n\t"
      "mov.b64 da, {%1, %5};\n\tmov.b64 db, {%2, %5};\n\t@e tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, p;\n\t"
      "add.u32 a1, %1, 2;\n\tadd.u32 b1, %2, 2;\n\tmov.b64 da, {a1, %5};\n\tmov.b64 db, {b1, %5};\n\t"
      "@e tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, t;\n\t"
      "add.u32 a1, %1, 4;\n\tadd.u32 b1, %2, 4;\n\tmov.b64 da, {a1, %5};\n\tmov.b64 db, {b1, %5};\n\t"
      "@e tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, t;\n\t"
      "add.u32 a1, %1, 6;\n\tadd.u32 b1, %2, 6;\n\tmov.b64 da, {a1, %5};\n\tmov.b64 db, {b1, %5};\n\t"
      "@e tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, t;\n\t}" ::"r"(td),
      "r"(al), "r"(bl), "r"(idesc), "r"(acc), "r"(DESC_HI)
      : "memory");
}

// mode 0: per chunk one N=256 block; mode 1: per chunk two N=128 blocks (B rows 0..127 and 128..255, accumulators 0 and 128)
__global__ void __launch_bounds__(128, 1) k_rate(int mode, int chunks, long long* cycles) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ uint64_t bar;
  __shared__ uint32_t tslot;
  uint8_t* A = smem;                 // 128 rows x 128 B
  uint8_t* B = smem + 16384;         // 256 rows x 128 B
  for (int i = threadIdx.x; i < (16384 + 32768) / 4; i += blockDim.x) {
    const uint32_t h = (uint32_t)i * 2654435761u + blockIdx.x;   // bf16 values in [-1, 1): the tensor pipe sees real data
    const uint32_t lo = 0x3C00u | ((h >> 9) & 0x7F) | ((h >> 8) & 0x8000u), hi = 0x3C00u | ((h >> 17) & 0x7F) | ((h >> 16) & 0x8000u);
    reinterpret_cast<uint32_t*>(smem)[i] = lo | (hi << 16);
  }
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&bar)));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (threadIdx.x < 32) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(&tslot)));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy operand writes -> tensor-core reads
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = tslot;
  if (threadIdx.x < 32) {
    const uint32_t al = desc_lo(smem_u32(A)), bl = desc_lo(smem_u32(B));
    const uint32_t id256 = (1u << 4) | (1u << 7) | (1u << 10) | ((256u >> 3) << 17) | ((128u >> 4) << 24);
    const uint32_t id128 = (1u << 4) | (1u << 7) | (1u << 10) | ((128u >> 3) << 17) | ((128u >> 4) << 24);
    const long long t0 = clock64();
    for (int c = 0; c < chunks; ++c) {
      const uint32_t acc = c > 0 ? 1u : 0u;
      if (mode == 0) {
        mma_k4(tmem, al, bl, id256, acc);
      } else {
        mma_k4(tmem, al, bl, id128, acc);
        mma_k4(tmem + 128, al, bl + (16384u >> 4), id128, acc);
      }
    }
    asm volatile(
        "{\n\t.reg .pred e;\n\telect.sync _|e, 0xffffffff;\n\t"
        "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::"r"(smem_u32(&bar))
        : "memory");
    asm volatile("{\n\t.reg .pred p;\n\tW: mbarrier.try_wait.parity.shared::cta.b64 p, [%0], 0;\n\t@p bra D;\n\tbra W;\n\tD:\n\t}" ::"r"(
                     smem_u32(&bar))
                 : "memory");
    if (threadIdx.x == 0) cycles[blockIdx.x] = clock64() - t0;
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (threadIdx.x < 32) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem));
  }
}

int main() {
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, 0);
  const int sms = prop.multiProcessorCount;
  printf("GPU: %s, %d SMs\n", prop.name, sms);
  if (FILE* f = popen("nvidia-smi --query-gpu=power.limit,clocks.max.sm,clocks.sm --format=csv,noheader -i 0", "r")) {
    char line[256];
    if (fgets(line, sizeof line, f)) printf("power.limit, clocks.max.sm, clocks.sm (before): %s", line);
    pclose(f);
  }
  const int smem = 120 * 1024;   // > half of the SM: one CTA per SM, so the 512-column TMEM allocation never waits
  cudaFuncSetAttribute(k_rate, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  long long* d_cyc;
  cudaMalloc(&d_cyc, sms * sizeof(long long));
  const int chunks = 400000;     // 400k x 4 x M128 N256 K16 per SM = 26.8 GFLOP per SM, ~0.1 s per run at the tensor peak
  const double flop = 2.0 * 128 * 256 * 64 * (double)chunks * sms;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  k_rate<<<sms, 128, smem>>>(0, 1000, d_cyc);   // warm-up of both modes
  k_rate<<<sms, 128, smem>>>(1, 1000, d_cyc);
  if (cudaDeviceSynchronize() != cudaSuccess) { printf("warm-up failed: %s\n", cudaGetErrorString(cudaGetLastError())); return 1; }
  const char* name[2] = {"N=256 x1     ", "N=128 x2 pair"};
  for (int rep = 0; rep < 3; ++rep)
    for (int mode = 0; mode < 2; ++mode) {
      cudaEventRecord(e0);
      k_rate<<<sms, 128, smem>>>(mode, chunks, d_cyc);
      cudaEventRecord(e1);
      cudaEventSynchronize(e1);
      float ms = 0.f;
      cudaEventElapsedTime(&ms, e0, e1);
      long long* h = (long long*)malloc(sms * sizeof(long long));
      cudaMemcpy(h, d_cyc, sms * sizeof(long long), cudaMemcpyDeviceToHost);
      long long mx = 0, mn = h[0];
      for (int i = 0; i < sms; ++i) { mx = h[i] > mx ? h[i] : mx; mn = h[i] < mn ? h[i] : mn; }
      free(h);
      printf("rep %d  %s  %8.3f ms  %7.1f TFLOP/s  SM cycles per M128xN256xK16 equivalent: %.1f .. %.1f\n", rep, name[mode], ms,
             flop / (ms * 1e-3) / 1e12, (double)mn / (4.0 * chunks), (double)mx / (4.0 * chunks));
    }
  if (FILE* f = popen("nvidia-smi --query-gpu=power.limit,clocks.max.sm,clocks.sm --format=csv,noheader -i 0", "r")) {
    char line[256];
    if (fgets(line, sizeof line, f)) printf("power.limit, clocks.max.sm, clocks.sm (after): %s", line);
    pclose(f);
  }
  const cudaError_t err = cudaGetLastError();
  if (err != cudaSuccess) { printf("CUDA error: %s\n", cudaGetErrorString(err)); return 1; }
  return 0;
}
