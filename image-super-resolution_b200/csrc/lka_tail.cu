// Tile-resident tail of an LKABlock on 64-channel fp32 token rows (Phase 3, the routing chain), on tcgen05 at fp32 accuracy:
//   x1 = x + s1 * BN1(x) * sigmoid(BN(pw(a)))        a = depthwise chain output          large_kernel_attention.py:96-105, 143-149
//   x2 = x1 + s2 * ffn2(GELU(ffn0(BN2(x1))))
// Three 1x1 contractions (64->64, 64->128, 128->64) that the fp32 path ran as three CUDA-core SGEMM launches (0.98 ms per
// 2040x1356 image at ~70 % of the FFMA peak, each streaming its operands through HBM).  Here a CTA keeps a 128-token tile on
// chip through all three, and the products run on the tensor cores WITHOUT giving up fp32 accuracy (the routing chain feeds
// the expert-selection indices, which must stay bit-exact): every fp32 operand is split into three bf16 terms
//   v = v1 + v2 + v3,   v1 = bf16(v), v2 = bf16(v - v1), v3 = bf16(v - v1 - v2)          (24 mantissa bits)
// and the six products that matter are accumulated in fp32 in TMEM:  a1 w1 + a1 w2 + a2 w1 + a2 w2 + a1 w3 + a3 w1;  the
// dropped terms are below 2^-24 of the result, i.e. below the rounding of an fp32 FMA chain.
//   operands : no-swizzle K-major planes (tc_ptx.cuh): activations [split][kg][row] = 16 B, weights [split][kg][n] = 16 B, all
//              three weight matrices resident (120 KB); the 128-wide hidden layer is consumed in two 64-channel halves.
//   threads  : 512 = 16 warps; warp w owns TMEM lanes 32 (w % 4) .. (the tcgen05.ld rule) = token rows, and channel quarter
//              w / 4 (16 of the 64 columns); warp 0 issues the MMAs (one PTX block of four K steps per split pair) between the
//              epilogue phases.
#include <cuda.h>
#include <stdlib.h>
#include "common.cuh"
#include "tc_ptx.cuh"
#include "../../include/ffsr_b200.h"

namespace {
using namespace tcx;

constexpr int LT_C = 64, LT_HID = 128;
constexpr int LT_TMEM_COLS = 256;                 // [0,64): stage 1 then stage 3; [64,192): stage 2
constexpr int LT_W1 = 3 * LT_C * LT_C * 2;        // 24,576 B  pw        [split][kg 8][n 64][8]
constexpr int LT_W0 = 3 * LT_HID * LT_C * 2;      // 49,152 B  ffn0      [split][kg 8][n 128][8]
constexpr int LT_W2 = 3 * LT_C * LT_HID * 2;      // 49,152 B  ffn2      [split][kg 16][n 64][8]
constexpr int LT_WBYTES = LT_W1 + LT_W0 + LT_W2;  // 122,880 B
constexpr int LT_SA = 3 * 8 * 128 * 16;           // 49,152 B  activation planes [split][kg 8][row 128]
constexpr int LT_PF = 64 * 3 + 128 + 64 + 8;      // fp32 parameters: b_pw[64] k1[64] d1[64] b0[128] b2[64] (s1 s2 come by pointer)
constexpr int LT_S_PAR = 64;
constexpr int LT_S_W = 2048;
constexpr int LT_S_A = LT_S_W + LT_WBYTES;
constexpr int LT_S_H = LT_S_A + LT_SA;
constexpr int LT_SMEM = LT_S_H + LT_SA;           // 223,232 B

// 8 fp32 values -> their three bf16 terms, as three 16-byte cells
__device__ __forceinline__ void split8(const float (&v)[8], uint4& c1, uint4& c2, uint4& c3) {
  uint32_t w1[4], w2[4], w3[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const float a = v[2 * k], b = v[2 * k + 1];
    const __nv_bfloat16 a1 = __float2bfloat16_rn(a), b1 = __float2bfloat16_rn(b);
    const float ra = a - __bfloat162float(a1), rb = b - __bfloat162float(b1);
    const __nv_bfloat16 a2 = __float2bfloat16_rn(ra), b2 = __float2bfloat16_rn(rb);
    const float sa = ra - __bfloat162float(a2), sb = rb - __bfloat162float(b2);
    const __nv_bfloat16 a3 = __float2bfloat16_rn(sa), b3 = __float2bfloat16_rn(sb);
    w1[k] = (uint32_t)__bfloat16_as_ushort(a1) | ((uint32_t)__bfloat16_as_ushort(b1) << 16);
    w2[k] = (uint32_t)__bfloat16_as_ushort(a2) | ((uint32_t)__bfloat16_as_ushort(b2) << 16);
    w3[k] = (uint32_t)__bfloat16_as_ushort(a3) | ((uint32_t)__bfloat16_as_ushort(b3) << 16);
  }
  c1 = make_uint4(w1[0], w1[1], w1[2], w1[3]);
  c2 = make_uint4(w2[0], w2[1], w2[2], w2[3]);
  c3 = make_uint4(w3[0], w3[1], w3[2], w3[3]);
}

// the six split products of one contraction: A planes [split][kg][128 rows], B planes [split][kg][n]; ksteps K=16 steps starting
// at activation plane 0 and weight plane kg0
__device__ __forceinline__ void lt_gemm(uint32_t tmem_d, uint32_t a32, uint32_t b32, int n, int kg_total_b, int kg0_b, int ksteps,
                                        uint32_t idesc, bool overwrite) {
  const uint32_t a_hi = desc_hi(128), b_hi = desc_hi(128);
  const uint32_t a_split = 8u * 2048u, b_split = (uint32_t)(kg_total_b * n * 16);
  const int pa[6] = {0, 0, 1, 1, 0, 2}, pb[6] = {0, 1, 0, 1, 2, 0};
  // (ksteps is 4 for every contraction here: one asm block per split pair issues its four K = 16 steps)
  (void)ksteps;
#pragma unroll
  for (int t = 0; t < 6; ++t) {
    const uint32_t al = desc_lo(a32 + (uint32_t)pa[t] * a_split, 2048u);
    const uint32_t bl = desc_lo(b32 + (uint32_t)pb[t] * b_split + (uint32_t)kg0_b * (uint32_t)(n * 16), (uint32_t)(n * 16));
    umma_taps_1x4(tmem_d, al, bl, idesc, (t == 0 && overwrite) ? 0u : 1u, a_hi, b_hi, (2u * 2048u) >> 4, (uint32_t)(2 * n), 0u);
  }
}

// 512 threads rather than 256: half the instructions per thread at four warps per scheduler.  The next tile's rows are
// prefetched into registers, and the second hidden half is written to the (dead) x1 planes so the two ffn2 MMA groups are
// issued without a wait in between.
__global__ void __launch_bounds__(512, 1) k_lka_tailw(const float* __restrict__ xin, const float* __restrict__ ain, long rows,
                                                      const uint8_t* __restrict__ wblob, const float* __restrict__ pblob,
                                                      const float* __restrict__ s1p, const float* __restrict__ s2p,
                                                      float* __restrict__ out) {
  extern __shared__ __align__(16) uint8_t smem[];
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + 8);
  float* par = reinterpret_cast<float*>(smem + LT_S_PAR);
  uint8_t* sW = smem + LT_S_W;
  uint8_t* sA = smem + LT_S_A;
  uint8_t* sH = smem + LT_S_H;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int row = (warp & 3) * 32 + lane;
  const int cq = warp >> 2;

  for (int i = tid; i < LT_WBYTES / 16; i += 512) reinterpret_cast<uint4*>(sW)[i] = __ldg(reinterpret_cast<const uint4*>(wblob) + i);
  for (int i = tid; i < LT_PF; i += 512) par[i] = __ldg(pblob + i);
  if (tid == 0) {
    mbar_init(bar, 1);
    fence_barrier_init();
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(LT_TMEM_COLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const float s1 = s1p[0], s2 = s2p[0];
  const float* b_pw = par;
  const float* k1 = par + 64;
  const float* d1 = par + 128;
  const float* b0 = par + 192;
  const float* b2 = par + 320;
  const uint32_t w1_32 = smem_u32(sW), w0_32 = w1_32 + LT_W1, w2_32 = w0_32 + LT_W0, a32 = smem_u32(sA), h32 = smem_u32(sH);
  const uint32_t id64 = idesc_bf16_m128(64), id128 = idesc_bf16_m128(128);
  const uint32_t trow = tmem + ((uint32_t)((warp & 3) * 32) << 16);
  uint32_t phase = 0;
  const long tiles = (rows + 127) / 128;
  const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);

  // 16 values -> their split cells in planes kg = 2 cq, 2 cq + 1 of `dst`
  auto put_split = [&](uint8_t* dst, const float* v16) {
#pragma unroll
    for (int g = 0; g < 2; ++g) {
      float v[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) v[i] = v16[8 * g + i];
      uint4 c1, c2, c3;
      split8(v, c1, c2, c3);
      uint8_t* cell = dst + (cq * 2 + g) * 2048 + row * 16;
      *reinterpret_cast<uint4*>(cell) = c1;
      *reinterpret_cast<uint4*>(cell + 8 * 2048) = c2;
      *reinterpret_cast<uint4*>(cell + 16 * 2048) = c3;
    }
  };
  float4 na[4], nx[4];
  bool nlive = false;
  if ((long)blockIdx.x < tiles) {
    const long r = (long)blockIdx.x * 128 + row;
    nlive = r < rows;
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      na[g] = nlive ? __ldg(reinterpret_cast<const float4*>(ain + r * LT_C + cq * 16) + g) : z4;
      nx[g] = nlive ? __ldg(reinterpret_cast<const float4*>(xin + r * LT_C + cq * 16) + g) : z4;
    }
  }
  for (long tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const long r = tile * 128 + row;
    const bool live = nlive;
    float x[16];
    {
      float a16[16];
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        a16[4 * g] = na[g].x; a16[4 * g + 1] = na[g].y; a16[4 * g + 2] = na[g].z; a16[4 * g + 3] = na[g].w;
        x[4 * g] = nx[g].x; x[4 * g + 1] = nx[g].y; x[4 * g + 2] = nx[g].z; x[4 * g + 3] = nx[g].w;
      }
      put_split(sA, a16);
    }
    if (tile + gridDim.x < tiles) {
      const long rn = (tile + gridDim.x) * 128 + row;
      nlive = rn < rows;
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        na[g] = nlive ? __ldg(reinterpret_cast<const float4*>(ain + rn * LT_C + cq * 16) + g) : z4;
        nx[g] = nlive ? __ldg(reinterpret_cast<const float4*>(xin + rn * LT_C + cq * 16) + g) : z4;
      }
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
      tc_fence_after();
      lt_gemm(tmem, a32, w1_32, 64, 8, 0, 4, id64, true);
      umma_commit(bar);
    }
    mbar_wait(bar, phase);
    phase ^= 1;
    tc_fence_after();
    {
      uint32_t v[16];
      tmem_ld16(trow + (uint32_t)(cq * 16), v);
      tmem_wait_ld(v);
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const int ch = cq * 16 + i;
        const float xr = x[i];
        x[i] = xr + s1 * (fmaf(xr, k1[ch], d1[ch]) * sigmoid_acc(__uint_as_float(v[i]) + b_pw[ch]));
      }
    }
    put_split(sA, x);                                // the a planes are dead: their MMAs completed
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
      tc_fence_after();
      lt_gemm(tmem + 64, a32, w0_32, 128, 8, 0, 4, id128, true);
      umma_commit(bar);
    }
    mbar_wait(bar, phase);
    phase ^= 1;
    tc_fence_after();
#pragma unroll 1
    for (int hh = 0; hh < 2; ++hh) {
      uint32_t v[16];
      tmem_ld16(trow + (uint32_t)(64 + hh * 64 + cq * 16), v);
      tmem_wait_ld(v);
      float y[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) y[i] = gelu_erf(__uint_as_float(v[i]) + b0[hh * 64 + cq * 16 + i]);
      put_split(hh == 0 ? sH : sA, y);               // second half: the x1 planes are dead (stage 2 completed)
      fence_proxy_async();
      tc_fence_before();
      __syncthreads();
      if (warp == 0) {
        tc_fence_after();
        lt_gemm(tmem, hh == 0 ? h32 : a32, w2_32, 64, 16, hh * 8, 4, id64, hh == 0);
        if (hh == 1) umma_commit(bar);
      }
    }
    mbar_wait(bar, phase);
    phase ^= 1;
    tc_fence_after();
    {
      uint32_t v[16];
      tmem_ld16(trow + (uint32_t)(cq * 16), v);
      tmem_wait_ld(v);
      if (live) {
        float4* op = reinterpret_cast<float4*>(out + r * LT_C + cq * 16);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          float o[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int j = q * 4 + i;
            o[i] = fmaf(s2, __uint_as_float(v[j]) + b2[cq * 16 + j], x[j]);
          }
          op[q] = make_float4(o[0], o[1], o[2], o[3]);
        }
      }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
  }
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(LT_TMEM_COLS));
}

// ---------------------------------------------------------------------------------------------------------------------
// bf16 variant for Phase 4 (128-channel tokens, hidden 256, bf16 residual stream): the same tail plus the first modulation
// layer (128 -> 32 per expert, the 1x1 conv that commutes with the bilinear upsampling), one kernel instead of four
// HBM-bound launches (pw 0.28 + ffn0 0.16 + ffn2 0.18 + mod0 0.07 ms).  Plain bf16 operands (this phase only feeds a sigmoid
// that is damped by 0.2).  Tiles are 128 tokens of ONE expert image; the expert's modulation weights are reloaded when the
// CTA's next tile belongs to another expert.  Only the 32-channel modulation features leave the kernel.
// ---------------------------------------------------------------------------------------------------------------------
constexpr int LB_C = 128, LB_HID = 256;
constexpr int LB_W1 = LB_C * LB_C * 2;            //  32,768 B  pw     [kg 16][n 128][8]
constexpr int LB_W0 = LB_HID * LB_C * 2;          //  65,536 B  ffn0   [kg 16][n 256][8]
constexpr int LB_W2 = LB_C * LB_HID * 2;          //  65,536 B  ffn2   [kg 32][n 128][8]
constexpr int LB_WM = 32 * LB_C * 2;              //   8,192 B  mod0 of ONE expert [kg 16][n 32][8]
constexpr int LB_WBYTES = LB_W1 + LB_W0 + LB_W2 + 4 * LB_WM;   // blob in global memory (all four experts)
constexpr int LB_PF = 128 * 3 + 256 + 128 + 128;  // b_pw k1 d1 | b0 | b2 | b_mod0[4][32]
constexpr int LB_S_PAR = 64;
constexpr int LB_S_W = 4096;
constexpr int LB_S_WM = LB_S_W + LB_W1 + LB_W0 + LB_W2;
constexpr int LB_S_A = LB_S_WM + LB_WM;           // activation planes [kg 16][row 128] = 32 KB
constexpr int LB_S_H = LB_S_A + 16 * 2048;        // hidden quarter planes [kg 8][row 128] = 16 KB
constexpr int LB_SMEM = LB_S_H + 8 * 2048;        // 225,280 B
constexpr int LB_TMEM_COLS = 512;                 // [0,128): stage 1 / 3; [128,384): stage 2; [128,160): modulation layer

// ---------------------------------------------------------------------------------------------------------------------
// k_lka_tail128w: 512 threads (warp w: TMEM lane group w % 4 = 32 token rows, channel quarter w / 4), the next tile's rows
// prefetched into registers, and the four hidden quarters written alternately to sH and to the two halves of the (by then
// dead) x1 planes, so the four ffn2 MMAs are issued back to back with the GELU epilogues instead of being waited for one by
// one.  ncu of an earlier 256-thread version: 3.3 k instructions per thread and tile at two warps per scheduler, 75 % of the
// issue cycles without an eligible warp (long-scoreboard on the un-prefetched loads, MMA waits).
// ---------------------------------------------------------------------------------------------------------------------
constexpr int LW_THREADS = 512;

__device__ __forceinline__ float bfl(uint32_t w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bfh(uint32_t w) { return __uint_as_float(w & 0xffff0000u); }

template <bool TANH>
__global__ void __launch_bounds__(LW_THREADS, 1) k_lka_tail128w(const __nv_bfloat16* __restrict__ xin, const __nv_bfloat16* __restrict__ ain,
                                                                int nimg, int HW, const uint8_t* __restrict__ wblob,
                                                                const float* __restrict__ pblob, const float* __restrict__ s1p,
                                                                const float* __restrict__ s2p, __nv_bfloat16* __restrict__ m32) {
  extern __shared__ __align__(16) uint8_t smem[];
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem);          // bar[0]: stage barrier, bar[1]: "ffn2 quarter 0 done" (sH reusable)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + 16);
  float* par = reinterpret_cast<float*>(smem + LB_S_PAR);
  uint8_t* sW = smem + LB_S_W;
  uint8_t* sWM = smem + LB_S_WM;
  uint8_t* sA = smem + LB_S_A;
  uint8_t* sH = smem + LB_S_H;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int row = (warp & 3) * 32 + lane;
  const int cq = warp >> 2;                          // 32 of the 128 columns

  for (int i = tid; i < (LB_W1 + LB_W0 + LB_W2) / 16; i += LW_THREADS) reinterpret_cast<uint4*>(sW)[i] = __ldg(reinterpret_cast<const uint4*>(wblob) + i);
  for (int i = tid; i < LB_PF; i += LW_THREADS) par[i] = __ldg(pblob + i);
  if (tid == 0) {
    mbar_init(bar, 1);
    mbar_init(bar + 1, 1);
    fence_barrier_init();
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(LB_TMEM_COLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const float s1 = s1p[0], s2 = s2p[0];
  const float* b_pw = par;
  const float* k1 = par + 128;
  const float* d1 = par + 256;
  const float* b0 = par + 384;
  const float* b2 = par + 640;
  const float* bm = par + 768;
  const uint32_t w1_32 = smem_u32(sW), w0_32 = w1_32 + LB_W1, w2_32 = w0_32 + LB_W0, wm_32 = smem_u32(sWM), a32 = smem_u32(sA), h32 = smem_u32(sH);
  const uint32_t hi = desc_hi(128);
  const uint32_t id128 = idesc_bf16_m128(128), id256 = idesc_bf16_m128(256), id32 = idesc_bf16_m128(32);
  const uint32_t trow = tmem + ((uint32_t)((warp & 3) * 32) << 16);
  uint32_t phase = 0, phase1 = 0;
  const int tpi = (HW + 127) / 128;
  const long tiles = (long)nimg * tpi;
  int cur_e = -1;
  const uint4 zero4 = make_uint4(0u, 0u, 0u, 0u);

  auto row_off = [&](long tile, bool& live) -> long {
    const int n = (int)(tile / tpi), pr = (int)(tile - (long)n * tpi) * 128 + row;
    live = pr < HW;
    return ((long)n * HW + (live ? pr : 0)) * LB_C + cq * 32;
  };
  uint4 na[4], nx[4];
  bool nlive = false;
  if ((long)blockIdx.x < tiles) {
    const long o = row_off(blockIdx.x, nlive);
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      na[g] = nlive ? __ldg(reinterpret_cast<const uint4*>(ain + o) + g) : zero4;
      nx[g] = nlive ? __ldg(reinterpret_cast<const uint4*>(xin + o) + g) : zero4;
    }
  }

  for (long tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const int n = (int)(tile / tpi);
    const int e = n & 3;
    const bool live = nlive;
    bool dummy;
    const long r32 = (row_off(tile, dummy) - cq * 32) / LB_C * 32;     // this row's offset in m32
    if (e != cur_e) {                                // (uniform) this expert's modulation weights; the previous tile's MMAs are done
      for (int i = tid; i < LB_WM / 16; i += LW_THREADS)
        reinterpret_cast<uint4*>(sWM)[i] = __ldg(reinterpret_cast<const uint4*>(wblob + LB_W1 + LB_W0 + LB_W2 + e * LB_WM) + i);
      cur_e = e;
    }
    float x[32];
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      *reinterpret_cast<uint4*>(sA + (cq * 4 + g) * 2048 + row * 16) = na[g];
      x[8 * g + 0] = bfl(nx[g].x); x[8 * g + 1] = bfh(nx[g].x); x[8 * g + 2] = bfl(nx[g].y); x[8 * g + 3] = bfh(nx[g].y);
      x[8 * g + 4] = bfl(nx[g].z); x[8 * g + 5] = bfh(nx[g].z); x[8 * g + 6] = bfl(nx[g].w); x[8 * g + 7] = bfh(nx[g].w);
    }
    if (tile + gridDim.x < tiles) {                  // next tile's rows: in flight during this tile's compute
      const long o = row_off(tile + gridDim.x, nlive);
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        na[g] = nlive ? __ldg(reinterpret_cast<const uint4*>(ain + o) + g) : zero4;
        nx[g] = nlive ? __ldg(reinterpret_cast<const uint4*>(xin + o) + g) : zero4;
      }
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    // ---- stage 1: G = a . Wpw^T (K = 128, N = 128)
    if (warp == 0) {
      tc_fence_after();
      umma_taps_1x4(tmem, desc_lo(a32, 2048u), desc_lo(w1_32, 128u * 16u), id128, 0u, hi, hi, (2u * 2048u) >> 4, 2u * 128u, 0u);
      umma_taps_1x4(tmem, desc_lo(a32 + 8u * 2048u, 2048u), desc_lo(w1_32 + 8u * 128u * 16u, 128u * 16u), id128, 1u, hi, hi, (2u * 2048u) >> 4, 2u * 128u, 0u);
      umma_commit(bar);
    }
    mbar_wait(bar, phase);
    phase ^= 1;
    tc_fence_after();
    // ---- epilogue 1: x1 = x + s1 * (x k1 + d1) * sigmoid(G + b) -> registers and planes (the a planes are dead)
    {
      uint32_t v0[16], v1[16];
      tmem_ld16(trow + (uint32_t)(cq * 32), v0);
      tmem_ld16(trow + (uint32_t)(cq * 32 + 16), v1);
      tmem_wait_ld(v0);
      tmem_wait_ld(v1);
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        const int ch = cq * 32 + i;
        const float g = __uint_as_float(i < 16 ? v0[i & 15] : v1[i & 15]) + b_pw[ch];
        const float sg = __fdividef(1.0f, 1.0f + __expf(-g));
        x[i] = fmaf(s1 * fmaf(x[i], k1[ch], d1[ch]), sg, x[i]);
      }
    }
#pragma unroll
    for (int g = 0; g < 4; ++g)
      *reinterpret_cast<uint4*>(sA + (cq * 4 + g) * 2048 + row * 16) =
          make_uint4(pack_bf16(x[g * 8], x[g * 8 + 1]), pack_bf16(x[g * 8 + 2], x[g * 8 + 3]), pack_bf16(x[g * 8 + 4], x[g * 8 + 5]),
                     pack_bf16(x[g * 8 + 6], x[g * 8 + 7]));
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    // ---- stage 2: Hd = x1 . W0^T (K = 128, N = 256) at TMEM column 128
    if (warp == 0) {
      tc_fence_after();
      umma_taps_1x4(tmem + 128, desc_lo(a32, 2048u), desc_lo(w0_32, 256u * 16u), id256, 0u, hi, hi, (2u * 2048u) >> 4, 2u * 256u, 0u);
      umma_taps_1x4(tmem + 128, desc_lo(a32 + 8u * 2048u, 2048u), desc_lo(w0_32 + 8u * 256u * 16u, 256u * 16u), id256, 1u, hi, hi, (2u * 2048u) >> 4, 2u * 256u, 0u);
      umma_commit(bar);
    }
    mbar_wait(bar, phase);
    phase ^= 1;
    tc_fence_after();
    // ---- stage 3: hidden quarters of 64 channels: GELU(Hd + b0) -> planes -> acc += . W2^T.  Quarter q goes to
    //      sH (q = 0, 3), x1 planes low half (q = 1), high half (q = 2): the MMAs are issued without waiting, except that
    //      quarter 3 reuses sH and waits for quarter 0's MMA (bar[1]), long complete by then.
#pragma unroll 1
    for (int q = 0; q < 4; ++q) {
      uint32_t v[16];
      tmem_ld16(trow + (uint32_t)(128 + q * 64 + cq * 16), v);
      tmem_wait_ld(v);
      float y[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const float z = __uint_as_float(v[i]) + b0[q * 64 + cq * 16 + i];
        y[i] = TANH ? gelu_tanh_fast(z) : gelu_erf_fast(z);
      }
      if (q == 3) {
        mbar_wait(bar + 1, phase1);
        phase1 ^= 1;
      }
      uint8_t* dst = (q == 0 || q == 3) ? sH : (q == 1 ? sA : sA + 8 * 2048);
#pragma unroll
      for (int g = 0; g < 2; ++g)
        *reinterpret_cast<uint4*>(dst + (cq * 2 + g) * 2048 + row * 16) =
            make_uint4(pack_bf16(y[g * 8], y[g * 8 + 1]), pack_bf16(y[g * 8 + 2], y[g * 8 + 3]), pack_bf16(y[g * 8 + 4], y[g * 8 + 5]),
                       pack_bf16(y[g * 8 + 6], y[g * 8 + 7]));
      fence_proxy_async();
      tc_fence_before();
      __syncthreads();
      if (warp == 0) {
        tc_fence_after();
        const uint32_t src = (q == 0 || q == 3) ? h32 : (q == 1 ? a32 : a32 + 8u * 2048u);
        umma_taps_1x4(tmem, desc_lo(src, 2048u), desc_lo(w2_32 + (uint32_t)(q * 8) * 128u * 16u, 128u * 16u), id128, q == 0 ? 0u : 1u, hi, hi,
                      (2u * 2048u) >> 4, 2u * 128u, 0u);
        if (q == 0) umma_commit(bar + 1);
        if (q == 3) umma_commit(bar);
      }
    }
    mbar_wait(bar, phase);
    phase ^= 1;
    tc_fence_after();
    // ---- epilogue 3: x2 = x1 + s2 * (acc + b2) -> planes
    {
      uint32_t v0[16], v1[16];
      tmem_ld16(trow + (uint32_t)(cq * 32), v0);
      tmem_ld16(trow + (uint32_t)(cq * 32 + 16), v1);
      tmem_wait_ld(v0);
      tmem_wait_ld(v1);
#pragma unroll
      for (int i = 0; i < 32; ++i)
        x[i] = fmaf(s2, __uint_as_float(i < 16 ? v0[i & 15] : v1[i & 15]) + b2[cq * 32 + i], x[i]);
    }
#pragma unroll
    for (int g = 0; g < 4; ++g)
      *reinterpret_cast<uint4*>(sA + (cq * 4 + g) * 2048 + row * 16) =
          make_uint4(pack_bf16(x[g * 8], x[g * 8 + 1]), pack_bf16(x[g * 8 + 2], x[g * 8 + 3]), pack_bf16(x[g * 8 + 4], x[g * 8 + 5]),
                     pack_bf16(x[g * 8 + 6], x[g * 8 + 7]));
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    // ---- stage 4: modulation layer 0 of this expert, m32 = x2 . Wm^T (K = 128, N = 32) at TMEM column 128
    if (warp == 0) {
      tc_fence_after();
      umma_taps_1x4(tmem + 128, desc_lo(a32, 2048u), desc_lo(wm_32, 32u * 16u), id32, 0u, hi, hi, (2u * 2048u) >> 4, 2u * 32u, 0u);
      umma_taps_1x4(tmem + 128, desc_lo(a32 + 8u * 2048u, 2048u), desc_lo(wm_32 + 8u * 32u * 16u, 32u * 16u), id32, 1u, hi, hi, (2u * 2048u) >> 4, 2u * 32u, 0u);
      umma_commit(bar);
    }
    mbar_wait(bar, phase);
    phase ^= 1;
    tc_fence_after();
    if (cq < 2) {
      uint32_t v[16];
      tmem_ld16(trow + (uint32_t)(128 + cq * 16), v);
      tmem_wait_ld(v);
      if (live) {
        const float* bb = bm + e * 32 + cq * 16;
        uint4* op = reinterpret_cast<uint4*>(m32 + r32 + cq * 16);
#pragma unroll
        for (int g = 0; g < 2; ++g)
          op[g] = make_uint4(pack_bf16(__uint_as_float(v[8 * g]) + bb[8 * g], __uint_as_float(v[8 * g + 1]) + bb[8 * g + 1]),
                             pack_bf16(__uint_as_float(v[8 * g + 2]) + bb[8 * g + 2], __uint_as_float(v[8 * g + 3]) + bb[8 * g + 3]),
                             pack_bf16(__uint_as_float(v[8 * g + 4]) + bb[8 * g + 4], __uint_as_float(v[8 * g + 5]) + bb[8 * g + 5]),
                             pack_bf16(__uint_as_float(v[8 * g + 6]) + bb[8 * g + 6], __uint_as_float(v[8 * g + 7]) + bb[8 * g + 7]));
      }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
  }
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(LB_TMEM_COLS));
}
}  // namespace

extern "C" size_t ffsr_lka_tail_weight_bytes(void) { return (size_t)LT_WBYTES; }
extern "C" size_t ffsr_lka_tail_param_floats(void) { return (size_t)LT_PF; }

// x, a, out: fp32 [rows][64] (out may alias neither input); wblob / pblob: isr_b200.pipeline.pack_lka_tail
extern "C" int ffsr_lka_tail64(const float* x, const float* a, long rows, const void* wblob, const float* pblob, const float* scale1,
                               const float* scale2, float* out, cudaStream_t stream) {
  FFSR_REQUIRE(x && a && wblob && pblob && scale1 && scale2 && out && rows > 0, FFSR_ERR_ARG, "lka_tail64: bad argument");
  FFSR_REQUIRE(((uintptr_t)x % 16) == 0 && ((uintptr_t)a % 16) == 0 && ((uintptr_t)out % 16) == 0 && ((uintptr_t)wblob % 16) == 0,
               FFSR_ERR_ALIGN, "lka_tail64: 16-byte alignment required");
  static int num_sms = 0;
  if (!num_sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
    cudaFuncSetAttribute(k_lka_tailw, cudaFuncAttributeMaxDynamicSharedMemorySize, LT_SMEM);
  }
  const long tiles = (rows + 127) / 128;
  const int grid = (int)(tiles < num_sms ? tiles : num_sms);
  k_lka_tailw<<<grid, 512, LT_SMEM, stream>>>(x, a, rows, (const uint8_t*)wblob, pblob, scale1, scale2, out);
  return ffsr_check_launch("lka_tail64");
}

extern "C" size_t ffsr_lka_tail128_weight_bytes(void) { return (size_t)LB_WBYTES; }
extern "C" size_t ffsr_lka_tail128_param_floats(void) { return (size_t)LB_PF; }

// x, a: bf16 [nimg][HW][128] (nimg = B * 4 expert images, expert = image index % 4); m32: bf16 [nimg][HW][32]
extern "C" int ffsr_lka_tail128_mod(const void* x, const void* a, int nimg, int HW, const void* wblob, const float* pblob,
                                    const float* scale1, const float* scale2, void* m32, cudaStream_t stream) {
  FFSR_REQUIRE(x && a && wblob && pblob && scale1 && scale2 && m32 && nimg > 0 && HW > 0, FFSR_ERR_ARG, "lka_tail128_mod: bad argument");
  FFSR_REQUIRE(((uintptr_t)x % 16) == 0 && ((uintptr_t)a % 16) == 0 && ((uintptr_t)m32 % 16) == 0 && ((uintptr_t)wblob % 16) == 0,
               FFSR_ERR_ALIGN, "lka_tail128_mod: 16-byte alignment required");
  static int num_sms = 0;
  static const bool erf_forced = getenv("FFSR_TC_GELU_ERF") != nullptr;
  if (!num_sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
    cudaFuncSetAttribute(k_lka_tail128w<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, LB_SMEM);
    cudaFuncSetAttribute(k_lka_tail128w<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, LB_SMEM);
  }
  const long tiles = (long)nimg * ((HW + 127) / 128);
  const int grid = (int)(tiles < num_sms ? tiles : num_sms);
  if (erf_forced)
    k_lka_tail128w<false><<<grid, LW_THREADS, LB_SMEM, stream>>>((const __nv_bfloat16*)x, (const __nv_bfloat16*)a, nimg, HW, (const uint8_t*)wblob,
                                                                  pblob, scale1, scale2, (__nv_bfloat16*)m32);
  else
    k_lka_tail128w<true><<<grid, LW_THREADS, LB_SMEM, stream>>>((const __nv_bfloat16*)x, (const __nv_bfloat16*)a, nimg, HW, (const uint8_t*)wblob,
                                                                 pblob, scale1, scale2, (__nv_bfloat16*)m32);
  return ffsr_check_launch("lka_tail128_mod");
}
