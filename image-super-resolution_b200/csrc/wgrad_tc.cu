// tcgen05 convolution weight gradient (1x1 / 3x3), bf16 operands, fp32 accumulation in TMEM.
//
//   dW[tap][ci][co] = sum_{n,y,x} X[n, y+dy, x+dx, ci] * dY[n, y, x, co]
//
//   GEMM view : D[ci, co] (one accumulator per tap) += A[ci, pixel] * B[pixel, co],  K = pixels.
//   Both operands are "MN-major" for the tensor core (the contraction index -- the pixel -- is the
//   slow index of the channels-last tensors), so NO transposed copy of the activations is needed:
//   the same SWIZZLE_128B TMA boxes the forward conv uses ({64 ch, 16 px, rows, 1}: one 128-byte
//   row per pixel) are read by tcgen05.mma with a_major = b_major = MN.  Canonical MN-major SW128
//   layout: 64 channels (128 B) contiguous, 8 pixel rows per 1024-byte swizzle atom (SBO = 1024),
//   next 64-channel block at LBO (= the next TMA box).
//   tile      : K chunk = 128 pixels (8 rows x 16 cols of one image) per pipeline stage.
//   A operand : row-haloed copy of the X tile at x offset (dx - pad): the operand of tap (dy, dx) for
//               K-step k (16 pixels = one image row of the tile) is the copy at byte offset
//               (dy + k) * 2048 -- one load serves the three dy taps.
//   B operand : the dY tile, K-step k at byte offset k * 2048.
//   work split: CTA = (pixel-tile subset p, dx, ci block of 128, co block of 64/128); ks accumulators
//               (dy = 0..ks-1) of 128 lanes x nblk columns live in TMEM for the whole kernel; partial
//               results go to a workspace [P][taps][CinPad][CoutPad] that a second kernel reduces
//               into dw (deterministic, no atomics).
//   warps     : 0 = TMA producer, 1 = MMA issuer (+ TMEM alloc), 2..5 = epilogue (TMEM lane quarters).
#include <cuda.h>
#include "common.cuh"
#include "../../include/ffsr_b200.h"

namespace {

constexpr int WT_TH = 8, WT_TW = 16;
constexpr int WT_ROW_BYTES = WT_TW * 128;       // one image row of a tile: 16 px x 64 bf16 channels
constexpr int WT_B_BYTES = WT_TH * WT_ROW_BYTES;   // 16 KB per 64-channel dY block
constexpr int WT_MAX_STAGES = 6;
constexpr int WT_SMEM_MAX = 232448;
constexpr int WT_SMEM_HDR = 1024;
constexpr int WT_THREADS = 192;
constexpr int WT_TMEM_COLS = 512;

struct WgArgs {
  int N, H, W, Cin, Cout, ks;
  int nblk;               // 64 or 128 output channels per CTA
  int a_chunks, b_chunks; // 64-channel blocks of the ci / co block actually loaded
  int a_bytes;            // bytes of one haloed 64-channel X copy
  int stage_bytes, nstages;
  int tiles_x, tiles_y;
  long long total_tiles;
  int P;                  // pixel-tile subsets
  int ci_blocks, co_blocks;
  int cin_pad, cout_pad;  // workspace extents: ci_blocks*128, co_blocks*nblk
  float* ws;
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WG_WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra WG_WAIT_DONE;\n\t"
      "bra WG_WAIT_LOOP;\n\t"
      "WG_WAIT_DONE:\n\t"
      "}" ::"r"(smem_u32(bar)), "r"(parity)
      : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tma_load_4d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2,
                                            int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void umma_bf16_ss(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum)
      : "memory");
}
// Eight K-steps of one accumulator in ONE asm block, issued by one elected lane of a converged warp: the descriptor
// low words advance by a_inc / b_inc (16-byte units) in PTX.  A single thread that builds two 64-bit descriptors and
// issues one tcgen05.mma per C++ statement spends ~100+ cycles per instruction, which bounds the small-N layers
// (N = 32: 16 cycles of tensor work per MMA); inside the block each further MMA costs a few uniform adds.
__device__ __forceinline__ void umma_wg_k8(uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                           uint32_t idesc, uint32_t acc_first, uint32_t a_inc, uint32_t b_inc) {
  asm volatile(
      "{\n\t"
      ".reg .pred p, e, t;\n\t"
      ".reg .b64 da, db;\n\t"
      ".reg .b32 al, bl;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "setp.eq.b32 t, 0, 0;\n\t"
      "mov.b32 al, %1;\n\t"
      "mov.b32 bl, %3;\n\t"
      "mov.b64 da, {al, %2};\n\t"
      "mov.b64 db, {bl, %4};\n\t"
      "@e tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t"
      "add.u32 al, al, %7;\n\t add.u32 bl, bl, %8;\n\t mov.b64 da, {al, %2};\n\t mov.b64 db, {bl, %4};\n\t"
      "@e tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, t;\n\t"
      "add.u32 al, al, %7;\n\t add.u32 bl, bl, %8;\n\t mov.b64 da, {al, %2};\n\t mov.b64 db, {bl, %4};\n\t"
      "@e tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, t;\n\t"
      "add.u32 al, al, %7;\n\t add.u32 bl, bl, %8;\n\t mov.b64 da, {al, %2};\n\t mov.b64 db, {bl, %4};\n\t"
      "@e tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, t;\n\t"
      "add.u32 al, al, %7;\n\t add.u32 bl, bl, %8;\n\t mov.b64 da, {al, %2};\n\t mov.b64 db, {bl, %4};\n\t"
      "@e tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, t;\n\t"
      "add.u32 al, al, %7;\n\t add.u32 bl, bl, %8;\n\t mov.b64 da, {al, %2};\n\t mov.b64 db, {bl, %4};\n\t"
      "@e tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, t;\n\t"
      "add.u32 al, al, %7;\n\t add.u32 bl, bl, %8;\n\t mov.b64 da, {al, %2};\n\t mov.b64 db, {bl, %4};\n\t"
      "@e tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, t;\n\t"
      "add.u32 al, al, %7;\n\t add.u32 bl, bl, %8;\n\t mov.b64 da, {al, %2};\n\t mov.b64 db, {bl, %4};\n\t"
      "@e tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, t;\n\t"
      "}" ::"r"(tmem_d),
      "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(acc_first), "r"(a_inc), "r"(b_inc)
      : "memory");
}
__device__ __forceinline__ void umma_commit_e(uint64_t* bar) {
  asm volatile(
      "{\n\t"
      ".reg .pred e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t"
      "}" ::"r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ uint32_t mn_lo(uint32_t smem_addr, uint32_t lbo_bytes) {
  return ((smem_addr & 0x3FFFFu) >> 4) | ((lbo_bytes >> 4) << 16);
}
__device__ __forceinline__ uint32_t mn_hi(uint32_t sbo_bytes, uint32_t layout) {
  return (sbo_bytes >> 4) | (1u << 14) | (layout << 29);
}

// MN-major SWIZZLE_128B descriptor: start>>4 [0,14) | LBO>>4 [16,30) | SBO>>4 [32,46) | version 1 [46,48) | layout 2 [61,64)
__device__ __forceinline__ uint64_t mn_desc(uint32_t smem_addr, uint32_t lbo_bytes) {
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(1024u >> 4) << 32) |
         (1ull << 46) | (2ull << 61);
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n\t"
      "tcgen05.wait::ld.sync.aligned;"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}

__global__ void __launch_bounds__(WT_THREADS, 1)
k_wgrad_tc(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmD, const WgArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full = reinterpret_cast<uint64_t*>(smem);       // [WT_MAX_STAGES]
  uint64_t* empty = full + WT_MAX_STAGES;                    // [WT_MAX_STAGES]
  uint64_t* tdone = empty + WT_MAX_STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tdone + 1);
  uint8_t* stages = smem + WT_SMEM_HDR;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int p = blockIdx.x / a.ks, dxi = blockIdx.x % a.ks;
  const int cib = blockIdx.y / a.co_blocks, cob = blockIdx.y % a.co_blocks;
  const int ci0 = cib * 128, co0 = cob * a.nblk;
  const int pad = a.ks / 2;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmX)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmD)) : "memory");
    for (int i = 0; i < WT_MAX_STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    mbar_init(tdone, 1);
    fence_barrier_init();
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(WT_TMEM_COLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const long long my_tiles = a.total_tiles > p ? (a.total_tiles - p + a.P - 1) / a.P : 0;

  if (warp == 0) {
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      const uint32_t tx_bytes = (uint32_t)(a.a_chunks * a.a_bytes + a.b_chunks * WT_B_BYTES);
      for (long long t = p; t < a.total_tiles; t += a.P) {
        const int tx = (int)(t % a.tiles_x);
        const long long r = t / a.tiles_x;
        const int ty = (int)(r % a.tiles_y);
        const int n = (int)(r / a.tiles_y);
        mbar_wait(&empty[s], ph ^ 1);
        uint8_t* st = stages + s * a.stage_bytes;
        mbar_expect_tx(&full[s], tx_bytes);
        for (int ch = 0; ch < a.a_chunks; ++ch)
          tma_load_4d(st + ch * a.a_bytes, &tmX, &full[s], ci0 + ch * 64, tx * WT_TW + dxi - pad, ty * WT_TH - pad, n);
        uint8_t* sb = st + 2 * a.a_bytes;
        for (int ch = 0; ch < a.b_chunks; ++ch)
          tma_load_4d(sb + ch * WT_B_BYTES, &tmD, &full[s], co0 + ch * 64, tx * WT_TW, ty * WT_TH, n);
        if (++s == a.nstages) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp == 1) {
    {
      // instruction descriptor: D fp32, A/B bf16, both MN-major, N = nblk, M = 128 (whole warp converged; one
      // elected lane issues inside umma_wg_k8)
      const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) |
                             ((uint32_t)(a.nblk >> 3) << 17) | ((128u >> 4) << 24);
      const uint32_t hi = mn_hi(1024u, 2u);
      int s = 0;
      uint32_t ph = 0;
      long long it = 0;
      for (long long t = p; t < a.total_tiles; t += a.P, ++it) {
        mbar_wait(&full[s], ph);
        tc_fence_after();
        const uint32_t a_addr = smem_u32(stages + s * a.stage_bytes);
        const uint32_t b_addr = a_addr + 2u * (uint32_t)a.a_bytes;
        const uint32_t bl = mn_lo(b_addr, (uint32_t)WT_B_BYTES);
        for (int dy = 0; dy < a.ks; ++dy)
          umma_wg_k8(tmem_base + (uint32_t)(dy * a.nblk), mn_lo(a_addr + (uint32_t)dy * WT_ROW_BYTES, (uint32_t)a.a_bytes), hi, bl,
                     hi, idesc, it > 0 ? 1u : 0u, WT_ROW_BYTES >> 4, WT_ROW_BYTES >> 4);
        umma_commit_e(&empty[s]);
        if (++s == a.nstages) { s = 0; ph ^= 1; }
      }
      umma_commit_e(tdone);
    }
  } else {
    // epilogue: warp w reads TMEM lanes [32*(w%4), +32) = ci rows, 16 co columns at a time
    if (my_tiles > 0) {
      mbar_wait(tdone, 0);
      tc_fence_after();
    }
    const int q = warp & 3;
    const int ci = ci0 + q * 32 + lane;
    for (int dy = 0; dy < a.ks; ++dy) {
      const int tap = dy * a.ks + dxi;
      float* dst = a.ws + (((long long)p * a.ks * a.ks + tap) * a.cin_pad + ci) * a.cout_pad + co0;
      for (int c = 0; c < a.nblk; c += 16) {
        uint32_t v[16];
        if (my_tiles > 0) {
          tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(dy * a.nblk + c), v);
        } else {
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = 0u;
        }
#pragma unroll
        for (int i = 0; i < 4; ++i)
          reinterpret_cast<float4*>(dst + c)[i] = make_float4(__uint_as_float(v[4 * i]), __uint_as_float(v[4 * i + 1]),
                                                              __uint_as_float(v[4 * i + 2]), __uint_as_float(v[4 * i + 3]));
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(WT_TMEM_COLS));
  }
}

// ------------------------------------------------------------------------------------------------------------
// Single-copy variant for 3x3 layers with Cout <= 32 (two 32-wide cout blocks re-read X and measured slower for Cout 64).
// The three-CTAs-per-dx kernel above moves each X tile and each dY tile three times from L2 and those layers are
// bound by exactly that traffic.  Here ONE CTA owns all nine taps of a (128-ci, 32-co) block:
//   * X: ONE haloed copy per 64-channel chunk {64 ch, 10 px, 18 rows} of a 16x8-pixel tile (SWIZZLE_128B); the
//     operand of tap (dy,dx), K-step k (16 pixels = 2 image rows) is that copy at byte offset
//     dy*1280 + dx*128 + k*2560, K-groups (8 pixels = one image row) SBO = 1280 B apart -- the swizzle is a function
//     of the absolute shared-memory address, so shifted starts need no base offset (measured, see conv_tc.cu);
//   * dY: {32 ch, 8 px, 16 rows} boxes, SWIZZLE_64B (64-byte rows: one MN-major atom of 32 channels), K-step k at
//     k*1024, K-groups 512 B apart;
//   * nine accumulators of 128 lanes x 32 columns (288 of 512 TMEM columns) live for the whole kernel.
// ------------------------------------------------------------------------------------------------------------
constexpr int W1_A_BYTES = 18 * 10 * 128, W1_A_STAGE = (W1_A_BYTES + 1023) / 1024 * 1024;   // 23040 -> 23552
constexpr int W1_B_BYTES = 16 * 8 * 64;                                                    // 8192
constexpr int W1_STAGE = 2 * W1_A_STAGE + W1_B_BYTES;

struct Wg1Args {
  int N, H, W, Cin, Cout;
  int a_chunks, nstages;
  int tiles_x, tiles_y;
  long long total_tiles;
  int P, ci_blocks, co_blocks, cin_pad, cout_pad;
  float* ws;
};

// MN-major descriptor with explicit SBO / swizzle mode (2 = 128B, 4 = 64B)
__device__ __forceinline__ uint64_t mn_desc2(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout) {
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(sbo_bytes >> 4) << 32) |
         (1ull << 46) | ((uint64_t)layout << 61);
}

__global__ void __launch_bounds__(WT_THREADS, 1)
k_wgrad_tc1c(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmD, const Wg1Args a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full = reinterpret_cast<uint64_t*>(smem);
  uint64_t* empty = full + WT_MAX_STAGES;
  uint64_t* tdone = empty + WT_MAX_STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tdone + 1);
  uint8_t* stages = smem + WT_SMEM_HDR;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int p = blockIdx.x;
  const int cib = blockIdx.y / a.co_blocks, cob = blockIdx.y % a.co_blocks;
  const int ci0 = cib * 128, co0 = cob * 32;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmX)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmD)) : "memory");
    for (int i = 0; i < WT_MAX_STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    mbar_init(tdone, 1);
    fence_barrier_init();
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(WT_TMEM_COLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const long long my_tiles = a.total_tiles > p ? (a.total_tiles - p + a.P - 1) / a.P : 0;

  if (warp == 0) {
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      const uint32_t tx_bytes = (uint32_t)(a.a_chunks * W1_A_BYTES + W1_B_BYTES);
      for (long long t = p; t < a.total_tiles; t += a.P) {
        const int tx = (int)(t % a.tiles_x);
        const long long r = t / a.tiles_x;
        const int ty = (int)(r % a.tiles_y);
        const int n = (int)(r / a.tiles_y);
        mbar_wait(&empty[s], ph ^ 1);
        uint8_t* st = stages + s * W1_STAGE;
        mbar_expect_tx(&full[s], tx_bytes);
        for (int ch = 0; ch < a.a_chunks; ++ch)
          tma_load_4d(st + ch * W1_A_STAGE, &tmX, &full[s], ci0 + ch * 64, tx * 8 - 1, ty * 16 - 1, n);
        tma_load_4d(st + 2 * W1_A_STAGE, &tmD, &full[s], co0, tx * 8, ty * 16, n);
        if (++s == a.nstages) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp == 1) {
    {
      const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((32u >> 3) << 17) | ((128u >> 4) << 24);
      const uint32_t a_hi = mn_hi(1280u, 2u), b_hi = mn_hi(512u, 4u);
      int s = 0;
      uint32_t ph = 0;
      long long it = 0;
      for (long long t = p; t < a.total_tiles; t += a.P, ++it) {
        mbar_wait(&full[s], ph);
        tc_fence_after();
        const uint32_t a_addr = smem_u32(stages + s * W1_STAGE);
        const uint32_t bl = mn_lo(a_addr + 2u * W1_A_STAGE, 0u);
#pragma unroll 1
        for (int tap = 0; tap < 9; ++tap) {
          const uint32_t tap_off = (uint32_t)(tap / 3) * 1280u + (uint32_t)(tap % 3) * 128u;
          umma_wg_k8(tmem_base + (uint32_t)(tap * 32), mn_lo(a_addr + tap_off, W1_A_STAGE), a_hi, bl, b_hi, idesc,
                     it > 0 ? 1u : 0u, 2560u >> 4, 1024u >> 4);
        }
        umma_commit_e(&empty[s]);
        if (++s == a.nstages) { s = 0; ph ^= 1; }
      }
      umma_commit_e(tdone);
    }
  } else {
    if (my_tiles > 0) {
      mbar_wait(tdone, 0);
      tc_fence_after();
    }
    const int q = warp & 3;
    const int ci = ci0 + q * 32 + lane;
    for (int tap = 0; tap < 9; ++tap) {
      float* dst = a.ws + (((long long)p * 9 + tap) * a.cin_pad + ci) * a.cout_pad + co0;
      for (int c = 0; c < 32; c += 16) {
        uint32_t v[16];
        if (my_tiles > 0) {
          tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(tap * 32 + c), v);
        } else {
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = 0u;
        }
#pragma unroll
        for (int i = 0; i < 4; ++i)
          reinterpret_cast<float4*>(dst + c)[i] = make_float4(__uint_as_float(v[4 * i]), __uint_as_float(v[4 * i + 1]),
                                                              __uint_as_float(v[4 * i + 2]), __uint_as_float(v[4 * i + 3]));
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(WT_TMEM_COLS));
  }
}

// dw[tap][ci][co] += sum_p ws[p][tap][ci][co] in blocks [0, dw_blocks); the blocks after them finish the bias sums
constexpr int WR_THREADS = 1024;
__global__ void __launch_bounds__(WR_THREADS) k_wgrad_reduce(const float* __restrict__ ws, int P, int taps, int Cin, int Cout,
                                                             int cin_pad, int cout_pad, float* __restrict__ dw,
                                                             long dw_blocks, const SlotSum<float> bias) {
  if ((long)blockIdx.x >= dw_blocks) {
    sum_slots_chunk(bias, blockIdx.x - dw_blocks);
    return;
  }
  const long total = (long)taps * Cin * Cout;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += dw_blocks * blockDim.x) {
    const int co = (int)(i % Cout);
    const int ci = (int)((i / Cout) % Cin);
    const int tap = (int)(i / ((long)Cout * Cin));
    float s = 0.f;
    for (int p = 0; p < P; ++p) s += ws[(((long)p * taps + tap) * cin_pad + ci) * cout_pad + co];
    dw[i] += s;
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn wg_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

struct WgPlan {
  int nblk, ci_blocks, co_blocks, cin_pad, cout_pad, P, tiles_x, tiles_y;
  long long total_tiles;
};
bool wg_single_copy(int H, int Cout, int ks) { return ks == 3 && Cout <= 32 && H >= 8; }

WgPlan wg_plan(int N, int H, int W, int Cin, int Cout, int ks) {
  WgPlan pl;
  if (wg_single_copy(H, Cout, ks)) {
    pl.nblk = 32;
    pl.ci_blocks = (Cin + 127) / 128;
    pl.co_blocks = (Cout + 31) / 32;
    pl.cin_pad = pl.ci_blocks * 128;
    pl.cout_pad = pl.co_blocks * 32;
    pl.tiles_x = ceil_div(W, 8);
    pl.tiles_y = ceil_div(H, 16);
    pl.total_tiles = (long long)pl.tiles_x * pl.tiles_y * N;
    long long P = 148 / ((long long)pl.ci_blocks * pl.co_blocks);
    if (P < 1) P = 1;
    const long long maxP = (pl.total_tiles + 3) / 4;
    if (P > maxP) P = maxP < 1 ? 1 : maxP;
    pl.P = (int)P;
    return pl;
  }
  pl.nblk = Cout > 64 ? 128 : 64;
  pl.ci_blocks = (Cin + 127) / 128;
  pl.co_blocks = (Cout + pl.nblk - 1) / pl.nblk;
  pl.cin_pad = pl.ci_blocks * 128;
  pl.cout_pad = pl.co_blocks * pl.nblk;
  pl.tiles_x = ceil_div(W, WT_TW);
  pl.tiles_y = ceil_div(H, WT_TH);
  pl.total_tiles = (long long)pl.tiles_x * pl.tiles_y * N;
  long long P = 148 / ((long long)ks * pl.ci_blocks * pl.co_blocks);
  if (P < 1) P = 1;
  const long long maxP = (pl.total_tiles + 3) / 4;     // at least ~4 tiles per CTA: the epilogue is per CTA
  if (P > maxP) P = maxP < 1 ? 1 : maxP;
  pl.P = (int)P;
  return pl;
}
}  // namespace

extern "C" size_t ffsr_conv2d_wgrad_tc_workspace_bytes(int N, int H, int W, int Cin, int Cout, int ksize) {
  const WgPlan pl = wg_plan(N, H, W, Cin, Cout, ksize);
  return ws_align((size_t)pl.P * ksize * ksize * pl.cin_pad * pl.cout_pad * sizeof(float)) +
         ffsr_colsum_workspace_bytes(N, H, W, Cout);
}

namespace {
// bias column-sum partials (after the weight-gradient partials in ws), then ONE launch reduces both
int wgrad_tc_finish(const ffsr_wgrad_params& p, const WgPlan& pl, int taps, void* ws, cudaStream_t stream) {
  SlotSum<float> bias{};
  if (p.dbias) {
    float* bpart = (float*)((char*)ws + ws_align((size_t)pl.P * taps * pl.cin_pad * pl.cout_pad * sizeof(float)));
    int nb;
    const int rc = colsum_partials(p.dy, p.dy_dtype, p.N, p.H, p.W, p.Cout, p.dy_sN, p.dy_sY, p.dy_sX, bpart, &nb, stream);
    if (rc) return rc;
    bias = slot_sum<float>(bpart, nb, p.Cout, p.dbias);
  }
  const long dw_blocks = ((long)taps * p.Cin * p.Cout + WR_THREADS - 1) / WR_THREADS;
  k_wgrad_reduce<<<(unsigned)(dw_blocks + slot_sum_blocks(bias)), WR_THREADS, 0, stream>>>(
      (const float*)ws, pl.P, taps, p.Cin, p.Cout, pl.cin_pad, pl.cout_pad, p.dw, dw_blocks, bias);
  return ffsr_check_launch("conv2d_wgrad_reduce");
}
}  // namespace

// x, dy: bf16 channels-last with 16-byte-multiple strides (pad the channel pitch to a multiple of 8)
extern "C" int ffsr_conv2d_wgrad_tc(const ffsr_wgrad_params* pp, void* ws, size_t ws_bytes, cudaStream_t stream) {
  FFSR_REQUIRE(pp && ws, FFSR_ERR_ARG, "conv2d_wgrad_tc: null pointer");
  const ffsr_wgrad_params& p = *pp;
  FFSR_REQUIRE(p.x && p.dy && p.dw, FFSR_ERR_ARG, "conv2d_wgrad_tc: null pointer");
  FFSR_REQUIRE(p.x_dtype == FFSR_DT_BF16 && p.dy_dtype == FFSR_DT_BF16 && p.x_sC == 1, FFSR_ERR_ARG,
               "conv2d_wgrad_tc: x and dy must be bf16 channels-last");
  FFSR_REQUIRE(p.ksize == 1 || p.ksize == 3, FFSR_ERR_ARG, "conv2d_wgrad_tc: ksize must be 1 or 3");
  FFSR_REQUIRE(p.N > 0 && p.H > 0 && p.W > 0 && p.Cin > 0 && p.Cout > 0, FFSR_ERR_ARG, "conv2d_wgrad_tc: bad shape");
  auto ok16 = [](const void* b, long long s0, long long s1, long long s2) {
    return ((uintptr_t)b % 16) == 0 && (s0 * 2) % 16 == 0 && (s1 * 2) % 16 == 0 && (s2 * 2) % 16 == 0;
  };
  FFSR_REQUIRE(ok16(p.x, p.x_sX, p.x_sY, p.x_sN) && ok16(p.dy, p.dy_sX, p.dy_sY, p.dy_sN), FFSR_ERR_ALIGN,
               "conv2d_wgrad_tc: TMA needs 16B-aligned bases and 16B-multiple strides");
  EncodeTiledFn enc = wg_encode_fn();
  FFSR_REQUIRE(enc, FFSR_ERR_DRIVER, "conv2d_wgrad_tc: cuTensorMapEncodeTiled entry point unavailable");
  const WgPlan pl = wg_plan(p.N, p.H, p.W, p.Cin, p.Cout, p.ksize);
  FFSR_REQUIRE(ws_bytes >= ffsr_conv2d_wgrad_tc_workspace_bytes(p.N, p.H, p.W, p.Cin, p.Cout, p.ksize), FFSR_ERR_ARG,
               "conv2d_wgrad_tc: workspace too small");
  const int pad = p.ksize / 2;
  if (wg_single_copy(p.H, p.Cout, p.ksize)) {
    CUtensorMap tX, tD;
    {
      cuuint64_t dims[4] = {(cuuint64_t)p.Cin, (cuuint64_t)p.W, (cuuint64_t)p.H, (cuuint64_t)p.N};
      cuuint64_t strides[3] = {(cuuint64_t)p.x_sX * 2, (cuuint64_t)p.x_sY * 2, (cuuint64_t)p.x_sN * 2};
      cuuint32_t box[4] = {64, 10, 18, 1};
      cuuint32_t es[4] = {1, 1, 1, 1};
      CUresult r = enc(&tX, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(p.x), dims, strides, box, es,
                       CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                       CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      FFSR_REQUIRE(r == CUDA_SUCCESS, FFSR_ERR_DRIVER, "conv2d_wgrad_tc: x tensor map encode failed (CUresult %d)", (int)r);
    }
    {
      cuuint64_t dims[4] = {(cuuint64_t)p.Cout, (cuuint64_t)p.W, (cuuint64_t)p.H, (cuuint64_t)p.N};
      cuuint64_t strides[3] = {(cuuint64_t)p.dy_sX * 2, (cuuint64_t)p.dy_sY * 2, (cuuint64_t)p.dy_sN * 2};
      cuuint32_t box[4] = {32, 8, 16, 1};
      cuuint32_t es[4] = {1, 1, 1, 1};
      CUresult r = enc(&tD, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(p.dy), dims, strides, box, es,
                       CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                       CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      FFSR_REQUIRE(r == CUDA_SUCCESS, FFSR_ERR_DRIVER, "conv2d_wgrad_tc: dy tensor map encode failed (CUresult %d)", (int)r);
    }
    Wg1Args a1;
    a1.N = p.N; a1.H = p.H; a1.W = p.W; a1.Cin = p.Cin; a1.Cout = p.Cout;
    a1.a_chunks = p.Cin > 64 ? 2 : 1;
    a1.nstages = (WT_SMEM_MAX - 1024 - WT_SMEM_HDR) / W1_STAGE;
    if (a1.nstages > WT_MAX_STAGES) a1.nstages = WT_MAX_STAGES;
    a1.tiles_x = pl.tiles_x; a1.tiles_y = pl.tiles_y; a1.total_tiles = pl.total_tiles;
    a1.P = pl.P; a1.ci_blocks = pl.ci_blocks; a1.co_blocks = pl.co_blocks; a1.cin_pad = pl.cin_pad; a1.cout_pad = pl.cout_pad;
    a1.ws = (float*)ws;
    static bool attr1 = false;
    if (!attr1) {
      cudaFuncSetAttribute(k_wgrad_tc1c, cudaFuncAttributeMaxDynamicSharedMemorySize, WT_SMEM_MAX);
      attr1 = true;
    }
    const int smem1 = 1024 + WT_SMEM_HDR + a1.nstages * W1_STAGE;
    dim3 grid1(pl.P, pl.ci_blocks * pl.co_blocks);
    k_wgrad_tc1c<<<grid1, WT_THREADS, smem1, stream>>>(tX, tD, a1);
    int rc1 = ffsr_check_launch("conv2d_wgrad_tc1c");
    if (rc1) return rc1;
    return wgrad_tc_finish(p, pl, 9, ws, stream);
  }
  CUtensorMap tmX, tmD;
  {
    cuuint64_t dims[4] = {(cuuint64_t)p.Cin, (cuuint64_t)p.W, (cuuint64_t)p.H, (cuuint64_t)p.N};
    cuuint64_t strides[3] = {(cuuint64_t)p.x_sX * 2, (cuuint64_t)p.x_sY * 2, (cuuint64_t)p.x_sN * 2};
    cuuint32_t box[4] = {64, WT_TW, (cuuint32_t)(WT_TH + 2 * pad), 1};
    cuuint32_t es[4] = {1, 1, 1, 1};
    CUresult r = enc(&tmX, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(p.x), dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    FFSR_REQUIRE(r == CUDA_SUCCESS, FFSR_ERR_DRIVER, "conv2d_wgrad_tc: x tensor map encode failed (CUresult %d)", (int)r);
  }
  {
    cuuint64_t dims[4] = {(cuuint64_t)p.Cout, (cuuint64_t)p.W, (cuuint64_t)p.H, (cuuint64_t)p.N};
    cuuint64_t strides[3] = {(cuuint64_t)p.dy_sX * 2, (cuuint64_t)p.dy_sY * 2, (cuuint64_t)p.dy_sN * 2};
    cuuint32_t box[4] = {64, WT_TW, WT_TH, 1};
    cuuint32_t es[4] = {1, 1, 1, 1};
    CUresult r = enc(&tmD, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(p.dy), dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    FFSR_REQUIRE(r == CUDA_SUCCESS, FFSR_ERR_DRIVER, "conv2d_wgrad_tc: dy tensor map encode failed (CUresult %d)", (int)r);
  }
  WgArgs a;
  a.N = p.N; a.H = p.H; a.W = p.W; a.Cin = p.Cin; a.Cout = p.Cout; a.ks = p.ksize;
  a.nblk = pl.nblk;
  a.a_bytes = (WT_TH + 2 * pad) * WT_ROW_BYTES;
  a.stage_bytes = 2 * a.a_bytes + 2 * WT_B_BYTES;
  a.nstages = (WT_SMEM_MAX - 1024 - WT_SMEM_HDR) / a.stage_bytes;
  if (a.nstages > WT_MAX_STAGES) a.nstages = WT_MAX_STAGES;
  a.tiles_x = pl.tiles_x; a.tiles_y = pl.tiles_y; a.total_tiles = pl.total_tiles;
  a.P = pl.P; a.ci_blocks = pl.ci_blocks; a.co_blocks = pl.co_blocks; a.cin_pad = pl.cin_pad; a.cout_pad = pl.cout_pad;
  a.ws = (float*)ws;
  // 64-channel blocks that hold any real channel (the rest of the 128 x nblk MMA reads zero-filled / stale rows
  // whose results are never stored)
  const int smem_bytes = 1024 + WT_SMEM_HDR + a.nstages * a.stage_bytes;
  static bool attr = false;
  if (!attr) {
    cudaFuncSetAttribute(k_wgrad_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, WT_SMEM_MAX);
    attr = true;
  }
  // a_chunks / b_chunks are per launch maxima; blocks past the tensor extent are zero-filled by TMA
  a.a_chunks = p.Cin > 64 ? 2 : 1;
  a.b_chunks = pl.nblk / 64;
  dim3 grid(pl.P * p.ksize, pl.ci_blocks * pl.co_blocks);
  k_wgrad_tc<<<grid, WT_THREADS, smem_bytes, stream>>>(tmX, tmD, a);
  int rc = ffsr_check_launch("conv2d_wgrad_tc");
  if (rc) return rc;
  return wgrad_tc_finish(p, pl, p.ksize * p.ksize, ws, stream);
}
