// tcgen05 implicit-GEMM convolution (1x1 / 3x3, zero pad, stride 1), bf16 operands, fp32
// accumulation in TMEM.  This is the tensor-core path of ffsr_conv2d for the contraction-heavy
// layers (SURVEY 2.3 K4/K5/K7/K8: refinement stack, hierarchical fusion, token GEMMs).
//
//   GEMM view : D[pixel, cout] = sum_{tap, cin} A[pixel shifted by tap, cin] * W[tap, cout, cin]
//   tile      : M = 128 output pixels (8 rows x 16 cols of one image), N = up to 128 cout
//   A operand : per (64-channel chunk, dx) ONE TMA tiled load of a row-haloed copy of the tile
//               from the NHWC bf16 activation tensor: 4-D tensor map {C, W, H, N}, box
//               {64, 16, 8+2*pad, 1}, SWIZZLE_128B, at (x0+dx-pad, y0-pad).  An image row of the
//               box is 16 px x 128 B = two 1024-byte swizzle atoms, so the operand of tap (dy,dx)
//               is the same copy at byte offset dy*2048: three loads serve nine taps and every
//               descriptor stays 1024-byte aligned.  Out-of-image coordinates (the conv halo) and
//               channels >= Cin are zero-filled by the TMA unit: padding costs no instructions.
//   B operand : weights pre-packed [group][dy][dx][CoutPad][CinPad] bf16 (K-major); one 5-D TMA
//               load {64, N, 1, ks, 1} brings the ks taps (all dy) of this dx.  When the whole
//               weight set of a cout block fits beside >= 3 A stages (every layer except
//               128->128 3x3) it is loaded ONCE per CTA and stays resident: the per-tile TMA
//               work (the measured limiter: ~4 cycles per 128-byte row per SM) is then A only.
//   MMA       : tcgen05.mma.cta_group::1.kind::f16, M=128, N=nblk, K=16, issued by one thread;
//               accumulators double-buffered in TMEM (2 x 128 columns) so the epilogue of
//               tile i overlaps the MMAs of tile i+1.
//   warps     : 0 = TMA producer, 1..3 = MMA issuers (warp 1 also allocates TMEM), 4..19 = epilogue: warp w reads
//               TMEM lane quarter w%4 (hardware rule) and the 16-column chunks (w-2)/4, +4, ...;
//               tcgen05.ld 32x32b -> bias/act/residual -> 16-byte vector stores.  16 warps keep
//               all four SM sub-partitions busy with the GELU math so that the epilogue of a
//               tile (~2k issue cycles) hides under the MMAs of the next one.
// Persistent: grid = min(tiles, #SMs), static round-robin over tiles.
//
// Four tile geometries, chosen per layer in ffsr_conv2d_tc:
//   g0   : the 8x16-pixel tile described above (1x1 layers; 3x3 layers only as a fallback);
//   g0x2 : 16x16-pixel tiles = two M=128 MMAs per (tap, K-step) that share every STREAMED weight stage (3x3 layers whose
//          nine-tap weight set does not fit beside the A stages, when g3 cannot take them);
//   g1   : 16x8-pixel tiles fed by ONE haloed copy {64 ch, 10 px, 18 rows} per 64-channel chunk -- every other 3x3
//          layer.  Measured: the 128-byte swizzle of tcgen05 shared-memory operands is a function of the ABSOLUTE
//          shared-memory address, so the operand of tap (dy, dx) is the same copy at byte offset dy*1280 + dx*128
//          (SBO = 1280, base offset 0).  These layers were bound by the L2 -> shared-memory traffic of three haloed
//          copies per tile, not by the tensor pipe.
//   g3   : SWAPPED operands for the streamed-weight 3x3 layers with bf16 inference outputs (128->128 refinement convs):
//          D[cout, pixel], the weights are the M=128 operand (single-tap 16 KB stages in a ring of 8) and an 8 px x 32 row
//          tile is the N=256 operand, fed by one haloed copy {64 ch, 10 px, 34 rows} per K chunk (ring of 2) with the
//          g1 tap offsets.  One M128 x N256 x K16 MMA reads 12 KB of shared memory per 128 cycles where the two
//          M128 x N128 MMAs of g0x2 read 16 KB: the refinement layers were bound by shared-memory operand bandwidth.
//          The transposing epilogue (swapped_epilogue) has one output channel per thread.
// Epilogue extras for the training graph: an optional bf16 copy of the pre-activation (out2) and FFSR_EPI_ACTGRAD
// (input gradient multiplied by act'(saved pre-activation of the previous layer)).
#include <cuda.h>
#include <stdio.h>
#include <stdlib.h>
#include "common.cuh"
#include "../../include/ffsr_b200.h"

namespace {

constexpr int TC_TH = 8, TC_TW = 16;           // output pixel tile (M = 128)
constexpr int TC_MAX_STAGES = 8;
constexpr int TC_ROW_BYTES = TC_TW * 128;      // one image row of the tile: 16 px x 64 bf16
constexpr int TC_SMEM_MAX = 232448;            // 227 KB opt-in limit per CTA
constexpr int TC_SMEM_HDR = 5120;              // barriers + TMEM slot (first 1 KB) + staged bias (1024 floats)
constexpr int TC_BIAS_OFF = 1024;              // byte offset of the staged bias inside the header
constexpr int TC_BIAS_MAX = 1024;              // output columns whose bias is staged (lean epilogue)
constexpr int TC_EPI_WARPS = 16;              // 4 per TMEM lane quarter: each owns a 16-column slice
constexpr int TC_MMA_WARPS = 3;               // warps 1..3 can issue MMAs (TcArgs.nmma of them do; see the MMA issuers).  20 warps = 5
                                              // per SM sub-partition keep the 96-register budget; a 21st would cut it to 80
constexpr int TC_EPI_WARP0 = 1 + TC_MMA_WARPS; // first epilogue warp
constexpr int TC_THREADS = 32 * (TC_EPI_WARP0 + TC_EPI_WARPS);
constexpr int TC_TMEM_COLS = 512;             // whole TMEM: ring of 512/slot accumulators (1 CTA per SM)
constexpr int TC_MAX_ACC = 12;
constexpr int TC_MAX_ASLOTS = 2;              // geom 3: activation ring depth

struct TcArgs {
  int N, H, W, Cin, Cout, taps, ks;
  int nblk;          // UMMA N (multiple of 16, <= 128)
  int n_nblocks;     // cout blocks
  int nchunks;       // 64-channel K chunks
  int ksteps_last;   // K=16 steps issued for the last chunk
  int a_bytes, b_bytes, stage_bytes, nstages;
  int acc_slot, nacc; // TMEM columns per accumulator (32/64/128) and ring depth
  int b_resident;     // weights of one (group, cout block) stay in smem across tiles
  int bres_bytes;     // bytes of that resident set (0 when streaming)
  int groups;
  int tiles_x, tiles_y;
  long long total_tiles;
  void* out;
  long long out_sN, out_sY, out_sX;
  int out_bf16;
  const float* bias;
  int act, epi;
  const void* r1;
  long long r1_sN, r1_sY, r1_sX;
  int r1_bf16;
  const void* r2;
  long long r2_sN, r2_sY, r2_sX;
  int r2_bf16;
  float sa, sb;
  const float* sa_ptr;
  const float* sb_ptr;
  const float* ch_k;
  const float* ch_d;
  void* out2;        // optional bf16 pre-activation copy (same strides as out)
  int halves;        // 1: tile = 8x16 px (M=128); 2: tile = 16x16 px as two M=128 MMAs sharing every weight stage
  int acc_half;      // TMEM columns of one half accumulator (acc_slot = halves * acc_half)
  int geom;          // 0: 8x16-px tile rows, one haloed A copy per dx;  1: 16x8-px tiles, ONE haloed copy per K chunk;
                     // 3: swapped operands (weights = M, 8x32-px tile = N = 256): ONE haloed copy {64 ch, 10 px, 34 rows} per
                     //    K chunk in its own ring + a ring of single-tap weight stages (see the kernel)
  int tile_h;        // output rows per tile (8 * halves, 16 for geom 1, 32 for geom 3)
  uint32_t a_step16; // geom 1: dy stride inside the haloed copy, in 16-byte units (10 px * 128 B)
  uint32_t a_desc_hi;// geom 1: A descriptor high word (SBO = haloed image-row pitch)
  int gelu_tanh;     // tanh-form GELU for bf16 outputs of inference launches (see gelu_tanh_fast)
  int epi_own;       // 1: epilogue warp group g owns every 4th tile of the CTA (all its column chunks); 0: chunks of every
                     //    tile are spread over the four groups.  See epilogue_loop.
  int lean;          // 1: lean_epilogue (bf16 inference outputs, bias staged in shared memory); see there
  int nmma;          // MMA-issuing warps (1, 2 or 3): warp 1+g issues the MMAs of tiles g, g+nmma, ... of this CTA
  int nb_fast;       // 1: the cout block varies FASTEST in the tile walk (multi-block 1x1 layers with streamed weights): the CTAs
                     //    of a wave then work on the same few pixel tiles, whose activations stay in L2 across the cout blocks
  int a_slot;        // geom 3: bytes of one slot of the activation ring (haloed copy rounded up to 1 KB)
  int na_slots;      // geom 3: slots of the activation ring (the weight ring has nstages slots of stage_bytes)
};

// ---------------------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
// "_e" variants: executed by a whole converged warp, one elected lane acts (see umma_bf16)
__device__ __forceinline__ void mbar_expect_tx_e(uint64_t* bar, uint32_t bytes) {
  asm volatile(
      "{\n\t"
      ".reg .pred e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "@e mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n\t"
      "}" ::"r"(smem_u32(bar)), "r"(bytes)
      : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra WAIT_DONE;\n\t"
      "bra WAIT_LOOP;\n\t"
      "WAIT_DONE:\n\t"
      "}" ::"r"(smem_u32(bar)), "r"(parity)
      : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tma_load_4d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2,
                                            int c3) {
  asm volatile(
      "{\n\t"
      ".reg .pred e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "@e cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];\n\t"
      "}" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_5d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2,
                                            int c3, int c4) {
  asm volatile(
      "{\n\t"
      ".reg .pred e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "@e cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];\n\t"
      "}" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

// K-major, SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor layout):
// start>>4 [0,14) | LBO>>4 [16,30) (unused for swizzled K-major: 1) | SBO>>4 [32,46) = 1024B
// (8 rows x 128B atom) | version=1 [46,48) | layout_type=2 (SWIZZLE_128B) [61,64);
// see desc_lo() / TC_DESC_HI below.

// Issued by the whole (converged) MMA warp: elect.sync picks one lane inside the asm block, so
// there is no divergent branch around the tensor-core instruction (a divergent guard makes the
// compiler wrap every UTCHMMA in an ELECT / R2UR.BROADCAST / BRA.U.ANY loop, and the single
// issuing thread -- not the tensor pipe -- becomes the limiter).  The two 64-bit shared-memory
// descriptors are assembled from 32-bit halves in PTX: the high half (SBO, version, swizzle)
// is a constant, only the 14-bit start address in the low half moves.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint32_t a_lo, uint32_t b_lo, uint32_t desc_hi, uint32_t idesc,
                                          uint32_t accum) {
  asm volatile(
      "{\n\t"
      ".reg .pred p, e;\n\t"
      ".reg .b64 da, db;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "mov.b64 da, {%1, %5};\n\t"
      "mov.b64 db, {%2, %5};\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "@e tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(accum), "r"(desc_hi)
      : "memory");
}
// Four K=16 steps of one (tap, 64-channel chunk) in ONE asm block: the descriptor increments
// (+32 B = +2 in 16-byte units) are done in PTX so that the operands cross to the uniform
// datapath once per block instead of once per MMA.
__device__ __forceinline__ void umma_bf16_x4(uint32_t tmem_d, uint32_t a_lo, uint32_t b_lo, uint32_t desc_hi, uint32_t idesc,
                                             uint32_t accum_first) {
  asm volatile(
      "{\n\t"
      ".reg .pred p, e, t;\n\t"
      ".reg .b64 da, db;\n\t"
      ".reg .b32 al, bl;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "setp.eq.b32 t, 0, 0;\n\t"
      "mov.b64 da, {%1, %5};\n\t"
      "mov.b64 db, {%2, %5};\n\t"
      "@e tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, p;\n\t"
      "add.u32 al, %1, 2;\n\t"
      "add.u32 bl, %2, 2;\n\t"
      "mov.b64 da, {al, %5};\n\t"
      "mov.b64 db, {bl, %5};\n\t"
      "@e tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, t;\n\t"
      "add.u32 al, %1, 4;\n\t"
      "add.u32 bl, %2, 4;\n\t"
      "mov.b64 da, {al, %5};\n\t"
      "mov.b64 db, {bl, %5};\n\t"
      "@e tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, t;\n\t"
      "add.u32 al, %1, 6;\n\t"
      "add.u32 bl, %2, 6;\n\t"
      "mov.b64 da, {al, %5};\n\t"
      "mov.b64 db, {bl, %5};\n\t"
      "@e tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, t;\n\t"
      "}" ::"r"(tmem_d),
      "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(accum_first), "r"(desc_hi)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile(
      "{\n\t"
      ".reg .pred e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t"
      "}" ::"r"(smem_u32(bar))
      : "memory");
}
#include "umma_blocks.inc"
constexpr uint32_t TC_DESC_HI = (1024u >> 4) | (1u << 14) | (2u << 29);   // SBO=1024B | version 1 | SWIZZLE_128B
__device__ __forceinline__ uint32_t desc_lo(uint32_t smem_addr) { return ((smem_addr & 0x3FFFFu) >> 4) | (1u << 16); }
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr));
}
// The wait names the loaded registers as in/out operands so that no use of them can be
// scheduled above it.
__device__ __forceinline__ void tmem_wait_ld(uint32_t (&v)[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]), "+r"(v[8]),
                 "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15])
               :
               : "memory");
}

// erf by Abramowitz-Stegun 7.1.26 (|abs err| <= 1.5e-7) on the fast-math units: the operands
// are bf16 here, so this is far inside the rounding noise and ~2x cheaper than erff().
__device__ __forceinline__ float gelu_fast(float x) {
  const float z = fabsf(x) * 0.70710678118654752440f;
  const float t = __fdividef(1.0f, fmaf(0.3275911f, z, 1.0f));
  float poly = fmaf(1.061405429f, t, -1.453152027f);
  poly = fmaf(poly, t, 1.421413741f);
  poly = fmaf(poly, t, -0.284496736f);
  poly = fmaf(poly, t, 0.254829592f);
  const float erf_abs = 1.0f - poly * t * __expf(-z * z);
  return 0.5f * x * (1.0f + copysignf(erf_abs, x));
}

// GELU through tanh.approx (6 instructions, 1 MUFU instead of ~21 / 2).  |error| <= 4.8e-4 absolute against the erf
// form (plus 2^-11 relative from the MUFU): below the bf16 rounding of the stored activation for positive inputs, a few
// bf16 ulps of the (|y| < 0.17) negative ones.  Used for INFERENCE launches with bf16 outputs only -- the path whose
// contract is |dPSNR| <= 0.01 dB, tested with it on; training launches (out2 != NULL: the backward pass differentiates
// the erf form) and every fp32 path keep the erf form.  FFSR_TC_GELU_ERF=1 forces the erf form everywhere.
// Measured on the C3 forward: 16.24 -> 15.52 ms; refine 128->128 layer 0.797 -> 0.868 of the sustained tensor peak
// (the epilogue's instructions compete with the MMA-issuing warp for the same schedulers).
__device__ __forceinline__ float gelu_tanh_fast(float x) {
  const float u = x * fmaf(0.0356774081f, x * x, 0.7978845608f);
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(u));
  const float hx = 0.5f * x;
  return fmaf(hx, t, hx);
}

enum { EM_NONE = 0, EM_GELU = 1, EM_RELU = 2, EM_SIGMOID = 3, EM_RESIDUAL = 4, EM_LKAGATE = 5, EM_ACTGRAD = 6 };

// d/dz of the activations (z = saved pre-activation); GELU' = Phi(z) + z phi(z) with the same fast erf
__device__ __forceinline__ float act_grad_fast(float z, int act) {
  if (act == ACT_GELU) {
    const float u = fabsf(z) * 0.70710678118654752440f;
    const float t = __fdividef(1.0f, fmaf(0.3275911f, u, 1.0f));
    float poly = fmaf(1.061405429f, t, -1.453152027f);
    poly = fmaf(poly, t, 1.421413741f);
    poly = fmaf(poly, t, -0.284496736f);
    poly = fmaf(poly, t, 0.254829592f);
    const float e = __expf(-u * u);
    const float erf_abs = 1.0f - poly * t * e;
    const float cdf = 0.5f * (1.0f + copysignf(erf_abs, z));
    return fmaf(z * 0.39894228040143267794f, e, cdf);
  }
  if (act == ACT_RELU) return z > 0.f ? 1.f : 0.f;
  if (act == ACT_SIGMOID) { const float sg = sigmoid_acc(z); return sg * (1.f - sg); }
  return 1.f;
}

// 16 consecutive residual channels -> fp32 registers; 16-byte vector loads when aligned.
__device__ __forceinline__ void load_res16(const void* base, int is_bf16, long long off, int nvalid, float (&o)[16]) {
  if (is_bf16) {
    const __nv_bfloat16* p = reinterpret_cast<const __nv_bfloat16*>(base) + off;
    if (nvalid == 16 && (reinterpret_cast<uintptr_t>(p) & 15) == 0) {
      const uint4 u0 = __ldg(reinterpret_cast<const uint4*>(p)), u1 = __ldg(reinterpret_cast<const uint4*>(p) + 1);
      const uint32_t w[8] = {u0.x, u0.y, u0.z, u0.w, u1.x, u1.y, u1.z, u1.w};
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const float2 f2 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w[k]));
        o[2 * k] = f2.x; o[2 * k + 1] = f2.y;
      }
    } else {
#pragma unroll
      for (int k = 0; k < 16; ++k) o[k] = k < nvalid ? __bfloat162float(p[k]) : 0.f;
    }
  } else {
    const float* p = reinterpret_cast<const float*>(base) + off;
    if (nvalid == 16 && (reinterpret_cast<uintptr_t>(p) & 15) == 0) {
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(p) + k);
        o[4 * k] = v.x; o[4 * k + 1] = v.y; o[4 * k + 2] = v.z; o[4 * k + 3] = v.w;
      }
    } else {
#pragma unroll
      for (int k = 0; k < 16; ++k) o[k] = k < nvalid ? p[k] : 0.f;
    }
  }
}

__device__ __forceinline__ float load_res(const void* base, int is_bf16, long long off) {
  return is_bf16 ? __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(base)[off])
                 : reinterpret_cast<const float*>(base)[off];
}

// Static round-robin tile walk without per-tile divisions: (tx, ty, n, nb) advance by the
// decomposed grid stride with carries.  The issuing threads of the producer and MMA warps are
// instruction-bound on small layers, so every instruction in their per-tile path counts.
struct TileIter {
  int tx, ty, n, nb;
  int dtx, dty, dn, dnb;
  long long t;
  __device__ __forceinline__ void init(const TcArgs& a) {
    unsigned r = blockIdx.x;
    unsigned d = gridDim.x;
    t = blockIdx.x;
    if (a.nb_fast) {
      nb = r % a.n_nblocks; r /= a.n_nblocks;
      tx = r % a.tiles_x; r /= a.tiles_x;
      ty = r % a.tiles_y; n = r / a.tiles_y;
      dnb = d % a.n_nblocks; d /= a.n_nblocks;
      dtx = d % a.tiles_x; d /= a.tiles_x;
      dty = d % a.tiles_y; dn = d / a.tiles_y;
      return;
    }
    tx = r % a.tiles_x; r /= a.tiles_x;
    ty = r % a.tiles_y; r /= a.tiles_y;
    n = r % a.N; nb = r / a.N;
    dtx = d % a.tiles_x; d /= a.tiles_x;
    dty = d % a.tiles_y; d /= a.tiles_y;
    dn = d % a.N; dnb = d / a.N;
  }
  __device__ __forceinline__ bool valid(const TcArgs& a) const { return t < a.total_tiles; }
  __device__ __forceinline__ void next(const TcArgs& a) {
    t += gridDim.x;
    if (a.nb_fast) {
      nb += dnb;
      int c = 0;
      if (nb >= a.n_nblocks) { nb -= a.n_nblocks; c = 1; }
      tx += dtx + c; c = 0;
      if (tx >= a.tiles_x) { tx -= a.tiles_x; c = 1; }
      ty += dty + c; c = 0;
      if (ty >= a.tiles_y) { ty -= a.tiles_y; c = 1; }
      n += dn + c;
      return;
    }
    tx += dtx;
    int c = 0;
    if (tx >= a.tiles_x) { tx -= a.tiles_x; c = 1; }
    ty += dty + c; c = 0;
    if (ty >= a.tiles_y) { ty -= a.tiles_y; c = 1; }
    n += dn + c; c = 0;
    if (n >= a.N) { n -= a.N; c = 1; }
    nb += dnb + c;
  }
};

// 16 fp32 -> 16 bf16 (two 16-byte stores) or 16 fp32 (four 16-byte stores); masked scalar tail
template <bool OUT_BF16>
__device__ __forceinline__ void store16_out(void* out, long long off, const float (&f)[16], int nvalid) {
  if (OUT_BF16) {
    __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(out) + off;
    if (nvalid == 16 && ((reinterpret_cast<uintptr_t>(o) & 15) == 0)) {
      uint32_t w[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        __nv_bfloat162 h = __floats2bfloat162_rn(f[2 * k], f[2 * k + 1]);
        w[k] = *reinterpret_cast<uint32_t*>(&h);
      }
      reinterpret_cast<uint4*>(o)[0] = make_uint4(w[0], w[1], w[2], w[3]);
      reinterpret_cast<uint4*>(o)[1] = make_uint4(w[4], w[5], w[6], w[7]);
    } else {
#pragma unroll
      for (int k = 0; k < 16; ++k)
        if (k < nvalid) o[k] = __float2bfloat16_rn(f[k]);
    }
  } else {
    float* o = reinterpret_cast<float*>(out) + off;
    if (nvalid == 16 && ((reinterpret_cast<uintptr_t>(o) & 15) == 0)) {
#pragma unroll
      for (int k = 0; k < 4; ++k) reinterpret_cast<float4*>(o)[k] = make_float4(f[4 * k], f[4 * k + 1], f[4 * k + 2], f[4 * k + 3]);
    } else {
#pragma unroll
      for (int k = 0; k < 16; ++k)
        if (k < nvalid) o[k] = f[k];
    }
  }
}

// Epilogue of one warp: TMEM lane quarter `warp & 3`, warp group (warp-2)>>2.  Chunk c (16
// accumulator columns) of the q-th tile of this CTA belongs to warp group (q*nch + c) & 3, so
// layers with fewer than four chunks per tile still spread over all 16 warps.
template <int MODE, bool OUT_BF16>
__device__ __forceinline__ void epilogue_loop(const TcArgs& a, uint64_t* tfull, uint64_t* tempty, uint32_t tmem_base,
                                              int warp, int lane) {
  const int wq = warp & 3;
  const int cgp = (warp - TC_EPI_WARP0) >> 2;
  const int row = wq * 32 + lane;                       // pixel within the tile (accumulator row)
  const int tw = a.geom ? 8 : TC_TW;
  const int py = row / tw, px = row % tw;
  const int nch = a.nblk >> 4;
  const int Cout = a.Cout, nblk = a.nblk, nacc = a.nacc, acc_slot = a.acc_slot;
  const float* __restrict__ bias = a.bias;
  float sa = 1.f, sb = 1.f;
  if (MODE == EM_RESIDUAL || MODE == EM_LKAGATE) {
    sa = a.sa * (a.sa_ptr ? a.sa_ptr[0] : 1.0f);
    sb = a.sb * (a.sb_ptr ? a.sb_ptr[0] : 1.0f);
  }
  // Small-N layers (<= 64 output columns per tile) are bound by the instructions of this loop, and with the chunk
  // split every one of the 16 warps pays the per-tile bookkeeping (iterator, barrier wait / arrive, addresses) for 1-2
  // useful chunks (measured on a 32->32 layer: 46 instructions per output, 72 % issue utilisation).  With `own` a
  // warp group takes whole tiles (tile q of this CTA belongs to group q & 3) and skips the others for ~15 instructions.
  const bool own = a.epi_own != 0;
  int as = 0, item0 = 0, q = 0;
  uint32_t aph = 0;
  TileIter ti;
  for (ti.init(a); ti.valid(a); ti.next(a), item0 = (item0 + nch) & 3, ++q) {
    if (own && (q & 3) != cgp) {
      if (++as == nacc) { as = 0; aph ^= 1; }
      continue;
    }
    const int n = ti.n;
    const int g = a.groups > 1 ? n % a.groups : 0;
    bool waited = false;
    for (int half = 0; half < a.halves; ++half, item0 = (item0 + (half < a.halves ? nch : 0)) & 3) {
    const int y = ti.ty * a.tile_h + half * TC_TH + py, x = ti.tx * tw + px;
    const bool inside = (y < a.H) && (x < a.W);
    const long long opix = (long long)n * a.out_sN + (long long)y * a.out_sY + (long long)x * a.out_sX;
    long long r1pix = 0, r2pix = 0;
    if (MODE == EM_RESIDUAL || MODE == EM_LKAGATE || MODE == EM_ACTGRAD) r1pix = (long long)n * a.r1_sN + (long long)y * a.r1_sY + (long long)x * a.r1_sX;
    if (MODE == EM_RESIDUAL) r2pix = (long long)n * a.r2_sN + (long long)y * a.r2_sY + (long long)x * a.r2_sX;
    uint32_t taddr = tmem_base + ((uint32_t)(wq * 32) << 16) + (uint32_t)(as * acc_slot + half * a.acc_half);
    for (int c = own ? 0 : ((cgp - item0) & 3); c < nch; c += own ? 1 : 4) {
      const int ocb = ti.nb * nblk + c * 16;
      const int nvalid = min(16, Cout - ocb);            // may be <= 0 for padded columns
      float f[16];
      // operands that do not depend on the accumulator are fetched before waiting for it
      if (bias != nullptr && nvalid > 0) {
        const float* bp = bias + (long long)g * Cout + ocb;
        if (nvalid == 16 && ((reinterpret_cast<uintptr_t>(bp) & 15) == 0)) {
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const float4 v4 = __ldg(reinterpret_cast<const float4*>(bp) + k);
            f[4 * k] = v4.x; f[4 * k + 1] = v4.y; f[4 * k + 2] = v4.z; f[4 * k + 3] = v4.w;
          }
        } else {
#pragma unroll
          for (int k = 0; k < 16; ++k) f[k] = (k < nvalid) ? __ldg(bp + k) : 0.f;
        }
      } else {
#pragma unroll
        for (int k = 0; k < 16; ++k) f[k] = 0.f;
      }
      float r1v[(MODE == EM_RESIDUAL || MODE == EM_LKAGATE || MODE == EM_ACTGRAD) ? 16 : 1];
      float r2v[MODE == EM_RESIDUAL ? 16 : 1];
      const bool has_r2 = MODE == EM_RESIDUAL && a.r2 != nullptr;
      if (MODE == EM_RESIDUAL || MODE == EM_LKAGATE || MODE == EM_ACTGRAD) {
        if (inside && nvalid > 0) load_res16(a.r1, a.r1_bf16, r1pix + ocb, nvalid, reinterpret_cast<float(&)[16]>(r1v));
      }
      if (MODE == EM_RESIDUAL) {
        if (inside && has_r2 && nvalid > 0) load_res16(a.r2, a.r2_bf16, r2pix + ocb, nvalid, reinterpret_cast<float(&)[16]>(r2v));
      }
      if (!waited) {
        mbar_wait(&tfull[as], aph);
        tc_fence_after();
        waited = true;
      }
      uint32_t v[16];
      tmem_ld16(taddr + (uint32_t)(c * 16), v);
      tmem_wait_ld(v);
      if (inside && nvalid > 0) {
#pragma unroll
        for (int k = 0; k < 16; ++k) f[k] += __uint_as_float(v[k]);
        if ((MODE == EM_GELU || MODE == EM_RELU || MODE == EM_SIGMOID) && a.out2 != nullptr)
          store16_out<true>(a.out2, opix + ocb, f, nvalid);          // pre-activation, kept for the backward pass
        if (MODE == EM_ACTGRAD) {
#pragma unroll
          for (int k = 0; k < 16; ++k) f[k] *= act_grad_fast(r1v[k % (sizeof(r1v) / 4)], a.act);
        } else if (MODE == EM_GELU) {
          if (OUT_BF16 && a.gelu_tanh) {
#pragma unroll
            for (int k = 0; k < 16; ++k) f[k] = gelu_tanh_fast(f[k]);
          } else {
#pragma unroll
            for (int k = 0; k < 16; ++k) f[k] = gelu_fast(f[k]);
          }
        } else if (MODE == EM_RELU) {
#pragma unroll
          for (int k = 0; k < 16; ++k) f[k] = fmaxf(f[k], 0.f);
        } else if (MODE == EM_SIGMOID) {
#pragma unroll
          for (int k = 0; k < 16; ++k) f[k] = sigmoid_acc(f[k]);
        } else if (MODE == EM_RESIDUAL) {
          if (a.act != ACT_NONE) {
#pragma unroll
            for (int k = 0; k < 16; ++k) f[k] = apply_act(f[k], a.act);
          }
#pragma unroll
          for (int k = 0; k < 16; ++k) f[k] = fmaf(sa, f[k], r1v[k % (sizeof(r1v) / 4)]);
          if (has_r2) {
#pragma unroll
            for (int k = 0; k < 16; ++k) f[k] = fmaf(sb, r2v[k % (sizeof(r2v) / 4)], f[k]);
          }
        } else if (MODE == EM_LKAGATE) {
#pragma unroll
          for (int k = 0; k < 16; ++k) {
            if (k < nvalid) {
              const float xr = r1v[k % (sizeof(r1v) / 4)];
              f[k] = xr + sa * (fmaf(xr, __ldg(a.ch_k + ocb + k), __ldg(a.ch_d + ocb + k)) * sigmoid_acc(f[k]));
            }
          }
        }
        store16_out<OUT_BF16>(a.out, opix + ocb, f, nvalid);
      }
    }
    }   // halves
    if (!waited) mbar_wait(&tfull[as], aph);          // warps without a column chunk still pace the ring
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(&tempty[as]);
    if (++as == nacc) { as = 0; aph ^= 1; }
  }
}


// ---------------------------------------------------------------------------- lean epilogue
// The generic epilogue_loop above spends most of its instructions on bookkeeping (round-1 ncu of a 32->32 layer:
// 46 executed instructions per output value, 72 % of the issue slots, 14 % tensor pipe): per 16-column chunk it
// recomputes three 64-bit pixel addresses, tests pointer alignment, fetches the bias from global memory and waits
// for its own TMEM load.  lean_epilogue serves the launches that dominate an inference forward -- bf16 outputs,
// Cout a multiple of 8, 16-byte aligned rows, one cout block, plain / activation / residual modes:
//   * the bias is staged once per CTA in shared memory (float4 broadcast reads);
//   * pixel addresses are computed once per tile (half);
//   * two chunks (32 accumulator columns) are fetched with back-to-back tcgen05.ld and one wait (four would spill: the
//     576-thread CTA caps a thread at 96 registers);
//   * the accumulator is handed back to the MMA warp as soon as the last tcgen05.ld of the tile has completed, before
//     the activation math and the stores;
//   * `own` layers (N <= 128 single-half tiles, >= 4 accumulators in flight): warp group g takes every 4th tile whole;
//     split layers (two-half 128-column tiles): warp group g takes columns [32 g, 32 g + 32) of both halves.
template <int MODE, bool TANH>
__device__ __forceinline__ void lean_chunk(const uint32_t (&v)[16], const float* __restrict__ sb16, __nv_bfloat16* __restrict__ o,
                                           int nv8, const TcArgs& a, long long r1off, long long r2off, float sa, float sb,
                                           bool has_r2) {
  float f[16];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const float4 b4 = *reinterpret_cast<const float4*>(sb16 + 4 * k);
    f[4 * k] = __uint_as_float(v[4 * k]) + b4.x;
    f[4 * k + 1] = __uint_as_float(v[4 * k + 1]) + b4.y;
    f[4 * k + 2] = __uint_as_float(v[4 * k + 2]) + b4.z;
    f[4 * k + 3] = __uint_as_float(v[4 * k + 3]) + b4.w;
  }
  if (MODE == EM_GELU) {
#pragma unroll
    for (int k = 0; k < 16; ++k) f[k] = TANH ? gelu_tanh_fast(f[k]) : gelu_fast(f[k]);
  } else if (MODE == EM_RELU) {
#pragma unroll
    for (int k = 0; k < 16; ++k) f[k] = fmaxf(f[k], 0.f);
  } else if (MODE == EM_SIGMOID) {
#pragma unroll
    for (int k = 0; k < 16; ++k) f[k] = sigmoid_acc(f[k]);
  } else if (MODE == EM_RESIDUAL) {
    float r[16];
    load_res16(a.r1, a.r1_bf16, r1off, nv8 * 8, r);
#pragma unroll
    for (int k = 0; k < 16; ++k) f[k] = fmaf(sa, f[k], r[k]);
    if (has_r2) {
      load_res16(a.r2, a.r2_bf16, r2off, nv8 * 8, r);
#pragma unroll
      for (int k = 0; k < 16; ++k) f[k] = fmaf(sb, r[k], f[k]);
    }
  }
  uint32_t w[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    __nv_bfloat162 h = __floats2bfloat162_rn(f[2 * k], f[2 * k + 1]);
    w[k] = *reinterpret_cast<uint32_t*>(&h);
  }
  reinterpret_cast<uint4*>(o)[0] = make_uint4(w[0], w[1], w[2], w[3]);
  if (nv8 > 1) reinterpret_cast<uint4*>(o)[1] = make_uint4(w[4], w[5], w[6], w[7]);
}

template <int MODE, bool TANH>
__device__ __forceinline__ void lean_epilogue(const TcArgs& a, uint64_t* tfull, uint64_t* tempty, uint32_t tmem_base, int warp,
                                              int lane, const float* __restrict__ sbias) {
  const int wq = warp & 3;
  const int cgp = (warp - TC_EPI_WARP0) >> 2;
  const int row = wq * 32 + lane;
  const int tw = a.geom ? 8 : TC_TW;
  const int py = row / tw, px = row % tw;
  const int nch = a.nblk >> 4;
  const int nv8_total = a.Cout >> 3;                   // Cout % 8 == 0 on this path
  const bool own = a.epi_own != 0;
  const int c_lo = own ? 0 : cgp * (nch >> 2);         // split mode: nch % 4 == 0
  const int c_hi = own ? nch : c_lo + (nch >> 2);
  const int nacc = a.nacc, halves = a.halves;
  float sa = 1.f, sb = 1.f;
  if (MODE == EM_RESIDUAL) {
    sa = a.sa * (a.sa_ptr ? a.sa_ptr[0] : 1.0f);
    sb = a.sb * (a.sb_ptr ? a.sb_ptr[0] : 1.0f);
  }
  const bool has_r2 = MODE == EM_RESIDUAL && a.r2 != nullptr;
  __nv_bfloat16* const outp = reinterpret_cast<__nv_bfloat16*>(a.out);
  int as = 0, q = 0;
  uint32_t aph = 0;
  TileIter ti;
  for (ti.init(a); ti.valid(a); ti.next(a), ++q) {
    if (own && (q & 3) != cgp) {
      if (++as == nacc) { as = 0; aph ^= 1; }
      continue;
    }
    const int n = ti.n;
    const int cb = ti.nb * a.nblk;                      // first output column of this cout block
    const int x0 = ti.tx * tw + px;
    if (MODE == EM_RESIDUAL) {
      // the residual rows of this thread's pixels are fetched towards L1 BEFORE the wait for the accumulator: their loads sat
      // behind the TMEM load in every chunk, and a residual layer cost twice its plain twin (stage3.r2 0.25 vs r0 0.11 ms)
      for (int half = 0; half < halves; ++half) {
        const int yy = ti.ty * a.tile_h + half * TC_TH + py;
        if (yy < a.H && x0 < a.W) {
          const long long e1 = (long long)n * a.r1_sN + (long long)yy * a.r1_sY + (long long)x0 * a.r1_sX + cb + c_lo * 16;
          const char* p1 = reinterpret_cast<const char*>(a.r1) + e1 * (a.r1_bf16 ? 2 : 4);
          const int bytes1 = (c_hi - c_lo) * 16 * (a.r1_bf16 ? 2 : 4);
          for (int o = 0; o < bytes1; o += 128) asm volatile("prefetch.global.L1 [%0];" ::"l"(p1 + o));
          if (has_r2) {
            const long long e2 = (long long)n * a.r2_sN + (long long)yy * a.r2_sY + (long long)x0 * a.r2_sX + cb + c_lo * 16;
            const char* p2 = reinterpret_cast<const char*>(a.r2) + e2 * (a.r2_bf16 ? 2 : 4);
            const int bytes2 = (c_hi - c_lo) * 16 * (a.r2_bf16 ? 2 : 4);
            for (int o = 0; o < bytes2; o += 128) asm volatile("prefetch.global.L1 [%0];" ::"l"(p2 + o));
          }
        }
      }
    }
    mbar_wait(&tfull[as], aph);
    tc_fence_after();
    for (int half = 0; half < halves; ++half) {
      const int y = ti.ty * a.tile_h + half * TC_TH + py;
      const bool inside = (y < a.H) && (x0 < a.W);
      const long long opix = (long long)n * a.out_sN + (long long)y * a.out_sY + (long long)x0 * a.out_sX + cb;
      long long r1pix = 0, r2pix = 0;
      if (MODE == EM_RESIDUAL) {
        r1pix = (long long)n * a.r1_sN + (long long)y * a.r1_sY + (long long)x0 * a.r1_sX + cb;
        if (has_r2) r2pix = (long long)n * a.r2_sN + (long long)y * a.r2_sY + (long long)x0 * a.r2_sX + cb;
      }
      const uint32_t taddr = tmem_base + ((uint32_t)(wq * 32) << 16) + (uint32_t)(as * a.acc_slot + half * a.acc_half);
      for (int c0 = c_lo; c0 < c_hi; c0 += 2) {
        const int nc = min(2, c_hi - c0);
        uint32_t v0[16], v1[16];
        tmem_ld16(taddr + (uint32_t)(c0 * 16), v0);
        if (nc > 1) tmem_ld16(taddr + (uint32_t)(c0 * 16 + 16), v1);
        tmem_wait_ld(v0);
        if (nc > 1) tmem_wait_ld(v1);
        if (half == halves - 1 && c0 + 2 >= c_hi) {      // every column of this tile is in registers: free the accumulator
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&tempty[as]);
        }
        if (inside) {
          const int col = cb + c0 * 16;                  // global output column of v0[0]
          const int g8 = nv8_total - (col >> 3);         // valid 8-column groups from here on
          if (g8 > 0) lean_chunk<MODE, TANH>(v0, sbias + col, outp + opix + c0 * 16, min(g8, 2), a, r1pix + c0 * 16, r2pix + c0 * 16, sa, sb, has_r2);
          if (nc > 1 && g8 > 2) lean_chunk<MODE, TANH>(v1, sbias + col + 16, outp + opix + c0 * 16 + 16, min(g8 - 2, 2), a, r1pix + c0 * 16 + 16, r2pix + c0 * 16 + 16, sa, sb, has_r2);
        }
      }
    }
    if (++as == nacc) { as = 0; aph ^= 1; }
  }
}

// ---------------------------------------------------------------------------- swapped epilogue (geom 3)
// The accumulator is D[cout, pixel]: TMEM lane = output channel, column j = pixel (row j / 8, column j % 8) of the 8x32 tile.
// Warp w reads lane quarter w % 4 (channels 32 (w%4) .. +31 of the cout block, one per thread, so the bias is one register)
// and column quarter (w - 4) / 4 (tile rows 8 q .. 8 q + 7).  After tcgen05.ld a thread holds one channel of consecutive
// pixels; one shfl.xor 1 per two values turns that into two adjacent channels of one pixel, so the 32 lanes of a warp store
// two pixels x 64 contiguous bytes per 4-byte store instruction.  Element math and bf16 rounding are those of lean_chunk.
template <int MODE, bool TANH>
__device__ __forceinline__ void swapped_rows2(const uint32_t (&v)[16], float bv, int odd, __nv_bfloat16* __restrict__ o,
                                              const TcArgs& a, long long r1off, long long r2off, int r0, int rows, int cols,
                                              bool cok, float sa, float sb, bool has_r2) {
  float f[16];
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    f[k] = __uint_as_float(v[k]) + bv;
    if (MODE == EM_GELU) f[k] = TANH ? gelu_tanh_fast(f[k]) : gelu_fast(f[k]);
    else if (MODE == EM_RELU) f[k] = fmaxf(f[k], 0.f);
    else if (MODE == EM_SIGMOID) f[k] = sigmoid_acc(f[k]);
  }
#pragma unroll
  for (int j = 0; j < 16; j += 2) {
    // columns j, j + 1: the even lane keeps pixel j, the odd lane pixel j + 1, each for channels (ce, ce + 1)
    const float recv = __shfl_xor_sync(0xffffffffu, odd ? f[j] : f[j + 1], 1);
    float lo = odd ? recv : f[j], hi = odd ? f[j + 1] : recv;
    const int r = r0 + (j >> 3), px = j & 7;
    if (cok && r < rows && px < cols) {
      const int oo = r * (int)a.out_sY + px * (int)a.out_sX;
      if (MODE == EM_RESIDUAL) {
        const int o1 = r * (int)a.r1_sY + px * (int)a.r1_sX;
        float2 r1;
        if (a.r1_bf16) r1 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(reinterpret_cast<const __nv_bfloat16*>(a.r1) + r1off + o1));
        else r1 = __ldg(reinterpret_cast<const float2*>(reinterpret_cast<const float*>(a.r1) + r1off + o1));
        lo = fmaf(sa, lo, r1.x);
        hi = fmaf(sa, hi, r1.y);
        if (has_r2) {
          const int o2 = r * (int)a.r2_sY + px * (int)a.r2_sX;
          float2 r2;
          if (a.r2_bf16) r2 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(reinterpret_cast<const __nv_bfloat16*>(a.r2) + r2off + o2));
          else r2 = __ldg(reinterpret_cast<const float2*>(reinterpret_cast<const float*>(a.r2) + r2off + o2));
          lo = fmaf(sb, r2.x, lo);
          hi = fmaf(sb, r2.y, hi);
        }
      }
      __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
      *reinterpret_cast<__nv_bfloat162*>(o + oo) = h;
    }
  }
}

template <int MODE, bool TANH>
__device__ __forceinline__ void swapped_epilogue(const TcArgs& a, uint64_t* tfull, uint64_t* tempty, uint32_t tmem_base, int warp,
                                                 int lane) {
  const int wq = warp & 3;
  const int cq = (warp - TC_EPI_WARP0) >> 2;
  const int odd = lane & 1;
  float sa = 1.f, sb = 1.f;
  if (MODE == EM_RESIDUAL) {
    sa = a.sa * (a.sa_ptr ? a.sa_ptr[0] : 1.0f);
    sb = a.sb * (a.sb_ptr ? a.sb_ptr[0] : 1.0f);
  }
  const bool has_r2 = MODE == EM_RESIDUAL && a.r2 != nullptr;
  __nv_bfloat16* const outp = reinterpret_cast<__nv_bfloat16*>(a.out);
  int as = 0;
  uint32_t aph = 0;
  TileIter ti;
  for (ti.init(a); ti.valid(a); ti.next(a)) {
    const int n = ti.n;
    const int co = ti.nb * 128 + wq * 32 + lane;       // this thread's accumulator lane
    const float bv = (a.bias != nullptr && co < a.Cout) ? __ldg(a.bias + co) : 0.f;
    const int ce = co - odd;                            // first of the two channels this thread stores (Cout is even)
    const bool cok = ce < a.Cout;
    const int y0 = ti.ty * 32 + cq * 8, x0 = ti.tx * 8 + odd;
    const int rows = a.H - y0, cols = a.W - x0;         // valid tile rows from y0 / stored columns px (+ odd) from x0
    const long long opix = (long long)n * a.out_sN + (long long)y0 * a.out_sY + (long long)x0 * a.out_sX + ce;
    long long r1pix = 0, r2pix = 0;
    if (MODE == EM_RESIDUAL) {
      r1pix = (long long)n * a.r1_sN + (long long)y0 * a.r1_sY + (long long)x0 * a.r1_sX + ce;
      if (has_r2) r2pix = (long long)n * a.r2_sN + (long long)y0 * a.r2_sY + (long long)x0 * a.r2_sX + ce;
      // the 64 pixels x 32 channels this warp adds are fetched towards L1 before the wait for the accumulator
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int p = lane + 32 * h, r = p >> 3, px = p & 7;
        if (r < rows && px < a.W - ti.tx * 8 && ti.nb * 128 + wq * 32 < a.Cout) {
          const long long e1 = (long long)n * a.r1_sN + (long long)(y0 + r) * a.r1_sY + (long long)(ti.tx * 8 + px) * a.r1_sX + ti.nb * 128 + wq * 32;
          asm volatile("prefetch.global.L1 [%0];" ::"l"(reinterpret_cast<const char*>(a.r1) + e1 * (a.r1_bf16 ? 2 : 4)));
          if (has_r2) {
            const long long e2 = (long long)n * a.r2_sN + (long long)(y0 + r) * a.r2_sY + (long long)(ti.tx * 8 + px) * a.r2_sX + ti.nb * 128 + wq * 32;
            asm volatile("prefetch.global.L1 [%0];" ::"l"(reinterpret_cast<const char*>(a.r2) + e2 * (a.r2_bf16 ? 2 : 4)));
          }
        }
      }
    }
    mbar_wait(&tfull[as], aph);
    tc_fence_after();
    const uint32_t taddr = tmem_base + ((uint32_t)(wq * 32) << 16) + (uint32_t)(as * a.acc_slot + cq * 64);
#pragma unroll 1
    for (int h = 0; h < 2; ++h) {                       // 32 columns = 4 tile rows per pass
      uint32_t v0[16], v1[16];
      tmem_ld16(taddr + (uint32_t)(h * 32), v0);
      tmem_ld16(taddr + (uint32_t)(h * 32 + 16), v1);
      tmem_wait_ld(v0);
      tmem_wait_ld(v1);
      if (h == 1) {                                     // every column of this warp is in registers: free the accumulator
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tempty[as]);
      }
      swapped_rows2<MODE, TANH>(v0, bv, odd, outp + opix, a, r1pix, r2pix, 4 * h, rows, cols, cok, sa, sb, has_r2);
      swapped_rows2<MODE, TANH>(v1, bv, odd, outp + opix, a, r1pix, r2pix, 4 * h + 2, rows, cols, cok, sa, sb, has_r2);
    }
    if (++as == a.nacc) { as = 0; aph ^= 1; }
  }
}

// ---------------------------------------------------------------------------- the kernel
__global__ void __launch_bounds__(TC_THREADS, 1)
k_conv_tc(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const TcArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem);
  uint64_t* full = bars;                           // [TC_MAX_STAGES]
  uint64_t* empty = bars + TC_MAX_STAGES;          // [TC_MAX_STAGES]
  uint64_t* tfull = bars + 2 * TC_MAX_STAGES;                  // [TC_MAX_ACC]
  uint64_t* tempty = bars + 2 * TC_MAX_STAGES + TC_MAX_ACC;    // [TC_MAX_ACC]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * TC_MAX_STAGES + 2 * TC_MAX_ACC);
  uint64_t* bfull = bars + 2 * TC_MAX_STAGES + 2 * TC_MAX_ACC + 1;   // resident-weights barrier
  uint64_t* afull = bfull + 1;                                       // geom 3: activation ring [TC_MAX_ASLOTS]
  uint64_t* aempty = afull + TC_MAX_ASLOTS;
  float* sbias = reinterpret_cast<float*>(smem + TC_BIAS_OFF);       // lean epilogue: bias of every output column
  uint8_t* bres = smem + TC_SMEM_HDR;                                // resident weights (may be empty)
  uint8_t* stages = bres + a.bres_bytes;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int i = 0; i < TC_MAX_STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    for (int i = 0; i < TC_MAX_ACC; ++i) { mbar_init(&tfull[i], 1); mbar_init(&tempty[i], a.epi_own ? 4 : TC_EPI_WARPS); }
    mbar_init(bfull, 1);
    for (int i = 0; i < TC_MAX_ASLOTS; ++i) { mbar_init(&afull[i], 1); mbar_init(&aempty[i], 1); }
    fence_barrier_init();
  }
  if (a.lean && threadIdx.x >= 32 * TC_EPI_WARP0) {
    const int ncols = a.n_nblocks * a.nblk;
    for (int c = threadIdx.x - 32 * TC_EPI_WARP0; c < ncols; c += TC_THREADS - 32 * TC_EPI_WARP0) sbias[c] = (a.bias != nullptr && c < a.Cout) ? a.bias[c] : 0.f;
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TC_TMEM_COLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int pad = a.ks / 2;
  const int kiters = a.geom ? a.nchunks : a.ks * a.nchunks;   // one pipeline stage per (chunk, dx) / per chunk (geom 1)
  const uint32_t stage_tx = (uint32_t)(a.a_bytes + (a.b_resident ? 0 : a.b_bytes));

  if (warp == 0) {
    // ================================ TMA producer (whole warp, converged) ===============
    {
      int s = 0;
      uint32_t ph = 0;
      int cur_g = -1, cur_nb = -1, last_s = 0;
      uint32_t last_ph = 0;
      bool have_last = false;
      int as_ = 0;                                   // geom 3: activation ring position
      uint32_t aph_ = 0;
      uint8_t* const wring = stages + a.na_slots * a.a_slot;
      TileIter ti;
      for (ti.init(a); ti.valid(a); ti.next(a)) {
        const int tx = ti.tx, ty = ti.ty, n = ti.n, nb = ti.nb;   // cout block varies slowest: resident weights change rarely
        const int g = a.groups > 1 ? n % a.groups : 0;
        if (a.b_resident && (g != cur_g || nb != cur_nb)) {
          // new weight set: every MMA that reads the old one must have retired first
          if (have_last) mbar_wait(&empty[last_s], last_ph);
          mbar_expect_tx_e(bfull, (uint32_t)a.bres_bytes);
          for (int ch = 0; ch < a.nchunks; ++ch)
            for (int dxi = 0; dxi < a.ks; ++dxi)
              tma_load_5d(bres + (ch * a.ks + dxi) * a.b_bytes, &tmB, bfull, ch * 64, nb * a.nblk, dxi, 0, g);
          cur_g = g;
          cur_nb = nb;
        }
        if (a.geom == 3) {
          // Streamed weights with a deep pipeline: the activations of a K chunk are ONE haloed copy {64 ch, 10 px, 34 rows}
          // (43.5 KB) in their own ring, and the weights stream through a ring of single-tap 16 KB stages (8 deep =
          // ~8,000 cycles of MMAs ahead).
          for (int ch = 0; ch < a.nchunks; ++ch) {
            mbar_wait(&aempty[as_], aph_ ^ 1);
            mbar_expect_tx_e(&afull[as_], (uint32_t)a.a_bytes);
            tma_load_4d(stages + as_ * a.a_slot, &tmA, &afull[as_], ch * 64, tx * 8 - 1, ty * 32 - 1, n);
            if (++as_ == a.na_slots) { as_ = 0; aph_ ^= 1; }
            for (int dxi = 0; dxi < 3; ++dxi)
              for (int dyi = 0; dyi < 3; ++dyi) {
                mbar_wait(&empty[s], ph ^ 1);
                mbar_expect_tx_e(&full[s], (uint32_t)a.b_bytes);
                tma_load_5d(wring + s * a.stage_bytes, &tmB, &full[s], ch * 64, nb * 128, dxi, dyi, g);
                if (++s == a.nstages) { s = 0; ph ^= 1; }
              }
          }
        } else if (a.geom) {
          // one row-haloed, column-haloed copy {64 ch, 10 px, 18 rows} per K chunk serves all nine taps
          for (int ch = 0; ch < a.nchunks; ++ch) {
            mbar_wait(&empty[s], ph ^ 1);
            uint8_t* sa_ = stages + s * a.stage_bytes;
            mbar_expect_tx_e(&full[s], stage_tx);
            tma_load_4d(sa_, &tmA, &full[s], ch * 64, tx * 8 - pad, ty * a.tile_h - pad, n);
            last_s = s; last_ph = ph; have_last = true;
            if (++s == a.nstages) { s = 0; ph ^= 1; }
          }
        } else
        for (int ch = 0; ch < a.nchunks; ++ch) {
          for (int dxi = 0; dxi < a.ks; ++dxi) {
            mbar_wait(&empty[s], ph ^ 1);
            uint8_t* sa_ = stages + s * a.stage_bytes;
            mbar_expect_tx_e(&full[s], stage_tx);
            tma_load_4d(sa_, &tmA, &full[s], ch * 64, tx * TC_TW + dxi - pad, ty * a.tile_h - pad, n);
            if (!a.b_resident) tma_load_5d(sa_ + a.a_bytes, &tmB, &full[s], ch * 64, nb * a.nblk, dxi, 0, g);
            last_s = s; last_ph = ph; have_last = true;
            if (++s == a.nstages) { s = 0; ph ^= 1; }
          }
        }
      }
    }
  } else if (warp < TC_EPI_WARP0) {
    // ================================ MMA issuers ========================================
    // One issuing warp is enough when a tile is many large MMAs (128->128 3x3: 144 x 64 cycles).  Small-N / small-K
    // layers are bound by the ISSUE path instead: ncu of a 32->32 3x3 layer shows the epilogue and producer warps
    // waiting while the MMA warp spends ~1,900 cycles on the ~300 instructions (descriptor assembly on the uniform
    // datapath, barrier waits, commits) that surround the 18 sixteen-cycle MMAs of a tile.  Tiles are independent
    // (own accumulator, own pipeline stages), so warp 1+g takes tiles g, g+nmma, ... of this CTA: stage and accumulator
    // positions advance by whole tiles, tcgen05.commit tracks the issuing thread's own MMAs.
    const int g = warp - 1;
    if (g < a.nmma) {
    const int nmma = a.nmma;
    const uint32_t umma_n = a.geom == 3 ? 256u : (uint32_t)a.nblk;   // geom 3: N = the 256 pixels of a tile
    const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((umma_n >> 3) << 17) | ((128u >> 4) << 24);
    const int k0 = g * kiters;
    int s = k0 % a.nstages;
    uint32_t ph = (uint32_t)((k0 / a.nstages) & 1);
    int as = g;                                     // nmma <= nacc, nacc % nmma == 0
    uint32_t aph = 0;
    int cur_g = -1, cur_nb = -1;
    uint32_t bph = 0;
    const uint32_t stages_u32 = smem_u32(stages), bres_u32 = smem_u32(bres);
    const uint32_t b_step = (uint32_t)(a.nblk * 128) >> 4;
    const int last_chunk_it = a.geom ? a.nchunks - 1 : (a.nchunks - 1) * a.ks;   // stages of the last (possibly partial) K chunk
    const int skip = (nmma - 1) * kiters;
    int g3_as = 0;                                  // geom 3: activation ring position
    uint32_t g3_aph = 0;
    TileIter ti;
    ti.init(a);                                     // tile coordinates matter only for weight-set changes (nmma == 1)
    for (int q = 0; q < g; ++q) ti.next(a);
    for (; ti.valid(a);) {
      if (a.b_resident) {
        const int nb = ti.nb;
        const int gg = a.groups > 1 ? ti.n % a.groups : 0;
        if (gg != cur_g || nb != cur_nb) {           // nmma > 1 launches have ONE weight set: every warp waits for phase 0 once
          mbar_wait(bfull, bph);
          bph ^= 1;
          cur_g = gg;
          cur_nb = nb;
        }
      }
      mbar_wait(&tempty[as], aph ^ 1);
      tc_fence_after();
      const uint32_t tmem_d = tmem_base + (uint32_t)(as * a.acc_slot);
      if (a.geom == 3) {
        // nmma == 1.  Per K chunk: wait for the haloed copy; per tap: wait for its weight stage, issue its K steps as
        // D[cout, pixel] += W_tap[cout, k] * X[pixel shifted by the tap, k] (A = the weight stage, SBO = 1024; B = the copy
        // at byte offset dy*1280 + dx*128, SBO = 1280), release the weight stage; after the ninth tap release the copy.
        // Chunk -> dx -> dy -> K step is the issue order of the g0x2 geometry this one replaced.
        const uint32_t wring_u32 = stages_u32 + (uint32_t)(a.na_slots * a.a_slot);
        for (int ch = 0; ch < a.nchunks; ++ch) {
          mbar_wait(&afull[g3_as], g3_aph);
          tc_fence_after();
          const uint32_t x_addr = stages_u32 + (uint32_t)(g3_as * a.a_slot);
          const int ksteps = (ch == a.nchunks - 1) ? a.ksteps_last : 4;
          for (int dxi = 0; dxi < 3; ++dxi)
            for (int dyi = 0; dyi < 3; ++dyi) {
              mbar_wait(&full[s], ph);
              tc_fence_after();
              const uint32_t wl = desc_lo(wring_u32 + (uint32_t)(s * a.stage_bytes));
              const uint32_t xl = desc_lo(x_addr + (uint32_t)dyi * (a.a_step16 << 4) + 128u * (uint32_t)dxi);
              const uint32_t acc0 = (ch > 0 || dxi > 0 || dyi > 0) ? 1u : 0u;
              switch (ksteps) {
                case 4: umma_tap1c_k4(tmem_d, wl, xl, idesc, acc0, TC_DESC_HI, a.a_desc_hi); break;
                case 3: umma_tap1c_k3(tmem_d, wl, xl, idesc, acc0, TC_DESC_HI, a.a_desc_hi); break;
                case 2: umma_tap1c_k2(tmem_d, wl, xl, idesc, acc0, TC_DESC_HI, a.a_desc_hi); break;
                default: umma_tap1c_k1(tmem_d, wl, xl, idesc, acc0, TC_DESC_HI, a.a_desc_hi); break;
              }
              umma_commit(&empty[s]);
              if (++s == a.nstages) { s = 0; ph ^= 1; }
            }
          umma_commit(&aempty[g3_as]);
          if (++g3_as == a.na_slots) { g3_as = 0; g3_aph ^= 1; }
        }
        umma_commit(&tfull[as]);
        as += nmma;
        if (as >= a.nacc) { as -= a.nacc; aph ^= 1; }
        ti.next(a);
        continue;
      }
      for (int it = 0; it < kiters; ++it) {
        mbar_wait(&full[s], ph);
        tc_fence_after();
        {
          const uint32_t a_addr = stages_u32 + (uint32_t)s * (uint32_t)a.stage_bytes;
          // weights: streamed next to the A copy, or the resident slice of this (chunk, dx)
          const uint32_t b_addr = a.b_resident ? bres_u32 + (uint32_t)it * (uint32_t)a.b_bytes : a_addr + (uint32_t)a.a_bytes;
          const int ksteps = (it >= last_chunk_it) ? a.ksteps_last : 4;
          if (a.geom) {
            // tap (dy, dx) = the same copy at byte offset dy*1280 + dx*128: the 128B swizzle is a function of the
            // absolute shared-memory address (measured), so unaligned starts and SBO = 1280 need no base offset
            for (int dxi = 0; dxi < 3; ++dxi) {
              const uint32_t al = desc_lo(a_addr + 128u * (uint32_t)dxi);
              const uint32_t blx = desc_lo(bres_u32 + (uint32_t)(it * 3 + dxi) * (uint32_t)a.b_bytes);
              const uint32_t accx = (it > 0 || dxi > 0) ? 1u : 0u;
              switch (ksteps) {
                case 4: umma_stage1c_ks3_k4(tmem_d, al, blx, idesc, accx, a.a_desc_hi, b_step, a.a_step16, TC_DESC_HI); break;
                case 3: umma_stage1c_ks3_k3(tmem_d, al, blx, idesc, accx, a.a_desc_hi, b_step, a.a_step16, TC_DESC_HI); break;
                case 2: umma_stage1c_ks3_k2(tmem_d, al, blx, idesc, accx, a.a_desc_hi, b_step, a.a_step16, TC_DESC_HI); break;
                default: umma_stage1c_ks3_k1(tmem_d, al, blx, idesc, accx, a.a_desc_hi, b_step, a.a_step16, TC_DESC_HI); break;
              }
            }
          } else {
          const uint32_t al0 = desc_lo(a_addr), bl = desc_lo(b_addr);
          const uint32_t acc0 = it > 0 ? 1u : 0u;
          // every MMA of this stage (ks taps along dy x ksteps K-steps) in one PTX block per tile half; the second
          // half (output rows 8..15 of a 16-row tile) reads the same haloed copy 8 image rows further down and the
          // SAME weight stage
          for (int half = 0; half < a.halves; ++half) {
            const uint32_t al = al0 + (uint32_t)half * (uint32_t)((TC_TH * TC_ROW_BYTES) >> 4);
            const uint32_t td = tmem_d + (uint32_t)(half * a.acc_half);
            if (a.ks == 3) {
              switch (ksteps) {
                case 4: umma_stage_ks3_k4(td, al, bl, idesc, acc0, TC_DESC_HI, b_step); break;
                case 3: umma_stage_ks3_k3(td, al, bl, idesc, acc0, TC_DESC_HI, b_step); break;
                case 2: umma_stage_ks3_k2(td, al, bl, idesc, acc0, TC_DESC_HI, b_step); break;
                default: umma_stage_ks3_k1(td, al, bl, idesc, acc0, TC_DESC_HI, b_step); break;
              }
            } else {
              switch (ksteps) {
                case 4: umma_stage_ks1_k4(td, al, bl, idesc, acc0, TC_DESC_HI, b_step); break;
                case 3: umma_stage_ks1_k3(td, al, bl, idesc, acc0, TC_DESC_HI, b_step); break;
                case 2: umma_stage_ks1_k2(td, al, bl, idesc, acc0, TC_DESC_HI, b_step); break;
                default: umma_stage_ks1_k1(td, al, bl, idesc, acc0, TC_DESC_HI, b_step); break;
              }
            }
          }
          }
          umma_commit(&empty[s]);                       // smem slot reusable once these MMAs retire
          if (it == kiters - 1) umma_commit(&tfull[as]);  // accumulator complete
        }
        if (++s == a.nstages) { s = 0; ph ^= 1; }
      }
      // on to this warp's next tile: skip the stages and accumulators of the other issuing warps' tiles
      s += skip;
      while (s >= a.nstages) { s -= a.nstages; ph ^= 1; }
      as += nmma;
      if (as >= a.nacc) { as -= a.nacc; aph ^= 1; }
      for (int q = 0; q < nmma; ++q) ti.next(a);
    }
    }
  } else {
    // ================================ epilogue (warps 4..19) ============================
    const int mode = a.epi == FFSR_EPI_LKAGATE ? EM_LKAGATE
                     : (a.epi == FFSR_EPI_RESIDUAL ? EM_RESIDUAL : (a.epi == FFSR_EPI_ACTGRAD ? EM_ACTGRAD : a.act));
    // one specialised loop per (epilogue mode, output type): no per-element switches, and the
    // plain modes do not carry the residual registers
    if (a.geom == 3) {
      switch (mode) {
        case EM_GELU:
          if (a.gelu_tanh) swapped_epilogue<EM_GELU, true>(a, tfull, tempty, tmem_base, warp, lane);
          else swapped_epilogue<EM_GELU, false>(a, tfull, tempty, tmem_base, warp, lane);
          break;
        case EM_RELU: swapped_epilogue<EM_RELU, false>(a, tfull, tempty, tmem_base, warp, lane); break;
        case EM_SIGMOID: swapped_epilogue<EM_SIGMOID, false>(a, tfull, tempty, tmem_base, warp, lane); break;
        case EM_RESIDUAL: swapped_epilogue<EM_RESIDUAL, false>(a, tfull, tempty, tmem_base, warp, lane); break;
        default: swapped_epilogue<EM_NONE, false>(a, tfull, tempty, tmem_base, warp, lane); break;
      }
    } else if (a.lean) {
      switch (mode) {
        case EM_GELU:
          if (a.gelu_tanh) lean_epilogue<EM_GELU, true>(a, tfull, tempty, tmem_base, warp, lane, sbias);
          else lean_epilogue<EM_GELU, false>(a, tfull, tempty, tmem_base, warp, lane, sbias);
          break;
        case EM_RELU: lean_epilogue<EM_RELU, false>(a, tfull, tempty, tmem_base, warp, lane, sbias); break;
        case EM_SIGMOID: lean_epilogue<EM_SIGMOID, false>(a, tfull, tempty, tmem_base, warp, lane, sbias); break;
        case EM_RESIDUAL: lean_epilogue<EM_RESIDUAL, false>(a, tfull, tempty, tmem_base, warp, lane, sbias); break;
        default: lean_epilogue<EM_NONE, false>(a, tfull, tempty, tmem_base, warp, lane, sbias); break;
      }
    } else if (a.out_bf16) {
      switch (mode) {
        case EM_GELU: epilogue_loop<EM_GELU, true>(a, tfull, tempty, tmem_base, warp, lane); break;
        case EM_RELU: epilogue_loop<EM_RELU, true>(a, tfull, tempty, tmem_base, warp, lane); break;
        case EM_SIGMOID: epilogue_loop<EM_SIGMOID, true>(a, tfull, tempty, tmem_base, warp, lane); break;
        case EM_RESIDUAL: epilogue_loop<EM_RESIDUAL, true>(a, tfull, tempty, tmem_base, warp, lane); break;
        case EM_LKAGATE: epilogue_loop<EM_LKAGATE, true>(a, tfull, tempty, tmem_base, warp, lane); break;
        case EM_ACTGRAD: epilogue_loop<EM_ACTGRAD, true>(a, tfull, tempty, tmem_base, warp, lane); break;
        default: epilogue_loop<EM_NONE, true>(a, tfull, tempty, tmem_base, warp, lane); break;
      }
    } else {
      switch (mode) {
        case EM_GELU: epilogue_loop<EM_GELU, false>(a, tfull, tempty, tmem_base, warp, lane); break;
        case EM_RELU: epilogue_loop<EM_RELU, false>(a, tfull, tempty, tmem_base, warp, lane); break;
        case EM_SIGMOID: epilogue_loop<EM_SIGMOID, false>(a, tfull, tempty, tmem_base, warp, lane); break;
        case EM_RESIDUAL: epilogue_loop<EM_RESIDUAL, false>(a, tfull, tempty, tmem_base, warp, lane); break;
        case EM_LKAGATE: epilogue_loop<EM_LKAGATE, false>(a, tfull, tempty, tmem_base, warp, lane); break;
        case EM_ACTGRAD: epilogue_loop<EM_ACTGRAD, false>(a, tfull, tempty, tmem_base, warp, lane); break;
        default: epilogue_loop<EM_NONE, false>(a, tfull, tempty, tmem_base, warp, lane); break;
      }
    }
  }

  // ---- teardown: everyone done with TMEM before the allocating warp frees it
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TC_TMEM_COLS));
  }
}

// ---------------------------------------------------------------------------- host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
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
}  // namespace

int ffsr_conv2d_tc(const ffsr_conv_params* pp, cudaStream_t stream) {
  const ffsr_conv_params& p = *pp;
  FFSR_REQUIRE(p.in_dtype == FFSR_DT_BF16, FFSR_ERR_ARG, "conv2d(tc): input must be bf16 NHWC (cast upstream)");
  FFSR_REQUIRE(p.w_dtype == FFSR_DT_BF16, FFSR_ERR_ARG, "conv2d(tc): weights must be packed bf16 [g*taps][CoutPad][CinPad]");
  FFSR_REQUIRE(p.in_sC == 1, FFSR_ERR_ARG, "conv2d(tc): input must be channels-last");
  FFSR_REQUIRE(((uintptr_t)p.in % 16) == 0 && (p.in_sX * 2) % 16 == 0 && (p.in_sY * 2) % 16 == 0 && (p.in_sN * 2) % 16 == 0,
               FFSR_ERR_ALIGN, "conv2d(tc): TMA needs a 16B-aligned base and 16B-multiple strides");
  EncodeTiledFn enc = get_encode_fn();
  FFSR_REQUIRE(enc, FFSR_ERR_DRIVER, "conv2d(tc): cuTensorMapEncodeTiled entry point unavailable");

  const int taps = p.ksize * p.ksize;
  const int cin_pad = (p.Cin + 63) / 64 * 64;
  const int cout_pad16 = (p.Cout + 15) / 16 * 16;
  const int nblk = cout_pad16 <= 128 ? cout_pad16 : 128;
  const int cout_pad = (cout_pad16 + nblk - 1) / nblk * nblk;
  FFSR_REQUIRE(((uintptr_t)p.w % 16) == 0, FFSR_ERR_ALIGN, "conv2d(tc): weights must be 16B aligned");

  // Streamed weights (the whole 3x3 set of a cout block does not fit beside three A stages: 128->128) are re-fetched
  // for every pixel tile and dominate the TMA traffic (2304 of 3264 128-byte rows per tile).  Those layers use
  // 16x16-pixel tiles: two M=128 MMAs per (tap, K-step) share each weight stage, halving the weight rows per pixel.
  // Multi-block 1x1 layers (the DRCT Linears: N = 360 .. 768 in 128-column blocks).  With the cout block slowest and resident
  // weights the whole activation tensor was re-read from HBM once per block (6 x 88 MB for a 244 -> 768 Linear: the launch sat on
  // the HBM roof of that schedule, 150 us for 12 GFLOP).  Here the cout block varies fastest, the weights stream beside the
  // activations and 16x16-pixel tiles share every weight stage between two M = 128 MMAs.
  const bool gemm_mode = p.ksize == 1 && cout_pad / nblk > 1 && p.groups == 1;
  int halves = 1;
  if (gemm_mode && p.H >= 16 && nblk * 2 * 2 <= TC_TMEM_COLS) halves = 2;
  {
    const int nch0 = (p.Cin + 63) / 64;
    const int a8 = (TC_TH + 2 * (p.ksize / 2)) * TC_ROW_BYTES;
    const int a16 = (2 * TC_TH + 2 * (p.ksize / 2)) * TC_ROW_BYTES;
    const int bb = p.ksize * nblk * 128;
    const int avail0 = TC_SMEM_MAX - 1024 - TC_SMEM_HDR;
    const bool resident = nch0 * p.ksize * bb + 3 * a8 <= avail0;
    if (!resident && p.ksize == 3 && p.H >= 16 && 2 * (a16 + bb) <= avail0 && nblk * 2 * 2 <= TC_TMEM_COLS) halves = 2;
  }
  // 3x3 layers whose weights stay resident use 16x8-pixel tiles fed by ONE haloed copy per 64-channel chunk
  // ({64 ch, 10 px, 18 rows} = 23 KB instead of three 20 KB copies per 128 output pixels): these layers are bound by
  // the L2 -> shared-memory traffic of the haloed A copies, not by the tensor pipe.
  int geom = 0;
  constexpr int A1C_BYTES = 18 * 10 * 128, A1C_STAGE = (A1C_BYTES + 1023) / 1024 * 1024;
  {
    const int nch0 = (p.Cin + 63) / 64;
    const int bb = p.ksize * nblk * 128;
    const int avail0 = TC_SMEM_MAX - 1024 - TC_SMEM_HDR;
    if (p.ksize == 3 && halves == 1 && nch0 * p.ksize * bb + 3 * A1C_STAGE <= avail0 && p.H >= 8)
      geom = 1;
  }
  // Streamed-weight 3x3 layers with bf16 inference outputs: swapped operands (weights = M, 8x32-px tiles = N = 256), see the
  // kernel.  Cout <= 64 (nblk 64) stays on g0x2: an M = 128 MMA would spend half its work on zero weight rows.  Images of
  // fewer than 32 rows stay there too: most of a 256-pixel tile would be padding.
  constexpr int A3_BYTES = 34 * 10 * 128, A3_SLOT = (A3_BYTES + 1023) / 1024 * 1024;
  // Outputs that both 16-byte-group epilogues (the lean one and geom 3's) can store: bf16, plain or residual without an
  // activation, aligned rows, residual inputs aligned to their own 16-byte groups.
  bool lean_ok = (p.epi == FFSR_EPI_PLAIN || (p.epi == FFSR_EPI_RESIDUAL && p.act == ACT_NONE)) && p.out_dtype == FFSR_DT_BF16 &&
                 p.out2 == nullptr && p.groups == 1 && p.Cout % 8 == 0 && ((uintptr_t)p.out % 16) == 0 && p.out_sX % 8 == 0 &&
                 p.out_sY % 8 == 0 && p.out_sN % 8 == 0;
  if (lean_ok && p.epi == FFSR_EPI_RESIDUAL) {
    const int r1q = p.r1_dtype == FFSR_DT_BF16 ? 8 : 4, r2q = p.r2_dtype == FFSR_DT_BF16 ? 8 : 4;
    lean_ok = p.r1 != nullptr && ((uintptr_t)p.r1 % 16) == 0 && p.r1_sX % r1q == 0 && p.r1_sY % r1q == 0 && p.r1_sN % r1q == 0 &&
              (p.r2 == nullptr || (((uintptr_t)p.r2 % 16) == 0 && p.r2_sX % r2q == 0 && p.r2_sY % r2q == 0 && p.r2_sN % r2q == 0));
  }
  if (halves == 2 && geom == 0 && p.ksize == 3 && lean_ok && nblk == 128 && p.H >= 32) geom = 3;
  CUtensorMap tmA, tmB;
  {
    cuuint64_t dims[4] = {(cuuint64_t)p.Cin, (cuuint64_t)p.W, (cuuint64_t)p.H, (cuuint64_t)p.N};
    cuuint64_t strides[3] = {(cuuint64_t)p.in_sX * 2, (cuuint64_t)p.in_sY * 2, (cuuint64_t)p.in_sN * 2};
    cuuint32_t box[4] = {64, TC_TW, (cuuint32_t)(TC_TH * halves + 2 * (p.ksize / 2)), 1};
    if (geom == 1) { box[1] = 10; box[2] = 18; }
    if (geom == 3) { box[1] = 10; box[2] = 34; }
    cuuint32_t es[4] = {1, 1, 1, 1};
    CUresult r = enc(&tmA, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(p.in), dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    FFSR_REQUIRE(r == CUDA_SUCCESS, FFSR_ERR_DRIVER, "conv2d(tc): activation tensor map encode failed (CUresult %d)", (int)r);
  }
  {
    // [g][dy][dx][CoutPad][CinPad] viewed as {K, N, dx, dy, g}
    const cuuint64_t tap_bytes = (cuuint64_t)cin_pad * cout_pad * 2;
    cuuint64_t dims[5] = {(cuuint64_t)cin_pad, (cuuint64_t)cout_pad, (cuuint64_t)p.ksize, (cuuint64_t)p.ksize, (cuuint64_t)p.groups};
    cuuint64_t strides[4] = {(cuuint64_t)cin_pad * 2, tap_bytes, tap_bytes * p.ksize, tap_bytes * taps};
    cuuint32_t box[5] = {64, (cuuint32_t)nblk, 1, (cuuint32_t)(geom == 3 ? 1 : p.ksize), 1};
    cuuint32_t es[5] = {1, 1, 1, 1, 1};
    CUresult r = enc(&tmB, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<float*>(p.w), dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    FFSR_REQUIRE(r == CUDA_SUCCESS, FFSR_ERR_DRIVER, "conv2d(tc): weight tensor map encode failed (CUresult %d)", (int)r);
  }

  TcArgs a;
  a.N = p.N; a.H = p.H; a.W = p.W; a.Cin = p.Cin; a.Cout = p.Cout; a.taps = taps; a.ks = p.ksize;
  a.nblk = nblk;
  a.n_nblocks = cout_pad / nblk;
  a.nchunks = cin_pad / 64;
  const int last = p.Cin - (a.nchunks - 1) * 64;
  a.ksteps_last = (last + 15) / 16;
  a.halves = halves;
  a.geom = geom;
  a.tile_h = geom ? 16 : TC_TH * halves;
  a.a_step16 = (10u * 128u) >> 4;
  a.a_desc_hi = ((10u * 128u) >> 4) | (1u << 14) | (2u << 29);
  a.a_bytes = geom ? A1C_BYTES : (TC_TH * halves + 2 * (p.ksize / 2)) * TC_ROW_BYTES;
  a.b_bytes = p.ksize * nblk * 128;
  const int smem_avail = TC_SMEM_MAX - 1024 - TC_SMEM_HDR;
  const int b_all = a.nchunks * p.ksize * a.b_bytes;          // all taps, all K chunks of one cout block
  a.b_resident = (b_all + 3 * a.a_bytes <= smem_avail && !gemm_mode) ? 1 : 0;
  a.nb_fast = gemm_mode ? 1 : 0;
  a.bres_bytes = a.b_resident ? b_all : 0;
  a.stage_bytes = geom ? A1C_STAGE : a.a_bytes + (a.b_resident ? 0 : a.b_bytes);
  if (geom) {                                                  // decided above with the same residency test
    a.b_resident = 1;
    a.bres_bytes = b_all;
  }
  a.nstages = (smem_avail - a.bres_bytes) / a.stage_bytes;
  if (a.nstages > TC_MAX_STAGES) a.nstages = TC_MAX_STAGES;
  int smem_bytes = 1024 + TC_SMEM_HDR + a.bres_bytes + a.nstages * a.stage_bytes;
  a.a_slot = 0;
  a.na_slots = 0;
  if (geom == 3) {
    a.tile_h = 32;
    a.a_bytes = A3_BYTES;
    a.a_slot = A3_SLOT;
    a.na_slots = TC_MAX_ASLOTS;
    a.b_bytes = nblk * 128;                                    // one tap of one K chunk
    a.b_resident = 0;
    a.bres_bytes = 0;
    a.stage_bytes = a.b_bytes;
    a.nstages = (smem_avail - a.na_slots * a.a_slot) / a.stage_bytes;
    if (a.nstages > TC_MAX_STAGES) a.nstages = TC_MAX_STAGES;
    smem_bytes = 1024 + TC_SMEM_HDR + a.na_slots * a.a_slot + a.nstages * a.stage_bytes;
  }
  a.acc_half = nblk <= 32 ? 32 : (nblk <= 64 ? 64 : 128);
  if (geom == 3) { a.halves = 1; a.acc_half = 256; }         // one accumulator: 128 lanes (couts) x 256 columns (pixels)
  a.acc_slot = a.acc_half * a.halves;
  a.nacc = TC_TMEM_COLS / a.acc_slot;
  if (a.nacc > TC_MAX_ACC) a.nacc = TC_MAX_ACC;
  a.groups = p.groups;
  a.epi_own = 0;
  a.tiles_x = ceil_div(p.W, geom == 1 || geom == 3 ? 8 : TC_TW);
  a.tiles_y = ceil_div(p.H, a.tile_h);
  a.total_tiles = (long long)a.tiles_x * a.tiles_y * p.N * a.n_nblocks;
  a.out = p.out; a.out_sN = p.out_sN; a.out_sY = p.out_sY; a.out_sX = p.out_sX;
  a.out_bf16 = p.out_dtype == FFSR_DT_BF16;
  a.bias = p.bias; a.act = p.act; a.epi = p.epi;
  a.r1 = p.r1; a.r1_sN = p.r1_sN; a.r1_sY = p.r1_sY; a.r1_sX = p.r1_sX; a.r1_bf16 = p.r1_dtype == FFSR_DT_BF16;
  a.r2 = p.r2; a.r2_sN = p.r2_sN; a.r2_sY = p.r2_sY; a.r2_sX = p.r2_sX; a.r2_bf16 = p.r2_dtype == FFSR_DT_BF16;
  a.sa = p.sa; a.sb = p.sb; a.sa_ptr = p.sa_ptr; a.sb_ptr = p.sb_ptr; a.ch_k = p.ch_k; a.ch_d = p.ch_d;
  a.out2 = p.out2;

  static int num_sms = 0;
  if (!num_sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
    cudaFuncSetAttribute(k_conv_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM_MAX);
  }
  const int grid = (int)(a.total_tiles < num_sms ? a.total_tiles : num_sms);
  // tile-per-group epilogue: needs >= 8 accumulators in flight (N <= 64, single-half tiles) and enough tiles per CTA
  static const bool erf_forced = getenv("FFSR_TC_GELU_ERF") != nullptr;
  a.gelu_tanh = (!erf_forced && p.out2 == nullptr) ? 1 : 0;
  const bool own_force = getenv("FFSR_TC_EPI_OWN_FORCE") != nullptr;     // tests: small images take the own path too (read per call)
  a.epi_own = (halves == 1 && a.nacc >= 8 && (own_force || a.total_tiles >= 8LL * grid)) ? 1 : 0;
  {
    // lean epilogue: bf16 inference outputs in 16-byte groups; own mode also for 128-column single-half tiles (4 accumulators)
    const bool own_lean = halves == 1 && a.nacc >= 4 && (own_force || a.total_tiles >= 8LL * grid);
    const bool split_lean = (a.nblk % 64) == 0;
    a.lean = (lean_ok && a.n_nblocks * a.nblk <= TC_BIAS_MAX && (own_lean || split_lean)) ? 1 : 0;
    if (a.lean) a.epi_own = own_lean ? 1 : 0;
    if (a.lean && !a.epi_own && !split_lean) a.lean = 0;
  }
  if (geom == 3) { a.lean = 0; a.epi_own = 0; }               // geom 3 has its own epilogue (swapped_epilogue)
  // several MMA-issuing warps for launches whose tiles are a few small MMAs (issue-bound, see the kernel): needs one weight
  // set for the whole launch and an accumulator ring that is a multiple of the warp count (3 warps: ring of 6)
  {
    a.nmma = 1;
    // Every barrier wait is by PARITY, which tells a phase only from its neighbours: whoever waits for use k of a pipeline
    // stage must KNOW that use k - nstages has completed.  With one issuer that is its own previous wait.  With several, a
    // stage whose consecutive uses fall to different warps would rest on "the producer issued the earlier load first" --
    // but TMA loads complete out of order, and a warp that starts waiting one phase early passes at once on the previous
    // phase's parity (seen on hardware: K = 192, 3 stages per tile in a ring of 8, two issuers -> nondeterministic hangs).
    // So the ring is trimmed to a multiple of nmma * (stages per tile): tile q and tile q + ring / kiters then use the same
    // stages AND belong to the same warp, and every wait follows that warp's own wait for the previous phase.
    const int kiters = geom ? a.nchunks : p.ksize * a.nchunks;
    if ((p.flags & FFSR_CONV_MULTI_ISSUE) && a.b_resident && p.groups == 1 && a.n_nblocks == 1 && halves == 1) {
      int n = TC_MMA_WARPS >= 3 ? 3 : TC_MMA_WARPS;
      while (n > 1 && n * kiters > a.nstages) --n;
      // The accumulator ring must likewise be a multiple of the issuing warps (a slot always belongs to the same warp) AND,
      // with tile ownership in the epilogue, of the four epilogue warp groups (a group waits for its tile's accumulator by
      // parity too, so the previous use of that slot must have been its own tile).  3 warps -> ring of 12 (N <= 32).
      int nm = 1, na = a.nacc;
      if (n == 3 && TC_TMEM_COLS / a.acc_slot >= 12) { nm = 3; na = 12; }
      else if (n >= 2 && a.nacc >= 8) { nm = 2; na = 8; }
      else if (n >= 2 && a.nacc >= 4) { nm = 2; na = 4; }
      else if (n >= 2 && a.nacc >= 2 && !a.epi_own) { nm = 2; na = 2; }
      if (nm > 1) {
        a.nmma = nm;
        a.nacc = na;
        a.nstages = a.nstages / (nm * kiters) * (nm * kiters);
      }
    }
  }
  if (getenv("FFSR_TC_DEBUG") != nullptr)
    fprintf(stderr, "[conv_tc] N=%d H=%d W=%d Cin=%d Cout=%d ks=%d groups=%d epi=%d act=%d out_bf16=%d out2=%d | geom=%d halves=%d nblk=%d nchunks=%d "
                    "kiters=%d nstages=%d resident=%d acc_slot=%d nacc=%d nmma=%d own=%d lean=%d tiles=%lld grid=%d\n",
            p.N, p.H, p.W, p.Cin, p.Cout, p.ksize, p.groups, p.epi, p.act, a.out_bf16, p.out2 != nullptr, a.geom, a.halves, a.nblk, a.nchunks,
            a.geom ? a.nchunks : p.ksize * a.nchunks, a.nstages, a.b_resident, a.acc_slot, a.nacc, a.nmma, a.epi_own, a.lean, a.total_tiles, grid);
  k_conv_tc<<<grid, TC_THREADS, smem_bytes, stream>>>(tmA, tmB, a);
  return ffsr_check_launch("conv2d_tc");
}
