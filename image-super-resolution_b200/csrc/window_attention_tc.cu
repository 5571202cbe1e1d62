// (Shifted-)window multi-head attention of the DRCT-L expert on tcgen05: both products of
//   softmax(q k^T / sqrt(dh) + relative-position bias [+ shift mask]) v          src/models/drct/drct_arch.py:175-206, 385-412
// for one 16 x 16 window (256 tokens) and one head per CTA, bf16 operands, fp32 accumulation in TMEM.  The CUDA-core
// kernel of window_attention.cu spends 14 ms per launch on the 352 x 512 DRCT-L image (2.4 TFLOP/s; 90 % of the whole
// expert forward); this one is bound by the softmax instead of the products.
//
//   operands : NO-SWIZZLE K-major planes (tc_ptx.cuh): q tile [128 rows][DP], k [256][DP] and the probabilities p [128][256]
//              as 8-element planes plane[kg][row] = 16 B; v in the SAME layout as k (planes [channel group][key]): p v takes it as
//              an MN-major B operand, so nothing is transposed on the way in.  DP = head dim padded to a multiple of 16 (30 -> 32, 53 -> 64,
//              122 -> 128, 46 -> 48, 77 -> 80) with zero columns.  The window gather (cyclic shift + partition) happens while
//              the tokens are copied from the channels-last qkv rows into the planes.
//   per tile : S = Q K^T (DP / 16 MMAs, M = 128, N = 256) -> TMEM columns [0, 256); thread = query row: two passes over
//              its 256 scores (max; then exp2, row sum, bf16 probabilities into the p planes); O = P V (16 MMAs, N = DP) ->
//              TMEM columns [0, DP) (S is dead by then); O / rowsum -> global at the token's ORIGINAL pixel.
//   bias     : chunk c of 16 score columns is key row c of the window, so the relative-position index of (query, key)
//              runs down by one per column: 16 consecutive table entries per chunk; the shift mask compares region ids.
#include <cuda.h>
#include <stdlib.h>
#include "common.cuh"
#include "tc_ptx.cuh"
#include "../../include/ffsr_b200.h"

namespace {
using namespace tcx;

constexpr int WT_THREADS = 256;             // two threads per query row: row = tid % 128, score-column half = tid / 128
constexpr int WT_N = 256;                 // tokens per window (16 x 16)
constexpr int WT_WS = 16;
constexpr int WT_HDR = 3072;              // barrier + TMEM slot | pix[256] | rid[256] | xch[256] (row max / row sum exchange)
constexpr int WT_TMEM_COLS = 256;

__device__ __forceinline__ int wt_region(int p, int n, int shift) { return p < n - WT_WS ? 0 : (p < n - shift ? 1 : 2); }

__device__ __forceinline__ float ex2f(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// 16-byte global -> shared copy that does not pass through registers: every cell of a gather is issued at once
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

__device__ __forceinline__ void umma_one(uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi, uint32_t idesc,
                                         uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      ".reg .b64 da, db;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t"
      "}" ::"r"(tmem_d),
      "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit_one(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// HEADPAD: qkv rows are [q | k | v], each heads x DP channels (every head's slice 16-byte aligned and zero padded by the
// qkv Linear itself, whose weight rows the host permutes): the gather is 16-byte loads and stores.  Otherwise rows are the
// reference's [3][heads][dh] order at pitch qp and the gather moves single elements.
template <bool HEADPAD>
__global__ void __launch_bounds__(WT_THREADS) k_window_attn_tc(const __nv_bfloat16* __restrict__ qkv, long qp, int B, int H, int W, int C,
                                                               int heads, int shift, const float* __restrict__ table,
                                                               __nv_bfloat16* __restrict__ out, long op, int DP) {
  extern __shared__ __align__(16) uint8_t smem[];
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + 8);
  int* pix = reinterpret_cast<int*>(smem + 64);
  uint8_t* rid = smem + 64 + WT_N * 4;
  float* xch = reinterpret_cast<float*>(smem + 1408);
  uint8_t* sQ = smem + WT_HDR;
  uint8_t* sK = sQ + 128 * DP * 2;
  uint8_t* sV = sK + WT_N * DP * 2;
  uint8_t* sP = sV + WT_N * DP * 2;
  const int tid = threadIdx.x, warp = tid >> 5;
  const int dh = C / heads;
  const int nwx = W / WT_WS, nwy = H / WT_WS;
  int wid = blockIdx.x;
  const int wx = wid % nwx; wid /= nwx;
  const int wy = wid % nwy;
  const int b = wid / nwy;
  const int h = blockIdx.y;

  if (tid == 0) {
    mbar_init(bar, 1);
    fence_barrier_init();
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(WT_TMEM_COLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  for (int t = tid; t < WT_N; t += WT_THREADS) {
    const int ys = wy * WT_WS + (t >> 4), xs = wx * WT_WS + (t & 15);       // position in the shifted frame
    int yo = ys + shift, xo = xs + shift;                                   // torch.roll(x, -shift)[i] = x[(i + shift) % n]
    if (yo >= H) yo -= H;
    if (xo >= W) xo -= W;
    pix[t] = yo * W + xo;
    rid[t] = shift ? (uint8_t)(wt_region(ys, H, shift) * 3 + wt_region(xs, W, shift)) : 0;
  }
  // zero K / V planes (element-wise gather: the padding channels dh..DP-1 must be zero; head-padded rows carry their zeros).
  // Q is not zeroed here: the bias table overwrites its planes after every S, so each tile's Q gather writes all DP channels.
  if (!HEADPAD) {
    uint4* z = reinterpret_cast<uint4*>(sK);
    const int n16 = (2 * WT_N * DP * 2) / 16;
    for (int i = tid; i < n16; i += WT_THREADS) z[i] = make_uint4(0u, 0u, 0u, 0u);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const size_t img = (size_t)b * H * W;

  const int lane = tid & 31;
  const int cpt = DP >> 3;                                                  // 16-byte cells per token and operand
  if (HEADPAD) {
    // K and V planes [channel group][key][8]: a cell = 8 channels of one key, copied whole with cp.async, so the loads of the
    // whole window are in flight together (with four register-staged loads per thread and round the gather was four to eight
    // dependent round trips to L2 / HBM: 16 % of the kernel's stall samples)
    const int total = WT_N * cpt;
    for (int i = tid; i < total; i += WT_THREADS) {
      const int t = i / cpt, g8 = i - t * cpt;
      const __nv_bfloat16* src = qkv + (img + (size_t)pix[t]) * (size_t)qp + (size_t)(h * DP + g8 * 8);
      cp_async16(sK + g8 * (WT_N * 16) + t * 16, src + heads * DP);
      cp_async16(sV + g8 * (WT_N * 16) + t * 16, src + 2 * heads * DP);
    }
  } else {
  // K planes [kg][key][8] and V^T planes [key group][channel][8 keys].  A warp copies four tokens at a time, lanes across the
  // head's channels (coalesced 2-byte loads), all eight loads of a step issued before the first store: the copy is bound by
  // global-load latency, and the pixel table lives in the same shared memory the stores go to, so the loads are hoisted by hand.
  for (int t0 = warp * 4; t0 < WT_N; t0 += WT_THREADS / 8) {
    size_t row[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) row[u] = (img + (size_t)pix[t0 + u]) * (size_t)qp + (size_t)(h * dh);
    for (int d = lane; d < dh; d += 32) {
      __nv_bfloat16 kv[4], vv[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        kv[u] = qkv[row[u] + C + d];
        vv[u] = qkv[row[u] + 2 * C + d];
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int t = t0 + u;
        *reinterpret_cast<__nv_bfloat16*>(sK + (d >> 3) * (WT_N * 16) + t * 16 + (d & 7) * 2) = kv[u];
        *reinterpret_cast<__nv_bfloat16*>(sV + (d >> 3) * (WT_N * 16) + t * 16 + (d & 7) * 2) = vv[u];
      }
    }
  }
  }

  const float scale2 = rsqrtf((float)dh) * 1.4426950408889634f;            // scores in log2 units: exp(x) = exp2(x log2 e)
  // max of this head's bias table (log2 units): warp maxima through the (not yet used) P buffer
  float bias_max;
  {
    float bm = -INFINITY;
    for (int i = tid; i < (2 * WT_WS - 1) * (2 * WT_WS - 1); i += WT_THREADS) bm = fmaxf(bm, __ldg(table + i * heads + h));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) bm = fmaxf(bm, __shfl_xor_sync(0xffffffffu, bm, o));
    float* red = reinterpret_cast<float*>(sP);
    if (lane == 0) red[warp] = bm;
    __syncthreads();
    bias_max = fmaxf(fmaxf(fmaxf(red[0], red[1]), fmaxf(red[2], red[3])), fmaxf(fmaxf(red[4], red[5]), fmaxf(red[6], red[7]))) * 1.4426950408889634f;
    __syncthreads();
  }
  const uint32_t hi128 = desc_hi(128);
  const uint32_t q32 = smem_u32(sQ), k32 = smem_u32(sK), v32 = smem_u32(sV), p32 = smem_u32(sP);
  // P V: B = V[key][channel] with the CHANNELS contiguous (planes [channel group][key] x 16 B, exactly the K layout) = an MN-major
  // operand (instruction-descriptor bit 16): LBO = 128 B to the next 8 keys, SBO = one plane to the next 8 channels, any 16-byte
  // aligned start (measured: tools/experiments/umma_mnmajor_b.cu).  No transposition of V on the way into shared memory.
  const uint32_t idesc_s = idesc_bf16_m128(256), idesc_o = idesc_bf16_m128(DP) | (1u << 16);
  const uint32_t hi_v = desc_hi(WT_N * 16);
  uint32_t phase = 0;

  for (int mt = 0; mt < 2; ++mt) {
    // ---- Q tile planes [kg][row][8]; rows = queries mt*128 .. +127
    if (HEADPAD) {
      const int total = 128 * cpt;
      for (int i = tid; i < total; i += WT_THREADS) {
        const int rr = i / cpt, gg = i - rr * cpt;
        cp_async16(sQ + gg * 2048 + rr * 16, qkv + (img + (size_t)pix[mt * 128 + rr]) * (size_t)qp + (size_t)(h * DP + gg * 8));
      }
      cp_async_wait_all();                           // also the K / V copies issued before the loop (first tile)
    } else
    for (int r0 = warp * 8; r0 < 128; r0 += WT_THREADS / 4) {
      size_t row[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) row[u] = (img + (size_t)pix[mt * 128 + r0 + u]) * (size_t)qp + (size_t)(h * dh);
      // channels dh..DP-1 are written as zeros: for dh < 16 they share planes 0 / 1 with the table of the previous tile, whose
      // bytes can read as bf16 Inf / NaN, and Inf x the zero K padding is NaN in the MMA
      for (int d = lane; d < DP; d += 32) {
        __nv_bfloat16 qv[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) qv[u] = d < dh ? qkv[row[u] + d] : __float2bfloat16_rn(0.f);
#pragma unroll
        for (int u = 0; u < 8; ++u) *reinterpret_cast<__nv_bfloat16*>(sQ + (d >> 3) * 2048 + (r0 + u) * 16 + (d & 7) * 2) = qv[u];
      }
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    if (tid == 0) {
      tc_fence_after();
      for (int ks = 0; ks < DP / 16; ++ks)
        umma_one(tmem, desc_lo(q32 + (uint32_t)(2 * ks) * 2048u, 2048u), hi128, desc_lo(k32 + (uint32_t)(2 * ks) * (WT_N * 16), WT_N * 16), hi128,
                 idesc_s, ks > 0 ? 1u : 0u);
      umma_commit_one(bar);
    }
    mbar_wait(bar, phase);
    phase ^= 1;
    tc_fence_after();

    // ---- this head's relative-position bias table (31 x 31 entries, log2 units) -> the Q planes, dead now that S is complete:
    //      the softmax below read one global word per score before
    float* tbl = reinterpret_cast<float*>(sQ);
    for (int i = tid; i < (2 * WT_WS - 1) * (2 * WT_WS - 1); i += WT_THREADS) tbl[i] = __ldg(table + i * heads + h) * 1.4426950408889634f;
    __syncthreads();
    // ---- softmax: thread = query row
    const int rowi = tid & 127, half = tid >> 7;                             // this thread's query row of the tile and its 8 of the 16 chunks
    const int q = mt * 128 + rowi;
    const int qy = q >> 4, qx = q & 15;
    const uint32_t qr = rid[q];
    const uint32_t trow = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    const float L2E = 1.4426950408889634f;
    // Row maximum: of the raw scores only (one pass of tcgen05.ld + max, no bias loads).  softmax is shift invariant, so any
    // m >= max_k s_k is as good as the true maximum for overflow; m = max_k(q k scale) + max(bias table of this head) is such
    // a bound (the mask only lowers scores), and it stays within the bias RANGE of the true maximum, far from underflow.
    float mx = -INFINITY;
#pragma unroll 1
    for (int c = half * 8; c < half * 8 + 8; ++c) {
      uint32_t v[16];
      tmem_ld16(trow + (uint32_t)(c * 16), v);
      tmem_wait_ld(v);
#pragma unroll
      for (int i = 0; i < 16; ++i) mx = fmaxf(mx, __uint_as_float(v[i]));
    }
    xch[tid] = mx;
    __syncthreads();
    mx = fmaxf(xch[rowi], xch[rowi + 128]);
    __syncthreads();                                                         // both maxima read: xch takes the row sums next
    mx = fmaf(mx, scale2, bias_max);
    float sum = 0.f;
#pragma unroll 1
    for (int c = half * 8; c < half * 8 + 8; ++c) {                          // 16 columns = key row c of the window
      uint32_t v[16];
      tmem_ld16(trow + (uint32_t)(c * 16), v);
      tmem_wait_ld(v);
      const float* tb = tbl + ((qy - c + WT_WS - 1) * (2 * WT_WS - 1) + (qx + WT_WS - 1));   // key column 0; -1 per column
      const uint4 rk = *reinterpret_cast<const uint4*>(rid + c * 16);
      const uint32_t rw[4] = {rk.x, rk.y, rk.z, rk.w};
      float pr[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        float a = fmaf(__uint_as_float(v[i]), scale2, tb[-i] - mx);
        if (shift && ((rw[i >> 2] >> ((i & 3) * 8)) & 0xffu) != qr) a -= 100.0f * L2E;
        pr[i] = ex2f(a);
        sum += pr[i];
      }
      // keys 16c .. 16c+7 -> plane 2c, keys 16c+8 .. -> plane 2c+1; row = this query
      *reinterpret_cast<uint4*>(sP + (2 * c) * 2048 + rowi * 16) =
          make_uint4(pack_bf16(pr[0], pr[1]), pack_bf16(pr[2], pr[3]), pack_bf16(pr[4], pr[5]), pack_bf16(pr[6], pr[7]));
      *reinterpret_cast<uint4*>(sP + (2 * c + 1) * 2048 + rowi * 16) =
          make_uint4(pack_bf16(pr[8], pr[9]), pack_bf16(pr[10], pr[11]), pack_bf16(pr[12], pr[13]), pack_bf16(pr[14], pr[15]));
    }
    xch[tid] = sum;
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();                                                         // every row of S has been read, P is complete
    const float inv = 1.0f / (xch[rowi] + xch[rowi + 128]);
    if (tid == 0) {
      tc_fence_after();
      for (int ks = 0; ks < WT_N / 16; ++ks)
        umma_one(tmem, desc_lo(p32 + (uint32_t)(2 * ks) * 2048u, 2048u), hi128, desc_lo(v32 + (uint32_t)ks * 256u, 128u), hi_v, idesc_o,
                 ks > 0 ? 1u : 0u);
      umma_commit_one(bar);
    }
    mbar_wait(bar, phase);
    phase ^= 1;
    tc_fence_after();

    // ---- O / rowsum -> bf16 rows in the (dead) P buffer -> global at the token's original pixel: a warp writes one row at a
    //      time, lanes along the channels (the thread-per-row version scattered every 2-byte store of a warp over 32 rows)
    {
      __nv_bfloat16* so = reinterpret_cast<__nv_bfloat16*>(sP);
      const int pitch = DP + 8;                                              // elements; 16-byte aligned rows, conflict-free
      for (int c = half; c < DP / 16; c += 2) {
        uint32_t v[16];
        tmem_ld16(trow + (uint32_t)(c * 16), v);
        tmem_wait_ld(v);
        uint4* d4 = reinterpret_cast<uint4*>(so + rowi * pitch + c * 16);
        d4[0] = make_uint4(pack_bf16(__uint_as_float(v[0]) * inv, __uint_as_float(v[1]) * inv), pack_bf16(__uint_as_float(v[2]) * inv, __uint_as_float(v[3]) * inv),
                           pack_bf16(__uint_as_float(v[4]) * inv, __uint_as_float(v[5]) * inv), pack_bf16(__uint_as_float(v[6]) * inv, __uint_as_float(v[7]) * inv));
        d4[1] = make_uint4(pack_bf16(__uint_as_float(v[8]) * inv, __uint_as_float(v[9]) * inv), pack_bf16(__uint_as_float(v[10]) * inv, __uint_as_float(v[11]) * inv),
                           pack_bf16(__uint_as_float(v[12]) * inv, __uint_as_float(v[13]) * inv), pack_bf16(__uint_as_float(v[14]) * inv, __uint_as_float(v[15]) * inv));
      }
      tc_fence_before();
      __syncthreads();                                                       // O read; rows staged
      const bool pair_ok = ((dh | (int)(op & 1)) & 1) == 0 && ((reinterpret_cast<uintptr_t>(out) & 3) == 0);
      for (int r = warp; r < 128; r += WT_THREADS / 32) {
        __nv_bfloat16* dst = out + (img + pix[mt * 128 + r]) * op + h * dh;
        if (pair_ok) {                                                       // even head dim and pitch: 4-byte stores
          for (int d = 2 * lane; d < dh; d += 64) *reinterpret_cast<uint32_t*>(dst + d) = *reinterpret_cast<const uint32_t*>(so + r * pitch + d);
        } else {
          for (int d = lane; d < dh; d += 32) dst[d] = so[r * pitch + d];
        }
      }
      __syncthreads();                                                       // Q / P free for the next tile
      tc_fence_after();
    }
  }
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(WT_TMEM_COLS));
}
}  // namespace

// returns 1 if the tcgen05 kernel was launched, 0 if the shape is not covered (caller falls back to the CUDA-core kernel), < 0 on error
static int wt_launch(bool headpad, const void* qkv, long qkv_pitch, int B, int H, int W, int C, int heads, int window, int shift,
                     const float* bias_table, void* out, long out_pitch, cudaStream_t stream) {
  if (window != WT_WS || getenv("FFSR_WATTN_TC0") != nullptr) return 0;
  const int dh = C / heads;
  const int DP = (dh + 15) / 16 * 16;
  if (DP < 16 || DP > 128) return 0;
  const size_t smem = (size_t)WT_HDR + (size_t)128 * DP * 2 + 2 * (size_t)WT_N * DP * 2 + 65536;
  if (smem > 232448) return 0;
  static bool attr = false;
  if (!attr) {
    attr = true;
    cudaFuncSetAttribute(k_window_attn_tc<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448);
    cudaFuncSetAttribute(k_window_attn_tc<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448);
  }
  const dim3 grid((unsigned)((long)B * (H / window) * (W / window)), (unsigned)heads);
  if (headpad)
    k_window_attn_tc<true><<<grid, WT_THREADS, smem, stream>>>((const __nv_bfloat16*)qkv, qkv_pitch, B, H, W, C, heads, shift, bias_table,
                                                               (__nv_bfloat16*)out, out_pitch, DP);
  else
    k_window_attn_tc<false><<<grid, WT_THREADS, smem, stream>>>((const __nv_bfloat16*)qkv, qkv_pitch, B, H, W, C, heads, shift, bias_table,
                                                                (__nv_bfloat16*)out, out_pitch, DP);
  const int rc = ffsr_check_launch("k_window_attn_tc");
  return rc ? rc : 1;
}

int ffsr_window_attention_tc_try(const void* qkv, long qkv_pitch, int B, int H, int W, int C, int heads, int window, int shift,
                                 const float* bias_table, void* out, long out_pitch, cudaStream_t stream) {
  return wt_launch(false, qkv, qkv_pitch, B, H, W, C, heads, window, shift, bias_table, out, out_pitch, stream);
}

// qkv rows in the head-padded order [q | k | v] x [heads][DP], DP = ffsr_window_attention_head_pad(C / heads): what a qkv Linear
// produces when the host permutes / zero-pads its weight rows.  bf16, 16 x 16 windows.  out: [B][H][W] rows of pitch out_pitch,
// channel = head * dh + d as the proj Linear expects.
extern "C" int ffsr_window_attention_head_pad(int head_dim) { return (head_dim + 15) / 16 * 16; }
extern "C" int ffsr_window_attention_headpadded(const void* qkv, int B, int H, int W, int C, int heads, int window, int shift,
                                                const float* bias_table, void* out, long out_pitch, cudaStream_t stream) {
  FFSR_REQUIRE(qkv && out && bias_table, FFSR_ERR_ARG, "window_attention_headpadded: null pointer");
  FFSR_REQUIRE(B > 0 && H > 0 && W > 0 && heads > 0 && C > 0 && C % heads == 0 && out_pitch >= C, FFSR_ERR_ARG,
               "window_attention_headpadded: B=%d H=%d W=%d C=%d heads=%d", B, H, W, C, heads);
  FFSR_REQUIRE(window == WT_WS && H % window == 0 && W % window == 0 && shift >= 0 && shift < window && C / heads <= 128, FFSR_ERR_ARG,
               "window_attention_headpadded: needs 16 x 16 windows and head dim <= 128 (window %d, head dim %d)", window, C / heads);
  FFSR_REQUIRE(((uintptr_t)qkv % 16) == 0, FFSR_ERR_ALIGN, "window_attention_headpadded: qkv must be 16-byte aligned");
  const int DP = ffsr_window_attention_head_pad(C / heads);
  const int r = wt_launch(true, qkv, 3L * heads * DP, B, H, W, C, heads, window, shift, bias_table, out, out_pitch, stream);
  FFSR_REQUIRE(r != 0, FFSR_ERR_ARG, "window_attention_headpadded: shape not covered by the tcgen05 kernel");
  return r == 1 ? 0 : r;
}
