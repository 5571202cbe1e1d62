// LR-side per-pixel token kernels:
//   * Phase 3 cross-band attention over the 9 sub-band tokens of each LR pixel
//     (EnhancedCrossBandWithLKA.forward, src/models/large_kernel_attention.py:207-233)
//   * Phase 3 tail: out_proj + band residual + routing_lr (:240-241, enhanced_fusion_v2.py:713)
//   * LayerNorm rows and the 4-token x 8-head attention core used by Phase 4 (:389-392)
//   * Phase 6 gate normalisation (DynamicExpertSelector.forward, enhanced_fusion_v2.py:462-465)
// All fp32: routing_lr feeds the expert-selection indices that must be bit-exact.
#include "common.cuh"

namespace {
constexpr int CB_DIM = 64, CB_BANDS = 9, CB_HD = 16;
}  // namespace

// ------------------------------------------------------------------------------------
// Cross-band attention with band_proj -> LayerNorm -> in_proj collapsed algebraically.  A token is an affine function of
// the 3 band values x:  t = Wp x + b;  t - mean(t) = A x + c;  LN(t) = (A x + c) * rstd * gamma + beta;  so
//   qkv = W_in LN(t) + b_in = rstd * (M x + m0) + n0,   M = W_in diag(gamma) A  [192x3],  m0 = W_in diag(gamma) c,
//   n0 = W_in beta + b_in  (folded on the host in fp64): 4 FMAs per qkv channel instead of 64, with the variance
// still taken from the 64 centred values themselves.  fold = [A|c : 64x4][M|m0 : 192x4][n0 : 192].
// Register-blocked (a block-per-8-pixels version ran at 0.87 ms per C3 image, ~15 % of the FMA peak, bound by one
// shared-memory load per FMA in the attention and out_proj loops and by five block barriers per 8 pixels).
// A WARP owns 8 pixels per iteration and never meets a block barrier; lane = (pixel, head):
//   * 1/std of the 9 tokens: each of a pixel's four lanes sums 16 of the 64 centred channels, two xor-shuffles combine them;
//   * q, k, v are never stored: channel d of head h is  rstd * (M[d] . x + m0[d]) + n0[d]  (4 FMAs), computed where it is used,
//     k / v once per pixel and head for all three query bands of a group;
//   * softmax(q k^T / 4) v in registers, context -> a per-warp shared tile [24 tokens][64];
//   * out_proj as a 6-token x 8-channel register tile per lane (48 FMAs per 14 vector loads), + bias + band_proj residual.
// Scores sum over d = 0..15, the context over j = 0..8 and out_proj over c = 0..63, each in ascending order.
// ------------------------------------------------------------------------------------
namespace {
constexpr int CB2_WARPS = 8, CB2_PX = 8, CB2_LD = 68;
struct CB2Smem {
  float4 fa[CB_DIM];                   // centred band_proj rows A | c
  float4 fm[3 * CB_DIM];               // folded in_proj rows M | m0   (q, k, v)
  float4 pw[CB_DIM];                   // band_proj rows W | b (residual)
  float n0[3 * CB_DIM];
  float ob[CB_DIM];
  float wo[CB_DIM][CB_DIM];            // out_proj transposed: wo[c][o]
  float xs[CB2_WARPS][CB2_PX][28];     // the 27 band values of the warp's pixels
  float ctx[CB2_WARPS][3 * CB2_PX][CB2_LD];
};
__device__ __forceinline__ float aff3(const float4& m, float x0, float x1, float x2) {
  return fmaf(m.z, x2, fmaf(m.y, x1, fmaf(m.x, x0, m.w)));
}
}  // namespace

template <int NG>   // query-band groups of three: 1 for the production nq = 3 (x and rstd die before out_proj), 3 for nq up to 9
__global__ void __launch_bounds__(CB2_WARPS * 32, 2) k_crossband_attn2(
    const float* __restrict__ fold, const float* __restrict__ raw9, int B, int HW, const float* __restrict__ proj_w,
    const float* __restrict__ proj_b, const float* __restrict__ out_w, const float* __restrict__ out_b, int nq,
    float* __restrict__ tok_out) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  CB2Smem& s = *reinterpret_cast<CB2Smem*>(smem_raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int i = tid; i < CB_DIM * CB_DIM; i += CB2_WARPS * 32) s.wo[i % CB_DIM][i / CB_DIM] = out_w[i];
  for (int i = tid; i < 3 * CB_DIM; i += CB2_WARPS * 32) {
    s.fm[i] = *reinterpret_cast<const float4*>(fold + CB_DIM * 4 + (long)i * 4);
    s.n0[i] = fold[CB_DIM * 4 + 3 * CB_DIM * 4 + i];
  }
  if (tid < CB_DIM) {
    s.fa[tid] = *reinterpret_cast<const float4*>(fold + tid * 4);
    s.pw[tid] = make_float4(proj_w[tid * 3], proj_w[tid * 3 + 1], proj_w[tid * 3 + 2], proj_b[tid]);
    s.ob[tid] = out_b[tid];
  }
  __syncthreads();

  const int px = lane >> 2, h = lane & 3;
  const int tb = lane >> 3, cb = lane & 7;            // out_proj tile: tokens 6 tb .. 6 tb + 5, channels 8 cb .. 8 cb + 7
  const int tiles_per_img = (HW + CB2_PX - 1) / CB2_PX;
  const long total = (long)B * tiles_per_img;
  float (*xs)[28] = s.xs[warp];
  float (*ctx)[CB2_LD] = s.ctx[warp];
  for (long tile = (long)blockIdx.x * CB2_WARPS + warp; tile < total; tile += (long)gridDim.x * CB2_WARPS) {
    const int b = (int)(tile / tiles_per_img);
    const int p0 = (int)(tile - (long)b * tiles_per_img) * CB2_PX;
    const int p = p0 + px;
    float x[27];
#pragma unroll
    for (int r = 0; r < 27; ++r) x[r] = (p < HW) ? __ldg(raw9 + ((long)b * 27 + r) * HW + p) : 0.f;
    if (h == 0) {
#pragma unroll
      for (int r = 0; r < 27; ++r) xs[px][r] = x[r];
    }
    // 1/std of the nine tokens
    float rstd[CB_BANDS];
    {
      float sq[CB_BANDS];
#pragma unroll
      for (int j = 0; j < CB_BANDS; ++j) sq[j] = 0.f;
#pragma unroll 4
      for (int cc = 0; cc < 16; ++cc) {
        const float4 a = s.fa[h * 16 + cc];
#pragma unroll
        for (int j = 0; j < CB_BANDS; ++j) {
          const float d = aff3(a, x[3 * j], x[3 * j + 1], x[3 * j + 2]);
          sq[j] = fmaf(d, d, sq[j]);
        }
      }
#pragma unroll
      for (int j = 0; j < CB_BANDS; ++j) {
        sq[j] += __shfl_xor_sync(0xffffffffu, sq[j], 1);
        sq[j] += __shfl_xor_sync(0xffffffffu, sq[j], 2);
        rstd[j] = rsqrtf(sq[j] * (1.0f / CB_DIM) + 1e-5f);
      }
    }
#pragma unroll
    for (int qg = 0; qg < NG; ++qg) {
      if (qg * 3 >= nq) break;
      // scores of this head for the three query bands of the group
      float sc[3][CB_BANDS];
#pragma unroll
      for (int t = 0; t < 3; ++t)
#pragma unroll
        for (int j = 0; j < CB_BANDS; ++j) sc[t][j] = 0.f;
#pragma unroll 2
      for (int d = 0; d < CB_HD; ++d) {
        const int ch = h * CB_HD + d;
        const float4 mk = s.fm[CB_DIM + ch], mq = s.fm[ch];
        const float nk = s.n0[CB_DIM + ch], nqv = s.n0[ch];
        float kd[CB_BANDS];
#pragma unroll
        for (int j = 0; j < CB_BANDS; ++j) kd[j] = fmaf(aff3(mk, x[3 * j], x[3 * j + 1], x[3 * j + 2]), rstd[j], nk);
#pragma unroll
        for (int t = 0; t < 3; ++t) {
          const int qt = qg * 3 + t;
          const float qv = fmaf(aff3(mq, x[3 * qt], x[3 * qt + 1], x[3 * qt + 2]), rstd[qt], nqv);
#pragma unroll
          for (int j = 0; j < CB_BANDS; ++j) sc[t][j] = fmaf(qv, kd[j], sc[t][j]);
        }
      }
#pragma unroll
      for (int t = 0; t < 3; ++t) {
        float mx = -INFINITY;
#pragma unroll
        for (int j = 0; j < CB_BANDS; ++j) {
          sc[t][j] *= 0.25f;
          mx = fmaxf(mx, sc[t][j]);
        }
        float den = 0.f;
#pragma unroll
        for (int j = 0; j < CB_BANDS; ++j) {
          sc[t][j] = expf(sc[t][j] - mx);
          den += sc[t][j];
        }
        const float inv = 1.0f / den;
#pragma unroll
        for (int j = 0; j < CB_BANDS; ++j) sc[t][j] *= inv;
      }
      __syncwarp();                                    // the previous group's out_proj reads of ctx are done
#pragma unroll 1
      for (int d4 = 0; d4 < CB_HD / 4; ++d4) {
        float cv[3][4];
#pragma unroll
        for (int dd = 0; dd < 4; ++dd) {
          const int ch = h * CB_HD + d4 * 4 + dd;
          const float4 mv = s.fm[2 * CB_DIM + ch];
          const float nv = s.n0[2 * CB_DIM + ch];
          float vd[CB_BANDS];
#pragma unroll
          for (int j = 0; j < CB_BANDS; ++j) vd[j] = fmaf(aff3(mv, x[3 * j], x[3 * j + 1], x[3 * j + 2]), rstd[j], nv);
#pragma unroll
          for (int t = 0; t < 3; ++t) {
            float a = 0.f;
#pragma unroll
            for (int j = 0; j < CB_BANDS; ++j) a = fmaf(sc[t][j], vd[j], a);
            cv[t][dd] = a;
          }
        }
#pragma unroll
        for (int t = 0; t < 3; ++t)
          *reinterpret_cast<float4*>(&ctx[px * 3 + t][h * CB_HD + d4 * 4]) = make_float4(cv[t][0], cv[t][1], cv[t][2], cv[t][3]);
      }
      __syncwarp();
      // out_proj + bias + band_proj residual for tokens 6 tb .. 6 tb + 5, channels 8 cb .. 8 cb + 7
      float acc[6][8];
      {
        const float4 o0 = *reinterpret_cast<const float4*>(&s.ob[cb * 8]), o1 = *reinterpret_cast<const float4*>(&s.ob[cb * 8 + 4]);
#pragma unroll
        for (int i = 0; i < 6; ++i) {
          acc[i][0] = o0.x; acc[i][1] = o0.y; acc[i][2] = o0.z; acc[i][3] = o0.w;
          acc[i][4] = o1.x; acc[i][5] = o1.y; acc[i][6] = o1.z; acc[i][7] = o1.w;
        }
      }
#pragma unroll 2
      for (int k4 = 0; k4 < CB_DIM / 4; ++k4) {
        float4 c4[6];
#pragma unroll
        for (int i = 0; i < 6; ++i) c4[i] = *reinterpret_cast<const float4*>(&ctx[tb * 6 + i][k4 * 4]);
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
          const float4 w0 = *reinterpret_cast<const float4*>(&s.wo[k4 * 4 + kk][cb * 8]);
          const float4 w1 = *reinterpret_cast<const float4*>(&s.wo[k4 * 4 + kk][cb * 8 + 4]);
#pragma unroll
          for (int i = 0; i < 6; ++i) {
            const float cvv = kk == 0 ? c4[i].x : kk == 1 ? c4[i].y : kk == 2 ? c4[i].z : c4[i].w;
            acc[i][0] = fmaf(cvv, w0.x, acc[i][0]); acc[i][1] = fmaf(cvv, w0.y, acc[i][1]);
            acc[i][2] = fmaf(cvv, w0.z, acc[i][2]); acc[i][3] = fmaf(cvv, w0.w, acc[i][3]);
            acc[i][4] = fmaf(cvv, w1.x, acc[i][4]); acc[i][5] = fmaf(cvv, w1.y, acc[i][5]);
            acc[i][6] = fmaf(cvv, w1.z, acc[i][6]); acc[i][7] = fmaf(cvv, w1.w, acc[i][7]);
          }
        }
      }
#pragma unroll
      for (int i = 0; i < 6; ++i) {
        const int tk = tb * 6 + i, pxo = tk / 3, qt = qg * 3 + tk % 3;
        const int po = p0 + pxo;
        if (po < HW && qt < nq) {
          const float x0 = xs[pxo][qt * 3], x1 = xs[pxo][qt * 3 + 1], x2 = xs[pxo][qt * 3 + 2];
          float r[8];
#pragma unroll
          for (int o = 0; o < 8; ++o) r[o] = acc[i][o] + aff3(s.pw[cb * 8 + o], x0, x1, x2);
          float4* dst = reinterpret_cast<float4*>(tok_out + (((long)b * nq + qt) * HW + po) * CB_DIM + cb * 8);
          dst[0] = make_float4(r[0], r[1], r[2], r[3]);
          dst[1] = make_float4(r[4], r[5], r[6], r[7]);
        }
      }
    }
    __syncwarp();                                      // xs / ctx are rewritten by the next tile
  }
}

extern "C" int ffsr_crossband_attention(const float* raw9, int B, int H, int W, const float* proj_w,
                                        const float* proj_b, const float* out_w, const float* out_b, int nq,
                                        float* tok_out, int num_sms, const float* fold, cudaStream_t stream) {
  FFSR_REQUIRE(raw9 && proj_w && proj_b && out_w && out_b && tok_out && fold, FFSR_ERR_ARG,
               "crossband_attention: null pointer");
  FFSR_REQUIRE(B > 0 && H > 0 && W > 0 && nq >= 1 && nq <= CB_BANDS, FFSR_ERR_ARG, "crossband_attention: bad shape");
  FFSR_REQUIRE(((uintptr_t)fold % 16) == 0 && ((uintptr_t)tok_out % 16) == 0, FFSR_ERR_ALIGN, "crossband_attention: fold / tok_out must be 16B aligned");
  const int HW = H * W;
  static bool attr_set = false;
  if (!attr_set) {
    cudaFuncSetAttribute(k_crossband_attn2<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(CB2Smem));
    cudaFuncSetAttribute(k_crossband_attn2<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(CB2Smem));
    attr_set = true;
  }
  const long wtiles = (long)B * ((HW + CB2_PX - 1) / CB2_PX);
  const long blocks = (wtiles + CB2_WARPS - 1) / CB2_WARPS;
  const int grid = (int)(blocks < 2L * num_sms ? blocks : 2L * num_sms);
  if (nq <= 3) k_crossband_attn2<1><<<grid, CB2_WARPS * 32, sizeof(CB2Smem), stream>>>(fold, raw9, B, HW, proj_w, proj_b, out_w, out_b, nq, tok_out);
  else k_crossband_attn2<3><<<grid, CB2_WARPS * 32, sizeof(CB2Smem), stream>>>(fold, raw9, B, HW, proj_w, proj_b, out_w, out_b, nq, tok_out);
  return ffsr_check_launch("crossband_attention");
}

// ------------------------------------------------------------------------------------
// Phase 3 tail: enhanced band = out_proj(x) + raw band; routing_lr = sum of bands 0..2.
// x: [B][nq][H][W][64] (after the LKA block); enh9/raw9: [B][9][3][H][W]; routing: [B][3][H][W]
// ------------------------------------------------------------------------------------
__global__ void k_cb_out(const float* __restrict__ x, const float* __restrict__ raw9, int B, int HW, int nq,
                         const float* __restrict__ w, const float* __restrict__ bias,
                         float* __restrict__ enh9, float* __restrict__ routing) {
  __shared__ float sw[3][CB_DIM];
  __shared__ float sb[3];
  for (int i = threadIdx.x; i < 3 * CB_DIM; i += blockDim.x) sw[i / CB_DIM][i % CB_DIM] = w[i];
  if (threadIdx.x < 3) sb[threadIdx.x] = bias[threadIdx.x];
  __syncthreads();
  const long gp = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (gp >= (long)B * HW) return;
  const int b = (int)(gp / HW), p = (int)(gp % HW);
  float r0 = 0.f, r1 = 0.f, r2 = 0.f;
  for (int band = 0; band < nq; ++band) {
    const float4* row = reinterpret_cast<const float4*>(x + (((long)b * nq + band) * HW + p) * CB_DIM);
    float a0 = sb[0], a1 = sb[1], a2 = sb[2];
#pragma unroll
    for (int c4 = 0; c4 < CB_DIM / 4; ++c4) {
      const float4 v = row[c4];
      a0 = fmaf(v.x, sw[0][4 * c4], a0); a0 = fmaf(v.y, sw[0][4 * c4 + 1], a0);
      a0 = fmaf(v.z, sw[0][4 * c4 + 2], a0); a0 = fmaf(v.w, sw[0][4 * c4 + 3], a0);
      a1 = fmaf(v.x, sw[1][4 * c4], a1); a1 = fmaf(v.y, sw[1][4 * c4 + 1], a1);
      a1 = fmaf(v.z, sw[1][4 * c4 + 2], a1); a1 = fmaf(v.w, sw[1][4 * c4 + 3], a1);
      a2 = fmaf(v.x, sw[2][4 * c4], a2); a2 = fmaf(v.y, sw[2][4 * c4 + 1], a2);
      a2 = fmaf(v.z, sw[2][4 * c4 + 2], a2); a2 = fmaf(v.w, sw[2][4 * c4 + 3], a2);
    }
    const long o = ((long)b * 9 + band) * 3 * HW + p;
    a0 += raw9[o]; a1 += raw9[o + HW]; a2 += raw9[o + 2 * (long)HW];
    enh9[o] = a0; enh9[o + HW] = a1; enh9[o + 2 * (long)HW] = a2;
    if (band == 0) { r0 = a0; r1 = a1; r2 = a2; }
    else if (band < 3) { r0 += a0; r1 += a1; r2 += a2; }
  }
  const long ro = (long)b * 3 * HW + p;
  routing[ro] = r0; routing[ro + HW] = r1; routing[ro + 2 * (long)HW] = r2;
}

extern "C" int ffsr_crossband_out(const float* x, const float* raw9, int B, int H, int W, int nq, const float* w,
                                  const float* bias, float* enh9, float* routing, cudaStream_t stream) {
  FFSR_REQUIRE(x && raw9 && w && bias && enh9 && routing, FFSR_ERR_ARG, "crossband_out: null pointer");
  FFSR_REQUIRE(nq >= 3 && nq <= 9, FFSR_ERR_ARG, "crossband_out: nq must be in [3,9]");
  FFSR_REQUIRE(((uintptr_t)x % 16) == 0, FFSR_ERR_ALIGN, "crossband_out: x must be 16B aligned");
  const long n = (long)B * H * W;
  k_cb_out<<<ceil_div(n, 128), 128, 0, stream>>>(x, raw9, B, H * W, nq, w, bias, enh9, routing);
  return ffsr_check_launch("crossband_out");
}

// ------------------------------------------------------------------------------------
// LayerNorm over the last dim (E in {64,128,256}): one warp per row.
// ------------------------------------------------------------------------------------
template <typename TO>
__global__ void k_layernorm_rows(const float* __restrict__ x, long rows, int E, const float* __restrict__ w,
                                 const float* __restrict__ b, TO* __restrict__ y) {
  const long row = (long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float* xr = x + row * E;
  float v[8];
  const int per = E / 32;   // 2, 4 or 8
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i)
    if (i < per) { v[i] = xr[lane + 32 * i]; sum += v[i]; }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  const float mean = sum / (float)E;
  float sq = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i)
    if (i < per) { v[i] -= mean; sq += v[i] * v[i]; }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
  const float rstd = rsqrtf(sq / (float)E + 1e-5f);
#pragma unroll
  for (int i = 0; i < 8; ++i)
    if (i < per) {
      const int c = lane + 32 * i;
      y[row * E + c] = from_f32<TO>(v[i] * rstd * w[c] + b[c]);
    }
}

extern "C" int ffsr_layernorm(const float* x, long rows, int E, const float* w, const float* b, void* y,
                              int out_bf16, cudaStream_t stream) {
  FFSR_REQUIRE(x && w && b && y, FFSR_ERR_ARG, "layernorm: null pointer");
  FFSR_REQUIRE(E % 32 == 0 && E >= 32 && E <= 256, FFSR_ERR_ARG, "layernorm: E must be a multiple of 32 in [32,256]");
  const int wpb = 8;
  if (out_bf16)
    k_layernorm_rows<__nv_bfloat16><<<ceil_div(rows, wpb), wpb * 32, 0, stream>>>(x, rows, E, w, b, (__nv_bfloat16*)y);
  else
    k_layernorm_rows<float><<<ceil_div(rows, wpb), wpb * 32, 0, stream>>>(x, rows, E, w, b, (float*)y);
  return ffsr_check_launch("layernorm");
}

// bf16 rows of 128 channels -> bf16 (Phase 4 in bf16 mode, where the residual stream is stored as bf16): one warp per row, one
// 8-byte load and store per lane, statistics in fp32.
__global__ void __launch_bounds__(256) k_layernorm128_bf16(const __nv_bfloat16* __restrict__ x, long rows, const float* __restrict__ w,
                                                           const float* __restrict__ b, __nv_bfloat16* __restrict__ y) {
  const long row = (long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const uint2 u = *reinterpret_cast<const uint2*>(x + row * 128 + lane * 4);
  const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.x));
  const float2 c = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.y));
  float v[4] = {a.x, a.y, c.x, c.y};
  float sum = (v[0] + v[1]) + (v[2] + v[3]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  const float mean = sum * (1.0f / 128.0f);
  float sq = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) { v[i] -= mean; sq = fmaf(v[i], v[i], sq); }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
  const float rstd = rsqrtf(sq * (1.0f / 128.0f) + 1e-5f);
  const float4 w4 = *reinterpret_cast<const float4*>(w + lane * 4), b4 = *reinterpret_cast<const float4*>(b + lane * 4);
  __nv_bfloat162 o0 = __floats2bfloat162_rn(fmaf(v[0] * rstd, w4.x, b4.x), fmaf(v[1] * rstd, w4.y, b4.y));
  __nv_bfloat162 o1 = __floats2bfloat162_rn(fmaf(v[2] * rstd, w4.z, b4.z), fmaf(v[3] * rstd, w4.w, b4.w));
  uint2 ou;
  ou.x = *reinterpret_cast<uint32_t*>(&o0);
  ou.y = *reinterpret_cast<uint32_t*>(&o1);
  *reinterpret_cast<uint2*>(y + row * 128 + lane * 4) = ou;
}

extern "C" int ffsr_layernorm128_bf16(const void* x, long rows, const float* w, const float* b, void* y, cudaStream_t stream) {
  FFSR_REQUIRE(x && w && b && y && rows > 0, FFSR_ERR_ARG, "layernorm128_bf16: bad argument");
  FFSR_REQUIRE(((uintptr_t)x % 8) == 0 && ((uintptr_t)y % 8) == 0 && ((uintptr_t)w % 16) == 0 && ((uintptr_t)b % 16) == 0, FFSR_ERR_ALIGN,
               "layernorm128_bf16: alignment");
  k_layernorm128_bf16<<<ceil_div(rows, 8), 256, 0, stream>>>((const __nv_bfloat16*)x, rows, w, b, (__nv_bfloat16*)y);
  return ffsr_check_launch("layernorm128_bf16");
}

// ------------------------------------------------------------------------------------
// Token attention core (Phase 4): softmax(q k^T / 4) v over the T tokens of each LR pixel.
// Token-major ("expert-major") layout: qkv[B][T][HW][3E] -> ctx[B][T][HW][E], head_dim 16.
// One thread per (b, pixel, query token, head); heads vary fastest so a warp reads
// contiguous 64-byte head slices.
// ------------------------------------------------------------------------------------
template <typename TI>
__device__ __forceinline__ void load16(const TI* p, float (&o)[16]);
template <>
__device__ __forceinline__ void load16<float>(const float* p, float (&o)[16]) {
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const float4 v = reinterpret_cast<const float4*>(p)[k];
    o[4 * k] = v.x; o[4 * k + 1] = v.y; o[4 * k + 2] = v.z; o[4 * k + 3] = v.w;
  }
}
template <>
__device__ __forceinline__ void load16<__nv_bfloat16>(const __nv_bfloat16* p, float (&o)[16]) {
  const uint4 u0 = reinterpret_cast<const uint4*>(p)[0], u1 = reinterpret_cast<const uint4*>(p)[1];
  const uint32_t w[8] = {u0.x, u0.y, u0.z, u0.w, u1.x, u1.y, u1.z, u1.w};
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const float2 f2 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w[k]));
    o[2 * k] = f2.x; o[2 * k + 1] = f2.y;
  }
}
template <typename TO>
__device__ __forceinline__ void store16(TO* p, const float (&o)[16]);
template <>
__device__ __forceinline__ void store16<float>(float* p, const float (&o)[16]) {
#pragma unroll
  for (int k = 0; k < 4; ++k) reinterpret_cast<float4*>(p)[k] = make_float4(o[4 * k], o[4 * k + 1], o[4 * k + 2], o[4 * k + 3]);
}
template <>
__device__ __forceinline__ void store16<__nv_bfloat16>(__nv_bfloat16* p, const float (&o)[16]) {
  uint32_t w[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    __nv_bfloat162 h = __floats2bfloat162_rn(o[2 * k], o[2 * k + 1]);
    w[k] = *reinterpret_cast<uint32_t*>(&h);
  }
  reinterpret_cast<uint4*>(p)[0] = make_uint4(w[0], w[1], w[2], w[3]);
  reinterpret_cast<uint4*>(p)[1] = make_uint4(w[4], w[5], w[6], w[7]);
}

template <typename TI, typename TO, int T>
__global__ void k_token_attention(const TI* __restrict__ qkv, int B, long HW, int E, TO* __restrict__ ctx) {
  const int heads = E / 16;
  const long it = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (it >= (long)B * HW * T * heads) return;
  const int h = (int)(it % heads);
  long rest = it / heads;
  const int qt = (int)(rest % T);
  rest /= T;
  const long p = rest % HW;
  const int b = (int)(rest / HW);
  const long tstride = HW * 3 * E;                       // between tokens of one pixel
  const TI* base = qkv + ((long)b * T * HW + p) * 3 * E + h * 16;
  float q[16];
  load16<TI>(base + qt * tstride, q);
  float sc[T];
  float mx = -INFINITY;
#pragma unroll
  for (int j = 0; j < T; ++j) {
    float kk[16];
    load16<TI>(base + j * tstride + E, kk);
    float a = 0.f;
#pragma unroll
    for (int d = 0; d < 16; ++d) a = fmaf(q[d], kk[d], a);
    sc[j] = a * 0.25f;
    mx = fmaxf(mx, sc[j]);
  }
  float den = 0.f;
#pragma unroll
  for (int j = 0; j < T; ++j) { sc[j] = expf(sc[j] - mx); den += sc[j]; }
  const float inv = 1.0f / den;
  float o[16];
#pragma unroll
  for (int d = 0; d < 16; ++d) o[d] = 0.f;
#pragma unroll
  for (int j = 0; j < T; ++j) {
    float vv[16];
    load16<TI>(base + j * tstride + 2 * E, vv);
    const float pj = sc[j] * inv;
#pragma unroll
    for (int d = 0; d < 16; ++d) o[d] = fmaf(pj, vv[d], o[d]);
  }
  store16<TO>(ctx + (((long)b * T + qt) * HW + p) * E + h * 16, o);
}

extern "C" int ffsr_token_attention(const void* qkv, int B, int T, long HW, int E, void* ctx, int is_bf16,
                                    cudaStream_t stream) {
  FFSR_REQUIRE(qkv && ctx, FFSR_ERR_ARG, "token_attention: null pointer");
  FFSR_REQUIRE(T == 4 && E % 16 == 0 && B > 0 && HW > 0, FFSR_ERR_ARG, "token_attention: built for T=4 tokens, E%%16==0");
  FFSR_REQUIRE(((uintptr_t)qkv % 16) == 0 && ((uintptr_t)ctx % 16) == 0, FFSR_ERR_ALIGN, "token_attention: 16B alignment");
  const long n = (long)B * HW * T * (E / 16);
  if (is_bf16)
    k_token_attention<__nv_bfloat16, __nv_bfloat16, 4><<<ceil_div(n, 128), 128, 0, stream>>>(
        (const __nv_bfloat16*)qkv, B, HW, E, (__nv_bfloat16*)ctx);
  else
    k_token_attention<float, float, 4><<<ceil_div(n, 128), 128, 0, stream>>>((const float*)qkv, B, HW, E, (float*)ctx);
  return ffsr_check_launch("token_attention");
}

// ------------------------------------------------------------------------------------
// Phase 6: gates = sigmoid(T*(raw - (0.7 - 0.5 d))) / max(sum + 1e-8, 0.3)
// raw: [B][H][W][4] (NHWC), diff: [B][1][H][W]; gates out: [B][4][H][W] planar.
// ------------------------------------------------------------------------------------
__global__ void k_gate_finalize(const float* __restrict__ raw, const float* __restrict__ diff, int B, int HW,
                                const float* __restrict__ temperature, float* __restrict__ gates) {
  const long gp = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (gp >= (long)B * HW) return;
  const int b = (int)(gp / HW), p = (int)(gp % HW);
  const float4 r = *reinterpret_cast<const float4*>(raw + gp * 4);
  const float thr = 0.7f - 0.5f * diff[gp];
  const float T = temperature[0];
  float g0 = sigmoid_acc(T * (r.x - thr)), g1 = sigmoid_acc(T * (r.y - thr));
  float g2 = sigmoid_acc(T * (r.z - thr)), g3 = sigmoid_acc(T * (r.w - thr));
  const float s = fmaxf(((g0 + g1) + g2) + g3 + 1e-8f, 0.3f);
  float* o = gates + (long)b * 4 * HW + p;
  o[0] = g0 / s; o[HW] = g1 / s; o[2 * (long)HW] = g2 / s; o[3 * (long)HW] = g3 / s;
}

extern "C" int ffsr_gate_finalize(const float* raw, const float* diff, int B, int H, int W,
                                  const float* temperature, float* gates, cudaStream_t stream) {
  FFSR_REQUIRE(raw && diff && temperature && gates, FFSR_ERR_ARG, "gate_finalize: null pointer");
  const long n = (long)B * H * W;
  k_gate_finalize<<<ceil_div(n, 256), 256, 0, stream>>>(raw, diff, B, H * W, temperature, gates);
  return ffsr_check_launch("gate_finalize");
}
