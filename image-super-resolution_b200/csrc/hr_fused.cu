// HR-side fused elementwise / resampling kernels (all HBM-bound; one thread per pixel or
// per pixel x 4-channel group, coalesced planar reads, channels-last vector writes).
// Each kernel cites the reference op sequence it replaces in include/ffsr_b200.h.
#include <type_traits>
#include "common.cuh"
#include "../../include/ffsr_b200.h"

namespace {
struct Img4 {
  const float* p[4];
};

template <typename T>
__device__ __forceinline__ void store_vec4(T* dst, float a, float b, float c, float d);
template <>
__device__ __forceinline__ void store_vec4<float>(float* dst, float a, float b, float c, float d) {
  *reinterpret_cast<float4*>(dst) = make_float4(a, b, c, d);
}
template <>
__device__ __forceinline__ void store_vec4<__nv_bfloat16>(__nv_bfloat16* dst, float a, float b, float c, float d) {
  __nv_bfloat162 lo = __floats2bfloat162_rn(a, b), hi = __floats2bfloat162_rn(c, d);
  uint2 u;
  u.x = *reinterpret_cast<uint32_t*>(&lo);
  u.y = *reinterpret_cast<uint32_t*>(&hi);
  *reinterpret_cast<uint2*>(dst) = u;
}
template <typename T>
__device__ __forceinline__ float4 load_vec4(const T* src);
template <>
__device__ __forceinline__ float4 load_vec4<float>(const float* src) {
  return *reinterpret_cast<const float4*>(src);
}
template <>
__device__ __forceinline__ float4 load_vec4<__nv_bfloat16>(const __nv_bfloat16* src) {
  const uint2 u = *reinterpret_cast<const uint2*>(src);
  const __nv_bfloat162 lo = *reinterpret_cast<const __nv_bfloat162*>(&u.x);
  const __nv_bfloat162 hi = *reinterpret_cast<const __nv_bfloat162*>(&u.y);
  const float2 a = __bfloat1622float2(lo), b = __bfloat1622float2(hi);
  return make_float4(a.x, a.y, b.x, b.y);
}
}  // namespace

// ------------------------------------------------------------------------------------------
// Phase 4 tail (modulation heads at HR)
// ------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(128) k_modulate_hr(Img4 imgs, const float* __restrict__ m32,
                                                     const float* __restrict__ w2, const float* __restrict__ b2,
                                                     int B, int H, int W, int mh, int mw, int clamp01,
                                                     float* __restrict__ ecol, T* __restrict__ cat3, long long cat3_sX) {
  __shared__ float sw[4][3][32];
  __shared__ float sb[4][3];
  if (m32) {
    for (int i = threadIdx.x; i < 384; i += blockDim.x) (&sw[0][0][0])[i] = w2[i];
    if (threadIdx.x < 12) (&sb[0][0])[threadIdx.x] = b2[threadIdx.x];
  }
  __syncthreads();
  const int Hh = 4 * H, Wh = 4 * W;
  const int X = blockIdx.x * blockDim.x + threadIdx.x;
  const int Y = blockIdx.y, b = blockIdx.z;
  if (X >= Wh) return;
  const long HWh = (long)Hh * Wh;
  const long pix = (long)Y * Wh + X;
  const BilinTap ty = bilin_tap(Y, mh, Hh), tx = bilin_tap(X, mw, Wh);      // m32 lives on an mh x mw grid (usually the LR grid)
  constexpr bool FAST = !std::is_same<T, float>::value;      // bf16 mode: A&S erf (1.5e-7), results are rounded to bf16
  float o[12];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    float mod[3] = {0.f, 0.f, 0.f};
    if (m32) {
      const float* base = m32 + ((long)(b * 4 + e) * mh) * mw * 32;
      const float4* p00 = reinterpret_cast<const float4*>(base + ((long)ty.i0 * mw + tx.i0) * 32);
      const float4* p01 = reinterpret_cast<const float4*>(base + ((long)ty.i0 * mw + tx.i1) * 32);
      const float4* p10 = reinterpret_cast<const float4*>(base + ((long)ty.i1 * mw + tx.i0) * 32);
      const float4* p11 = reinterpret_cast<const float4*>(base + ((long)ty.i1 * mw + tx.i1) * 32);
      mod[0] = sb[e][0]; mod[1] = sb[e][1]; mod[2] = sb[e][2];
#pragma unroll
      for (int c4 = 0; c4 < 8; ++c4) {
        const float4 a = p00[c4], bq = p01[c4], c = p10[c4], d = p11[c4];
        float g[4];
        g[0] = gelu_sel<FAST>(ty.w0 * (tx.w0 * a.x + tx.w1 * bq.x) + ty.w1 * (tx.w0 * c.x + tx.w1 * d.x));
        g[1] = gelu_sel<FAST>(ty.w0 * (tx.w0 * a.y + tx.w1 * bq.y) + ty.w1 * (tx.w0 * c.y + tx.w1 * d.y));
        g[2] = gelu_sel<FAST>(ty.w0 * (tx.w0 * a.z + tx.w1 * bq.z) + ty.w1 * (tx.w0 * c.z + tx.w1 * d.z));
        g[3] = gelu_sel<FAST>(ty.w0 * (tx.w0 * a.w + tx.w1 * bq.w) + ty.w1 * (tx.w0 * c.w + tx.w1 * d.w));
#pragma unroll
        for (int k = 0; k < 3; ++k)
#pragma unroll
          for (int i = 0; i < 4; ++i) mod[k] = fmaf(sw[e][k][4 * c4 + i], g[i], mod[k]);
      }
    }
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
      float v = imgs.p[e][((long)b * 3 + ch) * HWh + pix];
      if (m32) {
        v = v * (1.0f + 0.2f * (sigmoid_acc(mod[ch]) - 0.5f));
        if (clamp01) v = fminf(fmaxf(v, 0.f), 1.f);
      }
      o[e * 3 + ch] = v;
      ecol[((long)(b * 4 + e) * 3 + ch) * HWh + pix] = v;
    }
  }
  if (cat3) {
    T* dst = cat3 + ((long)b * HWh + pix) * cat3_sX;
    store_vec4<T>(dst, o[0], o[1], o[2], o[3]);
    store_vec4<T>(dst + 4, o[4], o[5], o[6], o[7]);
    store_vec4<T>(dst + 8, o[8], o[9], o[10], o[11]);
  }
}

static int modulate_hr_impl(const float* const* imgs, const float* m32, int mh, int mw, const float* w2, const float* b2,
                            int B, int H, int W, int clamp01, float* ecol, void* cat3, long long cat3_sX, int cat3_dtype,
                            cudaStream_t stream);

extern "C" int ffsr_modulate_hr(const float* const* imgs, const float* m32, const float* w2, const float* b2, int B,
                                int H, int W, int clamp01, float* ecol, void* cat3, long long cat3_sX, int cat3_dtype,
                                cudaStream_t stream) {
  return modulate_hr_impl(imgs, m32, H, W, w2, b2, B, H, W, clamp01, ecol, cat3, cat3_sX, cat3_dtype, stream);
}
// m32 on its own mh x mw grid (expert features cached at a resolution other than LR: large_kernel_attention.py:365-372, 410-414)
extern "C" int ffsr_modulate_hr_sized(const float* const* imgs, const float* m32, int mh, int mw, const float* w2,
                                      const float* b2, int B, int H, int W, int clamp01, float* ecol, void* cat3,
                                      long long cat3_sX, int cat3_dtype, cudaStream_t stream) {
  FFSR_REQUIRE(mh > 0 && mw > 0, FFSR_ERR_ARG, "modulate_hr_sized: bad feature grid");
  return modulate_hr_impl(imgs, m32, mh, mw, w2, b2, B, H, W, clamp01, ecol, cat3, cat3_sX, cat3_dtype, stream);
}

static int modulate_hr_impl(const float* const* imgs, const float* m32, int mh, int mw, const float* w2, const float* b2,
                            int B, int H, int W, int clamp01, float* ecol, void* cat3, long long cat3_sX, int cat3_dtype,
                            cudaStream_t stream) {
  FFSR_REQUIRE(imgs && imgs[0] && imgs[1] && imgs[2] && imgs[3] && ecol, FFSR_ERR_ARG, "modulate_hr: null pointer");
  FFSR_REQUIRE(!m32 || (w2 && b2), FFSR_ERR_ARG, "modulate_hr: modulation weights missing");
  FFSR_REQUIRE(B > 0 && B <= 65535 && H > 0 && W > 0 && 4 * H <= 65535, FFSR_ERR_ARG, "modulate_hr: bad shape");
  const int esz = cat3_dtype == FFSR_DT_BF16 ? 2 : 4;
  FFSR_REQUIRE(!cat3 || (((uintptr_t)cat3 % 16) == 0 && (cat3_sX * esz) % 16 == 0 && cat3_sX >= 12), FFSR_ERR_ALIGN,
               "modulate_hr: concat slice must be 16B aligned with a 16B-multiple pixel stride");
  FFSR_REQUIRE(!m32 || ((uintptr_t)m32 % 16) == 0, FFSR_ERR_ALIGN, "modulate_hr: m32 must be 16B aligned");
  Img4 im;
  for (int e = 0; e < 4; ++e) im.p[e] = imgs[e];
  dim3 grid(ceil_div(4 * W, 128), 4 * H, B);
  if (cat3_dtype == FFSR_DT_BF16)
    k_modulate_hr<__nv_bfloat16><<<grid, 128, 0, stream>>>(im, m32, w2, b2, B, H, W, mh, mw, clamp01, ecol, (__nv_bfloat16*)cat3, cat3_sX);
  else
    k_modulate_hr<float><<<grid, 128, 0, stream>>>(im, m32, w2, b2, B, H, W, mh, mw, clamp01, ecol, (float*)cat3, cat3_sX);
  return ffsr_check_launch("modulate_hr");
}

// v2: one thread = the four HR pixels 4k+2 .. 4k+5 of one row (they share the LR taps k, k+1 with x-weights 1/8, 3/8, 5/8,
// 7/8) x all four experts.  The v1 kernel above is bound by its loads and its erf: one thread per HR pixel issues 128 sixteen-
// byte loads, each of a different 128-byte line than its neighbours', for 128 GELUs.  Here the four taps are loaded once per
// four pixels (8x fewer load instructions per pixel with bf16 features), the vertical blend is shared by the four pixels, and the
// bf16 mode uses the tanh-form GELU (the result only feeds a sigmoid that is damped by 0.2).
template <typename TM>
struct ModLoad;
template <>
struct ModLoad<float> {
  static constexpr int CH = 4;
  __device__ static __forceinline__ void ld(const float* p, float (&f)[4]) {
    const float4 v = *reinterpret_cast<const float4*>(p);
    f[0] = v.x; f[1] = v.y; f[2] = v.z; f[3] = v.w;
  }
};
template <>
struct ModLoad<__nv_bfloat16> {
  static constexpr int CH = 8;
  __device__ static __forceinline__ void ld(const __nv_bfloat16* p, float (&f)[8]) {
    const uint4 u = *reinterpret_cast<const uint4*>(p);
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float2 f2 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w[k]));
      f[2 * k] = f2.x; f[2 * k + 1] = f2.y;
    }
  }
};

template <typename TM, typename T, bool FAST>
__global__ void __launch_bounds__(128) k_modulate_hr4(Img4 imgs, const TM* __restrict__ m32, const float* __restrict__ w2,
                                                      const float* __restrict__ b2, int B, int H, int W, int clamp01,
                                                      float* __restrict__ ecol, T* __restrict__ cat3, long long cat3_sX) {
  __shared__ float sw[4][3][32];
  __shared__ float sb[4][3];
  for (int i = threadIdx.x; i < 384; i += blockDim.x) (&sw[0][0][0])[i] = w2[i];
  if (threadIdx.x < 12) (&sb[0][0])[threadIdx.x] = b2[threadIdx.x];
  __syncthreads();
  const int Hh = 4 * H, Wh = 4 * W;
  const int k = blockIdx.x * blockDim.x + threadIdx.x - 1;       // LR column of the left tap: -1 .. W-1
  const int Y = blockIdx.y, b = blockIdx.z;
  if (k > W - 1) return;
  const int x0 = 4 * k + 2;                                      // HR column of pixel 0 (pixels 0,1 exist iff k >= 0; 2,3 iff k <= W-2)
  const int i0 = k < 0 ? 0 : k, i1 = k + 1 > W - 1 ? W - 1 : k + 1;
  const BilinTap ty = bilin_tap(Y, H, Hh);
  constexpr int CH = ModLoad<TM>::CH;
  float mod[4][12];
#pragma unroll
  for (int j = 0; j < 4; ++j)
#pragma unroll
    for (int q = 0; q < 12; ++q) mod[j][q] = sb[q / 3][q % 3];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const TM* base = m32 + ((long)(b * 4 + e) * H) * W * 32;
    const TM* p00 = base + ((long)ty.i0 * W + i0) * 32;
    const TM* p01 = base + ((long)ty.i0 * W + i1) * 32;
    const TM* p10 = base + ((long)ty.i1 * W + i0) * 32;
    const TM* p11 = base + ((long)ty.i1 * W + i1) * 32;
#pragma unroll 2
    for (int c = 0; c < 32; c += CH) {
      float a[CH], bq[CH], cc[CH], d[CH];
      ModLoad<TM>::ld(p00 + c, a);
      ModLoad<TM>::ld(p01 + c, bq);
      ModLoad<TM>::ld(p10 + c, cc);
      ModLoad<TM>::ld(p11 + c, d);
#pragma unroll
      for (int i = 0; i < CH; ++i) {
        const float l = ty.w0 * a[i] + ty.w1 * cc[i];            // vertical blend of the left / right tap column
        const float r = ty.w0 * bq[i] + ty.w1 * d[i];
        const float dlr = r - l;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float g = gelu_sel<FAST>(fmaf(0.125f + 0.25f * (float)j, dlr, l));
#pragma unroll
          for (int q = 0; q < 3; ++q) mod[j][e * 3 + q] = fmaf(sw[e][q][c + i], g, mod[j][e * 3 + q]);
        }
      }
    }
  }
  const long HWh = (long)Hh * Wh;
#pragma unroll
  for (int half = 0; half < 2; ++half) {
    if (half == 0 ? (k < 0) : (k > W - 2)) continue;
    const int X = x0 + 2 * half;
    const long pix = (long)Y * Wh + X;
    float o[2][12];
#pragma unroll
    for (int q = 0; q < 12; ++q) {
      const long off = ((long)(b * 4 + q / 3) * 3 + q % 3) * HWh + pix;
      const float2 v = *reinterpret_cast<const float2*>(imgs.p[q / 3] + ((long)b * 3 + q % 3) * HWh + pix);
      float v0 = v.x * (1.0f + 0.2f * (sigmoid_acc(mod[2 * half][q]) - 0.5f));
      float v1 = v.y * (1.0f + 0.2f * (sigmoid_acc(mod[2 * half + 1][q]) - 0.5f));
      if (clamp01) { v0 = fminf(fmaxf(v0, 0.f), 1.f); v1 = fminf(fmaxf(v1, 0.f), 1.f); }
      o[0][q] = v0; o[1][q] = v1;
      *reinterpret_cast<float2*>(ecol + off) = make_float2(v0, v1);
    }
    if (cat3) {
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        T* dst = cat3 + ((long)b * HWh + pix + j) * cat3_sX;
        store_vec4<T>(dst, o[j][0], o[j][1], o[j][2], o[j][3]);
        store_vec4<T>(dst + 4, o[j][4], o[j][5], o[j][6], o[j][7]);
        store_vec4<T>(dst + 8, o[j][8], o[j][9], o[j][10], o[j][11]);
      }
    }
  }
}

extern "C" int ffsr_modulate_hr_v2(const float* const* imgs, const void* m32, int m32_dtype, const float* w2, const float* b2,
                                   int B, int H, int W, int clamp01, float* ecol, void* cat3, long long cat3_sX,
                                   int cat3_dtype, cudaStream_t stream) {
  FFSR_REQUIRE(imgs && imgs[0] && imgs[1] && imgs[2] && imgs[3] && ecol && m32 && w2 && b2, FFSR_ERR_ARG, "modulate_hr_v2: null pointer");
  FFSR_REQUIRE(B > 0 && B <= 65535 && H > 0 && W > 0 && 4 * H <= 65535, FFSR_ERR_ARG, "modulate_hr_v2: bad shape");
  FFSR_REQUIRE(m32_dtype == FFSR_DT_F32 || (m32_dtype == FFSR_DT_BF16 && cat3_dtype == FFSR_DT_BF16), FFSR_ERR_ARG,
               "modulate_hr_v2: bf16 features belong to the bf16 mode (bf16 concat slice)");
  const int esz = cat3_dtype == FFSR_DT_BF16 ? 2 : 4;
  FFSR_REQUIRE(!cat3 || (((uintptr_t)cat3 % 16) == 0 && (cat3_sX * esz) % 16 == 0 && cat3_sX >= 12), FFSR_ERR_ALIGN,
               "modulate_hr_v2: concat slice must be 16B aligned with a 16B-multiple pixel stride");
  FFSR_REQUIRE(((uintptr_t)m32 % 16) == 0 && ((uintptr_t)ecol % 8) == 0, FFSR_ERR_ALIGN, "modulate_hr_v2: m32 must be 16B aligned");
  for (int e = 0; e < 4; ++e) FFSR_REQUIRE(((uintptr_t)imgs[e] % 8) == 0, FFSR_ERR_ALIGN, "modulate_hr_v2: expert images must be 8B aligned");
  Img4 im;
  for (int e = 0; e < 4; ++e) im.p[e] = imgs[e];
  dim3 grid(ceil_div(W + 1, 128), 4 * H, B);
  if (m32_dtype == FFSR_DT_BF16)
    k_modulate_hr4<__nv_bfloat16, __nv_bfloat16, true><<<grid, 128, 0, stream>>>(im, (const __nv_bfloat16*)m32, w2, b2, B, H, W, clamp01, ecol, (__nv_bfloat16*)cat3, cat3_sX);
  else if (cat3_dtype == FFSR_DT_BF16)
    k_modulate_hr4<float, __nv_bfloat16, true><<<grid, 128, 0, stream>>>(im, (const float*)m32, w2, b2, B, H, W, clamp01, ecol, (__nv_bfloat16*)cat3, cat3_sX);
  else
    k_modulate_hr4<float, float, false><<<grid, 128, 0, stream>>>(im, (const float*)m32, w2, b2, B, H, W, clamp01, ecol, (float*)cat3, cat3_sX);
  return ffsr_check_launch("modulate_hr_v2");
}

// ------------------------------------------------------------------------------------------
// /2 and /4 bilinear (exact 2-tap averages) of the 12-channel expert stack
// ------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(128) k_expert_downsample(const float* __restrict__ ecol, int B, int H, int W,
                                                           T* __restrict__ cat2, long long cat2_sX,
                                                           T* __restrict__ s1in, long long s1_sX) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y, b = blockIdx.z;
  if (x >= W) return;
  const int Wh = 4 * W;
  const long HWh = 16L * H * W;
  float d2[4][12];   // the 2x2 half-res outputs of this LR pixel
  float d4[12];
#pragma unroll
  for (int k = 0; k < 12; ++k) {
    const float* pl = ecol + ((long)b * 12 + k) * HWh + (long)(4 * y) * Wh + 4 * x;
    const float4 r0 = *reinterpret_cast<const float4*>(pl);
    const float4 r1 = *reinterpret_cast<const float4*>(pl + Wh);
    const float4 r2 = *reinterpret_cast<const float4*>(pl + 2 * Wh);
    const float4 r3 = *reinterpret_cast<const float4*>(pl + 3 * Wh);
    d2[0][k] = 0.5f * (0.5f * r0.x + 0.5f * r0.y) + 0.5f * (0.5f * r1.x + 0.5f * r1.y);
    d2[1][k] = 0.5f * (0.5f * r0.z + 0.5f * r0.w) + 0.5f * (0.5f * r1.z + 0.5f * r1.w);
    d2[2][k] = 0.5f * (0.5f * r2.x + 0.5f * r2.y) + 0.5f * (0.5f * r3.x + 0.5f * r3.y);
    d2[3][k] = 0.5f * (0.5f * r2.z + 0.5f * r2.w) + 0.5f * (0.5f * r3.z + 0.5f * r3.w);
    d4[k] = 0.5f * (0.5f * r1.y + 0.5f * r1.z) + 0.5f * (0.5f * r2.y + 0.5f * r2.z);   // centre 2x2
  }
  const int W2 = 2 * W;
#pragma unroll
  for (int s = 0; s < 4; ++s) {
    const long pix = ((long)b * 2 * H + 2 * y + (s >> 1)) * W2 + 2 * x + (s & 1);
    T* dst = cat2 + pix * cat2_sX;
    store_vec4<T>(dst, d2[s][0], d2[s][1], d2[s][2], d2[s][3]);
    store_vec4<T>(dst + 4, d2[s][4], d2[s][5], d2[s][6], d2[s][7]);
    store_vec4<T>(dst + 8, d2[s][8], d2[s][9], d2[s][10], d2[s][11]);
  }
  T* dst = s1in + (((long)b * H + y) * W + x) * s1_sX;
  store_vec4<T>(dst, d4[0], d4[1], d4[2], d4[3]);
  store_vec4<T>(dst + 4, d4[4], d4[5], d4[6], d4[7]);
  store_vec4<T>(dst + 8, d4[8], d4[9], d4[10], d4[11]);
}

extern "C" int ffsr_expert_downsample(const float* ecol, int B, int Hh, int Wh, void* cat2, long long cat2_sX,
                                      void* s1in, long long s1_sX, int dtype, cudaStream_t stream) {
  FFSR_REQUIRE(ecol && cat2 && s1in, FFSR_ERR_ARG, "expert_downsample: null pointer");
  FFSR_REQUIRE(Hh % 4 == 0 && Wh % 4 == 0 && Hh > 0 && Wh > 0, FFSR_ERR_ARG, "expert_downsample: HR size must be 4x LR");
  const int esz = dtype == FFSR_DT_BF16 ? 2 : 4;
  FFSR_REQUIRE(((uintptr_t)cat2 % 16) == 0 && ((uintptr_t)s1in % 16) == 0 && (cat2_sX * esz) % 16 == 0 &&
                   (s1_sX * esz) % 16 == 0 && ((uintptr_t)ecol % 16) == 0,
               FFSR_ERR_ALIGN, "expert_downsample: 16B alignment required");
  const int H = Hh / 4, W = Wh / 4;
  dim3 grid(ceil_div(W, 128), H, B);
  if (dtype == FFSR_DT_BF16)
    k_expert_downsample<__nv_bfloat16><<<grid, 128, 0, stream>>>(ecol, B, H, W, (__nv_bfloat16*)cat2, cat2_sX, (__nv_bfloat16*)s1in, s1_sX);
  else
    k_expert_downsample<float><<<grid, 128, 0, stream>>>(ecol, B, H, W, (float*)cat2, cat2_sX, (float*)s1in, s1_sX);
  return ffsr_check_launch("expert_downsample");
}

// ------------------------------------------------------------------------------------------
// generic bilinear resize of a channels-last tensor into a channel slice
// ------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) k_resize_nhwc(const T* __restrict__ src, int h, int w, int C4, long long src_sX,
                                                     T* __restrict__ dst, int H, int W, long long dst_sX, long total) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int c4 = (int)(i % C4);
  const long pix = i / C4;
  const int X = (int)(pix % W), Y = (int)((pix / W) % H);
  const long n = pix / ((long)W * H);
  const BilinTap ty = bilin_tap(Y, h, H), tx = bilin_tap(X, w, W);
  const T* base = src + n * h * w * src_sX + 4 * c4;
  const float4 a = load_vec4<T>(base + ((long)ty.i0 * w + tx.i0) * src_sX);
  const float4 b = load_vec4<T>(base + ((long)ty.i0 * w + tx.i1) * src_sX);
  const float4 c = load_vec4<T>(base + ((long)ty.i1 * w + tx.i0) * src_sX);
  const float4 d = load_vec4<T>(base + ((long)ty.i1 * w + tx.i1) * src_sX);
  store_vec4<T>(dst + pix * dst_sX + 4 * c4,
                ty.w0 * (tx.w0 * a.x + tx.w1 * b.x) + ty.w1 * (tx.w0 * c.x + tx.w1 * d.x),
                ty.w0 * (tx.w0 * a.y + tx.w1 * b.y) + ty.w1 * (tx.w0 * c.y + tx.w1 * d.y),
                ty.w0 * (tx.w0 * a.z + tx.w1 * b.z) + ty.w1 * (tx.w0 * c.z + tx.w1 * d.z),
                ty.w0 * (tx.w0 * a.w + tx.w1 * b.w) + ty.w1 * (tx.w0 * c.w + tx.w1 * d.w));
}

// bf16, 8 channels (16 bytes) per thread, row-structured grid (x = W*C8 items, y = output row, z = image)
__global__ void __launch_bounds__(256) k_resize_nhwc_bf16x8(const __nv_bfloat16* __restrict__ src, int h, int w, int C8,
                                                            long long src_sX, __nv_bfloat16* __restrict__ dst, int H, int W,
                                                            long long dst_sX) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const int X = t / C8, c8 = t - X * C8;
  const int Y = blockIdx.y, n = blockIdx.z;
  if (X >= W) return;
  const BilinTap ty = bilin_tap(Y, h, H), tx = bilin_tap(X, w, W);
  const __nv_bfloat16* base = src + (long)n * h * w * src_sX + 8 * c8;
  const uint4 a = *reinterpret_cast<const uint4*>(base + ((long)ty.i0 * w + tx.i0) * src_sX);
  const uint4 b = *reinterpret_cast<const uint4*>(base + ((long)ty.i0 * w + tx.i1) * src_sX);
  const uint4 c = *reinterpret_cast<const uint4*>(base + ((long)ty.i1 * w + tx.i0) * src_sX);
  const uint4 d = *reinterpret_cast<const uint4*>(base + ((long)ty.i1 * w + tx.i1) * src_sX);
  const uint32_t* pa = &a.x; const uint32_t* pb = &b.x; const uint32_t* pc = &c.x; const uint32_t* pd = &d.x;
  uint32_t o[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const float2 fa = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(pa + k));
    const float2 fb = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(pb + k));
    const float2 fc = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(pc + k));
    const float2 fd = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(pd + k));
    // same association as the 4-channel kernel: ty.w0*(tx.w0*a + tx.w1*b) + ty.w1*(tx.w0*c + tx.w1*d)
    const float r0 = ty.w0 * (tx.w0 * fa.x + tx.w1 * fb.x) + ty.w1 * (tx.w0 * fc.x + tx.w1 * fd.x);
    const float r1 = ty.w0 * (tx.w0 * fa.y + tx.w1 * fb.y) + ty.w1 * (tx.w0 * fc.y + tx.w1 * fd.y);
    __nv_bfloat162 hh = __floats2bfloat162_rn(r0, r1);
    o[k] = *reinterpret_cast<uint32_t*>(&hh);
  }
  *reinterpret_cast<uint4*>(dst + (((long)n * H + Y) * W + X) * dst_sX + 8 * c8) = make_uint4(o[0], o[1], o[2], o[3]);
}

// ------------------------------------------------------------------------------------------
// Bilinear upsampling by an INTEGER factor F (2 or 4; align_corners = False), bf16 channels-last, optionally of
// o * attn (edge refiners) scaled by the softmax level weight.  A thread owns one SOURCE cell and 8 channels: it loads the
// 3x3 clamped neighbourhood once (9 x 16 bytes) and writes the F x F output pixels of the cell (F = 4: 0.56 loads per output
// instead of 4, and the taps are compile-time constants).  With scale = 1/F the reference's tap arithmetic
// src = (dst + 0.5) / F - 0.5 is exact in fp32, so the weights and the association ty.w0*(tx.w0*a + tx.w1*b) + ty.w1*(...)
// below are those of bilin_tap / k_resize_nhwc_bf16x8 / k_edge_attn_up_bf16x8.
// ------------------------------------------------------------------------------------------
template <int F, bool ATTN>
__global__ void __launch_bounds__(256) k_upsample_int(const __nv_bfloat16* __restrict__ src, const float* __restrict__ attn, int h, int w,
                                                      int C8, long long src_sX, const float* __restrict__ level_w, int level,
                                                      __nv_bfloat16* __restrict__ dst, long long dst_sX) {
  __shared__ float s_lw;
  if (ATTN) {
    if (threadIdx.x == 0) {
      const float l0 = level_w[0], l1 = level_w[1], l2 = level_w[2];
      const float m = fmaxf(l0, fmaxf(l1, l2));
      const float e0 = expf(l0 - m), e1 = expf(l1 - m), e2 = expf(l2 - m);
      s_lw = (level == 0 ? e0 : (level == 1 ? e1 : e2)) / ((e0 + e1) + e2);
    }
    __syncthreads();
  }
  const int t = blockIdx.x * blockDim.x + threadIdx.x;       // over w * C8
  const int j = t / C8, c8 = t - j * C8;
  const int i = blockIdx.y, n = blockIdx.z;
  if (j >= w) return;
  const int ys[3] = {max(i - 1, 0), i, min(i + 1, h - 1)};
  const int xs[3] = {max(j - 1, 0), j, min(j + 1, w - 1)};
  const __nv_bfloat16* sb = src + (long)n * h * w * src_sX + 8 * c8;
  float v[3][3][8];
#pragma unroll
  for (int a = 0; a < 3; ++a)
#pragma unroll
    for (int b = 0; b < 3; ++b) {
      const long q = (long)ys[a] * w + xs[b];
      const uint4 u = __ldg(reinterpret_cast<const uint4*>(sb + q * src_sX));
      const float am = ATTN ? __ldg(attn + (long)n * h * w + q) : 1.0f;
      const uint32_t wv[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float lo = __uint_as_float(wv[k] << 16), hi = __uint_as_float(wv[k] & 0xffff0000u);
        v[a][b][2 * k] = ATTN ? lo * am : lo;
        v[a][b][2 * k + 1] = ATTN ? hi * am : hi;
      }
    }
  const float lw = ATTN ? s_lw : 1.0f;
  const int H = F * h, W = F * w;
  __nv_bfloat16* db = dst + (((long)n * H + (long)F * i) * W + (long)F * j) * dst_sX + 8 * c8;
#pragma unroll
  for (int b = 0; b < F; ++b) {
    // horizontal taps of output column F j + b: delta = (b + 0.5) / F - 0.5
    const float dx = ((float)b + 0.5f) / (float)F - 0.5f;
    const int cA = dx < 0.f ? 0 : 1, cB = cA + 1;
    float wx1 = dx < 0.f ? 1.0f + dx : dx, wx0 = 1.0f - wx1;
    if (dx < 0.f && j == 0) { wx0 = 1.0f; wx1 = 0.0f; }   // src clamped to 0: (i0, w1) = (0, 0)
    float hx[3][8];
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
      for (int k = 0; k < 8; ++k) hx[a][k] = wx0 * v[a][cA][k] + wx1 * v[a][cB][k];
#pragma unroll
    for (int a = 0; a < F; ++a) {
      const float dy = ((float)a + 0.5f) / (float)F - 0.5f;
      const int rA = dy < 0.f ? 0 : 1, rB = rA + 1;
      float wy1 = dy < 0.f ? 1.0f + dy : dy, wy0 = 1.0f - wy1;
      if (dy < 0.f && i == 0) { wy0 = 1.0f; wy1 = 0.0f; }
      uint32_t ow[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        float r0 = wy0 * hx[rA][2 * k] + wy1 * hx[rB][2 * k];
        float r1 = wy0 * hx[rA][2 * k + 1] + wy1 * hx[rB][2 * k + 1];
        if (ATTN) { r0 *= lw; r1 *= lw; }
        const __nv_bfloat162 hh = __floats2bfloat162_rn(r0, r1);
        ow[k] = *reinterpret_cast<const uint32_t*>(&hh);
      }
      *reinterpret_cast<uint4*>(db + ((long)a * W + b) * dst_sX) = make_uint4(ow[0], ow[1], ow[2], ow[3]);
    }
  }
}

extern "C" int ffsr_resize_nhwc(const void* src, int N, int h, int w, int C, long long src_sX, void* dst, int H, int W,
                                long long dst_sX, int dtype, cudaStream_t stream) {
  FFSR_REQUIRE(src && dst, FFSR_ERR_ARG, "resize_nhwc: null pointer");
  FFSR_REQUIRE(N > 0 && h > 0 && w > 0 && H > 0 && W > 0 && C > 0 && C % 4 == 0, FFSR_ERR_ARG, "resize_nhwc: C%%4 != 0 or bad shape");
  const int esz = dtype == FFSR_DT_BF16 ? 2 : 4;
  FFSR_REQUIRE(((uintptr_t)src % (4 * esz)) == 0 && ((uintptr_t)dst % (4 * esz)) == 0 && src_sX % 4 == 0 && dst_sX % 4 == 0,
               FFSR_ERR_ALIGN, "resize_nhwc: vector alignment");
  if (dtype == FFSR_DT_BF16 && C % 8 == 0 && ((uintptr_t)src % 16) == 0 && ((uintptr_t)dst % 16) == 0 && src_sX % 8 == 0 &&
      dst_sX % 8 == 0 && h <= 65535 && N <= 65535 && ((H == 2 * h && W == 2 * w) || (H == 4 * h && W == 4 * w))) {
    dim3 grid(ceil_div((long)w * (C / 8), 256), h, N);
    if (H == 2 * h)
      k_upsample_int<2, false><<<grid, 256, 0, stream>>>((const __nv_bfloat16*)src, nullptr, h, w, C / 8, src_sX, nullptr, 0, (__nv_bfloat16*)dst, dst_sX);
    else
      k_upsample_int<4, false><<<grid, 256, 0, stream>>>((const __nv_bfloat16*)src, nullptr, h, w, C / 8, src_sX, nullptr, 0, (__nv_bfloat16*)dst, dst_sX);
    return ffsr_check_launch("resize_nhwc");
  }
  if (dtype == FFSR_DT_BF16 && C % 8 == 0 && ((uintptr_t)src % 16) == 0 && ((uintptr_t)dst % 16) == 0 && src_sX % 8 == 0 &&
      dst_sX % 8 == 0 && H <= 65535 && N <= 65535) {
    dim3 grid(ceil_div((long)W * (C / 8), 256), H, N);
    k_resize_nhwc_bf16x8<<<grid, 256, 0, stream>>>((const __nv_bfloat16*)src, h, w, C / 8, src_sX, (__nv_bfloat16*)dst, H, W,
                                                   dst_sX);
    return ffsr_check_launch("resize_nhwc");
  }
  const long total = (long)N * H * W * (C / 4);
  if (dtype == FFSR_DT_BF16)
    k_resize_nhwc<__nv_bfloat16><<<ceil_div(total, 256), 256, 0, stream>>>((const __nv_bfloat16*)src, h, w, C / 4, src_sX, (__nv_bfloat16*)dst, H, W, dst_sX, total);
  else
    k_resize_nhwc<float><<<ceil_div(total, 256), 256, 0, stream>>>((const float*)src, h, w, C / 4, src_sX, (float*)dst, H, W, dst_sX, total);
  return ffsr_check_launch("resize_nhwc");
}

// ------------------------------------------------------------------------------------------
// SpatialGate: y = x * sigmoid(w2 . gelu(W1 x + b1) + b2), fp32 rows, one thread per pixel
// ------------------------------------------------------------------------------------------
template <int C>
__global__ void __launch_bounds__(128) k_spatial_gate(const float* __restrict__ x, long pixels, const float* __restrict__ w1,
                                                      const float* __restrict__ b1, const float* __restrict__ w2,
                                                      const float* __restrict__ b2, float* __restrict__ y) {
  constexpr int HID = C / 4;
  __shared__ __align__(16) float sw1[HID][C];
  __shared__ float sb1[HID], sw2[HID];
  for (int i = threadIdx.x; i < HID * C; i += blockDim.x) (&sw1[0][0])[i] = w1[i];
  if (threadIdx.x < HID) { sb1[threadIdx.x] = b1[threadIdx.x]; sw2[threadIdx.x] = w2[threadIdx.x]; }
  __syncthreads();
  const long p = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= pixels) return;
  float v[C];
#pragma unroll
  for (int c = 0; c < C; c += 4) {
    const float4 t = load_vec4<float>(x + p * C + c);
    v[c] = t.x; v[c + 1] = t.y; v[c + 2] = t.z; v[c + 3] = t.w;
  }
  float z = b2[0];
#pragma unroll 4
  for (int h = 0; h < HID; ++h) {
    float a = sb1[h];
#pragma unroll
    for (int c = 0; c < C; c += 4) {                 // broadcast 16-byte weight loads: one shared load per four FMAs
      const float4 w4 = *reinterpret_cast<const float4*>(&sw1[h][c]);
      a = fmaf(w4.x, v[c], a); a = fmaf(w4.y, v[c + 1], a); a = fmaf(w4.z, v[c + 2], a); a = fmaf(w4.w, v[c + 3], a);
    }
    z = fmaf(sw2[h], gelu_sel<false>(a), z);
  }
  const float g = sigmoid_acc(z);
#pragma unroll
  for (int c = 0; c < C; c += 4) store_vec4<float>(y + p * C + c, v[c] * g, v[c + 1] * g, v[c + 2] * g, v[c + 3] * g);
}

// bf16 rows, TPP = C / CH lanes per pixel with CH channels each, the lane's slice of W1 (HID x CH = 64 floats) in REGISTERS
// for the whole grid-stride loop.  ncu of a one-thread-per-pixel bf16 kernel: 65 % of the issue cycles without an eligible warp,
// short-scoreboard stalls on the 64 shared-memory weight loads per pixel (weights of all C channels cannot live in one thread's
// registers).  The HID partial sums are combined by a transposing butterfly: at each of the log2(TPP) steps a lane hands half of
// its values to its partner, so it ends with HID / TPP complete hidden units (HID - HID / TPP shuffles in total instead of
// HID log2(TPP)), applies GELU and the second layer to those, and a last xor-reduction sums the gate logit.
template <int C, int CH>
__global__ void __launch_bounds__(256) k_spatial_gate_rows(const __nv_bfloat16* __restrict__ x, long pixels, const float* __restrict__ w1,
                                                           const float* __restrict__ b1, const float* __restrict__ w2,
                                                           const float* __restrict__ b2, __nv_bfloat16* __restrict__ y) {
  constexpr int HID = C / 4, TPP = C / CH, OWN = HID / TPP;
  static_assert(OWN >= 1 && (TPP & (TPP - 1)) == 0, "lanes per pixel must be a power of two not above the hidden width");
  const int part = threadIdx.x % TPP;
  float w[HID][CH];
#pragma unroll
  for (int h = 0; h < HID; ++h)
#pragma unroll
    for (int k = 0; k < CH; ++k) w[h][k] = w1[h * C + part * CH + k];
  int base = 0;
  {
    int half = HID / 2;
#pragma unroll
    for (int o = TPP / 2; o >= 1; o >>= 1, half >>= 1) base += (part & o) ? half : 0;
  }
  float sb[OWN], sw[OWN];
#pragma unroll
  for (int k = 0; k < OWN; ++k) { sb[k] = b1[base + k]; sw[k] = w2[base + k]; }
  const float bias2 = b2[0];
  const long stride = (long)gridDim.x * (256 / TPP);
  const long rounds = (pixels + stride - 1) / stride;
  long p = (long)blockIdx.x * (256 / TPP) + threadIdx.x / TPP;
  // the rows of the next TWO rounds are loaded ahead (x is not __restrict__-aliased with y rows of later rounds: a row is read
  // before any lane writes it, and only its own lanes write it)
  auto ld = [&](long q) -> uint4 {
    if (q >= pixels) return make_uint4(0u, 0u, 0u, 0u);
    if (CH == 8) return *reinterpret_cast<const uint4*>(x + q * C + part * 8);
    const uint2 t = *reinterpret_cast<const uint2*>(x + q * C + part * 4);
    return make_uint4(t.x, t.y, 0u, 0u);
  };
  uint4 n0 = ld(p), n1 = ld(p + stride);
  for (long it = 0; it < rounds; ++it, p += stride) {
    const bool live = p < pixels;
    const uint4 u = n0;
    n0 = n1;
    n1 = ld(p + 2 * stride);
    float v[CH];
    {
      const uint32_t wv[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
      for (int k = 0; k < CH / 2; ++k) { v[2 * k] = __uint_as_float(wv[k] << 16); v[2 * k + 1] = __uint_as_float(wv[k] & 0xffff0000u); }
    }
    float a[HID];
#pragma unroll
    for (int h = 0; h < HID; ++h) {
      float t = w[h][0] * v[0];
#pragma unroll
      for (int k = 1; k < CH; ++k) t = fmaf(w[h][k], v[k], t);
      a[h] = t;
    }
    {
      int half = HID / 2;
#pragma unroll
      for (int o = TPP / 2; o >= 1; o >>= 1, half >>= 1) {
        const bool up = (part & o) != 0;
#pragma unroll
        for (int k = 0; k < HID / 2; ++k)
          if (k < half) {
            const float mine = up ? a[half + k] : a[k], other = up ? a[k] : a[half + k];
            a[k] = mine + __shfl_xor_sync(0xffffffffu, other, o);
          }
      }
    }
    float z = 0.f;
#pragma unroll
    for (int k = 0; k < OWN; ++k) z = fmaf(sw[k], gelu_tanh(a[k] + sb[k]), z);
#pragma unroll
    for (int o = TPP / 2; o >= 1; o >>= 1) z += __shfl_xor_sync(0xffffffffu, z, o);
    const float g = sigmoid_acc(z + bias2);
    if (live) {
      uint32_t ow[CH / 2];
#pragma unroll
      for (int k = 0; k < CH / 2; ++k) {
        const __nv_bfloat162 hh = __floats2bfloat162_rn(v[2 * k] * g, v[2 * k + 1] * g);
        ow[k] = *reinterpret_cast<const uint32_t*>(&hh);
      }
      if (CH == 8) *reinterpret_cast<uint4*>(y + p * C + part * 8) = make_uint4(ow[0], ow[1], ow[CH == 8 ? 2 : 0], ow[CH == 8 ? 3 : 0]);
      else *reinterpret_cast<uint2*>(y + p * C + part * 4) = make_uint2(ow[0], ow[1]);
    }
  }
}

extern "C" int ffsr_spatial_gate(const void* x, long pixels, int C, const float* w1, const float* b1, const float* w2,
                                 const float* b2, void* y, int dtype, cudaStream_t stream) {
  FFSR_REQUIRE(x && y && w1 && b1 && w2 && b2, FFSR_ERR_ARG, "spatial_gate: null pointer");
  FFSR_REQUIRE(C == 64 || C == 32, FFSR_ERR_ARG, "spatial_gate: C must be 32 or 64");
  FFSR_REQUIRE(((uintptr_t)x % 16) == 0 && ((uintptr_t)y % 16) == 0, FFSR_ERR_ALIGN, "spatial_gate: 16B alignment");
  if (dtype == FFSR_DT_BF16) {
    static int num_sms = 0;
    if (!num_sms) {
      int dev = 0;
      cudaGetDevice(&dev);
      cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
    }
    const int tpp = C == 64 ? 16 : 4;
    const long need = (pixels * tpp + 255) / 256;
    const int g2 = (int)(need < 8L * num_sms ? need : 8L * num_sms);
    if (C == 64) k_spatial_gate_rows<64, 4><<<g2, 256, 0, stream>>>((const __nv_bfloat16*)x, pixels, w1, b1, w2, b2, (__nv_bfloat16*)y);
    else k_spatial_gate_rows<32, 8><<<g2, 256, 0, stream>>>((const __nv_bfloat16*)x, pixels, w1, b1, w2, b2, (__nv_bfloat16*)y);
    return ffsr_check_launch("spatial_gate");
  }
  const int grid = ceil_div(pixels, 128);
  if (C == 64) k_spatial_gate<64><<<grid, 128, 0, stream>>>((const float*)x, pixels, w1, b1, w2, b2, (float*)y);
  else k_spatial_gate<32><<<grid, 128, 0, stream>>>((const float*)x, pixels, w1, b1, w2, b2, (float*)y);
  return ffsr_check_launch("spatial_gate");
}

// ------------------------------------------------------------------------------------------
// Phase 5b/5c/6 blend at HR
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float bilin_plane(const float* __restrict__ pl, int W, const BilinTap& ty, const BilinTap& tx) {
  const float top = tx.w0 * pl[(long)ty.i0 * W + tx.i0] + tx.w1 * pl[(long)ty.i0 * W + tx.i1];
  const float bot = tx.w0 * pl[(long)ty.i1 * W + tx.i0] + tx.w1 * pl[(long)ty.i1 * W + tx.i1];
  return ty.w0 * top + ty.w1 * bot;
}

__global__ void __launch_bounds__(128) k_blend_hr(const float* __restrict__ hier, long long hier_sX,
                                                  const float* __restrict__ ecol, const float* __restrict__ routing,
                                                  const float* __restrict__ gates, const float* __restrict__ diff,
                                                  const float* __restrict__ fw0_w, const float* __restrict__ fw0_b,
                                                  const float* __restrict__ fw2_w, const float* __restrict__ fw2_b,
                                                  int B, int H, int W, float* __restrict__ fused_before,
                                                  float* __restrict__ fused_nhwc, long long fused_sX,
                                                  __nv_bfloat16* __restrict__ fused_lp, long long fused_lp_sX) {
  __shared__ float s0w[16][3], s0b[16], s2w[4][16], s2b[4];
  if (threadIdx.x < 48) (&s0w[0][0])[threadIdx.x] = fw0_w[threadIdx.x];
  if (threadIdx.x < 16) s0b[threadIdx.x] = fw0_b[threadIdx.x];
  if (threadIdx.x < 64) (&s2w[0][0])[threadIdx.x] = fw2_w[threadIdx.x];
  if (threadIdx.x < 4) s2b[threadIdx.x] = fw2_b[threadIdx.x];
  __syncthreads();
  const int Hh = 4 * H, Wh = 4 * W;
  const int X = blockIdx.x * blockDim.x + threadIdx.x;
  const int Y = blockIdx.y, b = blockIdx.z;
  if (X >= Wh) return;
  const long HW = (long)H * W, HWh = (long)Hh * Wh, pix = (long)Y * Wh + X;
  const BilinTap ty = bilin_tap(Y, H, Hh), tx = bilin_tap(X, W, Wh);

  // 5b: frequency-guided softmax weights from routing_lr upsampled x4
  float r[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) r[c] = bilin_plane(routing + ((long)b * 3 + c) * HW, W, ty, tx);
  float lg[4] = {s2b[0], s2b[1], s2b[2], s2b[3]};
#pragma unroll
  for (int h = 0; h < 16; ++h) {
    const float a = gelu_erf(fmaf(s0w[h][2], r[2], fmaf(s0w[h][1], r[1], fmaf(s0w[h][0], r[0], s0b[h]))));
#pragma unroll
    for (int e = 0; e < 4; ++e) lg[e] = fmaf(s2w[e][h], a, lg[e]);
  }
  const float mx = fmaxf(fmaxf(lg[0], lg[1]), fmaxf(lg[2], lg[3]));
  float fw[4], den = 0.f;
#pragma unroll
  for (int e = 0; e < 4; ++e) { fw[e] = expf(lg[e] - mx); den += fw[e]; }
#pragma unroll
  for (int e = 0; e < 4; ++e) fw[e] /= den;

  // 6: gates / difficulty upsampled x4
  float g[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) g[e] = bilin_plane(gates + ((long)b * 4 + e) * HW, W, ty, tx);
  const float gsum = (((g[0] + g[1]) + g[2]) + g[3]) + 1e-8f;
  const float bw = 0.3f + 0.4f * bilin_plane(diff + (long)b * HW, W, ty, tx);

  const float* hp = hier + ((long)b * HWh + pix) * hier_sX;
  float out[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    float freq = 0.f, dyn = 0.f;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float v = ecol[((long)(b * 4 + e) * 3 + c) * HWh + pix];
      freq += v * fw[e];
      dyn += v * g[e];
    }
    const float f0 = hp[c] * 0.7f + freq * 0.3f;
    if (fused_before) fused_before[((long)b * 3 + c) * HWh + pix] = f0;
    out[c] = (1.0f - bw) * f0 + bw * (dyn / gsum);
  }
  float* fo = fused_nhwc + ((long)b * HWh + pix) * fused_sX;
  fo[0] = out[0]; fo[1] = out[1]; fo[2] = out[2];
  if (fused_sX > 3) fo[3] = 0.f;
  if (fused_lp) {
    __nv_bfloat16* lp = fused_lp + ((long)b * HWh + pix) * fused_lp_sX;
    store_vec4<__nv_bfloat16>(lp, out[0], out[1], out[2], 0.f);
    for (int c = 4; c + 4 <= (int)fused_lp_sX; c += 4) store_vec4<__nv_bfloat16>(lp + c, 0.f, 0.f, 0.f, 0.f);
  }
}

extern "C" int ffsr_blend_hr(const float* hier, long long hier_sX, const float* ecol, const float* routing,
                             const float* gates, const float* diff, const float* fw0_w, const float* fw0_b,
                             const float* fw2_w, const float* fw2_b, int B, int H, int W, float* fused_before,
                             float* fused_nhwc, long long fused_sX, void* fused_lp, long long fused_lp_sX,
                             cudaStream_t stream) {
  FFSR_REQUIRE(hier && ecol && routing && gates && diff && fw0_w && fw0_b && fw2_w && fw2_b && fused_nhwc, FFSR_ERR_ARG,
               "blend_hr: null pointer");
  FFSR_REQUIRE(B > 0 && B <= 65535 && 4 * H <= 65535 && fused_sX >= 3, FFSR_ERR_ARG, "blend_hr: bad shape");
  FFSR_REQUIRE(!fused_lp || (((uintptr_t)fused_lp % 8) == 0 && fused_lp_sX % 4 == 0 && fused_lp_sX >= 4), FFSR_ERR_ALIGN,
               "blend_hr: low-precision copy alignment");
  dim3 grid(ceil_div(4 * W, 128), 4 * H, B);
  k_blend_hr<<<grid, 128, 0, stream>>>(hier, hier_sX, ecol, routing, gates, diff, fw0_w, fw0_b, fw2_w, fw2_b, B, H, W,
                                       fused_before, fused_nhwc, fused_sX, (__nv_bfloat16*)fused_lp, fused_lp_sX);
  return ffsr_check_launch("blend_hr");
}

// ------------------------------------------------------------------------------------------
// Laplacian pyramid: down = avg_pool2(gauss5x5(x));  lap = x - bilinear(down)
// ------------------------------------------------------------------------------------------
// avg_pool2 o gauss5x5 is ONE 6x6 stride-2 kernel K6 = box2 * gauss5 (the same identity the backward kernel uses): 36 taps x 3
// channels per output instead of 4 x 25 x 3, and with channels-last rows of >= 4 floats each tap is one 16-byte load
// (the previous version: 108 predicated scalar loads + 300 FMAs per output, 0.63 TB/s).
template <bool VEC>
__global__ void __launch_bounds__(128) k_blur_pool(const float* __restrict__ x, long long x_sX, int H, int W,
                                                   const float* __restrict__ gauss25, float* __restrict__ down,
                                                   long long down_sX, __nv_bfloat16* __restrict__ down_lp,
                                                   long long down_lp_sX) {
  __shared__ float k6[6][6];
  if (threadIdx.x < 36) {
    const int a = threadIdx.x / 6, b = threadIdx.x % 6;
    float acc = 0.f;
    for (int da = 0; da < 2; ++da)
      for (int db = 0; db < 2; ++db) {
        const int ky = a - da, kx = b - db;
        if (ky >= 0 && ky < 5 && kx >= 0 && kx < 5) acc += gauss25[ky * 5 + kx];
      }
    k6[a][b] = 0.25f * acc;
  }
  __syncthreads();
  const int H2 = H / 2, W2 = W / 2;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  const int i = blockIdx.y, n = blockIdx.z;
  if (j >= W2) return;
  const float* img = x + (long)n * H * W * x_sX;
  float o0 = 0.f, o1 = 0.f, o2 = 0.f;
#pragma unroll
  for (int a = 0; a < 6; ++a) {
    const int yy = 2 * i + a - 2;
    if (yy < 0 || yy >= H) continue;
    const float* row = img + (long)yy * W * x_sX;
#pragma unroll
    for (int bb = 0; bb < 6; ++bb) {
      const int xx = 2 * j + bb - 2;
      if (xx < 0 || xx >= W) continue;
      const float kk = k6[a][bb];
      if (VEC) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(row + (long)xx * x_sX));
        o0 = fmaf(kk, v.x, o0); o1 = fmaf(kk, v.y, o1); o2 = fmaf(kk, v.z, o2);
      } else {
        const float* p = row + (long)xx * x_sX;
        o0 = fmaf(kk, p[0], o0); o1 = fmaf(kk, p[1], o1); o2 = fmaf(kk, p[2], o2);
      }
    }
  }
  float* o = down + (((long)n * H2 + i) * W2 + j) * down_sX;
  if (VEC && down_sX == 4) *reinterpret_cast<float4*>(o) = make_float4(o0, o1, o2, 0.f);
  else {
    o[0] = o0; o[1] = o1; o[2] = o2;
    if (down_sX > 3) o[3] = 0.f;
  }
  if (down_lp) store_vec4<__nv_bfloat16>(down_lp + (((long)n * H2 + i) * W2 + j) * down_lp_sX, o0, o1, o2, 0.f);
}

extern "C" int ffsr_blur_pool(const float* x, long long x_sX, int N, int H, int W, const float* gauss25, float* down,
                              long long down_sX, void* down_lp, long long down_lp_sX, cudaStream_t stream) {
  FFSR_REQUIRE(x && gauss25 && down, FFSR_ERR_ARG, "blur_pool: null pointer");
  FFSR_REQUIRE(N > 0 && H >= 2 && W >= 2 && x_sX >= 3 && down_sX >= 3, FFSR_ERR_ARG, "blur_pool: bad shape");
  dim3 grid(ceil_div(W / 2, 128), H / 2, N);
  FFSR_REQUIRE(!down_lp || (((uintptr_t)down_lp % 8) == 0 && down_lp_sX % 4 == 0 && down_lp_sX >= 4), FFSR_ERR_ALIGN,
               "blur_pool: bf16 copy alignment");
  const bool vec = x_sX % 4 == 0 && ((uintptr_t)x % 16) == 0 && (down_sX != 4 || ((uintptr_t)down % 16) == 0);
  if (vec) k_blur_pool<true><<<grid, 128, 0, stream>>>(x, x_sX, H, W, gauss25, down, down_sX, (__nv_bfloat16*)down_lp, down_lp_sX);
  else k_blur_pool<false><<<grid, 128, 0, stream>>>(x, x_sX, H, W, gauss25, down, down_sX, (__nv_bfloat16*)down_lp, down_lp_sX);
  return ffsr_check_launch("blur_pool");
}

// adjoint of down = avg_pool2(gauss5x5(x)): the two ops are one 6x6 stride-2 kernel K6 = box2 * gauss5, so
// gx[y][x] = sum over the <= 3x3 outputs (oy, ox) with 2*oy - 2 <= y <= 2*oy + 3 of K6[y-2oy+2][x-2ox+2] * g[oy][ox]
__global__ void __launch_bounds__(128) k_blur_pool_bwd(const float* __restrict__ g, long long g_sX, int H, int W,
                                                       const float* __restrict__ gauss25, float* __restrict__ gx,
                                                       long long gx_sX) {
  __shared__ float k6[6][6];
  if (threadIdx.x < 36) {
    const int a = threadIdx.x / 6, b = threadIdx.x % 6;
    float acc = 0.f;
    for (int da = 0; da < 2; ++da)
      for (int db = 0; db < 2; ++db) {
        const int ky = a - da, kx = b - db;
        if (ky >= 0 && ky < 5 && kx >= 0 && kx < 5) acc += gauss25[ky * 5 + kx];
      }
    k6[a][b] = 0.25f * acc;
  }
  __syncthreads();
  const int H2 = H / 2, W2 = W / 2;
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y, n = blockIdx.z;
  if (x >= W) return;
  const float* gi = g + (long)n * H2 * W2 * g_sX;
  float acc[3] = {0.f, 0.f, 0.f};
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const int a = (y & 1) + 2 * i;                 // a = y - 2*oy + 2, same parity as y
    const int oy = (y + 2 - a) >> 1;
    if (oy < 0 || oy >= H2) continue;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const int b = (x & 1) + 2 * j;
      const int ox = (x + 2 - b) >> 1;
      if (ox < 0 || ox >= W2) continue;
      const float wgt = k6[a][b];
      const float* p = gi + ((long)oy * W2 + ox) * g_sX;
      acc[0] = fmaf(wgt, p[0], acc[0]); acc[1] = fmaf(wgt, p[1], acc[1]); acc[2] = fmaf(wgt, p[2], acc[2]);
    }
  }
  float* o = gx + (((long)n * H + y) * W + x) * gx_sX;
  o[0] = acc[0]; o[1] = acc[1]; o[2] = acc[2];
}

extern "C" int ffsr_blur_pool_backward(const float* g, long long g_sX, int N, int H, int W, const float* gauss25, float* gx,
                                       long long gx_sX, cudaStream_t stream) {
  FFSR_REQUIRE(g && gauss25 && gx, FFSR_ERR_ARG, "blur_pool_backward: null pointer");
  FFSR_REQUIRE(N > 0 && N <= 65535 && H >= 2 && H <= 65535 && W >= 2 && g_sX >= 3 && gx_sX >= 3, FFSR_ERR_ARG, "blur_pool_backward: bad shape");
  dim3 grid(ceil_div(W, 128), H, N);
  k_blur_pool_bwd<<<grid, 128, 0, stream>>>(g, g_sX, H, W, gauss25, gx, gx_sX);
  return ffsr_check_launch("blur_pool_backward");
}

__global__ void __launch_bounds__(128) k_laplacian_sub(const float* __restrict__ x, long long x_sX,
                                                       const float* __restrict__ down, long long down_sX, int H, int W,
                                                       float* __restrict__ lap, long long lap_sX,
                                                       __nv_bfloat16* __restrict__ lap_lp, long long lap_lp_sX) {
  const int X = blockIdx.x * blockDim.x + threadIdx.x;
  const int Y = blockIdx.y, n = blockIdx.z;
  if (X >= W) return;
  const int h = H / 2, w = W / 2;
  const BilinTap ty = bilin_tap(Y, h, H), tx = bilin_tap(X, w, W);
  const float* d = down + (long)n * h * w * down_sX;
  const float* a = d + ((long)ty.i0 * w + tx.i0) * down_sX;
  const float* b = d + ((long)ty.i0 * w + tx.i1) * down_sX;
  const float* c = d + ((long)ty.i1 * w + tx.i0) * down_sX;
  const float* e = d + ((long)ty.i1 * w + tx.i1) * down_sX;
  const long pix = ((long)n * H + Y) * W + X;
  const float* xp = x + pix * x_sX;
  float* o = lap + pix * lap_sX;
#pragma unroll
  for (int ch = 0; ch < 3; ++ch)
    o[ch] = xp[ch] - (ty.w0 * (tx.w0 * a[ch] + tx.w1 * b[ch]) + ty.w1 * (tx.w0 * c[ch] + tx.w1 * e[ch]));
  if (lap_sX > 3) o[3] = 0.f;
  if (lap_lp) store_vec4<__nv_bfloat16>(lap_lp + pix * lap_lp_sX, o[0], o[1], o[2], 0.f);
}

extern "C" int ffsr_laplacian_sub(const float* x, long long x_sX, const float* down, long long down_sX, int N, int H,
                                  int W, float* lap, long long lap_sX, void* lap_lp, long long lap_lp_sX,
                                  cudaStream_t stream) {
  FFSR_REQUIRE(x && down && lap, FFSR_ERR_ARG, "laplacian_sub: null pointer");
  FFSR_REQUIRE(N > 0 && H >= 2 && W >= 2, FFSR_ERR_ARG, "laplacian_sub: bad shape");
  dim3 grid(ceil_div(W, 128), H, N);
  FFSR_REQUIRE(!lap_lp || (((uintptr_t)lap_lp % 8) == 0 && lap_lp_sX % 4 == 0 && lap_lp_sX >= 4), FFSR_ERR_ALIGN,
               "laplacian_sub: bf16 copy alignment");
  k_laplacian_sub<<<grid, 128, 0, stream>>>(x, x_sX, down, down_sX, H, W, lap, lap_sX, (__nv_bfloat16*)lap_lp, lap_lp_sX);
  return ffsr_check_launch("laplacian_sub");
}

// ------------------------------------------------------------------------------------------
// refiner tail: (o * attn), bilinear to HxW if needed, times softmax(level_weights)[level]
// ------------------------------------------------------------------------------------------
template <typename TI, typename T>
__global__ void __launch_bounds__(256) k_edge_attn_up(const TI* __restrict__ o, const float* __restrict__ attn, int h,
                                                      int w, int C4, const float* __restrict__ level_w, int level,
                                                      T* __restrict__ dst, int H, int W, long long dst_sX, long total) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const float l0 = level_w[0], l1 = level_w[1], l2 = level_w[2];
  const float m = fmaxf(l0, fmaxf(l1, l2));
  const float e0 = expf(l0 - m), e1 = expf(l1 - m), e2 = expf(l2 - m);
  const float lw = (level == 0 ? e0 : (level == 1 ? e1 : e2)) / ((e0 + e1) + e2);
  const int c4 = (int)(i % C4);
  const long pix = i / C4;
  const int X = (int)(pix % W), Y = (int)((pix / W) % H);
  const long n = pix / ((long)W * H);
  const int C = 4 * C4;
  const TI* ob = o + n * h * w * C + 4 * c4;
  const float* ab = attn + n * h * w;
  float4 r;
  if (h == H && w == W) {
    const long q = (long)Y * w + X;
    const float4 v = load_vec4<TI>(ob + q * C);
    const float a = ab[q];
    r = make_float4(v.x * a, v.y * a, v.z * a, v.w * a);
  } else {
    const BilinTap ty = bilin_tap(Y, h, H), tx = bilin_tap(X, w, W);
    const long q00 = (long)ty.i0 * w + tx.i0, q01 = (long)ty.i0 * w + tx.i1;
    const long q10 = (long)ty.i1 * w + tx.i0, q11 = (long)ty.i1 * w + tx.i1;
    const float4 v00 = load_vec4<TI>(ob + q00 * C), v01 = load_vec4<TI>(ob + q01 * C);
    const float4 v10 = load_vec4<TI>(ob + q10 * C), v11 = load_vec4<TI>(ob + q11 * C);
    const float a00 = ab[q00], a01 = ab[q01], a10 = ab[q10], a11 = ab[q11];
    r.x = ty.w0 * (tx.w0 * (v00.x * a00) + tx.w1 * (v01.x * a01)) + ty.w1 * (tx.w0 * (v10.x * a10) + tx.w1 * (v11.x * a11));
    r.y = ty.w0 * (tx.w0 * (v00.y * a00) + tx.w1 * (v01.y * a01)) + ty.w1 * (tx.w0 * (v10.y * a10) + tx.w1 * (v11.y * a11));
    r.z = ty.w0 * (tx.w0 * (v00.z * a00) + tx.w1 * (v01.z * a01)) + ty.w1 * (tx.w0 * (v10.z * a10) + tx.w1 * (v11.z * a11));
    r.w = ty.w0 * (tx.w0 * (v00.w * a00) + tx.w1 * (v01.w * a01)) + ty.w1 * (tx.w0 * (v10.w * a10) + tx.w1 * (v11.w * a11));
  }
  store_vec4<T>(dst + pix * dst_sX + 4 * c4, r.x * lw, r.y * lw, r.z * lw, r.w * lw);
}

// bf16 in / bf16 out, 8 channels (16 bytes) per thread, row-structured grid (no per-thread div/mod chain), the
// level softmax computed once per block: the 4-channel kernel above was issue-bound (3 expf + 64-bit index
// arithmetic per 8 output bytes).
__global__ void __launch_bounds__(256) k_edge_attn_up_bf16x8(const __nv_bfloat16* __restrict__ o, const float* __restrict__ attn,
                                                             int h, int w, int C8, const float* __restrict__ level_w,
                                                             int level, __nv_bfloat16* __restrict__ dst, int H, int W,
                                                             long long dst_sX) {
  __shared__ float s_lw;
  if (threadIdx.x == 0) {
    const float l0 = level_w[0], l1 = level_w[1], l2 = level_w[2];
    const float m = fmaxf(l0, fmaxf(l1, l2));
    const float e0 = expf(l0 - m), e1 = expf(l1 - m), e2 = expf(l2 - m);
    s_lw = (level == 0 ? e0 : (level == 1 ? e1 : e2)) / ((e0 + e1) + e2);
  }
  __syncthreads();
  const int t = blockIdx.x * blockDim.x + threadIdx.x;       // over W * C8
  const int X = t / C8, c8 = t - X * C8;
  const int Y = blockIdx.y, n = blockIdx.z;
  if (X >= W) return;
  const float lw = s_lw;
  const int C = 8 * C8;
  const __nv_bfloat16* ob = o + (long)n * h * w * C + 8 * c8;
  const float* ab = attn + (long)n * h * w;
  float r[8];
  auto unpack = [](const uint4& u, float (&f)[8]) {
    const uint32_t wv[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float2 f2 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&wv[k]));
      f[2 * k] = f2.x; f[2 * k + 1] = f2.y;
    }
  };
  if (h == H && w == W) {
    const int q = Y * w + X;
    float v[8];
    unpack(*reinterpret_cast<const uint4*>(ob + (long)q * C), v);
    const float a = ab[q];
#pragma unroll
    for (int k = 0; k < 8; ++k) r[k] = v[k] * a;
  } else {
    const BilinTap ty = bilin_tap(Y, h, H), tx = bilin_tap(X, w, W);
    const int q00 = ty.i0 * w + tx.i0, q01 = ty.i0 * w + tx.i1, q10 = ty.i1 * w + tx.i0, q11 = ty.i1 * w + tx.i1;
    float v00[8], v01[8], v10[8], v11[8];
    unpack(*reinterpret_cast<const uint4*>(ob + (long)q00 * C), v00);
    unpack(*reinterpret_cast<const uint4*>(ob + (long)q01 * C), v01);
    unpack(*reinterpret_cast<const uint4*>(ob + (long)q10 * C), v10);
    unpack(*reinterpret_cast<const uint4*>(ob + (long)q11 * C), v11);
    const float a00 = ab[q00], a01 = ab[q01], a10 = ab[q10], a11 = ab[q11];
#pragma unroll
    for (int k = 0; k < 8; ++k)
      r[k] = ty.w0 * (tx.w0 * (v00[k] * a00) + tx.w1 * (v01[k] * a01)) + ty.w1 * (tx.w0 * (v10[k] * a10) + tx.w1 * (v11[k] * a11));
  }
  uint32_t ow[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    __nv_bfloat162 hh = __floats2bfloat162_rn(r[2 * k] * lw, r[2 * k + 1] * lw);
    ow[k] = *reinterpret_cast<uint32_t*>(&hh);
  }
  *reinterpret_cast<uint4*>(dst + (((long)n * H + Y) * W + X) * dst_sX + 8 * c8) = make_uint4(ow[0], ow[1], ow[2], ow[3]);
}

extern "C" int ffsr_edge_attn_upsample(const void* o, int o_dtype, const float* attn, int N, int h, int w, int C,
                                       const float* level_w, int level, void* dst, int H, int W, long long dst_sX,
                                       int dtype, cudaStream_t stream) {
  FFSR_REQUIRE(o && attn && level_w && dst, FFSR_ERR_ARG, "edge_attn_upsample: null pointer");
  FFSR_REQUIRE(C % 4 == 0 && level >= 0 && level < 3, FFSR_ERR_ARG, "edge_attn_upsample: bad C/level");
  const int esz = dtype == FFSR_DT_BF16 ? 2 : 4;
  FFSR_REQUIRE(((uintptr_t)o % 16) == 0 && ((uintptr_t)dst % (4 * esz)) == 0 && dst_sX % 4 == 0, FFSR_ERR_ALIGN,
               "edge_attn_upsample: alignment");
  const long total = (long)N * H * W * (C / 4);
  FFSR_REQUIRE(o_dtype == FFSR_DT_F32 || dtype == FFSR_DT_BF16, FFSR_ERR_ARG, "edge_attn_upsample: bf16 input needs bf16 output");
  if (o_dtype == FFSR_DT_BF16 && C % 8 == 0 && ((uintptr_t)dst % 16) == 0 && dst_sX % 8 == 0 && h <= 65535 && N <= 65535 &&
      ((H == 2 * h && W == 2 * w) || (H == 4 * h && W == 4 * w))) {
    dim3 grid(ceil_div((long)w * (C / 8), 256), h, N);
    if (H == 2 * h)
      k_upsample_int<2, true><<<grid, 256, 0, stream>>>((const __nv_bfloat16*)o, attn, h, w, C / 8, C, level_w, level, (__nv_bfloat16*)dst, dst_sX);
    else
      k_upsample_int<4, true><<<grid, 256, 0, stream>>>((const __nv_bfloat16*)o, attn, h, w, C / 8, C, level_w, level, (__nv_bfloat16*)dst, dst_sX);
    return ffsr_check_launch("edge_attn_upsample");
  }
  if (o_dtype == FFSR_DT_BF16 && C % 8 == 0 && ((uintptr_t)dst % 16) == 0 && dst_sX % 8 == 0 && H <= 65535 && N <= 65535) {
    dim3 grid(ceil_div((long)W * (C / 8), 256), H, N);
    k_edge_attn_up_bf16x8<<<grid, 256, 0, stream>>>((const __nv_bfloat16*)o, attn, h, w, C / 8, level_w, level,
                                                    (__nv_bfloat16*)dst, H, W, dst_sX);
    return ffsr_check_launch("edge_attn_upsample");
  }
  if (o_dtype == FFSR_DT_BF16)
    k_edge_attn_up<__nv_bfloat16, __nv_bfloat16><<<ceil_div(total, 256), 256, 0, stream>>>((const __nv_bfloat16*)o, attn, h, w, C / 4, level_w, level, (__nv_bfloat16*)dst, H, W, dst_sX, total);
  else if (dtype == FFSR_DT_BF16)
    k_edge_attn_up<float, __nv_bfloat16><<<ceil_div(total, 256), 256, 0, stream>>>((const float*)o, attn, h, w, C / 4, level_w, level, (__nv_bfloat16*)dst, H, W, dst_sX, total);
  else
    k_edge_attn_up<float, float><<<ceil_div(total, 256), 256, 0, stream>>>((const float*)o, attn, h, w, C / 4, level_w, level, (float*)dst, H, W, dst_sX, total);
  return ffsr_check_launch("edge_attn_upsample");
}

// ------------------------------------------------------------------------------------------
// final: clamp(x + gate*strength*edge, 0, 1) + residual_scale * bilinear_x4(lr)  [clamp in eval]
// xe: channels-last, x in channels 0..2, edge map in 3..5; out: [B][3][4H][4W] planar
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_final_combine(const float* __restrict__ xe, long long xe_sX,
                                                       const float* __restrict__ gate, const float* __restrict__ strength,
                                                       const float* __restrict__ lr, const float* __restrict__ rs,
                                                       int H, int W, int clamp01, float* __restrict__ out) {
  const int Hh = 4 * H, Wh = 4 * W;
  const int X = blockIdx.x * blockDim.x + threadIdx.x;
  const int Y = blockIdx.y, b = blockIdx.z;
  if (X >= Wh) return;
  const long HW = (long)H * W, HWh = (long)Hh * Wh, pix = (long)Y * Wh + X;
  const BilinTap ty = bilin_tap(Y, H, Hh), tx = bilin_tap(X, W, Wh);
  const float* p = xe + ((long)b * HWh + pix) * xe_sX;
  const float gs = gate[(long)b * HWh + pix] * strength[0];
  const float scale = rs[0];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    float v = p[c] + gs * p[3 + c];
    v = fminf(fmaxf(v, 0.f), 1.f);
    v += scale * bilin_plane(lr + ((long)b * 3 + c) * HW, W, ty, tx);
    if (clamp01) v = fminf(fmaxf(v, 0.f), 1.f);
    out[((long)b * 3 + c) * HWh + pix] = v;
  }
}

extern "C" int ffsr_final_combine(const float* xe, long long xe_sX, const float* gate, const float* strength,
                                  const float* lr, const float* residual_scale, int B, int H, int W, int clamp01,
                                  float* out, cudaStream_t stream) {
  FFSR_REQUIRE(xe && gate && strength && lr && residual_scale && out, FFSR_ERR_ARG, "final_combine: null pointer");
  FFSR_REQUIRE(B > 0 && B <= 65535 && 4 * H <= 65535 && xe_sX >= 6, FFSR_ERR_ARG, "final_combine: bad shape");
  dim3 grid(ceil_div(4 * W, 128), 4 * H, B);
  k_final_combine<<<grid, 128, 0, stream>>>(xe, xe_sX, gate, strength, lr, residual_scale, H, W, clamp01, out);
  return ffsr_check_launch("final_combine");
}

// ------------------------------------------------------------------------------------------
// fp32 NCHW -> bf16 channels-last slice (expert features -> tcgen05 operand), 32x32 smem transpose
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_nchw_to_nhwc_bf16(const float* __restrict__ src, int C, long HW,
                                                           __nv_bfloat16* __restrict__ dst, long long dst_sN,
                                                           long long dst_sX) {
  __shared__ float tile[32][33];
  const long p0 = (long)blockIdx.x * 32;
  const int c0 = blockIdx.y * 32, n = blockIdx.z;
  const int tx = threadIdx.x, ty = threadIdx.y;           // (32, 8)
  const float* s = src + (long)n * C * HW;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int c = c0 + ty + 8 * j;
    const long p = p0 + tx;
    tile[ty + 8 * j][tx] = (c < C && p < HW) ? s[(long)c * HW + p] : 0.f;
  }
  __syncthreads();
  __nv_bfloat16* d = dst + (long long)n * dst_sN;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const long p = p0 + ty + 8 * j;
    const int c = c0 + tx;
    if (p < HW && c < C) d[p * dst_sX + c] = __float2bfloat16_rn(tile[tx][ty + 8 * j]);
  }
}

extern "C" int ffsr_nchw_to_nhwc_bf16(const float* src, int N, int C, long HW, void* dst, long long dst_sN,
                                      long long dst_sX, cudaStream_t stream) {
  FFSR_REQUIRE(src && dst && N > 0 && N <= 65535 && C > 0 && HW > 0, FFSR_ERR_ARG, "nchw_to_nhwc_bf16: bad args");
  dim3 grid(ceil_div(HW, 32), ceil_div(C, 32), N);
  k_nchw_to_nhwc_bf16<<<grid, dim3(32, 8), 0, stream>>>(src, C, HW, (__nv_bfloat16*)dst, dst_sN, dst_sX);
  return ffsr_check_launch("nchw_to_nhwc_bf16");
}

__global__ void __launch_bounds__(256) k_cast_bf16(const float4* __restrict__ src, uint2* __restrict__ dst, long n4) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n4) return;
  const float4 v = src[i];
  __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
  uint2 u;
  u.x = *reinterpret_cast<uint32_t*>(&lo);
  u.y = *reinterpret_cast<uint32_t*>(&hi);
  dst[i] = u;
}

extern "C" int ffsr_cast_f32_to_bf16(const float* src, void* dst, long n, cudaStream_t stream) {
  FFSR_REQUIRE(src && dst && n > 0 && n % 4 == 0, FFSR_ERR_ARG, "cast_f32_to_bf16: n must be a positive multiple of 4");
  FFSR_REQUIRE(((uintptr_t)src % 16) == 0 && ((uintptr_t)dst % 8) == 0, FFSR_ERR_ALIGN, "cast_f32_to_bf16: alignment");
  k_cast_bf16<<<ceil_div(n / 4, 256), 256, 0, stream>>>((const float4*)src, (uint2*)dst, n / 4);
  return ffsr_check_launch("cast_f32_to_bf16");
}
