// Small HBM-bound ops of the DRCT-L expert forward (SURVEY §8f N1) that the fusion path did not need:
// LayerNorm over a channel PREFIX of a wider row (the dense-growth buffer of an RDG), LeakyReLU in place on a channel
// slice, PixelShuffle(2) on channels-last tensors, and the RGB mean / range shifts at both ends of the network.
//
// STATUS: exercised on a B200 through `isr_b200.drct.DRCT.forward` (parity <= 1e-4 against the reference class's output,
// tests/test_gpu_drct.py); simple grid-stride kernels, not yet timed against the HBM roof.
#include "common.cuh"
#include "../../include/ffsr_b200.h"

namespace {

template <typename T>
__device__ __forceinline__ float ldf(const T* p, long i);
template <>
__device__ __forceinline__ float ldf<float>(const float* p, long i) { return p[i]; }
template <>
__device__ __forceinline__ float ldf<__nv_bfloat16>(const __nv_bfloat16* p, long i) { return __bfloat162float(p[i]); }
template <typename T>
__device__ __forceinline__ void stf(T* p, long i, float v);
template <>
__device__ __forceinline__ void stf<float>(float* p, long i, float v) { p[i] = v; }
template <>
__device__ __forceinline__ void stf<__nv_bfloat16>(__nv_bfloat16* p, long i, float v) { p[i] = __float2bfloat16_rn(v); }

// nn.LayerNorm(C), eps 1e-5, biased variance, over the first C channels of rows with pitch x_pitch; one warp per row.
template <typename TI, typename TO>
__global__ void __launch_bounds__(256) k_layernorm_strided(const TI* __restrict__ x, long rows, int C, long x_pitch,
                                                           const float* __restrict__ w, const float* __restrict__ b,
                                                           TO* __restrict__ y, long y_pitch) {
  const int lane = threadIdx.x & 31;
  const long warps = (long)gridDim.x * (blockDim.x >> 5);
  for (long r = (long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < rows; r += warps) {
    const TI* xr = x + r * x_pitch;
    float s = 0.f;
    for (int c = lane; c < C; c += 32) s += ldf<TI>(xr, c);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    const float mean = s / (float)C;
    float v = 0.f;
    for (int c = lane; c < C; c += 32) {
      const float d = ldf<TI>(xr, c) - mean;
      v = fmaf(d, d, v);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const float rstd = rsqrtf(v / (float)C + 1e-5f);
    TO* yr = y + r * y_pitch;
    for (int c = lane; c < C; c += 32) stf<TO>(yr, c, (ldf<TI>(xr, c) - mean) * rstd * __ldg(w + c) + __ldg(b + c));
  }
}

// fp32 rows -> bf16 rows, four channels per lane and step (16-byte loads, 8-byte stores): the DRCT-L LayerNorms in the bf16 mode
// (C, both pitches and both bases multiples of 4 elements).  Same two-pass statistics as above; the row is read from L1 on
// the second and third pass.
__global__ void __launch_bounds__(256) k_layernorm_strided_v4(const float* __restrict__ x, long rows, int C, long x_pitch,
                                                              const float* __restrict__ w, const float* __restrict__ b,
                                                              __nv_bfloat16* __restrict__ y, long y_pitch) {
  const int lane = threadIdx.x & 31;
  const int C4 = C >> 2;
  const long warps = (long)gridDim.x * (blockDim.x >> 5);
  for (long r = (long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < rows; r += warps) {
    const float4* xr = reinterpret_cast<const float4*>(x + r * x_pitch);
    float s = 0.f;
    for (int c = lane; c < C4; c += 32) {
      const float4 v = xr[c];
      s += (v.x + v.y) + (v.z + v.w);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    const float mean = s / (float)C;
    float q = 0.f;
    for (int c = lane; c < C4; c += 32) {
      const float4 v = xr[c];
      const float d0 = v.x - mean, d1 = v.y - mean, d2 = v.z - mean, d3 = v.w - mean;
      q = fmaf(d0, d0, q); q = fmaf(d1, d1, q); q = fmaf(d2, d2, q); q = fmaf(d3, d3, q);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
    const float rstd = rsqrtf(q / (float)C + 1e-5f);
    uint2* yr = reinterpret_cast<uint2*>(y + r * y_pitch);
    for (int c = lane; c < C4; c += 32) {
      const float4 v = xr[c];
      const float4 wv = __ldg(reinterpret_cast<const float4*>(w) + c), bv = __ldg(reinterpret_cast<const float4*>(b) + c);
      const __nv_bfloat162 lo = __floats2bfloat162_rn(fmaf((v.x - mean) * rstd, wv.x, bv.x), fmaf((v.y - mean) * rstd, wv.y, bv.y));
      const __nv_bfloat162 hi = __floats2bfloat162_rn(fmaf((v.z - mean) * rstd, wv.z, bv.z), fmaf((v.w - mean) * rstd, wv.w, bv.w));
      yr[c] = make_uint2(*reinterpret_cast<const uint32_t*>(&lo), *reinterpret_cast<const uint32_t*>(&hi));
    }
  }
}

template <typename T>
__global__ void k_leaky_relu(T* __restrict__ x, long rows, int C, long pitch, float slope) {
  const long total = rows * C;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const long r = i / C;
    const int c = (int)(i - r * C);
    const float v = ldf<T>(x, r * pitch + c);
    if (v < 0.f) stf<T>(x, r * pitch + c, v * slope);
  }
}

// nn.PixelShuffle(2) on channels-last data: y[b][2h+i][2w+j][c] = x[b][h][w][4c + 2i + j]
template <typename T>
__global__ void k_pixel_shuffle2(const T* __restrict__ x, int B, int H, int W, int C, T* __restrict__ y) {
  const long total = (long)B * 2 * H * 2 * W * C;
  for (long o = (long)blockIdx.x * blockDim.x + threadIdx.x; o < total; o += (long)gridDim.x * blockDim.x) {
    const int c = (int)(o % C);
    long r = o / C;
    const int xo = (int)(r % (2 * W)); r /= 2 * W;
    const int yo = (int)(r % (2 * H));
    const long b = r / (2 * H);
    const long src = ((b * H + (yo >> 1)) * W + (xo >> 1)) * (4L * C) + 4 * c + 2 * (yo & 1) + (xo & 1);
    y[o] = x[src];
  }
}

// in: [B][3][H][W] fp32 planar -> out: [B][H][W][pitch] channels-last, (x - mean[c]) * range (channels >= 3 untouched)
template <typename T>
__global__ void k_rgb_in(const float* __restrict__ x, int B, long HW, float m0, float m1, float m2, float range, T* __restrict__ y,
                         int pitch) {
  const long total = (long)B * HW;
  for (long p = (long)blockIdx.x * blockDim.x + threadIdx.x; p < total; p += (long)gridDim.x * blockDim.x) {
    const long b = p / HW, q = p - b * HW;
    const float* s = x + b * 3 * HW + q;
    stf<T>(y, p * pitch + 0, (s[0] - m0) * range);
    stf<T>(y, p * pitch + 1, (s[HW] - m1) * range);
    stf<T>(y, p * pitch + 2, (s[2 * HW] - m2) * range);
  }
}

// in: [B][H][W][pitch] channels-last -> out: [B][3][H][W] fp32 planar, x / range + mean[c]
template <typename T>
__global__ void k_rgb_out(const T* __restrict__ x, int B, long HW, int pitch, float m0, float m1, float m2, float inv_range,
                          float* __restrict__ y) {
  const long total = (long)B * HW;
  for (long p = (long)blockIdx.x * blockDim.x + threadIdx.x; p < total; p += (long)gridDim.x * blockDim.x) {
    const long b = p / HW, q = p - b * HW;
    float* d = y + b * 3 * HW + q;
    d[0] = ldf<T>(x, p * pitch + 0) * inv_range + m0;
    d[HW] = ldf<T>(x, p * pitch + 1) * inv_range + m1;
    d[2 * HW] = ldf<T>(x, p * pitch + 2) * inv_range + m2;
  }
}

inline int grid_for(long n, int per_block) {
  long g = (n + per_block - 1) / per_block;
  const long cap = 148L * 16;
  return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

}  // namespace

extern "C" int ffsr_layernorm_strided(const void* x, long rows, int C, long x_pitch, const float* w, const float* b, void* y,
                                      long y_pitch, int in_dtype, int out_dtype, cudaStream_t stream) {
  FFSR_REQUIRE(x && w && b && y && rows > 0 && C > 0 && x_pitch >= C && y_pitch >= C, FFSR_ERR_ARG,
               "layernorm_strided: rows=%ld C=%d pitches %ld / %ld", rows, C, x_pitch, y_pitch);
  const int grid = grid_for(rows, 8);
  const bool ib = in_dtype == FFSR_DT_BF16, ob = out_dtype == FFSR_DT_BF16;
  if (ib && ob) k_layernorm_strided<__nv_bfloat16, __nv_bfloat16><<<grid, 256, 0, stream>>>((const __nv_bfloat16*)x, rows, C, x_pitch, w, b, (__nv_bfloat16*)y, y_pitch);
  else if (ib) k_layernorm_strided<__nv_bfloat16, float><<<grid, 256, 0, stream>>>((const __nv_bfloat16*)x, rows, C, x_pitch, w, b, (float*)y, y_pitch);
  else if (ob && (C & 3) == 0 && (x_pitch & 3) == 0 && (y_pitch & 3) == 0 && ((uintptr_t)x & 15) == 0 && ((uintptr_t)y & 7) == 0 &&
           ((uintptr_t)w & 15) == 0 && ((uintptr_t)b & 15) == 0)
    k_layernorm_strided_v4<<<grid, 256, 0, stream>>>((const float*)x, rows, C, x_pitch, w, b, (__nv_bfloat16*)y, y_pitch);
  else if (ob) k_layernorm_strided<float, __nv_bfloat16><<<grid, 256, 0, stream>>>((const float*)x, rows, C, x_pitch, w, b, (__nv_bfloat16*)y, y_pitch);
  else k_layernorm_strided<float, float><<<grid, 256, 0, stream>>>((const float*)x, rows, C, x_pitch, w, b, (float*)y, y_pitch);
  return ffsr_check_launch("k_layernorm_strided");
}

extern "C" int ffsr_leaky_relu(void* x, long rows, int C, long pitch, float slope, int dtype, cudaStream_t stream) {
  FFSR_REQUIRE(x && rows > 0 && C > 0 && pitch >= C, FFSR_ERR_ARG, "leaky_relu: rows=%ld C=%d pitch=%ld", rows, C, pitch);
  const int grid = grid_for(rows * C, 256 * 4);
  if (dtype == FFSR_DT_BF16) k_leaky_relu<__nv_bfloat16><<<grid, 256, 0, stream>>>((__nv_bfloat16*)x, rows, C, pitch, slope);
  else k_leaky_relu<float><<<grid, 256, 0, stream>>>((float*)x, rows, C, pitch, slope);
  return ffsr_check_launch("k_leaky_relu");
}

extern "C" int ffsr_pixel_shuffle2(const void* x, int B, int H, int W, int C, void* y, int dtype, cudaStream_t stream) {
  FFSR_REQUIRE(x && y && B > 0 && H > 0 && W > 0 && C > 0, FFSR_ERR_ARG, "pixel_shuffle2: B=%d H=%d W=%d C=%d", B, H, W, C);
  const int grid = grid_for((long)B * 4 * H * W * C, 256 * 4);
  if (dtype == FFSR_DT_BF16) k_pixel_shuffle2<__nv_bfloat16><<<grid, 256, 0, stream>>>((const __nv_bfloat16*)x, B, H, W, C, (__nv_bfloat16*)y);
  else k_pixel_shuffle2<float><<<grid, 256, 0, stream>>>((const float*)x, B, H, W, C, (float*)y);
  return ffsr_check_launch("k_pixel_shuffle2");
}

extern "C" int ffsr_rgb_shift_in(const float* x, int B, int H, int W, const float* mean3_host, float range, void* y, int pitch, int dtype,
                                 cudaStream_t stream) {
  FFSR_REQUIRE(x && y && mean3_host && B > 0 && H > 0 && W > 0 && pitch >= 3, FFSR_ERR_ARG, "rgb_shift_in: bad argument");
  const int grid = grid_for((long)B * H * W, 256);
  if (dtype == FFSR_DT_BF16)
    k_rgb_in<__nv_bfloat16><<<grid, 256, 0, stream>>>(x, B, (long)H * W, mean3_host[0], mean3_host[1], mean3_host[2], range, (__nv_bfloat16*)y, pitch);
  else k_rgb_in<float><<<grid, 256, 0, stream>>>(x, B, (long)H * W, mean3_host[0], mean3_host[1], mean3_host[2], range, (float*)y, pitch);
  return ffsr_check_launch("k_rgb_in");
}

extern "C" int ffsr_rgb_shift_out(const void* x, int B, int H, int W, int pitch, const float* mean3_host, float range, float* y, int dtype,
                                  cudaStream_t stream) {
  FFSR_REQUIRE(x && y && mean3_host && B > 0 && H > 0 && W > 0 && pitch >= 3 && range != 0.f, FFSR_ERR_ARG, "rgb_shift_out: bad argument");
  const int grid = grid_for((long)B * H * W, 256);
  if (dtype == FFSR_DT_BF16)
    k_rgb_out<__nv_bfloat16><<<grid, 256, 0, stream>>>((const __nv_bfloat16*)x, B, (long)H * W, pitch, mean3_host[0], mean3_host[1], mean3_host[2], 1.0f / range, y);
  else k_rgb_out<float><<<grid, 256, 0, stream>>>((const float*)x, B, (long)H * W, pitch, mean3_host[0], mean3_host[1], mean3_host[2], 1.0f / range, y);
  return ffsr_check_launch("k_rgb_out");
}
