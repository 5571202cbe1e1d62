// Train-mode / backward kernels of the fusion hot path (fp32 CUDA-core versions):
//   * conv weight gradient (1x1 / 3x3) as a pixel-reduction GEMM  dW[tap][ci][co] = sum_p X[p+tap][ci] dY[p][co]
//   * channel sums (bias gradients)
//   * pointwise activation forward / backward on the saved pre-activation
//   * LayerNorm backward, BatchNorm batch statistics and backward reductions
//   * token attention (T tokens per LR pixel) forward with saved probabilities + dropout, and backward
// They are the autograd counterparts of nn.Conv2d / nn.GELU / nn.LayerNorm / nn.BatchNorm2d /
// nn.MultiheadAttention as the reference composes them (src/models/enhanced_fusion_v2.py:681-799,
// large_kernel_attention.py:92-149, 207-244, 324-426); the reference itself relies on ATen autograd.
#include "common.cuh"
#include "../../include/ffsr_b200.h"

namespace {

__device__ __forceinline__ float ld_any(const void* base, int dtype, long long off) {
  return dtype == FFSR_DT_BF16 ? __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(base)[off])
                               : reinterpret_cast<const float*>(base)[off];
}
__device__ __forceinline__ void st_any(void* base, int dtype, long long off, float v) {
  if (dtype == FFSR_DT_BF16) reinterpret_cast<__nv_bfloat16*>(base)[off] = __float2bfloat16_rn(v);
  else reinterpret_cast<float*>(base)[off] = v;
}

// 8 consecutive elements <-> fp32 registers (16-byte accesses for bf16, 2 x 16 bytes for fp32); p must be 16B aligned
template <typename T>
__device__ __forceinline__ void load8(const T* p, float (&f)[8]);
template <>
__device__ __forceinline__ void load8<float>(const float* p, float (&f)[8]) {
  const float4 a = reinterpret_cast<const float4*>(p)[0], b = reinterpret_cast<const float4*>(p)[1];
  f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w; f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
}
template <>
__device__ __forceinline__ void load8<__nv_bfloat16>(const __nv_bfloat16* p, float (&f)[8]) {
  const uint4 u = *reinterpret_cast<const uint4*>(p);
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const float2 f2 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w[k]));
    f[2 * k] = f2.x; f[2 * k + 1] = f2.y;
  }
}
template <typename T>
__device__ __forceinline__ void store8(T* p, const float (&f)[8]);
template <>
__device__ __forceinline__ void store8<float>(float* p, const float (&f)[8]) {
  reinterpret_cast<float4*>(p)[0] = make_float4(f[0], f[1], f[2], f[3]);
  reinterpret_cast<float4*>(p)[1] = make_float4(f[4], f[5], f[6], f[7]);
}
template <>
__device__ __forceinline__ void store8<__nv_bfloat16>(__nv_bfloat16* p, const float (&f)[8]) {
  uint32_t w[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    __nv_bfloat162 h = __floats2bfloat162_rn(f[2 * k], f[2 * k + 1]);
    w[k] = *reinterpret_cast<uint32_t*>(&h);
  }
  *reinterpret_cast<uint4*>(p) = make_uint4(w[0], w[1], w[2], w[3]);
}

// ------------------------------------------------------------------------------------
// conv weight gradient.  grid = (pixel chunks, taps, ci tiles * co tiles); 256 threads as a
// 16x16 grid of (TM/16)x(TN/16) register micro-tiles; K = pixels, staged 16 at a time.
// ------------------------------------------------------------------------------------
constexpr int WG_KP = 16;

template <int NI>
__device__ __forceinline__ void load_frag(const float* row, int t, float (&o)[NI]) {
  if constexpr (NI >= 4) {
#pragma unroll
    for (int g = 0; g < NI / 4; ++g) {
      const float4 v = *reinterpret_cast<const float4*>(row + g * 64 + 4 * t);
      o[4 * g] = v.x; o[4 * g + 1] = v.y; o[4 * g + 2] = v.z; o[4 * g + 3] = v.w;
    }
  } else if constexpr (NI == 2) {
    const float2 v = *reinterpret_cast<const float2*>(row + 2 * t);
    o[0] = v.x; o[1] = v.y;
  } else {
    o[0] = row[t];
  }
}
template <int NI>
__device__ __forceinline__ int frag_index(int t, int j) {
  if constexpr (NI >= 4) return (j / 4) * 64 + 4 * t + (j % 4);
  else if constexpr (NI == 2) return 2 * t + j;
  else return t;
}

template <int TM, int TN>
__global__ void __launch_bounds__(256) k_conv_wgrad(const ffsr_wgrad_params p, long chunk, float* __restrict__ part) {
  constexpr int MI = TM / 16, NI = TN / 16;
  __shared__ __align__(16) float sX[WG_KP][TM];
  __shared__ __align__(16) float sD[WG_KP][TN];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int tap = blockIdx.y;
  const int pad = p.ksize / 2;
  const int dy = tap / p.ksize - pad, dx = tap % p.ksize - pad;
  const int co_tiles = (p.Cout + TN - 1) / TN;
  const int ci0 = (blockIdx.z / co_tiles) * TM, co0 = (blockIdx.z % co_tiles) * TN;
  const long NP = (long)p.N * p.H * p.W;
  const long p_begin = (long)blockIdx.x * chunk;
  const long p_end = min(NP, p_begin + chunk);
  const bool x_cl = (p.x_sC == 1);

  float acc[MI][NI];
#pragma unroll
  for (int i = 0; i < MI; ++i)
#pragma unroll
    for (int j = 0; j < NI; ++j) acc[i][j] = 0.f;

  for (long pb = p_begin; pb < p_end; pb += WG_KP) {
    for (int i = tid; i < WG_KP * TM; i += 256) {
      int k, m;
      if (x_cl) { k = i / TM; m = i % TM; } else { m = i / WG_KP; k = i % WG_KP; }
      const long pix = pb + k;
      float v = 0.f;
      const int c = ci0 + m;
      if (pix < p_end && c < p.Cin) {
        const int x = (int)(pix % p.W);
        const long r = pix / p.W;
        const int y = (int)(r % p.H);
        const int n = (int)(r / p.H);
        const int yy = y + dy, xx = x + dx;
        if (yy >= 0 && yy < p.H && xx >= 0 && xx < p.W)
          v = ld_any(p.x, p.x_dtype, (long long)n * p.x_sN + (long long)yy * p.x_sY + (long long)xx * p.x_sX + (long long)c * p.x_sC);
      }
      sX[k][m] = v;
    }
    for (int i = tid; i < WG_KP * TN; i += 256) {
      const int k = i / TN, m = i % TN;
      const long pix = pb + k;
      float v = 0.f;
      const int c = co0 + m;
      if (pix < p_end && c < p.Cout) {
        const int x = (int)(pix % p.W);
        const long r = pix / p.W;
        const int y = (int)(r % p.H);
        const int n = (int)(r / p.H);
        v = ld_any(p.dy, p.dy_dtype, (long long)n * p.dy_sN + (long long)y * p.dy_sY + (long long)x * p.dy_sX + c);
      }
      sD[k][m] = v;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < WG_KP; ++k) {
      float a[MI], b[NI];
      load_frag<MI>(&sX[k][0], ty, a);
      load_frag<NI>(&sD[k][0], tx, b);
#pragma unroll
      for (int i = 0; i < MI; ++i)
#pragma unroll
        for (int j = 0; j < NI; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < MI; ++i) {
    const int ci = ci0 + frag_index<MI>(ty, i);
    if (ci >= p.Cin) continue;
#pragma unroll
    for (int j = 0; j < NI; ++j) {
      const int co = co0 + frag_index<NI>(tx, j);
      if (co < p.Cout) part[(((long)blockIdx.x * gridDim.y + tap) * p.Cin + ci) * p.Cout + co] = acc[i][j];
    }
  }
}

// register tile of the weight-gradient kernel and its pixel split P (chunk pixels per block): a function of the shape
struct WgradPlan {
  int TM, TN;
  long P, chunk;
};
inline WgradPlan wgrad_plan(int N, int H, int W, int Cin, int Cout, int ksize) {
  WgradPlan pl;
  pl.TM = Cin > 64 ? 128 : Cin > 32 ? 64 : Cin > 16 ? 32 : 16;
  pl.TN = Cout > 64 ? 128 : Cout > 32 ? 64 : Cout > 16 ? 32 : 16;
  const int taps = ksize * ksize;
  const int tiles = ceil_div(Cin, pl.TM) * ceil_div(Cout, pl.TN);
  const long NP = (long)N * H * W;
  long P = ceil_div(148 * 6, taps * tiles);
  const long maxP = (NP + 511) / 512;
  if (P > maxP) P = maxP;
  if (P < 1) P = 1;
  long chunk = (NP + P - 1) / P;
  chunk = (chunk + WG_KP - 1) / WG_KP * WG_KP;
  pl.P = (NP + chunk - 1) / chunk;
  pl.chunk = chunk;
  return pl;
}

// partials [P][taps][Cin][Cout] into part (reduced in pixel-chunk order by the caller)
template <int TM, int TN>
int launch_wgrad(const ffsr_wgrad_params& p, const WgradPlan& pl, float* part, cudaStream_t stream) {
  const int taps = p.ksize * p.ksize;
  dim3 grid((unsigned)pl.P, taps, ceil_div(p.Cin, TM) * ceil_div(p.Cout, TN));
  k_conv_wgrad<TM, TN><<<grid, 256, 0, stream>>>(p, pl.chunk, part);
  return ffsr_check_launch("conv2d_wgrad");
}

template <int TM>
int dispatch_wgrad_n(const ffsr_wgrad_params& p, const WgradPlan& pl, float* part, cudaStream_t s) {
  if (pl.TN == 128) return launch_wgrad<TM, 128>(p, pl, part, s);
  if (pl.TN == 64) return launch_wgrad<TM, 64>(p, pl, part, s);
  if (pl.TN == 32) return launch_wgrad<TM, 32>(p, pl, part, s);
  return launch_wgrad<TM, 16>(p, pl, part, s);
}

// ------------------------------------------------------------------------------------
// channel sums of a channels-last tensor: out[c] += sum_{n,y,x} v[n,y,x,c]
// ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_colsum(const void* __restrict__ v, int dtype, long long sN, long long sY,
                                                long long sX, int H, int W, long NP, int C, long rows_per_block,
                                                float* __restrict__ part) {
  extern __shared__ float sred[];          // [rows_in_block][CT]
  const int CT = blockDim.x;               // channel threads (power of two <= 64)
  const int RT = blockDim.y;
  const int c = blockIdx.y * CT + threadIdx.x;
  const long r0 = (long)blockIdx.x * rows_per_block;
  const long r1 = min(NP, r0 + rows_per_block);
  float acc = 0.f;
  if (c < C) {
    for (long r = r0 + threadIdx.y; r < r1; r += RT) {
      const int x = (int)(r % W);
      const long q = r / W;
      const int y = (int)(q % H);
      const long n = q / H;
      acc += ld_any(v, dtype, n * sN + (long long)y * sY + (long long)x * sX + c);
    }
  }
  sred[threadIdx.y * CT + threadIdx.x] = acc;
  __syncthreads();
  if (threadIdx.y == 0 && c < C) {
    float s = 0.f;
    for (int i = 0; i < RT; ++i) s += sred[i * CT + threadIdx.x];
    part[(long)blockIdx.x * C + c] = s;
  }
}

// dense channels-last fast path: rows of `pitch` elements, no index arithmetic per element, VEC channels per thread
template <typename T, int VEC>
__global__ void __launch_bounds__(256) k_colsum_rows(const T* __restrict__ v, long NP, int C, long pitch, int TPR,
                                                     long rows_per_block, float* __restrict__ part) {
  __shared__ float sred[256 * VEC];
  const int lane_c = threadIdx.x % TPR, rt = threadIdx.x / TPR, RT = 256 / TPR;
  const int c0 = lane_c * VEC;
  const long r0 = (long)blockIdx.x * rows_per_block, r1 = min(NP, r0 + rows_per_block);
  float acc[VEC];
#pragma unroll
  for (int i = 0; i < VEC; ++i) acc[i] = 0.f;
  if (c0 < C) {
    long r = r0 + rt;
    for (; r + 3 * RT < r1; r += 4 * RT) {
      float t[4][VEC];
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int i = 0; i < VEC; ++i) t[u][i] = (c0 + i < C) ? to_f32<T>(v[(r + (long)u * RT) * pitch + c0 + i]) : 0.f;
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int i = 0; i < VEC; ++i) acc[i] += t[u][i];
    }
    for (; r < r1; r += RT)
#pragma unroll
      for (int i = 0; i < VEC; ++i) acc[i] += (c0 + i < C) ? to_f32<T>(v[r * pitch + c0 + i]) : 0.f;
  }
#pragma unroll
  for (int i = 0; i < VEC; ++i) sred[(rt * TPR + lane_c) * VEC + i] = acc[i];
  __syncthreads();
  if (rt == 0 && c0 < C) {
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      if (c0 + i >= C) continue;
      float s = 0.f;
      for (int k = 0; k < RT; ++k) s += sred[(k * TPR + lane_c) * VEC + i];
      part[(long)blockIdx.x * C + c0 + i] = s;
    }
  }
}

// ------------------------------------------------------------------------------------
// pointwise activations
// ------------------------------------------------------------------------------------
__device__ __forceinline__ float act_grad(float x, int act) {
  switch (act) {
    case ACT_GELU: {
      const float cdf = 0.5f * (1.0f + erff(x * 0.70710678118654752440f));
      const float pdf = 0.39894228040143267794f * expf(-0.5f * x * x);
      return cdf + x * pdf;
    }
    case ACT_RELU: return x > 0.f ? 1.f : 0.f;
    case ACT_SIGMOID: {
      const float s = sigmoid_acc(x);
      return s * (1.f - s);
    }
    default: return 1.f;
  }
}

// 8 elements per thread-iteration (vector accesses) + scalar tail
template <typename T>
__global__ void __launch_bounds__(256) k_act_fwd(const T* __restrict__ x, T* __restrict__ y, long n, int act) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  const long stride = (long)gridDim.x * blockDim.x;
  const long n8 = n >> 3;
  for (long k = i; k < n8; k += stride) {
    float f[8];
    load8<T>(x + 8 * k, f);
#pragma unroll
    for (int j = 0; j < 8; ++j) f[j] = apply_act(f[j], act);
    store8<T>(y + 8 * k, f);
  }
  for (long k = 8 * n8 + i; k < n; k += stride) y[k] = from_f32<T>(apply_act(to_f32<T>(x[k]), act));
}
template <typename T>
__global__ void __launch_bounds__(256) k_act_bwd(const T* __restrict__ x, const T* __restrict__ dy, T* __restrict__ dx, long n,
                                                 int act) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  const long stride = (long)gridDim.x * blockDim.x;
  const long n8 = n >> 3;
  for (long k = i; k < n8; k += stride) {
    float f[8], g[8];
    load8<T>(x + 8 * k, f);
    load8<T>(dy + 8 * k, g);
#pragma unroll
    for (int j = 0; j < 8; ++j) g[j] *= act_grad(f[j], act);
    store8<T>(dx + 8 * k, g);
  }
  for (long k = 8 * n8 + i; k < n; k += stride) dx[k] = from_f32<T>(to_f32<T>(dy[k]) * act_grad(to_f32<T>(x[k]), act));
}

// ------------------------------------------------------------------------------------
// LayerNorm backward: one warp per row; per-block dw/db (warps summed in order) to slot blockIdx.x of part [grid][2E].
// ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_layernorm_bwd(const float* __restrict__ x, const float* __restrict__ dy,
                                                       long rows, int E, const float* __restrict__ w,
                                                       float* __restrict__ dx, float* __restrict__ part) {
  extern __shared__ float sacc[];            // [warps][2][E]
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, wpb = blockDim.x >> 5;
  const int per = E / 32;
  float lw[8], ldw[8], ldb[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) { ldw[i] = 0.f; ldb[i] = 0.f; lw[i] = (i < per) ? w[lane + 32 * i] : 0.f; }
  for (long row = (long)blockIdx.x * wpb + wib; row < rows; row += (long)gridDim.x * wpb) {
    const float* xr = x + row * E;
    const float* gr = dy + row * E;
    float v[8], g[8];
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i)
      if (i < per) { v[i] = xr[lane + 32 * i]; g[i] = gr[lane + 32 * i]; sum += v[i]; }
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
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i)
      if (i < per) {
        v[i] *= rstd;                               // xhat
        ldw[i] += g[i] * v[i];
        ldb[i] += g[i];
        g[i] *= lw[i];                              // dy * w
        s1 += g[i];
        s2 += g[i] * v[i];
      }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      s1 += __shfl_xor_sync(0xffffffffu, s1, o);
      s2 += __shfl_xor_sync(0xffffffffu, s2, o);
    }
    s1 /= (float)E;
    s2 /= (float)E;
#pragma unroll
    for (int i = 0; i < 8; ++i)
      if (i < per) dx[row * E + lane + 32 * i] = rstd * (g[i] - s1 - v[i] * s2);
  }
#pragma unroll
  for (int i = 0; i < 8; ++i)
    if (i < per) {
      sacc[wib * 2 * E + lane + 32 * i] = ldw[i];
      sacc[wib * 2 * E + E + lane + 32 * i] = ldb[i];
    }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * E; i += blockDim.x) {
    float s = 0.f;
    for (int k = 0; k < wpb; ++k) s += sacc[k * 2 * E + i];
    part[(long)blockIdx.x * 2 * E + i] = s;
  }
}

// ------------------------------------------------------------------------------------
// BatchNorm (train mode) on channels-last [G][R][C]: G independent statistic groups
// (one LKABlock call each), R = rows (images*H*W) per group.
//   stats : sum[g][c], sumsq[g][c]  (fp64 accumulation -> mean / biased var on the host side)
//   bwd   : sdy[g][c] = sum dy, sdyx[g][c] = sum dy * xhat   (xhat from mean / rstd)
// Both write slot blockIdx.x of part [grid.x][2][G][C] (the two sums of every (g, c)), reduced by k_sum_slots.
// ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_bn_stats(const float* __restrict__ x, long R, int C, long rows_per_block,
                                                  double* __restrict__ part) {
  extern __shared__ double sbn[];            // [2][RT][CT]
  const int CT = blockDim.x, RT = blockDim.y;
  const int c = blockIdx.y * CT + threadIdx.x;
  const int g = blockIdx.z;
  const long r0 = (long)blockIdx.x * rows_per_block, r1 = min(R, r0 + rows_per_block);
  const float* base = x + (long)g * R * C;
  float a = 0.f, b = 0.f;
  double da = 0.0, dbb = 0.0;
  int cnt = 0;
  if (c < C)
    for (long r = r0 + threadIdx.y; r < r1; r += RT) {
      const float v = base[r * C + c];
      a += v;
      b = fmaf(v, v, b);
      if (++cnt == 64) { da += a; dbb += b; a = 0.f; b = 0.f; cnt = 0; }
    }
  da += a; dbb += b;
  sbn[threadIdx.y * CT + threadIdx.x] = da;
  sbn[(RT + threadIdx.y) * CT + threadIdx.x] = dbb;
  __syncthreads();
  if (threadIdx.y == 0 && c < C) {
    double s = 0.0, q = 0.0;
    for (int i = 0; i < RT; ++i) { s += sbn[i * CT + threadIdx.x]; q += sbn[(RT + i) * CT + threadIdx.x]; }
    double* slot = part + (long)blockIdx.x * 2 * gridDim.z * C;
    slot[(long)g * C + c] = s;
    slot[(long)(gridDim.z + g) * C + c] = q;
  }
}

__global__ void __launch_bounds__(256) k_bn_bwd_reduce(const float* __restrict__ x, const float* __restrict__ dy, long R,
                                                       int C, long rows_per_block, const float* __restrict__ mean,
                                                       const float* __restrict__ rstd, float* __restrict__ part) {
  extern __shared__ float sbr[];             // [2][RT][CT]
  const int CT = blockDim.x, RT = blockDim.y;
  const int c = blockIdx.y * CT + threadIdx.x;
  const int g = blockIdx.z;
  const long r0 = (long)blockIdx.x * rows_per_block, r1 = min(R, r0 + rows_per_block);
  const float* xb = x + (long)g * R * C;
  const float* gb = dy + (long)g * R * C;
  float a = 0.f, b = 0.f;
  if (c < C) {
    const float mu = mean[(long)g * C + c], rs = rstd[(long)g * C + c];
    for (long r = r0 + threadIdx.y; r < r1; r += RT) {
      const float d = gb[r * C + c];
      a += d;
      b = fmaf(d, (xb[r * C + c] - mu) * rs, b);
    }
  }
  sbr[threadIdx.y * CT + threadIdx.x] = a;
  sbr[(RT + threadIdx.y) * CT + threadIdx.x] = b;
  __syncthreads();
  if (threadIdx.y == 0 && c < C) {
    float s = 0.f, q = 0.f;
    for (int i = 0; i < RT; ++i) { s += sbr[i * CT + threadIdx.x]; q += sbr[(RT + i) * CT + threadIdx.x]; }
    float* slot = part + (long)blockIdx.x * 2 * gridDim.z * C;
    slot[(long)g * C + c] = s;
    slot[(long)(gridDim.z + g) * C + c] = q;
  }
}

// y = (x - mean) * rstd * w + b   (per group g, channel c); float4 over channels (C % 4 == 0)
__global__ void __launch_bounds__(256) k_bn_apply(const float* __restrict__ x, long R, int C, int G, const float* __restrict__ mean,
                                                  const float* __restrict__ rstd, const float* __restrict__ w,
                                                  const float* __restrict__ b, float* __restrict__ y) {
  const int C4 = C >> 2;
  const long per_g = R * C4, total = (long)G * per_g;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int c = (int)(i % C4) << 2;
    const long gc = (i / per_g) * C + c;
    const float4 xv = reinterpret_cast<const float4*>(x)[i];
    const float4 mu = *reinterpret_cast<const float4*>(mean + gc), rs = *reinterpret_cast<const float4*>(rstd + gc);
    const float4 wv = *reinterpret_cast<const float4*>(w + c), bv = *reinterpret_cast<const float4*>(b + c);
    float4 o;
    o.x = fmaf((xv.x - mu.x) * rs.x, wv.x, bv.x);
    o.y = fmaf((xv.y - mu.y) * rs.y, wv.y, bv.y);
    o.z = fmaf((xv.z - mu.z) * rs.z, wv.z, bv.z);
    o.w = fmaf((xv.w - mu.w) * rs.w, wv.w, bv.w);
    reinterpret_cast<float4*>(y)[i] = o;
  }
}
// dx = w*rstd * (dy - sdy/R - xhat * sdyx/R)
__global__ void __launch_bounds__(256) k_bn_bwd_apply(const float* __restrict__ x, const float* __restrict__ dy, long R, int C,
                                                      int G, const float* __restrict__ mean, const float* __restrict__ rstd,
                                                      const float* __restrict__ w, const float* __restrict__ sdy,
                                                      const float* __restrict__ sdyx, float* __restrict__ dx) {
  const int C4 = C >> 2;
  const long per_g = R * C4, total = (long)G * per_g;
  const float invR = 1.0f / (float)R;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int c = (int)(i % C4) << 2;
    const long gc = (i / per_g) * C + c;
    const float4 xv = reinterpret_cast<const float4*>(x)[i], gv = reinterpret_cast<const float4*>(dy)[i];
    const float* xs = &xv.x;
    const float* gs = &gv.x;
    float o[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float rs = rstd[gc + k];
      const float xh = (xs[k] - mean[gc + k]) * rs;
      o[k] = w[c + k] * rs * (gs[k] - sdy[gc + k] * invR - xh * sdyx[gc + k] * invR);
    }
    reinterpret_cast<float4*>(dx)[i] = make_float4(o[0], o[1], o[2], o[3]);
  }
}

// ------------------------------------------------------------------------------------
// Token attention, train mode.  qkv[B][T][HW][3E] (token-major), head_dim 16.
//   fwd: probs[B][HW][heads][T][T] (pre-dropout softmax) saved; ctx = dropout(probs) v
//   bwd: kernel 1 (per query): dS -> scratch, dq;  kernel 2 (per key): dk, dv
// Dropout keep decision is a counter-based hash of (seed, element index): the backward
// regenerates the same mask.  nn.MultiheadAttention(dropout=0.1): large_kernel_attention.py:192-197, 294-299.
// ------------------------------------------------------------------------------------
__device__ __forceinline__ float keep_scale(unsigned long long seed, unsigned long long idx, float drop_p) {
  if (drop_p <= 0.f) return 1.f;
  unsigned long long z = seed + idx * 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  z ^= z >> 31;
  const float u = (float)(z >> 40) * (1.0f / 16777216.0f);
  return u < drop_p ? 0.f : 1.0f / (1.0f - drop_p);
}

template <int T>
__global__ void k_tokattn_fwd(const float* __restrict__ qkv, int B, long HW, int E, float* __restrict__ ctx,
                              float* __restrict__ probs, float drop_p, unsigned long long seed,
                              const unsigned long long* __restrict__ seed_dev) {
  if (seed_dev) seed += *seed_dev;
  const int heads = E / 16;
  const long it = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (it >= (long)B * HW * T * heads) return;
  const int h = (int)(it % heads);
  long rest = it / heads;
  const int qt = (int)(rest % T);
  rest /= T;
  const long p = rest % HW;
  const int b = (int)(rest / HW);
  const long tstride = HW * 3 * E;
  const float* base = qkv + ((long)b * T * HW + p) * 3 * E + h * 16;
  float q[16];
#pragma unroll
  for (int d = 0; d < 16; ++d) q[d] = base[qt * tstride + d];
  float sc[T];
  float mx = -INFINITY;
#pragma unroll
  for (int j = 0; j < T; ++j) {
    float a = 0.f;
#pragma unroll
    for (int d = 0; d < 16; ++d) a = fmaf(q[d], base[j * tstride + E + d], a);
    sc[j] = a * 0.25f;
    mx = fmaxf(mx, sc[j]);
  }
  float den = 0.f;
#pragma unroll
  for (int j = 0; j < T; ++j) { sc[j] = expf(sc[j] - mx); den += sc[j]; }
  const float inv = 1.0f / den;
  const long prow = ((((long)b * HW + p) * heads + h) * T + qt) * T;
  float o[16];
#pragma unroll
  for (int d = 0; d < 16; ++d) o[d] = 0.f;
#pragma unroll
  for (int j = 0; j < T; ++j) {
    const float pj = sc[j] * inv;
    probs[prow + j] = pj;
    const float pd = pj * keep_scale(seed, (unsigned long long)(prow + j), drop_p);
#pragma unroll
    for (int d = 0; d < 16; ++d) o[d] = fmaf(pd, base[j * tstride + 2 * E + d], o[d]);
  }
  float* op = ctx + (((long)b * T + qt) * HW + p) * E + h * 16;
#pragma unroll
  for (int d = 0; d < 16; ++d) op[d] = o[d];
}

template <int T>
__global__ void k_tokattn_bwd_q(const float* __restrict__ qkv, const float* __restrict__ probs,
                                const float* __restrict__ dctx, int B, long HW, int E, float* __restrict__ ds,
                                float* __restrict__ dqkv, float drop_p, unsigned long long seed,
                                const unsigned long long* __restrict__ seed_dev) {
  if (seed_dev) seed += *seed_dev;
  const int heads = E / 16;
  const long it = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (it >= (long)B * HW * T * heads) return;
  const int h = (int)(it % heads);
  long rest = it / heads;
  const int qt = (int)(rest % T);
  rest /= T;
  const long p = rest % HW;
  const int b = (int)(rest / HW);
  const long tstride = HW * 3 * E;
  const float* base = qkv + ((long)b * T * HW + p) * 3 * E + h * 16;
  const float* gp = dctx + (((long)b * T + qt) * HW + p) * E + h * 16;
  float g[16];
#pragma unroll
  for (int d = 0; d < 16; ++d) g[d] = gp[d];
  const long prow = ((((long)b * HW + p) * heads + h) * T + qt) * T;
  float dp[T], pr[T];
  float dot = 0.f;
#pragma unroll
  for (int j = 0; j < T; ++j) {
    float a = 0.f;
#pragma unroll
    for (int d = 0; d < 16; ++d) a = fmaf(g[d], base[j * tstride + 2 * E + d], a);
    pr[j] = probs[prow + j];
    dp[j] = a * keep_scale(seed, (unsigned long long)(prow + j), drop_p);
    dot = fmaf(pr[j], dp[j], dot);
  }
  float dq[16];
#pragma unroll
  for (int d = 0; d < 16; ++d) dq[d] = 0.f;
#pragma unroll
  for (int j = 0; j < T; ++j) {
    const float s = pr[j] * (dp[j] - dot) * 0.25f;
    ds[prow + j] = s;
#pragma unroll
    for (int d = 0; d < 16; ++d) dq[d] = fmaf(s, base[j * tstride + E + d], dq[d]);
  }
  float* oq = dqkv + (((long)b * T + qt) * HW + p) * 3 * E + h * 16;
#pragma unroll
  for (int d = 0; d < 16; ++d) oq[d] = dq[d];
}

template <int T>
__global__ void k_tokattn_bwd_kv(const float* __restrict__ qkv, const float* __restrict__ probs,
                                 const float* __restrict__ ds, const float* __restrict__ dctx, int B, long HW, int E,
                                 float* __restrict__ dqkv, float drop_p, unsigned long long seed,
                                const unsigned long long* __restrict__ seed_dev) {
  if (seed_dev) seed += *seed_dev;
  const int heads = E / 16;
  const long it = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (it >= (long)B * HW * T * heads) return;
  const int h = (int)(it % heads);
  long rest = it / heads;
  const int j = (int)(rest % T);          // key / value token
  rest /= T;
  const long p = rest % HW;
  const int b = (int)(rest / HW);
  const long tstride = HW * 3 * E;
  const float* base = qkv + ((long)b * T * HW + p) * 3 * E + h * 16;
  const long pbase = (((long)b * HW + p) * heads + h) * T * T;
  float dk[16], dv[16];
#pragma unroll
  for (int d = 0; d < 16; ++d) { dk[d] = 0.f; dv[d] = 0.f; }
#pragma unroll
  for (int qt = 0; qt < T; ++qt) {
    const float s = ds[pbase + qt * T + j];
    const float pd = probs[pbase + qt * T + j] * keep_scale(seed, (unsigned long long)(pbase + qt * T + j), drop_p);
    const float* gp = dctx + (((long)b * T + qt) * HW + p) * E + h * 16;
#pragma unroll
    for (int d = 0; d < 16; ++d) {
      dk[d] = fmaf(s, base[qt * tstride + d], dk[d]);
      dv[d] = fmaf(pd, gp[d], dv[d]);
    }
  }
  float* ok = dqkv + (((long)b * T + j) * HW + p) * 3 * E + h * 16;
#pragma unroll
  for (int d = 0; d < 16; ++d) { ok[E + d] = dk[d]; ok[2 * E + d] = dv[d]; }
}

// strided (NCHW / NHWC, fp32 / bf16) -> dense bf16 channels-last with the channel pitch padded to Cpad
__global__ void __launch_bounds__(256) k_to_bf16_nhwc(const void* __restrict__ src, int dtype, long long sN, long long sY,
                                                      long long sX, long long sC, int H, int W, int C, int Cpad,
                                                      long total, __nv_bfloat16* __restrict__ dst) {
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int c = (int)(i % Cpad);
    long r = i / Cpad;
    const int x = (int)(r % W);
    r /= W;
    const int y = (int)(r % H);
    const long n = r / H;
    const float v = c < C ? ld_any(src, dtype, n * sN + (long long)y * sY + (long long)x * sX + (long long)c * sC) : 0.f;
    dst[i] = __float2bfloat16_rn(v);
  }
}

// dense channels-last source (pixel pitch sX, channel stride 1): one thread per (pixel, 8-channel group), 16-byte stores
template <typename T>
__global__ void __launch_bounds__(256) k_to_bf16_rows(const T* __restrict__ src, long long sX, long NP, int C, int Cpad,
                                                      __nv_bfloat16* __restrict__ dst) {
  const int G = Cpad >> 3;
  const long total = NP * G;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const long pix = i / G;
    const int c0 = (int)(i - pix * G) << 3;
    const T* s = src + pix * sX + c0;
    uint32_t w[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float a = (c0 + 2 * k < C) ? to_f32<T>(s[2 * k]) : 0.f;
      const float b = (c0 + 2 * k + 1 < C) ? to_f32<T>(s[2 * k + 1]) : 0.f;
      __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
      w[k] = *reinterpret_cast<uint32_t*>(&h);
    }
    *reinterpret_cast<uint4*>(dst + pix * Cpad + c0) = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

// ------------------------------------------------------------------------------------
// bilinear resampling (align_corners=False) of dense channels-last tensors, forward and adjoint
// ------------------------------------------------------------------------------------
template <typename T, int VEC>
__global__ void __launch_bounds__(256) k_bilinear_fwd(const T* __restrict__ src, int h, int w, int C, T* __restrict__ dst,
                                                      int H, int W, long total) {
  const int G = C / VEC;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int cg = (int)(i % G);
    const long pix = i / G;
    const int X = (int)(pix % W), Y = (int)((pix / W) % H);
    const long n = pix / ((long)W * H);
    const BilinTap ty = bilin_tap(Y, h, H), tx = bilin_tap(X, w, W);
    const T* base = src + n * h * w * C + cg * VEC;
    const T* p00 = base + ((long)ty.i0 * w + tx.i0) * C;
    const T* p01 = base + ((long)ty.i0 * w + tx.i1) * C;
    const T* p10 = base + ((long)ty.i1 * w + tx.i0) * C;
    const T* p11 = base + ((long)ty.i1 * w + tx.i1) * C;
    T* o = dst + pix * C + cg * VEC;
#pragma unroll
    for (int k = 0; k < VEC; ++k)
      o[k] = from_f32<T>(ty.w0 * (tx.w0 * to_f32<T>(p00[k]) + tx.w1 * to_f32<T>(p01[k])) +
                         ty.w1 * (tx.w0 * to_f32<T>(p10[k]) + tx.w1 * to_f32<T>(p11[k])));
  }
}

// 8-channel vector versions (C % 8 == 0, 16-byte aligned rows)
template <typename T>
__global__ void __launch_bounds__(256) k_bilinear_fwd8(const T* __restrict__ src, int h, int w, int C, T* __restrict__ dst,
                                                       int H, int W, long total) {
  const int G = C >> 3;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int cg = (int)(i % G);
    const long pix = i / G;
    const int X = (int)(pix % W), Y = (int)((pix / W) % H);
    const long n = pix / ((long)W * H);
    const BilinTap ty = bilin_tap(Y, h, H), tx = bilin_tap(X, w, W);
    const T* base = src + n * h * w * C + cg * 8;
    float a[8], b[8], c[8], d[8], o[8];
    load8<T>(base + ((long)ty.i0 * w + tx.i0) * C, a);
    load8<T>(base + ((long)ty.i0 * w + tx.i1) * C, b);
    load8<T>(base + ((long)ty.i1 * w + tx.i0) * C, c);
    load8<T>(base + ((long)ty.i1 * w + tx.i1) * C, d);
#pragma unroll
    for (int k = 0; k < 8; ++k) o[k] = ty.w0 * (tx.w0 * a[k] + tx.w1 * b[k]) + ty.w1 * (tx.w0 * c[k] + tx.w1 * d[k]);
    store8<T>(dst + pix * C + cg * 8, o);
  }
}

// Candidate output indices per axis are visited in chunks of BL_MAXC (one chunk up to ~6x upscaling; any factor works).
constexpr int BL_MAXC = 16;

// candidates [lo, hi] of output indices whose taps may touch input index `i`
__device__ __forceinline__ void bilin_adjoint_range(int i, int in_size, int out_size, int& lo, int& hi) {
  const float inv_r = (float)out_size / (float)in_size;
  lo = max((int)floorf(((float)i - 0.5f) * inv_r - 0.5f) - 1, 0);
  hi = min((int)ceilf(((float)i + 1.5f) * inv_r - 0.5f) + 1, out_size - 1);
}

// weights of input index `i` in the taps of outputs lo .. lo + n - 1 (n = min(hi - lo + 1, BL_MAXC))
__device__ __forceinline__ int bilin_adjoint_taps(int i, int in_size, int out_size, int lo, int hi, float (&wt)[BL_MAXC]) {
  const int n = min(hi - lo + 1, BL_MAXC);
  for (int k = 0; k < BL_MAXC; ++k) {
    float wgt = 0.f;
    if (k < n) {
      const BilinTap t = bilin_tap(lo + k, in_size, out_size);
      if (t.i0 == i) wgt += t.w0;
      if (t.i1 == i) wgt += t.w1;
    }
    wt[k] = wgt;
  }
  return n;
}

template <typename T, int VEC>
__global__ void __launch_bounds__(256) k_bilinear_bwd(const T* __restrict__ gout, int H, int W, int C, T* __restrict__ gin,
                                                      int h, int w, long total) {
  const int G = C / VEC;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int cg = (int)(i % G);
    const long pix = i / G;
    const int x = (int)(pix % w), y = (int)((pix / w) % h);
    const long n = pix / ((long)w * h);
    float wy[BL_MAXC], wx[BL_MAXC];
    int ylo, yhi, xlo, xhi;
    bilin_adjoint_range(y, h, H, ylo, yhi);
    bilin_adjoint_range(x, w, W, xlo, xhi);
    float acc[VEC];
#pragma unroll
    for (int k = 0; k < VEC; ++k) acc[k] = 0.f;
    const T* base = gout + n * H * W * C + cg * VEC;
    for (int y0 = ylo; y0 <= yhi; y0 += BL_MAXC) {
      const int ny = bilin_adjoint_taps(y, h, H, y0, yhi, wy);
      for (int x0 = xlo; x0 <= xhi; x0 += BL_MAXC) {
        const int nx = bilin_adjoint_taps(x, w, W, x0, xhi, wx);
        for (int a = 0; a < ny; ++a) {
          if (wy[a] == 0.f) continue;
          for (int b = 0; b < nx; ++b) {
            const float wgt = wy[a] * wx[b];
            if (wgt == 0.f) continue;
            const T* p = base + ((long)(y0 + a) * W + x0 + b) * C;
#pragma unroll
            for (int k = 0; k < VEC; ++k) acc[k] = fmaf(wgt, to_f32<T>(p[k]), acc[k]);
          }
        }
      }
    }
    T* o = gin + pix * C + cg * VEC;
#pragma unroll
    for (int k = 0; k < VEC; ++k) o[k] = from_f32<T>(acc[k]);
  }
}

// ------------------------------------------------------------------------------------
// fused few-pass elementwise nodes of the training graph
// ------------------------------------------------------------------------------------
// out[p][c] = y[p][c] * g[p]        (SpatialGate / edge attention: a 1-channel map gating C channels)
// C % 8 == 0: 8 channels per thread-iteration with vector accesses
template <typename T>
__global__ void __launch_bounds__(256) k_gate_mul_fwd8(const T* __restrict__ y, const float* __restrict__ g, long NP, int C,
                                                       T* __restrict__ out) {
  const int G = C >> 3;
  const long total = NP * G;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const float gv = g[i / G];
    float f[8];
    load8<T>(y + 8 * i, f);
#pragma unroll
    for (int k = 0; k < 8; ++k) f[k] *= gv;
    store8<T>(out + 8 * i, f);
  }
}
// one warp-quarter (8 lanes) per pixel: each lane 8 channels per step, shuffle reduction for the gate gradient
template <typename T>
__global__ void __launch_bounds__(256) k_gate_mul_bwd8(const T* __restrict__ y, const float* __restrict__ g,
                                                       const T* __restrict__ gout, long NP, int C, T* __restrict__ dy,
                                                       float* __restrict__ dg) {
  const int sub = threadIdx.x & 7;
  const long pix0 = ((long)blockIdx.x * blockDim.x + threadIdx.x) >> 3;
  const long pstride = ((long)gridDim.x * blockDim.x) >> 3;
  const long trips = (NP + pstride - 1) / pstride;                 // uniform trip count: every lane joins the shuffles
  for (long it = 0; it < trips; ++it) {
    const long pix = pix0 + it * pstride;
    const bool live = pix < NP;
    float acc = 0.f;
    if (live) {
      const float gv = g[pix];
      for (int c = 8 * sub; c < C; c += 64) {
        float a[8], b[8];
        load8<T>(gout + pix * C + c, a);
        load8<T>(y + pix * C + c, b);
#pragma unroll
        for (int k = 0; k < 8; ++k) { acc = fmaf(a[k], b[k], acc); a[k] *= gv; }
        store8<T>(dy + pix * C + c, a);
      }
    }
    acc += __shfl_xor_sync(0xffffffffu, acc, 4);
    acc += __shfl_xor_sync(0xffffffffu, acc, 2);
    acc += __shfl_xor_sync(0xffffffffu, acc, 1);
    if (live && sub == 0) dg[pix] = acc;
  }
}

template <typename T>
__global__ void __launch_bounds__(256) k_gate_mul_fwd(const T* __restrict__ y, const float* __restrict__ g, long NP, int C,
                                                      T* __restrict__ out) {
  const int G = C >> 2;
  const long total = NP * G;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const long pix = i / G;
    const float gv = g[pix];
    const T* s = y + i * 4;
    T* o = out + i * 4;
#pragma unroll
    for (int k = 0; k < 4; ++k) o[k] = from_f32<T>(to_f32<T>(s[k]) * gv);
  }
}
// dy[p][c] = gout[p][c] * g[p];  dg[p] = sum_c gout[p][c] * y[p][c]   (one thread per pixel)
template <typename T>
__global__ void __launch_bounds__(128) k_gate_mul_bwd(const T* __restrict__ y, const float* __restrict__ g,
                                                      const T* __restrict__ gout, long NP, int C, T* __restrict__ dy,
                                                      float* __restrict__ dg) {
  for (long pix = (long)blockIdx.x * blockDim.x + threadIdx.x; pix < NP; pix += (long)gridDim.x * blockDim.x) {
    const float gv = g[pix];
    const T* ys = y + pix * C;
    const T* gs = gout + pix * C;
    T* o = dy + pix * C;
    float acc = 0.f;
    for (int c = 0; c < C; c += 4) {
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float go = to_f32<T>(gs[c + k]);
        acc = fmaf(go, to_f32<T>(ys[c + k]), acc);
        o[c + k] = from_f32<T>(go * gv);
      }
    }
    dg[pix] = acc;
  }
}

// vector versions (C % 8 == 0, 16-byte aligned): item i = (pixel, 8-channel group)
template <typename T>
__global__ void __launch_bounds__(256) k_axpby_fwd8(const T* __restrict__ a, const T* __restrict__ b, const T* __restrict__ c,
                                                    long c_pitch, const float* __restrict__ s1, const float* __restrict__ s2,
                                                    long NP, int C, T* __restrict__ out) {
  const float k1 = s1[0], k2 = c ? s2[0] : 0.f;
  const int G = C >> 3;
  const long total = NP * G;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    float fa[8], fb[8];
    load8<T>(a + 8 * i, fa);
    load8<T>(b + 8 * i, fb);
#pragma unroll
    for (int k = 0; k < 8; ++k) fa[k] = fmaf(k1, fb[k], fa[k]);
    if (c) {
      const long pix = i / G;
      float fc[8];
      load8<T>(c + pix * c_pitch + 8 * (i - pix * G), fc);
#pragma unroll
      for (int k = 0; k < 8; ++k) fa[k] = fmaf(k2, fc[k], fa[k]);
    }
    store8<T>(out + 8 * i, fa);
  }
}
template <typename T>
__global__ void __launch_bounds__(256) k_axpby_bwd8(const T* __restrict__ g, const T* __restrict__ b, const T* __restrict__ c,
                                                    long c_pitch, const float* __restrict__ s1, const float* __restrict__ s2,
                                                    long NP, int C, T* __restrict__ db, T* __restrict__ dc,
                                                    float* __restrict__ part) {
  __shared__ float sh[2][8];
  const float k1 = s1[0], k2 = c ? s2[0] : 0.f;
  const int G = C >> 3;
  const long total = NP * G;
  float a1 = 0.f, a2 = 0.f;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    float fg[8], fb[8], o[8];
    load8<T>(g + 8 * i, fg);
    load8<T>(b + 8 * i, fb);
#pragma unroll
    for (int k = 0; k < 8; ++k) { a1 = fmaf(fg[k], fb[k], a1); o[k] = k1 * fg[k]; }
    store8<T>(db + 8 * i, o);
    if (c) {
      const long pix = i / G;
      float fc[8];
      load8<T>(c + pix * c_pitch + 8 * (i - pix * G), fc);
#pragma unroll
      for (int k = 0; k < 8; ++k) { a2 = fmaf(fg[k], fc[k], a2); o[k] = k2 * fg[k]; }
      store8<T>(dc + 8 * i, o);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    a1 += __shfl_down_sync(0xffffffffu, a1, o);
    a2 += __shfl_down_sync(0xffffffffu, a2, o);
  }
  if ((threadIdx.x & 31) == 0) { sh[0][threadIdx.x >> 5] = a1; sh[1][threadIdx.x >> 5] = a2; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float t1 = 0.f, t2 = 0.f;
    for (int i = 0; i < 8; ++i) { t1 += sh[0][i]; t2 += sh[1][i]; }
    part[(long)blockIdx.x * (c ? 2 : 1)] = t1;
    if (c) part[(long)blockIdx.x * 2 + 1] = t2;
  }
}

// out = a + s1*b (+ s2*c);  c may be a channel slice (pixel pitch c_pitch >= C)
template <typename T>
__global__ void __launch_bounds__(256) k_axpby_fwd(const T* __restrict__ a, const T* __restrict__ b, const T* __restrict__ c,
                                                   long c_pitch, const float* __restrict__ s1, const float* __restrict__ s2,
                                                   long NP, int C, T* __restrict__ out) {
  const float k1 = s1[0], k2 = c ? s2[0] : 0.f;
  const long total = NP * C;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    float v = fmaf(k1, to_f32<T>(b[i]), to_f32<T>(a[i]));
    if (c) {
      const long pix = i / C;
      v = fmaf(k2, to_f32<T>(c[pix * c_pitch + (i - pix * C)]), v);
    }
    out[i] = from_f32<T>(v);
  }
}
// db = s1*g, dc = s2*g; slot blockIdx.x of part [grid][1 or 2] = partial sum g*b (, sum g*c)
template <typename T>
__global__ void __launch_bounds__(256) k_axpby_bwd(const T* __restrict__ g, const T* __restrict__ b, const T* __restrict__ c,
                                                   long c_pitch, const float* __restrict__ s1, const float* __restrict__ s2,
                                                   long NP, int C, T* __restrict__ db, T* __restrict__ dc,
                                                   float* __restrict__ part) {
  __shared__ float sh[2][8];
  const float k1 = s1[0], k2 = c ? s2[0] : 0.f;
  const long total = NP * C;
  float a1 = 0.f, a2 = 0.f;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const float gv = to_f32<T>(g[i]);
    a1 = fmaf(gv, to_f32<T>(b[i]), a1);
    db[i] = from_f32<T>(k1 * gv);
    if (c) {
      const long pix = i / C;
      a2 = fmaf(gv, to_f32<T>(c[pix * c_pitch + (i - pix * C)]), a2);
      dc[i] = from_f32<T>(k2 * gv);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    a1 += __shfl_down_sync(0xffffffffu, a1, o);
    a2 += __shfl_down_sync(0xffffffffu, a2, o);
  }
  if ((threadIdx.x & 31) == 0) { sh[0][threadIdx.x >> 5] = a1; sh[1][threadIdx.x >> 5] = a2; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float t1 = 0.f, t2 = 0.f;
    for (int i = 0; i < 8; ++i) { t1 += sh[0][i]; t2 += sh[1][i]; }
    part[(long)blockIdx.x * (c ? 2 : 1)] = t1;
    if (c) part[(long)blockIdx.x * 2 + 1] = t2;
  }
}

template <typename T>
__global__ void __launch_bounds__(256) k_bilinear_bwd8(const T* __restrict__ gout, int H, int W, int C, T* __restrict__ gin,
                                                       int h, int w, long total) {
  const int G = C >> 3;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int cg = (int)(i % G);
    const long pix = i / G;
    const int x = (int)(pix % w), y = (int)((pix / w) % h);
    const long n = pix / ((long)w * h);
    float wy[BL_MAXC], wx[BL_MAXC];
    int ylo, yhi, xlo, xhi;
    bilin_adjoint_range(y, h, H, ylo, yhi);
    bilin_adjoint_range(x, w, W, xlo, xhi);
    float acc[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) acc[k] = 0.f;
    const T* base = gout + n * H * W * C + cg * 8;
    for (int y0 = ylo; y0 <= yhi; y0 += BL_MAXC) {
      const int ny = bilin_adjoint_taps(y, h, H, y0, yhi, wy);
      for (int x0 = xlo; x0 <= xhi; x0 += BL_MAXC) {
        const int nx = bilin_adjoint_taps(x, w, W, x0, xhi, wx);
        for (int a = 0; a < ny; ++a) {
          if (wy[a] == 0.f) continue;
          for (int b = 0; b < nx; ++b) {
            const float wgt = wy[a] * wx[b];
            if (wgt == 0.f) continue;
            float v[8];
            load8<T>(base + ((long)(y0 + a) * W + x0 + b) * C, v);
#pragma unroll
            for (int k = 0; k < 8; ++k) acc[k] = fmaf(wgt, v[k], acc[k]);
          }
        }
      }
    }
    store8<T>(gin + pix * C + cg * 8, acc);
  }
}

inline void colsum_geom(int C, dim3& block, int& CT) {
  CT = 1;
  while (CT < C && CT < 64) CT <<= 1;
  block = dim3(CT, 256 / CT);
}

// grid of the BN reductions: (row chunks, channel tiles, groups)
inline void bn_geom(int G, long R, int C, dim3& block, dim3& grid, long& rpb) {
  int CT;
  colsum_geom(C, block, CT);
  long blocks = 148 * 4 / ((long)ceil_div(C, CT) * G);
  if (blocks < 1) blocks = 1;
  rpb = (R + blocks - 1) / blocks;
  if (rpb < 64) rpb = 64;
  grid = dim3(ceil_div(R, rpb), ceil_div(C, CT), G);
}

constexpr long COLSUM_MAX_BLOCKS = 148 * 8;     // row chunks of either colsum path
constexpr long LN_MAX_BLOCKS = 148 * 8;
constexpr long AXPBY_MAX_BLOCKS = 148 * 8;
}  // namespace

extern "C" size_t ffsr_conv2d_wgrad_workspace_bytes(int N, int H, int W, int Cin, int Cout, int ksize) {
  if (N <= 0 || H <= 0 || W <= 0 || Cin <= 0 || Cout <= 0 || (ksize != 1 && ksize != 3)) return 0;
  const WgradPlan pl = wgrad_plan(N, H, W, Cin, Cout, ksize);
  return ws_align((size_t)pl.P * ksize * ksize * Cin * Cout * sizeof(float)) + ffsr_colsum_workspace_bytes(N, H, W, Cout);
}

extern "C" int ffsr_conv2d_wgrad(const ffsr_wgrad_params* pp, void* ws, size_t ws_bytes, cudaStream_t stream) {
  FFSR_REQUIRE(pp, FFSR_ERR_ARG, "conv2d_wgrad: null params");
  const ffsr_wgrad_params& p = *pp;
  FFSR_REQUIRE(p.x && p.dy && p.dw && ws, FFSR_ERR_ARG, "conv2d_wgrad: null pointer");
  FFSR_REQUIRE(p.N > 0 && p.H > 0 && p.W > 0 && p.Cin > 0 && p.Cout > 0, FFSR_ERR_ARG, "conv2d_wgrad: bad shape");
  FFSR_REQUIRE(p.ksize == 1 || p.ksize == 3, FFSR_ERR_ARG, "conv2d_wgrad: ksize must be 1 or 3");
  FFSR_REQUIRE(ws_bytes >= ffsr_conv2d_wgrad_workspace_bytes(p.N, p.H, p.W, p.Cin, p.Cout, p.ksize), FFSR_ERR_ARG,
               "conv2d_wgrad: workspace too small");
  const WgradPlan pl = wgrad_plan(p.N, p.H, p.W, p.Cin, p.Cout, p.ksize);
  const int taps = p.ksize * p.ksize;
  float* part = (float*)ws;
  float* bpart = (float*)((char*)ws + ws_align((size_t)pl.P * taps * p.Cin * p.Cout * sizeof(float)));
  int rc;
  if (pl.TM == 128) rc = dispatch_wgrad_n<128>(p, pl, part, stream);
  else if (pl.TM == 64) rc = dispatch_wgrad_n<64>(p, pl, part, stream);
  else if (pl.TM == 32) rc = dispatch_wgrad_n<32>(p, pl, part, stream);
  else rc = dispatch_wgrad_n<16>(p, pl, part, stream);
  if (rc) return rc;
  SlotSum<float> bias{};
  if (p.dbias) {
    int nb;
    rc = colsum_partials(p.dy, p.dy_dtype, p.N, p.H, p.W, p.Cout, p.dy_sN, p.dy_sY, p.dy_sX, bpart, &nb, stream);
    if (rc) return rc;
    bias = slot_sum<float>(bpart, nb, p.Cout, p.dbias);
  }
  launch_sum_slots<float>(slot_sum<float>(part, (int)pl.P, (long)taps * p.Cin * p.Cout, p.dw), bias, stream);
  return ffsr_check_launch("conv2d_wgrad_reduce");
}

extern "C" size_t ffsr_wgrad_params_size(void) { return sizeof(ffsr_wgrad_params); }

extern "C" size_t ffsr_colsum_workspace_bytes(int N, int H, int W, int C) {
  (void)N; (void)H; (void)W;
  return C > 0 ? (size_t)COLSUM_MAX_BLOCKS * C * sizeof(float) : 0;
}

int colsum_partials(const void* v, int dtype, int N, int H, int W, int C, long long sN, long long sY, long long sX,
                    float* part, int* nslots, cudaStream_t stream) {
  if (sY == (long long)W * sX && sN == (long long)H * W * sX && C <= 512) {      // dense channels-last rows
    const long NP = (long)N * H * W;
    const int VEC = C >= 64 ? 4 : 1;
    int TPR = 1;
    while (TPR * VEC < C) TPR <<= 1;                   // power of two, <= 128
    long rpb = (NP + COLSUM_MAX_BLOCKS - 1) / COLSUM_MAX_BLOCKS;
    if (rpb < 256) rpb = 256;
    const unsigned grid = (unsigned)((NP + rpb - 1) / rpb);
    if (dtype == FFSR_DT_BF16) {
      if (VEC == 4) k_colsum_rows<__nv_bfloat16, 4><<<grid, 256, 0, stream>>>((const __nv_bfloat16*)v, NP, C, sX, TPR, rpb, part);
      else k_colsum_rows<__nv_bfloat16, 1><<<grid, 256, 0, stream>>>((const __nv_bfloat16*)v, NP, C, sX, TPR, rpb, part);
    } else {
      if (VEC == 4) k_colsum_rows<float, 4><<<grid, 256, 0, stream>>>((const float*)v, NP, C, sX, TPR, rpb, part);
      else k_colsum_rows<float, 1><<<grid, 256, 0, stream>>>((const float*)v, NP, C, sX, TPR, rpb, part);
    }
    *nslots = (int)grid;
    return ffsr_check_launch("colsum_rows");
  }
  dim3 block;
  int CT;
  colsum_geom(C, block, CT);
  const long NP = (long)N * H * W;
  long blocks = 148 * 4 / ceil_div(C, CT);
  if (blocks < 1) blocks = 1;
  long rpb = (NP + blocks - 1) / blocks;
  if (rpb < 64) rpb = 64;
  dim3 grid(ceil_div(NP, rpb), ceil_div(C, CT));
  k_colsum<<<grid, block, 256 * sizeof(float), stream>>>(v, dtype, sN, sY, sX, H, W, NP, C, rpb, part);
  *nslots = (int)grid.x;
  return ffsr_check_launch("colsum");
}

extern "C" int ffsr_colsum(const void* v, int dtype, int N, int H, int W, int C, long long sN, long long sY,
                           long long sX, float* out, void* ws, size_t ws_bytes, cudaStream_t stream) {
  FFSR_REQUIRE(v && out && ws && N > 0 && H > 0 && W > 0 && C > 0, FFSR_ERR_ARG, "colsum: bad argument");
  FFSR_REQUIRE(ws_bytes >= ffsr_colsum_workspace_bytes(N, H, W, C), FFSR_ERR_ARG, "colsum: workspace too small");
  int nslots;
  const int rc = colsum_partials(v, dtype, N, H, W, C, sN, sY, sX, (float*)ws, &nslots, stream);
  if (rc) return rc;
  launch_sum_slots<float>((const float*)ws, nslots, C, out, stream);
  return ffsr_check_launch("colsum_reduce");
}

extern "C" int ffsr_act_forward(const void* x, void* y, long n, int act, int dtype, cudaStream_t stream) {
  FFSR_REQUIRE(x && y && n > 0, FFSR_ERR_ARG, "act_forward: bad argument");
  const int grid = (int)min((long)148 * 16, (n + 255) / 256);
  if (dtype == FFSR_DT_BF16) k_act_fwd<__nv_bfloat16><<<grid, 256, 0, stream>>>((const __nv_bfloat16*)x, (__nv_bfloat16*)y, n, act);
  else k_act_fwd<float><<<grid, 256, 0, stream>>>((const float*)x, (float*)y, n, act);
  return ffsr_check_launch("act_forward");
}

extern "C" int ffsr_act_backward(const void* x, const void* dy, void* dx, long n, int act, int dtype,
                                 cudaStream_t stream) {
  FFSR_REQUIRE(x && dy && dx && n > 0, FFSR_ERR_ARG, "act_backward: bad argument");
  const int grid = (int)min((long)148 * 16, (n + 255) / 256);
  if (dtype == FFSR_DT_BF16)
    k_act_bwd<__nv_bfloat16><<<grid, 256, 0, stream>>>((const __nv_bfloat16*)x, (const __nv_bfloat16*)dy, (__nv_bfloat16*)dx, n, act);
  else k_act_bwd<float><<<grid, 256, 0, stream>>>((const float*)x, (const float*)dy, (float*)dx, n, act);
  return ffsr_check_launch("act_backward");
}

extern "C" size_t ffsr_layernorm_backward_workspace_bytes(long rows, int E) {
  if (rows <= 0 || E <= 0) return 0;
  return (size_t)min(LN_MAX_BLOCKS, (rows + 7) / 8) * 2 * E * sizeof(float);
}

extern "C" int ffsr_layernorm_backward(const float* x, const float* dy, long rows, int E, const float* w, float* dx,
                                       float* dw, float* db, void* ws, size_t ws_bytes, cudaStream_t stream) {
  FFSR_REQUIRE(x && dy && w && dx && dw && db && ws && rows > 0, FFSR_ERR_ARG, "layernorm_backward: null pointer");
  FFSR_REQUIRE(E % 32 == 0 && E >= 32 && E <= 256, FFSR_ERR_ARG, "layernorm_backward: E must be a multiple of 32 in [32,256]");
  FFSR_REQUIRE(ws_bytes >= ffsr_layernorm_backward_workspace_bytes(rows, E), FFSR_ERR_ARG, "layernorm_backward: workspace too small");
  const int grid = (int)min(LN_MAX_BLOCKS, (rows + 7) / 8);
  float* part = (float*)ws;
  k_layernorm_bwd<<<grid, 256, 8 * 2 * E * sizeof(float), stream>>>(x, dy, rows, E, w, dx, part);
  const int rc = ffsr_check_launch("layernorm_backward");
  if (rc) return rc;
  launch_sum_slots<float>(part, grid, 2L * E, dw, stream, db, E);
  return ffsr_check_launch("layernorm_backward_reduce");
}

extern "C" size_t ffsr_bn_stats_workspace_bytes(int G, long R, int C) {
  if (G <= 0 || R <= 0 || C <= 0) return 0;
  dim3 block, grid;
  long rpb;
  bn_geom(G, R, C, block, grid, rpb);
  return (size_t)grid.x * 2 * G * C * sizeof(double);
}

extern "C" int ffsr_bn_stats(const float* x, int G, long R, int C, double* sum, double* sumsq, void* ws, size_t ws_bytes,
                             cudaStream_t stream) {
  FFSR_REQUIRE(x && sum && sumsq && ws && G > 0 && R > 0 && C > 0 && G <= 65535, FFSR_ERR_ARG, "bn_stats: bad argument");
  FFSR_REQUIRE(ws_bytes >= ffsr_bn_stats_workspace_bytes(G, R, C), FFSR_ERR_ARG, "bn_stats: workspace too small");
  dim3 block, grid;
  long rpb;
  bn_geom(G, R, C, block, grid, rpb);
  double* part = (double*)ws;
  k_bn_stats<<<grid, block, 2 * 256 * sizeof(double), stream>>>(x, R, C, rpb, part);
  const int rc = ffsr_check_launch("bn_stats");
  if (rc) return rc;
  launch_sum_slots<double>(part, (int)grid.x, 2L * G * C, sum, stream, sumsq, (long)G * C);
  return ffsr_check_launch("bn_stats_reduce");
}

extern "C" int ffsr_bn_apply(const float* x, int G, long R, int C, const float* mean, const float* rstd, const float* w,
                             const float* b, float* y, cudaStream_t stream) {
  FFSR_REQUIRE(x && mean && rstd && w && b && y && G > 0 && R > 0 && C > 0 && C % 4 == 0, FFSR_ERR_ARG, "bn_apply: bad argument (C %% 4 == 0)");
  const long total = (long)G * R * (C / 4);
  k_bn_apply<<<(int)min((long)148 * 16, (total + 255) / 256), 256, 0, stream>>>(x, R, C, G, mean, rstd, w, b, y);
  return ffsr_check_launch("bn_apply");
}

extern "C" size_t ffsr_bn_backward_workspace_bytes(int G, long R, int C) {
  if (G <= 0 || R <= 0 || C <= 0) return 0;
  dim3 block, grid;
  long rpb;
  bn_geom(G, R, C, block, grid, rpb);
  return (size_t)grid.x * 2 * G * C * sizeof(float);
}

extern "C" int ffsr_bn_backward(const float* x, const float* dy, int G, long R, int C, const float* mean,
                                const float* rstd, const float* w, float* sdy, float* sdyx, float* dx, void* ws,
                                size_t ws_bytes, cudaStream_t stream) {
  FFSR_REQUIRE(x && dy && mean && rstd && w && sdy && sdyx && dx && ws && G > 0 && R > 0 && C > 0 && G <= 65535, FFSR_ERR_ARG,
               "bn_backward: bad argument");
  FFSR_REQUIRE(ws_bytes >= ffsr_bn_backward_workspace_bytes(G, R, C), FFSR_ERR_ARG, "bn_backward: workspace too small");
  dim3 block, grid;
  long rpb;
  bn_geom(G, R, C, block, grid, rpb);
  float* part = (float*)ws;
  k_bn_bwd_reduce<<<grid, block, 2 * 256 * sizeof(float), stream>>>(x, dy, R, C, rpb, mean, rstd, part);
  int rc = ffsr_check_launch("bn_backward_reduce");
  if (rc) return rc;
  launch_sum_slots<float>(part, (int)grid.x, 2L * G * C, sdy, stream, sdyx, (long)G * C);
  rc = ffsr_check_launch("bn_backward_sum");
  if (rc) return rc;
  FFSR_REQUIRE(C % 4 == 0, FFSR_ERR_ARG, "bn_backward: C must be a multiple of 4");
  const long total = (long)G * R * (C / 4);
  k_bn_bwd_apply<<<(int)min((long)148 * 16, (total + 255) / 256), 256, 0, stream>>>(x, dy, R, C, G, mean, rstd, w, sdy, sdyx, dx);
  return ffsr_check_launch("bn_backward_apply");
}

// eval-mode BatchNorm: the statistics are constants, so dx = dy * w * rstd (float4 over channels, C % 4 == 0)
__global__ void __launch_bounds__(256) k_bn_eval_dx(const float* __restrict__ dy, long n4, int C, const float* __restrict__ rstd,
                                                    const float* __restrict__ w, float* __restrict__ dx) {
  const int C4 = C >> 2;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long)gridDim.x * blockDim.x) {
    const int c = (int)(i % C4) << 2;
    const float4 g = reinterpret_cast<const float4*>(dy)[i];
    const float4 rs = *reinterpret_cast<const float4*>(rstd + c), wv = *reinterpret_cast<const float4*>(w + c);
    reinterpret_cast<float4*>(dx)[i] = make_float4(g.x * (wv.x * rs.x), g.y * (wv.y * rs.y), g.z * (wv.z * rs.z), g.w * (wv.w * rs.w));
  }
}

extern "C" int ffsr_bn_eval_backward(const float* x, const float* dy, long R, int C, const float* mean, const float* rstd,
                                     const float* w, float* sdy, float* sdyx, float* dx, void* ws, size_t ws_bytes,
                                     cudaStream_t stream) {
  FFSR_REQUIRE(x && dy && mean && rstd && w && sdy && sdyx && dx && ws && R > 0 && C > 0 && C % 4 == 0, FFSR_ERR_ARG,
               "bn_eval_backward: bad argument (C %% 4 == 0)");
  FFSR_REQUIRE(ws_bytes >= ffsr_bn_backward_workspace_bytes(1, R, C), FFSR_ERR_ARG, "bn_eval_backward: workspace too small");
  dim3 block, grid;
  long rpb;
  bn_geom(1, R, C, block, grid, rpb);
  float* part = (float*)ws;
  k_bn_bwd_reduce<<<grid, block, 2 * 256 * sizeof(float), stream>>>(x, dy, R, C, rpb, mean, rstd, part);
  int rc = ffsr_check_launch("bn_eval_backward_reduce");
  if (rc) return rc;
  launch_sum_slots<float>(part, (int)grid.x, 2L * C, sdy, stream, sdyx, (long)C);
  rc = ffsr_check_launch("bn_eval_backward_sum");
  if (rc) return rc;
  const long n4 = R * (C / 4);
  k_bn_eval_dx<<<(int)min((long)148 * 16, (n4 + 255) / 256), 256, 0, stream>>>(dy, n4, C, rstd, w, dx);
  return ffsr_check_launch("bn_eval_backward_dx");
}

extern "C" int ffsr_token_attention_train(const float* qkv, int B, int T, long HW, int E, float* ctx, float* probs,
                                          float drop_p, unsigned long long seed, const unsigned long long* seed_dev,
                                          cudaStream_t stream) {
  FFSR_REQUIRE(qkv && ctx && probs, FFSR_ERR_ARG, "token_attention_train: null pointer");
  FFSR_REQUIRE((T == 4 || T == 9) && E % 16 == 0 && B > 0 && HW > 0, FFSR_ERR_ARG, "token_attention_train: T must be 4 or 9, E%%16==0");
  FFSR_REQUIRE(drop_p >= 0.f && drop_p < 1.f, FFSR_ERR_ARG, "token_attention_train: dropout p must be in [0,1)");
  const long n = (long)B * HW * T * (E / 16);
  if (T == 4) k_tokattn_fwd<4><<<ceil_div(n, 128), 128, 0, stream>>>(qkv, B, HW, E, ctx, probs, drop_p, seed, seed_dev);
  else k_tokattn_fwd<9><<<ceil_div(n, 128), 128, 0, stream>>>(qkv, B, HW, E, ctx, probs, drop_p, seed, seed_dev);
  return ffsr_check_launch("token_attention_train");
}

extern "C" int ffsr_token_attention_backward(const float* qkv, const float* probs, const float* dctx, int B, int T,
                                             long HW, int E, float* ds_scratch, float* dqkv, float drop_p,
                                             unsigned long long seed, const unsigned long long* seed_dev,
                                             cudaStream_t stream) {
  FFSR_REQUIRE(qkv && probs && dctx && ds_scratch && dqkv, FFSR_ERR_ARG, "token_attention_backward: null pointer");
  FFSR_REQUIRE((T == 4 || T == 9) && E % 16 == 0 && B > 0 && HW > 0, FFSR_ERR_ARG, "token_attention_backward: T must be 4 or 9");
  const long n = (long)B * HW * T * (E / 16);
  if (T == 4) {
    k_tokattn_bwd_q<4><<<ceil_div(n, 128), 128, 0, stream>>>(qkv, probs, dctx, B, HW, E, ds_scratch, dqkv, drop_p, seed, seed_dev);
    k_tokattn_bwd_kv<4><<<ceil_div(n, 128), 128, 0, stream>>>(qkv, probs, ds_scratch, dctx, B, HW, E, dqkv, drop_p, seed, seed_dev);
  } else {
    k_tokattn_bwd_q<9><<<ceil_div(n, 128), 128, 0, stream>>>(qkv, probs, dctx, B, HW, E, ds_scratch, dqkv, drop_p, seed, seed_dev);
    k_tokattn_bwd_kv<9><<<ceil_div(n, 128), 128, 0, stream>>>(qkv, probs, ds_scratch, dctx, B, HW, E, dqkv, drop_p, seed, seed_dev);
  }
  return ffsr_check_launch("token_attention_backward");
}

extern "C" int ffsr_to_bf16_nhwc(const void* src, int src_dtype, long long sN, long long sY, long long sX, long long sC,
                                 int N, int H, int W, int C, int Cpad, void* dst, cudaStream_t stream) {
  FFSR_REQUIRE(src && dst && N > 0 && H > 0 && W > 0 && C > 0 && Cpad >= C, FFSR_ERR_ARG, "to_bf16_nhwc: bad argument");
  if (sC == 1 && sY == (long long)W * sX && sN == (long long)H * W * sX && Cpad % 8 == 0 && ((uintptr_t)dst % 16) == 0) {
    const long NP = (long)N * H * W;
    const long work = NP * (Cpad >> 3);
    const int grid = (int)min((long)148 * 16, (work + 255) / 256);
    if (src_dtype == FFSR_DT_BF16) k_to_bf16_rows<__nv_bfloat16><<<grid, 256, 0, stream>>>((const __nv_bfloat16*)src, sX, NP, C, Cpad, (__nv_bfloat16*)dst);
    else k_to_bf16_rows<float><<<grid, 256, 0, stream>>>((const float*)src, sX, NP, C, Cpad, (__nv_bfloat16*)dst);
    return ffsr_check_launch("to_bf16_rows");
  }
  const long total = (long)N * H * W * Cpad;
  k_to_bf16_nhwc<<<(int)min((long)148 * 16, (total + 255) / 256), 256, 0, stream>>>(src, src_dtype, sN, sY, sX, sC, H, W, C,
                                                                                     Cpad, total, (__nv_bfloat16*)dst);
  return ffsr_check_launch("to_bf16_nhwc");
}

// F.interpolate(mode="bilinear", align_corners=False) on dense channels-last tensors and its adjoint
// (SURVEY Appendix A; used by hierarchical_fusion.py:156-186, enhanced_fusion_v2.py:735-791, edge_enhancement.py:208-250)
template <bool BWD>
static int launch_bilinear(const void* a, int N, int h, int w, int C, void* b, int H, int W, int dtype, cudaStream_t stream) {
  // forward: a = src [N,h,w,C] -> b = dst [N,H,W,C];  backward: a = gout [N,H,W,C] -> b = gin [N,h,w,C]
  if (C % 8 == 0 && ((uintptr_t)a % 16) == 0 && ((uintptr_t)b % 16) == 0) {
    const long total8 = (long)N * (BWD ? (long)h * w : (long)H * W) * (C / 8);
    const int grid8 = (int)min((long)148 * 32, (total8 + 255) / 256);
    if (dtype == FFSR_DT_BF16) {
      using T = __nv_bfloat16;
      if (BWD) k_bilinear_bwd8<T><<<grid8, 256, 0, stream>>>((const T*)a, H, W, C, (T*)b, h, w, total8);
      else k_bilinear_fwd8<T><<<grid8, 256, 0, stream>>>((const T*)a, h, w, C, (T*)b, H, W, total8);
    } else {
      if (BWD) k_bilinear_bwd8<float><<<grid8, 256, 0, stream>>>((const float*)a, H, W, C, (float*)b, h, w, total8);
      else k_bilinear_fwd8<float><<<grid8, 256, 0, stream>>>((const float*)a, h, w, C, (float*)b, H, W, total8);
    }
    return ffsr_check_launch(BWD ? "bilinear_backward" : "bilinear_forward");
  }
  const int VEC = (C % 4 == 0) ? 4 : 1;
  const long total = (long)N * (BWD ? (long)h * w : (long)H * W) * (C / VEC);
  const int grid = (int)min((long)148 * 32, (total + 255) / 256);
  if (dtype == FFSR_DT_BF16) {
    using T = __nv_bfloat16;
    if (BWD) { if (VEC == 4) k_bilinear_bwd<T, 4><<<grid, 256, 0, stream>>>((const T*)a, H, W, C, (T*)b, h, w, total);
               else k_bilinear_bwd<T, 1><<<grid, 256, 0, stream>>>((const T*)a, H, W, C, (T*)b, h, w, total); }
    else { if (VEC == 4) k_bilinear_fwd<T, 4><<<grid, 256, 0, stream>>>((const T*)a, h, w, C, (T*)b, H, W, total);
           else k_bilinear_fwd<T, 1><<<grid, 256, 0, stream>>>((const T*)a, h, w, C, (T*)b, H, W, total); }
  } else {
    using T = float;
    if (BWD) { if (VEC == 4) k_bilinear_bwd<T, 4><<<grid, 256, 0, stream>>>((const T*)a, H, W, C, (T*)b, h, w, total);
               else k_bilinear_bwd<T, 1><<<grid, 256, 0, stream>>>((const T*)a, H, W, C, (T*)b, h, w, total); }
    else { if (VEC == 4) k_bilinear_fwd<T, 4><<<grid, 256, 0, stream>>>((const T*)a, h, w, C, (T*)b, H, W, total);
           else k_bilinear_fwd<T, 1><<<grid, 256, 0, stream>>>((const T*)a, h, w, C, (T*)b, H, W, total); }
  }
  return ffsr_check_launch(BWD ? "bilinear_backward" : "bilinear_forward");
}

extern "C" int ffsr_bilinear_forward(const void* src, int N, int h, int w, int C, void* dst, int H, int W, int dtype,
                                     cudaStream_t stream) {
  FFSR_REQUIRE(src && dst && N > 0 && h > 0 && w > 0 && H > 0 && W > 0 && C > 0, FFSR_ERR_ARG, "bilinear_forward: bad argument");
  return launch_bilinear<false>(src, N, h, w, C, dst, H, W, dtype, stream);
}

extern "C" int ffsr_bilinear_backward(const void* gout, int N, int H, int W, int C, void* gin, int h, int w, int dtype,
                                      cudaStream_t stream) {
  FFSR_REQUIRE(gout && gin && N > 0 && h > 0 && w > 0 && H > 0 && W > 0 && C > 0, FFSR_ERR_ARG, "bilinear_backward: bad argument");
  return launch_bilinear<true>(gout, N, h, w, C, gin, H, W, dtype, stream);
}

extern "C" int ffsr_gate_mul_forward(const void* y, const float* g, long NP, int C, void* out, int dtype, cudaStream_t stream) {
  FFSR_REQUIRE(y && g && out && NP > 0 && C > 0 && C % 4 == 0, FFSR_ERR_ARG, "gate_mul_forward: bad argument (C %% 4 == 0)");
  if (C % 8 == 0 && ((uintptr_t)y % 16) == 0 && ((uintptr_t)out % 16) == 0) {
    const long total8 = NP * (C / 8);
    const int grid8 = (int)min((long)148 * 16, (total8 + 255) / 256);
    if (dtype == FFSR_DT_BF16) k_gate_mul_fwd8<__nv_bfloat16><<<grid8, 256, 0, stream>>>((const __nv_bfloat16*)y, g, NP, C, (__nv_bfloat16*)out);
    else k_gate_mul_fwd8<float><<<grid8, 256, 0, stream>>>((const float*)y, g, NP, C, (float*)out);
    return ffsr_check_launch("gate_mul_forward");
  }
  const long total = NP * (C / 4);
  const int grid = (int)min((long)148 * 16, (total + 255) / 256);
  if (dtype == FFSR_DT_BF16) k_gate_mul_fwd<__nv_bfloat16><<<grid, 256, 0, stream>>>((const __nv_bfloat16*)y, g, NP, C, (__nv_bfloat16*)out);
  else k_gate_mul_fwd<float><<<grid, 256, 0, stream>>>((const float*)y, g, NP, C, (float*)out);
  return ffsr_check_launch("gate_mul_forward");
}

extern "C" int ffsr_gate_mul_backward(const void* y, const float* g, const void* gout, long NP, int C, void* dy, float* dg,
                                      int dtype, cudaStream_t stream) {
  FFSR_REQUIRE(y && g && gout && dy && dg && NP > 0 && C > 0 && C % 4 == 0, FFSR_ERR_ARG, "gate_mul_backward: bad argument");
  if (C % 8 == 0 && ((uintptr_t)y % 16) == 0 && ((uintptr_t)gout % 16) == 0 && ((uintptr_t)dy % 16) == 0) {
    const int grid8 = (int)min((long)148 * 16, (NP * 8 + 255) / 256);
    if (dtype == FFSR_DT_BF16)
      k_gate_mul_bwd8<__nv_bfloat16><<<grid8, 256, 0, stream>>>((const __nv_bfloat16*)y, g, (const __nv_bfloat16*)gout, NP, C, (__nv_bfloat16*)dy, dg);
    else k_gate_mul_bwd8<float><<<grid8, 256, 0, stream>>>((const float*)y, g, (const float*)gout, NP, C, (float*)dy, dg);
    return ffsr_check_launch("gate_mul_backward");
  }
  const int grid = (int)min((long)148 * 32, (NP + 127) / 128);
  if (dtype == FFSR_DT_BF16)
    k_gate_mul_bwd<__nv_bfloat16><<<grid, 128, 0, stream>>>((const __nv_bfloat16*)y, g, (const __nv_bfloat16*)gout, NP, C, (__nv_bfloat16*)dy, dg);
  else k_gate_mul_bwd<float><<<grid, 128, 0, stream>>>((const float*)y, g, (const float*)gout, NP, C, (float*)dy, dg);
  return ffsr_check_launch("gate_mul_backward");
}

extern "C" int ffsr_axpby_forward(const void* a, const void* b, const void* c, long c_pitch, const float* s1, const float* s2,
                                  long NP, int C, void* out, int dtype, cudaStream_t stream) {
  FFSR_REQUIRE(a && b && s1 && out && NP > 0 && C > 0 && (!c || s2), FFSR_ERR_ARG, "axpby_forward: bad argument");
  auto al16 = [](const void* p) { return ((uintptr_t)p % 16) == 0; };
  const int esz = dtype == FFSR_DT_BF16 ? 2 : 4;
  if (C % 8 == 0 && al16(a) && al16(b) && al16(out) && (!c || (al16(c) && (c_pitch * esz) % 16 == 0))) {
    const long total8 = NP * (C / 8);
    const int grid8 = (int)min((long)148 * 16, (total8 + 255) / 256);
    if (dtype == FFSR_DT_BF16)
      k_axpby_fwd8<__nv_bfloat16><<<grid8, 256, 0, stream>>>((const __nv_bfloat16*)a, (const __nv_bfloat16*)b, (const __nv_bfloat16*)c, c_pitch, s1, s2, NP, C, (__nv_bfloat16*)out);
    else k_axpby_fwd8<float><<<grid8, 256, 0, stream>>>((const float*)a, (const float*)b, (const float*)c, c_pitch, s1, s2, NP, C, (float*)out);
    return ffsr_check_launch("axpby_forward");
  }
  const long total = NP * C;
  const int grid = (int)min((long)148 * 16, (total + 255) / 256);
  if (dtype == FFSR_DT_BF16)
    k_axpby_fwd<__nv_bfloat16><<<grid, 256, 0, stream>>>((const __nv_bfloat16*)a, (const __nv_bfloat16*)b, (const __nv_bfloat16*)c, c_pitch, s1, s2, NP, C, (__nv_bfloat16*)out);
  else k_axpby_fwd<float><<<grid, 256, 0, stream>>>((const float*)a, (const float*)b, (const float*)c, c_pitch, s1, s2, NP, C, (float*)out);
  return ffsr_check_launch("axpby_forward");
}

extern "C" size_t ffsr_axpby_backward_workspace_bytes(long NP, int C) {
  (void)NP; (void)C;
  return (size_t)AXPBY_MAX_BLOCKS * 2 * sizeof(float);
}

extern "C" int ffsr_axpby_backward(const void* g, const void* b, const void* c, long c_pitch, const float* s1, const float* s2,
                                   long NP, int C, void* db, void* dc, float* ds, void* ws, size_t ws_bytes, int dtype,
                                   cudaStream_t stream) {
  FFSR_REQUIRE(g && b && s1 && db && ds && ws && NP > 0 && C > 0 && (!c || (s2 && dc)), FFSR_ERR_ARG, "axpby_backward: bad argument");
  FFSR_REQUIRE(ws_bytes >= ffsr_axpby_backward_workspace_bytes(NP, C), FFSR_ERR_ARG, "axpby_backward: workspace too small");
  float* part = (float*)ws;
  const int L = c ? 2 : 1;
  int grid;
  auto al16 = [](const void* p) { return ((uintptr_t)p % 16) == 0; };
  const int esz = dtype == FFSR_DT_BF16 ? 2 : 4;
  if (C % 8 == 0 && al16(g) && al16(b) && al16(db) && (!c || (al16(c) && al16(dc) && (c_pitch * esz) % 16 == 0))) {
    const long total8 = NP * (C / 8);
    grid = (int)min(AXPBY_MAX_BLOCKS, (total8 + 255) / 256);
    if (dtype == FFSR_DT_BF16)
      k_axpby_bwd8<__nv_bfloat16><<<grid, 256, 0, stream>>>((const __nv_bfloat16*)g, (const __nv_bfloat16*)b, (const __nv_bfloat16*)c, c_pitch, s1, s2, NP, C, (__nv_bfloat16*)db, (__nv_bfloat16*)dc, part);
    else k_axpby_bwd8<float><<<grid, 256, 0, stream>>>((const float*)g, (const float*)b, (const float*)c, c_pitch, s1, s2, NP, C, (float*)db, (float*)dc, part);
  } else {
    const long total = NP * C;
    grid = (int)min(AXPBY_MAX_BLOCKS, (total + 255) / 256);
    if (dtype == FFSR_DT_BF16)
      k_axpby_bwd<__nv_bfloat16><<<grid, 256, 0, stream>>>((const __nv_bfloat16*)g, (const __nv_bfloat16*)b, (const __nv_bfloat16*)c, c_pitch, s1, s2, NP, C, (__nv_bfloat16*)db, (__nv_bfloat16*)dc, part);
    else k_axpby_bwd<float><<<grid, 256, 0, stream>>>((const float*)g, (const float*)b, (const float*)c, c_pitch, s1, s2, NP, C, (float*)db, (float*)dc, part);
  }
  const int rc = ffsr_check_launch("axpby_backward");
  if (rc) return rc;
  launch_sum_slots<float>(part, grid, L, ds, stream);
  return ffsr_check_launch("axpby_backward_reduce");
}
