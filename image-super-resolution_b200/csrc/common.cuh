// Shared device helpers for the FreqFusionSR sm_100a kernels.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <math.h>

#define FFSR_OK 0
#define FFSR_ERR_ARG (-1)      // bad shape / null pointer / unsupported combination
#define FFSR_ERR_ALIGN (-2)    // pointer or stride misaligned for the vector path
#define FFSR_ERR_LAUNCH (-3)   // cudaGetLastError() after the launch was not cudaSuccess
#define FFSR_ERR_DRIVER (-4)   // driver entry point (tensor-map encode) unavailable

void ffsr_set_error(const char* fmt, ...);
int ffsr_check_launch(const char* what);

#define FFSR_REQUIRE(cond, code, ...)                 \
  do {                                                \
    if (!(cond)) {                                    \
      ffsr_set_error(__VA_ARGS__);                    \
      return (code);                                  \
    }                                                 \
  } while (0)

static inline int ceil_div(long a, long b) { return (int)((a + b - 1) / b); }

// Fixed-order cross-block reduction of the training kernels.  A partial kernel partitions its work by shape
// alone and writes one slot per block, slots[k][0..L), each entry of each slot exactly once (no atomics);
// k_sum_slots then adds sum_k slots[k][i] to out[i] (entries i >= L1 go to out2[i - L1]).  One 1024-thread block
// per 32 entries: thread (x = tid % 32, y = tid / 32) sums slots y, y+32, ... of entry x in order and row y == 0
// adds the 32 group sums in order, so the result depends on (nslots, L) only, never on block scheduling: training
// steps are bitwise reproducible.  Outputs keep their accumulate-into semantics.  One launch can finish two
// independent reductions (a weight gradient and its bias sums).
template <typename T>
struct SlotSum {
  const T* slots;
  int nslots;
  long L, L1;
  T* out;
  T* out2;
};
template <typename T>
inline SlotSum<T> slot_sum(const T* slots, int nslots, long L, T* out, T* out2 = nullptr, long L1 = -1) {
  return SlotSum<T>{slots, nslots, L, L1 < 0 ? L : L1, out, out2};
}
template <typename T>
__host__ __device__ inline long slot_sum_blocks(const SlotSum<T>& j) { return j.slots ? (j.L + 31) / 32 : 0; }

// the 32 entries [32*chunk, 32*chunk + 32) of j; every thread of a 1024-thread block calls it
template <typename T>
__device__ __forceinline__ void sum_slots_chunk(const SlotSum<T>& j, long chunk) {
  __shared__ T sh[32][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const long i = chunk * 32 + tx;
  T s = 0;
  if (i < j.L) {
#pragma unroll 4
    for (int k = ty; k < j.nslots; k += 32) s += j.slots[(long)k * j.L + i];
  }
  sh[ty][tx] = s;
  __syncthreads();
  if (ty == 0 && i < j.L) {
    T t = 0;
    for (int g = 0; g < 32; ++g) t += sh[g][tx];
    if (i < j.L1) j.out[i] += t;
    else j.out2[i - j.L1] += t;
  }
}

template <typename T>
__global__ void __launch_bounds__(1024) k_sum_slots(const SlotSum<T> a, const SlotSum<T> b) {
  const long na = slot_sum_blocks(a);
  if ((long)blockIdx.x < na) sum_slots_chunk(a, blockIdx.x);
  else sum_slots_chunk(b, blockIdx.x - na);
}

template <typename T>
static inline void launch_sum_slots(const SlotSum<T>& a, const SlotSum<T>& b, cudaStream_t stream) {
  k_sum_slots<T><<<(unsigned)(slot_sum_blocks(a) + slot_sum_blocks(b)), 1024, 0, stream>>>(a, b);
}
template <typename T>
static inline void launch_sum_slots(const T* slots, int nslots, long L, T* out, cudaStream_t stream, T* out2 = nullptr,
                                    long L1 = -1) {
  launch_sum_slots<T>(slot_sum(slots, nslots, L, out, out2, L1), SlotSum<T>{}, stream);
}

// bias sums of the weight-gradient entry points: column-sum partials [nslots][C] of ffsr_colsum into part
// (ffsr_colsum_workspace_bytes), finished by the caller's k_sum_slots launch
int colsum_partials(const void* v, int dtype, int N, int H, int W, int C, long long sN, long long sY, long long sX,
                    float* part, int* nslots, cudaStream_t stream);
// partial slots placed after `bytes` of other scratch in one workspace
inline size_t ws_align(size_t bytes) { return (bytes + 255) / 256 * 256; }

// activation codes shared with the host side
enum { ACT_NONE = 0, ACT_GELU = 1, ACT_RELU = 2, ACT_SIGMOID = 3 };

__device__ __forceinline__ float gelu_erf(float x) {
  return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f));
}
__device__ __forceinline__ float sigmoid_acc(float x) { return 1.0f / (1.0f + expf(-x)); }
// GELU with erf by Abramowitz-Stegun 7.1.26 (|abs err| <= 1.5e-7) on the fast-math units: used where the
// result is rounded to bf16 anyway (bf16 precision mode); ~2x cheaper than erff().
__device__ __forceinline__ float gelu_as(float x) {
  const float z = fabsf(x) * 0.70710678118654752440f;
  const float t = __fdividef(1.0f, fmaf(0.3275911f, z, 1.0f));
  float poly = fmaf(1.061405429f, t, -1.453152027f);
  poly = fmaf(poly, t, 1.421413741f);
  poly = fmaf(poly, t, -0.284496736f);
  poly = fmaf(poly, t, 0.254829592f);
  const float erf_abs = 1.0f - poly * t * __expf(-z * z);
  return 0.5f * x * (1.0f + copysignf(erf_abs, x));
}
// tanh-form GELU on the MUFU (6 instructions): |error| <= 4.8e-4 against the erf form.  Only for bf16-mode INFERENCE
// kernels whose GELU feeds a sigmoid gate head (k_modulate_hr, k_spatial_gate), where the error is damped again.
__device__ __forceinline__ float gelu_tanh(float x) {
  const float u = x * fmaf(0.0356774081f, x * x, 0.7978845608f);
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(u));
  const float hx = 0.5f * x;
  return fmaf(hx, t, hx);
}
template <bool FAST>
__device__ __forceinline__ float gelu_sel(float x) { return FAST ? gelu_tanh(x) : gelu_erf(x); }

__device__ __forceinline__ float apply_act(float v, int act) {
  switch (act) {
    case ACT_GELU: return gelu_erf(v);
    case ACT_RELU: return fmaxf(v, 0.0f);
    case ACT_SIGMOID: return sigmoid_acc(v);
    default: return v;
  }
}

// Bilinear, align_corners=False, explicit output size (SURVEY Appendix A):
//   src = max(0, (dst+0.5)*in/out - 0.5); i0 = floor(src); i1 = min(i0+1, in-1); w1 = src - i0
struct BilinTap {
  int i0, i1;
  float w0, w1;
};
__device__ __forceinline__ BilinTap bilin_tap(int dst, int in_size, int out_size) {
  const float scale = (float)in_size / (float)out_size;
  float src = scale * ((float)dst + 0.5f) - 0.5f;
  src = src < 0.0f ? 0.0f : src;
  int i0 = (int)src;
  if (i0 > in_size - 1) i0 = in_size - 1;
  BilinTap t;
  t.i0 = i0;
  t.i1 = i0 + (i0 < in_size - 1 ? 1 : 0);
  t.w1 = src - (float)i0;
  t.w0 = 1.0f - t.w1;
  return t;
}

// numpy-style reflect (edge not repeated); valid for -n < i < 2n-1
__device__ __forceinline__ int reflect_idx(int i, int n) {
  if (i < 0) i = -i;
  if (i >= n) i = 2 * n - 2 - i;
  return i;
}

template <typename T>
__device__ __forceinline__ float to_f32(T v);
template <>
__device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <>
__device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }

template <typename T>
__device__ __forceinline__ T from_f32(float v);
template <>
__device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <>
__device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }
