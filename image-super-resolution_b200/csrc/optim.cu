// Fused optimizer step over ONE flat fp32 parameter bucket (SURVEY 2.3 K11):
//   global-norm gradient clipping  torch.nn.utils.clip_grad_norm_(model.parameters(), 1.0)   train.py:344-348
//   AdamW                          torch.optim.AdamW(lr, betas, eps, weight_decay)           train.py:847-853
//   EMA shadow update              EMAModel.update                    src/utils/checkpoint_manager.py:352-359
// The reference runs these as ~600 small ATen launches per step (198 tensors x 3); here it is one
// reduction + one elementwise pass: 20 B read + 16 B written per parameter.  No host sync: the clip
// coefficient is derived on the device from the squared-norm accumulator.
#include <type_traits>

#include "common.cuh"
#include "../../include/ffsr_b200.h"

namespace {
// block sums of g^2 -> part[blockIdx.x], added in block order by k_sum_slots (bitwise reproducible clip coefficient)
__global__ void __launch_bounds__(256) k_sumsq(const float* __restrict__ g, long n, double* __restrict__ part) {
  __shared__ double sh[8];
  double acc = 0.0;
  float f = 0.f;
  int cnt = 0;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    f = fmaf(g[i], g[i], f);
    if (++cnt == 16) { acc += f; f = 0.f; cnt = 0; }
  }
  acc += f;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int i = 0; i < 8; ++i) s += sh[i];
    part[blockIdx.x] = s;
  }
}

__global__ void __launch_bounds__(256) k_adamw_ema(float* __restrict__ p, const float* __restrict__ g,
                                                   float* __restrict__ m, float* __restrict__ v,
                                                   float* __restrict__ ema, long n, float lr, float b1, float b2,
                                                   float eps, float wd, int step, const int* __restrict__ step_dev,
                                                   const float* __restrict__ lr_dev,
                                                   const double* __restrict__ gsumsq, float grad_scale,
                                                   float max_norm, float ema_decay) {
  if (step_dev) step += *step_dev;
  if (lr_dev) lr = *lr_dev;
  const float bc1 = 1.0f - (float)pow((double)b1, (double)step);
  const float bc2_sqrt = (float)sqrt(1.0 - pow((double)b2, (double)step));
  float clip = 1.0f;
  if (gsumsq && max_norm > 0.f) {
    const float norm = grad_scale * (float)sqrt(*gsumsq);
    clip = fminf(1.0f, max_norm / (norm + 1e-6f));
  }
  const float gs = grad_scale * clip;
  const float step_size = lr / bc1;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    const float gi = g[i] * gs;
    float pi = p[i] * (1.0f - lr * wd);
    const float mi = b1 * m[i] + (1.0f - b1) * gi;
    const float vi = b2 * v[i] + (1.0f - b2) * gi * gi;
    pi -= step_size * mi / (sqrtf(vi) / bc2_sqrt + eps);
    p[i] = pi; m[i] = mi; v[i] = vi;
    if (ema) ema[i] = ema_decay * ema[i] + (1.0f - ema_decay) * pi;
  }
}

// out[i] = (...((s_0[i] + s_1[i]) + s_2[i]) ... + s_{M-1}[i]) with s_m = slots + m * pitch: one thread owns VEC
// consecutive entries and adds the M slots in slot order, one fp32 rounding per add (__fadd_rn is never contracted
// into an FMA), so each entry depends on its M inputs only -- not on the grid, the block size or which path ran.
// The world-invariant training step sums its per-micro-batch gradient rows with it.
template <int VEC>
__global__ void __launch_bounds__(256) k_sum_slots_ordered(const float* __restrict__ slots, int M, long n, long pitch,
                                                           float* __restrict__ out) {
  using V = typename std::conditional<VEC == 4, float4, float>::type;
  const long nv = n / VEC, pv = pitch / VEC;
  const V* __restrict__ s = reinterpret_cast<const V*>(slots);
  V* __restrict__ o = reinterpret_cast<V*>(out);
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += (long)gridDim.x * blockDim.x) {
    V a = s[i];
#pragma unroll 4
    for (int m = 1; m < M; ++m) {
      const V b = s[(long)m * pv + i];
      if constexpr (VEC == 4) {
        a.x = __fadd_rn(a.x, b.x);
        a.y = __fadd_rn(a.y, b.y);
        a.z = __fadd_rn(a.z, b.z);
        a.w = __fadd_rn(a.w, b.w);
      } else {
        a = __fadd_rn(a, b);
      }
    }
    o[i] = a;
  }
  if (VEC > 1 && blockIdx.x == 0 && threadIdx.x < n - nv * VEC) {   // the last n % VEC entries
    const long i = nv * VEC + threadIdx.x;
    float a = slots[i];
    for (int m = 1; m < M; ++m) a = __fadd_rn(a, slots[(long)m * pitch + i]);
    out[i] = a;
  }
}
}  // namespace

extern "C" int ffsr_sum_slots_ordered(const float* slots, int M, long n, long pitch, float* out, cudaStream_t stream) {
  FFSR_REQUIRE(slots && out && M >= 1 && n >= 1 && pitch >= n, FFSR_ERR_ARG, "sum_slots_ordered: bad argument");
  FFSR_REQUIRE(out + n <= slots || out >= slots + (long)(M - 1) * pitch + n, FFSR_ERR_ARG,
               "sum_slots_ordered: out overlaps the slots");
  // 16-byte loads and stores when every slot row and the output start on a 16-byte boundary
  const bool vec = ((uintptr_t)slots % 16 == 0) && ((uintptr_t)out % 16 == 0) && (pitch % 4 == 0);
  const long items = vec ? n / 4 : n;
  const int grid = (int)(items <= 0 ? 1 : ((items + 255) / 256 < 148L * 8 ? (items + 255) / 256 : 148L * 8));
  if (vec) k_sum_slots_ordered<4><<<grid, 256, 0, stream>>>(slots, M, n, pitch, out);
  else k_sum_slots_ordered<1><<<grid, 256, 0, stream>>>(slots, M, n, pitch, out);
  return ffsr_check_launch("sum_slots_ordered");
}

static inline int sumsq_grid(long n) { return (int)((n + 255) / 256 < 148L * 4 ? (n + 255) / 256 : 148L * 4); }

extern "C" size_t ffsr_sumsq_workspace_bytes(long n) { return n > 0 ? (size_t)sumsq_grid(n) * sizeof(double) : 0; }

extern "C" int ffsr_sumsq(const float* g, long n, double* out, void* ws, size_t ws_bytes, cudaStream_t stream) {
  FFSR_REQUIRE(g && out && ws && n > 0, FFSR_ERR_ARG, "sumsq: bad argument");
  FFSR_REQUIRE(ws_bytes >= ffsr_sumsq_workspace_bytes(n), FFSR_ERR_ARG, "sumsq: workspace too small");
  const int grid = sumsq_grid(n);
  k_sumsq<<<grid, 256, 0, stream>>>(g, n, (double*)ws);
  const int rc = ffsr_check_launch("sumsq");
  if (rc) return rc;
  launch_sum_slots<double>((const double*)ws, grid, 1, out, stream);
  return ffsr_check_launch("sumsq_reduce");
}

extern "C" int ffsr_adamw_ema_step(float* p, const float* g, float* m, float* v, float* ema, long n, float lr,
                                   float beta1, float beta2, float eps, float weight_decay, int step,
                                   const int* step_dev, const float* lr_dev, const double* gsumsq, float grad_scale,
                                   float max_norm, float ema_decay, cudaStream_t stream) {
  FFSR_REQUIRE(p && g && m && v && n > 0 && (step >= 1 || step_dev), FFSR_ERR_ARG, "adamw_ema_step: bad argument");
  const int grid = (int)((n + 255) / 256 < 148L * 8 ? (n + 255) / 256 : 148L * 8);
  k_adamw_ema<<<grid, 256, 0, stream>>>(p, g, m, v, ema, n, lr, beta1, beta2, eps, weight_decay, step, step_dev, lr_dev,
                                        gsumsq, grad_scale, max_norm, ema_decay);
  return ffsr_check_launch("adamw_ema_step");
}
