// LKA depthwise chain on channels-last tensors [N][H][W][C]:
//   n  = BN1(x) inside the image, 0 outside      (LKABlock.forward, large_kernel_attention.py:146)
//   t1 = dw5x5(n)    zero pad 2                   (LargeKernelAttention.forward :98)
//   t2 = dw1x21(t1)  zero pad 10 along W          (:99)
//   t3 = dw21x1(t2)  zero pad 10 along H          (:100)
// Every conv zero-pads ITS OWN input, so intermediates are zero outside the image
// (three separately padded convs != one 25x25 conv at the borders; SURVEY §7 hard part 5).
// HBM/L1-bound: each thread owns one channel and a short run of outputs along the conv
// axis, keeps the sliding window in registers, and warps read 32 consecutive channels.
#include "common.cuh"

namespace {
constexpr int R5 = 4;    // 4x4 output patch per thread for the 5x5 (8x8 input window in registers)
}

// BN is folded to y = x*k + d (eval: running stats; train: batch stats computed upstream).
// CT: compile-time channel count (0 = run time).  With CT the x-direction offsets i * C of the interior path are immediates of
// the load / store instructions: the kernels are issue-bound and the address arithmetic was more than a third of their
// instructions (ncu: 125 M warp instructions for 58 M warp FFMAs in the Phase-4 1x21 pass).
template <typename TI, int CT = 0>
__global__ void __launch_bounds__(256) k_lka_dw5(const TI* __restrict__ x, int H, int W, int C_rt,
                                                 const float* __restrict__ bn_k, const float* __restrict__ bn_d,
                                                 const float* __restrict__ w5, float* __restrict__ out) {
  const int C = CT > 0 ? CT : C_rt;
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  const int runs_x = (W + R5 - 1) / R5, runs_y = (H + R5 - 1) / R5;
  const int idx = blockIdx.y * blockDim.y + threadIdx.y;      // over runs_y * runs_x
  const int y0 = (idx / runs_x) * R5, x0 = (idx % runs_x) * R5;
  const int n = blockIdx.z;
  if (c >= C || idx >= runs_y * runs_x) return;
  float w[25];
#pragma unroll
  for (int i = 0; i < 25; ++i) w[i] = w5[c * 25 + i];
  const float k = bn_k[c], d = bn_d[c];
  float acc[R5][R5];
#pragma unroll
  for (int a = 0; a < R5; ++a)
#pragma unroll
    for (int b = 0; b < R5; ++b) acc[a][b] = 0.f;
  const TI* img = x + (long)n * H * W * C;
  if (y0 >= 2 && y0 + R5 + 2 <= H && x0 >= 2 && x0 + R5 + 2 <= W) {
    // interior patch: no bounds tests, 32-bit strided offsets (the kernel is issue-bound, not HBM-bound)
    const TI* p = img + ((long)(y0 - 2) * W + (x0 - 2)) * C + c;
    const int rs = W * C;
#pragma unroll
    for (int iy = 0; iy < R5 + 4; ++iy) {
      float v[R5 + 4];
#pragma unroll
      for (int i = 0; i < R5 + 4; ++i) v[i] = fmaf(to_f32<TI>(p[iy * rs + i * C]), k, d);
#pragma unroll
      for (int a = 0; a < R5; ++a) {
        const int dy = iy - a;
        if (dy < 0 || dy > 4) continue;
#pragma unroll
        for (int b = 0; b < R5; ++b)
#pragma unroll
          for (int dx = 0; dx < 5; ++dx) acc[a][b] = fmaf(w[dy * 5 + dx], v[b + dx], acc[a][b]);
      }
    }
    float* o = out + (((long)n * H + y0) * W + x0) * C + c;
#pragma unroll
    for (int a = 0; a < R5; ++a)
#pragma unroll
      for (int b = 0; b < R5; ++b) o[a * rs + b * C] = acc[a][b];
    return;
  }
#pragma unroll
  for (int iy = 0; iy < R5 + 4; ++iy) {
    const int yy = y0 + iy - 2;
    if (yy < 0 || yy >= H) continue;                        // zero padding of n = BN1(x)
    float v[R5 + 4];
#pragma unroll
    for (int i = 0; i < R5 + 4; ++i) {
      const int xx = x0 + i - 2;
      v[i] = (xx >= 0 && xx < W) ? fmaf(to_f32<TI>(img[((long)yy * W + xx) * C + c]), k, d) : 0.f;
    }
#pragma unroll
    for (int a = 0; a < R5; ++a) {
      const int dy = iy - a;                                // tap row that maps input row iy to output row a
      if (dy < 0 || dy > 4) continue;
#pragma unroll
      for (int b = 0; b < R5; ++b)
#pragma unroll
        for (int dx = 0; dx < 5; ++dx) acc[a][b] = fmaf(w[dy * 5 + dx], v[b + dx], acc[a][b]);
    }
  }
#pragma unroll
  for (int a = 0; a < R5; ++a)
#pragma unroll
    for (int b = 0; b < R5; ++b)
      if (y0 + a < H && x0 + b < W) out[(((long)n * H + y0 + a) * W + x0 + b) * C + c] = acc[a][b];
}

// Rolling-window 21-tap pass, AXIS = 0: taps along W (1x21); AXIS = 1: taps along H (21x1).  A thread owns one channel and a
// STRIP of up to `strip` outputs along the conv axis and walks it in chunks of 16.  The 36-value window stays in registers;
// each chunk loads only its 16 new values, and loads them one chunk AHEAD, so their latency hides behind the 336 FMAs of the
// current chunk (a one-shot kernel that loaded 36 values per 16 outputs and then waited had 44 % of the issue cycles without
// an eligible warp at 29 % occupancy in ncu).  Every output sums its taps in the order t = 0..20.
template <int AXIS, typename TO, int CT>
__global__ void __launch_bounds__(256) k_lka_dw21_roll(const float* __restrict__ in, int H, int W, int C_rt, const float* __restrict__ w21,
                                                       TO* __restrict__ out, int strip, int nstrips) {
  const int C = CT > 0 ? CT : C_rt;
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  const int n = blockIdx.z;
  const int L = (AXIS == 0) ? W : H, lines = (AXIS == 0) ? H : W;
  const int idx = blockIdx.y * blockDim.y + threadIdx.y;
  if (c >= C || idx >= lines * nstrips) return;
  const int line = idx / nstrips, s0 = (idx - line * nstrips) * strip;
  const int s1 = min(s0 + strip, L);
  if (s0 >= s1) return;
  const long stride = (AXIS == 0) ? C : (long)W * C;
  const long lbase = (long)n * H * W * C + ((AXIS == 0) ? (long)line * W * C : (long)line * C) + c;
  const float* base = in + lbase;
  TO* obase = out + lbase;
  float w[21];
#pragma unroll
  for (int i = 0; i < 21; ++i) w[i] = w21[c * 21 + i];
  float v[36];
#pragma unroll
  for (int i = 0; i < 36; ++i) {
    const int q = s0 - 10 + i;
    v[i] = (q >= 0 && q < L) ? base[q * stride] : 0.f;
  }
#pragma unroll 1
  for (int pos = s0; pos < s1; pos += 16) {
    float nv[16];
    const bool more = pos + 16 < s1;
    const float* pn = base + (long)(pos + 26) * stride;
    if (more && pos + 42 <= L) {
#pragma unroll
      for (int i = 0; i < 16; ++i) nv[i] = pn[i * stride];
    } else {
#pragma unroll
      for (int i = 0; i < 16; ++i) nv[i] = (more && pos + 26 + i < L) ? pn[i * stride] : 0.f;
    }
    TO* po = obase + (long)pos * stride;
    if (pos + 16 <= s1) {
#pragma unroll
      for (int r = 0; r < 16; ++r) {
        float acc = 0.f;
#pragma unroll
        for (int t = 0; t < 21; ++t) acc = fmaf(w[t], v[r + t], acc);
        po[r * stride] = from_f32<TO>(acc);
      }
    } else {
#pragma unroll
      for (int r = 0; r < 16; ++r) {
        float acc = 0.f;
#pragma unroll
        for (int t = 0; t < 21; ++t) acc = fmaf(w[t], v[r + t], acc);
        if (pos + r < s1) po[r * stride] = from_f32<TO>(acc);
      }
    }
#pragma unroll
    for (int i = 0; i < 20; ++i) v[i] = v[i + 16];
#pragma unroll
    for (int i = 0; i < 16; ++i) v[20 + i] = nv[i];
  }
}

// A line of L outputs of the rolling-window passes as `n` strips of `len` <= 256 outputs (a multiple of 16)
struct DwStrips {
  int n, len;
};
static DwStrips dw_strips(int L) {
  const int n = ceil_div(L, 256);
  return {n, ceil_div(ceil_div(L, n), 16) * 16};
}

// x: [N][H][W][C] -> out: [N][H][W][C]; tmp1/tmp2: same-size scratch (tmp2 may alias out? no: distinct)
static int lka_depthwise_impl(const void* x, int x_dtype, int N, int H, int W, int C, const float* bn_k, const float* bn_d,
                              const float* w5, const float* wh, const float* wv, float* tmp1, float* tmp2, void* out,
                              int out_dtype, cudaStream_t stream);

extern "C" int ffsr_lka_depthwise(const float* x, int N, int H, int W, int C, const float* bn_k, const float* bn_d,
                                  const float* w5, const float* wh, const float* wv, float* tmp1, float* tmp2,
                                  void* out, int out_dtype, cudaStream_t stream) {
  return lka_depthwise_impl(x, 0, N, H, W, C, bn_k, bn_d, w5, wh, wv, tmp1, tmp2, out, out_dtype, stream);
}
// same chain with a bf16 input tensor (bf16 mode: the Phase-4 residual stream is stored as bf16)
extern "C" int ffsr_lka_depthwise_in(const void* x, int x_dtype, int N, int H, int W, int C, const float* bn_k,
                                     const float* bn_d, const float* w5, const float* wh, const float* wv, float* tmp1,
                                     float* tmp2, void* out, int out_dtype, cudaStream_t stream) {
  return lka_depthwise_impl(x, x_dtype, N, H, W, C, bn_k, bn_d, w5, wh, wv, tmp1, tmp2, out, out_dtype, stream);
}

static int lka_depthwise_impl(const void* x, int x_dtype, int N, int H, int W, int C, const float* bn_k, const float* bn_d,
                              const float* w5, const float* wh, const float* wv, float* tmp1, float* tmp2, void* out,
                              int out_dtype, cudaStream_t stream) {
  FFSR_REQUIRE(x && bn_k && bn_d && w5 && wh && wv && tmp1 && tmp2 && out, FFSR_ERR_ARG, "lka_depthwise: null pointer");
  FFSR_REQUIRE(N > 0 && H > 0 && W > 0 && C > 0 && C % 32 == 0, FFSR_ERR_ARG, "lka_depthwise: C must be a multiple of 32");
  FFSR_REQUIRE(N <= 65535 && (long)H * W / 4 < 65535L * 4, FFSR_ERR_ARG, "lka_depthwise: grid too large");
  const int cx = C < 64 ? C : 64;
  const int ty = 256 / cx;
  const dim3 block(cx, ty);
  const dim3 g5(C / cx, ceil_div((long)ceil_div(H, R5) * ceil_div(W, R5), ty), N);
  typedef __nv_bfloat16 bf;
  const DwStrips sw = dw_strips(W), sh = dw_strips(H);
  const dim3 rh(C / cx, ceil_div((long)H * sw.n, ty), N);
  const dim3 rv(C / cx, ceil_div((long)W * sh.n, ty), N);
#define FFSR_DW_CHAIN(CT)                                                                                                    \
  {                                                                                                                          \
    if (x_dtype == 1) k_lka_dw5<bf, CT><<<g5, block, 0, stream>>>((const bf*)x, H, W, C, bn_k, bn_d, w5, tmp1);             \
    else k_lka_dw5<float, CT><<<g5, block, 0, stream>>>((const float*)x, H, W, C, bn_k, bn_d, w5, tmp1);                     \
    k_lka_dw21_roll<0, float, CT><<<rh, block, 0, stream>>>(tmp1, H, W, C, wh, tmp2, sw.len, sw.n);                          \
    if (out_dtype == 1) k_lka_dw21_roll<1, bf, CT><<<rv, block, 0, stream>>>(tmp2, H, W, C, wv, (bf*)out, sh.len, sh.n);     \
    else k_lka_dw21_roll<1, float, CT><<<rv, block, 0, stream>>>(tmp2, H, W, C, wv, (float*)out, sh.len, sh.n);              \
  }
  if (C == 128) FFSR_DW_CHAIN(128) else if (C == 64) FFSR_DW_CHAIN(64) else FFSR_DW_CHAIN(0)
#undef FFSR_DW_CHAIN
  return ffsr_check_launch("lka_depthwise");
}

// ------------------------------------------------------------------------------------
// Train-mode access to the individual stages (the backward pass runs them with flipped taps:
// the input gradient of a zero-padded stride-1 depthwise conv is the same conv with reversed
// taps), and the depthwise weight gradients  dw[c][tap] = sum_{n,y,x} in[n,y+dy,x+dx,c] * g[n,y,x,c].
// kind: 0 = 5x5 (pad 2), 1 = 1x21 along W (pad 10), 2 = 21x1 along H (pad 10).
// ------------------------------------------------------------------------------------
extern "C" int ffsr_dwconv_stage(const float* in, int N, int H, int W, int C, int kind, const float* w,
                                 const float* bn_k, const float* bn_d, float* out, cudaStream_t stream) {
  FFSR_REQUIRE(in && w && out, FFSR_ERR_ARG, "dwconv_stage: null pointer");
  FFSR_REQUIRE(N > 0 && H > 0 && W > 0 && C > 0 && C % 32 == 0, FFSR_ERR_ARG, "dwconv_stage: C must be a multiple of 32");
  FFSR_REQUIRE(N <= 65535 && (long)H * W / 4 < 65535L * 4, FFSR_ERR_ARG, "dwconv_stage: grid too large");
  FFSR_REQUIRE(kind >= 0 && kind <= 2, FFSR_ERR_ARG, "dwconv_stage: kind must be 0, 1 or 2");
  FFSR_REQUIRE(kind != 0 || (bn_k && bn_d), FFSR_ERR_ARG, "dwconv_stage: the 5x5 stage needs the input affine (ones/zeros for none)");
  const int cx = C < 64 ? C : 64;
  const int ty = 256 / cx;
  dim3 block(cx, ty);
  if (kind == 0) {
    dim3 grid(C / cx, ceil_div((long)ceil_div(H, R5) * ceil_div(W, R5), ty), N);
    k_lka_dw5<float><<<grid, block, 0, stream>>>(in, H, W, C, bn_k, bn_d, w, out);
  } else {
    // the rolling-window passes of the inference chain, cut into the same strips
    const int lines = kind == 1 ? H : W;
    const DwStrips st = dw_strips(kind == 1 ? W : H);
    dim3 grid(C / cx, ceil_div((long)lines * st.n, ty), N);
    if (kind == 1) {
      if (C == 128) k_lka_dw21_roll<0, float, 128><<<grid, block, 0, stream>>>(in, H, W, C, w, out, st.len, st.n);
      else if (C == 64) k_lka_dw21_roll<0, float, 64><<<grid, block, 0, stream>>>(in, H, W, C, w, out, st.len, st.n);
      else k_lka_dw21_roll<0, float, 0><<<grid, block, 0, stream>>>(in, H, W, C, w, out, st.len, st.n);
    } else {
      if (C == 128) k_lka_dw21_roll<1, float, 128><<<grid, block, 0, stream>>>(in, H, W, C, w, out, st.len, st.n);
      else if (C == 64) k_lka_dw21_roll<1, float, 64><<<grid, block, 0, stream>>>(in, H, W, C, w, out, st.len, st.n);
      else k_lka_dw21_roll<1, float, 0><<<grid, block, 0, stream>>>(in, H, W, C, w, out, st.len, st.n);
    }
  }
  return ffsr_check_launch("dwconv_stage");
}

namespace {
constexpr int WG_R = 8;    // outputs per thread along the conv axis in the 21-tap weight-gradient kernel

// Both weight-gradient kernels: blockDim = (channels, item rows); grid = (channel blocks, Y, images), and
// thread row ty of block y takes items y*blockDim.y + ty, stepping by Y*blockDim.y, summing in registers.
// The rows of a block are summed in order in shared memory and the block's [channels][taps] partial goes to
// slot (n*Y + y) of part [N*Y][C][taps], reduced in slot order by k_sum_slots: no atomics, bitwise reproducible.
template <int TAPS>
__device__ __forceinline__ void dw_wgrad_store(const float (&acc)[TAPS], int C, float* sdw, float* __restrict__ part) {
  const int tl = threadIdx.y * blockDim.x + threadIdx.x;
  const int CB = blockDim.x * TAPS;
#pragma unroll
  for (int t = 0; t < TAPS; ++t) sdw[(threadIdx.y * blockDim.x + threadIdx.x) * TAPS + t] = acc[t];
  __syncthreads();
  float* slot = part + ((long)blockIdx.z * gridDim.y + blockIdx.y) * C * TAPS + (long)blockIdx.x * CB;
  for (int i = tl; i < CB; i += blockDim.x * blockDim.y) {
    float s = 0.f;
    for (int r = 0; r < (int)blockDim.y; ++r) s += sdw[r * CB + i];
    slot[i] = s;
  }
}

// AXIS 0: taps along W, AXIS 1: taps along H.  Each thread owns one channel and WG_R consecutive outputs per item.
template <int AXIS>
__global__ void __launch_bounds__(256) k_dw21_wgrad(const float* __restrict__ in, const float* __restrict__ g, int H,
                                                    int W, int C, long items, float* __restrict__ part) {
  extern __shared__ float sdw[];            // [blockDim.y][blockDim.x][21]
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  const int n = blockIdx.z;
  float acc[21];
#pragma unroll
  for (int t = 0; t < 21; ++t) acc[t] = 0.f;
  for (long idx = (long)blockIdx.y * blockDim.y + threadIdx.y; c < C && idx < items; idx += (long)gridDim.y * blockDim.y) {
    int y, x;
    if (AXIS == 0) {
      const int runs = (W + WG_R - 1) / WG_R;
      y = (int)(idx / runs);
      x = (int)(idx % runs) * WG_R;
    } else {
      y = (int)(idx / W) * WG_R;
      x = (int)(idx % W);
    }
    const float* img = in + (long)n * H * W * C;
    const float* gim = g + (long)n * H * W * C;
    float v[WG_R + 20], gr[WG_R];
#pragma unroll
    for (int i = 0; i < WG_R + 20; ++i) {
      if (AXIS == 0) {
        const int xx = x + i - 10;
        v[i] = (xx >= 0 && xx < W) ? img[((long)y * W + xx) * C + c] : 0.f;
      } else {
        const int yy = y + i - 10;
        v[i] = (yy >= 0 && yy < H) ? img[((long)yy * W + x) * C + c] : 0.f;
      }
    }
#pragma unroll
    for (int r = 0; r < WG_R; ++r) {
      if (AXIS == 0) gr[r] = (x + r < W) ? gim[((long)y * W + x + r) * C + c] : 0.f;
      else gr[r] = (y + r < H) ? gim[((long)(y + r) * W + x) * C + c] : 0.f;
    }
#pragma unroll
    for (int t = 0; t < 21; ++t) {
      float a = 0.f;
#pragma unroll
      for (int r = 0; r < WG_R; ++r) a = fmaf(v[r + t], gr[r], a);
      acc[t] += a;
    }
  }
  dw_wgrad_store<21>(acc, C, sdw, part);
}

__global__ void __launch_bounds__(256) k_dw5_wgrad(const float* __restrict__ in, const float* __restrict__ g, int H,
                                                   int W, int C, long items, float* __restrict__ part) {
  extern __shared__ float sdw[];            // [blockDim.y][blockDim.x][25]
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  const int n = blockIdx.z;
  float acc[25];
#pragma unroll
  for (int i = 0; i < 25; ++i) acc[i] = 0.f;
  for (long idx = (long)blockIdx.y * blockDim.y + threadIdx.y; c < C && idx < items; idx += (long)gridDim.y * blockDim.y) {
    const int runs_x = (W + R5 - 1) / R5;
    const int y0 = (int)(idx / runs_x) * R5, x0 = (int)(idx % runs_x) * R5;
    const float* img = in + (long)n * H * W * C;
    const float* gim = g + (long)n * H * W * C;
    float gr[R5][R5];
#pragma unroll
    for (int a = 0; a < R5; ++a)
#pragma unroll
      for (int b = 0; b < R5; ++b)
        gr[a][b] = (y0 + a < H && x0 + b < W) ? gim[((long)(y0 + a) * W + x0 + b) * C + c] : 0.f;
#pragma unroll
    for (int iy = 0; iy < R5 + 4; ++iy) {
      const int yy = y0 + iy - 2;
      float v[R5 + 4];
#pragma unroll
      for (int i = 0; i < R5 + 4; ++i) {
        const int xx = x0 + i - 2;
        v[i] = (yy >= 0 && yy < H && xx >= 0 && xx < W) ? img[((long)yy * W + xx) * C + c] : 0.f;
      }
#pragma unroll
      for (int a = 0; a < R5; ++a) {
        const int dy = iy - a;
        if (dy < 0 || dy > 4) continue;
#pragma unroll
        for (int b = 0; b < R5; ++b)
#pragma unroll
          for (int dx = 0; dx < 5; ++dx) acc[dy * 5 + dx] = fmaf(v[b + dx], gr[a][b], acc[dy * 5 + dx]);
      }
    }
  }
  dw_wgrad_store<25>(acc, C, sdw, part);
}

constexpr int DWG_CX = 32, DWG_TY = 8;

// items of one image and the item-row blocks Y per image (about 8 blocks per SM over the whole grid)
inline long dw_wgrad_items(int H, int W, int kind) {
  if (kind == 0) return (long)ceil_div(H, R5) * ceil_div(W, R5);
  if (kind == 1) return (long)H * ceil_div(W, WG_R);
  return (long)ceil_div(H, WG_R) * W;
}
inline int dw_wgrad_Y(int N, int H, int W, int C, int kind) {
  const long rows = ceil_div(dw_wgrad_items(H, W, kind), DWG_TY);
  long Y = (148L * 8) / ((long)(C / DWG_CX) * N);
  if (Y > rows) Y = rows;
  return Y < 1 ? 1 : (int)Y;
}
}  // namespace

extern "C" size_t ffsr_dwconv_wgrad_workspace_bytes(int N, int H, int W, int C, int kind) {
  if (N <= 0 || H <= 0 || W <= 0 || C <= 0 || C % DWG_CX != 0 || kind < 0 || kind > 2) return 0;
  return (size_t)N * dw_wgrad_Y(N, H, W, C, kind) * C * (kind == 0 ? 25 : 21) * sizeof(float);
}

// dw: [C][taps] fp32, ACCUMULATED into (caller zeroes)
extern "C" int ffsr_dwconv_wgrad(const float* in, const float* g, int N, int H, int W, int C, int kind, float* dw,
                                 void* ws, size_t ws_bytes, cudaStream_t stream) {
  FFSR_REQUIRE(in && g && dw && ws, FFSR_ERR_ARG, "dwconv_wgrad: null pointer");
  FFSR_REQUIRE(N > 0 && N <= 65535 && H > 0 && W > 0 && C > 0 && C % 32 == 0, FFSR_ERR_ARG, "dwconv_wgrad: bad shape");
  FFSR_REQUIRE(kind >= 0 && kind <= 2, FFSR_ERR_ARG, "dwconv_wgrad: kind must be 0, 1 or 2");
  FFSR_REQUIRE(ws_bytes >= ffsr_dwconv_wgrad_workspace_bytes(N, H, W, C, kind), FFSR_ERR_ARG, "dwconv_wgrad: workspace too small");
  const int Y = dw_wgrad_Y(N, H, W, C, kind);
  const long items = dw_wgrad_items(H, W, kind);
  const int taps = kind == 0 ? 25 : 21;
  dim3 block(DWG_CX, DWG_TY), grid(C / DWG_CX, Y, N);
  const size_t smem = (size_t)DWG_CX * DWG_TY * taps * sizeof(float);
  float* part = (float*)ws;
  if (kind == 0) k_dw5_wgrad<<<grid, block, smem, stream>>>(in, g, H, W, C, items, part);
  else if (kind == 1) k_dw21_wgrad<0><<<grid, block, smem, stream>>>(in, g, H, W, C, items, part);
  else k_dw21_wgrad<1><<<grid, block, smem, stream>>>(in, g, H, W, C, items, part);
  const int rc = ffsr_check_launch("dwconv_wgrad");
  if (rc) return rc;
  launch_sum_slots<float>(part, N * Y, (long)C * taps, dw, stream);
  return ffsr_check_launch("dwconv_wgrad_reduce");
}
