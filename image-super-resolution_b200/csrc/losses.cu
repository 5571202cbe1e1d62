// Fused stage-2/3 training losses with their backward passes (SURVEY 8a rows L-L1, L-SWT, L-FFT, L-SSIM):
// each entry point accumulates the loss partial sums (fp64) AND adds  weight * dLoss/dPred  into `dpred`
// in the same pass over the data, so loss.backward() costs nothing extra.  Each block writes its fp64 partial
// sums to a slot of the workspace and k_sum_slots adds them in slot order: the loss values are bitwise
// reproducible (no atomics).
//   L1    src/losses/perceptual_loss.py:86-104
//   SSIM  src/losses/perceptual_loss.py:225-291   (11x11 Gaussian sigma 1.5, zero pad 5, C1=1e-4, C2=9e-4)
//   FFT   src/losses/perceptual_loss.py:533-598   (fft2 ortho, |mag| + 0.1 |phase| L1, radial weights)
//   SWT   src/losses/perceptual_loss.py:661-733, 797-813  (Haar, 2 levels, reflect pad 2^l, dilation 2^l)
// pred / target / dpred: [P][H][W] fp32 planes (P = B*C, NCHW contiguous).  HBM-bound elementwise /
// small-stencil kernels; the 2-D FFT is a shared-memory Stockham transform (rows, then 4-column strips)
// with pred and target packed as the real and imaginary part of ONE complex transform.
#include "common.cuh"
#include "../../include/ffsr_b200.h"

namespace {

__device__ __forceinline__ float sgn(float v) { return (float)((v > 0.f) - (v < 0.f)); }

// block sum of v -> part[linear block index][0..NV)
template <int NV>
__device__ __forceinline__ void block_sum_slot(double (&v)[NV], double* part) {
  __shared__ double sh[NV][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v[i] += __shfl_down_sync(0xffffffffu, v[i], o);
    if (lane == 0) sh[i][warp] = v[i];
  }
  __syncthreads();
  if (warp == 0) {
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      double s = lane < nw ? sh[i][lane] : 0.0;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
      if (lane == 0) part[((long)(blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x) * NV + i] = s;
    }
  }
}

// ------------------------------------------------------------------------------------ L1
__global__ void __launch_bounds__(256) k_loss_l1(const float* __restrict__ p, const float* __restrict__ t, long n,
                                                 float gscale, double* __restrict__ sum, float* __restrict__ dpred) {
  double acc[1] = {0.0};
  float f = 0.f;
  int cnt = 0;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    const float d = p[i] - t[i];
    f += fabsf(d);
    dpred[i] += gscale * sgn(d);
    if (++cnt == 32) { acc[0] += f; f = 0.f; cnt = 0; }
  }
  acc[0] += f;
  block_sum_slot<1>(acc, sum);
}

// ------------------------------------------------------------------------------------ SWT
// One undecimated Haar level on cur = a - b (b optional):
//   c_b[y][x] = sum_ij f_b[i][j] * cur[refl(y+(i-1)d)][refl(x+(j-1)d)]
// Optionally stores the approximation, accumulates sum|c_b| and writes the four tap-gradient planes
//   G_ij = sum_b f_b[i][j] * g_b,   g_b = gscale*w_b*sign(c_b) (+ gA_in for the approximation band)
__global__ void __launch_bounds__(256) k_swt_level(const float* __restrict__ a, const float* __restrict__ b, long total,
                                                   int H, int W, int d, float* __restrict__ outA,
                                                   const float* __restrict__ gA_in, float gscale,
                                                   double* __restrict__ sums, float* __restrict__ G) {
  const float s = 0.70710677f;
  const float h = s * s;
  double acc[4] = {0.0, 0.0, 0.0, 0.0};
  float fa[4] = {0.f, 0.f, 0.f, 0.f};
  int cnt = 0;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    const int x = (int)(idx % W);
    const int y = (int)((idx / W) % H);
    const long base = idx - ((long)y * W + x);
    int ym = y - d, xm = x - d;
    ym = ym < 0 ? -ym : ym;
    xm = xm < 0 ? -xm : xm;
    const long i00 = base + (long)ym * W + xm, i01 = base + (long)ym * W + x, i10 = base + (long)y * W + xm;
    float v00 = a[i00], v01 = a[i01], v10 = a[i10], v11 = a[idx];
    if (b) { v00 -= b[i00]; v01 -= b[i01]; v10 -= b[i10]; v11 -= b[idx]; }
    const float cA = h * (((v00 + v01) + v10) + v11);
    const float cH = h * ((v10 + v11) - (v00 + v01));
    const float cV = h * ((v01 + v11) - (v00 + v10));
    const float cD = h * ((v00 + v11) - (v01 + v10));
    if (outA) outA[idx] = cA;
    if (sums) {
      fa[0] += fabsf(cA); fa[1] += fabsf(cH); fa[2] += fabsf(cV); fa[3] += fabsf(cD);
      if (++cnt == 32) {
#pragma unroll
        for (int k = 0; k < 4; ++k) { acc[k] += fa[k]; fa[k] = 0.f; }
        cnt = 0;
      }
    }
    if (G) {
      const float gA = gscale * 0.5f * sgn(cA) + (gA_in ? gA_in[idx] : 0.f);
      const float gH = gscale * 1.5f * sgn(cH), gV = gscale * 1.5f * sgn(cV), gD = gscale * 2.0f * sgn(cD);
      G[idx] = h * (gA - gH - gV + gD);
      G[total + idx] = h * (gA - gH + gV - gD);
      G[2 * total + idx] = h * (gA + gH - gV - gD);
      G[3 * total + idx] = h * (gA + gH + gV + gD);
    }
  }
  if (sums) {
#pragma unroll
    for (int k = 0; k < 4; ++k) acc[k] += fa[k];
    block_sum_slot<4>(acc, sums);
  }
}

// adjoint of the level operator: dcur[u][v] = sum over the outputs that read cur[u][v]
__global__ void __launch_bounds__(256) k_swt_gather(const float* __restrict__ G, long total, int H, int W, int d,
                                                    float* __restrict__ out, int accumulate) {
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    const int v = (int)(idx % W);
    const int u = (int)((idx / W) % H);
    const long base = idx - ((long)u * W + v);
    int ys[2], xs[2], ny = 0, nx = 0;
    if (u + d < H) ys[ny++] = u + d;
    if (u >= 1 && u <= d && d - u < H) ys[ny++] = d - u;
    if (v + d < W) xs[nx++] = v + d;
    if (v >= 1 && v <= d && d - v < W) xs[nx++] = d - v;
    float s = G[3 * total + idx];
    for (int i = 0; i < ny; ++i) {
      s += G[total + base + (long)ys[i] * W + v];
      for (int j = 0; j < nx; ++j) s += G[base + (long)ys[i] * W + xs[j]];
    }
    for (int j = 0; j < nx; ++j) s += G[2 * total + base + (long)u * W + xs[j]];
    out[idx] = accumulate ? out[idx] + s : s;
  }
}

// ------------------------------------------------------------------------------------ SSIM
constexpr int ST = 32, SR = 5, SP = ST + 2 * SR;
struct Gauss11 { float g[11]; };

__global__ void __launch_bounds__(256) k_ssim_fwd(const float* __restrict__ X, const float* __restrict__ Y, int H, int W,
                                                  Gauss11 gw, float gs, double* __restrict__ sum,
                                                  float* __restrict__ D, long total) {
  __shared__ float sx[SP][SP + 1], sy[SP][SP + 1];
  __shared__ float hq[5][SP][ST + 1];
  const int tid = threadIdx.x;
  const int ty0 = blockIdx.y * ST, tx0 = blockIdx.x * ST;
  const long base = (long)blockIdx.z * H * W;
  for (int i = tid; i < SP * SP; i += 256) {
    const int r = i / SP, c = i % SP;
    const int y = ty0 + r - SR, x = tx0 + c - SR;
    const bool in = (y >= 0 && y < H && x >= 0 && x < W);
    sx[r][c] = in ? X[base + (long)y * W + x] : 0.f;
    sy[r][c] = in ? Y[base + (long)y * W + x] : 0.f;
  }
  __syncthreads();
  for (int i = tid; i < SP * ST; i += 256) {
    const int r = i / ST, c = i % ST;
    float m1 = 0.f, m2 = 0.f, xx = 0.f, yy = 0.f, xy = 0.f;
#pragma unroll
    for (int k = 0; k < 11; ++k) {
      const float a = sx[r][c + k], b = sy[r][c + k], g = gw.g[k];
      m1 = fmaf(g, a, m1); m2 = fmaf(g, b, m2);
      xx = fmaf(g, a * a, xx); yy = fmaf(g, b * b, yy); xy = fmaf(g, a * b, xy);
    }
    hq[0][r][c] = m1; hq[1][r][c] = m2; hq[2][r][c] = xx; hq[3][r][c] = yy; hq[4][r][c] = xy;
  }
  __syncthreads();
  double acc[1] = {0.0};
  float f = 0.f;
  for (int i = tid; i < ST * ST; i += 256) {
    const int r = i / ST, c = i % ST;
    const int y = ty0 + r, x = tx0 + c;
    if (y >= H || x >= W) continue;
    float q[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int k = 0; k < 11; ++k) {
      const float g = gw.g[k];
#pragma unroll
      for (int j = 0; j < 5; ++j) q[j] = fmaf(g, hq[j][r + k][c], q[j]);
    }
    const float C1 = 1e-4f, C2 = 9e-4f;
    const float m1 = q[0], m2 = q[1];
    const float m11 = m1 * m1, m22 = m2 * m2, m12 = m1 * m2;
    const float s1 = q[2] - m11, s2 = q[3] - m22, s12 = q[4] - m12;
    const float A1 = 2.f * m12 + C1, A2 = 2.f * s12 + C2, B1 = m11 + m22 + C1, B2 = s1 + s2 + C2;
    const float inv = 1.0f / (B1 * B2);
    const float S = A1 * A2 * inv;
    f += S;
    const long o = base + (long)y * W + x;
    D[o] = gs * (2.f * m2 * (A2 - A1) * inv - S * 2.f * m1 * (B2 - B1) * inv);
    D[total + o] = gs * (-S / B2);
    D[2 * total + o] = gs * (2.f * A1 * inv);
  }
  acc[0] = f;
  block_sum_slot<1>(acc, sum);
}

__global__ void __launch_bounds__(256) k_ssim_bwd(const float* __restrict__ X, const float* __restrict__ Y, int H, int W,
                                                  Gauss11 gw, const float* __restrict__ D, long total,
                                                  float* __restrict__ dpred) {
  __shared__ float sd[3][SP][SP + 1];
  __shared__ float hq[3][SP][ST + 1];
  const int tid = threadIdx.x;
  const int ty0 = blockIdx.y * ST, tx0 = blockIdx.x * ST;
  const long base = (long)blockIdx.z * H * W;
  for (int i = tid; i < SP * SP; i += 256) {
    const int r = i / SP, c = i % SP;
    const int y = ty0 + r - SR, x = tx0 + c - SR;
    const bool in = (y >= 0 && y < H && x >= 0 && x < W);
    const long o = base + (long)y * W + x;
    sd[0][r][c] = in ? D[o] : 0.f;
    sd[1][r][c] = in ? D[total + o] : 0.f;
    sd[2][r][c] = in ? D[2 * total + o] : 0.f;
  }
  __syncthreads();
  for (int i = tid; i < SP * ST; i += 256) {
    const int r = i / ST, c = i % ST;
    float q0 = 0.f, q1 = 0.f, q2 = 0.f;
#pragma unroll
    for (int k = 0; k < 11; ++k) {
      const float g = gw.g[k];
      q0 = fmaf(g, sd[0][r][c + k], q0); q1 = fmaf(g, sd[1][r][c + k], q1); q2 = fmaf(g, sd[2][r][c + k], q2);
    }
    hq[0][r][c] = q0; hq[1][r][c] = q1; hq[2][r][c] = q2;
  }
  __syncthreads();
  for (int i = tid; i < ST * ST; i += 256) {
    const int r = i / ST, c = i % ST;
    const int y = ty0 + r, x = tx0 + c;
    if (y >= H || x >= W) continue;
    float q0 = 0.f, q1 = 0.f, q2 = 0.f;
#pragma unroll
    for (int k = 0; k < 11; ++k) {
      const float g = gw.g[k];
      q0 = fmaf(g, hq[0][r + k][c], q0); q1 = fmaf(g, hq[1][r + k][c], q1); q2 = fmaf(g, hq[2][r + k][c], q2);
    }
    const long o = base + (long)y * W + x;
    dpred[o] += q0 + 2.f * X[o] * q1 + Y[o] * q2;
  }
}

// ------------------------------------------------------------------------------------ FFT
struct Radices { int n; int r[12]; };

__device__ __forceinline__ float2 cmul(float2 a, float2 b) { return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }

template <int R>
__device__ __forceinline__ void dft_small(float2 (&v)[R], float dir) {
  if constexpr (R == 2) {
    const float2 a = v[0], b = v[1];
    v[0] = make_float2(a.x + b.x, a.y + b.y);
    v[1] = make_float2(a.x - b.x, a.y - b.y);
  } else if constexpr (R == 4) {
    const float2 a = v[0], b = v[1], c = v[2], d = v[3];
    const float2 s0 = make_float2(a.x + c.x, a.y + c.y), s1 = make_float2(a.x - c.x, a.y - c.y);
    const float2 s2 = make_float2(b.x + d.x, b.y + d.y), s3 = make_float2(b.x - d.x, b.y - d.y);
    // forward (dir = -1) multiplies s3 by -i, the inverse by +i:
    // -i * (x + iy) = y - ix ; +i * (x + iy) = -y + ix  ->  (-dir*y, dir*x)
    const float2 r3 = make_float2(-dir * s3.y, dir * s3.x);
    v[0] = make_float2(s0.x + s2.x, s0.y + s2.y);
    v[2] = make_float2(s0.x - s2.x, s0.y - s2.y);
    v[1] = make_float2(s1.x + r3.x, s1.y + r3.y);
    v[3] = make_float2(s1.x - r3.x, s1.y - r3.y);
  } else {
    float2 o[R];
#pragma unroll
    for (int k = 0; k < R; ++k) {
      float2 acc = v[0];
#pragma unroll
      for (int q = 1; q < R; ++q) {
        float sn, cs;
        sincospif(dir * 2.0f * (float)((q * k) % R) / (float)R, &sn, &cs);
        acc.x += v[q].x * cs - v[q].y * sn;
        acc.y += v[q].x * sn + v[q].y * cs;
      }
      o[k] = acc;
    }
#pragma unroll
    for (int k = 0; k < R; ++k) v[k] = o[k];
  }
}

// one Stockham pass of radix R over L independent length-N sequences stored back to back
template <int R>
__device__ __forceinline__ void fft_pass(const float2* __restrict__ src, float2* __restrict__ dst, int N, int Ns, int L,
                                         float dir) {
  const int nb = N / R;
  for (int w = threadIdx.x; w < L * nb; w += blockDim.x) {
    const int seq = w / nb, j = w % nb;
    const int k = j % Ns;
    const float2* s = src + seq * N;
    float2* o = dst + seq * N;
    float2 v[R];
#pragma unroll
    for (int q = 0; q < R; ++q) {
      v[q] = s[j + q * nb];
      if (q > 0 && Ns > 1) {
        float sn, cs;
        sincospif(dir * 2.0f * (float)((q * k) % (Ns * R)) / (float)(Ns * R), &sn, &cs);
        v[q] = cmul(v[q], make_float2(cs, sn));
      }
    }
    dft_small<R>(v, dir);
    const int j0 = (j / Ns) * Ns * R + k;
#pragma unroll
    for (int q = 0; q < R; ++q) o[j0 + q * Ns] = v[q];
  }
}

// transforms L sequences of length N held in bufA (scratch bufB); returns the buffer holding the result
__device__ float2* fft_smem(float2* bufA, float2* bufB, int N, int L, const Radices& rad, float dir) {
  int Ns = 1;
  float2 *src = bufA, *dst = bufB;
  for (int p = 0; p < rad.n; ++p) {
    const int R = rad.r[p];
    switch (R) {
      case 2: fft_pass<2>(src, dst, N, Ns, L, dir); break;
      case 3: fft_pass<3>(src, dst, N, Ns, L, dir); break;
      case 4: fft_pass<4>(src, dst, N, Ns, L, dir); break;
      case 5: fft_pass<5>(src, dst, N, Ns, L, dir); break;
      default: fft_pass<7>(src, dst, N, Ns, L, dir); break;
    }
    __syncthreads();
    Ns *= R;
    float2* t = src; src = dst; dst = t;
  }
  return src;
}

constexpr int FFT_ROWS = 4;   // rows per block (row pass), columns per block (column pass)

// rows: MODE 0: in = (re: a, im: b) real planes -> Z ; MODE 1: in = Z (complex) -> dpred += Re(out)
template <int MODE>
__global__ void __launch_bounds__(256) k_fft_rows(const float* __restrict__ a, const float* __restrict__ b,
                                                  float2* __restrict__ Z, long nrows, int W, Radices rad, float scale,
                                                  float* __restrict__ dpred) {
  extern __shared__ float2 fsm[];
  float2* A = fsm;
  float2* Bf = fsm + FFT_ROWS * W;
  const long row0 = (long)blockIdx.x * FFT_ROWS;
  const int L = (int)min((long)FFT_ROWS, nrows - row0);
  for (int i = threadIdx.x; i < L * W; i += blockDim.x) {
    const long g = row0 * W + i;
    A[i] = MODE == 0 ? make_float2(a[g], b[g]) : Z[g];
  }
  __syncthreads();
  float2* res = fft_smem(A, Bf, W, L, rad, MODE == 0 ? -1.f : 1.f);
  for (int i = threadIdx.x; i < L * W; i += blockDim.x) {
    const long g = row0 * W + i;
    if (MODE == 0) Z[g] = make_float2(res[i].x * scale, res[i].y * scale);
    else dpred[g] += res[i].x * scale;
  }
}

// columns, in place on Z [P][H][W]: block = (plane, strip of FFT_ROWS columns)
__global__ void __launch_bounds__(256) k_fft_cols(float2* __restrict__ Z, int H, int W, Radices rad, float dir,
                                                  float scale) {
  extern __shared__ float2 fsm[];
  float2* A = fsm;
  float2* Bf = fsm + FFT_ROWS * H;
  const int c0 = blockIdx.x * FFT_ROWS;
  const int L = min(FFT_ROWS, W - c0);
  float2* base = Z + (long)blockIdx.y * H * W;
  for (int i = threadIdx.x; i < H * FFT_ROWS; i += blockDim.x) {
    const int y = i / FFT_ROWS, c = i % FFT_ROWS;
    if (c < L) A[c * H + y] = base[(long)y * W + c0 + c];
  }
  __syncthreads();
  float2* res = fft_smem(A, Bf, H, L, rad, dir);
  for (int i = threadIdx.x; i < H * FFT_ROWS; i += blockDim.x) {
    const int y = i / FFT_ROWS, c = i % FFT_ROWS;
    if (c < L) base[(long)y * W + c0 + c] = make_float2(res[c * H + y].x * scale, res[c * H + y].y * scale);
  }
}

// spectrum loss: Z = F(pred) + i F(target).  P = (Z[k] + conj Z[-k])/2, T = (Z[k] - conj Z[-k])/(2i)
__global__ void __launch_bounds__(256) k_fft_spectrum(const float2* __restrict__ Z, long total, int H, int W,
                                                      float gscale, double* __restrict__ sums,
                                                      float2* __restrict__ G) {
  double acc[2] = {0.0, 0.0};
  float fm = 0.f, fp = 0.f;
  int cnt = 0;
  const int cy = H / 2, cx = W / 2;
  const float inv_max = rsqrtf((float)(cy * cy + cx * cx));
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    const int kx = (int)(idx % W);
    const int ky = (int)((idx / W) % H);
    const long base = idx - ((long)ky * W + kx);
    const int my = ky == 0 ? 0 : H - ky, mx = kx == 0 ? 0 : W - kx;
    const float2 z = Z[idx], zm = Z[base + (long)my * W + mx];
    const float pa = 0.5f * (z.x + zm.x), pb = 0.5f * (z.y - zm.y);       // P = (Z + conj Zm)/2
    const float ta = 0.5f * (z.y + zm.y), tb = 0.5f * (zm.x - z.x);       // T = (Z - conj Zm)/(2i); +0 (not -0) on
                                                                          // self-conjugate bins: angle(-|t|) = +pi like P's
    // fftshift puts frequency k at index (k + n/2) mod n; the weight is radial around (n/2, n/2)
    const int sy = (ky + cy) % H - cy, sx = (kx + cx) % W - cx;
    const float wgt = 1.0f + sqrtf((float)(sx * sx + sy * sy)) * inv_max;
    const float pm2 = pa * pa + pb * pb, tm2 = ta * ta + tb * tb;
    const float pm = sqrtf(pm2), tm = sqrtf(tm2);
    const float pang = atan2f(pb, pa), tang = atan2f(tb, ta);
    const float dm = pm - tm, dph = pang - tang;
    fm += wgt * fabsf(dm);
    fp += wgt * fabsf(dph);
    if (++cnt == 32) { acc[0] += fm; acc[1] += fp; fm = 0.f; fp = 0.f; cnt = 0; }
    float ga = 0.f, gb = 0.f;
    if (pm2 > 0.f) {
      const float c1 = gscale * wgt * sgn(dm) / pm;
      const float c2 = gscale * wgt * 0.1f * sgn(dph) / pm2;
      ga = c1 * pa - c2 * pb;
      gb = c1 * pb + c2 * pa;
    }
    G[idx] = make_float2(ga, gb);
  }
  acc[0] += fm; acc[1] += fp;
  block_sum_slot<2>(acc, sums);
}

bool factorize(int n, Radices& rad) {
  rad.n = 0;
  while (n % 4 == 0 && rad.n < 12) { rad.r[rad.n++] = 4; n /= 4; }
  const int primes[4] = {2, 3, 5, 7};
  for (int i = 0; i < 4; ++i)
    while (n % primes[i] == 0 && rad.n < 12) { rad.r[rad.n++] = primes[i]; n /= primes[i]; }
  return n == 1;
}

inline int ew_grid(long n) { return (int)((n + 255) / 256 < 148L * 16 ? (n + 255) / 256 : 148L * 16); }

// the partial-sum slots follow the entry point's own scratch in the workspace
constexpr size_t LOSS_PART_ALIGN = 256;
inline size_t part_offset(size_t scratch) { return (scratch + LOSS_PART_ALIGN - 1) / LOSS_PART_ALIGN * LOSS_PART_ALIGN; }
inline double* part_ptr(void* ws, size_t scratch) { return (double*)((char*)ws + part_offset(scratch)); }
inline long ssim_blocks(int P, int H, int W) { return (long)ceil_div(W, ST) * ceil_div(H, ST) * P; }
}  // namespace

extern "C" size_t ffsr_loss_l1_workspace_bytes(long n) { return n > 0 ? (size_t)ew_grid(n) * sizeof(double) : 0; }

extern "C" int ffsr_loss_l1(const float* pred, const float* target, long n, float gscale, double* sum, void* ws,
                            size_t ws_bytes, float* dpred, cudaStream_t stream) {
  FFSR_REQUIRE(pred && target && sum && ws && dpred && n > 0, FFSR_ERR_ARG, "loss_l1: bad argument");
  FFSR_REQUIRE(ws_bytes >= ffsr_loss_l1_workspace_bytes(n), FFSR_ERR_ARG, "loss_l1: workspace too small");
  const int grid = ew_grid(n);
  k_loss_l1<<<grid, 256, 0, stream>>>(pred, target, n, gscale, (double*)ws, dpred);
  const int rc = ffsr_check_launch("loss_l1");
  if (rc) return rc;
  launch_sum_slots<double>((const double*)ws, grid, 1, sum, stream);
  return ffsr_check_launch("loss_l1_reduce");
}

extern "C" size_t ffsr_loss_swt_workspace_bytes(int P, int H, int W) {
  const long total = (long)P * H * W;
  return part_offset((size_t)6 * total * sizeof(float)) + (size_t)ew_grid(total) * 4 * sizeof(double);
}

extern "C" int ffsr_loss_swt(const float* pred, const float* target, int P, int H, int W, float gscale, double* sums8,
                             void* ws, size_t ws_bytes, float* dpred, cudaStream_t stream) {
  FFSR_REQUIRE(pred && target && sums8 && ws && dpred && P > 0, FFSR_ERR_ARG, "loss_swt: bad argument");
  FFSR_REQUIRE(H >= 3 && W >= 3, FFSR_ERR_ARG, "loss_swt: H, W must be >= 3 (reflect pad 2 at level 1)");
  FFSR_REQUIRE(ws_bytes >= ffsr_loss_swt_workspace_bytes(P, H, W), FFSR_ERR_ARG, "loss_swt: workspace too small");
  const long total = (long)P * H * W;
  float* A0 = (float*)ws;
  float* gA0 = A0 + total;
  float* G = gA0 + total;
  const int grid = ew_grid(total);
  double* part = part_ptr(ws, (size_t)6 * total * sizeof(float));
  // level 0: approximation + sums;  level 1: sums + tap gradients;  adjoint to dA0;  level 0 again with dA0;  adjoint
  k_swt_level<<<grid, 256, 0, stream>>>(pred, target, total, H, W, 1, A0, nullptr, gscale, part, nullptr);
  launch_sum_slots<double>(part, grid, 4, sums8, stream);
  k_swt_level<<<grid, 256, 0, stream>>>(A0, nullptr, total, H, W, 2, nullptr, nullptr, gscale, part, G);
  launch_sum_slots<double>(part, grid, 4, sums8 + 4, stream);
  k_swt_gather<<<grid, 256, 0, stream>>>(G, total, H, W, 2, gA0, 0);
  k_swt_level<<<grid, 256, 0, stream>>>(pred, target, total, H, W, 1, nullptr, gA0, gscale, nullptr, G);
  k_swt_gather<<<grid, 256, 0, stream>>>(G, total, H, W, 1, dpred, 1);
  return ffsr_check_launch("loss_swt");
}

extern "C" size_t ffsr_loss_ssim_workspace_bytes(int P, int H, int W) {
  return part_offset((size_t)3 * P * H * W * sizeof(float)) + (size_t)ssim_blocks(P, H, W) * sizeof(double);
}

extern "C" int ffsr_loss_ssim(const float* pred, const float* target, int P, int H, int W, float gscale, double* sum,
                              void* ws, size_t ws_bytes, float* dpred, cudaStream_t stream) {
  FFSR_REQUIRE(pred && target && sum && ws && dpred && P > 0 && P <= 65535 && H > 0 && W > 0, FFSR_ERR_ARG, "loss_ssim: bad argument");
  FFSR_REQUIRE(ws_bytes >= ffsr_loss_ssim_workspace_bytes(P, H, W), FFSR_ERR_ARG, "loss_ssim: workspace too small");
  Gauss11 gw;
  float s = 0.f;
  for (int i = 0; i < 11; ++i) { gw.g[i] = (float)exp(-(double)((i - 5) * (i - 5)) / (2.0 * 1.5 * 1.5)); s += gw.g[i]; }
  for (int i = 0; i < 11; ++i) gw.g[i] /= s;
  const long total = (long)P * H * W;
  dim3 grid(ceil_div(W, ST), ceil_div(H, ST), P);
  // loss = 1 - mean(S): dLoss/dS = -1/n, the caller's gscale carries weight/n
  double* part = part_ptr(ws, (size_t)3 * total * sizeof(float));
  k_ssim_fwd<<<grid, 256, 0, stream>>>(pred, target, H, W, gw, -gscale, part, (float*)ws, total);
  launch_sum_slots<double>(part, (int)ssim_blocks(P, H, W), 1, sum, stream);
  k_ssim_bwd<<<grid, 256, 0, stream>>>(pred, target, H, W, gw, (const float*)ws, total, dpred);
  return ffsr_check_launch("loss_ssim");
}

extern "C" size_t ffsr_loss_fft_workspace_bytes(int P, int H, int W) {
  const long total = (long)P * H * W;
  return part_offset((size_t)2 * total * sizeof(float2)) + (size_t)ew_grid(total) * 2 * sizeof(double);
}

extern "C" int ffsr_loss_fft(const float* pred, const float* target, int P, int H, int W, float gscale, double* sums2,
                             void* ws, size_t ws_bytes, float* dpred, cudaStream_t stream) {
  FFSR_REQUIRE(pred && target && sums2 && ws && dpred && P > 0 && P <= 65535, FFSR_ERR_ARG, "loss_fft: bad argument");
  FFSR_REQUIRE(ws_bytes >= ffsr_loss_fft_workspace_bytes(P, H, W), FFSR_ERR_ARG, "loss_fft: workspace too small");
  Radices rh, rw;
  FFSR_REQUIRE(factorize(H, rh) && factorize(W, rw), FFSR_ERR_ARG,
               "loss_fft: H and W must factor into 2, 3, 5, 7 (got %dx%d)", H, W);
  FFSR_REQUIRE(H <= 4096 && W <= 4096, FFSR_ERR_ARG, "loss_fft: H, W must be <= 4096");
  const long total = (long)P * H * W;
  float2* Z = (float2*)ws;
  float2* G = Z + total;
  const size_t sm_rows = (size_t)2 * FFT_ROWS * W * sizeof(float2), sm_cols = (size_t)2 * FFT_ROWS * H * sizeof(float2);
  static size_t attr_rows = 0, attr_cols = 0;     // raise the opt-in shared-memory limit only when it has to grow
  if (sm_rows > attr_rows) {
    cudaFuncSetAttribute(k_fft_rows<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_rows);
    cudaFuncSetAttribute(k_fft_rows<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_rows);
    attr_rows = sm_rows;
  }
  if (sm_cols > attr_cols) {
    cudaFuncSetAttribute(k_fft_cols, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_cols);
    attr_cols = sm_cols;
  }
  const long nrows = (long)P * H;
  const float sc_w = 1.0f / sqrtf((float)W), sc_h = 1.0f / sqrtf((float)H);
  k_fft_rows<0><<<(unsigned)ceil_div(nrows, FFT_ROWS), 256, sm_rows, stream>>>(pred, target, Z, nrows, W, rw, sc_w, nullptr);
  dim3 cgrid(ceil_div(W, FFT_ROWS), P);
  k_fft_cols<<<cgrid, 256, sm_cols, stream>>>(Z, H, W, rh, -1.f, sc_h);
  double* part = part_ptr(ws, (size_t)2 * total * sizeof(float2));
  k_fft_spectrum<<<ew_grid(total), 256, 0, stream>>>(Z, total, H, W, gscale, part, G);
  launch_sum_slots<double>(part, ew_grid(total), 2, sums2, stream);
  k_fft_cols<<<cgrid, 256, sm_cols, stream>>>(G, H, W, rh, 1.f, sc_h);
  k_fft_rows<1><<<(unsigned)ceil_div(nrows, FFT_ROWS), 256, sm_rows, stream>>>(nullptr, nullptr, G, nrows, W, rw, sc_w, dpred);
  return ffsr_check_launch("loss_fft");
}
