// Phase 2: 9 sub-band decomposition of the LR image (DCT x3, db4 DWT x4, FFT x2).
// Replaces DCTDecomposition/DWTDecomposition/FFTDecomposition.forward
// (src/models/multi_domain_frequency.py:146-196, 251-299, 352-385).
// Output layout: raw9[B][9][3][H][W] fp32 (band-major planar), so raw9[:, i] is the
// reference's i-th [B,3,H,W] band.  HBM-bound, tiny next to the HR phases.
#include "common.cuh"
#include "../../include/ffsr_b200.h"

// ------------------------------------------------------------------------------------
// DCT: one 8x8 block of one channel per 64-thread CTA.
// ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(64) k_dct_bands(
    const float* __restrict__ x, int H, int W,
    const float* __restrict__ D, const float* __restrict__ Dt,
    const float* __restrict__ m_low, const float* __restrict__ m_mid, const float* __restrict__ m_high,
    const float* __restrict__ band_scale, float* __restrict__ raw9, int B) {
  __shared__ float sD[64], sDt[64], sX[64], sT[64], sY[64], sZ[64], sU[64];
  const int t = threadIdx.x, i = t >> 3, j = t & 7;
  const int bc = blockIdx.z, b = bc / 3, c = bc % 3;
  const int y = blockIdx.y * 8 + i, xx = blockIdx.x * 8 + j;
  sD[t] = D[t];
  sDt[t] = Dt[t];
  // bottom/right reflect pad to a multiple of 8 (:159-164)
  sX[t] = x[((long)bc * H + reflect_idx(y, H)) * W + reflect_idx(xx, W)];
  __syncthreads();
  float acc = 0.f;
#pragma unroll
  for (int k = 0; k < 8; ++k) acc = fmaf(sX[i * 8 + k], sDt[k * 8 + j], acc);   // T = X Dt
  sT[t] = acc;
  __syncthreads();
  acc = 0.f;
#pragma unroll
  for (int k = 0; k < 8; ++k) acc = fmaf(sD[i * 8 + k], sT[k * 8 + j], acc);    // Y = D T
  sY[t] = acc;
  const float* masks[3] = {m_low, m_mid, m_high};
  const bool inside = (y < H) && (xx < W);
#pragma unroll
  for (int band = 0; band < 3; ++band) {
    __syncthreads();
    sZ[t] = sY[t] * masks[band][t];
    __syncthreads();
    acc = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) acc = fmaf(sZ[i * 8 + k], sD[k * 8 + j], acc);  // U = Z D
    sU[t] = acc;
    __syncthreads();
    acc = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) acc = fmaf(sDt[i * 8 + k], sU[k * 8 + j], acc); // V = Dt U
    if (inside) raw9[(((long)b * 9 + band) * 3 + c) * H * W + (long)y * W + xx] = acc * band_scale[band];
  }
}

extern "C" int ffsr_dct_bands(const float* lr, int B, int H, int W, const float* basis, const float* basis_t,
                              const float* m_low, const float* m_mid, const float* m_high,
                              const float* band_scale, float* raw9, cudaStream_t stream) {
  FFSR_REQUIRE(lr && raw9 && basis && basis_t && m_low && m_mid && m_high && band_scale, FFSR_ERR_ARG, "dct_bands: null pointer");
  FFSR_REQUIRE(B > 0 && H >= 8 && W >= 8, FFSR_ERR_ARG, "dct_bands: need B>0 and H,W>=8 (got %d,%d,%d)", B, H, W);
  dim3 grid(ceil_div(W, 8), ceil_div(H, 8), B * 3);
  k_dct_bands<<<grid, 64, 0, stream>>>(lr, H, W, basis, basis_t, m_low, m_mid, m_high, band_scale, raw9, B);
  return ffsr_check_launch("dct_bands");
}

// ------------------------------------------------------------------------------------
// DWT: (1) db4 analysis at stride 2 with 7-px reflect pad -> sub[B][4][3][Hs][Ws];
//      (2) bilinear back to HxW, times subband_scale -> raw9 bands 3..6.
// ------------------------------------------------------------------------------------
__global__ void k_dwt_analysis(const float* __restrict__ x, int H, int W, int Hs, int Ws,
                               const float* __restrict__ lo_row, const float* __restrict__ hi_row,
                               const float* __restrict__ lo_col, const float* __restrict__ hi_col,
                               float* __restrict__ sub, int B) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  const int i = blockIdx.y;
  const int bc = blockIdx.z, b = bc / 3, c = bc % 3;
  if (j >= Ws) return;
  float lr_[8], hr_[8], lc_[8], hc_[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    lr_[k] = lo_row[k]; hr_[k] = hi_row[k]; lc_[k] = lo_col[k]; hc_[k] = hi_col[k];
  }
  const float* img = x + (long)bc * H * W;
  float LL = 0.f, LH = 0.f, HL = 0.f, HH = 0.f;
#pragma unroll
  for (int u = 0; u < 8; ++u) {
    const int r = reflect_idx(2 * i + u - 7, H);
    float rl = 0.f, rh = 0.f;
#pragma unroll
    for (int v = 0; v < 8; ++v) {
      const float val = img[(long)r * W + reflect_idx(2 * j + v - 7, W)];
      rl = fmaf(lr_[v], val, rl);
      rh = fmaf(hr_[v], val, rh);
    }
    LL = fmaf(lc_[u], rl, LL);   // lo_col on lo_rows
    LH = fmaf(hc_[u], rl, LH);   // hi_col on lo_rows
    HL = fmaf(lc_[u], rh, HL);   // lo_col on hi_rows
    HH = fmaf(hc_[u], rh, HH);   // hi_col on hi_rows
  }
  const long plane = (long)Hs * Ws;
  const long o = (long)i * Ws + j;
  sub[(((long)b * 4 + 0) * 3 + c) * plane + o] = LL;
  sub[(((long)b * 4 + 1) * 3 + c) * plane + o] = LH;
  sub[(((long)b * 4 + 2) * 3 + c) * plane + o] = HL;
  sub[(((long)b * 4 + 3) * 3 + c) * plane + o] = HH;
}

__global__ void k_dwt_resize(const float* __restrict__ sub, int Hs, int Ws, int H, int W,
                             const float* __restrict__ subband_scale, float* __restrict__ raw9, int B) {
  const int xx = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y;
  const int z = blockIdx.z;   // (b*4 + s)*3 + c
  if (xx >= W) return;
  const int c = z % 3, s = (z / 3) % 4, b = z / 12;
  const BilinTap ty = bilin_tap(y, Hs, H), tx = bilin_tap(xx, Ws, W);
  const float* p = sub + (long)z * Hs * Ws;
  const float top = tx.w0 * p[(long)ty.i0 * Ws + tx.i0] + tx.w1 * p[(long)ty.i0 * Ws + tx.i1];
  const float bot = tx.w0 * p[(long)ty.i1 * Ws + tx.i0] + tx.w1 * p[(long)ty.i1 * Ws + tx.i1];
  raw9[(((long)b * 9 + 3 + s) * 3 + c) * H * W + (long)y * W + xx] = (ty.w0 * top + ty.w1 * bot) * subband_scale[s];
}

extern "C" int ffsr_dwt_sub_size(int H, int W, int* Hs, int* Ws) {
  // conv output of the 7+7 padded axis with an 8-tap stride-2 filter
  *Hs = (H + 14 - 8) / 2 + 1;
  *Ws = (W + 14 - 8) / 2 + 1;
  return FFSR_OK;
}

extern "C" int ffsr_dwt_bands(const float* lr, int B, int H, int W, const float* lo_row, const float* hi_row,
                              const float* lo_col, const float* hi_col, const float* subband_scale,
                              float* sub_ws, float* raw9, cudaStream_t stream) {
  FFSR_REQUIRE(lr && raw9 && sub_ws && lo_row && hi_row && lo_col && hi_col && subband_scale, FFSR_ERR_ARG, "dwt_bands: null pointer");
  FFSR_REQUIRE(B > 0 && H >= 8 && W >= 8, FFSR_ERR_ARG, "dwt_bands: need H,W>=8 (reflect pad 7)");
  int Hs, Ws;
  ffsr_dwt_sub_size(H, W, &Hs, &Ws);
  dim3 g1(ceil_div(Ws, 128), Hs, B * 3);
  k_dwt_analysis<<<g1, 128, 0, stream>>>(lr, H, W, Hs, Ws, lo_row, hi_row, lo_col, hi_col, sub_ws, B);
  int rc = ffsr_check_launch("dwt_analysis");
  if (rc) return rc;
  dim3 g2(ceil_div(W, 128), H, B * 12);
  k_dwt_resize<<<g2, 128, 0, stream>>>(sub_ws, Hs, Ws, H, W, subband_scale, raw9, B);
  return ffsr_check_launch("dwt_resize");
}

// ------------------------------------------------------------------------------------
// Adjoints of the unit-scale DCT and DWT bands: the input gradient of Phase 2.  Gathers only: every output element
// is written by one thread that sums its sources in a fixed order (no atomics), so the gradient is bitwise
// reproducible like every training kernel.
// ------------------------------------------------------------------------------------
// Per 8x8 block of the padded grid: P = Dt (sum_b M_b .* (D G_b Dt)) D, with G_b the band gradient zero-extended to the
// padded grid.  X -> Dt (M .* (D X Dt)) D is its own adjoint for any D (the adjoint of X -> D X Dt is G -> Dt G D), so
// this is exact even though the fp32 basis is not exactly orthogonal.
__global__ void __launch_bounds__(64) k_dct_adjoint_blocks(
    const float* __restrict__ g3, int H, int W, int Hp, int Wp,
    const float* __restrict__ D, const float* __restrict__ Dt,
    const float* __restrict__ m_low, const float* __restrict__ m_mid, const float* __restrict__ m_high,
    float* __restrict__ pad) {
  __shared__ float sD[64], sDt[64], sG[64], sT[64];
  const int t = threadIdx.x, i = t >> 3, j = t & 7;
  const int bc = blockIdx.z, b = bc / 3, c = bc % 3;
  const int y = blockIdx.y * 8 + i, xx = blockIdx.x * 8 + j;
  sD[t] = D[t];
  sDt[t] = Dt[t];
  const bool inside = (y < H) && (xx < W);
  const float* masks[3] = {m_low, m_mid, m_high};
  float z = 0.f, acc;
#pragma unroll
  for (int band = 0; band < 3; ++band) {
    __syncthreads();
    sG[t] = inside ? g3[(((long)b * 3 + band) * 3 + c) * H * W + (long)y * W + xx] : 0.f;
    __syncthreads();
    acc = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) acc = fmaf(sG[i * 8 + k], sDt[k * 8 + j], acc);   // G Dt
    sT[t] = acc;
    __syncthreads();
    acc = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) acc = fmaf(sD[i * 8 + k], sT[k * 8 + j], acc);    // D G Dt
    z = fmaf(acc, masks[band][t], z);
  }
  __syncthreads();
  sG[t] = z;
  __syncthreads();
  acc = 0.f;
#pragma unroll
  for (int k = 0; k < 8; ++k) acc = fmaf(sG[i * 8 + k], sD[k * 8 + j], acc);     // Z D
  sT[t] = acc;
  __syncthreads();
  acc = 0.f;
#pragma unroll
  for (int k = 0; k < 8; ++k) acc = fmaf(sDt[i * 8 + k], sT[k * 8 + j], acc);    // Dt Z D
  pad[((long)bc * Hp + y) * Wp + xx] = acc;
}

// fold of the bottom/right reflect pad: dx[y][x] = sum of P over the padded positions that read (y, x)
__global__ void k_dct_adjoint_fold(const float* __restrict__ pad, int H, int W, int Hp, int Wp, float* __restrict__ dx) {
  const int xx = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y, bc = blockIdx.z;
  if (xx >= W) return;
  const int my = 2 * H - 2 - y, mx = 2 * W - 2 - xx;        // the mirror of y (x) in the pad, if it lies there
  const bool ry = my >= H && my < Hp, rx = mx >= W && mx < Wp;
  const float* p = pad + (long)bc * Hp * Wp;
  float v = p[(long)y * Wp + xx];
  if (rx) v += p[(long)y * Wp + mx];
  if (ry) {
    v += p[(long)my * Wp + xx];
    if (rx) v += p[(long)my * Wp + mx];
  }
  dx[((long)bc * H + y) * W + xx] = v;
}

extern "C" int ffsr_dct_bands_adjoint(const float* g3, int B, int H, int W, const float* basis, const float* basis_t,
                                      const float* m_low, const float* m_mid, const float* m_high, float* pad_ws, float* dx,
                                      cudaStream_t stream) {
  FFSR_REQUIRE(g3 && dx && pad_ws && basis && basis_t && m_low && m_mid && m_high, FFSR_ERR_ARG, "dct_bands_adjoint: null pointer");
  FFSR_REQUIRE(B > 0 && H >= 8 && W >= 8, FFSR_ERR_ARG, "dct_bands_adjoint: need B>0 and H,W>=8 (got %d,%d,%d)", B, H, W);
  const int Hp = ceil_div(H, 8) * 8, Wp = ceil_div(W, 8) * 8;
  k_dct_adjoint_blocks<<<dim3(Wp / 8, Hp / 8, B * 3), 64, 0, stream>>>(g3, H, W, Hp, Wp, basis, basis_t, m_low, m_mid, m_high, pad_ws);
  const int rc = ffsr_check_launch("dct_adjoint_blocks");
  if (rc) return rc;
  k_dct_adjoint_fold<<<dim3(ceil_div(W, 128), H, B * 3), 128, 0, stream>>>(pad_ws, H, W, Hp, Wp, dx);
  return ffsr_check_launch("dct_adjoint_fold");
}

// padded positions p in [-7, pmax] of a 7+7 reflect-padded axis of length n that read element y (pad 7 < n: at most
// one mirror on each side)
__device__ __forceinline__ int dwt_sources(int y, int n, int pmax, int (&p)[3]) {
  int k = 0;
  p[k++] = y;
  if (y >= 1 && y <= 7) p[k++] = -y;
  const int q = 2 * n - 2 - y;
  if (q >= n && q <= pmax) p[k++] = q;
  return k;
}

// dx[y][x] += adjoint of k_dwt_analysis at (y, x): the transposed 8x1 stride-2 column filters (into the lo-row / hi-row
// intermediates at (y, j)) and the transposed 1x8 stride-2 row filters, each folding its reflect pad.  Input: the
// subband gradients sub[B][4][3][Hs][Ws] (LL, LH, HL, HH).
__global__ void k_dwt_analysis_adjoint(const float* __restrict__ sub, int H, int W, int Hs, int Ws,
                                       const float* __restrict__ lo_row, const float* __restrict__ hi_row,
                                       const float* __restrict__ lo_col, const float* __restrict__ hi_col,
                                       float* __restrict__ dx) {
  const int xx = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y;
  const int bc = blockIdx.z, b = bc / 3, c = bc % 3;
  if (xx >= W) return;
  float lr_[8], hr_[8], lc_[8], hc_[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    lr_[k] = lo_row[k]; hr_[k] = hi_row[k]; lc_[k] = lo_col[k]; hc_[k] = hi_col[k];
  }
  const long plane = (long)Hs * Ws;
  const float* sLL = sub + (((long)b * 4 + 0) * 3 + c) * plane;
  const float* sLH = sub + (((long)b * 4 + 1) * 3 + c) * plane;
  const float* sHL = sub + (((long)b * 4 + 2) * 3 + c) * plane;
  const float* sHH = sub + (((long)b * 4 + 3) * 3 + c) * plane;
  int py[3], px[3];
  const int ny = dwt_sources(y, H, 2 * Hs - 2, py), nx = dwt_sources(xx, W, 2 * Ws - 2, px);
  float acc = 0.f;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    if (a >= nx) break;
#pragma unroll
    for (int v = 0; v < 8; ++v) {
      const int tj = px[a] + 7 - v;                  // p = 2 j + v - 7
      if (tj & 1) continue;
      const int j = tj >> 1;
      if (j < 0 || j >= Ws) continue;
      float tlo = 0.f, thi = 0.f;                    // gradients of the lo-row / hi-row intermediates at (y, j)
#pragma unroll
      for (int e = 0; e < 3; ++e) {
        if (e >= ny) break;
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int ti = py[e] + 7 - u;
          if (ti & 1) continue;
          const int i = ti >> 1;
          if (i < 0 || i >= Hs) continue;
          const long o = (long)i * Ws + j;
          tlo = fmaf(lc_[u], sLL[o], fmaf(hc_[u], sLH[o], tlo));
          thi = fmaf(lc_[u], sHL[o], fmaf(hc_[u], sHH[o], thi));
        }
      }
      acc = fmaf(lr_[v], tlo, fmaf(hr_[v], thi, acc));
    }
  }
  dx[((long)bc * H + y) * W + xx] += acc;
}

extern "C" int ffsr_dwt_bands_adjoint(const float* g4, int B, int H, int W, const float* lo_row, const float* hi_row,
                                      const float* lo_col, const float* hi_col, float* sub_ws, float* dx, cudaStream_t stream) {
  FFSR_REQUIRE(g4 && dx && sub_ws && lo_row && hi_row && lo_col && hi_col, FFSR_ERR_ARG, "dwt_bands_adjoint: null pointer");
  FFSR_REQUIRE(B > 0 && H >= 8 && W >= 8, FFSR_ERR_ARG, "dwt_bands_adjoint: need H,W>=8 (reflect pad 7)");
  int Hs, Ws;
  ffsr_dwt_sub_size(H, W, &Hs, &Ws);
  // bilinear (Hs,Ws) -> (H,W) adjoint of the B*12 planes: planar data is channels-last with one channel
  int rc = ffsr_bilinear_backward(g4, B * 12, H, W, 1, sub_ws, Hs, Ws, FFSR_DT_F32, stream);
  if (rc) return rc;
  k_dwt_analysis_adjoint<<<dim3(ceil_div(W, 128), H, B * 3), 128, 0, stream>>>(sub_ws, H, W, Hs, Ws, lo_row, hi_row, lo_col,
                                                                              hi_col, dx);
  return ffsr_check_launch("dwt_analysis_adjoint");
}

// ------------------------------------------------------------------------------------
// FFT bands.  Sizes are arbitrary (339x510 at full res), the transform is <0.1% of the
// forward's work, so it is evaluated as a dense DFT with exact table twiddles and fp64
// accumulation: four passes (rows R2C, cols C2C * mask, cols inverse, rows C2R).
// irfft2 semantics: imaginary parts of the DC and Nyquist columns are ignored
// (SURVEY Appendix A).  high = x - low (irfft2 is real-linear; SURVEY K3).
// ------------------------------------------------------------------------------------
__global__ void k_twiddles(int n, double2* out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double s, c;
  sincospi(2.0 * (double)i / (double)n, &s, &c);
  out[i] = make_double2(c, s);
}

extern "C" int ffsr_fft_twiddles(int n, void* out, cudaStream_t stream) {
  FFSR_REQUIRE(n > 0 && out, FFSR_ERR_ARG, "fft_twiddles: bad args");
  k_twiddles<<<ceil_div(n, 128), 128, 0, stream>>>(n, (double2*)out);
  return ffsr_check_launch("fft_twiddles");
}

__global__ void k_fft_mask(const float* __restrict__ logits, int ms, int H, int Wf,
                           const float* __restrict__ temperature, float* __restrict__ mask) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  const int l = blockIdx.y;
  if (k >= Wf) return;
  const BilinTap ty = bilin_tap(l, ms, H), tx = bilin_tap(k, ms, Wf);
  const float top = tx.w0 * logits[ty.i0 * ms + tx.i0] + tx.w1 * logits[ty.i0 * ms + tx.i1];
  const float bot = tx.w0 * logits[ty.i1 * ms + tx.i0] + tx.w1 * logits[ty.i1 * ms + tx.i1];
  const float T = fmaxf(temperature[0], 1.0f);
  mask[(long)l * Wf + k] = sigmoid_acc((ty.w0 * top + ty.w1 * bot) * T);
}

__global__ void __launch_bounds__(128) k_fft_rows_fwd(const float* __restrict__ x, int H, int W, int Wf,
                                                      const double2* __restrict__ tw, double2* __restrict__ A) {
  __shared__ float srow[256];
  __shared__ double2 stw[1024];               // twiddle table in shared memory (W <= 1024): the inner loop is
  const bool tw_s = W <= 1024;                // latency-bound on the table look-up, not on fp64 throughput
  if (tw_s)
    for (int t = threadIdx.x; t < W; t += blockDim.x) stw[t] = tw[t];
  const double2* __restrict__ twp = tw_s ? stw : tw;
  __syncthreads();
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y, bc = blockIdx.z;
  const float* row = x + ((long)bc * H + y) * W;
  double re = 0.0, im = 0.0;
  int idx = 0;
  for (int x0 = 0; x0 < W; x0 += 256) {
    const int n = min(256, W - x0);
    for (int t = threadIdx.x; t < n; t += blockDim.x) srow[t] = row[x0 + t];
    __syncthreads();
    if (k < Wf) {
      for (int t = 0; t < n; ++t) {
        const double v = (double)srow[t];
        const double2 w = twp[idx];
        re = fma(v, w.x, re);
        im = fma(-v, w.y, im);
        idx += k;
        if (idx >= W) idx -= W;
      }
    }
    __syncthreads();
  }
  if (k < Wf) A[((long)bc * H + y) * Wf + k] = make_double2(re, im);
}

// dir = -1: forward (then scaled and masked); dir = +1: inverse
template <int DIR>
__global__ void __launch_bounds__(256) k_fft_cols(const double2* __restrict__ A, int H, int Wf,
                                                  const double2* __restrict__ tw, const float* __restrict__ mask,
                                                  double scale, double2* __restrict__ Out) {
  __shared__ double2 stw[1024];
  const bool tw_s = H <= 1024;
  if (tw_s)
    for (int t = threadIdx.y * 32 + threadIdx.x; t < H; t += 256) stw[t] = tw[t];
  const double2* __restrict__ twp = tw_s ? stw : tw;
  __syncthreads();
  const int k = blockIdx.x * 32 + threadIdx.x;
  const int l = blockIdx.y * 8 + threadIdx.y;
  const int bc = blockIdx.z;
  if (k >= Wf || l >= H) return;
  const double2* col = A + (long)bc * H * Wf + k;
  double re = 0.0, im = 0.0;
  int idx = 0;
  for (int y = 0; y < H; ++y) {
    const double2 a = col[(long)y * Wf];
    const double2 w = twp[idx];
    if (DIR < 0) {            // (a)(c - i s)
      re = fma(a.x, w.x, fma(a.y, w.y, re));
      im = fma(a.y, w.x, fma(-a.x, w.y, im));
    } else {                  // (a)(c + i s)
      re = fma(a.x, w.x, fma(-a.y, w.y, re));
      im = fma(a.x, w.y, fma(a.y, w.x, im));
    }
    idx += l;
    if (idx >= H) idx -= H;
  }
  double m = scale;
  if (DIR < 0 && mask) m *= (double)mask[(long)l * Wf + k];
  Out[((long)bc * H + l) * Wf + k] = make_double2(re * m, im * m);
}

__global__ void __launch_bounds__(128) k_fft_rows_inv(const double2* __restrict__ G, const float* __restrict__ x,
                                                      int H, int W, int Wf, const double2* __restrict__ tw,
                                                      double scale, const float* __restrict__ band_scale,
                                                      float* __restrict__ raw9, int B, float* __restrict__ low_out) {
  __shared__ double2 sg[128];
  __shared__ double2 stw[1024];
  const bool tw_s = W <= 1024;
  if (tw_s)
    for (int t = threadIdx.x; t < W; t += blockDim.x) stw[t] = tw[t];
  const double2* __restrict__ twp = tw_s ? stw : tw;
  __syncthreads();
  const int xx = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y, bc = blockIdx.z, b = bc / 3, c = bc % 3;
  const double2* row = G + ((long)bc * H + y) * Wf;
  const bool even = (W % 2) == 0;
  const int kmax = even ? W / 2 - 1 : (W - 1) / 2;   // last strictly-interior bin
  double acc = 0.0;
  int idx = 0;   // (k * xx) mod W, advanced once per k
  for (int k0 = 0; k0 < Wf; k0 += 128) {
    const int n = min(128, Wf - k0);
    for (int t = threadIdx.x; t < n; t += blockDim.x) sg[t] = row[k0 + t];
    __syncthreads();
    if (xx < W) {
      for (int t = 0; t < n; ++t) {
        const int k = k0 + t;
        const double2 g = sg[t];
        if (k == 0) {
          acc += g.x;
        } else if (k <= kmax) {
          const double2 w = twp[idx];
          acc += 2.0 * fma(g.x, w.x, -g.y * w.y);
        } else {   // Nyquist column (W even): cos(pi*x) = (-1)^x, imaginary part ignored
          acc += (xx & 1) ? -g.x : g.x;
        }
        idx += xx;
        if (idx >= W) idx -= W;
      }
    }
    __syncthreads();
  }
  if (xx < W) {
    const float low = (float)(acc * scale);
    const long o = (long)y * W + xx;
    if (low_out) {                      // train mode: the unscaled low band only (scales / high band are applied upstream)
      low_out[(long)bc * H * W + o] = low;
      return;
    }
    const float xin = x[(long)bc * H * W + o];
    raw9[(((long)b * 9 + 7) * 3 + c) * H * W + o] = low * band_scale[0];
    raw9[(((long)b * 9 + 8) * 3 + c) * H * W + o] = (xin - low) * band_scale[1];
  }
}

// ------------------------------------------------------------------------------------
// Staged shared-memory FFT path (the default for H, W <= 2048: 212 KB of shared memory at 2048).  The dense-DFT kernels above cost O(N) complex MACs per
// point in fp64 with one thread per output (0.55 ms per 339x510 image, 0.5 % of the HBM roofline).  Here every 1-D transform is
// one Cooley-Tukey split N = N1 * N2 (N1 the divisor closest to sqrt(N); 510 = 17 * 30, 339 = 3 * 113, primes degenerate to the
// dense form) evaluated on CW independent sequences held in shared memory as [n][CW]:
//     t[n2][k1] = W_N^{n2 k1} * sum_{n1} x[N2 n1 + n2] W_N1^{n1 k1}        (N1 terms)
//     X[k1 + N1 k2] =          sum_{n2} t[n2][k1]    W_N2^{n2 k2}        (N2 terms)
// in fp32 with twiddles read from the fp64-generated table (all three twiddle families are powers of W_N).  Rows: CW image
// rows per block; columns: a strip of CW spectrum columns per block does forward transform, mask * scale and inverse
// transform without leaving shared memory.  Three launches, ~4 MB of fp32 complex intermediates.
// ------------------------------------------------------------------------------------
constexpr int FFT2_CW = 4;
constexpr int FFT2_THREADS = 256;

// in -> out over [N][CW] shared-memory arrays (tmp: scratch of the same size).  dir = -1: e^{-i...} (forward), +1: inverse.
// Callers synchronise before (inputs written) and after (outputs read).
template <int CW>
__device__ __forceinline__ void strip_fft(const float2* __restrict__ in, float2* __restrict__ tmp, float2* __restrict__ out,
                                          const float2* __restrict__ tw, int N, int N1, int N2, float sg) {
  const int total = N * CW;
  for (int o = threadIdx.x; o < total; o += blockDim.x) {
    const int c = o % CW, q = o / CW;
    const int n2 = q / N1, k1 = q - n2 * N1;
    const int inc = k1 * N2;                       // W_N1^{k1} = W_N^{k1 N2}
    const float2* p = in + n2 * CW + c;
    const int pstride = N2 * CW;
    float re = 0.f, im = 0.f;
    int idx = 0;
    for (int n1 = 0; n1 < N1; ++n1) {
      const float2 v = p[n1 * pstride];
      const float2 w = tw[idx];
      const float ws = sg * w.y;
      re = fmaf(v.x, w.x, fmaf(-v.y, ws, re));
      im = fmaf(v.x, ws, fmaf(v.y, w.x, im));
      idx += inc;
      if (idx >= N) idx -= N;
    }
    const float2 w = tw[n2 * k1];
    const float ws = sg * w.y;
    tmp[o] = make_float2(re * w.x - im * ws, re * ws + im * w.x);      // o = (n2 * N1 + k1) * CW + c
  }
  __syncthreads();
  for (int o = threadIdx.x; o < total; o += blockDim.x) {
    const int c = o % CW, k = o / CW;
    const int k2 = k / N1, k1 = k - k2 * N1;
    const int inc = k2 * N1;                       // W_N2^{k2} = W_N^{k2 N1}
    const float2* p = tmp + k1 * CW + c;
    const int pstride = N1 * CW;
    float re = 0.f, im = 0.f;
    int idx = 0;
    for (int n2 = 0; n2 < N2; ++n2) {
      const float2 v = p[n2 * pstride];
      const float2 w = tw[idx];
      const float ws = sg * w.y;
      re = fmaf(v.x, w.x, fmaf(-v.y, ws, re));
      im = fmaf(v.x, ws, fmaf(v.y, w.x, im));
      idx += inc;
      if (idx >= N) idx -= N;
    }
    out[o] = make_float2(re, im);
  }
  __syncthreads();
}

__device__ __forceinline__ void fft2_load_tw(float2* stw, const double2* __restrict__ tw, int N) {
  for (int t = threadIdx.x; t < N; t += blockDim.x) {
    const double2 w = tw[t];
    stw[t] = make_float2((float)w.x, (float)w.y);
  }
}

// rows, real -> half spectrum: A[bc][y][0..Wf)
__global__ void __launch_bounds__(FFT2_THREADS) k_fft2_rows_fwd(const float* __restrict__ x, int H, int W, int Wf, int N1, int N2,
                                                                const double2* __restrict__ tw, float2* __restrict__ A) {
  extern __shared__ float2 fsm[];
  constexpr int CW = FFT2_CW;
  float2* b0 = fsm;
  float2* b1 = b0 + W * CW;
  float2* b2 = b1 + W * CW;
  float2* stw = b2 + W * CW;
  fft2_load_tw(stw, tw, W);
  const int y0 = blockIdx.x * CW, bc = blockIdx.y;
  for (int o = threadIdx.x; o < W * CW; o += blockDim.x) {
    const int r = o / W, n = o - r * W;            // coalesced along the row
    const int y = y0 + r;
    b0[n * CW + r] = make_float2(y < H ? x[((long)bc * H + y) * W + n] : 0.f, 0.f);
  }
  __syncthreads();
  strip_fft<CW>(b0, b1, b2, stw, W, N1, N2, -1.f);
  for (int o = threadIdx.x; o < Wf * CW; o += blockDim.x) {
    const int r = o / Wf, k = o - r * Wf;
    const int y = y0 + r;
    if (y < H) A[((long)bc * H + y) * Wf + k] = b2[k * CW + r];
  }
}

// columns: forward, * mask * scale, inverse; in place on A (each block owns its CW columns)
__global__ void __launch_bounds__(FFT2_THREADS) k_fft2_cols(float2* __restrict__ A, int H, int Wf, int N1, int N2,
                                                            const double2* __restrict__ tw, const float* __restrict__ mask,
                                                            float scale, float2* __restrict__ spec_out) {
  extern __shared__ float2 fsm[];
  constexpr int CW = FFT2_CW;
  float2* b0 = fsm;
  float2* b1 = b0 + H * CW;
  float2* b2 = b1 + H * CW;
  float2* stw = b2 + H * CW;
  fft2_load_tw(stw, tw, H);
  const int k0 = blockIdx.x * CW, bc = blockIdx.y;
  float2* base = A + (long)bc * H * Wf;
  for (int o = threadIdx.x; o < H * CW; o += blockDim.x) {
    const int y = o / CW, c = o - y * CW;
    b0[o] = (k0 + c < Wf) ? base[(long)y * Wf + k0 + c] : make_float2(0.f, 0.f);
  }
  __syncthreads();
  strip_fft<CW>(b0, b1, b2, stw, H, N1, N2, -1.f);
  for (int o = threadIdx.x; o < H * CW; o += blockDim.x) {
    const int l = o / CW, c = o - l * CW;
    float mm = scale;
    if (mask && k0 + c < Wf) mm *= mask[(long)l * Wf + k0 + c];
    const float2 v = b2[o];
    b2[o] = make_float2(v.x * mm, v.y * mm);
    if (spec_out && k0 + c < Wf) spec_out[((long)bc * H + l) * Wf + k0 + c] = b2[o];    // training: the (scaled) spectrum itself
  }
  __syncthreads();
  if (spec_out) return;
  strip_fft<CW>(b2, b1, b0, stw, H, N1, N2, 1.f);
  for (int o = threadIdx.x; o < H * CW; o += blockDim.x) {
    const int y = o / CW, c = o - y * CW;
    if (k0 + c < Wf) base[(long)y * Wf + k0 + c] = b0[o];
  }
}

// rows, half spectrum -> real (irfft semantics: imaginary parts of the DC and Nyquist bins ignored), then the two bands
__global__ void __launch_bounds__(FFT2_THREADS) k_fft2_rows_inv(const float2* __restrict__ G, const float* __restrict__ x, int H,
                                                                int W, int Wf, int N1, int N2, const double2* __restrict__ tw,
                                                                float scale, const float* __restrict__ band_scale,
                                                                float* __restrict__ raw9, float* __restrict__ low_out) {
  extern __shared__ float2 fsm[];
  constexpr int CW = FFT2_CW;
  float2* b0 = fsm;
  float2* b1 = b0 + W * CW;
  float2* b2 = b1 + W * CW;
  float2* stw = b2 + W * CW;
  fft2_load_tw(stw, tw, W);
  const int y0 = blockIdx.x * CW, bc = blockIdx.y, b = bc / 3, ch = bc % 3;
  const bool even = (W % 2) == 0;
  for (int o = threadIdx.x; o < W * CW; o += blockDim.x) {
    const int r = o / W, k = o - r * W;
    const int y = y0 + r;
    float2 v = make_float2(0.f, 0.f);
    if (y < H) {
      const float2* row = G + ((long)bc * H + y) * Wf;
      if (k == 0 || (even && k == W / 2)) v = make_float2(row[k].x, 0.f);
      else if (k < Wf) v = row[k];
      else { const float2 g = row[W - k]; v = make_float2(g.x, -g.y); }
    }
    b0[k * CW + r] = v;
  }
  __syncthreads();
  strip_fft<CW>(b0, b1, b2, stw, W, N1, N2, 1.f);
  const float s0 = band_scale ? band_scale[0] : 1.f, s1 = band_scale ? band_scale[1] : 1.f;
  for (int o = threadIdx.x; o < W * CW; o += blockDim.x) {
    const int r = o / W, n = o - r * W;
    const int y = y0 + r;
    if (y >= H) continue;
    const float low = b2[n * CW + r].x * scale;
    const long pix = (long)y * W + n;
    if (low_out) { low_out[(long)bc * H * W + pix] = low; continue; }
    const float xin = x[(long)bc * H * W + pix];
    raw9[(((long)b * 9 + 7) * 3 + ch) * H * W + pix] = low * s0;
    raw9[(((long)b * 9 + 8) * 3 + ch) * H * W + pix] = (xin - low) * s1;
  }
}

static void fft2_split(int N, int* n1, int* n2) {
  int best = 1;
  for (int d = 1; (long)d * d <= N; ++d)
    if (N % d == 0) best = d;
  *n1 = best;
  *n2 = N / best;
}
static bool fft2_ok(int H, int W) { return H <= 2048 && W <= 2048; }
static size_t fft2_smem(int N) { return (size_t)(3 * FFT2_CW + 1) * N * sizeof(float2); }

// low-pass of B*3 planes through the staged path; A: fp32 complex scratch [B*3][H][Wf]
static int fft2_lowpass(const float* x, int B, int H, int W, const float* mask, const void* tw_h, const void* tw_w, float2* A,
                        const float* band_scale, float* raw9, float* low_out, cudaStream_t stream) {
  const int Wf = W / 2 + 1;
  int w1, w2, h1, h2;
  fft2_split(W, &w1, &w2);
  fft2_split(H, &h1, &h2);
  const float scale = (float)(1.0 / sqrt((double)H * (double)W));
  static bool attr = false;
  if (!attr) {
    attr = true;
    cudaFuncSetAttribute(k_fft2_rows_fwd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fft2_smem(2048));
    cudaFuncSetAttribute(k_fft2_cols, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fft2_smem(2048));
    cudaFuncSetAttribute(k_fft2_rows_inv, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fft2_smem(2048));
  }
  int rc;
  k_fft2_rows_fwd<<<dim3(ceil_div(H, FFT2_CW), B * 3), FFT2_THREADS, fft2_smem(W), stream>>>(x, H, W, Wf, w1, w2, (const double2*)tw_w, A);
  if ((rc = ffsr_check_launch("fft2_rows_fwd"))) return rc;
  k_fft2_cols<<<dim3(ceil_div(Wf, FFT2_CW), B * 3), FFT2_THREADS, fft2_smem(H), stream>>>(A, H, Wf, h1, h2, (const double2*)tw_h, mask, scale, nullptr);
  if ((rc = ffsr_check_launch("fft2_cols"))) return rc;
  k_fft2_rows_inv<<<dim3(ceil_div(H, FFT2_CW), B * 3), FFT2_THREADS, fft2_smem(W), stream>>>(A, x, H, W, Wf, w1, w2, (const double2*)tw_w, scale,
                                                                                               band_scale, raw9, low_out);
  return ffsr_check_launch("fft2_rows_inv");
}

extern "C" size_t ffsr_fft_workspace_bytes(int B, int H, int W) {
  const size_t Wf = (size_t)W / 2 + 1;
  const size_t cplx = (size_t)B * 3 * H * Wf * sizeof(double2);
  const size_t mask = ((size_t)H * Wf * sizeof(float) + 255) / 256 * 256;
  return 2 * cplx + mask;
}

extern "C" int ffsr_fft_bands(const float* lr, int B, int H, int W, const float* logits, int mask_size,
                              const float* temperature, const float* band_scale, const void* tw_h,
                              const void* tw_w, void* ws, size_t ws_bytes, float* raw9, cudaStream_t stream) {
  FFSR_REQUIRE(lr && raw9 && logits && temperature && band_scale && tw_h && tw_w && ws, FFSR_ERR_ARG, "fft_bands: null pointer");
  FFSR_REQUIRE(B > 0 && H > 0 && W > 1 && mask_size > 0, FFSR_ERR_ARG, "fft_bands: bad shape");
  FFSR_REQUIRE(ws_bytes >= ffsr_fft_workspace_bytes(B, H, W), FFSR_ERR_ARG, "fft_bands: workspace too small");
  FFSR_REQUIRE(((uintptr_t)ws % 16) == 0, FFSR_ERR_ALIGN, "fft_bands: workspace must be 16B aligned");
  const int Wf = W / 2 + 1;
  const size_t cplx = (size_t)B * 3 * H * Wf * sizeof(double2);
  double2* A = (double2*)ws;
  double2* F = (double2*)((char*)ws + cplx);
  float* mask = (float*)((char*)ws + 2 * cplx);
  const double scale = 1.0 / sqrt((double)H * (double)W);   // norm='ortho', applied once per direction
  int rc;
  k_fft_mask<<<dim3(ceil_div(Wf, 128), H), 128, 0, stream>>>(logits, mask_size, H, Wf, temperature, mask);
  if ((rc = ffsr_check_launch("fft_mask"))) return rc;
  if (fft2_ok(H, W)) return fft2_lowpass(lr, B, H, W, mask, tw_h, tw_w, (float2*)A, band_scale, raw9, nullptr, stream);
  k_fft_rows_fwd<<<dim3(ceil_div(Wf, 128), H, B * 3), 128, 0, stream>>>(lr, H, W, Wf, (const double2*)tw_w, A);
  if ((rc = ffsr_check_launch("fft_rows_fwd"))) return rc;
  dim3 gc(ceil_div(Wf, 32), ceil_div(H, 8), B * 3);
  k_fft_cols<-1><<<gc, dim3(32, 8), 0, stream>>>(A, H, Wf, (const double2*)tw_h, mask, scale, F);
  if ((rc = ffsr_check_launch("fft_cols_fwd"))) return rc;
  k_fft_cols<1><<<gc, dim3(32, 8), 0, stream>>>(F, H, Wf, (const double2*)tw_h, nullptr, 1.0, A);
  if ((rc = ffsr_check_launch("fft_cols_inv"))) return rc;
  k_fft_rows_inv<<<dim3(ceil_div(W, 128), H, B * 3), 128, 0, stream>>>(A, lr, H, W, Wf, (const double2*)tw_w, scale,
                                                                        band_scale, raw9, B, nullptr);
  return ffsr_check_launch("fft_rows_inv");
}

// ------------------------------------------------------------------------------------------------
// Train mode: low = irfft2(mask * rfft2(x)) with an explicit mask tensor, and the gradient of a scalar loss
// w.r.t. that mask:  dmask[l][k] = c_k * sum_{b,c} Re(conj(X[l][k]) * Q[l][k]),  X = rfft2(x), Q = rfft2(dL/dlow),
// c_k = 1 for the DC / Nyquist columns and 2 otherwise (the Hermitian half counted twice) -- identical to what
// autograd derives for torch.fft.irfft2 (multi_domain_frequency.py:362-383).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_fft_dmask(const double2* __restrict__ X, const double2* __restrict__ Q, int P, int H,
                                                   int Wf, int W, float* __restrict__ dmask) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  const int l = blockIdx.y;
  if (k >= Wf) return;
  double acc = 0.0;
  for (int p = 0; p < P; ++p) {
    const long i = ((long)p * H + l) * Wf + k;
    const double2 a = X[i], b = Q[i];
    acc += a.x * b.x + a.y * b.y;
  }
  const bool edge = (k == 0) || ((W % 2 == 0) && k == Wf - 1);
  dmask[(long)l * Wf + k] = (float)(edge ? acc : 2.0 * acc);
}

extern "C" size_t ffsr_fft_lowpass_workspace_bytes(int B, int H, int W) {
  return (size_t)3 * B * 3 * H * ((size_t)W / 2 + 1) * sizeof(double2);
}

extern "C" int ffsr_fft_lowpass(const float* x, int B, int H, int W, const float* mask, const void* tw_h, const void* tw_w,
                                void* ws, size_t ws_bytes, float* low, cudaStream_t stream) {
  FFSR_REQUIRE(x && mask && tw_h && tw_w && ws && low && B > 0 && H > 0 && W > 1, FFSR_ERR_ARG, "fft_lowpass: bad argument");
  FFSR_REQUIRE(ws_bytes >= ffsr_fft_lowpass_workspace_bytes(B, H, W) && ((uintptr_t)ws % 16) == 0, FFSR_ERR_ARG, "fft_lowpass: workspace");
  const int Wf = W / 2 + 1;
  const size_t cplx = (size_t)B * 3 * H * Wf * sizeof(double2);
  double2* A = (double2*)ws;
  double2* F = (double2*)((char*)ws + cplx);
  if (fft2_ok(H, W)) return fft2_lowpass(x, B, H, W, mask, tw_h, tw_w, (float2*)A, nullptr, nullptr, low, stream);
  const double scale = 1.0 / sqrt((double)H * (double)W);
  dim3 gc(ceil_div(Wf, 32), ceil_div(H, 8), B * 3);
  k_fft_rows_fwd<<<dim3(ceil_div(Wf, 128), H, B * 3), 128, 0, stream>>>(x, H, W, Wf, (const double2*)tw_w, A);
  k_fft_cols<-1><<<gc, dim3(32, 8), 0, stream>>>(A, H, Wf, (const double2*)tw_h, mask, scale, F);
  k_fft_cols<1><<<gc, dim3(32, 8), 0, stream>>>(F, H, Wf, (const double2*)tw_h, nullptr, 1.0, A);
  k_fft_rows_inv<<<dim3(ceil_div(W, 128), H, B * 3), 128, 0, stream>>>(A, x, H, W, Wf, (const double2*)tw_w, scale, nullptr,
                                                                        nullptr, B, low);
  return ffsr_check_launch("fft_lowpass");
}

extern "C" int ffsr_fft_lowpass_backward(const float* x, const float* dlow, int B, int H, int W, const void* tw_h,
                                         const void* tw_w, void* ws, size_t ws_bytes, float* dmask, cudaStream_t stream) {
  FFSR_REQUIRE(x && dlow && tw_h && tw_w && ws && dmask && B > 0 && H > 0 && W > 1, FFSR_ERR_ARG, "fft_lowpass_backward: bad argument");
  FFSR_REQUIRE(ws_bytes >= ffsr_fft_lowpass_workspace_bytes(B, H, W) && ((uintptr_t)ws % 16) == 0, FFSR_ERR_ARG, "fft_lowpass_backward: workspace");
  const int Wf = W / 2 + 1;
  const size_t cplx = (size_t)B * 3 * H * Wf * sizeof(double2);
  double2* A = (double2*)ws;
  double2* X = (double2*)((char*)ws + cplx);
  double2* Q = (double2*)((char*)ws + 2 * cplx);
  const double scale = 1.0 / sqrt((double)H * (double)W);
  dim3 gr(ceil_div(Wf, 128), H, B * 3), gc(ceil_div(Wf, 32), ceil_div(H, 8), B * 3);
  k_fft_rows_fwd<<<gr, 128, 0, stream>>>(x, H, W, Wf, (const double2*)tw_w, A);
  k_fft_cols<-1><<<gc, dim3(32, 8), 0, stream>>>(A, H, Wf, (const double2*)tw_h, nullptr, scale, X);
  k_fft_rows_fwd<<<gr, 128, 0, stream>>>(dlow, H, W, Wf, (const double2*)tw_w, A);
  k_fft_cols<-1><<<gc, dim3(32, 8), 0, stream>>>(A, H, Wf, (const double2*)tw_h, nullptr, scale, Q);
  k_fft_dmask<<<dim3(ceil_div(Wf, 128), H), 128, 0, stream>>>(X, Q, B * 3, H, Wf, W, dmask);
  return ffsr_check_launch("fft_lowpass_backward");
}
