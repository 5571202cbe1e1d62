/* ffsr_b200.h -- C ABI of libffsr_b200.so, the sm_100a kernel library behind the
 * drop-in CompleteEnhancedFusionSR module (image-super-resolution_b200/fusion.py).
 *
 * The reference (Nikhil-AI-Labs/Image-Super-Resolution) is pure Python/PyTorch: it has no
 * FFI of its own.  The "interface each entry point replaces" is therefore the PyTorch op
 * sequence at the cited reference file:line (all relative to the reference root); the
 * binding a maintainer adds is the ctypes stub shown in INTEGRATION.md.
 *
 * Conventions (SURVEY.md section 8b):
 *  - every pointer is a DEVICE pointer owned by the caller (PyTorch caching allocator),
 *    including scratch; kernels never allocate, free or synchronise the host;
 *  - work is enqueued on the cudaStream_t passed in (never the legacy default stream
 *    implicitly); entry points are re-entrant across streams;
 *  - return 0 on success, <0 on error (FFSR_ERR_*); ffsr_last_error() gives the message;
 *  - sm_100a only: there is no fallback path, ffsr_device_check() fails elsewhere.
 *  - scalar nn.Parameters (scales, temperatures) are passed as device pointers so that no
 *    host sync (.item()) is needed.
 */
#ifndef FFSR_B200_H
#define FFSR_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#ifndef __CUDA_RUNTIME_H__
typedef struct CUstream_st* cudaStream_t;
#endif

#define FFSR_OK 0
#define FFSR_ERR_ARG (-1)
#define FFSR_ERR_ALIGN (-2)
#define FFSR_ERR_LAUNCH (-3)
#define FFSR_ERR_DRIVER (-4)

#define FFSR_ACT_NONE 0
#define FFSR_ACT_GELU 1
#define FFSR_ACT_RELU 2
#define FFSR_ACT_SIGMOID 3

#define FFSR_EPI_PLAIN 0    /* out = act(conv + bias)                                        */
#define FFSR_EPI_RESIDUAL 1 /* out = r1 + sa*act(conv + bias) + sb*r2          (r2 optional) */
#define FFSR_EPI_LKAGATE 2  /* out = r1 + sa*(r1*ch_k[c] + ch_d[c])*sigmoid(conv + bias)     */
#define FFSR_EPI_ACTGRAD 3  /* out = (conv + bias) * act'(r1): input gradient of a conv fused with the
                               derivative of the activation that produced its input (r1 = that layer's
                               pre-activation); tcgen05 path only                                  */

#define FFSR_CONV_MULTI_ISSUE 1 /* ffsr_conv_params.flags: the tcgen05 path may spread a CTA's tiles over up to three MMA-issuing
                                  warps (issue-bound small layers; used by the inference pipeline) */

#define FFSR_DT_F32 0
#define FFSR_DT_BF16 1
#define FFSR_DT_F16 2  /* source dtype of cache records only (ffsr_cache_unpack) */

const char* ffsr_last_error(void);
const char* ffsr_version(void);
/* 0 iff the current device is compute capability 10.x; message otherwise. */
int ffsr_device_check(void);

/* ---- Phase 2: 9 sub-bands, raw9[B][9][3][H][W] fp32 ------------------------------------
 * DCTDecomposition.forward      src/models/multi_domain_frequency.py:146-196 */
int ffsr_dct_bands(const float* lr, int B, int H, int W, const float* basis, const float* basis_t,
                   const float* m_low, const float* m_mid, const float* m_high, const float* band_scale,
                   float* raw9, cudaStream_t stream);
/* DWTDecomposition.forward      src/models/multi_domain_frequency.py:251-299
 * sub_ws: float[B*12*Hs*Ws] with (Hs,Ws) from ffsr_dwt_sub_size */
int ffsr_dwt_sub_size(int H, int W, int* Hs, int* Ws);
int ffsr_dwt_bands(const float* lr, int B, int H, int W, const float* lo_row, const float* hi_row,
                   const float* lo_col, const float* hi_col, const float* subband_scale, float* sub_ws,
                   float* raw9, cudaStream_t stream);
/* Adjoints of the unit-scale DCT / DWT bands (input gradient of Phase 2; gathers, no atomics, fixed summation order).
 * ffsr_dct_bands_adjoint: g3[B][3][3][H][W] (low, mid, high) -> dx[B][3][H][W] (WRITTEN); pad_ws: float[B*3*Hp*Wp],
 *   Hp / Wp = H / W rounded up to a multiple of 8.
 * ffsr_dwt_bands_adjoint: g4[B][4][3][H][W] (LL, LH, HL, HH) -> dx[B][3][H][W] (ACCUMULATED); sub_ws as for ffsr_dwt_bands. */
int ffsr_dct_bands_adjoint(const float* g3, int B, int H, int W, const float* basis, const float* basis_t,
                           const float* m_low, const float* m_mid, const float* m_high, float* pad_ws, float* dx,
                           cudaStream_t stream);
int ffsr_dwt_bands_adjoint(const float* g4, int B, int H, int W, const float* lo_row, const float* hi_row,
                           const float* lo_col, const float* hi_col, float* sub_ws, float* dx, cudaStream_t stream);
/* FFTDecomposition.forward      src/models/multi_domain_frequency.py:352-385
 * tw_h / tw_w: double2[H] / double2[W] tables from ffsr_fft_twiddles; ws from ffsr_fft_workspace_bytes */
int ffsr_fft_twiddles(int n, void* out, cudaStream_t stream);
size_t ffsr_fft_workspace_bytes(int B, int H, int W);
int ffsr_fft_bands(const float* lr, int B, int H, int W, const float* logits, int mask_size,
                   const float* temperature, const float* band_scale, const void* tw_h, const void* tw_w,
                   void* ws, size_t ws_bytes, float* raw9, cudaStream_t stream);

/* ---- Phase 3: cross-band attention -------------------------------------------------------
 * EnhancedCrossBandWithLKA.forward steps 1-2  src/models/large_kernel_attention.py:219-233
 * tok_out[B][nq][H][W][64]: attention output (+residual) of the first nq bands.
 * fold (required, 16B aligned, [64x4 | 192x4 | 192] floats): band_proj -> LayerNorm -> in_proj collapsed on the host
 * (a token is an affine function of 3 band values): A|c = centred band_proj rows / bias, M|m0 = W_in diag(gamma) [A|c],
 * n0 = W_in beta + b_in; qkv = rstd * (M x + m0) + n0 -- 16x fewer FLOPs, same result up to fp32 rounding.
 * tok_out must be 16B aligned. */
int ffsr_crossband_attention(const float* raw9, int B, int H, int W, const float* proj_w, const float* proj_b,
                             const float* out_w, const float* out_b, int nq, float* tok_out, int num_sms,
                             const float* fold, cudaStream_t stream);
/* out_proj + band residual (:240-241) and routing_lr = bands 0+1+2 (enhanced_fusion_v2.py:713) */
int ffsr_crossband_out(const float* x, const float* raw9, int B, int H, int W, int nq, const float* w,
                       const float* bias, float* enh9, float* routing, cudaStream_t stream);

/* ---- LKA depthwise chain (BN1 affine -> dw5x5 -> dw1x21 -> dw21x1) -----------------------
 * LargeKernelAttention.forward  src/models/large_kernel_attention.py:98-100; x,out: [N][H][W][C] */
int ffsr_lka_depthwise(const float* x, int N, int H, int W, int C, const float* bn_k, const float* bn_d,
                       const float* w5, const float* wh, const float* wv, float* tmp1, float* tmp2, void* out,
                       int out_dtype, cudaStream_t stream);
/* the same chain reading a bf16 (x_dtype = FFSR_DT_BF16) or fp32 input tensor */
int ffsr_lka_depthwise_in(const void* x, int x_dtype, int N, int H, int W, int C, const float* bn_k, const float* bn_d,
                          const float* w5, const float* wh, const float* wv, float* tmp1, float* tmp2, void* out,
                          int out_dtype, cudaStream_t stream);

/* ---- token helpers (Phase 4) -------------------------------------------------------------
 * nn.LayerNorm rows (large_kernel_attention.py:389,392) and the softmax(QK^T/4)V core of
 * nn.MultiheadAttention (:390) for T tokens per LR pixel, head_dim 16; token-major layout
 * qkv[B][T][HW][3E] -> ctx[B][T][HW][E] */
/* Tail of an LKABlock on fp32 64-channel token rows, tile-resident on tcgen05 at fp32 accuracy (three-term bf16 split of
 * both operands, six products accumulated in fp32): x1 = x + s1 * BN1(x) * sigmoid(BN(pw(a))); out = x1 + s2 * ffn(BN2(x1))
 * src/models/large_kernel_attention.py:96-105 (pw + bn + sigmoid gate), :143-149 (LKABlock.forward).  Weights / parameters
 * are packed by the host into the kernel's shared-memory layout (isr_b200.pipeline: _prep_lka). */
size_t ffsr_lka_tail_weight_bytes(void);
size_t ffsr_lka_tail_param_floats(void);
int ffsr_lka_tail64(const float* x, const float* a, long rows, const void* wblob, const float* pblob, const float* scale1,
                    const float* scale2, float* out, cudaStream_t stream);
/* bf16 variant for Phase 4 (128-channel tokens): the same tail followed by the first modulation layer (128 -> 32 per
 * expert, large_kernel_attention.py:415-416), x / a bf16 [nimg][HW][128] with expert = image index % 4, m32 bf16 [nimg][HW][32]. */
size_t ffsr_lka_tail128_weight_bytes(void);
size_t ffsr_lka_tail128_param_floats(void);
int ffsr_lka_tail128_mod(const void* x, const void* a, int nimg, int HW, const void* wblob, const float* pblob,
                         const float* scale1, const float* scale2, void* m32, cudaStream_t stream);
int ffsr_layernorm(const float* x, long rows, int E, const float* w, const float* b, void* y, int out_bf16,
                   cudaStream_t stream);
/* nn.LayerNorm(128) on bf16 rows -> bf16 rows (Phase 4, bf16 mode: residual stream stored as bf16) */
int ffsr_layernorm128_bf16(const void* x, long rows, const float* w, const float* b, void* y, cudaStream_t stream);
int ffsr_token_attention(const void* qkv, int B, int T, long HW, int E, void* ctx, int is_bf16, cudaStream_t stream);
/* Phase 4 token pipeline (bf16 mode) as two tile-resident tcgen05 kernels (csrc/token_chain.cu), LayerNorm folded into the
 * contraction that follows it:
 *   ffsr_token_attn_chain: out = x + out_proj(MultiheadAttention(LN1(x)))  over the 4 expert tokens of every pixel
 *                          (large_kernel_attention.py:389-391); x / out bf16 [B][4][HW][128], out may alias x
 *   ffsr_token_ffn_chain : out = x + ffn2(GELU(ffn0(LN2(x))))  (:392); x / out bf16 [rows][128]
 * Weight / parameter blobs in the kernels' shared-memory layout: isr_b200.pipeline.pack_token_attn / pack_token_ffn. */
/* The four expert feature maps (fp32 NCHW, channel counts C[e] <= 192) -> aligned bf16 tokens [B][4][HW][128]:
 * align_layers[e] (1x1 conv + bias, large_kernel_attention.py:344-358) with the NCHW -> channels-last change done on the way
 * into shared memory.  wblob: per expert [kg 24][n 128][8] bf16 (K zero-padded to 192), bias fp32 [4][128]. */
size_t ffsr_align_tokens_weight_bytes(void);
int ffsr_align_tokens(const float* const* feat, const int* C, int B, int HW, const void* wblob, const float* bias, void* out,
                      cudaStream_t stream);
size_t ffsr_token_attn_weight_bytes(void);
size_t ffsr_token_attn_param_floats(void);
int ffsr_token_attn_chain(const void* x, int B, int HW, const void* wblob, const float* pblob, void* out, cudaStream_t stream);
size_t ffsr_token_ffn_weight_bytes(void);
size_t ffsr_token_ffn_param_floats(void);
int ffsr_token_ffn_chain(const void* x, long rows, const void* wblob, const float* pblob, void* out, cudaStream_t stream);

/* ---- Phase 6 gate normalisation  src/models/enhanced_fusion_v2.py:462-465 ---------------- */
/* Phase 6 as ONE kernel (csrc/selector.cu): difficulty_net + gate_net + gate normalisation on shared-memory tiles, fp32.
 * DynamicExpertSelector.forward, src/models/enhanced_fusion_v2.py:450-466.  routing [B][3][H][W] -> diff [B][1][H][W],
 * graw [B][H][W][4] (gate_net logits), gates [B][4][H][W].  blob: isr_b200.pipeline.pack_selector. */
size_t ffsr_selector_blob_floats(void);
int ffsr_selector_fused(const float* routing, int B, int H, int W, const float* blob, const float* temperature, float* diff,
                        float* graw, float* gates, cudaStream_t stream);
int ffsr_gate_finalize(const float* raw, const float* diff, int B, int H, int W, const float* temperature,
                       float* gates, cudaStream_t stream);

/* ---- generic convolution (1x1 / 3x3, zero pad k/2, stride 1) -----------------------------
 * Replaces every nn.Conv2d / nn.Linear on the path (SURVEY 2.3 K4/K5/K7/K8).  Input element
 * (n,y,x,c) lives at in + n*in_sN + y*in_sY + x*in_sX + c*in_sC (element strides: NHWC or
 * NCHW views, channel slices of concat buffers).  Output and residuals are channels-last
 * (channel stride 1).  Weights are packed [groups][k*k][Cin][Cout] fp32; image n uses weight
 * set n % groups. */
typedef struct ffsr_conv_params {
  const void* in;
  long long in_sN, in_sY, in_sX, in_sC;
  int N, H, W, Cin, Cout, ksize;
  const float* w;
  const float* bias; /* [groups][Cout] or NULL */
  int groups;
  void* out;
  long long out_sN, out_sY, out_sX;
  int act; /* FFSR_ACT_* */
  int epi; /* FFSR_EPI_* */
  const void* r1;
  long long r1_sN, r1_sY, r1_sX;
  const void* r2;
  long long r2_sN, r2_sY, r2_sX;
  float sa;
  const float* sa_ptr; /* effective sa = sa * (sa_ptr ? *sa_ptr : 1) */
  float sb;
  const float* sb_ptr;
  const float* ch_k; /* per-channel affine of FFSR_EPI_LKAGATE */
  const float* ch_d;
  int in_dtype, out_dtype; /* FFSR_DT_* */
  int w_dtype;             /* FFSR_DT_F32: w = [groups][k*k][Cin][Cout] fp32 (CUDA-core path);
                              FFSR_DT_BF16: w = [groups*k*k][CoutPad][CinPad] bf16, K-major (tcgen05 path,
                              taken iff in_dtype == FFSR_DT_BF16; CinPad = ceil64(Cin), CoutPad = ceil16(Cout)
                              rounded up to a multiple of 128 when > 128) */
  int r1_dtype, r2_dtype;  /* FFSR_DT_* of the residual tensors */
  void* out2;              /* optional (tcgen05 path, FFSR_EPI_PLAIN with an activation): bf16 copy of the
                              PRE-activation conv + bias, same strides as out -- saved for the backward pass */
  int flags;      /* FFSR_CONV_* bits; 0 = defaults */
} ffsr_conv_params;

int ffsr_conv2d(const ffsr_conv_params* p, cudaStream_t stream);
/* sizeof(ffsr_conv_params) as compiled into the library (bindings assert their layout against it) */
size_t ffsr_conv_params_size(void);

/* ---- HR-side fused elementwise kernels ---------------------------------------------------- */
/* Phase 4 tail: bilinear x4 of the LR modulation features, GELU, 1x1 32->3, sigmoid,
 * out*(1+0.2*(mod-0.5)), clamp (eval)   src/models/large_kernel_attention.py:410-424
 * imgs: 4 pointers to [B][3][Hh][Wh]; m32: [B][4][H][W][32] (NULL: Phase 4 skipped, E = imgs);
 * w2: [4][3][32], b2: [4][3];  ecol: [B][4][3][Hh][Wh] fp32;  cat3: NHWC concat buffer slice */
int ffsr_modulate_hr(const float* const* imgs, const float* m32, const float* w2, const float* b2, int B, int H,
                     int W, int clamp01, float* ecol, void* cat3, long long cat3_sX, int cat3_dtype,
                     cudaStream_t stream);
/* Same operation, four HR pixels (one LR cell phase) x four experts per thread; m32 may be bf16 ([B][4][H][W][32], bf16 mode).
 * Requires m32 != NULL (use ffsr_modulate_hr for the pass-through case). */
int ffsr_modulate_hr_sized(const float* const* imgs, const float* m32, int mh, int mw, const float* w2, const float* b2,
                           int B, int H, int W, int clamp01, float* ecol, void* cat3, long long cat3_sX, int cat3_dtype,
                           cudaStream_t stream);   /* m32 on an mh x mw grid != LR (large_kernel_attention.py:365-372) */
int ffsr_modulate_hr_v2(const float* const* imgs, const void* m32, int m32_dtype, const float* w2, const float* b2, int B,
                        int H, int W, int clamp01, float* ecol, void* cat3, long long cat3_sX, int cat3_dtype,
                        cudaStream_t stream);
/* bilinear /2 and /4 of the expert stack (hierarchical_fusion.py:156-159, 171-174) into the
 * stage-2 concat buffer slice and the stage-1 input */
int ffsr_expert_downsample(const float* ecol, int B, int Hh, int Wh, void* cat2, long long cat2_sX, void* s1in,
                           long long s1_sX, int dtype, cudaStream_t stream);
/* bilinear resize of a channels-last tensor into a channel slice (hierarchical_fusion.py:166-169,183-186) */
int ffsr_resize_nhwc(const void* src, int N, int h, int w, int C, long long src_sX, void* dst, int H, int W,
                     long long dst_sX, int dtype, cudaStream_t stream);
/* SpatialGate: x * sigmoid(w2 . gelu(W1 x + b1) + b2)   hierarchical_fusion.py:25-43 (in place allowed) */
int ffsr_spatial_gate(const void* x, long pixels, int C, const float* w1, const float* b1, const float* w2,
                      const float* b2, void* y, int dtype, cudaStream_t stream);
/* Phase 5b/5c/6 blend   src/models/enhanced_fusion_v2.py:735-774 */
int ffsr_blend_hr(const float* hier, long long hier_sX, const float* ecol, const float* routing, const float* gates,
                  const float* diff, const float* fw0_w, const float* fw0_b, const float* fw2_w, const float* fw2_b,
                  int B, int H, int W, float* fused_before, float* fused_nhwc, long long fused_sX, void* fused_lp,
                  long long fused_lp_sX, cudaStream_t stream);
/* Laplacian pyramid pieces   src/models/edge_enhancement.py:196-220 */
/* the optional *_lp outputs are bf16 channels-last copies (tcgen05 operands of the edge refiners) */
int ffsr_blur_pool(const float* x, long long x_sX, int N, int H, int W, const float* gauss25, float* down,
                   long long down_sX, void* down_lp, long long down_lp_sX, cudaStream_t stream);
/* adjoint of ffsr_blur_pool (gradient w.r.t. x of down = avg_pool2(gauss5x5(x))); g: [N][H/2][W/2] pitch g_sX */
int ffsr_blur_pool_backward(const float* g, long long g_sX, int N, int H, int W, const float* gauss25, float* gx,
                            long long gx_sX, cudaStream_t stream);
int ffsr_laplacian_sub(const float* x, long long x_sX, const float* down, long long down_sX, int N, int H, int W,
                       float* lap, long long lap_sX, void* lap_lp, long long lap_lp_sX, cudaStream_t stream);
/* refiner tail: (o * attn) [bilinear to HxW] * softmax(level_weights)[level] -> concat slice
 * src/models/edge_enhancement.py:118, 243-250 */
int ffsr_edge_attn_upsample(const void* o, int o_dtype, const float* attn, int N, int h, int w, int C,
                            const float* level_w, int level, void* dst, int H, int W, long long dst_sX, int dtype,
                            cudaStream_t stream);

/* Tile-resident edge refiner of ONE pyramid level (bf16 mode): EdgeRefineBlock + SpatialEdgeAttention in one tcgen05
 * kernel, 32-channel intermediates in shared memory (csrc/edge_chain.cu).
 * Replaces: r.proj / conv1 / conv2 / conv3 + identity, attn.attn[0..3] and the x * attn product --
 *   src/models/edge_enhancement.py:69-83 (SpatialEdgeAttention), :96-118 (EdgeRefineBlock.forward).
 * x: bf16 [N][H][W][8] (3 Laplacian channels + 5 zero); wblob / pblob: weights packed by the host into the kernel's
 * shared-memory layout (ffsr_edge_chain_weight_bytes() bytes of bf16, ffsr_edge_chain_param_floats() floats; layout in
 * csrc/edge_chain.cu).  mode 0: dst[n][y][x][0..31] = o3 * at * softmax(level_w)[level] (strided bf16 view, e.g. a slice
 * of the 96-channel concat); mode 1: dst = o3 (bf16) and attn_out[N][H][W] = at (fp32), for ffsr_edge_attn_upsample. */
size_t ffsr_edge_chain_weight_bytes(void);
size_t ffsr_edge_chain_param_floats(void);
int ffsr_edge_refiner_chain(const void* x, int N, int H, int W, const void* wblob, const float* pblob,
                            const float* level_w, int level, void* dst, long long dst_sN, long long dst_sY,
                            long long dst_sX, float* attn_out, int mode, cudaStream_t stream);
/* out = clamp(x + gate*strength*edge, 0, 1) + residual_scale*bilinear_x4(lr) [clamp in eval]
 * src/models/edge_enhancement.py:259-260, src/models/enhanced_fusion_v2.py:788-795 */
int ffsr_final_combine(const float* xe, long long xe_sX, const float* gate, const float* strength, const float* lr,
                       const float* residual_scale, int B, int H, int W, int clamp01, float* out,
                       cudaStream_t stream);

/* layout/precision staging for the tcgen05 path: fp32 NCHW -> bf16 channels-last slice
 * (expert features, cached_dataset.py layout -> align_layers operand), contiguous fp32 -> bf16 */
int ffsr_nchw_to_nhwc_bf16(const float* src, int N, int C, long HW, void* dst, long long dst_sN, long long dst_sX,
                           cudaStream_t stream);
int ffsr_cast_f32_to_bf16(const float* src, void* dst, long n, cudaStream_t stream);

/* =========================================================================================
 * Train-mode / backward entry points.  The reference relies on ATen autograd for these
 * (loss.backward() in train.py:331-357 over the modules cited below); each entry point is the
 * hand-written counterpart of one autograd node.  Gradient outputs marked ACCUMULATED are
 * added into (the caller zeroes them), everything else is overwritten.
 * ========================================================================================= */

/* nn.Conv2d weight / bias gradient (every conv of enhanced_fusion_v2.py:681-799):
 *   dw[tap][ci][co] += sum_{n,y,x} x[n, y+dy, x+dx, ci] * dy[n, y, x, co];  dbias[co] += sum dy
 * x: strided view (NHWC or NCHW, like ffsr_conv2d's input); dy channels-last. */
typedef struct ffsr_wgrad_params {
  const void* x;
  long long x_sN, x_sY, x_sX, x_sC;
  int x_dtype;
  const void* dy;
  long long dy_sN, dy_sY, dy_sX;
  int dy_dtype;
  int N, H, W, Cin, Cout, ksize;
  float* dw;    /* [k*k][Cin][Cout] fp32, ACCUMULATED */
  float* dbias; /* [Cout] fp32, ACCUMULATED, or NULL */
} ffsr_wgrad_params;
/* Reproducibility: every reduction of the training path below (weight / bias / scalar gradients, normalisation
 * statistics, loss sums, gradient norm) partitions its work by shape alone, writes one partial per block into the
 * caller's workspace `ws` (ws_bytes >= the matching *_workspace_bytes query; no initialisation needed) and adds
 * the partials to the output in a fixed order: no floating-point atomics, so results are bitwise reproducible
 * for the same shapes on the same GPU.  A workspace may be reused by calls ordered on one stream. */
size_t ffsr_conv2d_wgrad_workspace_bytes(int N, int H, int W, int Cin, int Cout, int ksize);
int ffsr_conv2d_wgrad(const ffsr_wgrad_params* p, void* ws, size_t ws_bytes, cudaStream_t stream);
size_t ffsr_wgrad_params_size(void);
/* out[c] += sum over (n,y,x) of a channels-last tensor (bias / scale gradients) */
size_t ffsr_colsum_workspace_bytes(int N, int H, int W, int C);
int ffsr_colsum(const void* v, int dtype, int N, int H, int W, int C, long long sN, long long sY, long long sX,
                float* out, void* ws, size_t ws_bytes, cudaStream_t stream);

/* nn.GELU / nn.ReLU / nn.Sigmoid forward on contiguous data and backward on the saved
 * pre-activation: dx = dy * act'(x) */
int ffsr_act_forward(const void* x, void* y, long n, int act, int dtype, cudaStream_t stream);
int ffsr_act_backward(const void* x, const void* dy, void* dx, long n, int act, int dtype, cudaStream_t stream);

/* nn.LayerNorm backward (large_kernel_attention.py:223, 389, 392); dw/db ACCUMULATED */
size_t ffsr_layernorm_backward_workspace_bytes(long rows, int E);
int ffsr_layernorm_backward(const float* x, const float* dy, long rows, int E, const float* w, float* dx, float* dw,
                            float* db, void* ws, size_t ws_bytes, cudaStream_t stream);

/* nn.BatchNorm2d in train mode (large_kernel_attention.py:84,128,131) on channels-last data
 * viewed as [G][R][C]: G independent statistic groups (one LKABlock call each), R rows per group.
 *   ffsr_bn_stats:    sum[g][c], sumsq[g][c] += (fp64; ACCUMULATED)
 *   ffsr_bn_apply:    y = (x - mean[g][c]) * rstd[g][c] * w[c] + b[c]
 *   ffsr_bn_backward: sdy[g][c] += sum dy, sdyx[g][c] += sum dy*xhat (ACCUMULATED), then
 *                     dx = w*rstd*(dy - sdy/R - xhat*sdyx/R) */
size_t ffsr_bn_stats_workspace_bytes(int G, long R, int C);
int ffsr_bn_stats(const float* x, int G, long R, int C, double* sum, double* sumsq, void* ws, size_t ws_bytes,
                  cudaStream_t stream);
int ffsr_bn_apply(const float* x, int G, long R, int C, const float* mean, const float* rstd, const float* w,
                  const float* b, float* y, cudaStream_t stream);
size_t ffsr_bn_backward_workspace_bytes(int G, long R, int C);
int ffsr_bn_backward(const float* x, const float* dy, int G, long R, int C, const float* mean, const float* rstd,
                     const float* w, float* sdy, float* sdyx, float* dx, void* ws, size_t ws_bytes, cudaStream_t stream);
/* nn.BatchNorm2d in eval mode with gradients (running statistics as constants) on channels-last [R][C]: forward is
 * ffsr_bn_apply with G = 1 and (running_mean, rsqrt(running_var + eps)); the backward gives
 *   sdy[c] += sum dy, sdyx[c] += sum dy*xhat (ACCUMULATED, fixed order), dx = dy * w * rstd;
 * ws sized by ffsr_bn_backward_workspace_bytes(1, R, C). */
int ffsr_bn_eval_backward(const float* x, const float* dy, long R, int C, const float* mean, const float* rstd,
                          const float* w, float* sdy, float* sdyx, float* dx, void* ws, size_t ws_bytes, cudaStream_t stream);

/* nn.MultiheadAttention core in train mode (T = 4 or 9 tokens per LR pixel, head_dim 16,
 * attention-probability dropout): probs[B][HW][E/16][T][T] saved for the backward; the dropout
 * mask is a counter-based hash of (seed, element index), regenerated by the backward.
 * ds_scratch: same size as probs.  The effective seed is seed + *seed_dev (seed_dev may be NULL): a device-side
 * counter keeps the masks changing when the step is replayed from a CUDA graph. */
int ffsr_token_attention_train(const float* qkv, int B, int T, long HW, int E, float* ctx, float* probs, float drop_p,
                               unsigned long long seed, const unsigned long long* seed_dev, cudaStream_t stream);
int ffsr_token_attention_backward(const float* qkv, const float* probs, const float* dctx, int B, int T, long HW, int E,
                                  float* ds_scratch, float* dqkv, float drop_p, unsigned long long seed,
                                  const unsigned long long* seed_dev, cudaStream_t stream);

/* single stages of the LKA depthwise chain (kind 0: 5x5 pad 2 with input affine bn_k/bn_d,
 * 1: 1x21 pad 10, 2: 21x1 pad 10; w: [C][taps]) -- the backward runs them with reversed taps --
 * and their weight gradients dw[C][taps] (ACCUMULATED).  large_kernel_attention.py:98-100 */
int ffsr_dwconv_stage(const float* in, int N, int H, int W, int C, int kind, const float* w, const float* bn_k,
                      const float* bn_d, float* out, cudaStream_t stream);
size_t ffsr_dwconv_wgrad_workspace_bytes(int N, int H, int W, int C, int kind);
int ffsr_dwconv_wgrad(const float* in, const float* g, int N, int H, int W, int C, int kind, float* dw, void* ws,
                      size_t ws_bytes, cudaStream_t stream);

/* ---- fused training losses (forward value + gradient w.r.t. pred in one pass) --------------
 * pred / target / dpred: [P][H][W] fp32 planes (P = B*C of an NCHW-contiguous tensor).
 * Each call ADDS its partial sums into the fp64 accumulators and ADDS gscale * dLoss/dPred into
 * dpred (the caller zeroes both); gscale = loss weight / element count (see losses.py).  The partial sums
 * go through the workspace (size queries below) and are added in a fixed order.
 *   ffsr_loss_l1    L1Loss        src/losses/perceptual_loss.py:86-104      sum[0] = sum |p-t|
 *   ffsr_loss_swt   SWTLoss       :661-733, 797-813   sums8 = sum|cA|,|cH|,|cV|,|cD| for level 0 then level 1
 *   ffsr_loss_ssim  SSIMLoss      :225-291            sum[0] = sum of the SSIM map
 *   ffsr_loss_fft   FFTLoss       :533-598            sums2 = sum w*||P|-|T||, sum w*|angle P - angle T|
 *                   (H, W must factor into 2,3,5,7: training patches are 256 / 384) */
size_t ffsr_loss_l1_workspace_bytes(long n);
int ffsr_loss_l1(const float* pred, const float* target, long n, float gscale, double* sum, void* ws, size_t ws_bytes,
                 float* dpred, cudaStream_t stream);
size_t ffsr_loss_swt_workspace_bytes(int P, int H, int W);
int ffsr_loss_swt(const float* pred, const float* target, int P, int H, int W, float gscale, double* sums8, void* ws,
                  size_t ws_bytes, float* dpred, cudaStream_t stream);
size_t ffsr_loss_ssim_workspace_bytes(int P, int H, int W);
int ffsr_loss_ssim(const float* pred, const float* target, int P, int H, int W, float gscale, double* sum, void* ws,
                   size_t ws_bytes, float* dpred, cudaStream_t stream);
size_t ffsr_loss_fft_workspace_bytes(int P, int H, int W);
int ffsr_loss_fft(const float* pred, const float* target, int P, int H, int W, float gscale, double* sums2, void* ws,
                  size_t ws_bytes, float* dpred, cudaStream_t stream);

/* ---- fused optimizer step over a flat fp32 bucket ------------------------------------------
 * ffsr_sumsq: out[0] += sum g^2 (fp64) -- the global gradient norm of clip_grad_norm_ (train.py:344-348)
 * ffsr_adamw_ema_step: g' = g*grad_scale*min(1, max_norm/(grad_scale*sqrt(*gsumsq)+1e-6)) (no clipping when
 *   gsumsq is NULL or max_norm <= 0); torch.optim.AdamW update with bias correction for `step` (1-based)
 *   (train.py:847-853); ema = decay*ema + (1-decay)*p (checkpoint_manager.py:352-359; ema may be NULL).
 *   step_dev / lr_dev (optional device scalars): effective step = step + *step_dev, lr = *lr_dev -- the values
 *   that change between replays of a CUDA-graph-captured training step.
 * ffsr_sum_slots_ordered: out[i] = (...((s_0[i] + s_1[i]) + s_2[i]) ... + s_{M-1}[i]), s_m = slots + m*pitch, i < n
 *   (pitch >= n floats; out must not overlap the slots).  One fp32 rounding per add, in slot order: the result is
 *   what a float32 left fold gives and depends on nothing else (grid, block size, alignment).  16-byte loads when
 *   slots, out and pitch allow.  Sums the per-micro-batch gradient rows of the world-invariant training step. */
size_t ffsr_sumsq_workspace_bytes(long n);
int ffsr_sumsq(const float* g, long n, double* out, void* ws, size_t ws_bytes, cudaStream_t stream);
int ffsr_adamw_ema_step(float* p, const float* g, float* m, float* v, float* ema, long n, float lr, float beta1,
                        float beta2, float eps, float weight_decay, int step, const int* step_dev, const float* lr_dev,
                        const double* gsumsq, float grad_scale, float max_norm, float ema_decay, cudaStream_t stream);
int ffsr_sum_slots_ordered(const float* slots, int M, long n, long pitch, float* out, cudaStream_t stream);

/* ---- bf16 / tcgen05 training path ------------------------------------------------------------
 * ffsr_to_bf16_nhwc: strided fp32/bf16 view (NCHW or NHWC) -> dense bf16 channels-last with the channel
 *   pitch padded to Cpad (zeros), the operand format of the TMA-fed tensor-core kernels.
 * ffsr_conv2d_wgrad_tc: same contract as ffsr_conv2d_wgrad for bf16 channels-last x / dy whose strides are
 *   multiples of 16 bytes; tcgen05 MMAs with both operands MN-major (no transposed copies), per-CTA partial
 *   results in `ws` (ffsr_conv2d_wgrad_tc_workspace_bytes) reduced deterministically into dw. */
int ffsr_to_bf16_nhwc(const void* src, int src_dtype, long long sN, long long sY, long long sX, long long sC, int N,
                      int H, int W, int C, int Cpad, void* dst, cudaStream_t stream);
size_t ffsr_conv2d_wgrad_tc_workspace_bytes(int N, int H, int W, int Cin, int Cout, int ksize);   /* covers the bias sums */
int ffsr_conv2d_wgrad_tc(const ffsr_wgrad_params* p, void* ws, size_t ws_bytes, cudaStream_t stream);

/* F.interpolate(mode="bilinear", align_corners=False) on dense channels-last tensors ([N][h][w][C] -> [N][H][W][C])
 * and its adjoint (gradient w.r.t. the source, a gather with no atomics); any C, any scale factor, fp32 or bf16
 * (fp32 arithmetic).
 * hierarchical_fusion.py:156-186, enhanced_fusion_v2.py:735-791, edge_enhancement.py:208-250 */
int ffsr_bilinear_forward(const void* src, int N, int h, int w, int C, void* dst, int H, int W, int dtype,
                          cudaStream_t stream);
int ffsr_bilinear_backward(const void* gout, int N, int H, int W, int C, void* gin, int h, int w, int dtype,
                           cudaStream_t stream);

/* fused elementwise nodes of the training graph on dense channels-last data ([NP pixels][C]):
 *   gate_mul : out = y * g[p] (1-channel gate: hierarchical_fusion.py:25-43, edge_enhancement.py:118);
 *              backward dy = gout*g, dg[p] = sum_c gout*y
 *   axpby    : out = a + s1*b (+ s2*c), s1/s2 learnable device scalars, c optionally a channel slice with pixel
 *              pitch c_pitch (ResBlock scale, residual_weight_1_2/2_3: hierarchical_fusion.py:46-64, 178-199;
 *              LKABlock scale1/scale2: large_kernel_attention.py:143-149); backward db = s1*g, dc = s2*g,
 *              ds[0] += sum g*b, ds[1] += sum g*c (ACCUMULATED); da = g is passed through by the caller */
int ffsr_gate_mul_forward(const void* y, const float* g, long NP, int C, void* out, int dtype, cudaStream_t stream);
int ffsr_gate_mul_backward(const void* y, const float* g, const void* gout, long NP, int C, void* dy, float* dg, int dtype,
                           cudaStream_t stream);
int ffsr_axpby_forward(const void* a, const void* b, const void* c, long c_pitch, const float* s1, const float* s2, long NP,
                       int C, void* out, int dtype, cudaStream_t stream);
size_t ffsr_axpby_backward_workspace_bytes(long NP, int C);
int ffsr_axpby_backward(const void* g, const void* b, const void* c, long c_pitch, const float* s1, const float* s2, long NP,
                        int C, void* db, void* dc, float* ds, void* ws, size_t ws_bytes, int dtype, cudaStream_t stream);

/* Train mode of FFTDecomposition (multi_domain_frequency.py:352-385): low = irfft2(mask * rfft2(x), ortho) with the
 * sigmoid mask [H][W/2+1] supplied by the caller, and d(loss)/d(mask) from d(loss)/d(low) (sum over batch and
 * channels, Hermitian half counted twice).  x / low / dlow: [B][3][H][W] fp32; tables from ffsr_fft_twiddles. */
size_t ffsr_fft_lowpass_workspace_bytes(int B, int H, int W);
int ffsr_fft_lowpass(const float* x, int B, int H, int W, const float* mask, const void* tw_h, const void* tw_w, void* ws,
                     size_t ws_bytes, float* low, cudaStream_t stream);
int ffsr_fft_lowpass_backward(const float* x, const float* dlow, int B, int H, int W, const void* tw_h, const void* tw_w,
                              void* ws, size_t ws_bytes, float* dmask, cudaStream_t stream);

/* Cache-shard records -> batch tensors (the collate step of src/data/cached_dataset.py:135-282 on the device).
 * `records`: B raw records of `record_bytes` each, already in device memory (one H2D copy of the pinned staging buffer).
 * Every segment describes one tensor of a record, stored dense [C][h][w] as fp32 or fp16 at `src_offset`; it is written
 * to dst[b] (dense [C][Ho][Wo], fp32 or bf16) after sample b's dihedral transform tf_codes[b] (device array, NULL = none):
 * out[y][x] = in[sy][sx], (sy, sx) = (code & 1) ? (x, y) : (y, x); sy = h-1-sy if (code & 2); sx = w-1-sx if (code & 4)
 * -- the 8 compositions of the loader's hflip / vflip / rot90 (cached_dataset.py:236-282).  At most 16 segments. */
typedef struct ffsr_cache_segment {
  unsigned long long src_offset; /* byte offset inside a record, multiple of 16 */
  void* dst;                     /* [B][C][Ho][Wo] dense, 16-byte aligned */
  int C, h, w;                   /* stored shape */
  int src_dtype;                 /* FFSR_DT_F32 | FFSR_DT_F16 */
  int dst_dtype;                 /* FFSR_DT_F32 | FFSR_DT_BF16 */
  int reserved;
} ffsr_cache_segment;
int ffsr_cache_segment_size(void); /* sizeof(ffsr_cache_segment), for binding layout checks */
int ffsr_cache_unpack(const void* records, size_t record_bytes, int B, const ffsr_cache_segment* segs, int nseg,
                      const int* tf_codes, int sm_count, cudaStream_t stream);

/* (Shifted-)window multi-head attention of the DRCT-L expert (SURVEY 8f N1; src/models/drct/drct_arch.py:175-206,
 * 385-412): everything between the qkv and the proj Linear of one SwinTransformerBlock -- cyclic shift, window
 * partition, q k^T / sqrt(dh) + relative-position bias (+ the -100 shift mask), softmax, attn @ v, window merge and
 * reverse shift.  qkv: [B][H][W][3*C] channels-last with channel = which*C + head*dh + d; out: [B][H][W][C] at the
 * un-shifted pixel; bias_table: [(2*window-1)^2][heads] fp32.  H, W multiples of window (callers pad), window^2 <= 256,
 * dh <= 128.  First CUDA-core version (parity-tested on a B200, used by isr_b200.drct; not yet timed). */
int ffsr_window_attention(const void* qkv, int B, int H, int W, int C, int heads, int window, int shift,
                          const float* bias_table, void* out, int dtype, cudaStream_t stream);
/* Same on bf16 rows PADDED to qkv_pitch >= 3*C / out_pitch >= C elements (the DRCT channel counts are 4 mod 8; bf16
 * operands of the tcgen05 Linears need 16-byte row pitches).  NOT yet run on hardware (caller and test gated). */
int ffsr_window_attention_pitched(const void* qkv, long qkv_pitch, int B, int H, int W, int C, int heads, int window,
                                  int shift, const float* bias_table, void* out, long out_pitch, cudaStream_t stream);

/* Small ops of the DRCT-L expert forward (SURVEY 8f N1; src/models/drct/drct_arch.py), used by isr_b200.drct.
 *   layernorm_strided : nn.LayerNorm(C) (eps 1e-5) over the first C channels of rows with pitch x_pitch (:292-299, the
 *                       dense-growth buffer of an RDG; :769 final norm)
 *   leaky_relu        : in place on a channel slice (rows x C at `pitch`)  (:283, slope 0.2; :728, slope 0.01)
 *   pixel_shuffle2    : nn.PixelShuffle(2) on channels-last data, x [B][H][W][4C] -> y [B][2H][2W][C]  (:612-614)
 *   rgb_shift_in/out  : (x - mean) * img_range from planar fp32 [B][3][H][W] into channels-last rows of `pitch`
 *                       channels, and back (x / img_range + mean) (:778-779, :787); mean3_host is a HOST array of 3 */
/* window attention on tcgen05 (16 x 16 windows, bf16) over HEAD-PADDED qkv rows [q | k | v] x [heads][DP], DP =
 * ffsr_window_attention_head_pad(C / heads): the layout a qkv Linear produces when its weight rows are permuted and zero
 * padded on the host (isr_b200.drct).  Same operation as ffsr_window_attention (drct_arch.py:175-206, 385-412). */
int ffsr_window_attention_head_pad(int head_dim);
int ffsr_window_attention_headpadded(const void* qkv, int B, int H, int W, int C, int heads, int window, int shift,
                                     const float* bias_table, void* out, long out_pitch, cudaStream_t stream);
int ffsr_layernorm_strided(const void* x, long rows, int C, long x_pitch, const float* w, const float* b, void* y,
                           long y_pitch, int in_dtype, int out_dtype, cudaStream_t stream);
int ffsr_leaky_relu(void* x, long rows, int C, long pitch, float slope, int dtype, cudaStream_t stream);
int ffsr_pixel_shuffle2(const void* x, int B, int H, int W, int C, void* y, int dtype, cudaStream_t stream);
int ffsr_rgb_shift_in(const float* x, int B, int H, int W, const float* mean3_host, float range, void* y, int pitch, int dtype,
                      cudaStream_t stream);
int ffsr_rgb_shift_out(const void* x, int B, int H, int W, int pitch, const float* mean3_host, float range, float* y, int dtype,
                       cudaStream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* FFSR_B200_H */
