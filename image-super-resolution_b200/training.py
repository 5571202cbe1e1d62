"""Train-mode forward + backward of the fusion path on the sm_100a kernels.

``train_forward`` is what ``CompleteEnhancedFusionSR._run_pipeline`` runs when the module is
in ``.train()`` mode (reference: ``src/models/enhanced_fusion_v2.py:681-799`` driven by
``train.py:331-357``).  The differentiable graph is assembled from ``torch.autograd.Function``
nodes whose forward AND backward are ``libffsr_b200.so`` kernels:

  conv2d        ffsr_conv2d (forward; input gradient = same kernel, rotated weights),
                ffsr_conv2d_wgrad / ffsr_conv2d_wgrad_tc (+ bias column sums)
  conv_chain    bf16 mode: conv -> act -> conv ... as ONE node on the tcgen05 kernels (activation in the forward
                epilogue, act' in the input-gradient epilogue)
  act           ffsr_act_forward / ffsr_act_backward        (GELU / ReLU / sigmoid)
  bilinear      ffsr_bilinear_forward / ffsr_bilinear_backward
  gate_mul      ffsr_gate_mul_forward / ffsr_gate_mul_backward     (1-channel gate x C channels)
  axpby         ffsr_axpby_forward / ffsr_axpby_backward           (x + s1*a (+ s2*b), learnable scalars)
  blur_pool     ffsr_blur_pool / ffsr_blur_pool_backward           (Laplacian pyramid reduction)
  fft_lowpass   ffsr_fft_lowpass / ffsr_fft_lowpass_backward       (learnable FFT mask, dense-DFT kernels)
  batchnorm     ffsr_bn_stats / ffsr_bn_apply / ffsr_bn_backward   (batch statistics per LKABlock call)
  layernorm     ffsr_layernorm / ffsr_layernorm_backward
  token_attn    ffsr_token_attention_train / ffsr_token_attention_backward  (dropout on the probabilities)
  dwconv        ffsr_dwconv_stage / ffsr_dwconv_wgrad       (LKA 5x5, 1x21, 21x1)

PyTorch autograd is the plumbing between those nodes: tensor bookkeeping, concatenation, dtype
casts and the 3/4-channel elementwise blends (softmax over experts, gate normalisation, image
modulation) are ordinary CUDA tensor ops (DESIGN.md section 4b lists them with their time share).
There is no CPU path: CPU tensors raise.

Tensors are logical NCHW in channels-last memory ([N][H][W][C]), the layout every kernel of
the library works in.
"""
from __future__ import annotations

import contextlib
import ctypes as C
from typing import Dict, List, Optional

import torch

from . import _cabi as K

EXPERT_ORDER = ("drct", "grl", "nafnet", "mamba")
_BN_EPS = 1e-5
CL = torch.channels_last


def _lib():
    return K.load()


def _S(t: torch.Tensor):
    return C.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def _ck(rc, what):
    if rc != 0:
        K.check(rc, what)


def _is_cl(t: torch.Tensor) -> bool:
    return t.permute(0, 2, 3, 1).is_contiguous()


def _cl(t: torch.Tensor) -> torch.Tensor:
    """Dense channels-last copy (no-op when the memory already is [N][H][W][C])."""
    if _is_cl(t):
        return t
    out = torch.empty(t.shape, device=t.device, dtype=t.dtype).contiguous(memory_format=CL)
    if not _is_cl(out):                       # C == 1 or H == W == 1: layouts coincide
        out = torch.empty_strided(t.shape, _cl_strides(t.shape), device=t.device, dtype=t.dtype)
    out.copy_(t)
    return out


def _cl_strides(shape):
    N, Cc, H, W = shape
    return (H * W * Cc, 1, W * Cc, Cc)


def _empty_cl(N, Cc, H, W, dev, dtype=torch.float32) -> torch.Tensor:
    return torch.empty_strided((N, Cc, H, W), (H * W * Cc, 1, W * Cc, Cc), device=dev, dtype=dtype)


def _empty_cl_padded(N, Cc, H, W, dev, dtype) -> torch.Tensor:
    """Channels-last [N,Cc,H,W] view of a buffer whose pixel pitch is padded to a multiple of 8 channels: keeps the
    16-byte vector stores of the conv epilogue aligned when Cc is e.g. 76 (a 152-byte bf16 pitch falls back to 2-byte
    stores: the stage-3 input gradient took 0.99 ms instead of ~0.4 ms)."""
    cp = (Cc + 7) // 8 * 8
    if cp == Cc:
        return _empty_cl(N, Cc, H, W, dev, dtype)
    buf = torch.empty(N, H, W, cp, device=dev, dtype=dtype)
    return buf.permute(0, 3, 1, 2)[:, :Cc]


def _zeros(shape, dev, dtype=torch.float32):
    return torch.zeros(shape, device=dev, dtype=dtype)


def _dt(t):
    return K.DT_BF16 if t.dtype == torch.bfloat16 else K.DT_F32


def _ws(nbytes: int, dev) -> torch.Tensor:
    """Workspace for the per-block partial sums of a reduction kernel (fixed-order, atomic-free: the training step is
    bitwise reproducible).  The kernels write every byte they read, so it needs no initialisation."""
    return torch.empty(max(int(nbytes), 16), device=dev, dtype=torch.uint8)


# --------------------------------------------------------------------------------------
# convolution
# --------------------------------------------------------------------------------------
def _launch_conv(x: torch.Tensor, wp: torch.Tensor, bias: Optional[torch.Tensor], out: torch.Tensor, ks: int):
    """x: [N,Cin,H,W] any strides (fp32); wp: [ks*ks][Cin][Cout] fp32; out: channels-last [N,Cout,H,W]."""
    N, Cin, H, W = x.shape
    Cout = out.shape[1]
    p = K.ConvParams()
    p.inp = x.data_ptr()
    p.in_sN, p.in_sC, p.in_sY, p.in_sX = x.stride(0), x.stride(1), x.stride(2), x.stride(3)
    if Cin == 1:
        p.in_sC = 1
    p.N, p.H, p.W, p.Cin, p.Cout, p.ksize = N, H, W, Cin, Cout, ks
    p.w = wp.data_ptr()
    p.bias = bias.data_ptr() if bias is not None else None
    p.groups = 1
    p.out = out.data_ptr()
    p.out_sN, p.out_sY, p.out_sX = H * W * Cout, W * Cout, Cout
    p.act, p.epi = K.ACT_NONE, K.EPI_PLAIN
    p.flags = K.CONV_MULTI_ISSUE
    p.sa = p.sb = 1.0
    p.in_dtype = p.out_dtype = p.w_dtype = K.DT_F32
    _ck(_lib().ffsr_conv2d(C.byref(p), _S(x)), "conv2d")


class _Conv2d(torch.autograd.Function):
    """nn.Conv2d (1x1 / 3x3, stride 1, zero pad k//2)."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        co, ci, kh, kw = weight.shape
        assert kh == kw and kh in (1, 3) and x.shape[1] == ci, (tuple(weight.shape), tuple(x.shape))
        x = x if x.dtype == torch.float32 else x.float()
        wp = weight.detach().permute(2, 3, 1, 0).reshape(kh * kw, ci, co).contiguous()
        N, _, H, W = x.shape
        out = _empty_cl(N, co, H, W, x.device)
        b = bias.detach().contiguous() if bias is not None else None
        _launch_conv(x, wp, b, out, kh)
        ctx.save_for_backward(x, weight)
        ctx.has_bias = bias is not None
        return out

    @staticmethod
    def backward(ctx, gy):
        x, weight = ctx.saved_tensors
        co, ci, kh, kw = weight.shape
        N, _, H, W = x.shape
        gy = _cl(gy)
        dx = None
        if ctx.needs_input_grad[0]:
            wr = weight.detach().flip(2, 3).permute(2, 3, 0, 1).reshape(kh * kw, co, ci).contiguous()
            dx = _empty_cl(N, ci, H, W, x.device)
            _launch_conv(gy, wr, None, dx, kh)
        dw = db = None
        if ctx.needs_input_grad[1] or (ctx.has_bias and ctx.needs_input_grad[2]):
            dwp = _zeros((kh * kw, ci, co), x.device)
            dbp = _zeros((co,), x.device) if ctx.has_bias else None
            p = K.WgradParams()
            p.x = x.data_ptr()
            p.x_sN, p.x_sC, p.x_sY, p.x_sX = x.stride(0), x.stride(1), x.stride(2), x.stride(3)
            if ci == 1:
                p.x_sC = 1
            p.x_dtype = K.DT_F32
            p.dy = gy.data_ptr()
            p.dy_sN, p.dy_sY, p.dy_sX = H * W * co, W * co, co
            p.dy_dtype = K.DT_F32
            p.N, p.H, p.W, p.Cin, p.Cout, p.ksize = N, H, W, ci, co, kh
            p.dw = dwp.data_ptr()
            p.dbias = dbp.data_ptr() if dbp is not None else None
            lib = _lib()
            ws = _ws(lib.ffsr_conv2d_wgrad_workspace_bytes(N, H, W, ci, co, kh), x.device)
            _ck(lib.ffsr_conv2d_wgrad(C.byref(p), ws.data_ptr(), ws.numel(), _S(x)), "conv2d_wgrad")
            dw = dwp.view(kh, kw, ci, co).permute(3, 2, 0, 1)
            db = dbp
        return dx, dw, db


# ---- tcgen05 path: bf16 operands (channel pitch padded to 8 for TMA), fp32 accumulation --------------
def _bf16_operand(x: torch.Tensor):
    """-> (buffer [N,H,W,Cpad] bf16 contiguous, C).  Zero-copy when x already is bf16 channels-last with a
    16-byte-multiple pixel pitch; otherwise one cast/pad kernel."""
    N, Cc, H, W = x.shape
    if x.dtype == torch.bfloat16 and x.stride(1) == 1 and Cc > 1:
        sN, sY, sX = x.stride(0), x.stride(2), x.stride(3)
        if sX % 8 == 0 and sX >= Cc and sY == W * sX and sN == H * W * sX and x.data_ptr() % 16 == 0:
            return torch.as_strided(x, (N, H, W, sX), (sN, sY, sX, 1)), Cc
    cpad = (Cc + 7) // 8 * 8
    buf = torch.empty(N, H, W, cpad, device=x.device, dtype=torch.bfloat16)
    if x.dtype == torch.float32 and Cc >= 16 and x.is_contiguous() and N <= 65535:
        # NCHW planes (cached expert features): tiled shared-memory transpose; pad channels are never read by TMA
        _ck(_lib().ffsr_nchw_to_nhwc_bf16(x.data_ptr(), N, Cc, H * W, buf.data_ptr(), H * W * cpad, cpad, _S(x)),
            "nchw_to_nhwc_bf16")
        return buf, Cc
    sC = x.stride(1) if Cc > 1 else 1
    _ck(_lib().ffsr_to_bf16_nhwc(x.data_ptr(), _dt(x), x.stride(0), x.stride(2), x.stride(3), sC, N, H, W, Cc, cpad,
                                 buf.data_ptr(), _S(x)), "to_bf16_nhwc")
    return buf, Cc


def _pack_tc(wp: torch.Tensor) -> torch.Tensor:
    """[taps][Cin][Cout] fp32 -> [taps][CoutPad][CinPad] bf16 K-major (layout of ffsr_conv2d's tcgen05 path)."""
    taps, ci, co = wp.shape
    cip = (ci + 63) // 64 * 64
    cop = (co + 15) // 16 * 16
    if cop > 128:
        cop = (cop + 127) // 128 * 128
    out = torch.zeros(taps, cop, cip, device=wp.device, dtype=torch.bfloat16)
    out[:, :co, :ci] = wp.transpose(1, 2)
    return out


def _launch_conv_tc(xb: torch.Tensor, Cin: int, wtc: torch.Tensor, bias, out: torch.Tensor, ks: int,
                    act: int = 0, out2: Optional[torch.Tensor] = None, actgrad_z: Optional[torch.Tensor] = None):
    """xb: [N,H,W,Cpad] bf16; out: channels-last [N,Cout,H,W] fp32 or bf16.
    act + out2: out = act(conv), out2 = bf16 pre-activation.  actgrad_z: out = conv * act'(actgrad_z)."""
    N, H, W, cpad = xb.shape
    Cout = out.shape[1]
    p = K.ConvParams()
    p.inp = xb.data_ptr()
    p.in_sN, p.in_sY, p.in_sX, p.in_sC = H * W * cpad, W * cpad, cpad, 1
    p.N, p.H, p.W, p.Cin, p.Cout, p.ksize = N, H, W, Cin, Cout, ks
    p.w = wtc.data_ptr()
    p.bias = bias.data_ptr() if bias is not None else None
    p.groups = 1
    p.out = out.data_ptr()
    p.out_sN, p.out_sY, p.out_sX = out.stride(0), out.stride(2), out.stride(3)      # dense or padded-pitch channels-last
    p.act, p.epi = act, K.EPI_PLAIN
    p.flags = K.CONV_MULTI_ISSUE    # tcgen05 launches: up to three MMA-issuing warps, as at inference
    p.sa = p.sb = 1.0
    p.in_dtype, p.w_dtype = K.DT_BF16, K.DT_BF16
    p.out_dtype = _dt(out)
    if out2 is not None:
        p.out2 = out2.data_ptr()
    if actgrad_z is not None:                 # z: dense channels-last [N,Cout,H,W]
        p.epi = K.EPI_ACTGRAD
        p.r1 = actgrad_z.data_ptr()
        p.r1_sN, p.r1_sY, p.r1_sX = H * W * Cout, W * Cout, Cout
        p.r1_dtype = _dt(actgrad_z)
    _ck(_lib().ffsr_conv2d(C.byref(p), _S(xb)), "conv2d(tc)")


class _Conv2dTC(torch.autograd.Function):
    """nn.Conv2d on the tcgen05 kernels: forward and input gradient through ffsr_conv2d's bf16 path,
    weight gradient through ffsr_conv2d_wgrad_tc.  Master weights / weight gradients stay fp32."""

    @staticmethod
    def forward(ctx, x, weight, bias, out_bf16):
        co, ci, kh, kw = weight.shape
        assert kh == kw and kh in (1, 3) and x.shape[1] == ci, (tuple(weight.shape), tuple(x.shape))
        xb, _ = _bf16_operand(x)
        N, _, H, W = x.shape
        wtc = _pack_tc(weight.detach().permute(2, 3, 1, 0).reshape(kh * kw, ci, co))
        out = _empty_cl(N, co, H, W, x.device, torch.bfloat16 if out_bf16 else torch.float32)
        b = bias.detach().float().contiguous() if bias is not None else None
        _launch_conv_tc(xb, ci, wtc, b, out, kh)
        ctx.save_for_backward(xb, weight)
        ctx.has_bias = bias is not None
        ctx.x_dtype = x.dtype
        return out

    @staticmethod
    def backward(ctx, gy):
        xb, weight = ctx.saved_tensors
        co, ci, kh, kw = weight.shape
        N, H, W, cpad = xb.shape
        gb, _ = _bf16_operand(gy)
        dx = None
        if ctx.needs_input_grad[0]:
            wr = _pack_tc(weight.detach().flip(2, 3).permute(2, 3, 0, 1).reshape(kh * kw, co, ci))
            dx = _empty_cl_padded(N, ci, H, W, xb.device, ctx.x_dtype if ctx.x_dtype == torch.bfloat16 else torch.float32)
            _launch_conv_tc(gb, co, wr, None, dx, kh)
        dw = db = None
        if ctx.needs_input_grad[1] or (ctx.has_bias and ctx.needs_input_grad[2]):
            dwp, db = _wgrad_tc(xb, gb, ci, co, kh, ctx.has_bias)
            dw = dwp.view(kh, kw, ci, co).permute(3, 2, 0, 1)
        return dx, dw, db, None


def _wgrad_tc(xb, gb, ci, co, ks, has_bias):
    """fp32 packed weight gradient [ks*ks][ci][co] (+ bias gradient) from bf16 operands xb / gb ([N,H,W,pitch])."""
    lib = _lib()
    N, H, W, cpad = xb.shape
    gpad = gb.shape[3]
    dwp = _zeros((ks * ks, ci, co), xb.device)
    dbp = _zeros((co,), xb.device) if has_bias else None
    p = K.WgradParams()
    p.x = xb.data_ptr()
    p.x_sN, p.x_sY, p.x_sX, p.x_sC = H * W * cpad, W * cpad, cpad, 1
    p.x_dtype = K.DT_BF16
    p.dy = gb.data_ptr()
    p.dy_sN, p.dy_sY, p.dy_sX = H * W * gpad, W * gpad, gpad
    p.dy_dtype = K.DT_BF16
    p.N, p.H, p.W, p.Cin, p.Cout, p.ksize = N, H, W, ci, co, ks
    p.dw = dwp.data_ptr()
    p.dbias = dbp.data_ptr() if dbp is not None else None
    nb = lib.ffsr_conv2d_wgrad_tc_workspace_bytes(N, H, W, ci, co, ks)
    ws = _ws(nb, xb.device)
    _ck(lib.ffsr_conv2d_wgrad_tc(C.byref(p), ws.data_ptr(), nb, _S(xb)), "conv2d_wgrad_tc")
    return dwp, dbp


class _ConvChainTC(torch.autograd.Function):
    """conv -> act -> conv -> act -> ... on the tcgen05 kernels as ONE autograd node.

    Forward: one launch per layer; the activation runs in the conv epilogue, which also stores the bf16
    pre-activation.  Backward: per layer one weight-gradient launch and one input-gradient launch whose epilogue
    multiplies by act'(pre-activation of the previous layer) (FFSR_EPI_ACTGRAD) -- no separate activation passes
    over the HR feature maps in either direction.  acts[i] is the activation after layer i (0 = none)."""

    @staticmethod
    def forward(ctx, x, acts, out_bf16, *wb):
        L = len(acts)
        cur, _ = _bf16_operand(x)
        N, _, H, W = x.shape
        ops, zs = [], []
        y = None
        for i in range(L):
            w, b = wb[2 * i], wb[2 * i + 1]
            if w.dim() == 2:
                w = w[:, :, None, None]
            co, ci, kh, _ = w.shape
            wtc = _pack_tc(w.detach().permute(2, 3, 1, 0).reshape(kh * kh, ci, co))
            bb = b.detach().float().contiguous() if b is not None else None
            last = i == L - 1
            odt = (torch.bfloat16 if out_bf16 else torch.float32) if last else torch.bfloat16
            y = _empty_cl(N, co, H, W, x.device, odt)
            z = _empty_cl(N, co, H, W, x.device, torch.bfloat16) if acts[i] != K.ACT_NONE else None
            _launch_conv_tc(cur, ci, wtc, bb, y, kh, acts[i], z)
            ops.append(cur)
            zs.append(z)
            if not last:
                assert co % 8 == 0, "intermediate channels of a fused conv chain must be a multiple of 8"
                cur = y.permute(0, 2, 3, 1)                      # [N,H,W,co] bf16 contiguous: next TMA operand
        ctx.save_for_backward(*ops, *[z for z in zs if z is not None], *[t for t in wb if t is not None])
        ctx.meta = (acts, [z is not None for z in zs], [t is not None for t in wb], x.dtype)
        return y

    @staticmethod
    def backward(ctx, gy):
        acts, zmask, wbmask, x_dtype = ctx.meta
        L = len(acts)
        saved = list(ctx.saved_tensors)
        ops = saved[:L]
        nz = sum(zmask)
        zlist = saved[L:L + nz]
        rest = saved[L + nz:]
        zs, k = [], 0
        for m_ in zmask:
            zs.append(zlist[k] if m_ else None)
            k += 1 if m_ else 0
        wb, k = [], 0
        for m_ in wbmask:
            wb.append(rest[k] if m_ else None)
            k += 1 if m_ else 0
        grads = [None] * (2 * L)
        g = gy
        if acts[L - 1] != K.ACT_NONE:                              # chain ends with an activation
            z = zs[L - 1]
            g2 = torch.empty_like(z)
            gsrc = g if (g.dtype == z.dtype and g.stride() == z.stride()) else torch.empty_like(z).copy_(g)
            _ck(_lib().ffsr_act_backward(z.data_ptr(), gsrc.data_ptr(), g2.data_ptr(), z.numel(), acts[L - 1], _dt(z), _S(z)),
                "act_backward")
            g = g2
        dx = None
        for i in range(L - 1, -1, -1):
            w, b = wb[2 * i], wb[2 * i + 1]
            w4 = w[:, :, None, None] if w.dim() == 2 else w
            co, ci, kh, _ = w4.shape
            gb, _ = _bf16_operand(g)
            xb = ops[i]
            N, H, W, _ = xb.shape
            need_w = ctx.needs_input_grad[3 + 2 * i]
            need_b = b is not None and ctx.needs_input_grad[4 + 2 * i]
            if need_w or need_b:
                dwp, dbp = _wgrad_tc(xb, gb, ci, co, kh, b is not None)
                dw = dwp.view(kh, kh, ci, co).permute(3, 2, 0, 1)
                grads[2 * i] = dw.reshape(w.shape) if w.dim() == 2 else dw
                grads[2 * i + 1] = dbp
            if i > 0 or ctx.needs_input_grad[0]:
                wr = _pack_tc(w4.detach().flip(2, 3).permute(2, 3, 0, 1).reshape(kh * kh, co, ci))
                if i > 0:
                    g = _empty_cl(N, ci, H, W, xb.device, torch.bfloat16)
                    _launch_conv_tc(gb, co, wr, None, g, kh, acts[i - 1], None, zs[i - 1])
                else:
                    dx = _empty_cl_padded(N, ci, H, W, xb.device, torch.bfloat16 if x_dtype == torch.bfloat16 else torch.float32)
                    _launch_conv_tc(gb, co, wr, None, dx, kh)
        return (dx, None, None, *grads)


def conv_chain(x, layers, tc: bool, out_bf16: bool = False):
    """layers: [(weight, bias, act)], act in {K.ACT_NONE, K.ACT_GELU, K.ACT_RELU, K.ACT_SIGMOID}.
    tc=True: one fused tcgen05 node; tc=False: fp32 conv / activation nodes in sequence."""
    if tc:
        flat = []
        for w, b, _ in layers:
            flat += [w, b]
        return _ConvChainTC.apply(x, tuple(a for _, _, a in layers), out_bf16, *flat)
    y = x
    for w, b, a in layers:
        y = conv2d(y, w, b)
        if a != K.ACT_NONE:
            y = _Act.apply(y, a)
    return y


def conv2d(x, weight, bias=None, tc: bool = False, out_bf16: bool = False):
    """tc=False: fp32 CUDA-core kernels; tc=True: tcgen05 kernels (bf16 operands), output fp32 or bf16."""
    if weight.dim() == 2:                      # nn.Linear weight [out, in] == 1x1 conv
        weight = weight[:, :, None, None]
    if tc:
        return _Conv2dTC.apply(x, weight, bias, out_bf16)
    return _Conv2d.apply(x, weight, bias)


def conv_mod(x, mod, tc: bool = False, out_bf16: bool = False):
    return conv2d(x, mod.weight, mod.bias, tc, out_bf16)


# --------------------------------------------------------------------------------------
# pointwise activations
# --------------------------------------------------------------------------------------
class _Act(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, kind):
        x = x if x.is_contiguous() or _is_cl(x) else x.contiguous()
        y = torch.empty_like(x)               # preserves the (dense) strides
        _ck(_lib().ffsr_act_forward(x.data_ptr(), y.data_ptr(), x.numel(), kind, _dt(x), _S(x)), "act_forward")
        ctx.save_for_backward(x)
        ctx.kind = kind
        return y

    @staticmethod
    def backward(ctx, gy):
        (x,) = ctx.saved_tensors
        if gy.stride() != x.stride() or gy.dtype != x.dtype:
            g2 = torch.empty_like(x)
            g2.copy_(gy)
            gy = g2
        dx = torch.empty_like(x)
        _ck(_lib().ffsr_act_backward(x.data_ptr(), gy.data_ptr(), dx.data_ptr(), x.numel(), ctx.kind, _dt(x), _S(x)),
            "act_backward")
        return dx, None


def gelu(x):
    return _Act.apply(x, K.ACT_GELU)


def relu(x):
    return _Act.apply(x, K.ACT_RELU)


def sigmoid(x):
    return _Act.apply(x, K.ACT_SIGMOID)


# --------------------------------------------------------------------------------------
# fused few-pass elementwise nodes
# --------------------------------------------------------------------------------------
class _GateMul(torch.autograd.Function):
    """out = y * g, g a 1-channel fp32 map broadcast over the channels of y."""

    @staticmethod
    def forward(ctx, y, g):
        y = _cl(y)
        N, Cc, H, W = y.shape
        g = g.float().contiguous()                       # [N,1,H,W]: layout-agnostic
        out = torch.empty_like(y)
        _ck(_lib().ffsr_gate_mul_forward(y.data_ptr(), g.data_ptr(), N * H * W, Cc, out.data_ptr(), _dt(y), _S(y)), "gate_mul_forward")
        ctx.save_for_backward(y, g)
        return out

    @staticmethod
    def backward(ctx, gout):
        y, g = ctx.saved_tensors
        N, Cc, H, W = y.shape
        if gout.dtype != y.dtype or gout.stride() != y.stride():
            gout = torch.empty_like(y).copy_(gout)
        dy = torch.empty_like(y)
        dg = torch.empty_like(g)
        _ck(_lib().ffsr_gate_mul_backward(y.data_ptr(), g.data_ptr(), gout.data_ptr(), N * H * W, Cc, dy.data_ptr(),
                                          dg.data_ptr(), _dt(y), _S(y)), "gate_mul_backward")
        return dy, dg


def gate_mul(y, g):
    if y.shape[1] % 4 != 0:
        return y * g.to(y.dtype)
    return _GateMul.apply(y, g)


class _Axpby(torch.autograd.Function):
    """out = a + s1*b (+ s2*c): learnable scalar-weighted residual sums in one pass each way."""

    @staticmethod
    def forward(ctx, a, b, s1, c, s2):
        a = _cl(a)
        b = _cl(b) if b.dtype == a.dtype else _cl(b.to(a.dtype))
        N, Cc, H, W = a.shape
        cp, cptr = 0, None
        if c is not None:
            if c.dtype != a.dtype:
                c = c.to(a.dtype)
            ok = c.stride(1) == 1 and c.stride(2) == W * c.stride(3) and c.stride(0) == H * W * c.stride(3)
            if not ok:
                c = _cl(c)
            cp, cptr = c.stride(3), c.data_ptr()
        out = torch.empty_like(a)
        s1c = s1.detach().reshape(1).float()
        s2c = s2.detach().reshape(1).float() if c is not None else None
        _ck(_lib().ffsr_axpby_forward(a.data_ptr(), b.data_ptr(), cptr, cp, s1c.data_ptr(),
                                      s2c.data_ptr() if s2c is not None else None, N * H * W, Cc, out.data_ptr(), _dt(a), _S(a)),
            "axpby_forward")
        ctx.save_for_backward(b, c if c is not None else b, s1c, s2c if s2c is not None else s1c)
        ctx.has_c = c is not None
        ctx.c_pitch = cp
        ctx.shape = (N, Cc, H, W)
        return out

    @staticmethod
    def backward(ctx, g):
        b, c, s1c, s2c = ctx.saved_tensors
        N, Cc, H, W = ctx.shape
        if g.dtype != b.dtype or g.stride() != b.stride():
            g = torch.empty_like(b).copy_(g)
        db = torch.empty_like(b)
        dc = torch.empty_like(b) if ctx.has_c else None
        ds = _zeros((2,), b.device)
        lib = _lib()
        ws = _ws(lib.ffsr_axpby_backward_workspace_bytes(N * H * W, Cc), b.device)
        _ck(lib.ffsr_axpby_backward(g.data_ptr(), b.data_ptr(), c.data_ptr() if ctx.has_c else None, ctx.c_pitch,
                                    s1c.data_ptr(), s2c.data_ptr() if ctx.has_c else None, N * H * W, Cc, db.data_ptr(),
                                    dc.data_ptr() if dc is not None else None, ds.data_ptr(), ws.data_ptr(), ws.numel(),
                                    _dt(b), _S(b)), "axpby_backward")
        return g, db, ds[0].reshape(()), dc, (ds[1].reshape(()) if ctx.has_c else None)


def axpby(a, b, s1, c=None, s2=None):
    return _Axpby.apply(a, b, s1, c, s2)


# --------------------------------------------------------------------------------------
# BatchNorm2d, train mode, G statistic groups (group-major images)
# --------------------------------------------------------------------------------------
class _BatchNormTrain(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias, G):
        x = _cl(x)
        N, Cc, H, W = x.shape
        assert N % G == 0
        R = (N // G) * H * W
        dev = x.device
        s = _zeros((2, G, Cc), dev, torch.float64)
        lib = _lib()
        ws = _ws(lib.ffsr_bn_stats_workspace_bytes(G, R, Cc), dev)
        _ck(lib.ffsr_bn_stats(x.data_ptr(), G, R, Cc, s[0].data_ptr(), s[1].data_ptr(), ws.data_ptr(), ws.numel(), _S(x)),
            "bn_stats")
        mean64 = s[0] / R
        var64 = (s[1] / R - mean64 * mean64).clamp_(min=0.0)
        mean = mean64.float()
        var = var64.float()
        rstd = torch.rsqrt(var + _BN_EPS)
        y = torch.empty_like(x)
        w = weight.detach().contiguous()
        b = bias.detach().contiguous()
        _ck(lib.ffsr_bn_apply(x.data_ptr(), G, R, Cc, mean.data_ptr(), rstd.data_ptr(), w.data_ptr(), b.data_ptr(),
                              y.data_ptr(), _S(x)), "bn_apply")
        ctx.save_for_backward(x, mean, rstd, w)
        ctx.G, ctx.R = G, R
        ctx.mark_non_differentiable(mean, var)
        return y, mean, var

    @staticmethod
    def backward(ctx, gy, _gm, _gv):
        x, mean, rstd, w = ctx.saved_tensors
        G, R = ctx.G, ctx.R
        Cc = x.shape[1]
        gy = _cl(gy)
        red = _zeros((2, G, Cc), x.device)
        dx = torch.empty_like(x)
        lib = _lib()
        ws = _ws(lib.ffsr_bn_backward_workspace_bytes(G, R, Cc), x.device)
        _ck(lib.ffsr_bn_backward(x.data_ptr(), gy.data_ptr(), G, R, Cc, mean.data_ptr(), rstd.data_ptr(),
                                 w.data_ptr(), red[0].data_ptr(), red[1].data_ptr(), dx.data_ptr(), ws.data_ptr(), ws.numel(),
                                 _S(x)), "bn_backward")
        return dx, red[1].sum(0), red[0].sum(0), None


class _BatchNormEval(torch.autograd.Function):
    """nn.BatchNorm2d in eval mode over the running statistics (constants of the graph): gradients to x, weight and
    bias; the running buffers and num_batches_tracked are not touched."""

    @staticmethod
    def forward(ctx, x, weight, bias, mean, rstd):
        x = _cl(x)
        N, Cc, H, W = x.shape
        y = torch.empty_like(x)
        w = weight.detach().contiguous()
        b = bias.detach().contiguous()
        _ck(_lib().ffsr_bn_apply(x.data_ptr(), 1, N * H * W, Cc, mean.data_ptr(), rstd.data_ptr(), w.data_ptr(), b.data_ptr(),
                                 y.data_ptr(), _S(x)), "bn_apply(eval)")
        ctx.save_for_backward(x, mean, rstd, w)
        return y

    @staticmethod
    def backward(ctx, gy):
        x, mean, rstd, w = ctx.saved_tensors
        N, Cc, H, W = x.shape
        R = N * H * W
        gy = _cl(gy)
        red = _zeros((2, Cc), x.device)
        dx = torch.empty_like(x)
        lib = _lib()
        ws = _ws(lib.ffsr_bn_backward_workspace_bytes(1, R, Cc), x.device)
        _ck(lib.ffsr_bn_eval_backward(x.data_ptr(), gy.data_ptr(), R, Cc, mean.data_ptr(), rstd.data_ptr(), w.data_ptr(),
                                      red[0].data_ptr(), red[1].data_ptr(), dx.data_ptr(), ws.data_ptr(), ws.numel(), _S(x)),
            "bn_eval_backward")
        return dx, red[1], red[0], None, None


def batchnorm_eval(x, bn: torch.nn.BatchNorm2d):
    mean = bn.running_mean.detach().float().contiguous()
    rstd = torch.rsqrt(bn.running_var.detach().float() + _BN_EPS)
    return _BatchNormEval.apply(x, bn.weight, bn.bias, mean, rstd)


def batchnorm_train(x, bn: torch.nn.BatchNorm2d, G: int, stats_sink: list):
    """Batch-statistic BN over G groups; the per-group (mean, biased var, n) are appended to
    ``stats_sink`` so the caller can fold the running-stat EMA in call order."""
    y, mean, var = _BatchNormTrain.apply(x, bn.weight, bn.bias, G)
    n = x.numel() // (x.shape[1] * G)
    stats_sink.append((bn, mean, var, n))
    return y


@torch.no_grad()
def fold_running_stats(records):
    """nn.BatchNorm2d side effect (momentum 0.1, unbiased variance, counter += 1 per call),
    applied for the G sequential LKABlock calls of one forward.  records: [(bn, mean[G,C], var[G,C], n)]
    in call order per BN module (large_kernel_attention.py:84,128,131).

    The records of M micro-batches, concatenated in micro-batch order, fold in one call: each module's G' = M*G
    groups go through the same closed form and ``num_batches_tracked`` grows by M*G, as M sequential forwards would
    leave it.  With one micro-batch this is the per-forward fold."""
    by_mod: Dict[int, list] = {}
    for bn, mean, var, n in records:
        by_mod.setdefault(id(bn), [bn, [], [], n])
        by_mod[id(bn)][1].append(mean)
        by_mod[id(bn)][2].append(var)
    for bn, means, vars_, n in by_mod.values():
        mean = torch.cat(means, 0)
        var = torch.cat(vars_, 0) * (n / max(n - 1, 1))
        G = mean.shape[0]
        mom = bn.momentum if bn.momentum is not None else 0.1
        wts = mom * (1.0 - mom) ** torch.arange(G - 1, -1, -1, device=mean.device, dtype=torch.float32)
        keep = (1.0 - mom) ** G
        bn.running_mean.mul_(keep).add_((wts[:, None] * mean).sum(0))
        bn.running_var.mul_(keep).add_((wts[:, None] * var).sum(0))
        bn.num_batches_tracked.add_(G)


# --------------------------------------------------------------------------------------
# LayerNorm over channels of a channels-last tensor
# --------------------------------------------------------------------------------------
class _LayerNorm(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias):
        x = _cl(x)
        N, E, H, W = x.shape
        rows = N * H * W
        y = torch.empty_like(x)
        w = weight.detach().contiguous()
        b = bias.detach().contiguous()
        _ck(_lib().ffsr_layernorm(x.data_ptr(), rows, E, w.data_ptr(), b.data_ptr(), y.data_ptr(), 0, _S(x)), "layernorm")
        ctx.save_for_backward(x, w)
        return y

    @staticmethod
    def backward(ctx, gy):
        x, w = ctx.saved_tensors
        N, E, H, W = x.shape
        gy = _cl(gy)
        dx = torch.empty_like(x)
        dwb = _zeros((2, E), x.device)
        lib = _lib()
        ws = _ws(lib.ffsr_layernorm_backward_workspace_bytes(N * H * W, E), x.device)
        _ck(lib.ffsr_layernorm_backward(x.data_ptr(), gy.data_ptr(), N * H * W, E, w.data_ptr(), dx.data_ptr(),
                                        dwb[0].data_ptr(), dwb[1].data_ptr(), ws.data_ptr(), ws.numel(), _S(x)),
            "layernorm_backward")
        return dx, dwb[0], dwb[1]


def layernorm(x, ln):
    return _LayerNorm.apply(x, ln.weight, ln.bias)


# --------------------------------------------------------------------------------------
# token attention core
# --------------------------------------------------------------------------------------
class _TokenAttention(torch.autograd.Function):
    """qkv: [B*T, 3E, H, W] channels-last (memory [B][T][HW][3E]) -> ctx [B*T, E, H, W]."""

    @staticmethod
    def forward(ctx, qkv, B, T, drop_p, seed, seed_dev=None):
        qkv = _cl(qkv)
        BT, E3, H, W = qkv.shape
        E = E3 // 3
        HW = H * W
        out = _empty_cl(BT, E, H, W, qkv.device)
        probs = torch.empty(B * HW * (E // 16) * T * T, device=qkv.device, dtype=torch.float32)
        sd_ptr = seed_dev.data_ptr() if (seed_dev is not None and drop_p > 0) else None
        _ck(_lib().ffsr_token_attention_train(qkv.data_ptr(), B, T, HW, E, out.data_ptr(), probs.data_ptr(),
                                              float(drop_p), int(seed), sd_ptr, _S(qkv)), "token_attention_train")
        ctx.save_for_backward(qkv, probs)
        ctx.cfg = (B, T, HW, E, float(drop_p), int(seed))
        ctx.seed_dev = seed_dev if sd_ptr is not None else None
        return out

    @staticmethod
    def backward(ctx, gy):
        qkv, probs = ctx.saved_tensors
        B, T, HW, E, drop_p, seed = ctx.cfg
        gy = _cl(gy)
        dqkv = torch.empty_like(qkv)
        ds = torch.empty_like(probs)
        sd_ptr = ctx.seed_dev.data_ptr() if ctx.seed_dev is not None else None
        _ck(_lib().ffsr_token_attention_backward(qkv.data_ptr(), probs.data_ptr(), gy.data_ptr(), B, T, HW, E,
                                                 ds.data_ptr(), dqkv.data_ptr(), drop_p, seed, sd_ptr, _S(qkv)),
            "token_attention_backward")
        return dqkv, None, None, None, None, None


def _draw_seed() -> int:
    # CPU default generator: reproducible under torch.manual_seed, no device sync
    return int(torch.randint(0, 2 ** 62, (1,)).item())


_M64 = (1 << 64) - 1


def _mix64(x: int) -> int:
    """splitmix64 finaliser: a bijection of 64-bit integers."""
    x = (x + 0x9E3779B97F4A7C15) & _M64
    x = ((x ^ (x >> 30)) * 0xBF58476D1CE4E5B9) & _M64
    x = ((x ^ (x >> 27)) * 0x94D049BB133111EB) & _M64
    return x ^ (x >> 31)


def dropout_seed(base: int, index: int, call: int) -> int:
    """Host seed of attention call ``call`` of global micro-batch ``index`` in a world-invariant step: a fixed hash of
    (base, index, call) in [0, 2**62), so a micro-batch draws the same masks whichever rank runs it."""
    return _mix64(_mix64((base & _M64) ^ _mix64(index)) ^ _mix64(call & _M64)) >> 2


class MicroBatch:
    """State of one micro-batch of a world-invariant training step (trainer.py), set by ``micro_batch``: its global
    index and the step's seed base key the dropout seeds (``seed_base=None``: the default ``_draw_seed`` draws), and
    the forward appends its BatchNorm records to ``records`` instead of folding them, so the step can fold every
    micro-batch's records in global order."""

    def __init__(self, index: int, seed_base: Optional[int]):
        self.index, self.seed_base, self.calls, self.records = int(index), seed_base, 0, []

    def seed(self) -> int:
        if self.seed_base is None:
            return _draw_seed()
        self.calls += 1
        return dropout_seed(self.seed_base, self.index, self.calls - 1)


_MICRO: Optional[MicroBatch] = None


@contextlib.contextmanager
def micro_batch(index: int, seed_base: Optional[int]):
    """``with micro_batch(i, base) as mb:`` -- train-mode forwards inside run as global micro-batch i (see MicroBatch)."""
    global _MICRO
    prev, _MICRO = _MICRO, MicroBatch(index, seed_base)
    try:
        yield _MICRO
    finally:
        _MICRO = prev


class SeedTape:
    """The host dropout seeds of one step, in call order.  ``seeds=None`` records: every seed the step hands a dropout
    kernel is appended, and nothing else changes.  A list replays: the default draws are taken from it in order
    instead of from torch's CPU generator (hashed world-invariant seeds are computed as usual), so an eager step can
    use exactly the frozen seeds of a CUDA-graph capture (trainer.py: resuming from a checkpoint)."""

    def __init__(self, seeds: Optional[List[int]] = None):
        self.replay = seeds is not None
        self.seeds = [int(s) for s in seeds] if seeds is not None else []
        self.pos = 0

    def take(self) -> int:
        if self.pos >= len(self.seeds):
            raise RuntimeError(f"seed tape holds {len(self.seeds)} dropout seeds; the step asked for more: it differs "
                               "from the step the seeds were recorded from")
        self.pos += 1
        return self.seeds[self.pos - 1]


_TAPE: Optional[SeedTape] = None


@contextlib.contextmanager
def seed_tape(seeds: Optional[List[int]] = None):
    """``with seed_tape() as t:`` records the step's host dropout seeds in ``t.seeds``; ``seed_tape(seeds)`` replays."""
    global _TAPE
    prev, _TAPE = _TAPE, SeedTape(seeds)
    try:
        yield _TAPE
    finally:
        _TAPE = prev


def dropout_host_seed() -> int:
    """Host seed of one train-mode dropout call: the micro-batch hash in a world-invariant step of several
    micro-batches, else the replaying tape's next seed, else a fresh ``_draw_seed``.  A recording tape logs it."""
    if _MICRO is not None and _MICRO.seed_base is not None:
        s = _MICRO.seed()
    elif _TAPE is not None and _TAPE.replay:
        return _TAPE.take()
    else:
        s = _draw_seed()
    if _TAPE is not None and not _TAPE.replay:
        _TAPE.seeds.append(s)
    return s


_SEED_COUNTERS: Dict[str, torch.Tensor] = {}
_CHECKED = set()


def seed_counter(dev) -> torch.Tensor:
    """Device-side int64 added to every dropout seed.  Eager steps draw a fresh host seed per call; a step
    replayed from a CUDA graph has its host seed frozen at capture time, so the trainer bumps this counter
    inside the graph instead (trainer.py)."""
    key = str(dev)
    t = _SEED_COUNTERS.get(key)
    if t is None:
        t = _SEED_COUNTERS[key] = torch.zeros(1, device=dev, dtype=torch.int64)
    return t


def mha_tokens(x, mha: torch.nn.MultiheadAttention, B: int, T: int, training: bool, tc: bool = False):
    """nn.MultiheadAttention self-attention over the T tokens of every LR pixel.
    x: [B*T, E, H, W] channels-last token-major.  (large_kernel_attention.py:192-197, 294-299)"""
    qkv = conv2d(x, mha.in_proj_weight, mha.in_proj_bias, tc)
    p = float(mha.dropout) if training else 0.0
    seed = dropout_host_seed() if p > 0 else 0
    ctx = _TokenAttention.apply(qkv, B, T, p, seed, seed_counter(x.device) if p > 0 else None)
    return conv2d(ctx, mha.out_proj.weight, mha.out_proj.bias, tc)


# --------------------------------------------------------------------------------------
# depthwise stages of the LKA chain
# --------------------------------------------------------------------------------------
class _DwStage(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, kind):
        x = _cl(x)
        N, Cc, H, W = x.shape
        w = weight.detach().reshape(Cc, -1).contiguous()
        out = torch.empty_like(x)
        ones = torch.ones(Cc, device=x.device)
        zeros = torch.zeros(Cc, device=x.device)
        _ck(_lib().ffsr_dwconv_stage(x.data_ptr(), N, H, W, Cc, kind, w.data_ptr(), ones.data_ptr(), zeros.data_ptr(),
                                     out.data_ptr(), _S(x)), "dwconv_stage")
        ctx.save_for_backward(x, weight)
        ctx.kind = kind
        return out

    @staticmethod
    def backward(ctx, gy):
        x, weight = ctx.saved_tensors
        kind = ctx.kind
        N, Cc, H, W = x.shape
        gy = _cl(gy)
        lib = _lib()
        dx = None
        if ctx.needs_input_grad[0]:
            wf = weight.detach().reshape(Cc, -1).flip(1).contiguous()
            dx = torch.empty_like(x)
            ones = torch.ones(Cc, device=x.device)
            zeros = torch.zeros(Cc, device=x.device)
            _ck(lib.ffsr_dwconv_stage(gy.data_ptr(), N, H, W, Cc, kind, wf.data_ptr(), ones.data_ptr(), zeros.data_ptr(),
                                      dx.data_ptr(), _S(x)), "dwconv_stage(bwd)")
        dw = _zeros((Cc, weight.numel() // Cc), x.device)
        ws = _ws(lib.ffsr_dwconv_wgrad_workspace_bytes(N, H, W, Cc, kind), x.device)
        _ck(lib.ffsr_dwconv_wgrad(x.data_ptr(), gy.data_ptr(), N, H, W, Cc, kind, dw.data_ptr(), ws.data_ptr(), ws.numel(),
                                  _S(x)), "dwconv_wgrad")
        return dx, dw.view(weight.shape), None


# --------------------------------------------------------------------------------------
# LKABlock (large_kernel_attention.py:92-105, 143-149), train mode, G statistic groups
# --------------------------------------------------------------------------------------
def lka_block_train(x, blk, G: int, sink: list, stats_only: bool = False, tc: bool = False, training: bool = True):
    """training=False: BatchNorm over the running statistics (the G groups share them)."""
    def norm(t, bn):
        return batchnorm_train(t, bn, G, sink) if training else batchnorm_eval(t, bn)

    n = norm(x, blk.norm1)
    a = _DwStage.apply(n, blk.lka.local_conv.weight, 0)
    a = _DwStage.apply(a, blk.lka.h_conv.weight, 1)
    a = _DwStage.apply(a, blk.lka.v_conv.weight, 2)
    a = conv2d(a, blk.lka.pw_conv.weight, None, tc)
    a = sigmoid(norm(a, blk.lka.bn))
    x1 = axpby(x, n * a, blk.scale1)
    h = norm(x1, blk.norm2)
    if stats_only:
        return None
    h = conv_chain(h, [(blk.ffn[0].weight, blk.ffn[0].bias, K.ACT_GELU), (blk.ffn[2].weight, blk.ffn[2].bias, K.ACT_NONE)], tc)
    return axpby(x1, h, blk.scale2)


class _Bilinear(torch.autograd.Function):
    """F.interpolate(mode="bilinear", align_corners=False) and its adjoint on channels-last tensors."""

    @staticmethod
    def forward(ctx, x, H, W):
        x = _cl(x)
        N, Cc, h, w = x.shape
        out = _empty_cl(N, Cc, H, W, x.device, x.dtype)
        _ck(_lib().ffsr_bilinear_forward(x.data_ptr(), N, h, w, Cc, out.data_ptr(), H, W, _dt(x), _S(x)), "bilinear_forward")
        ctx.shape = (N, Cc, h, w, H, W)
        return out

    @staticmethod
    def backward(ctx, gy):
        N, Cc, h, w, H, W = ctx.shape
        gy = _cl(gy)
        gin = _empty_cl(N, Cc, h, w, gy.device, gy.dtype)
        _ck(_lib().ffsr_bilinear_backward(gy.data_ptr(), N, H, W, Cc, gin.data_ptr(), h, w, _dt(gy), _S(gy)), "bilinear_backward")
        return gin, None, None


def _bilinear(x, size):
    if x.dtype not in (torch.float32, torch.bfloat16):
        x = x.float()
    return _Bilinear.apply(x, int(size[0]), int(size[1]))


class _BlurPool(torch.autograd.Function):
    """avg_pool2d(conv2d(x, gauss5x5, padding=2, groups=3), 2): one Laplacian-pyramid reduction
    (edge_enhancement.py:196-206) and its adjoint; x: [N,3,H,W] fp32."""

    @staticmethod
    def forward(ctx, x, kernel):
        x = _cl(x.float())
        N, Cc, H, W = x.shape
        assert Cc == 3
        g25 = kernel.detach().float()[0, 0].reshape(25).contiguous()
        out = _empty_cl(N, 3, H // 2, W // 2, x.device)
        _ck(_lib().ffsr_blur_pool(x.data_ptr(), 3, N, H, W, g25.data_ptr(), out.data_ptr(), 3, None, 0, _S(x)), "blur_pool")
        ctx.save_for_backward(g25)
        ctx.shape = (N, H, W)
        return out

    @staticmethod
    def backward(ctx, gy):
        (g25,) = ctx.saved_tensors
        N, H, W = ctx.shape
        gy = _cl(gy.float())
        gx = _empty_cl(N, 3, H, W, gy.device)
        _ck(_lib().ffsr_blur_pool_backward(gy.data_ptr(), 3, N, H, W, g25.data_ptr(), gx.data_ptr(), 3, _S(gy)), "blur_pool_backward")
        return gx, None


def _to_group_major(x, B, T):
    """[B*T, C, H, W] token-major (image b*T+t) -> [T*B, C, H, W] group-major (image t*B+b), channels-last."""
    BT, Cc, H, W = x.shape
    v = _cl(x).permute(0, 2, 3, 1).reshape(B, T, H, W, Cc).transpose(0, 1).contiguous()
    return v.view(T * B, H, W, Cc).permute(0, 3, 1, 2)


# --------------------------------------------------------------------------------------
# Phase 2 in train mode
# --------------------------------------------------------------------------------------
def _c32(t):
    t = t.detach()
    return t if (t.dtype == torch.float32 and t.is_contiguous()) else t.float().contiguous()


def _dwt_sub(B, H, W, dev):
    hs, ws_ = C.c_int(), C.c_int()
    _lib().ffsr_dwt_sub_size(H, W, C.byref(hs), C.byref(ws_))
    return torch.empty(B, 4, 3, hs.value, ws_.value, device=dev)


class _Phase2Bands(torch.autograd.Function):
    """Unit-scale DCT (bands 0-2) and DWT (bands 3-6) sub-bands of lr: raw [B,9,3,H,W], bands 7 and 8 left zero for
    the FFT pair.  The backward runs the adjoint kernels (ffsr_dct_bands_adjoint / ffsr_dwt_bands_adjoint)."""

    @staticmethod
    def forward(ctx, lr, fd):
        lib = _lib()
        B, _, H, W = lr.shape
        dev = lr.device
        S = _S(lr)
        raw = torch.zeros(B, 9, 3, H, W, device=dev)
        ones = torch.ones(4, device=dev)
        d = fd.dct
        keep = [_c32(d.dct_basis), _c32(d.dct_basis_t), _c32(d.low_mask), _c32(d.mid_mask), _c32(d.high_mask)]
        _ck(lib.ffsr_dct_bands(lr.data_ptr(), B, H, W, keep[0].data_ptr(), keep[1].data_ptr(), keep[2].data_ptr(),
                               keep[3].data_ptr(), keep[4].data_ptr(), ones.data_ptr(), raw.data_ptr(), S), "dct_bands")
        sub = _dwt_sub(B, H, W, dev)
        w_ = fd.dwt
        k2 = [_c32(w_.lo_row), _c32(w_.hi_row), _c32(w_.lo_col), _c32(w_.hi_col)]
        _ck(lib.ffsr_dwt_bands(lr.data_ptr(), B, H, W, k2[0].data_ptr(), k2[1].data_ptr(), k2[2].data_ptr(),
                               k2[3].data_ptr(), ones.data_ptr(), sub.data_ptr(), raw.data_ptr(), S), "dwt_bands")
        ctx.fd = fd
        return raw

    @staticmethod
    def backward(ctx, g):
        lib = _lib()
        B, _, _, H, W = g.shape
        dev = g.device
        S = _S(g)
        g = g.float()
        g3 = g[:, :3].contiguous()
        g4 = g[:, 3:7].contiguous()
        dx = torch.empty(B, 3, H, W, device=dev)
        d = ctx.fd.dct
        keep = [_c32(d.dct_basis), _c32(d.dct_basis_t), _c32(d.low_mask), _c32(d.mid_mask), _c32(d.high_mask)]
        pad = torch.empty(B * 3 * ((H + 7) // 8 * 8) * ((W + 7) // 8 * 8), device=dev)
        _ck(lib.ffsr_dct_bands_adjoint(g3.data_ptr(), B, H, W, keep[0].data_ptr(), keep[1].data_ptr(), keep[2].data_ptr(),
                                       keep[3].data_ptr(), keep[4].data_ptr(), pad.data_ptr(), dx.data_ptr(), S),
            "dct_bands_adjoint")
        w_ = ctx.fd.dwt
        k2 = [_c32(w_.lo_row), _c32(w_.hi_row), _c32(w_.lo_col), _c32(w_.hi_col)]
        sub = _dwt_sub(B, H, W, dev)
        _ck(lib.ffsr_dwt_bands_adjoint(g4.data_ptr(), B, H, W, k2[0].data_ptr(), k2[1].data_ptr(), k2[2].data_ptr(),
                                       k2[3].data_ptr(), sub.data_ptr(), dx.data_ptr(), S), "dwt_bands_adjoint")
        return dx, None


def _phase2_train(m, lr):
    """9 sub-bands [B,9,3,H,W] with gradients to band_scale / subband_scale / FFT mask parameters, and to lr when it
    requires grad.  The DCT and DWT analysis run on the library kernels with unit scales (_Phase2Bands; without an
    input gradient they are constants of the graph) and are scaled by the learnable factors here;
    the FFT low-pass and the gradient of its learnable mask run on the library's dense-DFT kernels
    (ffsr_fft_lowpass / ffsr_fft_lowpass_backward); the 64x64 -> HxWf mask resize runs on the bilinear node, the sigmoid is a
    tensor op."""
    fd = m.freq_decomp
    B, _, H, W = lr.shape
    raw = _Phase2Bands.apply(lr, fd)
    scale7 = torch.cat([fd.dct.band_scale, fd.dwt.subband_scale])
    b7 = raw[:, :7] * scale7[None, :, None, None, None]
    Wf = W // 2 + 1
    # [1,1,64,64] -> [1,1,H,Wf] on the library's bilinear node: its adjoint is a gather (no atomics), so the mask
    # gradient is reproducible and the step runs under torch.use_deterministic_algorithms(True)
    msk = _bilinear(fd.fft.freq_mask_logits, (H, Wf))
    msk = torch.sigmoid(msk * fd.fft.temperature.clamp(min=1.0))
    low = _FFTLowpass.apply(lr, msk)                                       # irfft2(rfft2(lr) * mask)
    low_s = low * fd.fft.band_scale[0]
    high_s = (lr - low) * fd.fft.band_scale[1]                             # irfft2(X (1 - m)) == x - low
    return torch.cat([b7, low_s[:, None], high_s[:, None]], dim=1)


_TWIDDLES: Dict = {}


def _twiddles(n: int, dev) -> torch.Tensor:
    key = (n, str(dev))
    t = _TWIDDLES.get(key)
    if t is None:
        t = torch.empty(n, 2, device=dev, dtype=torch.float64)
        with torch.cuda.device(dev):
            _ck(_lib().ffsr_fft_twiddles(n, t.data_ptr(), C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)), "fft_twiddles")
        _TWIDDLES[key] = t
    return t


class _FFTLowpass(torch.autograd.Function):
    """low = irfft2(mask * rfft2(x), ortho) on the library's dense-DFT kernels (any H, W) and its gradients.  For a real
    mask on the half spectrum the map is self-adjoint (on the DC and Nyquist columns irfft2 drops the imaginary parts,
    which symmetrises the mask there), so the input gradient is one more low-pass of the output gradient."""

    @staticmethod
    def forward(ctx, x, mask):
        B, _, H, W = x.shape
        lib = _lib()
        m = mask.detach().float().reshape(H, W // 2 + 1).contiguous()
        nb = lib.ffsr_fft_lowpass_workspace_bytes(B, H, W)
        ws = torch.empty(nb // 8 + 2, device=x.device, dtype=torch.float64)
        low = torch.empty_like(x)
        _ck(lib.ffsr_fft_lowpass(x.data_ptr(), B, H, W, m.data_ptr(), _twiddles(H, x.device).data_ptr(),
                                 _twiddles(W, x.device).data_ptr(), ws.data_ptr(), nb, low.data_ptr(), _S(x)), "fft_lowpass")
        ctx.save_for_backward(x, m)
        ctx.mask_shape = mask.shape
        return low

    @staticmethod
    def backward(ctx, g):
        x, m = ctx.saved_tensors
        B, _, H, W = x.shape
        lib = _lib()
        g = g.float().contiguous()
        nb = lib.ffsr_fft_lowpass_workspace_bytes(B, H, W)
        ws = torch.empty(nb // 8 + 2, device=x.device, dtype=torch.float64)
        dmask = torch.empty(H, W // 2 + 1, device=x.device, dtype=torch.float32)
        _ck(lib.ffsr_fft_lowpass_backward(x.data_ptr(), g.data_ptr(), B, H, W, _twiddles(H, x.device).data_ptr(),
                                          _twiddles(W, x.device).data_ptr(), ws.data_ptr(), nb, dmask.data_ptr(), _S(x)),
            "fft_lowpass_backward")
        dx = None
        if ctx.needs_input_grad[0]:
            dx = torch.empty_like(x)
            _ck(lib.ffsr_fft_lowpass(g.data_ptr(), B, H, W, m.data_ptr(), _twiddles(H, x.device).data_ptr(),
                                     _twiddles(W, x.device).data_ptr(), ws.data_ptr(), nb, dx.data_ptr(), _S(x)),
                "fft_lowpass(adjoint)")
        return dx, dmask.view(ctx.mask_shape)


# --------------------------------------------------------------------------------------
# whole pipeline, train mode
# --------------------------------------------------------------------------------------
def train_forward(m, lr: torch.Tensor, img_list: List[torch.Tensor], feats: Dict[str, torch.Tensor],
                  want_inter: bool = False):
    if not lr.is_cuda:
        raise RuntimeError("CompleteEnhancedFusionSR (sm_100a build) needs CUDA tensors: there is no CPU path")
    lib = _lib()
    with torch.cuda.device(lr.device):
        if str(lr.device) not in _CHECKED:
            _ck(lib.ffsr_device_check(), "device_check")
            _CHECKED.add(str(lr.device))
        return _train_forward(m, lr, img_list, feats, want_inter)


def _keep(t: torch.Tensor) -> torch.Tensor:
    """Inputs that require grad stay in the graph (their .float() casts return gradients in their own dtype)."""
    return t if t.requires_grad else t.detach()


def _train_forward(m, lr, img_list, feats, want_inter):
    """m.training=False: the eval forward as a differentiable graph (for input gradients): BatchNorm over the running
    statistics, no dropout, no running-stat update, the eval clamps, and phases 2/3/6 in fp32 in both precisions (as at
    inference, so the derived gate indices are those of the inference path)."""
    if len(img_list) != 4:
        raise ValueError(f"expected the 4 expert outputs drct/grl/nafnet/mamba, got {len(img_list)}")
    B, _, H, W = lr.shape
    Hh, Wh = 4 * H, 4 * W
    lr = _keep(lr).float().contiguous()
    imgs = [_keep(t).float() for t in img_list]
    training = m.training
    sink: list = []
    inter: Dict = {}
    if m.precision not in ("fp32", "bf16"):
        raise ValueError(f"precision must be 'fp32' or 'bf16', got {m.precision!r}")
    # bf16 mode: tcgen05 kernels for the contractions of phases 3/4/5/7 (bf16 operands, fp32 accumulate, HR feature
    # maps stored bf16); phases 2/6, the LR token streams and every residual / image stream stay fp32
    tc = m.precision == "bf16"

    def cv(x, mod, lp_out=False):
        return conv_mod(x, mod, tc, tc and lp_out)

    def cw(x, weight, bias=None, lp_out=False):
        return conv2d(x, weight, bias, tc, tc and lp_out)

    def chain(x, mods, lp_out=False):
        """[(conv module, activation)] as one fused tcgen05 node (bf16 mode) or exact fp32 nodes."""
        return conv_chain(x, [(mod.weight, mod.bias, a) for mod, a in mods], tc, tc and lp_out)

    # ---------------- Phase 2 ----------------
    raw9 = _phase2_train(m, lr)                                           # [B,9,3,H,W]

    # ---------------- Phase 3 ----------------
    cb = m.cross_band
    tc3 = tc and training                                                 # eval: fp32, as at inference
    tok_in = raw9.reshape(B * 9, 3, H, W)                                 # token-major images, NCHW planes
    proj = conv_mod(tok_in, cb.band_proj, tc3)                            # [B*9,64,H,W]
    att = mha_tokens(layernorm(proj, cb.norm), cb.band_attention, B, 9, training, tc3) + proj
    gm = _to_group_major(att, B, 9)                                       # [9*B,64,H,W], band-major
    x_used = lka_block_train(gm[:3 * B], cb.lka_block, 3, sink, tc=tc3, training=training)
    if training:
        with torch.no_grad():                                             # bands 3..8 feed nothing downstream:
            lka_block_train(gm[3 * B:].detach(), cb.lka_block, 6, sink, stats_only=True, tc=tc)   # BN running stats only
    enh = conv_mod(x_used, cb.out_proj, tc3).reshape(3, B, 3, H, W) + raw9[:, :3].transpose(0, 1)
    routing = enh.sum(0)                                                  # [B,3,H,W]

    # ---------------- Phase 6 nets ----------------
    ds = m.dynamic_selector
    d = relu(conv_mod(routing, ds.difficulty_net[0]))
    d = relu(conv_mod(d, ds.difficulty_net[2]))
    diff = sigmoid(conv_mod(d, ds.difficulty_net[4]))
    g = relu(conv_mod(routing, ds.gate_net[0]))
    g = relu(conv_mod(g, ds.gate_net[2]))
    graw = conv_mod(g, ds.gate_net[4])
    gt = torch.sigmoid(ds.temperature * (graw - (0.7 - 0.5 * diff)))
    gates = gt / (gt.sum(dim=1, keepdim=True) + 1e-8).clamp(min=0.3)

    # ---------------- Phase 4 ----------------
    co = m.collaborative
    have = [n for n in EXPERT_ORDER if n in feats]
    if have:
        for n in have:
            if feats[n].dim() != 4 or feats[n].shape[0] != B:
                raise ValueError(f"expert feature '{n}' has shape {tuple(feats[n].shape)}; expected [B={B}, C, h, w]")
        # Feature maps of different spatial sizes are brought to the smallest one (large_kernel_attention.py:365-372).  The
        # reference resizes AFTER the 1x1 align conv; a 1x1 conv (bias included: the bilinear weights sum to 1) commutes
        # with bilinear resampling, so resizing the raw features first gives the same tensor up to fp32 rounding.  Phase 4
        # then runs on that (Hp, Wp) grid, which need not be the LR grid; the modulation upsamples it to HR.
        Hp, Wp = min(feats[n].shape[2] for n in have), min(feats[n].shape[3] for n in have)
        H_lr, W_lr = H, W
        H, W = Hp, Wp
        aligned = []
        for n in EXPERT_ORDER:
            if n not in feats:
                aligned.append(None)
                continue
            f = _keep(feats[n]).float()
            if tuple(f.shape[2:]) != (H, W):
                f = _bilinear(_cl(f), (H, W))
            al = co.align_layers[n]
            cin_w = al.weight.shape[1]
            wgt = al.weight
            if f.shape[1] > cin_w:
                f = f[:, :cin_w]
            elif f.shape[1] < cin_w:
                wgt = wgt[:, :f.shape[1]]                                  # zero-padded channels contribute nothing
            aligned.append(cw(f, wgt, al.bias))
        E = co.norm1.weight.shape[0]
        zero = None
        rows = []
        for a in aligned:
            if a is None:
                if zero is None:
                    zero = torch.zeros(B, H, W, E, device=lr.device)
                rows.append(zero)
            else:
                rows.append(a.permute(0, 2, 3, 1))
        tokens = torch.stack(rows, dim=1).reshape(B * 4, H, W, E).permute(0, 3, 1, 2)   # token-major, channels-last
        x = tokens + mha_tokens(layernorm(tokens, co.norm1), co.cross_attn, B, 4, training, tc)
        x = x + conv_chain(layernorm(x, co.norm2), [(co.ffn[0].weight, co.ffn[0].bias, K.ACT_GELU),
                                                    (co.ffn[2].weight, co.ffn[2].bias, K.ACT_NONE)], tc)
        xg = lka_block_train(_to_group_major(x, B, 4), co.lka_global, 4, sink, tc=tc, training=training)  # [4*B,128,H,W]
        ecol = []
        for i in range(4):
            mod = co.modulation[i]
            f_i = xg[i * B:(i + 1) * B]
            m32 = cv(f_i, mod[0], True)                       # 1x1 conv commutes with the bilinear upsampling
            up = gelu(_bilinear(m32, (Hh, Wh)))
            mk = chain(up, [(mod[2], K.ACT_SIGMOID)])
            o = imgs[i] * (1.0 + 0.2 * (mk - 0.5))
            if not training:
                o = o.clamp(0, 1)
            ecol.append(o)
        H, W = H_lr, W_lr
    else:
        ecol = imgs

    # ---------------- Phase 5 ----------------
    mr = m.multi_res
    stack = torch.cat(ecol, dim=1)                                          # [B,12,Hh,Wh]

    def stage(xin, name, up=None, up_w=None):
        cvs = getattr(mr, name + "_conv")
        y = chain(xin, [(cvs[0], K.ACT_GELU), (cvs[2], K.ACT_GELU)], True)
        gate = getattr(mr, name + "_gate").gate
        y = gate_mul(y, chain(y, [(gate[0], K.ACT_GELU), (gate[2], K.ACT_SIGMOID)]))
        res = getattr(mr, name + "_res")
        r = chain(y, [(res.block[0], K.ACT_GELU), (res.block[2], K.ACT_NONE)], True)
        if up is None:
            return axpby(y, r, res.scale)
        return axpby(y, r, res.scale, up[:, :y.shape[1]], up_w)        # + residual_weight * upsampled coarser stage

    f1 = stage(_bilinear(stack, (H, W)), "stage1")
    f1u = _bilinear(f1, (2 * H, 2 * W))
    f2 = stage(torch.cat([f1u, _bilinear(stack, (2 * H, 2 * W)).to(f1u.dtype)], dim=1), "stage2", f1u, mr.residual_weight_1_2)
    f2u = _bilinear(f2, (Hh, Wh))
    f3 = stage(torch.cat([f2u, stack.to(f2u.dtype)], dim=1), "stage3", f2u, mr.residual_weight_2_3)
    hier = chain(f3, [(mr.to_rgb[0], K.ACT_GELU), (mr.to_rgb[2], K.ACT_SIGMOID)])

    # ---------------- Phase 5b / 6 blend ----------------
    r_hr = _bilinear(routing, (Hh, Wh))
    fl = chain(r_hr, [(m.freq_weight_conv[0], K.ACT_GELU), (m.freq_weight_conv[2], K.ACT_NONE)])
    fw = torch.softmax(fl, dim=1)
    freq = sum(o * fw[:, i:i + 1] for i, o in enumerate(ecol))
    fused = hier * 0.7 + freq * 0.3
    fused_before = fused
    g_hr = _bilinear(gates, (Hh, Wh))
    dyn = sum(o * g_hr[:, i:i + 1] for i, o in enumerate(ecol))
    dyn = dyn / (g_hr.sum(dim=1, keepdim=True) + 1e-8)
    bw = 0.3 + 0.4 * _bilinear(diff, (Hh, Wh))
    fused = (1 - bw) * fused + bw * dyn

    # ---------------- Phase 7a ----------------
    convs = [l for l in m.refine if isinstance(l, torch.nn.Conv2d)]
    y = chain(fused, [(layer, K.ACT_GELU if j < len(convs) - 1 else K.ACT_NONE) for j, layer in enumerate(convs)])
    fused = fused + 0.1 * y

    # ---------------- Phase 7b ----------------
    ee = m.edge_enhance
    kern = ee.gaussian.kernel
    pyr, cur = [], fused
    for lv in range(3):
        if lv < 2:
            hh, ww = cur.shape[2:]
            down = _BlurPool.apply(cur, kern)
            pyr.append(cur - _bilinear(down, (hh, ww)))
            cur = down
        else:
            pyr.append(cur)
    lw = torch.softmax(ee.level_weights, dim=0)
    fl_ = []
    for lv, lap in enumerate(pyr):
        r = ee.edge_refiners[lv]
        idt = cv(lap, r.proj, True)
        o = chain(lap, [(r.conv1, K.ACT_GELU), (r.conv2, K.ACT_GELU), (r.conv3, K.ACT_NONE)], True) + idt
        a = chain(o, [(r.attn.attn[0], K.ACT_GELU), (r.attn.attn[2], K.ACT_SIGMOID)])
        f = gate_mul(o, a)
        if f.shape[2:] != (Hh, Wh):
            f = _bilinear(f, (Hh, Wh))
        fl_.append(f * lw[lv])
    e = chain(torch.cat(fl_, dim=1), [(ee.fusion[0], K.ACT_GELU), (ee.fusion[2], K.ACT_NONE)])
    gte = chain(torch.cat([fused, e], dim=1), [(ee.edge_gate[0], K.ACT_GELU), (ee.edge_gate[2], K.ACT_SIGMOID)])
    fused = (fused + gte * ee.edge_strength * e).clamp(0, 1)

    # ---------------- output ----------------
    out = fused + m.residual_scale * _bilinear(lr, (Hh, Wh))
    if not training:
        out = out.clamp(0, 1)
    out = out.contiguous()
    if training:
        if _MICRO is not None:
            _MICRO.records.extend(sink)
        else:
            fold_running_stats(sink)
    if want_inter:
        inter["raw_9_bands"] = [raw9[:, i] for i in range(9)]
        inter["guidance_bands"] = inter["raw_9_bands"][:3]
        inter["enhanced_9_bands"] = [enh[i] for i in range(3)]
        inter["routing_lr"] = routing
        if have:
            inter["collaborative_outputs"] = ecol
        inter["fused_before_dynamic"] = fused_before
        inter["gates"] = gates
        inter["difficulty"] = diff
        if not training:
            inter["active"] = graw > (0.7 - 0.5 * diff)                   # as FusionEngine reports it
    return out, inter
