"""DRCT-L expert forward on the sm_100a kernels (SURVEY §8f N1) -- first correct path (fp32), not yet timed or tuned.

``DRCT`` mirrors the constructor arguments and the ``state_dict`` (names, shapes, order: ``DRCT-L_X4.pth`` loads with
``strict=True``) of ``src/models/drct/drct_arch.py:624-789`` as configured by ``create_drct_model``
(``src/models/drct/__init__.py:84-131``); the modules are parameter holders only.  ``forward`` runs the network in
fp32 through the C ABI: ``ffsr_conv2d`` for every Linear / Conv2d (residual adds fused in the epilogue),
``ffsr_layernorm_strided``, ``ffsr_window_attention`` (shift + partition + bias + mask + softmax + PV + merge in one
launch), ``ffsr_leaky_relu``, ``ffsr_pixel_shuffle2``, ``ffsr_rgb_shift_in/out``.  The five blocks of an RDG read channel
prefixes of ONE dense-growth buffer ``[B,H,W,dim+4*gc]`` and the adjust convs write their 32 channels straight into
it: no concatenation is ever materialised (``drct_arch.py:292-299``).

STATUS: parity-green on a B200 against the reference class's own output (``tests/golden/drct_small.npz``: 2 RDGs,
window 8, every channel count / head rule of DRCT-L; <= 1e-4 on the SR image and on the cached feature) and, kernel by
kernel, for the window attention at window 16 (``tests/test_gpu_drct.py``).  Every Linear / Conv2d still runs on the
fp32 CUDA-core path: bf16 / tcgen05 execution, timing and the roofline comparison are the next round's work.  One
shape of the FULL DRCT-L configuration has not run on hardware: swin3 (dim 244, 2 heads, head dim 122) at window 16,
whose fp32 K + V exceed shared memory and take the K-staged / V-through-L2 variant of the attention kernel.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, Optional, Tuple

import torch
import torch.nn as nn

from . import _cabi as K
from .pipeline import _View, _pack_conv, _pack_linear, _pack_tc, nhwc

RGB_MEAN = (0.4488, 0.4371, 0.4040)          # drct_arch.py:665-666


def _rel_index(ws: int) -> torch.Tensor:
    """drct_arch.py:153-165."""
    coords = torch.stack(torch.meshgrid([torch.arange(ws), torch.arange(ws)], indexing="ij"))
    flat = torch.flatten(coords, 1)
    rel = (flat[:, :, None] - flat[:, None, :]).permute(1, 2, 0).contiguous()
    rel[:, :, 0] += ws - 1
    rel[:, :, 1] += ws - 1
    rel[:, :, 0] *= 2 * ws - 1
    return rel.sum(-1)


def _shift_mask(H: int, W: int, ws: int, shift: int) -> torch.Tensor:
    """drct_arch.py:353-374 (kept only so that the buffer exists in the state_dict; the kernel derives the mask)."""
    img = torch.zeros(1, H, W, 1)
    cnt = 0
    for hs in (slice(0, -ws), slice(-ws, -shift), slice(-shift, None)):
        for wsl in (slice(0, -ws), slice(-ws, -shift), slice(-shift, None)):
            img[:, hs, wsl, :] = cnt
            cnt += 1
    x = img.view(1, H // ws, ws, W // ws, ws, 1).permute(0, 1, 3, 2, 4, 5).contiguous().view(-1, ws * ws)
    m = x.unsqueeze(1) - x.unsqueeze(2)
    return m.masked_fill(m != 0, -100.0).masked_fill(m == 0, 0.0)


class _Attn(nn.Module):
    def __init__(self, dim, ws, heads):
        super().__init__()
        self.relative_position_bias_table = nn.Parameter(torch.zeros((2 * ws - 1) ** 2, heads))
        self.register_buffer("relative_position_index", _rel_index(ws))
        self.qkv = nn.Linear(dim, 3 * dim)
        self.proj = nn.Linear(dim, dim)
        nn.init.trunc_normal_(self.relative_position_bias_table, std=0.02)


class _Mlp(nn.Module):
    def __init__(self, dim, hidden):
        super().__init__()
        self.fc1 = nn.Linear(dim, hidden)
        self.fc2 = nn.Linear(hidden, dim)


class _Swin(nn.Module):
    def __init__(self, dim, res, heads, ws, shift, mlp_ratio):
        super().__init__()
        if min(res) <= ws:                                  # drct_arch.py:331-334
            shift, ws = 0, min(res)
        self.dim, self.heads, self.window_size, self.shift_size = dim, heads, ws, shift
        self.norm1 = nn.LayerNorm(dim)
        self.attn = _Attn(dim, ws, heads)
        self.norm2 = nn.LayerNorm(dim)
        self.mlp = _Mlp(dim, int(dim * mlp_ratio))
        self.register_buffer("attn_mask", _shift_mask(res[0], res[1], ws, shift) if shift > 0 else None)


class _RDG(nn.Module):
    def __init__(self, dim, res, heads, ws, mlp_ratio, gc):
        super().__init__()
        for j in range(5):                                  # drct_arch.py:230-277
            d = dim + j * gc
            h = heads - (d % heads) if j else heads
            setattr(self, f"swin{j + 1}", _Swin(d, res, h, ws, ws // 2 if j % 2 else 0, mlp_ratio if j < 3 else 1))
            setattr(self, f"adjust{j + 1}", nn.Conv2d(d, gc if j < 4 else dim, 1))


class _PatchNorm(nn.Module):
    def __init__(self, dim):
        super().__init__()
        self.norm = nn.LayerNorm(dim)


class DRCT(nn.Module):
    """Parameter layout of the reference DRCT (pixelshuffle upsampler, '1conv' residual connection)."""

    def __init__(self, img_size=64, patch_size=1, in_chans=3, embed_dim=180, depths=(6,) * 12, num_heads=(6,) * 12,
                 window_size=16, mlp_ratio=2., upscale=4, img_range=1., upsampler="pixelshuffle", resi_connection="1conv",
                 gc=32, **unused):
        super().__init__()
        if upsampler != "pixelshuffle" or resi_connection != "1conv" or in_chans != 3 or patch_size != 1 or upscale != 4:
            raise NotImplementedError("the sm_100a DRCT is built for the DRCT-L x4 configuration "
                                      "(pixelshuffle, 1conv, RGB, patch 1; src/models/drct/__init__.py:84-131)")
        self.window_size, self.embed_dim, self.img_range, self.upscale, self.gc = window_size, embed_dim, img_range, upscale, gc
        res = (img_size // patch_size, img_size // patch_size)
        self.conv_first = nn.Conv2d(3, embed_dim, 3, 1, 1)
        self.patch_embed = _PatchNorm(embed_dim)
        self.layers = nn.ModuleList([_RDG(embed_dim, res, num_heads[i], window_size, mlp_ratio, gc) for i in range(len(depths))])
        self.norm = nn.LayerNorm(embed_dim)
        self.conv_after_body = nn.Conv2d(embed_dim, embed_dim, 3, 1, 1)
        self.conv_before_upsample = nn.Sequential(nn.Conv2d(embed_dim, 64, 3, 1, 1), nn.LeakyReLU(inplace=True))
        self.upsample = nn.Sequential(nn.Conv2d(64, 256, 3, 1, 1), nn.PixelShuffle(2), nn.Conv2d(64, 256, 3, 1, 1), nn.PixelShuffle(2))
        self.conv_last = nn.Conv2d(64, 3, 3, 1, 1)
        # "fp32": every Linear / Conv2d on the CUDA-core path (validated).  "bf16": LayerNorm outputs, qkv, attention output and
        # the MLP hidden activations are bf16 rows padded to 8 channels and the Linears run on tcgen05; the residual stream
        # stays fp32.  Both modes are validated on B200 (tests/test_gpu_drct.py).
        self.precision = "fp32"
        self.headpad_qkv = os.environ.get("FFSR_DRCT_QKV_PLAIN") is None   # bf16 mode, 16 x 16 windows: head-padded qkv rows
        self._packed: Optional[Tuple] = None
        self._ws: Dict[Tuple, torch.Tensor] = {}
        self.last_feature: Optional[torch.Tensor] = None     # conv_after_body output of the last forward ([B,180,H,W] view)

    # ---------------------------------------------------------------------------------- weights
    def _weights(self, dev) -> Dict[str, torch.Tensor]:
        key = (str(dev),) + tuple(p._version for p in self.parameters())
        if self._packed is not None and self._packed[0] == key:
            return self._packed[1]
        w: Dict[str, torch.Tensor] = {}
        for name, mod in self.named_modules():
            if isinstance(mod, nn.Conv2d):
                w[name] = _pack_conv(mod.weight).to(dev)
                w[name + ".b"] = mod.bias.detach().float().contiguous().to(dev)
            elif isinstance(mod, nn.Linear):
                w[name] = _pack_linear(mod.weight).to(dev)
                w[name + ".b"] = mod.bias.detach().float().contiguous().to(dev)
            elif isinstance(mod, nn.LayerNorm):
                w[name + ".w"] = mod.weight.detach().float().contiguous().to(dev)
                w[name + ".b"] = mod.bias.detach().float().contiguous().to(dev)
            elif isinstance(mod, _Attn):
                w[name + ".table"] = mod.relative_position_bias_table.detach().float().contiguous().to(dev)
                # bf16 mode: the qkv Linear writes HEAD-PADDED rows [q | k | v] x [heads][DP] (DP = head dim rounded up to 16):
                # its weight rows are permuted and zero padded here, so every head slice is 16-byte aligned and already
                # zero filled for the tcgen05 window attention (csrc/window_attention_tc.cu)
                heads = mod.relative_position_bias_table.shape[1]
                d = mod.qkv.in_features
                dh = d // heads
                DP = (dh + 15) // 16 * 16
                wq = mod.qkv.weight.detach().float().reshape(3, heads, dh, d)
                wp = torch.zeros(3, heads, DP, d)
                wp[:, :, :dh] = wq
                bp = torch.zeros(3, heads, DP)
                bp[:, :, :dh] = mod.qkv.bias.detach().float().reshape(3, heads, dh)
                w[name + ".qkvp"] = _pack_linear(wp.reshape(3 * heads * DP, d)).to(dev)
                w[name + ".qkvp.b"] = bp.reshape(-1).contiguous().to(dev)
        w["one"] = torch.ones(1, device=dev)
        self._packed = (key, w)
        return w

    def _buf(self, name, shape, dev, dtype=torch.float32):
        t = self._ws.get((name, tuple(shape), str(dev), dtype))
        if t is None:
            t = self._ws[(name, tuple(shape), str(dev), dtype)] = torch.zeros(shape, device=dev, dtype=dtype)
        return t

    # ---------------------------------------------------------------------------------- forward
    @torch.no_grad()
    def forward(self, x: torch.Tensor) -> torch.Tensor:
        if not x.is_cuda:
            raise RuntimeError("DRCT (sm_100a build) needs CUDA tensors: there is no CPU path")
        if self.precision not in ("fp32", "bf16"):
            raise ValueError(f"precision must be 'fp32' or 'bf16', got {self.precision!r}")
        lp = self.precision == "bf16"
        B, Cc, H, W = x.shape
        ws = self.window_size
        if Cc != 3 or H % ws or W % ws:
            raise ValueError(f"DRCT input must be [B,3,H,W] with H, W multiples of the window ({ws}); callers pad "
                             "(scripts/extract_test_tta_cache.py)")
        return self._run(x, K.load(), C.c_void_p(torch.cuda.current_stream(x.device).cuda_stream))

    def _run(self, x: torch.Tensor, lib, S) -> torch.Tensor:
        """The launch sequence (also driven with a recording fake of the library in the CPU tests)."""
        lp = self.precision == "bf16"
        B, Cc, H, W = x.shape
        ws = self.window_size
        dev = x.device
        w = self._weights(dev)
        mean3 = (C.c_float * 3)(*RGB_MEAN)
        E, gc = self.embed_dim, self.gc
        GW = E + 4 * gc                                        # width of the dense-growth buffer
        NP = B * H * W

        def call(fn, *a):
            K.check(fn(*a), fn.__name__)

        def conv(xv: _View, h, wd, cin, name, cout, ks, out: _View, act=K.ACT_NONE, r1: Optional[_View] = None, sa=1.0):
            p = K.ConvParams()
            p.inp, p.in_sN, p.in_sY, p.in_sX, p.in_sC = xv.ptr, xv.sN, xv.sY, xv.sX, xv.sC
            p.N, p.H, p.W, p.Cin, p.Cout, p.ksize = B, h, wd, cin, cout, ks
            wt = w[name]
            if xv.t.dtype == torch.bfloat16:                   # tcgen05 path: K-major bf16 weights, packed on first use
                wt = w.get(name + ".tc")
                if wt is None:
                    wt = w[name + ".tc"] = _pack_tc(w[name])
                p.w_dtype, p.in_dtype = K.DT_BF16, K.DT_BF16
            p.w, p.bias, p.groups = wt.data_ptr(), w[name + ".b"].data_ptr(), 1
            p.out, p.out_sN, p.out_sY, p.out_sX = out.ptr, out.sN, out.sY, out.sX
            p.out_dtype = K.DT_BF16 if out.t.dtype == torch.bfloat16 else K.DT_F32
            p.act, p.epi = act, (K.EPI_RESIDUAL if r1 is not None else K.EPI_PLAIN)
            p.flags = K.CONV_MULTI_ISSUE
            if r1 is not None:
                p.r1, p.r1_sN, p.r1_sY, p.r1_sX = r1.ptr, r1.sN, r1.sY, r1.sX
                p.r1_dtype = K.DT_BF16 if r1.t.dtype == torch.bfloat16 else K.DT_F32
            p.sa, p.sb = sa, 1.0
            call(lib.ffsr_conv2d, C.byref(p), S)

        def padded_out(name: str, cout_p: int) -> str:
            """Weights / bias of Linear `name` with zero output rows appended up to cout_p (packed once)."""
            key = f"{name}.o{cout_p}"
            if key not in w:
                wt = w[name]                                   # [1][in][out]
                wp = torch.zeros(1, wt.shape[1], cout_p, device=wt.device)
                wp[:, :, :wt.shape[2]] = wt
                bp = torch.zeros(cout_p, device=wt.device)
                bp[:wt.shape[2]] = w[name + ".b"]
                w[key], w[key + ".b"] = wp.contiguous(), bp
            return key

        def prefix(t: torch.Tensor, c0: int = 0) -> _View:
            """Channel slice starting at c0 of a [B,h,w,Cs] buffer (the conv takes the channel COUNT separately)."""
            return nhwc(t, c0)

        xin = self._buf("rgb", (B, H, W, 4), dev)
        call(lib.ffsr_rgb_shift_in, x.detach().float().contiguous().data_ptr(), B, H, W, mean3, float(self.img_range),
             xin.data_ptr(), 4, K.DT_F32, S)
        x0 = self._buf("x0", (B, H, W, E), dev)
        conv(nhwc(xin), H, W, 3, "conv_first", E, 3, nhwc(x0))
        G = self._buf("grow", (B, H, W, GW), dev)
        call(lib.ffsr_layernorm_strided, x0.data_ptr(), NP, E, E, w["patch_embed.norm.w"].data_ptr(), w["patch_embed.norm.b"].data_ptr(),
             G.data_ptr(), GW, K.DT_F32, K.DT_F32, S)

        for i, rdg in enumerate(self.layers):
            for j in range(5):
                sw: _Swin = getattr(rdg, f"swin{j + 1}")
                d, p = sw.dim, f"layers.{i}.swin{j + 1}"
                hid = sw.mlp.fc1.out_features
                adt = torch.bfloat16 if lp else torch.float32
                ADT = K.DT_BF16 if lp else K.DT_F32
                pad = (lambda c: (c + 7) // 8 * 8) if lp else (lambda c: c)     # bf16 rows: 16-byte pitch for the TMA loads
                n1 = self._buf("n", (B, H, W, pad(d)), dev, adt)
                call(lib.ffsr_layernorm_strided, G.data_ptr(), NP, d, GW, w[p + ".norm1.w"].data_ptr(), w[p + ".norm1.b"].data_ptr(),
                     n1.data_ptr(), pad(d), K.DT_F32, ADT, S)
                att = self._buf("att", (B, H, W, pad(d)), dev, adt)
                shift = ws // 2 if j % 2 else 0
                headpad = lp and ws == 16 and self.headpad_qkv
                if headpad:
                    nqkv = 3 * sw.heads * lib.ffsr_window_attention_head_pad(d // sw.heads)
                    qkv = self._buf("qkvp", (B, H, W, nqkv), dev, adt)
                    conv(nhwc(n1), H, W, d, p + ".attn.qkvp", nqkv, 1, nhwc(qkv))
                    call(lib.ffsr_window_attention_headpadded, qkv.data_ptr(), B, H, W, d, sw.heads, ws, shift,
                         w[p + ".attn.table"].data_ptr(), att.data_ptr(), pad(d), S)
                else:
                    qkv = self._buf("qkv", (B, H, W, pad(3 * d)), dev, adt)
                    conv(nhwc(n1), H, W, d, p + ".attn.qkv", 3 * d, 1, nhwc(qkv))
                    if lp:
                        call(lib.ffsr_window_attention_pitched, qkv.data_ptr(), pad(3 * d), B, H, W, d, sw.heads, ws, shift,
                             w[p + ".attn.table"].data_ptr(), att.data_ptr(), pad(d), S)
                    else:
                        call(lib.ffsr_window_attention, qkv.data_ptr(), B, H, W, d, sw.heads, ws, shift,
                             w[p + ".attn.table"].data_ptr(), att.data_ptr(), K.DT_F32, S)
                if lp:                                         # bf16 mode: the block's inner residual rows y1 / y2 as bf16 too
                    # Cout = d is 4 mod 8 for every DRCT-L width, which keeps these Linears off the 16-byte-store epilogue of
                    # k_conv_tc: their weights get four zero output rows (padded_out), the outputs land in the pad columns of the
                    # 8-channel-padded bf16 rows (never read: LayerNorm and the next Linear take d channels)
                    y1 = self._buf("y1b", (B, H, W, pad(d)), dev, adt)
                    conv(nhwc(att), H, W, d, padded_out(p + ".attn.proj", pad(d)), pad(d), 1, nhwc(y1), r1=prefix(G))
                else:
                    y1 = self._buf("y1", (B, H, W, d), dev)
                    conv(nhwc(att), H, W, d, p + ".attn.proj", d, 1, nhwc(y1), r1=prefix(G))      # x + proj(attn)
                n2 = n1
                call(lib.ffsr_layernorm_strided, y1.data_ptr(), NP, d, pad(d), w[p + ".norm2.w"].data_ptr(),
                     w[p + ".norm2.b"].data_ptr(), n2.data_ptr(), pad(d), ADT, ADT, S)
                hd = self._buf("hid", (B, H, W, pad(hid)), dev, adt)
                conv(nhwc(n2), H, W, d, p + ".mlp.fc1", hid, 1, nhwc(hd), act=K.ACT_GELU)
                # bf16 mode: y2 feeds only the adjust conv, so it is stored as bf16 rows (16-byte pitch) and that conv runs on tcgen05
                # too (it was an fp32 CUDA-core GEMM: 16 of the 147 ms of a 352x512 forward)
                y2 = self._buf("y2b", (B, H, W, pad(d)), dev, adt) if lp else att
                if lp:
                    conv(nhwc(hd), H, W, hid, padded_out(p + ".mlp.fc2", pad(d)), pad(d), 1, nhwc(y2), r1=nhwc(y1))
                else:
                    conv(nhwc(hd), H, W, hid, p + ".mlp.fc2", d, 1, nhwc(y2), r1=nhwc(y1))         # + mlp
                a = f"layers.{i}.adjust{j + 1}"
                if j < 4:                                      # 32 new channels straight into the growth buffer, LeakyReLU 0.2
                    c0 = E + j * gc
                    conv(nhwc(y2), H, W, d, a, gc, 1, prefix(G, c0))
                    call(lib.ffsr_leaky_relu, G.data_ptr() + 4 * c0, NP, gc, GW, 0.2, K.DT_F32, S)
                else:                                          # x5 * 0.2 + x, in place on the first `embed_dim` channels
                    conv(nhwc(y2), H, W, d, a, E, 1, prefix(G), r1=prefix(G), sa=0.2)

        if lp:
            # bf16 mode: the reconstruction tail on tcgen05 as well.  Its six 3x3 convs ran as fp32 CUDA-core launches (16.6 of the
            # 147 ms of a 352x512 forward, the 64 -> 256 conv at 2x resolution alone 7.1 ms at 30 TFLOP/s).  The cached feature
            # (expert_loader hook) stays an fp32 tensor; x0 + conv_after_body(.) is a second launch of the same conv with the
            # residual epilogue and a bf16 output (0.1 ms) instead of an add + cast pass.
            bf, pe = torch.bfloat16, (E + 7) // 8 * 8
            tb = self._buf("nb", (B, H, W, pe), dev, bf)
            call(lib.ffsr_layernorm_strided, G.data_ptr(), NP, E, GW, w["norm.w"].data_ptr(), w["norm.b"].data_ptr(), tb.data_ptr(), pe,
                 K.DT_F32, K.DT_BF16, S)
            feat = torch.empty(B, H, W, E, device=dev)
            conv(nhwc(tb), H, W, E, "conv_after_body", E, 3, nhwc(feat))
            self.last_feature = feat.permute(0, 3, 1, 2)
            yb = self._buf("yb", (B, H, W, pe), dev, bf)
            conv(nhwc(tb), H, W, E, "conv_after_body", E, 3, nhwc(yb), r1=nhwc(x0))
            ub = self._buf("ub", (B, H, W, 64), dev, bf)
            conv(nhwc(yb), H, W, E, "conv_before_upsample.0", 64, 3, nhwc(ub))
            call(lib.ffsr_leaky_relu, ub.data_ptr(), NP, 64, 64, 0.01, K.DT_BF16, S)
            u4 = self._buf("u4b", (B, H, W, 256), dev, bf)
            conv(nhwc(ub), H, W, 64, "upsample.0", 256, 3, nhwc(u4))
            s2 = self._buf("s2b", (B, 2 * H, 2 * W, 64), dev, bf)
            call(lib.ffsr_pixel_shuffle2, u4.data_ptr(), B, H, W, 64, s2.data_ptr(), K.DT_BF16, S)
            u8 = self._buf("u8b", (B, 2 * H, 2 * W, 256), dev, bf)
            conv(nhwc(s2), 2 * H, 2 * W, 64, "upsample.2", 256, 3, nhwc(u8))
            s4 = self._buf("s4b", (B, 4 * H, 4 * W, 64), dev, bf)
            call(lib.ffsr_pixel_shuffle2, u8.data_ptr(), B, 2 * H, 2 * W, 64, s4.data_ptr(), K.DT_BF16, S)
            o4 = self._buf("o4", (B, 4 * H, 4 * W, 4), dev)
            conv(nhwc(s4), 4 * H, 4 * W, 64, "conv_last", 3, 3, nhwc(o4))
            out = torch.empty(B, 3, 4 * H, 4 * W, device=dev)
            call(lib.ffsr_rgb_shift_out, o4.data_ptr(), B, 4 * H, 4 * W, 4, mean3, float(self.img_range), out.data_ptr(), K.DT_F32, S)
            return out
        t = self._buf("n", (B, H, W, E), dev)
        call(lib.ffsr_layernorm_strided, G.data_ptr(), NP, E, GW, w["norm.w"].data_ptr(), w["norm.b"].data_ptr(), t.data_ptr(), E,
             K.DT_F32, K.DT_F32, S)
        feat = torch.empty(B, H, W, E, device=dev)
        conv(nhwc(t), H, W, E, "conv_after_body", E, 3, nhwc(feat))
        self.last_feature = feat.permute(0, 3, 1, 2)           # the cached [B,180,H,W] feature (expert_loader hook)
        y = self._buf("y", (B, H, W, E), dev)
        call(lib.ffsr_axpby_forward, x0.data_ptr(), feat.data_ptr(), None, 0, w["one"].data_ptr(), None, NP, E, y.data_ptr(),
             K.DT_F32, S)
        u = self._buf("u", (B, H, W, 64), dev)
        conv(nhwc(y), H, W, E, "conv_before_upsample.0", 64, 3, nhwc(u))
        call(lib.ffsr_leaky_relu, u.data_ptr(), NP, 64, 64, 0.01, K.DT_F32, S)
        u4 = self._buf("u4", (B, H, W, 256), dev)
        conv(nhwc(u), H, W, 64, "upsample.0", 256, 3, nhwc(u4))
        s2 = self._buf("s2", (B, 2 * H, 2 * W, 64), dev)
        call(lib.ffsr_pixel_shuffle2, u4.data_ptr(), B, H, W, 64, s2.data_ptr(), K.DT_F32, S)
        u8 = self._buf("u8", (B, 2 * H, 2 * W, 256), dev)
        conv(nhwc(s2), 2 * H, 2 * W, 64, "upsample.2", 256, 3, nhwc(u8))
        s4 = self._buf("s4", (B, 4 * H, 4 * W, 64), dev)
        call(lib.ffsr_pixel_shuffle2, u8.data_ptr(), B, 2 * H, 2 * W, 64, s4.data_ptr(), K.DT_F32, S)
        o4 = self._buf("o4", (B, 4 * H, 4 * W, 4), dev)
        conv(nhwc(s4), 4 * H, 4 * W, 64, "conv_last", 3, 3, nhwc(o4))
        out = torch.empty(B, 3, 4 * H, 4 * W, device=dev)
        call(lib.ffsr_rgb_shift_out, o4.data_ptr(), B, 4 * H, 4 * W, 4, mean3, float(self.img_range), out.data_ptr(), K.DT_F32, S)
        return out


def create_drct_model(upscale: int = 4, img_size: int = 64, window_size: int = 16, embed_dim: int = 180, depths=None,
                      num_heads=None, img_range: float = 1.0, upsampler: str = "pixelshuffle",
                      resi_connection: str = "1conv") -> DRCT:
    """``create_drct_model`` of the reference (src/models/drct/__init__.py:84-131): DRCT-L x4."""
    return DRCT(upscale=upscale, img_size=img_size, window_size=window_size, embed_dim=embed_dim,
                depths=depths if depths is not None else [6] * 12, num_heads=num_heads if num_heads is not None else [6] * 12,
                img_range=img_range, mlp_ratio=2, upsampler=upsampler, resi_connection=resi_connection)


def flops_per_lr_pixel(model: DRCT) -> float:
    """2 x MAC per LR pixel of the forward (Linears, attention products, convs): the roofline unit of this path."""
    E, gc, N = model.embed_dim, model.gc, model.window_size ** 2
    f = 2 * 9 * 3 * E
    for rdg in model.layers:
        for j in range(5):
            sw = getattr(rdg, f"swin{j + 1}")
            d, hid = sw.dim, sw.mlp.fc1.out_features
            f += 2 * (4 * d * d + 2 * d * hid) + 4 * N * d + 2 * d * (gc if j < 4 else E)
    f += 2 * 9 * E * E + 2 * 9 * E * 64 + 2 * 9 * 64 * 256 * (1 + 4) + 16 * 2 * 9 * 64 * 3
    return float(f)

