"""Host-side orchestration of the sm_100a kernels for one fusion forward (eval mode).

``FusionEngine.forward`` is what ``CompleteEnhancedFusionSR._run_pipeline`` runs: it
enqueues ~110 kernel launches of ``libffsr_b200.so`` on the current CUDA stream.  PyTorch
is used for device memory (caching allocator / persistent workspaces), streams and the tiny
host-side weight re-packing (BN folding, [taps][Cin][Cout] packing), nothing else.

Phase map (reference file:line in include/ffsr_b200.h):
  P2  dct/dwt/fft bands      -> raw9 [B][9][3][H][W]
  P3  cross-band attention   -> tokens [B][nq][H][W][64] -> LKA block -> enhanced bands, routing_lr
  P6  selector convs on routing_lr -> gates, difficulty           (fp32 always)
  P4  align -> LN -> MHA -> FFN -> LKA(128) -> mod-head layer 0 at LR -> HR modulation
  P5  hierarchical conv pyramid; P5b/P6 blend; P7a refine; P7b Laplacian edge; residual
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Optional, Tuple

import torch

from . import _cabi as K

EXPERT_ORDER = ("drct", "grl", "nafnet", "mamba")
_BN_EPS = 1e-5


class _View:
    """Strided channels-last (or NCHW) view handed to ffsr_conv2d."""
    __slots__ = ("ptr", "sN", "sY", "sX", "sC", "t")

    def __init__(self, ptr, sN, sY, sX, sC, t):
        self.ptr, self.sN, self.sY, self.sX, self.sC, self.t = ptr, sN, sY, sX, sC, t


def nhwc(t: torch.Tensor, c_off: int = 0) -> _View:
    """t: [N,H,W,Cs] contiguous; view starting at channel c_off."""
    N, H, W, Cs = t.shape
    return _View(t.data_ptr() + c_off * t.element_size(), H * W * Cs, W * Cs, Cs, 1, t)


def nchw(t: torch.Tensor) -> _View:
    N, Cc, H, W = t.shape
    return _View(t.data_ptr(), Cc * H * W, W, 1, H * W, t)


def _pack_conv(w: torch.Tensor) -> torch.Tensor:
    """[Cout,Cin,kh,kw] -> [kh*kw][Cin][Cout] fp32 contiguous."""
    co, ci, kh, kw = w.shape
    return w.detach().float().permute(2, 3, 1, 0).reshape(kh * kw, ci, co).contiguous()


def _pack_tc(w_f32: torch.Tensor) -> torch.Tensor:
    """fp32 pack [G?][taps][Cin][Cout] -> tcgen05 pack [G*taps][CoutPad][CinPad] bf16 (K-major).
    CinPad = ceil64(Cin); CoutPad = ceil16(Cout), rounded up to a multiple of 128 when > 128."""
    if w_f32.dim() == 3:
        w_f32 = w_f32.unsqueeze(0)
    G, taps, ci, co = w_f32.shape
    cip = (ci + 63) // 64 * 64
    cop = (co + 15) // 16 * 16
    if cop > 128:
        cop = (cop + 127) // 128 * 128
    out = torch.zeros(G * taps, cop, cip, device=w_f32.device, dtype=torch.bfloat16)
    out[:, :co, :ci] = w_f32.reshape(G * taps, ci, co).transpose(1, 2).to(torch.bfloat16)
    return out.contiguous()


def _pack_planes(w: torch.Tensor, kgn: int, nout: int) -> torch.Tensor:
    """[Cout,Cin,kh,kw] -> [kh*kw][kgn][nout][8] fp32: the no-swizzle K-major shared-memory layout of the tile-resident
    kernels (8-input-channel groups, zero padded in both channel dimensions)."""
    co, ci, kh, kw = w.shape
    t = torch.zeros(kh * kw, kgn * 8, nout, device=w.device, dtype=torch.float32)
    t[:, :ci, :co] = w.detach().float().permute(2, 3, 1, 0).reshape(kh * kw, ci, co)
    return t.view(kh * kw, kgn, 8, nout).permute(0, 1, 3, 2).contiguous()


def pack_edge_chain(r):
    """EdgeRefineBlock -> (bf16 weight blob, fp32 parameter blob) of ffsr_edge_refiner_chain (layout: csrc/edge_chain.cu)."""
    a0, a2 = r.attn.attn[0], r.attn.attn[2]
    wb = torch.cat([_pack_planes(r.conv1.weight, 2, 32).reshape(-1), _pack_planes(r.conv2.weight, 4, 32).reshape(-1),
                    _pack_planes(r.conv3.weight, 4, 32).reshape(-1), _pack_planes(a0.weight, 4, 16).reshape(-1)]).to(torch.bfloat16)
    f = lambda t: t.detach().float().reshape(-1)
    ba = torch.zeros(16, device=wb.device)
    ba[:8] = f(a0.bias)
    wp = torch.cat([r.proj.weight.detach().float().reshape(32, 3), r.proj.bias.detach().float().reshape(32, 1)], 1)
    pb = torch.cat([f(r.conv1.bias), f(r.conv2.bias), f(r.conv3.bias), ba, wp.reshape(-1),
                    a2.weight.detach().float().permute(2, 3, 1, 0).reshape(-1), f(a2.bias),
                    torch.zeros(7, device=wb.device)])
    return wb.contiguous(), pb.contiguous()


def _planes_bf16(w2d: torch.Tensor) -> torch.Tensor:
    """fp32 [n][k] -> bf16 no-swizzle K-major planes [k/8][n][8] (B operand of the tile-resident kernels)."""
    n, k = w2d.shape
    return w2d.detach().float().to(torch.bfloat16).view(n, k // 8, 8).permute(1, 0, 2).contiguous()


def _split3_planes(w2d: torch.Tensor) -> torch.Tensor:
    """fp32 [n][k] -> its three bf16 terms w = w1 + w2 + w3 (24 mantissa bits) in the no-swizzle K-major plane layout
    [split][k/8][n][8] of the tile-resident kernels (csrc/lka_tail.cu)."""
    w = w2d.detach().float()
    w1 = w.to(torch.bfloat16)
    r = w - w1.float()
    w2 = r.to(torch.bfloat16)
    w3 = (r - w2.float()).to(torch.bfloat16)
    n, k = w.shape
    return torch.stack([w1, w2, w3]).view(3, n, k // 8, 8).permute(0, 2, 1, 3).contiguous()


def pack_align_tokens(co):
    """align_layers -> (bf16 weight blob [4][kg 24][n 128][8] with K zero-padded to 192, fp32 bias [4][128]) of ffsr_align_tokens."""
    ws, bs = [], []
    for n in EXPERT_ORDER:
        l = co.align_layers[n]
        w2 = torch.zeros(128, 192, device=l.weight.device)
        w2[:, :l.weight.shape[1]] = l.weight.detach().float().reshape(128, -1)
        ws.append(_planes_bf16(w2).reshape(-1))
        bs.append(l.bias.detach().float())
    return torch.cat(ws).contiguous(), torch.stack(bs).contiguous()


def pack_token_attn(co):
    """CollaborativeFeatureLearning norm1 + cross_attn -> (bf16 weight blob, fp32 parameter blob) of ffsr_token_attn_chain
    (layout: csrc/token_chain.cu).  LayerNorm folded into in_proj: g = gamma o W_in, colsum of the bf16-ROUNDED g (what the
    tensor cores multiply by), bias W_in beta + b_in; the 1/sqrt(head_dim) = 1/4 of the scores is folded into the q rows."""
    Win = co.cross_attn.in_proj_weight.detach().double()
    g = Win * co.norm1.weight.detach().double()[None, :]
    b = Win @ co.norm1.bias.detach().double() + co.cross_attn.in_proj_bias.detach().double()
    E = Win.shape[1]
    g[:E] *= 0.25
    b[:E] *= 0.25
    g16 = g.float().to(torch.bfloat16)
    wo = co.cross_attn.out_proj.weight.detach().float()
    wb = torch.cat([_planes_bf16(g16.float()).reshape(-1), _planes_bf16(wo).reshape(-1)]).contiguous()
    pb = torch.cat([g16.double().sum(1).float(), b.float(), co.cross_attn.out_proj.bias.detach().float()]).contiguous()
    return wb, pb


def pack_token_ffn(co):
    """norm2 + ffn -> blobs of ffsr_token_ffn_chain (LayerNorm folded into ffn.0 as in pack_token_attn)."""
    W0 = co.ffn[0].weight.detach().double()
    g = W0 * co.norm2.weight.detach().double()[None, :]
    b = W0 @ co.norm2.bias.detach().double() + co.ffn[0].bias.detach().double()
    g16 = g.float().to(torch.bfloat16)
    wb = torch.cat([_planes_bf16(g16.float()).reshape(-1), _planes_bf16(co.ffn[2].weight.detach().float()).reshape(-1)]).contiguous()
    pb = torch.cat([g16.double().sum(1).float(), b.float(), co.ffn[2].bias.detach().float()]).contiguous()
    return wb, pb


def pack_selector(ds):
    """DynamicExpertSelector difficulty_net / gate_net -> the fp32 blob of ffsr_selector_fused (layout: csrc/selector.cu):
    [taps][Cin][Cout] weights + bias per layer, the single-channel and 4-channel heads padded to 4 floats of bias."""
    f = lambda t: t.detach().float().reshape(-1)
    z3 = torch.zeros(3, device=ds.gate_net[0].weight.device)
    d, g = ds.difficulty_net, ds.gate_net
    return torch.cat([_pack_conv(d[0].weight).reshape(-1), f(d[0].bias), _pack_conv(d[2].weight).reshape(-1), f(d[2].bias),
                      _pack_conv(d[4].weight).reshape(-1), f(d[4].bias), z3,
                      _pack_conv(g[0].weight).reshape(-1), f(g[0].bias), _pack_conv(g[2].weight).reshape(-1), f(g[2].bias),
                      _pack_conv(g[4].weight).reshape(-1), f(g[4].bias)]).contiguous()


def _pack_linear(w: torch.Tensor) -> torch.Tensor:
    """[out,in] -> [1][in][out]."""
    return w.detach().float().t().contiguous().unsqueeze(0)


class FusionEngine:
    def __init__(self, model):
        self.m = model
        self.lib = K.load()
        self._wkey = None
        self._w: Dict[str, torch.Tensor] = {}
        self._ws: Dict[Tuple, torch.Tensor] = {}
        self._tw: Dict[Tuple, torch.Tensor] = {}
        self._checked_dev = None
        self.launches = 0          # kernels enqueued by the last forward (bench reports it)
        # optional per-launch CUDA-event timing of named conv layers (bench.py roofline):
        # {weight name: [(start_event, end_event), ...]}
        self.timed_layers = None
        # optional in-situ trace of EVERY launch: [(label, start_event, end_event), ...] (tools/trace_forward.py)
        self.trace = None
        self.overlap_routing = True    # phases 3 + 6 on a side stream, concurrent with phases 4 / 5
        # Tile-resident kernels in place of the layer-by-layer launches; tests turn them off to compare against the
        # layer-by-layer path, which also serves fp32 mode and missing experts.
        self.edge_chain = True       # bf16 mode: each edge refiner as ONE kernel (csrc/edge_chain.cu) instead of six conv launches
        self.token_chain = True      # bf16 mode: Phase-4 token pipeline as two kernels (csrc/token_chain.cu)
        self.selector_fused = True   # Phase 6 as one fp32 kernel (csrc/selector.cu)
        self._side: Dict[str, torch.cuda.Stream] = {}

    # ------------------------------------------------------------------ weights
    def _state_key(self, dev):
        m = self.m
        return (str(dev), m.training) + tuple(p._version for p in m.parameters()) + \
            tuple(b._version for b in m.buffers())

    def _bn_fold(self, bn):
        k = bn.weight.detach().float() / torch.sqrt(bn.running_var.detach().float() + _BN_EPS)
        d = bn.bias.detach().float() - bn.running_mean.detach().float() * k
        return k.contiguous(), d.contiguous()

    def _prep_lka(self, key, blk):
        w = self._w
        C_ = blk.norm1.weight.shape[0]
        w[key + ".k1"], w[key + ".d1"] = self._bn_fold(blk.norm1)
        w[key + ".w5"] = blk.lka.local_conv.weight.detach().float().reshape(C_, 25).contiguous()
        w[key + ".wh"] = blk.lka.h_conv.weight.detach().float().reshape(C_, 21).contiguous()
        w[key + ".wv"] = blk.lka.v_conv.weight.detach().float().reshape(C_, 21).contiguous()
        kb, db = self._bn_fold(blk.lka.bn)                      # BN after the 1x1: fold into it
        pw = blk.lka.pw_conv.weight.detach().float().reshape(C_, C_)      # [co][ci]
        w[key + ".pw"] = (pw * kb[:, None]).t().contiguous().unsqueeze(0)
        w[key + ".pwb"] = db
        k2, d2 = self._bn_fold(blk.norm2)                        # BN before ffn.0: fold into it
        f0 = blk.ffn[0].weight.detach().float().reshape(-1, C_)           # [2C][C]
        w[key + ".f0"] = (f0 * k2[None, :]).t().contiguous().unsqueeze(0)
        w[key + ".f0b"] = (blk.ffn[0].bias.detach().float() + f0 @ d2).contiguous()
        w[key + ".f2"] = _pack_conv(blk.ffn[2].weight)
        w[key + ".f2b"] = blk.ffn[2].bias.detach().float().contiguous()
        if C_ == 64:
            # tile-resident tail on tcgen05 at fp32 accuracy (three-term bf16 split of both operands): csrc/lka_tail.cu
            w[key + ".tail_w"] = torch.cat([_split3_planes(pw * kb[:, None]).reshape(-1), _split3_planes(f0 * k2[None, :]).reshape(-1),
                                            _split3_planes(blk.ffn[2].weight.detach().float().reshape(C_, 2 * C_)).reshape(-1)]).contiguous()
            w[key + ".tail_p"] = torch.cat([db, w[key + ".k1"], w[key + ".d1"], w[key + ".f0b"], w[key + ".f2b"],
                                            torch.zeros(8, device=db.device)]).contiguous()

    def _prepare(self, dev):
        key = self._state_key(dev)
        if key == self._wkey:
            return
        m, w = self.m, {}
        self._w = w
        # contiguous fp32 view of every parameter / buffer handed to the kernels by raw pointer
        # (e.g. dct_basis_t is registered as a transposed view: its storage is NOT D^T)
        self._P = {}
        for n, t in list(m.named_parameters()) + list(m.named_buffers()):
            if torch.is_floating_point(t):
                t = t.detach()
                self._P[n] = t if (t.dtype == torch.float32 and t.is_contiguous()) else t.float().contiguous()

        def conv(name, mod, bias=True):
            w[name] = _pack_conv(mod.weight)
            if bias and mod.bias is not None:
                w[name + ".b"] = mod.bias.detach().float().contiguous()

        with torch.no_grad():
            self._prep_lka("cb.lka", m.cross_band.lka_block)
            self._prep_lka("co.lka", m.collaborative.lka_global)
            cb = m.cross_band
            w["cb.proj_w"] = cb.band_proj.weight.detach().float().reshape(64, 3).contiguous()
            w["cb.out_w"] = cb.out_proj.weight.detach().float().reshape(3, 64).contiguous()
            # band_proj -> LayerNorm -> in_proj folded in fp64 (see k_crossband_attn2)
            Wp = cb.band_proj.weight.detach().double().reshape(64, 3)
            bp = cb.band_proj.bias.detach().double()
            A_ = Wp - Wp.mean(dim=0, keepdim=True)
            c_ = bp - bp.mean()
            Win = cb.band_attention.in_proj_weight.detach().double()            # [192, 64]
            gam, bet = cb.norm.weight.detach().double(), cb.norm.bias.detach().double()
            Wg = Win * gam[None, :]
            fold = torch.cat([torch.cat([A_, c_[:, None]], 1).reshape(-1),
                              torch.cat([Wg @ A_, (Wg @ c_)[:, None]], 1).reshape(-1),
                              Win @ bet + cb.band_attention.in_proj_bias.detach().double()])
            w["cb.fold"] = fold.float().contiguous()
            co = m.collaborative
            for n in EXPERT_ORDER:
                conv("co.align." + n, co.align_layers[n])
            w["co.qkv"] = _pack_linear(co.cross_attn.in_proj_weight)
            w["co.qkv.b"] = co.cross_attn.in_proj_bias.detach().float().contiguous()
            w["co.out"] = _pack_linear(co.cross_attn.out_proj.weight)
            w["co.out.b"] = co.cross_attn.out_proj.bias.detach().float().contiguous()
            w["co.f0"] = _pack_linear(co.ffn[0].weight)
            w["co.f0.b"] = co.ffn[0].bias.detach().float().contiguous()
            w["co.f2"] = _pack_linear(co.ffn[2].weight)
            w["co.f2.b"] = co.ffn[2].bias.detach().float().contiguous()
            if all(co.align_layers[n].weight.shape[0] == 128 and co.align_layers[n].weight.shape[1] <= 192 for n in EXPERT_ORDER):
                w["co.align_w"], w["co.align_b"] = pack_align_tokens(co)
            if (co.cross_attn.embed_dim, co.cross_attn.num_heads) == (128, 8) and tuple(co.ffn[0].weight.shape) == (256, 128):
                w["co.attn_w"], w["co.attn_p"] = pack_token_attn(co)
                w["co.ffn_w"], w["co.ffn_p"] = pack_token_ffn(co)
            w["co.m0"] = torch.stack([_pack_conv(co.modulation[i][0].weight) for i in range(4)]).contiguous()
            w["co.m0b"] = torch.stack([co.modulation[i][0].bias.detach().float() for i in range(4)]).contiguous()
            lg = co.lka_global
            if lg.norm1.weight.shape[0] == 128 and all(tuple(co.modulation[i][0].weight.shape[:2]) == (32, 128) for i in range(4)):
                # bf16 mode: LKA tail + modulation layer 0 as one tile-resident kernel (csrc/lka_tail.cu, k_lka_tail128w)
                kb, db = self._bn_fold(lg.lka.bn)
                k2, d2 = self._bn_fold(lg.norm2)
                pw = lg.lka.pw_conv.weight.detach().float().reshape(128, 128) * kb[:, None]
                f0 = lg.ffn[0].weight.detach().float().reshape(256, 128)
                w["co.tail_w"] = torch.cat([_planes_bf16(pw).reshape(-1), _planes_bf16(f0 * k2[None, :]).reshape(-1),
                                            _planes_bf16(lg.ffn[2].weight.detach().float().reshape(128, 256)).reshape(-1)]
                                           + [_planes_bf16(co.modulation[i][0].weight.detach().float().reshape(32, 128)).reshape(-1)
                                              for i in range(4)]).contiguous()
                w["co.tail_p"] = torch.cat([db, w["co.lka.k1"], w["co.lka.d1"], w["co.lka.f0b"], w["co.lka.f2b"]]
                                           + [co.modulation[i][0].bias.detach().float() for i in range(4)]).contiguous()
            w["co.m2"] = torch.stack([co.modulation[i][2].weight.detach().float().reshape(3, 32) for i in range(4)]).contiguous()
            w["co.m2b"] = torch.stack([co.modulation[i][2].bias.detach().float() for i in range(4)]).contiguous()
            mr = m.multi_res
            for s in ("stage1", "stage2", "stage3"):
                conv(f"mr.{s}.c0", getattr(mr, s + "_conv")[0])
                conv(f"mr.{s}.c2", getattr(mr, s + "_conv")[2])
                g = getattr(mr, s + "_gate").gate
                w[f"mr.{s}.g0"] = g[0].weight.detach().float().reshape(g[0].weight.shape[0], -1).contiguous()
                w[f"mr.{s}.g2"] = g[2].weight.detach().float().reshape(-1).contiguous()
                r = getattr(mr, s + "_res").block
                conv(f"mr.{s}.r0", r[0], bias=False)
                conv(f"mr.{s}.r2", r[2], bias=False)
            conv("mr.rgb0", mr.to_rgb[0])
            conv("mr.rgb2", mr.to_rgb[2])
            w["fw0"] = m.freq_weight_conv[0].weight.detach().float().reshape(16, 3).contiguous()
            w["fw2"] = m.freq_weight_conv[2].weight.detach().float().reshape(4, 16).contiguous()
            ds = m.dynamic_selector
            for i in (0, 2, 4):
                conv(f"ds.d{i}", ds.difficulty_net[i])
                conv(f"ds.g{i}", ds.gate_net[i])
            shapes = [tuple(l.weight.shape) for l in (ds.difficulty_net[0], ds.difficulty_net[2], ds.difficulty_net[4],
                                                        ds.gate_net[0], ds.gate_net[2], ds.gate_net[4])]
            if shapes == [(32, 3, 3, 3), (32, 32, 3, 3), (1, 32, 3, 3), (32, 3, 3, 3), (32, 32, 3, 3), (4, 32, 1, 1)]:
                w["ds.blob"] = pack_selector(ds)
            self._refine_idx = [i for i, l in enumerate(m.refine) if isinstance(l, torch.nn.Conv2d)]
            for i in self._refine_idx:
                conv(f"rf.{i}", m.refine[i])
            ee = m.edge_enhance
            for lv in range(3):
                r = ee.edge_refiners[lv]
                conv(f"ee.{lv}.c1", r.conv1)
                conv(f"ee.{lv}.c2", r.conv2)
                conv(f"ee.{lv}.c3", r.conv3)
                conv(f"ee.{lv}.proj", r.proj)
                conv(f"ee.{lv}.a0", r.attn.attn[0])
                conv(f"ee.{lv}.a2", r.attn.attn[2])
                if tuple(r.conv1.weight.shape) == (32, 3, 3, 3) and tuple(r.attn.attn[0].weight.shape[:2]) == (8, 32):
                    w[f"ee.{lv}.chain_w"], w[f"ee.{lv}.chain_p"] = pack_edge_chain(r)
            conv("ee.f0", ee.fusion[0])
            conv("ee.f2", ee.fusion[2])
            conv("ee.g0", ee.edge_gate[0])
            conv("ee.g2", ee.edge_gate[2])
            w["ee.gauss"] = ee.gaussian.kernel.detach().float()[0, 0].reshape(25).contiguous()
        self._wkey = key

    # ---------------------------------------------------------------- utilities
    @staticmethod
    def _get_stream(dev):
        return C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)

    @staticmethod
    def _sm_count(dev):
        return torch.cuda.get_device_properties(dev).multi_processor_count

    def _buf(self, name, shape, dev, dtype=torch.float32, zero=False, fresh=False):
        """Persistent workspace keyed by (name, shape): allocated once, reused across calls
        (padding channels are zeroed once and never written)."""
        if fresh:
            return torch.zeros(shape, device=dev, dtype=dtype) if zero else torch.empty(shape, device=dev, dtype=dtype)
        key = (name, tuple(shape), str(dev), dtype)
        t = self._ws.get(key)
        if t is None:
            t = torch.zeros(shape, device=dev, dtype=dtype)
            self._ws[key] = t
        return t

    def workspace(self, name):
        """Debug/test access to a persistent workspace buffer by name (latest shape)."""
        hits = [t for k, t in self._ws.items() if k[0] == name]
        if not hits:
            raise KeyError(name)
        return hits[-1]

    def _call(self, fn, *args, label=None):
        if self.trace is not None:
            st = torch.cuda.current_stream()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            rc = fn(*args)
            e1.record(st)
            self.trace.append((label or fn.__name__, e0, e1))
        else:
            rc = fn(*args)
        self.launches += 1
        if rc != 0:
            K.check(rc, fn.__name__)

    def conv(self, x: _View, N, H, W, Cin, wname, Cout, ks, out: _View, act=K.ACT_NONE, epi=K.EPI_PLAIN,
             bias=True, r1: Optional[_View] = None, r2: Optional[_View] = None, sa=1.0, sa_ptr=None, sb=1.0,
             sb_ptr=None, ch_k=None, ch_d=None, groups=1, bias_name=None):
        w = self._w[wname]
        assert w.shape[-3:] == (ks * ks, Cin, Cout) or w.numel() == groups * ks * ks * Cin * Cout, \
            (wname, tuple(w.shape), ks, Cin, Cout)
        b = self._w.get(bias_name or (wname + ".b")) if bias else None
        p = K.ConvParams()
        if x.t.dtype == torch.bfloat16:                    # tcgen05 path: K-major bf16 weights, packed lazily
            wt = self._w.get(wname + ".tc")
            if wt is None:
                wt = self._w[wname + ".tc"] = _pack_tc(w)
            w = wt
            p.w_dtype = K.DT_BF16
        p.inp, p.in_sN, p.in_sY, p.in_sX, p.in_sC = x.ptr, x.sN, x.sY, x.sX, x.sC
        p.N, p.H, p.W, p.Cin, p.Cout, p.ksize = N, H, W, Cin, Cout, ks
        p.w = w.data_ptr()
        p.bias = b.data_ptr() if b is not None else None
        p.groups = groups
        p.out, p.out_sN, p.out_sY, p.out_sX = out.ptr, out.sN, out.sY, out.sX
        p.act, p.epi = act, epi
        p.flags = K.CONV_MULTI_ISSUE      # inference launches: up to three MMA-issuing warps on issue-bound layers
        if r1 is not None:
            p.r1, p.r1_sN, p.r1_sY, p.r1_sX = r1.ptr, r1.sN, r1.sY, r1.sX
            p.r1_dtype = K.DT_BF16 if r1.t.dtype == torch.bfloat16 else K.DT_F32
        if r2 is not None:
            p.r2, p.r2_sN, p.r2_sY, p.r2_sX = r2.ptr, r2.sN, r2.sY, r2.sX
            p.r2_dtype = K.DT_BF16 if r2.t.dtype == torch.bfloat16 else K.DT_F32
        p.sa, p.sb = sa, sb
        p.sa_ptr = sa_ptr.data_ptr() if sa_ptr is not None else None
        p.sb_ptr = sb_ptr.data_ptr() if sb_ptr is not None else None
        p.ch_k = ch_k.data_ptr() if ch_k is not None else None
        p.ch_d = ch_d.data_ptr() if ch_d is not None else None
        p.in_dtype = K.DT_BF16 if x.t.dtype == torch.bfloat16 else K.DT_F32
        p.out_dtype = K.DT_BF16 if out.t.dtype == torch.bfloat16 else K.DT_F32
        ev = self.timed_layers.get(wname) if self.timed_layers is not None else None
        if ev is not None:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(torch.cuda.current_stream())
            self._call(self.lib.ffsr_conv2d, C.byref(p), self._stream)
            e1.record(torch.cuda.current_stream())
            ev.append((e0, e1))
            return
        self._call(self.lib.ffsr_conv2d, C.byref(p), self._stream,
                   label=f"conv {wname} {Cin}->{Cout} k{ks} {H}x{W}" + (" tc" if x.t.dtype == torch.bfloat16 else ""))

    def _lka_block(self, key, blk: str, x: torch.Tensor, name: str, lp: bool = False) -> torch.Tensor:
        """x: [N,H,W,C] fp32 -> LKABlock(x) (large_kernel_attention.py:143-149), eval-mode BN folded.
        lp: the three 1x1 contractions run on tcgen05 with bf16 activations (output bf16)."""
        N, H, W, Cc = x.shape
        dev, w = x.device, self._w
        adt = torch.bfloat16 if lp else torch.float32
        t1 = self._buf(name + ".lka_t1", x.shape, dev)                      # fp32 scratch of the depthwise chain
        t2 = self._buf(name + ".lka_t2", x.shape, dev)
        a = self._buf(name + ".lka_a", x.shape, dev, dtype=adt)
        self._call(self.lib.ffsr_lka_depthwise_in, x.data_ptr(), K.DT_BF16 if x.dtype == torch.bfloat16 else K.DT_F32, N, H, W, Cc,
                   w[key + ".k1"].data_ptr(), w[key + ".d1"].data_ptr(), w[key + ".w5"].data_ptr(), w[key + ".wh"].data_ptr(),
                   w[key + ".wv"].data_ptr(), t1.data_ptr(), t2.data_ptr(), a.data_ptr(),
                   K.DT_BF16 if lp else K.DT_F32, self._stream)
        self.launches += 2
        if not lp and (key + ".tail_w") in w and x.dtype == torch.float32:
            x2 = self._buf(name + ".lka_x2f", x.shape, dev)
            self._call(self.lib.ffsr_lka_tail64, x.data_ptr(), a.data_ptr(), N * H * W, w[key + ".tail_w"].data_ptr(),
                       w[key + ".tail_p"].data_ptr(), self._P[blk + ".scale1"].data_ptr(), self._P[blk + ".scale2"].data_ptr(),
                       x2.data_ptr(), self._stream)
            return x2
        x1 = self._buf(name + ".lka_x1", x.shape, dev, dtype=adt) if lp else t1   # fp32: t1 is free again
        self.conv(nhwc(a), N, H, W, Cc, key + ".pw", Cc, 1, nhwc(x1), epi=K.EPI_LKAGATE, bias_name=key + ".pwb",
                  r1=nhwc(x), sa_ptr=self._P[blk + ".scale1"], ch_k=w[key + ".k1"], ch_d=w[key + ".d1"])
        hdn = self._buf(name + ".lka_h", (N, H, W, 2 * Cc), dev, dtype=adt)
        self.conv(nhwc(x1), N, H, W, Cc, key + ".f0", 2 * Cc, 1, nhwc(hdn), act=K.ACT_GELU, bias_name=key + ".f0b")
        x2 = self._buf(name + ".lka_x2", x.shape, dev, dtype=adt) if lp else t2
        self.conv(nhwc(hdn), N, H, W, 2 * Cc, key + ".f2", Cc, 1, nhwc(x2), epi=K.EPI_RESIDUAL, bias_name=key + ".f2b",
                  r1=nhwc(x1), sa_ptr=self._P[blk + ".scale2"])
        return x2

    def _twiddles(self, n, dev):
        key = (n, str(dev))
        t = self._tw.get(key)
        if t is None:
            t = torch.empty(n, 2, device=dev, dtype=torch.float64)
            self._call(self.lib.ffsr_fft_twiddles, n, t.data_ptr(), self._stream)
            self._tw[key] = t
        return t

    # ------------------------------------------------------------------ forward
    @torch.no_grad()
    def forward(self, lr: torch.Tensor, img_list: List[torch.Tensor], feats: Dict[str, torch.Tensor],
                Hh: int, Wh: int, want_inter: bool, bands: Optional[torch.Tensor] = None):
        """``bands``: phase-2 output [B,9,3,H,W] computed elsewhere (tiled inference crops it from the bands of
        the WHOLE image, because the FFT / DWT bands of a window are not the window of the bands)."""
        m, lib = self.m, self.lib
        if not lr.is_cuda:
            raise RuntimeError("CompleteEnhancedFusionSR (sm_100a build) needs CUDA tensors: there is no CPU path")
        dev = lr.device
        if self._checked_dev != dev:
            with torch.cuda.device(dev):
                K.check(lib.ffsr_device_check(), "device_check")
            self._checked_dev = dev
        if len(img_list) != 4:
            raise ValueError(f"expected the 4 expert outputs drct/grl/nafnet/mamba, got {len(img_list)}")
        B, Cc, H, W = lr.shape
        if Cc != 3 or H < 8 or W < 8:
            raise ValueError("lr_input must be [B,3,H,W] with H,W >= 8 (7-px reflect pad of the db4 DWT)")
        for t in img_list:
            if tuple(t.shape) != (B, 3, 4 * H, 4 * W):
                raise ValueError(f"expert image shape {tuple(t.shape)} != {(B, 3, 4 * H, 4 * W)}")
        with torch.cuda.device(dev):
            entry_stream = torch.cuda.current_stream(dev)
            try:
                return self._forward(lr, img_list, feats, B, H, W, want_inter, bands)
            finally:
                if torch.cuda.current_stream(dev) != entry_stream:      # an error inside the side-stream section
                    torch.cuda.set_stream(entry_stream)

    @torch.no_grad()
    def frequency_bands(self, lr: torch.Tensor) -> torch.Tensor:
        """Phase 2 alone: the nine raw bands [B,9,3,H,W] (dct low/mid/high, dwt LL/LH/HL/HH, fft low/high) of ``lr``."""
        if not lr.is_cuda:
            raise RuntimeError("CompleteEnhancedFusionSR (sm_100a build) needs CUDA tensors: there is no CPU path")
        B, Cc, H, W = lr.shape
        if Cc != 3 or H < 8 or W < 8:
            raise ValueError("lr_input must be [B,3,H,W] with H,W >= 8 (7-px reflect pad of the db4 DWT)")
        dev = lr.device
        with torch.cuda.device(dev):
            self._stream = self._get_stream(dev)
            self._prepare(dev)
            self.launches = 0
            return self._phase2(lr.detach().to(torch.float32).contiguous(), B, H, W, True)

    def _phase2(self, lr, B, H, W, fresh):
        m, lib, P, S, dev = self.m, self.lib, self._P, self._stream, lr.device

        def pp(name):
            return P[name].data_ptr()

        fd = m.freq_decomp
        raw9 = self._buf("raw9", (B, 9, 3, H, W), dev, fresh=fresh)
        self._call(lib.ffsr_dct_bands, lr.data_ptr(), B, H, W, pp("freq_decomp.dct.dct_basis"), pp("freq_decomp.dct.dct_basis_t"),
                   pp("freq_decomp.dct.low_mask"), pp("freq_decomp.dct.mid_mask"), pp("freq_decomp.dct.high_mask"),
                   pp("freq_decomp.dct.band_scale"), raw9.data_ptr(), S)
        hs, ws_ = C.c_int(), C.c_int()
        lib.ffsr_dwt_sub_size(H, W, C.byref(hs), C.byref(ws_))
        sub = self._buf("dwt.sub", (B, 4, 3, hs.value, ws_.value), dev)
        self._call(lib.ffsr_dwt_bands, lr.data_ptr(), B, H, W, pp("freq_decomp.dwt.lo_row"), pp("freq_decomp.dwt.hi_row"),
                   pp("freq_decomp.dwt.lo_col"), pp("freq_decomp.dwt.hi_col"), pp("freq_decomp.dwt.subband_scale"),
                   sub.data_ptr(), raw9.data_ptr(), S)
        self.launches += 1
        fft_bytes = lib.ffsr_fft_workspace_bytes(B, H, W)
        fws = self._buf("fft.ws", (fft_bytes // 8 + 2,), dev, dtype=torch.float64)
        ms = fd.fft.freq_mask_logits.shape[-1]
        self._call(lib.ffsr_fft_bands, lr.data_ptr(), B, H, W, pp("freq_decomp.fft.freq_mask_logits"), ms,
                   pp("freq_decomp.fft.temperature"), pp("freq_decomp.fft.band_scale"), self._twiddles(H, dev).data_ptr(),
                   self._twiddles(W, dev).data_ptr(), fws.data_ptr(), fft_bytes, raw9.data_ptr(), S)
        self.launches += 4
        return raw9

    def _forward(self, lr, img_list, feats, B, H, W, want_inter, bands=None):
        m, lib, w = self.m, self.lib, None
        dev = lr.device
        self._stream = self._get_stream(dev)
        self._prepare(dev)
        w = self._w
        P = self._P

        def pp(name):
            return P[name].data_ptr()

        self.launches = 0
        S = self._stream
        f32 = torch.float32
        if m.precision not in ("fp32", "bf16"):
            raise ValueError(f"precision must be 'fp32' or 'bf16', got {m.precision!r}")
        lp = m.precision == "bf16"          # tcgen05 path for phases 4/5/7; phases 2/3/6 stay fp32
        adt = torch.bfloat16 if lp else f32
        ADT = K.DT_BF16 if lp else K.DT_F32
        esz = 2 if lp else 4
        Hh, Wh = 4 * H, 4 * W
        lr = lr.detach().to(f32).contiguous()            # fp16 caches are up-cast at the boundary (SURVEY App. C)
        imgs = [t.detach().to(f32).contiguous() for t in img_list]
        fr = want_inter                                   # intermediates are handed out: use fresh buffers

        # ---------------- Phase 2 ----------------
        if bands is None:
            raw9 = self._phase2(lr, B, H, W, fr)
        else:
            if tuple(bands.shape) != (B, 9, 3, H, W) or bands.dtype != f32 or bands.device != dev:
                raise ValueError(f"bands must be fp32 [B,9,3,H,W] = {(B, 9, 3, H, W)} on {dev}, got {tuple(bands.shape)}")
            raw9 = bands.contiguous()

        # Phases 3 + 6 (the fp32 LR routing chain: FFMA-bound kernels) only meet the rest of the network at the
        # blend, while phase 4 / the HR modulation / phase 5 depend on the expert features and images alone: run
        # the routing chain on a side stream so its CUDA-core kernels fill the SMs between the short tcgen05 and
        # latency-bound elementwise launches of the main chain.
        main_handle = self._stream
        overlap = self.overlap_routing and not want_inter and lr.is_cuda
        if overlap:
            side = self._side.get(str(dev))
            if side is None:
                side = self._side[str(dev)] = torch.cuda.Stream(dev)
            main_stream = torch.cuda.current_stream(dev)
            ev = torch.cuda.Event()
            ev.record(main_stream)
            side.wait_event(ev)
            torch.cuda.set_stream(side)          # first-use workspace fills of this block must be ordered with it
            S = self._stream = C.c_void_p(side.cuda_stream)

        # ---------------- Phase 3 ----------------
        cb = m.cross_band
        nq = 9 if want_inter else 3                       # bands 3..8 feed nothing downstream (SURVEY App. C)
        tok = self._buf("cb.tok", (B * nq, H, W, 64), dev)
        nsm = self._sm_count(dev)
        self._call(lib.ffsr_crossband_attention, raw9.data_ptr(), B, H, W, w["cb.proj_w"].data_ptr(),
                   pp("cross_band.band_proj.bias"), pp("cross_band.band_attention.out_proj.weight"),
                   pp("cross_band.band_attention.out_proj.bias"), nq, tok.data_ptr(), nsm, w["cb.fold"].data_ptr(), S)
        x2 = self._lka_block("cb.lka", "cross_band.lka_block", tok, "cb%d" % nq)
        enh9 = self._buf("enh9", (B, 9, 3, H, W), dev, fresh=fr)
        routing = self._buf("routing", (B, 3, H, W), dev, fresh=fr)
        self._call(lib.ffsr_crossband_out, x2.data_ptr(), raw9.data_ptr(), B, H, W, nq, w["cb.out_w"].data_ptr(),
                   pp("cross_band.out_proj.bias"), enh9.data_ptr(), routing.data_ptr(), S)

        # ---------------- Phase 6 (selector nets, fp32) ----------------
        ds = m.dynamic_selector
        s_a = self._buf("ds.a", (B, H, W, 32), dev)
        s_b = self._buf("ds.b", (B, H, W, 32), dev)
        diff = self._buf("diff", (B, 1, H, W), dev, fresh=fr)
        graw = self._buf("ds.raw", (B, H, W, 4), dev)
        gates = self._buf("gates", (B, 4, H, W), dev, fresh=fr)
        rv = nchw(routing)
        if self.selector_fused and "ds.blob" in w:
            self._call(lib.ffsr_selector_fused, routing.data_ptr(), B, H, W, w["ds.blob"].data_ptr(), pp("dynamic_selector.temperature"),
                       diff.data_ptr(), graw.data_ptr(), gates.data_ptr(), S)
        else:
          self.conv(rv, B, H, W, 3, "ds.d0", 32, 3, nhwc(s_a), act=K.ACT_RELU)
          self.conv(nhwc(s_a), B, H, W, 32, "ds.d2", 32, 3, nhwc(s_b), act=K.ACT_RELU)
          self.conv(nhwc(s_b), B, H, W, 32, "ds.d4", 1, 3, nhwc(diff.view(B, H, W, 1)), act=K.ACT_SIGMOID)
          self.conv(rv, B, H, W, 3, "ds.g0", 32, 3, nhwc(s_a), act=K.ACT_RELU)
          self.conv(nhwc(s_a), B, H, W, 32, "ds.g2", 32, 3, nhwc(s_b), act=K.ACT_RELU)
          self.conv(nhwc(s_b), B, H, W, 32, "ds.g4", 4, 1, nhwc(graw))
          self._call(lib.ffsr_gate_finalize, graw.data_ptr(), diff.data_ptr(), B, H, W, pp("dynamic_selector.temperature"),
                     gates.data_ptr(), S)

        if overlap:
            routing_done = torch.cuda.Event()
            routing_done.record(side)
            torch.cuda.set_stream(main_stream)
            S = self._stream = main_handle

        # ---------------- Phase 4 (LR part) ----------------
        co = m.collaborative
        have = [n for n in EXPERT_ORDER if n in feats]
        m32 = None
        if have:
            for n in have:
                f = feats[n]
                if f.dim() != 4 or f.shape[0] != B:
                    raise ValueError(f"expert feature '{n}' has shape {tuple(f.shape)}; expected [B={B}, C, h, w]")
            # Feature maps of different spatial sizes are brought to the smallest one (large_kernel_attention.py:365-372).
            # The reference resizes AFTER the 1x1 align conv; a 1x1 conv (bias included: bilinear weights sum to 1) commutes
            # with bilinear resampling, so the raw features are resized instead and the usual align path follows.  Phase 4
            # then runs on that (Hq, Wq) grid, which need not be the LR grid; the modulation kernel upsamples it to HR.
            Hq, Wq = min(feats[n].shape[2] for n in have), min(feats[n].shape[3] for n in have)
            if any(tuple(feats[n].shape[2:]) != (Hq, Wq) for n in have):
                feats = dict(feats)
                for n in have:
                    f = feats[n]
                    if tuple(f.shape[2:]) != (Hq, Wq):
                        src = f.detach().to(f32).permute(0, 2, 3, 1).contiguous()
                        dst = torch.empty(B, Hq, Wq, f.shape[1], device=dev, dtype=f32)
                        self._call(lib.ffsr_bilinear_forward, src.data_ptr(), B, f.shape[2], f.shape[3], f.shape[1],
                                   dst.data_ptr(), Hq, Wq, K.DT_F32, S)
                        feats[n] = dst.permute(0, 3, 1, 2).contiguous()
            # bf16 mode: the residual stream (tokens, t1, t2) is stored as bf16 -- every Phase-4 launch is bound by the HBM
            # round trip of these [4][H][W][128] tensors, and the phase only feeds a sigmoid damped by 0.2
            cin_exp = {n: co.align_layers[n].weight.shape[1] for n in EXPERT_ORDER}
            fast_align = lp and len(have) == 4 and all(feats[n].shape[1] == cin_exp[n] for n in EXPERT_ORDER)
            rdt = torch.bfloat16 if fast_align else f32
            tokens = self._buf("co.tok", (B, 4, Hq, Wq, 128), dev, dtype=rdt, zero=True)
            if fast_align and "co.align_w" in w:
                # NCHW fp32 features -> aligned bf16 tokens in one tile-resident kernel (csrc/token_chain.cu, k_align_tokens)
                fl = [feats[n].detach().to(f32).contiguous() for n in EXPERT_ORDER]
                fptr = (C.c_void_p * 4)(*[t.data_ptr() for t in fl])
                cnum = (C.c_int * 4)(*[cin_exp[n] for n in EXPERT_ORDER])
                self._call(lib.ffsr_align_tokens, fptr, cnum, B, Hq * Wq, w["co.align_w"].data_ptr(), w["co.align_b"].data_ptr(),
                           tokens.data_ptr(), S)
            else:
                if len(have) < 4:
                    tokens.zero_()                              # missing expert -> zero token (:378-381)
                for e, n in enumerate(EXPERT_ORDER):
                    if n not in feats:
                        continue
                    f = feats[n].detach().to(f32).contiguous()
                    cin_w = cin_exp[n]
                    cin = min(f.shape[1], cin_w)               # truncate / implicit zero-pad (:349-358)
                    wn = "co.align." + n
                    if cin != cin_w:
                        wn2 = wn + ".c%d" % cin
                        if wn2 not in w:
                            w[wn2] = w[wn][:, :cin, :].contiguous()
                            w[wn2 + ".b"] = w[wn + ".b"]
                        wn = wn2
                    tv = tokens[:, e]
                    ov = _View(tv.data_ptr(), tokens.stride(0), tokens.stride(2), tokens.stride(3), 1, tokens)
                    self.conv(nchw(f), B, Hq, Wq, cin, wn, 128, 1, ov)
            N4 = B * 4
            tok4 = tokens.view(N4, Hq, Wq, 128)
            rows = N4 * Hq * Wq
            n1 = self._buf("co.n", (N4, Hq, Wq, 128), dev, dtype=adt)
            def layernorm(src, wn, bn):
                if src.dtype == torch.bfloat16:
                    self._call(lib.ffsr_layernorm128_bf16, src.data_ptr(), rows, pp(wn), pp(bn), n1.data_ptr(), S)
                else:
                    self._call(lib.ffsr_layernorm, src.data_ptr(), rows, 128, pp(wn), pp(bn), n1.data_ptr(), int(lp), S)

            t1 = self._buf("co.t1", (N4, Hq, Wq, 128), dev, dtype=rdt)
            t2 = self._buf("co.t2", (N4, Hq, Wq, 128), dev, dtype=rdt)
            if lp and self.token_chain and rdt == torch.bfloat16 and "co.attn_w" in w:
                # LN1 -> qkv -> 4-token attention -> out_proj + residual, then LN2 -> ffn0 -> GELU -> ffn2 + residual: two
                # tile-resident tcgen05 kernels instead of seven launches (csrc/token_chain.cu)
                self._call(lib.ffsr_token_attn_chain, tok4.data_ptr(), B, Hq * Wq, w["co.attn_w"].data_ptr(), w["co.attn_p"].data_ptr(),
                           t1.data_ptr(), S)
                self._call(lib.ffsr_token_ffn_chain, t1.data_ptr(), rows, w["co.ffn_w"].data_ptr(), w["co.ffn_p"].data_ptr(),
                           t2.data_ptr(), S)
            else:
                layernorm(tok4, "collaborative.norm1.weight", "collaborative.norm1.bias")
                qkv = self._buf("co.qkv", (N4, Hq, Wq, 384), dev, dtype=adt)
                self.conv(nhwc(n1), N4, Hq, Wq, 128, "co.qkv", 384, 1, nhwc(qkv))
                ctx = self._buf("co.ctx", (N4, Hq, Wq, 128), dev, dtype=adt)
                self._call(lib.ffsr_token_attention, qkv.data_ptr(), B, 4, Hq * Wq, 128, ctx.data_ptr(), int(lp), S)
                self.conv(nhwc(ctx), N4, Hq, Wq, 128, "co.out", 128, 1, nhwc(t1), epi=K.EPI_RESIDUAL, r1=nhwc(tok4))
                layernorm(t1, "collaborative.norm2.weight", "collaborative.norm2.bias")
                hdn = self._buf("co.h", (N4, Hq, Wq, 256), dev, dtype=adt)
                self.conv(nhwc(n1), N4, Hq, Wq, 128, "co.f0", 256, 1, nhwc(hdn), act=K.ACT_GELU)
                self.conv(nhwc(hdn), N4, Hq, Wq, 256, "co.f2", 128, 1, nhwc(t2), epi=K.EPI_RESIDUAL, r1=nhwc(t1))
            m32 = self._buf("co.m32", (N4, Hq, Wq, 32), dev, dtype=adt if (Hq, Wq) == (H, W) else f32)
            if lp and "co.tail_w" in w and t2.dtype == torch.bfloat16 and m32.dtype == torch.bfloat16:
                # depthwise chain, then ONE tile-resident kernel: pw + gate, ffn0 + GELU, ffn2 + residual, modulation layer 0
                ta = self._buf("co.lka_t1", t2.shape, dev)
                tb = self._buf("co.lka_t2", t2.shape, dev)
                a_ = self._buf("co.lka_a", t2.shape, dev, dtype=adt)
                self._call(lib.ffsr_lka_depthwise_in, t2.data_ptr(), K.DT_BF16, N4, Hq, Wq, 128, w["co.lka.k1"].data_ptr(),
                           w["co.lka.d1"].data_ptr(), w["co.lka.w5"].data_ptr(), w["co.lka.wh"].data_ptr(), w["co.lka.wv"].data_ptr(),
                           ta.data_ptr(), tb.data_ptr(), a_.data_ptr(), K.DT_BF16, S)
                self.launches += 2
                self._call(lib.ffsr_lka_tail128_mod, t2.data_ptr(), a_.data_ptr(), N4, Hq * Wq, w["co.tail_w"].data_ptr(),
                           w["co.tail_p"].data_ptr(), P["collaborative.lka_global.scale1"].data_ptr(),
                           P["collaborative.lka_global.scale2"].data_ptr(), m32.data_ptr(), S)
            else:
                xg = self._lka_block("co.lka", "collaborative.lka_global", t2, "co", lp=lp)
                self.conv(nhwc(xg), N4, Hq, Wq, 128, "co.m0", 32, 1, nhwc(m32), groups=4, bias_name="co.m0b")

        # ---------------- HR: modulation + expert pyramid ----------------
        ecol = self._buf("ecol", (B, 4, 3, Hh, Wh), dev, fresh=fr)
        cat3 = self._buf("cat3", (B, Hh, Wh, 80), dev, dtype=adt, zero=True)
        cat2 = self._buf("cat2", (B, 2 * H, 2 * W, 80), dev, dtype=adt, zero=True)
        s1in = self._buf("s1in", (B, H, W, 16), dev, dtype=adt, zero=True)
        ptrs = (C.c_void_p * 4)(*[t.data_ptr() for t in imgs])
        if m32 is not None and tuple(m32.shape[1:3]) != (H, W):
            self._call(lib.ffsr_modulate_hr_sized, ptrs, m32.data_ptr(), m32.shape[1], m32.shape[2], w["co.m2"].data_ptr(),
                       w["co.m2b"].data_ptr(), B, H, W, 0 if m.training else 1, ecol.data_ptr(), cat3.data_ptr() + 64 * esz, 80, ADT, S)
        elif m32 is not None:
            self._call(lib.ffsr_modulate_hr_v2, ptrs, m32.data_ptr(), K.DT_BF16 if m32.dtype == torch.bfloat16 else K.DT_F32,
                       w["co.m2"].data_ptr(), w["co.m2b"].data_ptr(), B, H, W, 0 if m.training else 1, ecol.data_ptr(),
                       cat3.data_ptr() + 64 * esz, 80, ADT, S)
        else:
            self._call(lib.ffsr_modulate_hr, ptrs, None, w["co.m2"].data_ptr(), w["co.m2b"].data_ptr(), B, H, W,
                       0 if m.training else 1, ecol.data_ptr(), cat3.data_ptr() + 64 * esz, 80, ADT, S)
        self._call(lib.ffsr_expert_downsample, ecol.data_ptr(), B, Hh, Wh, cat2.data_ptr() + 64 * esz, 80,
                   s1in.data_ptr(), 16, ADT, S)

        # ---------------- Phase 5: hierarchical fusion ----------------
        mr = m.multi_res

        def stage(name, xin: _View, cin, h, wd, c_mid, c_out, r2=None, sb_ptr=None):
            a = self._buf(name + ".a", (B, h, wd, c_mid), dev, dtype=adt)
            b_ = self._buf(name + ".b", (B, h, wd, c_out), dev, dtype=adt)
            c_ = self._buf(name + ".c", (B, h, wd, c_out), dev, dtype=adt)
            self.conv(xin, B, h, wd, cin, f"mr.{name}.c0", c_mid, 3, nhwc(a), act=K.ACT_GELU)
            self.conv(nhwc(a), B, h, wd, c_mid, f"mr.{name}.c2", c_out, 3, nhwc(b_), act=K.ACT_GELU)
            g = getattr(mr, name + "_gate").gate
            self._call(lib.ffsr_spatial_gate, b_.data_ptr(), B * h * wd, c_out, w[f"mr.{name}.g0"].data_ptr(),
                       pp(f"multi_res.{name}_gate.gate.0.bias"), w[f"mr.{name}.g2"].data_ptr(), pp(f"multi_res.{name}_gate.gate.2.bias"), b_.data_ptr(),
                       ADT, S)
            d_ = self._buf(name + ".d", (B, h, wd, c_out), dev, dtype=adt)
            self.conv(nhwc(b_), B, h, wd, c_out, f"mr.{name}.r0", c_out, 3, nhwc(d_), act=K.ACT_GELU, bias=False)
            self.conv(nhwc(d_), B, h, wd, c_out, f"mr.{name}.r2", c_out, 3, nhwc(c_), bias=False, epi=K.EPI_RESIDUAL,
                      r1=nhwc(b_), sa_ptr=P[f"multi_res.{name}_res.scale"], r2=r2, sb_ptr=sb_ptr)
            return c_

        f1 = stage("stage1", nhwc(s1in), 12, H, W, 64, 64)
        self._call(lib.ffsr_resize_nhwc, f1.data_ptr(), B, H, W, 64, 64, cat2.data_ptr(), 2 * H, 2 * W, 80, ADT, S)
        f2 = stage("stage2", nhwc(cat2), 76, 2 * H, 2 * W, 64, 64, r2=nhwc(cat2), sb_ptr=P["multi_res.residual_weight_1_2"])
        self._call(lib.ffsr_resize_nhwc, f2.data_ptr(), B, 2 * H, 2 * W, 64, 64, cat3.data_ptr(), Hh, Wh, 80, ADT, S)
        f3 = stage("stage3", nhwc(cat3), 76, Hh, Wh, 64, 32, r2=nhwc(cat3), sb_ptr=P["multi_res.residual_weight_2_3"])
        u16 = self._buf("mr.u16", (B, Hh, Wh, 16), dev, dtype=adt)
        hier = self._buf("mr.hier", (B, Hh, Wh, 4), dev, zero=True)
        self.conv(nhwc(f3), B, Hh, Wh, 32, "mr.rgb0", 16, 3, nhwc(u16), act=K.ACT_GELU)
        self.conv(nhwc(u16), B, Hh, Wh, 16, "mr.rgb2", 3, 3, nhwc(hier), act=K.ACT_SIGMOID)

        if overlap:
            torch.cuda.current_stream(dev).wait_event(routing_done)

        # ---------------- Phase 5b / 6 blend ----------------
        fused_before = torch.empty(B, 3, Hh, Wh, device=dev, dtype=f32) if want_inter else None
        fusedx = self._buf("fusedx", (B, Hh, Wh, 4), dev, zero=True)
        fused_lp = self._buf("fused_lp", (B, Hh, Wh, 16), dev, dtype=torch.bfloat16, zero=True) if lp else None
        self._call(lib.ffsr_blend_hr, hier.data_ptr(), 4, ecol.data_ptr(), routing.data_ptr(), gates.data_ptr(),
                   diff.data_ptr(), w["fw0"].data_ptr(), pp("freq_weight_conv.0.bias"), w["fw2"].data_ptr(),
                   pp("freq_weight_conv.2.bias"), B, H, W,
                   fused_before.data_ptr() if fused_before is not None else None, fusedx.data_ptr(), 4,
                   fused_lp.data_ptr() if lp else None, 16 if lp else 0, S)

        # ---------------- Phase 7a: refinement ----------------
        idx = self._refine_idx
        rc = m.refine[idx[0]].weight.shape[0]
        ping = self._buf("rf.ping", (B, Hh, Wh, rc), dev, dtype=adt)
        pong = self._buf("rf.pong", (B, Hh, Wh, rc), dev, dtype=adt)
        cat6 = self._buf("cat6", (B, Hh, Wh, 8), dev, zero=True)
        self.conv(nhwc(fused_lp if lp else fusedx), B, Hh, Wh, 3, f"rf.{idx[0]}", rc, 3, nhwc(ping), act=K.ACT_GELU)
        cur, nxt = ping, pong
        for i in idx[1:-1]:
            self.conv(nhwc(cur), B, Hh, Wh, rc, f"rf.{i}", rc, 3, nhwc(nxt), act=K.ACT_GELU)
            cur, nxt = nxt, cur
        self.conv(nhwc(cur), B, Hh, Wh, rc, f"rf.{idx[-1]}", 3, 3, nhwc(cat6), epi=K.EPI_RESIDUAL, r1=nhwc(fusedx), sa=0.1)

        # ---------------- Phase 7b: Laplacian pyramid edge enhancement ----------------
        ee = m.edge_enhance
        g25 = w["ee.gauss"].data_ptr()
        down1 = self._buf("ee.down1", (B, 2 * H, 2 * W, 4), dev, zero=True)
        down2 = self._buf("ee.down2", (B, H, W, 4), dev, zero=True)
        lap0 = self._buf("ee.lap0", (B, Hh, Wh, 4), dev, zero=True)
        lap1 = self._buf("ee.lap1", (B, 2 * H, 2 * W, 4), dev, zero=True)
        bf = torch.bfloat16
        lap0_lp = self._buf("ee.lap0_lp", (B, Hh, Wh, 8), dev, dtype=bf, zero=True) if lp else None
        lap1_lp = self._buf("ee.lap1_lp", (B, 2 * H, 2 * W, 8), dev, dtype=bf, zero=True) if lp else None
        down2_lp = self._buf("ee.down2_lp", (B, H, W, 8), dev, dtype=bf, zero=True) if lp else None

        def ptr(t):
            return t.data_ptr() if t is not None else None

        self._call(lib.ffsr_blur_pool, cat6.data_ptr(), 8, B, Hh, Wh, g25, down1.data_ptr(), 4, None, 0, S)
        self._call(lib.ffsr_laplacian_sub, cat6.data_ptr(), 8, down1.data_ptr(), 4, B, Hh, Wh, lap0.data_ptr(), 4,
                   ptr(lap0_lp), 8, S)
        self._call(lib.ffsr_blur_pool, down1.data_ptr(), 4, B, 2 * H, 2 * W, g25, down2.data_ptr(), 4, ptr(down2_lp), 8, S)
        self._call(lib.ffsr_laplacian_sub, down1.data_ptr(), 4, down2.data_ptr(), 4, B, 2 * H, 2 * W, lap1.data_ptr(), 4,
                   ptr(lap1_lp), 8, S)
        cat96 = self._buf("ee.cat96", (B, Hh, Wh, 96), dev, dtype=adt)
        levels = ((lap0, lap0_lp, Hh, Wh), (lap1, lap1_lp, 2 * H, 2 * W), (down2, down2_lp, H, W))
        for lv, (lap, lap_lp, h, wd) in enumerate(levels):
            nm = f"ee{lv}"
            src = lap_lp if lp else lap                       # bf16 mode: every refiner conv is a tcgen05 launch
            if lp and self.edge_chain and f"ee.{lv}.chain_w" in w:
                # one tile-resident kernel per level; level 0 writes its weighted product straight into the concat slice
                cw, cp = w[f"ee.{lv}.chain_w"], w[f"ee.{lv}.chain_p"]
                if lv == 0:
                    self._call(lib.ffsr_edge_refiner_chain, src.data_ptr(), B, h, wd, cw.data_ptr(), cp.data_ptr(),
                               pp("edge_enhance.level_weights"), 0, cat96.data_ptr(), Hh * Wh * 96, Wh * 96, 96, None, 0, S)
                else:
                    o3 = self._buf(nm + ".o3", (B, h, wd, 32), dev, dtype=adt)
                    at = self._buf(nm + ".at", (B, h, wd, 1), dev)
                    self._call(lib.ffsr_edge_refiner_chain, src.data_ptr(), B, h, wd, cw.data_ptr(), cp.data_ptr(),
                               None, lv, o3.data_ptr(), h * wd * 32, wd * 32, 32, at.data_ptr(), 1, S)
                    self._call(lib.ffsr_edge_attn_upsample, o3.data_ptr(), ADT, at.data_ptr(), B, h, wd, 32,
                               pp("edge_enhance.level_weights"), lv, cat96.data_ptr() + 32 * lv * esz, Hh, Wh, 96, ADT, S)
                continue
            idt = self._buf(nm + ".idt", (B, h, wd, 32), dev)
            o1 = self._buf(nm + ".o1", (B, h, wd, 32), dev, dtype=adt)
            o2 = self._buf(nm + ".o2", (B, h, wd, 32), dev, dtype=adt)
            o3 = self._buf(nm + ".o3", (B, h, wd, 32), dev, dtype=adt) if lp else o1
            t8 = self._buf(nm + ".t8", (B, h, wd, 8), dev, dtype=adt)
            at = self._buf(nm + ".at", (B, h, wd, 1), dev)
            self.conv(nhwc(src), B, h, wd, 3, f"ee.{lv}.proj", 32, 1, nhwc(idt))
            self.conv(nhwc(src), B, h, wd, 3, f"ee.{lv}.c1", 32, 3, nhwc(o1), act=K.ACT_GELU)
            self.conv(nhwc(o1), B, h, wd, 32, f"ee.{lv}.c2", 32, 3, nhwc(o2), act=K.ACT_GELU)
            self.conv(nhwc(o2), B, h, wd, 32, f"ee.{lv}.c3", 32, 3, nhwc(o3), epi=K.EPI_RESIDUAL, r1=nhwc(idt))
            self.conv(nhwc(o3), B, h, wd, 32, f"ee.{lv}.a0", 8, 1, nhwc(t8), act=K.ACT_GELU)
            self.conv(nhwc(t8), B, h, wd, 8, f"ee.{lv}.a2", 1, 3, nhwc(at), act=K.ACT_SIGMOID)
            self._call(lib.ffsr_edge_attn_upsample, o3.data_ptr(), ADT, at.data_ptr(), B, h, wd, 32,
                       pp("edge_enhance.level_weights"), lv, cat96.data_ptr() + 32 * lv * esz, Hh, Wh, 96, ADT, S)
        e32 = self._buf("ee.e32", (B, Hh, Wh, 32), dev, dtype=adt)
        self.conv(nhwc(cat96), B, Hh, Wh, 96, "ee.f0", 32, 3, nhwc(e32), act=K.ACT_GELU)
        self.conv(nhwc(e32), B, Hh, Wh, 32, "ee.f2", 3, 3, nhwc(cat6, 3))
        g16 = self._buf("ee.g16", (B, Hh, Wh, 16), dev, dtype=adt)
        egate = self._buf("ee.gate", (B, Hh, Wh, 1), dev)
        gin = cat6
        if lp:
            gin = self._buf("cat6_lp", (B, Hh, Wh, 8), dev, dtype=bf, zero=True)
            self._call(lib.ffsr_cast_f32_to_bf16, cat6.data_ptr(), gin.data_ptr(), cat6.numel(), S)
        self.conv(nhwc(gin), B, Hh, Wh, 6, "ee.g0", 16, 3, nhwc(g16), act=K.ACT_GELU)
        self.conv(nhwc(g16), B, Hh, Wh, 16, "ee.g2", 1, 3, nhwc(egate), act=K.ACT_SIGMOID)

        # ---------------- output ----------------
        out = torch.empty(B, 3, Hh, Wh, device=dev, dtype=f32)
        self._call(lib.ffsr_final_combine, cat6.data_ptr(), 8, egate.data_ptr(), pp("edge_enhance.edge_strength"),
                   lr.data_ptr(), pp("residual_scale"), B, H, W, 0 if m.training else 1, out.data_ptr(), S)

        inter = {}
        if want_inter:
            inter["raw_9_bands"] = [raw9[:, i] for i in range(9)]
            inter["guidance_bands"] = inter["raw_9_bands"][:3]
            inter["enhanced_9_bands"] = [enh9[:, i] for i in range(9)]
            inter["routing_lr"] = routing
            if m32 is not None:
                inter["collaborative_outputs"] = [ecol[:, e] for e in range(4)]
            inter["fused_before_dynamic"] = fused_before
            inter["gates"] = gates
            inter["difficulty"] = diff
            # beyond the reference's dict: the raw selector logits and the second derived index of SURVEY §8a-P6,
            # active = gate_net(r) > 0.7 - 0.5 * difficulty_net(r)   (enhanced_fusion_v2.py:450-466)
            inter["gate_logits"] = graw.permute(0, 3, 1, 2).clone()
            inter["active"] = inter["gate_logits"] > (0.7 - 0.5 * diff)
        return out, inter
