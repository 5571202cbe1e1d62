"""DRCT-L window attention (SURVEY §8f N1): the (shifted-)window attention core of every SwinTransformerBlock against a
torch restatement of drct_arch.py (itself checked against the oracle block on the CPU); the tcgen05 kernels of window 16
against an fp64 emulation of what they compute; whole DRCT forwards against the oracle in fp64; argument validation on
the CPU."""
import ctypes as C
import math
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import isr_b200  # noqa: E402,F401
from isr_b200 import _cabi as K  # noqa: E402
from oracle import drct_oracle as DO  # noqa: E402


def expected_attention(qkv: torch.Tensor, heads: int, ws: int, shift: int, table: torch.Tensor) -> torch.Tensor:
    """drct_arch.py:385-412 around WindowAttention.forward :175-206 without the two Linears (torch ops, fp32)."""
    B, H, W, C3 = qkv.shape
    Cc = C3 // 3
    dh, N = Cc // heads, ws * ws
    x = torch.roll(qkv, shifts=(-shift, -shift), dims=(1, 2)) if shift else qkv
    xw = DO._partition(x, ws).view(-1, N, 3, heads, dh).permute(2, 0, 3, 1, 4)
    q, k, v = xw[0] * dh ** -0.5, xw[1], xw[2]
    attn = q @ k.transpose(-2, -1)
    bias = table[DO.relative_position_index(ws).view(-1)].view(N, N, -1).permute(2, 0, 1)
    attn = attn + bias.unsqueeze(0)
    if shift:
        mask = DO.shift_mask(H, W, ws, shift).to(attn)
        nW = mask.shape[0]
        attn = (attn.view(-1, nW, heads, N, N) + mask.unsqueeze(1).unsqueeze(0)).view(-1, heads, N, N)
    out = (attn.softmax(-1) @ v).transpose(1, 2).reshape(-1, ws, ws, Cc)
    out = DO._reverse(out, ws, H, W)
    return torch.roll(out, shifts=(shift, shift), dims=(1, 2)) if shift else out


L2E = 1.4426950408889634


def bf16_ulp(x: torch.Tensor) -> torch.Tensor:
    """One bf16 ulp at |x| (0 at 0)."""
    _, e = torch.frexp(x)
    return torch.where(x == 0, torch.zeros_like(x), torch.ldexp(torch.ones_like(x), e - 8))


def _bf16(t: torch.Tensor) -> torch.Tensor:
    return t.float().bfloat16().double()


def window16_reference(qkv: torch.Tensor, heads: int, shift: int, table: torch.Tensor, bf16_p: bool = True):
    """fp64 emulation of the 16 x 16 window attention kernels on bf16 qkv rows ([B,H,W,3C], the reference's [3][heads][dh]
    channel order) and a bound on their error.  Returns (out, tol), both [B,H,W,C] float64 on qkv's device.

    bf16_p=True is k_window_attn_tc (csrc/window_attention_tc.cu): scores s = q.k of the bf16 operands; the kernel's own
    shift m = max_k(s) scale log2e + max(table) log2e; p = 2^(s scale log2e + bias log2e - m), -100 log2e on masked keys;
    P rounded to bf16 (RNE) for P.V, divided by the sum of the unrounded p.  bf16_p=False is the fp32 softmax of the
    CUDA-core kernel (csrc/window_attention.cu), i.e. the exact softmax.

    tol is derived from the arithmetic, not fitted:
      * 1 bf16 ulp of |out|: 0.5 for the rounding of the output, the rest for the relative error of the row sum and 1/sum;
      * 2^-14 max|v| (window and head): fp32 accumulation of P.V over 256 keys is within 2^-16 of sum P|v|;
      * eta, the relative error of an fp32 p: the exponent's error in log2 units -- fp32 accumulation of the scores
        (<= (dh + 8) 2^-24 scale log2e sum_i |q_i k_i| with rsqrtf and the log2e product, for the key and for the row
        maximum) and four fp32 roundings of the bias / shift terms (2^-22 (|bias| + |m| + |exponent|)) -- times ln 2, plus
        2^-21 for ex2.approx / expf.  bf16 P: a key whose p lies within eta of a bf16 rounding boundary may round the other
        way, one bf16 ulp of p times |v| each.  fp32 P: 2 eta p |v| per key (numerator and row sum).
    """
    ws, N = 16, 256
    B, H, W, C3 = qkv.shape
    Cc = C3 // 3
    dh = Cc // heads
    nW = (H // ws) * (W // ws)
    x = torch.roll(qkv.double(), (-shift, -shift), (1, 2)) if shift else qkv.double()
    q, k, v = DO._partition(x, ws).view(-1, N, 3, heads, dh).permute(2, 0, 3, 1, 4)       # [B nW, heads, N, dh] each
    tbl = table.to(x.device, torch.float64)
    scale2 = dh ** -0.5 * L2E
    s = q @ k.transpose(-2, -1)
    bias = tbl[DO.relative_position_index(ws).view(-1)].view(N, N, heads).permute(2, 0, 1) * L2E
    m = s.amax(-1, keepdim=True) * scale2 + tbl.amax(0).view(heads, 1, 1) * L2E
    a = s * scale2 + bias - m
    if shift:
        a = (a.view(B, nW, heads, N, N) + DO.shift_mask(H, W, ws, shift).to(a).view(1, nW, 1, N, N) * L2E).view_as(a)
    p = torch.exp2(a)
    den = p.sum(-1, keepdim=True)
    out = (_bf16(p) if bf16_p else p) @ v / den
    sa = q.abs() @ k.abs().transpose(-2, -1)
    eta = ((dh + 8) * 2.0 ** -24 * scale2 * (sa + sa.amax(-1, keepdim=True)) + 2.0 ** -22 * (bias.abs() + m.abs() + a.abs())) \
        * math.log(2) + 2.0 ** -21
    if bf16_p:
        spread = (_bf16(p * (1 + eta)) - _bf16(p * (1 - eta))) @ v.abs() / den            # 0 where the rounding is unambiguous
    else:
        spread = 2 * (eta * p) @ v.abs() / den
    tol = bf16_ulp(out) + 2.0 ** -14 * v.abs().amax((-2, -1), keepdim=True) + spread

    def merge(t):
        t = DO._reverse(t.transpose(1, 2).reshape(-1, ws, ws, Cc), ws, H, W)
        return torch.roll(t, (shift, shift), (1, 2)) if shift else t
    return merge(out), merge(tol)


def assert_within(got: torch.Tensor, ref: torch.Tensor, tol: torch.Tensor, what) -> float:
    """|got - ref| <= tol everywhere; returns (and prints) the worst err / tol."""
    assert bool(torch.isfinite(got).all()), (what, "non-finite output")
    err = (got.double() - ref).abs()
    worst = float((err / tol).max())
    print(f"{what}: max|err| {float(err.max()):.3e}, worst err/tol {worst:.3f}")
    assert worst <= 1.0, (what, worst)
    return worst


def headpad_rows(qkv: torch.Tensor, heads: int) -> torch.Tensor:
    """[B,H,W,3C] rows in the [3][heads][dh] order -> the head-padded rows [3][heads][DP] (DP = dh rounded up to 16, zeros)."""
    B, H, W, C3 = qkv.shape
    dh = C3 // 3 // heads
    DP = (dh + 15) // 16 * 16
    out = torch.zeros(B, H, W, 3, heads, DP, dtype=qkv.dtype, device=qkv.device)
    out[..., :dh] = qkv.view(B, H, W, 3, heads, dh)
    return out.view(B, H, W, 3 * heads * DP)


def test_window16_reference_is_the_plain_attention():
    """The fp64 emulation of the window-16 kernels means what expected_attention means: without the bf16 rounding of P
    (its only approximation) the two agree to fp64 rounding, shifted or not, on a non-square window grid; its bound
    is positive and far below the 2e-2 of the semantic checks."""
    g = torch.Generator().manual_seed(3)
    heads = 2
    qkv = torch.randn(2, 16, 48, 3 * 40, generator=g).bfloat16()
    table = 0.5 * torch.randn(31 * 31, heads, generator=g)
    for shift in (0, 8, 3):
        want = expected_attention(qkv.double(), heads, 16, shift, table.double())
        got, tol = window16_reference(qkv, heads, shift, table, bf16_p=False)
        assert float((got - want).abs().max()) < 1e-12, shift
        got16, tol16 = window16_reference(qkv, heads, shift, table)
        assert float((got16 - want).abs().max()) < 2e-2 and bool((tol16 > 0).all()) and float(tol16.max()) < 2e-2, shift


def test_expected_attention_is_the_oracle_block_without_linears():
    """The torch restatement used as the checker equals oracle.swin_block's attention core (identity qkv / proj)."""
    torch.manual_seed(0)
    Cc, heads, ws = 12, 2, 4
    H, W = 8, 12
    x = torch.randn(1, H, W, Cc)
    Wqkv = torch.randn(3 * Cc, Cc) / Cc ** 0.5
    table = 0.5 * torch.randn((2 * ws - 1) ** 2, heads)
    for shift in (0, 2):
        sd = {"a.qkv.weight": Wqkv, "a.qkv.bias": torch.zeros(3 * Cc), "a.proj.weight": torch.eye(Cc), "a.proj.bias": torch.zeros(Cc),
              "a.relative_position_bias_table": table, "a.relative_position_index": DO.relative_position_index(ws)}
        h = torch.roll(x, (-shift, -shift), (1, 2)) if shift else x
        mask = DO.shift_mask(H, W, ws, shift) if shift else None
        want = DO._reverse(DO.window_attention(sd, "a", DO._partition(h, ws).view(-1, ws * ws, Cc), mask).view(-1, ws, ws, Cc), ws, H, W)
        want = torch.roll(want, (shift, shift), (1, 2)) if shift else want
        got = expected_attention(torch.nn.functional.linear(x, Wqkv), heads, ws, shift, table)
        assert float((got - want).abs().max()) < 1e-5


def test_window_attention_rejects_bad_arguments():
    lib = K.load()
    f = lib.ffsr_window_attention
    ok = (4096, 1, 16, 16, 180, 6, 8, 4, 4096, 4096, K.DT_F32, None)
    bad = [
        (0,) + ok[1:],                                        # null qkv
        ok[:2] + (15,) + ok[3:],                              # H not a multiple of the window
        ok[:5] + (7,) + ok[6:],                               # C % heads != 0
        ok[:6] + (17,) + ok[7:],                              # window^2 > 256
        ok[:7] + (8,) + ok[8:],                               # shift >= window
        ok[:10] + (K.DT_F16,) + ok[11:],                      # unsupported dtype
    ]
    for a in bad:
        assert f(*a) == -1, a
    assert b"window_attention" in lib.ffsr_last_error()


def test_headpadded_window_attention_rejects_bad_arguments():
    """Every check runs before a launch, so no device is needed (none of the calls below passes them)."""
    lib = K.load()
    assert [lib.ffsr_window_attention_head_pad(d) for d in (1, 8, 16, 17, 30, 53, 122, 128)] == [16, 16, 16, 32, 32, 64, 128, 128]
    f = lib.ffsr_window_attention_headpadded
    ok = (4096, 1, 16, 16, 180, 6, 16, 8, 4096, 4096, 184, None)
    bad = [
        ((0,) + ok[1:], -1),                                  # null qkv
        (ok[:8] + (0,) + ok[9:], -1),                         # null bias table
        (ok[:9] + (0,) + ok[10:], -1),                        # null out
        (ok[:6] + (8,) + ok[7:], -1),                         # window 8: the kernel is for 16 x 16 windows only
        (ok[:2] + (24,) + ok[3:], -1),                        # H not a multiple of 16
        (ok[:3] + (40,) + ok[4:], -1),                        # W not a multiple of 16
        (ok[:4] + (258, 2) + ok[6:], -1),                     # head dim 129 > 128
        (ok[:7] + (16,) + ok[8:], -1),                        # shift >= window
        (ok[:10] + (179,) + ok[11:], -1),                     # out_pitch < C
        ((4104,) + ok[1:], -2),                               # qkv not 16-byte aligned
    ]
    for a, rc in bad:
        assert f(*a) == rc, a
        assert b"window_attention_headpadded" in lib.ffsr_last_error(), a


@pytest.mark.gpu
@pytest.mark.parametrize("Cc,heads,ws,dtype", [(180, 6, 16, "fp32"), (212, 4, 16, "fp32"), (244, 2, 16, "bf16"), (276, 6, 8, "fp32"),
                                               (308, 4, 16, "bf16"), (60, 6, 8, "fp32"),
                                               # fp32 K + V of head dim 122 do not fit in shared memory: K staged, V read through L2
                                               (244, 2, 16, "fp32")])
def test_window_attention_matches_the_reference_block(Cc, heads, ws, dtype):
    dev = torch.device("cuda:0")
    lib = K.load()
    g = torch.Generator().manual_seed(Cc + ws)
    B, H, W = 2, 2 * ws, 3 * ws
    qkv = torch.randn(B, H, W, 3 * Cc, generator=g)
    table = 0.5 * torch.randn((2 * ws - 1) ** 2, heads, generator=g)
    tdt = torch.bfloat16 if dtype == "bf16" else torch.float32
    qd = qkv.to(dev, tdt).contiguous()
    td = table.to(dev)
    for shift in (0, ws // 2):
        out = torch.empty(B, H, W, Cc, device=dev, dtype=tdt)
        rc = lib.ffsr_window_attention(qd.data_ptr(), B, H, W, Cc, heads, ws, shift, td.data_ptr(), out.data_ptr(),
                                       K.DT_BF16 if dtype == "bf16" else K.DT_F32, C.c_void_p(torch.cuda.current_stream().cuda_stream))
        K.check(rc, "window_attention")
        want = expected_attention(qd.float().cpu(), heads, ws, shift, table)
        err = float((out.float().cpu() - want).abs().max())
        assert err <= (2e-2 if dtype == "bf16" else 2e-5), (Cc, heads, ws, shift, err)


@pytest.mark.gpu
def test_drct_forward_matches_oracle():
    """isr_b200.drct.DRCT.forward (fp32, C ABI kernels) against oracle/drct_oracle.py on the reduced configuration of the
    golden (2 RDGs, window 8, all DRCT-L channel counts), synthesised weights, a 16x24 input (shifted windows, 2x3 grid)."""
    import json
    import numpy as np
    from isr_b200 import drct as D
    g = np.load(os.path.join(ROOT, "tests", "golden", "drct_small.npz"))
    cfg = json.loads(str(g["cfg"]))
    m = D.DRCT(img_size=cfg["img_size"], window_size=cfg["window"], embed_dim=cfg["embed_dim"], depths=[6] * cfg["n_rdg"],
               num_heads=[cfg["num_heads"]] * cfg["n_rdg"], mlp_ratio=cfg["mlp_ratio"])
    sd = DO.synth_state_dict(DO.state_shapes(**cfg), seed=int(g["seed"]), img_size=cfg["img_size"])
    m.load_state_dict(sd, strict=True)
    dev = torch.device("cuda:0")
    m.to(dev).eval()
    x = torch.from_numpy(g["x"])
    y = m(x.to(dev))
    torch.cuda.synchronize()
    assert float((y.cpu() - torch.from_numpy(g["y"])).abs().max()) <= 1e-4           # the reference class's own output
    with torch.no_grad():
        want, feat = DO.forward(sd, x, return_feature=True)
    assert float((y.cpu() - want).abs().max()) <= 1e-4
    assert float((m.last_feature.cpu() - feat).abs().max()) <= 1e-4




@pytest.mark.gpu
@pytest.mark.parametrize("Cc,heads,ws", [(180, 6, 16), (212, 4, 16), (244, 2, 16), (276, 6, 16), (308, 4, 16), (308, 4, 8),
                                         # head dims 1, 8, 10, 12: padding channels in the Q planes the bias table reuses
                                         (6, 6, 16), (48, 6, 16), (40, 4, 16), (24, 2, 16)])
def test_pitched_window_attention_bf16(Cc, heads, ws):
    """Window 16 runs k_window_attn_tc<false>: also checked against its fp64 emulation (window16_reference)."""
    dev = torch.device("cuda:0")
    lib = K.load()
    g = torch.Generator().manual_seed(Cc)
    B, H, W = 1, 2 * ws, 2 * ws
    qp, op = (3 * Cc + 7) // 8 * 8, (Cc + 7) // 8 * 8
    qkv = torch.randn(B, H, W, 3 * Cc, generator=g)
    table = 0.5 * torch.randn((2 * ws - 1) ** 2, heads, generator=g)
    qd = torch.zeros(B, H, W, qp, device=dev, dtype=torch.bfloat16)
    qd[..., :3 * Cc] = qkv.to(dev)
    td = table.to(dev)
    for shift in (0, ws // 2):
        out = torch.full((B, H, W, op), 7.0, device=dev, dtype=torch.bfloat16)
        K.check(lib.ffsr_window_attention_pitched(qd.data_ptr(), qp, B, H, W, Cc, heads, ws, shift, td.data_ptr(), out.data_ptr(), op,
                                                  C.c_void_p(torch.cuda.current_stream().cuda_stream)), "window_attention_pitched")
        bad = int((~torch.isfinite(out[..., :Cc])).sum())
        assert bad == 0, (Cc, heads, shift, f"{bad} non-finite outputs")
        want = expected_attention(qd[..., :3 * Cc].float().cpu(), heads, ws, shift, table)
        assert float((out[..., :Cc].float().cpu() - want).abs().max()) <= 2e-2
        assert bool((out[..., Cc:] == 7.0).all())                      # padding channels are not touched
        if ws == 16:
            ref, tol = window16_reference(qd[..., :3 * Cc], heads, shift, td)
            assert_within(out[..., :Cc], ref, tol, ("pitched", Cc, heads, shift))


@pytest.mark.gpu
def test_drct_forward_bf16_mode():
    import json
    import numpy as np
    from isr_b200 import drct as D
    g = np.load(os.path.join(ROOT, "tests", "golden", "drct_small.npz"))
    cfg = json.loads(str(g["cfg"]))
    m = D.DRCT(img_size=cfg["img_size"], window_size=cfg["window"], embed_dim=cfg["embed_dim"], depths=[6] * cfg["n_rdg"],
               num_heads=[cfg["num_heads"]] * cfg["n_rdg"], mlp_ratio=cfg["mlp_ratio"])
    m.load_state_dict(DO.synth_state_dict(DO.state_shapes(**cfg), seed=int(g["seed"]), img_size=cfg["img_size"]), strict=True)
    dev = torch.device("cuda:0")
    m.to(dev).eval()
    m.precision = "bf16"
    y = m(torch.from_numpy(g["x"]).to(dev)).cpu()
    want = torch.from_numpy(g["y"])
    rel = float((y - want).norm() / want.norm())
    assert rel <= 2e-2, rel


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


@pytest.mark.gpu
@pytest.mark.parametrize("Cc,heads", [(180, 6), (212, 4), (244, 2), (276, 6), (308, 4),     # DRCT-L: head dims 30, 53, 122, 46, 77
                                      (96, 6), (256, 4), (256, 2),                          # 16, 64, 128: no padding (128 = 232448 B of smem)
                                      (48, 6), (40, 4)])                                    # 8, 10
def test_headpadded_window_attention(Cc, heads):
    """ffsr_window_attention_headpadded (k_window_attn_tc<true>, the bf16 DRCT-L path) on rows built here as
    [q|k|v] x heads x DP with zero padding, against its fp64 emulation and, at 2e-2, the plain attention; shifts 0, 8 and 3;
    B = 3 on a 2x5 window grid with output pitch pad8(C), and one 16x16 image (1x1 grid: the shift regions degenerate) with
    an odd output pitch (2-byte stores, as for odd head dims); the output's padding columns keep their sentinel.  On the
    same logical qkv the pitched entry point (k_window_attn_tc<false>) must give the same bits: the two differ only in
    how they gather into shared memory.
    Observed on a B200 (1000 W): worst err / tol 0.75 (DRCT-L shapes 0.64-0.75), max |err| 7.6e-3."""
    dev = torch.device("cuda:0")
    lib = K.load()
    g = torch.Generator().manual_seed(1000 + Cc + heads)
    table = (0.5 * torch.randn(31 * 31, heads, generator=g)).to(dev)
    for B, nwy, nwx, op in ((3, 2, 5, (Cc + 7) // 8 * 8), (1, 1, 1, Cc + 5)):
        H, W = 16 * nwy, 16 * nwx
        qkv = torch.randn(B, H, W, 3 * Cc, generator=g).to(dev, torch.bfloat16)
        qh = headpad_rows(qkv, heads)
        qp = (3 * Cc + 7) // 8 * 8
        qd = torch.zeros(B, H, W, qp, device=dev, dtype=torch.bfloat16)
        qd[..., :3 * Cc] = qkv
        for shift in (0, 8, 3):
            out = torch.full((B, H, W, op), 7.0, device=dev, dtype=torch.bfloat16)
            K.check(lib.ffsr_window_attention_headpadded(qh.data_ptr(), B, H, W, Cc, heads, 16, shift, table.data_ptr(), out.data_ptr(),
                                                         op, _stream()), "window_attention_headpadded")
            outp = torch.full_like(out, 7.0)
            K.check(lib.ffsr_window_attention_pitched(qd.data_ptr(), qp, B, H, W, Cc, heads, 16, shift, table.data_ptr(), outp.data_ptr(),
                                                      op, _stream()), "window_attention_pitched")
            ref, tol = window16_reference(qkv, heads, shift, table)
            assert_within(out[..., :Cc], ref, tol, ("headpadded", Cc, heads, B, H, W, op, shift))
            want = expected_attention(qkv.double(), heads, 16, shift, table.double())
            assert float((out[..., :Cc].double() - want).abs().max()) <= 2e-2
            assert bool((out[..., Cc:] == 7.0).all())
            assert torch.equal(out, outp), ("headpadded != pitched", Cc, heads, B, H, W, shift)


@pytest.mark.gpu
@pytest.mark.parametrize("qk_scale,table_scale", [(1.0, 0.5), (3.0, 0.5), (0.05, 0.5), (1.0, 5.0)],
                         ids=["randn", "peaky", "near-uniform", "wide-bias"])
@pytest.mark.parametrize("Cc,heads", [(212, 4), (256, 2)])
def test_window16_tcgen05_and_cuda_core_paths(Cc, heads, qk_scale, table_scale, monkeypatch):
    """ffsr_window_attention_pitched at window 16 on both of its kernels, the same inputs against fp64: tcgen05
    (k_window_attn_tc, bf16 P) and, with FFSR_WATTN_TC0 set, the CUDA-core k_window_attn (fp32 softmax).  Softmax edges:
    q, k ~ 3 randn (one key dominates), ~ 0.05 randn (near uniform), a bias table ~ 5 randn (the kernel's row-maximum
    bound m sits far above the true maximum of many rows).  B = 2, 2x3 window grid, shifts 0 and 8.
    Observed on a B200 (1000 W), worst err / tol: tcgen05 0.46 near-uniform, 0.57-0.61 randn, 0.81-0.89 peaky, 0.87-0.88
    wide bias; CUDA core 0.39-0.49."""
    dev = torch.device("cuda:0")
    lib = K.load()
    g = torch.Generator().manual_seed(int(100 * qk_scale) + int(10 * table_scale) + Cc)
    B, H, W = 2, 32, 48
    qkv = torch.randn(B, H, W, 3 * Cc, generator=g)
    qkv[..., :2 * Cc] *= qk_scale
    qp = (3 * Cc + 7) // 8 * 8
    qd = torch.zeros(B, H, W, qp, device=dev, dtype=torch.bfloat16)
    qd[..., :3 * Cc] = qkv.to(dev)
    table = (table_scale * torch.randn(31 * 31, heads, generator=g)).to(dev)
    for shift in (0, 8):
        for path in ("tcgen05", "cuda-core"):
            if path == "cuda-core":
                monkeypatch.setenv("FFSR_WATTN_TC0", "1")
            else:
                monkeypatch.delenv("FFSR_WATTN_TC0", raising=False)
            out = torch.empty(B, H, W, Cc, device=dev, dtype=torch.bfloat16)
            K.check(lib.ffsr_window_attention_pitched(qd.data_ptr(), qp, B, H, W, Cc, heads, 16, shift, table.data_ptr(), out.data_ptr(),
                                                      Cc, _stream()), "window_attention_pitched")
            ref, tol = window16_reference(qd[..., :3 * Cc], heads, shift, table, bf16_p=(path == "tcgen05"))
            assert_within(out, ref, tol, (path, Cc, heads, qk_scale, table_scale, shift))


def _fp64_oracle(sd, x, dev):
    """oracle/drct_oracle.py forward in float64 on the GPU (no TF32 anywhere in the reference)."""
    sd64 = {k: (v.to(dev, torch.float64) if v.is_floating_point() else v.to(dev)) for k, v in sd.items()}
    with torch.no_grad():
        return DO.forward(sd64, x.to(dev, torch.float64), return_feature=True)


def _rel(a, b):
    return float((a.double() - b).norm() / b.norm())


@pytest.mark.gpu
def test_drct_window16_forward_against_fp64():
    """DRCT.forward at window 16 on a reduced depth (2 RDGs, every DRCT-L channel count / head rule), B = 2, 32x48 input
    (2x3 window grid, shifted windows) against the fp64 oracle: fp32 mode <= 1e-4 max-abs on the SR image and the cached
    feature; bf16 mode with head-padded qkv rows (k_window_attn_tc<true>) and with plain rows (FFSR_DRCT_QKV_PLAIN,
    k_window_attn_tc<false>) rel-L2 <= 2e-2 on both.
    Observed on a B200 (1000 W): fp32 5.1e-6 (image) / 8.1e-6 (feature) max-abs; bf16 rel-L2 4.5e-3 / 2.8e-3 with either
    qkv layout, and the head-padded and plain forwards were bitwise equal (not asserted: nothing promises it)."""
    from isr_b200 import drct as D
    dev = torch.device("cuda:0")
    cfg = dict(embed_dim=180, n_rdg=2, window=16, num_heads=6, gc=32, mlp_ratio=2, num_feat=64, img_size=32)
    m = D.DRCT(img_size=32, window_size=16, embed_dim=180, depths=[6] * 2, num_heads=[6] * 2, mlp_ratio=2)
    sd = DO.synth_state_dict(DO.state_shapes(**cfg), seed=11, window=16, img_size=32)
    m.load_state_dict(sd, strict=True)
    m.to(dev).eval()
    x = torch.rand(2, 3, 32, 48, generator=torch.Generator().manual_seed(12))
    want, feat = _fp64_oracle(sd, x, dev)
    y = m(x.to(dev))
    e_y, e_f = float((y.double() - want).abs().max()), float((m.last_feature.double() - feat).abs().max())
    print(f"window 16, fp32 mode: max-abs image {e_y:.3e}, feature {e_f:.3e}")
    assert e_y <= 1e-4 and e_f <= 1e-4, (e_y, e_f)
    m.precision = "bf16"
    runs = {}
    for headpad in (True, False):
        m.headpad_qkv = headpad
        y = m(x.to(dev))
        runs[headpad] = (y, m.last_feature.clone())
        r_y, r_f = _rel(y, want), _rel(m.last_feature, feat)
        print(f"window 16, bf16 mode, headpad_qkv={headpad}: rel-L2 image {r_y:.3e}, feature {r_f:.3e}, "
              f"max-abs image {float((y.double() - want).abs().max()):.3e}")
        assert r_y <= 2e-2 and r_f <= 2e-2, (headpad, r_y, r_f)
    (yh, fh), (yp, fp) = runs[True], runs[False]
    print(f"head-padded vs plain qkv rows: image bitwise equal {torch.equal(yh, yp)} (max-abs {float((yh - yp).abs().max()):.3e}), "
          f"feature bitwise equal {torch.equal(fh, fp)} (max-abs {float((fh - fp).abs().max()):.3e})")


@pytest.mark.gpu
def test_drct_l_full_depth_against_fp64():
    """The full DRCT-L (create_drct_model after torch.manual_seed(0): 12 RDGs, window 16, default init) on one 64x96
    image against the fp64 oracle, fp32 and bf16 mode.
    Observed on a B200 (1000 W), max-abs image / feature: fp32 3.5e-7 / 5.2e-6, bf16 1.45e-3 / 7.3e-3 (image rel-L2
    6.2e-4).  The image bounds keep about 2x (bf16) and 30x (fp32) of headroom; the feature is held to the window-8 1e-4 in fp32."""
    from isr_b200 import drct as D
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    m = D.create_drct_model().eval()
    x = torch.rand(1, 3, 64, 96, generator=torch.Generator().manual_seed(13))
    want, feat = _fp64_oracle(m.state_dict(), x, dev)
    m.to(dev)
    for precision, bound in (("fp32", 1e-5), ("bf16", 3e-3)):
        m.precision = precision
        y = m(x.to(dev))
        e_y, e_f = float((y.double() - want).abs().max()), float((m.last_feature.double() - feat).abs().max())
        print(f"DRCT-L 64x96, {precision} mode: max-abs image {e_y:.3e}, feature {e_f:.3e}, rel-L2 image {_rel(y, want):.3e}")
        assert e_y <= bound, (precision, e_y)
        assert precision == "bf16" or e_f <= 1e-4, e_f
