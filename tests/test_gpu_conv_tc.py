"""tcgen05 implicit-GEMM conv (bf16 operands, fp32 accumulate) against F.conv2d evaluated on
the same bf16-rounded inputs and weights: differences are fp32 accumulation order only."""
import pytest
import torch
import torch.nn.functional as F

import isr_b200
from isr_b200 import _cabi as K
from isr_b200.pipeline import FusionEngine, nhwc, _pack_conv

pytestmark = pytest.mark.gpu


def _run(cin, cout, ks, N, H, W, act, epi, out_bf16, cs_in=None, c_off=0, groups=1, r_bf16=False):
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(cin * 7 + cout * 3 + ks + H)
    x = torch.randn(N, cin, H, W, generator=g).bfloat16().float()
    wt = (torch.randn(groups, cout, cin, ks, ks, generator=g) / (cin * ks * ks) ** 0.5).bfloat16().float()
    b = torch.randn(groups, cout, generator=g) * 0.1
    r1 = torch.randn(N, cout, H, W, generator=g)
    r2 = torch.randn(N, cout, H, W, generator=g)
    if r_bf16:
        r1, r2 = r1.bfloat16().float(), r2.bfloat16().float()
    chk, chd = torch.randn(cout, generator=g), torch.randn(cout, generator=g)
    refs = []
    for n in range(N):
        gi = n % groups
        refs.append(F.conv2d(x[n:n + 1].double(), wt[gi].double(), b[gi].double(), padding=ks // 2))
    ref = torch.cat(refs)
    if epi == K.EPI_LKAGATE:
        ref = r1.double() + 0.37 * (r1.double() * chk.double()[None, :, None, None] + chd.double()[None, :, None, None]) * torch.sigmoid(ref)
    else:
        ref = {K.ACT_NONE: lambda t: t, K.ACT_GELU: F.gelu, K.ACT_RELU: F.relu, K.ACT_SIGMOID: torch.sigmoid}[act](ref)
        if epi == K.EPI_RESIDUAL:
            ref = r1.double() + 0.37 * ref + 0.25 * r2.double()

    torch.manual_seed(0)
    eng = FusionEngine(isr_b200.CompleteEnhancedFusionSR(None))
    eng._stream = eng._get_stream(dev)
    eng._w = {"t": torch.stack([_pack_conv(wt[i]) for i in range(groups)]).to(dev), "t.b": b.to(dev).contiguous()}
    cs_in = cs_in or (cin + 7) // 8 * 8
    xin = torch.full((N, H, W, cs_in), 3.0, dtype=torch.bfloat16, device=dev)      # junk in unused channels
    xin[..., c_off:c_off + cin] = x.permute(0, 2, 3, 1).to(dev).bfloat16()
    odt = torch.bfloat16 if out_bf16 else torch.float32
    out = torch.full((N, H, W, cout + 8), 7.0, device=dev, dtype=odt)
    rdt = torch.bfloat16 if r_bf16 else torch.float32
    r1d = r1.permute(0, 2, 3, 1).contiguous().to(dev, rdt)
    r2d = r2.permute(0, 2, 3, 1).contiguous().to(dev, rdt)
    with torch.cuda.device(dev):
        eng.conv(nhwc(xin, c_off), N, H, W, cin, "t", cout, ks, nhwc(out, 8), act=act, epi=epi,
                 r1=nhwc(r1d) if epi else None, r2=nhwc(r2d) if epi == K.EPI_RESIDUAL else None,
                 sa=0.37 if epi else 1.0, sb=0.25, groups=groups,
                 ch_k=chk.to(dev) if epi == K.EPI_LKAGATE else None, ch_d=chd.to(dev) if epi == K.EPI_LKAGATE else None)
        torch.cuda.synchronize()
    got = out[..., 8:].float().permute(0, 3, 1, 2).cpu().double()
    tol = 2e-2 if out_bf16 else 2e-4
    err = (got - ref).abs().max().item()
    assert err < tol, f"max-abs {err}"
    assert torch.all(out[..., :8].float() == 7.0), "wrote outside its channel slice"


@pytest.mark.parametrize("cin,cout,ks,H,W,act,epi,out_bf16", [
    (64, 64, 1, 8, 16, K.ACT_NONE, K.EPI_PLAIN, False),          # single tile, single K chunk
    (64, 64, 3, 16, 32, K.ACT_NONE, K.EPI_PLAIN, False),
    (128, 128, 3, 19, 37, K.ACT_GELU, K.EPI_PLAIN, True),        # ragged tiles, refine layer shape
    (128, 128, 3, 64, 80, K.ACT_GELU, K.EPI_PLAIN, False),       # > 1 tile per CTA, TMEM double buffer
    (32, 32, 3, 19, 37, K.ACT_GELU, K.EPI_PLAIN, True),          # partial K chunk (2 k-steps)
    (3, 128, 3, 19, 37, K.ACT_GELU, K.EPI_PLAIN, True),          # 1 k-step per tap, zero-filled channels
    (128, 3, 3, 19, 37, K.ACT_NONE, K.EPI_RESIDUAL, False),      # N padded to 16, masked scalar stores
    (96, 32, 3, 19, 37, K.ACT_GELU, K.EPI_PLAIN, True),
    (244, 768, 1, 32, 48, K.ACT_NONE, K.EPI_PLAIN, True),        # multi-block 1x1 (DRCT qkv): activation-resident GEMM walk
    (180, 360, 1, 19, 37, K.ACT_GELU, K.EPI_PLAIN, True),        # ragged 16x16 tiles, 3 K chunks (last partial), 3 cout blocks
    (308, 180, 1, 32, 48, K.ACT_NONE, K.EPI_RESIDUAL, False),    # 5 K chunks, fp32 output with residual, 2 cout blocks
    (244, 768, 1, 8, 16, K.ACT_NONE, K.EPI_PLAIN, True),         # H < 16: streamed weights, cout block fastest
    (16, 3, 3, 9, 11, K.ACT_SIGMOID, K.EPI_PLAIN, False),        # image smaller than the TMA box
    (128, 384, 1, 19, 37, K.ACT_NONE, K.EPI_PLAIN, True),        # 3 cout blocks
    (256, 128, 1, 19, 37, K.ACT_NONE, K.EPI_RESIDUAL, False),    # 4 K chunks
    (64, 64, 1, 19, 37, K.ACT_NONE, K.EPI_LKAGATE, True),
])
def test_conv_tc_against_torch(cin, cout, ks, H, W, act, epi, out_bf16):
    _run(cin, cout, ks, 2, H, W, act, epi, out_bf16)


def test_conv_tc_concat_slice_and_groups():
    # 76 channels at offset 0 of an 80-channel pixel stride (stage2/3 concat buffers)
    _run(76, 64, 3, 1, 19, 37, K.ACT_GELU, K.EPI_PLAIN, True, cs_in=80)
    # input slice starting at channel 8 of a wider buffer
    _run(32, 32, 3, 1, 19, 37, K.ACT_NONE, K.EPI_PLAIN, False, cs_in=48, c_off=8)
    # per-image weight sets (modulation heads: image n uses weights n % 4), bf16 residuals
    _run(128, 32, 1, 8, 12, 20, K.ACT_NONE, K.EPI_PLAIN, False, groups=4)
    _run(64, 64, 3, 2, 12, 20, K.ACT_NONE, K.EPI_RESIDUAL, True, r_bf16=True)


# ---- lean epilogue (bf16 inference outputs): both tile-ownership modes, every activation, residual dtypes, Cout % 16 == 8
@pytest.mark.parametrize("force_own", [False, True])
@pytest.mark.parametrize("cin,cout,ks,act,epi,r_bf16", [
    (32, 32, 3, K.ACT_GELU, K.EPI_PLAIN, False),
    (64, 64, 3, K.ACT_GELU, K.EPI_PLAIN, False),
    (76, 64, 3, K.ACT_RELU, K.EPI_PLAIN, False),
    (32, 16, 3, K.ACT_GELU, K.EPI_PLAIN, False),
    (32, 8, 1, K.ACT_GELU, K.EPI_PLAIN, False),
    (32, 24, 3, K.ACT_SIGMOID, K.EPI_PLAIN, False),
    (32, 32, 3, K.ACT_NONE, K.EPI_RESIDUAL, False),
    (32, 32, 3, K.ACT_NONE, K.EPI_RESIDUAL, True),
    (16, 128, 3, K.ACT_GELU, K.EPI_PLAIN, False),
    (128, 128, 3, K.ACT_GELU, K.EPI_PLAIN, False),
    (128, 256, 1, K.ACT_GELU, K.EPI_PLAIN, False),
    (128, 384, 1, K.ACT_NONE, K.EPI_PLAIN, False),
    (64, 128, 1, K.ACT_NONE, K.EPI_RESIDUAL, True),
])
def test_conv_tc_lean_epilogue(monkeypatch, force_own, cin, cout, ks, act, epi, r_bf16):
    if force_own:
        monkeypatch.setenv("FFSR_TC_EPI_OWN_FORCE", "1")
    else:
        monkeypatch.delenv("FFSR_TC_EPI_OWN_FORCE", raising=False)
    _run(cin, cout, ks, 2, 37, 45, act, epi, True, r_bf16=r_bf16)


def test_conv_tc_lean_epilogue_many_tiles():
    # enough tiles per CTA (>= 8 x #SMs) for the tile-ownership heuristic to switch on by itself
    _run(32, 32, 3, 1, 400, 416, K.ACT_GELU, K.EPI_PLAIN, True)
    _run(64, 32, 3, 1, 400, 416, K.ACT_NONE, K.EPI_RESIDUAL, True, r_bf16=True)


# ---- several MMA-issuing warps: which warp issues a tile's MMAs must not change its accumulation order or its bits
@pytest.mark.parametrize("H,W", [(96, 96), (256, 256)])
@pytest.mark.parametrize("cin,cout,ks,act,out_bf16", [
    (32, 32, 3, K.ACT_GELU, True), (64, 64, 3, K.ACT_GELU, True), (76, 64, 3, K.ACT_GELU, True), (3, 32, 3, K.ACT_GELU, True),
    (32, 8, 1, K.ACT_GELU, True), (8, 1, 3, K.ACT_SIGMOID, False), (16, 3, 3, K.ACT_SIGMOID, False),
    (128, 3, 3, K.ACT_NONE, False), (3, 128, 3, K.ACT_GELU, True), (128, 128, 1, K.ACT_NONE, False),
    (96, 32, 3, K.ACT_GELU, True), (32, 32, 3, K.ACT_NONE, False),
])
def test_conv_tc_issue_warps_leave_bits_unchanged(monkeypatch, H, W, cin, cout, ks, act, out_bf16):
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(cin + cout)
    x = torch.randn(1, H, W, (cin + 7) // 8 * 8, generator=g).to(dev).bfloat16()
    wt = torch.randn(cout, cin, ks, ks, generator=g) / (cin * ks * ks) ** 0.5
    eng = FusionEngine(isr_b200.CompleteEnhancedFusionSR(None))
    eng._stream = eng._get_stream(dev)
    eng._w = {"t": _pack_conv(wt).to(dev), "t.b": torch.randn(cout, generator=g).to(dev)}

    def launch():
        out = torch.zeros(1, H, W, (cout + 7) // 8 * 8, device=dev, dtype=torch.bfloat16 if out_bf16 else torch.float32)
        with torch.cuda.device(dev):
            eng.conv(nhwc(x), 1, H, W, cin, "t", cout, ks, nhwc(out), act=act)
            torch.cuda.synchronize()
        return out.cpu()

    multi = launch()
    monkeypatch.setattr(K, "CONV_MULTI_ISSUE", 0)                  # one issuing warp
    single = launch()
    assert torch.equal(multi, single), f"{int((multi != single).sum())} values differ"
