"""Tile-resident (fused chain) tcgen05 kernels against the layer-by-layer tcgen05 path they replace, on the same bf16
inputs and weights: the two differ only by fp32 summation order and by where bf16 rounding of side inputs happens."""
import pytest
import torch

import isr_b200
from isr_b200 import _cabi as K
from oracle import fusion_oracle as O
from oracle.perturb import perturb_state_dict

pytestmark = pytest.mark.gpu


def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


def _model(dev):
    torch.manual_seed(0)
    m = isr_b200.CompleteEnhancedFusionSR(None)
    m.load_state_dict(perturb_state_dict(m.state_dict(), seed=3))
    m.eval().to(dev)
    m.precision = "bf16"
    return m


@pytest.mark.parametrize("B,H,W", [(1, 16, 16), (2, 13, 29), (1, 40, 56)])
def test_edge_refiner_chain_matches_layer_by_layer(B, H, W):
    """ffsr_edge_refiner_chain (csrc/edge_chain.cu) vs proj / conv1 / conv2 / conv3 / attn0 / attn2 as k_conv_tc launches
    + ffsr_edge_attn_upsample: the 96-channel concat of the three refined pyramid levels and the final image."""
    dev = _cuda()
    m = _model(dev)
    lr, imgs, fts, _ = O.synthetic_inputs(B, H, W)
    lr, imgs, fts = lr.to(dev), {k: v.to(dev) for k, v in imgs.items()}, {k: v.to(dev) for k, v in fts.items()}
    with torch.no_grad():
        m.forward_with_precomputed(lr, imgs, fts)
        eng = m._engine
        assert eng.edge_chain, "the edge-chain kernel must be the default path"
        sr_chain = m.forward_with_precomputed(lr, imgs, fts).float().cpu()
        cat_chain = eng.workspace("ee.cat96").float().cpu().clone()
        eng.edge_chain = False
        sr_ref = m.forward_with_precomputed(lr, imgs, fts).float().cpu()
        cat_ref = eng.workspace("ee.cat96").float().cpu().clone()
        eng.edge_chain = True
    scale = cat_ref.abs().max().item()
    for lv in range(3):
        a, b = cat_chain[..., 32 * lv:32 * lv + 32], cat_ref[..., 32 * lv:32 * lv + 32]
        err = (a - b).abs().max().item()
        # bf16 storage of three chained 32-channel layers: a few bf16 ulps of the feature scale
        assert err <= 0.04 * max(scale, 1e-3), f"level {lv}: max-abs {err:.4e} (feature scale {scale:.3e})"
        assert torch.nn.functional.cosine_similarity(a.reshape(-1), b.reshape(-1), dim=0).item() > 0.9995, lv
    assert (sr_chain - sr_ref).abs().max().item() <= 5e-3


@pytest.mark.parametrize("B,HW", [(1, 32), (2, 77), (1, 4999)])
def test_token_chain_against_torch(B, HW):
    """ffsr_token_attn_chain / ffsr_token_ffn_chain (csrc/token_chain.cu) against nn.LayerNorm -> nn.MultiheadAttention -> residual
    and nn.LayerNorm -> ffn -> residual in fp32 (large_kernel_attention.py:389-392) on the same bf16-rounded token rows.
    Tolerance: bf16 operands (weights and the attention context / hidden row) with fp32 accumulation, bf16 output rows."""
    import torch.nn.functional as F
    from isr_b200.pipeline import pack_token_attn, pack_token_ffn
    dev = _cuda()
    m = _model(dev)
    co = m.collaborative
    lib = K.load()
    g = torch.Generator().manual_seed(HW)
    x = (torch.randn(B, 4, HW, 128, generator=g) * 0.7 + 0.15 * torch.randn(B, 4, HW, 1, generator=g)).to(torch.bfloat16).to(dev)
    t1 = torch.full_like(x, float("nan"))
    t2 = torch.full_like(x, float("nan"))
    wa, pa = pack_token_attn(co)
    wf, pf = pack_token_ffn(co)
    assert wa.numel() * 2 == lib.ffsr_token_attn_weight_bytes() and pa.numel() == lib.ffsr_token_attn_param_floats()
    assert wf.numel() * 2 == lib.ffsr_token_ffn_weight_bytes() and pf.numel() == lib.ffsr_token_ffn_param_floats()
    K.check(lib.ffsr_token_attn_chain(x.data_ptr(), B, HW, wa.data_ptr(), pa.data_ptr(), t1.data_ptr(), None))
    K.check(lib.ffsr_token_ffn_chain(t1.data_ptr(), B * 4 * HW, wf.data_ptr(), pf.data_ptr(), t2.data_ptr(), None))
    torch.cuda.synchronize()
    with torch.no_grad():
        xf = x.float().permute(0, 2, 1, 3).reshape(B * HW, 4, 128)                # [pixel][expert token][128]
        n = co.norm1(xf)
        r1 = xf + co.cross_attn(n, n, n)[0]
        r1_rows = r1.reshape(B, HW, 4, 128).permute(0, 2, 1, 3)
        t1f = t1.float()
        r2 = t1f + co.ffn(co.norm2(t1f))                                           # the FFN kernel's own input
    s1, s2 = r1_rows.abs().max().item(), r2.abs().max().item()
    e1 = (t1f - r1_rows).abs().max().item()
    e2 = (t2.float() - r2).abs().max().item()
    assert torch.isfinite(t2.float()).all()
    assert e1 <= 0.02 * s1, f"attention chain: max-abs {e1:.4e} (scale {s1:.3e})"
    assert e2 <= 0.02 * s2, f"ffn chain: max-abs {e2:.4e} (scale {s2:.3e})"
    assert F.cosine_similarity((t1f - x.float()).reshape(-1), (r1_rows - x.float()).reshape(-1), dim=0).item() > 0.999
    assert F.cosine_similarity((t2.float() - t1f).reshape(-1), (r2 - t1f).reshape(-1), dim=0).item() > 0.999


def test_token_chain_matches_layer_by_layer_forward():
    """Whole bf16 forward with the token chain on and off (seven-launch path): same image within bf16 storage error."""
    dev = _cuda()
    m = _model(dev)
    lr, imgs, fts, _ = O.synthetic_inputs(1, 40, 56)
    lr, imgs, fts = lr.to(dev), {k: v.to(dev) for k, v in imgs.items()}, {k: v.to(dev) for k, v in fts.items()}
    with torch.no_grad():
        m.forward_with_precomputed(lr, imgs, fts)
        eng = m._engine
        assert eng.token_chain
        sr_chain = m.forward_with_precomputed(lr, imgs, fts).float().cpu()
        t2_chain = eng.workspace("co.t2").float().cpu().clone()
        eng.token_chain = False
        sr_ref = m.forward_with_precomputed(lr, imgs, fts).float().cpu()
        t2_ref = eng.workspace("co.t2").float().cpu().clone()
        eng.token_chain = True
    scale = t2_ref.abs().max().item()
    assert (t2_chain - t2_ref).abs().max().item() <= 0.03 * scale
    assert torch.nn.functional.cosine_similarity(t2_chain.reshape(-1), t2_ref.reshape(-1), dim=0).item() > 0.9995
    assert (sr_chain - sr_ref).abs().max().item() <= 5e-3


@pytest.mark.parametrize("B,H,W", [(1, 8, 16), (2, 13, 29), (1, 40, 56)])
def test_align_tokens_against_torch(B, H, W):
    """ffsr_align_tokens (csrc/token_chain.cu) against the four nn.Conv2d align layers in fp32 (large_kernel_attention.py:344-358):
    bf16 operands with fp32 accumulation, bf16 token rows."""
    import ctypes as C
    from isr_b200.pipeline import pack_align_tokens, EXPERT_ORDER
    dev = _cuda()
    m = _model(dev)
    co = m.collaborative
    lib = K.load()
    g = torch.Generator().manual_seed(B * 100 + H)
    feats = [torch.randn(B, co.align_layers[n].weight.shape[1], H, W, generator=g).to(dev) for n in EXPERT_ORDER]
    wb, bb = pack_align_tokens(co)
    assert wb.numel() * 2 == lib.ffsr_align_tokens_weight_bytes()
    out = torch.full((B, 4, H * W, 128), float("nan"), device=dev, dtype=torch.bfloat16)
    fptr = (C.c_void_p * 4)(*[t.data_ptr() for t in feats])
    cnum = (C.c_int * 4)(*[t.shape[1] for t in feats])
    K.check(lib.ffsr_align_tokens(fptr, cnum, B, H * W, wb.data_ptr(), bb.data_ptr(), out.data_ptr(), None))
    torch.cuda.synchronize()
    with torch.no_grad():
        ref = torch.stack([co.align_layers[n](f).permute(0, 2, 3, 1).reshape(B, H * W, 128) for n, f in zip(EXPERT_ORDER, feats)], 1)
    assert torch.isfinite(out.float()).all()
    err = (out.float() - ref).abs().max().item()
    assert err <= 0.02 * ref.abs().max().item(), err
    assert torch.nn.functional.cosine_similarity(out.float().reshape(-1), ref.reshape(-1), dim=0).item() > 0.9999


@pytest.mark.parametrize("B,H,W", [(1, 16, 16), (2, 13, 29), (1, 40, 56)])
def test_fused_selector_matches_layer_by_layer(B, H, W):
    """ffsr_selector_fused (csrc/selector.cu) vs the six fp32 conv launches + ffsr_gate_finalize it replaces
    (DynamicExpertSelector.forward, enhanced_fusion_v2.py:450-466): same fp32 math in another summation order."""
    dev = _cuda()
    m = _model(dev)
    m.precision = "fp32"
    lr, imgs, fts, _ = O.synthetic_inputs(B, H, W)
    lr, imgs, fts = lr.to(dev), {k: v.to(dev) for k, v in imgs.items()}, {k: v.to(dev) for k, v in fts.items()}
    with torch.no_grad():
        m.forward_with_precomputed(lr, imgs, fts)
        eng = m._engine
        assert eng.selector_fused, "the fused selector kernel must be the default path"
        run = lambda: m._run_pipeline(lr, [imgs[k] for k in O.EXPERT_ORDER], fts, 4 * H, 4 * W, {}, True)[1]
        a = run()
        a = {k: a[k].clone() for k in ("gates", "difficulty", "gate_logits", "active")}
        eng.selector_fused = False
        b = run()
        eng.selector_fused = True
    for k in ("gates", "difficulty", "gate_logits"):
        assert (a[k] - b[k]).abs().max().item() <= 2e-5, k
    assert a["gates"].argmax(1).eq(b["gates"].argmax(1)).all()
    assert a["active"].eq(b["active"]).all()
