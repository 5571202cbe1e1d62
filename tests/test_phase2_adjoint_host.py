"""CPU checks of the Phase-2 adjoint formulas that ffsr_dct_bands_adjoint / ffsr_dwt_bands_adjoint implement, and of
the self-adjointness of the FFT low-pass that the input gradient of the FFT bands relies on.

Each adjoint is restated here in fp64 torch in the kernels' own order of steps (zero-extend, per-block transform,
reflect fold for the DCT; bilinear adjoint, transposed stride-2 filters, reflect folds for the DWT) and compared with
autograd of the oracle's forward.  The sources of the new kernels are scanned for atomics."""
import os
import re

import pytest
import torch
import torch.nn.functional as F

import isr_b200
from oracle import fusion_oracle as O
from oracle.perturb import perturb_state_dict

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHAPES = [(1, 8, 8), (3, 9, 11), (1, 17, 23), (3, 64, 64), (1, 339, 510)]


def _sd():
    torch.manual_seed(0)
    m = isr_b200.CompleteEnhancedFusionSR(None)
    sd = perturb_state_dict(m.state_dict(), seed=7)
    return {k: v.double() if v.is_floating_point() else v for k, v in sd.items()}


def _fold_br(p, H, W):
    """Adjoint of the bottom/right reflect pad: padded grid -> [.., H, W]."""
    Hp, Wp = p.shape[-2:]
    out = p[..., :H, :W].clone()
    for py in range(H, Hp):
        out[..., 2 * H - 2 - py, :] += p[..., py, :W]
        for px in range(W, Wp):
            out[..., 2 * H - 2 - py, 2 * W - 2 - px] += p[..., py, px]
    for px in range(W, Wp):
        out[..., :, 2 * W - 2 - px] += p[..., :H, px]
    return out


def dct_adjoint(sd, g3, prefix="freq_decomp.dct"):
    """g3: [B,3(bands),3,H,W] -> dx [B,3,H,W] with unit band scales."""
    B, _, Cc, H, W = g3.shape
    D, Dt = sd[prefix + ".dct_basis"], sd[prefix + ".dct_basis_t"]
    Hp, Wp = (H + 7) // 8 * 8, (W + 7) // 8 * 8
    z = 0
    for b, name in enumerate(["low_mask", "mid_mask", "high_mask"]):
        gp = F.pad(g3[:, b], (0, Wp - W, 0, Hp - H))                      # zero-extend
        blk = gp.reshape(B, Cc, Hp // 8, 8, Wp // 8, 8).permute(0, 1, 2, 4, 3, 5)
        z = z + sd[prefix + "." + name] * (D @ blk @ Dt)
    P = (Dt @ z @ D).permute(0, 1, 2, 4, 3, 5).reshape(B, Cc, Hp, Wp)
    return _fold_br(P, H, W)


def _fold_reflect7(t, n, dim):
    """Adjoint of F.pad(..., 7, 7, mode='reflect') along dim (padded length n + 14)."""
    t = t.movedim(dim, -1)
    out = t[..., 7:7 + n].clone()
    for k in range(1, 8):
        out[..., k] += t[..., 7 - k]                  # p = -k
        out[..., n - 1 - k] += t[..., 7 + n - 1 + k]  # p = n - 1 + k
    return out.movedim(-1, dim)


def dwt_adjoint(sd, g4, prefix="freq_decomp.dwt"):
    """g4: [B,4(LL,LH,HL,HH),3,H,W] -> dx [B,3,H,W] with unit subband scales."""
    B, _, Cc, H, W = g4.shape
    Hs, Ws = (H + 6) // 2 + 1, (W + 6) // 2 + 1
    sub = []
    for s in range(4):                                                   # bilinear adjoint
        x0 = torch.zeros(B, Cc, Hs, Ws, dtype=g4.dtype, requires_grad=True)
        y = O._bilinear(x0, (H, W))
        sub.append(torch.autograd.grad(y, x0, g4[:, s])[0])
    LL, LH, HL, HH = sub

    def cols_t(ga, gb):                                                  # transposed 8x1 stride-(2,1) convs
        k = torch.stack([sd[prefix + ".lo_col"], sd[prefix + ".hi_col"]], 1).flatten(0, 1)   # per channel: (lo, hi)
        t = F.conv_transpose2d(torch.stack([ga, gb], 2).reshape(B, 2 * Cc, Hs, Ws), k, stride=(2, 1), groups=Cc)
        t = F.pad(t, (0, 0, 0, H + 14 - t.shape[2]))
        return _fold_reflect7(t, H, 2)

    lo, hi = cols_t(LL, LH), cols_t(HL, HH)
    k = torch.stack([sd[prefix + ".lo_row"], sd[prefix + ".hi_row"]], 1).flatten(0, 1)
    t = F.conv_transpose2d(torch.stack([lo, hi], 2).reshape(B, 2 * Cc, H, lo.shape[3]), k, stride=(1, 2), groups=Cc)
    t = F.pad(t, (0, W + 14 - t.shape[3]))
    return _fold_reflect7(t, W, 3)


@pytest.mark.parametrize("B,H,W", SHAPES)
def test_dct_and_dwt_adjoint_formulas_match_autograd(B, H, W):
    sd = _sd()
    sd["freq_decomp.dct.band_scale"] = torch.ones(3, dtype=torch.float64)
    sd["freq_decomp.dwt.subband_scale"] = torch.ones(4, dtype=torch.float64)
    g = torch.Generator().manual_seed(H * 1000 + W)
    x = torch.rand(B, 3, H, W, generator=g, dtype=torch.float64, requires_grad=True)
    g3 = torch.randn(B, 3, 3, H, W, generator=g, dtype=torch.float64)
    g4 = torch.randn(B, 4, 3, H, W, generator=g, dtype=torch.float64)
    fwd_dct = O.dct_bands(sd, x)
    ref = torch.autograd.grad(fwd_dct, x, list(g3.unbind(1)))[0]
    got = dct_adjoint(sd, g3)
    assert ((got - ref).norm() / ref.norm()).item() <= 1e-12
    # dot-product test <A x, g> = <x, A^T g>
    lhs = sum((a * b).sum() for a, b in zip(fwd_dct, g3.unbind(1))).item()
    assert abs(lhs - (x * got).sum().item()) <= 1e-10 * max(1.0, abs(lhs))
    fwd_dwt = O.dwt_bands(sd, x)
    ref = torch.autograd.grad(fwd_dwt, x, list(g4.unbind(1)))[0]
    got = dwt_adjoint(sd, g4)
    assert ((got - ref).norm() / ref.norm()).item() <= 1e-12
    lhs = sum((a * b).sum() for a, b in zip(fwd_dwt, g4.unbind(1))).item()
    assert abs(lhs - (x * got).sum().item()) <= 1e-10 * max(1.0, abs(lhs))


@pytest.mark.parametrize("H,W", [(8, 8), (9, 11), (17, 23), (64, 64), (339, 510)])
def test_fft_lowpass_is_self_adjoint_for_a_real_half_spectrum_mask(H, W):
    g = torch.Generator().manual_seed(H + W)
    m = torch.rand(H, W // 2 + 1, generator=g, dtype=torch.float64)     # not Hermitian-symmetric on DC / Nyquist

    def L(t):
        return torch.fft.irfft2(torch.fft.rfft2(t, norm="ortho") * m, s=(H, W), norm="ortho")

    x = torch.randn(2, 3, H, W, generator=g, dtype=torch.float64, requires_grad=True)
    y = torch.randn(2, 3, H, W, generator=g, dtype=torch.float64)
    assert abs((L(x) * y).sum().item() - (x * L(y)).sum().item()) <= 1e-10 * y.norm().item() * x.norm().item()
    ref = torch.autograd.grad(L(x), x, y)[0]
    assert ((L(y) - ref).norm() / ref.norm()).item() <= 1e-12


def test_phase2_adjoint_kernels_use_no_atomics():
    src = open(os.path.join(ROOT, "image-super-resolution_b200", "csrc", "phase2_bands.cu")).read()
    start = src.index("Adjoints of the unit-scale DCT and DWT bands")
    end = src.index("ffsr_dwt_bands_adjoint(const float* g4")
    body = src[start:src.index("\n}\n", end)]
    assert "k_dct_adjoint_blocks" in body and "k_dwt_analysis_adjoint" in body
    assert not re.search(r"\batomic\w*\s*\(|\bred\.", body), "the Phase-2 adjoints must be atomic-free gathers"
    bn = open(os.path.join(ROOT, "image-super-resolution_b200", "csrc", "train_ops.cu")).read()
    i = bn.index("k_bn_eval_dx")
    body = bn[i:bn.index("\n}\n", bn.index("ffsr_bn_eval_backward(const float* x"))]
    assert not re.search(r"\batomic\w*\s*\(", body)
