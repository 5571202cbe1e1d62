"""The swapped-operand geometry of k_conv_tc (geom 3: weights as the M operand, an 8x32-pixel tile as N = 256) against
F.conv2d in fp64 on the same bf16-rounded operands, and the shape rule that selects it."""
import re

import pytest
import torch

import isr_b200
from isr_b200 import _cabi as K
from isr_b200.pipeline import FusionEngine, nhwc, _pack_conv
from test_gpu_conv_tc import _run

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("cin,cout,N,H,W,act,epi,r_bf16", [
    (128, 128, 2, 37, 45, K.ACT_GELU, K.EPI_PLAIN, False),       # refinement layer, ragged tiles in x and y
    (128, 128, 1, 400, 416, K.ACT_GELU, K.EPI_PLAIN, False),     # ~80 tiles per CTA: many laps of the accumulator ring
    (128, 128, 2, 37, 45, K.ACT_NONE, K.EPI_PLAIN, False),
    (128, 128, 2, 37, 45, K.ACT_RELU, K.EPI_PLAIN, False),
    (128, 128, 2, 37, 45, K.ACT_SIGMOID, K.EPI_PLAIN, False),
    (184, 184, 2, 37, 45, K.ACT_NONE, K.EPI_RESIDUAL, False),    # r1 + r2 fp32, 2 cout blocks, partial last K chunk
    (184, 184, 2, 37, 45, K.ACT_NONE, K.EPI_RESIDUAL, True),     # bf16 residuals
    (136, 136, 1, 70, 21, K.ACT_GELU, K.EPI_PLAIN, False),       # second cout block with 8 channels, 1 k-step last chunk
    (256, 256, 1, 33, 50, K.ACT_GELU, K.EPI_PLAIN, False),       # 4 K chunks, 2 full cout blocks
    (128, 128, 2, 32, 45, K.ACT_GELU, K.EPI_PLAIN, False),       # smallest image that takes geom 3
    (128, 128, 2, 31, 45, K.ACT_GELU, K.EPI_PLAIN, False),       # one row fewer: the 16x16-pixel fallback
])
def test_conv_tc_swapped_against_torch(cin, cout, N, H, W, act, epi, r_bf16):
    _run(cin, cout, 3, N, H, W, act, epi, True, r_bf16=r_bf16)


def _geom_of(capfd, monkeypatch, cin, cout, H, W, N=1):
    """Launch one bf16 3x3 GELU conv with FFSR_TC_DEBUG set and return the geometry its launch line reports."""
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    dev = torch.device("cuda:0")
    monkeypatch.setenv("FFSR_TC_DEBUG", "1")
    eng = FusionEngine(isr_b200.CompleteEnhancedFusionSR(None))
    eng._stream = eng._get_stream(dev)
    wt = torch.randn(cout, cin, 3, 3) / (9 * cin) ** 0.5
    eng._w = {"t": _pack_conv(wt)[None].to(dev), "t.b": torch.zeros(1, cout).to(dev)}
    xin = torch.randn(N, H, W, cin, device=dev).bfloat16()
    out = torch.empty(N, H, W, cout, device=dev, dtype=torch.bfloat16)
    capfd.readouterr()
    with torch.cuda.device(dev):
        eng.conv(nhwc(xin), N, H, W, cin, "t", cout, 3, nhwc(out), act=K.ACT_GELU)
        torch.cuda.synchronize()
    lines = [l for l in capfd.readouterr().err.splitlines() if l.startswith("[conv_tc]")]
    assert len(lines) == 1, lines
    return int(re.search(r"geom=(\d+)", lines[0]).group(1))


def test_conv_tc_refinement_shape_selects_swapped(capfd, monkeypatch):
    # the C3 refinement layers (1 x 1356 x 2040, 128 -> 128): a silent fallback would pass every numeric test
    assert _geom_of(capfd, monkeypatch, 128, 128, 1356, 2040) == 3
    assert _geom_of(capfd, monkeypatch, 128, 128, 32, 45) == 3
    assert _geom_of(capfd, monkeypatch, 128, 128, 31, 45) == 0
    assert _geom_of(capfd, monkeypatch, 192, 64, 64, 64) == 0      # Cout <= 64 stays on the 16x16-pixel tiles
