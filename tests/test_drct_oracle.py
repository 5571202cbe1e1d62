"""DRCT-L expert forward (SURVEY §8f N1): the oracle restatement pinned to the reference class -- prepared ahead of the
CUDA path.  CPU only."""
import hashlib
import json
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import drct_oracle as DO  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden", "drct_small.npz")


def test_oracle_reproduces_the_reference_class_golden():
    g = np.load(GOLD)
    cfg = json.loads(str(g["cfg"]))
    sd = DO.synth_state_dict(DO.state_shapes(**cfg), seed=int(g["seed"]), img_size=cfg["img_size"])
    x = torch.from_numpy(g["x"])
    with torch.no_grad():
        y, feat = DO.forward(sd, x, return_feature=True)
    assert tuple(y.shape) == (1, 3, 64, 96) and tuple(feat.shape) == (1, 180, 16, 24)
    assert float((y - torch.from_numpy(g["y"])).abs().max()) <= 2e-5
    assert float((feat.reshape(-1)[::5] - torch.from_numpy(g["feat_sub"])).abs().max()) <= 2e-5


def test_full_drct_l_state_layout_matches_the_reference():
    """Names, shapes and order of the DRCT-L state_dict (create_drct_model) as digested when the golden was made."""
    g = np.load(GOLD)
    ours = [(k, s) for k, (s, _) in DO.state_shapes().items()]
    assert hashlib.sha256(repr(ours).encode()).hexdigest() == bytes(g["full_shapes_sha"]).decode()
    n_float = sum(int(np.prod(s)) for k, (s, kind) in DO.state_shapes().items() if kind == "float")
    assert 27_000_000 < n_float < 29_000_000                          # DRCT-L: ~27.6 M parameters
    dims = DO.swin_dims(180, 6, 32, 2)
    assert [(d, h) for d, h, _, _ in dims] == [(180, 6), (212, 4), (244, 2), (276, 6), (308, 4)]
    assert [hid for _, _, hid, _ in dims] == [360, 424, 488, 276, 308]


def test_shift_mask_and_window_round_trip():
    m = DO.shift_mask(16, 24, 8, 4)
    assert tuple(m.shape) == (6, 64, 64) and set(m.unique().tolist()) == {-100.0, 0.0}
    assert float(m[0].abs().max()) == 0.0                              # an interior window attends everywhere
    x = torch.arange(2 * 16 * 24 * 3, dtype=torch.float32).view(2, 16, 24, 3)
    assert torch.equal(DO._reverse(DO._partition(x, 8), 8, 16, 24), x)
    idx = DO.relative_position_index(16)
    assert tuple(idx.shape) == (256, 256) and int(idx.max()) == 31 * 31 - 1 and int(idx.min()) == 0
    assert DO.flops_per_lr_pixel() > 2.0e7


def test_module_mirror_has_the_reference_state_layout():
    """isr_b200.drct.DRCT (parameter holders of the WIP sm_100a expert) against the reference layout restated in the oracle,
    itself checked against create_drct_model(): names, shapes, order; strict load of a synthesised checkpoint."""
    import isr_b200  # noqa: F401
    from isr_b200 import drct as D
    g = np.load(GOLD)
    cfg = json.loads(str(g["cfg"]))
    small = D.DRCT(img_size=cfg["img_size"], window_size=cfg["window"], embed_dim=cfg["embed_dim"], depths=[6] * cfg["n_rdg"],
                   num_heads=[cfg["num_heads"]] * cfg["n_rdg"], mlp_ratio=cfg["mlp_ratio"])
    want = [(k, s) for k, (s, _) in DO.state_shapes(**cfg).items()]
    assert [(k, tuple(v.shape)) for k, v in small.state_dict().items()] == want
    sd = DO.synth_state_dict(DO.state_shapes(**cfg), seed=1, img_size=cfg["img_size"])
    small.load_state_dict(sd, strict=True)
    for k, v in small.state_dict().items():                       # our index / mask buffers equal the reference's
        if DO.state_shapes(**cfg)[k][1] != "float":
            assert torch.equal(v.float(), sd[k].float()), k
    full = D.create_drct_model()
    assert [(k, tuple(v.shape)) for k, v in full.state_dict().items()] == [(k, s) for k, (s, _) in DO.state_shapes().items()]
    assert abs(D.flops_per_lr_pixel(full) - DO.flops_per_lr_pixel()) < 1.0
    with pytest.raises(RuntimeError, match="no CPU path"):
        full(torch.zeros(1, 3, 16, 16))
    if torch.cuda.is_available():
        with pytest.raises(ValueError, match="multiples of the window"):
            full.cuda()(torch.zeros(1, 3, 20, 16, device="cuda"))
    with pytest.raises(NotImplementedError):
        D.DRCT(upsampler="nearest+conv")


@pytest.mark.parametrize("precision,ws,headpad", [pytest.param("fp32", 8, True, id="fp32"), pytest.param("bf16", 8, True, id="bf16"),
                                                  pytest.param("fp32", 16, True, id="fp32-ws16"),
                                                  pytest.param("bf16", 16, True, id="bf16-ws16"),
                                                  pytest.param("bf16", 16, False, id="bf16-ws16-plain-qkv")])
def test_drct_launch_sequence_dry_run(precision, ws, headpad):
    """Every line of the orchestration runs against a recording fake of the library (no compute without a GPU).  bf16 mode
    at window 16 writes head-padded qkv rows (Cout = 3 heads DP) and runs ffsr_window_attention_headpadded on exactly those
    rows; headpad_qkv = False (FFSR_DRCT_QKV_PLAIN) runs the pitched entry point instead."""
    import ctypes as C
    import isr_b200  # noqa: F401
    from isr_b200 import drct as D

    class Fake:
        def __init__(self):
            self.calls = []

        def __getattr__(self, name):
            def f(*a):
                self.calls.append((name, a))
                return 0
            f.__name__ = name
            return f

        def ffsr_window_attention_head_pad(self, dh):
            return (dh + 15) // 16 * 16

    n = 2
    m = D.DRCT(img_size=2 * ws, window_size=ws, depths=[6] * n, num_heads=[6] * n).eval()
    m.precision = precision
    m.headpad_qkv = headpad
    lib = Fake()
    H, W = 2 * ws, 3 * ws
    y = m._run(torch.rand(1, 3, H, W), lib, C.c_void_p(0))
    assert tuple(y.shape) == (1, 3, 4 * H, 4 * W) and tuple(m.last_feature.shape) == (1, 180, H, W)
    names = [c[0] for c in lib.calls]
    # bf16 mode: conv_after_body runs twice (the cached fp32 feature; x0 + conv as the bf16 input of the tcgen05 tail)
    assert names.count("ffsr_conv2d") == 1 + 25 * n + 5 + (1 if precision == "bf16" else 0)
    assert names.count("ffsr_layernorm_strided") == 1 + 10 * n + 1
    hp = precision == "bf16" and ws == 16 and headpad
    att = "ffsr_window_attention_headpadded" if hp else ("ffsr_window_attention_pitched" if precision == "bf16" else "ffsr_window_attention")
    others = {"ffsr_window_attention_headpadded", "ffsr_window_attention_pitched", "ffsr_window_attention"} - {att}
    assert names.count(att) == 5 * n and not any(names.count(o) for o in others)
    assert names.count("ffsr_leaky_relu") == 4 * n + 1
    assert names.count("ffsr_pixel_shuffle2") == 2 and names[0] == "ffsr_rgb_shift_in" and names[-1] == "ffsr_rgb_shift_out"
    hi, si = (5, 7) if att != "ffsr_window_attention_pitched" else (6, 8)
    heads = [c[1][hi] for c in lib.calls if c[0] == att]
    assert heads[:5] == [6, 4, 2, 6, 4]
    shifts = [c[1][si] for c in lib.calls if c[0] == att]
    assert shifts[:5] == [0, ws // 2] * 2 + [0]
    if hp:                                              # the qkv conv right before each launch writes its input rows
        for i, (name, a) in enumerate(lib.calls):
            if name == att:
                d, h = a[4], a[5]
                conv = lib.calls[i - 1]
                assert conv[0] == "ffsr_conv2d"
                p = conv[1][0]._obj
                assert (p.Cin, p.Cout, p.ksize) == (d, 3 * h * ((d // h + 15) // 16 * 16), 1)
                assert p.out == a[0] and a[6] == ws and a[10] == (d + 7) // 8 * 8


def test_headpadded_qkv_weights():
    """bf16 mode at window 16: the packed `.attn.qkvp` Linear of DRCT._weights writes the rows [q|k|v] x heads x DP whose
    [3][heads][:dh] slices are the module's own qkv Linear and whose padding channels are exactly 0 (the tcgen05 window
    attention multiplies them with each other)."""
    import isr_b200  # noqa: F401
    from isr_b200 import drct as D
    torch.manual_seed(0)
    m = D.DRCT(img_size=32, window_size=16, depths=[6], num_heads=[6]).eval()
    for mod in m.modules():                             # non-zero biases: a misplaced bias row shows too
        if isinstance(mod, torch.nn.Linear):
            torch.nn.init.normal_(mod.bias)
    w = m._weights(torch.device("cpu"))
    x = torch.randn(5, 7, 308)
    for j in range(5):
        sw = getattr(m.layers[0], f"swin{j + 1}")
        d, heads = sw.dim, sw.heads
        dh = d // heads
        DP = (dh + 15) // 16 * 16
        p = f"layers.0.swin{j + 1}.attn"
        assert tuple(w[p + ".qkvp"].shape) == (1, d, 3 * heads * DP) and tuple(w[p + ".qkvp.b"].shape) == (3 * heads * DP,)
        xd = x[..., :d].double()
        got = (xd @ w[p + ".qkvp"][0].double() + w[p + ".qkvp.b"].double()).view(5, 7, 3, heads, DP)
        want = torch.nn.functional.linear(xd, sw.attn.qkv.weight.detach().double(), sw.attn.qkv.bias.detach().double()).view(5, 7, 3, heads, dh)
        assert float((got[..., :dh] - want).abs().max()) < 1e-12, (j, d, heads)
        assert bool((got[..., dh:] == 0).all()), (j, d, heads)
