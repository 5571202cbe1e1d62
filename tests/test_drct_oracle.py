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


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_drct_launch_sequence_dry_run(precision):
    """Every line of the orchestration runs against a recording fake of the library (no compute without a GPU)."""
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

    n = 2
    m = D.DRCT(img_size=16, window_size=8, depths=[6] * n, num_heads=[6] * n).eval()
    m.precision = precision
    lib = Fake()
    y = m._run(torch.rand(1, 3, 16, 24), lib, C.c_void_p(0))
    assert tuple(y.shape) == (1, 3, 64, 96) and tuple(m.last_feature.shape) == (1, 180, 16, 24)
    names = [c[0] for c in lib.calls]
    # bf16 mode: conv_after_body runs twice (the cached fp32 feature; x0 + conv as the bf16 input of the tcgen05 tail)
    assert names.count("ffsr_conv2d") == 1 + 25 * n + 5 + (1 if precision == "bf16" else 0)
    assert names.count("ffsr_layernorm_strided") == 1 + 10 * n + 1
    att = "ffsr_window_attention_pitched" if precision == "bf16" else "ffsr_window_attention"
    assert names.count(att) == 5 * n and names.count("ffsr_leaky_relu") == 4 * n + 1
    assert names.count("ffsr_pixel_shuffle2") == 2 and names[0] == "ffsr_rgb_shift_in" and names[-1] == "ffsr_rgb_shift_out"
    heads = [c[1][5] if precision == "fp32" else c[1][6] for c in lib.calls if c[0] == att]
    assert heads[:5] == [6, 4, 2, 6, 4]
    shifts = [c[1][7] if precision == "fp32" else c[1][8] for c in lib.calls if c[0] == att]
    assert shifts[:5] == [0, 4, 0, 4, 0]
