"""Pin the CPU oracle (oracle/fusion_oracle.py) to fixtures produced by the reference itself.

Fixtures: tests/golden/*.npz written by oracle/make_golden.py (which imports /root/reference in
the build container).  Nothing here touches /root/reference.
"""
import hashlib
import json
import os

import numpy as np
import pytest
import torch

import isr_b200
from oracle import fusion_oracle as O
from oracle.perturb import perturb_state_dict

TOL = 2e-6   # same torch CPU ops in a different composition: fp32 re-association noise only


def _model(perturbed):
    torch.manual_seed(0)
    m = isr_b200.CompleteEnhancedFusionSR(None)
    if perturbed:
        m.load_state_dict(perturb_state_dict(m.state_dict(), seed=7), strict=True)
    return m


def test_init_matches_reference_bit_for_bit(golden_dir):
    """Our parameter holders consume the RNG like the reference: same seed, same 226 tensors."""
    ref = json.load(open(os.path.join(golden_dir, "state_hashes.json")))
    sd = _model(False).state_dict()
    assert list(sd.keys()) == list(ref.keys())
    assert len(sd) == 226
    for k, v in sd.items():
        shape, dtype, h = ref[k]
        assert list(v.shape) == shape and str(v.dtype) == dtype, k
        assert hashlib.sha256(v.contiguous().numpy().tobytes()).hexdigest() == h, k
    assert sum(p.numel() for p in _model(False).parameters()) == 1_433_217


def _check(g, key, val, tol=TOL):
    ref = torch.from_numpy(g[key])
    err = (val - ref).abs().max().item()
    assert err <= tol, f"{key}: max-abs {err:.3e} > {tol}"


@pytest.mark.parametrize("name,perturbed,B,H,W,feats", [
    ("case_default_16x16", False, 1, 16, 16, True),
    ("case_perturbed_17x23", True, 1, 17, 23, True),
    ("case_perturbed_b2_9x11", True, 2, 9, 11, True),
    ("case_nofeat_16x24", True, 1, 16, 24, False),
])
def test_eval_forward_against_reference_fixtures(golden_dir, name, perturbed, B, H, W, feats):
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    sd = _model(perturbed).state_dict()
    lr, imgs, fts, _ = O.synthetic_inputs(B, H, W, feats=feats)
    with torch.no_grad():
        sr, ints = O.run_pipeline(sd, lr, imgs, fts, training=False, return_intermediates=True)
    _check(g, "sr", sr)
    _check(g, "gates", ints["gates"])
    _check(g, "difficulty", ints["difficulty"])
    if "raw_9_bands" in g:
        _check(g, "raw_9_bands", torch.stack(ints["raw_9_bands"], 1))
        _check(g, "enhanced_9_bands", torch.stack(ints["enhanced_9_bands"], 1))
        _check(g, "routing_lr", ints["routing_lr"])
        _check(g, "fused_before_dynamic", ints["fused_before_dynamic"])
        _check(g, "collaborative_outputs", torch.stack(ints["collaborative_outputs"], 1))
    # derived expert-selection indices are bit-exact (SURVEY §8a-P6)
    top1 = ints["gates"].argmax(1)
    assert torch.equal(top1, torch.from_numpy(g["gates"]).argmax(1))
    assert sr.min() >= 0 and sr.max() <= 1


def test_train_forward_and_bn_side_effects(golden_dir):
    g = np.load(os.path.join(golden_dir, "case_train_b2_12x12.npz"))
    sd = _model(True).state_dict()
    lr, imgs, fts, _ = O.synthetic_inputs(2, 12, 12)
    upd = {}
    with torch.no_grad():
        sr, ints = O.run_pipeline(sd, lr, imgs, fts, training=True, bn_updates=upd, return_intermediates=True)
    _check(g, "sr", sr, 5e-6)
    _check(g, "gates", ints["gates"], 5e-6)
    bn_keys = [k[4:] for k in g.files if k.startswith("bn::")]
    assert len(bn_keys) == 18           # 6 BatchNorms x (mean, var, counter)
    for k in bn_keys:
        ref = torch.from_numpy(g["bn::" + k])
        if k.endswith("num_batches_tracked"):
            assert int(upd[k]) == int(ref), k        # +9 (cross_band) / +4 (collaborative) per forward
        else:
            assert (upd[k] - ref).abs().max().item() <= 1e-6, k


def test_loss_oracle_matches_reference_losses(golden_dir):
    """oracle/loss_oracle.py against the values the reference's own L1Loss / SSIMLoss / FFTLoss /
    SWTLoss classes produced (oracle/make_golden.py, losses_24x24.npz)."""
    import numpy as np
    from oracle import loss_oracle as L
    d = np.load(os.path.join(golden_dir, "losses_24x24.npz"))
    a, b = torch.from_numpy(d["pred"]), torch.from_numpy(d["target"])
    for name, fn in L.LOSSES.items():
        assert abs(float(fn(a, b)) - float(d[name])) <= 2e-7, name
    total, comps = L.combined_loss(a, b, L.STAGE_WEIGHTS[3])
    want = sum(L.STAGE_WEIGHTS[3][k] * float(d[k]) for k in L.STAGE_WEIGHTS[3])
    assert abs(float(total) - want) <= 1e-6 and set(comps) == {"l1", "swt", "fft", "ssim"}
