"""The drop-in boundary exercised the way the reference's own scripts use it on a GPU: scripts written against the
reference's names only run through ``python -m isr_b200.install``, which pre-seeds ``src.models.enhanced_fusion_v2``
with the sm_100a module.  Their ``src`` package is ``oracle.reference_layout`` (the reference's import layout; its own
enhanced_fusion_v2 refuses to import, its loader and metrics are the oracle restatements pinned to the reference)."""
import os
import subprocess
import sys
import textwrap

import pytest
import torch

from oracle.reference_layout import write_reference_layout

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu

# mock cache pickles in the reference's format (three parts per image), as the reference's self-test builds them
MOCK_CACHE = """
    d = Path(tempfile.mkdtemp())
    g = torch.Generator().manual_seed(0)
    for i in range(3):
        stem = f"img_{i:03d}"
        hr = torch.rand(3, 128, 128, generator=g)
        torch.save({"outputs": {"drct": (hr + 0.02 * torch.randn(3, 128, 128, generator=g)).clamp(0, 1).unsqueeze(0)},
                    "features": {"drct": torch.randn(1, 180, 32, 32, generator=g)},
                    "lr": torch.nn.functional.avg_pool2d(hr, 4), "hr": hr}, d / f"{stem}_drct_part.pt")
        torch.save({"outputs": {k: (hr + 0.02 * torch.randn(3, 128, 128, generator=g)).clamp(0, 1).unsqueeze(0) for k in ("grl", "nafnet")},
                    "features": {"grl": torch.randn(1, 180, 32, 32, generator=g), "nafnet": torch.randn(1, 64, 32, 32, generator=g)}},
                   d / f"{stem}_rest_part.pt")
        torch.save({"outputs": {"mamba": (hr + 0.02 * torch.randn(3, 128, 128, generator=g)).clamp(0, 1).unsqueeze(0).half()},
                    "features": {"mamba": torch.randn(1, 180, 32, 32, generator=g).half()}}, d / f"{stem}_mamba_part.pt")
"""


def _run(ref, script, timeout=900):
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE="1", PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    return subprocess.run([sys.executable, "-m", "isr_b200.install", str(script)], cwd=ref, env=env, capture_output=True,
                          text=True, timeout=timeout)


def _script(tmp_path, ref, body):
    script = tmp_path / "script.py"
    script.write_text(f"import sys, tempfile\nfrom pathlib import Path\nsys.path.insert(0, {ref!r})\nimport torch\n"
                      + textwrap.dedent(MOCK_CACHE) + textwrap.dedent(body))
    return script


def test_reference_cached_training_script_passes_on_the_installed_module(tmp_path):
    """The checks of the reference's scripts/test_cached_training.py: its CachedSRDataset over mock pickles, the model in
    cached mode, forward_with_precomputed, gradient flow to all parameters, a torch.optim.Adam step, forward() raising in
    cached mode."""
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    ref = write_reference_layout(tmp_path / "ref")
    script = _script(tmp_path, ref, """
        from torch.utils.data import DataLoader
        from src.data import CachedSRDataset
        from src.models import CompleteEnhancedFusionSR
        import isr_b200
        assert CompleteEnhancedFusionSR is isr_b200.CompleteEnhancedFusionSR, "install did not take effect"
        ds = CachedSRDataset(str(d), augment=True, repeat_factor=2)
        assert len(ds) == 6
        batch = next(iter(DataLoader(ds, batch_size=2, shuffle=True, num_workers=0)))
        assert sorted(batch["expert_imgs"]) == ["drct", "grl", "mamba", "nafnet"] and batch["expert_imgs"]["mamba"].dtype == torch.float32
        print("[PASSED] dataset")
        model = CompleteEnhancedFusionSR(expert_ensemble=None).cuda().train()
        assert model.cached_mode
        print("[PASSED] cached mode")
        lr = batch["lr"].cuda()
        imgs = {k: v.cuda() for k, v in batch["expert_imgs"].items()}
        feats = {k: v.cuda() for k, v in batch["expert_feats"].items()}
        sr = model.forward_with_precomputed(lr, imgs, feats)
        assert sr.shape == batch["hr"].shape and torch.isfinite(sr).all()
        print("[PASSED] forward_with_precomputed")
        loss = (sr - batch["hr"].cuda()).abs().mean()
        loss.backward()
        params = [p for p in model.parameters() if p.requires_grad]
        n_grad = sum(p.grad is not None and bool(torch.isfinite(p.grad).all()) for p in params)
        print(f"Params with gradients: {n_grad}/{len(params)}")
        assert n_grad == len(params)
        print("[PASSED] gradient flow")
        before = [p.detach().clone() for p in params]
        opt = torch.optim.Adam(params, lr=1e-4)
        opt.step()
        assert any(not torch.equal(a, p.detach()) for a, p in zip(before, params))
        print("[PASSED] optimizer step")
        try:
            model(lr)
        except RuntimeError as exc:
            assert "cached mode" in str(exc)
            print("[PASSED] forward() refuses cached mode")
        else:
            raise AssertionError("forward() ran in cached mode")
        print("CACHED TRAINING OK")
        """)
    r = _run(ref, script)
    out = r.stdout + r.stderr
    assert r.returncode == 0 and "CACHED TRAINING OK" in r.stdout, out[-3000:]
    assert out.count("[PASSED]") == 6 and "Params with gradients: 198/198" in out, out[-3000:]


def test_reference_validation_loop_over_its_own_dataset(tmp_path):
    """A test.py / validate_epoch-style loop written against the reference's names only (src.data.CachedSRDataset, DataLoader,
    src.models.CompleteEnhancedFusionSR, src.utils.metrics): train.py:415-515 in cached mode on mock pickles."""
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    ref = write_reference_layout(tmp_path / "ref")
    script = _script(tmp_path, ref, """
        from torch.utils.data import DataLoader
        from src.data import CachedSRDataset
        from src.models import CompleteEnhancedFusionSR
        from src.utils.metrics import calculate_psnr, calculate_ssim
        import isr_b200
        assert CompleteEnhancedFusionSR is isr_b200.CompleteEnhancedFusionSR, "install did not take effect"
        ds = CachedSRDataset(str(d), augment=False, repeat_factor=1)
        loader = DataLoader(ds, batch_size=1, shuffle=False, num_workers=0)
        model = CompleteEnhancedFusionSR(expert_ensemble=None).cuda().eval()
        psnrs = []
        with torch.no_grad():
            for batch in loader:
                lr = batch["lr"].cuda()
                imgs = {k: v.cuda() for k, v in batch["expert_imgs"].items()}
                feats = {k: v.cuda() for k, v in batch["expert_feats"].items()}
                sr = model.forward_with_precomputed(lr, imgs, feats).clamp(0, 1)
                psnrs.append(float(calculate_psnr(sr, batch["hr"].cuda(), crop_border=4)))
                float(calculate_ssim(sr, batch["hr"].cuda(), crop_border=4))
        assert len(psnrs) == 3 and all(10.0 < p < 60.0 for p in psnrs), psnrs     # random-init weights: a sanity band only
        print("VALIDATION LOOP OK", psnrs)
        """)
    r = _run(ref, script)
    assert r.returncode == 0 and "VALIDATION LOOP OK" in r.stdout, (r.stdout + r.stderr)[-3000:]
