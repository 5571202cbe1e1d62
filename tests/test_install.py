"""The sys.modules pre-seeding that drops the module into an unmodified reference checkout."""
import os
import subprocess
import sys

import pytest

from oracle.reference_layout import write_reference_layout

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_install_exports_reference_names():
    import isr_b200
    from isr_b200 import install as I
    mod = I.install()
    assert sys.modules["src.models.enhanced_fusion_v2"] is mod
    for n in ("CompleteEnhancedFusionSR", "create_enhanced_fusion", "AdaptiveFrequencyDecomposition",
              "CrossBandAttention", "CollaborativeFeatureLearning", "MultiResolutionFusion", "DynamicExpertSelector"):
        assert hasattr(mod, n), n
    assert mod.CompleteEnhancedFusionSR is isr_b200.CompleteEnhancedFusionSR
    with pytest.raises(NotImplementedError):
        mod.CrossBandAttention()
    del sys.modules["src.models.enhanced_fusion_v2"]


def test_reference_package_import_resolves_to_our_module(tmp_path):
    """Through a package with the reference's layout whose own enhanced_fusion_v2 refuses to import."""
    ref = write_reference_layout(tmp_path)
    code = (
        "import sys; sys.path.insert(0, %r); import isr_b200, isr_b200.install as I; I.install();"
        "sys.path.insert(0, %r);"
        "from src.models import CompleteEnhancedFusionSR as A, create_enhanced_fusion;"
        "from src.models.enhanced_fusion_v2 import CompleteEnhancedFusionSR as B2;"
        "assert A is isr_b200.CompleteEnhancedFusionSR and B2 is A;"
        "m = create_enhanced_fusion(None); assert m.cached_mode and len(m.state_dict()) == 226; print('ok')"
    ) % (ROOT, ref)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600,
                       env=dict(os.environ, PYTHONDONTWRITEBYTECODE="1"))
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr[-2000:]


def test_reference_data_package_resolves_to_shard_loader(tmp_path):
    """Through a package with the reference's layout whose own cached_dataset is the pickle loader."""
    ref = write_reference_layout(tmp_path)
    code = (
        "import sys; sys.path.insert(0, %r); import isr_b200, isr_b200.install as I; I.install(loader=True);"
        "sys.path.insert(0, %r);"
        "from src.data import CachedSRDataset, create_cached_dataloader;"
        "from isr_b200 import cache as CA;"
        "assert CachedSRDataset is CA.ShardDataset and create_cached_dataloader.__module__ == 'isr_b200.install'; print('ok')"
    ) % (ROOT, ref)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600,
                       env=dict(os.environ, PYTHONDONTWRITEBYTECODE="1"))
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr[-2000:]


def test_install_fused_losses_module():
    from isr_b200 import install as I
    from isr_b200 import losses as FL
    I.install(losses=True)
    mod = sys.modules["src.losses"]
    assert mod.CombinedLoss is FL.CombinedLoss and mod.PYWT_AVAILABLE is True
    crit = mod.CombinedLoss()
    crit.set_weights({"l1": 0.6, "swt": 0.25, "fft": 0.1, "ssim": 0.05})
    assert crit.current_stage == 3 and crit.weights["swt"] == 0.25
    with pytest.raises(NotImplementedError):
        mod.VGGPerceptualLoss()
    del sys.modules["src.losses"], sys.modules["src.models.enhanced_fusion_v2"]


def test_install_shard_loader_module(tmp_path):
    """--shard-loader: `from src.data.cached_dataset import CachedSRDataset` is the shard dataset, a reference cache
    DIRECTORY is packed on first use, and the samples equal the restated reference loader's."""
    import random
    import torch
    from isr_b200 import install as I
    from isr_b200 import cache as CA
    from oracle import cache_oracle as CO
    I.install(loader=True)
    mod = sys.modules["src.data.cached_dataset"]
    assert mod.CachedSRDataset is CA.ShardDataset and callable(mod.create_cached_dataloader)
    d = tmp_path / "cached_features_train"
    CO.write_mock_cache(d, n=3, lr_hw=(8, 8), seed=6)
    ds = mod.CachedSRDataset(feature_dir=str(d), augment=True, repeat_factor=2, load_features=True)
    assert (d / CA.SHARD_NAME).exists() and len(ds) == 6
    ref = CO.OracleCachedDataset(str(d), augment=True, repeat_factor=2)
    random.seed(4)
    a = [ds[i] for i in range(6)]
    random.seed(4)
    b = [ref[i] for i in range(6)]
    for x, y in zip(a, b):
        assert x["filename"] == y["filename"] and torch.equal(x["lr"], y["lr"])
        assert all(torch.equal(x["expert_feats"][k], y["expert_feats"][k]) for k in y["expert_feats"])
    mt = (d / CA.SHARD_NAME).stat().st_mtime
    mod.CachedSRDataset(feature_dir=str(d), augment=False)                  # second open reuses the shard
    assert (d / CA.SHARD_NAME).stat().st_mtime == mt
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError, match="no CPU path"):
            mod.create_cached_dataloader(str(d), batch_size=2)
    with pytest.raises(RuntimeError):
        mod.CachedSRDataset(feature_dir=str(tmp_path / "missing"))
    del sys.modules["src.data.cached_dataset"], sys.modules["src.models.enhanced_fusion_v2"]
