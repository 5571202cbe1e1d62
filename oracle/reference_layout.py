"""A minimal ``src`` package with the reference's import layout (TEST INFRASTRUCTURE ONLY).

The reference is not part of this repository, yet the drop-in boundary (``isr_b200.install``) is defined by how the
reference's packages import their modules.  ``write_reference_layout(root)`` writes those packages, not the reference's
own files:

* ``src/models/__init__.py`` re-exports the names of ``src.models.enhanced_fusion_v2`` (src/models/__init__.py:50-58)
  and ``src/models/enhanced_fusion_v2.py`` refuses to import, so only the module the installer pre-seeds can answer;
* ``src/data`` holds the pickle-cache loader as restated by ``oracle.cache_oracle`` (pinned to the reference class by
  ``tests/golden/cache_golden.json``), re-exported as ``from src.data import CachedSRDataset, create_cached_dataloader``;
* ``src/utils/metrics.py`` is ``calculate_psnr`` / ``calculate_ssim`` as restated by ``oracle.loss_oracle``.

The oracle modules must be importable by whoever imports this package (the repository root on ``sys.path``).
"""
import os
import textwrap

FILES = {
    "src/__init__.py": "",
    "src/models/__init__.py": """
        from .enhanced_fusion_v2 import (CompleteEnhancedFusionSR, create_enhanced_fusion, AdaptiveFrequencyDecomposition,
                                         CrossBandAttention, CollaborativeFeatureLearning, MultiResolutionFusion,
                                         DynamicExpertSelector)
        """,
    "src/models/enhanced_fusion_v2.py": """
        raise ImportError("stand-in for the reference's enhanced_fusion_v2: run under python -m isr_b200.install, "
                          "which pre-seeds src.models.enhanced_fusion_v2 with the sm_100a module")
        """,
    "src/data/__init__.py": """
        from .cached_dataset import CachedSRDataset, create_cached_dataloader
        """,
    "src/data/cached_dataset.py": """
        from torch.utils.data import DataLoader

        from oracle.cache_oracle import OracleCachedDataset as CachedSRDataset


        def create_cached_dataloader(feature_dir, batch_size=16, num_workers=4, augment=True, repeat_factor=20,
                                     load_features=True, **_):
            ds = CachedSRDataset(feature_dir, augment=augment, repeat_factor=repeat_factor, load_features=load_features)
            return DataLoader(ds, batch_size=batch_size, shuffle=True, num_workers=num_workers)
        """,
    "src/utils/__init__.py": "",
    "src/utils/metrics.py": """
        from oracle.loss_oracle import metric_psnr as calculate_psnr, metric_ssim as calculate_ssim
        """,
}


def write_reference_layout(root) -> str:
    """Write the packages under ``root`` and return ``root`` (the directory a reference script puts on sys.path)."""
    root = str(root)
    for rel, body in FILES.items():
        path = os.path.join(root, rel)
        os.makedirs(os.path.dirname(path), exist_ok=True)
        with open(path, "w") as f:
            f.write(textwrap.dedent(body).lstrip("\n"))
    return root
