"""CPU oracle for the cached-sample loader (TEST INFRASTRUCTURE ONLY; SURVEY §8f N2).

Restates what ``CachedSRDataset`` does with the reference's on-disk cache (three ``torch.save`` pickles per sample,
``src/data/cached_dataset.py``): which stems form the dataset (:84-118), how one sample is assembled (:135-232) and
how the geometric augmentation draws from ``random`` and transforms every tensor (:236-282).  Only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py`` / ``tools/bench_loader.py`` baseline legs may import this module.

Parity pin: ``tests/golden/cache_golden.json`` holds SHA-256 digests of the samples the *reference class itself*
returns on a seeded mock cache (``oracle/make_cache_golden.py``); ``tests/test_cache_format.py`` checks this
restatement against them.
"""
from __future__ import annotations

import hashlib
import random
from pathlib import Path
from typing import Dict, List

import torch

PARTS = ("drct", "rest", "mamba")


def write_mock_cache(root, n: int = 3, lr_hw=(8, 8), seed: int = 0, mamba_missing=(), rest_missing=(),
                     batch_dim: bool = True, scale: int = 4) -> List[str]:
    """A cache directory in the reference's format, as its own self-test builds one (cached_dataset.py:354-389):
    drct part (output, feature, lr, hr, filename) + rest part (grl, nafnet) + fp16 mamba part."""
    root = Path(root)
    root.mkdir(parents=True, exist_ok=True)
    g = torch.Generator().manual_seed(seed)
    h, w = lr_hw
    lead = (1,) if batch_dim else ()
    stems = []
    for i in range(n):
        stem = f"img_{i:03d}"
        stems.append(stem)
        torch.save({"outputs": {"drct": torch.rand(*lead, 3, scale * h, scale * w, generator=g)},
                    "features": {"drct": torch.randn(*lead, 180, h, w, generator=g)},
                    "lr": torch.rand(3, h, w, generator=g), "hr": torch.rand(3, scale * h, scale * w, generator=g),
                    "filename": stem}, root / f"{stem}_drct_part.pt")
        rest = {"outputs": {"grl": torch.rand(*lead, 3, scale * h, scale * w, generator=g),
                            "nafnet": torch.rand(*lead, 3, scale * h, scale * w, generator=g)},
                "features": {"grl": torch.randn(*lead, 180, h, w, generator=g),
                             "nafnet": torch.randn(*lead, 64, h, w, generator=g)}, "filename": stem}
        mamba = {"outputs": {"mamba": torch.rand(*lead, 3, scale * h, scale * w, generator=g).half()},
                 "features": {"mamba": torch.randn(*lead, 180, h, w, generator=g).half()}, "filename": stem}
        if i not in rest_missing:
            torch.save(rest, root / f"{stem}_rest_part.pt")
        if i not in mamba_missing:
            torch.save(mamba, root / f"{stem}_mamba_part.pt")
    return stems


def list_stems(feature_dir) -> List[str]:
    """cached_dataset.py:84-109: sorted ``*_drct_part.pt``; stems without a rest part are dropped."""
    d = Path(feature_dir)
    stems = [f.name.replace("_drct_part.pt", "") for f in sorted(d.glob("*_drct_part.pt"))]
    return [s for s in stems if (d / f"{s}_rest_part.pt").exists()]


def _squeeze(d: Dict[str, torch.Tensor]) -> None:
    for k in d:
        if d[k].dim() == 4:
            d[k] = d[k].squeeze(0)


def load_sample(feature_dir, stem: str, load_features: bool = True) -> dict:
    """One un-augmented sample, cached_dataset.py:150-214 (mamba part fp16 -> fp32; zeros when it is missing)."""
    d = Path(feature_dir)
    a = torch.load(d / f"{stem}_drct_part.pt", weights_only=False)
    b = torch.load(d / f"{stem}_rest_part.pt", weights_only=False)
    lr, hr = a["lr"], a["hr"]
    imgs = dict(a["outputs"])
    imgs.update(b["outputs"])
    mp = d / f"{stem}_mamba_part.pt"
    c = torch.load(mp, weights_only=False) if mp.exists() else None
    if c is not None:
        for k, v in c["outputs"].items():
            imgs[k] = v.float()
    else:
        imgs["mamba"] = torch.zeros(next(iter(imgs.values())).shape)
    _squeeze(imgs)
    feats = None
    if load_features:
        feats = dict(a.get("features", {}))
        feats.update(b.get("features", {}))
        if c is not None:
            for k, v in c.get("features", {}).items():
                feats[k] = v.float()
        else:
            feats["mamba"] = torch.zeros(1, 180, lr.shape[-2], lr.shape[-1])
        _squeeze(feats)
    return {"lr": lr, "hr": hr, "expert_imgs": imgs, "expert_feats": feats, "filename": stem}


def draw_augmentation(rng=random):
    """cached_dataset.py:262-264: three draws per sample, in this order."""
    hflip = rng.random() < 0.5
    vflip = rng.random() < 0.5
    rot_k = rng.randint(0, 3)
    return hflip, vflip, rot_k


def transform(t: torch.Tensor, hflip: bool, vflip: bool, rot_k: int) -> torch.Tensor:
    """cached_dataset.py:266-274: hflip, then vflip, then rot90 by k quarter turns on the last two dims."""
    if hflip:
        t = torch.flip(t, dims=[-1])
    if vflip:
        t = torch.flip(t, dims=[-2])
    if rot_k > 0:
        t = torch.rot90(t, k=rot_k, dims=[-2, -1])
    return t


class OracleCachedDataset:
    """``CachedSRDataset`` restated (same constructor arguments, ``__len__`` / ``__getitem__`` results)."""

    def __init__(self, feature_dir: str, augment: bool = True, repeat_factor: int = 1, load_features: bool = True):
        self.feature_dir = Path(feature_dir)
        if not self.feature_dir.exists():
            raise RuntimeError(f"Feature cache directory not found: {feature_dir}")
        self.file_stems = list_stems(feature_dir)
        if not list(self.feature_dir.glob("*_drct_part.pt")):
            raise RuntimeError(f"No cached features found in {feature_dir}!")
        self.augment, self.repeat_factor, self.load_features = augment, repeat_factor, load_features

    def __len__(self) -> int:
        return len(self.file_stems) * self.repeat_factor

    def __getitem__(self, idx: int) -> dict:
        s = load_sample(self.feature_dir, self.file_stems[idx % len(self.file_stems)], self.load_features)
        lr, hr, imgs, feats = s["lr"], s["hr"], s["expert_imgs"], s["expert_feats"]
        if self.augment:
            hf, vf, k = draw_augmentation()
            lr, hr = transform(lr, hf, vf, k), transform(hr, hf, vf, k)
            imgs = {n: transform(v, hf, vf, k) for n, v in imgs.items()}
            if feats is not None:
                feats = {n: transform(v, hf, vf, k) for n, v in feats.items()}
        out = {"lr": lr, "hr": hr, "expert_imgs": imgs, "filename": s["filename"]}
        if feats is not None:
            out["expert_feats"] = feats
        return out


def sample_digest(sample: dict) -> Dict[str, str]:
    """SHA-256 of every tensor of a sample (dtype, shape and bytes), keyed ``lr``, ``hr``, ``img.<name>``, ``feat.<name>``."""
    def dg(t: torch.Tensor) -> str:
        t = t.contiguous()
        h = hashlib.sha256(f"{t.dtype}{tuple(t.shape)}".encode())
        h.update(t.numpy().tobytes())
        return h.hexdigest()[:32]
    out = {"lr": dg(sample["lr"]), "hr": dg(sample["hr"])}
    for k, v in sample["expert_imgs"].items():
        out["img." + k] = dg(v)
    for k, v in (sample.get("expert_feats") or {}).items():
        out["feat." + k] = dg(v)
    return out


GOLDEN_CASES = [  # (augment, load_features, random.seed, indices)
    (False, True, 0, [0, 1, 2]),
    (True, True, 11, [0, 1, 2, 3, 4, 5]),
    (True, False, 12, [2, 0, 1]),
]
GOLDEN_MOCK = dict(n=3, lr_hw=(8, 12), seed=5, mamba_missing=(1,))


def golden_digests(dataset_cls, root) -> list:
    """Digests of ``dataset_cls`` (the reference class or the oracle) over GOLDEN_CASES on the GOLDEN_MOCK cache."""
    res = []
    for augment, load_features, seed, idxs in GOLDEN_CASES:
        ds = dataset_cls(str(root), augment=augment, repeat_factor=2, load_features=load_features)
        random.seed(seed)
        res.append({"len": len(ds), "samples": [sample_digest(ds[i]) for i in idxs]})
    return res
