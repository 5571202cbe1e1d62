"""Cache shards (SURVEY §8f N2): oracle pinned to the reference's CachedSRDataset; pack -> ShardDataset round trip
bit-exact against the oracle; header / layout invariants.  CPU only (the device loader is tests/test_gpu_cache.py)."""
import contextlib
import io
import json
import os
import random
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import isr_b200  # noqa: E402,F401
from isr_b200 import cache as CA  # noqa: E402
from oracle import cache_oracle as CO  # noqa: E402


def _same(a: dict, b: dict):
    assert list(a.keys()) == list(b.keys())
    assert a["filename"] == b["filename"]
    for k in ("lr", "hr"):
        assert a[k].dtype == b[k].dtype and torch.equal(a[k], b[k]), k
    for grp in ("expert_imgs", "expert_feats"):
        if grp not in a:
            continue
        assert sorted(a[grp].keys()) == sorted(b[grp].keys())
        for k in a[grp]:
            assert a[grp][k].dtype == b[grp][k].dtype and a[grp][k].shape == b[grp][k].shape, (grp, k)
            assert torch.equal(a[grp][k], b[grp][k]), (grp, k)


def test_oracle_matches_reference_golden_digests(tmp_path):
    """The restated loader reproduces the digests of what the reference class returned (oracle/make_cache_golden.py)."""
    g = json.load(open(os.path.join(ROOT, "tests", "golden", "cache_golden.json")))
    CO.write_mock_cache(tmp_path, **CO.GOLDEN_MOCK)
    assert CO.golden_digests(CO.OracleCachedDataset, tmp_path) == g["cases"]


@pytest.mark.parametrize("load_features", [True, False])
def test_source_shard_is_bit_exact_with_the_loader(tmp_path, load_features):
    d = tmp_path / "cache"
    CO.write_mock_cache(d, n=5, lr_hw=(8, 12), seed=1, mamba_missing=(3,), rest_missing=(0,))
    shard = tmp_path / "train.ffsrc"
    hdr = CA.pack_cache(str(d), str(shard), dtype="source", load_features=load_features)
    assert hdr["count"] == 4 and hdr["stems"] == CO.list_stems(d) and hdr["has_mamba"] == [True, True, False, True]
    for augment in (False, True):
        ref = CO.OracleCachedDataset(str(d), augment=augment, repeat_factor=2, load_features=load_features)
        ours = CA.ShardDataset(str(shard), augment=augment, repeat_factor=2, load_features=load_features)
        assert len(ref) == len(ours) == 8
        random.seed(17)
        want = [ref[i] for i in range(len(ref))]
        random.seed(17)
        got = [ours[i] for i in range(len(ours))]
        for a, b in zip(got, want):
            _same(a, b)
            assert a["expert_imgs"]["mamba"].dtype == torch.float32


def test_fp16_shard_rounds_once_and_is_half_the_size(tmp_path):
    d = tmp_path / "cache"
    CO.write_mock_cache(d, n=2, lr_hw=(8, 8), seed=2)
    CA.pack_cache(str(d), str(tmp_path / "a.ffsrc"), dtype="source")
    CA.pack_cache(str(d), str(tmp_path / "b.ffsrc"), dtype="fp16")
    sa, sb = os.path.getsize(tmp_path / "a.ffsrc"), os.path.getsize(tmp_path / "b.ffsrc")
    assert sb < 0.62 * sa
    ref = CO.OracleCachedDataset(str(d), augment=False)
    ours = CA.ShardDataset(str(tmp_path / "b.ffsrc"), augment=False)
    for i in range(2):
        a, b = ours[i], ref[i]
        assert torch.equal(a["lr"], b["lr"]) and torch.equal(a["hr"], b["hr"])          # lr / hr stay fp32
        for k in b["expert_imgs"]:
            assert torch.equal(a["expert_imgs"][k], b["expert_imgs"][k].half().float())
        for k in b["expert_feats"]:
            assert torch.equal(a["expert_feats"][k], b["expert_feats"][k].half().float())


def test_layout_alignment_and_header(tmp_path):
    d = tmp_path / "cache"
    CO.write_mock_cache(d, n=2, lr_hw=(9, 11), seed=3)          # odd sizes: segment byte counts not multiples of 16
    CA.pack_cache(str(d), str(tmp_path / "s.ffsrc"))
    c = CA.ShardCache(str(tmp_path / "s.ffsrc"))
    segs, rbytes = c.layout(0)
    assert rbytes % 512 == 0 and c.data_start % 4096 == 0 and c.uniform
    assert [s[0] for s in segs] == ["lr", "hr", "img.drct", "img.grl", "img.nafnet", "img.mamba",
                                    "feat.drct", "feat.grl", "feat.nafnet", "feat.mamba"]
    ends = 0
    for key, Cc, hh, ww, dt, off in segs:
        assert off % 16 == 0 and off >= ends
        ends = off + Cc * hh * ww * (2 if dt == "f16" else 4)
    assert ends <= rbytes and c.record(1).nbytes == rbytes
    assert dict((s[0], s[4]) for s in segs)["img.mamba"] == "f16" and dict((s[0], s[4]) for s in segs)["feat.drct"] == "f32"
    c.close()
    with open(tmp_path / "bad.ffsrc", "wb") as f:
        f.write(b"not a shard at all")
    with pytest.raises(ValueError):
        CA.ShardCache(str(tmp_path / "bad.ffsrc"))
    with pytest.raises(RuntimeError):
        CA.pack_cache(str(tmp_path / "nope"), str(tmp_path / "x.ffsrc"))


def test_tta_style_cache_without_hr_and_mixed_sizes(tmp_path):
    """Val / TTA caches: everything fp16, lr fp16, no hr, per-image sizes, tta_info (extract_test_tta_cache.py:296-326)."""
    d = tmp_path / "tta"
    d.mkdir()
    g = torch.Generator().manual_seed(4)
    for i, (h, w) in enumerate([(8, 12), (12, 8)]):
        stem = f"im_t{i}"
        torch.save({"outputs": {"drct": torch.rand(1, 3, 4 * h, 4 * w, generator=g).half()},
                    "features": {"drct": torch.randn(1, 180, h, w, generator=g).half()},
                    "lr": torch.rand(3, h, w, generator=g).half(), "filename": stem, "original_stem": "im",
                    "original_size": (4 * h, 4 * w), "tta_info": {"hflip": bool(i), "rot": i, "t_idx": i}}, d / f"{stem}_drct_part.pt")
        torch.save({"outputs": {"grl": torch.rand(1, 3, 4 * h, 4 * w, generator=g).half(),
                                "nafnet": torch.rand(1, 3, 4 * h, 4 * w, generator=g).half()},
                    "features": {"grl": torch.randn(1, 180, h, w, generator=g).half(),
                                 "nafnet": torch.randn(1, 64, h, w, generator=g).half()}, "filename": stem}, d / f"{stem}_rest_part.pt")
        torch.save({"outputs": {"mamba": torch.rand(1, 3, 4 * h, 4 * w, generator=g).half()},
                    "features": {"mamba": torch.randn(1, 180, h, w, generator=g).half()}, "filename": stem}, d / f"{stem}_mamba_part.pt")
    hdr = CA.pack_cache(str(d), str(tmp_path / "tta.ffsrc"))
    assert not hdr["uniform"] and hdr["meta"][1]["tta_info"] == {"hflip": True, "rot": 1, "t_idx": 1}
    assert hdr["meta"][0]["original_size"] == [32, 48]
    c = CA.ShardCache(str(tmp_path / "tta.ffsrc"))
    s = c.sample(1)
    ref = torch.load(d / "im_t1_rest_part.pt", weights_only=False)
    assert s["hr"] is None and s["lr"].dtype == torch.float16 and tuple(s["lr"].shape) == (3, 12, 8)
    assert torch.equal(s["expert_feats"]["nafnet"], ref["features"]["nafnet"][0])
    ds = CA.ShardDataset(str(tmp_path / "tta.ffsrc"), augment=False)
    assert "hr" not in ds[0] and ds[0]["expert_imgs"]["drct"].dtype == torch.float16      # like the reference: only mamba up-cast


def test_dihedral_codes_cover_every_augmentation():
    t = torch.arange(3 * 4 * 5, dtype=torch.float32).view(3, 4, 5)
    seen = set()
    for hf in (False, True):
        for vf in (False, True):
            for k in range(4):
                code = CA.dihedral_code(hf, vf, k)
                seen.add(code)
                want = CO.transform(t, hf, vf, k)
                tr, fy, fx = code & 1, code & 2, code & 4
                src = t
                if fy:
                    src = torch.flip(src, dims=[-2])
                if fx:
                    src = torch.flip(src, dims=[-1])
                got = src.transpose(-1, -2) if tr else src
                assert torch.equal(got, want), (hf, vf, k, code)
    assert seen == set(range(8))


def test_device_loader_refuses_cpu(tmp_path):
    d = tmp_path / "cache"
    CO.write_mock_cache(d, n=1, lr_hw=(8, 8))
    CA.pack_cache(str(d), str(tmp_path / "s.ffsrc"))
    with pytest.raises(RuntimeError, match="no CPU path"):
        CA.DeviceBatchLoader(str(tmp_path / "s.ffsrc"), 1, "cpu")


def test_epoch_batches_partition_the_epoch_over_ranks():
    for world in (1, 2, 8):
        seen = []
        for rank in range(world):
            bs = CA.epoch_batches(103, 4, True, seed=7, epoch=2, rank=rank, world=world, drop_last=False)
            assert all(len(b) == 4 for b in bs[:-1]) and 1 <= len(bs[-1]) <= 4
            seen += [i for b in bs for i in b]
        # every index at least once (padding wraps around, as DistributedSampler does), every rank the same permutation
        assert sorted(set(seen)) == list(range(103)) and len(seen) == -(-103 // world) * world
    a = CA.epoch_batches(50, 8, True, 1, 0)
    assert a == CA.epoch_batches(50, 8, True, 1, 0) and a != CA.epoch_batches(50, 8, True, 1, 1)
    assert len(a) == 6 and all(len(b) == 8 for b in a)                # drop_last
    assert CA.epoch_batches(10, 4, False, 0, 0, drop_last=False) == [[0, 1, 2, 3], [4, 5, 6, 7], [8, 9]]


def test_every_rank_gets_the_same_number_of_batches():
    """Each training step is a collective: a rank with one batch more would hang in NCCL at the end of the epoch
    (the advisor's case: total=65, world=8, B=3 used to give [3,2,2,2,2,2,2,2])."""
    for total, world, B in [(65, 8, 3), (103, 2, 4), (7, 8, 1), (64, 8, 8), (1000, 4, 32)]:
        for drop_last in (True, False):
            counts = [len(CA.epoch_batches(total, B, True, 3, 1, rank=r, world=world, drop_last=drop_last)) for r in range(world)]
            assert len(set(counts)) == 1, (total, world, B, drop_last, counts)
            assert counts[0] == CA.batches_per_epoch(total, B, world, drop_last)
            idx = [i for r in range(world) for b in CA.epoch_batches(total, B, True, 3, 1, rank=r, world=world, drop_last=drop_last) for i in b]
            if drop_last:
                assert len(idx) == len(set(idx)) == counts[0] * world * B          # no index twice, full batches only
            else:
                assert set(idx) == set(range(total))                               # padded by wrap-around


def test_shard_writer_uses_unique_temporaries_and_resolve_repacks_on_dtype_change(tmp_path):
    import glob
    lr, hr = torch.rand(3, 8, 8), torch.rand(3, 32, 32)
    imgs = {k: torch.rand(3, 32, 32) for k in ("drct", "grl", "nafnet", "mamba")}
    out = str(tmp_path / "a.ffsrc")
    w1, w2 = CA.ShardWriter(out), CA.ShardWriter(out)            # two writers of the same target (two ranks / workers)
    assert w1._tmp != w2._tmp
    for w in (w1, w2):
        w.add("s0", lr, hr, imgs)
        w.close()
    assert CA.ShardCache(out).count == 1 and not glob.glob(str(tmp_path / "*.tmp")) and not glob.glob(str(tmp_path / "*.part"))
    assert CA.ShardCache.read_header(out)["dtype_mode"] == "source"


def test_shard_writer_rejects_inconsistent_samples(tmp_path):
    lr, hr = torch.rand(3, 8, 8), torch.rand(3, 32, 32)
    imgs = {k: torch.rand(3, 32, 32) for k in ("drct", "grl", "nafnet", "mamba")}
    feats = {"drct": torch.randn(180, 8, 8), "grl": torch.randn(180, 8, 8), "nafnet": torch.randn(64, 8, 8), "mamba": torch.randn(180, 8, 8)}
    with pytest.raises(ValueError, match="expected"):
        with CA.ShardWriter(str(tmp_path / "a.ffsrc")) as w:
            w.add("a", lr, hr, imgs, feats)
            w.add("b", lr, hr, {**imgs, "grl": torch.rand(3, 16, 16)}, feats)
    assert not os.path.exists(tmp_path / "a.ffsrc") and not os.path.exists(str(tmp_path / "a.ffsrc") + ".records.tmp")
    with pytest.raises(ValueError, match="no tensor"):
        with CA.ShardWriter(str(tmp_path / "b.ffsrc")) as w:
            w.add("a", lr, hr, imgs, feats)
            w.add("b", lr, hr, {k: v for k, v in imgs.items() if k != "grl"}, feats)
    with pytest.raises(ValueError):
        CA.ShardWriter(str(tmp_path / "c.ffsrc"), dtype="int8")
    with CA.ShardWriter(str(tmp_path / "d.ffsrc"), dtype="fp16") as w:       # in-memory samples straight into a shard
        w.add("a", lr, hr, imgs, feats)
        w.add("b", lr, hr, {k: v for k, v in imgs.items() if k != "mamba"}, {k: v for k, v in feats.items() if k != "mamba"})
    c = CA.ShardCache(str(tmp_path / "d.ffsrc"))
    assert c.count == 2 and c.header["has_mamba"] == [True, False]
    s1 = c.sample(1)
    assert float(s1["expert_imgs"]["mamba"].abs().max()) == 0.0 and torch.equal(s1["expert_imgs"]["drct"], imgs["drct"].half())


def test_shard_dataset_survives_pickling_and_worker_processes(tmp_path):
    """DataLoader workers: fork inherits the mapping, spawn pickles the dataset -- the cache re-opens itself."""
    import pickle
    d = tmp_path / "cache"
    CO.write_mock_cache(d, n=4, lr_hw=(8, 8), seed=3)
    ds = CA.ShardDataset(str(d), augment=False)
    ds2 = pickle.loads(pickle.dumps(ds))
    assert ds2.cache is not ds.cache and len(ds2) == 4
    _same(ds2[2], ds[2])
    dl = torch.utils.data.DataLoader(ds, batch_size=2, num_workers=2, multiprocessing_context="spawn")
    names = [f for b in dl for f in b["filename"]]
    assert names == ["img_000", "img_001", "img_002", "img_003"]
