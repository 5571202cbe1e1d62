"""Flat cache shards and the device-side batch loader (SURVEY §8f N2).

The reference stores one training sample as three ``torch.save`` pickles (``{stem}_{drct,rest,mamba}_part.pt``) and
reads them with ``torch.load(weights_only=False)`` in DataLoader workers, up-casting and flipping on the CPU
(``src/data/cached_dataset.py:135-282``).  One 64x64 sample is 13.9 MB of fp32, so a B200 that trains hundreds of
patches per second needs several GB/s of unpickling -- the loader, not the GPU, sets the pace.  Here:

* ``pack_cache`` converts a reference cache directory once into ONE flat file: a JSON header and fixed-layout raw
  records (every tensor dense ``[C][h][w]``, 16-byte aligned), readable through ``mmap`` with no parsing.
  ``dtype="source"`` keeps the stored dtypes (fp32, fp16 for the MambaIR part) and is bit-exact with the reference
  loader; ``dtype="fp16"`` stores expert images / features as fp16 (what the reference's own val / TTA caches do).
* ``ShardDataset`` has ``CachedSRDataset``'s constructor and ``__getitem__`` contract on top of a shard (host tensors,
  same ``random`` draws for the augmentation) -- the drop-in for unchanged callers.
* ``DeviceBatchLoader`` is the B200 path: B records are gathered into a pinned staging buffer, cross PCIe in ONE copy
  on a side stream, and ONE kernel (``ffsr_cache_unpack``) up-casts, applies each sample's flip / rot90 and writes the
  dense batch tensors; the next batch is in flight while the current one trains.

No pickles of our own are ever written (SURVEY App. C).
"""
from __future__ import annotations

import ctypes as C
import json
import mmap
import os
import queue
import random
import struct
import tempfile
import threading
import warnings
from pathlib import Path
from typing import Dict, Iterator, List, Optional, Sequence, Tuple

import numpy as np
import torch

EXPERT_ORDER = ("drct", "grl", "nafnet", "mamba")
MAGIC = b"FFSRC1\x00\x00"
_ALIGN_SEG, _ALIGN_REC, _ALIGN_DATA = 16, 512, 4096
_NP = {"f32": np.float32, "f16": np.float16}


def _round_up(x: int, a: int) -> int:
    return (x + a - 1) // a * a


def _dihedral_table() -> Dict[Tuple[bool, bool, int], int]:
    """Brute force over a non-square index tensor: for each (hflip, vflip, rot_k) the code whose gather reproduces the
    torch ops (built once at import: 16 tiny tensor ops)."""
    h, w = 2, 3
    src = torch.arange(h * w).view(h, w)
    table = {}
    for hf in (False, True):
        for vf in (False, True):
            for k in range(4):
                t = src
                if hf:
                    t = torch.flip(t, dims=[-1])
                if vf:
                    t = torch.flip(t, dims=[-2])
                if k:
                    t = torch.rot90(t, k=k, dims=[-2, -1])
                hit = None
                for code in range(8):
                    tr, fy, fx = code & 1, code & 2, code & 4
                    ho, wo = (w, h) if tr else (h, w)
                    if tuple(t.shape) != (ho, wo):
                        continue
                    ok = True
                    for y in range(ho):
                        for x in range(wo):
                            sy, sx = (x, y) if tr else (y, x)
                            if fy:
                                sy = h - 1 - sy
                            if fx:
                                sx = w - 1 - sx
                            ok = ok and int(t[y, x]) == int(src[sy, sx])
                    if ok:
                        hit = code
                        break
                assert hit is not None
                table[(hf, vf, k)] = hit
    return table


_DIHEDRAL = _dihedral_table()


def dihedral_code(hflip: bool, vflip: bool, rot_k: int) -> int:
    """The loader's ``hflip -> vflip -> rot90(k)`` (cached_dataset.py:266-274) as one of the 8 dihedral maps of
    ``ffsr_cache_unpack``: bit 0 transpose, bit 1 reverse source rows, bit 2 reverse source columns, i.e.
    ``out[y][x] = in[sy][sx]`` with ``(sy, sx) = (x, y) if transpose else (y, x)``, then ``sy = h-1-sy`` / ``sx = w-1-sx``."""
    return _DIHEDRAL[(bool(hflip), bool(vflip), int(rot_k) % 4)]


# ---------------------------------------------------------------------------------------------------
# record layout
# ---------------------------------------------------------------------------------------------------
def _layout(tensors: Sequence[dict], h: int, w: int, scale: int):
    """[(key, C, hh, ww, dtype, offset)], record_bytes for an LR size (h, w)."""
    segs, off = [], 0
    for t in tensors:
        s = scale if t["hr"] else 1
        hh, ww = h * s, w * s
        nbytes = t["C"] * hh * ww * (2 if t["dtype"] == "f16" else 4)
        segs.append((t["key"], t["C"], hh, ww, t["dtype"], off))
        off = _round_up(off + nbytes, _ALIGN_SEG)
    return segs, _round_up(off, _ALIGN_REC)


def _read_parts(d: Path, stem: str):
    """The three pickles of one sample in their STORED dtypes (no up-cast), batch dim squeezed
    (cached_dataset.py:150-214); a missing mamba part is ``None`` (zero-filled by the caller, as :178-185 does)."""
    a = torch.load(d / f"{stem}_drct_part.pt", weights_only=False)
    b = torch.load(d / f"{stem}_rest_part.pt", weights_only=False)
    mp = d / f"{stem}_mamba_part.pt"
    c = torch.load(mp, weights_only=False) if mp.exists() else None
    imgs, feats = dict(a["outputs"]), dict(a.get("features") or {})
    imgs.update(b["outputs"])
    feats.update(b.get("features") or {})
    if c is not None:
        imgs.update(c["outputs"])
        feats.update(c.get("features") or {})
    sq = lambda t: t.squeeze(0) if t.dim() == 4 else t                      # noqa: E731
    imgs = {k: sq(v) for k, v in imgs.items() if v is not None}
    feats = {k: sq(v) for k, v in feats.items() if v is not None}
    meta = {k: a[k] for k in ("original_stem", "original_size", "tta_info") if k in a}
    return a["lr"], a.get("hr"), imgs, feats, c is not None, meta


class ShardWriter:
    """Writes a shard sample by sample (what an extractor would use directly instead of three pickles per sample):

        with ShardWriter("train.ffsrc", dtype="fp16") as w:
            w.add(stem, lr, hr, {"drct": sr, ...}, {"drct": feat, ...})

    The first sample fixes the tensor table (names, channel counts, stored dtypes); a later sample without a MambaIR
    tensor gets zeros (the reference loader's fallback, cached_dataset.py:178-185, 203-206)."""

    def __init__(self, out_path: str, dtype: str = "source", load_features: bool = True):
        if dtype not in ("source", "fp16"):
            raise ValueError("dtype must be 'source' (bit-exact with the reference loader) or 'fp16'")
        self.out_path, self.dtype, self.load_features = str(out_path), dtype, bool(load_features)
        self.tensors: Optional[List[dict]] = None
        self.hw, self.offsets, self.has_mamba, self.metas, self.stems = [], [], [], [], []
        self.scale, self._pos = 4, 0
        # unique temporaries beside the target (several processes may pack the same directory: torchrun ranks, DataLoader
        # workers); the finished shard appears atomically through os.replace
        fd, self._tmp = tempfile.mkstemp(prefix=os.path.basename(self.out_path) + ".", suffix=".records.tmp",
                                         dir=os.path.dirname(os.path.abspath(self.out_path)))
        self._rec = os.fdopen(fd, "wb")
        self.header: Optional[dict] = None

    def _sdt(self, t: torch.Tensor, lossy: bool) -> str:
        if t.dtype not in (torch.float32, torch.float16):
            raise ValueError(f"unsupported cache dtype {t.dtype}")
        return "f16" if (t.dtype == torch.float16 or (lossy and self.dtype == "fp16")) else "f32"

    def add(self, stem: str, lr: torch.Tensor, hr: Optional[torch.Tensor], imgs: Dict[str, torch.Tensor],
            feats: Optional[Dict[str, torch.Tensor]] = None, has_mamba: Optional[bool] = None, meta: Optional[dict] = None):
        feats = feats or {}
        h, w = int(lr.shape[-2]), int(lr.shape[-1])
        if self.tensors is None:
            self.scale = int(next(iter(imgs.values())).shape[-1]) // w
            ts = [{"key": "lr", "C": int(lr.shape[0]), "hr": False, "dtype": self._sdt(lr, False)}]
            if hr is not None:
                ts.append({"key": "hr", "C": int(hr.shape[0]), "hr": True, "dtype": self._sdt(hr, False)})
            for n in EXPERT_ORDER:
                if n in imgs or n == "mamba":
                    ts.append({"key": "img." + n, "C": 3, "hr": True, "dtype": self._sdt(imgs[n], True) if n in imgs else "f16"})
            if self.load_features:
                for n in EXPERT_ORDER:
                    if n in feats or n == "mamba":
                        ts.append({"key": "feat." + n, "C": int(feats[n].shape[0]) if n in feats else 180, "hr": False,
                                   "dtype": self._sdt(feats[n], True) if n in feats else "f16"})
            self.tensors = ts
        segs, rbytes = _layout(self.tensors, h, w, self.scale)
        buf = np.zeros(rbytes, dtype=np.uint8)
        src = {"lr": lr, "hr": hr}
        src.update({"img." + k: v for k, v in imgs.items()})
        src.update({"feat." + k: v for k, v in feats.items()})
        for key, Cc, hh, ww, dt, off in segs:
            t = src.get(key)
            if t is None:
                if key.endswith(".mamba"):
                    continue                          # zeros: the reference's fallback for a missing MambaIR part
                raise ValueError(f"sample '{stem}' has no tensor '{key}' (the first sample defines the tensor set)")
            if tuple(t.shape) != (Cc, hh, ww):
                raise ValueError(f"sample '{stem}': '{key}' is {tuple(t.shape)}, expected {(Cc, hh, ww)}")
            arr = t.detach().cpu().contiguous().numpy().astype(_NP[dt], copy=False)
            buf[off:off + arr.nbytes] = arr.reshape(-1).view(np.uint8)
        self._rec.write(buf.tobytes())
        self.stems.append(stem)
        self.hw.append([h, w])
        self.offsets.append(self._pos)
        self._pos += rbytes
        self.has_mamba.append(bool("mamba" in imgs if has_mamba is None else has_mamba))
        self.metas.append(meta or {})

    def close(self) -> dict:
        if self.header is not None:
            return self.header
        self._rec.close()
        header = {"version": 1, "count": len(self.stems), "scale": self.scale, "dtype_mode": self.dtype,
                  "tensors": self.tensors or [], "hw": self.hw, "offsets": self.offsets, "stems": self.stems,
                  "has_mamba": self.has_mamba, "load_features": self.load_features,
                  "uniform": len({tuple(x) for x in self.hw}) <= 1}
        if any(self.metas):
            header["meta"] = [json.loads(json.dumps(m, default=lambda o: list(o) if isinstance(o, tuple) else str(o)))
                              for m in self.metas]
        hj = json.dumps(header).encode("utf-8")
        data_start = _round_up(len(MAGIC) + 8 + len(hj), _ALIGN_DATA)
        fd, part = tempfile.mkstemp(prefix=os.path.basename(self.out_path) + ".", suffix=".part",
                                    dir=os.path.dirname(os.path.abspath(self.out_path)))
        with os.fdopen(fd, "wb") as f:                # written beside the target and renamed: readers never see half a shard
            f.write(MAGIC)
            f.write(struct.pack("<Q", len(hj)))
            f.write(hj)
            f.write(b"\x00" * (data_start - f.tell()))
            with open(self._tmp, "rb") as rec:
                while True:
                    chunk = rec.read(64 << 20)
                    if not chunk:
                        break
                    f.write(chunk)
        os.remove(self._tmp)
        os.replace(part, self.out_path)
        self.header = header
        return header

    def __enter__(self):
        return self

    def __exit__(self, et, ev, tb):
        if et is None:
            self.close()
        else:
            self._rec.close()
            if os.path.exists(self._tmp):
                os.remove(self._tmp)
        return False


def pack_cache(feature_dir: str, out_path: str, dtype: str = "source", load_features: bool = True) -> dict:
    """Convert a reference cache directory (``*_drct_part.pt`` + ``*_rest_part.pt`` [+ ``*_mamba_part.pt``]) into one
    flat shard.  Stems follow the reference's rule (cached_dataset.py:84-109: sorted, incomplete pairs dropped).
    Returns the header."""
    d = Path(feature_dir)
    if not d.exists():
        raise RuntimeError(f"Feature cache directory not found: {feature_dir}")
    stems = [f.name.replace("_drct_part.pt", "") for f in sorted(d.glob("*_drct_part.pt"))]
    if not stems:
        raise RuntimeError(f"No cached features found in {feature_dir}!")
    stems = [s for s in stems if (d / f"{s}_rest_part.pt").exists()]
    with ShardWriter(out_path, dtype, load_features) as w:
        for stem in stems:
            lr, hr, imgs, feats, hm, meta = _read_parts(d, stem)
            w.add(stem, lr, hr, imgs, feats, hm, meta)
    return w.header


SHARD_NAME = "_cache.ffsrc"


def resolve_shard(feature_dir: str, dtype: str = "source", load_features: bool = True) -> str:
    """A shard path for what the reference calls ``feature_dir``: a shard file is returned as is; a reference cache
    DIRECTORY (the argument unchanged callers pass, train.py:594-646) is packed once into ``<dir>/_cache.ffsrc`` and
    that file is reused afterwards (re-packed when a ``*_part.pt`` is newer than the shard)."""
    p = Path(feature_dir)
    if p.is_file():
        return str(p)
    if not p.exists():
        raise RuntimeError(f"Feature cache directory not found: {feature_dir}")
    shard = p / SHARD_NAME
    parts = list(p.glob("*_part.pt"))
    if not parts and not shard.exists():
        raise RuntimeError(f"No cached features found in {feature_dir}!")
    def stale():
        if not shard.exists():
            return True
        if parts and max(f.stat().st_mtime for f in parts) > shard.stat().st_mtime:
            return True
        try:                                          # an existing shard packed for another request (dtype / features)
            hdr = ShardCache.read_header(str(shard))
        except Exception:
            return True
        return hdr.get("dtype_mode") != dtype or (load_features and not hdr.get("load_features", False))

    import torch.distributed as dist
    multi = dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
    if stale() and (not multi or dist.get_rank() == 0):           # one packer per job; the others wait at the barrier
        print(f"[isr_b200.cache] packing {feature_dir} -> {shard} ({dtype}) ...", flush=True)
        pack_cache(str(p), str(shard), dtype=dtype, load_features=load_features)
    if multi:
        dist.barrier()
    return str(shard)


class ShardCache:
    """Read-only view of a shard: header + memory-mapped records."""

    @staticmethod
    def read_header(path: str) -> dict:
        with open(path, "rb") as f:
            if f.read(len(MAGIC)) != MAGIC:
                raise ValueError(f"{path} is not an FFSRC1 cache shard")
            (n,) = struct.unpack("<Q", f.read(8))
            return json.loads(f.read(n).decode("utf-8"))

    def __init__(self, path: str):
        self.path = str(path)
        with open(self.path, "rb") as f:
            if f.read(len(MAGIC)) != MAGIC:
                raise ValueError(f"{path} is not an FFSRC1 cache shard")
            (n,) = struct.unpack("<Q", f.read(8))
            self.header = json.loads(f.read(n).decode("utf-8"))
        if self.header.get("version") != 1:
            raise ValueError(f"unsupported shard version {self.header.get('version')}")
        self.data_start = _round_up(len(MAGIC) + 8 + n, _ALIGN_DATA)
        self._file = open(self.path, "rb")
        self._mm = mmap.mmap(self._file.fileno(), 0, access=mmap.ACCESS_READ)
        self._bytes = np.frombuffer(self._mm, dtype=np.uint8)
        self.count = int(self.header["count"])
        self.stems: List[str] = self.header["stems"]
        self.scale = int(self.header["scale"])
        self.tensors = self.header["tensors"]
        self.uniform = bool(self.header["uniform"])
        self._layouts: Dict[Tuple[int, int], tuple] = {}

    def __getstate__(self):
        return {"path": self.path}                     # DataLoader workers started by spawn re-open the mapping

    def __setstate__(self, state):
        self.__init__(state["path"])

    def layout(self, i: int):
        h, w = self.header["hw"][i]
        lay = self._layouts.get((h, w))
        if lay is None:
            lay = self._layouts[(h, w)] = _layout(self.tensors, h, w, self.scale)
        return lay

    def record(self, i: int) -> np.ndarray:
        """The raw bytes of record i (a view into the mapping)."""
        _, rbytes = self.layout(i)
        o = self.data_start + self.header["offsets"][i]
        return self._bytes[o:o + rbytes]

    def sample(self, i: int, load_features: bool = True, copy: bool = True) -> dict:
        """Record i as host tensors in their stored dtypes.  ``copy=False`` returns read-only VIEWS of the mapping (for
        callers that transform every tensor into a new one anyway); the default copies."""
        segs, _ = self.layout(i)
        rec = self.record(i)
        out = {"lr": None, "hr": None, "expert_imgs": {}, "expert_feats": {} if load_features else None,
               "filename": self.stems[i]}
        for key, Cc, hh, ww, dt, off in segs:
            if key.startswith("feat.") and not load_features:
                continue
            n = Cc * hh * ww * (2 if dt == "f16" else 4)
            arr = rec[off:off + n].view(_NP[dt]).reshape(Cc, hh, ww)
            if copy:
                t = torch.from_numpy(arr.copy())
            else:
                with warnings.catch_warnings():
                    warnings.simplefilter("ignore", UserWarning)         # "array is not writable": it is never written
                    t = torch.from_numpy(arr)
            if key in ("lr", "hr"):
                out[key] = t
            elif key.startswith("img."):
                out["expert_imgs"][key[4:]] = t
            else:
                out["expert_feats"][key[5:]] = t
        return out

    def close(self):
        self._bytes = None
        try:
            self._mm.close()
        except BufferError:            # views handed out are still alive; the mapping goes with them
            pass
        self._file.close()


class ShardDataset(torch.utils.data.Dataset):
    """``CachedSRDataset`` (cached_dataset.py:50-232) over a shard: same arguments, same sample dict, same ``random``
    draws.  With a ``dtype="source"`` shard every tensor is bit-identical to what the reference class returns."""

    def __init__(self, feature_dir: str, augment: bool = True, repeat_factor: int = 1, load_features: bool = True):
        super().__init__()
        self.cache = ShardCache(resolve_shard(feature_dir))          # a reference cache directory is packed on first use
        self.file_stems = self.cache.stems
        self.has_mamba = dict(zip(self.cache.stems, self.cache.header["has_mamba"]))
        self.augment, self.repeat_factor = augment, repeat_factor
        self.load_features = load_features and self.cache.header["load_features"]
        self._upcast_all = self.cache.header["dtype_mode"] == "fp16"

    def __len__(self) -> int:
        return self.cache.count * self.repeat_factor

    def __getitem__(self, idx: int) -> dict:
        # every returned tensor is produced by exactly ONE pass over its bytes: views of the mapping go through a single
        # fused flip (+ transpose) / up-cast / clone, instead of copy -> flip -> flip -> rot90 (each a full copy)
        s = self.cache.sample(idx % self.cache.count, self.load_features, copy=False)
        code = 0
        if self.augment:
            hflip = random.random() < 0.5                    # the reference's three draws, in its order (:262-264)
            vflip = random.random() < 0.5
            rot_k = random.randint(0, 3)
            code = dihedral_code(hflip, vflip, rot_k)
        tr, fy, fx = bool(code & 1), bool(code & 2), bool(code & 4)

        def tf(t, up):
            # out = T?(flip_rows_if_fy(flip_cols_if_fx(t)))  ==  flip(t.T, rows if fx, cols if fy) when transposed
            v = t.transpose(-1, -2) if tr else t
            dims = [d for d, f in ((-2, fx if tr else fy), (-1, fy if tr else fx)) if f]
            if dims:
                v = torch.flip(v, dims)
                v = v.float() if (up and v.dtype != torch.float32) else v
                return v.contiguous()
            if up and v.dtype != torch.float32:
                return v.float().contiguous()
            return v.contiguous().clone() if v.is_contiguous() else v.contiguous()
        lr = tf(s["lr"], False)                              # lr / hr keep their stored dtype, as in the reference
        hr = tf(s["hr"], False) if s["hr"] is not None else None
        imgs = {k: tf(v, self._upcast_all or k == "mamba") for k, v in s["expert_imgs"].items()}
        feats = None
        if s["expert_feats"] is not None:
            feats = {k: tf(v, self._upcast_all or k == "mamba") for k, v in s["expert_feats"].items()}
        out = {"lr": lr, "hr": hr, "expert_imgs": imgs, "filename": s["filename"]}
        if hr is None:
            del out["hr"]
        if feats is not None:
            out["expert_feats"] = feats
        return out


# ---------------------------------------------------------------------------------------------------
# device loader
# ---------------------------------------------------------------------------------------------------
def epoch_batches(total: int, batch_size: int, shuffle: bool, seed: int, epoch: int, rank: int = 0, world: int = 1,
                  drop_last: bool = True) -> List[List[int]]:
    """Index batches of one epoch for one rank: a permutation shared by all ranks (seeded by ``seed + epoch``), every
    world-th index from position ``rank``, cut into batches.  Ranks never share an index within an epoch."""
    order = _epoch_order(total, shuffle, seed, epoch)
    if world > 1:
        # every rank must run the SAME number of steps: each step is a collective (gradient all-reduce, BatchNorm buffer
        # sync), so a rank with one batch more would wait in NCCL for ever at the end of the epoch.  With drop_last the
        # permutation is cut to a multiple of world * batch_size; without it, it is padded by wrapping around, as
        # torch.utils.data.DistributedSampler does.
        if drop_last:
            order = order[:len(order) // (world * batch_size) * (world * batch_size)]
        elif order:
            per = -(-len(order) // world)
            order = (order * (1 + (per * world) // len(order)))[:per * world]
    order = order[rank::world]
    out = [order[i:i + batch_size] for i in range(0, len(order), batch_size)]
    if out and drop_last and len(out[-1]) < batch_size:
        out.pop()
    return out


def _epoch_order(total: int, shuffle: bool, seed: int, epoch: int) -> List[int]:
    if shuffle:
        g = torch.Generator().manual_seed(seed + epoch)
        return torch.randperm(total, generator=g).tolist()
    return list(range(total))


def world_invariant_batches(total: int, batch_size: int, shuffle: bool, seed: int, epoch: int, rank: int = 0,
                            world: int = 1, drop_last: bool = True) -> List[Tuple[List[int], List[int]]]:
    """(positions, sample indices) of one rank's batches in the world-invariant layout: at step t rank r takes
    positions [t*world*B + r*B, t*world*B + (r+1)*B) of the epoch permutation shared by all ranks, which is cut to a
    multiple of world*B (drop_last) or padded by wrapping around.  With world*B fixed, a position lands on the same
    step and, cut into micro-batches of b = B/k, in the same global micro-batch (r*k + j) for every world size."""
    order = _epoch_order(total, shuffle, seed, epoch)
    span = world * batch_size
    if drop_last:
        order = order[:len(order) // span * span]
    elif order:
        target = -(-len(order) // span) * span
        order = (order * -(-target // len(order)))[:target]
    out = []
    for t in range(len(order) // span):
        pos = list(range(t * span + rank * batch_size, t * span + (rank + 1) * batch_size))
        out.append((pos, [order[p] for p in pos]))
    return out


def augment_code(seed: int, epoch: int, position: int) -> int:
    """Dihedral code of the sample at ``position`` of the epoch permutation, drawn (the reference's three draws, in its
    order) from a generator keyed by (seed, epoch, position) alone: the same on whichever rank loads the sample."""
    rng = random.Random(f"ffsr-augment:{seed}:{epoch}:{position}")
    hflip = rng.random() < 0.5
    vflip = rng.random() < 0.5
    return dihedral_code(hflip, vflip, rng.randint(0, 3))


def epoch_schedule(total: int, batch_size: int, shuffle: bool, seed: int, epoch: int, rank: int = 0, world: int = 1,
                   drop_last: bool = True, world_invariant: bool = False, augment: bool = True,
                   rng: Optional[random.Random] = None, start: int = 0):
    """``DeviceBatchLoader``'s host plan of one epoch from batch ``start`` on: yields (sample indices, dihedral codes,
    state of ``rng`` after the batch's draws or None).  World-invariant codes come from ``augment_code`` by position;
    default codes are the reference's three draws per sample from ``rng``, in batch order.  The batches before
    ``start`` are skipped without a draw: resuming restores the ``rng`` state those draws left."""
    if world_invariant:
        plan = world_invariant_batches(total, batch_size, shuffle, seed, epoch, rank, world, drop_last)
    else:
        plan = [(None, b) for b in epoch_batches(total, batch_size, shuffle, seed, epoch, rank, world, drop_last)]
    for pos, idxs in plan[start:]:
        codes = [0] * len(idxs)
        if augment and pos is not None:
            codes = [augment_code(seed, epoch, p) for p in pos]
        elif augment:
            for j in range(len(idxs)):
                hflip = rng.random() < 0.5
                vflip = rng.random() < 0.5
                codes[j] = dihedral_code(hflip, vflip, rng.randint(0, 3))
        yield idxs, codes, (rng.getstate() if augment and pos is None else None)


_LOADER_KEYS = ("samples", "seed", "shuffle", "drop_last", "augment", "world_invariant")


def check_loader_resume(saved: dict, now: dict) -> None:
    """Raise ``ValueError`` naming the field when a ``DeviceBatchLoader.state_dict()`` ``saved`` cannot continue in a
    loader configured as ``now`` (the same keys).  World-invariant mode resumes on another world size when
    world * batch_size is unchanged: a position keeps its step and augmentation.  The default mode keeps its world
    size and batch size, except that the world size may change at an epoch boundary (batch 0)."""
    for k in _LOADER_KEYS:
        if saved[k] != now[k]:
            raise ValueError(f"loader state: {k} is {saved[k]!r} in the checkpoint, {now[k]!r} here")
    if now["world_invariant"]:
        if saved["world"] * saved["B"] != now["world"] * now["B"]:
            raise ValueError(f"loader state: world * batch_size is {saved['world']} * {saved['B']} in the checkpoint, "
                             f"{now['world']} * {now['B']} here; a world-invariant resume keeps the product")
        return
    if saved["B"] != now["B"]:
        raise ValueError(f"loader state: batch_size is {saved['B']} in the checkpoint, {now['B']} here")
    if saved["world"] != now["world"] and saved["batch"] != 0:
        raise ValueError(f"loader state: world is {saved['world']} in the checkpoint, {now['world']} here, and the "
                         f"checkpoint is mid-epoch (batch {saved['batch']}): the default mode's batches depend on the "
                         "world size, so it changes only at an epoch boundary")


def batches_per_epoch(total: int, batch_size: int, world: int = 1, drop_last: bool = True) -> int:
    """len(epoch_batches(...)) without building them (identical on every rank)."""
    if world > 1:
        if drop_last:
            return total // (world * batch_size)
        per = -(-total // world) if total else 0
        return -(-per // batch_size)
    return total // batch_size if drop_last else -(-total // batch_size)


class DeviceBatchLoader:
    """Batches of a shard as DEVICE tensors, shaped like the reference DataLoader's collated dict
    (``lr [B,3,h,w]``, ``hr``, ``expert_imgs{name}``, ``expert_feats{name}``, ``filename`` list; train.py:300-322).

    Per batch: B records -> pinned staging (a few host threads; plain memcpy out of the page cache), one async H2D on a
    copy stream, one ``ffsr_cache_unpack`` launch (up-cast + per-sample flip/rot90 + collate).  ``depth`` batches are
    in flight; the consumer's stream waits on the batch's event, never the host.

    ``rng``: a ``random.Random`` (default seeded from ``seed``) from which the augmentation of every sample is drawn in
    the reference's order, so a run seeded like ``random.seed(s)`` reproduces the reference's augmentations.
    Under ``world > 1`` rank r takes every world-th index of the (shared-seed) epoch permutation.

    ``world_invariant=True``: rank r's batch at step t is the contiguous block of positions
    [t*world*B + r*B, t*world*B + (r+1)*B) of the shared permutation, and each sample's augmentation is drawn from a
    generator keyed by (seed, epoch, position) (``world_invariant_batches``, ``augment_code``).  For a fixed world*B,
    every micro-batch of a step then gets the same samples and flips for any world size: the loader of
    ``FusionTrainer(world_invariant=True)``.  ``rng`` is not used in this mode.

    ``state_dict()`` / ``load_state_dict()``: the epoch and the index of the next batch the consumer has not received
    yet, the ``rng`` state those batches' draws leave (default mode), and the settings the batch plan depends on.  A
    loaded loader's next iteration yields exactly the remaining batches of that epoch -- same samples, dihedral codes
    and tensor bits, skipped batches never read -- then continues into the next epochs.  A world-invariant state
    resumes on another world size when world * batch_size is unchanged (``check_loader_resume``)."""

    def __init__(self, shard: str, batch_size: int, device, augment: bool = True, shuffle: bool = True,
                 drop_last: bool = True, load_features: bool = True, repeat_factor: int = 1, rank: int = 0, world: int = 1,
                 seed: int = 0, depth: int = 2, copy_threads: int = 4, rng: Optional[random.Random] = None,
                 out_dtype: torch.dtype = torch.float32, reuse_buffers: bool = True, world_invariant: bool = False):
        from . import _cabi as K
        self.K = K
        self.lib = K.load()                                   # raises FusionLibraryError when the library is missing
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("DeviceBatchLoader needs a CUDA device: there is no CPU path (use ShardDataset on the host)")
        self.cache = shard if isinstance(shard, ShardCache) else ShardCache(shard)
        if batch_size > 1 and not self.cache.uniform:
            raise ValueError("batch_size > 1 needs a shard whose samples all have the same LR size")
        if out_dtype not in (torch.float32, torch.bfloat16):
            raise ValueError("out_dtype must be torch.float32 or torch.bfloat16")
        self.B, self.augment, self.shuffle, self.drop_last = int(batch_size), augment, shuffle, drop_last
        self.load_features = load_features and self.cache.header["load_features"]
        self.repeat_factor, self.rank, self.world, self.seed = repeat_factor, rank, world, seed
        self.world_invariant = bool(world_invariant)
        self.depth = max(2, int(depth))
        self.rng = rng if rng is not None else random.Random(seed * 1000003 + rank)
        self.out_dtype = out_dtype
        # Batch tensors are recycled round-robin (a batch stays valid until `depth` further batches have been fetched;
        # clone what must live longer).  Allocating fresh tensors per batch from a producer thread makes the caching
        # allocator wait for blocks still in use by the training step (measured: +35 ms per step).
        self.reuse_buffers = bool(reuse_buffers)
        self.epoch = 0
        self._start = 0                                       # first batch of the next iteration (load_state_dict)
        self._cursor = None                                   # (epoch, next batch, rng state) of the consumer
        self.copy_threads = max(1, int(copy_threads))
        self._codes_bytes = _round_up(4 * self.B, _ALIGN_REC)
        self._slots = None
        self._copy_stream = torch.cuda.Stream(self.device)
        self._sm = torch.cuda.get_device_properties(self.device).multi_processor_count
        self.launches = 0

    def __len__(self) -> int:
        total = self.cache.count * self.repeat_factor
        if self.world_invariant:
            span = self.world * self.B
            return total // span if self.drop_last else -(-total // span)
        return batches_per_epoch(total, self.B, self.world, self.drop_last)

    def set_epoch(self, epoch: int) -> None:
        """The epoch the next iteration runs.  Setting the epoch a loaded state resumes keeps its batch position."""
        if int(epoch) != self.epoch:
            self._start = 0
        self.epoch = int(epoch)
        self._cursor = None

    # ---- one batch --------------------------------------------------------------------------------
    def _slot(self, k: int, rbytes: int):
        if self._slots is None or self._slots[0]["host"].numel() < self._codes_bytes + self.B * rbytes:
            n = self._codes_bytes + self.B * rbytes
            self._slots = [{"host": torch.empty(n, dtype=torch.uint8).pin_memory(),
                            "dev": torch.empty(n, dtype=torch.uint8, device=self.device), "ev": None, "consumed": None,
                            "outs": {}} for _ in range(self.depth + 1)]
        return self._slots[k % len(self._slots)]

    def _produce(self, k: int, idxs: List[int], batch_codes: List[int]) -> dict:
        K, cache = self.K, self.cache
        n = len(idxs)
        recs = [i % cache.count for i in idxs]
        segs, rbytes = cache.layout(recs[0])
        slot = self._slot(k, rbytes)
        if slot["ev"] is not None:
            slot["ev"].synchronize()                          # the H2D that last used this staging buffer has finished
        host = slot["host"].numpy()
        codes = np.zeros(self.B, dtype=np.int32)
        codes[:n] = batch_codes
        host[:4 * self.B] = codes.view(np.uint8)
        base = self._codes_bytes

        def copy(j):
            host[base + j * rbytes: base + (j + 1) * rbytes] = cache.record(recs[j])
        if self.copy_threads > 1 and n > 1:
            ts = [threading.Thread(target=lambda a=a: [copy(j) for j in range(a, n, self.copy_threads)])
                  for a in range(min(self.copy_threads, n))]
            for t in ts:
                t.start()
            for t in ts:
                t.join()
        else:
            for j in range(n):
                copy(j)

        h0, w0 = cache.header["hw"][recs[0]]
        transposed = {bool(c & 1) for c in codes[:n]}
        if h0 != w0 and len(transposed) > 1:
            raise ValueError("quarter-turn augmentation of non-square samples changes the shape per sample: "
                             "use batch_size=1 or square patches")
        tr = bool(codes[0] & 1)
        nbytes = base + n * rbytes
        out = {"lr": None, "expert_imgs": {}, "filename": [cache.stems[r] for r in recs]}
        if self.load_features:
            out["expert_feats"] = {}
        with torch.cuda.stream(self._copy_stream):
            slot["dev"][:nbytes].copy_(slot["host"][:nbytes], non_blocking=True)
            if self.reuse_buffers and slot["consumed"] is not None:
                self._copy_stream.wait_event(slot["consumed"])       # the consumer's reads of this slot's last batch
            arr = (K.CacheSegment * len(segs))()
            m = 0
            tensors = []
            for key, Cc, hh, ww, dt, off in segs:
                if key.startswith("feat.") and not self.load_features:
                    continue
                ho, wo = (ww, hh) if tr else (hh, ww)
                if self.reuse_buffers:
                    t = slot["outs"].get((key, n, Cc, ho, wo))
                    if t is None:
                        t = slot["outs"][(key, n, Cc, ho, wo)] = torch.empty(n, Cc, ho, wo, device=self.device, dtype=self.out_dtype)
                else:
                    t = torch.empty(n, Cc, ho, wo, device=self.device, dtype=self.out_dtype)
                tensors.append(t)
                s = arr[m]
                s.src_offset, s.dst, s.C, s.h, s.w = off, t.data_ptr(), Cc, hh, ww
                s.src_dtype = K.DT_F16 if dt == "f16" else K.DT_F32
                s.dst_dtype = K.DT_BF16 if self.out_dtype == torch.bfloat16 else K.DT_F32
                m += 1
                if key in ("lr", "hr"):
                    out[key] = t
                elif key.startswith("img."):
                    out["expert_imgs"][key[4:]] = t
                else:
                    out["expert_feats"][key[5:]] = t
            dev_ptr = slot["dev"].data_ptr()
            K.check(self.lib.ffsr_cache_unpack(dev_ptr + base, rbytes, n, arr, m, dev_ptr if self.augment else None, self._sm,
                                               C.c_void_p(self._copy_stream.cuda_stream)), "cache_unpack")
            self.launches += 1
            ev = torch.cuda.Event()
            ev.record(self._copy_stream)
        slot["ev"] = ev
        out["_event"], out["_tensors"], out["_slot"] = ev, tensors, slot
        return out

    # ---- resuming ---------------------------------------------------------------------------------
    def _resume_config(self) -> dict:
        return {"samples": self.cache.count * self.repeat_factor, "seed": self.seed, "shuffle": bool(self.shuffle),
                "drop_last": bool(self.drop_last), "augment": bool(self.augment),
                "world_invariant": self.world_invariant, "B": self.B, "world": self.world}

    def state_dict(self) -> dict:
        """Position of the consumer: the epoch and index of the next batch it has not received (a state taken after an
        epoch's last batch is batch 0 of the next epoch), the ``rng`` state (default mode) and the plan's settings.
        The producer thread runs ahead; what it drew for batches not yet handed out is not part of the state."""
        epoch, nxt, rng = self._cursor if self._cursor is not None else (self.epoch, self._start, None)
        if nxt >= len(self):
            epoch, nxt = epoch + 1, 0
        if rng is None and not self.world_invariant:
            rng = self.rng.getstate()
        return dict(self._resume_config(), epoch=int(epoch), batch=int(nxt), rng=rng)

    def load_state_dict(self, state: dict) -> None:
        """Continue from ``state``: the next iteration yields the remaining batches of its epoch.  Raises ValueError
        (``check_loader_resume``) when this loader's settings cannot continue it."""
        check_loader_resume(state, self._resume_config())
        self.epoch, self._start, self._cursor = int(state["epoch"]), int(state["batch"]), None
        if not self.world_invariant and state["world"] == self.world and state["rng"] is not None:
            self.rng.setstate(state["rng"])

    def __iter__(self) -> Iterator[dict]:
        epoch, start = self.epoch, self._start
        self.epoch += 1
        self._start = 0
        self._cursor = (epoch, start, None if self.world_invariant else self.rng.getstate())
        sched = epoch_schedule(self.cache.count * self.repeat_factor, self.B, self.shuffle, self.seed, epoch, self.rank,
                               self.world, self.drop_last, self.world_invariant, self.augment, self.rng, start)
        q: "queue.Queue" = queue.Queue(maxsize=self.depth - 1)
        stop = threading.Event()

        def worker():
            try:
                with torch.cuda.device(self.device):
                    for k, (idxs, codes, rng_after) in enumerate(sched):
                        if stop.is_set():
                            return
                        item = self._produce(k, idxs, codes)
                        item["_rng"] = rng_after
                        q.put(item)
                q.put(None)
            except BaseException as exc:                      # surface loader errors in the consumer
                q.put(exc)

        th = threading.Thread(target=worker, daemon=True)
        th.start()
        nxt = start
        try:
            while True:
                item = q.get()
                if item is None:
                    break
                if isinstance(item, BaseException):
                    raise item
                cur = torch.cuda.current_stream(self.device)
                cur.wait_event(item.pop("_event"))
                for t in item.pop("_tensors"):
                    t.record_stream(cur)
                slot = item.pop("_slot")
                nxt += 1
                rng_after = item.pop("_rng")
                self._cursor = (epoch, nxt, rng_after if rng_after is not None else self._cursor[2])
                yield item
                if self.reuse_buffers:                         # the consumer is done enqueueing work on this batch
                    done = torch.cuda.Event()
                    done.record(torch.cuda.current_stream(self.device))
                    slot["consumed"] = done
        finally:
            stop.set()
            while th.is_alive():
                try:
                    q.get_nowait()
                except queue.Empty:
                    pass
                th.join(timeout=0.05)


def create_cached_dataloader(feature_dir: str, batch_size: int = 16, num_workers: int = 4, augment: bool = True,
                             repeat_factor: int = 20, pin_memory: bool = True, persistent_workers: bool = True,
                             prefetch_factor: int = 4, load_features: bool = True, device=None, **kw):
    """``create_cached_dataloader`` of the reference (cached_dataset.py:285-337) over a shard (or a reference cache
    directory, packed on first use).  With ``device`` it returns the ``DeviceBatchLoader`` (batches already on the GPU);
    without, a torch ``DataLoader`` over ``ShardDataset`` with the reference's settings (shuffle, drop_last, workers)."""
    feature_dir = resolve_shard(feature_dir)
    if device is not None:
        return DeviceBatchLoader(feature_dir, batch_size, device, augment=augment, shuffle=True, drop_last=True,
                                 load_features=load_features, repeat_factor=repeat_factor, **kw)
    ds = ShardDataset(feature_dir, augment=augment, repeat_factor=repeat_factor, load_features=load_features)
    return torch.utils.data.DataLoader(ds, batch_size=batch_size, shuffle=True, num_workers=num_workers, pin_memory=pin_memory,
                                       drop_last=True, persistent_workers=persistent_workers and num_workers > 0,
                                       prefetch_factor=prefetch_factor if num_workers > 0 else None)
