"""Host-side pieces of resuming a training run: the loader's batch plan and augmentation draws continued from a saved
position, world-invariant loader positions on another world size, the refusals of trainer and loader states, the
dropout seed tape and the atomic checkpoint write."""
import io
import os
import random

import pytest
import torch

from isr_b200 import cache as CA
from isr_b200 import training as T
from isr_b200 import trainer as TR

TOTAL, SEED = 45, 13


def _roundtrip(obj):
    """Through torch.save / torch.load(weights_only=True), as a checkpoint file carries it."""
    buf = io.BytesIO()
    torch.save(obj, buf)
    buf.seek(0)
    return torch.load(buf, weights_only=True)


def _run(B, world_invariant, epochs, rank=0, world=1, drop_last=True, epoch0=0, start=0, rng=None):
    """(epoch, batch index, sample indices, codes, rng state after) of every batch from (epoch0, start) on."""
    rng = rng if rng is not None else random.Random(SEED * 1000003 + rank)
    out = []
    for e in range(epoch0, epochs):
        sched = CA.epoch_schedule(TOTAL, B, True, SEED, e, rank, world, drop_last, world_invariant, True, rng,
                                  start if e == epoch0 else 0)
        for k, (idxs, codes, after) in enumerate(sched, start if e == epoch0 else 0):
            out.append((e, k, idxs, codes, after))
    return out


def _position(entry, per_epoch):
    """The loader's state after the consumer received ``entry``: its next batch, an epoch's end counting as batch 0
    of the next epoch."""
    e, k = entry[0], entry[1] + 1
    return (e + 1, 0) if k >= per_epoch else (e, k)


@pytest.mark.parametrize("world_invariant", [False, True])
@pytest.mark.parametrize("drop_last", [True, False])
def test_resumed_schedule_is_the_tail_of_the_uninterrupted_one(world_invariant, drop_last):
    B, world, rank = 4, 2, 1
    full = _run(B, world_invariant, 3, rank, world, drop_last)
    per_epoch = sum(1 for x in full if x[0] == 0)
    span = world * B
    want_len = (TOTAL // span if drop_last else -(-TOTAL // span)) if world_invariant else \
        CA.batches_per_epoch(TOTAL, B, world, drop_last)
    assert per_epoch == want_len and len(full) == 3 * per_epoch
    # the plan is the host helpers' plan
    for e in range(3):
        got = [x[2] for x in full if x[0] == e]
        if world_invariant:
            plan = CA.world_invariant_batches(TOTAL, B, True, SEED, e, rank, world, drop_last)
            assert got == [idx for _, idx in plan]
            assert [x[3] for x in full if x[0] == e] == [[CA.augment_code(SEED, e, p) for p in pos] for pos, _ in plan]
        else:
            assert got == CA.epoch_batches(TOTAL, B, True, SEED, e, rank, world, drop_last)
    # save after a mid-epoch batch, after an epoch's last batch, and after the first batch of the next epoch
    for cut in (2, per_epoch - 1, per_epoch):
        epoch, nxt = _position(full[cut], per_epoch)
        rng = None
        if not world_invariant:
            rng = random.Random(0)
            rng.setstate(_roundtrip(full[cut][4]))
        tail = _run(B, world_invariant, 3, rank, world, drop_last, epoch, nxt, rng)
        assert [x[:4] for x in tail] == [x[:4] for x in full[cut + 1:]], cut


@pytest.mark.parametrize("drop_last", [True, False])
def test_world_invariant_position_resumes_on_fewer_ranks(drop_last):
    """Saved at N=4 (B=2) mid-epoch 1: N'=2 (B=4) and N'=1 (B=8) continue with the same global batches and codes."""
    def steps(world, epoch0, start):
        B = 8 // world
        runs = [_run(B, True, 3, r, world, drop_last, epoch0, start) for r in range(world)]
        return [[i for run in runs for i in run[t][2]] for t in range(len(runs[0]))], \
               [[c for run in runs for c in run[t][3]] for t in range(len(runs[0]))]
    ref_idx, ref_codes = steps(4, 0, 0)
    per_epoch = len(ref_idx) // 3
    cut = per_epoch + 3
    epoch, nxt = 1, 4
    saved = {"samples": TOTAL, "seed": SEED, "shuffle": True, "drop_last": drop_last, "augment": True,
             "world_invariant": True, "B": 2, "world": 4, "epoch": epoch, "batch": nxt, "rng": None}
    for world in (2, 1):
        now = dict(saved, B=8 // world, world=world)
        CA.check_loader_resume(_roundtrip(saved), now)
        idx, codes = steps(world, epoch, nxt)
        assert idx == ref_idx[cut + 1:] and codes == ref_codes[cut + 1:], world


def _loader_state(**kw):
    st = {"samples": TOTAL, "seed": SEED, "shuffle": True, "drop_last": True, "augment": True,
          "world_invariant": False, "B": 4, "world": 2, "epoch": 1, "batch": 3, "rng": random.Random(1).getstate()}
    st.update(kw)
    return st


@pytest.mark.parametrize("field,value", [("samples", TOTAL + 1), ("seed", SEED + 1), ("shuffle", False),
                                         ("drop_last", False), ("augment", False), ("world_invariant", True),
                                         ("B", 8), ("world", 4)])
def test_loader_refusals_name_the_field(field, value):
    saved = _loader_state()
    now = {k: v for k, v in saved.items() if k not in ("epoch", "batch", "rng")}
    CA.check_loader_resume(saved, now)
    with pytest.raises(ValueError, match=field if field != "B" else "batch_size"):
        CA.check_loader_resume(saved, dict(now, **{field: value}))


def test_loader_world_rules():
    # default mode: another world size only at an epoch boundary
    CA.check_loader_resume(_loader_state(batch=0), _loader_state(world=4))
    # world-invariant: world * B must stay
    wi = _loader_state(world_invariant=True, rng=None)
    CA.check_loader_resume(wi, _loader_state(world_invariant=True, world=1, B=8))
    CA.check_loader_resume(wi, _loader_state(world_invariant=True, world=8, B=1))
    with pytest.raises(ValueError, match="world \\* batch_size"):
        CA.check_loader_resume(wi, _loader_state(world_invariant=True, world=1, B=4))


def _config(**kw):
    c = {"bucket": (1433220, [0, 4, 20]), "precision": "bf16", "world_invariant": False, "accumulation_steps": 1,
         "world": 2, "micro_batches": 2}
    c.update(kw)
    return c


def test_trainer_refusals_name_the_field():
    saved = _roundtrip(_config())
    TR.check_resume(saved, _config())
    with pytest.raises(ValueError, match="bucket layout"):
        TR.check_resume(saved, _config(bucket=(1433220, [0, 8, 20])))
    with pytest.raises(ValueError, match="precision"):
        TR.check_resume(saved, _config(precision="fp32"))
    with pytest.raises(ValueError, match="world_invariant"):
        TR.check_resume(saved, _config(world_invariant=True))
    with pytest.raises(ValueError, match="accumulation_steps"):
        TR.check_resume(saved, _config(accumulation_steps=2, micro_batches=4))
    # default mode: another world size only at an epoch boundary (not bitwise there)
    with pytest.raises(ValueError, match="world size"):
        TR.check_resume(saved, _config(world=1, micro_batches=1))
    TR.check_resume(saved, _config(world=1, micro_batches=1), at_epoch_boundary=True)
    # world-invariant: any N dividing M, with N * k = M
    wi = _config(world_invariant=True, world=4, accumulation_steps=1, micro_batches=4)
    for world in (1, 2, 4):
        TR.check_resume(wi, _config(world_invariant=True, world=world, accumulation_steps=4 // world,
                                    micro_batches=4))
    with pytest.raises(ValueError, match="does not divide"):
        TR.check_resume(wi, _config(world_invariant=True, world=3, accumulation_steps=1, micro_batches=3))
    with pytest.raises(ValueError, match="micro_batches"):
        TR.check_resume(wi, _config(world_invariant=True, world=2, accumulation_steps=1, micro_batches=2))


def test_seed_tape_records_without_changing_draws_and_replays_without_drawing():
    torch.manual_seed(5)
    plain = [T.dropout_host_seed() for _ in range(4)]
    torch.manual_seed(5)
    with T.seed_tape() as tape:
        recorded = [T.dropout_host_seed() for _ in range(4)]
    assert recorded == plain == tape.seeds
    after = torch.get_rng_state()
    with T.seed_tape(_roundtrip(tape.seeds)):
        replayed = [T.dropout_host_seed() for _ in range(4)]
        with pytest.raises(RuntimeError):
            T.dropout_host_seed()                       # the step asked for more seeds than its capture froze
    assert replayed == plain
    assert torch.equal(torch.get_rng_state(), after)   # replaying consumed nothing from the CPU generator
    # world-invariant micro-batches of a step of several keep their hash, recorded or replayed
    with T.seed_tape() as tape, T.micro_batch(3, 77):
        hashed = [T.dropout_host_seed(), T.dropout_host_seed()]
    assert hashed == tape.seeds == [T.dropout_seed(77, 3, 0), T.dropout_seed(77, 3, 1)]
    with T.seed_tape([1]), T.micro_batch(3, 77):
        assert [T.dropout_host_seed(), T.dropout_host_seed()] == hashed


def test_atomic_save_leaves_no_partial_file(tmp_path):
    path = tmp_path / "ckpt.pt"
    TR.atomic_save({"step": 1, "w": torch.arange(4.0)}, str(path))
    before = path.read_bytes()
    bad = {"w": torch.zeros(1 << 16), "fn": lambda: 0}             # torch.save fails after it has started writing
    with pytest.raises(Exception):
        TR.atomic_save(bad, str(path))
    assert path.read_bytes() == before
    assert os.listdir(tmp_path) == ["ckpt.pt"]
    fresh = tmp_path / "new.pt"
    with pytest.raises(Exception):
        TR.atomic_save(bad, str(fresh))
    assert sorted(os.listdir(tmp_path)) == ["ckpt.pt"]
    TR.atomic_save({"step": 2}, str(path))
    assert torch.load(str(path), weights_only=True) == {"step": 2}
