"""Host-side pieces of world-invariant data-parallel training: the loader layout and augmentation keys, the BatchNorm
fold over several micro-batches, and the dropout seed hash."""
import pytest
import torch

from isr_b200 import cache as CA
from isr_b200 import training as T

TOTAL, SPAN, b = 1000, 32, 4          # N * B fixed at 32 patches per step, micro-batches of 4 (M = 8)


def _micro_batches(world, drop_last, epoch=3):
    """global micro-batch i of every step -> (positions, indices, augmentation codes), as the ranks would load them."""
    B = SPAN // world
    k = B // b
    per_rank = [CA.world_invariant_batches(TOTAL, B, True, 11, epoch, r, world, drop_last) for r in range(world)]
    steps = {len(p) for p in per_rank}
    assert len(steps) == 1
    out = []
    for t in range(steps.pop()):
        for r in range(world):
            pos, idx = per_rank[r][t]
            for j in range(k):
                sl = slice(j * b, (j + 1) * b)
                out.append((pos[sl], idx[sl], [CA.augment_code(11, epoch, p) for p in pos[sl]]))
    return out


@pytest.mark.parametrize("drop_last", [True, False])
def test_loader_micro_batches_do_not_depend_on_world_size(drop_last):
    ref = _micro_batches(1, drop_last)
    assert len(ref) == (TOTAL // SPAN if drop_last else -(-TOTAL // SPAN)) * (SPAN // b)
    for world in (2, 4, 8):
        assert _micro_batches(world, drop_last) == ref, world
    seen = [i for _, idx, _ in ref for i in idx]
    if drop_last:
        assert len(set(seen)) == len(seen) == TOTAL // SPAN * SPAN
    else:
        assert set(seen) == set(range(TOTAL))                   # every sample once, the tail padded by wrapping around


def test_augment_code_is_keyed_by_seed_epoch_position():
    codes = [CA.augment_code(5, 0, p) for p in range(256)]
    assert codes == [CA.augment_code(5, 0, p) for p in range(256)]
    assert set(codes) == set(range(8))
    assert codes != [CA.augment_code(5, 1, p) for p in range(256)]
    assert codes != [CA.augment_code(6, 0, p) for p in range(256)]


def _bn_records(M, G=3, C=8, n=50, seed=0):
    """M micro-batches of G groups: (bn, mean, biased var, n) per group batch, and the raw group batches."""
    g = torch.Generator().manual_seed(seed)
    xs = [torch.randn(G, n, C, generator=g, dtype=torch.float64) * (1 + i) + i for i in range(M)]
    return xs, [(x.mean(1).float(), x.var(1, unbiased=False).float()) for x in xs]


def _fold(bn, stats, n):
    T.fold_running_stats([(bn, m, v, n) for m, v in stats])


def test_bn_fold_of_many_micro_batches_matches_sequential_batchnorm():
    M, G, C, n = 8, 3, 8, 50
    xs, stats = _bn_records(M, G, C, n)
    bn = torch.nn.BatchNorm2d(C)
    _fold(bn, stats, n)
    ref = torch.nn.BatchNorm2d(C).double().train()
    for x in xs:                                                # M * G sequential BatchNorm2d calls (fp64)
        for grp in x:
            ref(grp.t().reshape(1, C, n, 1))
    for a, r in ((bn.running_mean, ref.running_mean), (bn.running_var, ref.running_var)):
        assert ((a.double() - r).norm() / r.norm()).item() < 1e-6
    assert int(bn.num_batches_tracked) == int(ref.num_batches_tracked) == M * G


def test_bn_fold_of_one_micro_batch_is_the_per_forward_fold():
    _, stats = _bn_records(1)
    bn1, bn2 = torch.nn.BatchNorm2d(8), torch.nn.BatchNorm2d(8)
    _fold(bn1, stats, 50)
    # the per-forward fold as it was written before it took several micro-batches
    mean, var = stats[0][0], stats[0][1] * (50 / 49)
    G = mean.shape[0]
    wts = 0.1 * (1.0 - 0.1) ** torch.arange(G - 1, -1, -1, dtype=torch.float32)
    keep = (1.0 - 0.1) ** G
    bn2.running_mean.mul_(keep).add_((wts[:, None] * mean).sum(0))
    bn2.running_var.mul_(keep).add_((wts[:, None] * var).sum(0))
    assert torch.equal(bn1.running_mean, bn2.running_mean) and torch.equal(bn1.running_var, bn2.running_var)
    assert int(bn1.num_batches_tracked) == G


def test_bn_fold_of_gathered_ranks_equals_one_rank():
    """Records of two emulated ranks, concatenated in rank order, fold to the same bits as one rank holding all."""
    _, stats = _bn_records(4, seed=3)
    one, two = torch.nn.BatchNorm2d(8), torch.nn.BatchNorm2d(8)
    _fold(one, stats, 50)
    rank0, rank1 = stats[:2], stats[2:]
    _fold(two, rank0 + rank1, 50)
    for name in ("running_mean", "running_var", "num_batches_tracked"):
        assert torch.equal(getattr(one, name), getattr(two, name)), name


def test_dropout_seed_hash():
    base = 0x1234_5678_9ABC
    seeds = {T.dropout_seed(base, i, c) for i in range(1000) for c in range(100)}
    assert len(seeds) == 100_000                                # no collisions over 10^5 (micro-batch, call) pairs
    assert all(0 <= s < 2 ** 62 for s in seeds)
    # a pure function of (base, global micro-batch, call): rank r of N running micro-batches r*k .. r*k+k-1 asks
    # for the same seeds for every N
    M = 8
    ref = [[T.dropout_seed(base, i, c) for c in range(2)] for i in range(M)]
    for N in (1, 2, 4, 8):
        k = M // N
        got = [[T.dropout_seed(base, r * k + j, c) for c in range(2)] for r in range(N) for j in range(k)]
        assert got == ref
    assert T.dropout_seed(base + 1, 0, 0) != T.dropout_seed(base, 0, 0)


def test_micro_batch_context_draws_seeds():
    """Inside micro_batch the seeds come from the hash (call counter per micro-batch); without a base they are the
    default CPU-generator draws."""
    with T.micro_batch(5, 77) as mb:
        assert [mb.seed(), mb.seed()] == [T.dropout_seed(77, 5, 0), T.dropout_seed(77, 5, 1)]
    torch.manual_seed(0)
    ref = T._draw_seed()
    torch.manual_seed(0)
    with T.micro_batch(0, None) as mb:
        assert mb.seed() == ref
    assert T._MICRO is None

