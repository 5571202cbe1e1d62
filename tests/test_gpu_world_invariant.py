"""World-invariant data-parallel training (``FusionTrainer(world_invariant=True)``) and gradient accumulation.

The ordered slot sum against a numpy float32 left fold; the mode at one GPU and one micro-batch against the default
step; ranks emulated in one process (local pass per rank, rows concatenated as the all-gather would, finish on every
instance) against the single-GPU run of the same micro-batches; both accumulation modes against the reference's
``loss/k``-backward loop; two real NCCL processes where the box has the GPUs; the deterministic-algorithms flag."""
import ctypes as C
import os
import sys

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

import isr_b200
from isr_b200 import _cabi as K
from oracle import fusion_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu
STAGE3 = {"charbonnier": 0, "l2": 0, "vgg": 0, "edge": 0, "clip": 0, "l1": 0.6, "swt": 0.25, "fft": 0.1, "ssim": 0.05}
BN_BUFS = ("running_mean", "running_var", "num_batches_tracked")


def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


def _rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return ((a - b).norm() / (b.norm() + 1e-30)).item()


# ------------------------------------------------------------------------------------------
# ffsr_sum_slots_ordered
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("pitch_kind", ["padded", "odd"])
@pytest.mark.parametrize("n", [1, 3, 1_433_217, 2 ** 24 + 5])
@pytest.mark.parametrize("M", [1, 2, 3, 8, 64])
def test_sum_slots_ordered_is_a_float32_left_fold(M, n, pitch_kind):
    """padded: rows on 16-byte boundaries (16-byte loads); odd: an odd pitch and an output off the 16-byte grid."""
    dev = _cuda()
    lib = K.load()
    pitch = (n + 3) // 4 * 4 + 4 if pitch_kind == "padded" else n + 1
    g = torch.Generator(device=dev).manual_seed(M * 7 + n)
    scale = torch.logspace(-4, 4, M, device=dev)[:, None]          # magnitudes that make the order visible
    slots = torch.randn(M, pitch, device=dev, generator=g) * scale
    off = 0 if pitch_kind == "padded" else 1
    S = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)

    def run():
        out = torch.full((n + off,), float("nan"), device=dev)
        K.check(lib.ffsr_sum_slots_ordered(slots.data_ptr(), M, n, pitch, out.data_ptr() + 4 * off, S), "sum_slots_ordered")
        return out[off:]

    a, b = run(), run()
    torch.cuda.synchronize()
    assert torch.equal(a, b)
    s = slots[:, :n].cpu().numpy()
    ref = s[0].copy()
    for m in range(1, M):
        ref += s[m]                                                  # one float32 rounding per add, in slot order
    assert np.array_equal(a.cpu().numpy(), ref)


def test_sum_slots_ordered_rejects_bad_arguments():
    dev = _cuda()
    lib = K.load()
    x = torch.zeros(4, 16, device=dev)
    S = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    assert lib.ffsr_sum_slots_ordered(x.data_ptr(), 0, 16, 16, x.data_ptr(), S) != 0               # M < 1
    assert lib.ffsr_sum_slots_ordered(x.data_ptr(), 2, 16, 8, x[3].data_ptr(), S) != 0             # pitch < n
    assert lib.ffsr_sum_slots_ordered(x.data_ptr(), 2, 16, 16, x[1].data_ptr(), S) != 0            # out overlaps


# ------------------------------------------------------------------------------------------
# trainer
# ------------------------------------------------------------------------------------------
def _inputs(dev, B, S, seed=0):
    torch.manual_seed(seed)
    lr, imgs, fts, hr = O.synthetic_inputs(B, S, S)
    return (lr.to(dev), {k: v.to(dev) for k, v in imgs.items()}, {k: v.to(dev) for k, v in fts.items()}, hr.to(dev))


def _trainer(dev, precision="fp32", dropout=True, **kw):
    from isr_b200.losses import CombinedLoss
    from isr_b200.trainer import FusionTrainer
    torch.manual_seed(0)
    m = isr_b200.CompleteEnhancedFusionSR(None).to(dev)
    m.precision = precision
    if not dropout:
        m.cross_band.band_attention.dropout = 0.0
        m.collaborative.cross_attn.dropout = 0.0
    crit = CombinedLoss()
    crit.set_weights(STAGE3)
    tr = FusionTrainer(m, crit, lr=2e-4, **kw)
    # the gradient bucket each step applies (the default step zeroes it afterwards); a clone recorded during a graph
    # capture is refreshed by every replay
    tr.grad_snaps = []
    apply = tr.optimizer.apply_summed

    def snap_then_apply(count):
        tr.grad_snaps.append(tr.optimizer.grads.clone())
        apply(count)
    tr.optimizer.apply_summed = snap_then_apply
    return tr


def _state(tr, loss, comps):
    o = tr.optimizer
    st = {"loss": loss.detach().clone(), "grads": tr.grad_snaps[-1].clone(), "flat": o.bucket.flat.clone(),
          "exp_avg": o.exp_avg.clone(), "exp_avg_sq": o.exp_avg_sq.clone(), "ema": o.ema.clone()}
    st.update({"comp." + k: v.detach().clone() for k, v in comps.items()})
    st.update({n: b.clone() for n, b in tr.model.named_buffers() if n.endswith(BN_BUFS)})
    return st


def _run(tr, batches):
    out = []
    for args in batches:
        loss, comps = tr.step(*args)
        out.append(_state(tr, loss, comps))
    torch.cuda.synchronize()
    return out


def _assert_same(r1, r2, what=""):
    assert len(r1) == len(r2)
    for s, (a, b) in enumerate(zip(r1, r2)):
        assert a.keys() == b.keys() and any(k.endswith("running_var") for k in a)
        for k in a:
            assert torch.equal(a[k], b[k]), (what, s, k, float((a[k].double() - b[k].double()).abs().max()))


@pytest.mark.timeout(900)
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_invariant_one_gpu_one_micro_batch_is_the_default_step(precision):
    """N=1, k=1 with dropout on: 3 eager steps, capture, 3 replays -- bit for bit the default trainer's."""
    dev = _cuda()
    args = _inputs(dev, 8, 64)
    runs = []
    for inv in (False, True):
        tr = _trainer(dev, precision, cuda_graph=True, graph_warmup=3, world_invariant=inv)
        runs.append(_run(tr, [args] * 6))
        assert tr._graph is not None
    assert all(torch.isfinite(s["loss"]) for s in runs[0])
    _assert_same(runs[0], runs[1])


def _emulated_run(dev, world, M, batches):
    """`world` trainer instances in one process, each the rank of a world-size run; every step runs each rank's
    local pass on its micro-batches, concatenates the rows in rank order (what all_gather_into_tensor does) and
    finishes the step on every instance.  Returns every instance's per-step states."""
    from isr_b200.training import seed_counter
    k = M // world
    ranks = [_trainer(dev, cuda_graph=False, accumulation_steps=k, world_invariant=True) for _ in range(world)]
    base = ranks[0]._seed_base if ranks[0]._seed_base is not None else _trainer(
        dev, cuda_graph=False, accumulation_steps=M, world_invariant=True)._seed_base
    for t in ranks:
        t._seed_base = base                                          # rank 0's base, as the broadcast hands it out
    out = [[] for _ in ranks]
    for s, (lr, imgs, fts, hr) in enumerate(batches):
        B = lr.shape[0] // world
        rows = []
        for r, t in enumerate(ranks):
            t.model.train()
            seed_counter(dev).fill_(s)                               # each process has its own step counter
            sl = slice(r * B, (r + 1) * B)
            micro = t._split(lr[sl], {n: v[sl] for n, v in imgs.items()}, {n: v[sl] for n, v in fts.items()}, hr[sl])
            rows.append(t._local_rows(micro, r * k))
        gathered = torch.cat(rows, 0)
        for r, t in enumerate(ranks):
            seed_counter(dev).fill_(s)
            loss, comps = t._finish(gathered)
            out[r].append(_state(t, loss, comps))
    torch.cuda.synchronize()
    return out


@pytest.mark.timeout(1200)
def test_emulated_ranks_are_bitwise_the_single_gpu_run():
    """M=4 micro-batches of 2 patches, dropout on: N in {1, 2, 4} emulated ranks and the N=1, k=4 trainer (eager, and
    graph-replayed) agree bit for bit over 3 steps in losses, gradients, parameters, Adam moments, EMA and BN buffers."""
    dev = _cuda()
    M, b, S = 4, 2, 32
    batches = [_inputs(dev, M * b, S, seed=s) for s in range(3)]
    ref = _run(_trainer(dev, cuda_graph=False, accumulation_steps=M, world_invariant=True), batches)
    graph_tr = _trainer(dev, cuda_graph=True, graph_warmup=1, accumulation_steps=M, world_invariant=True)
    _assert_same(ref, _run(graph_tr, batches), "graph")
    assert graph_tr._graph is not None
    assert all(torch.isfinite(s["loss"]) for s in ref)
    for world in (1, 2, 4):
        for r, got in enumerate(_emulated_run(dev, world, M, batches)):
            _assert_same(ref, got, f"N={world} rank {r}")


@pytest.mark.timeout(900)
def test_accumulation_matches_the_reference_loop():
    """One fp32 step (dropout 0) of the reference's loop -- loss/4 backward x4, clip_grad_norm_, torch.optim.AdamW --
    against world_invariant k=4 and the default mode's accumulation_steps=4."""
    dev = _cuda()
    k, b, S = 4, 2, 48
    lr, imgs, fts, hr = _inputs(dev, k * b, S)
    from isr_b200.losses import CombinedLoss
    torch.manual_seed(0)
    m = isr_b200.CompleteEnhancedFusionSR(None).to(dev).train()
    m.cross_band.band_attention.dropout = 0.0
    m.collaborative.cross_attn.dropout = 0.0
    crit = CombinedLoss()
    crit.set_weights(STAGE3)
    before = torch.cat([p.detach().reshape(-1) for p in m.parameters()]).clone()
    opt = torch.optim.AdamW(m.parameters(), lr=2e-4, weight_decay=1e-4)
    opt.zero_grad()
    for j in range(k):
        sl = slice(j * b, (j + 1) * b)
        sr = m.forward_with_precomputed(lr[sl], {n: v[sl] for n, v in imgs.items()}, {n: v[sl] for n, v in fts.items()})
        (crit(sr.clamp(0, 1), hr[sl]) / k).backward()
    ref_grads = torch.cat([p.grad.reshape(-1) for p in m.parameters()]) * k
    torch.nn.utils.clip_grad_norm_(m.parameters(), 1.0)
    opt.step()
    ref_update = torch.cat([p.detach().reshape(-1) for p in m.parameters()]) - before
    ref_bufs = {n: t for n, t in m.named_buffers() if n.endswith(BN_BUFS)}

    for inv in (True, False):
        tr = _trainer(dev, dropout=False, cuda_graph=False, accumulation_steps=k, world_invariant=inv)
        o = tr.optimizer
        unpack = lambda flat: torch.cat([flat[off:off + p.numel()] for off, p in zip(o.bucket.offsets, o._params)])
        start = unpack(o.bucket.flat).clone()
        tr.step(lr, imgs, fts, hr)
        torch.cuda.synchronize()
        assert _rel(unpack(tr.grad_snaps[-1]), ref_grads) < 1e-6, inv
        assert _rel(unpack(o.bucket.flat) - start, ref_update) < 1e-3, inv
        for n, t in tr.model.named_buffers():
            if n.endswith("num_batches_tracked"):
                assert int(t) == int(ref_bufs[n]), (inv, n)
            elif n.endswith(BN_BUFS):
                assert _rel(t, ref_bufs[n]) < 1e-6, (inv, n)


@pytest.mark.timeout(900)
def test_invariant_step_under_deterministic_algorithms():
    """N=1, k=2 (hash-seeded dropout, rows, ordered sum) under torch.use_deterministic_algorithms(True): same bits."""
    dev = _cuda()
    batches = [_inputs(dev, 8, 32, seed=s) for s in range(4)]
    ref = _run(_trainer(dev, "bf16", cuda_graph=True, graph_warmup=2, accumulation_steps=2, world_invariant=True), batches)
    prev, prev_warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        got = _run(_trainer(dev, "bf16", cuda_graph=True, graph_warmup=2, accumulation_steps=2, world_invariant=True),
                   batches)
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=prev_warn)
    _assert_same(ref, got)


def test_micro_batch_count_must_divide_over_the_ranks():
    dev = _cuda()
    with pytest.raises(ValueError):
        _trainer(dev, cuda_graph=False, accumulation_steps=0)
    with pytest.raises(ValueError):
        _trainer(dev, cuda_graph=False, global_micro_batches=4)                  # needs world_invariant
    tr = _trainer(dev, cuda_graph=False, world_invariant=True, global_micro_batches=3)
    assert tr.accumulation_steps == 3
    with pytest.raises(ValueError):
        tr.step(*_inputs(dev, 4, 16))                                            # 4 patches do not split into 3


# ------------------------------------------------------------------------------------------
# real NCCL ranks
# ------------------------------------------------------------------------------------------
def _nccl_worker(rank, world, k, port, q):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    M, b, S = world * k, 2, 32
    batches = [_inputs(dev, M * b, S, seed=s) for s in range(4)]
    B = k * b
    mine = [(lr[rank * B:(rank + 1) * B], {n: v[rank * B:(rank + 1) * B] for n, v in imgs.items()},
             {n: v[rank * B:(rank + 1) * B] for n, v in fts.items()}, hr[rank * B:(rank + 1) * B])
            for lr, imgs, fts, hr in batches]
    got = _run(_trainer(dev, cuda_graph=True, graph_warmup=2, accumulation_steps=k, world_invariant=True), mine)
    dist.barrier()
    same = None
    if rank == 0:                     # the N=1 run of the same M micro-batches, in this process
        dist.destroy_process_group()
        ref = _run(_trainer(dev, cuda_graph=True, graph_warmup=2, accumulation_steps=M, world_invariant=True), batches)
        try:
            _assert_same(ref, got)
            same = "ok"
        except AssertionError as e:
            same = str(e)
    else:
        dist.destroy_process_group()
    q.put((rank, same))


@pytest.mark.timeout(1200)
@pytest.mark.parametrize("world,k", [(2, 2), (4, 1)])
def test_nccl_ranks_equal_the_single_gpu_run(world, k):
    if not torch.cuda.is_available() or torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} CUDA devices (one process per GPU)")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29811 + world
    procs = [ctx.Process(target=_nccl_worker, args=(r, world, k, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=1100) for _ in range(world))
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    assert res[0] == "ok", res[0]
