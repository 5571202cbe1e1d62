"""Resuming training from a checkpoint gives the bits of the uninterrupted run.

Default mode on a mock shard (augmentation and shuffle on, stage-3 fused losses, attention dropout on), eager and
CUDA-graph steps, fp32 and bf16, saved during warm-up, right after the capture and several replays later, across epoch
boundaries; the resumed process is rebuilt after a different ``torch.manual_seed``.  World-invariant mode with ranks
emulated in one process (as tests/test_gpu_world_invariant.py does) saved at N ranks and resumed at fewer; two real
NCCL ranks saving and one process resuming where the box has the GPUs; a reference ``torch.optim.AdamW`` checkpoint."""
import gc
import os
import sys

import pytest
import torch
import torch.multiprocessing as mp

import isr_b200
from isr_b200 import cache as CA
from oracle import cache_oracle as CO
from oracle import fusion_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu
STAGE3 = {"charbonnier": 0, "l2": 0, "vgg": 0, "edge": 0, "clip": 0, "l1": 0.6, "swt": 0.25, "fft": 0.1, "ssim": 0.05}
BN_BUFS = ("running_mean", "running_var", "num_batches_tracked")


def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


def _trainer(dev, seed, precision="fp32", **kw):
    from isr_b200.losses import CombinedLoss
    from isr_b200.trainer import FusionTrainer
    torch.manual_seed(seed)
    m = isr_b200.CompleteEnhancedFusionSR(None).to(dev)
    m.precision = precision
    crit = CombinedLoss()
    crit.set_weights(STAGE3)
    return FusionTrainer(m, crit, lr=2e-4, **kw)


def _final(tr):
    o = tr.optimizer
    st = {"flat": o.bucket.flat.clone(), "exp_avg": o.exp_avg.clone(), "exp_avg_sq": o.exp_avg_sq.clone(),
          "ema": o.ema.clone(), "steps": torch.tensor(o.steps)}
    st.update({n: b.clone() for n, b in tr.model.named_buffers() if n.endswith(BN_BUFS)})
    return st


def _assert_equal_dicts(a, b, what):
    assert a.keys() == b.keys(), what
    for k in a:
        assert torch.equal(a[k], b[k]), (what, k, float((a[k].double() - b[k].double()).abs().max()))


def _step_record(loss, comps):
    rec = {"loss": loss.detach().clone()}
    rec.update({"comp." + k: v.detach().clone() for k, v in comps.items()})
    return rec


def _train(tr, loader, steps, out):
    """``steps`` steps over the loader's epochs; appends each step's loss and components to ``out``."""
    it = iter(loader)
    done = 0
    while done < steps:
        try:
            b = next(it)
        except StopIteration:
            it = iter(loader)
            continue
        out.append(_step_record(*tr.step(b["lr"], b["expert_imgs"], b.get("expert_feats"), b["hr"])))
        done += 1
    torch.cuda.synchronize()
    it.close()


@pytest.fixture(scope="module")
def shard(tmp_path_factory):
    d = tmp_path_factory.mktemp("resume")
    CO.write_mock_cache(d / "cache", n=7, lr_hw=(16, 16), seed=31)
    CA.pack_cache(str(d / "cache"), str(d / "s.ffsrc"))
    return str(d / "s.ffsrc")


def _loader(shard, dev):
    return CA.DeviceBatchLoader(shard, 2, dev, augment=True, shuffle=True, seed=9)   # 3 batches per epoch


TOTAL = 14


@pytest.mark.timeout(1800)
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("graph", [False, True])
def test_default_mode_resume_is_bitwise_the_uninterrupted_run(tmp_path, shard, precision, graph):
    """Graph warm-up 2: a save after step 1 is mid-warm-up, after step 3 right after the capture (step 3 is the first
    replay), after step 7 five replays later; every k crosses or ends on an epoch boundary of 3 batches."""
    from isr_b200.trainer import load_checkpoint, save_checkpoint
    dev = _cuda()
    kw = dict(cuda_graph=graph, graph_warmup=2)
    ref_steps = []
    tr = _trainer(dev, 0, precision, **kw)
    _train(tr, _loader(shard, dev), TOTAL, ref_steps)
    assert tr._graph is not None or not graph
    assert all(torch.isfinite(s["loss"]) for s in ref_steps)
    ref = _final(tr)
    del tr
    for k in ((1, 3, 7) if graph else (4,)):
        path = str(tmp_path / f"ckpt{k}.pt")
        tr, loader, steps = _trainer(dev, 0, precision, **kw), _loader(shard, dev), []
        _train(tr, loader, k, steps)
        save_checkpoint(path, tr, loader, extra={"step": k})
        del tr, loader
        gc.collect()
        tr, loader = _trainer(dev, 1234, precision, **kw), _loader(shard, dev)    # nothing may leak from this seed
        assert load_checkpoint(path, tr, loader) == {"step": k}
        _train(tr, loader, TOTAL - k, steps)
        for s, (a, b) in enumerate(zip(ref_steps, steps)):
            _assert_equal_dicts(a, b, (k, "step", s))
        _assert_equal_dicts(ref, _final(tr), (k, "final"))
        assert len(tr.model.state_dict()) == 226
        del tr, loader
        gc.collect()


def _inputs(dev, B, S, seed):
    torch.manual_seed(seed)
    lr, imgs, fts, hr = O.synthetic_inputs(B, S, S)
    return (lr.to(dev), {k: v.to(dev) for k, v in imgs.items()}, {k: v.to(dev) for k, v in fts.items()}, hr.to(dev))


def _emulated(ranks, batches, first_step, out):
    """``ranks``: the trainer instances of a world-size-len(ranks) run, in rank order.  Per step: each rank's local pass
    on its slice, rows concatenated as all_gather_into_tensor would, the finish on every instance."""
    from isr_b200.training import seed_counter
    world = len(ranks)
    dev = ranks[0].optimizer.bucket.flat.device
    for s, (lr, imgs, fts, hr) in enumerate(batches, first_step):
        B = lr.shape[0] // world
        k = ranks[0].accumulation_steps
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
            rec = _step_record(*t._finish(gathered))
            if r == 0:
                out.append(rec)
    torch.cuda.synchronize()


def _emulated_ranks(dev, world, M, seed):
    """The instances of a world-size run.  Each sees a world of one in this process, so its resume configuration
    (what state_dict() records and load_state_dict() checks against) is that of a rank of the emulated run."""
    from isr_b200.trainer import FusionTrainer
    ranks = [_trainer(dev, seed, cuda_graph=False, accumulation_steps=M // world, world_invariant=True)
             for _ in range(world)]
    base = _trainer(dev, seed, cuda_graph=False, accumulation_steps=M, world_invariant=True)._seed_base
    for t in ranks:
        t._seed_base = base                                          # rank 0's base, as the broadcast hands it out
        t._resume_config = lambda t=t: dict(FusionTrainer._resume_config(t), world=world, micro_batches=M)
    return ranks


@pytest.mark.timeout(1800)
@pytest.mark.parametrize("M,save_world,resume_world", [(2, 2, 1), (4, 4, 2)])
def test_world_invariant_resume_on_fewer_ranks(M, save_world, resume_world):
    """Saved by emulated ranks at N after k steps, resumed at N' (emulated ranks, or one CUDA-graph trainer at N'=1):
    bitwise the uninterrupted run at N and at N'."""
    dev = _cuda()
    b, S, k = 2, 32, 2
    batches = [_inputs(dev, M * b, S, seed=s) for s in range(2 * k)]
    runs = {}
    for world in (save_world, resume_world):
        steps = []
        ranks = _emulated_ranks(dev, world, M, 0)
        _emulated(ranks, batches, 0, steps)
        runs[world] = (steps, _final(ranks[0]))
        del ranks
    _assert_equal_dicts(runs[save_world][1], runs[resume_world][1], "uninterrupted N vs N'")
    steps = []
    ranks = _emulated_ranks(dev, save_world, M, 0)
    _emulated(ranks, batches[:k], 0, steps)
    state = ranks[0].state_dict()
    del ranks
    gc.collect()
    if resume_world == 1:
        tr = _trainer(dev, 77, cuda_graph=True, graph_warmup=1, accumulation_steps=M, world_invariant=True)
        tr.load_state_dict(state)
        for args in batches[k:]:
            steps.append(_step_record(*tr.step(*args)))
        torch.cuda.synchronize()
        final = _final(tr)
    else:
        ranks = _emulated_ranks(dev, resume_world, M, 77)
        for t in ranks:
            t.load_state_dict(state)
        _emulated(ranks, batches[k:], k, steps)
        final = _final(ranks[0])
    for world in (save_world, resume_world):
        for s, (a, got) in enumerate(zip(runs[world][0], steps)):
            _assert_equal_dicts(a, got, (world, "step", s))
        _assert_equal_dicts(runs[world][1], final, (world, "final"))


def _nccl_worker(rank, world, port, path, q):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    from isr_b200.trainer import load_checkpoint, save_checkpoint
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    b, S, k = 2, 32, 2
    batches = [_inputs(dev, world * b, S, seed=s) for s in range(2 * k)]
    mine = [(lr[rank * b:(rank + 1) * b], {n: v[rank * b:(rank + 1) * b] for n, v in imgs.items()},
             {n: v[rank * b:(rank + 1) * b] for n, v in fts.items()}, hr[rank * b:(rank + 1) * b])
            for lr, imgs, fts, hr in batches]
    tr = _trainer(dev, 0, cuda_graph=True, graph_warmup=1, world_invariant=True)
    ref = []
    for s, args in enumerate(mine):
        ref.append(_step_record(*tr.step(*args)))
        if s == k - 1:
            save_checkpoint(path, tr, extra={"step": k})
    torch.cuda.synchronize()
    ref_final = _final(tr)
    dist.barrier()
    dist.destroy_process_group()
    res = None
    if rank == 0:                     # resume the N=2 run in this process alone: N'=1, two micro-batches per step
        del tr
        gc.collect()
        tr = _trainer(dev, 5, cuda_graph=True, graph_warmup=1, world_invariant=True, global_micro_batches=world)
        try:
            assert load_checkpoint(path, tr) == {"step": k}
            got = [_step_record(*tr.step(*args)) for args in batches[k:]]
            torch.cuda.synchronize()
            for s, (a, g) in enumerate(zip(ref[k:], got)):
                _assert_equal_dicts(a, g, ("step", k + s))
            _assert_equal_dicts(ref_final, _final(tr), "final")
            res = "ok"
        except AssertionError as e:
            res = str(e)
    q.put((rank, res))


@pytest.mark.timeout(1200)
def test_nccl_save_resumes_in_one_process(tmp_path):
    world = 2
    if not torch.cuda.is_available() or torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} CUDA devices (one process per GPU)")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_nccl_worker, args=(r, world, 29851, str(tmp_path / "ckpt.pt"), q))
             for r in range(world)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=1100) for _ in range(world))
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    assert res[0] == "ok", res[0]


def test_reference_adamw_checkpoint_still_loads(tmp_path):
    """torch.optim.AdamW's per-parameter state, through a file, into FusedAdamW: moments scattered into the flat
    buckets, the step count kept, the EMA shadow restarted from the weights."""
    from isr_b200.trainer import FusedAdamW
    dev = _cuda()
    torch.manual_seed(0)
    m = isr_b200.CompleteEnhancedFusionSR(None).to(dev)
    params = [p for p in m.parameters() if p.requires_grad]
    ref = torch.optim.AdamW(params, lr=1e-3, weight_decay=1e-4)
    g = torch.Generator(device=dev).manual_seed(3)
    for _ in range(2):
        for p in params:
            p.grad = torch.randn(p.shape, device=dev, generator=g)
        ref.step()
    torch.save(ref.state_dict(), tmp_path / "adamw.pt")
    opt = FusedAdamW(params, lr=2e-4, ema_decay=0.999)
    with torch.no_grad():
        opt.bucket.flat.add_(0.01)                                   # the shadow must follow the weights, not this
    opt.load_state_dict(torch.load(tmp_path / "adamw.pt", weights_only=True))
    assert opt.steps == 2 and opt.param_groups[0]["lr"] == 1e-3
    torch.cuda.synchronize()
    assert torch.equal(opt.ema, opt.bucket.flat)
    for i, p in enumerate(params):
        st, o = ref.state[p], opt.bucket.offsets[i]
        assert torch.equal(opt.exp_avg[o:o + p.numel()].view(p.shape), st["exp_avg"])
        assert torch.equal(opt.exp_avg_sq[o:o + p.numel()].view(p.shape), st["exp_avg_sq"])
