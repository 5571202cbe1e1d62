"""Data-parallel training step of the fusion network: flat parameter / gradient buckets, ONE
NCCL all-reduce per optimizer step, fused clip + AdamW + EMA kernel.

Mirrors the reference's cached training loop (``train.py:300-357``: forward_with_precomputed ->
clamp -> criterion -> backward -> clip_grad_norm_(1.0) -> AdamW.step -> EMA.update) with the
per-tensor ATen loops replaced by two kernels over a flat bucket (``csrc/optim.cu``) and, under
``torchrun``, one ``ncclAllReduce`` of the 1,433,217-float gradient bucket over NVLink/NVSwitch
(SURVEY §8e: the reference has no DDP).  ``FusionTrainer(accumulation_steps=k)`` runs k micro-batches per rank and
step, accumulating their gradients into the bucket as ``train.py:331-357`` does.  In this default mode an N-rank step
equals its own ``accumulation_steps=N`` run only up to rounding: the all-reduce's ring order depends on N, and the
ranks' BatchNorm running statistics are averaged EMAs.

``world_invariant=True`` makes the step bitwise independent of N for a fixed sequence of M = N*k micro-batches of b
patches: every micro-batch's gradient, BatchNorm records and loss terms go into a row of their own, ONE all-gather puts
all M rows on every rank in micro-batch order, and every rank sums them in that order (``ffsr_sum_slots_ordered``),
folds the BatchNorm records of all M micro-batches in one closed form and applies the optimizer with grad_scale 1/M.
Dropout seeds are a hash of (run base, global micro-batch, call).  With the same build, GPU model, precision mode,
``torch.manual_seed``, data and step sequence, losses, gradients, parameters, optimizer / EMA state and BatchNorm
buffers match bit for bit for every N dividing M (feed it from ``DeviceBatchLoader(world_invariant=True)``).  With one
micro-batch per step it is exactly the default step.

``FusedAdamW`` is a ``torch.optim.Optimizer`` so LR schedulers and ``optimizer.state_dict()`` keep
working in an unchanged ``train.py``; parameters stay ordinary leaf ``nn.Parameter``s whose storage
is re-pointed into the flat bucket.
"""
from __future__ import annotations

import ctypes as C
import os
import uuid
from typing import Dict, Iterable, List, Optional

import torch
import torch.distributed as dist

from . import _cabi as K


class FlatBucket:
    """Flattens tensors into one contiguous fp32 buffer and re-points them at views of it."""

    def __init__(self, tensors: List[torch.Tensor], align: int = 4):
        self.shapes = [tuple(t.shape) for t in tensors]
        self.offsets, off = [], 0
        for t in tensors:
            self.offsets.append(off)
            off += (t.numel() + align - 1) // align * align
        self.numel = off
        dev = tensors[0].device if tensors else torch.device("cpu")
        self.flat = torch.zeros(self.numel, device=dev, dtype=torch.float32)
        for t, o in zip(tensors, self.offsets):
            self.flat[o:o + t.numel()].view(t.shape).copy_(t.detach())

    def view(self, i: int) -> torch.Tensor:
        o, s = self.offsets[i], self.shapes[i]
        n = 1
        for d in s:
            n *= d
        return self.flat[o:o + n].view(s)

    def new_like(self) -> torch.Tensor:
        return torch.zeros_like(self.flat)


def _world():
    return dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1


def allreduce_mean_(flat: torch.Tensor) -> None:
    """In-place mean over ranks (sum + scale; gloo has no AVG)."""
    w = _world()
    if w > 1:
        dist.all_reduce(flat, op=dist.ReduceOp.SUM)
        flat.mul_(1.0 / w)


def sync_bn_buffers(model: torch.nn.Module) -> None:
    """Per-rank BatchNorm statistics (no SyncBN in the reference); the running buffers are
    mean-all-reduced so every rank checkpoints the same state (SURVEY §8e)."""
    if _world() == 1:
        return
    bufs = [b for n, b in model.named_buffers() if n.endswith("running_mean") or n.endswith("running_var")]
    if not bufs:
        return
    flat = torch.cat([b.reshape(-1) for b in bufs])
    allreduce_mean_(flat)
    o = 0
    for b in bufs:
        b.copy_(flat[o:o + b.numel()].view_as(b))
        o += b.numel()


class FusedAdamW(torch.optim.Optimizer):
    """AdamW over a flat bucket with optional fused global-norm clipping, data-parallel gradient
    all-reduce and EMA shadow update (one kernel pass: csrc/optim.cu).

    One documented difference from ``torch.optim.AdamW``: a parameter that received no gradient in a step has a
    zero gradient in the bucket (not ``None``), so it still gets weight decay and moment decay.  In the cached
    training loop every parameter receives a gradient every step (198/198, scripts/test_cached_training.py:212-218);
    the difference only shows when ``expert_feats`` is omitted and Phase 4 is skipped."""

    def __init__(self, params: Iterable[torch.nn.Parameter], lr: float = 2e-4, betas=(0.9, 0.999), eps: float = 1e-8,
                 weight_decay: float = 1e-4, max_grad_norm: float = 0.0, ema_decay: Optional[float] = None):
        params = [p for p in params if p.requires_grad]
        if not params:
            raise ValueError("FusedAdamW got no trainable parameters")
        if not all(p.is_cuda and p.dtype == torch.float32 for p in params):
            raise RuntimeError("FusedAdamW (sm_100a build) needs fp32 CUDA parameters: there is no CPU path")
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay))
        self.lib = K.load()
        self.max_grad_norm = float(max_grad_norm)
        self.ema_decay = ema_decay
        self._params = params
        self.bucket = FlatBucket(params)
        self.grads = self.bucket.new_like()
        self.exp_avg = self.bucket.new_like()
        self.exp_avg_sq = self.bucket.new_like()
        self.ema = self.bucket.flat.clone() if ema_decay is not None else None
        dev = self.bucket.flat.device
        self._gsq = torch.zeros(1, device=dev, dtype=torch.float64)
        self._gsq_ws = torch.empty(self.lib.ffsr_sumsq_workspace_bytes(self.bucket.numel), device=dev, dtype=torch.uint8)
        # step counter and learning rate live on the device so that a CUDA-graph replay sees fresh values
        self._step_dev = torch.zeros(1, device=dev, dtype=torch.int32)
        self._lr_dev = torch.full((1,), float(lr), device=dev, dtype=torch.float32)
        self._lr_host = float(lr)
        self.steps = 0
        # micro-batch gradients each rank sums into `grads` per step (FusionTrainer's accumulation_steps): step()
        # scales the all-reduced bucket by 1 / (world * micro_batches)
        self.micro_batches = 1
        self._grad_count = 1
        for i, p in enumerate(params):
            p.data = self.bucket.view(i)                       # same values, storage now inside the bucket
        self.attach_grads(self.grads)                          # autograd accumulates in place into the bucket
        self.sync_from_rank0()

    def attach_grads(self, flat: torch.Tensor) -> None:
        """Point every parameter's ``.grad`` at its slice of ``flat`` (a buffer laid out like the bucket)."""
        for i, p in enumerate(self._params):
            o = self.bucket.offsets[i]
            p.grad = flat[o:o + p.numel()].view(p.shape)

    @torch.no_grad()
    def sync_from_rank0(self) -> None:
        """Data-parallel replicas must start from (and resume with) ONE state: parameters, Adam moments, EMA shadow and
        step count are broadcast from rank 0 (what DistributedDataParallel does for parameters at construction).  Only
        gradients and BatchNorm statistics are reduced afterwards, so ranks that were seeded differently, or where only
        rank 0 loaded a checkpoint, would otherwise train diverging replicas silently.  No-op without a process group."""
        if _world() == 1:
            return
        for t in (self.bucket.flat, self.exp_avg, self.exp_avg_sq, self.ema):
            if t is not None:
                dist.broadcast(t, src=0)
        dist.broadcast(self._step_dev, src=0)
        self.steps = int(self._step_dev.item())
        self.bump_versions()

    @torch.no_grad()
    def reset_ema(self) -> None:
        """Re-initialise the EMA shadow from the current parameters (call after loading weights into the model once the
        optimizer exists: the shadow was taken from the construction-time weights)."""
        if self.ema is not None:
            self.ema.copy_(self.bucket.flat)

    # -- torch.optim API -------------------------------------------------------------------
    def zero_grad(self, set_to_none: bool = False):
        self.grads.zero_()
        for i, p in enumerate(self._params):                   # re-attach if a caller set .grad = None
            if p.grad is None or p.grad.data_ptr() != self.grads.data_ptr() + 4 * self.bucket.offsets[i]:
                o = self.bucket.offsets[i]
                p.grad = self.grads[o:o + p.numel()].view(p.shape)

    def _gather_stray_grads(self):
        for i, p in enumerate(self._params):
            o = self.bucket.offsets[i]
            if p.grad is not None and p.grad.data_ptr() != self.grads.data_ptr() + 4 * o:
                self.grads[o:o + p.numel()].view(p.shape).copy_(p.grad)

    @torch.no_grad()
    def step(self, closure=None):
        loss = closure() if closure is not None else None
        self._gather_stray_grads()
        world = _world()
        if world > 1:
            dist.all_reduce(self.grads, op=dist.ReduceOp.SUM)   # ONE collective: the flat 5.7 MB gradient bucket
        self.apply_summed(world * self.micro_batches)
        return loss

    @torch.no_grad()
    def apply_summed(self, count: int) -> None:
        """Clip + AdamW + EMA from ``grads`` holding the sum of ``count`` micro-batch gradients, each of its own mean
        loss: the update uses their mean (grad_scale = 1 / count).  No collective."""
        g = self.param_groups[0]
        self._grad_count = count
        dev = self.bucket.flat.device
        capturing = torch.cuda.is_current_stream_capturing()
        if not capturing:                    # a capture records the step without running it (the replay loop counts it)
            self.steps += 1
        if not capturing and float(g["lr"]) != self._lr_host:   # scheduler changed the LR: refresh the device scalar
            self._lr_host = float(g["lr"])
            self._lr_dev.fill_(self._lr_host)
        self._step_dev.add_(1)
        with torch.cuda.device(dev):
            S = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
            n = self.bucket.numel
            gsq = None
            if self.max_grad_norm > 0:
                self._gsq.zero_()
                K.check(self.lib.ffsr_sumsq(self.grads.data_ptr(), n, self._gsq.data_ptr(), self._gsq_ws.data_ptr(),
                                            self._gsq_ws.numel(), S), "sumsq")
                gsq = self._gsq.data_ptr()
            K.check(self.lib.ffsr_adamw_ema_step(
                self.bucket.flat.data_ptr(), self.grads.data_ptr(), self.exp_avg.data_ptr(), self.exp_avg_sq.data_ptr(),
                self.ema.data_ptr() if self.ema is not None else None, n, float(g["lr"]), float(g["betas"][0]),
                float(g["betas"][1]), float(g["eps"]), float(g["weight_decay"]), 0, self._step_dev.data_ptr(),
                self._lr_dev.data_ptr(), gsq, 1.0 / count, self.max_grad_norm, float(self.ema_decay or 0.0), S),
                "adamw_ema_step")
        self.bump_versions()      # the kernel wrote through raw pointers: tell the version-keyed weight caches (pipeline.py)

    # -- checkpointing (train.py saves optimizer.state_dict(): src/utils/checkpoint_manager.py:120-160) --------
    def state_dict(self):
        """param_groups as torch.optim does, plus the flat Adam moments, EMA shadow and step count."""
        sd = super().state_dict()
        sd["fused"] = {"exp_avg": self.exp_avg.detach().clone(), "exp_avg_sq": self.exp_avg_sq.detach().clone(),
                       "ema": self.ema.detach().clone() if self.ema is not None else None, "steps": int(self.steps),
                       "offsets": list(self.bucket.offsets), "numel": int(self.bucket.numel)}
        return sd

    def load_state_dict(self, state_dict):
        fused = state_dict.get("fused")
        rest = {k: v for k, v in state_dict.items() if k != "fused"}
        per_param = rest.get("state") or {}
        if fused is None and per_param:
            # a torch.optim.AdamW checkpoint as the reference writes it (src/utils/checkpoint_manager.py:120-160):
            # state[i] = {step, exp_avg, exp_avg_sq} per parameter index -> scatter into the flat buckets
            if len(per_param) != len(self._params):
                raise ValueError(f"FusedAdamW.load_state_dict: checkpoint has state for {len(per_param)} parameters, "
                                 f"this optimizer owns {len(self._params)}")
            steps = 0
            for i, p in enumerate(self._params):
                st = per_param.get(i, per_param.get(str(i)))
                if st is None or tuple(st["exp_avg"].shape) != tuple(p.shape):
                    raise ValueError(f"FusedAdamW.load_state_dict: no matching AdamW state for parameter {i}")
                o = self.bucket.offsets[i]
                self.exp_avg[o:o + p.numel()].view(p.shape).copy_(st["exp_avg"])
                self.exp_avg_sq[o:o + p.numel()].view(p.shape).copy_(st["exp_avg_sq"])
                steps = max(steps, int(st["step"]))
            rest = dict(rest)
            rest["state"] = {}
            super().load_state_dict(rest)
            self.steps = steps
            self._step_dev.fill_(steps)
            self.reset_ema()                 # a plain AdamW checkpoint carries no shadow: restart it from the weights
            self.set_lr(float(self.param_groups[0]["lr"]))
            self.sync_from_rank0()
            return
        super().load_state_dict(rest)
        if fused is not None:
            if fused["numel"] != self.bucket.numel or list(fused["offsets"]) != list(self.bucket.offsets):
                raise ValueError("FusedAdamW.load_state_dict: bucket layout differs from the checkpoint's")
            self.exp_avg.copy_(fused["exp_avg"])
            self.exp_avg_sq.copy_(fused["exp_avg_sq"])
            if self.ema is not None and fused.get("ema") is not None:
                self.ema.copy_(fused["ema"])
            elif self.ema is not None:
                self.reset_ema()             # checkpoint written with EMA disabled
            self.steps = int(fused["steps"])
            self._step_dev.fill_(self.steps)
        self.set_lr(float(self.param_groups[0]["lr"]))
        self.sync_from_rank0()

    # -- extras ----------------------------------------------------------------------------
    def set_lr(self, lr: float) -> None:
        """Scheduler hook usable between CUDA-graph replays (also picked up from param_groups[0]['lr'])."""
        self.param_groups[0]["lr"] = float(lr)
        self._lr_host = float(lr)
        self._lr_dev.fill_(float(lr))

    def bump_versions(self) -> None:
        for p in self._params:
            torch.autograd.graph.increment_version(p)

    def grad_norm(self) -> torch.Tensor:
        """Global gradient norm seen by the last step (device scalar, no sync)."""
        return self._gsq.sqrt() / self._grad_count

    @torch.no_grad()
    def swap_ema(self) -> None:
        """Exchange the parameters with their EMA shadow in place (call again to undo).  ``EMAModel.save`` + ``apply``
        + ``restore`` (checkpoint_manager.py:359-377, train.py:450-452, 515) clone every parameter twice and copy 198
        tensors three times; with flat buckets the swap is three copies of one 5.7 MB buffer and no allocation beyond
        the temporary."""
        if self.ema is None:
            raise RuntimeError("EMA is disabled (ema_decay=None)")
        tmp = self.bucket.flat.clone()
        self.bucket.flat.copy_(self.ema)
        self.ema.copy_(tmp)
        self.bump_versions()                                   # packed / bf16 weight caches are keyed on _version

    def ema_shadow(self, names: List[str]) -> Dict[str, torch.Tensor]:
        """EMAModel.shadow-compatible dict (checkpoint_manager.py:344-350): name -> view of the flat shadow."""
        if self.ema is None:
            raise RuntimeError("EMA is disabled (ema_decay=None)")
        out = {}
        for i, nme in enumerate(names):
            o, s = self.bucket.offsets[i], self.bucket.shapes[i]
            out[nme] = self.ema[o:o + self._params[i].numel()].view(s)
        return out


class FusionTrainer:
    """One data-parallel training step (BASELINE configs[1] / configs[3]).

    ``cuda_graph=True`` (default): after ``graph_warmup`` eager steps the whole step -- forward, fused losses,
    backward, gradient all-reduce, clip + AdamW + EMA, BatchNorm buffer sync -- is captured once into a CUDA
    graph and replayed from static input buffers: the ~2,000 kernel launches of a step cost one graph launch
    instead of ~80 us of Python / driver time each.  The values that change between steps (optimizer step
    count, learning rate, dropout seed) are device-side scalars.  A change of input shapes re-captures.

    Reproducibility: every reduction of the step runs in a fixed order (no floating-point atomics) and the dropout
    seeds come from torch's CPU generator plus a device counter that construction resets, so two trainers built
    after the same ``torch.manual_seed`` (before the model, and on the same GPU, precision mode and inputs) give
    bitwise-identical losses, gradients, parameters, optimizer / EMA state and BatchNorm buffers, eager or
    graph-replayed, with or without ``torch.use_deterministic_algorithms(True)``.

    ``accumulation_steps=k``: ``step()`` takes the rank's k*b patches and runs them as k contiguous micro-batches along
    dim 0; the returned loss and components are their mean.  ``world_invariant=True`` (module docstring): the same
    results for every world size N dividing M = N*k; ``global_micro_batches=M`` instead of k sets M directly and
    raises ``ValueError`` when N does not divide it.

    Resuming: ``state_dict()`` / ``load_state_dict()`` (and ``save_checkpoint`` / ``load_checkpoint`` with the
    loader's state) continue a run bit for bit -- in the default mode on the same world size, in world-invariant mode on
    any N dividing M.  Each capture records the host dropout seeds it freezes; a trainer loaded from a checkpoint
    taken after a capture runs its warm-up steps and its own capture on those seeds, so with the restored device
    counter they compute what the interrupted run's replays would."""

    def __init__(self, model, criterion, lr: float = 2e-4, betas=(0.9, 0.999), eps: float = 1e-8,
                 weight_decay: float = 1e-4, max_grad_norm: float = 1.0, ema_decay: Optional[float] = 0.999,
                 cuda_graph: bool = True, graph_warmup: int = 3, accumulation_steps: int = 1,
                 world_invariant: bool = False, global_micro_batches: Optional[int] = None):
        from .training import _draw_seed, seed_counter
        world = _world()
        if global_micro_batches is not None:
            if not world_invariant:
                raise ValueError("global_micro_batches needs world_invariant=True")
            if accumulation_steps != 1:
                raise ValueError("give accumulation_steps (per rank) or global_micro_batches, not both")
            if global_micro_batches < 1 or global_micro_batches % world:
                raise ValueError(f"global_micro_batches={global_micro_batches} is not a positive multiple of the "
                                 f"world size {world}")
            accumulation_steps = global_micro_batches // world
        if accumulation_steps < 1:
            raise ValueError(f"accumulation_steps must be >= 1, got {accumulation_steps}")
        self.model, self.criterion = model, criterion
        self.names = [n for n, p in model.named_parameters() if p.requires_grad]
        self.optimizer = FusedAdamW(model.parameters(), lr, betas, eps, weight_decay, max_grad_norm, ema_decay)
        dev = self.optimizer.bucket.flat.device
        seed_counter(dev).zero_()                                   # dropout masks start over with each trainer
        if world > 1:                         # BatchNorm statistics / counters start from rank 0's too (parameters: FusedAdamW)
            for n, b in model.named_buffers():
                if n.endswith(("running_mean", "running_var", "num_batches_tracked")):
                    dist.broadcast(b, src=0)
        self.accumulation_steps = int(accumulation_steps)
        self.world_invariant = bool(world_invariant)
        self.optimizer.micro_batches = 1 if self.world_invariant else self.accumulation_steps
        # world-invariant mode: dropout seeds hash (base, global micro-batch, call) with ONE base per run, rank 0's.
        # A step of one micro-batch keeps the default per-call draws, so it is exactly the default step.
        self._seed_base = None
        if self.world_invariant and world * self.accumulation_steps > 1:
            base = torch.tensor([_draw_seed()], dtype=torch.int64, device=dev)
            if world > 1:
                dist.broadcast(base, src=0)
            self._seed_base = int(base.item())
        self._layout = None
        self._rows = self._rows_all = None
        self.optimizer.zero_grad()
        self.cuda_graph = cuda_graph
        self.graph_warmup = graph_warmup
        self._eager_steps = 0
        self._graph = None
        self._static = None
        self._sig = None
        # host dropout seeds of the current capture, in call order (recorded by it, or loaded with a checkpoint taken
        # after one): a step that uses them plus the device counter gives the bits of that capture's replay
        self._capture_seeds: Optional[List[int]] = None

    def _split(self, lr_img, expert_imgs, expert_feats, hr_img):
        """The rank's batch as accumulation_steps contiguous micro-batches along dim 0."""
        k = self.accumulation_steps
        if k == 1:
            return [(lr_img, expert_imgs, expert_feats, hr_img)]
        B = lr_img.shape[0]
        if B % k:
            raise ValueError(f"a batch of {B} patches does not split into accumulation_steps={k} micro-batches")
        b = B // k

        def cut(j):
            return (lr_img[j * b:(j + 1) * b], {n: v[j * b:(j + 1) * b] for n, v in expert_imgs.items()},
                    {n: v[j * b:(j + 1) * b] for n, v in expert_feats.items()} if expert_feats else expert_feats,
                    hr_img[j * b:(j + 1) * b])
        return [cut(j) for j in range(k)]

    def _step_body(self, lr_img, expert_imgs, expert_feats, hr_img):
        from .training import seed_counter
        micro = self._split(lr_img, expert_imgs, expert_feats, hr_img)
        if self.world_invariant:
            world = _world()
            rows = self._local_rows(micro, (dist.get_rank() if world > 1 else 0) * len(micro))
            if world > 1:                     # ONE collective; rank order is global micro-batch order; moves bits only
                if self._rows_all is None or self._rows_all.shape[0] != world * rows.shape[0]:
                    self._rows_all = rows.new_empty((world * rows.shape[0], rows.shape[1]))
                dist.all_gather_into_tensor(self._rows_all, rows)
                rows = self._rows_all
            return self._finish(rows)
        out = []
        for lr_j, imgs_j, feats_j, hr_j in micro:      # train.py:331-357: backward per micro-batch into one bucket
            sr = self.model.forward_with_precomputed(lr_j, imgs_j, feats_j).clamp(0, 1)   # train.py:326
            loss, comps = self.criterion(sr, hr_j, return_components=True)
            loss.backward()
            out.append((loss, comps))
        self.optimizer.step()
        sync_bn_buffers(self.model)
        self.optimizer.zero_grad()
        seed_counter(lr_img.device).add_(1)
        if len(out) == 1:
            loss, comps = out[0]
            return loss.detach(), {k: v.detach() for k, v in comps.items()}
        k = len(out)
        return (sum(l.detach() for l, _ in out) / k,
                {n: sum(c[n].detach() for _, c in out) / k for n in out[0][1]})

    # ---- world-invariant step: local pass -> all-gather -> finish ---------------------------------------------
    def _local_rows(self, micro_batches, first_index: int) -> torch.Tensor:
        """Forward + backward of the rank's micro-batches, which are global micro-batches first_index, first_index+1,
        ...  Row j of the returned [k, L] buffer holds micro-batch j's gradient bucket (of its own mean loss,
        unscaled), then its BatchNorm records (per BN call, in call order: mean[G,C], biased var[G,C]), then its
        loss and loss components.  Nothing is reduced here."""
        from .training import micro_batch
        opt = self.optimizer
        rows = None
        for j, (lr_j, imgs_j, feats_j, hr_j) in enumerate(micro_batches):
            with micro_batch(first_index + j, self._seed_base) as mb:
                sr = self.model.forward_with_precomputed(lr_j, imgs_j, feats_j).clamp(0, 1)   # train.py:326
            loss, comps = self.criterion(sr, hr_j, return_components=True)
            if j == 0:
                rows = self._row_buffer(mb.records, comps, len(micro_batches))
            lay = self._layout
            if [(id(r[0]),) + tuple(r[1].shape) + (r[3],) for r in mb.records] != lay["key"] or list(comps) != lay["comps"]:
                raise RuntimeError("world-invariant step: micro-batches of one step differ in their BatchNorm calls or "
                                   "loss components")
            row = rows[j]
            parts = [t.reshape(-1) for r in mb.records for t in (r[1], r[2])]
            parts += [loss.detach().float().reshape(1)] + [comps[n].detach().float().reshape(1) for n in lay["comps"]]
            torch.cat(parts, out=row[lay["nb"]:lay["end"]])
            opt.attach_grads(row)             # backward accumulates into the zeroed row j
            loss.backward()
        return rows

    def _row_buffer(self, records, comps, k: int) -> torch.Tensor:
        """The zeroed [k, L] row buffer; its layout follows the BN calls and loss components of the first micro-batch."""
        key = [(id(r[0]),) + tuple(r[1].shape) + (r[3],) for r in records]
        if self._layout is None or self._layout["key"] != key or self._layout["comps"] != list(comps) \
                or self._rows.shape[0] != k:
            nb = self.optimizer.bucket.numel
            bn, off = [], nb
            for bnm, mean, _var, n in records:
                G, Cc = mean.shape
                bn.append((bnm, G, Cc, n, off))
                off += 2 * G * Cc
            loss_off = off
            end = loss_off + 1 + len(comps)
            L = (end + 63) // 64 * 64                 # rows start on 256-byte boundaries: 16-byte loads in the sum
            self._layout = {"key": key, "comps": list(comps), "nb": nb, "bn": bn, "loss_off": loss_off, "end": end}
            dev = self.optimizer.grads.device
            self._rows = torch.zeros((k, L), device=dev, dtype=torch.float32)
            self._loss_sum = torch.zeros(1 + len(comps), device=dev, dtype=torch.float32)
            return self._rows
        return self._rows.zero_()

    def _finish(self, rows: torch.Tensor):
        """The step from the gathered rows [M, L] of all M global micro-batches, identical on every rank: gradient
        bucket and loss terms summed in micro-batch order (ffsr_sum_slots_ordered), the BatchNorm records of all M
        micro-batches folded in one closed form, then clip + AdamW + EMA with grad_scale = 1 / M."""
        from .training import fold_running_stats, seed_counter
        opt, lay = self.optimizer, self._layout
        M, L = rows.shape
        ncomp = lay["end"] - lay["loss_off"]
        with torch.cuda.device(rows.device):
            S = C.c_void_p(torch.cuda.current_stream(rows.device).cuda_stream)
            K.check(opt.lib.ffsr_sum_slots_ordered(rows.data_ptr(), M, lay["nb"], L, opt.grads.data_ptr(), S),
                    "sum_slots_ordered")
            K.check(opt.lib.ffsr_sum_slots_ordered(rows.data_ptr() + 4 * lay["loss_off"], M, ncomp, L,
                                                   self._loss_sum.data_ptr(), S), "sum_slots_ordered")
        vals = self._loss_sum / M
        fold_running_stats([(bn, rows[i, o:o + G * Cc].view(G, Cc), rows[i, o + G * Cc:o + 2 * G * Cc].view(G, Cc), n)
                            for i in range(M) for bn, G, Cc, n, o in lay["bn"]])
        opt.attach_grads(opt.grads)
        opt.apply_summed(M)
        seed_counter(rows.device).add_(1)
        return vals[0], {n: vals[1 + i] for i, n in enumerate(lay["comps"])}

    def _signature(self, lr_img, expert_imgs, expert_feats, hr_img):
        """Everything a capture bakes in: input shapes / dtypes, and the host scalars and Python control flow of the step --
        the loss weights and component set (the curriculum calls ``criterion.set_weights`` every epoch, train.py:296), the
        optimizer hyper-parameters passed by value, the precision mode.  A change re-warms and re-captures."""
        f = expert_feats or {}
        crit, g = self.criterion, self.optimizer.param_groups[0]
        cw = tuple(sorted((k, float(v)) for k, v in getattr(crit, "weights", {}).items()))
        return (tuple(lr_img.shape), lr_img.dtype, tuple(sorted((k, tuple(v.shape), v.dtype) for k, v in expert_imgs.items())),
                tuple(sorted((k, tuple(v.shape), v.dtype) for k, v in f.items())), tuple(hr_img.shape),
                cw, bool(getattr(crit, "use_swt", True)), bool(getattr(crit, "use_fft", True)),
                float(g["weight_decay"]), tuple(float(b) for b in g["betas"]), float(g["eps"]),
                float(self.optimizer.max_grad_norm), self.optimizer.ema_decay, getattr(self.model, "precision", None),
                self.accumulation_steps)

    def _capture(self, lr_img, expert_imgs, expert_feats, hr_img):
        from .training import seed_tape
        self._static = (lr_img.clone(), {k: v.clone() for k, v in expert_imgs.items()},
                        {k: v.clone() for k, v in expert_feats.items()} if expert_feats else None, hr_img.clone())
        self._graph = torch.cuda.CUDAGraph()
        torch.cuda.synchronize()
        with seed_tape(self._capture_seeds) as tape:          # records the seeds it freezes (replays loaded ones)
            with torch.cuda.graph(self._graph):
                self._out = self._step_body(*self._static)
        self._capture_seeds = tape.seeds
        self._sig = self._signature(lr_img, expert_imgs, expert_feats, hr_img)

    def _eager_step(self, lr_img, expert_imgs, expert_feats, hr_img):
        """An executed step outside a graph.  After loading a checkpoint taken after a capture it takes that capture's
        seeds instead of drawing: with the restored counter it computes what the interrupted run's replay would."""
        import contextlib
        from .training import seed_tape
        with seed_tape(self._capture_seeds) if self._capture_seeds is not None else contextlib.nullcontext():
            return self._step_body(lr_img, expert_imgs, expert_feats, hr_img)

    def step(self, lr_img, expert_imgs, expert_feats, hr_img):
        """forward -> clamp -> loss -> backward -> all-reduce -> clip + AdamW + EMA.  Returns the
        (device) loss and its components; nothing here synchronises the host."""
        self.model.train()
        opt = self.optimizer
        if not self.cuda_graph:
            if self._capture_seeds is not None and self._signature(lr_img, expert_imgs, expert_feats, hr_img) != self._sig:
                self._capture_seeds = None
            return self._eager_step(lr_img, expert_imgs, expert_feats, hr_img)
        sig = self._signature(lr_img, expert_imgs, expert_feats, hr_img)
        if self._capture_seeds is not None and sig != self._sig:      # new shapes: warm up and re-capture
            self._graph, self._static, self._eager_steps, self._capture_seeds = None, None, 0, None
        if self._graph is None:
            if self._eager_steps < self.graph_warmup:
                self._eager_steps += 1
                return self._eager_step(lr_img, expert_imgs, expert_feats, hr_img)
            self._capture(lr_img, expert_imgs, expert_feats, hr_img)     # capture does not execute the step
        lr_now = float(opt.param_groups[0]["lr"])
        if lr_now != opt._lr_host:
            opt.set_lr(lr_now)
        s_lr, s_imgs, s_feats, s_hr = self._static
        s_lr.copy_(lr_img, non_blocking=True)
        for k, v in expert_imgs.items():
            s_imgs[k].copy_(v, non_blocking=True)
        if s_feats:
            for k, v in expert_feats.items():
                s_feats[k].copy_(v, non_blocking=True)
        s_hr.copy_(hr_img, non_blocking=True)
        self._graph.replay()
        opt.steps += 1
        opt.bump_versions()
        return self._out

    # ---- checkpointing ----------------------------------------------------------------------------
    def _resume_config(self) -> dict:
        o = self.optimizer
        return {"bucket": (int(o.bucket.numel), [int(x) for x in o.bucket.offsets]),
                "precision": getattr(self.model, "precision", None), "world_invariant": self.world_invariant,
                "accumulation_steps": self.accumulation_steps, "world": _world(),
                "micro_batches": _world() * self.accumulation_steps}

    def state_dict(self) -> dict:
        """Everything the next steps depend on: the model's parameters and buffers (BatchNorm statistics and
        ``num_batches_tracked``), ``optimizer.state_dict()``, the dropout state (device counter, world-invariant seed
        base, the seeds of the current capture, torch's CPU generator), the eager-step count and capture signature,
        the criterion's weights and the configuration a resume is checked against."""
        from .training import seed_counter
        crit = self.criterion
        captured = self._capture_seeds is not None
        return {"model": {k: v.detach().clone() for k, v in self.model.state_dict().items()},
                "optimizer": self.optimizer.state_dict(),
                "seed_counter": int(seed_counter(self.optimizer.bucket.flat.device).item()),
                "seed_base": self._seed_base,
                "eager_steps": int(self._eager_steps),
                "capture_seeds": list(self._capture_seeds) if captured else None,
                "signature": self._sig if captured else None,
                "cpu_rng": torch.get_rng_state(),
                "criterion": {"weights": dict(getattr(crit, "weights", {})), "use_swt": getattr(crit, "use_swt", None),
                              "use_fft": getattr(crit, "use_fft", None)},
                "config": self._resume_config()}

    @torch.no_grad()
    def load_state_dict(self, state: dict, at_epoch_boundary: bool = False) -> None:
        """Continue the run ``state`` was taken from: the next steps give the bits the uninterrupted run's would (same
        build, GPU model, inputs and step sequence).  Drops any captured graph; a checkpoint taken after a capture
        warms up and re-captures on that capture's seeds, one taken during warm-up finishes the remaining warm-up steps
        from the restored CPU generator.  Restores torch's CPU generator state.  With a process group every rank ends
        with rank 0's state.  Raises ``ValueError`` naming the field when this trainer cannot continue it
        (``check_resume``); ``at_epoch_boundary`` allows a default-mode resume on another world size (not bitwise)."""
        from .training import seed_counter
        check_resume(state["config"], self._resume_config(), at_epoch_boundary)
        world = _world()
        self.model.load_state_dict(state["model"])
        if world > 1:
            for n, b in self.model.named_buffers():
                if n.endswith(("running_mean", "running_var", "num_batches_tracked")):
                    dist.broadcast(b, src=0)
        self.optimizer.load_state_dict(state["optimizer"])          # moments, EMA, step, LR; sync_from_rank0
        self.optimizer.bump_versions()                               # the packed-weight caches are version-keyed
        self.optimizer.zero_grad()
        dev = self.optimizer.bucket.flat.device
        counter = seed_counter(dev)
        counter.fill_(int(state["seed_counter"]))
        base = state["seed_base"]
        if world > 1:
            dist.broadcast(counter, src=0)
            if base is not None:
                b = torch.tensor([base], dtype=torch.int64, device=dev)
                dist.broadcast(b, src=0)
                base = int(b.item())
        self._seed_base = base
        self._graph, self._static, self._out = None, None, None
        if state["capture_seeds"] is not None:
            self._capture_seeds, self._sig, self._eager_steps = list(state["capture_seeds"]), state["signature"], 0
        else:
            self._capture_seeds, self._sig, self._eager_steps = None, None, int(state["eager_steps"])
        crit = state["criterion"]
        if hasattr(self.criterion, "set_weights"):
            self.criterion.set_weights(crit["weights"])
        for k in ("use_swt", "use_fft"):
            if crit[k] is not None:
                setattr(self.criterion, k, crit[k])
        torch.set_rng_state(state["cpu_rng"])

    # ---- validation -----------------------------------------------------------------------------
    def ema_weights(self):
        """``with trainer.ema_weights():`` -- the model runs on its EMA weights inside the block."""
        import contextlib

        @contextlib.contextmanager
        def cm():
            self.optimizer.swap_ema()
            try:
                yield self.model
            finally:
                self.optimizer.swap_ema()
        return cm()

    def validate(self, val_loader, crop_border: int = 4, test_y_channel: bool = True, use_ema: bool = True) -> Dict[str, float]:
        """``validate_epoch`` of the reference's cached mode (train.py:415-515) on this trainer's model."""
        return validate_epoch(self.model, val_loader, self.model.residual_scale.device, crop_border, test_y_channel,
                              self.optimizer if (use_ema and self.optimizer.ema is not None) else None)


def check_resume(saved: dict, now: dict, at_epoch_boundary: bool = False) -> None:
    """Raise ``ValueError`` naming the field when a trainer configured as ``now`` cannot continue a checkpoint whose
    configuration is ``saved`` (both ``FusionTrainer._resume_config()``): another bucket layout or precision mode; in
    world-invariant mode a world size N that does not divide the checkpoint's M micro-batches per step, or a trainer
    whose N * accumulation_steps is not M; in the default mode another accumulation_steps, or another world size
    unless the checkpoint was taken at an epoch boundary (the default step's bits depend on N)."""
    if saved["bucket"] != now["bucket"]:
        raise ValueError("trainer checkpoint: the parameter bucket layout differs from this model's")
    if saved["precision"] != now["precision"]:
        raise ValueError(f"trainer checkpoint: precision is {saved['precision']!r} in the checkpoint, "
                         f"{now['precision']!r} here")
    if saved["world_invariant"] != now["world_invariant"]:
        raise ValueError(f"trainer checkpoint: world_invariant is {saved['world_invariant']} in the checkpoint, "
                         f"{now['world_invariant']} here")
    if now["world_invariant"]:
        M = saved["micro_batches"]
        if M % now["world"]:
            raise ValueError(f"trainer checkpoint: world size {now['world']} does not divide the checkpoint's "
                             f"micro_batches M={M}")
        if now["micro_batches"] != M:
            raise ValueError(f"trainer checkpoint: micro_batches is M={M} in the checkpoint, {now['micro_batches']} "
                             f"here: use accumulation_steps={M // now['world']} (or global_micro_batches={M})")
        return
    if saved["accumulation_steps"] != now["accumulation_steps"]:
        raise ValueError(f"trainer checkpoint: accumulation_steps is {saved['accumulation_steps']} in the checkpoint, "
                         f"{now['accumulation_steps']} here")
    if saved["world"] != now["world"] and not at_epoch_boundary:
        raise ValueError(f"trainer checkpoint: world size is {saved['world']} in the checkpoint, {now['world']} here; "
                         "the default mode changes it only at an epoch boundary (use world_invariant=True to resume "
                         "mid-epoch on another GPU count)")


def atomic_save(obj, path: str) -> None:
    """``torch.save`` to a temporary file beside ``path``, flushed to disk, then renamed over it: a reader sees the old
    file or the complete new one, and an interrupted write leaves neither a partial file nor the temporary."""
    path = os.fspath(path)
    tmp = f"{path}.{os.getpid()}.{uuid.uuid4().hex}.tmp"
    try:
        with open(tmp, "xb") as f:
            torch.save(obj, f)
            f.flush()
            os.fsync(f.fileno())
        os.replace(tmp, path)
    except BaseException:
        if os.path.exists(tmp):
            os.unlink(tmp)
        raise


def save_checkpoint(path: str, trainer: FusionTrainer, loader=None, extra=None) -> None:
    """Write ``trainer.state_dict()``, the loader's state (every rank's, for the default mode's per-rank augmentation
    generators) and ``extra`` (caller state such as an LR scheduler's ``state_dict()`` or the epoch: plain containers,
    numbers, strings and tensors) to ``path``.  Under a process group every rank calls it and rank 0 writes the file
    (``atomic_save``).  Take it between steps, after the step's loader batch was consumed."""
    world = _world()
    state = {"trainer": trainer.state_dict(), "loader": None, "extra": extra}
    if loader is not None:
        mine = loader.state_dict()
        if world > 1:
            states = [None] * world
            dist.all_gather_object(states, mine)
        else:
            states = [mine]
        state["loader"] = states
    if world == 1 or dist.get_rank() == 0:
        atomic_save(state, path)
    if world > 1:
        dist.barrier()


def load_checkpoint(path: str, trainer: FusionTrainer, loader=None):
    """Load a ``save_checkpoint`` file into ``trainer`` (and ``loader``) on every rank and return its ``extra``.  The
    default mode may change the world size only when the loader state is at an epoch boundary; a file written
    without a loader counts as mid-epoch."""
    ck = torch.load(path, map_location="cpu", weights_only=True)
    states = ck["loader"]
    if loader is not None and states is None:
        raise ValueError(f"checkpoint {path} holds no loader state")
    trainer.load_state_dict(ck["trainer"], at_epoch_boundary=states is not None and all(s["batch"] == 0 for s in states))
    if loader is not None:
        rank = dist.get_rank() if _world() > 1 else 0
        loader.load_state_dict(states[rank] if rank < len(states) else states[0])
    return ck["extra"]


@torch.no_grad()
def validate_epoch(model, val_loader, device, crop_border: int = 4, test_y_channel: bool = True,
                   ema: Optional[FusedAdamW] = None) -> Dict[str, float]:
    """Cached-mode ``validate_epoch`` (train.py:415-515): eval mode, EMA weights if given, full-image
    ``forward_with_precomputed`` per batch, clamp, Y-channel PSNR / SSIM with border crop -- with the metrics kept on
    the device (ONE host sync per epoch instead of two per image) and the EMA exchange done on the flat bucket.
    ``val_loader`` yields the reference's batch dict (host tensors from a DataLoader, fp16 allowed) or device batches
    (``cache.DeviceBatchLoader``).  The model's train / eval mode is restored on exit."""
    from .metrics import MetricCalculator
    was_training = model.training
    model.eval()
    if ema is not None:
        ema.swap_ema()
    calc = MetricCalculator(crop_border, test_y_channel)
    try:
        for batch in val_loader:
            lr_img = batch["lr"].to(device, non_blocking=True).float()
            hr_img = batch["hr"].to(device, non_blocking=True).float()
            imgs = {k: v.to(device, non_blocking=True).float() for k, v in batch["expert_imgs"].items()}
            feats = None
            if batch.get("expert_feats") is not None:
                feats = {k: v.to(device, non_blocking=True).float() for k, v in batch["expert_feats"].items()}
            sr = model.forward_with_precomputed(lr_img, imgs, feats).clamp(0, 1)
            calc.update(sr, hr_img)
    finally:
        if ema is not None:
            ema.swap_ema()
        model.train(was_training)
    return calc.get_metrics()
