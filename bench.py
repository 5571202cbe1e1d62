#!/usr/bin/env python
"""Headline benchmark: fusion forward throughput in HR MPix/s (BASELINE.json metric).

Workload (config.workload = "C3"): BASELINE.json configs[2] -- full-res DIV2K-shape inference,
510x339 LR -> 2040x1356 HR fusion forward over synthetic cached expert outputs + features,
random-init weights.  One "step" = one image per GPU (images are independent units: weak
scaling, no data-path collective -- SURVEY §8e).  configs[1] (training step) needs the backward
kernels, which are not built yet; configs[0] is the CPU-runnable parity case.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--precision fp32|bf16] [--dump-outputs DIR]

* value : whole-job HR MPix/s with the inputs resident in HBM (CUDA events, barrier + sync on both
          sides, max over ranks).  The 553 MB of inputs per step exceed the 126 MB L2.
* e2e   : same metric through forward_with_precomputed with pinned HOST buffers: every step
          copies the inputs host->device and the SR image device->host inside the timed region.
* roofline : the dominant kernel (3x3 128->128 refinement conv), algorithmic FLOPs per launch /
          mean CUDA-event duration of those launches inside the timed region, against the
          measured bf16 tensor peak of MEASURED_PEAKS.json.
* cpu_baseline : the oracle (CPU port of the reference forward) on the host cores, rank 0, N=1.
* --impl reference : the reference's CPU implementation of the path = the oracle port (the
          reference is pure Python and does not travel to the GPU box), all host threads.
* --dump-outputs DIR : after the timed steps of the C3 job, DIR/sr_sample.npy (float32, one row per image of this rank's
          last timed step; sr_sample_rank<r>.npy per rank with several GPUs) holds a fixed, seeded sample of the SR images
          that step returned (dump_sample_index).  Inputs and weights are seeded, so two builds run with the same
          arguments can be compared output for output.  The gathers that take the sample run inside the last timed step:
          the line then carries a `dump_outputs` note, and timings are taken from runs without the option.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

LR_H, LR_W = 339, 510                       # config 3
FLOP_PER_HR_PIXEL = 1_774_222                # SURVEY §8d, whole forward
HOT_LAYER_FLOP_PER_HR_PIXEL = 2 * 9 * 128 * 128   # one 3x3 128->128 conv


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1371.0), d.get("hbm_gbs", 6555.2), "measured (MEASURED_PEAKS.json, sustained)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """SM clock / throttle reasons sampled DURING the timed region (NVML every 10 ms; nvidia-smi
    fallback if NVML is unavailable)."""

    _REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self._stop_evt = index, threading.Event()
        self.sm, self.reasons, self.sm_max = [], set(), None
        self._nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
            self._nvml = pynvml
        except Exception:
            self._nvml = None

    def _sample_nvml(self):
        n = self._nvml
        self.sm.append(float(n.nvmlDeviceGetClockInfo(self._h, n.NVML_CLOCK_SM)))
        try:
            mask = n.nvmlDeviceGetCurrentClocksEventReasons(self._h)
        except Exception:
            mask = n.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
        for bit, name in self._REASONS.items():
            if mask & bit:
                self.reasons.add(name)

    def _sample_smi(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=5).stdout.strip()
        c = [x.strip() for x in out.split(",")]
        if len(c) >= 6:
            self.sm.append(float(c[0]))
            self.sm_max = float(c[1])
            for i, name in enumerate(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]):
                if c[2 + i].lower().startswith("active"):
                    self.reasons.add(name)

    def run(self):
        while not self._stop_evt.is_set():
            try:
                self._sample_nvml() if self._nvml else self._sample_smi()
            except Exception:
                pass
            self._stop_evt.wait(0.01 if self._nvml else 0.2)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=6)
        return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": self.sm_max,
                "reasons": sorted(self.reasons), "samples": len(self.sm),
                "source": "nvml" if self._nvml else "nvidia-smi"}


def cpu_oracle_throughput(H, W, steps, warmup, threads):
    """HR MPix/s of the CPU oracle (port of the reference forward) on a LR HxW image."""
    import torch
    import isr_b200
    from oracle import fusion_oracle as O
    torch.set_num_threads(threads)
    torch.manual_seed(0)
    m = isr_b200.CompleteEnhancedFusionSR(None).eval()
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    lr, imgs, fts, _ = O.synthetic_inputs(1, H, W)
    times = []
    with torch.no_grad():
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            O.run_pipeline(sd, lr, imgs, fts)
            if i >= warmup:
                times.append(time.perf_counter() - t0)
    t = sum(times) / len(times)
    return 16 * H * W / t / 1e6, t


def gpu_eager_throughput(model, dev, H, W, steps=5, warmup=2):
    """BASELINE.md §3 item 2, "the real bar": the same algorithm in PyTorch eager (cuDNN / cuBLAS / cuFFT / ATen) on the
    SAME B200.  The reference tree does not travel to the GPU box, so this times the oracle's restatement of the module
    (plain torch ops, pinned to the reference on CPU) with its tensors on the device: fp32 and under bf16 autocast."""
    import torch
    from oracle import fusion_oracle as O
    sd = {k: v.detach().to(dev) for k, v in model.state_dict().items()}
    lr, imgs, fts, _ = O.synthetic_inputs(1, H, W, seed=1234)
    lr, imgs, fts = lr.to(dev), {k: v.to(dev) for k, v in imgs.items()}, {k: v.to(dev) for k, v in fts.items()}
    out = {}
    for name, ctx in (("fp32", None), ("bf16_autocast", torch.autocast("cuda", dtype=torch.bfloat16))):
        def fwd():
            with torch.no_grad():
                if ctx is None:
                    return O.run_pipeline(sd, lr, imgs, fts)
                with ctx:
                    return O.run_pipeline(sd, lr, imgs, fts)
        for _ in range(warmup):
            fwd()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fwd()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        out[name] = {"value": 16 * H * W / 1e6 / (ms * 1e-3), "unit": "HR MPix/s", "ms_per_image": ms}
    out["kind"] = "port: oracle restatement in PyTorch eager on the same GPU (cudnn.allow_tf32=%s, matmul.allow_tf32=%s)" % (
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    out["steps"] = steps
    return out


def cpu_oracle_train_throughput(hw, batch, steps, warmup, threads, weights):
    """patches/s of one CPU training step of the oracle port (forward + losses + autograd backward + AdamW)."""
    import torch
    import isr_b200
    from oracle import fusion_oracle as O
    from oracle import loss_oracle as LO
    torch.set_num_threads(threads)
    torch.manual_seed(0)
    m = isr_b200.CompleteEnhancedFusionSR(None)
    pn = dict(m.named_parameters())
    sd = {k: (v.detach().clone().requires_grad_() if k in pn else v.detach().clone()) for k, v in m.state_dict().items()}
    opt = torch.optim.AdamW([sd[k] for k in pn], lr=2e-4, betas=(0.9, 0.999), weight_decay=1e-4)
    lr, imgs, fts, hr = O.synthetic_inputs(batch, hw, hw)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        opt.zero_grad()
        sr = O.run_pipeline(sd, lr, imgs, fts, training=True, bn_updates={}).clamp(0, 1)
        loss, _ = LO.combined_loss(sr, hr, weights)
        loss.backward()
        torch.nn.utils.clip_grad_norm_([sd[k] for k in pn], 1.0)
        opt.step()
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    t = sum(times) / len(times)
    return batch / t, t


def gpu_eager_train_throughput(dev, hw, batch, weights, steps=4, warmup=2):
    """The training step as plain PyTorch eager on the SAME GPU (autograd over the oracle's restatement, torch losses,
    clip_grad_norm_, torch.optim.AdamW, EMA as a foreach lerp): fp32 and with the forward under bf16 autocast."""
    import torch
    import isr_b200
    from oracle import fusion_oracle as O
    from oracle import loss_oracle as LO
    out = {}
    lr, imgs, fts, hr = O.synthetic_inputs(batch, hw, hw)
    lr, hr = lr.to(dev), hr.to(dev)
    imgs, fts = {k: v.to(dev) for k, v in imgs.items()}, {k: v.to(dev) for k, v in fts.items()}
    for name, auto in (("fp32", False), ("bf16_autocast", True)):
        torch.manual_seed(0)
        m = isr_b200.CompleteEnhancedFusionSR(None)
        pn = dict(m.named_parameters())
        sd = {k: (v.detach().to(dev).requires_grad_() if k in pn else v.detach().to(dev)) for k, v in m.state_dict().items()}
        params = [sd[k] for k in pn]
        ema = [p.detach().clone() for p in params]
        opt = torch.optim.AdamW(params, lr=2e-4, betas=(0.9, 0.999), weight_decay=1e-4)

        def step():
            opt.zero_grad(set_to_none=True)
            with torch.autocast("cuda", dtype=torch.bfloat16, enabled=auto):
                sr = O.run_pipeline(sd, lr, imgs, fts, training=True, bn_updates={})
            loss, _ = LO.combined_loss(sr.float().clamp(0, 1), hr, weights)
            loss.backward()
            torch.nn.utils.clip_grad_norm_(params, 1.0)
            opt.step()
            with torch.no_grad():
                torch._foreach_lerp_(ema, params, 1.0 - 0.999)
        for _ in range(warmup):
            step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        out[name] = {"value": batch / (ms * 1e-3), "unit": "patches/s", "ms_per_step": ms}
        del sd, params, ema, opt
        torch.cuda.empty_cache()
    out["kind"] = "port: oracle restatement + torch autograd / AdamW in PyTorch eager on the same GPU"
    out["steps"] = steps
    return out


def run_reference_train(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    hw = 64 if args.workload == "c2" else 96
    batch = 2                                                   # bounded sample of the global batch
    v, t = cpu_oracle_train_throughput(hw, batch, args.steps, args.warmup, threads, STAGE_WEIGHTS[args.workload])
    line = {
        "impl": "reference", "metric": "fusion_train_patches_per_s", "value": v, "unit": "patches/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": train_config(args.workload, batch, batch, hw, "fp32"),
        "cpu_baseline": {"value": v, "unit": "patches/s", "cores": threads, "kind": "port",
                         "sample": f"each step = forward + losses + autograd backward + clip + AdamW of the oracle port on "
                                   f"{batch} patches of {hw}x{hw} LR (the metric is linear in patches)"},
        "e2e": {"value": v, "unit": "patches/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


HOT_LAYER_DRAM_BYTES = 710.2e6 + 662.0e6       # per launch, bf16 path, from the ncu capture named in traffic_source
TRAIN_FLOP_PER_HR_PIXEL = 5_921_000          # SURVEY 8(d): forward + backward (parameter gradients)
STAGE_WEIGHTS = {"c2": {"l1": 1.0}, "c4": {"l1": 0.60, "swt": 0.25, "fft": 0.10, "ssim": 0.05}}


def measure_train(args, workload, dev, world, rank, local, steps, warmup, e2e=True):
    """Device-timed data-parallel training steps of one workload; returns the result dict (rank 0 view)."""
    import torch
    import torch.distributed as dist
    import isr_b200
    from isr_b200.losses import CombinedLoss
    from isr_b200.trainer import FusionTrainer
    from isr_b200.dist import max_over_ranks as _mor
    from oracle import fusion_oracle as O

    gb, hw = (32, 64) if workload == "c2" else (64, 96)
    if args.batch:
        gb = args.batch
    B = max(gb // world, 1)
    torch.manual_seed(0)
    m = isr_b200.CompleteEnhancedFusionSR(None).to(dev)
    m.precision = args.precision
    crit = CombinedLoss()
    crit.set_weights({"charbonnier": 0, "l2": 0, "vgg": 0, "edge": 0, "clip": 0, "swt": 0, "fft": 0, "ssim": 0,
                      **STAGE_WEIGHTS[workload]})
    tr = FusionTrainer(m, crit, lr=2e-4, betas=(0.9, 0.999), weight_decay=1e-4, max_grad_norm=1.0, ema_decay=0.999)
    lr, imgs, fts, hr = O.synthetic_inputs(B, hw, hw, seed=1234 + rank)
    host = [lr.pin_memory(), {k: v.pin_memory() for k, v in imgs.items()}, {k: v.pin_memory() for k, v in fts.items()},
            hr.pin_memory()]
    devs = [lr.to(dev), {k: v.to(dev) for k, v in imgs.items()}, {k: v.to(dev) for k, v in fts.items()}, hr.to(dev)]
    h2d = 4 * (lr.numel() + hr.numel() + sum(v.numel() for v in imgs.values()) + sum(v.numel() for v in fts.values()))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(warmup, 4)):                      # 3 eager steps + the CUDA-graph capture + 1 replay
        tr.step(*devs)
    sampler = ClockSampler(local)
    sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss, _ = tr.step(*devs)
    e1.record()
    barrier()
    ms = _mor(e0.elapsed_time(e1), dev)
    clocks = sampler.stop()
    res = {"patches": B * world, "B": B, "hw": hw, "ms": ms / steps, "clocks": clocks, "h2d": h2d, "trainer": tr,
           "launches": None}
    if e2e:
        def e2e_step():
            d = [host[0].to(dev, non_blocking=True), {k: v.to(dev, non_blocking=True) for k, v in host[1].items()},
                 {k: v.to(dev, non_blocking=True) for k, v in host[2].items()}, host[3].to(dev, non_blocking=True)]
            l, _ = tr.step(*d)
            return float(l)                                     # device -> host read of the step's loss

        e2e_step()
        barrier()
        t0 = time.perf_counter()
        e0.record()
        for _ in range(steps):
            last = e2e_step()
        e1.record()
        barrier()
        res["ms_e2e"] = _mor(max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3), dev) / steps
        res["last_loss"] = last

        # The same loop fed by the repo's loader: flat fp16 cache shard -> pinned staging -> ONE H2D copy + ONE unpack
        # kernel per batch on a side stream (augmentation included), prefetched while the previous step trains.
        import tempfile
        from isr_b200.cache import DeviceBatchLoader, ShardWriter
        with tempfile.TemporaryDirectory() as tmp:
            shard = os.path.join(tmp, f"train_r{rank}.ffsrc")
            with ShardWriter(shard, dtype="fp16") as w:
                for rep in range(2):
                    for i in range(B):
                        w.add(f"p{rep}_{i:03d}", lr[i], hr[i], {k: v[i] for k, v in imgs.items()}, {k: v[i] for k, v in fts.items()})
            loader = DeviceBatchLoader(shard, B, dev, augment=True, shuffle=True, repeat_factor=steps + 4, seed=rank)
            rec_bytes = loader.cache.layout(0)[1]
            it = iter(loader)

            def loader_step():
                b = next(it)
                l, _ = tr.step(b["lr"], b["expert_imgs"], b["expert_feats"], b["hr"])
                return float(l)

            loader_step()
            barrier()
            t0 = time.perf_counter()
            e0.record()
            for _ in range(steps):
                last = loader_step()
            e1.record()
            barrier()
            res["ms_e2e_loader"] = _mor(max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3), dev) / steps
            res["h2d_loader"] = B * rec_bytes
            res["last_loss_loader"] = last
            it.close()
            del it, loader
    return res


def _leave(world, trainer=None):
    """The captured CUDA graph holds NCCL kernels; tearing the communicator down underneath it can hang at exit
    (seen at N=2).  Drop the graph, drain the device, then leave without the NCCL destructor."""
    import torch
    import torch.distributed as dist
    if world > 1:
        if trainer is not None:
            trainer._graph = None
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def run_train(args):
    """BASELINE configs[1] (c2: batch 32 x 64x64 LR, L1 + AdamW) / configs[3] (c4: batch 64 x 96x96 LR,
    stage-3 fused losses): one data-parallel training step = forward + loss + backward + gradient
    all-reduce + clip/AdamW/EMA.  Global batch fixed (strong scaling): each rank takes batch/world."""
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the fusion path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    warmup = max(args.warmup, 4)
    r = measure_train(args, args.workload, dev, world, rank, local, args.steps, warmup)
    if rank == 0:
        tensor_peak, hbm_peak, peak_src = _peaks()
        patches, hw, ms = r["patches"], r["hw"], r["ms"]
        tfl = TRAIN_FLOP_PER_HR_PIXEL * patches * 16 * hw * hw / (ms * 1e-3) / 1e12
        line = {
            "metric": "fusion_train_patches_per_s", "value": patches / (ms * 1e-3), "unit": "patches/s",
            "n_gpus": world, "steps": args.steps, "warmup": warmup, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32" if args.precision == "fp32" else "bf16", "data": "synthetic",
            "config": train_config(args.workload, patches, r["B"], hw, args.precision),
            "e2e": {"value": patches / (r["ms_e2e"] * 1e-3), "unit": "patches/s", "h2d_bytes_per_step": r["h2d"],
                    "d2h_bytes_per_step": 4, "ms_per_step": r["ms_e2e"], "last_loss": r["last_loss"]},
            "e2e_loader": {"value": patches / (r["ms_e2e_loader"] * 1e-3), "unit": "patches/s",
                           "h2d_bytes_per_step": r["h2d_loader"], "d2h_bytes_per_step": 4, "ms_per_step": r["ms_e2e_loader"],
                           "last_loss": r["last_loss_loader"],
                           "note": "fed by isr_b200.cache.DeviceBatchLoader from an fp16 flat shard (augmentation on): one "
                                   "H2D copy + one unpack kernel per batch on a side stream, prefetched during the step"},
            "gpu_launches": "one CUDA-graph replay per step (~2,000 captured kernel launches)",
            "clocks": r["clocks"],
            "roofline": {"bound": "tensor", "achieved": tfl / world, "achieved_all_gpus": tfl, "peak": tensor_peak, "unit": "TFLOP/s",
                         "frac": tfl / world / tensor_peak, "traffic": None,
                         "kernel": "whole training step (fwd+bwd), algorithmic FLOPs; per-kernel figures: "
                                   "profiles/r01_conv_train_microbench.txt, profiles/r01_wgrad_tc_128x128_ncu_full.txt",
                         "peak_source": peak_src},
        }
        if world == 1 and not args.no_gpu_eager:
            try:
                import gc
                import torch
                tr_ = r.pop("trainer")
                tr_._graph = None
                del tr_
                gc.collect()
                torch.cuda.empty_cache()
                eb = min(r["B"], 32 if hw <= 64 else 16)       # autograd keeps every fp32 activation: bound the footprint
                line["gpu_eager_baseline"] = gpu_eager_train_throughput(dev, hw, eb, STAGE_WEIGHTS[args.workload])
                line["gpu_eager_baseline"]["batch"] = eb
            except Exception as exc:
                line["gpu_eager_baseline"] = {"error": repr(exc)[:300]}
        if world == 1 and not args.no_cpu_baseline:
            threads = os.cpu_count() or 1
            v, t = cpu_oracle_train_throughput(hw, 2, 2, 1, threads, STAGE_WEIGHTS[args.workload])
            line["cpu_baseline"] = {"value": v, "unit": "patches/s", "cores": threads, "kind": "port",
                                    "sample": f"2 training steps (forward + losses + autograd backward + clip + AdamW) of the "
                                              f"fp32 oracle port on 2 patches of {hw}x{hw} LR, {t:.1f} s per step on {threads} threads"}
        print(json.dumps(line), flush=True)
    _leave(world, r.get("trainer"))


def run_tiled(args):
    """`--workload c3t`: ONE C3 image across all ranks (SURVEY §8e row 2) -- halo tiles, bands of the whole image on every
    rank, cores assembled by one NCCL all-reduce.  Strong scaling: value = the image's HR pixels / max-over-ranks time."""
    import torch
    import torch.distributed as dist
    import isr_b200
    from isr_b200.serving import fuse_tiled, tile_grid, TILE_HALO_LR
    from isr_b200.dist import max_over_ranks
    from oracle import fusion_oracle as O

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the fusion path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    warmup = max(args.warmup, 3)
    H, W = args.lr
    grid = {1: (1, 1), 2: (1, 2), 4: (2, 2), 8: (2, 4)}.get(world, (1, world))
    torch.manual_seed(0)
    m = isr_b200.CompleteEnhancedFusionSR(None).eval().to(dev)
    m.precision = args.precision
    lr, imgs, fts, _ = O.synthetic_inputs(1, H, W, seed=1234)            # the SAME image on every rank (replicated inputs)
    lrd, imd, ftd = lr.to(dev), {k: v.to(dev) for k, v in imgs.items()}, {k: v.to(dev) for k, v in fts.items()}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(warmup):
        sr = fuse_tiled(m, lrd, imd, ftd, grid=grid, rank=rank, world=world)
    sampler = ClockSampler(local)
    sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        sr = fuse_tiled(m, lrd, imd, ftd, grid=grid, rank=rank, world=world)
    e1.record()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1), dev)
    clocks = sampler.stop()
    launches_tile = m._engine.launches
    whole = m.forward_with_precomputed(lrd, imd, ftd)
    err = float((whole - sr).abs().max())
    if rank == 0:
        tiles = tile_grid(H, W, *grid)
        y0, y1, x0, x1 = tiles[0]
        hal = TILE_HALO_LR
        win = (min(H, y1 + hal) - max(0, y0 - hal)) * (min(W, x1 + hal) - max(0, x0 - hal))
        print(json.dumps({
            "metric": "fusion_forward_hr_mpix_per_s", "value": 16 * H * W / 1e6 * args.steps / (ms * 1e-3), "unit": "HR MPix/s",
            "n_gpus": world, "steps": args.steps, "warmup": warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32" if args.precision == "fp32" else "bf16", "data": "synthetic",
            "config": {"workload": "C3 fusion forward, ONE 2040x1356 image split over all ranks (latency mode)",
                       "lr": [H, W], "grid": list(grid), "halo_lr_px": hal, "window_over_core": win * len(tiles) / (H * W),
                       "partition": "halo tiles; phase-2 bands recomputed on the whole LR image by every rank; cores "
                                    "assembled by one all-reduce(sum) of the fp32 output" if world > 1 else "single tile",
                       "precision": args.precision},
            "max_abs_vs_whole_image": err, "gpu_launches": (launches_tile + 7) * args.steps, "clocks": clocks}), flush=True)
    if world > 1:
        _leave(world)


def run_drct(args):
    """`--workload n1`: the DRCT-L expert forward (SURVEY §8f N1) on one C3-sized LR image padded to the window
    (352x512), fp32 first version, against the same algorithm as PyTorch eager ops on the same GPU (the oracle's
    restatement).  Not a headline line: N=1 only, reports HR MPix/s of the x4 output and algorithmic TFLOP/s."""
    import torch
    from isr_b200 import drct as D
    from oracle import drct_oracle as DO
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device")
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        if int(os.environ.get("RANK", "0")) == 0:
            print(json.dumps({"workload": "n1", "unavailable": "single-GPU measurement only"}), flush=True)
        return
    dev = torch.device("cuda", 0)
    H, W = (352, 512) if tuple(args.lr) == (LR_H, LR_W) else tuple(args.lr)
    torch.manual_seed(0)
    m = D.create_drct_model().to(dev).eval()
    x = torch.rand(1, 3, H, W, generator=torch.Generator().manual_seed(1234)).to(dev)
    warmup, steps = max(args.warmup, 3), args.steps

    def timed(fn):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps

    res = {}
    sampler = ClockSampler(0)
    sampler.start()
    for prec in ("fp32", "bf16"):
        m.precision = prec
        with torch.no_grad():
            res[prec] = timed(lambda: m(x))
    clocks = sampler.stop()
    sd = {k: v.detach() for k, v in m.state_dict().items()}
    with torch.no_grad():
        ms_eager = timed(lambda: DO.forward(sd, x))
        with torch.autocast("cuda", dtype=torch.bfloat16):
            ms_eager16 = timed(lambda: DO.forward(sd, x))
        ref = DO.forward(sd, x)
        errs = {}
        for prec in ("fp32", "bf16"):
            m.precision = prec
            errs[prec] = float((m(x) - ref).abs().max())
    m.precision = args.precision
    ms = res[args.precision]
    flop = D.flops_per_lr_pixel(m) * H * W
    tensor_peak, hbm_peak, peak_src = _peaks()
    print(json.dumps({
        "metric": "drct_forward_hr_mpix_per_s", "value": 16 * H * W / 1e6 / (ms * 1e-3), "unit": "HR MPix/s", "n_gpus": 1,
        "steps": steps, "warmup": warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32" if args.precision == "fp32" else "bf16", "data": "synthetic",
        "config": {"workload": "N1 DRCT-L x4 expert forward (12 RDG x 5 Swin blocks, window 16, dims 180..308), one LR image "
                               "padded to the 16-px window, random-init weights", "lr": [H, W], "precision": args.precision},
        "modes": {p_: {"ms": res[p_], "hr_mpix_per_s": 16 * H * W / 1e6 / (res[p_] * 1e-3), "tflops_algorithmic": flop / (res[p_] * 1e-3) / 1e12,
                       "max_abs_vs_fp32_eager": errs[p_]} for p_ in res},
        "roofline": {"bound": "tensor", "achieved": flop / (ms * 1e-3) / 1e12, "peak": tensor_peak, "unit": "TFLOP/s",
                     "frac": flop / (ms * 1e-3) / 1e12 / tensor_peak, "traffic": None, "peak_source": peak_src,
                     "kernel": "whole DRCT-L forward, algorithmic FLOPs (70.3 MFLOP per LR pixel)"},
        "gpu_eager_baseline": {"fp32": {"value": 16 * H * W / 1e6 / (ms_eager * 1e-3), "ms_per_image": ms_eager},
                               "bf16_autocast": {"value": 16 * H * W / 1e6 / (ms_eager16 * 1e-3), "ms_per_image": ms_eager16},
                               "unit": "HR MPix/s", "kind": "port: oracle restatement in PyTorch eager on the same GPU"},
        "clocks": clocks}), flush=True)


def run_c5(args):
    """`--workload c5` = BASELINE configs[4]: end-to-end x4 SR of one 2040x1356 image per rank per step with the DRCT-L expert
    forward (180-dim, window 16) feeding the fusion, x8 self-ensemble TTA.  Per image: the 8 dihedral variants of the LR image
    (scripts/extract_test_tta_cache.py:253-256) are padded to the 16-px window (reflect), DRCT-L produces the SR image and the
    180-channel feature of each (io.py:226-235), the other three experts' outputs come from the cache (synthetic here), the fusion
    runs on the variants batched by shape (serving.fuse_tta), outputs are un-transformed and averaged on the device
    (scripts/generate_fast_submission.py:190-250).  Images are independent: rank r takes images r, r+N, ... (weak scaling)."""
    import torch
    import torch.distributed as dist
    import torch.nn.functional as F
    import isr_b200
    from isr_b200 import drct as D
    from isr_b200.serving import fuse_tta
    from isr_b200.dist import max_over_ranks as _mor

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    H, W = args.lr
    warmup, steps = max(args.warmup, 3), args.steps
    torch.manual_seed(0)
    fusion = isr_b200.CompleteEnhancedFusionSR(None).eval().to(dev)
    fusion.precision = args.precision
    drct = D.create_drct_model().to(dev).eval()
    drct.precision = args.precision
    g = torch.Generator(device=dev).manual_seed(4321 + rank)
    lr0 = torch.rand(1, 3, H, W, device=dev, generator=g)
    others = {}                                   # cached outputs / features of the experts that are not built (per variant shape)

    def cached(shape_key, h, w):
        if shape_key not in others:
            gg = torch.Generator(device=dev).manual_seed(99 + len(others))
            others[shape_key] = ({k: torch.rand(1, 3, 4 * h, 4 * w, device=dev, generator=gg) for k in ("grl", "nafnet", "mamba")},
                                 {k: torch.randn(1, 64 if k == "nafnet" else 180, h, w, device=dev, generator=gg) for k in ("grl", "nafnet", "mamba")})
        return others[shape_key]

    def one_image():
        variants = []
        for hflip in (False, True):
            for rot in range(4):
                x = torch.flip(lr0, [3]) if hflip else lr0
                x = torch.rot90(x, rot, [2, 3]) if rot else x
                h, w = x.shape[2:]
                ph, pw = (16 - h % 16) % 16, (16 - w % 16) % 16
                xp = F.pad(x, (0, pw, 0, ph), mode="reflect") if (ph or pw) else x
                sr_d = drct(xp)[:, :, :4 * h, :4 * w].float().clamp(0, 1)
                feat_d = drct.last_feature[:, :, :h, :w].float()
                imgs_o, feats_o = cached((h, w), h, w)
                variants.append((x, {"drct": sr_d, **imgs_o}, {"drct": feat_d, **feats_o}, hflip, rot))
        return fuse_tta(fusion, variants)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.no_grad():
        for _ in range(warmup):
            out = one_image()
        sampler = ClockSampler(local)
        sampler.start()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            out = one_image()
        e1.record()
        barrier()
        ms = _mor(e0.elapsed_time(e1), dev) / steps
        clocks = sampler.stop()
        # split of one image: expert vs fusion
        torch.cuda.synchronize()
        e0.record()
        xp = F.pad(lr0, (0, (16 - W % 16) % 16, 0, (16 - H % 16) % 16), mode="reflect")
        for _ in range(3):
            drct(xp)
        e1.record()
        torch.cuda.synchronize()
        ms_drct = e0.elapsed_time(e1) / 3
    if rank == 0:
        tensor_peak, hbm_peak, peak_src = _peaks()
        flop = (D.flops_per_lr_pixel(drct) * xp.shape[2] * xp.shape[3] + FLOP_PER_HR_PIXEL * 16 * H * W) * 8
        print(json.dumps({
            "metric": "end_to_end_sr_hr_mpix_per_s", "value": world * 16 * H * W / 1e6 / (ms * 1e-3), "unit": "HR MPix/s", "n_gpus": world,
            "steps": steps, "warmup": warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32" if args.precision == "fp32" else "bf16", "data": "synthetic",
            "config": {"workload": "C5 (BASELINE configs[4]): end-to-end x4 SR, DRCT-L expert forward (180-dim, window 16) feeding the fusion, "
                                   "x8 self-ensemble TTA, one 2040x1356 HR image per GPU per step; the GRL / NAFNet / MambaIR expert outputs "
                                   "come from the cache (synthetic)", "lr": [H, W], "hr": [4 * H, 4 * W], "tta_variants": 8,
                       "precision": args.precision, "partition": "independent images round-robin over ranks, no collective"},
            "ms_per_image": ms, "ms_drct_forward_one_variant": ms_drct, "drct_share_of_image": 8 * ms_drct / ms,
            "roofline": {"bound": "tensor", "achieved": flop / (ms * 1e-3) / 1e12, "peak": tensor_peak, "unit": "TFLOP/s",
                         "frac": flop / (ms * 1e-3) / 1e12 / tensor_peak, "traffic": None, "peak_source": peak_src,
                         "kernel": "whole image: 8 x (DRCT-L forward + fusion forward), algorithmic FLOPs"},
            "output_range": [float(out.min()), float(out.max())], "clocks": clocks}), flush=True)
    if world > 1:
        _leave(world)


def train_config(workload, patches, B, hw, precision):
    return {"workload": f"{workload.upper()} fusion training step (BASELINE configs[{1 if workload == 'c2' else 3}]): "
                        f"global batch {patches} x {hw}x{hw} LR patches, losses {STAGE_WEIGHTS[workload]}, "
                        "clip 1.0 + AdamW + EMA, random-init weights",
            "global_batch": patches, "batch_per_gpu": B, "lr_patch": [hw, hw], "precision": precision,
            "partition": "data-parallel patches, one NCCL all-reduce of the flat 1.43M-float gradient bucket",
            "l2": "per-step activations (GBs) exceed the 126 MB L2; no explicit flush"}


N_JOB_IMAGES = 100                            # BASELINE configs[2]: "100 images tiled across 1/2/4/8 B200"
N_INPUT_SETS = 4                              # distinct synthetic images cycled through (4 x 553 MB > the 126 MB L2)
DUMP_BUDGET_BYTES = 48 << 20                  # --dump-outputs: the float32 samples of all ranks together


def dump_sample_index(rows, numel, world=1):
    """Indices into the flattened SR images (rows x k, each row sorted) that --dump-outputs keeps: every element while
    rows x numel x world floats fit DUMP_BUDGET_BYTES, else k seeded random elements per image.  Each row draws its own
    elements, so the images of one input set (the job cycles N_INPUT_SETS inputs) together cover more of that output."""
    import torch
    if rows == 0:                                 # a rank the job schedule gives no image
        return torch.empty(0, 0, dtype=torch.long)
    k = DUMP_BUDGET_BYTES // (4 * rows * world)
    if k >= numel:
        return torch.arange(numel).repeat(rows, 1)
    g = torch.Generator().manual_seed(0)
    return torch.randint(0, numel, (rows, k), generator=g).sort(dim=1).values


def c3_config(H, W):
    """The config both arms (ours / --impl reference) name: BASELINE configs[2]."""
    return {"workload": "C3 fusion forward job (BASELINE configs[2]): %d images of 510x339 LR -> 2040x1356 HR, cached 4-expert "
                        "outputs + features, random-init weights, eval" % N_JOB_IMAGES,
            "lr": [H, W], "hr": [4 * H, 4 * W], "images_per_job": N_JOB_IMAGES,
            "partition": "whole images items[rank::world] (scripts/extract_test_tta_cache.py:196), no collective; the n % world "
                         "left-over images split into halo tiles over rank groups (serving.fuse_tiled, one all-reduce per group)",
            "l2": "%d distinct input sets of 553 MB cycled: every forward reads inputs that are not in the 126 MB L2" % N_INPUT_SETS}


def load_reference_class():
    """The reference's own CompleteEnhancedFusionSR from the git-ignored baseline/_ref copy (tools/install_reference.py), or
    None where that copy does not exist."""
    ref = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref, "src", "models")):
        return None
    try:
        if ref not in sys.path:
            sys.path.insert(1, ref)
        import contextlib
        import io
        with contextlib.redirect_stdout(io.StringIO()):       # "diffusers not available" banner
            from src.models.enhanced_fusion_v2 import CompleteEnhancedFusionSR as RefModel
        return RefModel
    except Exception:
        return None


def device_inputs(H, W, dev, set_idx):
    """Synthetic cached inputs of one image generated ON the device (same values on every rank for the same set)."""
    import torch
    g = torch.Generator(device=dev).manual_seed(1234 + set_idx)
    names = ("drct", "grl", "nafnet", "mamba")
    lr = torch.rand(1, 3, H, W, device=dev, generator=g)
    imgs = {k: torch.rand(1, 3, 4 * H, 4 * W, device=dev, generator=g) for k in names}
    fts = {k: torch.randn(1, 64 if k == "nafnet" else 180, H, W, device=dev, generator=g) for k in names}
    return lr, imgs, fts


def parity_at_headline_size(model, dev, H, W, threads):
    """One full-size forward of the CPU oracle (the cpu_baseline sample) compared with this library on the same inputs:
    fp32 max-abs, bf16 dPSNR, flips of the two derived expert-selection indices over all LR pixels."""
    import math
    import torch
    import torch.nn.functional as F
    from oracle import fusion_oracle as O
    torch.set_num_threads(threads)
    sd = {k: v.detach().cpu().clone() for k, v in model.state_dict().items()}
    lr, imgs, fts, _ = O.synthetic_inputs(1, H, W)
    g = torch.Generator().manual_seed(77)
    up = F.interpolate(lr, scale_factor=4, mode="bicubic", align_corners=False)
    imgs = {k: (up + 0.02 * torch.randn(up.shape, generator=g)).clamp(0, 1) for k in O.EXPERT_ORDER}
    hr = (up + 0.01 * torch.randn(up.shape, generator=g)).clamp(0, 1)
    t0 = time.perf_counter()
    with torch.no_grad():
        ref, rint = O.run_pipeline(sd, lr, imgs, fts, return_intermediates=True)
    t_cpu = time.perf_counter() - t0
    top1, active = O.derived_indices(sd, rint["routing_lr"], rint["gates"])

    def psnr(a, b):
        return -10.0 * math.log10(max(float(((a - b) ** 2).mean()), 1e-20))

    lrd, imd, ftd = lr.to(dev), {k: v.to(dev) for k, v in imgs.items()}, {k: v.to(dev) for k, v in fts.items()}
    out = {"lr": [H, W], "lr_pixels": H * W}
    prev = model.precision
    try:
        for prec in ("fp32", "bf16"):
            model.precision = prec
            sr, ints = model._run_pipeline(lrd, [imd[k] for k in O.EXPERT_ORDER], ftd, 4 * H, 4 * W, {}, True)
            sr = sr.cpu()
            out[prec] = {"max_abs": float((sr - ref).abs().max()), "dpsnr_db": abs(psnr(sr, hr) - psnr(ref, hr)),
                         "psnr_vs_oracle_db": psnr(sr, ref),
                         "top1_flips": int((ints["gates"].cpu().argmax(1) != top1).sum()),
                         "active_flips": int((ints["active"].cpu() != active).sum())}
    finally:
        model.precision = prev
    out["tolerance"] = {"fp32_max_abs": 1e-4, "bf16_dpsnr_db": 0.01, "index_flips": 0}
    return out, 16 * H * W / t_cpu / 1e6, t_cpu


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on the box's host cores, on OUR config.  Each
    step is a bounded sample of the job: one full-size image (1/100 of a step's images; the metric is linear in images)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.workload not in ("c3",):
        return run_reference_train(args)
    import torch
    from oracle import fusion_oracle as O
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    H, W = args.lr
    RefModel = load_reference_class()
    torch.manual_seed(0)
    lr, imgs, fts, _ = O.synthetic_inputs(1, H, W)
    if RefModel is not None:
        import contextlib
        import io
        with contextlib.redirect_stdout(io.StringIO()):
            m = RefModel(None).eval()
        kind = "reference"
        fwd = lambda: m.forward_with_precomputed(lr, imgs, fts)
    else:
        import isr_b200
        mm = isr_b200.CompleteEnhancedFusionSR(None).eval()
        sd = {k: v.clone() for k, v in mm.state_dict().items()}
        kind = "port"
        fwd = lambda: O.run_pipeline(sd, lr, imgs, fts)
    budget_s = 330.0                                            # the whole arm stays within "a few minutes"
    times = []
    with torch.no_grad():
        t0 = time.perf_counter()
        fwd()                                                   # first warm-up step, also the estimate for the budget
        t_first = time.perf_counter() - t0
        n_all = max(1, int(budget_s / t_first) - 1)
        warm_more = max(0, min(args.warmup - 1, n_all // 5))
        for _ in range(warm_more):
            fwd()
        steps = max(1, min(args.steps, n_all - warm_more))
        for _ in range(steps):
            t0 = time.perf_counter()
            fwd()
            times.append(time.perf_counter() - t0)
    t = sum(times) / len(times)
    v = 16 * H * W / t / 1e6
    line = {
        "impl": "reference", "metric": "fusion_forward_hr_mpix_per_s", "value": v, "unit": "HR MPix/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": 1 + warm_more, "ms_per_step": t * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": c3_config(H, W),
        "cpu_baseline": {"value": v, "unit": "HR MPix/s", "cores": threads, "kind": kind,
                         "sample": f"each timed step = ONE full-size image ({16 * H * W / 1e6:.3f} HR MPix, 1/{N_JOB_IMAGES} of the "
                                   f"job; the metric is linear in images) through "
                                   + ("the unmodified reference module (baseline/_ref) forward_with_precomputed"
                                      if kind == "reference" else "the oracle port of the reference forward")
                                   + f", {t:.1f} s per image on {threads} threads ({steps} of {args.steps} requested steps and "
                                     f"{1 + warm_more} of {args.warmup} warm-up steps fit the {budget_s:.0f} s budget of this arm)"},
        "e2e": {"value": v, "unit": "HR MPix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def gpu_reference_eager_throughput(dev, H, W, steps=3, warmup=1):
    """BASELINE.md §3 item 2, "the real bar", with the reference MODULE itself: the unmodified CompleteEnhancedFusionSR of
    baseline/_ref in PyTorch eager on the same GPU (fp32, and under bf16 autocast)."""
    import contextlib
    import io
    import torch
    RefModel = load_reference_class()
    if RefModel is None:
        return None
    torch.manual_seed(0)
    with contextlib.redirect_stdout(io.StringIO()):
        m = RefModel(None).eval().to(dev)
    lr, imgs, fts = device_inputs(H, W, dev, 0)
    out = {}
    for name, auto in (("fp32", False), ("bf16_autocast", True)):
        def fwd():
            with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16, enabled=auto):
                return m.forward_with_precomputed(lr, imgs, fts)
        for _ in range(warmup):
            fwd()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fwd()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        out[name] = {"value": 16 * H * W / 1e6 / (ms * 1e-3), "unit": "HR MPix/s", "ms_per_image": ms}
    out["kind"] = "reference: unmodified reference module (baseline/_ref) in PyTorch eager on the same GPU"
    out["steps"] = steps
    del m
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="c3", choices=["c3", "c2", "c4", "c3t", "n1", "c5"],
                    help="c3: the 100-image full-res inference job (headline, default); c2 / c4: training steps (BASELINE "
                         "configs[1] / [3]); c3t: one image across all ranks; n1: DRCT-L expert forward; c5: configs[4], DRCT-L -> fusion, x8 TTA")
    ap.add_argument("--batch", type=int, default=0, help="override the global batch of a training workload")
    ap.add_argument("--images", type=int, default=N_JOB_IMAGES, help="images per job step (debug runs only)")
    ap.add_argument("--in-flight", type=int, default=2, help="C3 job: images in flight per GPU (serving.ConcurrentFusion; 1 = one stream)")
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default=os.environ.get("FFSR_PRECISION", "bf16"), choices=["fp32", "bf16"])
    ap.add_argument("--lr", type=int, nargs=2, default=[LR_H, LR_W], help="LR size (parity/debug runs only)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-eager", action="store_true", help="skip the PyTorch-eager-on-the-same-GPU baseline of the C3 line")
    ap.add_argument("--no-train", action="store_true", help="skip the C2 training-step figure added to the C3 line")
    ap.add_argument("--dump-outputs", metavar="DIR", help="C3 job: write a seeded sample of the SR images of the last timed "
                                                          "step to DIR/sr_sample.npy (float32, at most 48 MiB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "c3"):
        ap.error("--dump-outputs is implemented for the c3 workload of --impl ours")
    if args.impl == "reference":
        return run_reference(args)
    if args.workload == "c3t":
        return run_tiled(args)
    if args.workload == "n1":
        return run_drct(args)
    if args.workload == "c5":
        return run_c5(args)
    if args.workload != "c3":
        return run_train(args)

    import torch
    import torch.distributed as dist
    import isr_b200
    from isr_b200.dist import job_schedule
    from isr_b200.serving import PackedImage, PipelinedFusion, fuse_tiled

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the fusion path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    warmup = max(args.warmup, 3)
    H, W = args.lr
    n_images = args.images
    mpix_img = 16 * H * W / 1e6

    torch.manual_seed(0)
    m = isr_b200.CompleteEnhancedFusionSR(None).eval().to(dev)
    m.precision = args.precision
    whole, tail = job_schedule(n_images, world)
    mine = whole[rank]
    my_tail = [(img, ranks, grid) for img, ranks, grid in tail if rank in ranks]
    groups = {}
    if world > 1:
        for img, ranks, grid in tail:                           # every rank creates every group, in the same order
            groups[img] = dist.new_group(ranks)
    sets = [device_inputs(H, W, dev, i) for i in range(N_INPUT_SETS)]
    h2d32 = 4 * (3 * H * W + 4 * 3 * 16 * H * W + (3 * 180 + 64) * H * W)
    d2h = 3 * 16 * H * W * 4

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    from isr_b200.dist import max_over_ranks as _mor

    def max_over_ranks(ms):
        return _mor(ms, dev)

    from isr_b200.serving import ConcurrentFusion
    conc = ConcurrentFusion(m, ways=args.in_flight, device=dev) if args.in_flight > 1 else None

    def job_resident(sink=None):
        """sink(i, sr): called with the SR image of this rank's i-th image of the step, on the stream that computed it."""
        if conc is not None:                                    # whole images of this rank: `in_flight` forwards on as many streams
            conc.run((sets[i % N_INPUT_SETS] for i in mine), sink)
        else:
            for j, i in enumerate(mine):
                lr_, im_, ft_ = sets[i % N_INPUT_SETS]
                sr = m.forward_with_precomputed(lr_, im_, ft_)
                if sink is not None:
                    sink(j, sr)
        for j, (img, ranks, grid) in enumerate(my_tail):
            lr_, im_, ft_ = sets[img % N_INPUT_SETS]
            sr = fuse_tiled(m, lr_, im_, ft_, grid=grid, rank=ranks.index(rank), world=len(ranks), group=groups.get(img))
            if sink is not None:
                sink(len(mine) + j, sr)

    keep = dump = None
    if args.dump_outputs:
        dump_idx = dump_sample_index(len(mine) + len(my_tail), 3 * 16 * H * W, world).to(dev)
        dump = torch.empty(dump_idx.shape, device=dev)

        def keep(i, sr):                                        # one gather kernel per image, last timed step only
            torch.index_select(sr.reshape(-1), 0, dump_idx[i], out=dump[i])

    for _ in range(warmup):                                     # >= 3 warm-up forwards per distinct path (not whole jobs)
        lr_, im_, ft_ = sets[0]
        m.forward_with_precomputed(lr_, im_, ft_)
    if keep is not None and dump.shape[0]:                      # first launch (module load) of the gather before the timed region
        keep(0, m.forward_with_precomputed(*sets[0]))
    if conc is not None:
        for _ in range(warmup):
            conc.run(sets[i % N_INPUT_SETS] for i in range(args.in_flight))
    for img, ranks, grid in my_tail[:1]:
        for _ in range(2):
            fuse_tiled(m, *sets[img % N_INPUT_SETS], grid=grid, rank=ranks.index(rank), world=len(ranks), group=groups.get(img))
    eng = m._engine
    hot = [f"rf.{i}" for i in eng._refine_idx[1:-1]]

    # ---- timed region: inputs resident in HBM ---------------------------------------------
    sampler = ClockSampler(local)
    sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for step in range(args.steps):
        job_resident(keep if step == args.steps - 1 else None)
    e1.record()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1))
    clocks = sampler.stop()
    if dump is not None:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        name = "sr_sample" if world == 1 else f"sr_sample_rank{rank}"
        np.save(os.path.join(args.dump_outputs, name + ".npy"), dump.cpu().numpy())
        keep = dump = dump_idx = None
    # the dominant kernel's launch time: CUDA-event pairs around the hot layers of 100 further forwards on ONE stream (with
    # several images in flight a launch's wall time would include kernels of the other stream)
    eng.timed_layers = timed = {n: [] for n in hot}
    for i in range(100):
        m.forward_with_precomputed(*sets[i % N_INPUT_SETS])
    torch.cuda.synchronize()
    eng.timed_layers = None
    launches = eng.launches * (len(mine) + len(my_tail)) * args.steps
    hot_ms = [a.elapsed_time(b) for evs in timed.values() for a, b in evs]

    # ---- in-situ trace of one forward (every launch, single stream): per-phase time and the memory-bound kernels' roofline
    trace_rows = None
    if rank == 0:
        prev_overlap = eng.overlap_routing
        eng.overlap_routing = False
        eng.trace = []
        m.forward_with_precomputed(*sets[1 % N_INPUT_SETS])
        torch.cuda.synchronize()
        trace_rows = [(lab, a.elapsed_time(b)) for lab, a, b in eng.trace]
        eng.trace = None
        eng.overlap_routing = prev_overlap

    # ---- e2e: host caches -> SR image in host memory, copies inside the timed region -------------------------
    # Serving format = fp16 host caches (what the reference's val / TTA extractors store: scripts/extract_val_cache.py:
    # 167-209, scripts/extract_test_tta_cache.py:296-326), one packed pinned buffer and ONE host->device copy per image.
    out_host = torch.empty(1, 3, 4 * H, 4 * W).pin_memory()
    packed = [PackedImage(sets[i][0].cpu(), {k: v.cpu() for k, v in sets[i][1].items()}, {k: v.cpu() for k, v in sets[i][2].items()},
                          dtype=torch.float16) for i in range(N_INPUT_SETS)]
    pipe = PipelinedFusion(m, depth=2, device=dev)
    tail_dev = None
    if my_tail:
        tail_dev = torch.empty(packed[0].nbytes, dtype=torch.uint8, device=dev)

    def job_e2e(p_list):
        for i in mine:
            pipe.submit_packed(p_list[i % N_INPUT_SETS], out_host)
        pipe.finish()
        for img, ranks, grid in my_tail:                        # tile group: every member stages the image, the leader copies out
            pk = p_list[img % N_INPUT_SETS]
            tail_dev.copy_(pk.buf, non_blocking=True)
            lr_, im_, ft_ = pk.views(tail_dev)
            sr = fuse_tiled(m, lr_, im_, ft_, grid=grid, rank=ranks.index(rank), world=len(ranks), group=groups.get(img))
            if ranks[0] == rank:
                out_host.copy_(sr, non_blocking=True)
            torch.cuda.synchronize()

    for i in range(min(4, len(mine))):                          # warm-up: graph capture of both pipeline slots
        pipe.submit_packed(packed[i % N_INPUT_SETS], out_host)
    pipe.finish()
    barrier()
    t0 = time.perf_counter()
    e0.record()
    for _ in range(args.steps):
        job_e2e(packed)
    e1.record()
    barrier()
    ms_e2e = max_over_ranks(max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3))
    h2d16 = packed[0].payload_bytes

    # the same loop from fp32 host buffers (553 MB per image: PCIe- / host-memory-bound with several GPUs behind one host)
    e2e32 = None
    try:
        packed32 = [PackedImage(sets[i][0].cpu(), {k: v.cpu() for k, v in sets[i][1].items()},
                                {k: v.cpu() for k, v in sets[i][2].items()}, dtype=torch.float32) for i in range(2)]
        pipe32 = PipelinedFusion(m, depth=2, device=dev)
        n32 = min(len(mine), 12)
        for i in range(min(4, n32)):
            pipe32.submit_packed(packed32[i % 2], out_host)
        pipe32.finish()
        barrier()
        t0 = time.perf_counter()
        e0.record()
        for i in range(n32):
            pipe32.submit_packed(packed32[i % 2], out_host)
        pipe32.finish()
        e1.record()
        barrier()
        ms32 = max_over_ranks(max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3))
        if n32:
            e2e32 = {"value": world * n32 * mpix_img / (ms32 * 1e-3), "unit": "HR MPix/s", "h2d_bytes_per_image": packed32[0].payload_bytes,
                     "images_per_rank": n32, "ms_per_image": ms32 / n32,
                     "note": "fp32 pinned host buffers instead of the fp16 cache format; whole images only"}
        del pipe32, packed32
    except Exception as exc:
        e2e32 = {"error": repr(exc)[:200]}
    del pipe

    # ---- second half of BASELINE.json's metric: training patches/s (C2 step, same ranks) -------------
    train = None
    trainer = None
    if not args.no_train and tuple(args.lr) == (LR_H, LR_W) and os.environ.get("FFSR_BENCH_NO_TRAIN") is None:
        m._engine = None
        sets = None
        packed = None
        torch.cuda.empty_cache()
        try:
            r = measure_train(args, "c2", dev, world, rank, local, 5, 4, e2e=False)
            trainer = r["trainer"]
            tfl = TRAIN_FLOP_PER_HR_PIXEL * r["patches"] * 16 * r["hw"] ** 2 / (r["ms"] * 1e-3) / 1e12
            train = {"metric": "fusion_train_patches_per_s", "value": r["patches"] / (r["ms"] * 1e-3), "unit": "patches/s",
                     "ms_per_step": r["ms"], "steps": 5, "scaling": "strong", "n_gpus": world,
                     "config": train_config("c2", r["patches"], r["B"], r["hw"], args.precision),
                     "tflops_algorithmic": tfl, "tflops_algorithmic_per_gpu": tfl / world}
            r = None
        except Exception as exc:                               # the headline line must survive a training failure
            train = {"error": repr(exc)[:300]}

    gpu_eager = None
    if world == 1 and not args.no_gpu_eager:
        if trainer is not None:
            trainer._graph = None
        trainer = None
        m._engine = None
        sets = None
        import gc
        gc.collect()
        torch.cuda.empty_cache()
        try:
            gpu_eager = gpu_reference_eager_throughput(dev, H, W) or gpu_eager_throughput(m, dev, H, W)
        except Exception as exc:                                   # a baseline must not take the headline line down
            gpu_eager = {"error": repr(exc)[:300]}
        torch.cuda.empty_cache()

    if rank == 0:
        tensor_peak, hbm_peak, peak_src = _peaks()
        hot_flop = HOT_LAYER_FLOP_PER_HR_PIXEL * 16 * H * W
        hot_mean_ms = sum(hot_ms) / max(len(hot_ms), 1)
        achieved = hot_flop / (hot_mean_ms * 1e-3) / 1e12 if hot_ms else None
        total_img = n_images * args.steps
        ms_img = ms / total_img * world                         # per image per GPU
        whole_tflops = FLOP_PER_HR_PIXEL * 16 * H * W * total_img / (ms * 1e-3) / 1e12 / world
        line = {
            "metric": "fusion_forward_hr_mpix_per_s", "value": total_img * mpix_img / (ms * 1e-3),
            "unit": "HR MPix/s", "n_gpus": world, "steps": args.steps, "warmup": warmup,
            "ms_per_step": ms / args.steps, "ms_per_image_per_gpu": ms_img, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32" if args.precision == "fp32" else "bf16", "data": "synthetic",
            "config": c3_config(H, W), "precision": args.precision,
            "images_in_flight": args.in_flight,    # per GPU, on as many CUDA streams (serving.ConcurrentFusion): `value` only
            "schedule": {"whole_images_per_rank": [len(w) for w in whole],
                         "tail": [{"image": img, "ranks": ranks, "grid": list(grid)} for img, ranks, grid in tail]},
            "e2e": {"value": total_img * mpix_img / (ms_e2e * 1e-3), "unit": "HR MPix/s",
                    "h2d_bytes_per_step": h2d16 * n_images, "d2h_bytes_per_step": d2h * n_images, "ms_per_step": ms_e2e / args.steps,
                    "h2d_gb_per_s_per_gpu": h2d16 * n_images * args.steps / world / (ms_e2e * 1e-3) / 1e9,
                    "format": "fp16 host caches (the reference's val / TTA cache format) in one packed pinned buffer per image: "
                              "one cudaMemcpyAsync in, CUDA-graph forward, one copy out (serving.PipelinedFusion.submit_packed)"},
            "e2e_fp32_host": e2e32,
            "gpu_launches": launches,
            "clocks": clocks,
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": tensor_peak, "unit": "TFLOP/s",
                         "frac": (achieved / tensor_peak) if achieved else None,
                         "traffic": HOT_LAYER_DRAM_BYTES if args.precision == "bf16" else None,
                         "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full capture of this "
                                           "kernel at this size (profiles/r02_convtc_refine_c3_ncu_full.txt); algorithmic "
                                           "bytes = 128 ch x 2 B x 2.766 MPix in + out = 1.416e9",
                         "kernel": "3x3 128->128 refinement conv (refine.2/4/6/8), "
                                   + ("k_conv_ffma<64,3> fp32 CUDA-core path" if args.precision == "fp32" else "tcgen05 implicit GEMM"),
                         "launch_ms": hot_mean_ms, "launches_timed": len(hot_ms), "flop_per_launch": hot_flop,
                         "peak_source": peak_src,
                         "whole_forward_tflops": whole_tflops, "whole_forward_frac": whole_tflops / tensor_peak,
                         "whole_forward_target_frac": 0.40},
        }
        if args.dump_outputs:
            line["dump_outputs"] = {"dir": args.dump_outputs,
                                    "note": "the timed region of this run includes one gather kernel per image of its last step "
                                            "(the sample written to the dump); take timings from runs without --dump-outputs"}
        if trace_rows:
            line["forward_breakdown"] = forward_breakdown(trace_rows, H, W, hbm_peak, tensor_peak)
        if train is not None:
            line["train"] = train
        if gpu_eager is not None:
            line["gpu_eager_baseline"] = gpu_eager
        if world == 1 and not args.no_cpu_baseline:
            threads = os.cpu_count() or 1
            try:
                torch.manual_seed(0)
                mp = isr_b200.CompleteEnhancedFusionSR(None).eval().to(dev)
                par, v, t = parity_at_headline_size(mp, dev, H, W, threads)
                line["parity"] = par
                line["cpu_baseline"] = {"value": v, "unit": "HR MPix/s", "cores": threads, "kind": "port",
                                        "sample": f"one fp32 oracle forward with intermediates, LR {H}x{W} ({16 * H * W / 1e6:.3f} HR "
                                                  f"MPix = one image of the job), {t:.1f} s on {threads} threads; its output is the "
                                                  "checker of the `parity` block"}
            except Exception as exc:
                line["cpu_baseline"] = {"error": repr(exc)[:300]}
        print(json.dumps(line), flush=True)
    if world > 1:
        _leave(world, trainer)


def forward_breakdown(rows, H, W, hbm_peak, tensor_peak):
    """Per-phase in-situ time of ONE forward (CUDA events around every launch, single stream) and the roofline position of
    the kernels that matter besides the refinement convs: algorithmic bytes (or FLOPs) / measured duration / measured peak."""
    P = H * W                                                 # LR pixels
    phases = {"P2 bands": 0.0, "P3 cross-band + LKA": 0.0, "P6 selector": 0.0, "P4 collaborative (LR)": 0.0, "P4 modulation (HR)": 0.0,
              "P5 hierarchical": 0.0, "P5b/P6 blend": 0.0, "P7a refine": 0.0, "P7b edge": 0.0, "output": 0.0}
    kern = {}
    lka_seen = 0
    for lab, ms in rows:
        if lab.startswith(("ffsr_dct", "ffsr_dwt", "ffsr_fft")):
            ph = "P2 bands"
        elif lab.startswith("ffsr_crossband") or " cb." in lab:
            ph = "P3 cross-band + LKA"
        elif " ds." in lab or lab.startswith(("ffsr_gate_finalize", "ffsr_selector_fused")):
            ph = "P6 selector"
        elif lab.startswith("ffsr_lka_tail64"):
            ph = "P3 cross-band + LKA"
        elif lab.startswith(("ffsr_lka_tail128", "ffsr_token_", "ffsr_align_tokens")):
            ph = "P4 collaborative (LR)"
        elif lab.startswith("ffsr_lka_depthwise"):
            ph = "P3 cross-band + LKA" if lka_seen == 0 else "P4 collaborative (LR)"
            kern["lka_dw_p3" if lka_seen == 0 else "lka_dw_p4"] = ms
            lka_seen += 1
        elif " co." in lab or lab.startswith(("ffsr_nchw", "ffsr_layernorm", "ffsr_token_attention")):
            ph = "P4 collaborative (LR)"
        elif lab.startswith(("ffsr_modulate", "ffsr_expert_downsample")):
            ph = "P4 modulation (HR)"
            if lab.startswith("ffsr_modulate"):
                kern["modulate_hr"] = ms
        elif " mr." in lab or lab.startswith(("ffsr_spatial_gate", "ffsr_resize")):
            ph = "P5 hierarchical"
        elif lab.startswith("ffsr_blend"):
            ph = "P5b/P6 blend"
        elif " rf." in lab:
            ph = "P7a refine"
        elif lab.startswith("ffsr_final"):
            ph = "output"
        else:
            ph = "P7b edge"
        phases[ph] += ms
        if lab.startswith("ffsr_resize_nhwc"):
            kern["resize_hr"] = ms                           # last call = the 2x -> HR upsampling into the stage-3 concat
        if lab.startswith("ffsr_spatial_gate"):
            kern["spatial_gate_hr"] = ms                     # last call = stage 3 (HR, 32 channels)
        if lab.startswith("ffsr_blend"):
            kern["blend_hr"] = ms
        if lab.startswith("ffsr_fft"):
            kern["fft_bands"] = ms
        if lab.startswith("ffsr_crossband_attention"):
            kern["crossband_attn"] = ms
    total = sum(phases.values())
    out = {"ms_per_forward_sum": total, "phase_ms": {k: round(v, 4) for k, v in phases.items()}}
    hbm = []
    if "lka_dw_p4" in kern:    # reads the bf16 token tensor once, writes bf16 once: 4 experts x 128 ch x (2 + 2) B per LR pixel
        b = 4 * 128 * 4 * P
        hbm.append({"kernel": "LKA depthwise chain, Phase 4 (BN -> dw5x5 -> dw1x21 -> dw21x1)", "algorithmic_bytes": b, "ms": kern["lka_dw_p4"],
                    "achieved_gb_s": b / kern["lka_dw_p4"] / 1e6, "frac_of_hbm": b / kern["lka_dw_p4"] / 1e6 / hbm_peak})
    if "modulate_hr" in kern:  # 4 expert images in (fp32) + ecol out (fp32) + 12-ch bf16 concat slice
        b = (4 * 3 * 4 * 2 + 12 * 2) * 16 * P
        hbm.append({"kernel": "HR modulation (bilinear x4 + GELU + 32->3 + sigmoid, 4 experts)", "algorithmic_bytes": b, "ms": kern["modulate_hr"],
                    "achieved_gb_s": b / kern["modulate_hr"] / 1e6, "frac_of_hbm": b / kern["modulate_hr"] / 1e6 / hbm_peak})
    if "fft_bands" in kern:    # 120 B per LR pixel for the two FFT bands (SURVEY 8d)
        b = 3 * 4 * 3 * P
        hbm.append({"kernel": "FFT low/high bands (staged shared-memory FFT)", "algorithmic_bytes": b, "ms": kern["fft_bands"],
                    "achieved_gb_s": b / kern["fft_bands"] / 1e6, "frac_of_hbm": b / kern["fft_bands"] / 1e6 / hbm_peak})
    if "resize_hr" in kern:    # 64 bf16 channels: a quarter of the HR pixels in, every HR pixel out
        b = 64 * 2 * (4 + 16) * P
        hbm.append({"kernel": "x2 bilinear upsampling into the stage-3 concat (64 ch bf16)", "algorithmic_bytes": b, "ms": kern["resize_hr"],
                    "achieved_gb_s": b / kern["resize_hr"] / 1e6, "frac_of_hbm": b / kern["resize_hr"] / 1e6 / hbm_peak})
    if "spatial_gate_hr" in kern:   # 32 bf16 channels in place
        b = 32 * 2 * 2 * 16 * P
        hbm.append({"kernel": "SpatialGate at HR (32 ch bf16, in place)", "algorithmic_bytes": b, "ms": kern["spatial_gate_hr"],
                    "achieved_gb_s": b / kern["spatial_gate_hr"] / 1e6, "frac_of_hbm": b / kern["spatial_gate_hr"] / 1e6 / hbm_peak})
    if "blend_hr" in kern:     # SURVEY 8d: 72 B per HR pixel (hier + 12 expert planes in, fused fp32 out) + the 32 B bf16 copy for the refine input
        b = (72 + 32) * 16 * P
        hbm.append({"kernel": "P5b / P6 blend at HR", "algorithmic_bytes": b, "ms": kern["blend_hr"],
                    "achieved_gb_s": b / kern["blend_hr"] / 1e6, "frac_of_hbm": b / kern["blend_hr"] / 1e6 / hbm_peak})
    out["memory_bound_kernels"] = hbm
    if hbm:
        out["worst_memory_bound_frac"] = min(h["frac_of_hbm"] for h in hbm)
        big = [h["frac_of_hbm"] for h in hbm if h["ms"] >= 0.1]
        if big:
            out["worst_memory_bound_frac_of_kernels_over_0.1ms"] = min(big)
    return out


if __name__ == "__main__":
    main()
