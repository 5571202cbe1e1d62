"""Cost of world-invariant training against the default data-parallel step, on the C2 geometry of bench.py: a global
batch of 32 patches of 64x64 LR, bf16, L1 loss, CUDA-graph steps.

    python tools/bench_invariant_train.py [--steps 20] [--rounds 3]
    torchrun --nproc-per-node N tools/bench_invariant_train.py

Per configuration (mode, M global micro-batches of 32/M patches; k = M/N per rank) one trainer is built and warmed
up; the configurations are then timed in alternating rounds of --steps graph replays (CUDA events, max over ranks), and
the median round is reported.  Before timing, at N=1, the invariant k=1 step is checked to equal the default step bit
for bit over 3 eager + 3 graph steps.  Prints one JSON line per configuration after a line naming the GPU and its power
limit; writes no files.
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

GLOBAL_BATCH, HW = 32, 64


def gpu_info(index):
    try:
        out = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = ""
    return {"gpu": torch.cuda.get_device_name(index), "nvidia_smi": out or "unavailable"}


def make_trainer(dev, world, rank, invariant, M):
    import isr_b200
    from isr_b200.losses import CombinedLoss
    from isr_b200.trainer import FusionTrainer
    from oracle import fusion_oracle as O
    torch.manual_seed(0)
    m = isr_b200.CompleteEnhancedFusionSR(None).to(dev)
    m.precision = "bf16"
    crit = CombinedLoss()
    crit.set_weights({"charbonnier": 0, "l2": 0, "vgg": 0, "edge": 0, "clip": 0, "swt": 0, "fft": 0, "ssim": 0, "l1": 1.0})
    tr = FusionTrainer(m, crit, lr=2e-4, weight_decay=1e-4, max_grad_norm=1.0, ema_decay=0.999,
                       accumulation_steps=M // world, world_invariant=invariant)
    B = GLOBAL_BATCH // world
    lr, imgs, fts, hr = O.synthetic_inputs(GLOBAL_BATCH, HW, HW, seed=1234)
    sl = slice(rank * B, (rank + 1) * B)
    args = (lr[sl].to(dev), {k: v[sl].to(dev) for k, v in imgs.items()}, {k: v[sl].to(dev) for k, v in fts.items()},
            hr[sl].to(dev))
    return tr, args


def state(tr):
    o = tr.optimizer
    return [o.bucket.flat.clone(), o.exp_avg.clone(), o.exp_avg_sq.clone(), o.ema.clone()] + \
        [b.clone() for n, b in tr.model.named_buffers() if n.endswith(("running_mean", "running_var", "num_batches_tracked"))]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_invariant_train.py needs a CUDA device")
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    rank = dist.get_rank() if world > 1 else 0
    if rank == 0:
        print(json.dumps({"world": world, **gpu_info(local)}), flush=True)

    if world == 1:                    # the anchor: invariant N=1, k=1 is the default step, bit for bit
        finals = []
        for inv in (False, True):
            tr, a = make_trainer(dev, 1, 0, inv, 1)
            losses = [tr.step(*a)[0].clone() for _ in range(6)]
            finals.append((losses, state(tr)))
            del tr
        equal = all(torch.equal(x, y) for x, y in zip(finals[0][0] + finals[0][1], finals[1][0] + finals[1][1]))
        print(json.dumps({"check": "invariant N=1 k=1 == default, 3 eager + 3 graph steps", "bitwise_equal": equal}),
              flush=True)
        del finals

    configs = []
    for M in sorted({world, 8} if 8 % world == 0 else {world}):
        for inv in (False, True):
            configs.append((inv, M))
    runs = []
    for inv, M in configs:
        tr, a = make_trainer(dev, world, rank, inv, M)
        for _ in range(5):            # 3 eager steps, the capture, one replay
            tr.step(*a)
        runs.append((tr, a))
    times = {c: [] for c in configs}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(args.rounds):
        for c, (tr, a) in zip(configs, runs):
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            e0.record()
            for _ in range(args.steps):
                tr.step(*a)
            e1.record()
            torch.cuda.synchronize()
            t = torch.tensor([e0.elapsed_time(e1) / args.steps], device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            times[c].append(float(t))
    if rank == 0:
        for inv, M in configs:
            ts = sorted(times[(inv, M)])
            print(json.dumps({"mode": "world_invariant" if inv else "default", "N": world, "M": M, "k": M // world,
                              "b": GLOBAL_BATCH // M, "ms_per_step_median": round(ts[len(ts) // 2], 3),
                              "ms_per_step_rounds": [round(x, 3) for x in times[(inv, M)]], "steps_per_round": args.steps}),
                  flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
