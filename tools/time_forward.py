"""Wall-clock-free timing of the C3 fusion forward in its launch modes (CUDA events, inputs resident):
eager launches with / without the routing side stream, CUDA-graph replay, and host time per eager forward.
    python tools/time_forward.py [--lr 339 510] [--steps 10] [--precision bf16]
"""
import argparse
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import isr_b200  # noqa: E402
from oracle import fusion_oracle as O  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--lr", type=int, nargs=2, default=[339, 510])
ap.add_argument("--steps", type=int, default=10)
ap.add_argument("--precision", default="bf16")
a = ap.parse_args()
dev = torch.device("cuda:0")
torch.manual_seed(0)
m = isr_b200.CompleteEnhancedFusionSR(None).eval().to(dev)
m.precision = a.precision
lr, imgs, fts, _ = O.synthetic_inputs(1, a.lr[0], a.lr[1])
lr, imgs, fts = lr.to(dev), {k: v.to(dev) for k, v in imgs.items()}, {k: v.to(dev) for k, v in fts.items()}


def fwd():
    return m.forward_with_precomputed(lr, imgs, fts)


def timed(fn, steps=a.steps):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    host = (time.perf_counter() - t0) * 1e3 / steps
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps, host


fwd()
eng = m._engine
ms, host = timed(fwd)
print(f"eager, routing side stream : {ms:7.3f} ms / forward  (host enqueue time {host:.3f} ms, {eng.launches} launches)")
eng.overlap_routing = False
ms, host = timed(fwd)
print(f"eager, single stream       : {ms:7.3f} ms / forward  (host enqueue time {host:.3f} ms)")
g = torch.cuda.CUDAGraph()
with torch.cuda.graph(g):
    out = fwd()
ms, host = timed(g.replay)
print(f"CUDA graph, single stream  : {ms:7.3f} ms / forward  (host enqueue time {host:.3f} ms)")
