"""Cost of input gradients through the fusion.  Prints the GPU and its power limit, then one JSON line per figure:
  1. C2 shape (32 x 64x64 LR, bf16, train mode, L1): eager forward + backward with and without input gradients;
  2. an eval attribution pass at C3 (one 510x339 LR image, 4 experts with features, fp32 and bf16): forward + backward
     to every input, its time and torch.cuda.max_memory_allocated;
  3. the two Phase-2 adjoint kernels at C3 (B = 1) against their algorithmic bytes.
CUDA-event timing after warm-up; steps end in a device synchronise.
    python tools/bench_input_grad.py [--out profiles/r04_input_grad.txt]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import isr_b200  # noqa: E402
from isr_b200 import training as T  # noqa: E402
from oracle import fusion_oracle as O  # noqa: E402
from oracle.perturb import perturb_state_dict  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = ""
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": out or "unavailable"}


def timed(fn, warm=2, reps=5):
    for _ in range(warm):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def model(dev, precision, train):
    torch.manual_seed(0)
    m = isr_b200.CompleteEnhancedFusionSR(None)
    m.load_state_dict(perturb_state_dict(m.state_dict(), seed=7))
    m.precision = precision
    return m.train(train).to(dev)


def inputs(dev, B, H, W, grad):
    lr, imgs, fts, hr = O.synthetic_inputs(B, H, W)
    to = lambda t: t.to(dev).requires_grad_(grad)
    return (to(lr), {k: to(v) for k, v in imgs.items()}, {k: to(v) for k, v in fts.items()}), hr.to(dev)


def c2_step(dev):
    m = model(dev, "bf16", True)
    res = {}
    for grad in (False, True):
        args, hr = inputs(dev, 32, 64, 64, grad)

        def step():
            m.zero_grad(set_to_none=True)
            (m.forward_with_precomputed(*args) - hr).abs().mean().backward()
        res["with_input_grad_ms" if grad else "without_input_grad_ms"] = round(timed(step), 3)
    res["overhead_pct"] = round(100 * (res["with_input_grad_ms"] / res["without_input_grad_ms"] - 1), 2)
    return {"figure": "C2 train step, bf16, 32 x 64x64 LR, eager forward + backward", **res}


def c3_attribution(dev, precision):
    m = model(dev, precision, False)
    args, _ = inputs(dev, 1, 339, 510, True)
    leaves = [args[0], *args[1].values(), *args[2].values()]

    def attribution():
        for t in leaves:
            t.grad = None
        m.forward_with_precomputed(*args).sum().backward()
    attribution()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    ms = timed(attribution, warm=1, reps=3)
    return {"figure": f"C3 eval attribution pass ({precision}): 510x339 LR -> 2040x1356, forward + backward to lr, 4 images, "
                      "4 features", "ms": round(ms, 2),
            "max_memory_allocated_GB": round(torch.cuda.max_memory_allocated() / 1e9, 2)}


def adjoint_kernels(dev):
    m = model(dev, "fp32", True)
    lib = T._lib()
    B, H, W = 1, 339, 510
    fd = m.freq_decomp
    g3 = torch.randn(B, 3, 3, H, W, device=dev)
    g4 = torch.randn(B, 4, 3, H, W, device=dev)
    dx = torch.zeros(B, 3, H, W, device=dev)
    d, w_ = fd.dct, fd.dwt
    keep = [T._c32(t) for t in (d.dct_basis, d.dct_basis_t, d.low_mask, d.mid_mask, d.high_mask)]
    k2 = [T._c32(t) for t in (w_.lo_row, w_.hi_row, w_.lo_col, w_.hi_col)]
    Hp, Wp = (H + 7) // 8 * 8, (W + 7) // 8 * 8
    pad = torch.empty(B * 3 * Hp * Wp, device=dev)
    sub = T._dwt_sub(B, H, W, dev)
    S = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)

    def dct():
        T._ck(lib.ffsr_dct_bands_adjoint(g3.data_ptr(), B, H, W, *[t.data_ptr() for t in keep], pad.data_ptr(),
                                         dx.data_ptr(), S), "dct_bands_adjoint")

    def dwt():
        T._ck(lib.ffsr_dwt_bands_adjoint(g4.data_ptr(), B, H, W, *[t.data_ptr() for t in k2], sub.data_ptr(),
                                         dx.data_ptr(), S), "dwt_bands_adjoint")
    px = B * 3 * H * W
    # algorithmic bytes: band gradients read once, dx written once (DWT: read-modify-write)
    rows = []
    for name, fn, nbytes in (("ffsr_dct_bands_adjoint", dct, (3 + 1) * 4 * px), ("ffsr_dwt_bands_adjoint", dwt, (4 + 2) * 4 * px)):
        ms = timed(fn, warm=5, reps=50)
        rows.append({"figure": f"{name} at C3 (B=1, 510x339)", "ms": round(ms, 4), "algorithmic_MB": round(nbytes / 1e6, 2),
                     "GB_per_s": round(nbytes / ms / 1e6, 1)})
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_input_grad.py needs a CUDA device")
    dev = torch.device("cuda:0")
    lines = [json.dumps(gpu_info()), json.dumps(c2_step(dev))]
    for prec in ("fp32", "bf16"):
        lines.append(json.dumps(c3_attribution(dev, prec)))
    lines += [json.dumps(r) for r in adjoint_kernels(dev)]
    for ln in lines:
        print(ln, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
