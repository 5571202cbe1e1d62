"""bench.py --dump-outputs: the sample of the last timed step's SR images that lets two builds be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402


def test_dump_sample_is_fixed_and_fits_the_budget():
    rows, numel = bench.N_JOB_IMAGES, 3 * 16 * bench.LR_H * bench.LR_W          # the default C3 job: 100 x 2040x1356 images
    idx = bench.dump_sample_index(rows, numel)
    assert idx.shape[0] == rows and 4 * idx.numel() <= bench.DUMP_BUDGET_BYTES <= 64 * 10**6
    assert int(idx.min()) >= 0 and int(idx.max()) < numel
    assert bool((idx[:, 1:] >= idx[:, :-1]).all()) and not torch.equal(idx[0], idx[1])
    assert torch.equal(idx, bench.dump_sample_index(rows, numel))
    for world in (2, 8):                                                          # one file per rank, same budget in all
        assert 4 * world * bench.dump_sample_index(rows // world, numel, world).numel() <= bench.DUMP_BUDGET_BYTES
    small = bench.dump_sample_index(3, 3 * 16 * 24 * 32)                          # small images are kept whole
    assert torch.equal(small, torch.arange(3 * 16 * 24 * 32).repeat(3, 1))
    assert bench.dump_sample_index(0, numel, 8).shape == (0, 0)                     # a rank the schedule gives no image


@pytest.mark.gpu
def test_dump_outputs_are_what_the_timed_path_returned(tmp_path):
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import isr_b200
    H, W, n = 24, 32, 3
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--lr", str(H), str(W), "--images", str(n),
                        "--steps", "2", "--warmup", "1", "--precision", "bf16", "--no-cpu-baseline", "--no-gpu-eager",
                        "--no-train", "--dump-outputs", str(out)],
                       cwd=ROOT, capture_output=True, text=True, timeout=900,
                       env=dict(os.environ, PYTHONDONTWRITEBYTECODE="1"))
    assert r.returncode == 0, r.stderr[-3000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
    assert sorted(os.listdir(out)) == ["sr_sample.npy"]
    got = np.load(out / "sr_sample.npy")
    assert got.dtype == np.float32 and got.shape == (n, 3 * 16 * H * W)
    # the same seeded weights and inputs in this process: image i of a step is input set i % N_INPUT_SETS
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    m = isr_b200.CompleteEnhancedFusionSR(None).eval().to(dev)
    m.precision = "bf16"
    idx = bench.dump_sample_index(n, 3 * 16 * H * W)
    for i in range(n):
        sr = m.forward_with_precomputed(*bench.device_inputs(H, W, dev, i % bench.N_INPUT_SETS))
        assert torch.equal(torch.from_numpy(got[i]), sr.reshape(-1).cpu()[idx[i]]), i
