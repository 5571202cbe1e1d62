"""Bitwise reproducibility of the training path.

Every reduction of the backward, loss and optimizer kernels writes per-block partials to a workspace and adds them in
a fixed order, so the same inputs give bitwise-identical results on the same GPU.  Checked per entry point (twice, and
against a CPU fp64 torch reference), for the bilinear adjoint beyond a 6x factor, for two ``FusionTrainer`` runs (eager
and CUDA-graph steps, fp32 and bf16, attention dropout on), for the reference-style loop with ``torch.optim.AdamW``,
and under ``torch.use_deterministic_algorithms(True)``.
"""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

import isr_b200
from isr_b200 import _cabi as K
from isr_b200 import losses as FL
from isr_b200 import training as T
from oracle import fusion_oracle as O
from oracle import loss_oracle as L

pytestmark = pytest.mark.gpu

N, H, W = 32, 128, 128          # 32 x 128^2 rows: hundreds of blocks per reduction
STAGE3 = {"charbonnier": 0, "l2": 0, "vgg": 0, "edge": 0, "clip": 0, "l1": 0.6, "swt": 0.25, "fft": 0.1, "ssim": 0.05}


def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


def _rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return ((a - b).norm() / (b.norm() + 1e-30)).item()


def _twice(fn):
    """fn() -> tuple of tensors; run it twice and require bitwise-equal results."""
    r1 = [t.detach().clone() for t in fn()]
    r2 = [t.detach().clone() for t in fn()]
    torch.cuda.synchronize()
    for i, (a, b) in enumerate(zip(r1, r2)):
        assert torch.equal(a, b), (i, float((a.double() - b.double()).abs().max()))
    return r1


def _cl(t, dev):
    return t.to(dev).contiguous(memory_format=torch.channels_last)


# ------------------------------------------------------------------------------------------
# per entry point
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("Cc", [3, 32, 64, 128])
@pytest.mark.parametrize("pitch", ["dense", "padded"])
def test_colsum_is_reproducible(Cc, pitch):
    """ffsr_colsum: dense channels-last rows path and the strided path (pixel pitch padded beyond C)."""
    dev = _cuda()
    lib = K.load()
    g = torch.Generator().manual_seed(Cc)
    cp = Cc if pitch == "dense" else Cc + 5
    buf = torch.randn(N, H, W, cp, generator=g)
    v = buf.to(dev)
    ws = torch.empty(lib.ffsr_colsum_workspace_bytes(N, H, W, Cc), device=dev, dtype=torch.uint8)

    def run():
        out = torch.zeros(Cc, device=dev)
        S = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        K.check(lib.ffsr_colsum(v.data_ptr(), K.DT_F32, N, H, W, Cc, H * W * cp, W * cp, cp, out.data_ptr(),
                                ws.data_ptr(), ws.numel(), S), "colsum")
        return (out,)

    (out,) = _twice(run)
    assert _rel(out, buf[..., :Cc].double().sum((0, 1, 2))) < 5e-6


@pytest.mark.parametrize("cin,cout,ks", [(3, 32, 3), (32, 32, 3), (64, 64, 1), (128, 128, 1)])
def test_conv_wgrad_fp32_is_reproducible(cin, cout, ks):
    """ffsr_conv2d_wgrad (fp32 FFMA path) + its bias sums."""
    dev = _cuda()
    g = torch.Generator().manual_seed(cin + cout)
    x = torch.randn(N, cin, H, W, generator=g)
    w = torch.randn(cout, cin, ks, ks, generator=g) / (cin * ks * ks) ** 0.5
    b = torch.randn(cout, generator=g)
    gy = torch.randn(N, cout, H, W, generator=g)
    xd, gyd = _cl(x, dev), _cl(gy, dev)

    def run():
        wd, bd = w.to(dev).requires_grad_(), b.to(dev).requires_grad_()
        T.conv2d(xd, wd, bd).backward(gyd)
        return wd.grad, bd.grad

    dw, db = _twice(run)
    xr, wr, br = x.double(), w.double().requires_grad_(), b.double().requires_grad_()
    F.conv2d(xr, wr, br, padding=ks // 2).backward(gy.double())
    assert _rel(dw, wr.grad) < 5e-6
    assert _rel(db, br.grad) < 5e-6


@pytest.mark.parametrize("cin,cout,ks", [(64, 64, 3), (128, 128, 1)])
def test_conv_wgrad_tc_bias_is_reproducible(cin, cout, ks):
    """ffsr_conv2d_wgrad_tc (bf16 tcgen05 path): its bias gradient goes through the fixed-order column sums."""
    dev = _cuda()
    g = torch.Generator().manual_seed(cin * 3 + ks)
    x = torch.randn(N, cin, H, W, generator=g).bfloat16().float()
    w = (torch.randn(cout, cin, ks, ks, generator=g) / (cin * ks * ks) ** 0.5).bfloat16().float()
    b = torch.randn(cout, generator=g)
    gy = torch.randn(N, cout, H, W, generator=g).bfloat16().float()
    xd, gyd = _cl(x, dev), _cl(gy, dev)

    def run():
        wd, bd = w.to(dev).requires_grad_(), b.to(dev).requires_grad_()
        T.conv2d(xd, wd, bd, tc=True).backward(gyd)
        return wd.grad, bd.grad

    dw, db = _twice(run)
    xr, wr, br = x.double(), w.double().requires_grad_(), b.double().requires_grad_()
    F.conv2d(xr, wr, br, padding=ks // 2).backward(gy.double())
    assert _rel(dw, wr.grad) < 1e-4
    assert _rel(db, br.grad) < 5e-6


@pytest.mark.parametrize("E", [32, 64, 128])
def test_layernorm_backward_is_reproducible(E):
    dev = _cuda()
    g = torch.Generator().manual_seed(E)
    x = torch.randn(N, E, H, W, generator=g)
    w = 1 + 0.1 * torch.randn(E, generator=g)
    b = 0.1 * torch.randn(E, generator=g)
    gy = torch.randn(N, E, H, W, generator=g)
    xd, gyd = _cl(x, dev), _cl(gy, dev)

    def run():
        ln = torch.nn.LayerNorm(E).to(dev)
        with torch.no_grad():
            ln.weight.copy_(w)
            ln.bias.copy_(b)
        xx = xd.clone().requires_grad_()
        T.layernorm(xx, ln).backward(gyd)
        return xx.grad, ln.weight.grad, ln.bias.grad

    dx, dw, db = _twice(run)
    xr, wr, br = x.double().requires_grad_(), w.double().requires_grad_(), b.double().requires_grad_()
    y = F.layer_norm(xr.permute(0, 2, 3, 1), (E,), wr, br, 1e-5).permute(0, 3, 1, 2)
    y.backward(gy.double())
    assert _rel(dx, xr.grad) < 1e-5
    assert _rel(dw, wr.grad) < 1e-5
    assert _rel(db, br.grad) < 1e-5


@pytest.mark.parametrize("Cc", [32, 64, 128])
def test_batchnorm_stats_and_backward_are_reproducible(Cc):
    dev = _cuda()
    G = 2
    g = torch.Generator().manual_seed(Cc + 1)
    x = torch.randn(N, Cc, H, W, generator=g) * 2 + 0.5
    w = 1 + 0.1 * torch.randn(Cc, generator=g)
    b = 0.1 * torch.randn(Cc, generator=g)
    gy = torch.randn(N, Cc, H, W, generator=g)
    xd, gyd = _cl(x, dev), _cl(gy, dev)

    def run():
        bn = torch.nn.BatchNorm2d(Cc).to(dev)
        with torch.no_grad():
            bn.weight.copy_(w)
            bn.bias.copy_(b)
        xx = xd.clone().requires_grad_()
        sink = []
        y = T.batchnorm_train(xx, bn, G, sink)
        y.backward(gyd)
        return y, sink[0][1], sink[0][2], xx.grad, bn.weight.grad, bn.bias.grad

    y, mean, var, dx, dw, db = _twice(run)
    xr, wr, br = x.double().requires_grad_(), w.double().requires_grad_(), b.double().requires_grad_()
    xg = xr.view(G, N // G, Cc, H, W)
    mu = xg.mean((1, 3, 4), keepdim=True)
    vr = xg.var((1, 3, 4), unbiased=False, keepdim=True)
    yr = ((xg - mu) / torch.sqrt(vr + 1e-5)).view(N, Cc, H, W) * wr[:, None, None] + br[:, None, None]
    yr.backward(gy.double())
    assert _rel(mean, mu.view(G, Cc)) < 1e-6
    assert _rel(var, vr.view(G, Cc)) < 1e-6
    assert _rel(y, yr) < 1e-5
    assert _rel(dx, xr.grad) < 1e-5
    assert _rel(dw, wr.grad) < 1e-5
    assert _rel(db, br.grad) < 1e-5


@pytest.mark.parametrize("Cc", [3, 64])          # scalar and 8-channel vector kernels
@pytest.mark.parametrize("with_c", [False, True])
def test_axpby_backward_is_reproducible(Cc, with_c):
    dev = _cuda()
    g = torch.Generator().manual_seed(Cc * 2 + with_c)
    a, bb, cc, gy = (torch.randn(N, Cc, H, W, generator=g) for _ in range(4))
    s1, s2 = torch.tensor(0.7), torch.tensor(-0.3)
    ad, bd, cd, gyd = (_cl(t, dev) for t in (a, bb, cc, gy))

    def run():
        t1, t2 = s1.to(dev).requires_grad_(), s2.to(dev).requires_grad_()
        out = T.axpby(ad, bd, t1, cd if with_c else None, t2 if with_c else None)
        out.backward(gyd)
        return (t1.grad, t2.grad) if with_c else (t1.grad,)

    res = _twice(run)
    assert _rel(res[0], (gy.double() * bb.double()).sum()) < 1e-5
    if with_c:
        assert _rel(res[1], (gy.double() * cc.double()).sum()) < 1e-5


@pytest.mark.parametrize("kind,kh,kw", [(0, 5, 5), (1, 1, 21), (2, 21, 1)])
@pytest.mark.parametrize("Cc", [32, 64, 128])
def test_depthwise_wgrad_is_reproducible(kind, kh, kw, Cc):
    dev = _cuda()
    n, h, w = 8, 64, 64            # 8 x 64^2 x C: the LKA stage shapes of a C2 step
    g = torch.Generator().manual_seed(kind * 7 + Cc)
    x = torch.randn(n, Cc, h, w, generator=g)
    wt = torch.randn(Cc, 1, kh, kw, generator=g) * 0.1
    gy = torch.randn(n, Cc, h, w, generator=g)
    xd, gyd = _cl(x, dev), _cl(gy, dev)

    def run():
        wd = wt.to(dev).requires_grad_()
        T._DwStage.apply(xd, wd, kind).backward(gyd)
        return (wd.grad,)

    (dw,) = _twice(run)
    wr = wt.double().requires_grad_()
    F.conv2d(x.double(), wr, padding=(kh // 2, kw // 2), groups=Cc).backward(gy.double())
    assert _rel(dw, wr.grad) < 1e-5


@pytest.mark.parametrize("name", ["l1", "swt", "ssim", "fft"])
def test_losses_are_reproducible(name):
    dev = _cuda()
    g = torch.Generator().manual_seed(3)
    a = torch.rand(8, 4, H, W, generator=g)                     # 32 planes of 128^2
    b = (a + 0.1 * torch.randn(8, 4, H, W, generator=g)).clamp(0, 1)
    ad, bd = a.to(dev), b.to(dev)

    def run():
        p = ad.clone().requires_grad_()
        total, _ = FL.fused_losses(p, bd, {name: 1.0})
        total.backward()
        return total, p.grad

    total, grad = _twice(run)
    ar = a.clone().requires_grad_()
    ref = L.LOSSES[name](ar, b)
    ref.backward()
    vtol = 2e-5 * max(1.0, abs(float(ref))) + (L.fft_branch_cut_slack(a, b) if name == "fft" else 0.0)
    assert abs(float(total) - float(ref)) <= vtol, (float(total), float(ref))
    assert _rel(grad, ar.grad) <= (2e-3 if name == "fft" else 1e-4)


def test_sumsq_is_reproducible():
    dev = _cuda()
    lib = K.load()
    n = N * H * W * 3
    gr = torch.randn(n, generator=torch.Generator().manual_seed(11))
    gd = gr.to(dev)
    ws = torch.empty(lib.ffsr_sumsq_workspace_bytes(n), device=dev, dtype=torch.uint8)

    def run():
        out = torch.zeros(1, device=dev, dtype=torch.float64)
        K.check(lib.ffsr_sumsq(gd.data_ptr(), n, out.data_ptr(), ws.data_ptr(), ws.numel(),
                               C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)), "sumsq")
        return (out,)

    (out,) = _twice(run)
    assert abs(float(out) - float((gr.double() ** 2).sum())) <= 1e-9 * float((gr.double() ** 2).sum())


# ------------------------------------------------------------------------------------------
# bilinear adjoint beyond a 6x factor (the FFT mask resize: 64^2 -> H x (W/2+1))
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("C_,h,w,H_,W_", [(1, 64, 64, 512, 257), (3, 8, 8, 100, 100), (8, 8, 8, 100, 77)])
def test_bilinear_adjoint_beyond_factor_6(C_, h, w, H_, W_):
    dev = _cuda()
    g = torch.Generator().manual_seed(h + H_)
    x = torch.randn(2, C_, h, w, generator=g)
    gy = torch.randn(2, C_, H_, W_, generator=g)
    xr = x.clone().requires_grad_()
    yr = F.interpolate(xr, size=(H_, W_), mode="bilinear", align_corners=False)
    yr.backward(gy)
    xd = _cl(x, dev).requires_grad_()
    y = T._bilinear(xd, (H_, W_))
    y.backward(_cl(gy, dev))
    assert _rel(y, yr) < 2e-6
    assert _rel(xd.grad, xr.grad) < 2e-6


# ------------------------------------------------------------------------------------------
# whole trainer and the reference-style loop
# ------------------------------------------------------------------------------------------
def _inputs(dev, B=8, S=64):
    lr, imgs, fts, hr = O.synthetic_inputs(B, S, S)
    return (lr.to(dev), {k: v.to(dev) for k, v in imgs.items()}, {k: v.to(dev) for k, v in fts.items()}, hr.to(dev))


def _trainer_run(dev, precision, args, steps=6):
    """Seeded model (dropout at its default 0.1) + FusionTrainer: 3 eager steps, capture, 3 replays."""
    from isr_b200.losses import CombinedLoss
    from isr_b200.trainer import FusionTrainer
    torch.manual_seed(0)
    m = isr_b200.CompleteEnhancedFusionSR(None).to(dev)
    m.precision = precision
    crit = CombinedLoss()
    crit.set_weights(STAGE3)
    tr = FusionTrainer(m, crit, lr=2e-4, cuda_graph=True, graph_warmup=3)
    losses, comps = [], []
    for _ in range(steps):
        loss, cp = tr.step(*args)
        losses.append(loss.detach().clone())
        comps.append({k: v.detach().clone() for k, v in cp.items()})
    torch.cuda.synchronize()
    assert tr._graph is not None
    o = tr.optimizer
    state = {"flat": o.bucket.flat.clone(), "exp_avg": o.exp_avg.clone(), "exp_avg_sq": o.exp_avg_sq.clone(),
             "ema": o.ema.clone()}
    bufs = {n: b.clone() for n, b in m.named_buffers() if n.endswith(("running_mean", "running_var", "num_batches_tracked"))}
    return losses, comps, state, bufs


def _assert_same_run(r1, r2):
    (l1, c1, s1, b1), (l2, c2, s2, b2) = r1, r2
    for i, (a, b) in enumerate(zip(l1, l2)):
        assert torch.equal(a, b), (i, float(a), float(b))
    for a, b in zip(c1, c2):
        assert a.keys() == b.keys() and all(torch.equal(a[k], b[k]) for k in a)
    for k in s1:
        assert torch.equal(s1[k], s2[k]), (k, float((s1[k] - s2[k]).abs().max()))
    assert b1.keys() == b2.keys() and len(b1) > 0
    for k in b1:
        assert torch.equal(b1[k], b2[k]), k


@pytest.mark.timeout(900)
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_two_trainers_are_bitwise_identical(precision):
    dev = _cuda()
    args = _inputs(dev)
    r1 = _trainer_run(dev, precision, args)
    r2 = _trainer_run(dev, precision, args)
    assert all(torch.isfinite(l) for l in r1[0])
    _assert_same_run(r1, r2)


@pytest.mark.timeout(900)
def test_reference_style_loop_is_bitwise_reproducible():
    """model.train() + CombinedLoss + loss.backward() + clip_grad_norm_ + torch.optim.AdamW, twice."""
    from isr_b200.losses import CombinedLoss
    dev = _cuda()
    lr, imgs, fts, hr = _inputs(dev)

    def run():
        torch.manual_seed(0)
        m = isr_b200.CompleteEnhancedFusionSR(None).to(dev).train()
        crit = CombinedLoss()
        crit.set_weights(STAGE3)
        opt = torch.optim.AdamW(m.parameters(), lr=2e-4, weight_decay=1e-4)
        grads = []
        for _ in range(2):
            opt.zero_grad()
            sr = m.forward_with_precomputed(lr, imgs, fts).clamp(0, 1)
            crit(sr, hr).backward()
            torch.nn.utils.clip_grad_norm_(m.parameters(), 1.0)
            grads = [p.grad.clone() for p in m.parameters()]
            opt.step()
        return grads + [p.detach().clone() for p in m.parameters()]

    res = _twice(run)
    assert len(res) == 2 * 198


@pytest.mark.timeout(900)
def test_deterministic_algorithms_flag_runs_and_matches():
    """Under torch.use_deterministic_algorithms(True) (uninitialised memory filled with NaN) the bf16 step runs,
    stays finite and equals the run without the flag."""
    dev = _cuda()
    args = _inputs(dev)
    ref = _trainer_run(dev, "bf16", args)
    prev, prev_warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        got = _trainer_run(dev, "bf16", args)
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=prev_warn)
    assert all(torch.isfinite(l) for l in got[0])
    _assert_same_run(ref, got)
