"""Gradients of the fusion with respect to its inputs (LR image, expert images, expert features), in train and eval mode,
against fp64 autograd over the CPU oracle.

Losses are sums (not means), so input gradients are O(1) per element and fp16 gradients stay normal numbers."""
import math

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

import isr_b200
from isr_b200 import training as T
from oracle import fusion_oracle as O
from oracle.perturb import perturb_state_dict

pytestmark = pytest.mark.gpu

NAMES = O.EXPERT_ORDER


def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


def _rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return ((a - b).norm() / (b.norm() + 1e-30)).item()


def _cos(a, b):
    a, b = a.double().cpu().reshape(-1), b.double().cpu().reshape(-1)
    return float(a @ b / (a.norm() * b.norm() + 1e-30))


def _psnr(a, b):
    return 10 * math.log10(1.0 / float(((a.double() - b.double()) ** 2).mean()))


def _model(seed=0):
    torch.manual_seed(seed)
    m = isr_b200.CompleteEnhancedFusionSR(None)
    m.load_state_dict(perturb_state_dict(m.state_dict(), seed=7), strict=True)
    m.cross_band.band_attention.dropout = 0.0
    m.collaborative.cross_attn.dropout = 0.0
    return m


def _sd64(m):
    return {k: (v.double() if v.is_floating_point() else v.clone()) for k, v in m.state_dict().items()}


def _leaves(lr, imgs, fts, dev=None, dtype=None, which=("lr", "imgs", "fts")):
    """Copies of the inputs (on dev, in dtype) with requires_grad set on the groups named in `which`."""
    def mk(t, on):
        t = t.detach().clone()
        if dev is not None:
            t = t.to(dev)
        if dtype is not None:
            t = t.to(dtype)
        return t.requires_grad_(on)
    return (mk(lr, "lr" in which), {k: mk(v, "imgs" in which) for k, v in imgs.items()},
            {k: mk(v, "fts" in which) for k, v in fts.items()} if fts else None)


def _grads(lr, imgs, fts):
    out = {"lr": lr.grad}
    out.update({"img." + k: v.grad for k, v in imgs.items()})
    if fts:
        out.update({"feat." + k: v.grad for k, v in fts.items()})
    return out


# ------------------------------------------------------------------------------------------
# 1. Phase 2: input gradient of the nine bands (DCT / DWT adjoint kernels, FFT low-pass as its own adjoint)
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B", [1, 3])
@pytest.mark.parametrize("H,W", [(8, 8), (9, 11), (17, 23), (64, 64), (339, 510)])
def test_phase2_input_gradient_against_oracle(B, H, W):
    dev = _cuda()
    m = _model()
    with torch.no_grad():                                              # non-unit scales, perturbed FFT mask
        m.freq_decomp.dct.band_scale.copy_(torch.tensor([0.7, 1.3, 0.9]))
        m.freq_decomp.dwt.subband_scale.copy_(torch.tensor([1.1, 0.6, 1.4, 0.8]))
        m.freq_decomp.fft.band_scale.copy_(torch.tensor([1.2, 0.75]))
        m.freq_decomp.fft.freq_mask_logits.add_(torch.randn(m.freq_decomp.fft.freq_mask_logits.shape,
                                                            generator=torch.Generator().manual_seed(3)))
    sd = _sd64(m)
    g = torch.Generator().manual_seed(B * 7 + H * 31 + W)
    x = torch.rand(B, 3, H, W, generator=g)
    G = torch.randn(B, 9, 3, H, W, generator=g)
    x64 = x.double().requires_grad_()
    bands = O.decompose9(sd, x64)
    torch.autograd.backward(bands, list(G.double().unbind(1)))
    m.to(dev)
    xd = x.to(dev).requires_grad_()
    with torch.cuda.device(dev):
        raw9 = T._phase2_train(m, xd)
        (raw9 * G.to(dev)).sum().backward()
    torch.cuda.synchronize()
    assert _rel(xd.grad, x64.grad) <= 1e-5
    # dot-product test on the kernels' own forward and adjoint: <A x, g> = <x, A^T g>, fp64 sums
    lhs = (raw9.detach().double() * G.to(dev).double()).sum().item()
    rhs = (xd.detach().double() * xd.grad.double()).sum().item()
    scale = raw9.detach().double().norm().item() * G.double().norm().item()
    assert abs(lhs - rhs) <= 1e-6 * scale, (lhs, rhs)


# ------------------------------------------------------------------------------------------
# 2. train mode, fp32: every input gradient against fp64 autograd of the oracle
# ------------------------------------------------------------------------------------------
def _variant(name):
    """-> (B, H, W, lr, imgs, fts, dtype, which)"""
    shapes = {"12x12": (2, 12, 12, True), "17x23": (1, 17, 23, True), "9x11_nofeat": (2, 9, 11, False)}
    B, H, W, feats = shapes.get(name, (2, 12, 12, True))
    lr, imgs, fts, _ = O.synthetic_inputs(B, H, W, feats=feats)
    dtype, which = None, ("lr", "imgs", "fts")
    g = torch.Generator().manual_seed(11)
    if name == "partial":                          # two of the four experts have features; lr needs no gradient
        fts = {k: fts[k] for k in ("grl", "nafnet")}
        which = ("imgs", "fts")
    elif name == "small_grid":                     # features at a coarser grid than LR (resized to the smallest)
        fts = {k: F.interpolate(v, size=(H // 2, W // 2 + 1), mode="bilinear", align_corners=False) for k, v in fts.items()}
        fts["mamba"] = torch.randn(B, 180, 8, 9, generator=g)
    elif name == "channels":                       # above and below the align width: truncated / zero-padded
        fts["drct"] = torch.randn(B, 200, H, W, generator=g)
        fts["nafnet"] = torch.randn(B, 40, H, W, generator=g)
    elif name == "fp16":
        dtype = torch.float16
        lr, imgs, fts = lr.half(), {k: v.half() for k, v in imgs.items()}, {k: v.half() for k, v in fts.items()}
    return B, H, W, lr, imgs, fts, dtype, which


@pytest.mark.parametrize("name", ["12x12", "17x23", "9x11_nofeat", "partial", "small_grid", "channels", "fp16"])
def test_train_input_gradients_match_oracle(name):
    dev = _cuda()
    B, H, W, lr, imgs, fts, dtype, which = _variant(name)
    m = _model().train()
    sd = _sd64(m)
    hr = torch.rand(B, 3, 4 * H, 4 * W, generator=torch.Generator().manual_seed(5))
    r_lr, r_imgs, r_fts = _leaves(lr, imgs, fts, dtype=torch.float64, which=which)
    ref = O.run_pipeline(sd, r_lr, r_imgs, r_fts, training=True, bn_updates={})
    ((ref - hr.double()) ** 2).sum().backward()
    m.to(dev)
    d_lr, d_imgs, d_fts = _leaves(lr, imgs, fts, dev=dev, which=which)
    out = m.forward_with_precomputed(d_lr, d_imgs, d_fts)
    ((out - hr.to(dev)) ** 2).sum().backward()
    torch.cuda.synchronize()
    assert (out.detach().cpu() - ref.detach()).abs().max().item() <= 1e-4
    got, want = _grads(d_lr, d_imgs, d_fts), _grads(r_lr, r_imgs, r_fts)
    tol = 2e-3 if dtype == torch.float16 else 1e-4                   # fp16: the rounding of the gradient itself
    for k, gr in want.items():
        if gr is None:
            assert got[k] is None, f"{k}: gradient although the input does not require grad"
            continue
        assert got[k] is not None, f"{k}: no gradient"
        assert got[k].dtype == (dtype or torch.float32) and got[k].shape == gr.shape, k
        assert _rel(got[k], gr) <= tol, f"{k}: rel-L2 {_rel(got[k], gr):.3e}"


# ------------------------------------------------------------------------------------------
# 3. bf16 mode: input gradients close to the fp32 oracle
# ------------------------------------------------------------------------------------------
def test_train_bf16_input_gradients_close_to_fp32_oracle():
    dev = _cuda()
    B, H, W = 2, 16, 16
    lr, imgs, fts, hr = O.synthetic_inputs(B, H, W)
    m = _model().train()
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    r = _leaves(lr, imgs, fts)
    ref = O.run_pipeline(sd, *r, training=True, bn_updates={})
    (ref - hr).abs().sum().backward()
    m.to(dev)
    m.precision = "bf16"
    d = _leaves(lr, imgs, fts, dev=dev)
    out = m.forward_with_precomputed(*d)
    (out - hr.to(dev)).abs().sum().backward()
    want, got = _grads(*r), _grads(*d)
    bad = {k: _cos(got[k], want[k]) for k in want if _cos(got[k], want[k]) < 0.99}
    assert not bad, bad


# ------------------------------------------------------------------------------------------
# 4. eval mode with an input that requires grad: the differentiable path with eval semantics
# ------------------------------------------------------------------------------------------
def test_eval_input_gradients_match_oracle_and_leave_bn_buffers():
    dev = _cuda()
    B, H, W = 2, 12, 12
    lr, imgs, fts, hr = O.synthetic_inputs(B, H, W)
    m = _model().eval()
    sd = _sd64(m)
    r = _leaves(lr, imgs, fts, dtype=torch.float64)
    ref = O.run_pipeline(sd, *r, training=False)
    ((ref - hr.double()) ** 2).sum().backward()
    m.to(dev)
    buf0 = {k: v.clone() for k, v in m.state_dict().items() if "running_" in k or "num_batches" in k}
    outs, grads = [], []
    for _ in range(2):
        d = _leaves(lr, imgs, fts, dev=dev)
        out = m.forward_with_precomputed(*d)
        assert out.grad_fn is not None
        ((out - hr.to(dev)) ** 2).sum().backward()
        outs.append(out.detach().clone())
        grads.append(_grads(*d))
    torch.cuda.synchronize()
    assert (outs[0].cpu() - ref.detach().float()).abs().max().item() <= 1e-4
    want = _grads(*r)
    for k in want:
        assert _rel(grads[0][k], want[k]) <= 1e-4, f"{k}: rel-L2 {_rel(grads[0][k], want[k]):.3e}"
        assert torch.equal(grads[0][k], grads[1][k]), f"{k}: two calls differ"
    assert torch.equal(outs[0], outs[1])
    after = m.state_dict()
    for k, v in buf0.items():
        assert torch.equal(after[k], v), f"{k} changed in eval mode"
    # no input requires grad: the inference engine, output without grad_fn, as before
    out = m.forward_with_precomputed(*_leaves(lr, imgs, fts, dev=dev, which=()))
    assert out.grad_fn is None


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_eval_with_input_grad_keeps_inference_indices_and_quality(prec):
    """64x64 LR, realistic experts: output against the eval oracle (fp32 1e-4 max-abs; bf16 0.01 dB PSNR) and 0 flips of
    the derived expert-selection indices."""
    dev = _cuda()
    B, H, W = 1, 64, 64
    lr, imgs, fts, _ = O.synthetic_inputs(B, H, W)
    g = torch.Generator().manual_seed(77)
    up = F.interpolate(lr, scale_factor=4, mode="bicubic", align_corners=False)
    imgs = {k: (up + 0.02 * torch.randn(up.shape, generator=g)).clamp(0, 1) for k in NAMES}
    hr = (up + 0.01 * torch.randn(up.shape, generator=g)).clamp(0, 1)
    m = _model().eval()
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    with torch.no_grad():
        ref, rint = O.run_pipeline(sd, lr, imgs, fts, return_intermediates=True)
        top1, active = O.derived_indices(sd, rint["routing_lr"], rint["gates"])
    m.to(dev)
    m.precision = prec
    d = _leaves(lr, imgs, fts, dev=dev, which=("lr",))
    sr, ints = m._run_pipeline(d[0], [d[1][k] for k in NAMES], d[2], 4 * H, 4 * W, {}, True)
    assert sr.grad_fn is not None
    sr.sum().backward()
    assert d[0].grad is not None and torch.isfinite(d[0].grad).all()
    sr = sr.detach().cpu()
    if prec == "fp32":
        assert (sr - ref).abs().max().item() <= 1e-4
    else:
        assert abs(_psnr(sr, hr) - _psnr(ref, hr)) <= 0.01
    flips = (ints["gates"].detach().cpu().argmax(1) != top1).sum().item()
    aflips = (ints["active"].cpu() != active).sum().item()
    assert flips == 0 and aflips == 0, f"{flips} top-1 flips, {aflips} active flips"


# ------------------------------------------------------------------------------------------
# 5. / 6. no side effects on the parameter graph; reproducible input gradients
# ------------------------------------------------------------------------------------------
def test_input_grad_leaves_the_train_step_bitwise_unchanged():
    dev = _cuda()
    lr, imgs, fts, hr = O.synthetic_inputs(2, 16, 16)
    m = _model().train().to(dev)
    sd0 = {k: v.clone() for k, v in m.state_dict().items()}
    res = []
    for which in ((), ("lr", "imgs", "fts")):
        m.load_state_dict(sd0)
        m.zero_grad(set_to_none=True)
        out = m.forward_with_precomputed(*_leaves(lr, imgs, fts, dev=dev, which=which))
        (out - hr.to(dev)).abs().mean().backward()
        res.append((out.detach().clone(), {n: p.grad.clone() for n, p in m.named_parameters()},
                    {k: v.clone() for k, v in m.state_dict().items() if "running_" in k or "num_batches" in k}))
    (o0, g0, b0), (o1, g1, b1) = res
    assert torch.equal(o0, o1)
    assert len(g0) == 198 and all(torch.equal(g0[n], g1[n]) for n in g0), [n for n in g0 if not torch.equal(g0[n], g1[n])]
    assert all(torch.equal(b0[k], b1[k]) for k in b0)


@pytest.mark.parametrize("deterministic", [False, True])
def test_input_gradients_are_bitwise_reproducible(deterministic):
    dev = _cuda()
    lr, imgs, fts, hr = O.synthetic_inputs(2, 16, 16)
    m = _model().train().to(dev)
    sd0 = {k: v.clone() for k, v in m.state_dict().items()}
    prev = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(deterministic)
    try:
        runs = []
        for _ in range(2):
            m.load_state_dict(sd0)
            d = _leaves(lr, imgs, fts, dev=dev)
            (m.forward_with_precomputed(*d) - hr.to(dev)).abs().sum().backward()
            runs.append(_grads(*d))
    finally:
        torch.use_deterministic_algorithms(prev)
    for k in runs[0]:
        assert torch.equal(runs[0][k], runs[1][k]), k


# ------------------------------------------------------------------------------------------
# 7. full size: directional derivative of the kernels' own forward along the input gradient
# ------------------------------------------------------------------------------------------
def _directional_check(m, lr, imgs, fts, hr, eps):
    sd0 = {k: v.clone() for k, v in m.state_dict().items()}

    def loss(d):
        m.load_state_dict(sd0)
        return (m.forward_with_precomputed(*d).double() - hr.double()).abs().sum()

    d = _leaves(lr, imgs, fts)
    loss(d).backward()
    leaves = [d[0], *d[1].values(), *d[2].values()]
    grads = [t.grad.detach().clone() for t in leaves]
    gnorm = math.sqrt(sum(float((g.double() ** 2).sum()) for g in grads))
    assert gnorm > 0
    vals = []
    with torch.no_grad():
        for sgn in (1.0, -1.0):
            sh = [(t + g * (sgn * eps / gnorm)).detach() for t, g in zip(leaves, grads)]
            k = iter(sh[1:])
            vals.append(float(loss((sh[0], {n: next(k) for n in d[1]}, {n: next(k) for n in d[2]}))))
    fd = (vals[0] - vals[1]) / (2 * eps)
    assert abs(fd - gnorm) <= 0.03 * gnorm, (fd, gnorm)


def test_full_patch_size_input_directional_derivative():
    dev = _cuda()
    lr, imgs, fts, hr = O.synthetic_inputs(4, 64, 64)
    m = _model().train().to(dev)
    to = lambda t: t.to(dev)
    _directional_check(m, to(lr), {k: to(v) for k, v in imgs.items()}, {k: to(v) for k, v in fts.items()}, to(hr), 0.05)


@pytest.mark.timeout(900)
def test_c3_eval_attribution_pass_and_directional_derivative():
    dev = _cuda()
    lr, imgs, fts, hr = O.synthetic_inputs(1, 339, 510)
    m = _model().eval().to(dev)
    to = lambda t: t.to(dev)
    _directional_check(m, to(lr), {k: to(v) for k, v in imgs.items()}, {k: to(v) for k, v in fts.items()}, to(hr), 0.05)


# ------------------------------------------------------------------------------------------
# 8. live path: a trainable expert ensemble learns through model.forward(lr)
# ------------------------------------------------------------------------------------------
class _TinyEnsemble(nn.Module):
    """Bilinear x4 + a learnable 1x1 conv per expert image, a learnable 1x1 conv per expert feature map."""

    def __init__(self):
        super().__init__()
        self.img = nn.ModuleDict({k: nn.Conv2d(3, 3, 1) for k in NAMES})
        self.feat = nn.ModuleDict({k: nn.Conv2d(3, 64 if k == "nafnet" else 180, 1) for k in NAMES})

    def forward_all_with_hooks(self, lr):
        up = F.interpolate(lr, scale_factor=4, mode="bilinear", align_corners=False)
        return {k: self.img[k](up) for k in NAMES}, {k: self.feat[k](lr) for k in NAMES}


@pytest.mark.parametrize("mode", ["train", "eval"])
def test_live_forward_trains_an_expert_ensemble(mode):
    dev = _cuda()
    torch.manual_seed(0)
    ens = _TinyEnsemble()
    with torch.no_grad():
        for mod in ens.img.values():
            mod.weight.copy_(torch.eye(3)[:, :, None, None] + 0.05 * torch.randn(3, 3, 1, 1))
            mod.bias.mul_(0.1)
    m = isr_b200.CompleteEnhancedFusionSR(ens)
    ref_m = _model()
    m.load_state_dict({**m.state_dict(), **ref_m.state_dict()})
    m.cross_band.band_attention.dropout = 0.0
    m.collaborative.cross_attn.dropout = 0.0
    for p in ens.parameters():
        p.requires_grad_(True)                                         # the constructor froze the experts
    m.train(mode == "train")
    B, H, W = 1, 12, 12
    lr, _, _, hr = O.synthetic_inputs(B, H, W)
    ens64 = _TinyEnsemble().double()
    ens64.load_state_dict(ens.state_dict())
    sd = {k: v for k, v in _sd64(m).items() if not k.startswith("expert_ensemble.")}
    outs, feats = ens64.forward_all_with_hooks(lr.double())
    ref = O.run_pipeline(sd, lr.double(), outs, feats, training=(mode == "train"), bn_updates={})
    ((ref - hr.double()) ** 2).sum().backward()
    m.to(dev)
    out = m(lr.to(dev))
    ((out - hr.to(dev)) ** 2).sum().backward()
    torch.cuda.synchronize()
    ref_g = dict(ens64.named_parameters())
    for n, p in ens.named_parameters():
        assert p.grad is not None, n
        assert _rel(p.grad, ref_g[n].grad) <= 1e-4, f"{n}: rel-L2 {_rel(p.grad, ref_g[n].grad):.3e}"
