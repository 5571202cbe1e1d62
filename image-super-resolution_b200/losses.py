"""Fused training losses on the sm_100a kernels: drop-in for the ``src.losses`` names the
training loop uses (``from src.losses import CombinedLoss, PYWT_AVAILABLE``, train.py:549,
817-830; ``CombinedLoss(**weights)``, ``.set_weights(dict)``, ``.weights``,
``forward(pred, target, return_components)`` -- src/losses/perceptual_loss.py:1077-1284).

One autograd node evaluates every active component AND d(total)/d(pred) in the same passes over
the data (``ffsr_loss_l1 / _swt / _ssim / _fft``), so ``loss.backward()`` only scales a stored
gradient.  Components whose weight is 0 are not evaluated (the reference is weight-driven the
same way).  Components outside the stage-1/2/3 curriculum of ``configs/train_config.yaml:140-175``
(charbonnier, l2, vgg, edge, clip) are not built: a positive weight for one of them raises.
There is no CPU path.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Tuple, Union

import torch
import torch.nn as nn

from . import _cabi as K

PYWT_AVAILABLE = True          # the Haar taps are compiled in; PyWavelets is not needed
LPIPS_AVAILABLE = False
CLIP_AVAILABLE = False
_BUILT = ("l1", "swt", "fft", "ssim")
_SWT_BANDS = (0.5, 1.5, 1.5, 2.0)
_SWT_LEVELS = 2


def _S(t):
    return C.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


_CONSTS: Dict = {}


def _const(dev, name, values, dtype):
    """Small device constants, cached so that no host->device copy happens inside a CUDA-graph capture."""
    key = (str(dev), name, tuple(values), dtype)
    t = _CONSTS.get(key)
    if t is None:
        t = _CONSTS[key] = torch.tensor(list(values), device=dev, dtype=dtype)
    return t


class _FusedLosses(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pred, target, w_l1, w_swt, w_fft, w_ssim):
        if not pred.is_cuda:
            raise RuntimeError("fused losses (sm_100a build) need CUDA tensors: there is no CPU path")
        lib = K.load()
        p = pred.detach().float().contiguous()
        t = target.detach().float().contiguous()
        if p.shape != t.shape or p.dim() != 4:
            raise ValueError(f"pred {tuple(pred.shape)} and target {tuple(target.shape)} must be equal [B,C,H,W]")
        B, Cc, H, W = p.shape
        P, n = B * Cc, p.numel()
        dev = p.device
        dpred = torch.zeros_like(p)
        sums = torch.zeros(16, device=dev, dtype=torch.float64)   # l1 | swt x8 | ssim | fft x2
        S = _S(p)
        with torch.cuda.device(dev):
            if w_l1 > 0:
                nb = lib.ffsr_loss_l1_workspace_bytes(n)
                ws = torch.empty(nb, device=dev, dtype=torch.uint8)
                K.check(lib.ffsr_loss_l1(p.data_ptr(), t.data_ptr(), n, w_l1 / n, sums.data_ptr(), ws.data_ptr(), nb,
                                         dpred.data_ptr(), S), "loss_l1")
            if w_swt > 0:
                nb = lib.ffsr_loss_swt_workspace_bytes(P, H, W)
                ws = torch.empty(nb, device=dev, dtype=torch.uint8)
                K.check(lib.ffsr_loss_swt(p.data_ptr(), t.data_ptr(), P, H, W, w_swt / (n * _SWT_LEVELS),
                                          sums.data_ptr() + 8, ws.data_ptr(), nb, dpred.data_ptr(), S), "loss_swt")
            if w_ssim > 0:
                nb = lib.ffsr_loss_ssim_workspace_bytes(P, H, W)
                ws = torch.empty(nb, device=dev, dtype=torch.uint8)
                K.check(lib.ffsr_loss_ssim(p.data_ptr(), t.data_ptr(), P, H, W, w_ssim / n, sums.data_ptr() + 9 * 8,
                                           ws.data_ptr(), nb, dpred.data_ptr(), S), "loss_ssim")
            if w_fft > 0:
                nb = lib.ffsr_loss_fft_workspace_bytes(P, H, W)
                ws = torch.empty(nb, device=dev, dtype=torch.uint8)
                K.check(lib.ffsr_loss_fft(p.data_ptr(), t.data_ptr(), P, H, W, w_fft / n, sums.data_ptr() + 10 * 8,
                                          ws.data_ptr(), nb, dpred.data_ptr(), S), "loss_fft")
        bw = _const(dev, "swt_bands", _SWT_BANDS * _SWT_LEVELS, torch.float64)
        l1 = sums[0] / n
        swt = (sums[1:9] * bw).sum() / (n * _SWT_LEVELS)
        ssim = 1.0 - sums[9] / n
        fft = (sums[10] + 0.1 * sums[11]) / n
        comps = torch.stack([l1, swt, fft, ssim]).float()
        wts = _const(dev, "weights", (w_l1, w_swt, w_fft, w_ssim), torch.float32)
        total = (comps * wts).sum()
        ctx.save_for_backward(dpred)
        ctx.pred_dtype = pred.dtype
        ctx.mark_non_differentiable(comps)
        return total, comps

    @staticmethod
    def backward(ctx, g_total, _g_comps):
        (dpred,) = ctx.saved_tensors
        return (dpred * g_total).to(ctx.pred_dtype), None, None, None, None, None


def fused_losses(pred, target, weights: Dict[str, float]):
    """(total, {name: value}) for the active components among l1 / swt / fft / ssim."""
    w = {k: float(weights.get(k, 0.0) or 0.0) for k in _BUILT}
    total, comps = _FusedLosses.apply(pred, target, max(w["l1"], 0.0), max(w["swt"], 0.0), max(w["fft"], 0.0),
                                      max(w["ssim"], 0.0))
    out = {}
    for i, name in enumerate(("l1", "swt", "fft", "ssim")):
        if w[name] > 0:
            out[name] = comps[i]
    return total, out


class _Single(nn.Module):
    name = ""

    def forward(self, pred, target):
        return fused_losses(pred, target, {self.name: 1.0})[0]


class L1Loss(_Single):
    """perceptual_loss.py:86-104 (mean reduction)."""
    name = "l1"


class SSIMLoss(_Single):
    """perceptual_loss.py:205-291 (window 11, mean reduction)."""
    name = "ssim"


class FFTLoss(_Single):
    """perceptual_loss.py:505-598 (loss_type l1, focus_high_freq, high_freq_weight 2)."""
    name = "fft"

    def __init__(self, loss_type: str = "l1", focus_high_freq: bool = True, high_freq_weight: float = 2.0):
        super().__init__()
        if loss_type != "l1" or not focus_high_freq or high_freq_weight != 2.0:
            raise NotImplementedError("the fused FFT loss implements the configuration CombinedLoss uses "
                                      "(l1, focus_high_freq=True, high_freq_weight=2.0)")


class SWTLoss(_Single):
    """perceptual_loss.py:604-813 (haar, level 2, GPU approximation path)."""
    name = "swt"

    def __init__(self, wavelet: str = "haar", level: int = 2, band_weights=None, use_gpu_approximation: bool = True):
        super().__init__()
        if wavelet not in ("haar", "db1") or level != 2 or band_weights is not None or not use_gpu_approximation:
            raise NotImplementedError("the fused SWT loss implements the configuration CombinedLoss hard-codes "
                                      "(haar, level=2, default band weights, use_gpu_approximation=True)")


class CombinedLoss(nn.Module):
    """Weight-driven combination with the reference's constructor and methods
    (perceptual_loss.py:1053-1300).  VGG19 is NOT constructed (the reference downloads it eagerly,
    :1122-1125, which cannot work offline); asking for it through a positive weight raises."""

    def __init__(self, l1_weight: float = 1.0, charbonnier_weight: float = 0.5, l2_weight: float = 0.5,
                 vgg_weight: float = 0.1, swt_weight: float = 0.2, fft_weight: float = 0.15,
                 edge_weight: float = 0.1, ssim_weight: float = 0.1, clip_weight: float = 0.0,
                 use_swt: bool = True, use_fft: bool = True, use_clip: bool = False, clip_threshold: float = 0.5):
        super().__init__()
        self.weights = {"l1": l1_weight, "charbonnier": charbonnier_weight, "l2": l2_weight, "vgg": vgg_weight,
                        "swt": swt_weight, "fft": fft_weight, "edge": edge_weight, "ssim": ssim_weight,
                        "clip": clip_weight}
        self.use_swt, self.use_fft, self.use_clip = use_swt, use_fft, False
        self.current_stage = 1

    def set_stage(self, stage: int):
        self.current_stage = stage

    def set_weights(self, weights: Dict[str, float]):
        for name, w in weights.items():
            self.weights[name] = w
        if self.weights.get("swt", 0) > 0 or self.weights.get("fft", 0) > 0:
            self.current_stage = 3
        elif self.weights.get("vgg", 0) > 0 or self.weights.get("ssim", 0) > 0:
            self.current_stage = 2
        else:
            self.current_stage = 1

    def get_active_weights(self) -> Dict[str, float]:
        return {k: v for k, v in self.weights.items() if v > 0}

    def get_loss_info(self) -> Dict:
        return {"weights": self.weights, "current_stage": self.current_stage, "use_swt": self.use_swt,
                "use_fft": self.use_fft, "use_clip": self.use_clip,
                "available_losses": ["l1", "ssim", "fft" if self.use_fft else None, "swt" if self.use_swt else None]}

    def forward(self, pred: torch.Tensor, target: torch.Tensor, return_components: bool = False
                ) -> Union[torch.Tensor, Tuple[torch.Tensor, Dict[str, torch.Tensor]]]:
        unbuilt = [k for k, v in self.weights.items() if v and v > 0 and k not in _BUILT]
        if unbuilt:
            raise NotImplementedError(f"loss components {unbuilt} are not built in the sm_100a fused-loss path "
                                      f"(built: {list(_BUILT)}); set their weights to 0 as the stage-1/2/3 "
                                      "curriculum of configs/train_config.yaml does")
        w = dict(self.weights)
        if not self.use_swt:
            w["swt"] = 0.0
        if not self.use_fft:
            w["fft"] = 0.0
        total, comps = fused_losses(pred, target, w)
        return (total, comps) if return_components else total
