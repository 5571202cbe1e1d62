"""Drop-in ``CompleteEnhancedFusionSR`` backed by hand-written sm_100a kernels.

Replaces ``src.models.enhanced_fusion_v2`` of the reference
(enhanced_fusion_v2.py:473-870): same constructor, same
``forward_with_precomputed(lr_input, expert_imgs, expert_feats)`` signature, same
226-entry ``state_dict`` (SURVEY.md Appendix B / §8b).  All arithmetic runs in
``libffsr_b200.so`` (C-ABI declared in ``include/ffsr_b200.h``); there is no CPU
or PyTorch-eager fallback: without the CUDA library or a CUDA device the forward
raises.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Tuple, Union

import torch
import torch.nn as nn

from .modules import (Collaborative, CrossBand, DynamicExpertSelector, FrequencyBands,
                      HierarchicalFusion, LaplacianEdge)

EXPERT_ORDER = ("drct", "grl", "nafnet", "mamba")


class CompleteEnhancedFusionSR(nn.Module):
    """7-phase expert fusion over cached expert outputs (phases 2-7 on the GPU).

    ``precision``: ``"fp32"`` (FFMA kernels everywhere, <=1e-4 max-abs of the
    reference) or ``"bf16"`` (tcgen05 tensor-core kernels for the contraction-heavy
    phases 4/5/7, fp32 for phases 2/3/6 so derived gate indices stay bit-exact).
    It is an attribute, not a constructor argument, so the constructor stays
    byte-compatible with the reference's call sites (train.py:693-709,
    models/team29_FreqFusionSR/io.py:179-194).
    """

    def __init__(self, expert_ensemble, num_experts: int = 4, fusion_dim: int = 128,
                 refine_channels: int = 128, refine_depth: int = 6, base_channels: int = 64,
                 block_size: int = 8, upscale: int = 4,
                 enable_dynamic_selection: bool = True, enable_cross_band_attn: bool = True,
                 enable_adaptive_bands: bool = True, enable_multi_resolution: bool = True,
                 enable_collaborative: bool = True, enable_edge_enhance: bool = True):
        super().__init__()
        self.expert_ensemble = expert_ensemble
        self.cached_mode = expert_ensemble is None
        self.num_experts = num_experts
        self.upscale = upscale
        self.enable_dynamic_selection = enable_dynamic_selection
        self.enable_cross_band_attn = enable_cross_band_attn
        self.enable_adaptive_bands = enable_adaptive_bands
        self.enable_multi_resolution = enable_multi_resolution
        self.enable_collaborative = enable_collaborative
        self.enable_edge_enhance = enable_edge_enhance
        self.precision = "fp32"

        if expert_ensemble is not None:
            for p in self.expert_ensemble.parameters():
                p.requires_grad = False

        # construction order == reference order (enhanced_fusion_v2.py:526-583): the
        # RNG is consumed identically, so manual_seed(s) gives bit-identical weights.
        if enable_adaptive_bands:
            self.freq_decomp = FrequencyBands(block_size, 3, 64)
        if enable_cross_band_attn:
            self.cross_band = CrossBand(64, 9, 4, 21)
        if enable_collaborative:
            self.collaborative = Collaborative(num_experts, fusion_dim, 8, 21)
        if enable_multi_resolution:
            self.multi_res = HierarchicalFusion(num_experts, base_channels)
            self.freq_weight_conv = nn.Sequential(nn.Conv2d(3, 16, 1), nn.GELU(), nn.Conv2d(16, num_experts, 1))
        else:
            self.simple_fusion = nn.Conv2d(num_experts * 3, 3, 1)
        if enable_dynamic_selection:
            self.dynamic_selector = DynamicExpertSelector(3, 32, num_experts)
        layers: List[nn.Module] = [nn.Conv2d(3, refine_channels, 3, 1, 1), nn.GELU()]
        for _ in range(refine_depth - 2):
            layers += [nn.Conv2d(refine_channels, refine_channels, 3, 1, 1), nn.GELU()]
        layers.append(nn.Conv2d(refine_channels, 3, 3, 1, 1))
        self.refine = nn.Sequential(*layers)
        self.residual_scale = nn.Parameter(torch.tensor(0.1))
        if enable_edge_enhance:
            self.edge_enhance = LaplacianEdge(3, 32, 0.15)

        self._all_on = all((enable_dynamic_selection, enable_cross_band_attn, enable_adaptive_bands,
                            enable_multi_resolution, enable_collaborative, enable_edge_enhance)) \
            and num_experts == 4 and upscale == 4 and block_size == 8 and fusion_dim == 128 \
            and base_channels == 64 and refine_depth >= 3
        self._engine = None

    # ------------------------------------------------------------------ forward
    def forward(self, lr_input: torch.Tensor, return_intermediates: bool = False):
        """Live-expert path (enhanced_fusion_v2.py:589-636)."""
        if self.cached_mode:
            raise RuntimeError("Cannot call forward() in cached mode (expert_ensemble=None). "
                               "Use forward_with_precomputed() instead.")
        outs, feats = self.expert_ensemble.forward_all_with_hooks(lr_input)
        names = list(outs.keys())
        H, W = lr_input.shape[2] * self.upscale, lr_input.shape[3] * self.upscale
        inter: Dict = {}
        if return_intermediates:
            inter["expert_outputs"], inter["expert_features"] = outs, feats
        return self._run_pipeline(lr_input, [outs[n] for n in names], feats, H, W, inter, return_intermediates)

    def forward_with_precomputed(self, lr_input: torch.Tensor, expert_imgs: Dict[str, torch.Tensor],
                                 expert_feats: Optional[Dict[str, torch.Tensor]] = None) -> torch.Tensor:
        """Cached-expert path (enhanced_fusion_v2.py:642-675): dict order is normalised to
        drct, grl, nafnet, mamba; missing feature entries are tolerated."""
        H, W = lr_input.shape[2] * self.upscale, lr_input.shape[3] * self.upscale
        img_list = [expert_imgs[k] for k in EXPERT_ORDER if k in expert_imgs]
        feats = {k: expert_feats[k] for k in EXPERT_ORDER if k in expert_feats} if expert_feats is not None else {}
        return self._run_pipeline(lr_input, img_list, feats, H, W, {}, False)

    def _run_pipeline(self, lr_input: torch.Tensor, expert_output_list: List[torch.Tensor],
                      expert_features: Dict[str, torch.Tensor], H_hr: int, W_hr: int,
                      intermediates: Dict, return_intermediates: bool
                      ) -> Union[torch.Tensor, Tuple[torch.Tensor, Dict]]:
        """Phases 2-7 (enhanced_fusion_v2.py:681-799) on the GPU."""
        if not self._all_on:
            raise NotImplementedError(
                "the sm_100a path implements the all-phases-on 4-expert x4 configuration "
                "(configs/train_config.yaml:63-80); other flag combinations are not built")
        wants_input_grad = torch.is_grad_enabled() and any(
            t.requires_grad for t in (lr_input, *expert_output_list, *expert_features.values()))
        if self.training or wants_input_grad:
            # train mode: differentiable graph of library kernels (BN batch statistics, attention
            # dropout, no output clamps) -- train.py:331-357 calls this under autograd.  Eval mode with an input that
            # requires grad (gradient attribution, an upstream module learning through the fusion): the same graph
            # with eval semantics (BN running statistics, no dropout, the eval clamps)
            from .training import train_forward
            sr, inter = train_forward(self, lr_input, expert_output_list, expert_features, return_intermediates)
            if return_intermediates:
                intermediates.update(inter)
                return sr, intermediates
            return sr
        from .pipeline import FusionEngine
        if self._engine is None:
            self._engine = FusionEngine(self)
        sr, inter = self._engine.forward(lr_input, expert_output_list, expert_features,
                                         H_hr, W_hr, return_intermediates)
        if return_intermediates:
            intermediates.update(inter)
            return sr, intermediates
        return sr

    # ---------------------------------------------------------------- utilities
    def get_trainable_params(self) -> int:
        return sum(p.numel() for p in self.parameters() if p.requires_grad)

    def get_frozen_params(self) -> int:
        return sum(p.numel() for p in self.expert_ensemble.parameters()) if self.expert_ensemble is not None else 0

    def get_improvement_status(self) -> Dict[str, bool]:
        return {
            "dynamic_expert_selection": self.enable_dynamic_selection,
            "cross_band_attention": self.enable_cross_band_attn,
            "adaptive_frequency_bands": self.enable_adaptive_bands,
            "multi_resolution_fusion": self.enable_multi_resolution,
            "collaborative_learning": self.enable_collaborative,
            "edge_enhancement": self.enable_edge_enhance,
        }

    def __repr__(self) -> str:
        return (f"CompleteEnhancedFusionSR(num_experts={self.num_experts}, "
                f"trainable={self.get_trainable_params():,}, frozen={self.get_frozen_params():,})")


def create_enhanced_fusion(expert_ensemble, config: Optional[Dict] = None) -> CompleteEnhancedFusionSR:
    """Factory with dict overrides (enhanced_fusion_v2.py:836-870)."""
    cfg = dict(num_experts=4, fusion_dim=128, refine_channels=128, refine_depth=6, base_channels=64,
               block_size=8, upscale=4, enable_dynamic_selection=True, enable_cross_band_attn=True,
               enable_adaptive_bands=True, enable_multi_resolution=True, enable_collaborative=True,
               enable_edge_enhance=True)
    if config:
        cfg.update(config)
    return CompleteEnhancedFusionSR(expert_ensemble=expert_ensemble, **cfg)
