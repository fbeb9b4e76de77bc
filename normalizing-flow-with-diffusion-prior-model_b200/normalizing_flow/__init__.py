"""normalizing_flow — B200-native drop-in for the Glow flow hot path of NFDPM.

Same import surface as the reference package for everything on the hot path (reference
normalizing_flow/__init__.py:8-13, :109-111): the transforms, StepFlow / GlowBlock / Glow, the priors, NFBackbone
and the step glue.  The trainers, data loaders, metrics and logging helpers of the reference are outside the hot
path; INTEGRATION.md shows how the reference tree picks this package up.
"""
from typing import Optional, Tuple

import torch
import torch.nn as nn
from torch import Tensor

from . import _native
from .glow import StepFlow, GlowBlock, Glow
from ._dp import GradAllReduce, shard, combine_init_stats
from ._optim import FusedClipAdam
from .prior import IsotropicGaussian, GaussianPrior, save_model
from .transforms import InvConv2d, ActNorm, AffineCoupling, Squeeze, Split, IdentityTransform
from .utils import (init_optimizer, preprocess_batch, postprocess_batch, initialize_with_zeros,
                    calculate_output_shapes, calculate_loss, data_dependent_nf_initialization, get_item,
                    ZeroConv2d, Conv2dActNorm, coupling_network)


class NFBackbone(nn.Module):
    """Frozen-or-trainable Glow wrapper used by the diffusion-prior experiment (reference __init__.py:16-106)."""

    def __init__(self, model_dir: str, in_channel: int, L: int, K: int, learn_prior_mean_logs: bool, freeze_flow: bool):
        super().__init__()
        self.L, self.K, self.learn_prior_mean_logs = L, K, learn_prior_mean_logs
        self.model = Glow(in_channel=in_channel, L=L, K=K, learn_prior_mean_logs=learn_prior_mean_logs)
        self.device = self.model.device
        self.model.to(self.device)
        self.freeze_flow = freeze_flow
        if model_dir:
            checkpoint = torch.load(model_dir, map_location=torch.device("cpu"))
            self.model.load_state_dict(checkpoint["flow"])
        for p in self.model.parameters():
            p.requires_grad = not self.freeze_flow

    def is_frozen(self) -> bool:
        return self.freeze_flow

    def set_train_mode(self):
        self.train() if not self.is_frozen() else self.eval()

    def set_eval_mode(self):
        self.eval()

    def transform(self, x: Tensor, log_det_jac: Tensor) -> Tuple[list, Tensor]:
        parts, log_det_jac, _ = self.model.transform(x, log_det_jac, None)
        return parts, log_det_jac

    def invert(self, latents: list, log_det_jac: Optional[Tensor] = None) -> Tensor:
        """Glow.invert; ``log_det_jac`` (optional) receives the flow's log|det dz/dx| at the returned x, as ``transform``
        would add it (the Split priors are not evaluated, as in ``transform``)."""
        return self.model.invert(latents, log_det_jac=log_det_jac)

    def invert_with_density(self, latents: list, log_det_jac: Tensor) -> Tuple[Tensor, Tensor]:
        """Glow.invert_with_density without the Split priors (as ``transform``): ``(x, log_det_jac)``, differentiable in
        both; a frozen flow still passes gradients to the latents."""
        x, log_det_jac, _ = self.model.invert_with_density(latents, log_det_jac=log_det_jac)
        return x, log_det_jac

    @torch.no_grad()
    def sample(self, latents: list, postprocess_func=None, log_det_jac: Optional[Tensor] = None) -> Tensor:
        """Glow.sample; ``log_det_jac`` as in ``invert``, at the sample before ``postprocess_func``."""
        return self.model.sample(latents, postprocess_func, log_det_jac=log_det_jac)


__all__ = ["InvConv2d", "ActNorm", "AffineCoupling", "StepFlow", "Squeeze", "Split", "GlowBlock", "Glow",
           "IsotropicGaussian", "GaussianPrior", "NFBackbone", "init_optimizer", "preprocess_batch",
           "postprocess_batch", "calculate_output_shapes", "calculate_loss", "initialize_with_zeros",
           "data_dependent_nf_initialization", "IdentityTransform", "ZeroConv2d", "Conv2dActNorm",
           "coupling_network", "get_item", "save_model", "GradAllReduce", "shard", "combine_init_stats", "FusedClipAdam"]
