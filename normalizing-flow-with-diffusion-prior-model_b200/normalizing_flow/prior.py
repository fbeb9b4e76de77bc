"""Gaussian priors with the reference's interface (normalizing_flow/prior.py:11-99).

``GaussianPrior`` keeps the ZeroConv2d(2C,2C) parameter container under the reference's mangled name
(``_GaussianPrior__conv``) so checkpoints interchange, but does not run the convolution: the reference feeds it
an all-zero map (prior.py:79-81), whose output is exactly bias*exp(3*logs) per channel, so mean / log-sd are
per-channel constants and log p(z) is a single reduction kernel (K-G).  ``save_model`` writes the reference's
checkpoint wire format (prior.py:102-115), so checkpoints travel in both directions (SURVEY §8(f) row 3).
"""
import os
from typing import Optional

import numpy as np
import torch
from torch import Tensor

from . import _engine as E
from . import _native as N
from .base import Prior
from .utils import ZeroConv2d


class IsotropicGaussian(Prior):
    """Diagonal Gaussian with explicit ``mean`` / ``logsd`` tensors (reference prior.py:20-50).  Kept for API
    compatibility; Split and GaussianPrior use fused kernels instead of constructing this object."""

    def __init__(self, mean: Tensor, logsd: Tensor):
        super().__init__()
        self.Log2PI = float(np.log(2 * np.pi))
        self.mean = mean
        self.logsd = logsd

    def compute_log_prob(self, x: Tensor) -> Tensor:
        x = E.check_input(x)
        mean, logsd = E.check_input(self.mean, "mean"), E.check_input(self.logsd, "logsd")
        if mean.shape != x.shape or logsd.shape != x.shape:
            raise ValueError("IsotropicGaussian: mean / logsd must have the shape of x")
        B = x.shape[0]
        n = x[0].numel()
        # [B, 2n] view of (mean | logsd) rows is what the split-prior kernel consumes: C=2n "channels", P=1
        h = torch.empty(B, 2 * n, dtype=torch.float32, device=x.device)
        N.copy_channels(mean, h, B, n, 1, n, 2 * n)
        N.copy_channels(logsd, h.view(-1)[n:], B, n, 1, n, 2 * n)
        xx = torch.empty(B, 2 * n, dtype=torch.float32, device=x.device)
        N.copy_channels(x, xx.view(-1)[n:], B, n, 1, n, 2 * n)
        part = torch.empty(B, dtype=torch.float32, device=x.device)
        zeros = E.WS.get("zeros2n", 2 * n, torch.float32, x.device)
        zeros.zero_()
        N.split_prior_logp(h, 2 * n, zeros, zeros, xx, 2 * n, None, part, B, 2 * n, 1, 1)
        return part

    def sample(self, shape: tuple = None, temperature: float = 1.0) -> Tensor:
        mean, logsd = E.check_input(self.mean, "mean"), E.check_input(self.logsd, "logsd")
        if E.invert_grad_enabled() and torch.is_grad_enabled() and (mean.requires_grad or logsd.requires_grad):
            from ._invgrad import IsotropicSampleFn
            return IsotropicSampleFn.apply(float(temperature), mean, logsd)
        B = mean.shape[0]
        n = mean[0].numel()
        eps = torch.empty_like(mean).normal_()
        h = torch.empty(B, 2 * n, dtype=torch.float32, device=mean.device)
        N.copy_channels(mean, h, B, n, 1, n, 2 * n)
        N.copy_channels(logsd, h.view(-1)[n:], B, n, 1, n, 2 * n)
        out2 = torch.empty(B, 2 * n, dtype=torch.float32, device=mean.device)
        zeros = E.WS.get("zeros2n", 2 * n, torch.float32, mean.device)
        zeros.zero_()
        N.split_prior_sample(h, 2 * n, zeros, zeros, eps, temperature, out2, 2 * n, B, 2 * n, 1, 1)
        out = torch.empty_like(mean)
        N.copy_channels(out2.view(-1)[n:], out, B, n, 1, 2 * n, n)
        return out


class GaussianPrior(Prior):
    """Learned per-channel Gaussian on the final latent (reference prior.py:53-99)."""

    def __init__(self, in_channels: int, learn_prior_mean_logs: bool = True):
        super().__init__()
        self.__conv = ZeroConv2d(2 * in_channels, 2 * in_channels, padding=(3 - 1) // 2) \
            if learn_prior_mean_logs else None
        if self.__conv is not None:
            self.__conv.to(self.device)
        self._C = in_channels

    def _params(self):
        c = self.__conv
        return (c.bias, c.logs) if c is not None else (None, None)

    def compute_log_prob(self, x: Tensor) -> Tensor:
        x = E.check_input(x)
        B, C, H, W = x.shape
        if C != self._C:
            raise ValueError(f"GaussianPrior built for {self._C} channels got {C}")
        bias, logs = self._params()
        if E.autograd_needed(x, self):
            from ._train import GaussianPriorFn
            weight = self.__conv.weight if self.__conv is not None else None
            return GaussianPriorFn.apply(x, weight, bias, logs)
        out = torch.empty(B, dtype=torch.float32, device=x.device)
        N.gauss_logp_const(x, bias, logs, out, B, C, H * W)
        return out

    def sample(self, shape: tuple = None, temperature: float = 1.0) -> Tensor:
        B, C, H, W = shape
        if C != self._C:
            raise ValueError(f"GaussianPrior built for {self._C} channels got {C}")
        dev = self.__conv.bias.device if self.__conv is not None else self.device
        bias, logs = self._params()
        if E.invert_grad_enabled() and bias is not None and E.autograd_needed(bias, self):
            from ._invgrad import GaussianSampleFn
            return GaussianSampleFn.apply((B, C, H, W), float(temperature), bias, logs)
        eps = torch.empty(B, C, H, W, dtype=torch.float32, device=dev).normal_()
        out = torch.empty_like(eps)
        N.gauss_sample_const(eps, bias, logs, temperature, out, B, C, H * W)
        return out


def save_model(logger_obj, model, p_dist, optim, current_epoch, current_iteration, checkpoint_directory, text=""):
    """Checkpoint writer with the reference's wire format (prior.py:102-115): one ``torch.save`` dict holding the
    flow's and the prior's ``state_dict()``, the optimiser state and the iteration counter.  With a ``GaussianPrior``
    the keys are ``flow`` / ``prior_dist`` and the file is ``model_gaussian_<epoch:03d>.pt`` (what ``NFBackbone`` and
    ``run_baseline_experiment.py:112-114`` read back); with any other prior (the diffusion prior) they are
    ``nf_backbone`` / ``diffusion_prior`` and the file is ``model_diffusion_<epoch:03d>.pt``.  Returns the path."""
    if logger_obj is not None:
        logger_obj.info(f"Saving the model. {text}")
    gaussian = isinstance(p_dist, GaussianPrior)
    names = ("flow", "prior_dist") if gaussian else ("nf_backbone", "diffusion_prior")
    path = os.path.join(checkpoint_directory,
                        f"model_{'gaussian' if gaussian else 'diffusion'}_{str(current_epoch).zfill(3)}.pt")
    torch.save({names[0]: model.state_dict(), names[1]: p_dist.state_dict(), "optimizer": optim.state_dict(),
                "current_iter": current_iteration}, path)
    return path
