"""Primitive invertible transforms, API-compatible with the reference's normalizing_flow/transforms.py
(ActNorm :28-94, InvConv2d :97-145, AffineCoupling :148-201, Squeeze :204-239, Split :242-309), executed by
the sm_100a kernels of libnfdpm_b200 instead of ATen/cuDNN op chains.

Shared semantics kept from the reference: ``transform(x, log_det_jac, logp)`` adds into both accumulators IN
PLACE (any of fp32/fp64) and returns them; inputs are NCHW fp32; outputs are fresh NCHW fp32 tensors.
"""
from typing import Optional, Tuple

import torch
import torch.nn as nn
from torch import Tensor

from . import _engine as E
from . import _native as N
from .base import Transform
from .utils import ZeroConv2d, coupling_network


class _NoBackward(torch.autograd.Function):
    """Identity whose backward raises.  ``transform`` of the granular modules (ActNorm, InvConv2d, AffineCoupling, Squeeze,
    Split — and StepFlow / GlowBlock, which compose them) is differentiable through normalizing_flow/_modgrad.py; ``invert``
    is differentiable only with NFDPM_INVERT_GRAD=1 (the reference inverts under ``torch.no_grad()``: sampling and decoding); without it its forward
    runs in any grad mode — the reference's own unit tests call it with autograd enabled (tests/transformations.py) —
    and back-propagating through it fails loudly instead of silently dropping gradients."""

    @staticmethod
    def forward(ctx, t, what, inplace, *deps):
        ctx.what = what
        if inplace:
            ctx.mark_dirty(t)
            return t
        return t.view_as(t)

    @staticmethod
    def backward(ctx, g):
        raise NotImplementedError(
            f"{ctx.what}: backward through invert() is not implemented (the reference inverts under torch.no_grad(): "
            f"sampling and decoding); transform() is differentiable.")


def _no_autograd(x: Tensor, mod: nn.Module, what: str) -> None:
    if E.autograd_needed(x, mod):
        raise NotImplementedError(
            f"{what}: not available under autograd; call under torch.no_grad().")


def _granular(what: str):
    """Decorator for stand-alone transform / invert methods.  Without autograd: the kernels, nothing recorded.  Under
    autograd ``transform`` goes through the module's autograd Function (normalizing_flow/_modgrad.py; StepFlow composes its
    three parts); ``invert`` does the same with ``NFDPM_INVERT_GRAD=1`` and otherwise runs the kernels without recording
    and attaches the loud-failure node to its result."""
    def deco(fn):
        def wrapper(self, x, *args, **kw):
            latent_grad = fn.__name__ == "invert" and E.invert_grad_enabled() and torch.is_grad_enabled() and \
                any(isinstance(t, Tensor) and t.requires_grad for t in tuple(args) + tuple(kw.values()))
            if not E.autograd_needed(x, self) and not latent_grad:
                return fn(self, x, *args, **kw)
            if fn.__name__ == "transform":
                from . import _modgrad as MG
                ld = args[0] if len(args) > 0 else kw.get("log_det_jac")
                lp = args[1] if len(args) > 1 else kw.get("logp")
                if what == "StepFlow":
                    return self._transform_composed(x, ld, lp)
                if what in MG.SUPPORTED:
                    return MG.transform(self, what, fn, E.check_input(x), ld, lp)
            elif E.invert_grad_enabled():
                from . import _modgrad as MG
                if what == "StepFlow":
                    return self._invert_composed(x)
                if what == "Split":
                    latent = args[0] if len(args) > 0 else kw.get("inv_y_split")
                    temperature = args[1] if len(args) > 1 else kw.get("temperature", 1.0)
                    return MG.invert(self, what, fn, x, latent, temperature)
                return MG.invert(self, what, fn, x)
            ins = [t for t in (x,) + tuple(args) + tuple(kw.values()) if isinstance(t, Tensor)]
            deps = [t for t in ins if t.requires_grad] + [p for p in self.parameters() if p.requires_grad]
            with torch.no_grad():
                out = fn(self, x, *args, **kw)

            def poison(t):
                if not isinstance(t, Tensor) or not t.is_floating_point():
                    return t
                inplace = any(t is i for i in ins)
                if inplace and t.requires_grad:
                    return t
                return _NoBackward.apply(t, what, inplace, *deps)
            return tuple(poison(t) for t in out) if isinstance(out, tuple) else poison(out)
        wrapper.__name__, wrapper.__doc__ = fn.__name__, fn.__doc__
        return wrapper
    return deco


class IdentityTransform(Transform):
    def transform(self, x, log_det_jac, logp):
        return x, log_det_jac, logp

    def invert(self, y):
        return y


class ActNorm(Transform):
    """Per-channel affine y = exp(scale)*(x+bias) with data-dependent initialisation on the first call
    (reference transforms.py:56-94).  Parameters ``scale``/``bias`` (C,1,1) and the uint8 buffer
    ``is_initialized`` keep the reference's names."""

    def __init__(self, in_channels: int = 3):
        super().__init__()
        self.scale = nn.Parameter(torch.zeros(in_channels, 1, 1, device=self.device))
        self.bias = nn.Parameter(torch.zeros(in_channels, 1, 1, device=self.device))
        self.register_buffer("is_initialized", torch.tensor(0, dtype=torch.uint8, device=self.device))
        self._mix = E.MixCache()
        self._init_known: Optional[bool] = None

    # The reference reads the flag with .item() on every call (transforms.py:74: one host sync per ActNorm,
    # 144 per L3/K16 forward).  Here the flag is read once and cached on the host; loading a state_dict or
    # moving the module resets the cache.
    def _initialized(self) -> bool:
        if self._init_known is None:
            self._init_known = bool(self.is_initialized.item() != 0)
        return self._init_known

    def _mark_initialized(self) -> None:
        self.is_initialized.fill_(1)
        self._init_known = True
        self._mix.invalidate()

    def _load_from_state_dict(self, *args, **kwargs):
        self._init_known = None
        self._mix.invalidate()
        return super()._load_from_state_dict(*args, **kwargs)

    def _apply(self, fn, *a, **k):
        self._init_known = None
        self._mix = E.MixCache()
        return super()._apply(fn, *a, **k)

    @torch.no_grad()
    def _maybe_init(self, x: Tensor, xbs: int, B: int, C: int, P: int) -> None:
        if not self._initialized():
            E.channel_stats(x, 0, B, C, P, xbs, self.scale, self.bias)
            self._mark_initialized()

    @_granular("ActNorm")
    def transform(self, x: Tensor, log_det_jac: Tensor, logp: Tensor) -> Tuple[Tensor, Tensor, Tensor]:
        x = E.check_input(x)
        B, C, H, W = x.shape
        E.check_acc(log_det_jac, B, "log_det_jac")
        self._maybe_init(x, C * H * W, B, C, H * W)
        y = torch.empty_like(x)
        N.actnorm_apply(x, y, self.scale, self.bias, B, C, H * W, 0)
        if log_det_jac is not None:
            E.prepare_mix([(self._mix, None, self.scale, self.bias, C, None)])
            N.accumulate(log_det_jac, None, 0, B, self._mix.logdet, E.scalar_f32(x.device, H * W), 1)
        return y, log_det_jac, logp

    @_granular("ActNorm")
    def invert(self, y: Tensor) -> Tensor:
        y = E.check_input(y)
        B, C, H, W = y.shape
        out = torch.empty_like(y)
        N.actnorm_apply(y, out, self.scale, self.bias, B, C, H * W, 1)
        return out


class InvConv2d(Transform):
    """Invertible 1x1 convolution with a dense (C,C,1,1) ``weight`` initialised to a random orthogonal matrix
    (reference transforms.py:104-145).  log|det W| and W^-1 come from one fp64 LU kernel, cached until the
    weight changes."""

    def __init__(self, in_channels: int = 3):
        super().__init__()
        q, _ = torch.linalg.qr(torch.randn(in_channels, in_channels, dtype=torch.float32, device=self.device))
        self.weight = nn.Parameter(q.reshape(in_channels, in_channels, 1, 1).contiguous())
        self._mix = E.MixCache()

    def _load_from_state_dict(self, *args, **kwargs):
        self._mix.invalidate()
        return super()._load_from_state_dict(*args, **kwargs)

    def _apply(self, fn, *a, **k):
        self._mix = E.MixCache()
        return super()._apply(fn, *a, **k)

    @_granular("InvConv2d")
    def transform(self, x: Tensor, log_det_jac: Tensor, logp: Tensor) -> Tuple[Tensor, Tensor, Tensor]:
        x = E.check_input(x)
        B, C, H, W = x.shape
        E.check_acc(log_det_jac, B, "log_det_jac")
        E.prepare_mix([(self._mix, self.weight, None, None, C, None)])
        y = torch.empty_like(x)
        N.channel_mix(x, y, self._mix.fwd_mt, self._mix.fwd_beta, B, C, H * W, C * H * W, C * H * W)
        if log_det_jac is not None:
            N.accumulate(log_det_jac, None, 0, B, self._mix.logdet, E.scalar_f32(x.device, H * W), 1)
        return y, log_det_jac, logp

    @_granular("InvConv2d")
    def invert(self, y: Tensor) -> Tensor:
        y = E.check_input(y)
        B, C, H, W = y.shape
        E.prepare_mix([(self._mix, self.weight, None, None, C, None)])
        out = torch.empty_like(y)
        N.channel_mix(y, out, self._mix.inv_mt, self._mix.inv_beta, B, C, H * W, C * H * W, C * H * W)
        return out


class AffineCoupling(Transform):
    """Affine coupling layer (reference transforms.py:155-201).  ``net`` keeps the reference's Sequential layout
    so state_dicts interchange; the arithmetic is three GEMMs plus the fused coupling epilogue."""

    def __init__(self, in_channels: int = 2, n_features: int = 512):
        super().__init__()
        if in_channels % 2 != 0:
            raise ValueError("AffineCoupling needs an even number of channels")
        self.net = coupling_network(in_channels=in_channels // 2, n_features=n_features,
                                    out_channels=in_channels).to(self.device)
        self._cache = E.CouplingCache()

    def _parts(self):
        n = self.net
        return n[0].conv, n[0].actnorm, n[2].conv, n[2].actnorm, n[4]

    def _load_from_state_dict(self, *args, **kwargs):
        self._cache = E.CouplingCache()
        return super()._load_from_state_dict(*args, **kwargs)

    def _apply(self, fn, *a, **k):
        self._cache = E.CouplingCache()
        return super()._apply(fn, *a, **k)

    def _run(self, x: Tensor, xbs: int, y: Tensor, ybs: int, B: int, C: int, H: int, W: int, inverse: bool,
             ld_part: Optional[Tensor]) -> None:
        """x -> y on [B,C,P] views (may be the same memory: in place on the second channel half)."""
        zc = self.net[4]
        pm, ldp = E.coupling_rows(self, x, xbs, B, C, H, W, init=True)
        N.coupling_apply(pm, ldp, zc.bias, zc.logs, x, y, ld_part, B, C, H, W, xbs, ybs, inverse)

    @_granular("AffineCoupling")
    def transform(self, x: Tensor, log_det_jac: Tensor, logp: Tensor) -> Tuple[Tensor, Tensor, Tensor]:
        x = E.check_input(x)
        B, C, H, W = x.shape
        E.check_acc(log_det_jac, B, "log_det_jac")
        T = N.ld_tiles(H * W)
        part = E.WS.get("ldp1", T * B, torch.float32, x.device) if log_det_jac is not None else None
        y = torch.empty_like(x)
        self._run(x, C * H * W, y, C * H * W, B, C, H, W, False, part)
        if log_det_jac is not None:
            N.accumulate(log_det_jac, part, T, B)
        return y, log_det_jac, logp

    @_granular("AffineCoupling")
    def invert(self, y: Tensor) -> Tensor:
        y = E.check_input(y)
        B, C, H, W = y.shape
        out = torch.empty_like(y)
        self._run(y, C * H * W, out, C * H * W, B, C, H, W, True, None)
        return out


class Squeeze(Transform):
    """Space-to-depth by 2 (reference transforms.py:212-239): out channel = c*4 + h1*2 + w1."""

    @_granular("Squeeze")
    def transform(self, x: Tensor, log_det_jac: Tensor, logp: Tensor) -> Tuple[Tensor, Tensor, Tensor]:
        x = E.check_input(x)
        B, C, H, W = x.shape
        if H % 2 or W % 2:
            raise ValueError("Squeeze needs even height and width")
        y = torch.empty(B, C * 4, H // 2, W // 2, dtype=torch.float32, device=x.device)
        N.squeeze(x, y, B, C, H, W, C * H * W, C * H * W)
        return y, log_det_jac, logp

    @_granular("Squeeze")
    def invert(self, y: Tensor) -> Tensor:
        y = E.check_input(y)
        B, C, H, W = y.shape
        if C % 4:
            raise ValueError("Squeeze.invert needs a channel count divisible by 4")
        out = torch.empty(B, C // 4, H * 2, W * 2, dtype=torch.float32, device=y.device)
        N.unsqueeze(y, out, B, C, H, W, C * H * W, C * H * W)
        return out


class Split(Transform):
    """Channel split with an optional learned Gaussian prior on the split-off half (reference
    transforms.py:246-309).  ``conv`` is the ZeroConv2d(C/2 -> C) producing mean/log-sd."""

    def __init__(self, in_channels, learn_prior_mean_logs: bool = True):
        super().__init__()
        self.conv = ZeroConv2d(in_channels // 2, in_channels, padding=(3 - 1) // 2) if learn_prior_mean_logs else None
        self._cache = E.SplitCache()

    def _load_from_state_dict(self, *args, **kwargs):
        self._cache = E.SplitCache()
        return super()._load_from_state_dict(*args, **kwargs)

    def _apply(self, fn, *a, **k):
        self._cache = E.SplitCache()
        return super()._apply(fn, *a, **k)

    def _forward_views(self, x: Tensor, xbs: int, B: int, C: int, H: int, W: int, z_out: Tensor,
                       logp_part: Optional[Tensor]) -> None:
        """z_out <- x[:, C/2:], logp_part[t*B+b] <- log N(z; mean, exp(logs)) (skipped when logp_part is None)."""
        if logp_part is None:
            N.copy_channels(x[0, C // 2:] if xbs == C * H * W else x.view(-1)[(C // 2) * H * W:], z_out, B, C // 2,
                            H * W, xbs, (C // 2) * H * W)
            return
        h, ldh = E.split_rows(self, x, xbs, B, C, H, W)
        bias = self.conv.bias if self.conv is not None else None
        logs = self.conv.logs if self.conv is not None else None
        N.split_prior_logp(h, ldh, bias, logs, x, xbs, z_out, logp_part, B, C, H, W)

    @_granular("Split")
    def transform(self, x: Tensor, log_det_jac: Tensor, logp: Tensor) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
        x = E.check_input(x)
        B, C, H, W = x.shape
        E.check_acc(logp, B, "logp")
        Ch, P = C // 2, H * W
        y = torch.empty(B, Ch, H, W, dtype=torch.float32, device=x.device)
        z = torch.empty(B, Ch, H, W, dtype=torch.float32, device=x.device)
        N.copy_channels(x, y, B, Ch, P, C * P, Ch * P)
        T = N.ld_tiles(P)
        part = E.WS.get("lpp1", T * B, torch.float32, x.device) if logp is not None else None
        self._forward_views(x, C * P, B, C, H, W, z, part)
        if logp is not None:
            N.accumulate(logp, part, T, B)
        return y, log_det_jac, z, logp

    @_granular("Split")
    def invert(self, y: Tensor, inv_y_split: Tensor = None, temperature: float = 1.0) -> Tensor:
        y = E.check_input(y)
        B, Ch, H, W = y.shape
        C, P = 2 * Ch, H * W
        out = torch.empty(B, C, H, W, dtype=torch.float32, device=y.device)
        N.copy_channels(y, out, B, Ch, P, Ch * P, C * P)
        self._fill_second_half(out, C * P, B, C, H, W, inv_y_split, temperature)
        return out

    def _fill_second_half(self, out: Tensor, obs: int, B: int, C: int, H: int, W: int, z: Optional[Tensor],
                          temperature: float, eps_sink: Optional[list] = None,
                          logp_part: Optional[Tensor] = None) -> None:
        """Write the latent (given, or drawn from the conditional prior, reference transforms.py:305-307 and
        prior.py:49-50) into channels C/2..C of ``out`` whose first half is already in place.  ``eps_sink`` receives the
        standard-normal tensor a draw used (the inverse's backward needs it).  ``logp_part`` receives the partials of
        log N(z; mean, exp(logs)) of the written half, as ``transform`` writes them (the model's density, whatever the
        temperature of a draw)."""
        Ch, P = C // 2, H * W
        second = out.view(-1)[Ch * P:]
        bias = self.conv.bias if self.conv is not None else None
        logs = self.conv.logs if self.conv is not None else None
        if z is not None:
            z = E.check_input(z, "latent")
            if tuple(z.shape) != (B, Ch, H, W):
                raise ValueError(f"latent has shape {tuple(z.shape)}, expected {(B, Ch, H, W)}")
            N.copy_channels(z, second, B, Ch, P, Ch * P, obs)
            if logp_part is not None:
                h, ldh = E.split_rows(self, out, obs, B, C, H, W)
                N.split_prior_logp(h, ldh, bias, logs, out, obs, None, logp_part, B, C, H, W)
            return
        eps = torch.empty(B, Ch, H, W, dtype=torch.float32, device=out.device).normal_()
        if eps_sink is not None:
            eps_sink.append(eps)
        h, ldh = E.split_rows(self, out, obs, B, C, H, W)
        N.split_prior_sample(h, ldh, bias, logs, eps, temperature, out, obs, B, C, H, W)
        if logp_part is not None:           # the prior conv rows h of the draw serve the density too
            N.split_prior_logp(h, ldh, bias, logs, out, obs, None, logp_part, B, C, H, W)
