"""Autograd through ``Glow.invert`` and the priors' ``sample`` (``NFDPM_INVERT_GRAD=1``).

``Glow.invert`` records ONE ``GlowInvertFn``.  Its forward is the no-grad inverse's kernel chain, level by level with the
same per-level kernel choice (``Glow._level_mode``), with sinks added: fresh per-step buffers for the coupling network's
operands (im2col rows A1, hidden maps h1 / h2, ZeroConv taps pm) and the step boundary's pre-mix sink for u_k, the coupling
inverse's output (``gemm3_boundary(pm_out, xs, inverse)`` where the fused GEMM runs, ``flow_boundary_inv_stash`` at the
other one-CTA-per-image levels, ``flow_boundary_tiled(xs)`` at row-band levels, the unfused kernels elsewhere).  Each step
writes a fresh state tensor, so the state stack y_k costs no extra writes; x is the output of that one chain.  Per
sampling Split it keeps the eps its prior draw used (drawn eagerly by ``normal_()`` on torch's CUDA generator, deepest
first, as the no-grad inverse draws it).  The backward walks the levels 0..L-1 and the steps k = 0..K-1: mix_bwd with
inv_mt (fusing the col2im of the previous step's im2col gradient) + mix_inv_param_grad, coupling_inv_bwd + the shared
coupling-network backward (_modgrad._net_backward); at the level end col2im_add, then the Split (split_sample_bwd + the
prior conv's GEMMs, or the gradient of a supplied latent) and the squeeze.

Parameter gradients are returned to autograd (nothing writes ``.grad`` directly); a module whose parameters do not
require grad launches no weight-gradient GEMM and no parameter fold.
"""
from __future__ import annotations

from types import SimpleNamespace
from typing import List, Optional

import torch
from torch import Tensor

from . import _engine as E
from . import _modgrad as MG
from . import _native as N
from .utils import get_item


def _net_rows(cp, A1: Tensor, M: int, dt: torch.dtype):
    """GEMM1 and GEMM2 of coupling network ``cp`` into fresh buffers (the launches of E.coupling_gemms)."""
    conv1, an1, conv2, an2, _ = cp._parts()
    F = conv1.weight.shape[0]
    cache, K1p = cp._cache.at(dt), cp._cache.K1p
    h1 = torch.empty(M * F, dtype=dt, device=A1.device)
    N.gemm_nt(A1, K1p, cache.w1, K1p, h1, F, M, F, K1p, N.EPI_ACTNORM_RELU, an1.scale, an1.bias)
    h2 = torch.empty(M * F, dtype=dt, device=A1.device)
    N.gemm_nt(h1, F, cache.w2 if dt != torch.float32 else conv2.weight, F, h2, F, M, F, F, N.EPI_ACTNORM_RELU, an2.scale,
              an2.bias)
    return h1, h2


def _a1(cp, M: int, dt: torch.dtype, dev) -> Tensor:
    conv1, _, conv2, _, zc = cp._parts()
    E._pack_coupling(cp._cache, conv1.weight, conv2.weight, zc.weight, dt)
    return torch.empty(M * cp._cache.K1p, dtype=dt, device=dev)


def _level_stash(flows, src: Tensor, mode: str, B: int, C: int, h: int, w: int):
    """The K inverse StepFlows of one level (input ``src``, only read) with the operands of every step kept.
    Returns (level output, [(y_k, stash_k, u_k) for k = 0..K-1])."""
    dev = src.device
    P, M = h * w, B * h * w
    K = len(flows)
    recs = [None] * K
    cur = src
    if mode == "unfused":
        for k in range(K - 1, -1, -1):
            step = flows[k]
            E.prepare_mix([step._mix_entry(None)])
            u, st = MG.coupling_invert_stash(step.affcoupling, cur)
            x = torch.empty_like(u)
            N.channel_mix(u, x, step._mix.inv_mt, step._mix.inv_beta, B, C, P, C * P, C * P)
            recs[k] = (cur, st, u)
            cur = x
        return cur, recs
    dt = E.coupling_dtype()
    A1 = _a1(flows[-1].affcoupling, M, dt, dev)
    K1p = flows[-1].affcoupling._cache.K1p
    if mode == "tiled":                                 # im2col of the level's entry state
        N.flow_boundary_tiled(src, C * P, False, None, 0, None, None, None, None, None, None, 0, None, 0, A1, K1p, B, C, h,
                              w, False, N.flow_boundary_tiles(B, C, h, w, 0, 0, 1))
    else:
        N.flow_boundary(src, C * P, False, None, 0, None, None, None, None, None, None, 0, A1, K1p, B, C, h, w, False)
    for k in range(K - 1, -1, -1):
        step = flows[k]
        cp = step.affcoupling
        zc = cp._parts()[4]
        F = cp._parts()[0].weight.shape[0]
        K1p, ldp = cp._cache.K1p, cp._cache.ldp
        h1, h2 = _net_rows(cp, A1, M, dt)
        pm = torch.empty(M * ldp, dtype=torch.float32, device=dev)
        u, x = torch.empty_like(src), torch.empty_like(src)
        A1n = _a1(flows[k - 1].affcoupling, M, dt, dev) if k > 0 else None
        K1n = flows[k - 1].affcoupling._cache.K1p if k > 0 else 0
        mt, beta = step._mix.inv_mt, step._mix.inv_beta
        if mode == "tiled":
            N.gemm_nt(h2, F, cp._cache.at(dt).w3, F, pm, ldp, M, ldp, F)
            N.flow_boundary_tiled(cur, C * P, False, pm, ldp, zc.bias, zc.logs, None, mt, beta, x, C * P, u, C * P, A1n, K1n,
                                  B, C, h, w, True, N.flow_boundary_tiles(B, C, h, w, 1, 1, int(k > 0)))
        elif E.fused_g3_ok(B, C, h, w, F, ldp, dt):
            N.gemm3_boundary(h2, F, cp._cache.at(dt).w3, pm, ldp, cur, C * P, zc.bias, zc.logs, None, mt, beta, x, C * P, u,
                             C * P, A1n, K1n, B, C, h, w, F, ldp, True)
        else:
            N.gemm_nt(h2, F, cp._cache.at(dt).w3, F, pm, ldp, M, ldp, F)
            N.flow_boundary_inv_stash(cur, C * P, pm, ldp, zc.bias, zc.logs, mt, beta, x, C * P, u, C * P, A1n, K1n, B, C, h,
                                      w)
        recs[k] = (cur, SimpleNamespace(A1=A1, h1=h1, h2=h2, pm=pm, dt=dt, K1p=K1p, ldp=ldp), u)
        cur, A1 = x, A1n
    return cur, recs


def invert_stash(glow, latents, temperature: float):
    """Glow.invert returning (x, per-level step records, per-Split (input, eps)).  The kernels are those of the no-grad
    inverse (uncaptured), with sinks added; an uninitialised model takes the unfused chain, which initialises the coupling
    networks' ActNorms on the way (without gradient), as the no-grad inverse does."""
    levels = glow._levels()
    L = glow.L
    z_last = latents[-1]
    B, C, h, w = z_last.shape
    dev = z_last.device
    steps = [s for flows, _ in levels for s in flows]
    ready = all(s._ready() for s in steps)
    fast = ready and glow._fast_ok(h * 2 ** L, w * 2 ** L)
    if ready:
        slots = glow._slots(dev)
        E.prepare_mix([s._mix_entry(slots[i:i + 1]) for i, s in enumerate(steps)])
    steps_rec, split_rec = [None] * L, [None] * L
    cur = z_last
    for li in range(L - 1, -1, -1):
        flows, _ = levels[li]
        P = h * w
        mode = glow._level_mode(B, C, h, w) if fast else "unfused"
        cur, steps_rec[li] = _level_stash(flows, cur, mode, B, C, h, w)
        if li == 0:
            out = torch.empty(B, C // 4, h * 2, w * 2, dtype=torch.float32, device=dev)
            N.unsqueeze(cur, out, B, C, h, w, C * P, (C // 4) * P * 4)
            return out, steps_rec, split_rec
        Cn, hn, wn = 2 * (C // 4), h * 2, w * 2
        nxt = torch.empty(B, Cn, hn, wn, dtype=torch.float32, device=dev)
        N.unsqueeze(cur, nxt, B, C, h, w, C * P, Cn * hn * wn)
        sink = []
        levels[li - 1][1]._fill_second_half(nxt, Cn * hn * wn, B, Cn, hn, wn, get_item(latents, -(L - li + 1)),
                                            temperature, eps_sink=sink)
        split_rec[li - 1] = (nxt, sink[0] if sink else None)
        cur, C, h, w = nxt, Cn, hn, wn
    raise AssertionError("unreachable")


class GlowInvertFn(torch.autograd.Function):
    """(glow, temperature, n_latents, *latents, *parameters) -> x."""

    @staticmethod
    def forward(ctx, glow, temperature, n_lat, *args):
        latents = [t.detach() if isinstance(t, Tensor) else t for t in args[:n_lat]]
        ctx.glow, ctx.temperature, ctx.n_lat, ctx.params = glow, temperature, n_lat, args[n_lat:]
        x, steps_rec, split_rec = invert_stash(glow, latents, temperature)
        ctx.rec = (steps_rec, split_rec)
        # the deepest level's first step keeps the caller's last latent: saved so that an in-place change is detected
        ctx.save_for_backward(*[t for t in args[:n_lat] if isinstance(t, Tensor)])
        return x

    @staticmethod
    def backward(ctx, dx):
        if ctx.rec is None:
            raise RuntimeError("Glow.invert: the stash of this call was released by an earlier backward")
        ctx.saved_tensors                               # raises if a latent was modified in place since the forward
        glow, T, n_lat = ctx.glow, ctx.temperature, ctx.n_lat
        steps_rec, split_rec = ctx.rec
        ctx.rec = None
        levels = glow._levels()
        L = glow.L
        dx = dx.to(torch.float32).contiguous()
        B, c, H, W = dx.shape
        C, h, w = 4 * c, H // 2, W // 2
        d = torch.empty(B, C, h, w, dtype=torch.float32, device=dx.device)
        N.squeeze(dx, d, B, c, H, W, c * H * W, C * h * w)
        g = {}
        d_lat: List[Optional[Tensor]] = [None] * n_lat
        for li in range(L):
            flows, split = levels[li]
            da1, lda1 = None, 0
            for step, (y_k, st_k, u_k) in zip(flows, steps_rec[li]):
                an, ic = step.actnorm, step.invconv2d
                du, dW, dS, dB = MG._mix_inv_backward(step._mix, u_k, d, ic.weight, an.scale, an.bias,
                                                      MG._wants_grad(an) or MG._wants_grad(ic), da1, lda1)
                g[ic.weight], g[an.scale], g[an.bias] = dW, dS, dB
                d, gc, da1 = MG._coupling_backward(step.affcoupling, st_k, y_k, du, None, inverse=True,
                                                   wgrad=MG._wants_grad(step.affcoupling), col2im=False)
                lda1 = st_k.K1p
                g.update(gc)
            N.col2im_add(da1, lda1, d, C * h * w, B, C // 2, h, w)
            if li == L - 1:
                d_lat[n_lat - 1] = d
                break
            nxt, eps = split_rec[li]
            dy, dz, gs = MG._split_sample_backward(split, nxt, eps, T, d, MG._wants_grad(split))
            g.update(gs)
            if dz is not None:
                d_lat[n_lat - (L - li)] = dz
            Ch, P = C // 2, h * w
            C, h, w = 4 * Ch, h // 2, w // 2
            d = torch.empty(B, C, h, w, dtype=torch.float32, device=dx.device)
            N.squeeze(dy, d, B, Ch, 2 * h, 2 * w, Ch * P, C * h * w)
        lat_g = [gl if ctx.needs_input_grad[3 + i] else None for i, gl in enumerate(d_lat)]
        par_g = [g.get(p) if p.requires_grad else None for p in ctx.params]
        return (None, None, None) + tuple(lat_g) + tuple(par_g)


def glow_invert(glow, latents: list, temperature: float) -> Tensor:
    lat = [E.check_input(t, "latent") if isinstance(t, Tensor) else t for t in latents]
    return GlowInvertFn.apply(glow, float(temperature), len(lat), *lat, *glow.parameters())


# ------------------------------------------------------------------------------------------- priors
class GaussianSampleFn(torch.autograd.Function):
    """GaussianPrior.sample: z = bias*e^(3 logs) (mean half) + exp(log-sd half)*T*eps, per channel."""

    @staticmethod
    def forward(ctx, shape, temperature, bias, logs):
        B, C, H, W = shape
        eps = torch.empty(B, C, H, W, dtype=torch.float32, device=bias.device).normal_()
        out = torch.empty_like(eps)
        N.gauss_sample_const(eps, bias, logs, temperature, out, B, C, H * W)
        ctx.temperature = temperature
        ctx.save_for_backward(eps, bias, logs)
        return out

    @staticmethod
    def backward(ctx, dz):
        eps, bias, logs = ctx.saved_tensors
        B, C, H, W = eps.shape
        dz = dz.to(torch.float32).contiguous()
        dpar = torch.empty(B * 4 * C, dtype=torch.float32, device=dz.device)
        N.split_sample_bwd(dz, C * H * W, eps, ctx.temperature, None, 0, bias, logs, None, dpar, B, 2 * C, H, W)
        db, dl = torch.empty_like(bias), torch.empty_like(logs)
        N.reduce_rows2(dpar, db, dl, B, 2 * C, 2 * C, 4 * C)
        return None, None, db if ctx.needs_input_grad[2] else None, dl if ctx.needs_input_grad[3] else None


class IsotropicSampleFn(torch.autograd.Function):
    """IsotropicGaussian.sample: z = mean + exp(logsd)*T*eps, elementwise."""

    @staticmethod
    def forward(ctx, temperature, mean, logsd):
        B = mean.shape[0]
        n = mean[0].numel()
        eps = torch.empty_like(mean).normal_()
        h = torch.empty(B, 2 * n, dtype=torch.float32, device=mean.device)
        N.copy_channels(mean, h, B, n, 1, n, 2 * n)
        N.copy_channels(logsd, h.view(-1)[n:], B, n, 1, n, 2 * n)
        zeros = torch.zeros(2 * n, dtype=torch.float32, device=mean.device)
        out2 = torch.empty(B, 2 * n, dtype=torch.float32, device=mean.device)
        N.split_prior_sample(h, 2 * n, zeros, zeros, eps, temperature, out2, 2 * n, B, 2 * n, 1, 1)
        out = torch.empty_like(mean)
        N.copy_channels(out2.view(-1)[n:], out, B, n, 1, 2 * n, n)
        ctx.temperature = temperature
        ctx.save_for_backward(eps, h, zeros)
        return out

    @staticmethod
    def backward(ctx, dz):
        eps, h, zeros = ctx.saved_tensors
        B, n = h.shape[0], h.shape[1] // 2
        dz = dz.to(torch.float32).contiguous()
        dh = torch.empty(B, 2 * n, dtype=torch.float32, device=dz.device)
        dpar = torch.empty(B * 4 * n, dtype=torch.float32, device=dz.device)
        N.split_sample_bwd(dz, n, eps, ctx.temperature, h, 2 * n, zeros, zeros, dh, dpar, B, 2 * n, 1, 1)
        dmean, dlogsd = torch.empty_like(eps), torch.empty_like(eps)
        N.copy_channels(dh, dmean, B, n, 1, 2 * n, n)
        N.copy_channels(dh.view(-1)[n:], dlogsd, B, n, 1, 2 * n, n)
        return None, dmean if ctx.needs_input_grad[1] else None, dlogsd if ctx.needs_input_grad[2] else None
