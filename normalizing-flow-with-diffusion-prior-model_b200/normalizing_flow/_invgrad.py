"""Autograd through ``Glow.invert`` and the priors' ``sample`` (``NFDPM_INVERT_GRAD=1``).

``Glow.invert`` records ONE ``GlowInvertFn``.  Its forward is the no-grad inverse's walk (``Glow._invert_walk``: the same
level transitions and per-level kernel choice, ``Glow._level_mode``) with each level's StepFlows run by ``_level_stash``,
which adds sinks: fresh per-step buffers for the coupling network's operands (im2col rows A1, hidden maps h1 / h2,
ZeroConv taps pm) and the step boundary's pre-mix sink for u_k, the coupling inverse's output (``gemm3_boundary(pm_out,
xs, inverse)`` where the fused GEMM runs, ``flow_boundary_inv_stash`` at the other one-CTA-per-image levels,
``flow_boundary_tiled(xs)`` at row-band levels, the unfused kernels elsewhere).  Each step
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


def _level_stash(flows, src: Tensor, mode: str, B: int, C: int, h: int, w: int, ld_part: Optional[Tensor] = None,
                 row: int = 0):
    """The K inverse StepFlows of one level (input ``src``, only read) with the operands of every step kept.  The log-det
    partials go to the rows of ``ld_part`` from ``row`` on that the no-grad level function of ``mode`` writes (none when
    ``ld_part`` is None).  Returns (level output, [(y_k, stash_k, u_k) for k = 0..K-1], partial rows)."""
    dev = src.device
    P, M = h * w, B * h * w
    K = len(flows)
    recs = [None] * K
    cur = src
    rows = 0

    def part():
        return ld_part[(row + rows) * B:] if ld_part is not None else None

    if mode == "unfused":
        T = N.ld_tiles(P)
        for k in range(K - 1, -1, -1):
            step = flows[k]
            E.prepare_mix([step._mix_entry(None)])
            u, st = MG.coupling_invert_stash(step.affcoupling, cur, part())
            x = torch.empty_like(u)
            N.channel_mix(u, x, step._mix.inv_mt, step._mix.inv_beta, B, C, P, C * P, C * P)
            recs[k] = (cur, st, u)
            cur = x
            rows += T
        return cur, recs, rows
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
            T = N.flow_boundary_tiles(B, C, h, w, 1, 1, int(k > 0))
            N.gemm_nt(h2, F, cp._cache.at(dt).w3, F, pm, ldp, M, ldp, F)
            N.flow_boundary_tiled(cur, C * P, False, pm, ldp, zc.bias, zc.logs, part(), mt, beta, x, C * P, u, C * P, A1n,
                                  K1n, B, C, h, w, True, T)
        elif E.fused_g3_ok(B, C, h, w, F, ldp, dt):
            T = 1
            N.gemm3_boundary(h2, F, cp._cache.at(dt).w3, pm, ldp, cur, C * P, zc.bias, zc.logs, part(), mt, beta, x, C * P,
                             u, C * P, A1n, K1n, B, C, h, w, F, ldp, True)
        else:
            T = 1
            N.gemm_nt(h2, F, cp._cache.at(dt).w3, F, pm, ldp, M, ldp, F)
            N.flow_boundary_inv_stash_ld(cur, C * P, pm, ldp, zc.bias, zc.logs, part(), mt, beta, x, C * P, u, C * P, A1n,
                                         K1n, B, C, h, w)
        recs[k] = (cur, SimpleNamespace(A1=A1, h1=h1, h2=h2, pm=pm, dt=dt, K1p=K1p, ldp=ldp), u)
        cur, A1 = x, A1n
        rows += T
    return cur, recs, rows


def invert_stash(glow, latents, temperature, with_ld: bool = False, with_lp: bool = False,
                 seeds: Optional[Tensor] = None):
    """Glow.invert returning (x, per-level step records, per-Split (input, eps), density partials as `_invert_walk`
    returns them).  The walk and the kernels are those of the no-grad inverse (uncaptured, ``Glow._invert_walk``), with
    `_level_stash` for each level's StepFlows; an uninitialised model takes the unfused chain, which initialises the
    coupling networks' ActNorms on the way (without gradient), as the no-grad inverse does."""
    steps_rec, split_rec = [], []

    def level(mode, flows, src, B, C, h, w, ld_part, row):
        x, recs, rows = _level_stash(flows, src, mode, B, C, h, w, ld_part, row)
        steps_rec.insert(0, recs)                       # the walk runs deepest first
        return x, rows

    x, parts = glow._invert_walk(latents, temperature, glow._ready(), with_ld, with_lp, level=level, eps_sink=split_rec,
                                 seeds=seeds)
    return x, steps_rec, split_rec[::-1], parts


class GlowInvertFn(torch.autograd.Function):
    """(glow, (temperature, seeds), n_latents, log_det_jac | None, logp | None, *latents, *parameters) -> x, or (x,
    log_det_jac?, logp?) when an accumulator is given: the accumulators receive the density of x in place
    (``Glow._add_density``, as the no-grad inverse) and are marked dirty; their gradients reach the log-det and Split log-p
    terms.  The temperature is a number or a per-image [B] vector; with seeds the draws come from the kernels' counter-based
    generator and are kept for the backward like torch's."""

    @staticmethod
    def forward(ctx, glow, draw, n_lat, ld, lp, *args):
        temperature, seeds = draw
        latents = [t.detach() if isinstance(t, Tensor) else t for t in args[:n_lat]]
        ctx.glow, ctx.temperature, ctx.n_lat, ctx.params = glow, temperature, n_lat, args[n_lat:]
        ctx.have_ld, ctx.have_lp = ld is not None, lp is not None
        x, steps_rec, split_rec, parts = invert_stash(glow, latents, temperature, ld is not None, lp is not None, seeds)
        ctx.rec = (steps_rec, split_rec)
        # the deepest level's first step keeps the caller's last latent: saved so that an in-place change is detected
        ctx.save_for_backward(*[t for t in args[:n_lat] if isinstance(t, Tensor)])
        accs = [a for a in (ld, lp) if a is not None]
        if not accs:
            return x
        glow._add_density(ld, lp, parts, x.shape[2], x.shape[3])
        ctx.mark_dirty(*accs)
        return (x,) + tuple(accs)

    @staticmethod
    def backward(ctx, dx, *g_acc):
        if ctx.rec is None:
            raise RuntimeError("Glow.invert: the stash of this call was released by an earlier backward")
        ctx.saved_tensors                               # raises if a latent was modified in place since the forward
        glow, T, n_lat = ctx.glow, ctx.temperature, ctx.n_lat
        steps_rec, split_rec = ctx.rec
        ctx.rec = None
        L = glow.L
        dy = dx.to(torch.float32).contiguous()
        B, _, H, W = dy.shape
        g_acc = list(g_acc)
        dld = g_acc.pop(0).to(torch.float32).contiguous() if ctx.have_ld else None
        dlp = g_acc.pop(0).to(torch.float32).contiguous() if ctx.have_lp else None
        dld_sum = MG._dld_sum(dld) if dld is not None else None
        g = {}
        d_lat: List[Optional[Tensor]] = [None] * n_lat
        for li, (flows, split, C, h, w) in enumerate(glow._geometry(H, W)):
            # gradient of the level's output state: squeeze of the gradient of what it unsqueezed into
            d = torch.empty(B, C, h, w, dtype=torch.float32, device=dy.device)
            N.squeeze(dy, d, B, C // 4, 2 * h, 2 * w, C * h * w, C * h * w)
            da1, lda1 = None, 0
            for step, (y_k, st_k, u_k) in zip(flows, steps_rec[li]):
                an, ic = step.actnorm, step.invconv2d
                du, dW, dS, dB = MG._mix_inv_backward(step._mix, u_k, d, ic.weight, an.scale, an.bias,
                                                      MG._wants_grad(an) or MG._wants_grad(ic), da1, lda1, dld_sum)
                g[ic.weight], g[an.scale], g[an.bias] = dW, dS, dB
                d, gc, da1 = MG._coupling_backward(step.affcoupling, st_k, y_k, du, dld, inverse=True,
                                                   wgrad=MG._wants_grad(step.affcoupling), col2im=False)
                lda1 = st_k.K1p
                g.update(gc)
            N.col2im_add(da1, lda1, d, C * h * w, B, C // 2, h, w)
            if split is None:
                d_lat[n_lat - 1] = d
                break
            nxt, eps = split_rec[li]
            dy, dz, gs = MG._split_sample_backward(split, nxt, eps, T, d, MG._wants_grad(split), dlp)
            g.update(gs)
            if dz is not None:
                d_lat[n_lat - (L - li)] = dz
        lat_g = [gl if ctx.needs_input_grad[5 + i] else None for i, gl in enumerate(d_lat)]
        par_g = [g.get(p) if p.requires_grad else None for p in ctx.params]
        return (None, None, None, None, None) + tuple(lat_g) + tuple(par_g)


def glow_invert(glow, latents: list, temperature, log_det_jac: Optional[Tensor] = None,
                logp: Optional[Tensor] = None, seeds: Optional[Tensor] = None):
    """The recorded Glow.invert: x, or (x, log_det_jac, logp) when an accumulator is given (``None`` stays ``None``).
    ``temperature`` / ``seeds`` as ``E.sampling_inputs`` returns them."""
    lat = [E.check_input(t, "latent") if isinstance(t, Tensor) else t for t in latents]
    draw = (temperature if isinstance(temperature, Tensor) else float(temperature), seeds)
    out = GlowInvertFn.apply(glow, draw, len(lat), log_det_jac, logp, *lat, *glow.parameters())
    if log_det_jac is None and logp is None:
        return out
    out = list(out)
    x = out.pop(0)
    ld = out.pop(0) if log_det_jac is not None else None
    lp = out.pop(0) if logp is not None else None
    return x, ld, lp


# ------------------------------------------------------------------------------------------- priors
class GaussianSampleFn(torch.autograd.Function):
    """GaussianPrior.sample: z = bias*e^(3 logs) (mean half) + exp(log-sd half)*T*eps, per channel.  ``draw``: (temperature,
    seeds) as ``E.sampling_inputs`` returns them."""

    @staticmethod
    def forward(ctx, shape, draw, bias, logs):
        temperature, seeds = draw
        B, C, H, W = shape
        eps = torch.empty(B, C, H, W, dtype=torch.float32, device=bias.device)
        out = torch.empty_like(eps)
        if seeds is None and not isinstance(temperature, Tensor):
            N.gauss_sample_const(eps.normal_(), bias, logs, temperature, out, B, C, H * W)
        elif seeds is None:
            N.gauss_sample_const_ex(eps.normal_(), None, 0, bias, logs, 1.0, temperature, None, out, B, C, H * W)
        else:
            N.gauss_sample_const_ex(None, seeds, N.PRIOR_STREAM, bias, logs, 1.0, temperature, eps, out, B, C, H * W)
        ctx.temperature = temperature
        ctx.save_for_backward(eps, bias, logs)
        return out

    @staticmethod
    def backward(ctx, dz):
        eps, bias, logs = ctx.saved_tensors
        B, C, H, W = eps.shape
        dz = dz.to(torch.float32).contiguous()
        dpar = torch.empty(B * 4 * C, dtype=torch.float32, device=dz.device)
        if isinstance(ctx.temperature, Tensor):
            N.split_sample_bwd_ex(dz, C * H * W, eps, 1.0, ctx.temperature, None, None, 0, bias, logs, None, dpar, B, 2 * C,
                                  H, W)
        else:
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
