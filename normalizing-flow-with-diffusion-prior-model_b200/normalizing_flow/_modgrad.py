"""Autograd for the transforms called ON THEIR OWN (reference normalizing_flow/transforms.py:56-309, glow.py:46-48,107-111
are ordinary autograd modules): ``ActNorm``, ``InvConv2d``, ``AffineCoupling``, ``Squeeze``, ``Split`` — and through them
``StepFlow`` and ``GlowBlock``, which compose the granular calls like the reference does.  One ``torch.autograd.Function``
per ``transform`` call: the forward runs the module's own kernels and keeps what the backward needs, the backward is
composed from the SAME backward kernels the whole-``Glow`` training path uses (normalizing_flow/_train.py) — no torch
arithmetic.  The whole-Glow Function stays the fast training entry point (fused step boundaries, side-stream weight
gradients, captured chains); this path serves unit tests, ablations and custom stacks of the primitives.

Both accumulators are updated in place (``+=`` semantics, transforms.py:81,131,184,288) and marked dirty; their incoming
gradients pass through unchanged and the log-det / log-p terms of the module receive them.

``invert`` is differentiable the same way when ``NFDPM_INVERT_GRAD=1`` (``ModuleInvertFn``): the inverse kernels run with
their operands kept, and the backward uses the inverse-direction kernels (coupling_inv_bwd, mix_inv_param_grad,
split_sample_bwd) plus the shared coupling-network backward.  Without the knob ``invert`` has no backward.
"""
from __future__ import annotations

from types import SimpleNamespace
from typing import Optional

import torch
from torch import Tensor

from . import _engine as E
from . import _native as N

SUPPORTED = ("ActNorm", "InvConv2d", "AffineCoupling", "Squeeze", "Split")


def _f32(t: Optional[Tensor], B: int, dev) -> Tensor:
    if t is None:
        return torch.zeros(B, dtype=torch.float32, device=dev)
    return t.to(torch.float32).contiguous()


def _dld_sum(dld32: Tensor) -> Tensor:
    out = torch.empty(1, dtype=torch.float32, device=dld32.device)
    N.reduce_rows(dld32, out, dld32.numel(), 1, 1)
    return out


# ------------------------------------------------------------------------------------------- per-module forward / backward
def _mix_backward(mod, x: Tensor, dy: Tensor, dld32: Tensor, weight, scale, bias):
    """Backward of y = W diag(e^s) (x + b) with log-det P (sum s + log|det W|): dx and the parameter gradients
    (nfdpm_mix_bwd + nfdpm_mix_param_grad, the kernels of the fused ActNorm + 1x1 conv backward)."""
    B, C, H, W = x.shape
    P = H * W
    f32 = dict(dtype=torch.float32, device=x.device)
    E.prepare_mix([(mod._mix, weight, scale, bias, C, None)])
    T_m = N.mix_bwd_tiles(C, H, W)
    part = torch.empty(B * T_m * (C * C + C), **f32)
    dx = torch.empty_like(x)
    N.mix_bwd(dy, C * P, None, 0, x, C * P, mod._mix.fwd_mt, dx, C * P, part, B, C, H, W)
    eye = torch.eye(C, **f32) if weight is None else None
    dW = torch.empty_like(weight) if weight is not None else None
    dS = torch.empty_like(scale) if scale is not None else None
    dB = torch.empty_like(bias) if bias is not None else None
    scratch = torch.empty(C * C + C, **f32)
    wptr = weight.data_ptr() if weight is not None else eye.data_ptr()
    winv = mod._mix.winv.data_ptr() if weight is not None else eye.data_ptr()
    item = N.MixGradItem(part=part.data_ptr(), B=B * T_m, C=C, weight=wptr, scale=N._p(scale), bias=N._p(bias), winv=winv,
                         dld_sum=_dld_sum(dld32).data_ptr(), P=float(P), pad_=0, d_weight=N._p(dW), d_scale=N._p(dS),
                         d_bias=N._p(dB), scratch=scratch.data_ptr())
    N.mix_param_grad([item])
    return dx, dW, dS, dB


def _mix_inv_backward(mix, u: Tensor, dx: Tensor, weight, scale, bias, wgrad: bool = True, da1: Optional[Tensor] = None,
                      lda1: int = 0, dld_sum: Optional[Tensor] = None):
    """Backward of the inverse mix x = diag(e^-s) W^-1 u - b: du (nfdpm_mix_bwd with inv_mt) and, with ``wgrad``, the
    parameter gradients (nfdpm_mix_inv_param_grad).  ``da1``: im2col-row gradient of a coupling network that read ``x``;
    its col2im is added to ``dx`` inside mix_bwd.  ``dld_sum`` ([1], sum over the batch of d(log_det_jac)): the gradient of
    the constant H*W*(sum s + log|det W|) the inverse accumulates is folded into the parameter gradients."""
    B, C, H, W = u.shape
    P = H * W
    f32 = dict(dtype=torch.float32, device=u.device)
    E.prepare_mix([(mix, weight, scale, bias, C, None)])
    T_m = N.mix_bwd_tiles(C, H, W)
    part = torch.empty(B * T_m * (C * C + C), **f32)
    du = torch.empty_like(u)
    N.mix_bwd(dx, C * P, da1, lda1, u, C * P, mix.inv_mt, du, C * P, part, B, C, H, W)
    if not wgrad:
        return du, None, None, None
    eye = torch.eye(C, **f32) if weight is None else None
    dW = torch.empty_like(weight) if weight is not None else None
    dS = torch.empty_like(scale) if scale is not None else None
    dB = torch.empty_like(bias) if bias is not None else None
    scratch = torch.empty(C * C + C, **f32)
    item = N.MixGradItem(part=part.data_ptr(), B=B * T_m, C=C, weight=N._p(weight), scale=N._p(scale), bias=N._p(bias),
                         winv=mix.winv.data_ptr() if weight is not None else eye.data_ptr(), dld_sum=N._p(dld_sum),
                         P=float(P) if dld_sum is not None else 0.0, pad_=0,
                         d_weight=N._p(dW), d_scale=N._p(dS), d_bias=N._p(dB), scratch=scratch.data_ptr())
    N.mix_inv_param_grad([item])
    return du, dW, dS, dB


def _split_sample_backward(sp, out: Tensor, eps: Optional[Tensor], temperature, d_out: Tensor, wgrad: bool = True,
                           dlp: Optional[Tensor] = None):
    """Backward of Split.invert: ``out`` = (y | z) [B,C,H,W], ``d_out`` its gradient.  Returns (dy, d_latent, grads).  A
    sampled half (``eps`` given) z = mean(y) + exp(lg(y))*T*eps back-propagates into y and the prior conv's parameters
    (nfdpm_split_sample_bwd + the conv's fp32 wgrad / dgrad GEMMs); a supplied latent receives the second half.
    ``temperature``: the draw's number or per-image [B] vector.  ``dlp`` ([B] fp32): gradient of the log-density log N(z; mean(y), exp(lg(y))) the inverse accumulated for this Split.
    A sampled half takes it inside nfdpm_split_sample_bwd_lp (-dlp on lg); a supplied one through nfdpm_split_prior_bwd on
    the assembled ``out``, into the latent and, through the prior conv, into y and the conv's parameters (it adds to the
    second half of ``d_out`` in place)."""
    B, C, H, W = out.shape
    Ch, P = C // 2, H * W
    f32 = dict(dtype=torch.float32, device=out.device)
    dy = torch.empty(B, Ch, H, W, **f32)
    N.copy_channels(d_out, dy, B, Ch, P, C * P, Ch * P)
    g = {}
    conv = sp.conv
    if eps is None:
        if dlp is not None and conv is None:            # the standard-normal prior ignores y: only the latent's term
            N.split_prior_bwd(dlp, None, 0, None, None, out, C * P, d_out, C * P, None, None, B, C, H, W)
        elif dlp is not None:
            _prior_conv_backward(sp, out, dy, Ch * P, wgrad, g, lambda hs, ldh, dh, dpar: N.split_prior_bwd(
                dlp, hs, ldh, conv.bias, conv.logs, out, C * P, d_out, C * P, dh, dpar, B, C, H, W))
        dz = torch.empty(B, Ch, H, W, **f32)
        N.copy_channels(d_out.view(-1)[Ch * P:], dz, B, Ch, P, C * P, Ch * P)
        return dy, dz, g
    if conv is None:                                    # the standard-normal prior has no parameters and ignores y
        return dy, None, g
    if isinstance(temperature, Tensor):                 # per-image temperatures [B]
        _prior_conv_backward(sp, out, dy, Ch * P, wgrad, g, lambda hs, ldh, dh, dpar: N.split_sample_bwd_ex(
            d_out.view(-1)[Ch * P:], C * P, eps, 1.0, temperature, dlp, hs, ldh, conv.bias, conv.logs, dh, dpar, B, C, H, W))
    else:
        _prior_conv_backward(sp, out, dy, Ch * P, wgrad, g, lambda hs, ldh, dh, dpar: N.split_sample_bwd_lp(
            d_out.view(-1)[Ch * P:], C * P, dlp, eps, temperature, hs, ldh, conv.bias, conv.logs, dh, dpar, B, C, H, W))
    return dy, None, g


def _prior_conv_backward(sp, out: Tensor, dy: Tensor, dy_bs: int, wgrad: bool, g: dict, prior_bwd) -> None:
    """The Split prior conv's part of a Split backward: recompute its rows hs from the first half of ``out`` [B,C,H,W]
    (im2col + fp32 GEMM), run ``prior_bwd(hs, ldh, dh, dpar)`` (the prior kernel's backward, which writes dh and the
    per-image bias / logs partials), then the conv's wgrad (with ``wgrad``, into ``g``) and dgrad + col2im into the first
    C/2 channels of ``dy`` (batch stride ``dy_bs``)."""
    B, C, H, W = out.shape
    Ch, P, M = C // 2, H * W, B * H * W
    f32 = dict(dtype=torch.float32, device=out.device)
    conv = sp.conv
    Ks, Kp, ldh = Ch * 9, E.round_up(Ch * 9, 16), E.round_up(C, 16)
    wp = torch.empty(ldh * Kp, **f32)
    N.pack_matrix(conv.weight, wp, 1, C, Ks, 0, Ks, 1, Kp, ldh)
    wst = torch.empty(Kp * ldh, **f32)
    N.pack_matrix(conv.weight, wst, Ks, 1, C, 1, 0, Ks, ldh, Kp)
    As = torch.empty(M * Kp, **f32)
    N.im2col3x3(out, As, B, Ch, H, W, C * P, Kp)
    hs = torch.empty(M * ldh, **f32)
    N.gemm_nt(As, Kp, wp, Kp, hs, ldh, M, C, Kp)
    dh = torch.empty(M * ldh, **f32)
    dpar = torch.empty(B * 2 * C, **f32)
    prior_bwd(hs, ldh, dh, dpar)
    if wgrad:
        g[conv.bias], g[conv.logs] = torch.empty_like(conv.bias), torch.empty_like(conv.logs)
        N.reduce_rows2(dpar, g[conv.bias], g[conv.logs], B, C, C, 2 * C)
        dws = torch.empty(C * Kp, **f32)
        ws = torch.empty(N.gemm_tn_workspace(M, C, Kp), **f32)
        N.gemm_tn(dh, ldh, As, Kp, dws, M, C, Kp, ws, fused_reduce=False)
        g[conv.weight] = torch.empty_like(conv.weight)
        N.pack_matrix(dws, g[conv.weight], C, 1, Ks, Kp, 0, 1, Ks, C)        # drop the K padding
    dAs = torch.empty(M * Kp, **f32)
    N.gemm_nt(dh, ldh, wst, ldh, dAs, Kp, M, Kp, ldh)
    N.col2im_add(dAs, Kp, dy, dy_bs, B, Ch, H, W)


def _wants_grad(mod) -> bool:
    return any(p.requires_grad for p in mod.parameters())


def _coupling_forward(cp, x: Tensor, ld: Optional[Tensor]):
    """AffineCoupling.transform keeping the coupling network's operands (im2col rows, hidden maps, ZeroConv taps)."""
    B, C, H, W = x.shape
    P = H * W
    zc = cp.net[4]
    pm, ldp = E.coupling_rows(cp, x, C * P, B, C, H, W, init=True, stash=True)
    y = torch.empty_like(x)
    T = N.ld_tiles(P)
    part = torch.empty(T * B, dtype=torch.float32, device=x.device) if ld is not None else None
    N.coupling_apply(pm, ldp, zc.bias, zc.logs, x, y, part, B, C, H, W, C * P, C * P, False)
    if ld is not None:
        N.accumulate(ld, part, T, B)
    return y


def _coupling_backward(cp, st: SimpleNamespace, x: Tensor, dy: Tensor, dld32: Optional[Tensor], inverse: bool = False,
                       wgrad: bool = True, col2im: bool = True):
    """Backward of AffineCoupling.transform (``x`` its input) or, with ``inverse``, of AffineCoupling.invert (``x`` the
    inverse's input y, ``dy`` the gradient of its output; ``dld32`` None or the gradient of the log-det the inverse
    accumulated): coupling_bwd / coupling_inv_bwd_ld, then the coupling
    network (``_net_backward``).  ``wgrad=False`` skips every parameter gradient (frozen network).  With
    ``col2im=False`` the network's im2col-row gradient dA1 is returned as a third value instead of being added to du (the
    caller fuses it into the next mix_bwd)."""
    B, C, H, W = x.shape
    P, M = H * W, B * H * W
    f32 = dict(dtype=torch.float32, device=x.device)
    zc = cp._parts()[4]
    Kp3 = E.round_up(9 * C, 64)
    g = {}
    du = torch.empty_like(x)
    dpm = torch.empty(M * Kp3, dtype=st.dt, device=x.device)
    T_c = N.coupling_bwd_tiles(C, H, W)
    dpar3 = torch.empty(B * T_c * 2 * C, **f32)
    if wgrad:
        g[zc.bias], g[zc.logs] = torch.empty_like(zc.bias), torch.empty_like(zc.logs)
    fused = dict(dbias=g[zc.bias], dlogs=g[zc.logs]) if wgrad and T_c == 1 else {}
    tiled = dict(dp_scratch=torch.empty(M * C, **f32)) if T_c > 1 else {}
    if inverse:
        N.coupling_inv_bwd_ld(dy, C * P, dld32, x, C * P, st.pm, st.ldp, zc.bias, zc.logs, du, C * P, dpm, Kp3, dpar3, B, C,
                              H, W, **fused, **tiled)
    else:
        N.coupling_bwd(dy, C * P, dld32, x, C * P, st.pm, st.ldp, zc.bias, zc.logs, du, C * P, dpm, Kp3, dpar3, B, C, H, W,
                       **fused, **tiled)
    if wgrad and T_c > 1:
        N.reduce_rows2(dpar3, g[zc.bias], g[zc.logs], B * T_c, C, C, 2 * C)
    dA1 = _net_backward(cp, st, dpm, du if col2im else None, B, C, H, W, g, wgrad)
    return (du, g) if col2im else (du, g, dA1)


def _net_backward(cp, st: SimpleNamespace, dpm: Tensor, dstate: Optional[Tensor], B: int, C: int, H: int, W: int, g: dict,
                  wgrad: bool) -> Tensor:
    """The coupling network's backward from d(pm): dgrad3 + wgrad3 -> ActNorm/ReLU bwd -> wgrad2 + dgrad2 -> ActNorm/ReLU
    bwd -> wgrad1 + dgrad1 -> col2im into the first C/2 channels of ``dstate`` (the per-StepFlow section of
    _train.backward_train on one stream; ``dstate=None`` leaves the col2im to the caller).  Parameter gradients go into
    ``g``; ``wgrad=False`` runs the dgrad chain only.  Returns the im2col-row gradient dA1 [M, K1p]."""
    from . import _train as T
    Ch, P, M = C // 2, H * W, B * H * W
    dev = dpm.device
    f32 = dict(dtype=torch.float32, device=dev)
    conv1, an1, conv2, an2, zc = cp._parts()
    F = conv1.weight.shape[0]
    dt, K1p, ldp = st.dt, st.K1p, st.ldp
    tc = dt in E.TC_DTYPES
    Kp3 = E.round_up(9 * C, 64)
    # transposed (dgrad) weight operands of THIS coupling network, packed like the whole-Glow path packs them
    plan = getattr(cp, "_granular_plan", None)
    if plan is None or plan.dt != dt or not plan.valid():
        plan = cp._granular_plan = E.PackPlan([SimpleNamespace(affcoupling=cp)], dt, True)
    plan.refresh()
    bc = cp._bwd_caches[dt]
    ws = torch.empty(max(N.gemm_tn_workspace(M, F, F), N.gemm_tn_workspace(M, ldp, F), N.gemm_tn_workspace(M, F, K1p)),
                     **f32) if wgrad else None
    rows_cta = T.ROWS_PER_CTA
    while rows_cta > 8 and (M + rows_cta - 1) // rows_cta < 256:
        rows_cta //= 2
    n_cta = (M + rows_cta - 1) // rows_cta
    an_part = torch.empty(n_cta * 2 * F, **f32)
    dh = torch.empty(M * F, dtype=dt if dt == torch.bfloat16 else torch.float32, device=dev)
    dpre, dpre1 = torch.empty(M * F, dtype=dt, device=dev), torch.empty(M * F, dtype=dt, device=dev)
    # ZeroConv 3x3
    if wgrad:
        g[zc.weight] = torch.empty_like(zc.weight)
        if tc:
            N.gemm_tn(dpm, Kp3, st.h2, F, g[zc.weight], M, ldp, F, ws, out_mode=N.TN_OUT_TAPS, out_c=C)
        else:
            d3 = torch.empty(ldp * F, **f32)
            N.gemm_tn(dpm, Kp3, st.h2, F, d3, M, ldp, F, ws, fused_reduce=False)
            N.pack_matrix(d3, g[zc.weight], C, F, 9, F, 1, C * F, 9, C * F)
    # second Conv2dActNorm (1x1)
    N.gemm_nt(dpm, Kp3, bc.w3t, Kp3, dh, F, M, F, Kp3)
    N.actnorm_relu_bwd(dh, F, st.h2, F, an2.scale, dpre, F, an_part, M, F, rows_cta)
    if wgrad:
        g[an2.scale], g[an2.bias] = torch.empty_like(an2.scale), torch.empty_like(an2.bias)
        N.reduce_rows2(an_part, g[an2.scale], g[an2.bias], n_cta, F, F, 2 * F)
        g[conv2.weight] = torch.empty_like(conv2.weight)
        N.gemm_tn(dpre, F, st.h1, F, g[conv2.weight], M, F, F, ws, fused_reduce=tc)
    # first Conv2dActNorm (3x3)
    N.gemm_nt(dpre, F, bc.w2t, F, dh, F, M, F, F)
    N.actnorm_relu_bwd(dh, F, st.h1, F, an1.scale, dpre1, F, an_part, M, F, rows_cta)
    if wgrad:
        g[an1.scale], g[an1.bias] = torch.empty_like(an1.scale), torch.empty_like(an1.bias)
        N.reduce_rows2(an_part, g[an1.scale], g[an1.bias], n_cta, F, F, 2 * F)
        g[conv1.weight] = torch.empty_like(conv1.weight)
        if tc:
            N.gemm_tn(dpre1, F, st.A1, K1p, g[conv1.weight], M, F, K1p, ws, out_mode=N.TN_OUT_STRIP, out_c=Ch * 9)
        else:
            d1 = torch.empty(F * K1p, **f32)
            N.gemm_tn(dpre1, F, st.A1, K1p, d1, M, F, K1p, ws, fused_reduce=False)
            T._strip_cols(d1, g[conv1.weight], F, K1p, Ch * 9)
    dA1 = torch.empty(M * K1p, **f32)
    N.gemm_nt(dpre1, F, bc.w1t, F, dA1, K1p, M, K1p, F)
    if dstate is not None:
        N.col2im_add(dA1, K1p, dstate, C * P, B, Ch, H, W)  # the kept half also feeds the coupling network
    return dA1


def _split_backward(sp, x: Tensor, dy_kept: Optional[Tensor], dz: Optional[Tensor], dlp32: Optional[Tensor]):
    """Backward of (y, z) = chunk(x), logp += N(z; mean(y), exp(logs(y))) (transforms.py:285-289)."""
    B, C, H, W = x.shape
    Ch, P = C // 2, H * W
    dx = torch.zeros_like(x)
    if dy_kept is not None:
        N.copy_channels(dy_kept.to(torch.float32).contiguous(), dx, B, Ch, P, Ch * P, C * P)
    if dz is not None:
        N.copy_channels(dz.to(torch.float32).contiguous(), dx.view(-1)[Ch * P:], B, Ch, P, Ch * P, C * P)
    g = {}
    if dlp32 is None:
        return dx, g
    conv = sp.conv
    if conv is None:
        N.split_prior_bwd(dlp32, None, 0, None, None, x, C * P, dx, C * P, None, None, B, C, H, W)
        return dx, g
    _prior_conv_backward(sp, x, dx, C * P, True, g, lambda hs, ldh, dh, dpar: N.split_prior_bwd(
        dlp32, hs, ldh, conv.bias, conv.logs, x, C * P, dx, C * P, dh, dpar, B, C, H, W))
    return dx, g


# ------------------------------------------------------------------------------------------- the Function
class ModuleTransformFn(torch.autograd.Function):
    """(x, log_det_jac | None, logp | None, *parameters) -> (outputs..., log_det_jac?, logp?) for one granular transform."""

    @staticmethod
    def forward(ctx, mod, what, raw_forward, x, ld, lp, *params):
        ctx.mod, ctx.what = mod, what
        ctx.have_ld, ctx.have_lp = ld is not None, lp is not None
        ctx.params = params
        st = None
        if what == "AffineCoupling":
            E.last_coupling_stash = None
            y = _coupling_forward(mod, x, ld)
            st = E.last_coupling_stash
            E.last_coupling_stash = None
            outs = (y,)
        else:
            out = raw_forward(mod, x, ld, lp)              # the module's own kernels (no recording: we are inside forward())
            outs = (out[0], out[2]) if what == "Split" else (out[0],)
        ctx.stash = st
        ctx.save_for_backward(x)
        dirty = [t for t in (ld, lp) if t is not None]
        if dirty:
            ctx.mark_dirty(*dirty)
        return tuple(outs) + tuple(dirty)

    @staticmethod
    def backward(ctx, *gout):
        (x,) = ctx.saved_tensors
        mod, what = ctx.mod, ctx.what
        B = x.shape[0]
        dev = x.device
        n_out = 2 if what == "Split" else 1
        g_outs = gout[:n_out]
        rest = list(gout[n_out:])
        g_ld = rest.pop(0) if ctx.have_ld else None
        g_lp = rest.pop(0) if ctx.have_lp else None
        dy = g_outs[0]
        dy32 = dy.to(torch.float32).contiguous() if dy is not None else (None if what in ("Squeeze", "Split") else torch.zeros_like(x))
        grads = {}
        if what == "Squeeze":
            Bc, C, H, W = x.shape
            dx = torch.empty_like(x)
            if dy is None:
                dx.zero_()
            else:
                N.unsqueeze(dy32, dx, Bc, 4 * C, H // 2, W // 2, C * H * W, C * H * W)
        elif what == "ActNorm":
            dx, _, dS, dB = _mix_backward(mod, x, dy32, _f32(g_ld, B, dev), None, mod.scale, mod.bias)
            grads = {mod.scale: dS, mod.bias: dB}
        elif what == "InvConv2d":
            dx, dW, _, _ = _mix_backward(mod, x, dy32, _f32(g_ld, B, dev), mod.weight, None, None)
            grads = {mod.weight: dW}
        elif what == "AffineCoupling":
            dx, grads = _coupling_backward(mod, ctx.stash, x, dy32, _f32(g_ld, B, dev))
        elif what == "Split":
            dx, grads = _split_backward(mod, x, g_outs[0], g_outs[1], _f32(g_lp, B, dev) if ctx.have_lp else None)
        else:                                               # pragma: no cover
            raise NotImplementedError(what)
        ctx.stash = None
        pg = []
        for p in ctx.params:
            gp = grads.get(p) if p.requires_grad else None
            if p.requires_grad and gp is None:
                gp = torch.zeros_like(p)
            pg.append(gp)
        return (None, None, None, dx if ctx.needs_input_grad[3] else None, g_ld, g_lp) + tuple(pg)


def transform(mod, what: str, raw_forward, x: Tensor, ld: Optional[Tensor], lp: Optional[Tensor]):
    """Run ``mod.transform(x, ld, lp)`` under autograd; returns the module's usual tuple."""
    params = [p for p in mod.parameters()]
    for a, name in ((ld, "log_det_jac"), (lp, "logp")):
        if a is not None and a.requires_grad and a.is_leaf:
            raise RuntimeError(f"{name} is updated in place and must not be a leaf that requires grad")
    out = ModuleTransformFn.apply(mod, what, raw_forward, x, ld, lp, *params)
    n_out = 2 if what == "Split" else 1
    outs, rest = out[:n_out], list(out[n_out:])
    ld_o = rest.pop(0) if ld is not None else None
    lp_o = rest.pop(0) if lp is not None else None
    if what == "Split":
        return outs[0], ld_o, outs[1], lp_o
    return outs[0], ld_o, lp_o


# ------------------------------------------------------------------------------------------- invert (NFDPM_INVERT_GRAD=1)
def coupling_invert_stash(cp, y: Tensor, ld_part: Optional[Tensor] = None):
    """AffineCoupling.invert keeping the coupling network's operands, in the operand format of the no-grad inverse.
    ``ld_part``: the log-det partial rows, as the no-grad inverse writes them."""
    B, C, H, W = y.shape
    E.last_coupling_stash = None
    E.coupling_rows(cp, y, C * H * W, B, C, H, W, init=True, stash=True, fmt=E.coupling_dtype())
    st = E.last_coupling_stash
    E.last_coupling_stash = None
    x = torch.empty_like(y)
    zc = cp._parts()[4]
    N.coupling_apply(st.pm, st.ldp, zc.bias, zc.logs, y, x, ld_part, B, C, H, W, C * H * W, C * H * W, True)
    return x, st


class ModuleInvertFn(torch.autograd.Function):
    """(y, latent | None, *parameters) -> x for one granular ``invert``.  ``draw``: (temperature, seeds) of a Split, as
    ``E.sampling_inputs`` returns them."""

    @staticmethod
    def forward(ctx, mod, what, raw_invert, draw, y, latent, *params):
        temperature, seeds = draw
        ctx.mod, ctx.what, ctx.temperature, ctx.params = mod, what, temperature, params
        ctx.stash = ctx.eps = None
        if what == "AffineCoupling":
            x, ctx.stash = coupling_invert_stash(mod, y)
        elif what == "Split":                              # Split.invert, keeping the drawn eps
            B, Ch, H, W = y.shape
            x = torch.empty(B, 2 * Ch, H, W, dtype=torch.float32, device=y.device)
            N.copy_channels(y, x, B, Ch, H * W, Ch * H * W, 2 * Ch * H * W)
            sink = []
            mod._fill_second_half(x, 2 * Ch * H * W, B, 2 * Ch, H, W, latent, temperature, eps_sink=sink, seeds=seeds)
            ctx.eps = sink[0] if sink else None
            ctx.save_for_backward(y, x)
            return x
        else:
            x = raw_invert(mod, y)
        ctx.save_for_backward(y)
        return x

    @staticmethod
    def backward(ctx, dx):
        if ctx.what == "AffineCoupling" and ctx.stash is None:
            raise RuntimeError("AffineCoupling.invert: the stash of this call was released by an earlier backward")
        mod, what = ctx.mod, ctx.what
        y = ctx.saved_tensors[0]
        dx = dx.to(torch.float32).contiguous()
        wgrad = any(p.requires_grad for p in ctx.params)
        grads, d_lat = {}, None
        if what == "Squeeze":
            B, C, H, W = y.shape
            dy = torch.empty_like(y)
            N.squeeze(dx, dy, B, C // 4, 2 * H, 2 * W, C * H * W, C * H * W)
        elif what == "ActNorm":
            dy, _, dS, dB = _mix_inv_backward(mod._mix, y, dx, None, mod.scale, mod.bias, wgrad)
            grads = {mod.scale: dS, mod.bias: dB}
        elif what == "InvConv2d":
            dy, dW, _, _ = _mix_inv_backward(mod._mix, y, dx, mod.weight, None, None, wgrad)
            grads = {mod.weight: dW}
        elif what == "AffineCoupling":
            dy, grads = _coupling_backward(mod, ctx.stash, y, dx, None, inverse=True, wgrad=wgrad)
        elif what == "Split":
            dy, d_lat, grads = _split_sample_backward(mod, ctx.saved_tensors[1], ctx.eps, ctx.temperature, dx, wgrad)
        else:                                               # pragma: no cover
            raise NotImplementedError(what)
        ctx.stash = None
        pg = [grads.get(p) if p.requires_grad else None for p in ctx.params]
        return (None, None, None, None, dy if ctx.needs_input_grad[4] else None,
                d_lat if ctx.needs_input_grad[5] else None) + tuple(pg)


def invert(mod, what: str, raw_invert, y: Tensor, latent: Optional[Tensor] = None, temperature=1.0,
           seeds: Optional[Tensor] = None):
    """Run ``mod.invert`` under autograd (one ModuleInvertFn node)."""
    y = E.check_input(y)
    if isinstance(temperature, Tensor) or seeds is not None:
        draw = E.sampling_inputs(temperature, seeds, y.shape[0], y.device)
    else:
        draw = (float(temperature), None)
    return ModuleInvertFn.apply(mod, what, raw_invert, draw, y, latent, *mod.parameters())
