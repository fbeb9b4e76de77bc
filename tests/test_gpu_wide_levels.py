"""Levels wider than 192 channels (GPU): the final levels of L6 / L7 models on RGB input (384 and 768 channels), whose C x C
mix matrix does not fit shared memory.  nfdpm_channel_mix, nfdpm_mix_bwd and nfdpm_mix_inv_param_grad run them with the
multi-CTA kernels of csrc/wide_mix.cu; every other kernel such a level reaches is covered through the model tests
against the CPU oracle.

Tolerances: kernel sinks by the fp32 rule of kernel_refs (relative L2 1e-5, max |error| 1e-4 of max |ref|; d(weight)
1e-4 as in test_gpu_train_kernels.py); model outputs as the config-4 test (z 1e-4 relative, log-det / log-p rtol 1e-5 with
atol 5e-2, round trip 1e-3); training gradients as test_gpu_train.py (fp32_simt 2e-4 per tensor, bf16 8e-2); the
recorded inverse as test_gpu_invert_density_grad.py."""
import math
import os

import numpy as np
import pytest
import torch

import normalizing_flow as nf
from normalizing_flow import _engine as E
from normalizing_flow import _native as N
from oracle import glow_oracle as O
from kernel_refs import DEV, WORST, Sink, check, im2col_rows, mix_ref, report_worst, rnd, same_bits

pytestmark = pytest.mark.gpu
TOL_DW = 1e-4


@pytest.fixture(autouse=True)
def _report_worst(request):
    WORST.clear()
    yield
    report_worst(request.node.name)


def relerr(a, b):
    a, b = a.detach().cpu().double(), torch.as_tensor(b).detach().cpu().double()
    return float((a - b).norm() / (b.norm() + 1e-30))


def _prepare(w, s, b, C):
    cache = E.MixCache()
    dv = lambda t: None if t is None else t.to(DEV).contiguous()
    E.prepare_mix([(cache, dv(w), dv(s), dv(b), C, None)])
    return cache


def _wsb(C, seed):
    w = (torch.linalg.qr(rnd(C, C, seed=seed).double())[0].float() + 0.1 * rnd(C, C, seed=seed + 1) / math.sqrt(C))
    return w.contiguous(), rnd(C, seed=seed + 2, scale=0.3), rnd(C, seed=seed + 3, scale=0.3)


def _kernel_names(fn):
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}


# ------------------------------------------------------------------------------------------------ wide K-A / K-A^-1
_KA = [(C, P) for C in (193, 194, 256, 390, 512, 768, 1024) for P in (1, 3, 4, 16, 64)]


@pytest.mark.parametrize("C,P", _KA, ids=[f"C{c}-P{p}" for c, p in _KA])
def test_wide_channel_mix(C, P):
    """Forward and inverse matrices of mix_prepare, strided batches (gaps of 4 and 8 floats keep the V = 4 path when
    P % 4 == 0), against fp64; the stride gaps and the slack stay untouched."""
    B = 3
    w, s, b = _wsb(C, 10 + C)
    mix = _prepare(w, s, b, C)
    x = rnd(B, C * P + 4, seed=C + P)
    xbs, ybs = C * P + 4, C * P + 8
    written = (torch.arange(ybs) < C * P).expand(B, ybs)
    for mt, beta in ((mix.fwd_mt, mix.fwd_beta), (mix.inv_mt, mix.inv_beta)):
        y = Sink(B * ybs)
        N.channel_mix(x.to(DEV), y.t, mt, beta, B, C, P, xbs, ybs)
        torch.cuda.synchronize()
        got = y.get(written).view(B, ybs)[:, :C * P].view(B, C, P)
        m64, b64 = mt.cpu().double().view(C, C), beta.cpu().double()
        ref = torch.einsum("io,bip->bop", m64, x[:, :C * P].double().view(B, C, P)) + b64.view(1, C, 1)
        check(f"y C={C} P={P}", got, ref)


def test_channel_mix_192_keeps_the_single_pass_kernel():
    """C = 192 still runs chanmix_generic_kernel (bit-identical to before: the same launch); C = 193 the wide kernel."""
    for C, want in ((192, "chanmix_generic_kernel"), (193, "chanmix_wide_kernel")):
        w, s, b = _wsb(C, 5)
        mix = _prepare(w, s, b, C)
        x = rnd(2, C, 16, seed=1).to(DEV)
        y = torch.empty_like(x)
        names = _kernel_names(lambda: N.channel_mix(x, y, mix.fwd_mt, mix.fwd_beta, 2, C, 16, C * 16, C * 16))
        assert any(want in n for n in names), names
        assert not any(("chanmix_wide_kernel" if want != "chanmix_wide_kernel" else "chanmix_generic") in n for n in names)


def test_channel_mix_rejects_1025_before_any_launch():
    x = torch.zeros(1, 1025, 1, device=DEV)
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        with pytest.raises(RuntimeError, match="1025 > 1024"):
            N.channel_mix(x, x, x, x, 1, 1025, 1, 1025, 1025)
        with pytest.raises(RuntimeError, match="1025 > 1024"):
            N.mix_bwd(x, 1025, None, 0, x, 1025, x, x, 1025, x, 1, 1025, 1, 1)
        torch.cuda.synchronize()
    assert not [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


# ------------------------------------------------------------------------------------------------ wide mix backward
_BWD = [(2, 256, 2, 2), (2, 384, 4, 4), (3, 384, 1, 1), (2, 768, 2, 2), (2, 768, 1, 1), (2, 256, 5, 3)]


@pytest.mark.parametrize("with_da1", [False, True])
@pytest.mark.parametrize("B,C,H,W", _BWD, ids=[f"{c}x{h}x{w}" for _, c, h, w in _BWD])
def test_wide_mix_bwd(B, C, H, W, with_da1):
    """Objective <y, du> (+ <im2col(y_a), da1>) + sum_b dld[b] P (sum s + log|det W|), y = W exp(s)(x + b): dx and the
    per-image partials from mix_bwd (one row per image), d(W, s, b) from mix_param_grad, against fp64 autograd."""
    P, Ch, M = H * W, C // 2, B * H * W
    assert N.mix_bwd_tiles(C, H, W) == 1
    w, s, b = _wsb(C, 20 + C)
    x, du, dld = rnd(B, C, P, seed=5), rnd(B, C, P, seed=6), rnd(B, seed=7)
    lda1 = 9 * Ch + 8
    da1 = rnd(M, lda1, seed=8)
    mix = _prepare(w, s, b, C)
    dx_bs = (C + 1) * P
    dx = Sink(B * dx_bs)
    part = Sink(B * (C * C + C))
    N.mix_bwd(du.to(DEV), C * P, da1.to(DEV) if with_da1 else None, lda1 if with_da1 else 0, x.to(DEV), C * P,
              mix.fwd_mt, dx.t, dx_bs, part.t, B, C, H, W)
    dW, dS, dB, scratch = Sink(C * C), Sink(C), Sink(C), Sink(C * C + C)
    wd, sd, bd = w.to(DEV), s.to(DEV), b.to(DEV)
    dld_sum = dld.sum().view(1).to(DEV)
    N.mix_param_grad([N.MixGradItem(part=part.t.data_ptr(), B=B, C=C, weight=wd.data_ptr(), scale=sd.data_ptr(),
                                    bias=bd.data_ptr(), winv=mix.winv.data_ptr(), dld_sum=dld_sum.data_ptr(), P=float(P),
                                    pad_=0, d_weight=dW.t.data_ptr(), d_scale=dS.t.data_ptr(), d_bias=dB.t.data_ptr(),
                                    scratch=scratch.t.data_ptr())])
    torch.cuda.synchronize()
    got_dx = dx.get((torch.arange(C + 1) < C).view(1, C + 1, 1).expand(B, C + 1, P)).view(B, C + 1, P)[:, :C]
    got_part = part.get().view(B, C * C + C)
    scratch.get()
    xl, wl, sl, bl = (t.double().requires_grad_(True) for t in (x.view(B, C, H, W), w, s, b))
    y, ld = mix_ref(xl, wl, sl, bl)
    obj = (y * du.double().view(B, C, H, W)).sum()
    du_full = du.double().clone()
    if with_da1:
        yl = y[:, :Ch]
        obj = obj + (im2col_rows(yl) * da1.double()[:, :9 * Ch]).sum()
        # the complete du of the K-A output: du plus the col2im of da1 on the first half
        ya = torch.zeros(B, Ch, H, W, dtype=torch.float64, requires_grad=True)
        (im2col_rows(ya) * da1.double()[:, :9 * Ch]).sum().backward()
        du_full[:, :Ch] += ya.grad.view(B, Ch, P)
    (obj + dld.double().sum() * ld).backward()
    check("dx", got_dx, xl.grad.view(B, C, P))
    # partial layout: [b][o*C + i] = sum_p du[o] x[i], [b][C*C + o] = sum_p du[o]
    xm = x.double()
    check("part dW^", got_part[:, :C * C].view(B, C, C), torch.einsum("bop,bip->boi", du_full, xm))
    check("part db^", got_part[:, C * C:], du_full.sum(2))
    check("dW", dW.get(), wl.grad, TOL_DW, TOL_DW)
    check("ds", dS.get(), sl.grad)
    check("db", dB.get(), bl.grad)


@pytest.mark.parametrize("C,H,W,with_w,with_dld", [(256, 2, 2, True, True), (384, 2, 2, True, False), (384, 1, 1, False, True),
                                                   (768, 1, 1, True, True), (768, 2, 2, False, False)])
def test_wide_mix_inv_param_grad(C, H, W, with_w, with_dld):
    """mix_bwd (inv_mt) + mix_inv_param_grad of the inverse x = diag(e^-s) W^-1 u - b, with and without dld_sum and
    with weight NULL (a lone ActNorm), against fp64 autograd."""
    from normalizing_flow import _modgrad as MG
    B, P = 3, H * W
    w, s, b = _wsb(C, 30 + C)
    w = w.double() if with_w else None
    s, b = s.double(), b.double()
    u, dx, dld = rnd(B, C, H, W, seed=5), rnd(B, C, H, W, seed=6), rnd(B, seed=7)
    dv = lambda t: t.float().to(DEV).contiguous()
    wg = None if w is None else dv(w).view(C, C, 1, 1)
    du, dW, dS, dB = MG._mix_inv_backward(E.MixCache(), u.to(DEV), dx.to(DEV), wg, dv(s).view(C, 1, 1),
                                          dv(b).view(C, 1, 1), True, None, 0,
                                          MG._dld_sum(dld.to(DEV)) if with_dld else None)
    torch.cuda.synchronize()
    leaves = [t.float().double().requires_grad_(True) if t is not None else None for t in (w, s, b)]
    ul = u.double().requires_grad_(True)
    x, const = ul, 0.0
    if leaves[0] is not None:
        x = torch.einsum("oi,bihw->bohw", torch.linalg.inv(leaves[0]), x)
        const = const + torch.linalg.slogdet(leaves[0])[1]
    x = x * torch.exp(-leaves[1]).view(1, C, 1, 1) - leaves[2].view(1, C, 1, 1)
    const = const + leaves[1].sum()
    obj = (x * dx.double()).sum()
    if with_dld:
        obj = obj + dld.double().sum() * P * const
    obj.backward()
    check("du", du.cpu(), ul.grad)
    if w is not None:
        check("dW", dW.view(C, C).cpu(), leaves[0].grad, TOL_DW, TOL_DW)
    check("ds", dS.view(C).cpu(), leaves[1].grad)
    check("db", dB.view(C).cpu(), leaves[2].grad)


def test_mix_bwd_192_keeps_the_single_pass_kernel():
    for C, want in ((192, "mix_bwd_kernel"), (194, "mix_bwd_part_wide_kernel")):
        x = rnd(2, C, 16, seed=1).to(DEV)
        mix = _prepare(*_wsb(C, 3), C)
        part = torch.empty(2 * N.mix_bwd_tiles(C, 4, 4) * (C * C + C), device=DEV)
        dx = torch.empty_like(x)
        names = _kernel_names(lambda: N.mix_bwd(x, C * 16, None, 0, x, C * 16, mix.fwd_mt, dx, C * 16, part, 2, C, 4, 4))
        assert any(n.split("(")[0].endswith(want) or want in n for n in names), names


# ------------------------------------------------------------------------------------------------ the model vs the oracle
_GEO = [(6, 2, 64, 3), (6, 2, 128, 2), (7, 1, 128, 2)]


def _flow(c, L, K, seed):
    sd, psd = O.seeded_state(c, L, K, seed)
    flow = nf.Glow(c, L, K).to(DEV)
    flow.load_state_dict(sd, strict=True)
    return flow, sd, psd


@pytest.mark.parametrize("L,K,S,B", _GEO, ids=[f"L{g[0]}K{g[1]}-{g[2]}px" for g in _GEO])
def test_model_against_oracle(L, K, S, B, monkeypatch):
    monkeypatch.setenv("NFDPM_PRECISION", "fp32")
    c = 3
    flow, sd, _ = _flow(c, L, K, 40 + L)
    x = O.seeded_input((B, c, S, S), 41).to(DEV)
    shapes = [tuple(z) for z in O.output_shapes(L, c, S)]
    assert max(s[0] for s in shapes) == 2 ** (L + 1) * c
    ld_o, lp_o = torch.zeros(B, dtype=torch.float64), torch.zeros(B, dtype=torch.float64)
    zo, ld_o, lp_o = O.glow_transform(sd, x.cpu(), L, K, ld_o, lp_o)
    xo = O.glow_invert(sd, zo, L, K)
    # the reference's own round trip is not exact (s forward, s + 1e-6 inverse): it grows with the number of steps
    rt = max(1e-3, 2 * float((xo - x.cpu()).abs().max()))
    results = {}
    for graphs, fused in (("1", "1"), ("0", "1"), ("1", "0")):
        monkeypatch.setenv("NFDPM_GRAPHS", graphs)
        monkeypatch.setenv("NFDPM_FUSED_BOUNDARY", fused)
        with torch.no_grad():
            ld = torch.zeros(B, dtype=torch.float64, device=DEV)
            lp = torch.zeros(B, dtype=torch.float64, device=DEV)
            zs, ld, lp = flow.transform(x, ld, lp)
            xr = flow.invert(zs)
        results[(graphs, fused)] = (zs, ld, lp, xr)
    zs, ld, lp, xr = results[("1", "1")]
    assert [tuple(z.shape[1:]) for z in zs] == shapes
    for key, (zs2, ld2, lp2, xr2) in results.items():
        for a, b in zip(zs2, zs):
            assert relerr(a, b) < 1e-5, key
        assert relerr(ld2, ld) < 1e-6 and relerr(lp2, lp) < 1e-6, key
        assert (xr2 - x).abs().max() < rt, key
    for a, b in zip(zs, zo):
        assert relerr(a, b) < 1e-4
    np.testing.assert_allclose(ld.cpu().numpy(), ld_o.numpy(), rtol=1e-5, atol=5e-2)
    np.testing.assert_allclose(lp.cpu().numpy(), lp_o.numpy(), rtol=1e-5, atol=5e-2)
    # decoding the oracle's latents: the inverse chain of these seeded weights amplifies fp32 rounding, so the bound is
    # the oracle's own round-trip error (its decode of its latents against the image they came from)
    with torch.no_grad():
        xd = flow.invert([z.float().to(DEV) for z in zo])
    e_dec, e_own = relerr(xd, xo), relerr(xo, x)
    print(f"decode vs oracle {e_dec:.2e}, oracle round trip {e_own:.2e}")
    assert e_dec < max(1e-4, 4 * e_own)
    # seeded sampling with per-image temperatures: level 0's Split draws, the deeper latents (the wide levels included)
    # are supplied (draws at every Split of these seeded random weights overflow, in the oracle too).  The same image
    # whatever the batch, and transform(sample) returns the supplied latents.
    seeds = torch.arange(B, dtype=torch.int64, device=DEV) * 7 + 1
    temps = torch.linspace(0.5, 0.9, B, device=DEV)
    with torch.no_grad():
        lat = [z.contiguous() for z in zs[1:]]
        xs = flow.sample(lat, temperature=temps, seeds=seeds)
        x1 = flow.sample([z[1:2].contiguous() for z in lat], temperature=temps[1:2].contiguous(),
                         seeds=seeds[1:2].contiguous())
        zb, _, _ = flow.transform(xs, torch.zeros(B, device=DEV), None)
    assert bool(torch.isfinite(xs).all())
    assert relerr(x1, xs[1:2]) < 1e-5
    for a, b in zip(zb[1:], lat):
        assert relerr(a, b) < 1e-3


def test_wider_than_1024_is_refused_before_init():
    """L8 on RGB: the final level has 1536 channels.  The calls refuse it before the data-dependent initialisation."""
    flow = nf.Glow(3, 8, 1).to(DEV)
    x = torch.randn(1, 3, 256, 256, device=DEV)
    with pytest.raises(ValueError, match="1536 channels"):
        flow.transform(x, torch.zeros(1, device=DEV), None)
    assert all(int(m.is_initialized) == 0 for m in flow.modules() if isinstance(m, nf.ActNorm))
    with pytest.raises(ValueError, match="1536 channels"):
        flow.invert([torch.zeros(1, 1536, 1, 1, device=DEV)])
    for mod, shape in ((nf.InvConv2d(1536), (1, 1536, 1, 1)), (nf.ActNorm(1536), (1, 1536, 1, 1)),
                       (nf.StepFlow(1536), (1, 1536, 1, 1))):
        mod = mod.to(DEV)
        with pytest.raises(ValueError, match="1536 channels"):
            mod.transform(torch.zeros(shape, device=DEV), None, None)
        with pytest.raises(ValueError, match="1536 channels"):
            mod.invert(torch.zeros(shape, device=DEV))


# ------------------------------------------------------------------------------------------------ gradients
def _train_grads(flow, prior, x, S):
    B = x.shape[0]
    flow.zero_grad(set_to_none=True)
    ld, lp = nf.initialize_with_zeros(2, B, DEV)
    zs, ld, lp = flow.transform(x, ld, lp)
    lp += prior.compute_log_prob(zs[-1])
    loss = nf.calculate_loss(ld + lp, 32.0, S * S * 3.0)
    loss.backward()
    return loss, {k: p.grad.detach().clone() for k, p in flow.named_parameters()}


# fp32_simt: 2e-3 as test_gpu_train.py::test_gradients_large_images, the fp32 oracle's own error at these image sizes
# (measured worst 1.2e-3: a level-2 coupling conv, not a wide level); fp32 (split pairs) additionally runs the weight-
# gradient GEMMs whose grids exceed the SM count at 384 channels (gemm_tn_reduce_kernel)
@pytest.mark.parametrize("mode,tol", [("fp32_simt", 2e-3), ("fp32", 1e-2), ("bf16", 8e-2)])
def test_training_step_L6_against_oracle(mode, tol, monkeypatch):
    monkeypatch.setenv("NFDPM_PRECISION", mode)
    c, L, K, S, B = 3, 6, 2, 64, 2
    sd, psd = O.seeded_state(c, L, K, 61)
    flow = nf.Glow(c, L, K).to(DEV)
    flow.load_state_dict(sd)
    prior = nf.GaussianPrior(2 ** (L + 1) * c).to(DEV)
    prior.load_state_dict(psd)
    x_cpu = O.seeded_input((B, c, S, S), 62)
    lo, g_o, _ = O.train_grads(sd, psd, x_cpu, L, K, 32.0, S * S * 3.0)
    loss, g = _train_grads(flow, prior, x_cpu.to(DEV), S)
    assert abs(float(loss.detach()) - float(lo)) < (1e-4 if mode != "bf16" else 1e-3)
    worst = max((relerr(g[k], g_o[k]), k) for k in g)
    print(f"[{mode}] worst gradient {worst}")
    assert worst[0] <= tol, worst
    if mode != "bf16":
        _, g2 = _train_grads(flow, prior, x_cpu.to(DEV), S)
        assert all(same_bits(g[k], g2[k]) for k in g), "two identical training steps differ"


def test_invert_with_density_L6_against_oracle(monkeypatch):
    """Decoding (all latents supplied) with the density, back-propagated: the inverse-direction mix kernels at 384
    channels."""
    from test_gpu_invert_density_grad import TOL_SIMT, _density_case
    monkeypatch.delenv("NFDPM_INVERT_GRAD", raising=False)
    monkeypatch.setenv("NFDPM_PRECISION", "fp32_simt")
    e = _density_case("fp32_simt", False, False, c=3, L=6, K=1, B=2, S=64)
    assert e["x"] <= 1e-4 and e["ld"] <= 1e-4 and e["lp"] <= 1e-4, e
    assert max(v for k, v in e.items() if k not in ("x", "ld", "lp", "worst")) <= TOL_SIMT, e


@pytest.mark.parametrize("inverse", [False, True])
def test_standalone_modules_384_under_autograd(inverse, monkeypatch):
    """InvConv2d, ActNorm and StepFlow of a 384-channel level under autograd (the inverse with NFDPM_INVERT_GRAD=1)
    against torch's fp64 autograd over the oracle's arithmetic."""
    monkeypatch.setenv("NFDPM_PRECISION", "fp32_simt")
    monkeypatch.setenv("NFDPM_INVERT_GRAD", "1")
    C, B, H, W = 384, 2, 2, 2
    sd, _ = O.seeded_state(3, 6, 1, 71)
    pre = "final_flows.0."
    ssd = {k[len(pre):]: v for k, v in sd.items() if k.startswith(pre)}
    step = nf.StepFlow(C).to(DEV)
    step.load_state_dict(ssd)
    x = rnd(B, C, H, W, seed=72)
    gy, gl = rnd(B, C, H, W, seed=73), rnd(B, seed=74)
    mods = {"invconv2d": step.invconv2d, "actnorm": step.actnorm, "step": step}

    def ref(name, xo, p):
        """(output, per-image log-det) of the oracle's arithmetic"""
        ld = torch.zeros(B, dtype=torch.float64)
        if name == "step":
            return (O.step_inv(xo, p, ""), ld) if inverse else (O.step_fwd(xo, p, "", ld), ld)
        if name == "invconv2d":
            w = p["invconv2d.weight"]
            if inverse:
                return O.invconv_inv(xo, w), ld
            y, l = O.invconv_fwd(xo, w)
        else:
            if inverse:
                return O.actnorm_inv(xo, p["actnorm.scale"], p["actnorm.bias"]), ld
            y, l = O.actnorm_fwd(xo, p["actnorm.scale"], p["actnorm.bias"])
        return y, ld + l

    for name, mod in mods.items():
        mod.zero_grad(set_to_none=True)
        xg = x.to(DEV).requires_grad_(True)
        if inverse:
            y = mod.invert(xg)
            (y * gy.to(DEV)).sum().backward()
        else:
            ld = torch.zeros(B, device=DEV)
            y, ld, _ = mod.transform(xg, ld, None)
            ((y * gy.to(DEV)).sum() + (ld * gl.to(DEV)).sum()).backward()
        p = {k: v.double().clone().requires_grad_(v.dtype.is_floating_point) for k, v in ssd.items()}
        xo = x.double().requires_grad_(True)
        yo, ldo = ref(name, xo, p)
        obj = (yo * gy.double()).sum()
        if not inverse:
            obj = obj + (ldo * gl.double()).sum()
        obj.backward()
        assert relerr(y, yo) < 1e-5, name
        assert relerr(xg.grad, xo.grad) < 2e-4, name
        for k, prm in mod.named_parameters():
            full = k if name == "step" else f"{name}.{k}"
            if p[full].grad is None or float(p[full].grad.abs().max()) == 0.0:
                continue
            assert relerr(prm.grad, p[full].grad) < 2e-4, (name, k, relerr(prm.grad, p[full].grad))


# ------------------------------------------------------------------------------------------------ 256x256 L6
def test_256_L6_K4_against_oracle(monkeypatch):
    monkeypatch.setenv("NFDPM_PRECISION", "fp32")
    c, L, K, S, B = 3, 6, 4, 256, 2
    flow, sd, _ = _flow(c, L, K, 81)
    x = O.seeded_input((B, c, S, S), 82).to(DEV)
    with torch.no_grad():
        ld = torch.zeros(B, dtype=torch.float64, device=DEV)
        lp = torch.zeros(B, dtype=torch.float64, device=DEV)
        zs, ld, lp = flow.transform(x, ld, lp)
        xr = flow.invert(zs)
    assert zs[-1].shape == (B, 384, 4, 4)
    ld_o, lp_o = torch.zeros(1, dtype=torch.float64), torch.zeros(1, dtype=torch.float64)
    zo, ld_o, lp_o = O.glow_transform(sd, x.cpu()[1:2], L, K, ld_o, lp_o)
    for a, b in zip(zs, zo):
        assert relerr(a[1:2], b) < 1e-4
    np.testing.assert_allclose(ld.cpu().numpy()[1:2], ld_o.numpy(), rtol=1e-5, atol=5e-2)
    np.testing.assert_allclose(lp.cpu().numpy()[1:2], lp_o.numpy(), rtol=1e-5, atol=5e-2)
    # the round trip of these seeded weights is not exact in the reference either (s forward, s + 1e-6 inverse, fp32)
    xo = O.glow_invert(sd, zo, L, K)
    e_own = float((xo - x.cpu()[1:2]).abs().max())
    print(f"round trip {float((xr - x).abs().max()):.2e}, oracle's own {e_own:.2e}")
    assert (xr - x).abs().max() < max(1e-3, 2 * e_own)


def test_256_L6_K32_properties(tmp_path):
    from diffusion_prior import CatFormater
    c, L, K, S, B = 3, 6, 32, 256, 2
    torch.manual_seed(0)
    flow = nf.Glow(c, L, K).to(DEV)
    prior = nf.GaussianPrior(2 ** (L + 1) * c).to(DEV)
    x = O.seeded_input((B, c, S, S), 91).to(DEV) * 0.5
    with torch.no_grad():
        zs, ld, lp = flow.transform(x, *nf.initialize_with_zeros(2, B, DEV))      # data-dependent init
    assert flow._ready()
    with torch.no_grad():
        err = float((flow.invert(zs) - x).abs().max())
    print(f"256x256 L6 K32 round trip max error {err:.2e}")
    assert err < 1e-4
    opt = nf.FusedClipAdam(list(flow.parameters()) + list(prior.parameters()), lr=1e-5)
    ld, lp = nf.initialize_with_zeros(2, B, DEV)
    zs, ld, lp = flow.transform(x, ld, lp)
    lp += prior.compute_log_prob(zs[-1])
    loss = nf.calculate_loss(ld + lp, 256.0, S * S * 3.0)
    assert math.isfinite(float(loss))
    loss.backward()
    assert all(p.grad is None or bool(torch.isfinite(p.grad).all()) for p in flow.parameters())
    before = flow.final_flows[0].invconv2d.weight.detach().clone()
    opt.step()
    assert not torch.equal(before, flow.final_flows[0].invconv2d.weight.detach())
    with torch.no_grad():
        zs, _, _ = flow.transform(x, torch.zeros(B, device=DEV), None)
        xs = flow.sample([zs[-1].contiguous()], temperature=0.7)
    assert xs.shape == x.shape and bool(torch.isfinite(xs).all())
    fm = CatFormater(L, c, S)
    cat = fm.process_latents(zs)
    back = fm.postprocess(cat)
    assert len(back) == L and all(torch.equal(a, b) for a, b in zip(back, zs))
    path = str(tmp_path / "flow.pt")
    torch.save({"flow": flow.state_dict()}, path)
    bb = nf.NFBackbone(path, c, L, K, True, True).to(DEV)
    with torch.no_grad():
        xb = bb.sample(fm.postprocess(cat))
    assert relerr(xb, x) < 1e-3
