"""Back-propagation through ``invert`` (NFDPM_INVERT_GRAD=1): the inverse-direction backward kernels against fp64 torch
restatements, the granular inverses and the whole Glow against torch autograd over the CPU oracle, the forward left
unchanged by recording, the inverse-function property at benchmark size, and the autograd contract (no side-effect
``.grad`` writes, frozen flows launch no weight-gradient GEMM, accumulation, released stash, knob off)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import normalizing_flow as nf
from normalizing_flow import _native as N
from oracle import glow_oracle as O
import split_pairs as SP

DEV = torch.device("cuda")
TOL_SIMT = 2e-4          # exact fp32 GEMMs (fp32_simt): per tensor, relative L2
TOL_FP32 = 3e-3          # split-pair tensor-core operands (fp32): measured worst tensor, see DESIGN.md §5
TOL_BF16 = 1e-1          # plain bf16 operands: measured worst tensor, see DESIGN.md §5
INV_PROP_TOL = 5e-2      # inverse-function property at config-2 size (fp32): measured, see DESIGN.md §5


@pytest.fixture
def knob(monkeypatch):
    monkeypatch.setenv("NFDPM_INVERT_GRAD", "1")
    torch.set_grad_enabled(True)


def rel(a, b):
    a, b = a.detach().cpu().double(), b.detach().cpu().double()
    return float((a - b).norm() / (b.norm() + 1e-30))


def rnd(*shape, seed=0, scale=1.0):
    return torch.from_numpy((scale * np.random.default_rng(seed).standard_normal(shape)).astype(np.float32))


# ------------------------------------------------------------------------------------------------ CPU: argument checks
def test_new_entry_points_reject_null_pointers():
    rc = N.lib.nfdpm_coupling_inv_bwd(None, 0, None, 0, None, 108, None, None, None, 0, None, 0, 128, None, None, None,
                                      None, None, 1, 12, 4, 4, None)
    assert rc != 0 and b"nfdpm_coupling_inv_bwd: null pointer" in N.lib.nfdpm_last_error_string()
    rc = N.lib.nfdpm_split_sample_bwd(None, 0, None, 1.0, None, 0, None, None, None, None, 1, 2, 1, 1, None)
    assert rc != 0 and b"nfdpm_split_sample_bwd: null pointer" in N.lib.nfdpm_last_error_string()
    rc = N.lib.nfdpm_flow_boundary_inv_stash(None, 0, None, 108, None, None, None, None, None, 0, None, 0, None, 0, 0, 1, 12,
                                             4, 4, None)
    assert rc != 0 and b"nfdpm_flow_boundary_inv_stash: null pointer" in N.lib.nfdpm_last_error_string()
    item = N.MixGradItem(part=None, B=1, C=4)
    rc = N.lib.nfdpm_mix_inv_param_grad((N.MixGradItem * 1)(item), 1, None)
    assert rc != 0 and b"nfdpm_mix_inv_param_grad: item 0 incomplete" in N.lib.nfdpm_last_error_string()


# ------------------------------------------------------------------------------------------------ kernels
def _coupling_inv_ref(y, pm, bias3, logs3, B, C, H, W):
    """fp64 x = (y_a, y_b/(s+1e-6) - t) with (log_s, t) gathered from the taps-as-N rows pm (the kernel's inputs)."""
    ldp = pm.shape[1]
    p4 = pm.view(B, H, W, ldp)[..., :9 * C].reshape(B, H, W, 9, C).permute(0, 3, 4, 1, 2)      # [B, tap, C, H, W]
    pp = F.pad(p4.reshape(B, 9 * C, H, W), (1, 1, 1, 1)).view(B, 9, C, H + 2, W + 2)
    net = sum(pp[:, tap, :, 1 + tap // 3 - 1 + 0:1 + tap // 3 - 1 + H, 1 + tap % 3 - 1:1 + tap % 3 - 1 + W]
              for tap in range(9))
    net = (net + bias3.view(1, C, 1, 1)) * torch.exp(3 * logs3.view(1, C, 1, 1))
    log_s, t = net.chunk(2, 1)
    s = torch.sigmoid(log_s + 2)
    ya, yb = y.view(B, C, H, W).chunk(2, 1)
    return torch.cat([ya, yb / (s + 1e-6) - t], 1)


@pytest.mark.gpu
@pytest.mark.parametrize("B,C,H,W", [(3, 12, 16, 16), (4, 48, 4, 4), (2, 12, 32, 32)])
@pytest.mark.parametrize("fmt", ["f32", "bf16", "split"])
def test_coupling_inv_bwd(B, C, H, W, fmt):
    """All three d(pm) formats, one-CTA-per-image and pixel-tiled (2x12x32x32) forms, against fp64 autograd."""
    P = H * W
    ldp, Kp3, M = (9 * C + 15) // 16 * 16, (9 * C + 63) // 64 * 64, B * H * W
    y, dx = rnd(B, C, P, seed=1), rnd(B, C, P, seed=2)
    pm = rnd(M, ldp, seed=3) * 0.1
    bias3, logs3 = rnd(C, seed=4, scale=0.1), rnd(C, seed=5, scale=0.1)
    T_c = N.coupling_bwd_tiles(C, H, W)
    assert (T_c > 1) == (H == 32)
    dt = {"f32": torch.float32, "bf16": torch.bfloat16, "split": N.SPLIT}[fmt]
    dy = torch.zeros(B, C, P, device=DEV)
    dpm = torch.full((M, Kp3), 7, dtype=dt, device=DEV)
    dpar = torch.zeros(B * T_c * 2 * C, device=DEV)
    db, dl = torch.zeros(C, device=DEV), torch.zeros(C, device=DEV)
    args = (dx.to(DEV), C * P, y.to(DEV), C * P, pm.to(DEV), ldp, bias3.to(DEV), logs3.to(DEV), dy, C * P, dpm, Kp3, dpar,
            B, C, H, W)
    if T_c == 1:
        N.coupling_inv_bwd(*args, db, dl)
    else:
        N.coupling_inv_bwd(*args, dp_scratch=torch.empty(M * C, device=DEV))
        N.reduce_rows2(dpar, db, dl, B * T_c, C, C, 2 * C)
    torch.cuda.synchronize()
    yd, pd, bd, ld = (t.double().requires_grad_(True) for t in (y, pm, bias3, logs3))
    (_coupling_inv_ref(yd, pd, bd, ld, B, C, H, W) * dx.double().view(B, C, H, W)).sum().backward()
    assert rel(dy, yd.grad) < 1e-5
    assert rel(db, bd.grad) < 1e-5 and rel(dl, ld.grad) < 1e-5
    got = dpm.cpu()
    if dt == N.SPLIT:
        want32 = torch.zeros(M, Kp3)
        want32[:, :9 * C] = pd.grad[:, :9 * C].float()
        assert rel(SP.value(got, M, Kp3).float(), want32) < 1e-5
    else:
        assert float(got.float()[:, 9 * C:].abs().max()) == 0.0
        assert rel(got.float()[:, :9 * C], pd.grad[:, :9 * C]) < (1e-5 if dt == torch.float32 else 5e-3)


@pytest.mark.gpu
@pytest.mark.parametrize("C,H,W,with_w,with_s", [(12, 8, 8, True, True), (48, 4, 4, True, True), (12, 16, 16, False, True),
                                                 (24, 8, 8, True, False)])
def test_mix_inv_param_grad(C, H, W, with_w, with_s):
    """mix_bwd (mt = inv_mt) + mix_inv_param_grad against fp64 autograd of x = diag(e^-s) W^-1 u - b."""
    from normalizing_flow import _engine as E
    from normalizing_flow import _modgrad as MG
    B = 5
    w = torch.linalg.qr(rnd(C, C, seed=1).double())[0] + 0.1 * rnd(C, C, seed=2).double() if with_w else None
    s = rnd(C, seed=3, scale=0.3).double() if with_s else None
    b = rnd(C, seed=4, scale=0.3).double() if with_s else None
    u, dx = rnd(B, C, H, W, seed=5), rnd(B, C, H, W, seed=6)
    dev = lambda t: None if t is None else t.float().to(DEV).contiguous()
    wg = None if w is None else dev(w).view(C, C, 1, 1)
    sg, bg = (None, None) if s is None else (dev(s).view(C, 1, 1), dev(b).view(C, 1, 1))
    du, dW, dS, dB = MG._mix_inv_backward(E.MixCache(), u.to(DEV), dx.to(DEV), wg, sg, bg)
    torch.cuda.synchronize()
    ud = u.double().requires_grad_(True)
    leaves = [t.clone().requires_grad_(True) if t is not None else None for t in (w, s, b)]
    x = ud
    if leaves[0] is not None:
        x = torch.einsum("oi,bihw->bohw", torch.linalg.inv(leaves[0].float().double()), x)
    if leaves[1] is not None:
        x = x * torch.exp(-leaves[1].float().double()).view(1, C, 1, 1) - leaves[2].float().double().view(1, C, 1, 1)
    (x * dx.double()).sum().backward()
    assert rel(du, ud.grad) < 1e-5
    if w is not None:
        assert rel(dW.view(C, C), leaves[0].grad) < 1e-4
    if s is not None:
        assert rel(dS.view(C), leaves[1].grad) < 1e-5 and rel(dB.view(C), leaves[2].grad) < 1e-5


@pytest.mark.gpu
@pytest.mark.parametrize("conditional", [True, False])
@pytest.mark.parametrize("B,Ch,H,W", [(3, 6, 8, 8), (2, 300, 1, 1)])
def test_split_sample_bwd(conditional, B, Ch, H, W):
    """d(mean) = dz, d(lg) = dz*exp(lg)*T*eps, through (h + bias)*exp(3 logs) (conditional) or per-channel constants;
    the one-pixel, many-channel case is IsotropicGaussian's (channels in two chunks)."""
    T = 0.7
    C, P, M = 2 * Ch, H * W, B * H * W
    ldh = (C + 15) // 16 * 16 + 16
    h = rnd(M, ldh, seed=1, scale=0.3)
    bias, logs = rnd(C, seed=2, scale=0.3), rnd(C, seed=3, scale=0.1)
    eps, dz = rnd(B, Ch, H, W, seed=4), rnd(B, Ch, H, W, seed=5)
    dh = torch.full((M, ldh), 7.0, device=DEV)
    dpar = torch.zeros(B * 2 * C, device=DEV)
    N.split_sample_bwd(dz.to(DEV), Ch * P, eps.to(DEV), T, h.to(DEV) if conditional else None, ldh, bias.to(DEV),
                       logs.to(DEV), dh if conditional else None, dpar, B, C, H, W)
    torch.cuda.synchronize()
    hd, bd, ld = (t.double().requires_grad_(True) for t in (h, bias, logs))
    hh = hd[:, :C] if conditional else torch.zeros(M, C, dtype=torch.float64)
    net = (hh + bd) * torch.exp(3 * ld)
    net = net.view(B, H, W, C).permute(0, 3, 1, 2)
    mean, lg = net.chunk(2, 1)
    z = mean + torch.exp(lg) * T * eps.double()
    (z * dz.double()).sum().backward()
    dp = dpar.view(B, 2 * C).sum(0).cpu()
    assert rel(dp[:C], bd.grad) < 1e-5 and rel(dp[C:], ld.grad) < 1e-5
    if conditional:
        got = dh.cpu()
        assert rel(got[:, :C], hd.grad[:, :C]) < 1e-5 and float(got[:, C:].abs().max()) == 0.0


# ------------------------------------------------------------------------------------------------ granular inverses
def _sub(sd, pre):
    return {k[len(pre):]: v for k, v in sd.items() if k.startswith(pre)}


def leafify(sd):
    return {k: (v.clone().requires_grad_(True) if v.dtype.is_floating_point else v) for k, v in sd.items()}


def check_params(mod, sd_g, tol, prefix=""):
    worst = 0.0
    for k, p in mod.named_parameters():
        ref = sd_g[prefix + k].grad
        if ref is None or float(ref.abs().max()) == 0.0:
            assert p.grad is None or float(p.grad.abs().max()) < 1e-6, k
            continue
        assert p.grad is not None, k
        r = rel(p.grad, ref)
        worst = max(worst, r)
        assert r <= tol, (k, r)
    return worst


@pytest.mark.gpu
@pytest.mark.parametrize("B,C,H,W", [(3, 12, 8, 8), (5, 48, 4, 4)])
def test_granular_inverses(knob, monkeypatch, B, C, H, W):
    monkeypatch.setenv("NFDPM_PRECISION", "fp32_simt")
    sd, _ = O.seeded_state(C // 4, 2, 1, 31)
    sd = _sub(sd, "blocks.0.flows.0.")
    y = rnd(B, C, H, W, seed=32)
    wx = rnd(B, C, H, W, seed=33)
    cases = [("actnorm.", nf.ActNorm(C), lambda t, s: O.actnorm_inv(t, s["scale"], s["bias"])),
             ("invconv2d.", nf.InvConv2d(C), lambda t, s: O.invconv_inv(t, s["weight"])),
             ("affcoupling.", nf.AffineCoupling(C), lambda t, s: O.coupling_inv(t, s, "net.")),
             ("", nf.StepFlow(C), lambda t, s: O.step_inv(t, s, ""))]
    for pre, mod, ref in cases:
        mod = mod.to(DEV)
        sub = _sub(sd, pre)
        mod.load_state_dict(sub)
        yg = y.to(DEV).requires_grad_(True)
        x = mod.invert(yg)
        (x * wx.to(DEV)).sum().backward()
        sg = leafify(sub)
        yo = y.clone().requires_grad_(True)
        xo = ref(yo, sg)
        (xo * wx).sum().backward()
        assert rel(x, xo) <= 1e-5, pre
        assert rel(yg.grad, yo.grad) <= TOL_SIMT, pre
        check_params(mod, sg, TOL_SIMT)
    sq = nf.Squeeze().to(DEV)
    yg = y.to(DEV).requires_grad_(True)
    (sq.invert(yg) * O.unsqueeze2x2(wx).to(DEV)).sum().backward()
    assert torch.equal(yg.grad.cpu(), wx)


@pytest.mark.gpu
@pytest.mark.parametrize("learn_prior", [True, False])
@pytest.mark.parametrize("sampled", [False, True])
def test_glowblock_invert(knob, monkeypatch, learn_prior, sampled):
    monkeypatch.setenv("NFDPM_PRECISION", "fp32_simt")
    c, B, S, T = 3, 3, 16, 0.7
    sd, _ = O.seeded_state(c, 2, 2, 41, learn_prior=learn_prior)
    sd = _sub(sd, "blocks.0.")
    blk = nf.GlowBlock(c, K=2, learn_prior_mean_logs=learn_prior).to(DEV)
    blk.load_state_dict(sd)
    C = 4 * c
    y = rnd(B, C // 2, S // 2, S // 2, seed=42)
    z = rnd(B, C // 2, S // 2, S // 2, seed=43)
    wx = rnd(B, c, S, S, seed=44)
    yg = y.to(DEV).requires_grad_(True)
    zg = None if sampled else z.to(DEV).requires_grad_(True)
    torch.cuda.manual_seed(5)
    x = blk.invert(yg, zg, temperature=T)
    torch.cuda.manual_seed(5)
    eps = torch.empty(B, C // 2, S // 2, S // 2, device=DEV).normal_().cpu()
    (x * wx.to(DEV)).sum().backward()
    sg = leafify(sd)
    yo = y.clone().requires_grad_(True)
    zo = None if sampled else z.clone().requires_grad_(True)
    if sampled:
        mean, logs = O.split_prior_params(yo, sg, "split.")
        zz = mean + torch.exp(logs) * T * eps
    else:
        zz = zo
    t = torch.cat([yo, zz], 1)
    for k in reversed(range(2)):
        t = O.step_inv(t, sg, f"flows.{k}.")
    xo = O.unsqueeze2x2(t)
    (xo * wx).sum().backward()
    assert rel(x, xo) <= 1e-5
    assert rel(yg.grad, yo.grad) <= TOL_SIMT
    if not sampled:
        assert rel(zg.grad, zo.grad) <= TOL_SIMT
    check_params(blk, sg, TOL_SIMT)


# ------------------------------------------------------------------------------------------------ whole Glow
def _glow(c, L, K, seed, learn_prior=True):
    sd, psd = O.seeded_state(c, L, K, seed, learn_prior=learn_prior)
    flow = nf.Glow(c, L, K, learn_prior_mean_logs=learn_prior).to(DEV)
    flow.load_state_dict(sd, strict=True)
    return flow, sd, psd


def _lat_shapes(c, L, S, B):
    return [(B,) + s for s in O.output_shapes(L, c, S)]


def _glow_case(mode, sampled, c=3, L=3, K=2, B=3, S=32, T=0.7, seed=51):
    flow, sd, _ = _glow(c, L, K, seed)
    shapes = _lat_shapes(c, L, S, B)
    lats = [rnd(*s, seed=60 + i) for i, s in enumerate(shapes)]
    if sampled:
        lats = lats[-1:]
    wx = rnd(B, c, S, S, seed=70)
    lg = [t.to(DEV).requires_grad_(True) for t in lats]
    torch.cuda.manual_seed(9)
    x = flow.invert(lg, temperature=T if sampled else 1.0)
    (x * wx.to(DEV)).sum().backward()
    eps = None
    if sampled:
        torch.cuda.manual_seed(9)
        eps = {i: torch.empty(shapes[i], device=DEV).normal_().cpu() for i in reversed(range(L - 1))}
    sg = leafify(sd)
    lo = [t.clone().requires_grad_(True) for t in lats]
    xo = O.glow_invert(sg, lo, L, K, temperature=T if sampled else 1.0, eps=eps)
    (xo * wx).sum().backward()
    errs = {"x": rel(x, xo)}
    for i, (a, b) in enumerate(zip(lg, lo)):
        errs[f"dz{i}"] = rel(a.grad, b.grad)
    worst, worst_k = 0.0, None
    for k, p in flow.named_parameters():
        ref = sg[k].grad
        if ref is None or float(ref.abs().max()) == 0.0:
            assert p.grad is None or float(p.grad.abs().max()) < 1e-6, k
            continue
        r = rel(p.grad, ref)
        if r > worst:
            worst, worst_k = r, k
    errs["param"] = worst
    print(f"invert-grad {mode} sampled={sampled}: {errs} (worst parameter {worst_k})")
    return errs


@pytest.mark.gpu
@pytest.mark.parametrize("mode,tol", [("fp32_simt", TOL_SIMT), ("fp32", TOL_FP32), ("bf16", TOL_BF16)])
@pytest.mark.parametrize("sampled", [False, True])
def test_glow_invert_grad_matches_oracle(knob, monkeypatch, mode, tol, sampled):
    monkeypatch.setenv("NFDPM_PRECISION", mode)
    errs = _glow_case(mode, sampled)
    assert errs["x"] <= (1e-4 if mode != "bf16" else 5e-2)
    assert max(v for k, v in errs.items() if k != "x") <= tol, errs


@pytest.mark.gpu
@pytest.mark.parametrize("B,S", [(64, 32), (8, 64)])
def test_forward_unchanged_by_recording(knob, monkeypatch, B, S):
    """With the knob, grad-mode invert returns what the no-grad invert returns: exactly at the one-CTA-per-image geometry
    (decoding and T = 0), within 1e-6 at a row-band geometry."""
    monkeypatch.setenv("NFDPM_PRECISION", "fp32")
    c, L, K = 3, 3, 2
    flow, _, _ = _glow(c, L, K, 81)
    lats = [rnd(*s, seed=90 + i).to(DEV) for i, s in enumerate(_lat_shapes(c, L, S, B))]
    for args in ((lats, 1.0), (lats[-1:], 0.0)):
        with torch.no_grad():
            ref = flow.invert(*args)
        got = flow.invert([t.clone().requires_grad_(True) for t in args[0]], args[1])
        assert got.grad_fn is not None
        if S == 32:
            assert torch.equal(got.detach(), ref)
        else:
            assert rel(got, ref) <= 1e-6


@pytest.mark.gpu
def test_inverse_function_property_config2(knob, monkeypatch):
    """v back through invert at z = transform(x), then back through transform at x, returns v (J_f^T J_{f^-1}^T = I):
    L3 K16, B = 128, 3x32x32, fp32, the benchmark's weights."""
    monkeypatch.setenv("NFDPM_PRECISION", "fp32")
    c, L, K, B, S = 3, 3, 16, 128, 32
    flow, _, _ = _glow(c, L, K, 0)
    x = (torch.rand(B, c, S, S, device=DEV, generator=torch.Generator(DEV).manual_seed(1)) - 0.5)
    with torch.no_grad():
        ld = torch.zeros(B, device=DEV)
        zs, _, _ = flow.transform(x, ld, None)
    zg = [z.clone().requires_grad_(True) for z in zs]
    v = torch.randn(B, c, S, S, device=DEV, generator=torch.Generator(DEV).manual_seed(2))
    xi = flow.invert(zg)
    gz = torch.autograd.grad(xi, zg, v)
    for p in flow.parameters():
        p.requires_grad_(False)
    xg = x.clone().requires_grad_(True)
    ld = torch.zeros(B, device=DEV)
    zs2, _, _ = flow.transform(xg, ld, None)
    (back,) = torch.autograd.grad(zs2, xg, list(gz))
    err = rel(back, v)
    print(f"inverse-function property: relL2 {err:.3e}")
    assert err <= INV_PROP_TOL


# ------------------------------------------------------------------------------------------------ contract
@pytest.mark.gpu
def test_autograd_contract(knob, monkeypatch):
    monkeypatch.setenv("NFDPM_PRECISION", "fp32")
    c, L, K, B, S = 3, 2, 2, 4, 16
    flow, _, _ = _glow(c, L, K, 7)
    lats = [rnd(*s, seed=i).to(DEV).requires_grad_(True) for i, s in enumerate(_lat_shapes(c, L, S, B))]
    w = rnd(B, c, S, S, seed=9).to(DEV)
    # torch.autograd.grad wrt the latents leaves every .grad as it was
    x = flow.invert(lats)
    g1 = torch.autograd.grad((x * w).sum(), lats)
    assert all(p.grad is None for p in flow.parameters()) and all(t.grad is None for t in lats)
    # two forwards, one backward each: gradients accumulate to 2x
    xa, xb = flow.invert(lats), flow.invert(lats)
    (xa * w).sum().backward()
    once = [p.grad.clone() for p in flow.parameters() if p.grad is not None]
    (xb * w).sum().backward()
    twice = [p.grad for p in flow.parameters() if p.grad is not None]
    assert once and all(rel(b, 2 * a) < 1e-6 for a, b in zip(once, twice))
    assert rel(lats[-1].grad, 2 * g1[-1]) < 1e-6
    # a second backward through one graph raises
    xc = flow.invert(lats)
    loss = (xc * w).sum()
    loss.backward(retain_graph=True)
    with pytest.raises(RuntimeError, match="released"):
        loss.backward()
    # a latent modified in place between forward and backward is detected
    xd = flow.invert(lats)
    with torch.no_grad():
        lats[-1].add_(1.0)
    with pytest.raises(RuntimeError, match="modified by an inplace operation"):
        (xd * w).sum().backward()
    # knob unset: NotImplementedError as before
    monkeypatch.setenv("NFDPM_INVERT_GRAD", "0")
    with pytest.raises(NotImplementedError):
        (flow.invert(lats) * w).sum().backward()


@pytest.mark.gpu
def test_frozen_flow_launches_no_weight_gradient_gemm(knob, monkeypatch):
    monkeypatch.setenv("NFDPM_PRECISION", "fp32")
    c, L, K, B, S = 1, 3, 2, 4, 32
    calls = []
    real = N.gemm_tn
    monkeypatch.setattr(N, "gemm_tn", lambda *a, **k: (calls.append(1), real(*a, **k))[1])
    sd, _ = O.seeded_state(c, L, K, 3)
    bb = nf.NFBackbone("", in_channel=c, L=L, K=K, learn_prior_mean_logs=True, freeze_flow=True)
    bb.model.load_state_dict(sd, strict=True)
    bb.to(DEV)
    assert not any(p.requires_grad for p in bb.model.parameters())
    lats = [rnd(*s, seed=i).to(DEV).requires_grad_(True) for i, s in enumerate(_lat_shapes(c, L, S, B))]
    x = bb.invert(lats)
    (x * x).sum().backward()
    assert lats[0].grad is not None and float(lats[0].grad.abs().max()) > 0
    assert not calls


@pytest.mark.gpu
def test_prior_sample_grads(knob):
    C, B, H, W, T = 24, 3, 4, 4, 0.7
    _, psd = O.seeded_state(3, 2, 1, 5)                  # GaussianPrior over 2**(L+1)*c = 24 channels
    prior = nf.GaussianPrior(C).to(DEV)
    prior.load_state_dict(psd, strict=True)
    wz = rnd(B, C, H, W, seed=1)
    torch.cuda.manual_seed(3)
    z = prior.sample((B, C, H, W), temperature=T)
    torch.cuda.manual_seed(3)
    eps = torch.empty(B, C, H, W, device=DEV).normal_().cpu()
    (z * wz.to(DEV)).sum().backward()
    pg = leafify(psd)
    zo = O.gaussian_prior_sample(pg, (B, C, H, W), T, eps)
    (zo * wz).sum().backward()
    assert rel(z, zo) <= 1e-5
    for k, p in prior.named_parameters():
        ref = pg[k].grad
        if ref is None or float(ref.abs().max()) == 0.0:
            assert p.grad is None or float(p.grad.abs().max()) < 1e-6, k
        else:
            assert rel(p.grad, ref) <= 1e-5, k
    # IsotropicGaussian: gradients wrt mean / logsd
    mean = rnd(B, 6, 1, 1, seed=4).to(DEV).requires_grad_(True)
    logsd = rnd(B, 6, 1, 1, seed=5, scale=0.2).to(DEV).requires_grad_(True)
    torch.cuda.manual_seed(4)
    zi = nf.IsotropicGaussian(mean, logsd).sample(temperature=T)
    torch.cuda.manual_seed(4)
    e = torch.empty(B, 6, 1, 1, device=DEV).normal_()
    (zi * 2).sum().backward()
    assert rel(mean.grad, torch.full_like(mean, 2.0)) < 1e-6
    assert rel(logsd.grad, 2 * torch.exp(logsd.detach()) * T * e) < 1e-6
