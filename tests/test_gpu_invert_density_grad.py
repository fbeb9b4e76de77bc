"""Back-propagation through the density of ``Glow.invert``: ``Glow.invert_with_density`` / ``NFBackbone.invert_with_density``.

The three new entry points (coupling_inv_bwd_ld, flow_boundary_inv_stash_ld, split_sample_bwd_lp) and the log-det fold of
mix_inv_param_grad against fp64 autograd; the whole model against an fp64 oracle that accumulates the density along the
inverse's own walk; the recorded forward against the no-grad inverse bit for bit; the call contract; and the reverse-KL
recipe end to end."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import normalizing_flow as nf
from normalizing_flow import _native as N
from oracle import glow_oracle as O

DEV = torch.device("cuda")
TOL_SIMT = 2e-4          # exact fp32 GEMMs (fp32_simt): per tensor, relative L2
TOL_FP32 = 3e-3          # split-pair tensor-core operands (fp32)
TOL_BF16 = 1e-1          # plain bf16 operands
TOL_CFG2 = 5e-2          # config-2 size, fp32, density-only loss: 2x the measured worst tensor (2.5e-2), DESIGN.md §5


@pytest.fixture
def grad(monkeypatch):
    """invert_with_density records without NFDPM_INVERT_GRAD."""
    monkeypatch.delenv("NFDPM_INVERT_GRAD", raising=False)
    torch.set_grad_enabled(True)


def rel(a, b):
    a, b = a.detach().cpu().double(), b.detach().cpu().double()
    return float((a - b).norm() / (b.norm() + 1e-30))


def rnd(*shape, seed=0, scale=1.0):
    return torch.from_numpy((scale * np.random.default_rng(seed).standard_normal(shape)).astype(np.float32))


# ------------------------------------------------------------------------------------------------ CPU
def test_new_entry_points_reject_null_pointers():
    rc = N.lib.nfdpm_coupling_inv_bwd_ld(None, 0, None, None, 0, None, 108, None, None, None, 0, None, 0, 128, None, None,
                                         None, None, None, 1, 12, 4, 4, None)
    assert rc != 0 and b"nfdpm_coupling_inv_bwd_ld: null pointer" in N.lib.nfdpm_last_error_string()
    rc = N.lib.nfdpm_flow_boundary_inv_stash_ld(None, 0, None, 108, None, None, None, None, None, None, 0, None, 0, None, 0,
                                                0, 1, 12, 4, 4, None)
    assert rc != 0 and b"nfdpm_flow_boundary_inv_stash_ld: null pointer" in N.lib.nfdpm_last_error_string()
    rc = N.lib.nfdpm_split_sample_bwd_lp(None, 0, None, None, 1.0, None, 0, None, None, None, None, 1, 2, 1, 1, None)
    assert rc != 0 and b"nfdpm_split_sample_bwd_lp: null pointer" in N.lib.nfdpm_last_error_string()


def test_invert_with_density_argument_checks():
    flow = nf.Glow(3, 2, 1)
    shapes = [(2,) + s for s in O.output_shapes(2, 3, 8)]
    lats = [torch.zeros(s) for s in shapes]
    with pytest.raises(ValueError, match="invert"):
        flow.invert_with_density(lats)
    with pytest.raises(RuntimeError, match="CUDA"):
        flow.invert_with_density(lats, 1.0, torch.zeros(2))


# ------------------------------------------------------------------------------------------------ kernels
def _coupling_inv_ref(y, pm, bias3, logs3, B, C, H, W):
    """fp64 (x, sum log(s+1e-6)) of the inverse coupling, with (log_s, t) gathered from the taps-as-N rows pm."""
    ldp = pm.shape[1]
    p4 = pm.view(B, H, W, ldp)[..., :9 * C].reshape(B, H, W, 9, C).permute(0, 3, 4, 1, 2)      # [B, tap, C, H, W]
    pp = F.pad(p4.reshape(B, 9 * C, H, W), (1, 1, 1, 1)).view(B, 9, C, H + 2, W + 2)
    net = sum(pp[:, tap, :, tap // 3:tap // 3 + H, tap % 3:tap % 3 + W] for tap in range(9))
    net = (net + bias3.view(1, C, 1, 1)) * torch.exp(3 * logs3.view(1, C, 1, 1))
    log_s, t = net.chunk(2, 1)
    s = torch.sigmoid(log_s + 2)
    ya, yb = y.view(B, C, H, W).chunk(2, 1)
    return torch.cat([ya, yb / (s + 1e-6) - t], 1), torch.log(s + 1e-6).reshape(B, -1).sum(1)


@pytest.mark.gpu
@pytest.mark.parametrize("B,C,H,W", [(3, 12, 16, 16), (4, 48, 4, 4), (2, 12, 32, 32)])
@pytest.mark.parametrize("fmt", ["f32", "bf16", "split"])
def test_coupling_inv_bwd_ld(B, C, H, W, fmt):
    """One-CTA-per-image and pixel-tiled (2x12x32x32) forms, all d(pm) formats, against fp64 autograd of
    (x*dx).sum() + (dld*sum log(s+1e-6)).sum(); with dld = NULL the old entry point's bits."""
    import split_pairs as SP
    P = H * W
    ldp, Kp3, M = (9 * C + 15) // 16 * 16, (9 * C + 63) // 64 * 64, B * H * W
    y, dx = rnd(B, C, P, seed=1), rnd(B, C, P, seed=2)
    pm = rnd(M, ldp, seed=3) * 0.1
    bias3, logs3 = rnd(C, seed=4, scale=0.1), rnd(C, seed=5, scale=0.1)
    dld = rnd(B, seed=6)
    T_c = N.coupling_bwd_tiles(C, H, W)
    assert (T_c > 1) == (H == 32)
    dt = {"f32": torch.float32, "bf16": torch.bfloat16, "split": N.SPLIT}[fmt]

    def run(fn, *extra):
        dy = torch.zeros(B, C, P, device=DEV)
        dpm = torch.full((M, Kp3), 7, dtype=dt, device=DEV)
        dpar = torch.zeros(B * T_c * 2 * C, device=DEV)
        db, dl = torch.zeros(C, device=DEV), torch.zeros(C, device=DEV)
        args = (dx.to(DEV), C * P) + extra + (y.to(DEV), C * P, pm.to(DEV), ldp, bias3.to(DEV), logs3.to(DEV), dy, C * P,
                                              dpm, Kp3, dpar, B, C, H, W)
        if T_c == 1:
            fn(*args, db, dl)
        else:
            fn(*args, dp_scratch=torch.empty(M * C, device=DEV))
            N.reduce_rows2(dpar, db, dl, B * T_c, C, C, 2 * C)
        return dy, dpm, dpar, db, dl

    dy, dpm, _, db, dl = run(N.coupling_inv_bwd_ld, dld.to(DEV))
    torch.cuda.synchronize()
    yd, pd, bd, lsd = (t.double().requires_grad_(True) for t in (y, pm, bias3, logs3))
    x, ldc = _coupling_inv_ref(yd, pd, bd, lsd, B, C, H, W)
    ((x * dx.double().view(B, C, H, W)).sum() + (ldc * dld.double()).sum()).backward()
    assert rel(dy, yd.grad) < 1e-5
    assert rel(db, bd.grad) < 1e-5 and rel(dl, lsd.grad) < 1e-5
    got = dpm.cpu()
    if dt == N.SPLIT:
        want32 = torch.zeros(M, Kp3)
        want32[:, :9 * C] = pd.grad[:, :9 * C].float()
        assert rel(SP.value(got, M, Kp3).float(), want32) < 1e-5
    else:
        assert float(got.float()[:, 9 * C:].abs().max()) == 0.0
        assert rel(got.float()[:, :9 * C], pd.grad[:, :9 * C]) < (1e-5 if dt == torch.float32 else 5e-3)
    new = run(N.coupling_inv_bwd_ld, None)
    old = run(N.coupling_inv_bwd)
    assert all(torch.equal(a, b) for a, b in zip(new, old))


@pytest.mark.gpu
@pytest.mark.parametrize("B,C,H,W", [(3, 12, 16, 16), (5, 48, 4, 4), (2, 24, 8, 8)])
def test_flow_boundary_inv_stash_ld(B, C, H, W):
    """ld_part equals flow_boundary(inverse=1)'s partial on the same inputs; every other sink equals
    flow_boundary_inv_stash's."""
    P = H * W
    ldp = (9 * C + 15) // 16 * 16
    K1p = (9 * (C // 2) + 63) // 64 * 64
    src = rnd(B, C, P, seed=1).to(DEV)
    pm = (rnd(B * P, ldp, seed=2) * 0.1).to(DEV)
    bias3, logs3 = rnd(C, seed=3, scale=0.1).to(DEV), rnd(C, seed=4, scale=0.1).to(DEV)
    mt, beta = (rnd(C, C, seed=5) * 0.3).to(DEV), rnd(C, seed=6).to(DEV)
    ld_ref = torch.full((B,), 7.0, device=DEV)
    y_ref = torch.empty(B, C, P, device=DEV)
    a1_ref = torch.zeros(B * P * K1p, device=DEV)
    N.flow_boundary(src, C * P, False, pm, ldp, bias3, logs3, ld_ref, mt, beta, y_ref, C * P, a1_ref, K1p, B, C, H, W, True)
    outs = []
    for with_ld in (True, False):
        ld = torch.full((B,), 7.0, device=DEV)
        y, xs = torch.empty(B, C, P, device=DEV), torch.empty(B, C, P, device=DEV)
        a1 = torch.zeros(B * P * K1p, device=DEV)
        N.flow_boundary_inv_stash_ld(src, C * P, pm, ldp, bias3, logs3, ld if with_ld else None, mt, beta, y, C * P, xs,
                                     C * P, a1, K1p, B, C, H, W)
        outs.append((ld, y, xs, a1))
    y_old, xs_old = torch.empty(B, C, P, device=DEV), torch.empty(B, C, P, device=DEV)
    a1_old = torch.zeros(B * P * K1p, device=DEV)
    N.flow_boundary_inv_stash(src, C * P, pm, ldp, bias3, logs3, mt, beta, y_old, C * P, xs_old, C * P, a1_old, K1p, B, C,
                              H, W)
    torch.cuda.synchronize()
    assert torch.equal(outs[0][0], ld_ref)
    assert bool((outs[1][0] == 7.0).all())                # NULL sink: nothing written
    for ld, y, xs, a1 in outs:
        assert torch.equal(y, y_old) and torch.equal(xs, xs_old) and torch.equal(a1, a1_old)
    assert torch.equal(y_old, y_ref) and torch.equal(a1_old, a1_ref)


@pytest.mark.gpu
@pytest.mark.parametrize("conditional", [True, False])
@pytest.mark.parametrize("B,Ch,H,W", [(3, 6, 8, 8), (2, 300, 1, 1)])
def test_split_sample_bwd_lp(conditional, B, Ch, H, W):
    """Against fp64 autograd of (z*dz).sum() + (dlp*log N(z; mean, exp(lg))).sum() with z = mean + exp(lg)*T*eps, in the
    conditional and the per-channel-constant form; with dlp = NULL the old entry point's bits."""
    T = 0.7
    C, P, M = 2 * Ch, H * W, B * H * W
    ldh = (C + 15) // 16 * 16 + 16
    h = rnd(M, ldh, seed=1, scale=0.3)
    bias, logs = rnd(C, seed=2, scale=0.3), rnd(C, seed=3, scale=0.1)
    eps, dz, dlp = rnd(B, Ch, H, W, seed=4), rnd(B, Ch, H, W, seed=5), rnd(B, seed=6)

    def run(fn, *extra):
        dh = torch.full((M, ldh), 7.0, device=DEV)
        dpar = torch.zeros(B * 2 * C, device=DEV)
        fn(dz.to(DEV), Ch * P, *extra, eps.to(DEV), T, h.to(DEV) if conditional else None, ldh, bias.to(DEV),
           logs.to(DEV), dh if conditional else None, dpar, B, C, H, W)
        return dh, dpar

    dh, dpar = run(N.split_sample_bwd_lp, dlp.to(DEV))
    torch.cuda.synchronize()
    hd, bd, ld = (t.double().requires_grad_(True) for t in (h, bias, logs))
    hh = hd[:, :C] if conditional else torch.zeros(M, C, dtype=torch.float64)
    net = ((hh + bd) * torch.exp(3 * ld)).view(B, H, W, C).permute(0, 3, 1, 2)
    mean, lg = net.chunk(2, 1)
    z = mean + torch.exp(lg) * T * eps.double()
    ((z * dz.double()).sum() + (O.gaussian_logp(z, mean, lg) * dlp.double()).sum()).backward()
    dp = dpar.view(B, 2 * C).sum(0).cpu()
    assert rel(dp[:C], bd.grad) < 1e-5 and rel(dp[C:], ld.grad) < 1e-5
    if conditional:
        got = dh.cpu()
        assert rel(got[:, :C], hd.grad[:, :C]) < 1e-5 and float(got[:, C:].abs().max()) == 0.0
    new, old = run(N.split_sample_bwd_lp, None), run(N.split_sample_bwd)
    assert all(torch.equal(a, b) for a, b in zip(new, old))


@pytest.mark.gpu
@pytest.mark.parametrize("C,H,W,with_w,with_s", [(12, 8, 8, True, True), (48, 4, 4, True, True), (12, 16, 16, False, True),
                                                 (24, 8, 8, True, False)])
def test_mix_inv_param_grad_dld(C, H, W, with_w, with_s):
    """mix_bwd + mix_inv_param_grad with dld_sum against fp64 autograd of x*dx + dld*P*(sum s + log|det W|)."""
    from normalizing_flow import _engine as E
    from normalizing_flow import _modgrad as MG
    B, P = 5, H * W
    w = torch.linalg.qr(rnd(C, C, seed=1).double())[0] + 0.1 * rnd(C, C, seed=2).double() if with_w else None
    s = rnd(C, seed=3, scale=0.3).double() if with_s else None
    b = rnd(C, seed=4, scale=0.3).double() if with_s else None
    u, dx, dld = rnd(B, C, H, W, seed=5), rnd(B, C, H, W, seed=6), rnd(B, seed=7)
    dev = lambda t: None if t is None else t.float().to(DEV).contiguous()
    wg = None if w is None else dev(w).view(C, C, 1, 1)
    sg, bg = (None, None) if s is None else (dev(s).view(C, 1, 1), dev(b).view(C, 1, 1))
    _, dW, dS, dB = MG._mix_inv_backward(E.MixCache(), u.to(DEV), dx.to(DEV), wg, sg, bg, True, None, 0,
                                         MG._dld_sum(dld.to(DEV)))
    torch.cuda.synchronize()
    leaves = [t.float().double().requires_grad_(True) if t is not None else None for t in (w, s, b)]
    x, const = u.double(), 0.0
    if leaves[0] is not None:
        x = torch.einsum("oi,bihw->bohw", torch.linalg.inv(leaves[0]), x)
        const = const + torch.linalg.slogdet(leaves[0])[1]
    if leaves[1] is not None:
        x = x * torch.exp(-leaves[1]).view(1, C, 1, 1) - leaves[2].view(1, C, 1, 1)
        const = const + leaves[1].sum()
    ((x * dx.double()).sum() + dld.double().sum() * P * const).backward()
    if w is not None:
        assert rel(dW.view(C, C), leaves[0].grad) < 1e-4
    if s is not None:
        assert rel(dS.view(C), leaves[1].grad) < 1e-5 and rel(dB.view(C), leaves[2].grad) < 1e-5


# ------------------------------------------------------------------------------------------------ fp64 oracle
def _double(sd):
    return {k: (v.double().clone().requires_grad_(True) if v.dtype.is_floating_point else v) for k, v in sd.items()}


def oracle_invert_density(sd, latents, L, K, temperature=1.0, eps=None):
    """O.glow_invert's walk, accumulating the density it inverts: per step sum log(s+1e-6) plus P*(sum scale +
    log|det W|), and per Split log N(z; mean, exp(logs)) of the supplied or drawn half.  Returns (x, ld, lp)."""
    levels = O._step_prefixes(L, K)
    B = latents[-1].shape[0]
    ld = torch.zeros(B, dtype=torch.float64)
    lp = torch.zeros(B, dtype=torch.float64)

    def step_inv(y, pre):
        nonlocal ld
        y_a, y_b = y.chunk(2, dim=1)
        log_s, t = O.coupling_net(y_a, sd, pre + "affcoupling.net.").chunk(2, dim=1)
        s = torch.sigmoid(log_s + 2.0)
        x = torch.cat([y_a, y_b / (s + 1e-6) - t], dim=1)
        W = sd[pre + "invconv2d.weight"]
        c = W.shape[0]
        x = O.invconv_inv(x, W)
        x = O.actnorm_inv(x, sd[pre + "actnorm.scale"], sd[pre + "actnorm.bias"])
        P = y.shape[2] * y.shape[3]
        ld = ld + torch.log(s + 1e-6).reshape(B, -1).sum(1) + \
            P * (sd[pre + "actnorm.scale"].sum() + torch.linalg.slogdet(W.reshape(c, c))[1])
        return x

    y = latents[-1]
    for pre in reversed(levels[L - 1]):
        y = step_inv(y, pre)
    y = O.unsqueeze2x2(y)
    for n, i in enumerate(reversed(range(L - 1))):
        idx = -(n + 2)
        z = latents[idx] if len(latents) >= -idx else None
        mean, logs = O.split_prior_params(y, sd, f"blocks.{i}.split.")
        mean, logs = mean.double(), logs.double()
        if z is None:
            z = mean + (torch.exp(logs) * temperature) * eps[i]
        lp = lp + O.gaussian_logp(z, mean, logs)
        y = torch.cat([y, z], dim=1)
        for pre in reversed(levels[i]):
            y = step_inv(y, pre)
        y = O.unsqueeze2x2(y)
    return y, ld, lp


def _glow(c, L, K, seed, learn_prior=True):
    sd, psd = O.seeded_state(c, L, K, seed, learn_prior=learn_prior)
    flow = nf.Glow(c, L, K, learn_prior_mean_logs=learn_prior).to(DEV)
    flow.load_state_dict(sd, strict=True)
    return flow, sd, psd


def _lat_shapes(c, L, S, B):
    return [(B,) + s for s in O.output_shapes(L, c, S)]


def _draw_eps(shapes, L, seed):
    torch.cuda.manual_seed(seed)
    return {i: torch.empty(shapes[i], device=DEV).normal_().cpu().double() for i in reversed(range(L - 1))}


def _grad_errs(flow, lg, lo, sdo):
    errs = {f"dz{i}": rel(a.grad, b.grad) for i, (a, b) in enumerate(zip(lg, lo)) if b.grad is not None}
    worst, worst_k = 0.0, None
    for k, p in flow.named_parameters():
        ref = sdo[k].grad
        if ref is None or float(ref.abs().max()) == 0.0:
            assert p.grad is None or float(p.grad.abs().max()) < 1e-6, k
            continue
        assert p.grad is not None, k
        r = rel(p.grad, ref)
        if r > worst:
            worst, worst_k = r, k
    errs["param"] = worst
    errs["worst"] = worst_k
    return errs


def _density_case(mode, sampled, density_only, c=3, L=3, K=2, B=3, S=32, T=0.7, seed=51, learn_prior=True):
    flow, sd, _ = _glow(c, L, K, seed, learn_prior)
    shapes = _lat_shapes(c, L, S, B)
    lats = [rnd(*s, seed=60 + i) for i, s in enumerate(shapes)]
    if sampled:
        lats = lats[-1:]
    temp = T if sampled else 1.0
    wx = torch.zeros(B, c, S, S) if density_only else rnd(B, c, S, S, seed=70)
    a, cc = rnd(B, seed=71), rnd(B, seed=72)
    lg = [t.to(DEV).requires_grad_(True) for t in lats]
    torch.cuda.manual_seed(9)
    x, ld, lp = flow.invert_with_density(lg, temp, torch.zeros(B, device=DEV), torch.zeros(B, device=DEV))
    ((x * wx.to(DEV)).sum() + (ld * a.to(DEV)).sum() + (lp * cc.to(DEV)).sum()).backward()
    eps = _draw_eps(shapes, L, 9) if sampled else None
    sdo = _double(sd)
    lo = [t.double().requires_grad_(True) for t in lats]
    xo, ldo, lpo = oracle_invert_density(sdo, lo, L, K, temp, eps)
    ((xo * wx.double()).sum() + (ldo * a.double()).sum() + (lpo * cc.double()).sum()).backward()
    errs = {"x": rel(x, xo), "ld": rel(ld, ldo), "lp": rel(lp, lpo)}
    errs.update(_grad_errs(flow, lg, lo, sdo))
    print(f"invert-density-grad {mode} sampled={sampled} density_only={density_only} c={c} "
          f"learn_prior={learn_prior}: {errs}")
    return errs


@pytest.mark.gpu
def test_oracle_matches_transform_of_invert():
    """The oracle's density equals the oracle transform's density at its returned x (the 1e-6 asymmetry aside)."""
    c, L, K, B, S = 3, 3, 2, 3, 32
    _, sd, _ = _glow(c, L, K, 51)
    lats = [rnd(*s, seed=60 + i).double() for i, s in enumerate(_lat_shapes(c, L, S, B))]
    sdo = {k: (v.double() if v.dtype.is_floating_point else v) for k, v in sd.items()}
    with torch.no_grad():
        x, ld, lp = oracle_invert_density(sdo, lats, L, K)
        ld2, lp2 = torch.zeros(B, dtype=torch.float64), torch.zeros(B, dtype=torch.float64)
        O.glow_transform(sdo, x, L, K, ld2, lp2)
    assert rel(ld, ld2) <= 1e-4 and rel(lp, lp2) <= 1e-4


@pytest.mark.gpu
@pytest.mark.parametrize("mode,tol", [("fp32_simt", TOL_SIMT), ("fp32", TOL_FP32), ("bf16", TOL_BF16)])
@pytest.mark.parametrize("sampled", [False, True])
@pytest.mark.parametrize("density_only", [False, True])
def test_invert_with_density_grad_matches_oracle(grad, monkeypatch, mode, tol, sampled, density_only):
    monkeypatch.setenv("NFDPM_PRECISION", mode)
    e = _density_case(mode, sampled, density_only)
    assert e["x"] <= (1e-4 if mode != "bf16" else 5e-2)
    assert e["ld"] <= (1e-4 if mode != "bf16" else 2e-4) and e["lp"] <= (1e-4 if mode != "bf16" else 2e-4), e
    assert max(v for k, v in e.items() if k not in ("x", "ld", "lp", "worst")) <= tol, e


@pytest.mark.gpu
@pytest.mark.parametrize("sampled", [False, True])
def test_one_channel_and_no_learned_prior(grad, monkeypatch, sampled):
    monkeypatch.setenv("NFDPM_PRECISION", "fp32_simt")
    for c, learn_prior in ((1, True), (3, False)):
        e = _density_case("fp32_simt", sampled, True, c=c, learn_prior=learn_prior)
        assert max(v for k, v in e.items() if k not in ("worst",)) <= TOL_SIMT, e


@pytest.mark.gpu
def test_split_conv_gets_logp_gradient_at_supplied_levels(grad, monkeypatch):
    """Decoding with a loss on logp only: every Split conv's gradient comes from the log-p term alone and matches the
    oracle (non-zero)."""
    monkeypatch.setenv("NFDPM_PRECISION", "fp32_simt")
    c, L, K, B, S = 3, 3, 2, 3, 32
    flow, sd, _ = _glow(c, L, K, 52)
    lats = [rnd(*s, seed=80 + i) for i, s in enumerate(_lat_shapes(c, L, S, B))]
    lg = [t.to(DEV).requires_grad_(True) for t in lats]
    _, _, lp = flow.invert_with_density(lg, 1.0, None, torch.zeros(B, device=DEV))
    lp.sum().backward()
    sdo = _double(sd)
    lo = [t.double().requires_grad_(True) for t in lats]
    _, _, lpo = oracle_invert_density(sdo, lo, L, K)
    lpo.sum().backward()
    for i in range(L - 1):
        p = flow.blocks[i].split.conv.weight
        ref = sdo[f"blocks.{i}.split.conv.weight"].grad
        assert float(ref.abs().max()) > 0 and rel(p.grad, ref) <= TOL_SIMT
    e = _grad_errs(flow, lg, lo, sdo)
    assert max(v for k, v in e.items() if k != "worst") <= TOL_SIMT, e


# ------------------------------------------------------------------------------------------------ forward identity
@pytest.mark.gpu
@pytest.mark.parametrize("case", ["image", "row_band", "unfused", "not_ready"])
def test_recorded_forward_equals_no_grad(grad, monkeypatch, case):
    """x, log_det_jac and logp of the recorded call equal the no-grad invert with accumulators bit for bit, and x equals
    the recorded call without accumulators: image levels with the fused GEMM3 (16x16 at B = 64), row bands (B = 3),
    every level unfused, and a model that is not ready."""
    monkeypatch.setenv("NFDPM_PRECISION", "fp32")
    c, L, K, S = 3, 3, 2, 32
    B = 64 if case == "image" else 3
    if case == "unfused":
        monkeypatch.setenv("NFDPM_FUSED_BOUNDARY", "0")
    if case == "not_ready":
        flow = nf.Glow(c, L, K).to(DEV)
    else:
        flow, _, _ = _glow(c, L, K, 81)
    if case == "image":
        assert flow._level_mode(B, 4 * c, S // 2, S // 2) == "image"
    if case == "row_band":
        assert flow._level_mode(B, 4 * c, S // 2, S // 2) == "tiled"
    lats = [rnd(*s, seed=90 + i).to(DEV) for i, s in enumerate(_lat_shapes(c, L, S, B))]
    for args in ((lats, 1.0), (lats[-1:], 0.0)):
        ld0, lp0 = torch.zeros(B, device=DEV), torch.zeros(B, device=DEV)
        with torch.no_grad():
            ref = flow.invert(*args, ld0, lp0)
        assert flow._ready() == (case != "not_ready")
        lg = [t.clone().requires_grad_(True) for t in args[0]]
        ld1, lp1 = torch.zeros(B, device=DEV), torch.zeros(B, device=DEV)
        got, ld, lp = flow.invert_with_density(lg, args[1], ld1, lp1)
        assert got.grad_fn is not None and ld is ld1 and lp is lp1 and ld.grad_fn is not None
        assert torch.equal(got.detach(), ref), (case, rel(got, ref))
        assert torch.equal(ld1.detach(), ld0) and torch.equal(lp1.detach(), lp0), case
        monkeypatch.setenv("NFDPM_INVERT_GRAD", "1")
        plain = flow.invert(lg, args[1])
        monkeypatch.delenv("NFDPM_INVERT_GRAD")
        assert torch.equal(plain.detach(), got.detach())


# ------------------------------------------------------------------------------------------------ config-2 size
@pytest.mark.gpu
def test_config2_density_grad_vs_oracle(grad, monkeypatch):
    """L3 K16, B = 128, 3x32x32, fp32, the benchmark's weights, decoding latents of real-looking images: a density-only
    loss on two images; their latent gradients and the parameter gradients against the fp64 oracle on those two."""
    monkeypatch.setenv("NFDPM_PRECISION", "fp32")
    c, L, K, B, S = 3, 3, 16, 128, 32
    flow, sd, _ = _glow(c, L, K, 0)
    x = (torch.rand(B, c, S, S, device=DEV, generator=torch.Generator(DEV).manual_seed(1)) - 0.5)
    with torch.no_grad():
        zs, _, _ = flow.transform(x, torch.zeros(B, device=DEV), None)
    a, cc = torch.zeros(B), torch.zeros(B)
    a[:2], cc[:2] = rnd(2, seed=3), rnd(2, seed=4)
    lg = [z.clone().requires_grad_(True) for z in zs]
    _, ld, lp = flow.invert_with_density(lg, 1.0, torch.zeros(B, device=DEV), torch.zeros(B, device=DEV))
    ((ld * a.to(DEV)).sum() + (lp * cc.to(DEV)).sum()).backward()
    assert all(float(t.grad[2:].abs().max()) == 0.0 for t in lg)
    sdo = _double(sd)
    lo = [z[:2].detach().cpu().double().requires_grad_(True) for z in zs]
    _, ldo, lpo = oracle_invert_density(sdo, lo, L, K)
    ((ldo * a[:2].double()).sum() + (lpo * cc[:2].double()).sum()).backward()
    e = {f"dz{i}": rel(t.grad[:2], o.grad) for i, (t, o) in enumerate(zip(lg, lo))}
    e["ld"], e["lp"] = rel(ld[:2], ldo), rel(lp[:2], lpo)
    pe = _grad_errs(flow, [], [], sdo)
    print(f"config-2 density grad: {e} {pe}")
    assert max(e.values()) <= TOL_CFG2 and pe["param"] <= TOL_CFG2, (e, pe)


# ------------------------------------------------------------------------------------------------ contract
@pytest.mark.gpu
def test_contract(grad, monkeypatch):
    monkeypatch.setenv("NFDPM_PRECISION", "fp32")
    c, L, K, B, S = 3, 2, 2, 4, 16
    flow, _, _ = _glow(c, L, K, 7)
    lats = [rnd(*s, seed=i).to(DEV).requires_grad_(True) for i, s in enumerate(_lat_shapes(c, L, S, B))]
    a = rnd(B, seed=9).to(DEV)
    # fp32 and fp64 accumulators, logp None: same gradients
    g32 = torch.autograd.grad((flow.invert_with_density(lats, 1.0, torch.zeros(B, device=DEV))[1] * a).sum(), lats)
    ld64 = torch.zeros(B, dtype=torch.float64, device=DEV)
    x, ld, lp = flow.invert_with_density(lats, 1.0, ld64)
    assert lp is None and ld is ld64 and ld.dtype == torch.float64
    g64 = torch.autograd.grad((ld * a.double()).sum(), lats)
    assert all(rel(p, q) < 1e-6 for p, q in zip(g32, g64))
    with torch.no_grad():
        want = torch.zeros(B, dtype=torch.float64, device=DEV)
        flow.invert([t.detach() for t in lats], 1.0, want)
    assert torch.equal(ld64.detach(), want)
    # an accumulator that requires grad on entry
    with pytest.raises(RuntimeError, match="must not require grad"):
        flow.invert_with_density(lats, 1.0, torch.zeros(B, device=DEV, requires_grad=True))
    # .grad accumulates over two backwards
    for t in lats:
        t.grad = None
    (flow.invert_with_density(lats, 1.0, torch.zeros(B, device=DEV))[1] * a).sum().backward()
    once = [t.grad.clone() for t in lats]
    (flow.invert_with_density(lats, 1.0, torch.zeros(B, device=DEV))[1] * a).sum().backward()
    assert all(rel(t.grad, 2 * o) < 1e-6 for t, o in zip(lats, once))
    # a second backward through one graph raises
    loss = (flow.invert_with_density(lats, 1.0, torch.zeros(B, device=DEV))[1] * a).sum()
    loss.backward(retain_graph=True)
    with pytest.raises(RuntimeError, match="released"):
        loss.backward()
    # a latent modified in place between forward and backward is detected
    ld = flow.invert_with_density(lats, 1.0, torch.zeros(B, device=DEV))[1]
    with torch.no_grad():
        lats[-1].add_(1.0)
    with pytest.raises(RuntimeError, match="modified by an inplace operation"):
        (ld * a).sum().backward()
    # NFDPM_INVERT_GRAD=1: Glow.invert with accumulators still refuses to record
    monkeypatch.setenv("NFDPM_INVERT_GRAD", "1")
    with pytest.raises(NotImplementedError, match="not differentiable"):
        flow.invert(lats, 1.0, torch.zeros(B, device=DEV))


@pytest.mark.gpu
def test_no_grad_call_is_invert(grad, monkeypatch):
    """Under torch.no_grad() the method returns exactly what invert accumulates, through the same captured graph entry."""
    monkeypatch.setenv("NFDPM_PRECISION", "fp32")
    c, L, K, B, S = 3, 3, 2, 8, 32
    flow, _, _ = _glow(c, L, K, 11)
    lats = [rnd(*s, seed=20 + i).to(DEV) for i, s in enumerate(_lat_shapes(c, L, S, B))]
    with torch.no_grad():
        ld0, lp0 = torch.zeros(B, device=DEV), torch.zeros(B, device=DEV)
        x0 = flow.invert(lats, 1.0, ld0, lp0)
        keys = set(flow._graphs)
        ld1, lp1 = torch.zeros(B, device=DEV), torch.zeros(B, device=DEV)
        x1, ld, lp = flow.invert_with_density(lats, 1.0, ld1, lp1)
    assert ld is ld1 and lp is lp1 and set(flow._graphs) == keys and len(keys) > 0
    assert torch.equal(x0, x1) and torch.equal(ld0, ld1) and torch.equal(lp0, lp1)


@pytest.mark.gpu
def test_frozen_backbone(grad, monkeypatch):
    """A frozen NFBackbone launches no gemm_tn and still gives the latents the gradient of log_det_jac."""
    monkeypatch.setenv("NFDPM_PRECISION", "fp32_simt")
    c, L, K, B, S = 1, 3, 2, 4, 32
    calls = []
    real = N.gemm_tn
    monkeypatch.setattr(N, "gemm_tn", lambda *a, **k: (calls.append(1), real(*a, **k))[1])
    sd, _ = O.seeded_state(c, L, K, 3)
    bb = nf.NFBackbone("", in_channel=c, L=L, K=K, learn_prior_mean_logs=True, freeze_flow=True)
    bb.model.load_state_dict(sd, strict=True)
    bb.to(DEV)
    lats = [rnd(*s, seed=i) for i, s in enumerate(_lat_shapes(c, L, S, B))]
    lg = [t.to(DEV).requires_grad_(True) for t in lats]
    x, ld = bb.invert_with_density(lg, torch.zeros(B, device=DEV))
    ld.sum().backward()
    assert not calls
    sdo = {k: (v.double() if v.dtype.is_floating_point else v) for k, v in sd.items()}
    lo = [t.double().requires_grad_(True) for t in lats]
    _, ldo, _ = oracle_invert_density(sdo, lo, L, K)
    ldo.sum().backward()
    assert rel(ld, ldo) <= 1e-4
    for a, b in zip(lg, lo):
        assert rel(a.grad, b.grad) <= TOL_SIMT


# ------------------------------------------------------------------------------------------------ reverse KL
@pytest.mark.gpu
def test_reverse_kl_recipe(monkeypatch):
    """z = prior.sample; x, ld, lp = flow.invert_with_density([z], T, ld, lp); loss = mean(ld + lp + log p(z)): flow and
    prior gradients against the oracle."""
    monkeypatch.setenv("NFDPM_INVERT_GRAD", "1")
    monkeypatch.setenv("NFDPM_PRECISION", "fp32_simt")
    torch.set_grad_enabled(True)
    c, L, K, B, S, T = 3, 3, 2, 3, 32, 0.7
    flow, sd, psd = _glow(c, L, K, 61)
    shapes = _lat_shapes(c, L, S, B)
    Cf = shapes[-1][1]
    prior = nf.GaussianPrior(Cf).to(DEV)
    prior.load_state_dict(psd, strict=True)
    torch.cuda.manual_seed(13)
    z = prior.sample(shapes[-1], T)
    x, ld, lp = flow.invert_with_density([z], T, torch.zeros(B, device=DEV), torch.zeros(B, device=DEV))
    loss = (ld + lp + prior.compute_log_prob(z)).mean()
    loss.backward()
    torch.cuda.manual_seed(13)
    e_prior = torch.empty(shapes[-1], device=DEV).normal_().cpu().double()
    eps = {i: torch.empty(shapes[i], device=DEV).normal_().cpu().double() for i in reversed(range(L - 1))}
    sdo, pso = _double(sd), _double(psd)
    # GaussianPrior: the ZeroConv of an all-zero map is its bias, (mean, logs) = bias*exp(3*logs) per channel
    key = "_GaussianPrior__conv."
    pb = pso[key + "bias"].reshape(-1) * torch.exp(3.0 * pso[key + "logs"].reshape(-1))
    pm, pl = pb.view(1, 2 * Cf, 1, 1).chunk(2, dim=1)
    zo = pm + torch.exp(pl) * T * e_prior
    xo, ldo, lpo = oracle_invert_density(sdo, [zo], L, K, T, eps)
    loss_o = (ldo + lpo + O.gaussian_logp(zo, pm.expand_as(zo), pl.expand_as(zo))).mean()
    loss_o.backward()
    assert rel(x, xo) <= 1e-4 and abs(float(loss) - float(loss_o)) <= 1e-4 * abs(float(loss_o))
    e = _grad_errs(flow, [], [], sdo)
    pe = _grad_errs(prior, [], [], pso)
    print(f"reverse-KL recipe: flow {e} prior {pe}")
    assert e["param"] <= TOL_SIMT and pe["param"] <= TOL_SIMT, (e, pe)
