"""Seeded sampling and per-image temperatures on the GPU: the three _ex entry points against the numpy oracle of the draw
contract and against the old entry points bit for bit; batch invariance of Glow sampling at config-2 size; the temperature
grid; one captured chain for every temperature and seed vector; density and gradients against the fp64 oracle; and the
unchanged default path."""
import numpy as np
import pytest
import torch

import normalizing_flow as nf
from normalizing_flow import _native as N
from oracle import glow_oracle as O
import philox_oracle as PO
from test_gpu_benchmarked_path import bench_style_model
from test_gpu_invert_density import check, errors, oracle_density, own_density
from test_gpu_invert_density_grad import TOL_FP32, TOL_SIMT, _glow, _grad_errs, _lat_shapes, oracle_invert_density

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")


@pytest.fixture(autouse=True)
def _defaults(monkeypatch):
    for k in ("NFDPM_PRECISION", "NFDPM_TILED", "NFDPM_INVERT_GRAD"):
        monkeypatch.delenv(k, raising=False)
    monkeypatch.setenv("NFDPM_GRAPHS", "1")
    monkeypatch.setenv("NFDPM_FUSED_BOUNDARY", "1")
    torch.set_grad_enabled(False)
    yield
    torch.set_grad_enabled(True)


def rnd(*shape, seed=0, scale=1.0):
    return torch.from_numpy((scale * np.random.default_rng(seed).standard_normal(shape)).astype(np.float32))


def seeds_of(n, seed=0):
    return torch.from_numpy(np.random.default_rng(seed).integers(-2 ** 63, 2 ** 63 - 1, n, dtype=np.int64)).to(DEV)


def oracle_eps(seeds, stream, shape):
    """The contract's draws of a [B, *shape] tensor, fp64 on the CPU."""
    n = int(np.prod(shape))
    return torch.from_numpy(PO.normals(seeds.cpu().numpy(), stream, n)).view(len(seeds), *shape)


def worst_vs_oracle(eps, ref):
    """max |d| / max(1, |ref|); the uniforms are exact, so this is the rounding of fp32 logf / sincospif."""
    d = (eps.detach().cpu().double() - ref).abs() / ref.abs().clamp(min=1.0)
    return float(d.max())


# ------------------------------------------------------------------------------------------------ kernels
@pytest.mark.parametrize("B,Ch,H,W,pad", [(1, 3, 5, 3, 0), (3, 4, 4, 4, 7), (2, 12, 16, 16, 0)])
def test_split_prior_sample_ex(B, Ch, H, W, pad):
    """eps_out against the oracle (P % 4 != 0 with an odd C/2 at B = 1; a strided y); y of the seeded call is the old entry
    point fed with eps_out; temp_b = T everywhere is scalar T; per-image temp_b is the old entry point per image."""
    C, P, M = 2 * Ch, H * W, B * H * W
    ldh = (C + 15) // 16 * 16
    ybs = C * P + pad
    h = rnd(M, ldh, seed=1, scale=0.3).to(DEV)
    bias, logs = rnd(C, seed=2, scale=0.3).to(DEV), rnd(C, seed=3, scale=0.1).to(DEV)
    seeds = seeds_of(B, 4)
    temp_b = (torch.rand(B, generator=torch.Generator().manual_seed(5)) + 0.25).to(DEV)
    T = 0.7

    def y0():
        return rnd(B * ybs, seed=6).to(DEV)

    y_seed, eps = y0(), torch.full((B, Ch, H, W), 7.0, device=DEV)
    N.split_prior_sample_ex(h, ldh, bias, logs, None, seeds, 5, T, None, eps, y_seed, ybs, B, C, H, W)
    torch.cuda.synchronize()
    w = worst_vs_oracle(eps, oracle_eps(seeds, 5, (Ch, H, W)))
    print(f"split_prior_sample_ex B={B} C/2={Ch} P={P}: worst |d|/max(1,|ref|) = {w:.2e}")
    assert w <= 1e-6
    y_old = y0()
    N.split_prior_sample(h, ldh, bias, logs, eps, T, y_old, ybs, B, C, H, W)
    assert torch.equal(y_seed, y_old)
    y_vec = y0()
    N.split_prior_sample_ex(h, ldh, bias, logs, None, seeds, 5, 0.0, torch.full((B,), T, device=DEV), None, y_vec, ybs, B, C,
                            H, W)
    assert torch.equal(y_vec, y_old)
    y_pi = y0()
    N.split_prior_sample_ex(h, ldh, bias, logs, None, seeds, 5, 0.0, temp_b, None, y_pi, ybs, B, C, H, W)
    want = y0()
    for b in range(B):
        N.split_prior_sample(h[b * P:], ldh, bias, logs, eps[b:b + 1], float(temp_b[b]), want[b * ybs:], ybs, 1, C, H, W)
    assert torch.equal(y_pi, want)
    # NULL new arguments: the old entry point's bits
    y_null = y0()
    N.split_prior_sample_ex(h, ldh, bias, logs, eps, None, 0, T, None, None, y_null, ybs, B, C, H, W)
    assert torch.equal(y_null, y_old)
    # unconditional form (h NULL)
    y_u, y_uo = y0(), y0()
    eps_u = torch.empty(B, Ch, H, W, device=DEV)
    N.split_prior_sample_ex(None, 0, None, None, None, seeds, 0, T, None, eps_u, y_u, ybs, B, C, H, W)
    N.split_prior_sample(None, 0, None, None, eps_u, T, y_uo, ybs, B, C, H, W)
    assert torch.equal(y_u, y_uo) and worst_vs_oracle(eps_u, oracle_eps(seeds, 0, (Ch, H, W))) <= 1e-6


@pytest.mark.parametrize("B,C,P,learned", [(1, 3, 15, True), (4, 8, 16, True), (2, 5, 9, False)])
def test_gauss_sample_const_ex(B, C, P, learned):
    bias = rnd(2 * C, seed=1, scale=0.3).to(DEV) if learned else None
    logs = rnd(2 * C, seed=2, scale=0.1).to(DEV) if learned else None
    seeds = seeds_of(B, 3)
    temp_b = (torch.rand(B, generator=torch.Generator().manual_seed(4)) + 0.25).to(DEV)
    T = 0.6
    out, eps = torch.empty(B, C, P, device=DEV), torch.full((B, C, P), 7.0, device=DEV)
    N.gauss_sample_const_ex(None, seeds, PO.PRIOR_STREAM, bias, logs, T, None, eps, out, B, C, P)
    torch.cuda.synchronize()
    w = worst_vs_oracle(eps, oracle_eps(seeds, PO.PRIOR_STREAM, (C, P)))
    print(f"gauss_sample_const_ex B={B} C={C} P={P}: worst |d|/max(1,|ref|) = {w:.2e}")
    assert w <= 1e-6
    old = torch.empty_like(out)
    N.gauss_sample_const(eps, bias, logs, T, old, B, C, P)
    assert torch.equal(out, old)
    vec = torch.empty_like(out)
    N.gauss_sample_const_ex(None, seeds, PO.PRIOR_STREAM, bias, logs, 0.0, torch.full((B,), T, device=DEV), None, vec, B, C, P)
    assert torch.equal(vec, old)
    pi, want = torch.empty_like(out), torch.empty_like(out)
    N.gauss_sample_const_ex(None, seeds, PO.PRIOR_STREAM, bias, logs, 0.0, temp_b, None, pi, B, C, P)
    for b in range(B):
        N.gauss_sample_const(eps[b], bias, logs, float(temp_b[b]), want[b], 1, C, P)
    assert torch.equal(pi, want)
    null = torch.empty_like(out)
    N.gauss_sample_const_ex(eps, None, 0, bias, logs, T, None, None, null, B, C, P)
    assert torch.equal(null, old)


@pytest.mark.parametrize("conditional", [True, False])
@pytest.mark.parametrize("B,Ch,H,W", [(3, 6, 8, 8), (2, 300, 1, 1)])
def test_split_sample_bwd_ex(conditional, B, Ch, H, W):
    """Per-image temp_b against fp64 autograd (the fp32-sink rule of test_gpu_train_kernels: relative L2 1e-5); NULL temp_b
    is split_sample_bwd_lp's and split_sample_bwd's bits."""
    C, P, M = 2 * Ch, H * W, B * H * W
    ldh = (C + 15) // 16 * 16 + 16
    h = rnd(M, ldh, seed=1, scale=0.3)
    bias, logs = rnd(C, seed=2, scale=0.3), rnd(C, seed=3, scale=0.1)
    eps, dz, dlp = rnd(B, Ch, H, W, seed=4), rnd(B, Ch, H, W, seed=5), rnd(B, seed=6)
    temp = torch.rand(B, generator=torch.Generator().manual_seed(7)) + 0.25

    def run(fn, *args):
        dh = torch.full((M, ldh), 7.0, device=DEV)
        dpar = torch.zeros(B * 2 * C, device=DEV)
        fn(dz.to(DEV), Ch * P, *args, h.to(DEV) if conditional else None, ldh, bias.to(DEV), logs.to(DEV),
           dh if conditional else None, dpar, B, C, H, W)
        return dh, dpar

    dh, dpar = run(N.split_sample_bwd_ex, eps.to(DEV), 0.0, temp.to(DEV), dlp.to(DEV))
    torch.cuda.synchronize()
    with torch.enable_grad():
        hd, bd, ld = (t.double().requires_grad_(True) for t in (h, bias, logs))
        hh = hd[:, :C] if conditional else torch.zeros(M, C, dtype=torch.float64)
        net = ((hh + bd) * torch.exp(3 * ld)).view(B, H, W, C).permute(0, 3, 1, 2)
        mean, lg = net.chunk(2, 1)
        z = mean + torch.exp(lg) * temp.double().view(B, 1, 1, 1) * eps.double()
        ((z * dz.double()).sum() + (O.gaussian_logp(z, mean, lg) * dlp.double()).sum()).backward()
    rel = lambda a, b: float((a.double() - b).norm() / (b.norm() + 1e-30))         # noqa: E731
    dp = dpar.view(B, 2 * C).sum(0).cpu()
    assert rel(dp[:C], bd.grad) < 1e-5 and rel(dp[C:], ld.grad) < 1e-5
    if conditional:
        got = dh.cpu()
        assert rel(got[:, :C], hd.grad[:, :C]) < 1e-5 and float(got[:, C:].abs().max()) == 0.0
    T = 0.7
    new = run(N.split_sample_bwd_ex, eps.to(DEV), T, None, dlp.to(DEV))
    assert all(torch.equal(a, b) for a, b in zip(new, run(N.split_sample_bwd_lp, dlp.to(DEV), eps.to(DEV), T)))
    new = run(N.split_sample_bwd_ex, eps.to(DEV), T, None, None)
    assert all(torch.equal(a, b) for a, b in zip(new, run(N.split_sample_bwd, eps.to(DEV), T)))


# ------------------------------------------------------------------------------------------------ model
def _drawn(flow, z_last, temp, seeds):
    """(x, [assembled Split states, level 0 first], ld, lp) of one seeded sampling call through the captured chain, and
    the assembled states of the same draw from an uncaptured walk."""
    B = z_last.shape[0]
    ld, lp = torch.zeros(B, device=DEV), torch.zeros(B, device=DEV)
    x = flow.invert([z_last], temp, ld, lp, seeds=seeds)
    sink = []
    flow._invert_walk([z_last], temp, True, eps_sink=sink, seeds=seeds)
    return x, [s for s, _ in sink[::-1]], ld, lp


def test_batch_invariance_config2(monkeypatch):
    """L3 K16 3x32x32, bench weights, fp32: B = 128 in one call, as two shards of 64 and in permuted order give the same
    drawn latents, x, log_det_jac and logp bit for bit (every level in "image" mode at both sizes)."""
    monkeypatch.setenv("NFDPM_PRECISION", "fp32")
    c, L, K, B, S = 3, 3, 16, 128, 32
    flow, prior, _, _, _ = bench_style_model(c, L, K, B, S, 1e-3)
    for Bn in (B, B // 2):
        assert all(flow._level_mode(Bn, C, h, w) == "image" for _, _, C, h, w in flow._geometry(S, S))
    s = seeds_of(B, 11)
    T = torch.linspace(0.3, 1.0, B, device=DEV)
    shape = (B,) + O.output_shapes(L, c, S)[-1]
    z_last = prior.sample(shape, T, seeds=s)
    full = _drawn(flow, z_last, T, s)
    halves = [_drawn(flow, z_last[i:i + 64].contiguous(), T[i:i + 64].contiguous(), s[i:i + 64].contiguous())
              for i in (0, 64)]
    perm = torch.randperm(B, generator=torch.Generator().manual_seed(3)).to(DEV)
    zp = prior.sample(shape, T[perm].contiguous(), seeds=s[perm].contiguous())
    assert torch.equal(zp, z_last[perm])
    permuted = _drawn(flow, zp, T[perm].contiguous(), s[perm].contiguous())
    x, states, ld, lp = full
    for a, b in zip(states, [torch.cat(t) for t in zip(*[hv[1] for hv in halves])]):
        assert torch.equal(a, b)
    for a, b in zip(states, permuted[1]):
        assert torch.equal(a[perm], b)
    for i in (0, 2, 3):
        assert torch.equal(full[i], torch.cat([hv[i] for hv in halves])), i
        assert torch.equal(full[i][perm], permuted[i]), i


def test_temperature_grid(monkeypatch):
    """One seed over T = 0, 0.25, ..., 1: every row draws the same eps, and each row is a seeded scalar-T call at its T."""
    monkeypatch.setenv("NFDPM_PRECISION", "fp32")
    c, L, K, S = 3, 3, 2, 32
    flow, _, _ = _glow(c, L, K, 21)
    temps = [0.0, 0.25, 0.5, 0.75, 1.0]
    B = len(temps)
    s = seeds_of(1, 22).repeat(B)
    T = torch.tensor(temps, device=DEV)
    z_last = rnd(*_lat_shapes(c, L, S, 1)[-1], seed=23).to(DEV).repeat(B, 1, 1, 1)
    sink = []
    flow._invert_walk([z_last], T, True, eps_sink=sink, seeds=s)
    for _, eps in sink:
        assert all(torch.equal(eps[0], eps[i]) for i in range(B))
    x = flow.invert([z_last], T, seeds=s)
    for i, t in enumerate(temps):
        assert torch.equal(x[i], flow.invert([z_last], t, seeds=s)[i]), t


def test_split_and_prior_draws_are_the_glow_draws(monkeypatch):
    monkeypatch.setenv("NFDPM_PRECISION", "fp32")
    c, L, K, B, S = 3, 3, 2, 6, 32
    flow, sd, psd = _glow(c, L, K, 31)
    s = seeds_of(B, 32)
    T = torch.linspace(0.2, 1.0, B, device=DEV)
    prior = nf.GaussianPrior(2 ** (L + 1) * c).to(DEV)
    prior.load_state_dict(psd, strict=True)
    shape = (B,) + O.output_shapes(L, c, S)[-1]
    z = prior.sample(shape, T, seeds=s)
    key = "_GaussianPrior__conv."
    pb = psd[key + "bias"].double().reshape(-1) * torch.exp(3.0 * psd[key + "logs"].double().reshape(-1))
    pm, pl = pb.view(1, -1, 1, 1).chunk(2, dim=1)
    want = pm + torch.exp(pl) * T.cpu().double().view(B, 1, 1, 1) * oracle_eps(s, PO.PRIOR_STREAM, shape[1:])
    assert float((z.cpu().double() - want).abs().max()) <= 1e-5
    sink = []
    flow._invert_walk([z], T, True, eps_sink=sink, seeds=s)
    for li, (state, eps) in enumerate(sink[::-1]):
        Ch = state.shape[1] // 2
        assert worst_vs_oracle(eps, oracle_eps(s, li, eps.shape[1:])) <= 1e-6
        if li == 0:
            got = flow.blocks[0].split.invert(state[:, :Ch].contiguous(), None, T, seeds=s)
            assert torch.equal(got, state)
            y = state[:, :Ch].contiguous()
            blk = flow.blocks[0]
            inv = blk.split.invert(y, None, T, seeds=s)
            for f in reversed(blk.flows):
                inv = f.invert(inv)
            assert torch.equal(blk.invert(y, None, T, seeds=s), blk.squeeze.invert(inv))


def test_one_captured_chain_for_every_temperature_and_seed(monkeypatch):
    """Ten temperature and seed vectors replay one "inv" entry, each returning its own draw, equal to the eager call bit for
    bit; a tensor temperature without seeds shares no entry with the seeded chain."""
    monkeypatch.setenv("NFDPM_PRECISION", "fp32")
    c, L, K, B, S = 3, 3, 2, 8, 32
    flow, _, _ = _glow(c, L, K, 41)
    z_last = rnd(*_lat_shapes(c, L, S, B)[-1], seed=42).to(DEV)
    outs = []
    for i in range(10):
        s = seeds_of(B, 100 + i)
        T = (torch.rand(B, generator=torch.Generator().manual_seed(i)) + 0.1).to(DEV)
        ld = torch.zeros(B, dtype=torch.float64, device=DEV)
        x = flow.invert([z_last], T, ld, seeds=s)
        assert sum(k[0] == "inv" for k in flow._graphs) == 1
        monkeypatch.setenv("NFDPM_GRAPHS", "0")
        ld_e = torch.zeros(B, dtype=torch.float64, device=DEV)
        x_e = flow.invert([z_last], T, ld_e, seeds=s)
        monkeypatch.setenv("NFDPM_GRAPHS", "1")
        assert torch.equal(x, x_e) and torch.equal(ld, ld_e), i
        assert all(not torch.equal(x, o) for o in outs)
        outs.append(x)
    keys = [k for k in flow._graphs if k[0] == "inv"]
    assert keys[0][6:9] == (1, "ex", True)
    monkeypatch.setenv("NFDPM_GRAPHS", "0")
    torch.cuda.manual_seed(5)
    a = flow.invert([z_last], torch.full((B,), 0.5, device=DEV))
    torch.cuda.manual_seed(5)
    b = flow.invert([z_last], 0.5)
    assert torch.equal(a, b)                          # per-image T = T everywhere, torch's draws: the scalar call's bits
    monkeypatch.setenv("NFDPM_GRAPHS", "1")
    flow.invert([z_last], torch.full((B,), 0.5, device=DEV))
    assert sum(k[0] == "inv" for k in flow._graphs) == 2


def test_sampling_density_with_seeds(monkeypatch):
    """ld + lp + prior(z) of a seeded per-image-T draw at config-2 size is the model's density at the returned x."""
    c, L, K, B, S = 3, 3, 16, 128, 32
    flow, prior, sd, psd, _ = bench_style_model(c, L, K, B, S, 1e-3)
    s = seeds_of(B, 51)
    T = torch.linspace(0.0, 1.0, B, device=DEV)
    z = prior.sample((B,) + O.output_shapes(L, c, S)[-1], T, seeds=s)
    for _ in range(2):
        ld, lp = torch.zeros(B, dtype=torch.float64, device=DEV), torch.zeros(B, dtype=torch.float64, device=DEV)
        xs = flow.invert([z], T, ld, lp, seeds=s)
    pl = prior.compute_log_prob(z).double()
    n_pix = float(S * S * c)
    check(errors((ld, lp, pl), own_density(flow, prior, xs), n_pix))
    idx = [0, B - 1]
    check(errors((ld[idx], lp[idx], pl[idx]), oracle_density(sd, psd, xs.cpu()[idx], L, K), n_pix))


@pytest.mark.parametrize("mode,tol", [("fp32_simt", TOL_SIMT), ("fp32", TOL_FP32)])
@pytest.mark.parametrize("recorded_invert", [False, True])
def test_gradients_with_seeds_and_per_image_temperature(monkeypatch, mode, tol, recorded_invert):
    """invert_with_density, and the recorded invert (NFDPM_INVERT_GRAD=1), at L3 K2 3x32x32 B = 3 with seeds and per-image
    T: x, density and every gradient against fp64 autograd over the oracle fed the contract's draws."""
    monkeypatch.setenv("NFDPM_PRECISION", mode)
    torch.set_grad_enabled(True)
    c, L, K, B, S = 3, 3, 2, 3, 32
    flow, sd, _ = _glow(c, L, K, 61)
    shapes = _lat_shapes(c, L, S, B)
    s = seeds_of(B, 62)
    T = torch.tensor([0.3, 0.7, 1.0], device=DEV)
    lat = rnd(*shapes[-1], seed=63)
    wx, a, cc = rnd(B, c, S, S, seed=64), rnd(B, seed=65), rnd(B, seed=66)
    lg = [lat.to(DEV).requires_grad_(True)]
    if recorded_invert:
        monkeypatch.setenv("NFDPM_INVERT_GRAD", "1")
        x = flow.invert(lg, T, seeds=s)
        (x * wx.to(DEV)).sum().backward()
    else:
        x, ld, lp = flow.invert_with_density(lg, T, torch.zeros(B, device=DEV), torch.zeros(B, device=DEV), seeds=s)
        ((x * wx.to(DEV)).sum() + (ld * a.to(DEV)).sum() + (lp * cc.to(DEV)).sum()).backward()
    sdo = {k: (v.double().clone().requires_grad_(True) if v.dtype.is_floating_point else v) for k, v in sd.items()}
    lo = [lat.double().requires_grad_(True)]
    eps = {i: oracle_eps(s, i, shapes[i][1:]) for i in range(L - 1)}
    xo, ldo, lpo = oracle_invert_density(sdo, lo, L, K, T.cpu().double().view(B, 1, 1, 1), eps)
    loss = (xo * wx.double()).sum()
    if not recorded_invert:
        loss = loss + (ldo * a.double()).sum() + (lpo * cc.double()).sum()
    loss.backward()
    rel = lambda p, q: float((p.detach().cpu().double() - q.detach()).norm() / (q.detach().norm() + 1e-30))   # noqa: E731
    e = {"x": rel(x, xo)}
    if not recorded_invert:
        e["ld"], e["lp"] = rel(ld, ldo), rel(lp, lpo)
    e.update(_grad_errs(flow, lg, lo, sdo))
    print(f"seeded gradients {mode} recorded_invert={recorded_invert}: {e}")
    assert e["x"] <= 1e-4 and e.get("ld", 0) <= 1e-4 and e.get("lp", 0) <= 1e-4, e
    assert max(v for k, v in e.items() if k not in ("x", "ld", "lp", "worst")) <= tol, e


def test_keyword_checks(monkeypatch):
    c, L, K, B, S = 3, 2, 1, 4, 16
    flow, _, psd = _glow(c, L, K, 71)
    z = rnd(*_lat_shapes(c, L, S, B)[-1], seed=72).to(DEV)
    before = N.launch_count
    bad = [dict(seeds=torch.zeros(B, dtype=torch.int32, device=DEV)), dict(seeds=torch.zeros(B + 1, dtype=torch.int64,
                                                                                                 device=DEV)),
           dict(seeds=torch.zeros(2 * B, dtype=torch.int64, device=DEV)[::2]),
           dict(temperature=torch.ones(B, dtype=torch.float64, device=DEV)),
           dict(temperature=torch.ones(B, 1, device=DEV)), dict(temperature=torch.ones(B - 1, device=DEV))]
    for kw in bad:
        with pytest.raises(ValueError):
            flow.invert([z], **kw)
    with pytest.raises(RuntimeError, match="CUDA"):
        flow.invert([z], torch.ones(B), seeds=seeds_of(B))
    with torch.enable_grad(), pytest.raises(ValueError, match="gradient with respect to the temperature"):
        flow.invert([z], torch.ones(B, device=DEV, requires_grad=True))
    prior = nf.GaussianPrior(z.shape[1]).to(DEV)
    with pytest.raises(ValueError):
        prior.sample(tuple(z.shape), torch.ones(B + 1, device=DEV))
    y = rnd(B, 6, 8, 8, seed=73).to(DEV)
    with pytest.raises(ValueError):
        flow.blocks[0].split.invert(y, None, 1.0, seeds=torch.zeros(B, 1, dtype=torch.int64, device=DEV))
    assert N.launch_count == before
    # seeds on a call that draws nothing are accepted and unused
    lats = [rnd(*s, seed=74 + i).to(DEV) for i, s in enumerate(_lat_shapes(c, L, S, B))]
    assert torch.equal(flow.invert(lats, 1.0, seeds=seeds_of(B)), flow.invert(lats))


def test_default_path_unchanged(monkeypatch):
    """Without seeds and with a float temperature no _ex entry point runs, the graph keys keep their form (temperature in
    the sampling key, at most four sampling graphs) and a replay launches what it launched."""
    monkeypatch.setenv("NFDPM_PRECISION", "fp32")
    for name in ("split_prior_sample_ex", "gauss_sample_const_ex", "split_sample_bwd_ex"):
        monkeypatch.setattr(N, name, lambda *a, _n=name: pytest.fail(f"{_n} called on the default path"))
    c, L, K, B, S = 3, 3, 2, 4, 32
    flow, _, psd = _glow(c, L, K, 81)
    prior = nf.GaussianPrior(2 ** (L + 1) * c).to(DEV)
    prior.load_state_dict(psd, strict=True)
    z = prior.sample((B,) + O.output_shapes(L, c, S)[-1], 0.7)
    counts = []
    for t in (0.1, 0.2, 0.3, 0.4, 0.5, 0.5, 0.5):
        n0 = N.launch_count
        flow.sample([z], temperature=t)
        counts.append(N.launch_count - n0)
    keys = [k for k in flow._graphs if k[0] == "inv"]
    assert len(keys) == 4 and all(k[6] == 1 and isinstance(k[7], float) for k in keys)
    assert counts[-1] == counts[-2]
    monkeypatch.setenv("NFDPM_INVERT_GRAD", "1")
    with torch.enable_grad():
        zg = z.clone().requires_grad_(True)
        flow.invert([zg], 0.7).sum().backward()
    assert zg.grad is not None
