"""The density of what Glow.invert / Glow.sample return (GPU).

``invert(latents, T, log_det_jac, logp)`` adds exactly what ``transform(x, log_det_jac, logp)`` would add at the returned x.
Kernel level: every inverse-mode step boundary writes the forward's log-det partial bit for bit (same pm, same pass-through
half) and its other outputs do not change with the sink.  Model level, against the CPU oracle's transform of the oracle's
inverse (north-star bar: log-det / log-p relative <= 1e-4, bits/dim |d| <= 1e-3) and against this package's own transform:
decoding at config 2 with the weight sets of test_gpu_benchmarked_path.py, sampling at three temperatures, every inverse
path (one CTA per image, row bands, unfused, eager, replayed graphs, a model that is not ready), the
bf16 mode at its stated tolerance, and the call contract."""
import numpy as np
import pytest
import torch

import normalizing_flow as nf
from normalizing_flow import _native as N
from oracle import glow_oracle as O
import split_pairs as SP
from test_gpu_benchmarked_path import bench_style_model, seeded_model

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")


@pytest.fixture(autouse=True)
def _no_grad_default_mode(monkeypatch):
    for k in ("NFDPM_PRECISION", "NFDPM_TILED", "NFDPM_INVERT_GRAD"):
        monkeypatch.delenv(k, raising=False)
    monkeypatch.setenv("NFDPM_GRAPHS", "1")
    monkeypatch.setenv("NFDPM_FUSED_BOUNDARY", "1")
    torch.set_grad_enabled(False)
    yield
    torch.set_grad_enabled(True)


def rnd(*shape, seed=0, scale=1.0):
    return torch.from_numpy((scale * np.random.default_rng(seed).standard_normal(shape)).astype(np.float32))


def zeros2(B, dtype=torch.float64):
    return torch.zeros(B, dtype=dtype, device=DEV), torch.zeros(B, dtype=dtype, device=DEV)


# ------------------------------------------------------------------------------------------------ kernels
def _pm(B, C, H, W, seed=2):
    ldp = (9 * C + 15) // 16 * 16
    return (rnd(B * H * W, ldp, seed=seed) * 0.1).cuda(), ldp


@pytest.mark.parametrize("B,C,H,W", [(3, 4, 28, 28), (5, 12, 16, 16), (19, 48, 4, 4), (2, 6, 5, 7), (2, 12, 64, 64)])
def test_coupling_apply_inverse_ld_part(B, C, H, W):
    P = H * W
    x = rnd(B, C, H, W, seed=1).cuda()
    pm, ldp = _pm(B, C, H, W)
    bias3, logs3 = rnd(C, seed=3, scale=0.1).cuda(), rnd(C, seed=4, scale=0.1).cuda()
    T = N.ld_tiles(P)
    fwd, inv = torch.full((T * B,), np.nan, device=DEV), torch.full((T * B,), np.nan, device=DEV)
    y = torch.empty_like(x)
    N.coupling_apply(pm, ldp, bias3, logs3, x, y, fwd, B, C, H, W, C * P, C * P, False)
    x_plain, x_sink = torch.empty_like(x), torch.empty_like(x)
    N.coupling_apply(pm, ldp, bias3, logs3, y, x_plain, None, B, C, H, W, C * P, C * P, True)
    N.coupling_apply(pm, ldp, bias3, logs3, y, x_sink, inv, B, C, H, W, C * P, C * P, True)
    torch.cuda.synchronize()
    assert torch.equal(inv, fwd)
    assert torch.equal(x_sink, x_plain)


@pytest.mark.parametrize("B,C,H,W", [(3, 4, 16, 16), (5, 12, 16, 16), (4, 24, 8, 8), (7, 48, 4, 4), (2, 6, 5, 7)])
@pytest.mark.parametrize("a1_dt", [torch.float32, torch.bfloat16, N.SPLIT])
def test_flow_boundary_inverse_ld_part(B, C, H, W, a1_dt):
    P, Ch = H * W, C // 2
    lda = (9 * Ch + 63) // 64 * 64
    x = rnd(B, C, H, W, seed=1).cuda()
    pm, ldp = _pm(B, C, H, W)
    bias3, logs3 = rnd(C, seed=3, scale=0.1).cuda(), rnd(C, seed=4, scale=0.1).cuda()
    mt, beta = rnd(C, C, seed=5, scale=0.4).cuda(), rnd(C, seed=6).cuda()
    fwd = torch.full((B,), np.nan, device=DEV)
    N.flow_boundary(x, C * P, False, pm, ldp, bias3, logs3, fwd, mt, beta, torch.empty_like(x), C * P, None, 0, B, C, H, W,
                    False)
    outs = []
    for part in (None, torch.full((B,), np.nan, device=DEV)):
        y, a1 = torch.empty_like(x), torch.zeros(B * P, lda, dtype=a1_dt, device=DEV)
        N.flow_boundary(x, C * P, False, pm, ldp, bias3, logs3, part, mt, beta, y, C * P, a1, lda, B, C, H, W, True)
        outs.append((y, a1, part))
    torch.cuda.synchronize()
    assert torch.equal(outs[1][2], fwd)
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])


@pytest.mark.parametrize("B,C,H,W", [(2, 12, 32, 32), (3, 24, 16, 16), (2, 12, 64, 64), (8, 48, 8, 8)])
@pytest.mark.parametrize("a1_dt", [torch.float32, torch.bfloat16, N.SPLIT])
def test_flow_boundary_tiled_inverse_ld_part(B, C, H, W, a1_dt):
    P, Ch = H * W, C // 2
    lda = (9 * Ch + 63) // 64 * 64
    x = rnd(B, C, H, W, seed=1).cuda()
    pm, ldp = _pm(B, C, H, W)
    bias3, logs3 = rnd(C, seed=3, scale=0.1).cuda(), rnd(C, seed=4, scale=0.1).cuda()
    mt, beta = rnd(C, C, seed=5, scale=0.4).cuda(), rnd(C, seed=6).cuda()
    for with_a1 in (True, False):
        T = N.flow_boundary_tiles(B, C, H, W, 1, 1, int(with_a1))
        assert T > 0
        fwd = torch.full((T * B,), np.nan, device=DEV)
        N.flow_boundary_tiled(x, C * P, False, pm, ldp, bias3, logs3, fwd, mt, beta, torch.empty_like(x), C * P, None, 0,
                              torch.zeros(B * P, lda, dtype=a1_dt, device=DEV) if with_a1 else None,
                              lda if with_a1 else 0, B, C, H, W, False, T)
        outs = []
        for part in (None, torch.full((T * B,), np.nan, device=DEV)):
            y = torch.empty_like(x)
            a1 = torch.zeros(B * P, lda, dtype=a1_dt, device=DEV) if with_a1 else None
            N.flow_boundary_tiled(x, C * P, False, pm, ldp, bias3, logs3, part, mt, beta, y, C * P, None, 0, a1,
                                  lda if with_a1 else 0, B, C, H, W, True, T)
            outs.append((y, a1, part))
        torch.cuda.synchronize()
        assert torch.equal(outs[1][2], fwd)
        assert torch.equal(outs[0][0], outs[1][0])
        if with_a1:
            assert torch.equal(outs[0][1], outs[1][1])


@pytest.mark.parametrize("B,C,H,W", [(5, 12, 16, 16), (5, 24, 8, 8), (11, 48, 4, 4), (8, 16, 4, 4)])
@pytest.mark.parametrize("a1_dt,op_dt", [(torch.float32, torch.bfloat16), (torch.bfloat16, torch.bfloat16),
                                         (N.SPLIT, N.SPLIT), (torch.float32, N.SPLIT)])
def test_gemm3_boundary_inverse_ld_part(B, C, H, W, a1_dt, op_dt):
    P, Ch, F = H * W, C // 2, 512
    ldp = (9 * C + 15) // 16 * 16
    lda = (9 * Ch + 63) // 64 * 64
    M = B * P
    assert N.gemm3_boundary_ok(B, C, H, W, F * (2 if op_dt == N.SPLIT else 1), ldp)
    x = rnd(B, C, H, W, seed=1).cuda()
    h2 = rnd(M, F, seed=2).clamp_min(0) * 0.5
    w3 = rnd(ldp, F, seed=3, scale=0.02)
    w3[9 * C:] = 0
    if op_dt == N.SPLIT:
        h2, w3 = SP.encode(h2).cuda(), SP.encode(w3).cuda()
    else:
        h2, w3 = h2.cuda().to(torch.bfloat16), w3.cuda().to(torch.bfloat16)
    bias3, logs3 = rnd(C, seed=4, scale=0.1).cuda(), rnd(C, seed=5, scale=0.1).cuda()
    mt, beta = rnd(C, C, seed=6, scale=0.4).cuda(), rnd(C, seed=7).cuda()
    for with_mix in (True, False):
        m_, b_ = (mt, beta) if with_mix else (None, None)
        fwd = torch.full((B,), np.nan, device=DEV)
        N.gemm3_boundary(h2, F, w3, None, 0, x, C * P, bias3, logs3, fwd, m_, b_, torch.empty_like(x), C * P, None, 0, None,
                         0, B, C, H, W, F, ldp, False)
        outs = []
        for part in (None, torch.full((B,), np.nan, device=DEV)):
            y = torch.empty_like(x)
            a1 = torch.zeros(M, lda, dtype=a1_dt, device=DEV) if with_mix else None
            N.gemm3_boundary(h2, F, w3, None, 0, x, C * P, bias3, logs3, part, m_, b_, y, C * P, None, 0, a1,
                             lda if with_mix else 0, B, C, H, W, F, ldp, True)
            outs.append((y, a1, part))
        torch.cuda.synchronize()
        assert torch.equal(outs[1][2], fwd)
        assert torch.equal(outs[0][0], outs[1][0])
        if with_mix:
            assert torch.equal(outs[0][1], outs[1][1])


# ------------------------------------------------------------------------------------------------ model level
def oracle_density(sd, psd, xs, L, K):
    """The oracle's transform of images xs: (log-det, Split log-p, final prior log-p), fp64."""
    n = xs.shape[0]
    ld, lp = torch.zeros(n, dtype=torch.float64), torch.zeros(n, dtype=torch.float64)
    zo, ld, lp = O.glow_transform(sd, xs, L, K, ld, lp)
    return ld, lp, O.gaussian_prior_logp(psd, zo[-1]).double()


def own_density(flow, prior, x):
    ld, lp = zeros2(x.shape[0])
    zs, ld, lp = flow.transform(x, ld, lp)
    return ld, lp, prior.compute_log_prob(zs[-1]).double()


def errors(got, want, n_pix):
    """got / want: (ld, lp, prior) on the same images -> log-det and log-p relative, bits/dim absolute."""
    (ld, lp, pl), (ld_w, lp_w, pl_w) = [[t.detach().cpu().double() for t in g] for g in (got, want)]
    bpd = lambda a: O.bpd_loss(a, 32.0, n_pix)                                           # noqa: E731
    return {"ld_rel": float(((ld - ld_w).abs() / ld_w.abs()).max()),
            "lp_rel": float(((lp + pl - lp_w - pl_w).abs() / (lp_w + pl_w).abs()).max()),
            "bpd_abs": float(abs(bpd(ld + lp + pl) - bpd(ld_w + lp_w + pl_w)))}


def check(e, ld_tol=1e-4, lp_tol=1e-4, bpd_tol=1e-3):
    assert e["ld_rel"] <= ld_tol and e["lp_rel"] <= lp_tol and e["bpd_abs"] <= bpd_tol, e


def decode_vs_oracle(flow, prior, sd, psd, x, L, K, idx, calls=2):
    """Invert the oracle's latents of x (scattered into the batch) with both accumulators; -> (errors against the oracle's
    transform of its own inverse on idx, errors against this package's transform of the returned x, x, ld, lp)."""
    B, c, S, _ = x.shape
    zs, _, _ = flow.transform(x.to(DEV), torch.zeros(B, device=DEV), None)
    ld_o = torch.zeros(len(idx), dtype=torch.float64)
    zo, _, _ = O.glow_transform(sd, x[idx], L, K, ld_o, None)
    lat = [z.clone() for z in zs]
    for a, b in zip(lat, zo):
        a[idx] = b.to(DEV)
    for _ in range(calls):                                          # the second call replays the captured chain
        ld, lp = zeros2(B)
        xi = flow.invert(lat, 1.0, ld, lp)
    pl = prior.compute_log_prob(lat[-1]).double()
    n_pix = float(S * S * c)
    want = oracle_density(sd, psd, O.glow_invert(sd, zo, L, K), L, K)
    e_oracle = errors((ld[idx], lp[idx], pl[idx]), want, n_pix)
    e_own = errors((ld, lp, pl), own_density(flow, prior, xi), n_pix)
    return e_oracle, e_own, xi, lat, ld, lp


@pytest.mark.parametrize("weights,zero_sigma", [("bench", 1e-3), ("bench", 5e-3), ("seeded", 1e-3), ("seeded", 5e-3),
                                                ("seeded", 2e-2)])
def test_config2_decode_density_vs_oracle(weights, zero_sigma):
    c, L, K, B, S = 3, 3, 16, 128, 32
    make = bench_style_model if weights == "bench" else seeded_model
    flow, prior, sd, psd, x = make(c, L, K, B, S, zero_sigma)
    e_o, e_own, xi, lat, ld, lp = decode_vs_oracle(flow, prior, sd, psd, x, L, K, [0, 63, 100, 127])
    print("config2 decode", weights, zero_sigma, e_o, e_own)
    assert any(k[0] == "inv" and k[-1] == (True, True) for k in flow._graphs), "graph path not taken"
    check(e_o)
    check(e_own)
    assert torch.equal(flow.invert(lat), xi)                        # the sinks leave the decoded images unchanged


@pytest.mark.parametrize("cfg", [(3, 3, 16, 128, 32), (1, 3, 4, 128, 32)])
@pytest.mark.parametrize("temperature", [0.0, 0.7, 1.0])
def test_sampling_density(cfg, temperature):
    """invert([z_last], T, ld, lp): ld + lp + prior(z_last) is the model's density at the sample (config 2 and config 5
    shapes), against this package's transform of the sample and the oracle's."""
    c, L, K, B, S = cfg
    flow, prior, sd, psd, _ = bench_style_model(c, L, K, B, S, 1e-3)
    z_last = rnd(B, 2 ** (L + 1) * c, S >> L, S >> L, seed=5).to(DEV)
    for _ in range(2):
        ld, lp = zeros2(B)
        xs = flow.invert([z_last], temperature, ld, lp)
    pl = prior.compute_log_prob(z_last).double()
    n_pix = float(S * S * c)
    check(errors((ld, lp, pl), own_density(flow, prior, xs), n_pix))
    idx = [0, B - 1]
    check(errors((ld[idx], lp[idx], pl[idx]), oracle_density(sd, psd, xs.cpu()[idx], L, K), n_pix))


def _paths_model(B):
    return bench_style_model(3, 3, 16, B, 32, 5e-3)


@pytest.mark.parametrize("path", ["graph", "eager", "unfused", "unfused_eager", "tiled"])
def test_every_inverse_path_agrees(path, monkeypatch):
    """Config-2 geometry through each inverse path: captured and replayed (image mode), eager (NFDPM_GRAPHS=0), unfused
    (NFDPM_FUSED_BOUNDARY=0 and NFDPM_TILED=0, captured and eager) and row bands (a small batch)."""
    B = 16 if path == "tiled" else 128
    env = {"eager": {"NFDPM_GRAPHS": "0"}, "unfused": {"NFDPM_FUSED_BOUNDARY": "0", "NFDPM_TILED": "0"},
           "unfused_eager": {"NFDPM_FUSED_BOUNDARY": "0", "NFDPM_TILED": "0", "NFDPM_GRAPHS": "0"}}.get(path, {})
    flow, prior, sd, psd, x = _paths_model(B)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    flow._drop_graphs()                                             # graph keys do not carry these switches
    if path == "tiled":
        assert flow._level_mode(B, 12, 16, 16) == "tiled"
    e_o, e_own, xi, lat, _, _ = decode_vs_oracle(flow, prior, sd, psd, x, 3, 16, [0, B - 1])
    print(path, e_o, e_own)
    check(e_o)
    check(e_own)
    assert torch.equal(flow.invert(lat), xi)


def test_config4_row_bands_and_image_mode(monkeypatch):
    """Config-4 geometry (L5 K16 3x128x128, B = 8): row bands at every level by default; with NFDPM_TILED=0 the levels of
    at most 256 pixels take the one-CTA-per-image kernels and the larger ones the unfused chain.  One image against the
    oracle."""
    c, L, K, B, S = 3, 5, 16, 8, 128
    flow, prior, sd, psd, x = bench_style_model(c, L, K, B, S, 1e-3)
    zs, _, _ = flow.transform(x.to(DEV), torch.zeros(B, device=DEV), None)
    idx = [5]
    want = oracle_density(sd, psd, O.glow_invert(sd, [z.cpu()[idx] for z in zs], L, K), L, K)
    n_pix = float(S * S * c)
    for tiled in ("1", "0"):
        monkeypatch.setenv("NFDPM_TILED", tiled)
        flow._drop_graphs()
        modes = {flow._level_mode(B, (12 << i), S >> (i + 1), S >> (i + 1)) for i in range(L)}
        assert ("tiled" in modes) == (tiled == "1") and ("image" in modes) == (tiled == "0"), modes
        ld, lp = zeros2(B)
        xi = flow.invert(zs, 1.0, ld, lp)
        pl = prior.compute_log_prob(zs[-1]).double()
        e = errors((ld[idx], lp[idx], pl[idx]), want, n_pix)
        print("config4 tiled" if tiled == "1" else "config4 image/unfused", e)
        check(e)
        check(errors((ld, lp, pl), own_density(flow, prior, xi), n_pix))


def test_not_ready_model_eager_path():
    """A model whose StepFlow ActNorms are not initialised inverts through the eager unfused chain (`_invert_walk`); the
    density it returns is that of the model as it stands (the inverse initialises no StepFlow ActNorm)."""
    c, L, K, B, S = 3, 3, 2, 4, 32
    sd, psd = O.seeded_state(c, L, K, 3)
    for k in sd:
        if k.endswith("actnorm.is_initialized") and ".net." not in k:
            sd[k] = torch.tensor(0, dtype=torch.uint8)
    flow = nf.Glow(c, L, K).to(DEV)
    flow.load_state_dict(sd)
    assert not flow.blocks[0].flows[0]._ready()
    lat = [t.to(DEV) for t in O.glow_transform(sd, O.seeded_input((B, c, S, S), 4), L, K,
                                                torch.zeros(B, dtype=torch.float64), None)[0]]
    ld, lp = zeros2(B)
    xi = flow.invert(lat, 1.0, ld, lp)
    assert not flow.blocks[0].flows[0]._ready()
    ld_o, lp_o = torch.zeros(B, dtype=torch.float64), torch.zeros(B, dtype=torch.float64)
    O.glow_transform(sd, xi.cpu(), L, K, ld_o, lp_o)
    assert float(((ld.cpu() - ld_o).abs() / ld_o.abs()).max()) <= 1e-4
    assert float(((lp.cpu() - lp_o).abs() / lp_o.abs()).max()) <= 1e-4


def test_bf16_mode_stated_tolerance(monkeypatch):
    monkeypatch.setenv("NFDPM_PRECISION", "bf16")
    flow, prior, sd, psd, x = bench_style_model(3, 3, 16, 128, 32, 1e-3)
    e_o, e_own, _, _, _, _ = decode_vs_oracle(flow, prior, sd, psd, x, 3, 16, [0, 127])
    print("bf16", e_o, e_own)
    check(e_o, ld_tol=2e-4, lp_tol=2e-4)
    check(e_own, ld_tol=2e-4, lp_tol=2e-4)


# ------------------------------------------------------------------------------------------------ contract
@pytest.fixture
def small():
    c, L, K, B, S = 3, 3, 4, 64, 32
    flow, prior, sd, psd, x = bench_style_model(c, L, K, B, S, 5e-3)
    zs, _, _ = flow.transform(x.to(DEV), torch.zeros(B, device=DEV), None)
    return flow, prior, sd, psd, x, zs


def test_accumulator_dtypes_and_logp_none(small):
    flow, prior, sd, psd, x, zs = small
    B = x.shape[0]
    flow.invert(zs)
    n0 = N.launch_count
    x_plain = flow.invert(zs)
    n_plain = N.launch_count - n0
    res = {}
    for dt in (torch.float32, torch.float64):
        ld, lp = zeros2(B, dt)
        flow.invert(zs, log_det_jac=ld, logp=lp)
        res[dt] = (ld, lp)
        ld2, lp2 = ld + 1.0, lp - 2.0                               # += into what is there
        flow.invert(zs, log_det_jac=ld2, logp=lp2)
        assert torch.allclose(ld2, 2 * ld + 1.0, rtol=1e-6) and torch.allclose(lp2, 2 * lp - 2.0, rtol=1e-6)
    for a, b in zip(res[torch.float32], res[torch.float64]):
        assert torch.allclose(a.double(), b, rtol=1e-6, atol=1e-2)
    ld = torch.zeros(B, dtype=torch.float64, device=DEV)
    flow.invert(zs, log_det_jac=ld)
    n0 = N.launch_count
    x_ld = flow.invert(zs, log_det_jac=ld.zero_())
    assert N.launch_count - n0 == n_plain + 1                       # no prior work: the same chain plus one accumulate
    assert torch.equal(ld, res[torch.float64][0]) and torch.equal(x_ld, x_plain)
    lp = torch.zeros(B, dtype=torch.float64, device=DEV)
    flow.invert(zs, logp=lp)
    assert torch.equal(lp, res[torch.float64][1])


def test_learn_prior_mean_logs_false():
    c, L, K, B, S = 3, 3, 4, 64, 32
    sd, psd = O.seeded_state(c, L, K, 7, learn_prior=False)
    flow = nf.Glow(c, L, K, learn_prior_mean_logs=False).to(DEV)
    flow.load_state_dict(sd)
    z_last = rnd(B, 2 ** (L + 1) * c, S >> L, S >> L, seed=8).to(DEV)
    ld, lp = zeros2(B)
    xs = flow.invert([z_last], 0.8, ld, lp)
    ld_t, lp_t = zeros2(B)
    flow.transform(xs, ld_t, lp_t)
    assert float(((ld - ld_t).abs() / ld_t.abs()).max()) <= 1e-4
    assert float(((lp - lp_t).abs() / lp_t.abs()).max()) <= 1e-4
    ld_o, lp_o = torch.zeros(2, dtype=torch.float64), torch.zeros(2, dtype=torch.float64)
    O.glow_transform(sd, xs.cpu()[:2], L, K, ld_o, lp_o)
    assert float(((lp.cpu()[:2] - lp_o).abs() / lp_o.abs()).max()) <= 1e-4


def test_nfbackbone_invert_and_sample(small):
    flow, prior, sd, psd, x, zs = small
    B = x.shape[0]
    bb = nf.NFBackbone("", 3, 3, 4, True, True).to(DEV)
    bb.model.load_state_dict(sd)
    want = torch.zeros(B, dtype=torch.float64, device=DEV)
    x_want = flow.invert(zs, log_det_jac=want)
    ld = torch.zeros(B, dtype=torch.float64, device=DEV)
    assert torch.allclose(bb.invert(zs, ld), x_want, rtol=1e-6, atol=1e-6) and torch.allclose(ld, want, rtol=1e-9)
    torch.manual_seed(3)
    ld = torch.zeros(B, dtype=torch.float64, device=DEV)
    xs = bb.sample([zs[-1]], log_det_jac=ld)
    ld_t = torch.zeros(B, dtype=torch.float64, device=DEV)
    bb.model.transform(xs, ld_t, None)
    assert float(((ld - ld_t).abs() / ld_t.abs()).max()) <= 1e-4
    lp = torch.zeros(B, dtype=torch.float64, device=DEV)
    xp = flow.sample([zs[-1]], lambda t: t * 2, 0.5, log_det_jac=None, logp=lp)
    assert xp.shape == x.shape and bool(torch.isfinite(lp).all()) and bool((lp != 0).all())


def test_parameter_update_between_replays(small):
    flow, prior, sd, psd, x, zs = small
    B = x.shape[0]
    ld1 = torch.zeros(B, dtype=torch.float64, device=DEV)
    for _ in range(2):
        flow.invert(zs, log_det_jac=ld1.zero_())
    key = next(k for k in flow._graphs if k[0] == "inv" and k[-1] == (True, False))
    graph = flow._graphs[key]["graph"]
    flow.final_flows[1].actnorm.scale.add_(0.05)                    # in place: picked up through the version counters
    flow.blocks[0].flows[2].affcoupling.net[4].weight.mul_(1.5)
    ld2 = torch.zeros(B, dtype=torch.float64, device=DEV)
    x2 = flow.invert(zs, log_det_jac=ld2)
    assert flow._graphs[key]["graph"] is graph                      # replayed, not re-captured
    assert not torch.allclose(ld1, ld2)
    ld_t = torch.zeros(B, dtype=torch.float64, device=DEV)
    flow.transform(x2, ld_t, None)
    assert float(((ld2 - ld_t).abs() / ld_t.abs()).max()) <= 1e-4


def test_graph_entries_with_and_without_accumulators_coexist(small):
    flow, prior, sd, psd, x, zs = small
    B = x.shape[0]
    x_plain = flow.invert(zs)
    plain = [k for k in flow._graphs if k[0] == "inv"]
    assert len(plain) == 1 and len(plain[0]) == 6, plain            # the key of a call without accumulators
    g_plain = flow._graphs[plain[0]]["graph"]
    ld, lp = zeros2(B)
    x_acc = flow.invert(zs, 1.0, ld, lp)
    x_plain2 = flow.invert(zs)
    keys = [k for k in flow._graphs if k[0] == "inv"]
    assert sorted(keys, key=len) == [plain[0], plain[0] + ((True, True),)], keys
    assert flow._graphs[plain[0]]["graph"] is g_plain
    assert torch.equal(x_plain, x_acc) and torch.equal(x_plain, x_plain2)
    ld2, lp2 = zeros2(B)
    flow.invert(zs, 1.0, ld2, lp2)
    assert torch.equal(ld, ld2) and torch.equal(lp, lp2)


def test_bad_accumulators_raise(small, monkeypatch):
    flow, prior, sd, psd, x, zs = small
    B = x.shape[0]
    for bad in (torch.zeros(B + 1, device=DEV), torch.zeros(B, dtype=torch.float16, device=DEV),
                torch.zeros(B, 2, device=DEV)[:, 0], torch.zeros(B, dtype=torch.int64, device=DEV)):
        with pytest.raises(ValueError):
            flow.invert(zs, log_det_jac=bad)
        with pytest.raises(ValueError):
            flow.invert(zs, logp=bad)
    torch.set_grad_enabled(True)
    with pytest.raises(RuntimeError, match="must not require grad"):
        flow.invert(zs, log_det_jac=torch.zeros(B, device=DEV, requires_grad=True))
    # a recorded invert (NFDPM_INVERT_GRAD=1) does not take accumulators: refused before any launch
    monkeypatch.setenv("NFDPM_INVERT_GRAD", "1")
    lat = [z.clone().requires_grad_(True) for z in zs]
    n0 = N.launch_count
    with pytest.raises(NotImplementedError, match="not differentiable"):
        flow.invert(lat, log_det_jac=torch.zeros(B, device=DEV))
    assert N.launch_count == n0
    # without the knob the call computes without recording and fills the accumulators
    monkeypatch.delenv("NFDPM_INVERT_GRAD")
    ld = torch.zeros(B, dtype=torch.float64, device=DEV)
    xr = flow.invert(lat, log_det_jac=ld)
    with torch.no_grad():
        want = torch.zeros(B, dtype=torch.float64, device=DEV)
        assert torch.equal(flow.invert(zs, log_det_jac=want), xr.detach()) and torch.equal(ld, want)
