"""Parity of the paths bench.py times, at BASELINE.json's sizes, in the modes it times them in (GPU).

The module-level suite (test_gpu_modules.py) runs small batches under an explicit NFDPM_PRECISION=fp32 fixture; this file
runs the benchmarked configurations themselves — default precision (NFDPM_PRECISION unset: "auto" = inference in the
fp32-faithful split-bf16-pair tensor-core mode), fused kernels, CUDA-graph replay — and compares an image subset with
the CPU oracle (every image of a batch is independent, so a subset pins the whole batch's arithmetic):

  fp32-faithful mode (default)   north-star bar: z relL2 <= 1e-4, log-det / log-p relative <= 1e-4, bits/dim |d| <= 1e-3,
                                 invert vs the oracle's inverse of the SAME latents <= max(1e-4, 2 x the oracle's own
                                 reconstruction error)  [the reference's inverse divides by s + 1e-6 where its forward
                                 multiplies by s (transforms.py:182,199): with non-zero ZeroConvs a 48-step flow is itself
                                 only invertible to ~1e-3 in fp32, so the bound is relative to what the reference achieves]
  bf16 mode (opt-in)             stated tolerance: z relL2 <= 5e-3, log-det relative <= 2e-4, bits/dim |d| <= 1e-3; the
                                 inverse is conditioning-limited (asserted at the benchmark's weights only)
"""
import os

import numpy as np
import pytest
import torch

import normalizing_flow as nf
from oracle import glow_oracle as O

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")


@pytest.fixture(autouse=True)
def _no_grad_default_precision(monkeypatch):
    monkeypatch.delenv("NFDPM_PRECISION", raising=False)       # the DEFAULT mode is what the bench times
    monkeypatch.setenv("NFDPM_GRAPHS", "1")
    monkeypatch.setenv("NFDPM_FUSED_BOUNDARY", "1")
    torch.set_grad_enabled(False)
    yield
    torch.set_grad_enabled(True)


def relerr(a, b):
    a, b = a.detach().cpu().double(), torch.as_tensor(b).detach().cpu().double()
    return float((a - b).norm() / (b.norm() + 1e-30))


def bench_style_model(c, L, K, B, S, zero_sigma):
    """bench.py's weight recipe (SURVEY 8d): reference constructors under seed 0, data-dependent ActNorm initialisation on
    the first batch, then N(0, zero_sigma) on every ZeroConv tensor."""
    torch.manual_seed(0)
    flow = nf.Glow(c, L, K).to(DEV)
    prior = nf.GaussianPrior(2 ** (L + 1) * c).to(DEV)
    x = O.seeded_input((B, c, S, S), 1)
    ld, lp = nf.initialize_with_zeros(2, B, DEV)
    flow.transform(x.to(DEV), ld, lp)
    sd = {k: v.detach().cpu().clone() for k, v in flow.state_dict().items()}
    psd = {k: v.detach().cpu().clone() for k, v in prior.state_dict().items()}
    g = torch.Generator().manual_seed(1)
    for d in (sd, psd):
        for k in d:
            if ".net.4." in k or ".split.conv." in k or "_GaussianPrior__conv." in k:
                d[k] = d[k] + zero_sigma * torch.randn(d[k].shape, generator=g)
    flow.load_state_dict(sd)
    prior.load_state_dict(psd)
    return flow, prior, sd, psd, x


def run_against_oracle(flow, prior, sd, psd, x, L, K, idx):
    """-> dict of errors of the CUDA path (whole batch) against the oracle on the images `idx`."""
    B, c, S, _ = x.shape
    ld, lp = nf.initialize_with_zeros(2, B, DEV)
    for _ in range(2):                                         # second call replays the captured chain
        ld.zero_(); lp.zero_()
        zs, ld, lp = flow.transform(x.to(DEV), ld, lp)
    pl = prior.compute_log_prob(zs[-1])
    xr = flow.invert(zs)
    n = len(idx)
    xs = x[idx]
    ld_o, lp_o = torch.zeros(n, dtype=torch.float64), torch.zeros(n, dtype=torch.float64)
    zo, ld_o, lp_o = O.glow_transform(sd, xs, L, K, ld_o, lp_o)
    pl_o = O.gaussian_prior_logp(psd, zo[-1])
    xo = O.glow_invert(sd, zo, L, K)
    # the CUDA inverse of the ORACLE's latents (scattered into a full batch) against the oracle's inverse of them
    lat = [z.clone() for z in zs]
    for a, b in zip(lat, zo):
        a[idx] = b.to(DEV)
    xi = flow.invert(lat)
    n_pix = float(S * S * 3.0)
    bpd = float(O.bpd_loss((ld + lp + pl).cpu()[idx], 32.0, n_pix))
    bpd_o = float(O.bpd_loss(ld_o + lp_o + pl_o.double(), 32.0, n_pix))
    return {"z_rel": max(relerr(a[idx], b) for a, b in zip(zs, zo)),
            "ld_rel": float(((ld.cpu()[idx] - ld_o).abs() / ld_o.abs()).max()),
            "lp_rel": float((((lp + pl).cpu()[idx] - (lp_o + pl_o)).abs() / (lp_o + pl_o).abs()).max()),
            "bpd_abs": abs(bpd - bpd_o),
            "recon_own": float((xr.cpu() - x).abs().max()),
            "recon_oracle": float((xo - xs).abs().max()),
            "inv_vs_oracle": float((xi.cpu()[idx] - xo).abs().max())}


def seeded_model(c, L, K, B, S, zero_sigma):
    """The parity suite's seeded non-degenerate weights (synthetic.seeded_state: ZeroConv entries ~ zero_sigma * 16 /
    sqrt(fan_in)); zero_sigma = 0.02 is the strongly contracting case of profiles/r01_bf16_parity.jsonl, where plain bf16
    reconstructs to 0.27 and the fp32 reference itself only to 1.6e-3."""
    sd, psd = O.seeded_state(c, L, K, 14, zero_sigma=zero_sigma)
    flow = nf.Glow(c, L, K).to(DEV)
    flow.load_state_dict(sd)
    prior = nf.GaussianPrior(2 ** (L + 1) * c).to(DEV)
    prior.load_state_dict(psd)
    return flow, prior, sd, psd, O.seeded_input((B, c, S, S), 15)


@pytest.mark.parametrize("weights,zero_sigma", [("bench", 1e-3), ("bench", 5e-3), ("seeded", 1e-3), ("seeded", 5e-3),
                                                ("seeded", 2e-2)])
def test_config2_default_mode_b128_k16_fused_graph_vs_oracle(weights, zero_sigma):
    """BASELINE config 2 exactly as bench.py runs it (B=128, L3/K16, fused-graph path, default precision): the bench's
    own weight recipe (its N(0, 1e-3) ZeroConv perturbation and a 5x stronger one; at 2e-2 of THAT recipe the fp32
    reference itself overflows) and the parity suite's seeded weights at zero_sigma 1e-3 / 5e-3 / 2e-2."""
    c, L, K, B, S = 3, 3, 16, 128, 32
    make = bench_style_model if weights == "bench" else seeded_model
    flow, prior, sd, psd, x = make(c, L, K, B, S, zero_sigma)
    idx = [0, 1, 2, 63, 64, 100, 126, 127]
    r = run_against_oracle(flow, prior, sd, psd, x, L, K, idx)
    print("config2 default mode", weights, zero_sigma, r)
    assert any(k[0] == "fwd" for k in flow._graphs) and any(k[0] == "inv" for k in flow._graphs), "graph path not taken"
    assert r["z_rel"] <= 1e-4 and r["ld_rel"] <= 1e-4 and r["lp_rel"] <= 1e-4 and r["bpd_abs"] <= 1e-3, r
    assert r["inv_vs_oracle"] <= max(1e-4, 2 * r["recon_oracle"]), r
    assert r["recon_own"] <= max(1e-4, 2 * r["recon_oracle"]), r


def test_config2_bf16_mode_b128_k16_stated_tolerance(monkeypatch):
    """The opt-in fast mode at the benchmarked size and weights: the stated bf16 tolerance, incl. a NUMERIC bound on the
    inverse (measured r1: 8.6e-4 round trip at these weights; the bound documents that plain bf16 inverses degrade with
    larger ZeroConv weights, which is why bf16 is not the default for Glow.invert)."""
    monkeypatch.setenv("NFDPM_PRECISION", "bf16")
    c, L, K, B, S = 3, 3, 16, 128, 32
    flow, prior, sd, psd, x = bench_style_model(c, L, K, B, S, 1e-3)
    r = run_against_oracle(flow, prior, sd, psd, x, L, K, [0, 1, 64, 127])
    print("config2 bf16 mode", r)
    assert r["z_rel"] <= 5e-3 and r["ld_rel"] <= 2e-4 and r["bpd_abs"] <= 1e-3, r
    assert r["recon_own"] <= 5e-3 and r["inv_vs_oracle"] <= 1e-2, r


def test_config3_b1024_default_mode_vs_oracle():
    """BASELINE config 3's single-GPU shard at N=1: batch 1024 (M = 262 144 rows at level 0)."""
    c, L, K, B, S = 3, 3, 16, 1024, 32
    flow, prior, sd, psd, x = bench_style_model(c, L, K, B, S, 1e-3)
    r = run_against_oracle(flow, prior, sd, psd, x, L, K, [0, 511, 512, 1023])
    print("config3", r)
    assert r["z_rel"] <= 1e-4 and r["ld_rel"] <= 1e-4 and r["lp_rel"] <= 1e-4 and r["bpd_abs"] <= 1e-3, r
    assert r["inv_vs_oracle"] <= max(1e-4, 2 * r["recon_oracle"]) and r["recon_own"] <= max(1e-4, 2 * r["recon_oracle"]), r


def test_config4_k16_celeba_128_default_mode_vs_oracle():
    """BASELINE config 4 at its real depth (L5, K16, 3x128x128, batch 8): row-band boundary kernels at the 64x64 / 32x32
    levels, 9C > 512 multi-tile GEMMs at the deepest level; the oracle runs one image."""
    c, L, K, B, S = 3, 5, 16, 8, 128
    flow, prior, sd, psd, x = bench_style_model(c, L, K, B, S, 1e-3)
    r = run_against_oracle(flow, prior, sd, psd, x, L, K, [5])
    print("config4", r)
    assert r["z_rel"] <= 1e-4 and r["ld_rel"] <= 1e-4 and r["lp_rel"] <= 1e-4 and r["bpd_abs"] <= 1e-3, r
    assert r["inv_vs_oracle"] <= max(1e-4, 2 * r["recon_oracle"]) and r["recon_own"] <= max(1e-4, 2 * r["recon_oracle"]), r


@pytest.mark.parametrize("cfg", [(3, 3, 16, 128, 32), (1, 3, 4, 128, 32)])
def test_sampling_variant_decodes_what_it_drew(cfg):
    """The sampling variant bench.py times (Glow.invert([z_last]): every Split draws its half from its conditional prior,
    glow.py:203-246 / transforms.py:305-307; config 2 and config 5 shapes).  The draws are internal, so parity is pinned
    through invertibility: transform(sample) returns the latents that were used; (a) the deepest one is the supplied
    z_last, (b) the oracle's inverse of those latents is the sample, (c) the drawn halves are standardised correctly:
    eps = (z - mean) / exp(logs) with the ORACLE's conditional-prior parameters is ~N(0, 1), and at temperature 0 the
    sample equals the oracle's mean decode exactly to fp32 tolerance."""
    c, L, K, B, S = cfg
    flow, prior, sd, psd, x = bench_style_model(c, L, K, B, S, 1e-3)
    rng = np.random.default_rng(5)
    z_last = torch.from_numpy(rng.standard_normal((B, 2 ** (L + 1) * c, S // 2 ** L, S // 2 ** L)).astype(np.float32))
    idx = [0, 37, B - 1]
    xs = flow.invert([z_last.to(DEV)], temperature=1.0)
    xs = flow.invert([z_last.to(DEV)], temperature=1.0)        # replayed chain, fresh noise
    ld = torch.zeros(B, dtype=torch.float64, device=DEV)
    zs, ld, _ = flow.transform(xs, ld, None)
    assert relerr(zs[-1], z_last) < 1e-3
    xo = O.glow_invert(sd, [z.cpu()[idx] for z in zs], L, K)
    rec = float((xs.cpu()[idx] - xo).abs().max())
    assert rec < 5e-3, rec                                     # (round trip through transform: twice the flow's own error)
    # temperature 0: the prior means, against the oracle with eps = 0
    x0 = flow.invert([z_last.to(DEV)], temperature=0.0)
    x0_o = O.glow_invert(sd, [z_last[idx]], L, K, temperature=0.0)
    assert float((x0.cpu()[idx] - x0_o).abs().max()) < 1e-3
    # the draws: standard normal after standardising with the oracle's conditional prior
    ld_o = torch.zeros(len(idx), dtype=torch.float64)
    zo, _, _ = O.glow_transform(sd, xs.cpu()[idx], L, K, ld_o, None)
    for a, b in zip(zs[:-1], zo[:-1]):
        assert relerr(a[idx], b) < 1e-4
    eps_all = []
    for z in zs[:-1]:
        eps_all.append(z.flatten())
    e = torch.cat(eps_all).double().cpu()
    assert torch.isfinite(e).all()
    # with near-zero split ZeroConvs (zero_sigma 1e-3) mean ~ 0 and exp(logs) ~ 1: the latents themselves are ~N(0,1)
    assert abs(float(e.mean())) < 0.02 and abs(float(e.std()) - 1.0) < 0.02, (float(e.mean()), float(e.std()))


def test_bench_dump_outputs_hold_what_the_headline_path_returns(tmp_path):
    """bench.py --dump-outputs writes what its timed headline step returned: the same arrays the public API gives for the
    bench's own weights and inputs in this process."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--steps", "2", "--warmup", "1", "--no-train",
                        "--no-cpu-baseline", "--no-eager-gpu", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=900, cwd=str(tmp_path))
    assert r.returncode == 0, r.stderr[-4000:]
    c, L, K, B, S = 3, 3, 16, 128, 32
    flow, prior, _, _, x = bench_style_model(c, L, K, B, S, 1e-3)
    ld, lp = nf.initialize_with_zeros(2, B, DEV)
    zs, ld, lp = flow.transform(x.to(DEV), ld, lp)
    lp += prior.compute_log_prob(zs[-1])
    want = {"log_likelihood": ld + lp, "x_reconstructed": flow.invert(zs), **{f"z{i}": z for i, z in enumerate(zs)}}
    assert sorted(os.listdir(out)) == sorted(k + ".npy" for k in want)
    for k, v in want.items():
        a = np.load(out / f"{k}.npy")
        v = v.cpu().numpy()
        assert a.dtype == v.dtype and a.shape == v.shape, (k, a.dtype, a.shape)
        np.testing.assert_allclose(a, v, rtol=1e-6, atol=1e-6, err_msg=k)
