"""Generate tests/golden/*.npz by running the UNMODIFIED reference package.

Needs a checkout of the reference named by NFDPM_REFERENCE; the tests use the committed
fixtures.  Usage:  NFDPM_REFERENCE=<checkout> python oracle/make_golden.py

For every case: weights/inputs come from oracle.glow_oracle.seeded_state / seeded_input
(numpy PCG64 — regenerated bit-identically by the tests; a checksum is stored to prove it),
are loaded into the reference modules with load_state_dict(strict=True) (which also pins the
state_dict key layout), and the reference's own transform / invert / compute_log_prob
outputs are stored.
"""
from __future__ import annotations

import os
import sys
from unittest.mock import MagicMock

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
REF = os.environ.get("NFDPM_REFERENCE", "")


def import_reference():
    """Import the reference's normalizing_flow package; its non-hot-path imports (aim,
    skimage, cleanfid, ignite) are absent from this image and are stubbed."""
    for m in ["aim", "skimage", "skimage.transform", "cleanfid", "cleanfid.fid", "cleanfid.features",
              "cleanfid.utils", "cleanfid.resize", "ignite", "ignite.metrics"]:
        sys.modules.setdefault(m, MagicMock())
    if not REF or not os.path.isdir(os.path.join(REF, "normalizing_flow")):
        raise SystemExit("set NFDPM_REFERENCE to a checkout of the reference project")
    sys.path.insert(0, REF)
    import normalizing_flow as nf  # noqa
    assert os.path.realpath(nf.__file__).startswith(os.path.realpath(REF)), nf.__file__
    return nf


def np_(t):
    return t.detach().cpu().numpy()


def main():
    import warnings
    warnings.filterwarnings("ignore")
    nf = import_reference()
    from oracle import glow_oracle as O
    out_dir = os.path.join(ROOT, "tests", "golden")
    os.makedirs(out_dir, exist_ok=True)
    torch.set_grad_enabled(False)

    def glow_case(name, c, L, K, B, S, seed, learn_prior=True):
        sd, psd = O.seeded_state(c, L, K, seed, learn_prior=learn_prior)
        ref = nf.Glow(in_channel=c, L=L, K=K, learn_prior_mean_logs=learn_prior)
        ref.load_state_dict(sd, strict=True)
        assert [k for k in ref.state_dict()] == [k for k, _, _ in O.glow_param_shapes(c, L, K, learn_prior)]
        x = O.seeded_input((B, c, S, S), seed + 1000)
        ld = torch.zeros(B, dtype=torch.float64)
        lp = torch.zeros(B, dtype=torch.float64)
        zs, ld, lp = ref.transform(x, ld, lp)
        ld_nolp = torch.zeros(B, dtype=torch.float64)
        zs2, ld_nolp, none = ref.transform(x, ld_nolp, None)
        assert none is None
        rec = {"x": np_(x), "ld": np_(ld), "logp": np_(lp), "ld_nolp": np_(ld_nolp),
               "cfg": np.array([c, L, K, B, S, seed, int(learn_prior)]),
               "checksum": np.array(O.state_checksum(sd))}
        for i, z in enumerate(zs):
            rec[f"z{i}"] = np_(z)
        if learn_prior:
            gp = nf.GaussianPrior(in_channels=2 ** (L + 1) * c)
            gp.load_state_dict(psd, strict=True)
            rec["prior_logp"] = np_(gp.compute_log_prob(zs[-1]))
            eps = torch.from_numpy(np.random.default_rng(seed + 7).standard_normal(tuple(zs[-1].shape)).astype(np.float32))
            # GaussianPrior.sample draws eps itself; pin its parameters through T=0 and the eps path via oracle check
            rec["prior_sample_T0"] = np_(gp.sample(tuple(zs[-1].shape), temperature=0.0))
            rec["prior_eps"] = np_(eps)
            m, lg = O.gaussian_prior_params(psd, zs[-1].shape)
            rec["prior_sample_eps"] = np_(m + torch.exp(lg) * 0.7 * eps)
            rec["prior_checksum"] = np.array(O.state_checksum(psd))
        rec["x_rec"] = np_(ref.invert(list(zs)))
        rec["x_T0"] = np_(ref.invert([zs[-1]], temperature=0.0))
        # oracle agreement, checked at generation time too
        ld_o = torch.zeros(B, dtype=torch.float64)
        lp_o = torch.zeros(B, dtype=torch.float64)
        zo, ld_o, lp_o = O.glow_transform(sd, x, L, K, ld_o, lp_o)
        for a, b in zip(zo, zs):
            assert torch.allclose(a, b, rtol=1e-5, atol=1e-6), name
        assert torch.allclose(ld_o, ld, rtol=1e-7) and torch.allclose(lp_o, lp, rtol=1e-7), name
        assert torch.allclose(O.glow_invert(sd, list(zs), L, K), ref.invert(list(zs)), rtol=1e-5, atol=1e-6)
        np.savez_compressed(os.path.join(out_dir, name + ".npz"), **rec)
        print(name, "ok", {k: v.shape for k, v in rec.items() if k.startswith("z")})

    glow_case("glow_c1_L3_K2_b3_s32", 1, 3, 2, 3, 32, 11)
    glow_case("glow_c3_L3_K1_b2_s32", 3, 3, 1, 2, 32, 12)
    glow_case("glow_c3_L2_K1_b5_s16", 3, 2, 1, 5, 16, 13)
    glow_case("glow_c1_L2_K1_b2_s8_noprior", 1, 2, 1, 2, 8, 14, learn_prior=False)

    # ---- one training step's loss and gradients (trainer.py:154-164) from the reference's own autograd
    def grad_case(name, c, L, K, B, S, seed):
        sd, psd = O.seeded_state(c, L, K, seed)
        ref = nf.Glow(in_channel=c, L=L, K=K)
        ref.load_state_dict(sd, strict=True)
        gp = nf.GaussianPrior(in_channels=2 ** (L + 1) * c)
        gp.load_state_dict(psd, strict=True)
        x = O.seeded_input((B, c, S, S), seed + 1000)
        from normalizing_flow.utils import calculate_loss, initialize_with_zeros
        n_bins, n_pixel = 32.0, S * S * 3.0
        with torch.enable_grad():
            ld, lp = initialize_with_zeros(2, B, torch.device("cpu"))
            zs, ld, lp = ref.transform(x, ld, lp)
            lp += gp.compute_log_prob(zs[-1])
            loss = calculate_loss(ld + lp, n_bins, n_pixel)
            loss.backward()
        rec = {"x": np_(x), "loss": np_(loss), "cfg": np.array([c, L, K, B, S, seed, 1]),
               "checksum": np.array(O.state_checksum(sd))}
        lo, g_o, pg_o = O.train_grads(sd, psd, x, L, K, n_bins, n_pixel)
        assert torch.allclose(lo, loss.detach(), rtol=1e-9), name
        names = []
        for i, (k, p) in enumerate(list(ref.named_parameters()) + [("prior/" + k, p) for k, p in gp.named_parameters()]):
            g = p.grad if p.grad is not None else torch.zeros_like(p)
            rec["sig/" + k] = np.array(O.grad_signature(g, 5000 + i))
            if g.numel() <= 4096:
                rec["grad/" + k] = np_(g)
            go = pg_o[k[len("prior/"):]] if k.startswith("prior/") else g_o[k]
            assert torch.allclose(go, g, rtol=1e-4, atol=1e-7), (name, k, float((go - g).abs().max()))
            names.append(k)
        rec["names"] = np.array(names)
        np.savez_compressed(os.path.join(out_dir, name + ".npz"), **rec)
        print(name, "ok", float(loss), len(names), "parameters")

    grad_case("glow_grad_c3_L2_K2_b3_s16", 3, 2, 2, 3, 16, 51)
    grad_case("glow_grad_c1_L3_K1_b2_s32", 1, 3, 1, 2, 32, 52)

    # ---- data-dependent initialisation (transforms.py:74-78 through the whole model)
    c, L, K, B, S, seed = 1, 2, 1, 6, 16, 21
    sd, _ = O.seeded_state(c, L, K, seed, initialized=False)
    ref = nf.Glow(in_channel=c, L=L, K=K)
    ref.load_state_dict(sd, strict=True)
    x = O.seeded_input((B, c, S, S), seed + 1000)
    ld = torch.zeros(B, dtype=torch.float64)
    lp = torch.zeros(B, dtype=torch.float64)
    zs, ld, lp = ref.transform(x, ld, lp)
    rec = {"x": np_(x), "ld": np_(ld), "logp": np_(lp), "cfg": np.array([c, L, K, B, S, seed, 1]),
           "checksum": np.array(O.state_checksum(sd))}
    for i, z in enumerate(zs):
        rec[f"z{i}"] = np_(z)
    after = ref.state_dict()
    for k, v in after.items():
        if "actnorm" in k:
            rec["sd/" + k] = np_(v)
    np.savez_compressed(os.path.join(out_dir, "glow_init_c1_L2_K1_b6_s16.npz"), **rec)
    print("glow_init ok")

    # ---- the three transforms the reference's own tests exercise (tests/transformations.py)
    rng = np.random.default_rng(31)
    x3 = torch.from_numpy(rng.standard_normal((8, 3, 28, 28)).astype(np.float32))
    an = nf.ActNorm(in_channels=3)
    ld = torch.zeros(8)
    y, ld, _ = an.transform(x3, ld, torch.zeros(8))
    rec = {"x": np_(x3), "y": np_(y), "ld": np_(ld), "scale": np_(an.scale), "bias": np_(an.bias),
           "inv": np_(an.invert(y))}
    w = torch.from_numpy(rng.standard_normal((3, 3)).astype(np.float32)).reshape(3, 3, 1, 1)
    ic = nf.InvConv2d(in_channels=3)
    ic.weight.data.copy_(w)
    ld = torch.zeros(8)
    y, ld, _ = ic.transform(x3, ld, torch.zeros(8))
    rec.update({"ic_w": np_(w), "ic_y": np_(y), "ic_ld": np_(ld), "ic_inv": np_(ic.invert(y))})
    x4 = torch.from_numpy(rng.standard_normal((4, 4, 28, 28)).astype(np.float32))
    ac = nf.AffineCoupling(4)
    sdc, _ = O.seeded_state(1, 2, 1, 41)          # blocks.0.flows.0 has C=4
    pre = "blocks.0.flows.0.affcoupling."
    ac.load_state_dict({k[len(pre):]: v for k, v in sdc.items() if k.startswith(pre)}, strict=True)
    ld = torch.zeros(4)
    y, ld, _ = ac.transform(x4, ld, torch.zeros(4))
    rec.update({"ac_x": np_(x4), "ac_y": np_(y), "ac_ld": np_(ld), "ac_inv": np_(ac.invert(y))})
    # squeeze / unsqueeze channel order
    xs = torch.arange(2 * 3 * 4 * 6, dtype=torch.float32).reshape(2, 3, 4, 6)
    sq = nf.Squeeze()
    ys = sq.transform(xs, None, None)[0]
    rec.update({"sq_x": np_(xs), "sq_y": np_(ys), "sq_inv": np_(sq.invert(ys))})
    np.savez_compressed(os.path.join(out_dir, "transforms.npz"), **rec)
    print("transforms ok")

    # ---- step glue: preprocess / postprocess / loss (utils.py:175-256)
    img = torch.from_numpy(rng.random((2, 3, 8, 8)).astype(np.float32))
    pp = nf.preprocess_batch(img, 5, 32.0)
    from normalizing_flow.utils import calculate_loss
    ll = torch.from_numpy(rng.standard_normal(7) * 100 - 5000)
    rec = {"img": np_(img), "pre": np_(pp), "post": np_(nf.postprocess_batch(pp, 32.0)),
           "ll": np_(ll), "loss": np_(calculate_loss(ll, 32.0, 32 * 32 * 3.0)),
           "shapes": np.array(nf.calculate_output_shapes(3, 3, 32))}
    np.savez_compressed(os.path.join(out_dir, "glue.npz"), **rec)
    print("glue ok")


if __name__ == "__main__":
    main()
