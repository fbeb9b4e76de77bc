"""Generate tests/golden/formats.npz from the UNMODIFIED reference: CatFormater.process_latents / postprocess
(diffusion_prior/latent_formaters.py), postprocess_batch over its whole clipping range and preprocess_batch + the
dequantisation noise add (normalizing_flow/utils.py:175-210, trainer.py:155).  Needs a checkout of the reference
named by NFDPM_REFERENCE.  Usage:  NFDPM_REFERENCE=<checkout> python oracle/make_golden_formats.py

The reference's diffusion_prior/__init__.py imports its trainer (UNet, denoising_diffusion_pytorch ... absent here), so
latent_formaters.py is loaded as a stand-alone module from its file; nothing in it is modified."""
from __future__ import annotations

import importlib.util
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle.make_golden import import_reference, REF, np_  # noqa: E402

CASES = [("L3_c1_s32", 3, 1, 32, 2), ("L3_c3_s32", 3, 3, 32, 2), ("L4_c1_s32", 4, 1, 32, 1), ("L5_c3_s32", 5, 3, 32, 2),
         ("L5_c3_s64", 5, 3, 64, 1)]


def seeded_latents(dims, B, seed):
    rng = np.random.default_rng(seed)
    return [torch.from_numpy(rng.standard_normal((B,) + tuple(int(v) for v in d)).astype(np.float32)) for d in dims]


def main():
    nf = import_reference()
    spec = importlib.util.spec_from_file_location("ref_latent_formaters",
                                                  os.path.join(REF, "diffusion_prior", "latent_formaters.py"))
    lf = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(lf)
    rec = {}
    for i, (name, L, c, S, B) in enumerate(CASES):
        fm = lf.CatFormater(L, c, S)
        lat = seeded_latents(fm.latent_dims, B, 700 + i)
        cat = fm.process_latents([t.clone() for t in lat])
        assert len(cat) == 1
        back = fm.postprocess([cat[0].clone()])
        assert len(back) == L and all(torch.equal(a, b) for a, b in zip(back, lat)), name
        rec[name + "_cat"] = np_(cat[0])
        rec[name + "_dims"] = np.array(fm.latent_dims)
        rec[name + "_input_shapes"] = np.array(fm.get_input_shapes())
        # postprocess of an independent tensor (not a process_latents output)
        rng = np.random.default_rng(800 + i)
        q = torch.from_numpy(rng.standard_normal(tuple(cat[0].shape)).astype(np.float32))
        for j, t in enumerate(fm.postprocess([q.clone()])):
            rec[f"{name}_post{j}"] = np_(t)
        idf = lf.IdentityFormater(L, c, S)
        assert idf.get_num_latent_parts() == L and fm.get_num_latent_parts() == 1
        rec[name + "_id_shapes"] = np.array(idf.get_input_shapes())
    # pixel formats: values beyond both clipping ends, every bin edge, n_bits 5 and 8
    rng = np.random.default_rng(900)
    xs = torch.from_numpy(np.concatenate([rng.uniform(-0.8, 0.8, 4000), np.arange(-40, 40) / 32.0 - 0.5,
                                          np.nextafter(np.arange(-40, 40) / 32.0 - 0.5, -10)]).astype(np.float32))
    rec["post_x"] = np_(xs)
    rec["post_u8_32"] = np_(nf.postprocess_batch(xs, 32.0))
    rec["post_u8_256"] = np_(nf.postprocess_batch(xs, 256.0))
    img = torch.from_numpy(rng.random((3, 3, 9, 7)).astype(np.float32))       # 567 values: not a multiple of 4
    u = torch.from_numpy(rng.random((3, 3, 9, 7)).astype(np.float32))
    rec["pre_img"], rec["pre_noise"] = np_(img), np_(u)
    for n_bits in (5, 8, 3):
        n_bins = 2.0 ** n_bits
        pre = nf.preprocess_batch(img, n_bits, n_bins)
        rec[f"pre_{n_bits}"] = np_(pre)
        rec[f"dq_{n_bits}"] = np_(pre + u / n_bins)
    out = os.path.join(ROOT, "tests", "golden", "formats.npz")
    np.savez_compressed(out, **rec)
    print("formats ok", os.path.getsize(out), "bytes")


if __name__ == "__main__":
    main()
