"""Generate tests/golden/checkpoint_manifest.json from a checkpoint written by the UNMODIFIED reference.

TEST INFRASTRUCTURE ONLY.  Needs a checkout of the reference named by NFDPM_REFERENCE.  The reference's own `save_model`
(normalizing_flow/prior.py:102-115) writes `model_gaussian_XXX.pt` for a small Glow + GaussianPrior + Adam after one
real CPU training step (trainer.py:150-167 recipe); the manifest records the wire format that a drop-in must keep:
file name, top-level keys, every state_dict key with shape and dtype (in order), the optimiser's param_group keys and
per-parameter state keys / dtypes.  tests/test_checkpoint_cpu.py holds the product package to it everywhere; when
NFDPM_REFERENCE names a checkout the same test file also exchanges real checkpoint files with the reference both ways.

Usage:  python oracle/make_golden_checkpoint.py                 # (re)write the manifest
        python oracle/make_golden_checkpoint.py --write DIR     # the reference writes DIR/model_gaussian_007.pt
        python oracle/make_golden_checkpoint.py --read FILE     # the reference loads FILE (strict), re-saves it as
                                                                # FILE.ref and prints a per-dict tensor checksum
(the two sub-commands exist because the product package has the reference's package name: the reference has to run in
its own process)
"""
from __future__ import annotations

import json
import logging
import os
import sys
import tempfile

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle.make_golden import import_reference  # noqa: E402

CASE = dict(c=1, L=2, K=1, B=2, S=8)


def describe(sd):
    return [[k, list(v.shape), str(v.dtype).replace("torch.", "")] for k, v in sd.items()]


def reference_checkpoint(nf, directory, steps=1):
    """One reference training step on CPU, then the reference's save_model.  Returns (path, flow, prior, optimiser)."""
    torch.manual_seed(0)
    c, L, K, B, S = (CASE[k] for k in "cLKBS")
    flow = nf.Glow(in_channel=c, L=L, K=K)
    prior = nf.GaussianPrior(2 ** (L + 1) * c)
    opt = torch.optim.Adam(list(flow.parameters()) + list(prior.parameters()), lr=1e-4)
    x = torch.rand(B, c, S, S) - 0.5
    for _ in range(steps):
        ld, lp = nf.initialize_with_zeros(2, B, torch.device("cpu"))
        zs, ld, lp = flow.transform(x, ld, lp)
        lp = lp + prior.compute_log_prob(zs[-1])
        loss = sys.modules["normalizing_flow.utils"].calculate_loss(ld + lp, 32.0, S * S * 3.0)
        opt.zero_grad()
        loss.backward()
        torch.nn.utils.clip_grad_value_(flow.parameters(), 1)
        torch.nn.utils.clip_grad_norm_(flow.parameters(), 1)
        opt.step()
    nf.save_model(logging.getLogger("golden"), flow, prior, opt, 7, 123, directory)
    return os.path.join(directory, "model_gaussian_007.pt"), flow, prior, opt


def checksum(sd) -> float:
    return float(sum(v.double().abs().sum() for v in sd.values() if torch.is_tensor(v)))


def reference_reads(nf, path):
    """The reference's own load path (__init__.py:43-45 for the flow; strict load for prior and optimiser)."""
    c, L, K = CASE["c"], CASE["L"], CASE["K"]
    ck = torch.load(path, map_location="cpu")
    bb = nf.NFBackbone(model_dir=path, in_channel=c, L=L, K=K, learn_prior_mean_logs=True, freeze_flow=True)
    prior = nf.GaussianPrior(2 ** (L + 1) * c)
    prior.load_state_dict(ck["prior_dist"], strict=True)
    flow = bb.model
    opt = torch.optim.Adam(list(flow.parameters()) + list(prior.parameters()), lr=1e-4)
    opt.load_state_dict(ck["optimizer"])
    torch.save({"flow": flow.state_dict(), "prior_dist": prior.state_dict(), "optimizer": opt.state_dict(),
                "current_iter": ck["current_iter"]}, path + ".ref")
    print(json.dumps({"ok": True, "flow": checksum(flow.state_dict()), "prior_dist": checksum(prior.state_dict()),
                      "current_iter": ck["current_iter"], "n_state": len(opt.state_dict()["state"])}))


def main():
    import warnings
    warnings.filterwarnings("ignore")
    nf = import_reference()
    if len(sys.argv) == 3 and sys.argv[1] == "--write":
        print(reference_checkpoint(nf, sys.argv[2])[0])
        return
    if len(sys.argv) == 3 and sys.argv[1] == "--read":
        reference_reads(nf, sys.argv[2])
        return
    with tempfile.TemporaryDirectory() as d:
        path, flow, prior, opt = reference_checkpoint(nf, d)
        assert os.listdir(d) == ["model_gaussian_007.pt"], os.listdir(d)
        ck = torch.load(path, map_location="cpu")
    ost = ck["optimizer"]
    first = ost["state"][0]
    man = {
        "case": CASE, "file": "model_gaussian_007.pt", "top_level_keys": list(ck.keys()),
        "current_iter": ck["current_iter"],
        "flow": describe(ck["flow"]), "prior_dist": describe(ck["prior_dist"]),
        "optimizer": {"keys": list(ost.keys()), "param_group_keys": sorted(ost["param_groups"][0].keys()),
                      "n_params": len(ost["param_groups"][0]["params"]), "n_state": len(ost["state"]),
                      "state_keys": list(first.keys()),
                      "state_dtypes": {k: str(v.dtype).replace("torch.", "") for k, v in first.items()}},
        "torch": torch.__version__,
    }
    out = os.path.join(ROOT, "tests", "golden", "checkpoint_manifest.json")
    with open(out, "w") as f:
        json.dump(man, f)
    print("wrote", out, len(man["flow"]), "flow tensors,", len(man["prior_dist"]), "prior tensors")


if __name__ == "__main__":
    main()
