"""Checkpoint wire format (SURVEY §8(f) row 3; reference normalizing_flow/prior.py:102-115, __init__.py:43-45,
run_baseline_experiment.py:112-114).  CPU only: constructing modules and moving state needs no kernel.

* against tests/golden/checkpoint_manifest.json — written by oracle/make_golden_checkpoint.py from a file the UNMODIFIED
  reference's own save_model produced after one real training step: file name, top-level keys, every key / shape / dtype
  in order, the optimiser layout;
* when NFDPM_REFERENCE names a checkout of the reference (it is not part of this repository): real files travel both
  ways — the reference writes, this package loads strictly, saves again, the reference loads strictly — and every tensor
  must be bit-identical.
"""
import json
import os
import subprocess
import sys

import pytest
import torch

import normalizing_flow as nf

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("NFDPM_REFERENCE", "")
GEN = os.path.join(ROOT, "oracle", "make_golden_checkpoint.py")


def _manifest(golden_dir):
    with open(os.path.join(golden_dir, "checkpoint_manifest.json")) as f:
        return json.load(f)


def _describe(sd):
    return [[k, list(v.shape), str(v.dtype).replace("torch.", "")] for k, v in sd.items()]


def _build(case):
    torch.manual_seed(1)
    flow = nf.Glow(in_channel=case["c"], L=case["L"], K=case["K"])
    prior = nf.GaussianPrior(2 ** (case["L"] + 1) * case["c"])
    opt = nf.init_optimizer("adam", list(flow.parameters()) + list(prior.parameters()), 1e-4)
    return flow, prior, opt


def test_save_model_writes_the_reference_wire_format(golden_dir, tmp_path):
    man = _manifest(golden_dir)
    flow, prior, opt = _build(man["case"])
    path = nf.save_model(None, flow, prior, opt, 7, 123, str(tmp_path))
    assert os.path.basename(path) == man["file"] and os.listdir(tmp_path) == [man["file"]]
    ck = torch.load(path, map_location="cpu")
    assert list(ck.keys()) == man["top_level_keys"] and ck["current_iter"] == man["current_iter"]
    assert _describe(ck["flow"]) == man["flow"]
    assert _describe(ck["prior_dist"]) == man["prior_dist"]
    o = ck["optimizer"]
    assert list(o.keys()) == man["optimizer"]["keys"]
    assert sorted(o["param_groups"][0].keys()) == man["optimizer"]["param_group_keys"]
    assert len(o["param_groups"][0]["params"]) == man["optimizer"]["n_params"]
    # what NFBackbone and run_baseline_experiment.py read back
    bb = nf.NFBackbone(path, man["case"]["c"], man["case"]["L"], man["case"]["K"], True, True)
    assert bb.is_frozen() and not any(p.requires_grad for p in bb.parameters())
    for k, v in flow.state_dict().items():
        assert torch.equal(bb.model.state_dict()[k], v), k
    assert list(bb.state_dict().keys()) == ["model." + k for k, _, _ in man["flow"]]


def test_save_model_diffusion_prior_naming(golden_dir, tmp_path):
    # any prior that is not a GaussianPrior (the diffusion prior) switches keys and file name (prior.py:106-109)
    man = _manifest(golden_dir)
    flow, _, opt = _build(man["case"])
    other = torch.nn.Linear(2, 2)
    path = nf.save_model(None, flow, other, opt, 12, 5, str(tmp_path))
    assert os.path.basename(path) == "model_diffusion_012.pt"
    assert list(torch.load(path, map_location="cpu").keys()) == ["nf_backbone", "diffusion_prior", "optimizer",
                                                                 "current_iter"]


def test_strict_load_rejects_foreign_layouts(golden_dir):
    man = _manifest(golden_dir)
    flow, _, _ = _build(man["case"])
    sd = flow.state_dict()
    missing = dict(sd)
    missing.pop(man["flow"][3][0])
    with pytest.raises(RuntimeError, match="Missing key"):
        flow.load_state_dict(missing, strict=True)
    wrong = dict(sd)
    wrong[man["flow"][3][0]] = torch.zeros(5, 5, 1, 1)
    with pytest.raises(RuntimeError, match="size mismatch"):
        flow.load_state_dict(wrong, strict=True)


def _run_reference(*args):
    env = dict(os.environ, NFDPM_REFERENCE=REF, PYTHONPATH="")
    r = subprocess.run([sys.executable, GEN, *args], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    return r.stdout.strip().splitlines()[-1]


@pytest.mark.skipif(not REF or not os.path.isdir(os.path.join(REF, "normalizing_flow")),
                    reason="needs a checkout of the reference project named by NFDPM_REFERENCE")
def test_checkpoints_travel_both_ways_with_the_reference(golden_dir, tmp_path):
    man = _manifest(golden_dir)
    case = man["case"]
    # 1. the reference trains one step and writes; we load strictly
    src = _run_reference("--write", str(tmp_path))
    ck = torch.load(src, map_location="cpu")
    assert _describe(ck["flow"]) == man["flow"] and _describe(ck["prior_dist"]) == man["prior_dist"]
    bb = nf.NFBackbone(src, case["c"], case["L"], case["K"], True, False)
    prior = nf.GaussianPrior(2 ** (case["L"] + 1) * case["c"])
    prior.load_state_dict(ck["prior_dist"], strict=True)
    for k, v in ck["flow"].items():
        assert torch.equal(bb.model.state_dict()[k], v), k
    assert int(bb.model.state_dict()["blocks.0.flows.0.actnorm.is_initialized"]) == 1
    opt = nf.init_optimizer("adam", list(bb.model.parameters()) + list(prior.parameters()), 1e-4)
    opt.load_state_dict(ck["optimizer"])
    # 2. we write; the reference loads strictly (NFBackbone + GaussianPrior + Adam) and saves its view again
    out = tmp_path / "ours"
    out.mkdir()
    path = nf.save_model(None, bb.model, prior, opt, 7, ck["current_iter"], str(out))
    rep = json.loads(_run_reference("--read", path))
    assert rep["ok"] and rep["current_iter"] == man["current_iter"] and rep["n_state"] == man["optimizer"]["n_state"]
    back = torch.load(path + ".ref", map_location="cpu")
    for name in ("flow", "prior_dist"):
        assert list(back[name].keys()) == list(ck[name].keys())
        for k, v in ck[name].items():
            assert torch.equal(back[name][k], v), (name, k)
    for pid, st in ck["optimizer"]["state"].items():
        for k, v in st.items():
            assert torch.equal(back["optimizer"]["state"][pid][k], v), (pid, k)
