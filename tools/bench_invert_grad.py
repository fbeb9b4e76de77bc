"""Time back-propagation through Glow.invert (NFDPM_INVERT_GRAD=1) on one GPU and, in the same run, the training step.

    python tools/bench_invert_grad.py [--steps 10] [--warmup 3] [--out profiles/r03_invert_grad.jsonl]

Configurations: config 2 (L3 K16, 3x32x32, B = 128) in fp32 and bf16 with every parameter trainable, and the config-5
decode geometry (L3 K4, 1x32x32, B = 128) with a frozen flow (latent gradient only).  Per configuration: the no-grad
invert, the recorded invert (stash), its backward, their total, and the training step both uncaptured
(NFDPM_TRAIN_GRAPHS=0, the same execution model as the uncaptured invert backward) and with its captured chains (the
default).  CUDA events around each phase, means over --steps after --warmup.  L2 is not flushed between timed steps; the
config-2 stash (several GB) far exceeds the 126 MB L2, so only the config-5 deep levels can stay resident.  One JSON line
per configuration; the card name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "normalizing-flow-with-diffusion-prior-model_b200")]
import normalizing_flow as nf  # noqa: E402
from oracle import glow_oracle as O  # noqa: E402

DEV = torch.device("cuda")
CONFIGS = [("config2", 3, 3, 16, 128, 32, "fp32", False), ("config2", 3, 3, 16, 128, 32, "bf16", False),
           ("config5_decode_frozen", 1, 3, 4, 128, 32, "fp32", True)]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name()


def timed(fn, steps):
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(steps):
        fn()
    ev[1].record()
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[1]) / steps


def run(name, c, L, K, B, S, mode, frozen, steps, warmup):
    os.environ["NFDPM_PRECISION"] = mode
    sd, psd = O.seeded_state(c, L, K, 0)
    flow = nf.Glow(c, L, K).to(DEV)
    flow.load_state_dict(sd)
    prior = nf.GaussianPrior(2 ** (L + 1) * c).to(DEV)
    prior.load_state_dict(psd)
    for p in flow.parameters():
        p.requires_grad_(not frozen)
    g = torch.Generator(DEV).manual_seed(0)
    x = torch.rand(B, c, S, S, device=DEV, generator=g) - 0.5
    with torch.no_grad():
        zs, _, _ = flow.transform(x, torch.zeros(B, device=DEV), None)
    lats = [z.clone().requires_grad_(True) for z in zs]
    v = torch.randn(B, c, S, S, device=DEV, generator=g)
    holder = {}

    def nograd():
        with torch.no_grad():
            flow.invert(zs)

    def stash():
        holder["x"] = flow.invert(lats)

    def backward():
        holder.pop("x").backward(v)

    def both():
        stash()
        backward()

    def train(captured: bool):
        os.environ["NFDPM_TRAIN_GRAPHS"] = "1" if captured else "0"
        for p in flow.parameters():
            p.requires_grad_(True)
        ld, lp = nf.initialize_with_zeros(2, B, DEV)
        z, ld, lp = flow.transform(x, ld, lp)
        lp += prior.compute_log_prob(z[-1])
        nf.calculate_loss(ld + lp, 32.0, S * S * c).backward()
        for p in flow.parameters():
            p.requires_grad_(not frozen)

    for fn in (nograd, both, lambda: train(False), lambda: train(True)):
        for _ in range(warmup):
            fn()
    torch.cuda.synchronize()
    t_ng = timed(nograd, steps)
    # stash and backward: events between the phases of each iteration, one synchronise at the end
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(steps)]
    for e in ev:
        e[0].record()
        stash()
        e[1].record()
        backward()
        e[2].record()
    torch.cuda.synchronize()
    ts = sum(e[0].elapsed_time(e[1]) for e in ev)
    tb = sum(e[1].elapsed_time(e[2]) for e in ev)
    t_tot = timed(both, steps)
    t_train = timed(lambda: train(False), steps)
    t_train_g = timed(lambda: train(True), steps)
    os.environ.pop("NFDPM_TRAIN_GRAPHS")
    return {"config": name, "precision": mode, "batch": B, "L": L, "K": K, "image": [c, S, S], "frozen_flow": frozen,
            "invert_nograd_ms": round(t_ng, 3), "invert_stash_ms": round(ts / steps, 3),
            "backward_ms": round(tb / steps, 3), "total_ms": round(t_tot, 3), "train_step_uncaptured_ms": round(t_train, 3),
            "train_step_captured_ms": round(t_train_g, 3), "steps": steps, "warmup": warmup,
            "l2": "not flushed between steps; the stash exceeds L2 at config 2"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_invert_grad.jsonl"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_invert_grad: needs a CUDA device")
    os.environ["NFDPM_INVERT_GRAD"] = "1"
    gpu = card()
    lines = []
    for cfg in CONFIGS:
        r = run(*cfg, a.steps, a.warmup)
        r["gpu"] = gpu
        print(json.dumps(r), flush=True)
        lines.append(json.dumps(r))
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
