"""Time back-propagation through the density of Glow.invert (``invert_with_density``) against the recorded invert without
accumulators, on one GPU, the two arms alternating in one run.

    python tools/bench_invert_density_grad.py [--steps 10] [--rounds 5] [--warmup 3]
                                              [--out profiles/r04_invert_density_grad.jsonl]

Arms, per configuration:
  plain    x = invert(latents) (NFDPM_INVERT_GRAD=1), then x.backward(v)
  density  x, ld, lp = invert_with_density(latents, 1.0, ld, lp), then backward of (x*v).sum() + ld.sum() + lp.sum()
The difference is the cost of the density: its partial rows and accumulates in the forward, the log-det terms in every
coupling and mix backward, the per-Split log-p backward and one reduction.  Configurations: config 2 (L3 K16, 3x32x32,
B = 128) in fp32 and bf16 with every parameter trainable, and the config-5 decode geometry (L3 K4, 1x32x32, B = 128) with
a frozen flow.  Each round times --steps iterations of one arm, then of the other (CUDA events, one synchronise per
round); the medians over --rounds are reported.  L2 is not flushed; the config-2 stash (several GB) far exceeds the
126 MB L2.  One JSON line per configuration; the card name and power limit are read in the same run."""
import argparse
import json
import os
import statistics
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


def run(name, c, L, K, B, S, mode, frozen, steps, rounds, warmup):
    os.environ["NFDPM_PRECISION"] = mode
    sd, _ = O.seeded_state(c, L, K, 0)
    flow = nf.Glow(c, L, K).to(DEV)
    flow.load_state_dict(sd)
    for p in flow.parameters():
        p.requires_grad_(not frozen)
    g = torch.Generator(DEV).manual_seed(0)
    x = torch.rand(B, c, S, S, device=DEV, generator=g) - 0.5
    with torch.no_grad():
        zs, _, _ = flow.transform(x, torch.zeros(B, device=DEV), None)
    lats = [z.clone().requires_grad_(True) for z in zs]
    v = torch.randn(B, c, S, S, device=DEV, generator=g)

    def plain():
        flow.invert(lats).backward(v)

    def density():
        xi, ld, lp = flow.invert_with_density(lats, 1.0, torch.zeros(B, device=DEV), torch.zeros(B, device=DEV))
        ((xi * v).sum() + ld.sum() + lp.sum()).backward()

    for fn in (plain, density):
        for _ in range(warmup):
            fn()
    torch.cuda.synchronize()
    t = {"plain": [], "density": []}
    for _ in range(rounds):
        t["plain"].append(timed(plain, steps))
        t["density"].append(timed(density, steps))
    mp, md = statistics.median(t["plain"]), statistics.median(t["density"])
    return {"config": name, "precision": mode, "batch": B, "L": L, "K": K, "image": [c, S, S], "frozen_flow": frozen,
            "invert_backward_ms": round(mp, 3), "invert_with_density_backward_ms": round(md, 3),
            "overhead_pct": round(100.0 * (md / mp - 1.0), 2),
            "rounds_ms": {k: [round(x, 3) for x in xs] for k, xs in t.items()},
            "steps_per_round": steps, "rounds": rounds, "warmup": warmup,
            "l2": "not flushed between steps; the stash exceeds L2 at config 2"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_invert_density_grad.jsonl"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_invert_density_grad: needs a CUDA device")
    os.environ["NFDPM_INVERT_GRAD"] = "1"
    torch.set_grad_enabled(True)
    gpu = card()
    lines = []
    for cfg in CONFIGS:
        r = run(*cfg, a.steps, a.rounds, a.warmup)
        r["gpu"] = gpu
        print(json.dumps(r), flush=True)
        lines.append(json.dumps(r))
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
