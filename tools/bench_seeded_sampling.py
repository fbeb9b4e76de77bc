"""Time Glow sampling with torch's generator and a float temperature against seeded draws with a per-image temperature.

    python tools/bench_seeded_sampling.py [--steps 50] [--warmup 5] [--rounds 5] [--out profiles/r05_seeded_sampling.jsonl]

Configurations: config 2 (L3 K16, 3x32x32, B = 128) and config 5 (L3 K4, 1x32x32, B = 128), sampling from the last latent;
default precision, captured chains (the default).  Per configuration, in the same process: ``invert([z], 0.7)`` (one
``normal_()`` per Split, the draws read back by the prior kernel) and ``invert([z], T, seeds=s)`` with a [B] temperature
vector (the draws made inside the prior kernel).  CUDA events around --steps calls after --warmup; the variants alternate
within each of --rounds rounds and the median round is reported.  L2 is not flushed between calls.  One JSON line per
configuration; the card name and power limit are read in the same run."""
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
CONFIGS = [("config2_sample", 3, 3, 16, 128, 32), ("config5_sample", 1, 3, 4, 128, 32)]


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


def run(name, c, L, K, B, S, steps, warmup, rounds):
    sd, _ = O.seeded_state(c, L, K, 0)
    flow = nf.Glow(c, L, K).to(DEV)
    flow.load_state_dict(sd)
    x = O.seeded_input((B, c, S, S), 1).to(DEV)
    zs, _, _ = flow.transform(x, torch.zeros(B, device=DEV), None)
    lat = [zs[-1]]
    temp = torch.full((B,), 0.7, device=DEV)
    seeds = torch.arange(B, dtype=torch.int64, device=DEV) + 12345
    variants = {
        "float_T_torch_generator_ms": lambda: flow.invert(lat, 0.7),
        "tensor_T_seeded_ms": lambda: flow.invert(lat, temp, seeds=seeds),
    }
    launches = {}
    for k, fn in variants.items():
        for _ in range(warmup):
            fn()
        n0 = nf._native.launch_count
        fn()
        launches[k.replace("_ms", "_launches")] = nf._native.launch_count - n0
    torch.cuda.synchronize()
    times = {k: [] for k in variants}
    for _ in range(rounds):
        for k, fn in variants.items():
            times[k].append(timed(fn, steps))
    med = {k: statistics.median(v) for k, v in times.items()}
    out = {"config": name, "batch": B, "L": L, "K": K, "image": [c, S, S], "latents_given": len(lat),
           "precision": nf._engine.precision(), "captured": True}
    out.update({k: round(v, 4) for k, v in med.items()})
    out.update({k.replace("_ms", "_spread_ms"): round(max(v) - min(v), 4) for k, v in times.items()})
    out["seeded_vs_float_pct"] = round(100 * (med["tensor_T_seeded_ms"] / med["float_T_torch_generator_ms"] - 1), 2)
    out.update(launches)
    out.update({"steps": steps, "warmup": warmup, "rounds": rounds, "l2": "not flushed between calls"})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_seeded_sampling.jsonl"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_seeded_sampling: needs a CUDA device")
    gpu = card()
    lines = []
    with torch.no_grad():
        for cfg in CONFIGS:
            r = run(*cfg, a.steps, a.warmup, a.rounds)
            r["gpu"] = gpu
            print(json.dumps(r), flush=True)
            lines.append(json.dumps(r))
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
