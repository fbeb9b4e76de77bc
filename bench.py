#!/usr/bin/env python
"""bench.py — Glow L3/K16 32x32 forward(+log-det, +log-p) and inverse images/s on 1..8 B200.

Contract (see the task statement): `python bench.py --gpus N --steps K --warmup W [--impl reference]`, launched
under torchrun for N>1 (one rank per GPU).  One "step" = one pass of the hot path over one batch of synthetic
images: Glow.transform + GaussianPrior.compute_log_prob (x -> z, log-det, log-p) followed by Glow.invert (z -> x).
Rank 0 prints ONE JSON line.

  value        images/s (whole job) in the DEFAULT precision mode (NFDPM_PRECISION=auto: inference in the fp32-faithful
               split-bf16-pair tensor-core mode that meets the reference's 1e-4 parity bar), inputs resident in HBM,
               device-timed with CUDA events, L2 flushed between timed steps, max over ranks
  e2e          same metric through the public module API with HOST (pinned) inputs: H2D of the batch and D2H of
               the per-image log-likelihood and the decoded images inside the timed region
  directions   forward(+log-det,+log-p), inverse (all L latents) and the sampling variant (last latent only) separately
  modes        the same measurements + parity checks per precision mode ("fp32" = the headline, "bf16" = the opt-in fast
               mode with its stated tolerance)
  roofline     the dominant kernel (coupling-net 512x512 GEMM at level 0) timed alone (16 back-to-back launches per
               CUDA-graph replay): algorithmic FLOP/s vs the measured bf16 BURST peak in MEASURED_PEAKS.json (peak/3 in
               the 3-MMA fp32-faithful mode), with cuBLAS on the same shape beside it; roofline_hbm: the step-boundary
               (ActNorm + 1x1 conv + affine coupling) kernels against the measured HBM copy bandwidth
  cpu_baseline the UNMODIFIED reference module (baseline/_ref, staged by __graft_entry__.build()) on the host CPU, all
               host threads, on a bounded sample of the same workload (rank 0 / N=1 only; own process)
  gpu_eager_reference  the same unmodified module on cuda:0 through torch eager / cuDNN (SURVEY §2b: the number the
               kernels must beat), own process

`--impl reference`: the reference arm — the unmodified reference module on the host CPU for the same config (batch 128).

`--dump-outputs DIR`: after the timed steps, rank 0 writes what the headline path returned in its last timed step as
DIR/<name>.npy: log_likelihood (float64, per image), x_reconstructed and the latents z0..z{L-1} (float32).  Inputs and
weights are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "normalizing-flow-with-diffusion-prior-model_b200")

CFG = dict(in_channel=3, L=3, K=16, S=32, batch=128)          # BASELINE.json configs[1]
WORKLOAD = "Glow L3 K16, CIFAR-10 shape 3x32x32, batch 128 per GPU, fwd+logdet+logp then inverse"
METRIC = "Glow L3/K16 32×32 fwd+logdet & inverse imgs/sec"      # BASELINE.json's metric (its leading clause)
FLOP_PER_IMG_FWD = 4.0119e9                                   # SURVEY.md §8 (verified with torch flop counter)
WEIGHTS = ("reference constructors (seed 0) + data-dependent ActNorm init on the first batch + N(0,1e-3) on every "
           "ZeroConv tensor (SURVEY 8d)")
DTYPE_NAME = {"auto": "bf16x3 (split bf16 pairs on tcgen05, fp32 accumulate: fp32-faithful)",
              "fp32": "bf16x3 (split bf16 pairs on tcgen05, fp32 accumulate: fp32-faithful)",
              "bf16": "bf16", "fp32_simt": "fp32 (CUDA cores)"}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops", 1590.0), d.get("bf16_tflops_sustained", 1400.0), "measured"
    return 6650.0, 1590.0, 1400.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu: int):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(gpu), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0: float, t1: float):
        if self.proc is None:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = [r for t, r in self.rows if t0 - 0.05 <= t <= t1 + 0.15] or [r for _, r in self.rows]
        for r in rows:
            f = [v.strip() for v in r.split(",")]
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except Exception:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return None
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def perturb_zero_convs(torch, sd, psd):
    """N(0, 1e-3) (generator seed 1) on every ZeroConv2d tensor, in key order: no term of the path is degenerate."""
    g = torch.Generator().manual_seed(1)
    for d in (sd, psd):
        for k in d:
            if ".net.4." in k or ".split.conv." in k or "_GaussianPrior__conv." in k:
                d[k] = d[k] + 1e-3 * torch.randn(d[k].shape, generator=g)
    return sd, psd


def reference_style_state(nf, torch, dev, x_first):
    """Weights as SURVEY §8(d) specifies them: the module constructors under torch.manual_seed(0) (QR-initialised 1x1
    convs, N(0, 0.05) coupling convs, zero ZeroConvs: transforms.py:112-114, utils.py:37-38,64-65), the data-dependent
    ActNorm initialisation on the first batch (transforms.py:74-78, always fp32), then `perturb_zero_convs`.  Works with
    the product package AND with the unmodified reference (same constructors, same state_dict).  Returns CPU state dicts."""
    c, L, K = CFG["in_channel"], CFG["L"], CFG["K"]
    torch.manual_seed(0)
    flow = nf.Glow(c, L, K).to(dev)
    prior = nf.GaussianPrior(2 ** (L + 1) * c).to(dev)
    x = x_first.to(dev)
    with torch.no_grad():
        ld, lp = nf.initialize_with_zeros(2, x.shape[0], dev)
        flow.transform(x, ld, lp)
    sd = {k: v.detach().cpu().clone() for k, v in flow.state_dict().items()}
    psd = {k: v.detach().cpu().clone() for k, v in prior.state_dict().items()}
    return perturb_zero_convs(torch, sd, psd)


# ------------------------------------------------------------------------------------------- reference arms (own process)
def run_reference(args, on_gpu: bool):
    """--impl reference: the UNMODIFIED reference module (baseline/_ref) through its own public API — Glow.transform +
    GaussianPrior.compute_log_prob + Glow.invert under no_grad, fp32 — on the host CPU with all host threads (the
    reference arm / cpu_baseline), or with `--impl reference-gpu` on cuda:0 through torch eager + cuDNN (the
    gpu_eager_reference comparator).  Falls back to the oracle port (kind "port") when no copy of the reference exists."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if not on_gpu:
        os.environ["CUDA_VISIBLE_DEVICES"] = ""            # the reference picks cuda whenever it is visible (base.py:18)
    import torch
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    import synthetic as SY
    from oracle import reference_module as RM
    # torchrun exports OMP_NUM_THREADS=1 to every rank; the other ranks have exited, so rank 0 takes all host cores
    if not on_gpu:
        torch.set_num_threads(max(torch.get_num_threads(), os.cpu_count() or 1))
    c, L, K, S, B = CFG["in_channel"], CFG["L"], CFG["K"], CFG["S"], args.batch
    dev = torch.device("cuda", 0) if on_gpu else torch.device("cpu")
    x = SY.seeded_input((B, c, S, S), 1)
    kind = "reference"
    try:
        nf = RM.import_reference()
        sd, psd = reference_style_state(nf, torch, dev, x)
        flow = nf.Glow(c, L, K).to(dev)
        flow.load_state_dict(sd)
        prior = nf.GaussianPrior(2 ** (L + 1) * c).to(dev)
        prior.load_state_dict(psd)
        flow.eval()
        xd = x.to(dev)

        def fwd():
            ld, lp = nf.initialize_with_zeros(2, B, dev)
            zs, ld, lp = flow.transform(xd, ld, lp)
            lp = lp + prior.compute_log_prob(zs[-1])
            return zs, ld + lp

        def inv(zs):
            return flow.invert(zs)
    except ImportError as e:
        if on_gpu:
            print(json.dumps({"impl": "reference-gpu", "unavailable": str(e).splitlines()[0]}))
            return
        kind = "port"
        from oracle import glow_oracle as O
        sd, psd = O.seeded_state(c, L, K, 0)

        def fwd():
            ld = torch.zeros(B, dtype=torch.float64)
            lp = torch.zeros(B, dtype=torch.float64)
            zs, ld, lp = O.glow_transform(sd, x, L, K, ld, lp)
            return zs, ld + lp + O.gaussian_prior_logp(psd, zs[-1])

        def inv(zs):
            return O.glow_invert(sd, zs, L, K)

    def sync():
        if on_gpu:
            torch.cuda.synchronize()

    def step():
        zs, ll = fwd()
        sync()
        t_mid = time.perf_counter()
        xr = inv(zs)
        sync()
        return t_mid, xr

    tf32 = None
    if on_gpu:
        # torch's defaults: cuDNN convolutions may use TF32 (allow_tf32=True), matmuls may not
        tf32 = bool(torch.backends.cudnn.allow_tf32) if args.tf32 is None else bool(args.tf32)
        torch.backends.cudnn.allow_tf32 = tf32
    budget = args.time_budget
    with torch.no_grad():
        t0 = time.perf_counter()
        step()
        first = time.perf_counter() - t0
        warm = max(0, min(args.warmup - 1, int(0.2 * budget / max(first, 1e-3))))
        for _ in range(warm):
            step()
        t0 = time.perf_counter()
        step()
        one = time.perf_counter() - t0
        steps = max(1, min(args.steps, int(0.8 * budget / max(one, 1e-3))))
        t_f = t_i = 0.0
        recon = 0.0
        for _ in range(steps):
            sync()
            a = time.perf_counter()
            t_mid, xr = step()
            b = time.perf_counter()
            t_f += t_mid - a
            t_i += b - t_mid
        recon = float((xr.cpu() - x).abs().max())
    dt = (t_f + t_i) / steps
    val = B / dt
    cores = torch.get_num_threads()
    what = "unmodified reference module (baseline/_ref)" if kind == "reference" else "oracle port (no copy of the reference on this box)"
    if on_gpu:
        print(json.dumps({"impl": "reference-gpu", "value": val, "unit": "img/s", "ms_per_step": dt * 1e3, "steps": steps,
                          "warmup": warm + 1, "batch": B, "forward_ms": t_f / steps * 1e3, "inverse_ms": t_i / steps * 1e3,
                          "dtype": "fp32 tensors; cuDNN conv allow_tf32=%s" % tf32, "recon_max_abs_err": recon,
                          "how": f"{what} on cuda:0, torch {torch.__version__} eager, wall clock around synchronised steps"}))
        return
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "img/s", "n_gpus": args.gpus, "steps": steps,
            "warmup": warm + 1, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "fp32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "global_batch": B, "weights": WEIGHTS,
                       "steps_requested": args.steps, "warmup_requested": args.warmup,
                       "note": f"steps bounded by a {budget:.0f} s budget" if steps < args.steps else "as requested"},
            "directions": {"forward": {"value": B / (t_f / steps), "unit": "img/s", "ms": t_f / steps * 1e3},
                           "inverse": {"value": B / (t_i / steps), "unit": "img/s", "ms": t_i / steps * 1e3}},
            "checks": {"recon_max_abs_err": recon},
            "cpu_baseline": {"value": val, "unit": "img/s", "cores": cores, "kind": kind,
                             "sample": f"{what}: batch {B}, {steps} steps after {warm + 1} warm-up, "
                                       f"os.cpu_count={os.cpu_count()}"},
            "e2e": {"value": val, "unit": "img/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def spawn_arm(impl: str, extra, timeout: float):
    """Run a reference arm in its own process (it imports a package of the same name as the product's) -> parsed JSON."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", impl] + [str(a) for a in extra]
    env = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "OMP_NUM_THREADS", "NFDPM_PRECISION"):
        env.pop(k, None)
    try:
        r = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=timeout)
    except subprocess.TimeoutExpired:
        return {"unavailable": f"timed out after {timeout:.0f} s"}
    for ln in reversed(r.stdout.strip().splitlines()):
        if ln.startswith("{"):
            return json.loads(ln)
    return {"unavailable": (r.stderr.strip().splitlines() or ["no output"])[-1][:300]}


# ------------------------------------------------------------------------------------------- training step
def bench_train(args, torch, dist, nf, N, dev, world, rank, B, x_host, timed, flush_buf, state):
    """Full training step of the reference recipe (normalizing_flow/trainer.py:150-167): dequantisation noise,
    transform, prior log-prob, bits/dim loss, backward, [gradient all-reduce over NCCL when N > 1], clip value 1,
    clip norm 1, Adam(1e-4).  The whole step is captured once in a CUDA graph and replayed (host launch overhead of
    the ~1100 kernels would otherwise dominate); `e2e` adds the H2D copy of the batch and the D2H read of the loss."""
    c, L, K, S = CFG["in_channel"], CFG["L"], CFG["K"], CFG["S"]
    n_bins, n_pixel = 32.0, S * S * 3.0
    sd, psd = state
    flow = nf.Glow(c, L, K).to(dev)
    flow.load_state_dict(sd)
    prior = nf.GaussianPrior(2 ** (L + 1) * c).to(dev)
    prior.load_state_dict(psd)
    params = list(flow.parameters()) + list(prior.parameters())
    if args.torch_optimizer:
        opt = torch.optim.Adam(params, lr=1e-4, capturable=True, foreach=True)
    else:       # clip value 1 + clip norm 1 (flow parameters, trainer.py:165-166) + Adam in three fused launches
        opt = nf.FusedClipAdam(params, lr=1e-4, clip_params=list(flow.parameters()), clip_value=1.0, max_norm=1.0)
    dp = None
    if world > 1:
        dp = nf.GradAllReduce(flow, prior)
        dp.broadcast_parameters(src=0)
    x_static = x_host.to(dev)
    loss_host = torch.empty((), dtype=torch.float64).pin_memory()

    def step():
        opt.zero_grad(set_to_none=True)
        ld, lp = nf.initialize_with_zeros(2, B, dev)
        zs, ld, lp = flow.transform(x_static + torch.rand_like(x_static) / n_bins, ld, lp)
        lp += prior.compute_log_prob(zs[-1])
        loss = nf.calculate_loss(ld + lp, n_bins, n_pixel)
        loss.backward()
        if dp is not None:
            dp.finish()
        if args.torch_optimizer:
            torch.nn.utils.clip_grad_value_(list(flow.parameters()), 1.0)
            torch.nn.utils.clip_grad_norm_(list(flow.parameters()), 1.0)
        opt.step()
        return loss

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            loss0 = step()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    first_loss = float(loss0)
    graph, n_launch = None, None
    if not args.train_eager:
        try:
            graph = torch.cuda.CUDAGraph()
            l0 = N.launch_count
            with torch.cuda.graph(graph):
                loss_static = step()
            n_launch = N.launch_count - l0
        except Exception as e:                      # pragma: no cover - reported, eager numbers follow
            graph = None
            if rank == 0:
                print(f"# train-step graph capture failed ({type(e).__name__}: {e}); timing eagerly", file=sys.stderr)
            torch.cuda.synchronize()
    if graph is not None:
        def run_dev():
            graph.replay()
            return loss_static

        def run_e2e():
            x_static.copy_(x_host, non_blocking=True)
            graph.replay()
            loss_host.copy_(loss_static, non_blocking=True)
    else:
        def run_dev():
            return step()

        def run_e2e():
            x_static.copy_(x_host, non_blocking=True)
            loss_host.copy_(step().detach(), non_blocking=True)
    for _ in range(max(args.warmup, 3)):
        run_dev()
    torch.cuda.synchronize()
    steps = args.steps
    l0 = N.launch_count
    ms = timed(run_dev, steps)
    launches = (n_launch * steps) if graph is not None else (N.launch_count - l0)
    ms_e2e = timed(run_e2e, steps)
    torch.cuda.synchronize()
    last_loss = float(loss_host)
    # HBM roofline of the fused optimiser step (3 launches): 4 fp32 reads + 4 writes per parameter element
    opt_roof = None
    if not args.torch_optimizer:
        hbm = peaks()[0]
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(10)]
        for s_, e_ in evs:
            flush_buf.zero_()
            s_.record()
            opt.step()
            e_.record()
        torch.cuda.synchronize()
        o_ms = sorted(s_.elapsed_time(e_) for s_, e_ in evs)[len(evs) // 2]
        n_el = sum(p.numel() for p in params)
        gbs = 32.0 * n_el / (o_ms * 1e-3) / 1e9
        opt_roof = {"bound": "hbm", "kernel": "opt_clip_sumsq + opt_finalize + opt_adam (FusedClipAdam.step)",
                    "achieved": gbs, "peak": hbm, "unit": "GB/s", "frac": gbs / hbm, "ms": o_ms,
                    "bytes_per_launch": 32.0 * n_el}
    imgs = B * world * steps
    # exposed communication: the same captured step with the collectives skipped (every rank does so: no mismatch), timed
    # the same way; the difference is what the all-reduce adds to the step after overlap
    exposed = None
    if dp is not None and graph is not None:
        dp.enabled = False
        try:
            g2 = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g2):
                step()
            for _ in range(3):
                g2.replay()
            ms_nc = timed(lambda: g2.replay(), steps)
            exposed = (ms - ms_nc) / steps * 1e3
        finally:
            dp.enabled = True
    return {"metric": "Glow L3/K16 32x32 full train step imgs/sec (fwd + bwd + clip + Adam)", "value": imgs / (ms * 1e-3),
            "unit": "img/s", "ms_per_step": ms / steps, "dtype": "bf16 coupling GEMMs (tcgen05), fp32 elsewhere",
            "e2e": {"value": imgs / (ms_e2e * 1e-3), "unit": "img/s", "ms_per_step": ms_e2e / steps,
                    "h2d_bytes_per_step": x_host.numel() * 4, "d2h_bytes_per_step": 8},
            "gpu_launches": launches, "cuda_graph": graph is not None,
            "optimizer": "torch clip_grad_value_/clip_grad_norm_/Adam(foreach)" if args.torch_optimizer else
                         "FusedClipAdam (clip value + clip norm + Adam, 3 launches)",
            "grad_allreduce": dp.describe() if dp is not None else None,
            "exposed_comm_us_per_step": exposed,
            "step_tflops": 3 * FLOP_PER_IMG_FWD * B / (ms / steps * 1e-3) / 1e12,
            "optimizer_roofline": opt_roof, "loss_first": first_loss, "loss_last": last_loss}


def graph_time(torch, fn, reps=16, replays=10):
    """us per call of fn the way the product runs it: `reps` back-to-back launches per CUDA-graph replay (no launch
    gaps, operands L2-resident), CUDA events around `replays` replays on the launching stream."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            fn()
        side.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for _ in range(reps):
                fn()
        g.replay()
        side.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(replays):
            g.replay()
        e.record()
        side.synchronize()
    torch.cuda.current_stream().wait_stream(side)
    return s.elapsed_time(e) * 1e3 / (reps * replays)


def ncu_traffic(kernel_key: str):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu --set full summary of THIS round
    (profiles/r02_ncu_traffic.json, written by tools/summarise_ncu.py), or None."""
    path = os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")
    try:
        d = json.load(open(path))
        return d.get(kernel_key)
    except Exception:
        return None


DUMP_LIMIT = 64 * 1024 * 1024


def dump_outputs(path: str, arrays: dict) -> None:
    """--dump-outputs: each tensor (batch-major) -> path/<name>.npy on the host.  Above DUMP_LIMIT bytes in all, the first
    n images of every array are written, n the most that fit (the inputs are seeded, so that sample is fixed)."""
    import numpy as np
    host = {k: v.detach().cpu().numpy() for k, v in arrays.items()}
    for k, a in host.items():
        assert a.dtype in (np.float32, np.float64), (k, a.dtype)
    B = next(iter(host.values())).shape[0]
    per_image = sum(a.nbytes for a in host.values()) // B
    n = min(B, DUMP_LIMIT // per_image)
    os.makedirs(path, exist_ok=True)
    for k, a in host.items():
        np.save(os.path.join(path, k + ".npy"), a[:n])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-gpu"])
    ap.add_argument("--batch", type=int, default=CFG["batch"])
    ap.add_argument("--time-budget", type=float, default=150.0, help="reference arms: seconds of steps at most")
    ap.add_argument("--tf32", type=int, default=None, help="reference-gpu arm: force cuDNN allow_tf32 (default: torch's)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager-gpu", action="store_true", help="skip the torch-eager-on-GPU reference comparator")
    ap.add_argument("--no-train", action="store_true", help="skip the full-train-step measurement")
    ap.add_argument("--only-train", action="store_true", help="development: print only the training record")
    ap.add_argument("--train-eager", action="store_true", help="do not capture the train step in a CUDA graph")
    ap.add_argument("--torch-optimizer", action="store_true",
                    help="train arm: torch clip_grad_value_/clip_grad_norm_/Adam instead of the fused optimiser step")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the headline path returned in its last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.only_train):
        ap.error("--dump-outputs records the headline path: it needs --impl ours and no --only-train")
    if args.impl == "reference":
        return run_reference(args, on_gpu=False)
    if args.impl == "reference-gpu":
        return run_reference(args, on_gpu=True)
    args.warmup = max(args.warmup, 3)
    for p in (ROOT, PKG):
        if p not in sys.path:
            sys.path.insert(0, p)

    import torch
    import torch.distributed as dist
    import normalizing_flow as nf
    from normalizing_flow import _native as N, _engine as E
    import synthetic as SY            # synthetic inputs; the oracle is imported only as the checker of `checks`

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    c, L, K, S, B = CFG["in_channel"], CFG["L"], CFG["K"], CFG["S"], args.batch
    head_mode = E.precision()                       # "auto" unless the caller exported NFDPM_PRECISION
    head_infer = "bf16" if head_mode == "bf16" else ("fp32_simt" if head_mode == "fp32_simt" else "fp32")

    # random-init weights of the named architecture (SURVEY §8(d) recipe), synthetic dequantised images
    state = reference_style_state(nf, torch, dev, SY.seeded_input((CFG["batch"], c, S, S), 1))
    sd, psd = state
    flow = nf.Glow(c, L, K).to(dev)
    flow.load_state_dict(sd)
    prior = nf.GaussianPrior(2 ** (L + 1) * c).to(dev)
    prior.load_state_dict(psd)
    x_host = SY.seeded_input((B, c, S, S), 1 + rank).pin_memory()
    x_dev = x_host.to(dev)
    ll_host = torch.empty(B, dtype=torch.float64).pin_memory()
    xr_host = torch.empty(B, c, S, S).pin_memory()
    flush_buf = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)   # > 126 MB L2

    def fwd_dev(x):
        ld, lp = nf.initialize_with_zeros(2, B, dev)
        zs, ld, lp = flow.transform(x, ld, lp)
        lp += prior.compute_log_prob(zs[-1])
        return zs, ld + lp

    def step_dev():
        zs, ll = fwd_dev(x_dev)
        return ll, flow.invert(zs), zs

    def step_e2e():
        xd = x_host.to(dev, non_blocking=True)
        zs, ll = fwd_dev(xd)
        xr = flow.invert(zs)
        ll_host.copy_(ll, non_blocking=True)
        xr_host.copy_(xr, non_blocking=True)

    def timed(fn, steps):
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        for s, e in ev:
            flush_buf.zero_()                      # evict L2 between timed iterations (not timed)
            s.record()
            fn()
            e.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        tot = sum(s.elapsed_time(e) for s, e in ev)          # ms
        t = torch.tensor([tot], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def rate(ms_total, steps):
        return B * world * steps / (ms_total * 1e-3)

    def oracle_checks(n_img=8):
        """This mode's CUDA path against the CPU oracle on the first n_img images of the batch (the oracle is the checker
        here, never the thing measured)."""
        from oracle import glow_oracle as O
        xs = x_host[:n_img].clone()
        ld = torch.zeros(n_img, dtype=torch.float64)
        lp = torch.zeros(n_img, dtype=torch.float64)
        zo, ld, lp = O.glow_transform(sd, xs, L, K, ld, lp)
        ll_o = ld + lp + O.gaussian_prior_logp(psd, zo[-1])
        xo = O.glow_invert(sd, zo, L, K)
        zs, ll = fwd_dev(x_dev)
        xr_from_oracle_z = flow.invert([torch.cat([z, z.new_zeros(B - n_img, *z.shape[1:])]).to(dev) for z in zo])[:n_img].cpu()
        n_px = S * S * 3.0
        zg = torch.cat([z[:n_img].reshape(n_img, -1).cpu() for z in zs], 1).double()
        zr = torch.cat([z.reshape(n_img, -1) for z in zo], 1).double()
        bpd_g = float(nf.calculate_loss(ll[:n_img].cpu(), 32.0, n_px))
        bpd_o = float(nf.calculate_loss(ll_o, 32.0, n_px))
        return {"images": n_img,
                "z_rel_l2_vs_oracle": float((zg - zr).norm() / zr.norm()),
                "loglik_rel_err_vs_oracle": float(((ll[:n_img].cpu() - ll_o).abs() / ll_o.abs()).max()),
                "bits_per_dim": bpd_g, "bits_per_dim_abs_err_vs_oracle": abs(bpd_g - bpd_o),
                "inverse_max_abs_err_vs_oracle": float((xr_from_oracle_z - xo).abs().max()),
                "oracle_own_recon_max_abs_err": float((xo - xs).abs().max())}

    def measure_mode(mode, full):
        """All device-timed numbers of one precision mode (the graphs are keyed on the mode string)."""
        prev = os.environ.get("NFDPM_PRECISION")
        os.environ["NFDPM_PRECISION"] = mode
        try:
            for _ in range(args.warmup):
                step_dev()
                step_e2e()
            torch.cuda.synchronize()
            l0 = N.launch_count
            last = {}

            def step_kept():
                last["out"] = step_dev()
            ms = timed(step_kept if full and args.dump_outputs else step_dev, args.steps)
            launches = N.launch_count - l0
            if rank == 0 and "out" in last:
                ll, xr, zs = last.pop("out")
                dump_outputs(args.dump_outputs, {"log_likelihood": ll, "x_reconstructed": xr,
                                                 **{f"z{i}": z for i, z in enumerate(zs)}})
            ms_e2e = timed(step_e2e, args.steps)
            zs, _ = fwd_dev(x_dev)
            flow.invert(zs)
            ms_f = timed(lambda: fwd_dev(x_dev), args.steps)
            ms_i = timed(lambda: flow.invert(zs), args.steps)
            out = {"dtype": DTYPE_NAME[mode], "value": rate(ms, args.steps), "unit": "img/s", "ms_per_step": ms / args.steps,
                   "e2e": {"value": rate(ms_e2e, args.steps), "unit": "img/s", "ms_per_step": ms_e2e / args.steps},
                   "gpu_launches": launches,
                   "forward": {"value": rate(ms_f, args.steps), "unit": "img/s", "ms": ms_f / args.steps},
                   "inverse": {"value": rate(ms_i, args.steps), "unit": "img/s", "ms": ms_i / args.steps},
                   "step_tflops_algorithmic": 2 * FLOP_PER_IMG_FWD * B / (ms / args.steps * 1e-3) / 1e12}
            if full:
                for _ in range(3):
                    flow.invert([zs[-1]])
                ms_s = timed(lambda: flow.invert([zs[-1]]), args.steps)
                out["sample_last_latent"] = {"value": rate(ms_s, args.steps), "unit": "img/s", "ms": ms_s / args.steps,
                                             "what": "Glow.invert([z_last]): every Split draws its half from the learned "
                                                     "conditional prior (glow.py:203-246), T=1"}
            ll, xr, _ = step_dev()
            torch.cuda.synchronize()
            out["checks"] = {"recon_max_abs_err": float((xr - x_dev).abs().max())}
            if rank == 0 and not args.no_cpu_baseline:
                out["checks"].update(oracle_checks())
            return out
        finally:
            if prev is None:
                os.environ.pop("NFDPM_PRECISION", None)
            else:
                os.environ["NFDPM_PRECISION"] = prev

    hbm, tf_burst, tf_sust, src = peaks()
    if args.only_train:                             # development switch: just the training record
        train = bench_train(args, torch, dist, nf, N, dev, world, rank, B, x_host, timed, flush_buf, state)
        if rank == 0:
            print(json.dumps({"only_train": True, "n_gpus": world, "train": train}))
        if world > 1:
            dist.destroy_process_group()
        return
    with torch.no_grad():
        sampler = ClockSampler(local) if rank == 0 else None
        t_wall0 = time.time()
        head = measure_mode(head_infer, True)
        t_wall1 = time.time()
        clocks = sampler.stop(t_wall0, t_wall1) if sampler else None
        modes = {head_infer: head}
        if head_infer != "bf16":
            modes["bf16"] = measure_mode("bf16", False)

        # ---- roofline of the dominant kernel: coupling-net conv2 (512x512) GEMM at level 0, M = B*256
        M, F = B * (S // 2) * (S // 2), 512
        es, eb = torch.zeros(F, device=dev), torch.zeros(F, device=dev)

        def operand(rows, cols, scale, dt):
            v = torch.randn(rows, cols, device=dev) * scale
            if dt != N.SPLIT:
                return v.to(dt)
            hi = v.bfloat16()
            lo = (v - hi.float()).bfloat16()
            w = torch.stack([hi.reshape(rows, cols // 32, 32), lo.reshape(rows, cols // 32, 32)], dim=2).contiguous()
            return w.view(torch.int32).reshape(rows, cols)

        def gemm_roofline(dt):
            a, w = operand(M, F, 0.5, dt), operand(F, F, 0.05, dt)
            d = torch.empty(M, F, dtype=dt, device=dev)
            call = lambda: N.gemm_nt(a, F, w, F, d, F, M, F, F, N.EPI_ACTNORM_RELU, es, eb)
            us = graph_time(torch, call)
            for _ in range(3):
                call()
            evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(10)]
            for s_, e_ in evs:
                flush_buf.zero_()
                s_.record()
                call()
                e_.record()
            torch.cuda.synchronize()
            cold_us = sum(s_.elapsed_time(e_) for s_, e_ in evs) / len(evs) * 1e3
            mmas = 3 if dt == N.SPLIT else 1
            alg = 2.0 * M * F * F
            tf = alg / (us * 1e-6) / 1e12
            name = {torch.bfloat16: "gemm_nt_tc_kernel<ACTNORM_RELU, bf16, X3=false> (tcgen05, bf16 operands)",
                    N.SPLIT: "gemm_nt_tc_kernel<ACTNORM_RELU, bf16x2, X3=true> (tcgen05, split bf16 pairs, 3 MMAs per product)",
                    torch.float32: "gemm_nt_f32_kernel (CUDA cores)"}[dt]
            key = {torch.bfloat16: "gemm_nt_tc_bf16", N.SPLIT: "gemm_nt_tc_x3", torch.float32: "gemm_nt_f32"}[dt]
            tr = ncu_traffic(key)
            return {"bound": "tensor", "kernel": f"{name} M={M} N=512 K=512", "achieved": tf, "peak": tf_burst / mmas,
                    "unit": "TFLOP/s", "frac": tf / (tf_burst / mmas), "kernel_us": us, "launches_timed": 160,
                    "flop_per_launch_algorithmic": alg, "mma_flop_issued_per_launch": alg * mmas,
                    "issued_tflops": tf * mmas,
                    "peak_source": f"{src} bf16 burst ({tf_burst:.1f} TFLOP/s)" + (" / 3 MMAs per product" if mmas == 3 else ""),
                    "how": "16 back-to-back launches per CUDA-graph replay (as the product runs them), CUDA events around "
                           "10 replays on the launching stream: a ~5 ms burst, hence the burst peak",
                    "isolated_cold": {"kernel_us": cold_us, "achieved": alg / (cold_us * 1e-6) / 1e12,
                                      "frac": alg / (cold_us * 1e-6) / 1e12 / (tf_burst / mmas),
                                      "note": "event pair around single launches, L2 flushed before each (includes the launch gap)"},
                    "traffic": tr.get("bytes") if tr else None, "traffic_source": tr.get("source") if tr else None}

        head_dt = {"fp32": N.SPLIT, "bf16": torch.bfloat16, "fp32_simt": torch.float32}[head_infer]
        roof = gemm_roofline(head_dt)
        roof_bf16 = gemm_roofline(torch.bfloat16) if head_dt != torch.bfloat16 else None
        # cuBLAS on the same shape, timed the same way: the bar for the kernel
        a16 = (torch.randn(M, F, device=dev) * 0.5).bfloat16()
        w16 = (torch.randn(F, F, device=dev) * 0.05).bfloat16()
        a32, w32 = a16.float(), w16.float()
        o16, o32 = torch.empty(M, F, dtype=torch.bfloat16, device=dev), torch.empty(M, F, device=dev)
        cublas = {"bf16_us": graph_time(torch, lambda: torch.matmul(a16, w16.t(), out=o16))}
        prev_tf32 = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = True
        cublas["tf32_us"] = graph_time(torch, lambda: torch.matmul(a32, w32.t(), out=o32))
        torch.backends.cuda.matmul.allow_tf32 = False
        cublas["fp32_us"] = graph_time(torch, lambda: torch.matmul(a32, w32.t(), out=o32))
        torch.backends.cuda.matmul.allow_tf32 = prev_tf32
        cublas["note"] = ("torch.matmul (cuBLASLt) on M=%d N=K=512, no epilogue, same 16-per-replay timing; tf32 has 2^-11 "
                          "operand rounding (not fp32-faithful), fp32 runs on CUDA cores" % M)
        roof["cublas_same_shape"] = cublas

        # ---- HBM roofline of the step-boundary kernels (ActNorm + 1x1 conv + affine coupling epilogue) at this batch
        def boundary_roofline():
            recs = []
            for lvl, (C, hw) in enumerate([(12, 16), (24, 8), (48, 4)]):
                P = hw * hw
                Mr = B * P
                K1p = (9 * (C // 2) + 63) // 64 * 64
                ldp = (9 * C + 15) // 16 * 16
                x = torch.randn(B, C, hw, hw, device=dev)
                pm = torch.randn(Mr, ldp, device=dev) * 0.05
                a1 = torch.empty(Mr, K1p, dtype=head_dt if head_dt != torch.float32 else torch.float32, device=dev)
                mt, beta = torch.randn(C, C, device=dev) * 0.3, torch.randn(C, device=dev)
                b3, l3 = torch.zeros(C, device=dev), torch.zeros(C, device=dev)
                part = torch.empty(B, device=dev)
                us = graph_time(torch, lambda: N.flow_boundary(x, C * P, False, pm, ldp, b3, l3, part, mt, beta, x, C * P, a1,
                                                               K1p, B, C, hw, hw, False))
                alg = 8.0 * C * P * B
                moved = alg + 4.0 * Mr * ldp + a1.element_size() * Mr * K1p
                recs.append({"level": lvl, "C": C, "P": P, "kernel_us": us, "algorithmic_bytes": alg,
                             "achieved": alg / (us * 1e-6) / 1e9, "frac": alg / (us * 1e-6) / 1e9 / hbm,
                             "bytes_moved_incl_pm_and_im2col": moved, "moved_gbs": moved / (us * 1e-6) / 1e9})
            # the unfused K-A kernel (fused ActNorm + invertible 1x1 conv, north-star item 2) at a size beyond L2, where it IS
            # bandwidth-bound: x [8192, 12, 256] fp32 read once, y written once = 201 MB
            Bk, Ck, Pk = 8192, 12, 256
            xk = torch.randn(Bk, Ck, Pk, device=dev)
            yk = torch.empty_like(xk)
            mk, bk = torch.randn(Ck, Ck, device=dev) * 0.3, torch.randn(Ck, device=dev)
            for _ in range(3):
                N.channel_mix(xk, yk, mk, bk, Bk, Ck, Pk, Ck * Pk, Ck * Pk)
            evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(10)]
            for s_, e_ in evs:
                s_.record()
                N.channel_mix(xk, yk, mk, bk, Bk, Ck, Pk, Ck * Pk, Ck * Pk)
                e_.record()
            torch.cuda.synchronize()
            ka_us = sorted(s_.elapsed_time(e_) for s_, e_ in evs)[len(evs) // 2] * 1e3
            ka_bytes = 8.0 * Bk * Ck * Pk
            ka = {"kernel": "chanmix kernel (nfdpm_channel_mix: fused ActNorm + 1x1 conv, unfused form) on [8192,12,256] fp32",
                  "bytes_per_launch": ka_bytes, "kernel_us": ka_us, "achieved": ka_bytes / (ka_us * 1e-6) / 1e9,
                  "frac": ka_bytes / (ka_us * 1e-6) / 1e9 / hbm,
                  "note": "inputs larger than L2 (201 MB), timed alone with CUDA events; not on the default fused path at batch 128"}
            del xk, yk
            tr = ncu_traffic("flow_boundary_level1")
            top = recs[1]
            return {"bound": "hbm", "kernel": "flow_boundary_kernel<coupling, im2col sink> (levels 1-2 of the default path; "
                    "level 0 runs it fused into gemm3_boundary_kernel)", "achieved": top["achieved"], "peak": hbm,
                    "unit": "GB/s", "frac": top["frac"], "kernel_us": top["kernel_us"],
                    "algorithmic_bytes_per_launch": top["algorithmic_bytes"],
                    "what": "algorithmic bytes = read x + write y = 8*C*P per image per StepFlow (SURVEY 8d); the kernel also "
                            "reads the ZeroConv taps (36*C*P) and writes the next im2col rows; one CTA per image: "
                            "latency/issue-bound at batch 128, not bandwidth-bound",
                    "per_level": recs, "bandwidth_bound_size": ka, "peak_source": f"{src} copy bandwidth",
                    "traffic": tr.get("bytes") if tr else None, "traffic_source": tr.get("source") if tr else None}
        roof_hbm = boundary_roofline()

    train = None
    if not args.no_train:
        train = bench_train(args, torch, dist, nf, N, dev, world, rank, B, x_host, timed, flush_buf, state)
        if head_mode == "auto" and world == 1:
            # the same step with the fp32-faithful (split bf16 pair) operand format in the stash, dgrad and wgrad GEMMs
            os.environ["NFDPM_PRECISION"] = "fp32"
            try:
                t32 = bench_train(args, torch, dist, nf, N, dev, world, rank, B, x_host, timed, flush_buf, state)
            finally:
                os.environ.pop("NFDPM_PRECISION", None)
            t32["dtype"] = "bf16x3 coupling GEMMs (split bf16 pairs on tcgen05: forward, dgrad, wgrad), fp32 elsewhere"
            train["fp32_faithful_mode"] = {k: t32[k] for k in ("value", "unit", "ms_per_step", "dtype", "e2e", "gpu_launches",
                                                               "step_tflops", "loss_first", "loss_last")}

    if rank == 0:
        line = {
            "metric": METRIC, "value": head["value"], "unit": "img/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": head["dtype"], "data": "synthetic",
            "config": {"workload": WORKLOAD, "global_batch": B * world, "precision_mode": head_mode,
                       "parallelism": f"dp{world} (independent shards, no data-path collective)",
                       "l2": "flushed between timed steps (256 MiB memset)", "weights": WEIGHTS},
            "e2e": {"value": head["e2e"]["value"], "unit": "img/s", "h2d_bytes_per_step": x_host.numel() * 4,
                    "d2h_bytes_per_step": ll_host.numel() * 8 + xr_host.numel() * 4,
                    "ms_per_step": head["e2e"]["ms_per_step"]},
            "gpu_launches": head["gpu_launches"],
            "directions": {k: head[k] for k in ("forward", "inverse", "sample_last_latent") if k in head},
            "modes": modes,
            "roofline": roof, "roofline_bf16_mode": roof_bf16, "roofline_hbm": roof_hbm,
            "clocks": clocks,
            "checks": dict(head["checks"], step_tflops_algorithmic=head["step_tflops_algorithmic"]),
        }
        if train is not None:
            line["train"] = train
        if world == 1 and not args.no_cpu_baseline:
            # the unmodified reference on the host CPU: bounded sample (same batch, few steps), own process
            cpu = spawn_arm("reference", ["--batch", B, "--steps", 3, "--warmup", 1, "--time-budget", 25], 240)
            if "cpu_baseline" in cpu:
                line["cpu_baseline"] = cpu["cpu_baseline"]
                line["cpu_baseline"]["directions"] = cpu.get("directions")
            else:
                line["cpu_baseline"] = {"value": None, "unit": "img/s", "cores": os.cpu_count(), "kind": "reference",
                                        "sample": "unavailable: " + str(cpu.get("unavailable"))}
        if world == 1 and not args.no_eager_gpu:
            torch.cuda.empty_cache()
            g = spawn_arm("reference-gpu", ["--batch", B, "--steps", 10, "--warmup", 3, "--time-budget", 60], 300)
            g["speedup_of_this_repo_device_timed"] = (head["value"] / g["value"]) if g.get("value") else None
            line["gpu_eager_reference"] = g
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
