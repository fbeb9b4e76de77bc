"""Wide levels (192 < C <= 1024 channels) at 256x256 L6 K32, B = 8 per GPU, fp32 and bf16: end-to-end times of the
forward (+ log-det + log-p), the decoding inverse, sampling and the training step; the in-graph time of each level's K
StepFlows (forward and inverse), so the wide final level's share is visible; and kernel times of the wide K-A, the wide
mix_bwd, the wide mix_inv_param_grad, mix_param_grad and mix_prepare at 384 and 768 channels.  Appends JSON lines to
profiles/r06_wide_levels.jsonl (OUT=... to redirect), each with the card's name and power limit read in the same run.

CUDA-event timing.  End-to-end: WARM calls, then ROUNDS rounds of STEPS calls, median round reported.  Kernels: REPS
back-to-back calls captured in one CUDA graph, replayed ITERS times (working sets of a few MB: L2-resident, as in the
model, where the previous kernel just wrote them)."""
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "normalizing-flow-with-diffusion-prior-model_b200"))
import torch

import normalizing_flow as nf
from normalizing_flow import _engine as E
from normalizing_flow import _native as N

DEV = torch.device("cuda")
OUT = os.environ.get("OUT", os.path.join(ROOT, "profiles", "r06_wide_levels.jsonl"))
c, L, K, S, B = 3, 6, int(os.environ.get("K", 32)), 256, int(os.environ.get("B", 8))
WARM, ROUNDS, STEPS = 3, 5, int(os.environ.get("STEPS", 5))
REPS, ITERS = 16, 20


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # pragma: no cover
        q = f"{torch.cuda.get_device_name()}, power limit unknown ({e})"
    return q


def timed(fn):
    """Median over ROUNDS rounds of STEPS calls, ms per call."""
    for _ in range(WARM):
        fn()
    torch.cuda.synchronize()
    rounds = []
    for _ in range(ROUNDS):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(STEPS):
            fn()
        e.record()
        torch.cuda.synchronize()
        rounds.append(s.elapsed_time(e) / STEPS)
    return round(statistics.median(rounds), 4), [round(r, 4) for r in rounds]


def graph_us(fn, reps=REPS, iters=ITERS):
    fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(reps):
            fn()
    g.replay()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(iters):
        g.replay()
    e.record()
    torch.cuda.synchronize()
    return round(s.elapsed_time(e) * 1e3 / (iters * reps), 2)


def own_graph_us(scope, fn, iters=10):
    """fn captured as the model captures its chains (E.capture, own=True: parameter caches stay outside the graph)."""
    g, _, _ = E.capture(scope, fn, own=True)
    g.replay()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(iters):
        g.replay()
    e.record()
    torch.cuda.synchronize()
    E.WS.drop_scope(scope)
    return round(s.elapsed_time(e) * 1e3 / iters, 2)


def event_us(fn, iters=10):
    """For host-driven sequences that are not captured (mix_prepare runs outside the model's graphs)."""
    fn()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(iters):
        fn()
    e.record()
    torch.cuda.synchronize()
    return round(s.elapsed_time(e) * 1e3 / iters, 2)


def model(prec):
    os.environ["NFDPM_PRECISION"] = prec
    torch.manual_seed(0)
    flow = nf.Glow(c, L, K).to(DEV)
    prior = nf.GaussianPrior(2 ** (L + 1) * c).to(DEV)
    x = torch.rand(B, c, S, S, device=DEV) - 0.5
    with torch.no_grad():
        flow.transform(x, *nf.initialize_with_zeros(2, B, DEV))      # data-dependent init
    return flow, prior, x


def end_to_end(prec, gpu):
    flow, prior, x = model(prec)
    ld, lp = nf.initialize_with_zeros(2, B, DEV)

    def fwd():
        with torch.no_grad():
            ld.zero_(); lp.zero_()
            zs, _, _ = flow.transform(x, ld, lp)
            lp.add_(prior.compute_log_prob(zs[-1]))
        return zs
    zs = fwd()
    zs = [z.clone() for z in zs]
    zl = [zs[-1].clone()]

    def inv():
        with torch.no_grad():
            flow.invert(zs)

    def smp():
        flow.sample(zl, temperature=0.7)
    opt = nf.FusedClipAdam(list(flow.parameters()) + list(prior.parameters()), lr=1e-6)

    def train():
        opt.zero_grad(set_to_none=False)
        l2, p2 = nf.initialize_with_zeros(2, B, DEV)
        z2, l2, p2 = flow.transform(x, l2, p2)
        p2 += prior.compute_log_prob(z2[-1])
        nf.calculate_loss(l2 + p2, 256.0, S * S * 3.0).backward()
        opt.step()
    rec = dict(kind="end_to_end", precision=prec, B=B, L=L, K=K, image=[c, S, S], gpu=gpu)
    for name, fn in (("forward_ld_lp_ms", fwd), ("invert_ms", inv), ("sample_ms", smp), ("train_step_ms", train)):
        rec[name], rec[name.replace("_ms", "_rounds")] = timed(fn)
    return rec, flow


def per_level(prec, flow, gpu):
    """Each level's K no-grad StepFlows (the kernels of its _level_mode) captured in one graph, forward and inverse, as
    Glow captures its chains: the LU/fold refresh runs outside."""
    os.environ["NFDPM_PRECISION"] = prec
    flow._prepare_mix(DEV)
    out = []
    for li, (flows, split, C, h, w) in enumerate(flow._geometry(S, S)):
        mode = flow._level_mode(B, C, h, w)
        src = torch.randn(B, C // 4, 2 * h, 2 * w, device=DEV) * 0.5
        st = torch.randn(B, C, h, w, device=DEV) * 0.5
        R = max(K * N.ld_tiles(h * w), K * N.flow_boundary_tiles(B, C, h, w, 1, 1, 1) + 1, K)
        ldp = torch.empty(R * B, device=DEV)
        slots = flow._slots(DEV)[li * K:(li + 1) * K]
        fwd = {"image": flow._transform_level_image, "tiled": flow._transform_level_tiled,
               "unfused": flow._transform_level_unfused}[mode]
        inv = {"image": flow._invert_level_image, "tiled": flow._invert_level_tiled,
               "unfused": flow._invert_level_unfused}[mode]
        f_us = own_graph_us(("wide-bench", li, "fwd"), lambda: fwd(flows, slots, src, (C // 4) * 4 * h * w, B, C, h, w,
                                                                    ldp, 0))
        i_us = own_graph_us(("wide-bench", li, "inv"), lambda: inv(flows, st, False, B, C, h, w, None, 0))
        out.append(dict(level=li, C=C, hw=[h, w], mode=mode, fwd_us=f_us, inv_us=i_us))
    tf, ti = sum(r["fwd_us"] for r in out), sum(r["inv_us"] for r in out)
    for r in out:
        r["fwd_share"], r["inv_share"] = round(r["fwd_us"] / tf, 4), round(r["inv_us"] / ti, 4)
    return dict(kind="per_level_in_graph", precision=prec, B=B, L=L, K=K, image=[c, S, S], levels=out, gpu=gpu)


def kernels(gpu):
    recs = []
    for C, hw in ((384, 4), (768, 2)):
        P = hw * hw
        q = torch.linalg.qr(torch.randn(C, C, dtype=torch.float64))[0].float()
        w = (q + 0.01 * torch.randn(C, C)).to(DEV)
        s, b = (0.1 * torch.randn(C)).to(DEV), (0.1 * torch.randn(C)).to(DEV)
        caches = [E.MixCache() for _ in range(K)]
        E.prepare_mix([(m, w, s, b, C, None) for m in caches])
        items = [N.MixItem(weight=w.data_ptr(), scale=s.data_ptr(), bias=b.data_ptr(), C=C, pad_=0,
                           fwd_mt=m.fwd_mt.data_ptr(), fwd_beta=m.fwd_beta.data_ptr(), inv_mt=m.inv_mt.data_ptr(),
                           inv_beta=m.inv_beta.data_ptr(), winv=m.winv.data_ptr(), logdet=m.logdet.data_ptr(),
                           lu_ws=m.lu_ws.data_ptr()) for m in caches]
        mix = caches[0]
        x = torch.randn(B, C, P, device=DEV)
        y = torch.empty_like(x)
        du = torch.randn(B, C, P, device=DEV)
        K1p = 9 * (C // 2)
        da1 = torch.randn(B * P, K1p, device=DEV)
        part = torch.empty(K, B * (C * C + C), device=DEV)
        dld = torch.ones(1, device=DEV)
        dW = torch.empty(K, C * C, device=DEV)
        dS, dB = torch.empty(K, C, device=DEV), torch.empty(K, C, device=DEV)
        scratch = torch.empty(K, C * C + C, device=DEV)
        N.mix_bwd(du, C * P, da1, K1p, x, C * P, mix.fwd_mt, y, C * P, part[0], B, C, hw, hw)
        for k in range(1, K):
            part[k].copy_(part[0])

        def gitem(k, inv=False):
            return N.MixGradItem(part=part[k].data_ptr(), B=B, C=C, weight=w.data_ptr(), scale=s.data_ptr(),
                                 bias=b.data_ptr(), winv=mix.winv.data_ptr(), dld_sum=dld.data_ptr(), P=float(P), pad_=0,
                                 d_weight=dW[k].data_ptr(), d_scale=dS[k].data_ptr(), d_bias=dB[k].data_ptr(),
                                 scratch=scratch[k].data_ptr())
        g16 = [gitem(k) for k in range(16)]
        rec = dict(kind="kernels", C=C, B=B, hw=[hw, hw], gpu=gpu,
                   wide_channel_mix_us=graph_us(lambda: N.channel_mix(x, y, mix.fwd_mt, mix.fwd_beta, B, C, P, C * P, C * P)),
                   wide_mix_bwd_da1_us=graph_us(lambda: N.mix_bwd(du, C * P, da1, K1p, x, C * P, mix.fwd_mt, y, C * P,
                                                                  part[0], B, C, hw, hw)),
                   wide_mix_inv_param_grad_us=graph_us(lambda: N.mix_inv_param_grad([gitem(0)])),
                   mix_param_grad_16_items_us=graph_us(lambda: N.mix_param_grad(g16), reps=2, iters=10),
                   mix_prepare_1_item_us=event_us(lambda: N.mix_prepare(items[:1])),
                   mix_prepare_K_items_us=event_us(lambda: N.mix_prepare(items)))
        recs.append(rec)
    return recs


def main():
    gpu = gpu_info()
    print("#", gpu, flush=True)
    os.makedirs(os.path.dirname(OUT), exist_ok=True)

    def emit(rec):
        print(json.dumps(rec), flush=True)
        with open(OUT, "a") as f:
            f.write(json.dumps(rec) + "\n")
    for k in kernels(gpu):
        emit(k)
    for prec in ("fp32", "bf16"):
        rec, flow = end_to_end(prec, gpu)
        emit(rec)
        emit(per_level(prec, flow, gpu))
        del flow
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
