"""Training path of the Glow flow: forward with activation stash + hand-written backward kernel chain, exposed to
autograd as ONE ``torch.autograd.Function`` per ``Glow.transform`` call (and one per ``GaussianPrior.compute_log_prob``).

What autograd computes for the reference module (normalizing_flow/trainer.py:155-164 drives
glow.py:172-201 -> transforms.py:56-82, 116-133, 166-185, 270-290 and utils.py:43-44, 68-69) is reproduced by the
kernel sequence below; no torch arithmetic is involved (torch supplies memory, dtype casts of the incoming [B]
gradient vectors and the autograd plumbing).

Per StepFlow, backward order (k = K-1 .. 0), with M = B*P rows:
    coupling_bwd      dy, d(ld)            -> du (partial), dpm, d(bias3), d(logs3)
    dgrad3  (NT GEMM) dpm  x W3p           -> dh2           wgrad3 (TN GEMM) dpm^T h2  -> d(W3)
    actnorm_relu_bwd  dh2, h2              -> dpre2, d(scale2), d(bias2)
    wgrad2  (TN GEMM) dpre2^T h1 -> d(W2)  dgrad2 (NT GEMM) dpre2 x W2 -> dh1
    actnorm_relu_bwd  dh1, h1              -> dpre1, d(scale1), d(bias1)
    wgrad1  (TN GEMM) dpre1^T A1 -> d(W1)  dgrad1 (NT GEMM) dpre1 x W1 -> dA1
    mix_bwd           du + col2im(dA1), x  -> dx, per-image partials of d(W^), d(b^)
and per level one mix_param_grad launch folding those partials and the log-det terms P*sum(d ld)*W^-T, P*sum(d ld)
into d(InvConv2d.weight), d(ActNorm.scale), d(ActNorm.bias).
"""
from __future__ import annotations

import os
import weakref
from typing import Dict, List, Optional, Tuple

import torch
from torch import Tensor

from . import _engine as E
from . import _native as N

#: write parameter gradients straight into ``p.grad`` (views of one flat buffer) when it is empty; set to False to
#: hand every gradient to autograd instead (needed for torch.autograd.grad(), which must not touch ``.grad``)
DIRECT_GRADS = True
ROWS_PER_CTA = 64          # rows of one actnorm_relu_bwd CTA at large M (fewer at deep levels: >= ~256 CTAs)


def _f32(t: Optional[Tensor], B: int, dev) -> Tensor:
    """[B] gradient vector as contiguous fp32 (zeros when autograd passed None)."""
    if t is None:
        return torch.zeros(B, dtype=torch.float32, device=dev)
    return t.to(torch.float32).contiguous()


class _BwdCache:
    """Transposed (dgrad) copies of the three conv weights of one coupling network (filled by _engine.PackPlan):
    w1t[k, o] = W1[o, k] (rows K1..K1p zero), w2t[i, o] = W2[o, i], w3t[ci, tap*C+co] = W3[co, ci, tap]."""

    def __init__(self):
        self.key = None
        self.w1t = self.w2t = self.w3t = None
        self.Kp3 = 0


_SIDE = {}


def _side_stream(dev: torch.device) -> "torch.cuda.Stream":
    s = _SIDE.get(dev.index)
    if s is None:
        s = _SIDE[dev.index] = torch.cuda.Stream(device=dev)
    return s


class _LevelStash:
    __slots__ = ("C", "h", "w", "u", "x", "A1", "h1", "h2", "pm", "K1p", "ldp", "state_out")


class Stash:
    def __init__(self):
        self.levels: List[_LevelStash] = []
        self.B = 0
        self.with_logp = False
        self.in_shape = None
        self.dt = torch.bfloat16


def forward_train(glow, x: Tensor, with_logp: bool):
    """Glow.transform with every tensor the backward needs kept alive: per StepFlow the K-A input x_k, the K-A output
    u_k (= coupling input), the im2col rows A1_k, the hidden maps h1_k / h2_k and the taps-as-N rows pm_k."""
    B, c, H, W = x.shape
    dev = x.device
    glow._prepare_mix(dev)
    K = glow.K
    dt = E.coupling_dtype(train=True)
    glow._pack_plan(glow._steps(), dt, True).refresh()      # every forward / transposed weight layout in one launch
    st = Stash()
    st.B, st.with_logp, st.in_shape, st.dt = B, with_logp, (B, c, H, W), dt
    geo = glow._geometry(H, W)
    R_ld = sum(K * (1 if glow._level_fast(C, h, w) else N.ld_tiles(h * w)) for _, _, C, h, w in geo)
    R_lp = sum(N.ld_tiles(h * w) for _, split, _, h, w in geo if split is not None)
    ld_part = torch.empty(R_ld * B, dtype=torch.float32, device=dev)
    lp_part = torch.empty(max(R_lp, 1) * B, dtype=torch.float32, device=dev) if with_logp else None
    latents: List[Tensor] = []
    cur, cur_bs = x, c * H * W
    row = lrow = 0
    for flows, split, C, h, w in geo:
        P, M = h * w, B * h * w
        first = flows[0].affcoupling
        conv1 = first._parts()[0]
        F = conv1.weight.shape[0]
        K1p, ldp = first._cache.K1p, first._cache.ldp
        lv = _LevelStash()
        lv.C, lv.h, lv.w, lv.K1p, lv.ldp = C, h, w, K1p, ldp
        f32 = dict(dtype=torch.float32, device=dev)
        lv.u = torch.empty(K, B, C, P, **f32)
        lv.x = torch.empty(K, B, C, P, **f32)
        lv.A1 = torch.empty(K, M, K1p, dtype=dt, device=dev)
        lv.h1 = torch.empty(K, M, F, dtype=dt, device=dev)
        lv.h2 = torch.empty(K, M, F, dtype=dt, device=dev)
        lv.pm = torch.empty(K, M, ldp, **f32)
        lv.state_out = torch.empty(B, C, h, w, **f32)
        fused_g3 = E.fused_g3_ok(B, C, h, w, F, ldp, dt)
        fast = glow._level_fast(C, h, w)
        T_ld = 1 if fast else N.ld_tiles(P)
        if fast:
            # level entry: squeeze + stash x_0 + K-A of step 0 + im2col
            N.flow_boundary_stash(cur, cur_bs, True, None, 0, None, None, None, flows[0]._mix.fwd_mt,
                                  flows[0]._mix.fwd_beta, lv.u[0], C * P, lv.x[0], C * P, lv.A1[0], K1p, B, C, h, w)
        else:
            N.squeeze(cur, lv.x[0], B, C // 4, 2 * h, 2 * w, cur_bs, C * P)
        for k, step in enumerate(flows):
            cp = step.affcoupling
            conv1, an1, conv2, an2, zc = cp._parts()
            cache = cp._cache.at(dt)
            if not fast:      # images larger than one CTA: unfused K-A + im2col (any size)
                N.channel_mix(lv.x[k], lv.u[k], step._mix.fwd_mt, step._mix.fwd_beta, B, C, P, C * P, C * P)
                N.im2col3x3(lv.u[k], lv.A1[k], B, C // 2, h, w, C * P, K1p)
            N.gemm_nt(lv.A1[k], K1p, cache.w1, K1p, lv.h1[k], F, M, F, K1p, N.EPI_ACTNORM_RELU, an1.scale, an1.bias)
            w2 = cache.w2 if dt != torch.float32 else conv2.weight
            N.gemm_nt(lv.h1[k], F, w2, F, lv.h2[k], F, M, F, F, N.EPI_ACTNORM_RELU, an2.scale, an2.bias)
            nxt = flows[k + 1] if k + 1 < K else None
            mt, beta = (nxt._mix.fwd_mt, nxt._mix.fwd_beta) if nxt is not None else (None, None)
            y = lv.u[k + 1] if nxt is not None else lv.state_out
            xs = lv.x[k + 1] if nxt is not None else None
            a1n = lv.A1[k + 1] if nxt is not None else None
            if not fast:
                N.gemm_nt(lv.h2[k], F, cache.w3, F, lv.pm[k], ldp, M, ldp, F)
                N.coupling_apply(lv.pm[k], ldp, zc.bias, zc.logs, lv.u[k], xs if nxt is not None else lv.state_out,
                                 ld_part[row * B:], B, C, h, w, C * P, C * P, False)
            elif fused_g3:
                # ZeroConv GEMM + coupling + next mix + sinks in one kernel; pm is also written out for the backward
                N.gemm3_boundary(lv.h2[k], F, cache.w3, lv.pm[k], ldp, lv.u[k], C * P, zc.bias, zc.logs,
                                 ld_part[row * B:], mt, beta, y, C * P, xs, C * P if xs is not None else 0, a1n,
                                 K1p if a1n is not None else 0, B, C, h, w, F, ldp, False)
            else:
                N.gemm_nt(lv.h2[k], F, cache.w3, F, lv.pm[k], ldp, M, ldp, F)
                N.flow_boundary_stash(lv.u[k], C * P, False, lv.pm[k], ldp, zc.bias, zc.logs, ld_part[row * B:],
                                      mt, beta, y, C * P, xs, C * P if xs is not None else 0, a1n,
                                      K1p if a1n is not None else 0, B, C, h, w)
            row += T_ld
        st.levels.append(lv)
        if split is None:
            latents.append(lv.state_out)
            break
        z = torch.empty(B, C // 2, h, w, **f32)
        split._forward_views(lv.state_out, C * P, B, C, h, w, z, lp_part[lrow * B:] if lp_part is not None else None)
        lrow += N.ld_tiles(P)
        latents.append(z)
        cur, cur_bs = lv.state_out, C * P
    assert (row, lrow) == (R_ld, R_lp), f"wrote {row} / {lrow} partial rows, allotted {R_ld} / {R_lp}"
    return latents, ld_part, R_ld, lp_part, (R_lp if with_logp else 0), st


class GradSink:
    """Destination of every parameter gradient of one backward pass: ONE flat fp32 buffer in ``parameters()`` order
    (each tensor padded to 64 floats), so that the data-parallel all-reduce (normalizing_flow/_dp.py) and the
    optimizer work on contiguous memory and the backward kernels write their results in place (no per-parameter
    copies).  ``flat`` is allocated per backward: gradients of an earlier step that the caller still holds stay valid."""
    ALIGN = 64

    def __init__(self, params: List[Tensor]):
        self.offsets: Dict[int, Tuple[int, torch.Size]] = {}
        off = 0
        for p in params:
            self.offsets[id(p)] = (off, p.shape)
            off += (p.numel() + self.ALIGN - 1) // self.ALIGN * self.ALIGN
        self.numel = off
        dev = params[0].device
        self.flat = torch.empty(off, dtype=torch.float32, device=dev)
        self.written = set()

    def get(self, p: Tensor) -> Tensor:
        off, shape = self.offsets[id(p)]
        self.written.add(id(p))
        return self.flat[off:off + p.numel()].view(shape)

    def span(self, first: Tensor, last: Tensor) -> Tuple[int, int]:
        """[start, end) element range of the flat buffer from parameter ``first`` to the (padded) end of ``last``."""
        lo = self.offsets[id(first)][0]
        o, _ = self.offsets[id(last)]
        return lo, o + (last.numel() + self.ALIGN - 1) // self.ALIGN * self.ALIGN

    def level_ranges(self, glow) -> List[Tuple[int, int]]:
        """[start, end) element range of every level's parameters (levels are contiguous in parameters() order)."""
        out = []
        for blk in list(glow.blocks) + [glow.final_flows]:
            ps = list(blk.parameters())
            lo = self.offsets[id(ps[0])][0]
            o, shp = self.offsets[id(ps[-1])]
            hi = o + (ps[-1].numel() + self.ALIGN - 1) // self.ALIGN * self.ALIGN
            out.append((lo, hi))
        return out


def _strip_cols(src: Tensor, out: Tensor, rows: int, ld: int, cols: int) -> None:
    """[rows, ld] -> contiguous [rows, cols] (drops the GEMM padding columns)."""
    N.pack_matrix(src, out, rows, 1, cols, ld, 0, 1, cols, rows)


#: StepFlows per gradient bucket of the data-parallel all-reduce (``bucket_done``).  Measured at N = 2 on the config-2 step
#: (profiles/r02_dp_cta_sweep.txt): 2 / 4 / 8 / 16 StepFlows per bucket -> 9.16 / 9.01 / 8.88 / 8.70 ms per step (N = 1 on the
#: same box: 8.73 ms).  Finer buckets shorten the last, exposed all-reduce (22 MB -> 5.6 MB at 4) but every bucket costs a
#: parameter-gradient fold launch, stream events and an NCCL kernel that takes SMs from the persistent GEMM grids, which
#: outweighs it — so the default is one bucket per level (K = 16 and larger values mean "the whole level").
BUCKET_STEPS = int(os.environ.get("NFDPM_BUCKET_STEPS", "16"))


def backward_train(glow, st: Stash, d_lat: List[Optional[Tensor]], dld: Optional[Tensor], dlp: Optional[Tensor],
                   need_dx: bool, sink: GradSink, bucket_done=None) -> Optional[Tensor]:
    """Writes every parameter gradient into ``sink`` and returns d x (or None).  ``bucket_done(lo, hi, events)`` is called
    once every gradient in the flat-buffer range [lo, hi) has been enqueued — a group of BUCKET_STEPS consecutive
    StepFlows, in backward order (deepest level first, last StepFlow first; the range of a level's first bucket also
    holds its Split prior) — on the current stream or on the streams whose ``events`` are passed: the hook the
    data-parallel gradient all-reduce uses to overlap communication with the rest of the backward."""
    B = st.B
    levels = glow._levels()
    dev = st.levels[0].u.device
    dt = st.dt
    K = glow.K
    f32 = dict(dtype=torch.float32, device=dev)
    dld32 = _f32(dld, B, dev)
    dlp32 = _f32(dlp, B, dev) if st.with_logp else None
    dld_sum = torch.empty(1, **f32)
    N.reduce_rows(dld32, dld_sum, B, 1, 1)
    dx_next: Optional[Tensor] = None     # grad wrt the squeezed input of the level processed last
    for li in range(glow.L - 1, -1, -1):
        lv = st.levels[li]
        flows, split = levels[li]
        C, h, w = lv.C, lv.h, lv.w
        Ch, P, M = C // 2, h * w, B * h * w
        K1p, ldp = lv.K1p, lv.ldp
        F = lv.h1.shape[-1]
        # ---- gradient wrt the level's final state
        if split is None:
            g = d_lat[li]
            dy = g.to(torch.float32).contiguous() if g is not None else torch.zeros(B, C, h, w, **f32)
        else:
            dy = torch.empty(B, C, h, w, **f32)
            # first half <- squeeze backward of the next level's input gradient
            N.unsqueeze(dx_next, dy, B, 2 * C, h // 2, w // 2, 2 * C * (P // 4), C * P)
            second = dy.view(-1)[Ch * P:]
            g = d_lat[li]
            if g is not None:
                N.copy_channels(g.to(torch.float32).contiguous(), second, B, Ch, P, Ch * P, C * P)
            else:
                dy[:, Ch:].zero_()
            if st.with_logp:
                conv = split.conv
                if conv is None:
                    N.split_prior_bwd(dlp32, None, 0, None, None, lv.state_out, C * P, dy, C * P, None, None, B, C, h, w)
                else:
                    Ks, Kp, ldh = Ch * 9, E.round_up(Ch * 9, 16), E.round_up(C, 16)
                    wp = torch.empty(ldh * Kp, **f32)
                    N.pack_matrix(conv.weight, wp, 1, C, Ks, 0, Ks, 1, Kp, ldh)
                    wst = torch.empty(Kp * ldh, **f32)
                    N.pack_matrix(conv.weight, wst, Ks, 1, C, 1, 0, Ks, ldh, Kp)
                    As = torch.empty(M * Kp, **f32)
                    N.im2col3x3(lv.state_out, As, B, Ch, h, w, C * P, Kp)
                    hs = torch.empty(M * ldh, **f32)
                    N.gemm_nt(As, Kp, wp, Kp, hs, ldh, M, C, Kp)
                    dh = torch.empty(M * ldh, **f32)
                    dpar = torch.empty(B * 2 * C, **f32)
                    N.split_prior_bwd(dlp32, hs, ldh, conv.bias, conv.logs, lv.state_out, C * P, dy, C * P, dh, dpar,
                                      B, C, h, w)
                    N.reduce_rows2(dpar, sink.get(conv.bias), sink.get(conv.logs), B, C, C, 2 * C)
                    dws = torch.empty(C * Kp, **f32)
                    ws = torch.empty(N.gemm_tn_workspace(M, C, Kp), **f32)
                    N.gemm_tn(dh, ldh, As, Kp, dws, M, C, Kp, ws, fused_reduce=False)
                    _strip_cols(dws, sink.get(conv.weight), C, Kp, Ks)
                    dAs = torch.empty(M * Kp, **f32)
                    N.gemm_nt(dh, ldh, wst, ldh, dAs, Kp, M, Kp, ldh)
                    N.col2im_add(dAs, Kp, dy, C * P, B, Ch, h, w)
            elif split.conv is not None:
                for p_ in (split.conv.weight, split.conv.bias, split.conv.logs):
                    sink.get(p_).zero_()
        # ---- K StepFlows in reverse
        rows_cta = ROWS_PER_CTA
        while rows_cta > 8 and (M + rows_cta - 1) // rows_cta < 256:
            rows_cta //= 2
        n_cta = (M + rows_cta - 1) // rows_cta
        du = torch.empty(B, C, P, **f32)
        pong = (torch.empty(B, C, P, **f32), torch.empty(B, C, P, **f32))   # dx of successive steps alternate
        Kp3 = E.round_up(9 * C, 64)
        # dgrad GEMM output: bf16 in bf16 mode; fp32 in the fp32-faithful (split-pair) and CUDA-core modes
        dh = torch.empty(M * F, dtype=dt if dt == torch.bfloat16 else torch.float32, device=dev)
        tc = dt in E.TC_DTYPES               # tensor-core wgrad: in-kernel split reduction + direct weight layouts
        # The weight-gradient GEMMs feed only the optimiser: they run on a SIDE stream, concurrently with the
        # dgrad / elementwise chain of the same and the next StepFlow.  Their operands (dpm, dpre2, dpre1) are therefore
        # double-buffered across steps, and a buffer set is rewritten only after the side stream has read it.
        side = _side_stream(dev) if (tc and os.environ.get("NFDPM_WGRAD_STREAM", "1") != "0") else None
        main = torch.cuda.current_stream(dev)
        nbuf = 2 if side is not None else 1
        dpm_b = [torch.empty(M * Kp3, dtype=dt, device=dev) for _ in range(nbuf)]
        dpre2_b = [torch.empty(M * F, dtype=dt, device=dev) for _ in range(nbuf)]
        dpre1_b = [torch.empty(M * F, dtype=dt, device=dev) for _ in range(nbuf)]
        read_done = [None, None]
        dA1 = torch.empty(M * K1p, **f32)
        # ActNorm partial-sum buffers: one per (buffer set, layer) so their reductions can run on the side stream too
        an_part_b = [[torch.empty(n_cta * 2 * F, **f32) for _ in range(2)] for _ in range(nbuf)]
        keep = []                                  # scratch of the mix_param_grad launches (alive until the level is done)
        bucket = BUCKET_STEPS if bucket_done is not None else K      # without a data-parallel hook: one fold per level
        T_c, T_m = N.coupling_bwd_tiles(C, h, w), N.mix_bwd_tiles(C, h, w)     # pixel tiles per image (1: image per CTA)
        dpar3 = torch.empty(B * T_c * 2 * C, **f32)
        dp_scratch = torch.empty(M * C, **f32) if T_c > 1 else None
        mix_part = torch.empty(K, B * T_m * (C * C + C), **f32)
        d1 = torch.empty(F * K1p, **f32)
        d3 = torch.empty(ldp * F, **f32)
        ws = torch.empty(max(N.gemm_tn_workspace(M, F, F), N.gemm_tn_workspace(M, ldp, F),
                             N.gemm_tn_workspace(M, F, K1p)), **f32)

        ablate = int(os.environ.get("NFDPM_ABLATE", "0"))     # timing experiments only (results are wrong when set)

        def wgrad(fn):
            """Run a weight-gradient launch on the side stream once everything enqueued so far on main is done."""
            if ablate & 1:
                return
            if side is None:
                fn()
                return
            side.wait_stream(main)
            with torch.cuda.stream(side):
                fn()

        for k in range(K - 1, -1, -1):
            step = flows[k]
            sb = (K - 1 - k) % nbuf
            dpm, dpre, dpre1 = dpm_b[sb], dpre2_b[sb], dpre1_b[sb]
            an_part, an_part1 = an_part_b[sb]
            if side is not None and read_done[sb] is not None:
                main.wait_event(read_done[sb])          # the wgrads of two steps ago have read this buffer set
            cp = step.affcoupling
            conv1, an1, conv2, an2, zc = cp._parts()
            bc = cp._bwd_caches[dt]              # refreshed by the forward's PackPlan
            if ablate & 2:
                pass
            elif T_c == 1:
                N.coupling_bwd(dy, C * P, dld32, lv.u[k], C * P, lv.pm[k], ldp, zc.bias, zc.logs, du, C * P, dpm, Kp3,
                               dpar3, B, C, h, w, sink.get(zc.bias), sink.get(zc.logs))
            else:
                N.coupling_bwd(dy, C * P, dld32, lv.u[k], C * P, lv.pm[k], ldp, zc.bias, zc.logs, du, C * P, dpm, Kp3,
                               dpar3, B, C, h, w, dp_scratch=dp_scratch)
                N.reduce_rows2(dpar3, sink.get(zc.bias), sink.get(zc.logs), B * T_c, C, C, 2 * C)
            # ZeroConv 3x3: weight gradient in the taps-as-N layout, then back to [C, F, 3, 3]
            if tc:      # the split reduction writes d(W3) straight in its [C, F, 3, 3] layout
                wgrad(lambda: N.gemm_tn(dpm, Kp3, lv.h2[k], F, sink.get(zc.weight), M, ldp, F, ws,
                                        out_mode=N.TN_OUT_TAPS, out_c=C))
            else:
                N.gemm_tn(dpm, Kp3, lv.h2[k], F, d3, M, ldp, F, ws, fused_reduce=False)
                N.pack_matrix(d3, sink.get(zc.weight), C, F, 9, F, 1, C * F, 9, C * F)
            # second Conv2dActNorm (1x1).  (A dgrad GEMM with the ActNorm+ReLU backward fused into its epilogue was measured
            # in round 1 and was epilogue-bound: 32.9 / 40.7 us against 10.8+18.3 / 18.2+18.3 us for GEMM + elementwise
            # kernel at level 0, profiles/r01_levels_bwd_in_graph.txt; it left the library.)
            N.gemm_nt(dpm, Kp3, bc.w3t, Kp3, dh, F, M, F, Kp3)
            N.actnorm_relu_bwd(dh, F, lv.h2[k], F, an2.scale, dpre, F, an_part, M, F, rows_cta)
            n_red = n_cta

            def side2():
                N.reduce_rows2(an_part, sink.get(an2.scale), sink.get(an2.bias), n_red, F, F, 2 * F)
                N.gemm_tn(dpre, F, lv.h1[k], F, sink.get(conv2.weight), M, F, F, ws, fused_reduce=tc)
            wgrad(side2)
            # first Conv2dActNorm (3x3)
            N.gemm_nt(dpre, F, bc.w2t, F, dh, F, M, F, F)
            N.actnorm_relu_bwd(dh, F, lv.h1[k], F, an1.scale, dpre1, F, an_part1, M, F, rows_cta)

            def side1():
                N.reduce_rows2(an_part1, sink.get(an1.scale), sink.get(an1.bias), n_red, F, F, 2 * F)
                if tc:
                    N.gemm_tn(dpre1, F, lv.A1[k], K1p, sink.get(conv1.weight), M, F, K1p, ws, out_mode=N.TN_OUT_STRIP,
                              out_c=Ch * 9)
                else:
                    N.gemm_tn(dpre1, F, lv.A1[k], K1p, d1, M, F, K1p, ws, fused_reduce=False)
                    _strip_cols(d1, sink.get(conv1.weight), F, K1p, Ch * 9)
            wgrad(side1)
            if side is not None:
                ev = torch.cuda.Event()
                ev.record(side)
                read_done[sb] = ev
            N.gemm_nt(dpre1, F, bc.w1t, F, dA1, K1p, M, K1p, F)
            # fused ActNorm + 1x1 conv
            dxb = pong[k & 1]
            if not (ablate & 4):
                    N.mix_bwd(du, C * P, dA1, K1p, lv.x[k], C * P, step._mix.fwd_mt, dxb, C * P, mix_part[k], B, C, h, w)
            dy = dxb
            if k % bucket == 0:
                # a bucket of StepFlows [k, k_hi] is complete once their InvConv / ActNorm parameter gradients are folded
                # and their weight gradients have run (both on the side stream)
                k_hi = min(k + bucket, K) - 1
                items = []
                for kk in range(k, k_hi + 1):
                    stp = flows[kk]
                    wgt, sc, bi = stp.invconv2d.weight, stp.actnorm.scale, stp.actnorm.bias
                    scratch = torch.empty(C * C + C, **f32)
                    keep.append(scratch)
                    items.append(N.MixGradItem(part=mix_part[kk].data_ptr(), B=B * T_m, C=C, weight=wgt.data_ptr(),
                                               scale=sc.data_ptr(), bias=bi.data_ptr(), winv=stp._mix.winv.data_ptr(),
                                               dld_sum=dld_sum.data_ptr(), P=float(P), pad_=0,
                                               d_weight=sink.get(wgt).data_ptr(), d_scale=sink.get(sc).data_ptr(),
                                               d_bias=sink.get(bi).data_ptr(), scratch=scratch.data_ptr()))
                # (side stream: the fold feeds only the optimiser / the all-reduce, and one launch is ~50 us of latency)
                wgrad(lambda items=items: N.mix_param_grad(items))
                if bucket_done is not None:
                    first_p = next(flows[k].parameters())
                    last_mod = flows[k_hi] if (k_hi < K - 1 or split is None or split.conv is None) else split
                    last_p = list(last_mod.parameters())[-1]
                    lo_, hi_ = sink.span(first_p, last_p)
                    evs = []
                    if side is not None:
                        ev_b = torch.cuda.Event()
                        ev_b.record(side)
                        evs.append(ev_b)
                    bucket_done(lo_, hi_, evs)
        if side is not None:
            main.wait_stream(side)                # every weight gradient of the level is complete (buffers are reused)
        dx_next = dy
    dx = None
    if need_dx:
        Bc, c, H, W = st.in_shape
        lv = st.levels[0]
        dx = torch.empty(B, c, H, W, **f32)
        N.unsqueeze(dx_next, dx, B, lv.C, lv.h, lv.w, lv.C * lv.h * lv.w, c * H * W)
    return dx


# ------------------------------------------------------------------------------------------- captured training chains
# An UNCAPTURED training loop (the reference trainer as is) issues ~1 600 launches per step from Python and is host-bound
# (25.9 ms per 128-image step against 8.7 ms when the whole step sits in a torch.cuda.graph).  The autograd Function
# therefore captures its stash-forward chain and its backward chain once per (shape, precision) and replays them, like the
# inference entry points do: the reference trainer's unchanged step then takes 9.07 ms (bench.py --train-eager, round 2;
# profiles/r02_train_chains.txt).  Bit-identical to the eager chain over several optimiser steps
# (tests/test_gpu_train.py::test_captured_training_chains_equal_eager); the whole GPU suite passes with the chains on.
# NFDPM_TRAIN_GRAPHS=0 turns them off.  Not used under a caller's own capture or with the data-parallel hook (NCCL launches
# from inside the backward); parameter caches are refreshed INSIDE the chains (E.own_capture stays False), because the
# parameters change between replays.
def train_graphs_enabled() -> bool:
    return os.environ.get("NFDPM_TRAIN_GRAPHS", "1") != "0"


class _TrainChains:
    """Static buffers and graphs of one key.  ``busy`` marks a forward whose backward has not run yet: its stash lives in
    the graph's buffers, so a second forward before that backward (gradient accumulation over micro-batches in one
    autograd graph) takes the eager path instead of overwriting it."""

    def __init__(self):
        self.x = None
        self.fwd = None
        self.fwd_out = None
        self.n_fwd = 0
        self.bwd = {}
        self.owner = None             # weak reference to the autograd context whose stash is in the buffers
        self.epoch = -1
        self.scope = None

    @property
    def busy(self) -> bool:
        o = self.owner() if self.owner is not None else None
        return o is not None and getattr(o, "chains", None) is self

    def claim(self, ctx) -> None:
        try:
            self.owner = weakref.ref(ctx)
        except TypeError:             # context objects that cannot be weakly referenced: hold it until backward
            self.owner = lambda c=ctx: c

    def release(self) -> None:
        self.owner = None


def _train_chains(glow, x: Tensor, with_logp: bool) -> Optional["_TrainChains"]:
    if not train_graphs_enabled() or torch.cuda.is_current_stream_capturing() or \
            getattr(glow, "_grad_hook", None) is not None:
        return None
    store = glow.__dict__.setdefault("_train_chains", {})
    key = (tuple(x.shape), with_logp, E.precision(), x.device.index)
    tc = store.get(key)
    if tc is not None and tc.epoch != E.alloc_epoch:  # a cache was re-allocated: the captured addresses are stale
        E.WS.drop_scope(tc.scope + ("fwd",))
        for i in range(len(tc.bwd)):
            E.WS.drop_scope(tc.scope + ("bwd", i))
        tc = None
    if tc is None:
        tc = _TrainChains()
        tc.scope = ("train", id(glow), key)
        tc.x = torch.empty_like(x)
        tc.x.copy_(x)
        tc.fwd, tc.fwd_out, tc.n_fwd = E.capture(tc.scope + ("fwd",), lambda: forward_train(glow, tc.x, with_logp),
                                                 own=False)
        tc.epoch = E.alloc_epoch
        store[key] = tc
    return None if tc.busy else tc


def _bwd_chain(tc: "_TrainChains", glow, params, g_lat, g_ld, g_lp, need_dx: bool):
    """Static gradient inputs + captured backward of ``tc``'s stash for this pattern of present / absent gradients."""
    key = (tuple(None if g is None else (tuple(g.shape), g.dtype) for g in g_lat),
           None if g_ld is None else g_ld.dtype, None if g_lp is None else g_lp.dtype, need_dx)
    ent = tc.bwd.get(key)
    if ent is None:
        s_lat = [None if g is None else torch.empty_like(g) for g in g_lat]
        s_ld = None if g_ld is None else torch.empty_like(g_ld)
        s_lp = None if g_lp is None else torch.empty_like(g_lp)
        for s_, g in zip(s_lat + [s_ld, s_lp], list(g_lat) + [g_ld, g_lp]):
            if s_ is not None:
                s_.copy_(g)

        def build():
            sink = GradSink(params)
            dx = backward_train(glow, tc.fwd_out[5], s_lat, s_ld, s_lp, need_dx, sink, None)
            for p in params:                           # parameters the backward does not reach: exact zeros
                if p.requires_grad and id(p) not in sink.written:
                    sink.get(p).zero_()
            return sink, dx
        g, (sink, dx), n = E.capture(tc.scope + ("bwd", len(tc.bwd)), build, own=False)
        ent = tc.bwd[key] = dict(graph=g, sink=sink, dx=dx, n=n, lat=s_lat, ld=s_ld, lp=s_lp)
    return ent


class GlowTransformFn(torch.autograd.Function):
    """(x, log_det_jac, logp, *parameters) -> (log_det_jac, logp, *latents); both accumulators are updated in place
    like the reference (`+=`, transforms.py:81,131,184,288) and marked dirty."""

    @staticmethod
    def forward(ctx, glow, x, ld, lp, *params):
        with_logp = lp is not None
        H, W = x.shape[2:]
        tc = _train_chains(glow, x, with_logp)
        if tc is not None:
            tc.x.copy_(x)
            tc.fwd.replay()
            N.launch_count += tc.n_fwd
            latents, ld_part, R_ld, lp_part, R_lp, st = tc.fwd_out
            latents = [t.clone() for t in latents]      # the caller may keep latents across steps
            tc.claim(ctx)
        else:
            latents, ld_part, R_ld, lp_part, R_lp, st = forward_train(glow, x, with_logp)
        ctx.chains = tc
        glow._add_density(ld, lp, (ld_part, R_ld, lp_part, R_lp), H, W)
        ctx.mark_dirty(*([ld, lp] if with_logp else [ld]))
        ctx.glow, ctx.stash, ctx.with_logp = glow, st, with_logp
        ctx.params = params
        if with_logp:
            return (ld, lp) + tuple(latents)
        return (ld,) + tuple(latents)

    @staticmethod
    def backward(ctx, *gout):
        st = ctx.stash
        if st is None:
            raise RuntimeError("Glow.transform: backward called twice (the activation stash was released)")
        if ctx.with_logp:
            g_ld, g_lp, g_lat = gout[0], gout[1], list(gout[2:])
        else:
            g_ld, g_lp, g_lat = gout[0], None, list(gout[1:])
        glow, params = ctx.glow, list(ctx.params)
        tc = ctx.chains
        if tc is not None:
            ent = _bwd_chain(tc, glow, params, g_lat, g_ld, g_lp, ctx.needs_input_grad[1])
            for s_, g in zip(ent["lat"] + [ent["ld"], ent["lp"]], g_lat + [g_ld, g_lp]):
                if s_ is not None:
                    s_.copy_(g)
            sink = ent["sink"]
            # a .grad that still IS a view of this chain's flat buffer (zero_grad(set_to_none=False), or accumulation
            # over several backward calls) would be overwritten by the replay: keep its values and add them back
            aliased = {id(p) for p in params if p.grad is not None and p.requires_grad and
                       p.grad.data_ptr() == sink.flat.data_ptr() + 4 * sink.offsets[id(p)][0]}
            old = sink.flat.clone() if aliased else None
            ent["graph"].replay()
            N.launch_count += ent["n"]
            if old is not None:
                sink.flat.add_(old)
            dx = ent["dx"].clone() if ent["dx"] is not None else None
            tc.release()
            ctx.stash = None
            ctx.params = None
            ctx.chains = None
            glow._last_grad_flat = sink.flat
            pg = []
            for p in params:
                if not p.requires_grad:
                    pg.append(None)
                elif p.grad is None and DIRECT_GRADS:
                    p.grad = sink.get(p)
                    pg.append(None)
                elif id(p) in aliased:
                    pg.append(None)                        # already accumulated in place above
                else:
                    pg.append(sink.get(p).clone())         # autograd accumulates into a .grad held elsewhere
            return (None, dx, g_ld, g_lp) + tuple(pg)
        sink = GradSink(params)
        hook = getattr(glow, "_grad_hook", None)           # data-parallel all-reduce (normalizing_flow/_dp.py)
        if hook is not None:
            hook.begin(glow, sink)
        dx = backward_train(glow, st, g_lat, g_ld, g_lp, ctx.needs_input_grad[1], sink,
                            hook.bucket_done if hook is not None else None)
        ctx.stash = None
        ctx.params = None
        glow._last_grad_flat = sink.flat                   # contiguous view of all gradients of this step
        # Parameters whose .grad is empty receive their slice of the flat buffer DIRECTLY (no AccumulateGrad copy: 700+
        # small kernels per step otherwise); a parameter that already holds a gradient gets the usual accumulation.
        pg = []
        for p in params:
            if not p.requires_grad:
                pg.append(None)
                continue
            untouched = id(p) not in sink.written
            g = sink.get(p)
            if untouched:
                g.zero_()
            if p.grad is None and DIRECT_GRADS:
                p.grad = g
                pg.append(None)
            else:
                pg.append(g)
        del sink
        return (None, dx, g_ld, g_lp) + tuple(pg)


class GaussianPriorFn(torch.autograd.Function):
    """(z, weight, bias, logs) -> log p(z) [B] for the per-channel-constant prior (prior.py:79-83)."""

    @staticmethod
    def forward(ctx, z, weight, bias, logs):
        B, C, H, W = z.shape
        out = torch.empty(B, dtype=torch.float32, device=z.device)
        N.gauss_logp_const(z, bias, logs, out, B, C, H * W)
        ctx.save_for_backward(z, weight, bias, logs)
        return out

    @staticmethod
    def backward(ctx, g):
        z, weight, bias, logs = ctx.saved_tensors
        B, C, H, W = z.shape
        f32 = dict(dtype=torch.float32, device=z.device)
        g32 = g.to(torch.float32).contiguous()
        dz = torch.empty_like(z)
        if bias is None:
            N.gauss_const_bwd(g32, z, None, None, dz, None, B, C, H * W)
            return dz, None, None, None
        dpar = torch.empty(B * 4 * C, **f32)
        N.gauss_const_bwd(g32, z, bias, logs, dz, dpar, B, C, H * W)
        gp = torch.empty(4 * C, **f32)
        N.reduce_rows(dpar, gp, B, 4 * C, 4 * C)
        # the reference convolves an all-zero map: the weight receives an exactly-zero gradient
        return dz, torch.zeros_like(weight), gp[:2 * C].view_as(bias), gp[2 * C:].view_as(logs)
