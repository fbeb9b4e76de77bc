"""Composite flows StepFlow / GlowBlock / Glow with the reference's constructor signatures, attribute and
parameter names (reference normalizing_flow/glow.py:12-246), scheduled as one kernel chain per call:

    forward step   : [K-LU+fold, cached] -> K-A (ActNorm+1x1 conv, fused) -> im2col -> GEMM1 -> GEMM2 -> GEMM3
                     -> coupling epilogue (in place on the K-A output)
    inverse step   : im2col -> GEMM1 -> GEMM2 -> GEMM3 -> inverse coupling epilogue -> K-A^-1
    level boundary : squeeze reads the kept half in place (batch stride); Split writes z and the prior term
    whole call     : ONE accumulate kernel adds every per-step log-det partial and the K*L data-independent
                     constants H*W*(sum(scale) + log|det W|) into the caller's accumulator (in place)

``Glow.transform`` / ``Glow.invert`` never copy activations for chunk/concat: halves are addressed through batch
strides.
"""
import os
from typing import List, Optional, Tuple

import torch
import torch.nn as nn
from torch import Tensor

from . import _engine as E
from . import _native as N
from .base import Transform
from .transforms import ActNorm, AffineCoupling, InvConv2d, Split, Squeeze, _granular, _no_autograd
from .utils import get_item


class StepFlow(Transform):
    """ActNorm -> InvConv2d -> AffineCoupling (reference glow.py:21-63).  ActNorm and the 1x1 convolution run as
    ONE memory-bound kernel with pre-folded weights."""

    def __init__(self, in_channels: int = 3, coupling_net_n_features: int = 512):
        super().__init__()
        self.actnorm = ActNorm(in_channels=in_channels)
        self.invconv2d = InvConv2d(in_channels=in_channels)
        self.affcoupling = AffineCoupling(in_channels=in_channels, n_features=coupling_net_n_features)
        self._mix = E.MixCache()
        self._C = in_channels

    def _load_from_state_dict(self, *args, **kwargs):
        self._mix.invalidate()
        return super()._load_from_state_dict(*args, **kwargs)

    def _apply(self, fn, *a, **k):
        self._mix = E.MixCache()
        return super()._apply(fn, *a, **k)

    def _mix_entry(self, slot: Optional[Tensor] = None):
        return (self._mix, self.invconv2d.weight, self.actnorm.scale, self.actnorm.bias, self._C, slot)

    def _ready(self) -> bool:
        _, an1, _, an2, _ = self.affcoupling._parts()
        return self.actnorm._initialized() and an1._initialized() and an2._initialized()

    def _forward_views(self, x: Tensor, xbs: int, y: Tensor, ybs: int, B: int, H: int, W: int,
                       ld_part: Optional[Tensor], slot: Optional[Tensor] = None) -> None:
        C, P = self._C, H * W
        if not self.actnorm._initialized():
            self.actnorm._maybe_init(x, xbs, B, C, P)
            self._mix.invalidate()
        E.prepare_mix([self._mix_entry(slot)])
        N.channel_mix(x, y, self._mix.fwd_mt, self._mix.fwd_beta, B, C, P, xbs, ybs)
        self.affcoupling._run(y, ybs, y, ybs, B, C, H, W, False, ld_part)

    def _inverse_views(self, y: Tensor, ybs: int, t: Tensor, tbs: int, x: Tensor, xbs: int, B: int, H: int,
                       W: int, ld_part: Optional[Tensor] = None) -> None:
        """y --coupling^-1--> t (t may be y: in place) --K-A^-1--> x.  ``ld_part``: the coupling's log-det partials at x,
        the rows the forward writes."""
        C, P = self._C, H * W
        E.prepare_mix([self._mix_entry(None)])
        self.affcoupling._run(y, ybs, t, tbs, B, C, H, W, True, ld_part)
        N.channel_mix(t, x, self._mix.inv_mt, self._mix.inv_beta, B, C, P, tbs, xbs)

    def _transform_composed(self, x: Tensor, log_det_jac: Tensor, logp: Tensor) -> Tuple[Tensor, Tensor, Tensor]:
        """Under autograd a stand-alone StepFlow is the composition of its three differentiable parts, like the reference's
        (glow.py:46-48); the fused single-kernel form below serves the no-grad call."""
        y, log_det_jac, logp = self.actnorm.transform(x, log_det_jac, logp)
        y, log_det_jac, logp = self.invconv2d.transform(y, log_det_jac, logp)
        return self.affcoupling.transform(y, log_det_jac, logp)

    @_granular("StepFlow")
    def transform(self, x: Tensor, log_det_jac: Tensor, logp: Tensor) -> Tuple[Tensor, Tensor, Tensor]:
        x = E.check_input(x)
        B, C, H, W = x.shape
        if C != self._C:
            raise ValueError(f"StepFlow built for {self._C} channels got {C}")
        E.check_acc(log_det_jac, B, "log_det_jac")
        T = N.ld_tiles(H * W)
        part = E.WS.get("ldp1", T * B, torch.float32, x.device)
        y = torch.empty_like(x)
        self._forward_views(x, C * H * W, y, C * H * W, B, H, W, part)
        if log_det_jac is not None:
            N.accumulate(log_det_jac, part, T, B, self._mix.logdet, E.scalar_f32(x.device, H * W), 1)
        return y, log_det_jac, logp

    def _invert_composed(self, y: Tensor) -> Tensor:
        """Under autograd (NFDPM_INVERT_GRAD=1) the inverse is the composition of the three parts' inverses."""
        return self.actnorm.invert(self.invconv2d.invert(self.affcoupling.invert(y)))

    @_granular("StepFlow")
    def invert(self, y: Tensor) -> Tensor:
        y = E.check_input(y)
        B, C, H, W = y.shape
        t, x = torch.empty_like(y), torch.empty_like(y)
        self._inverse_views(y, C * H * W, t, C * H * W, x, C * H * W, B, H, W)
        return x


class GlowBlock(Transform):
    """Squeeze -> K StepFlows -> Split (reference glow.py:75-137)."""

    def __init__(self, in_channels: int = 3, K: int = 32, learn_prior_mean_logs: bool = True):
        super().__init__()
        flow_channels = 4 * in_channels
        self.squeeze = Squeeze()
        self.flows = nn.ModuleList([StepFlow(in_channels=flow_channels) for _ in range(K)])
        self.split = Split(flow_channels, learn_prior_mean_logs=learn_prior_mean_logs)

    def transform(self, x: Tensor, log_det_jac: Tensor, logp: Tensor) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
        y, log_det_jac, logp = self.squeeze.transform(x, log_det_jac, logp)
        for flow in self.flows:
            y, log_det_jac, logp = flow.transform(y, log_det_jac, logp)
        return self.split.transform(y, log_det_jac, logp)

    def invert(self, y: Tensor, latent: Tensor = None, temperature: float = 1.0) -> Tensor:
        inv = self.split.invert(y, latent, temperature=temperature)
        for flow in reversed(self.flows):
            inv = flow.invert(inv)
        return self.squeeze.invert(inv)


class Glow(Transform):
    """L-1 GlowBlocks, a final squeeze and K final StepFlows (reference glow.py:149-246)."""

    def __init__(self, in_channel: int = 3, L: int = 3, K: int = 32, learn_prior_mean_logs: bool = True):
        super().__init__()
        self.L, self.K, self.in_channel = L, K, in_channel
        self.blocks = nn.ModuleList(GlowBlock(in_channels=(2 ** i * in_channel), K=K,
                                              learn_prior_mean_logs=learn_prior_mean_logs) for i in range(L - 1))
        self.final_squeeze = Squeeze()
        self.final_flows = nn.ModuleList(StepFlow(in_channels=(2 ** (L + 1) * in_channel)) for _ in range(K))
        self._logdet_all: Optional[Tensor] = None
        self._cmul = {}
        self._graphs = {}
        self._plist = None
        self._pver = None
        self._plans = {}

    def _pack_plan(self, steps, dt, train: bool) -> "E.PackPlan":
        """The batched weight-packing job table for (dtype, train); built once, dropped when the module moves."""
        key = (dt, train)
        plan = self._plans.get(key)
        if plan is None or not plan.valid():
            plan = self._plans[key] = E.PackPlan(steps, dt, train)
        return plan

    def _apply(self, fn, *a, **k):
        self._plans = {}
        self.__dict__.pop("_train_chains", None)      # captured training chains hold the old parameter addresses
        self._logdet_all = None
        self._cmul = {}
        self._drop_graphs()
        self._plist = None
        return super()._apply(fn, *a, **k)

    def invalidate_caches(self) -> None:
        """Forget everything derived from the parameter VALUES (LU/fold matrices, packed weights, batched packing plans);
        the next call recomputes them.  Needed only after writes that bypass the tensors' version counters
        (``p.data.copy_(...)``, ``torch.Tensor.set_``): ordinary in-place updates, optimizer steps and
        ``load_state_dict`` are detected on their own."""
        for m in self.modules():
            if isinstance(m, StepFlow):
                m._mix.invalidate()
            elif isinstance(m, AffineCoupling):
                for ws in m._cache.sets.values():
                    ws.key = None
                for b in getattr(m, "_bwd_caches", {}).values():
                    b.key = None
            elif isinstance(m, Split):
                m._cache.key = None
        for plan in self._plans.values():
            plan.key = None
        self._pver = None

    def _load_from_state_dict(self, *args, **kwargs):
        # the coupling networks start new weight caches on load (transforms.py): the batched packing plans hold the OLD
        # cache objects and buffer addresses, so they are rebuilt too (found by the checkpoint-resume test: a model that
        # had already run, then loaded a checkpoint, packed into the orphaned buffers and launched with null operands)
        self._pver = None
        self._plans = {}
        return super()._load_from_state_dict(*args, **kwargs)

    # ---- CUDA graphs: the ~300-kernel chain of one call is captured once per (direction, shape, precision) and
    # replayed; only the parameter-version check and the final accumulate into the caller's tensors stay outside.
    def _drop_graphs(self) -> None:
        for key in list(self._graphs):
            E.WS.drop_scope(("glow", id(self), key))
        self._graphs = {}

    def _params_changed(self) -> bool:
        if self._plist is None:
            self._plist = list(self.parameters())
            self._pver = None
        ver = [p._version for p in self._plist]
        if ver != self._pver:
            self._pver = ver
            return True
        return False

    def _refresh_caches(self, steps, slots) -> None:
        """Re-run LU/fold and weight packing for parameters that changed (outside any graph)."""
        E.prepare_mix([s._mix_entry(slots[i:i + 1]) for i, s in enumerate(steps)])
        self._pack_plan(steps, E.coupling_dtype(), False).refresh()
        for blk in self.blocks:
            E.refresh_split(blk.split, blk.flows[0]._C)

    def _use_graph(self, ready: bool) -> bool:
        return ready and E.graphs_enabled() and not torch.cuda.is_current_stream_capturing()

    def _graph_entry(self, key, build):
        """build() -> dict of static tensors; called once eagerly (warm-up) and once under capture."""
        ent = self._graphs.get(key)
        if ent is not None and ent["epoch"] == E.alloc_epoch:
            return ent
        scope = ("glow", id(self), key)
        E.WS.drop_scope(scope)
        prev = E.WS.scope
        try:
            E.WS.scope = ("warm", id(self))
            build()                                   # eager warm-up: parameter caches, one-time kernel attributes
            torch.cuda.current_stream().synchronize()
            E.WS.drop_scope(("warm", id(self)))
            E.WS.scope = scope                        # buffers baked into the graph live (only) under this scope
            g = torch.cuda.CUDAGraph()
            n0 = N.launch_count
            E.own_capture = True                      # parameter caches were refreshed above, outside the graph
            with torch.cuda.graph(g):
                out = build()
            n_launch = N.launch_count - n0
        finally:
            E.own_capture = False
            E.WS.scope = prev
        N.launch_count -= n_launch                    # counted per replay instead
        ent = dict(out)
        ent["graph"], ent["epoch"], ent["n_launch"] = g, E.alloc_epoch, n_launch
        self._graphs[key] = ent
        return ent

    # ---- helpers
    def _levels(self) -> List[Tuple[nn.ModuleList, Optional[Split]]]:
        lv = [(blk.flows, blk.split) for blk in self.blocks]
        lv.append((self.final_flows, None))
        return lv

    def _slots(self, device: torch.device) -> Tensor:
        n = self.L * self.K
        if self._logdet_all is None or self._logdet_all.device != device:
            self._logdet_all = torch.zeros(n, dtype=torch.float32, device=device)
        return self._logdet_all

    def _multipliers(self, H: int, W: int, device: torch.device) -> Tensor:
        key = (H, W, device.index)
        t = self._cmul.get(key)
        if t is None:
            vals = []
            h, w = H, W
            for _ in range(self.L):
                h, w = h // 2, w // 2
                vals += [float(h * w)] * self.K
            t = torch.tensor(vals, dtype=torch.float32, device=device)
            self._cmul[key] = t
        return t

    def _check_image(self, x: Tensor) -> Tuple[int, int, int, int]:
        B, C, H, W = x.shape
        if C != self.in_channel:
            raise ValueError(f"Glow built for {self.in_channel} input channels got {C}")
        if H % (2 ** self.L) or W % (2 ** self.L):
            raise ValueError(f"input {H}x{W} is not divisible by 2^L = {2 ** self.L}")
        return B, C, H, W

    # ---- forward: x -> ([z_0..z_{L-1}], log_det_jac, logp)
    def transform(self, x: Tensor, log_det_jac: Tensor, logp: Tensor) -> Tuple[list, Tensor, Tensor]:
        x = E.check_input(x)
        B, c, H, W = self._check_image(x)
        if log_det_jac is None:
            raise ValueError("log_det_jac accumulator is required")
        E.check_acc(log_det_jac, B, "log_det_jac")
        E.check_acc(logp, B, "logp")
        dev = x.device
        levels = self._levels()
        slots = self._slots(dev)
        steps = [s for flows, _ in levels for s in flows]
        ready = all(s._ready() for s in steps)
        if E.autograd_needed(x, self):
            return self._transform_autograd(x, log_det_jac, logp, levels, slots, steps, ready)
        if self._use_graph(ready):
            if self._params_changed():
                self._refresh_caches(steps, slots)
            key = ("fwd", B, H, W, logp is not None, E.precision(), dev.index)
            x_static = self._graphs.get(key, {}).get("x")
            if x_static is None:
                x_static = torch.empty_like(x)
            x_static.copy_(x)

            nsub = self._n_sub(B)
            Bs = B // nsub

            def build():
                # images are independent: sub-batches run on concurrent streams inside the graph, so that the deep
                # levels (few rows per kernel, < 148 CTAs) of one sub-batch overlap with kernels of the other
                parts = self._fork_join(nsub, lambda i: self._transform_core(
                    x_static[i * Bs:(i + 1) * Bs], logp is not None, levels, slots, steps, True))
                return {"x": x_static, "parts": parts}
            ent = self._graph_entry(key, build)
            if ent["x"] is not x_static:              # entry was (re)built around another buffer
                ent["x"].copy_(x)
            ent["graph"].replay()
            N.launch_count += ent["n_launch"]
            parts = ent["parts"]
            latents = [torch.cat([p[0][j] for p in parts]) if nsub > 1 else parts[0][0][j].clone()
                       for j in range(len(parts[0][0]))]
            cm = self._multipliers(H, W, dev)
            for i, (_, ld_part, R_ld, lp_part, R_lp) in enumerate(parts):
                N.accumulate(log_det_jac[i * Bs:(i + 1) * Bs], ld_part, R_ld, Bs, slots, cm, self.L * self.K)
                if logp is not None and R_lp > 0:
                    N.accumulate(logp[i * Bs:(i + 1) * Bs], lp_part, R_lp, Bs)
            return latents, log_det_jac, logp
        latents, ld_part, R_ld, lp_part, R_lp = self._transform_core(x, logp is not None, levels, slots, steps, ready)
        N.accumulate(log_det_jac, ld_part, R_ld, B, slots, self._multipliers(H, W, dev), self.L * self.K)
        if logp is not None and R_lp > 0:
            N.accumulate(logp, lp_part, R_lp, B)
        return latents, log_det_jac, logp

    # ---- concurrent sub-batches inside a captured graph
    def _n_sub(self, B: int) -> int:
        # measured (profiles/): with batch 128 two concurrent sub-batches are 6% SLOWER than one stream (the deep-level
        # kernels are latency-, not occupancy-bound), so the default is one stream; the knob stays for large batches
        n = int(os.environ.get("NFDPM_STREAMS", "1"))
        if n <= 1 or B % n != 0 or B // n < 16:
            return 1
        return n

    @staticmethod
    def _deep_sub(B: int, h: int, w: int) -> int:
        """Concurrent sub-batches for ONE level's StepFlow chain.  At the deep levels (8x8 and smaller) every kernel of the
        chain is latency-bound on a fraction of the SMs (one 128-row tile per CTA: 16...128 CTAs, 8-15 us per launch of which
        2-6 us are MMA work), and the images of a batch are independent: running the chain of several image groups on
        concurrent streams inside the captured graph overlaps those latencies.  Level 0 stays on one stream (its persistent
        GEMM grids already fill the GPU; splitting it was measured 6 % slower).  NFDPM_DEEP_STREAMS="n1:n2" = sub-batches
        at 64-pixel / 16-pixel-and-smaller levels.  MEASURED SLOWER in every combination (profiles/r02_deep_streams.txt:
        5.60 ms per config-2 step on one stream, 5.90 / 5.92 / 6.71 ms with 2:2 / 2:4 / 4:4) — the deep-level GEMMs turn out
        to be bound by the depth of their TMA operand ring (two 32 KB stages in flight per ~1 us L2 round trip = 64 GB/s per
        CTA), not by idle SMs, and concurrent chains compete for the same L2 — so the default is one stream ("1:1")."""
        if h * w >= 256:
            return 1
        spec = os.environ.get("NFDPM_DEEP_STREAMS", "1:1").split(":")
        try:
            n = int(spec[0] if h * w >= 64 else spec[-1])
        except ValueError:
            n = 1
        while n > 1 and (B % n != 0 or (B // n) * h * w < 256):      # whole sub-batches of at least two 128-row tiles
            n -= 1
        return max(n, 1)

    def _fork_join(self, n: int, fn, pool: str = "_streams"):
        """fn(0) ... fn(n-1) on n concurrent streams forked from / joined into the current one (inside a capture: parallel
        branches of the graph).  `pool`: attribute holding the streams, so that nested forks do not share them."""
        if n == 1:
            return [fn(0)]
        cur = torch.cuda.current_stream()
        if getattr(self, pool, None) is None or len(getattr(self, pool)) < n:
            setattr(self, pool, [torch.cuda.Stream() for _ in range(n)])
        streams = getattr(self, pool)
        out = []
        for i in range(n):
            s = streams[i]
            s.wait_stream(cur)
            with torch.cuda.stream(s):
                out.append(fn(i))
        for i in range(n):
            cur.wait_stream(streams[i])
        return out

    def _transform_autograd(self, x, log_det_jac, logp, levels, slots, steps, ready):
        """Training path (reference trainer.py:155-164): forward with activation stash, hand-written backward kernels
        behind one autograd Function (normalizing_flow/_train.py)."""
        from . import _train as T
        B, c, H, W = x.shape
        if not T.supported(self, H, W):
            raise NotImplementedError(
                f"Glow.transform under autograd: the training kernels need every level's image to fit one CTA "
                f"(H*W/4 <= 256 at level 0); got {H}x{W}.  Use torch.no_grad() for likelihood evaluation.")
        if not ready:
            # data-dependent ActNorm initialisation happens inside the first transform (transforms.py:74-78), without
            # gradient; run it once on this batch, then take the training path
            with torch.no_grad():
                self._transform_core(x.detach(), logp is not None, levels, slots, steps, False)
        if torch.is_grad_enabled() and (log_det_jac.requires_grad or (logp is not None and logp.requires_grad)):
            raise RuntimeError("log_det_jac / logp are updated in place and must not require grad on entry")
        out = T.GlowTransformFn.apply(self, x, log_det_jac, logp, *list(self.parameters()))
        if logp is not None:
            return list(out[2:]), out[0], out[1]
        return list(out[1:]), out[0], None

    def _fast_ok(self, H: int, W: int) -> bool:
        """Use the fused step-boundary kernels?  They are chosen PER LEVEL (`_level_fast`): a level whose image does not
        fit one CTA (more than 256 pixels, e.g. the 64x64 and 32x32 levels of a 128x128 input) runs the unfused
        kernels, the deeper levels of the same model still run the fused ones."""
        return os.environ.get("NFDPM_FUSED_BOUNDARY", "1") != "0"

    @staticmethod
    def _level_fast(C: int, h: int, w: int) -> bool:
        return h * w <= 256 and N.flow_boundary_smem(C, h, w, 1, 1) <= 200 * 1024

    @classmethod
    def _level_mode(cls, B: int, C: int, h: int, w: int) -> str:
        """Which kernels run the StepFlow boundaries of a level:
          "image"   one CTA per image (flow_boundary / gemm3_boundary): images of at most 256 pixels in batches that fill the GPU
          "tiled"   row bands with a recomputed halo (flow_boundary_tiled): larger images (the 64x64 / 32x32 levels of a
                    128x128 input) and small batches (config 4: 8 images per GPU would occupy 8 of 148 SMs)
          "unfused" separate K-A / im2col / coupling kernels (NFDPM_TILED=0, or a single image row beyond shared memory)"""
        tiled = os.environ.get("NFDPM_TILED", "1") != "0" and N.flow_boundary_tiles(B, C, h, w, 1, 1, 1) > 0
        deep = os.environ.get("NFDPM_TILED_DEEP", "0") == "1" and h * w < 256        # experiment knob
        if cls._level_fast(C, h, w) and ((B >= 64 and not deep) or not tiled):
            return "image"
        return "tiled" if tiled else "unfused"

    def _transform_core(self, x: Tensor, with_logp: bool, levels, slots, steps, ready: bool):
        B, c, H, W = x.shape
        dev = x.device
        if ready and self._fast_ok(H, W):
            return self._transform_fast(x, with_logp, levels, slots, steps)
        if ready:
            # one batched LU/fold launch for every StepFlow whose parameters changed since the last call
            E.prepare_mix([s._mix_entry(slots[i:i + 1]) for i, s in enumerate(steps)])
        # partial-sum rows: per step T_l rows of B
        geo = []
        h, w, ch = H, W, c
        for li in range(self.L):
            h, w = h // 2, w // 2
            C = ch * 4
            geo.append((C, h, w, N.ld_tiles(h * w)))
            ch = C // 2
        R_ld = sum(g[3] for g in geo) * self.K
        R_lp = sum(g[3] for g in geo[:-1])
        ld_part = E.WS.get("ld_part", max(R_ld, 1) * B, torch.float32, dev)
        lp_part = E.WS.get("lp_part", max(R_lp, 1) * B, torch.float32, dev) if with_logp else None
        latents: List[Tensor] = []
        cur, cur_bs, cur_c, cur_h, cur_w = x, c * H * W, c, H, W
        row = lrow = si = 0
        for li, (flows, split) in enumerate(levels):
            C, h, w, T = geo[li]
            P = h * w
            a = torch.empty(B, C, h, w, dtype=torch.float32, device=dev)
            b = torch.empty_like(a)
            N.squeeze(cur, a, B, cur_c, cur_h, cur_w, cur_bs, C * P)
            for step in flows:
                step._forward_views(a, C * P, b, C * P, B, h, w, ld_part[row * B:], slots[si:si + 1])
                a, b = b, a
                row += T
                si += 1
            if split is None:
                latents.append(a)
                break
            z = torch.empty(B, C // 2, h, w, dtype=torch.float32, device=dev)
            split._forward_views(a, C * P, B, C, h, w, z, lp_part[lrow * B:] if lp_part is not None else None)
            lrow += T
            latents.append(z)
            cur, cur_bs, cur_c, cur_h, cur_w = a, C * P, C // 2, h, w
        return latents, ld_part, R_ld, lp_part, R_lp

    # ---- inverse: latents -> x
    def invert(self, latents: list, temperature: float = 1.0, log_det_jac: Optional[Tensor] = None,
               logp: Optional[Tensor] = None) -> Tensor:
        """latents -> x.  ``latents`` holds all L parts (decoding) or the last ones only: every Split without a latent draws
        its half from its conditional prior at ``temperature``.

        ``log_det_jac`` / ``logp`` (optional [B] fp32/fp64 CUDA vectors, ``+=`` in place, ``None`` = not requested) receive
        exactly the terms ``transform(x, log_det_jac, logp)`` would add at the returned x, without a second pass:
          log_det_jac += sum over steps of P*sum(actnorm scale) + P*log|det W| + sum log(s + 1e-6), which is
                         -log|det dx/dz| of this inverse (it divides by exactly s + 1e-6);
          logp        += sum over the L-1 Split halves of log N(z_l; mean_l, exp(logs_l)), supplied or drawn; the final
                         latent's prior is not included, as in ``transform``.
        Under a temperature this is the model's density at the returned sample, not the tempered one.  The accumulated
        density is not differentiable: a call that NFDPM_INVERT_GRAD=1 would record raises NotImplementedError."""
        z_last = E.check_input(latents[-1], "latents[-1]")
        B, Cf, h, w = z_last.shape
        if Cf != 2 ** (self.L + 1) * self.in_channel:
            raise ValueError(f"final latent has {Cf} channels, expected {2 ** (self.L + 1) * self.in_channel}")
        E.check_acc(log_det_jac, B, "log_det_jac")
        E.check_acc(logp, B, "logp")
        accs = [a for a in (log_det_jac, logp) if a is not None]
        if torch.is_grad_enabled() and any(a.requires_grad for a in accs):
            raise RuntimeError("log_det_jac / logp are updated in place and must not require grad on entry")
        if E.autograd_needed(z_last, self) or any(isinstance(t, Tensor) and t.requires_grad for t in latents):
            if E.invert_grad_enabled():
                if accs:
                    raise NotImplementedError(
                        "Glow.invert: the accumulated log_det_jac / logp are not differentiable; a recorded invert "
                        "(NFDPM_INVERT_GRAD=1) takes no accumulators.  Call it under torch.no_grad() for the density.")
                from ._invgrad import glow_invert
                return glow_invert(self, latents, temperature)
            # without NFDPM_INVERT_GRAD: compute it without recording and fail loudly on back-propagation
            from .transforms import _NoBackward
            deps = [t for t in latents if isinstance(t, Tensor) and t.requires_grad] + \
                   [p for p in self.parameters() if p.requires_grad]
            with torch.no_grad():
                out = self.invert([t.detach() if isinstance(t, Tensor) else t for t in latents], temperature,
                                  log_det_jac, logp)
            return _NoBackward.apply(out, "Glow.invert", False, *deps)
        with_ld, with_lp = log_det_jac is not None, logp is not None
        dev = z_last.device
        levels = self._levels()
        slots = self._slots(dev)
        steps = [s for flows, _ in levels for s in flows]
        ready = all(s._ready() for s in steps)
        H, W = h << self.L, w << self.L
        if self._use_graph(ready) and 1 <= len(latents) <= self.L and all(isinstance(t, Tensor) for t in latents):
            # decoding (all L latents supplied) and sampling (fewer: every Split without a latent draws its half from the
            # learned conditional prior, transforms.py:305-307) replay one captured chain; the normal draws inside a
            # captured chain come from torch's default CUDA generator, whose Philox offset advances on every replay
            lat_in = [E.check_input(t, "latent") for t in latents]
            if self._params_changed():
                self._refresh_caches(steps, slots)
            sampling = len(latents) < self.L
            key = ("inv", B, h, w, E.precision(), dev.index)
            if sampling:
                key += (len(latents), float(temperature))
            if with_ld or with_lp:                    # a chain that also writes the density partials
                key += ((with_ld, with_lp),)
            ent = self._graphs.get(key)
            if ent is None and sampling:
                # the temperature is baked into a sampling graph: keep at most four of them (a temperature sweep would
                # otherwise pin one captured chain and its workspace per value)
                old = [k for k in self._graphs if k[0] == "inv" and len(k) >= 8]
                for k in old[:max(0, len(old) - 3)]:
                    E.WS.drop_scope(("glow", id(self), k))
                    del self._graphs[k]
            statics = ent["lat"] if ent is not None else [torch.empty_like(t) for t in lat_in]
            for s_, t in zip(statics, lat_in):
                if s_.shape != t.shape:
                    raise ValueError(f"latent has shape {tuple(t.shape)}, expected {tuple(s_.shape)}")
                s_.copy_(t)

            nsub = self._n_sub(B)
            Bs = B // nsub

            def build():
                outs = self._fork_join(nsub, lambda i: self._invert_core(
                    [t[i * Bs:(i + 1) * Bs] for t in statics], temperature, levels, slots, steps, True, with_ld, with_lp))
                return {"lat": statics, "outs": outs}
            ent = self._graph_entry(key, build)
            if ent["lat"] is not statics:
                for s_, t in zip(ent["lat"], lat_in):
                    s_.copy_(t)
            ent["graph"].replay()
            N.launch_count += ent["n_launch"]
            outs = ent["outs"]
            for i, (_, ld_part, R_ld, lp_part, R_lp) in enumerate(outs):     # after the replay, into the caller's tensors
                sl = slice(i * Bs, (i + 1) * Bs)
                self._add_density(log_det_jac[sl] if with_ld else None, logp[sl] if with_lp else None, ld_part, R_ld,
                                  lp_part, R_lp, Bs, H, W, slots)
            return torch.cat([o[0] for o in outs]) if nsub > 1 else outs[0][0].clone()
        x, ld_part, R_ld, lp_part, R_lp = self._invert_core(latents, temperature, levels, slots, steps, ready, with_ld,
                                                            with_lp)
        self._add_density(log_det_jac, logp, ld_part, R_ld, lp_part, R_lp, B, H, W, slots)
        return x

    def _add_density(self, log_det_jac, logp, ld_part, R_ld: int, lp_part, R_lp: int, B: int, H: int, W: int,
                     slots: Tensor) -> None:
        """The final accumulates of an inverse, as ``transform`` runs them: the log-det partial rows plus the L*K
        data-independent constants, and the Split log-prob rows."""
        if log_det_jac is not None:
            N.accumulate(log_det_jac, ld_part, R_ld, B, slots, self._multipliers(H, W, slots.device), self.L * self.K)
        if logp is not None and R_lp > 0:
            N.accumulate(logp, lp_part, R_lp, B)

    def _part_rows(self, B: int, H: int, W: int, inverse: bool = False, fused: bool = True) -> Tuple[int, int]:
        """Rows of B per-image partials that one call writes for [B, c, H, W] images: (log-det rows, Split log-prob rows).
        Log-det: one per step at "image" levels, ld_tiles(P) per step at unfused ones, one per band at "tiled" levels, where
        K-1 boundaries carry an im2col sink and the level's last one does not (and has a mix in the inverse only, which can
        change the band height).  ``fused=False``: every level unfused (NFDPM_FUSED_BOUNDARY=0, or a model not ready)."""
        R_ld = R_lp = 0
        hh, ww, cc = H, W, self.in_channel
        for li in range(self.L):
            hh, ww, CC = hh // 2, ww // 2, cc * 4
            mode = self._level_mode(B, CC, hh, ww) if fused else "unfused"
            if mode == "tiled":
                R_ld += (self.K - 1) * N.flow_boundary_tiles(B, CC, hh, ww, 1, 1, 1) + \
                    N.flow_boundary_tiles(B, CC, hh, ww, 1, int(inverse), 0)
            else:
                R_ld += self.K * (1 if mode == "image" else N.ld_tiles(hh * ww))
            if li < self.L - 1:
                R_lp += N.ld_tiles(hh * ww)
            cc = CC // 2
        return R_ld, R_lp

    def _transform_fast(self, x: Tensor, with_logp: bool, levels, slots, steps):
        """Forward with the fused step-boundary kernel: 4 launches per StepFlow (boundary + 3 GEMMs)."""
        B, c, H, W = x.shape
        dev = x.device
        E.prepare_mix([s._mix_entry(slots[i:i + 1]) for i, s in enumerate(steps)])
        R_ld, R_lp = self._part_rows(B, H, W)
        ld_part = E.WS.get("ld_part", R_ld * B, torch.float32, dev)
        lp_part = E.WS.get("lp_part", max(R_lp, 1) * B, torch.float32, dev) if with_logp else None
        latents: List[Tensor] = []
        cur, cur_bs = x, c * H * W
        h, w, ch = H, W, c
        row = lrow = 0
        for li, (flows, split) in enumerate(levels):
            h, w, C = h // 2, w // 2, ch * 4
            P = h * w
            mode = self._level_mode(B, C, h, w)
            if mode == "tiled":
                st, rows = self._transform_level_tiled(flows, cur, cur_bs, B, C, h, w, ld_part, row, dev)
                row += rows
                if split is None:
                    latents.append(st)
                    break
                z = torch.empty(B, C // 2, h, w, dtype=torch.float32, device=dev)
                split._forward_views(st, C * P, B, C, h, w, z, lp_part[lrow * B:] if lp_part is not None else None)
                lrow += N.ld_tiles(P)
                latents.append(z)
                cur, cur_bs, ch = st, C * P, C // 2
                continue
            if mode == "unfused":
                # NFDPM_TILED=0: squeeze + unfused K-A / im2col / GEMMs / coupling per step
                T = N.ld_tiles(P)
                a = torch.empty(B, C, h, w, dtype=torch.float32, device=dev)
                b = torch.empty_like(a)
                N.squeeze(cur, a, B, ch, 2 * h, 2 * w, cur_bs, C * P)
                for step in flows:
                    step._forward_views(a, C * P, b, C * P, B, h, w, ld_part[row * B:], None)
                    a, b = b, a
                    row += T
                st = a
                if split is None:
                    latents.append(st)
                    break
                z = torch.empty(B, C // 2, h, w, dtype=torch.float32, device=dev)
                split._forward_views(st, C * P, B, C, h, w, z, lp_part[lrow * B:] if lp_part is not None else None)
                lrow += T
                latents.append(z)
                cur, cur_bs, ch = st, C * P, C // 2
                continue
            st = torch.empty(B, C, h, w, dtype=torch.float32, device=dev)     # flow state of this level (in place)
            nsub = self._deep_sub(B, h, w) if torch.cuda.is_current_stream_capturing() else 1
            Bs = B // nsub
            row0 = row

            def level_chain(i, cur=cur, cur_bs=cur_bs, st=st, flows=flows, C=C, h=h, w=w, P=P, Bs=Bs, row0=row0):
                """The K StepFlows of this level for images [i*Bs, (i+1)*Bs): views of the level's tensors."""
                src_i, st_i = cur[i * Bs:(i + 1) * Bs], st[i * Bs:(i + 1) * Bs]
                first = flows[0]
                A1, K1p = E.coupling_a1(first.affcoupling, Bs, C, h, w, dev)
                # level entry: squeeze + K-A of step 0 + im2col
                N.flow_boundary(src_i, cur_bs, True, None, 0, None, None, None, first._mix.fwd_mt, first._mix.fwd_beta,
                                st_i, C * P, A1, K1p, Bs, C, h, w, False)
                r = row0
                for k, step in enumerate(flows):
                    cp = step.affcoupling
                    nxt = flows[k + 1] if k + 1 < len(flows) else None
                    part = ld_part[r * B + i * Bs:]
                    if nxt is not None:
                        A1n, K1p = E.coupling_a1(nxt.affcoupling, Bs, C, h, w, dev)     # same scratch buffer as A1
                        E.coupling_boundary(cp, A1, Bs, C, h, w, st_i, C * P, part, nxt._mix.fwd_mt,
                                            nxt._mix.fwd_beta, st_i, C * P, A1n, K1p, False)
                        A1 = A1n
                    else:
                        E.coupling_boundary(cp, A1, Bs, C, h, w, st_i, C * P, part, None, None, st_i, C * P,
                                            None, 0, False)
                    r += 1
            self._fork_join(nsub, level_chain, pool="_deep_streams")
            row += len(flows)
            if split is None:
                latents.append(st)
                break
            z = torch.empty(B, C // 2, h, w, dtype=torch.float32, device=dev)
            split._forward_views(st, C * P, B, C, h, w, z, lp_part[lrow * B:] if lp_part is not None else None)
            lrow += N.ld_tiles(P)
            latents.append(z)
            cur, cur_bs, ch = st, C * P, C // 2
        return latents, ld_part, R_ld, lp_part, (R_lp if with_logp else 0)

    def _density_parts(self, B: int, H: int, W: int, dev, with_ld: bool, with_lp: bool, fused: bool):
        """Partial buffers of one inverse that also returns its density (None where not requested), with their row
        counts: the rows the forward writes (`_part_rows`)."""
        R_ld, R_lp = self._part_rows(B, H, W, inverse=True, fused=fused)
        ld_part = E.WS.get("ld_part", R_ld * B, torch.float32, dev) if with_ld else None
        lp_part = E.WS.get("lp_part", max(R_lp, 1) * B, torch.float32, dev) if with_lp else None
        return ld_part, R_ld, lp_part, R_lp

    def _invert_fast(self, latents, temperature, levels, slots, steps, with_ld: bool = False, with_lp: bool = False):
        """Inverse with the fused step-boundary kernel -> (x, ld_part, R_ld, lp_part, R_lp); the partials are written
        only when requested (``with_ld`` / ``with_lp``), in level order from the deepest level."""
        z_last = latents[-1]
        B, C, h, w = z_last.shape
        dev = z_last.device
        E.prepare_mix([s._mix_entry(slots[i:i + 1]) for i, s in enumerate(steps)])
        ld_part, R_ld, lp_part, R_lp = self._density_parts(B, h << self.L, w << self.L, dev, with_ld, with_lp, True)
        src = z_last                                   # caller memory: read only
        row = lrow = 0
        for li in range(self.L - 1, -1, -1):
            flows, _ = levels[li]
            P = h * w
            mode = self._level_mode(B, C, h, w)
            if mode == "tiled":
                st, rows = self._invert_level_tiled(flows, src, B, C, h, w, dev, ld_part, row)
                row += rows
            elif mode == "unfused":
                # NFDPM_TILED=0: unfused inverse steps (coupling^-1 in place, then K-A^-1)
                cur, own = src, li < self.L - 1        # the deepest level reads caller memory
                other = torch.empty(B, C, h, w, dtype=torch.float32, device=dev)
                for step in reversed(flows):
                    part = ld_part[row * B:] if ld_part is not None else None
                    if own:
                        step._inverse_views(cur, C * P, cur, C * P, other, C * P, B, h, w, part)
                        cur, other = other, cur
                    else:
                        tmp = torch.empty(B, C, h, w, dtype=torch.float32, device=dev)
                        step._inverse_views(cur, C * P, tmp, C * P, other, C * P, B, h, w, part)
                        cur, other, own = other, tmp, True
                    row += N.ld_tiles(P)
                st = cur
            else:
                st = self._invert_level_fast(flows, src, li < self.L - 1, B, C, h, w, dev, ld_part, row)
                row += len(flows)
            if li == 0:
                out = torch.empty(B, C // 4, h * 2, w * 2, dtype=torch.float32, device=dev)
                N.unsqueeze(st, out, B, C, h, w, C * P, (C // 4) * P * 4)
                return out, ld_part, R_ld, lp_part, R_lp
            Cn, hn, wn = 2 * (C // 4), h * 2, w * 2
            nxt = torch.empty(B, Cn, hn, wn, dtype=torch.float32, device=dev)
            N.unsqueeze(st, nxt, B, C, h, w, C * P, Cn * hn * wn)
            latent = get_item(latents, -(self.L - li + 1))
            levels[li - 1][1]._fill_second_half(nxt, Cn * hn * wn, B, Cn, hn, wn, latent, temperature,
                                                logp_part=lp_part[lrow * B:] if lp_part is not None else None)
            lrow += N.ld_tiles(hn * wn)
            src, C, h, w = nxt, Cn, hn, wn
        raise AssertionError("unreachable")

    def _transform_level_tiled(self, flows, cur, cur_bs: int, B: int, C: int, h: int, w: int, ld_part, row: int, dev):
        """K forward StepFlows of one level with the row-band boundary kernel.  A band reads halo rows that a neighbouring
        band writes, so the flow state ping-pongs between two buffers.  Returns (state, log-det partial rows used)."""
        P = h * w
        bufs = [torch.empty(B, C, h, w, dtype=torch.float32, device=dev) for _ in range(2)]
        first = flows[0]
        A1, K1p = E.coupling_a1(first.affcoupling, B, C, h, w, dev)
        N.flow_boundary_tiled(cur, cur_bs, True, None, 0, None, None, None, first._mix.fwd_mt, first._mix.fwd_beta,
                              bufs[0], C * P, None, 0, A1, K1p, B, C, h, w, False,
                              N.flow_boundary_tiles(B, C, h, w, 0, 1, 1))       # level entry: squeeze + K-A + im2col
        src, rows = 0, 0
        for k, step in enumerate(flows):
            nxt = flows[k + 1] if k + 1 < len(flows) else None
            T = N.flow_boundary_tiles(B, C, h, w, 1, int(nxt is not None), int(nxt is not None))
            if nxt is not None:
                A1n, K1p = E.coupling_a1(nxt.affcoupling, B, C, h, w, dev)
                E.coupling_boundary(step.affcoupling, A1, B, C, h, w, bufs[src], C * P, ld_part[(row + rows) * B:],
                                    nxt._mix.fwd_mt, nxt._mix.fwd_beta, bufs[1 - src], C * P, A1n, K1p, False, tiles=T)
                A1 = A1n
            else:
                E.coupling_boundary(step.affcoupling, A1, B, C, h, w, bufs[src], C * P, ld_part[(row + rows) * B:],
                                    None, None, bufs[1 - src], C * P, None, 0, False, tiles=T)
            src = 1 - src
            rows += T
        return bufs[src], rows

    def _invert_level_tiled(self, flows, src, B: int, C: int, h: int, w: int, dev, ld_part=None, row: int = 0):
        """K inverse StepFlows of one level with the row-band boundary kernel (state ping-pongs between two buffers;
        `src` — caller memory or the previous level's output — is only read).  Returns (state, log-det partial rows used
        from `row` on; written only when `ld_part` is given)."""
        P = h * w
        rows = 0
        bufs = [torch.empty(B, C, h, w, dtype=torch.float32, device=dev) for _ in range(2)]
        A1, K1p = E.coupling_a1(flows[-1].affcoupling, B, C, h, w, dev)
        N.flow_boundary_tiled(src, C * P, False, None, 0, None, None, None, None, None, None, 0, None, 0, A1, K1p, B, C,
                              h, w, False, N.flow_boundary_tiles(B, C, h, w, 0, 0, 1))   # im2col of the level's entry state
        cur, dst = src, 0
        for k in range(len(flows) - 1, -1, -1):
            step = flows[k]
            T = N.flow_boundary_tiles(B, C, h, w, 1, 1, int(k > 0))
            part = ld_part[(row + rows) * B:] if ld_part is not None else None
            if k > 0:
                A1n, K1p = E.coupling_a1(flows[k - 1].affcoupling, B, C, h, w, dev)
                E.coupling_boundary(step.affcoupling, A1, B, C, h, w, cur, C * P, part, step._mix.inv_mt,
                                    step._mix.inv_beta, bufs[dst], C * P, A1n, K1p, True, tiles=T)
                A1 = A1n
            else:
                E.coupling_boundary(step.affcoupling, A1, B, C, h, w, cur, C * P, part, step._mix.inv_mt,
                                    step._mix.inv_beta, bufs[dst], C * P, None, 0, True, tiles=T)
            cur, dst = bufs[dst], 1 - dst
            rows += T
        return cur, rows

    def _invert_level_fast(self, flows, src, own: bool, B: int, C: int, h: int, w: int, dev, ld_part=None,
                           row: int = 0) -> Tensor:
        """K inverse StepFlows of one level with the fused kernels; returns the level's input state.  Deep levels run as
        concurrent sub-batches inside a captured graph (`_deep_sub`).  Step k writes its log-det partial to row `row + k`
        of `ld_part` when given."""
        P = h * w
        st = src if own else torch.empty(B, C, h, w, dtype=torch.float32, device=dev)
        nsub = self._deep_sub(B, h, w) if torch.cuda.is_current_stream_capturing() else 1
        Bs = B // nsub

        def level_chain(i):
            src_i, st_i = src[i * Bs:(i + 1) * Bs], st[i * Bs:(i + 1) * Bs]
            last = flows[-1]
            A1, K1p = E.coupling_a1(last.affcoupling, Bs, C, h, w, dev)
            N.flow_boundary(src_i, C * P, False, None, 0, None, None, None, None, None, None, 0, A1, K1p, Bs, C, h, w,
                            False)                     # im2col of the level's entry state
            for k in range(len(flows) - 1, -1, -1):
                step = flows[k]
                cp = step.affcoupling
                part = ld_part[(row + k) * B + i * Bs:] if ld_part is not None else None
                if k > 0:
                    A1n, K1p = E.coupling_a1(flows[k - 1].affcoupling, Bs, C, h, w, dev)
                    E.coupling_boundary(cp, A1, Bs, C, h, w, src_i, C * P, part, step._mix.inv_mt, step._mix.inv_beta,
                                        st_i, C * P, A1n, K1p, True)
                    A1 = A1n
                else:
                    E.coupling_boundary(cp, A1, Bs, C, h, w, src_i, C * P, part, step._mix.inv_mt, step._mix.inv_beta,
                                        st_i, C * P, None, 0, True)
                src_i = st_i
        self._fork_join(nsub, level_chain, pool="_deep_streams")
        return st

    def _invert_core(self, latents, temperature, levels, slots, steps, ready: bool, with_ld: bool = False,
                     with_lp: bool = False):
        """-> (x, ld_part, R_ld, lp_part, R_lp), as `_invert_fast`."""
        z_last = E.check_input(latents[-1], "latents[-1]")
        B, Cf, h, w = z_last.shape
        dev = z_last.device
        if ready and self._fast_ok(h * 2 ** self.L, w * 2 ** self.L):
            return self._invert_fast([z_last] if len(latents) == 1 else list(latents), temperature, levels, slots, steps,
                                     with_ld, with_lp)
        if ready or with_ld:
            # (the inverse initialises no StepFlow ActNorm, so the log-det constants of a model that is not ready are
            # final here too)
            E.prepare_mix([s._mix_entry(slots[i:i + 1]) for i, s in enumerate(steps)])
        ld_part, R_ld, lp_part, R_lp = self._density_parts(B, h << self.L, w << self.L, dev, with_ld, with_lp, False)
        C, P = Cf, h * w
        cur = z_last
        own = False          # `cur` is caller memory until the first step has produced a copy
        row = lrow = 0
        for li in range(self.L - 1, -1, -1):
            flows, _ = levels[li]
            other = torch.empty(B, C, h, w, dtype=torch.float32, device=dev)
            for step in reversed(flows):
                part = ld_part[row * B:] if ld_part is not None else None
                if own:
                    step._inverse_views(cur, C * P, cur, C * P, other, C * P, B, h, w, part)
                    cur, other = other, cur
                else:
                    tmp = torch.empty(B, C, h, w, dtype=torch.float32, device=dev)
                    step._inverse_views(cur, C * P, tmp, C * P, other, C * P, B, h, w, part)
                    cur, other, own = other, tmp, True
                row += N.ld_tiles(P)
            # undo the squeeze of this level into the first half of the previous level's tensor
            if li == 0:
                out = torch.empty(B, C // 4, h * 2, w * 2, dtype=torch.float32, device=dev)
                N.unsqueeze(cur, out, B, C, h, w, C * P, (C // 4) * P * 4)
                return out, ld_part, R_ld, lp_part, R_lp
            Cn, hn, wn = 2 * (C // 4), h * 2, w * 2
            nxt = torch.empty(B, Cn, hn, wn, dtype=torch.float32, device=dev)
            N.unsqueeze(cur, nxt, B, C, h, w, C * P, Cn * hn * wn)
            latent = get_item(latents, -(self.L - li + 1))   # None -> draw from the conditional prior
            levels[li - 1][1]._fill_second_half(nxt, Cn * hn * wn, B, Cn, hn, wn, latent, temperature,
                                                logp_part=lp_part[lrow * B:] if lp_part is not None else None)
            lrow += N.ld_tiles(hn * wn)
            cur, own, C, h, w, P = nxt, True, Cn, hn, wn, hn * wn
        raise AssertionError("unreachable")

    @torch.no_grad()
    def sample(self, latents: list, postprocess_func=None, temperature: float = 1.0,
               log_det_jac: Optional[Tensor] = None, logp: Optional[Tensor] = None) -> Tensor:
        """eval() -> invert -> optional postprocess -> train(), like the reference (glow.py:230-246; note the
        unconditional switch back to train mode).  ``log_det_jac`` / ``logp`` as in ``invert``: the density of the
        continuous sample before ``postprocess_func``."""
        self.eval()
        new_samples = self.invert(latents, temperature, log_det_jac, logp)
        out = postprocess_func(new_samples.float()) if postprocess_func else new_samples.float()
        self.train()
        return out
