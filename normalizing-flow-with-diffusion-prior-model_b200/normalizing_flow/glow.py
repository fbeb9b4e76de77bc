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
        E.check_width(self.flows[0]._C if len(self.flows) else 0, "GlowBlock")
        y, log_det_jac, logp = self.squeeze.transform(x, log_det_jac, logp)
        for flow in self.flows:
            y, log_det_jac, logp = flow.transform(y, log_det_jac, logp)
        return self.split.transform(y, log_det_jac, logp)

    def invert(self, y: Tensor, latent: Tensor = None, temperature: float = 1.0, *,
               seeds: Optional[Tensor] = None) -> Tensor:
        """``temperature`` / ``seeds`` as in ``Split.invert`` (draw site 0: the draw of ``Glow`` level 0)."""
        E.check_width(self.flows[0]._C if len(self.flows) else 0, "GlowBlock")
        inv = self.split.invert(y, latent, temperature=temperature, seeds=seeds)
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

    def _refresh_caches(self, device: torch.device) -> None:
        """Re-run LU/fold and weight packing for parameters that changed (outside any graph)."""
        self._prepare_mix(device)
        self._pack_plan(self._steps(), E.coupling_dtype(), False).refresh()
        for blk in self.blocks:
            E.refresh_split(blk.split, blk.flows[0]._C)

    def _use_graph(self, ready: bool) -> bool:
        return ready and E.graphs_enabled() and not torch.cuda.is_current_stream_capturing()

    def _replay(self, key, inputs: List[Tensor], walk):
        """The captured call ``key``: refresh the parameter caches if a parameter changed, copy ``inputs`` into the entry's
        static tensors, capture ``walk(statics)`` when the entry is missing or stale, replay.  Returns what the captured
        walk returned (graph-static tensors)."""
        if self._params_changed():
            self._refresh_caches(inputs[0].device)
        ent = self._graphs.get(key)
        statics = ent["in"] if ent is not None else [torch.empty_like(t) for t in inputs]
        for s_, t in zip(statics, inputs):
            if s_.shape != t.shape:
                raise ValueError(f"input has shape {tuple(t.shape)}, expected {tuple(s_.shape)}")
            s_.copy_(t)
        if ent is None or ent["epoch"] != E.alloc_epoch:
            scope = ("glow", id(self), key)
            E.WS.drop_scope(scope)
            # parameter caches were refreshed above, outside the graph
            g, out, n_launch = E.capture(scope, lambda: walk(statics), own=True)
            ent = self._graphs[key] = {"in": statics, "out": out, "graph": g, "n_launch": n_launch,
                                       "epoch": E.alloc_epoch}
        ent["graph"].replay()
        N.launch_count += ent["n_launch"]
        return ent["out"]

    # ---- helpers
    def _levels(self) -> List[Tuple[nn.ModuleList, Optional[Split]]]:
        lv = [(blk.flows, blk.split) for blk in self.blocks]
        lv.append((self.final_flows, None))
        return lv

    def _geometry(self, H: int, W: int) -> List[Tuple[nn.ModuleList, Optional[Split], int, int, int]]:
        """Per level, in forward order, for [B, c, H, W] images: (StepFlows, Split or None at the last level, channels C,
        height h and width w of the level's squeezed flow state)."""
        return [(flows, split, (4 * self.in_channel) << li, H >> (li + 1), W >> (li + 1))
                for li, (flows, split) in enumerate(self._levels())]

    def _steps(self) -> List[StepFlow]:
        return [s for flows, _ in self._levels() for s in flows]

    def _ready(self) -> bool:
        """Every StepFlow's ActNorms are initialised (the first transform of a fresh model initialises them)."""
        return all(s._ready() for s in self._steps())

    def _slots(self, device: torch.device) -> Tensor:
        n = self.L * self.K
        if self._logdet_all is None or self._logdet_all.device != device:
            self._logdet_all = torch.zeros(n, dtype=torch.float32, device=device)
        return self._logdet_all

    def _prepare_mix(self, device: torch.device) -> None:
        """One batched LU/fold launch for every StepFlow whose parameters changed since the last call; step i's
        log|det W| lands in slot i, which the final accumulate reads."""
        slots = self._slots(device)
        E.prepare_mix([s._mix_entry(slots[i:i + 1]) for i, s in enumerate(self._steps())])

    def _multipliers(self, H: int, W: int, device: torch.device) -> Tensor:
        key = (H, W, device.index)
        t = self._cmul.get(key)
        if t is None:
            vals = [float(h * w) for _, _, _, h, w in self._geometry(H, W) for _ in range(self.K)]
            t = torch.tensor(vals, dtype=torch.float32, device=device)
            self._cmul[key] = t
        return t

    def _check_width(self) -> None:
        """The final level is the widest (2^(L+1) * in_channel channels).  The constructor accepts any L, as the reference's
        does (a checkpoint of such a model loads); the calls refuse one wider than the kernels run, before any launch."""
        E.check_width(2 ** (self.L + 1) * self.in_channel, f"Glow(in_channel={self.in_channel}, L={self.L})")

    def _check_image(self, x: Tensor) -> Tuple[int, int, int, int]:
        B, C, H, W = x.shape
        if C != self.in_channel:
            raise ValueError(f"Glow built for {self.in_channel} input channels got {C}")
        if H % (2 ** self.L) or W % (2 ** self.L):
            raise ValueError(f"input {H}x{W} is not divisible by 2^L = {2 ** self.L}")
        return B, C, H, W

    # ---- forward: x -> ([z_0..z_{L-1}], log_det_jac, logp)
    def transform(self, x: Tensor, log_det_jac: Tensor, logp: Tensor) -> Tuple[list, Tensor, Tensor]:
        self._check_width()
        x = E.check_input(x)
        B, c, H, W = self._check_image(x)
        if log_det_jac is None:
            raise ValueError("log_det_jac accumulator is required")
        E.check_acc(log_det_jac, B, "log_det_jac")
        E.check_acc(logp, B, "logp")
        ready = self._ready()
        if E.autograd_needed(x, self):
            return self._transform_autograd(x, log_det_jac, logp, ready)
        with_logp = logp is not None
        if self._use_graph(ready):
            key = ("fwd", B, H, W, with_logp, E.precision(), x.device.index)
            latents, parts = self._replay(key, [x], lambda xs: self._transform_walk(xs[0], with_logp, True))
            latents = [z.clone() for z in latents]
        else:
            latents, parts = self._transform_walk(x, with_logp, ready)
        self._add_density(log_det_jac, logp, parts, H, W)
        return latents, log_det_jac, logp

    def _transform_autograd(self, x, log_det_jac, logp, ready: bool):
        """Training path (reference trainer.py:155-164): forward with activation stash, hand-written backward kernels
        behind one autograd Function (normalizing_flow/_train.py)."""
        from . import _train as T
        if not ready:
            # data-dependent ActNorm initialisation happens inside the first transform (transforms.py:74-78), without
            # gradient; run it once on this batch, then take the training path
            with torch.no_grad():
                self._transform_walk(x.detach(), logp is not None, False)
        if torch.is_grad_enabled() and (log_det_jac.requires_grad or (logp is not None and logp.requires_grad)):
            raise RuntimeError("log_det_jac / logp are updated in place and must not require grad on entry")
        out = T.GlowTransformFn.apply(self, x, log_det_jac, logp, *list(self.parameters()))
        if logp is not None:
            return list(out[2:]), out[0], out[1]
        return list(out[1:]), out[0], None

    @staticmethod
    def _level_fast(C: int, h: int, w: int) -> bool:
        """Can the fused step-boundary kernel hold one image of this level in a CTA?"""
        return h * w <= 256 and N.flow_boundary_smem(C, h, w, 1, 1) <= 200 * 1024

    @classmethod
    def _level_mode(cls, B: int, C: int, h: int, w: int) -> str:
        """Which kernels run the StepFlow boundaries of a level:
          "image"   one CTA per image (flow_boundary / gemm3_boundary): images of at most 256 pixels in batches that fill the GPU
          "tiled"   row bands with a recomputed halo (flow_boundary_tiled): larger images (the 64x64 / 32x32 levels of a
                    128x128 input) and small batches (config 4: 8 images per GPU would occupy 8 of 148 SMs)
          "unfused" separate K-A / im2col / coupling kernels (NFDPM_TILED=0, or a single image row beyond shared memory)
        Levels wider than 192 channels (the final levels of L6 / L7 models on RGB) take "unfused": both fused-boundary
        queries refuse them, because their C x C mix matrix does not fit shared memory; nfdpm_channel_mix / nfdpm_mix_bwd
        run them with their multi-CTA wide kernels."""
        tiled = os.environ.get("NFDPM_TILED", "1") != "0" and N.flow_boundary_tiles(B, C, h, w, 1, 1, 1) > 0
        if cls._level_fast(C, h, w) and (B >= 64 or not tiled):
            return "image"
        return "tiled" if tiled else "unfused"

    def _part_rows(self, B: int, H: int, W: int, inverse: bool = False, fused: bool = True) -> Tuple[int, int]:
        """Rows of B per-image partials that one call writes for [B, c, H, W] images: (log-det rows, Split log-prob rows).
        Log-det: one per step at "image" levels, ld_tiles(P) per step at unfused ones, one per band at "tiled" levels, where
        K-1 boundaries carry an im2col sink and the level's last one does not (and has a mix in the inverse only, which can
        change the band height).  ``fused=False``: every level unfused (NFDPM_FUSED_BOUNDARY=0, or a model not ready)."""
        R_ld = R_lp = 0
        for _, split, C, h, w in self._geometry(H, W):
            mode = self._level_mode(B, C, h, w) if fused else "unfused"
            if mode == "tiled":
                R_ld += (self.K - 1) * N.flow_boundary_tiles(B, C, h, w, 1, 1, 1) + \
                    N.flow_boundary_tiles(B, C, h, w, 1, int(inverse), 0)
            else:
                R_ld += self.K * (1 if mode == "image" else N.ld_tiles(h * w))
            if split is not None:
                R_lp += N.ld_tiles(h * w)
        return R_ld, R_lp

    def _density_parts(self, B: int, H: int, W: int, dev, inverse: bool, fused: bool, with_ld: bool, with_lp: bool):
        """(ld_part, R_ld, lp_part, R_lp): the partial buffers of one call (None where not requested) with the row counts
        of `_part_rows`."""
        R_ld, R_lp = self._part_rows(B, H, W, inverse, fused)
        ld_part = E.WS.get("ld_part", R_ld * B, torch.float32, dev) if with_ld else None
        lp_part = E.WS.get("lp_part", max(R_lp, 1) * B, torch.float32, dev) if with_lp else None
        return ld_part, R_ld, lp_part, R_lp

    def _add_density(self, log_det_jac, logp, parts, H: int, W: int) -> None:
        """The final accumulates of a call, after its chain or its replay: the log-det partial rows plus the L*K
        data-independent constants H*W*(sum(scale) + log|det W|), and the Split log-prob rows (``None``: not requested)."""
        ld_part, R_ld, lp_part, R_lp = parts
        if log_det_jac is not None:
            dev = ld_part.device
            N.accumulate(log_det_jac, ld_part, R_ld, log_det_jac.shape[0], self._slots(dev), self._multipliers(H, W, dev),
                         self.L * self.K)
        if logp is not None and R_lp > 0:
            N.accumulate(logp, lp_part, R_lp, logp.shape[0])

    def _transform_walk(self, x: Tensor, with_logp: bool, ready: bool):
        """x -> (latents, (ld_part, R_ld, lp_part, R_lp)): the levels in forward order.  Each level squeezes its input, runs
        its K StepFlows with the kernels of its `_level_mode` (every level unfused for a model that is not ready or under
        NFDPM_FUSED_BOUNDARY=0) and splits off its latent."""
        B, c, H, W = x.shape
        dev = x.device
        fused = ready and E.fused_boundary_enabled()
        if ready:
            self._prepare_mix(dev)
        parts = ld_part, R_ld, lp_part, R_lp = self._density_parts(B, H, W, dev, False, fused, True, with_logp)
        slots = self._slots(dev)
        run = {"image": self._transform_level_image, "tiled": self._transform_level_tiled,
               "unfused": self._transform_level_unfused}
        latents: List[Tensor] = []
        cur, cur_bs = x, c * H * W
        row = lrow = 0
        for li, (flows, split, C, h, w) in enumerate(self._geometry(H, W)):
            mode = self._level_mode(B, C, h, w) if fused else "unfused"
            st, rows = run[mode](flows, slots[li * self.K:(li + 1) * self.K], cur, cur_bs, B, C, h, w, ld_part, row)
            row += rows
            if split is None:
                latents.append(st)
                break
            z = torch.empty(B, C // 2, h, w, dtype=torch.float32, device=dev)
            split._forward_views(st, C * h * w, B, C, h, w, z, lp_part[lrow * B:] if lp_part is not None else None)
            lrow += N.ld_tiles(h * w)
            latents.append(z)
            cur, cur_bs = st, C * h * w
        assert (row, lrow) == (R_ld, R_lp), f"wrote {row} / {lrow} partial rows, allotted {R_ld} / {R_lp}"
        return latents, parts

    def _transform_level_image(self, flows, slots, src, src_bs: int, B: int, C: int, h: int, w: int, ld_part, row: int):
        """K forward StepFlows with one CTA per image, in place on the level's state: the level entry (squeeze + K-A of
        step 0 + im2col), then per step GEMM1, GEMM2 and [GEMM3 +] the step boundary.  Returns (state, log-det partial rows
        written from `row` on)."""
        P, dev = h * w, src.device
        st = torch.empty(B, C, h, w, dtype=torch.float32, device=dev)
        first = flows[0]
        A1, K1p = E.coupling_a1(first.affcoupling, B, C, h, w, dev)
        N.flow_boundary(src, src_bs, True, None, 0, None, None, None, first._mix.fwd_mt, first._mix.fwd_beta, st, C * P,
                        A1, K1p, B, C, h, w, False)
        for k, step in enumerate(flows):
            cp = step.affcoupling
            nxt = flows[k + 1] if k + 1 < len(flows) else None
            part = ld_part[(row + k) * B:]
            if nxt is not None:
                A1n, K1p = E.coupling_a1(nxt.affcoupling, B, C, h, w, dev)     # same scratch buffer as A1
                E.coupling_boundary(cp, A1, B, C, h, w, st, C * P, part, nxt._mix.fwd_mt, nxt._mix.fwd_beta, st, C * P,
                                    A1n, K1p, False)
                A1 = A1n
            else:
                E.coupling_boundary(cp, A1, B, C, h, w, st, C * P, part, None, None, st, C * P, None, 0, False)
        return st, len(flows)

    def _transform_level_tiled(self, flows, slots, src, src_bs: int, B: int, C: int, h: int, w: int, ld_part, row: int):
        """K forward StepFlows of one level with the row-band boundary kernel.  A band reads halo rows that a neighbouring
        band writes, so the flow state ping-pongs between two buffers.  Returns (state, log-det partial rows written)."""
        P, dev = h * w, src.device
        bufs = [torch.empty(B, C, h, w, dtype=torch.float32, device=dev) for _ in range(2)]
        first = flows[0]
        A1, K1p = E.coupling_a1(first.affcoupling, B, C, h, w, dev)
        N.flow_boundary_tiled(src, src_bs, True, None, 0, None, None, None, first._mix.fwd_mt, first._mix.fwd_beta,
                              bufs[0], C * P, None, 0, A1, K1p, B, C, h, w, False,
                              N.flow_boundary_tiles(B, C, h, w, 0, 1, 1))       # level entry: squeeze + K-A + im2col
        cur, rows = 0, 0
        for k, step in enumerate(flows):
            nxt = flows[k + 1] if k + 1 < len(flows) else None
            T = N.flow_boundary_tiles(B, C, h, w, 1, int(nxt is not None), int(nxt is not None))
            if nxt is not None:
                A1n, K1p = E.coupling_a1(nxt.affcoupling, B, C, h, w, dev)
                E.coupling_boundary(step.affcoupling, A1, B, C, h, w, bufs[cur], C * P, ld_part[(row + rows) * B:],
                                    nxt._mix.fwd_mt, nxt._mix.fwd_beta, bufs[1 - cur], C * P, A1n, K1p, False, tiles=T)
                A1 = A1n
            else:
                E.coupling_boundary(step.affcoupling, A1, B, C, h, w, bufs[cur], C * P, ld_part[(row + rows) * B:],
                                    None, None, bufs[1 - cur], C * P, None, 0, False, tiles=T)
            cur = 1 - cur
            rows += T
        return bufs[cur], rows

    def _transform_level_unfused(self, flows, slots, src, src_bs: int, B: int, C: int, h: int, w: int, ld_part,
                                 row: int):
        """Squeeze, then per StepFlow the separate K-A / im2col / GEMMs / coupling kernels.  A step of a model that is not
        ready initialises its ActNorm from this batch first, then runs its LU/fold into its log-det slot (``slots[k]``).
        Returns (state, log-det partial rows written)."""
        P, T = h * w, N.ld_tiles(h * w)
        a = torch.empty(B, C, h, w, dtype=torch.float32, device=src.device)
        b = torch.empty_like(a)
        N.squeeze(src, a, B, C // 4, 2 * h, 2 * w, src_bs, C * P)
        for k, step in enumerate(flows):
            step._forward_views(a, C * P, b, C * P, B, h, w, ld_part[(row + k * T) * B:], slots[k:k + 1])
            a, b = b, a
        return a, len(flows) * T

    # ---- inverse: latents -> x
    def invert(self, latents: list, temperature: float = 1.0, log_det_jac: Optional[Tensor] = None,
               logp: Optional[Tensor] = None, *, seeds: Optional[Tensor] = None) -> Tensor:
        """latents -> x.  ``latents`` holds all L parts (decoding) or the last ones only: every Split without a latent draws
        its half from its conditional prior at ``temperature``.

        ``log_det_jac`` / ``logp`` (optional [B] fp32/fp64 CUDA vectors, ``+=`` in place, ``None`` = not requested) receive
        exactly the terms ``transform(x, log_det_jac, logp)`` would add at the returned x, without a second pass:
          log_det_jac += sum over steps of P*sum(actnorm scale) + P*log|det W| + sum log(s + 1e-6), which is
                         -log|det dx/dz| of this inverse (it divides by exactly s + 1e-6);
          logp        += sum over the L-1 Split halves of log N(z_l; mean_l, exp(logs_l)), supplied or drawn; the final
                         latent's prior is not included, as in ``transform``.
        Under a temperature this is the model's density at the returned sample, not the tempered one.  The accumulated
        density is not differentiable here: a call that NFDPM_INVERT_GRAD=1 would record raises NotImplementedError.
        ``invert_with_density`` returns the same values and back-propagates through them.

        ``temperature`` may also be a float32 CUDA vector [B], one temperature per image.  ``seeds`` (int64 CUDA [B],
        optional) makes every draw of the call a pure function of (seeds[b], level of the Split, element): image b does
        not depend on the batch it is drawn in, its position there, earlier draws or graph replays (the contract is in
        include/nfdpm_b200.h).  Without seeds the draws come from torch's CUDA generator.  A call that draws nothing (all
        L latents supplied) accepts seeds and a tensor temperature and uses neither.  With seeds or a tensor temperature
        one captured chain serves every temperature and seed vector of its shape."""
        z_last, recorded = self._check_invert_args(latents, log_det_jac, logp)
        accs = [a for a in (log_det_jac, logp) if a is not None]
        B, _, h, w = z_last.shape
        temperature, seeds = E.sampling_inputs(temperature, seeds, B, z_last.device)
        if recorded:
            if E.invert_grad_enabled():
                if accs:
                    raise NotImplementedError(
                        "Glow.invert: the accumulated log_det_jac / logp are not differentiable; a recorded invert "
                        "(NFDPM_INVERT_GRAD=1) takes no accumulators.  Call it under torch.no_grad() for the density, "
                        "or Glow.invert_with_density to back-propagate through it.")
                from ._invgrad import glow_invert
                return glow_invert(self, latents, temperature, seeds=seeds)
            # without NFDPM_INVERT_GRAD: compute it without recording and fail loudly on back-propagation
            from .transforms import _NoBackward
            deps = [t for t in latents if isinstance(t, Tensor) and t.requires_grad] + \
                   [p for p in self.parameters() if p.requires_grad]
            with torch.no_grad():
                out = self.invert([t.detach() if isinstance(t, Tensor) else t for t in latents], temperature,
                                  log_det_jac, logp, seeds=seeds)
            return _NoBackward.apply(out, "Glow.invert", False, *deps)
        with_ld, with_lp = log_det_jac is not None, logp is not None
        ready = self._ready()
        H, W = h << self.L, w << self.L
        if self._use_graph(ready) and 1 <= len(latents) <= self.L and all(isinstance(t, Tensor) for t in latents):
            # decoding (all L latents supplied) and sampling (fewer: every Split without a latent draws its half from the
            # learned conditional prior, transforms.py:305-307) replay one captured chain; without seeds the normal draws
            # inside a captured chain come from torch's default CUDA generator, whose Philox offset advances on every
            # replay, and with seeds the prior kernels draw from the static seed vector
            lat_in = [E.check_input(t, "latent") for t in latents]
            sampling = len(latents) < self.L
            # seeds or per-image temperatures: the [B] vectors are static inputs of the chain, so its key has no temperature
            ex = sampling and isinstance(temperature, Tensor)
            key = ("inv", B, h, w, E.precision(), z_last.device.index)
            if ex:
                key += (len(latents), "ex", seeds is not None)
            elif sampling:
                key += (len(latents), float(temperature))
            if with_ld or with_lp:                    # a chain that also writes the density partials
                key += ((with_ld, with_lp),)
            if key not in self._graphs and sampling and not ex:
                # the temperature is baked into a sampling graph: keep at most four of them (a temperature sweep would
                # otherwise pin one captured chain and its workspace per value)
                old = [k for k in self._graphs if k[0] == "inv" and len(k) >= 8 and k[7] != "ex"]
                for k in old[:max(0, len(old) - 3)]:
                    E.WS.drop_scope(("glow", id(self), k))
                    del self._graphs[k]
            n = len(lat_in)
            if ex:
                ins = lat_in + [temperature] + ([seeds] if seeds is not None else [])
                walk = lambda st: self._invert_walk(st[:n], st[n], True, with_ld, with_lp,
                                                    seeds=st[n + 1] if len(st) > n + 1 else None)
            else:
                ins, walk = lat_in, lambda lat: self._invert_walk(lat, temperature, True, with_ld, with_lp)
            x, parts = self._replay(key, ins, walk)
            self._add_density(log_det_jac, logp, parts, H, W)     # after the replay, into the caller's tensors
            return x.clone()
        x, parts = self._invert_walk(latents, temperature, ready, with_ld, with_lp, seeds=seeds)
        self._add_density(log_det_jac, logp, parts, H, W)
        return x

    def _check_invert_args(self, latents: list, log_det_jac: Optional[Tensor], logp: Optional[Tensor]):
        """The argument checks of `invert` / `invert_with_density`, before any launch.  Returns (final latent, whether the
        call is to be recorded by autograd: a latent or a parameter requires grad)."""
        self._check_width()
        z_last = E.check_input(latents[-1], "latents[-1]")
        B, Cf, h, w = z_last.shape
        if Cf != 2 ** (self.L + 1) * self.in_channel:
            raise ValueError(f"final latent has {Cf} channels, expected {2 ** (self.L + 1) * self.in_channel}")
        E.check_acc(log_det_jac, B, "log_det_jac")
        E.check_acc(logp, B, "logp")
        accs = [a for a in (log_det_jac, logp) if a is not None]
        if torch.is_grad_enabled() and any(a.requires_grad for a in accs):
            raise RuntimeError("log_det_jac / logp are updated in place and must not require grad on entry")
        return z_last, E.autograd_needed(z_last, self) or any(isinstance(t, Tensor) and t.requires_grad for t in latents)

    def invert_with_density(self, latents: list, temperature: float = 1.0, log_det_jac: Optional[Tensor] = None,
                            logp: Optional[Tensor] = None, *,
                            seeds: Optional[Tensor] = None) -> Tuple[Tensor, Optional[Tensor], Optional[Tensor]]:
        """``invert(latents, temperature, log_det_jac, logp)`` returning ``(x, log_det_jac, logp)``, differentiable in all
        three: the density of generated images as a function of the latents and the weights (reverse-KL / variational
        training, entropy terms, distillation through the flow).  The arguments and the accumulated values are exactly
        those of ``invert``; at least one accumulator is required (``None`` stays ``None``), and both are updated in place.

        Without autograd (no latent and no parameter requires grad, or under ``torch.no_grad()``) this is ``invert``, with
        the same captured chain.  Otherwise it records ONE autograd node whose outputs are x and the accumulators (marked
        dirty, like ``transform``'s): gradients reach the latents, every StepFlow parameter and every Split prior conv,
        at sampled Splits (through the draw and its log-density) and at supplied ones (through the log-density).  It
        records whether or not NFDPM_INVERT_GRAD is set: that knob guards ``invert``, ``sample`` and the granular inverses,
        whose callers did not ask for a graph.  The recorded call is not captured in a CUDA graph.  ``temperature`` /
        ``seeds`` as in ``invert``; the backward uses each image's temperature and the draws the forward made."""
        if log_det_jac is None and logp is None:
            raise ValueError("Glow.invert_with_density needs log_det_jac and/or logp; Glow.invert returns the images alone")
        z_last, recorded = self._check_invert_args(latents, log_det_jac, logp)
        if recorded:
            temperature, seeds = E.sampling_inputs(temperature, seeds, z_last.shape[0], z_last.device)
            from ._invgrad import glow_invert
            return glow_invert(self, latents, temperature, log_det_jac, logp, seeds)
        return self.invert(latents, temperature, log_det_jac, logp, seeds=seeds), log_det_jac, logp

    def _invert_walk(self, latents, temperature, ready: bool, with_ld: bool = False, with_lp: bool = False,
                     level=None, eps_sink: Optional[list] = None, seeds: Optional[Tensor] = None):
        """latents -> (x, (ld_part, R_ld, lp_part, R_lp)): the levels deepest first.  Each level runs its K inverse
        StepFlows with the kernels of its `_level_mode` (as `_transform_walk`) and unsqueezes into the first half of the
        previous level's state, whose Split fills the second half with the supplied latent or a draw from its conditional
        prior.  The partials are written only when requested (``with_ld`` / ``with_lp``).
        ``level(mode, flows, src, B, C, h, w, ld_part, row) -> (state, rows)`` replaces the no-grad kernels of a level (the
        recorded inverse keeps the operands of every step) and writes the log-det partial rows the no-grad level function
        of ``mode`` writes; ``eps_sink`` receives (assembled Split state, eps of its draw or None) per Split.
        ``temperature``: a number or a [B] device vector; ``seeds``: the Split of level l draws with draw site l."""
        z_last = E.check_input(latents[-1], "latents[-1]")
        B, _, h, w = z_last.shape
        H, W = h << self.L, w << self.L
        dev = z_last.device
        fused = ready and E.fused_boundary_enabled()
        if ready or with_ld:
            # (the inverse initialises no StepFlow ActNorm, so the log-det constants of a model that is not ready are
            # final here too)
            self._prepare_mix(dev)
        parts = ld_part, R_ld, lp_part, R_lp = self._density_parts(B, H, W, dev, True, fused, with_ld, with_lp)
        run = {"image": self._invert_level_image, "tiled": self._invert_level_tiled,
               "unfused": self._invert_level_unfused}
        geo = self._geometry(H, W)
        st = z_last
        row = lrow = 0
        for li in range(self.L - 1, -1, -1):
            flows, _, C, h, w = geo[li]
            mode = self._level_mode(B, C, h, w) if fused else "unfused"
            if level is None:          # (the deepest level's input is caller memory: `own` False, only read)
                st, rows = run[mode](flows, st, li < self.L - 1, B, C, h, w, ld_part, row)
            else:
                st, rows = level(mode, flows, st, B, C, h, w, ld_part, row)
            row += rows
            # undo the squeeze of this level into the first half of the previous level's state (the image at level 0)
            Cn = C // 4 if li == 0 else C // 2
            nxt = torch.empty(B, Cn, 2 * h, 2 * w, dtype=torch.float32, device=dev)
            N.unsqueeze(st, nxt, B, C, h, w, C * h * w, Cn * 4 * h * w)
            st = nxt
            if li > 0:
                drawn = [] if eps_sink is not None else None
                geo[li - 1][1]._fill_second_half(nxt, Cn * 4 * h * w, B, Cn, 2 * h, 2 * w,
                                                 get_item(latents, li - self.L - 1), temperature, eps_sink=drawn,
                                                 logp_part=lp_part[lrow * B:] if lp_part is not None else None,
                                                 seeds=seeds, stream_id=li - 1)
                lrow += N.ld_tiles(4 * h * w)
                if eps_sink is not None:
                    eps_sink.append((nxt, drawn[0] if drawn else None))
        assert (row, lrow) == (R_ld, R_lp), f"wrote {row} / {lrow} partial rows, allotted {R_ld} / {R_lp}"
        return st, parts

    def _invert_level_image(self, flows, src, own: bool, B: int, C: int, h: int, w: int, ld_part, row: int):
        """K inverse StepFlows with one CTA per image, in place on the level's state (on a copy when `src` is caller memory,
        ``own`` False).  Step k writes its log-det partial to row `row + k` of `ld_part` when given.  Returns (state,
        rows)."""
        P, dev = h * w, src.device
        st = src if own else torch.empty(B, C, h, w, dtype=torch.float32, device=dev)
        last = flows[-1]
        A1, K1p = E.coupling_a1(last.affcoupling, B, C, h, w, dev)
        N.flow_boundary(src, C * P, False, None, 0, None, None, None, None, None, None, 0, A1, K1p, B, C, h, w,
                        False)                         # im2col of the level's entry state
        for k in range(len(flows) - 1, -1, -1):
            step = flows[k]
            cp = step.affcoupling
            part = ld_part[(row + k) * B:] if ld_part is not None else None
            if k > 0:
                A1n, K1p = E.coupling_a1(flows[k - 1].affcoupling, B, C, h, w, dev)
                E.coupling_boundary(cp, A1, B, C, h, w, src, C * P, part, step._mix.inv_mt, step._mix.inv_beta,
                                    st, C * P, A1n, K1p, True)
                A1 = A1n
            else:
                E.coupling_boundary(cp, A1, B, C, h, w, src, C * P, part, step._mix.inv_mt, step._mix.inv_beta,
                                    st, C * P, None, 0, True)
            src = st
        return st, len(flows)

    def _invert_level_tiled(self, flows, src, own: bool, B: int, C: int, h: int, w: int, ld_part, row: int):
        """K inverse StepFlows of one level with the row-band boundary kernel (state ping-pongs between two buffers;
        `src` is only read).  Returns (state, log-det partial rows from `row` on; written only when `ld_part` is given)."""
        P, dev = h * w, src.device
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

    def _invert_level_unfused(self, flows, src, own: bool, B: int, C: int, h: int, w: int, ld_part, row: int):
        """K inverse StepFlows with the separate kernels: coupling^-1 in place, then K-A^-1 into the other buffer (caller
        memory, ``own`` False, is only read).  Returns (state, log-det partial rows from `row` on)."""
        P, T = h * w, N.ld_tiles(h * w)
        cur, other = src, torch.empty(B, C, h, w, dtype=torch.float32, device=src.device)
        for k, step in enumerate(reversed(flows)):
            part = ld_part[(row + k * T) * B:] if ld_part is not None else None
            if own:
                step._inverse_views(cur, C * P, cur, C * P, other, C * P, B, h, w, part)
                cur, other = other, cur
            else:
                tmp = torch.empty(B, C, h, w, dtype=torch.float32, device=src.device)
                step._inverse_views(cur, C * P, tmp, C * P, other, C * P, B, h, w, part)
                cur, other, own = other, tmp, True
        return cur, len(flows) * T

    @torch.no_grad()
    def sample(self, latents: list, postprocess_func=None, temperature: float = 1.0,
               log_det_jac: Optional[Tensor] = None, logp: Optional[Tensor] = None, *,
               seeds: Optional[Tensor] = None) -> Tensor:
        """eval() -> invert -> optional postprocess -> train(), like the reference (glow.py:230-246; note the
        unconditional switch back to train mode).  ``log_det_jac`` / ``logp`` as in ``invert``: the density of the
        continuous sample before ``postprocess_func``.  ``temperature`` / ``seeds`` as in ``invert``."""
        self.eval()
        new_samples = self.invert(latents, temperature, log_det_jac, logp, seeds=seeds)
        out = postprocess_func(new_samples.float()) if postprocess_func else new_samples.float()
        self.train()
        return out
