"""Host-side orchestration of the libnfdpm_b200 kernels: parameter caches, scratch memory and the
launch sequences of one StepFlow / coupling network.  No arithmetic happens here — every number is
produced by a kernel of the C-ABI library; torch supplies device memory and the current stream.

Precision modes (env ``NFDPM_PRECISION``); everything outside the coupling networks is fp32 in every mode:
  * ``fp32`` — the reference's arithmetic (fp32 convolutions, utils.py:36,64) on the tcgen05 tensor cores: operands are SPLIT
    bf16 pairs (v = hi + lo, NFDPM_BF16X2) and every product is formed as hi*hi + lo*hi + hi*lo with fp32 TMEM
    accumulation (2^-17 operand error instead of bf16's 2^-9).  Parity bar: z / log-det within 1e-4 relative of the
    reference, reconstruction < 1e-4.  Training in this mode uses the same operand format for the stash, the dgrad
    GEMMs and the weight-gradient GEMMs (gradients within 2e-4 of the reference's autograd).
  * ``bf16`` — plain bf16 operands, one MMA per product: 3x the tensor throughput, stated tolerance in DESIGN.md / tests.
  * ``auto`` (default) — inference (``torch.no_grad()`` transform / invert / sample: likelihood evaluation, decoding,
    sampling) in ``fp32``, the training step (autograd-recorded transform + backward) in ``bf16``.
  * ``fp32_simt`` — coupling GEMMs in exact fp32 FMA on CUDA cores everywhere (debugging reference, ~10x slower).
"""
from __future__ import annotations

import os
from typing import List, Optional, Sequence, Tuple

import torch

from . import _native as N


#: installed by _dp.GradAllReduce.global_initialization(): called as ``hook(scale, bias, n_local)`` right after every
#: data-dependent ActNorm initialisation so that the statistics of the ranks' shards can be combined (SURVEY §8(f) row 2)
stats_hook = None


def channel_stats(x, layout: int, B: int, C: int, P: int, xs: int, scale, bias) -> None:
    """Data-dependent ActNorm initialisation from this rank's batch (reference transforms.py:74-78): one launch writes
    ``scale = -log(std_unbiased + 1e-6)`` and ``bias = -mean`` per channel; under data parallelism the hook replaces them
    by the values of the GLOBAL batch."""
    N.channel_stats(x, layout, B, C, P, xs, scale, bias)
    if stats_hook is not None:
        stats_hook(scale, bias, B * P)


def precision() -> str:
    p = os.environ.get("NFDPM_PRECISION", "auto").lower()
    if p not in ("auto", "fp32", "bf16", "fp32_simt"):
        raise ValueError(f"NFDPM_PRECISION must be 'auto', 'fp32', 'bf16' or 'fp32_simt', got {p!r}")
    return p


#: storage dtypes of the coupling-network operands: torch.float32 (CUDA-core GEMMs), torch.bfloat16, N.SPLIT (bf16 pairs)
TC_DTYPES = (torch.bfloat16, N.SPLIT)


def coupling_dtype(train: bool = False) -> torch.dtype:
    """Operand format of the coupling-network GEMMs for the inference chains or (``train``) the training step."""
    p = precision()
    if p == "bf16":
        return torch.bfloat16
    if p == "fp32_simt":
        return torch.float32
    if p == "fp32":
        return N.SPLIT
    return torch.bfloat16 if train else N.SPLIT


def invert_grad_enabled() -> bool:
    """``NFDPM_INVERT_GRAD=1``: ``invert`` (Glow, the granular transforms) and the priors' ``sample`` record an autograd
    node with hand-written backward kernels.  Off by default: ``invert`` then refuses to back-propagate."""
    return os.environ.get("NFDPM_INVERT_GRAD", "0") == "1"


def round_up(a: int, b: int) -> int:
    return (a + b - 1) // b * b


class _Workspace:
    """Grow-only scratch buffers keyed by (scope, tag, dtype, device, stream).  Kernels of one flow run in stream
    order and each buffer is consumed before it is overwritten, so one set per stream is enough.  A CUDA-graph
    capture runs under its own ``scope`` so that the buffers baked into the graph are never re-allocated."""

    def __init__(self):
        self._bufs = {}
        self.scope = None

    def drop_scope(self, scope) -> None:
        for k in [k for k in self._bufs if k[0] == scope]:
            del self._bufs[k]

    def get(self, tag: str, numel: int, dtype: torch.dtype, device: torch.device) -> torch.Tensor:
        key = (self.scope, tag, dtype, device.index, torch.cuda.current_stream(device).cuda_stream)
        t = self._bufs.get(key)
        if t is None or t.numel() < numel:
            t = torch.empty(max(numel, 1), dtype=dtype, device=device)
            self._bufs[key] = t
        return t

    def clear(self):
        self._bufs.clear()


WS = _Workspace()
_SCALARS = {}
#: bumped whenever a parameter-derived cache buffer is (re)allocated; CUDA graphs that baked the old pointers
#: compare it with the value at capture time and re-capture
alloc_epoch = 0


def _bump_epoch() -> None:
    global alloc_epoch
    alloc_epoch += 1


def graphs_enabled() -> bool:
    return os.environ.get("NFDPM_GRAPHS", "1") != "0"


def fused_boundary_enabled() -> bool:
    """``NFDPM_FUSED_BOUNDARY=0`` runs every level of Glow's inference chains on the unfused kernels: the reference the
    fused and row-band step boundaries are tested against."""
    return os.environ.get("NFDPM_FUSED_BOUNDARY", "1") != "0"


def scalar_f32(device: torch.device, value: float) -> torch.Tensor:
    """Cached 1-element device tensor (multipliers for nfdpm_accumulate)."""
    key = (device.index, float(value))
    t = _SCALARS.get(key)
    if t is None:
        t = torch.full((1,), float(value), dtype=torch.float32, device=device)
        _SCALARS[key] = t
    return t


MAX_LEVEL_CHANNELS = 1024      # widest flow level the kernels run (nfdpm_mix_prepare, nfdpm_channel_mix, nfdpm_mix_bwd)


def check_width(C: int, what: str) -> None:
    """Refuses a flow level wider than MAX_LEVEL_CHANNELS, before any launch (e.g. L8 on RGB: 1536 channels)."""
    if C > MAX_LEVEL_CHANNELS:
        raise ValueError(f"{what}: a level of {C} channels is wider than the {MAX_LEVEL_CHANNELS} this package supports")


def check_input(x: torch.Tensor, what: str = "input") -> torch.Tensor:
    N.require_cuda(x, what)
    if x.dtype != torch.float32:
        raise TypeError(f"{what} must be float32 (got {x.dtype})")
    if x.dim() != 4:
        raise ValueError(f"{what} must be [B, C, H, W] (got shape {tuple(x.shape)})")
    return x if x.is_contiguous() else x.contiguous()


def check_acc(a: Optional[torch.Tensor], B: int, what: str) -> None:
    if a is None:
        return
    N.require_cuda(a, what)
    if a.dtype not in (torch.float32, torch.float64) or a.dim() != 1 or a.shape[0] != B or not a.is_contiguous():
        raise ValueError(f"{what} must be a contiguous float32/float64 vector of length {B} "
                         f"(got {a.dtype}, shape {tuple(a.shape)})")


def sampling_inputs(temperature, seeds: Optional[torch.Tensor], B: int, device: torch.device):
    """The checks of the sampling keywords of a call that draws B images, before any launch.  ``temperature``: a Python
    number, or a contiguous float32 CUDA vector [B] (one per image, no gradient); ``seeds``: None or a contiguous int64
    CUDA vector [B].  Returns (temperature, seeds): the number unchanged when neither is a tensor (the torch-generator
    draw with a scalar temperature), else a [B] float32 device vector (a number is broadcast) and the seeds."""
    device = torch.device(device)
    if device.type == "cuda" and device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    if seeds is not None:
        if not isinstance(seeds, torch.Tensor):
            raise TypeError(f"seeds must be an int64 CUDA tensor [B] (got {type(seeds).__name__})")
        N.require_cuda(seeds, "seeds")
        if seeds.dtype != torch.int64 or seeds.dim() != 1 or seeds.shape[0] != B or not seeds.is_contiguous():
            raise ValueError(f"seeds must be a contiguous int64 vector of length {B} (got {seeds.dtype}, shape "
                             f"{tuple(seeds.shape)})")
        if seeds.device != device:
            raise ValueError(f"seeds live on {seeds.device}, the call runs on {device}")
    if isinstance(temperature, torch.Tensor):
        N.require_cuda(temperature, "temperature")
        if temperature.dtype != torch.float32 or temperature.dim() != 1 or temperature.shape[0] != B or \
                not temperature.is_contiguous():
            raise ValueError(f"a tensor temperature must be a contiguous float32 vector of length {B} (got "
                             f"{temperature.dtype}, shape {tuple(temperature.shape)})")
        if temperature.device != device:
            raise ValueError(f"temperature lives on {temperature.device}, the call runs on {device}")
        if temperature.requires_grad:
            raise ValueError("temperature requires grad: sampling has no gradient with respect to the temperature")
        return temperature, seeds
    if seeds is None:
        return temperature, None
    return torch.full((B,), float(temperature), dtype=torch.float32, device=device), seeds


def autograd_needed(x: torch.Tensor, module: torch.nn.Module) -> bool:
    if not torch.is_grad_enabled():
        return False
    if x.requires_grad:
        return True
    return any(p.requires_grad for p in module.parameters())


def _vkey(*tensors) -> tuple:
    return tuple((t.data_ptr(), t._version) if t is not None else None for t in tensors)


#: True while Glow captures its own inference graph (parameter caches are refreshed OUTSIDE that graph)
own_capture = False


def cache_hit(cached_key, key) -> bool:
    """Parameter-derived caches (LU/fold, packed weights) are keyed on tensor version counters.  Inside a CUDA-graph
    capture started by the CALLER (e.g. a whole training step: forward, backward, optimizer) the refresh kernels
    must be part of the graph, because the parameters change between replays without the host noticing."""
    if cached_key != key:
        return False
    return own_capture or not torch.cuda.is_current_stream_capturing()


def capture(scope, build, own: bool):
    """``build()`` once eagerly (parameter caches, one-time kernel attributes), then under capture into a CUDA graph ->
    (graph, what the captured ``build()`` returned, launches per replay).  Workspace buffers taken inside the captured
    chain live under ``scope``.  ``own``: the caller refreshed the parameter caches outside the graph (``own_capture``);
    a chain whose parameters change between replays refreshes them inside it."""
    global own_capture
    warm = ("warm",) + tuple(scope)
    prev = WS.scope
    try:
        WS.scope = warm
        build()
        torch.cuda.current_stream().synchronize()
        WS.drop_scope(warm)
        WS.scope = scope                              # buffers baked into the graph live (only) under this scope
        g = torch.cuda.CUDAGraph()
        n0 = N.launch_count
        own_capture = own
        with torch.cuda.graph(g):
            out = build()
        n_launch = N.launch_count - n0
    finally:
        own_capture = False
        WS.scope = prev
    N.launch_count -= n_launch                        # counted per replay instead
    return g, out, n_launch


# ------------------------------------------------------------------------------------------- mix cache
class MixCache:
    """Prepared mixing matrices of one (ActNorm, InvConv2d) pair: see nfdpm_mix_prepare."""

    def __init__(self):
        self.key = None
        self.C = 0
        self.fwd_mt = self.fwd_beta = self.inv_mt = self.inv_beta = self.winv = self.logdet = self.lu_ws = None

    def invalidate(self):
        self.key = None

    def _alloc(self, C: int, device: torch.device, logdet_slot: Optional[torch.Tensor]):
        if self.fwd_mt is not None and self.C == C and self.fwd_mt.device == device:
            if logdet_slot is not None and (self.logdet is None or self.logdet.data_ptr() != logdet_slot.data_ptr()):
                self.logdet = logdet_slot
                self.key = None
                _bump_epoch()
            return
        f = dict(dtype=torch.float32, device=device)
        _bump_epoch()
        self.C = C
        self.fwd_mt = torch.empty(C * C, **f)
        self.fwd_beta = torch.empty(C, **f)
        self.inv_mt = torch.empty(C * C, **f)
        self.inv_beta = torch.empty(C, **f)
        self.winv = torch.empty(C * C, **f)
        self.logdet = logdet_slot if logdet_slot is not None else torch.empty(1, **f)
        self.lu_ws = torch.empty(2 * C * C, dtype=torch.float64, device=device)
        self.key = None


def prepare_mix(entries: Sequence[Tuple[MixCache, Optional[torch.Tensor], Optional[torch.Tensor],
                                        Optional[torch.Tensor], int, Optional[torch.Tensor]]]) -> None:
    """entries: (cache, weight|None, scale|None, bias|None, C, logdet_slot|None).  Re-runs the batched
    LU/fold kernel only for entries whose parameters changed (tensor version counters)."""
    items = []
    for cache, w, s, b, C, slot in entries:
        dev = (w if w is not None else s).device
        cache._alloc(C, dev, slot)
        key = _vkey(w, s, b)
        if cache_hit(cache.key, key):
            continue
        cache.key = key
        items.append(N.MixItem(weight=N._p(w), scale=N._p(s), bias=N._p(b), C=C, pad_=0,
                               fwd_mt=cache.fwd_mt.data_ptr(), fwd_beta=cache.fwd_beta.data_ptr(),
                               inv_mt=cache.inv_mt.data_ptr(), inv_beta=cache.inv_beta.data_ptr(),
                               winv=cache.winv.data_ptr(), logdet=cache.logdet.data_ptr(),
                               lu_ws=cache.lu_ws.data_ptr()))
    if items:
        N.mix_prepare(items)


# ------------------------------------------------------------------------------------------- coupling net
class WeightSet:
    """The three packed conv weights of one coupling network in ONE operand format."""

    def __init__(self):
        self.key = None
        self.w1 = self.w2 = self.w3 = None

    def alloc(self, dt: torch.dtype, F: int, K1p: int, ldp: int, dev: torch.device) -> None:
        if self.w1 is None or self.w1.numel() != F * K1p or self.w1.device != dev:
            _bump_epoch()
            self.w1 = torch.empty(F * K1p, dtype=dt, device=dev)
            self.w3 = torch.empty(ldp * F, dtype=dt, device=dev)
            self.w2 = torch.empty(F * F, dtype=dt, device=dev) if dt != torch.float32 else None
            self.key = None


class CouplingCache:
    """GEMM-ready copies of the three conv weights of one coupling network (nfdpm_pack_matrix), one WeightSet per operand
    format: evaluation (split pairs) and training (bf16) alternate in one process without re-allocating — and thereby
    invalidating captured graphs and batched packing plans of — each other's buffers."""

    def __init__(self):
        self.sets = {}
        self.K1 = self.K1p = self.ldp = 0

    def at(self, dt: torch.dtype) -> WeightSet:
        ws = self.sets.get(dt)
        if ws is None:
            ws = self.sets[dt] = WeightSet()
        return ws

    def geometry(self, w1: torch.Tensor, w3: torch.Tensor) -> None:
        self.K1 = w1.shape[1] * 9
        self.K1p = round_up(self.K1, 64)
        self.ldp = round_up(9 * w3.shape[0], 16)


def _pack_coupling(cache: CouplingCache, w1: torch.Tensor, w2: torch.Tensor, w3: torch.Tensor, dt: torch.dtype) -> WeightSet:
    ws = cache.at(dt)
    key = _vkey(w1, w2, w3)
    if cache_hit(ws.key, key):
        return ws
    F, C = w1.shape[0], w3.shape[0]
    cache.geometry(w1, w3)
    K1, K1p, ldp = cache.K1, cache.K1p, cache.ldp
    ws.alloc(dt, F, K1p, ldp, w1.device)
    # conv1 [F, Ch, 3, 3] -> rows n, cols c*9+tap (natural), zero-padded to K1p
    N.pack_matrix(w1, ws.w1, 1, F, K1, 0, K1, 1, K1p, F)
    if dt != torch.float32:
        N.pack_matrix(w2, ws.w2, 1, F, F, 0, F, 1, F, F)
    # zero conv [C, F, 3, 3] -> rows (tap, co), cols ci ("taps as N"); rows 9C..ldp zero
    N.pack_matrix(w3, ws.w3, 9, C, F, 1, F * 9, 9, F, ldp)
    ws.key = key
    return ws


class PackPlan:
    """All weight layouts of all coupling networks of one Glow (forward operands, and the transposed dgrad operands
    when ``train``) refreshed by ONE nfdpm_pack_batch launch whenever a parameter changed — instead of 3 (+4)
    nfdpm_pack_matrix launches per StepFlow."""

    def __init__(self, steps, dt: torch.dtype, train: bool):
        import numpy as np
        from . import _train as T
        self.dt, self.train = dt, train
        self.weights, self.marks, jobs = [], [], []
        self.owners = [(s.affcoupling, s.affcoupling._cache) for s in steps]
        code = {torch.float32: N.F32, torch.bfloat16: N.BF16, N.SPLIT: N.BF16X2}[dt]
        pe = N.pack_elems()
        blocks = 0

        def job(src, out, na, nb, nk, sa, sb, sk, ld, rows, nk2=1, sk2=0, out_code=code):
            nonlocal blocks
            jobs.append([src.data_ptr(), out.data_ptr(), sa, sb, sk, ld, na | (nb << 32), nk | (rows << 32),
                         out_code | (blocks << 32), nk2 | (sk2 << 32)])
            blocks += ((rows + 63) // 64) * ((ld + 63) // 64)

        for s in steps:
            cp = s.affcoupling
            conv1, _, conv2, _, zc = cp._parts()
            w1, w2, w3 = conv1.weight, conv2.weight, zc.weight
            F, Ch, C = w1.shape[0], w1.shape[1], w3.shape[0]
            dev = w1.device
            K1, K1p, ldp, Kp3 = Ch * 9, round_up(Ch * 9, 64), round_up(9 * C, 16), round_up(9 * C, 64)
            cp._cache.geometry(w1, w3)
            c = cp._cache.at(dt)
            c.alloc(dt, F, K1p, ldp, dev)
            job(w1, c.w1, 1, F, K1, 0, K1, 1, K1p, F)
            if dt != torch.float32:
                job(w2, c.w2, 1, F, F, 0, F, 1, F, F)
            job(w3, c.w3, 9, C, F, 1, F * 9, 9, F, ldp)
            caches = [c]
            if train:
                # one set of transposed operands per operand format (like the forward WeightSets)
                b = cp.__dict__.setdefault("_bwd_caches", {}).get(dt)
                if b is None:
                    b = cp._bwd_caches[dt] = T._BwdCache()
                if b.w1t is None or b.w1t.device != dev:
                    b.w1t = torch.empty(K1p * F, dtype=dt, device=dev)
                    b.w2t = torch.empty(F * F, dtype=dt, device=dev)
                    b.w3t = torch.empty(F * Kp3, dtype=dt, device=dev)
                b.Kp3 = Kp3
                job(w1, b.w1t, K1, 1, F, 1, 0, K1, F, K1p)
                job(w2, b.w2t, F, 1, F, 1, 0, F, F, F)
                # w3t[ci, tap*C + co] = W3[co, ci, tap]: two-level column index (tap, co)
                job(w3, b.w3t, F, 1, 9 * C, 9, 0, 1, Kp3, F, nk2=C, sk2=F * 9)
                caches.append(b)
            self.weights += [w1, w2, w3]
            self.marks.append((caches, (w1, w2, w3)))
        self.n_jobs, self.n_blocks = len(jobs), blocks
        self.table = torch.tensor(np.asarray(jobs, dtype=np.int64).reshape(-1), device=self.weights[0].device)
        self.key = None

    def valid(self) -> bool:
        """False once a coupling network started a new cache (its own load_state_dict / .to()): the job table then
        points at orphaned buffers and the plan must be rebuilt."""
        return all(cp._cache is c for cp, c in self.owners)

    def refresh(self) -> None:
        key = _vkey(*self.weights)
        if cache_hit(self.key, key):
            return
        N.pack_batch(self.table, self.n_jobs, self.n_blocks)
        self.key = key
        for caches, ws in self.marks:
            k = _vkey(*ws)
            for c in caches:
                c.key = k


def coupling_a1(cp, B: int, C: int, H: int, W: int, dev: torch.device) -> Tuple[torch.Tensor, int]:
    """The im2col operand buffer of coupling network ``cp`` (filled by nfdpm_flow_boundary / nfdpm_im2col3x3)."""
    conv1, _, conv2, _, zc = cp._parts()
    dt = coupling_dtype()
    _pack_coupling(cp._cache, conv1.weight, conv2.weight, zc.weight, dt)
    K1p = cp._cache.K1p
    return WS.get("A1", B * H * W * K1p, dt, dev), K1p     # (numel counts logical columns: a split pair is one int32)


def coupling_gemms(cp, A1: torch.Tensor, B: int, C: int, H: int, W: int) -> Tuple[torch.Tensor, int]:
    """GEMM1 -> GEMM2 -> GEMM3 of an initialised coupling network from its im2col rows ``A1``.
    Returns the taps-as-N rows (pm, ldp)."""
    conv1, an1, conv2, an2, zc = cp._parts()
    F = conv1.weight.shape[0]
    dt = A1.dtype
    K1p, ldp = cp._cache.K1p, cp._cache.ldp
    cache = cp._cache.at(dt)
    dev = A1.device
    M = B * H * W
    h1 = WS.get("h1", M * F, dt, dev)
    N.gemm_nt(A1, K1p, cache.w1, K1p, h1, F, M, F, K1p, N.EPI_ACTNORM_RELU, an1.scale, an1.bias)
    w2 = cache.w2 if dt != torch.float32 else conv2.weight
    h2 = WS.get("h2", M * F, dt, dev)
    N.gemm_nt(h1, F, w2, F, h2, F, M, F, F, N.EPI_ACTNORM_RELU, an2.scale, an2.bias)
    pm = WS.get("pm", M * ldp, torch.float32, dev)
    N.gemm_nt(h2, F, cache.w3, F, pm, ldp, M, ldp, F)
    return pm, ldp


def fused_g3_ok(B: int, C: int, H: int, W: int, F: int, ldp: int, dt: torch.dtype = torch.bfloat16) -> bool:
    """Use nfdpm_gemm3_boundary?  Measured in situ (tools/bench_levels.py, profiles/): with ONE image per CTA
    (16x16 images: 128 CTAs) it beats GEMM3 + boundary (54.6 vs 61.4 us per StepFlow chain); at the deeper levels a
    128-row tile holds 2..8 images, only 64 / 16 CTAs exist and the separate kernels win — so only H*W == 256 takes it."""
    if dt not in TC_DTYPES or not N.gemm3_boundary_ok(B, C, H, W, F * (2 if dt == N.SPLIT else 1), ldp):
        return False
    return H * W == 256


def coupling_boundary(cp, A1: torch.Tensor, B: int, C: int, H: int, W: int, src, src_bs, ld_part, mt, beta, y, y_bs,
                      a1_next, lda1_next, inverse: bool, pm_out=None, xs=None, tiles: int = 0) -> None:
    """One StepFlow's coupling network + everything up to the next network's first GEMM:
    GEMM1 -> GEMM2 -> [GEMM3 + coupling + next mix + sinks].  In tensor-core mode the bracketed part is ONE kernel
    (nfdpm_gemm3_boundary: the ZeroConv output stays in tensor/shared memory); otherwise GEMM3 and
    nfdpm_flow_boundary run separately."""
    conv1, an1, conv2, an2, zc = cp._parts()
    F = conv1.weight.shape[0]
    dt = A1.dtype
    K1p, ldp = cp._cache.K1p, cp._cache.ldp
    cache = cp._cache.at(dt)
    dev = A1.device
    M = B * H * W
    if tiles > 0:
        # row-band boundary (images beyond one CTA, small batches): GEMM1 -> GEMM2 -> GEMM3, then nfdpm_flow_boundary_tiled
        pm, _ = coupling_gemms(cp, A1, B, C, H, W)
        N.flow_boundary_tiled(src, src_bs, False, pm, ldp, zc.bias, zc.logs, ld_part, mt, beta, y, y_bs, None, 0, a1_next,
                              lda1_next, B, C, H, W, inverse, tiles)
        return
    fused = fused_g3_ok(B, C, H, W, F, ldp, dt)
    if not fused:
        if pm_out is None:
            pm, _ = coupling_gemms(cp, A1, B, C, H, W)
        else:
            raise RuntimeError("coupling_boundary: the training stash path needs the fused kernel or explicit GEMMs")
        if xs is None:
            N.flow_boundary(src, src_bs, False, pm, ldp, zc.bias, zc.logs, ld_part, mt, beta, y, y_bs, a1_next,
                            lda1_next, B, C, H, W, inverse)
        return
    h1 = WS.get("h1", M * F, dt, dev)
    N.gemm_nt(A1, K1p, cache.w1, K1p, h1, F, M, F, K1p, N.EPI_ACTNORM_RELU, an1.scale, an1.bias)
    h2 = WS.get("h2", M * F, dt, dev)
    N.gemm_nt(h1, F, cache.w2, F, h2, F, M, F, F, N.EPI_ACTNORM_RELU, an2.scale, an2.bias)
    N.gemm3_boundary(h2, F, cache.w3, pm_out, ldp if pm_out is not None else 0, src, src_bs, zc.bias, zc.logs, ld_part,
                     mt, beta, y, y_bs, xs, (C * H * W) if xs is not None else 0, a1_next, lda1_next, B, C, H, W, F, ldp,
                     inverse)


#: set by coupling_rows(stash=True): the operands the backward of a stand-alone AffineCoupling needs (normalizing_flow/_modgrad.py)
last_coupling_stash = None


def coupling_rows(cp, y: torch.Tensor, ybs: int, B: int, C: int, H: int, W: int, init: bool = False,
                  stash: bool = False, fmt: Optional[torch.dtype] = None) -> Tuple[torch.Tensor, int]:
    """Run the coupling network of AffineCoupling ``cp`` on the first C/2 channels of ``y`` ([B,C,P], batch
    stride ``ybs``).  Returns (pm, ldp): the taps-as-N ZeroConv rows consumed by nfdpm_coupling_apply.
    ``init`` performs the data-dependent initialisation of inner ActNorms that are not initialised yet
    (always in exact fp32).  ``stash``: the training form — operands in the TRAINING format, in fresh tensors that are
    published as ``last_coupling_stash`` for the module's backward.  ``fmt`` overrides the operand format (the inverse
    keeps the no-grad inference format, see coupling_dtype)."""
    global last_coupling_stash
    conv1, an1, conv2, an2, zc = cp._parts()
    F = conv1.weight.shape[0]
    if F % 64 != 0:
        raise ValueError(f"coupling_net_n_features must be a multiple of 64 (got {F})")
    need_init = init and not (an1._initialized() and an2._initialized())
    if stash and need_init:
        coupling_rows(cp, y, ybs, B, C, H, W, init=True)          # initialise first (exact fp32), then run the stash pass
        need_init = False
    dt = torch.float32 if need_init else (fmt or coupling_dtype(train=stash))   # the data-dependent init runs in exact fp32
    cache = _pack_coupling(cp._cache, conv1.weight, conv2.weight, zc.weight, dt)
    dev = y.device
    M = B * H * W
    K1p, ldp = cp._cache.K1p, cp._cache.ldp

    def buf(tag, numel, dtype):
        return torch.empty(numel, dtype=dtype, device=dev) if stash else WS.get(tag, numel, dtype, dev)
    A1 = buf("A1", M * K1p, dt)
    N.im2col3x3(y, A1, B, C // 2, H, W, ybs, K1p)
    h1 = buf("h1", M * F, dt)
    if need_init and not an1._initialized():
        raw = WS.get("raw", M * F, torch.float32, dev)
        N.gemm_nt(A1, K1p, cache.w1, K1p, raw, F, M, F, K1p)
        channel_stats(raw, 1, B, F, H * W, F, an1.scale, an1.bias)
        an1._mark_initialized()
    N.gemm_nt(A1, K1p, cache.w1, K1p, h1, F, M, F, K1p, N.EPI_ACTNORM_RELU, an1.scale, an1.bias)
    w2 = cache.w2 if dt != torch.float32 else conv2.weight
    h2 = buf("h2", M * F, dt)
    if need_init and not an2._initialized():
        raw = WS.get("raw", M * F, torch.float32, dev)
        N.gemm_nt(h1, F, w2, F, raw, F, M, F, F)
        channel_stats(raw, 1, B, F, H * W, F, an2.scale, an2.bias)
        an2._mark_initialized()
    N.gemm_nt(h1, F, w2, F, h2, F, M, F, F, N.EPI_ACTNORM_RELU, an2.scale, an2.bias)
    pm = buf("pm", M * ldp, torch.float32)
    N.gemm_nt(h2, F, cache.w3, F, pm, ldp, M, ldp, F)
    if stash:
        from types import SimpleNamespace
        last_coupling_stash = SimpleNamespace(A1=A1, h1=h1, h2=h2, pm=pm, dt=dt, K1p=K1p, ldp=ldp)
    return pm, ldp


class SplitCache:
    def __init__(self):
        self.key = None
        self.w = None
        self.Kp = self.ldh = 0


def refresh_split(sp, C: int) -> None:
    """(Re)pack the Split prior's ZeroConv weight if it changed."""
    conv = sp.conv
    if conv is None:
        return
    cache = sp._cache
    w = conv.weight
    K = (C // 2) * 9
    Kp = round_up(K, 16)
    ldh = round_up(C, 8)
    key = _vkey(w)
    if not cache_hit(cache.key, key):
        if cache.w is None or cache.w.numel() != ldh * Kp:
            _bump_epoch()
            cache.w = torch.empty(ldh * Kp, dtype=torch.float32, device=w.device)
        N.pack_matrix(w, cache.w, 1, C, K, 0, K, 1, Kp, ldh)
        cache.key, cache.Kp, cache.ldh = key, Kp, ldh


def split_rows(sp, y: torch.Tensor, ybs: int, B: int, C: int, H: int, W: int) -> Tuple[Optional[torch.Tensor], int]:
    """Raw ZeroConv3x3 (C/2 -> C) rows of the Split prior, always exact fp32 (the conv is tiny).
    Returns (h, ldh) or (None, 0) when the prior is not learned."""
    if sp.conv is None:
        return None, 0
    refresh_split(sp, C)
    cache = sp._cache
    Kp, ldh = cache.Kp, cache.ldh
    M = B * H * W
    A = WS.get("As", M * Kp, torch.float32, y.device)
    N.im2col3x3(y, A, B, C // 2, H, W, ybs, Kp)
    h = WS.get("hs", M * ldh, torch.float32, y.device)
    N.gemm_nt(A, Kp, cache.w, Kp, h, ldh, M, C, Kp)
    return h, ldh


def conv3x3_rows(conv, x: torch.Tensor, xbs: int, B: int, Cin: int, Cout: int, H: int, W: int) -> Tuple[torch.Tensor, int]:
    """Exact-fp32 3x3 "same" convolution of the first ``Cin`` channels of x as im2col + GEMM.  Returns the raw
    rows [M, ld] (no bias).  Used by the stand-alone ZeroConv2d / Conv2dActNorm module calls."""
    K, Kp, ld = Cin * 9, round_up(Cin * 9, 16), round_up(Cout, 8)
    wp = WS.get("wp", ld * Kp, torch.float32, x.device)
    N.pack_matrix(conv.weight, wp, 1, Cout, K, 0, K, 1, Kp, ld)
    M = B * H * W
    A = WS.get("As", M * Kp, torch.float32, x.device)
    N.im2col3x3(x, A, B, Cin, H, W, xbs, Kp)
    h = WS.get("hs", M * ld, torch.float32, x.device)
    N.gemm_nt(A, Kp, wp, Kp, h, ld, M, Cout, Kp)
    return h, ld
