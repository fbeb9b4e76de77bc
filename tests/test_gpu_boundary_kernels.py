"""The step-boundary kernels of the forward, inverse and sampling paths (csrc/flow_boundary.cu + boundary_body.cuh,
flow_boundary_tiled.cu, gemm3_boundary.cu), every entry point against one fp64 restatement of the reference's arithmetic
(``boundary_ref``), at the dispatch branches each kernel has.

Every output is a guarded sink (kernel_refs.Sink): sentinel-filled with slack on both sides; the NCHW state and the
pre-mix stash are strided into wider tensors whose gaps must stay bit-identical; the im2col rows have padding columns
that must be exactly zero; the pm copy has columns past ldp that must stay untouched.  Tolerances are those of
kernel_refs (fp32 rule, one bf16 ulp, split pairs decoded then the fp32 rule).  Wherever a kernel writes both the state
and the im2col rows, the rows must also be bit-identical to the im2col gather of the kernel's own state (its RN bf16
rounding, or its split-pair encoding).

Each parametrised case asserts, through the Python replicas of the host dispatch below, the branch it claims to cover;
the unmarked tests check the replicas against the library's own host queries and the restatement against the CPU
oracle.  The replicas assume the default band tuning (NFDPM_TILE_PIX 256, NFDPM_TILE_CTAS 112)."""
import os

import pytest
import torch
import torch.nn.functional as F

from normalizing_flow import _native as N
from oracle import glow_oracle as O
import split_pairs as SP
from kernel_refs import (DEV, WORST, Sink, check, check_bf16, gather_taps, im2col_rows, report_worst, rnd, same_bits)

gpu = pytest.mark.gpu
pytestmark = pytest.mark.skipif(bool(os.environ.get("NFDPM_TILE_PIX") or os.environ.get("NFDPM_TILE_CTAS")),
                                reason="the band replicas assume the default NFDPM_TILE_PIX / NFDPM_TILE_CTAS")
CAP = 200 * 1024                  # shared-memory budget of flow_boundary / flow_boundary_tiled
_FMT = {"f32": torch.float32, "bf16": torch.bfloat16, "split": N.SPLIT}


@pytest.fixture(autouse=True)
def _report_worst(request):
    """Prints the worst value of each measure a test took (pytest -s)."""
    WORST.clear()
    yield
    report_worst(request.node.name)


@pytest.fixture(scope="module", autouse=True)
def _report_device():
    if torch.cuda.is_available():
        print(f"\n[device] {torch.cuda.get_device_name()}")


# ------------------------------------------------------------------------------------------------ fp64 restatement
def boundary_ref(x, C, H, W, squeeze_in=False, pm=None, bias3=None, logs3=None, inverse=False, mt=None, beta=None,
                 R=None):
    """One step boundary in fp64.  Source: x [B, C, H, W], or with ``squeeze_in`` the [B, C/4, 2H, 2W] map that
    O.squeeze2x2 turns into it.  Coupling (pm given): net = (gather_taps(pm) + bias3) exp(3 logs3), (log_s, t) its
    halves, s = sigmoid(log_s + 2); forward (x_a, (x_b + t) s), inverse (x_a, x_b / (s + 1e-6) - t); log-det
    sum log(s + 1e-6) per image, or with ``R`` per band of R rows ([T, B], band t = rows [tR, min(H, (t+1)R))).  Mix
    (mt given): u[o] = sum_i mt[i, o] x[i] + beta[o].  Returns xs (pre-mix), y = u, a1 = im2col_rows(u[:, :C/2]), ld,
    log_s."""
    x = x.double()
    if squeeze_in:
        x = O.squeeze2x2(x)
    B = x.shape[0]
    x = x.reshape(B, C, H, W)
    ld = log_s = None
    if pm is not None:
        net = (gather_taps(pm.double(), B, C, H, W) + bias3.double().view(1, C, 1, 1)) * \
            torch.exp(3 * logs3.double().view(1, C, 1, 1))
        log_s, t = net.chunk(2, 1)
        s = torch.sigmoid(log_s + 2)
        xa, xb = x.chunk(2, 1)
        x = torch.cat([xa, xb / (s + 1e-6) - t if inverse else (xb + t) * s], 1)
        terms = torch.log(s + 1e-6)
        if R is None:
            ld = terms.reshape(B, -1).sum(1)
        else:
            ld = torch.stack([terms[:, :, r0:r0 + R].reshape(B, -1).sum(1) for r0 in range(0, H, R)])
    u = x if mt is None else \
        torch.einsum("io,bihw->bohw", mt.double().reshape(C, C), x) + beta.double().view(1, C, 1, 1)
    return {"xs": x, "y": u, "a1": im2col_rows(u[:, :C // 2]), "ld": ld, "log_s": log_s}


# ------------------------------------------------------------------------------------------------ CPU: restatement
def _oracle_setup(B, C, H, W, seed):
    """pm of a random ZeroConv, the net it stands for, and one (ActNorm, InvConv2d) pair, all fp64."""
    Cin = C // 2
    h, w3 = rnd(B, Cin, H, W, seed=seed).double(), rnd(C, Cin, 3, 3, seed=seed + 1, scale=0.3).double()
    bias3, logs3 = rnd(C, seed=seed + 2, scale=0.3).double(), rnd(C, seed=seed + 3, scale=0.2).double()
    pm = torch.einsum("bihw,oiyx->bhwyxo", h, w3).reshape(B * H * W, 9 * C)
    pm = torch.cat([pm, torch.full((B * H * W, 3), 1e3, dtype=torch.float64)], 1)    # padding columns are not read
    net = O.zeroconv(h, w3, bias3, logs3.view(1, C, 1, 1))
    wq = torch.linalg.qr(rnd(C, C, seed=seed + 4).double())[0] + 0.1 * rnd(C, C, seed=seed + 5).double()
    s, b = rnd(C, seed=seed + 6, scale=0.3).double(), rnd(C, seed=seed + 7, scale=0.3).double()
    return pm, bias3, logs3, net, wq, s, b


def test_restatement_forward_is_coupling_then_actnorm_invconv(monkeypatch):
    B, C, H, W = 2, 8, 5, 7
    pm, bias3, logs3, net, wq, s, b = _oracle_setup(B, C, H, W, 10)
    monkeypatch.setattr(O, "coupling_net", lambda x_a, sd, pre, init=False: net)
    src = rnd(B, C // 4, 2 * H, 2 * W, seed=1).double()
    x = O.squeeze2x2(src)
    y1, ld1 = O.coupling_fwd(x, {}, "")
    y2 = O.actnorm_fwd(y1, s.view(C, 1, 1), b.view(C, 1, 1))[0]
    y3 = O.invconv_fwd(y2, wq.view(C, C, 1, 1))[0]
    mt = (wq * torch.exp(s)[None, :]).T                 # [i, o], as nfdpm_mix_prepare builds fwd_mt
    beta = mt.T @ b
    for squeeze in (False, True):
        r = boundary_ref(src if squeeze else x, C, H, W, squeeze, pm, bias3, logs3, False, mt, beta)
        assert torch.allclose(r["xs"], y1, rtol=0, atol=1e-12)
        assert torch.allclose(r["y"], y3, rtol=0, atol=1e-12)
        assert torch.allclose(r["ld"], ld1, rtol=1e-13, atol=0)
        assert torch.equal(r["a1"], im2col_rows(r["y"][:, :C // 2]))
    for R in (1, 2, 3, 5, 7):                             # bands, the last one ragged or clamped to H
        bands = boundary_ref(x, C, H, W, False, pm, bias3, logs3, False, R=R)["ld"]
        assert bands.shape == (-(-H // R), B) and torch.allclose(bands.sum(0), ld1, rtol=1e-13, atol=0)
    assert torch.equal(boundary_ref(x, C, H, W)["y"], x)  # no coupling, no mix: the source itself


def test_restatement_inverse_is_coupling_inv_then_invconv_inv_actnorm_inv(monkeypatch):
    B, C, H, W = 2, 6, 4, 3
    pm, bias3, logs3, net, wq, s, b = _oracle_setup(B, C, H, W, 20)
    monkeypatch.setattr(O, "coupling_net", lambda x_a, sd, pre, init=False: net)
    y = rnd(B, C, H, W, seed=2).double()
    x1 = O.coupling_inv(y, {}, "")
    x2 = O.invconv_inv(x1, wq.view(C, C, 1, 1))
    x3 = O.actnorm_inv(x2, s.view(C, 1, 1), b.view(C, 1, 1))
    inv_mt = (torch.exp(-s)[:, None] * torch.linalg.inv(wq)).T     # [i, o] = exp(-s[o]) W^-1[o, i]
    inv_beta = -b
    r = boundary_ref(y, C, H, W, False, pm, bias3, logs3, True, inv_mt, inv_beta)
    assert torch.allclose(r["xs"], x1, rtol=0, atol=1e-12)
    assert torch.allclose(r["y"], x3, rtol=0, atol=1e-12)
    # the inverse's log-det partial is the forward's term of the same s (x_a passes through unchanged)
    assert torch.allclose(r["ld"], O.coupling_fwd(x1, {}, "")[1], rtol=1e-13, atol=0)


# ------------------------------------------------------------------------------------------------ dispatch replicas
def _fb_smem(C, H, W, coupling, mix):
    """boundary_scratch_floats (boundary_body.cuh) in bytes: nfdpm_flow_boundary_smem."""
    P, Cp, Ch = H * W, (C + 3) & ~3, C // 2
    fl = C * (P + 1) * (2 if mix else 1)
    if mix:
        fl += C * Cp + Cp
    if coupling:
        fl += 2 * C + P * Ch
    fl = (fl + 3) & ~3
    fl += (Ch * (H + 2) * (W + 2) + 3) & ~3
    fl += (9 * Ch + 3) & ~3
    return 4 * fl


def _fb_threads(C, H, W, lda1):
    """flow_boundary_impl: one thread per item of the largest phase, rounded to warps, clamped to [128, 1024]."""
    items = max(H * W * (C // 2), H * W * (lda1 // 8) if lda1 else 0)
    return min(1024, max(128, (items + 31) // 32 * 32))


def _fb_bulk(C, H, W, ldp, mix, aligned):
    """flow_boundary_impl's PM_BULK: the image's pm block is bulk-copied into shared memory when ldp % 4 == 0, pm is
    16-byte aligned and the block fits next to the scratch in 200 KB."""
    return aligned and ldp % 4 == 0 and _fb_smem(C, H, W, True, mix) + 4 * H * W * ldp <= CAP


def _fb_tails(C, H, W, lda1, squeeze, coupling, mix):
    """Phase-0 loops of boundary_body.cuh past the first four items per thread: the state (C*P > 4 threads), the mix
    matrix (C*Cp > 4 threads) and the per-channel parameters (beta: Cp > threads, bias3 / logs3: C > threads)."""
    nt, Cp = _fb_threads(C, H, W, lda1), (C + 3) & ~3
    tails = set()
    if not squeeze and C * H * W > 4 * nt:
        tails.add("state")
    if mix and C * Cp > 4 * nt:
        tails.add("matrix")
    if (mix and Cp > nt) or (coupling and C > nt):
        tails.add("param")
    return tails


def _tiled_smem(C, W, R, halo, coupling, mix):
    """tiled_scratch_floats (flow_boundary_tiled.cu) in bytes."""
    Pv, Cp, Ch = (R + 2 * halo) * W, (C + 3) & ~3, C // 2
    fl = C * (Pv + 1) * (2 if mix else 1)
    if mix:
        fl += C * Cp + Cp
    if coupling:
        fl += 2 * C + R * W * Ch
    fl = (fl + 3) & ~3
    if halo:
        fl += (Ch * (R + 2) * (W + 2) + 3) & ~3
        fl += (9 * Ch + 3) & ~3
    return 4 * fl


def _rows(B, C, H, W, coupling, mix, a1):
    """choose_rows, step by step: (R from 256 pixels per band clamped to [1, H], after the 112-CTA rule, after the
    shared-memory rule)."""
    R0 = min(max(256 // W, 1), H)
    R1 = R0
    while R1 > 1 and B * -(-H // R1) < 112:
        R1 -= 1
    R = R1
    while R > 1 and _tiled_smem(C, W, R, int(a1), coupling, mix) > CAP:
        R -= 1
    return R0, R1, R


def _tiles(B, C, H, W, coupling, mix, a1):
    """nfdpm_flow_boundary_tiles: ceil(H / R), or 0 when even one row does not fit."""
    R = _rows(B, C, H, W, coupling, mix, a1)[2]
    return 0 if _tiled_smem(C, W, R, int(a1), coupling, mix) > CAP else -(-H // R)


def _bulk_m(C, mix, aligned):
    """TileGeom::bulk_m: the mix matrix and beta arrive by bulk copy when C % 4 == 0 and both are 16-byte aligned."""
    return mix and C % 4 == 0 and aligned


def _g3_plan(B, C, H, W, K, ldp, mix):
    """g3_plan (gemm3_boundary.cu): None when unsupported, else images per CTA, images per pm pass, pipeline stages."""
    P = H * W
    if C % 2 or K % 64 or ldp % 16 or ldp < 9 * C or ldp > 512:
        return None
    if P == 256:
        ipc = 1
    elif P <= 128 and 128 % P == 0:
        ipc = 128 // P
    else:
        return None
    rows = ipc * P
    if rows > 128 and ldp > 256:
        return None
    a_bytes = 32768 if rows > 128 else 16384
    n_bbox = 2 if ldp > 256 else 1
    if (ldp // n_bbox) % 8:
        return None
    stage = a_bytes + ldp * 128
    lds = ldp + 4
    ipp = ipc
    while ipp > 1 and ipp * P * lds * 4 > 122880:
        ipp = (ipp + 1) // 2
    if (ipp * P) % 32 and ipp != ipc:
        return None
    if ipp > 16 or ipp * P * lds * 4 > 122880:
        return None
    pm_bytes = ipp * P * lds * 4
    Cp, Ch = (C + 3) & ~3, C // 2
    body = 4 * (ipc * C * (P + 1) * (2 if mix else 1) + (C * Cp + Cp if mix else 0) + 2 * C + ipp * P * Ch)
    pad = 4 * (((ipc * Ch * (H + 2) * (W + 2) + 3) & ~3) + 9 * Ch)
    stages = 3
    while stages > 2 and 1024 + max(stages * stage, pm_bytes) + body > 224 * 1024:
        stages -= 1
    region = (max(stages * stage, pm_bytes, pad) + 15) & ~15
    if 1024 + region + body > 224 * 1024:
        return None
    return {"ipc": ipc, "ipp": ipp, "stages": stages, "passes": -(-ipc // ipp), "m_tiles": 2 if rows > 128 else 1}


_SHAPES = [(C, H, W) for C in (2, 4, 6, 8, 12, 24, 48, 96, 192) for H, W in
           ((1, 1), (2, 2), (1, 16), (16, 1), (5, 7), (4, 4), (8, 8), (14, 14), (16, 16), (32, 32), (3, 300), (64, 64))]


def test_replica_flow_boundary_smem():
    for C, H, W in _SHAPES:
        for cp in (0, 1):
            for mx in (0, 1):
                assert N.flow_boundary_smem(C, H, W, cp, mx) == _fb_smem(C, H, W, cp, mx), (C, H, W, cp, mx)


def test_replica_tiles():
    for C, H, W in _SHAPES:
        for B in (1, 2, 3, 8, 28, 40, 64, 120):
            for cp, mx, a1 in ((1, 1, 1), (1, 1, 0), (1, 0, 0), (0, 1, 1), (0, 0, 1), (1, 0, 1)):
                assert N.flow_boundary_tiles(B, C, H, W, cp, mx, a1) == _tiles(B, C, H, W, cp, mx, a1), \
                    (B, C, H, W, cp, mx, a1)


def test_replica_gemm3_plan():
    n = 0
    for C in (2, 4, 6, 8, 12, 14, 24, 48, 56):
        for H, W in ((16, 16), (8, 8), (4, 4), (4, 2), (2, 4), (2, 2), (1, 1), (14, 14), (8, 16), (32, 32), (5, 5)):
            for K in (256, 512, 1024, 100):
                for ldp in {(9 * C + 15) // 16 * 16, 9 * C, 9 * C + 16, 512}:
                    got = N.gemm3_boundary_ok(3, C, H, W, K, ldp)
                    assert got == (_g3_plan(3, C, H, W, K, ldp, True) is not None), (C, H, W, K, ldp)
                    n += got
    assert n > 50
    assert _g3_plan(3, 48, 4, 4, 512, 432, True)["stages"] == 2 and _g3_plan(3, 12, 16, 16, 512, 112, True)["stages"] == 3


# ------------------------------------------------------------------------------------------------ GPU plumbing
def _lda1(C, fmt):
    """An im2col leading dimension with padding columns past 9*C/2 (a multiple of 8, of 32 for split pairs)."""
    m = 32 if fmt == "split" else 8
    return (9 * (C // 2) + m - 1) // m * m + m


def _ldp(C):
    return (9 * C + 15) // 16 * 16


class Case:
    """Host inputs of one boundary and the device buffers holding them (source strided into a wider tensor)."""

    def __init__(self, B, C, H, W, seed=0, squeeze=False, coupling=True, mix=True, wide=False, pm_aligned=True,
                 mt_aligned=True, pm=None):
        self.B, self.C, self.H, self.W = B, C, H, W
        P = H * W
        self.P, self.M, self.Ch = P, B * P, C // 2
        self.squeeze = squeeze
        if squeeze:     # the first C/4 channels of a [B, C/4 + 2, 2H, 2W] map (Glow entering a level after a Split)
            cw = C // 4 + 2
            self.in_bs = cw * 4 * P
            full = rnd(B, cw, 2 * H, 2 * W, seed=seed)
            self.x = full[:, :C // 4]
        else:
            self.in_bs = C * P + 6
            full = rnd(B, self.in_bs, seed=seed)
            self.x = full[:, :C * P].reshape(B, C, H, W)
        self.src_host = full.reshape(-1)
        self.src = self.src_host.to(DEV)
        self.ldp = _ldp(C)
        self.pm = self.bias3 = self.logs3 = self.pm_dev = None
        if coupling:
            if pm is None:      # (a given pm is the fp64 product of gemm3_boundary's operands: no device copy)
                pm = rnd(self.M, self.ldp, seed=seed + 1, scale=1.4 if wide else 0.1)
                self.pm_dev = pm.to(DEV) if pm_aligned else _misaligned(pm)
            self.pm = pm
            self.bias3, self.logs3 = rnd(C, seed=seed + 2, scale=0.1), rnd(C, seed=seed + 3, scale=0.1)
            if wide:    # log_s ~ N(-4, 4.2): s = sigmoid(log_s + 2) from below 1e-6 (the +1e-6 matters) to ~1
                self.bias3[:self.Ch] = -4.0
                self.logs3.zero_()
        self.mt = self.beta = self.mt_dev = self.beta_dev = None
        if mix:
            self.mt, self.beta = rnd(C, C, seed=seed + 4, scale=1.2 / C ** 0.5), rnd(C, seed=seed + 5, scale=0.5)
            self.mt_dev = self.mt.to(DEV) if mt_aligned else _misaligned(self.mt)
            self.beta_dev = self.beta.to(DEV)
        self.dev = [None if t is None else t.to(DEV) for t in (self.bias3, self.logs3)]

    def ref(self, inverse, R=None, on_device=False):
        d = DEV if on_device else "cpu"
        mv = lambda t: None if t is None else t.to(d)
        r = boundary_ref(mv(self.x), self.C, self.H, self.W, self.squeeze, mv(self.pm), mv(self.bias3), mv(self.logs3),
                         inverse, mv(self.mt), mv(self.beta), R)
        return {k: (None if v is None else v.cpu()) for k, v in r.items()}


def _misaligned(t):
    """A device copy of t whose pointer is 4 bytes past a 16-byte boundary."""
    buf = torch.empty(t.numel() + 4, device=DEV)
    v = buf[1:1 + t.numel()]
    v.copy_(t.reshape(-1).to(DEV))
    assert v.data_ptr() % 16 == 4
    return v


class Sinks:
    """The guarded outputs of one launch: y and xs strided (image stride C*P + gap), a1 with padding columns, ld."""

    def __init__(self, cs, want, fmt="f32", ld_rows=0, src_sink=None):
        B, C, P = cs.B, cs.C, cs.P
        self.cs, self.fmt = cs, fmt
        self.y = self.xs = self.a1 = self.ld = None
        self.y_bs = self.xs_bs = self.lda1 = 0
        if "y" in want:
            if src_sink is not None:                       # in place: y aliases the (strided) source
                self.y, self.y_bs = src_sink, cs.in_bs
            else:
                self.y_bs = C * P + 10
                self.y = Sink(B * self.y_bs)
        if "xs" in want:
            self.xs_bs = C * P + 14
            self.xs = Sink(B * self.xs_bs)
        if "a1" in want:
            self.lda1 = _lda1(C, fmt)
            self.a1 = Sink(cs.M * self.lda1, _FMT[fmt])
        if ld_rows:
            self.ld = Sink(ld_rows * B)

    def t(self, name):
        s = getattr(self, name)
        return None if s is None else s.t


def _strided(sink, B, bs, n):
    """The first n elements of each image of a sink with image stride bs; the gaps must be untouched."""
    return sink.get((torch.arange(bs) < n).expand(B, bs)).view(B, bs)[:, :n]


def _verify(sk, ref):
    """Every sink of sk against the restatement, and the im2col rows against the kernel's own state."""
    cs = sk.cs
    B, C, H, W, P, M, Ch = cs.B, cs.C, cs.H, cs.W, cs.P, cs.M, cs.Ch
    y = None
    if sk.y is not None:
        y = _strided(sk.y, B, sk.y_bs, C * P).reshape(B, C, H, W)
        check("y", y, ref["y"])
    if sk.xs is not None:
        check("xs", _strided(sk.xs, B, sk.xs_bs, C * P), ref["xs"].reshape(B, C * P))
    if sk.a1 is not None:
        K, ld = 9 * Ch, sk.lda1
        words = sk.a1.get().view(M, ld)
        val = SP.value(words, M, ld) if sk.fmt == "split" else words.double()
        assert float(val[:, K:].abs().max()) == 0.0, "a1 padding columns are not zero"          # (NaN fails too)
        (check_bf16 if sk.fmt == "bf16" else check)("a1", val[:, :K], ref["a1"])
        if y is not None:
            im = F.pad(im2col_rows(y[:, :Ch].float()), (0, ld - K))
            want = SP.encode(im) if sk.fmt == "split" else im.to(_FMT[sk.fmt])
            assert same_bits(words, want), "a1 is not the im2col gather of the kernel's own y"
    if sk.ld is not None:
        check("ld_part", sk.ld.get(), ref["ld"])


# ------------------------------------------------------------------------------------------------ flow_boundary
# (id, entry, B, C, H, W, source, pm staging ("none" / "bulk" / "global" / "unaligned"), mix, sinks, inverse, ld,
#  in place, phase-0 tails, a1 formats, wide-range log_s)
_FB = [
    ("level_entry_squeeze", "fb", 3, 12, 16, 16, "squeeze", "none", True, "y a1", False, False, False, set(),
     ("f32", "bf16", "split"), False),
    ("im2col_only", "fb", 3, 12, 8, 8, "plain", "none", False, "a1", False, False, False, set(),
     ("f32", "bf16", "split"), False),
    ("entry_stash_squeeze", "stash", 2, 8, 5, 7, "squeeze", "none", True, "y xs a1", False, False, False, set(),
     ("f32",), False),
    ("bulk_in_place", "fb", 3, 12, 16, 16, "plain", "bulk", True, "y a1", False, True, True, set(),
     ("f32", "bf16", "split"), False),
    ("global_c24", "fb", 2, 24, 16, 16, "plain", "global", True, "y a1", False, True, False, {"state"},
     ("f32", "bf16"), False),
    ("unaligned_pm_5x7", "fb", 3, 6, 5, 7, "plain", "unaligned", True, "y a1", False, True, False, set(),
     ("f32", "split"), False),
    ("last_step_no_mix", "fb", 3, 12, 16, 16, "plain", "bulk", False, "y", False, True, False, set(), ("f32",), False),
    ("coupling_no_mix_a1", "stash", 2, 12, 8, 8, "plain", "bulk", False, "y xs a1", False, True, False, set(),
     ("bf16",), False),
    ("state_tail_c48", "stash", 2, 48, 16, 16, "plain", "global", True, "y xs", False, True, False, {"state"},
     ("f32",), False),
    ("matrix_tail_c48_2x2", "stash", 3, 48, 2, 2, "plain", "bulk", True, "y xs a1", False, True, False, {"matrix"},
     ("f32", "split"), False),
    ("param_tail_c192_1x1", "fb", 3, 192, 1, 1, "plain", "bulk", True, "y a1", False, True, False,
     {"matrix", "param"}, ("f32", "bf16"), False),
    ("row_1x16_inverse", "fb", 2, 8, 1, 16, "plain", "bulk", True, "y a1", True, True, False, set(), ("f32",), False),
    ("col_16x1", "stash", 2, 8, 16, 1, "plain", "bulk", True, "y xs a1", False, True, False, set(), ("f32",), False),
    ("inverse_in_place_no_ld", "fb", 3, 12, 16, 16, "plain", "bulk", True, "y a1", True, False, True, set(),
     ("f32", "split"), False),
    ("inv_stash", "inv_stash", 3, 12, 16, 16, "plain", "bulk", True, "y xs a1", True, False, False, set(),
     ("f32", "bf16", "split"), False),
    ("inv_stash_ld", "inv_stash_ld", 3, 24, 8, 8, "plain", "bulk", True, "y xs a1", True, True, False, set(),
     ("f32", "split"), False),
    ("inv_stash_ld_last", "inv_stash_ld", 2, 6, 5, 7, "plain", "unaligned", True, "y xs", True, True, False, set(),
     ("f32",), False),
    ("inv_stash_ld_null", "inv_stash_ld", 2, 24, 16, 16, "plain", "global", True, "y xs a1", True, False, False,
     {"state"}, ("f32",), False),
    ("wide_forward", "stash", 3, 12, 16, 16, "plain", "bulk", True, "y xs a1", False, True, False, set(), ("f32",),
     True),
    ("wide_inverse", "inv_stash_ld", 3, 12, 16, 16, "plain", "bulk", True, "y xs a1", True, True, False, set(),
     ("f32",), True),
]


def _check_wide(ref):
    ls = ref["log_s"]
    s = torch.sigmoid(ls + 2)
    assert float(s.min()) < 2e-6 and float(s.max()) > 0.9999, (float(ls.min()), float(ls.max()))


@gpu
@pytest.mark.parametrize("case,entry,B,C,H,W,source,staging,mix,sinks,inverse,with_ld,in_place,tails,fmt,wide", [
    pytest.param(*c[:14], f, c[15], id=f"{c[0]}-{f}") for c in _FB for f in c[14]])
def test_flow_boundary(case, entry, B, C, H, W, source, staging, mix, sinks, inverse, with_ld, in_place, tails, fmt,
                       wide):
    coupling = staging != "none"
    want = set(sinks.split())
    cs = Case(B, C, H, W, seed=len(case), squeeze=source == "squeeze", coupling=coupling, mix=mix, wide=wide,
              pm_aligned=staging != "unaligned")
    lda1 = _lda1(C, fmt) if "a1" in want else 0
    assert _fb_smem(C, H, W, coupling, mix) <= CAP
    if coupling:
        assert _fb_bulk(C, H, W, cs.ldp, mix, cs.pm_dev.data_ptr() % 16 == 0) == (staging == "bulk")
    assert _fb_tails(C, H, W, lda1, cs.squeeze, coupling, mix) == tails
    src_sink = Sink(cs.src_host.numel(), init=cs.src_host) if in_place else None
    src = src_sink.t if in_place else cs.src
    sk = Sinks(cs, want, fmt, 1 if with_ld else 0, src_sink)
    b3, l3 = cs.dev
    common = (cs.pm_dev, cs.ldp, b3, l3)
    if entry == "fb":
        assert "xs" not in want
        N.flow_boundary(src, cs.in_bs, cs.squeeze, *common, sk.t("ld"), cs.mt_dev, cs.beta_dev, sk.t("y"), sk.y_bs,
                        sk.t("a1"), lda1, B, C, H, W, inverse)
    elif entry == "stash":
        assert not inverse
        N.flow_boundary_stash(src, cs.in_bs, cs.squeeze, *common, sk.t("ld"), cs.mt_dev, cs.beta_dev, sk.t("y"),
                              sk.y_bs, sk.t("xs"), sk.xs_bs, sk.t("a1"), lda1, B, C, H, W)
    elif entry == "inv_stash":
        assert inverse and not with_ld
        N.flow_boundary_inv_stash(src, cs.in_bs, *common, cs.mt_dev, cs.beta_dev, sk.t("y"), sk.y_bs, sk.t("xs"),
                                  sk.xs_bs, sk.t("a1"), lda1, B, C, H, W)
    else:
        assert inverse
        N.flow_boundary_inv_stash_ld(src, cs.in_bs, *common, sk.t("ld"), cs.mt_dev, cs.beta_dev, sk.t("y"), sk.y_bs,
                                     sk.t("xs"), sk.xs_bs, sk.t("a1"), lda1, B, C, H, W)
    torch.cuda.synchronize()
    ref = cs.ref(inverse)
    if wide:
        _check_wide(ref)
    _verify(sk, ref)


# ------------------------------------------------------------------------------------------------ flow_boundary_tiled
# (id, B, C, H, W, source, coupling, mix, sinks, inverse, ld, mt aligned, expected (R, T, R-rule), a1 formats, wide)
# R-rule: "pixels" (256 / W unchanged), "ctas" (lowered by the 112-CTA rule), "smem" (lowered by shared memory),
# "clamp" (256 / W > H: T = 1), "wide_row" (W > 256: R = 1)
_TILED = [
    ("r256w_t4", 64, 12, 32, 32, "plain", True, True, "y a1", False, True, True, (8, 4, "pixels"), ("f32", "bf16"),
     False),
    ("cta_rule_r1", 2, 12, 32, 32, "plain", True, True, "y a1", False, True, True, (1, 32, "ctas"),
     ("f32", "bf16", "split"), False),
    ("smem_c96_a1", 28, 96, 32, 32, "plain", True, True, "y a1", False, True, True, (2, 16, "smem"), ("bf16",), False),
    ("smem_c96_ragged", 28, 96, 32, 32, "plain", True, True, "y", False, True, True, (5, 7, "smem"), ("f32",), False),
    ("mnist_b40_ragged", 40, 4, 14, 14, "plain", True, True, "y a1", False, True, True, (6, 3, "ctas"),
     ("f32", "split"), False),
    ("c192_ragged_inverse", 64, 192, 8, 8, "plain", True, True, "y xs", True, True, True, (3, 3, "smem"), ("f32",),
     False),
    ("clamp_t1_c6", 120, 6, 5, 7, "plain", True, True, "y a1", False, True, False, (5, 1, "clamp"), ("f32",), False),
    ("wide_row_c2", 2, 2, 3, 300, "plain", True, True, "y a1", False, True, False, (1, 3, "wide_row"), ("f32", "bf16"),
     False),
    ("entry_squeeze", 2, 12, 32, 32, "squeeze", False, True, "y a1", False, False, True, (1, 32, "ctas"),
     ("f32", "split"), False),
    ("entry_squeeze_t1", 120, 8, 4, 4, "squeeze", False, True, "y a1", False, False, True, (4, 1, "clamp"), ("f32",),
     False),
    ("im2col_only", 2, 12, 32, 32, "plain", False, False, "a1", False, False, True, (1, 32, "ctas"), ("f32", "bf16"),
     False),
    ("inverse_recorded", 2, 12, 32, 32, "plain", True, True, "y xs a1", True, True, True, (1, 32, "ctas"),
     ("f32", "split"), False),
    ("inverse_ld_null", 16, 12, 16, 16, "plain", True, True, "y xs", True, False, True, (2, 8, "ctas"), ("f32",), False),
    ("forward_ld_null", 8, 24, 16, 16, "plain", True, True, "y a1", False, False, True, (1, 16, "ctas"), ("f32",),
     False),
    ("mt_unaligned", 4, 12, 32, 32, "plain", True, True, "y a1", False, True, False, (1, 32, "ctas"), ("f32",), False),
    ("no_mix", 4, 12, 32, 32, "plain", True, False, "y a1", False, True, True, (1, 32, "ctas"), ("f32",), False),
    ("wide_forward", 64, 12, 32, 32, "plain", True, True, "y a1", False, True, True, (8, 4, "pixels"), ("f32",), True),
    ("wide_inverse", 40, 4, 14, 14, "plain", True, True, "y xs a1", True, True, True, (6, 3, "ctas"), ("f32",), True),
]


@gpu
@pytest.mark.parametrize("case,B,C,H,W,source,coupling,mix,sinks,inverse,with_ld,mt_aligned,expect,fmt,wide", [
    pytest.param(*c[:13], f, c[14], id=f"{c[0]}-{f}") for c in _TILED for f in c[13]])
def test_flow_boundary_tiled(case, B, C, H, W, source, coupling, mix, sinks, inverse, with_ld, mt_aligned, expect, fmt,
                             wide):
    want = set(sinks.split())
    a1 = "a1" in want
    R_want, T_want, rule = expect
    R0, R1, R = _rows(B, C, H, W, coupling, mix, a1)
    T = N.flow_boundary_tiles(B, C, H, W, coupling, mix, a1)
    assert (R, T) == (R_want, T_want) == (R, _tiles(B, C, H, W, coupling, mix, a1))
    assert {"pixels": R0 == R1 == R == 256 // W, "ctas": R0 > R1 == R, "smem": R1 > R,
            "clamp": 256 // W > H and R == H, "wide_row": W > 256 and R == 1}[rule]
    cs = Case(B, C, H, W, seed=len(case) + 7, squeeze=source == "squeeze", coupling=coupling, mix=mix, wide=wide,
              mt_aligned=mt_aligned)
    if mix:
        assert _bulk_m(C, mix, cs.mt_dev.data_ptr() % 16 == 0 and cs.beta_dev.data_ptr() % 16 == 0) == \
            (C % 4 == 0 and mt_aligned)
    sk = Sinks(cs, want, fmt, T if with_ld else 0)
    b3, l3 = cs.dev
    N.flow_boundary_tiled(cs.src, cs.in_bs, cs.squeeze, cs.pm_dev, cs.ldp, b3, l3, sk.t("ld"), cs.mt_dev, cs.beta_dev,
                          sk.t("y"), sk.y_bs, sk.t("xs"), sk.xs_bs, sk.t("a1"), sk.lda1, B, C, H, W, inverse, T)
    torch.cuda.synchronize()
    ref = cs.ref(inverse, R=R, on_device=B * C * H * W > 1 << 20)
    if wide:
        _check_wide(ref)
    _verify(sk, ref)


@gpu
def test_flow_boundary_tiled_rejects_bad_shapes():
    """A tiles count other than the query's, and a shape whose one row does not fit, raise before any launch."""
    cs = Case(2, 12, 32, 32, seed=3)
    sk = Sinks(cs, {"y", "a1"}, "f32", 32)
    T = N.flow_boundary_tiles(2, 12, 32, 32, 1, 1, 1)
    b3, l3 = cs.dev
    for bad in (T - 1, T + 1):
        with pytest.raises(RuntimeError, match="tiles"):
            N.flow_boundary_tiled(cs.src, cs.in_bs, False, cs.pm_dev, cs.ldp, b3, l3, sk.t("ld"), cs.mt_dev, cs.beta_dev,
                                  sk.t("y"), sk.y_bs, None, 0, sk.t("a1"), sk.lda1, 2, 12, 32, 32, False, bad)
    B, C, H, W = 64, 192, 8, 8
    assert N.flow_boundary_tiles(B, C, H, W, 1, 1, 1) == 0 == _tiles(B, C, H, W, True, True, True)
    big = Case(B, C, H, W, seed=4)
    bsk = Sinks(big, {"y", "a1"}, "f32", 3)
    b3, l3 = big.dev
    with pytest.raises(RuntimeError, match="does not fit"):
        N.flow_boundary_tiled(big.src, big.in_bs, False, big.pm_dev, big.ldp, b3, l3, bsk.t("ld"), big.mt_dev,
                              big.beta_dev, bsk.t("y"), bsk.y_bs, None, 0, bsk.t("a1"), bsk.lda1, B, C, H, W, False, 3)
    torch.cuda.synchronize()
    for s in (sk.y, sk.a1, sk.ld, bsk.y, bsk.a1, bsk.ld):
        assert same_bits(s.buf.cpu(), s.before)


# ------------------------------------------------------------------------------------------------ gemm3_boundary
F_HID = 256           # hidden width of the coupling network: 4 (bf16) / 8 (split pairs) k-blocks, more than the stages
# (id, B, C, H, W, expected (ipc, ipp, stages), mix, sinks, inverse, ld, pm_out, in place, operand x a1 formats, wide)
_G3 = [
    ("ipc1_two_mtiles", 3, 12, 16, 16, (1, 1, 3), True, "y xs a1", False, True, True, False,
     (("bf16", "f32"), ("bf16", "bf16"), ("split", "split"), ("split", "f32")), False),
    ("ipc1_in_place_inverse", 3, 12, 16, 16, (1, 1, 3), True, "y a1", True, True, False, True,
     (("bf16", "bf16"), ("split", "f32")), False),
    ("ipc2_ragged_inverse", 5, 24, 8, 8, (2, 2, 3), True, "y xs a1", True, True, True, False,
     (("split", "f32"), ("bf16", "bf16")), False),
    ("ipc8_ragged_two_passes", 11, 48, 4, 4, (8, 4, 2), True, "y xs a1", False, True, True, False,
     (("bf16", "f32"), ("split", "split")), False),
    ("ipc8_ragged_inverse_no_ld", 20, 48, 4, 4, (8, 4, 2), True, "y xs", True, False, False, False,
     (("bf16", "f32"), ("split", "f32")), False),
    ("ipc16_4x2_ragged_no_mix", 21, 8, 4, 2, (16, 16, 3), False, "y a1", False, True, True, False,
     (("bf16", "f32"), ("split", "bf16")), False),
    ("ipc16_2x4_b_lt_ipc", 5, 8, 2, 4, (16, 16, 3), True, "y a1", False, True, False, True,
     (("bf16", "split"), ("split", "f32")), False),
    ("ipc16_2x4_b_lt_ipc_last_step", 5, 8, 2, 4, (16, 16, 3), False, "y", True, True, True, False, (("bf16", "f32"),), False),
    ("wide_forward", 3, 12, 16, 16, (1, 1, 3), True, "y xs a1", False, True, True, False, (("bf16", "f32"),), True),
    ("wide_inverse_ragged", 5, 24, 8, 8, (2, 2, 3), True, "y xs a1", True, True, False, False, (("split", "f32"),), True),
]


@gpu
@pytest.mark.parametrize("case,B,C,H,W,expect,mix,sinks,inverse,with_ld,with_pm_out,in_place,op,fmt,wide", [
    pytest.param(*c[:12], o, f, c[13], id=f"{c[0]}-{o}-{f}") for c in _G3 for o, f in c[12]])
def test_gemm3_boundary(case, B, C, H, W, expect, mix, sinks, inverse, with_ld, with_pm_out, in_place, op, fmt, wide):
    want = set(sinks.split())
    P, ldp = H * W, _ldp(C)
    M = B * P
    kmul = 2 if op == "split" else 1
    plan = _g3_plan(B, C, H, W, F_HID * kmul, ldp, mix)
    assert plan is not None and (plan["ipc"], plan["ipp"], plan["stages"]) == expect
    assert N.gemm3_boundary_ok(B, C, H, W, F_HID * kmul, ldp) == (_g3_plan(B, C, H, W, F_HID * kmul, ldp, True) is not None)
    assert (B % plan["ipc"] != 0) == ("ragged" in case or "b_lt_ipc" in case)      # a partial last CTA
    assert (B < plan["ipc"]) == ("b_lt_ipc" in case)
    assert (plan["passes"] > 1) == ("two_passes" in case or case.startswith("ipc8"))
    h2 = rnd(M, F_HID, seed=11) * 0.5
    w3 = rnd(ldp, F_HID, seed=12, scale=(2.8 if wide else 0.2) / F_HID ** 0.5)
    if op == "split":
        h2k, w3k = SP.encode(h2), SP.encode(w3)
        h2v, w3v = SP.value(h2k, M, F_HID), SP.value(w3k, ldp, F_HID)
    else:
        h2k, w3k = h2.bfloat16(), w3.bfloat16()
        h2v, w3v = h2k.double(), w3k.double()
    pm = h2v @ w3v.T                                     # fp64 from the operands the kernel decodes
    cs = Case(B, C, H, W, seed=len(case) + 13, mix=mix, wide=wide, pm=pm)
    src_sink = Sink(cs.src_host.numel(), init=cs.src_host) if in_place else None
    src = src_sink.t if in_place else cs.src
    sk = Sinks(cs, want, fmt, 1 if with_ld else 0, src_sink)
    ld_pm = ldp + 20
    pm_out = Sink(M * ld_pm) if with_pm_out else None
    b3, l3 = cs.dev
    N.gemm3_boundary(h2k.to(DEV), F_HID, w3k.to(DEV), pm_out and pm_out.t, ld_pm if with_pm_out else 0, src, cs.in_bs,
                     b3, l3, sk.t("ld"), cs.mt_dev, cs.beta_dev, sk.t("y"), sk.y_bs, sk.t("xs"), sk.xs_bs, sk.t("a1"),
                     sk.lda1, B, C, H, W, F_HID, ldp, inverse)
    torch.cuda.synchronize()
    ref = cs.ref(inverse)
    if wide:
        _check_wide(ref)
    if with_pm_out:
        got = pm_out.get((torch.arange(ld_pm) < ldp).expand(M, ld_pm)).view(M, ld_pm)
        check("pm_out", got[:, :ldp], pm)
    _verify(sk, ref)
