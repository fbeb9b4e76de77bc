"""Helpers of the kernel-level tests (test_gpu_train_kernels.py, test_gpu_boundary_kernels.py): guarded output buffers,
the tolerance rules, and fp64 restatements of the reference's arithmetic that more than one kernel is checked against.

Tolerances (per tensor): fp32 sinks relative L2 <= 1e-5 and max |error| <= 1e-4 * max |ref| (one wrong border pixel
fails the second); bf16 sinks within one bf16 ulp of the bf16 rounding of the fp64 value per element; split-pair sinks
decoded, then the fp32 rule.  ``check`` and ``check_bf16`` record their worst values in ``WORST`` for the tests to
print (run with -s)."""
import numpy as np
import torch
import torch.nn.functional as F

from normalizing_flow import _native as N

DEV = "cuda"
TOL_REL, TOL_MAX = 1e-5, 1e-4     # fp32 sinks: relative L2, max |error| / max |ref|
WORST = {}


def rnd(*shape, seed=0, scale=1.0):
    return torch.from_numpy((scale * np.random.default_rng(seed).standard_normal(shape)).astype(np.float32))


def note(key, v):
    WORST[key] = max(WORST.get(key, 0.0), v)


def report_worst(name):
    """Prints and clears the worst value of each measure taken since the last call."""
    if WORST:
        print(f"\n[worst] {name}: " + ", ".join(f"{k} {v:.2e}" for k, v in sorted(WORST.items())))
    WORST.clear()


def check(name, got, ref, rel_tol=TOL_REL, max_tol=TOL_MAX):
    """The fp32 rule: relative L2 and max |error| / max |ref| of one tensor."""
    got, ref = got.double().reshape(-1), ref.detach().double().reshape(-1)
    assert bool(torch.isfinite(got).all()), f"{name}: non-finite values"
    d = got - ref
    r = float(d.norm() / ref.norm()) if float(ref.norm()) > 0 else float(d.norm())
    scale = float(ref.abs().max())
    m = float(d.abs().max() / scale) if scale > 0 else float(d.abs().max())
    note("relL2", r)
    note("max/max|ref|", m)
    assert r <= rel_tol and m <= max_tol, f"{name}: relL2 {r:.3e} (<= {rel_tol}), max {m:.3e} (<= {max_tol})"


def check_bf16(name, got, ref):
    """A bf16 sink: per element within one bf16 ulp of the bf16 rounding of the fp64 value.  An element that is the sum
    of terms far larger than itself carries their fp32 rounding (~1e-7 of the terms) before the kernel rounds it to bf16,
    so the bound also admits 1e-6 * max |ref|, which is 2^-8 of one ulp of the largest element."""
    ref = ref.detach().double().reshape(-1)
    want = ref.to(torch.bfloat16).double()
    got = got.double().reshape(-1)
    assert bool(torch.isfinite(got).all()), f"{name}: non-finite values"
    _, e = torch.frexp(want)
    ulp = torch.where(want == 0, torch.full_like(want, 2.0 ** -133), torch.ldexp(torch.ones_like(want), e - 8))
    err = float(((got - want).abs() / (ulp + 1e-6 * float(ref.abs().max()))).max())
    note("bf16 ulps", err)
    assert err <= 1.0, f"{name}: {err:.3f} bf16 ulps"


_INT = {4: torch.int32, 2: torch.int16}


def same_bits(a, b):
    return torch.equal(a.reshape(-1).view(_INT[a.element_size()]), b.reshape(-1).view(_INT[b.element_size()]))


class Sink:
    """A device output of n elements inside a buffer with SLACK guard elements on both sides, all sentinel-filled (NaN;
    the int32 word 7 for split pairs) or set to ``init`` (outputs the kernel adds to).  ``slack`` widens the guards."""
    SLACK = 64

    def __init__(self, n, dtype=torch.float32, init=None, slack=None):
        S = self.S = slack or self.SLACK
        fill = 7 if dtype == N.SPLIT else float("nan")
        host = torch.full((n + 2 * S,), fill, dtype=dtype)
        if init is not None:
            host[S:S + n] = init.reshape(-1).to(dtype)
        self.n, self.before = n, host
        self.buf = host.to(DEV, copy=True)
        self.t = self.buf[S:S + n]

    def get(self, written=None):
        """The n elements after the kernel.  The slack and the elements outside the boolean mask ``written`` must hold
        exactly what they held before."""
        S, n = self.S, self.n
        got = self.buf.cpu()
        assert same_bits(got[:S], self.before[:S]) and same_bits(got[S + n:], self.before[S + n:]), \
            "write outside the output"
        g = got[S:S + n]
        if written is not None:
            keep = ~written.reshape(-1)
            assert same_bits(g[keep], self.before[S:S + n][keep]), "write into a region of the output it must not touch"
        return g


def cols_below(rows, ld, k):
    """[rows, ld] mask of the columns < k."""
    return (torch.arange(ld) < k).expand(rows, ld)


def split_words(mask):
    """Logical [rows, ld] mask -> mask of the int32 words of the split-pair layout that hold those elements (group
    g = k // 32 of a row is [hi(32) | lo(32)] bf16, two bf16 per word)."""
    rows, ld = mask.shape
    m = mask.reshape(rows, ld // 32, 1, 32).expand(rows, ld // 32, 2, 32).reshape(rows, 2 * ld)
    return m.reshape(rows, ld, 2).any(-1)


# ------------------------------------------------------------------------------------------------ fp64 restatements
def gather_taps(pm, B, C, H, W):
    """The ZeroConv output from its taps-as-N GEMM rows pm [B*H*W, >= 9C]: net[b, co, y, x] = sum over the taps inside
    the image of pm[(b, y + dy, x + dx), tap*C + co], (dy, dx) = (tap // 3 - 1, tap % 3 - 1)."""
    p5 = pm[:, :9 * C].reshape(B, H, W, 9, C).permute(0, 3, 4, 1, 2)       # [B, tap, C, H, W]
    pp = F.pad(p5, (1, 1, 1, 1))
    return sum(pp[:, tap, :, tap // 3:tap // 3 + H, tap % 3:tap % 3 + W] for tap in range(9))


def coupling_ref(u, pm, bias3, logs3, B, C, H, W):
    """transforms.py:179-184 with the ZeroConv of utils.py:43-44 given as taps-as-N rows: net = (conv + bias)*exp(3 logs),
    (log_s, t) its halves, s = sigmoid(log_s + 2), y = (u_a, (u_b + t)*s), per-image log-det sum log(s + 1e-6)."""
    net = (gather_taps(pm, B, C, H, W) + bias3.view(1, C, 1, 1)) * torch.exp(3 * logs3.view(1, C, 1, 1))
    log_s, t = net.chunk(2, 1)
    s = torch.sigmoid(log_s + 2)
    ua, ub = u.view(B, C, H, W).chunk(2, 1)
    return torch.cat([ua, (ub + t) * s], 1), torch.log(s + 1e-6).reshape(B, -1).sum(1)


def mix_ref(x, w, s, b):
    """transforms.py:80-81 then :131-132: y = W exp(s)(x + b); log-det P (sum s + log|det W|) (P = H*W)."""
    C, P = x.shape[1], x.shape[2] * x.shape[3]
    y = torch.einsum("oi,bihw->bohw", w, torch.exp(s).view(1, C, 1, 1) * (x + b.view(1, C, 1, 1)))
    return y, P * (s.sum() + torch.linalg.slogdet(w)[1])


def im2col_rows(x):
    """F.unfold(x, 3, padding=1) as GEMM rows [B*H*W, 9C], column c*9 + tap (the coupling network's first operand)."""
    B, C, H, W = x.shape
    return F.unfold(x, 3, padding=1).transpose(1, 2).reshape(B * H * W, 9 * C)
