"""Training-direction backward kernels (csrc/backward.cu), one entry point at a time, against fp64 torch autograd over
restatements of the reference's arithmetic, at the dispatch branches each kernel has.

Every output is a guarded sink: sentinel-filled (NaN, or the word 7 for split pairs) with slack on both sides, strided
into a wider tensor where the ABI takes a batch stride, and with padding columns where it takes a leading dimension.
A test asserts that the written region matches the reference, that padding columns the header says are zero-filled are
exactly zero, and that every element outside the output is bit-identical to before.

Tolerances (per tensor): fp32 sinks relative L2 <= 1e-5 and max |error| <= 1e-4 * max |ref| (one wrong border pixel
fails the second); bf16 sinks within one bf16 ulp of the bf16 rounding of the fp64 value per element; split-pair sinks
decoded, then the fp32 rule.  Each test prints its worst measured values (run with -s).

The unmarked tests at the top check each fp64 restatement against the CPU oracle's forward on the same values, so a
wrong tap order or sign in a restatement cannot hide the same mistake in a kernel."""
import contextlib
import math

import pytest
import torch
import torch.nn.functional as F

from normalizing_flow import _native as N
from oracle import glow_oracle as O
import split_pairs as SP
from kernel_refs import (DEV, WORST, Sink, check, check_bf16, cols_below, coupling_ref, gather_taps, im2col_rows, mix_ref,
                         report_worst, rnd, same_bits, split_words)

gpu = pytest.mark.gpu
TOL_DW = 1e-4                     # d(weight) of mix_param_grad: W^-1 is the fp32 inverse from mix_prepare


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


@contextlib.contextmanager
def default_fp64():
    prev = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        yield
    finally:
        torch.set_default_dtype(prev)


# ------------------------------------------------------------------------------------------------ fp64 restatements
def actnorm_relu_ref(pre, scale, bias):
    """utils.py:69 (ActNorm, transforms.py:80) followed by the ReLU of utils.py:84-87 on rows [M, N]."""
    return torch.relu(torch.exp(scale) * (pre + bias))


def col2im_ref(da, B, Cin, H, W):
    """The adjoint of :func:`im2col_rows` written out: dx[b, c, y, x] = sum over the taps inside the image of
    da[(b, y - dy, x - dx), c*9 + tap]."""
    d5 = da[:, :9 * Cin].reshape(B, H, W, Cin, 9).permute(0, 4, 3, 1, 2)    # [B, tap, Cin, H, W]
    pp = F.pad(d5, (1, 1, 1, 1))
    return sum(pp[:, tap, :, 2 - tap // 3:2 - tap // 3 + H, 2 - tap % 3:2 - tap % 3 + W] for tap in range(9))


def gauss_logp(z, mean, lg):
    """prior.py:36-37: log N(z; mean, exp(lg)) summed per image."""
    v = -0.5 * (math.log(2 * math.pi) + 2 * lg + (z - mean) ** 2 * torch.exp(-2 * lg))
    return v.reshape(z.shape[0], -1).sum(1)


def split_prior_ref(hh, bias, logs, z):
    """transforms.py:286-289: log-density of the split-off half z under (mean, lg), the halves of the ZeroConv output
    (h + bias)*exp(3 logs) given as rows hh [B*H*W, C]."""
    B, Ch, H, W = z.shape
    net = ((hh + bias) * torch.exp(3 * logs)).view(B, H, W, 2 * Ch).permute(0, 3, 1, 2)
    mean, lg = net.chunk(2, 1)
    return gauss_logp(z, mean, lg)


def gauss_const_ref(z, bias, logs):
    """prior.py:79-83: the ZeroConv of an all-zero map is bias*exp(3 logs) per channel; (mean, lg) its halves."""
    C = z.shape[1]
    net = (bias * torch.exp(3 * logs)).view(1, 2 * C, 1, 1)
    return gauss_logp(z, net[:, :C], net[:, C:])


# ------------------------------------------------------------------------------------------------ CPU: restatements
def test_taps_gather_is_the_zeroconv(monkeypatch):
    B, Cin, C, H, W = 2, 5, 6, 5, 7
    h, w = rnd(B, Cin, H, W, seed=1).double(), rnd(C, Cin, 3, 3, seed=2).double()
    bias, logs = rnd(C, seed=3).double(), rnd(C, seed=4, scale=0.3).double()
    pm = torch.einsum("bihw,oiyx->bhwyxo", h, w).reshape(B * H * W, 9 * C)          # column (ky*3 + kx)*C + co
    pm = torch.cat([pm, torch.full((B * H * W, 5), 1e3, dtype=torch.float64)], 1)   # padding columns are not read
    assert torch.allclose(gather_taps(pm, B, C, H, W), F.conv2d(h, w, padding=1), rtol=0, atol=1e-12)
    net = O.zeroconv(h, w, bias, logs.view(1, C, 1, 1))
    u = rnd(B, C, H, W, seed=5).double()
    monkeypatch.setattr(O, "coupling_net", lambda x_a, sd, pre, init=False: net)
    y_o, ld_o = O.coupling_fwd(u, {}, "")
    y, ld = coupling_ref(u, pm, bias, logs, B, C, H, W)
    assert torch.allclose(y, y_o, rtol=0, atol=1e-12) and torch.allclose(ld, ld_o, rtol=1e-13, atol=0)


def test_mix_restatement_is_actnorm_then_invconv():
    B, C, H, W = 2, 6, 3, 5
    x = rnd(B, C, H, W, seed=1).double()
    w = torch.linalg.qr(rnd(C, C, seed=2).double())[0] + 0.1 * rnd(C, C, seed=3).double()
    s, b = rnd(C, seed=4, scale=0.3).double(), rnd(C, seed=5, scale=0.3).double()
    y1, ld1 = O.actnorm_fwd(x, s.view(C, 1, 1), b.view(C, 1, 1))
    y_o = F.conv2d(y1, w.view(C, C, 1, 1))                          # invconv_fwd, without its fp32 log-det cast
    ld_o = ld1 + H * W * torch.slogdet(w)[1]
    y, ld = mix_ref(x, w, s, b)
    assert torch.allclose(y, y_o, rtol=0, atol=1e-12) and abs(float(ld - ld_o)) <= 1e-12 * abs(float(ld_o))


def test_split_prior_restatement_is_gaussian_logp():
    B, Ch, H, W = 3, 3, 4, 5
    C = 2 * Ch
    y, z = rnd(B, Ch, H, W, seed=1).double(), rnd(B, Ch, H, W, seed=2).double()
    sd = {"p.conv.weight": rnd(C, Ch, 3, 3, seed=3, scale=0.3).double(), "p.conv.bias": rnd(C, seed=4).double(),
          "p.conv.logs": rnd(1, C, 1, 1, seed=5, scale=0.2).double()}
    mean, logs = O.split_prior_params(y, sd, "p.")
    want = O.gaussian_logp(z, mean, logs)
    hh = F.conv2d(y, sd["p.conv.weight"], padding=1).permute(0, 2, 3, 1).reshape(B * H * W, C)
    got = split_prior_ref(hh, sd["p.conv.bias"], sd["p.conv.logs"].view(C), z)
    assert torch.allclose(got, want, rtol=1e-13, atol=1e-12)
    assert torch.allclose(gauss_logp(z, 0.0 * z, 0.0 * z), O.gaussian_logp(z, 0.0 * z, 0.0 * z), rtol=1e-13, atol=0)


def test_gauss_restatement_is_gaussian_prior_logp():
    B, C, H, W = 3, 4, 5, 3
    z = rnd(B, C, H, W, seed=1).double()
    psd = {"_GaussianPrior__conv.weight": rnd(2 * C, 2 * C, 3, 3, seed=2).double(),
           "_GaussianPrior__conv.bias": rnd(2 * C, seed=3).double(),
           "_GaussianPrior__conv.logs": rnd(1, 2 * C, 1, 1, seed=4, scale=0.2).double()}
    with default_fp64():                            # the oracle builds its all-zero map in the default dtype
        want = O.gaussian_prior_logp(psd, z)
        want0 = O.gaussian_prior_logp({}, z)
    got = gauss_const_ref(z, psd["_GaussianPrior__conv.bias"], psd["_GaussianPrior__conv.logs"].view(2 * C))
    assert torch.allclose(got, want, rtol=1e-13, atol=1e-12)
    assert torch.allclose(gauss_logp(z, 0.0 * z, 0.0 * z), want0, rtol=1e-13, atol=0)


def test_col2im_restatement_is_the_unfold_adjoint():
    for B, Cin, H, W in ((2, 3, 5, 7), (1, 2, 1, 1), (2, 1, 2, 3)):
        da = rnd(B * H * W, 9 * Cin + 4, seed=H * W).double()
        x = torch.zeros(B, Cin, H, W, dtype=torch.float64, requires_grad=True)
        (im2col_rows(x) * da[:, :9 * Cin]).sum().backward()
        assert torch.allclose(col2im_ref(da, B, Cin, H, W), x.grad, rtol=0, atol=1e-12)


def test_branch_replicas_agree_with_the_library():
    """The Python replicas of backward.cu's dispatch conditions that the GPU tests rely on, against the library's own
    tile queries (host code: no device needed)."""
    for C, H, W in ((48, 4, 4), (12, 16, 16), (24, 8, 8), (4, 14, 14), (8, 7, 7), (6, 5, 7), (12, 8, 8), (12, 32, 32),
                    (12, 64, 64)):
        assert (N.coupling_bwd_tiles(C, H, W) == 1) == (_coupling_smem(C, H, W) <= 200 * 1024)
    for C, H, W in ((12, 16, 16), (4, 28, 28), (24, 14, 14), (24, 7, 7), (48, 4, 4), (12, 64, 64), (96, 16, 16),
                    (192, 4, 4)):
        assert N.mix_bwd_tiles(C, H, W) == -(-(H * W) // _mix_tp(C, H * W))


# ------------------------------------------------------------------------------------------------ dispatch replicas
def _coupling_smem(C, H, W):
    """coupling_bwd_floats (backward.cu) in bytes: the one-CTA-per-image kernel's shared memory without the pm block."""
    P, Ch, PP = H * W, C // 2, (H + 2) * (W + 2)
    fl = (C * (P + 1) + Ch * (P + 1) + 4 * P * Ch + 2 * C + 3) & ~3
    fl += (C * PP + 3) & ~3
    fl += (9 * C + 3) & ~3
    return 4 * fl


def _coupling_pm_bulk(C, H, W, ldp):
    """coupling_bwd_launch: pm is staged by bulk copy when ldp % 4 == 0, pm is 16-byte aligned (a fresh allocation) and
    the pm block fits next to the kernel's shared memory in 200 KB."""
    return ldp % 4 == 0 and _coupling_smem(C, H, W) + 4 * H * W * ldp <= 200 * 1024


def _last_cta_loops(B, C, P):
    """Trip counts of the last-CTA reduction's 32-wide, 8-wide and tail loops for row group 0: coupling_bwd_launch runs
    threads = clamp(roundup32(P*C/2), 128, 1024), the kernel RG = clamp(threads / 2C, 1, 32) row groups."""
    threads = min(1024, max(128, (P * (C // 2) + 31) // 32 * 32))
    RG = min(32, max(1, threads // (2 * C)))
    bb, n = 0, [0, 0, 0]
    while bb + 31 * RG < B:
        bb, n[0] = bb + 32 * RG, n[0] + 1
    while bb + 7 * RG < B:
        bb, n[1] = bb + 8 * RG, n[1] + 1
    while bb < B:
        bb, n[2] = bb + RG, n[2] + 1
    return tuple(n)


def _mix_tp(C, P):
    """mix_bwd_tile (backward.cu, default cap 256): pixels per CTA tile, halved until 2C(TP+1) + C^2 floats fit 200 KB."""
    tp = min(P, 256)
    while tp > 8 and 4 * (2 * C * (tp + 1) + C * C) > 200 * 1024:
        tp = (tp + 1) // 2
    return tp


# ------------------------------------------------------------------------------------------------ coupling_bwd
_FMT = {"f32": torch.float32, "bf16": torch.bfloat16, "split": N.SPLIT}
# (id, B, C, H, W, path, pm staging, dpm store, dld given, formats)
_COUPLING = [
    ("last_cta_three_loops", 165, 48, 4, 4, "fused", "bulk", "vec", True, ("f32", "bf16", "split")),
    ("level0_bench", 5, 12, 16, 16, "fused", "bulk", "vec", True, ("f32", "bf16", "split")),
    ("level1_bench", 4, 24, 8, 8, "fused", "bulk", "vec", True, ("f32", "bf16", "split")),
    ("mnist_196px", 3, 4, 14, 14, "rows2", "bulk", "vec", True, ("f32", "bf16", "split")),
    ("scalar_store", 5, 8, 7, 7, "rows2", "bulk", "scalar", True, ("f32", "bf16")),
    ("pm_global_no_dld", 2, 6, 5, 7, "fused", "global", "vec", False, ("f32", "bf16", "split")),
    ("pm_global_scalar", 3, 12, 8, 8, "rows2", "global", "scalar", True, ("f32", "bf16")),
    ("no_dld", 4, 24, 8, 8, "rows2", "bulk", "vec", False, ("f32",)),
    ("one_image", 1, 12, 8, 8, "fused", "bulk", "vec", True, ("f32", "bf16")),
    ("tiled_32", 2, 12, 32, 32, "tiled", "bulk", "vec", True, ("f32", "bf16", "split")),
    ("tiled_64_config4", 2, 12, 64, 64, "tiled", "bulk", "vec", True, ("f32", "bf16", "split")),
    ("tiled_no_dld", 2, 12, 32, 32, "tiled", "bulk", "vec", False, ("f32",)),
]


@gpu
@pytest.mark.parametrize("case,B,C,H,W,path,staging,store,with_dld,fmt", [
    pytest.param(*c[:9], f, id=f"{c[0]}-{f}") for c in _COUPLING for f in c[9]])
def test_coupling_bwd(case, B, C, H, W, path, staging, store, with_dld, fmt):
    """Forward coupling backward: objective <y, dy> + sum_b dld[b] * sum log(s + 1e-6) with leaves u, pm, bias3, logs3."""
    P, Ch, M = H * W, C // 2, B * H * W
    T_c = N.coupling_bwd_tiles(C, H, W)
    assert (T_c > 1) == (path == "tiled")
    ldp = (9 * C + 15) // 16 * 16 if staging == "bulk" else (9 * C + 2 if (9 * C + 2) % 4 else 9 * C + 1)
    if path != "tiled":
        assert _coupling_pm_bulk(C, H, W, ldp) == (staging == "bulk")
    ld_dpm = (9 * C + 63) // 64 * 64 + 32 if store == "vec" else (9 * C + 4 if (9 * C + 4) % 8 else 9 * C + 2)
    assert ld_dpm > 9 * C and (ld_dpm % 8 == 0) == (store == "vec")      # vector dpm stores need ld % 8 == 0
    if case == "last_cta_three_loops":
        assert min(_last_cta_loops(B, C, P)) > 0
    dy, u = rnd(B, C, P, seed=1), rnd(B, C, P, seed=3)
    dld = rnd(B, seed=2) if with_dld else None
    pm = rnd(M, ldp, seed=4, scale=0.1)
    bias3, logs3 = rnd(C, seed=5, scale=0.1), rnd(C, seed=6, scale=0.1)
    dev = [None if t is None else t.to(DEV) for t in (dy, dld, u, pm, bias3, logs3)]
    du_bs = (C + 1) * P                                     # du strided into a wider tensor

    def run():
        du = Sink(B * du_bs)
        dpm = Sink(M * ld_dpm, _FMT[fmt])
        dpar = Sink(B * T_c * 2 * C)
        db, dl = Sink(C), Sink(C)
        args = (dev[0], C * P, dev[1], dev[2], C * P, dev[3], ldp, dev[4], dev[5], du.t, du_bs, dpm.t, ld_dpm, dpar.t,
                B, C, H, W)
        if path == "fused":
            N.coupling_bwd(*args, db.t, dl.t)
        elif path == "rows2":
            N.coupling_bwd(*args)
            N.reduce_rows2(dpar.t, db.t, dl.t, B * T_c, C, C, 2 * C)
        else:
            N.coupling_bwd(*args, dp_scratch=torch.empty(M * C, device=DEV))
            N.reduce_rows2(dpar.t, db.t, dl.t, B * T_c, C, C, 2 * C)
        torch.cuda.synchronize()
        du_w = (torch.arange(C + 1) < C).view(1, C + 1, 1).expand(B, C + 1, P)
        return (du.get(du_w).view(B, C + 1, P)[:, :C], dpm.get(), dpar.get(), db.get(), dl.get())

    out = run()
    if path == "fused":                     # the last CTA re-arms its counter: a second call gives the same bits
        again = run()
        assert all(same_bits(a, b) for a, b in zip(out, again))
    du, dpm, _, db, dl = out
    ud, pd, bd, lsd = (t.double().requires_grad_(True) for t in (u, pm, bias3, logs3))
    y, ld = coupling_ref(ud, pd, bd, lsd, B, C, H, W)
    obj = (y * dy.double().view(B, C, H, W)).sum()
    if with_dld:
        obj = obj + (ld * dld.double()).sum()
    obj.backward()
    assert torch.equal(du[:, :Ch], dy[:, :Ch])
    check("du_b", du[:, Ch:], ud.grad.view(B, C, P)[:, Ch:])
    check("dbias3", db, bd.grad)
    check("dlogs3", dl, lsd.grad)
    want = pd.grad[:, :9 * C]
    if fmt == "split":
        val = SP.value(dpm, M, ld_dpm)
        assert float(val[:, 9 * C:].abs().max()) == 0.0
        check("dpm", val[:, :9 * C], want)
    else:
        got = dpm.view(M, ld_dpm).float()
        assert float(got[:, 9 * C:].abs().max()) == 0.0                 # (NaN fails too)
        (check if fmt == "f32" else check_bf16)("dpm", got[:, :9 * C], want)


# ------------------------------------------------------------------------------------------------ actnorm_relu_bwd
_AN_FORMS = [(a, b, c) for a in ("f32", "bf16") for b in ("f32", "bf16") for c in ("f32", "bf16")] + \
            [("f32", "split", "split")]
# (N, rows_per_cta, forms): the kernel runs cg = N/8 column groups, rg = 256/cg row groups of a CTA's rows
_AN = [(512, 64, _AN_FORMS), (512, 3, [("f32", "f32", "f32"), ("f32", "split", "split")]),
       (432, 64, [("f32", "f32", "f32"), ("bf16", "bf16", "bf16")]), (432, 3, [("f32", "f32", "f32"), ("f32", "split", "split")]),
       (2048, 8, [("f32", "f32", "f32"), ("bf16", "f32", "bf16"), ("f32", "split", "split")]),
       (2048, 3, [("f32", "bf16", "f32")])]


@gpu
@pytest.mark.parametrize("Nn,rows,form", [pytest.param(n, r, f, id=f"N{n}-rows{r}-{'_'.join(f)}")
                                          for n, r, forms in _AN for f in forms])
def test_actnorm_relu_bwd(Nn, rows, form):
    """h = relu(exp(s)(pre + b)) with pre a leaf, objective <h, dh>: dpre and the column partials (d scale, d bias)
    reduced by reduce_rows2.  About a third of h is exactly 0 and must be masked, half of it on the ReLU's boundary."""
    cg = Nn // 8
    rg = 256 // cg
    if Nn == 432:
        assert 256 % cg != 0                       # threads r0 >= rg idle
    if rows == 3 and Nn < 2048:
        assert rg > rows                           # some row groups of each CTA have no rows
    if Nn == 2048:
        assert rg == 1                             # one row group
    M, ld = 203, (Nn + 63) // 32 * 32              # M not a multiple of rows_per_cta; ld > N (a multiple of 32)
    assert M % rows != 0 and ld % 32 == 0
    n_cta = -(-M // rows)
    fd, fh, fo = form
    scale, bias = rnd(Nn, seed=3, scale=0.2), rnd(Nn, seed=4, scale=0.5)
    hv = rnd(M, ld, seed=2).abs()
    sel = rnd(M, ld, seed=5)
    hv[sel < -0.4] = 0.0
    dh = rnd(M, ld, seed=1)
    if fd == "bf16":
        dh = dh.bfloat16()
    if fh == "split":
        h_k = SP.encode(hv)
        h_val = SP.value(h_k, M, ld)
    else:
        h_k = hv.bfloat16() if fh == "bf16" else hv
        h_val = h_k.double()
    dpre = Sink(M * ld, _FMT[fo])
    part = Sink(n_cta * 2 * Nn)
    d_s, d_b = Sink(Nn), Sink(Nn)
    N.actnorm_relu_bwd(dh.to(DEV), ld, h_k.to(DEV), ld, scale.to(DEV), dpre.t, ld, part.t, M, Nn, rows)
    N.reduce_rows2(part.t, d_s.t, d_b.t, n_cta, Nn, Nn, 2 * Nn)
    torch.cuda.synchronize()
    written = cols_below(M, ld, Nn)
    got = dpre.get(split_words(written) if fo == "split" else written).view(M, ld)
    part.get()
    # the pre-activation the kernel's h belongs to: exp(s)(pre + b) = h for h > 0; for h == 0 half the entries sit on the
    # ReLU's boundary (pre = -b exactly), half below it
    s64, b64 = scale.double(), bias.double()
    hv64 = h_val[:, :Nn]
    below = -b64 - 0.5 - rnd(M, Nn, seed=6).double().abs()
    pre = torch.where(hv64 > 0, hv64 / torch.exp(s64) - b64, torch.where(sel[:, :Nn] < -1.0, -b64.expand(M, Nn), below))
    pre_l, s_l, b_l = (t.clone().requires_grad_(True) for t in (pre, s64, b64))
    h_ref = actnorm_relu_ref(pre_l, s_l, b_l)
    assert torch.equal(h_ref > 0, hv64 > 0) and bool((h_ref[hv64 == 0] == 0).all())
    (h_ref * dh.double()[:, :Nn]).sum().backward()
    if fo == "split":
        check("dpre", SP.value(got, M, ld)[:, :Nn], pre_l.grad)
    elif fo == "bf16":
        check_bf16("dpre", got[:, :Nn].float(), pre_l.grad)
    else:
        check("dpre", got[:, :Nn], pre_l.grad)
    check("dscale", d_s.get(), s_l.grad)
    check("dbias", d_b.get(), b_l.grad)


# ------------------------------------------------------------------------------------------------ mix_bwd + mix_param_grad
def _prepare(w, s, b, C):
    """fwd_mt and winv of one (ActNorm, InvConv2d) pair from nfdpm_mix_prepare, as production prepares them."""
    from normalizing_flow import _engine as E
    cache = E.MixCache()
    dv = lambda t: None if t is None else t.to(DEV).contiguous()
    E.prepare_mix([(cache, dv(w), dv(s), dv(b), C, None)])
    return cache


def _mix_item(part, R, C, w, s, b, winv, dld_sum, P, dW, dS, dB, scratch):
    p = lambda t: None if t is None else t.data_ptr()
    return N.MixGradItem(part=part.data_ptr(), B=R, C=C, weight=w.data_ptr(), scale=p(s), bias=p(b), winv=winv.data_ptr(),
                         dld_sum=dld_sum.data_ptr(), P=float(P), pad_=0, d_weight=p(dW), d_scale=p(dS), d_bias=p(dB),
                         scratch=scratch.data_ptr())


# (B, C, H, W, tiles, partial-sum branches of the tiles): the warp branch runs for tiles of >= 64 pixels, the per-thread
# branch below
_MIX = [(3, 12, 16, 16, 1, {"warp"}), (2, 4, 28, 28, 4, {"warp", "thread"}), (3, 24, 14, 14, 1, {"warp"}),
        (4, 24, 7, 7, 1, {"thread"}), (5, 48, 4, 4, 1, {"thread"}), (2, 12, 64, 64, 16, {"warp"}),
        (2, 96, 16, 16, 2, {"warp"}), (3, 192, 4, 4, 1, {"thread"})]


@gpu
@pytest.mark.parametrize("B,C,H,W,tiles,branches", _MIX, ids=[f"{m[1]}x{m[2]}x{m[3]}" for m in _MIX])
def test_mix_bwd(B, C, H, W, tiles, branches):
    """Forward mix y = W exp(s)(x + b) with the coupling network's im2col gradient fused: objective <y, du> +
    <im2col(y_a), da1> + sum_b dld[b] P (sum s + log|det W|) with leaves x, W, s, b; dx from mix_bwd, d(W, s, b) from
    mix_param_grad over its partials."""
    P, Ch, M = H * W, C // 2, B * H * W
    T = N.mix_bwd_tiles(C, H, W)
    tp = _mix_tp(C, P)
    assert T == tiles == -(-P // tp)
    sizes = [min(tp, P - t * tp) for t in range(T)]
    assert {"warp" if n >= 64 else "thread" for n in sizes} == branches
    w = (torch.linalg.qr(rnd(C, C, seed=1).double())[0].float() + 0.1 * rnd(C, C, seed=2)).contiguous()   # (Q is column-major)
    s, b = rnd(C, seed=3, scale=0.3), rnd(C, seed=4, scale=0.3)
    x, du, dld = rnd(B, C, P, seed=5), rnd(B, C, P, seed=6), rnd(B, seed=7)
    lda1 = 9 * Ch + 8
    da1 = rnd(M, lda1, seed=8)
    mix = _prepare(w, s, b, C)
    dx_bs = (C + 1) * P
    dx = Sink(B * dx_bs)
    part = Sink(B * T * (C * C + C))
    N.mix_bwd(du.to(DEV), C * P, da1.to(DEV), lda1, x.to(DEV), C * P, mix.fwd_mt, dx.t, dx_bs, part.t, B, C, H, W)
    dW, dS, dB, scratch = Sink(C * C), Sink(C), Sink(C), Sink(C * C + C)
    wd, sd, bd = w.to(DEV), s.to(DEV), b.to(DEV)
    dld_sum = dld.sum().view(1).to(DEV)
    N.mix_param_grad([_mix_item(part.t, B * T, C, wd, sd, bd, mix.winv, dld_sum, P, dW.t, dS.t, dB.t, scratch.t)])
    torch.cuda.synchronize()
    got_dx = dx.get((torch.arange(C + 1) < C).view(1, C + 1, 1).expand(B, C + 1, P)).view(B, C + 1, P)[:, :C]
    part.get()
    scratch.get()
    xl, wl, sl, bl = (t.double().requires_grad_(True) for t in (x.view(B, C, H, W), w, s, b))
    y, ld = mix_ref(xl, wl, sl, bl)
    obj = (y * du.double().view(B, C, H, W)).sum() + (im2col_rows(y[:, :Ch]) * da1.double()[:, :9 * Ch]).sum()
    (obj + dld.double().sum() * ld).backward()
    check("dx", got_dx, xl.grad.view(B, C, P))
    check("dW", dW.get(), wl.grad, TOL_DW, TOL_DW)
    check("ds", dS.get(), sl.grad)
    check("db", dB.get(), bl.grad)


@gpu
def test_mix_param_grad_two_launches():
    """17 StepFlows in one nfdpm_mix_param_grad call (16 per launch): item 7 is a lone ActNorm (identity weight and
    inverse, no d(weight), as _modgrad._mix_backward builds it), item 16 an InvConv2d with scale / bias NULL."""
    B, H, W = 3, 4, 4
    P = H * W
    items, keep, refs = [], [], []
    for k in range(17):
        C = (4, 6, 8, 12)[k % 4]
        kind = "actnorm" if k == 7 else ("invconv" if k == 16 else "both")
        w = None if kind == "actnorm" else (torch.linalg.qr(rnd(C, C, seed=10 * k).double())[0].float() +
                                            0.1 * rnd(C, C, seed=10 * k + 1)).contiguous()
        s, b = (None, None) if kind == "invconv" else (rnd(C, seed=10 * k + 2, scale=0.3), rnd(C, seed=10 * k + 3, scale=0.3))
        x, du, dld = rnd(B, C, P, seed=10 * k + 4), rnd(B, C, P, seed=10 * k + 5), rnd(B, seed=10 * k + 6)
        mix = _prepare(w, s, b, C)
        T = N.mix_bwd_tiles(C, H, W)
        part = torch.empty(B * T * (C * C + C), device=DEV)
        dx = torch.empty(B, C, P, device=DEV)
        N.mix_bwd(du.to(DEV), C * P, None, 0, x.to(DEV), C * P, mix.fwd_mt, dx, C * P, part, B, C, H, W)
        eye = torch.eye(C, device=DEV)
        wd = eye if w is None else w.to(DEV)
        winv = eye if w is None else mix.winv
        sd, bd = (None, None) if s is None else (s.to(DEV), b.to(DEV))
        dW = None if w is None else Sink(C * C)
        dS, dB = (None, None) if s is None else (Sink(C), Sink(C))
        scratch = Sink(C * C + C)
        dld_sum = dld.sum().view(1).to(DEV)
        items.append(_mix_item(part, B * T, C, wd, sd, bd, winv, dld_sum, P, dW and dW.t, dS and dS.t, dB and dB.t,
                               scratch.t))
        keep.append((mix, part, dx, eye, wd, winv, sd, bd, dld_sum))
        refs.append((C, w, s, b, x, du, dld, dW, dS, dB, scratch))
    N.mix_param_grad(items)
    torch.cuda.synchronize()
    for k, (C, w, s, b, x, du, dld, dW, dS, dB, scratch) in enumerate(refs):
        scratch.get()
        wl = torch.eye(C, dtype=torch.float64) if w is None else w.double().requires_grad_(True)
        sl = torch.zeros(C, dtype=torch.float64) if s is None else s.double().requires_grad_(True)
        bl = torch.zeros(C, dtype=torch.float64) if b is None else b.double().requires_grad_(True)
        y, ld = mix_ref(x.double().view(B, C, H, W), wl, sl, bl)
        ((y * du.double().view(B, C, H, W)).sum() + dld.double().sum() * ld).backward()
        if w is not None:
            check(f"dW[{k}]", dW.get(), wl.grad, TOL_DW, TOL_DW)
        if s is not None:
            check(f"ds[{k}]", dS.get(), sl.grad)
            check(f"db[{k}]", dB.get(), bl.grad)


# ------------------------------------------------------------------------------------------------ priors
@gpu
@pytest.mark.parametrize("learned", [True, False], ids=["learned", "standard"])
@pytest.mark.parametrize("C", [6, 12, 48])
@pytest.mark.parametrize("H,W", [(4, 4), (7, 7), (16, 16), (32, 32)])
def test_split_prior_bwd(learned, C, H, W):
    """Split's log N(z; mean, exp(lg)) with (mean, lg) from the prior conv rows h (learned) or zeros: objective
    sum_b dlp[b] logp_b with leaves h, bias, logs, z.  dz adds into the second half of a pre-filled state (the first half
    stays as it was), dh's padding columns are zero-filled, dpar is reduced by reduce_rows2."""
    B, P, Ch = 3, H * W, C // 2
    M = B * P
    xs = (C + 2) * P                                       # state and its gradient strided into wider tensors
    x = rnd(B, C + 2, P, seed=1)
    dlp = rnd(B, seed=2)
    ldh = C + 10
    h = rnd(M, ldh, seed=3, scale=0.3)
    bias, logs = rnd(C, seed=4, scale=0.3), rnd(C, seed=5, scale=0.1)
    dstate = Sink(B * xs, init=rnd(B, C + 2, P, seed=6))
    dh, dpar, d_b, d_l = Sink(M * ldh), Sink(B * 2 * C), Sink(C), Sink(C)
    if learned:
        N.split_prior_bwd(dlp.to(DEV), h.to(DEV), ldh, bias.to(DEV), logs.to(DEV), x.to(DEV), xs, dstate.t, xs, dh.t,
                          dpar.t, B, C, H, W)
        N.reduce_rows2(dpar.t, d_b.t, d_l.t, B, C, C, 2 * C)
    else:
        N.split_prior_bwd(dlp.to(DEV), None, 0, None, None, x.to(DEV), xs, dstate.t, xs, None, None, B, C, H, W)
    torch.cuda.synchronize()
    ch = torch.arange(C + 2)
    got = dstate.get(((ch >= Ch) & (ch < C)).view(1, C + 2, 1).expand(B, C + 2, P)).view(B, C + 2, P)
    delta = got[:, Ch:C].double() - dstate.before[Sink.SLACK:Sink.SLACK + B * xs].view(B, C + 2, P)[:, Ch:C].double()
    zl = x[:, Ch:C].double().contiguous().view(B, Ch, H, W).requires_grad_(True)
    hl, bl, ll = (t.double().requires_grad_(True) for t in (h[:, :C], bias, logs))
    lp = split_prior_ref(hl, bl, ll, zl) if learned else gauss_logp(zl, 0.0 * zl.detach(), 0.0 * zl.detach())
    (lp * dlp.double()).sum().backward()
    check("dz", delta, zl.grad.view(B, Ch, P))
    if learned:
        g = dh.get().view(M, ldh)
        assert float(g[:, C:].abs().max()) == 0.0                          # (NaN fails too)
        check("dh", g[:, :C], hl.grad)
        dpar.get()
        check("dbias", d_b.get(), bl.grad)
        check("dlogs", d_l.get(), ll.grad)
    else:
        for s in (dh, dpar, d_b, d_l):
            assert same_bits(s.buf.cpu(), s.before)


@gpu
@pytest.mark.parametrize("with_params", [True, False], ids=["bias_logs", "standard"])
@pytest.mark.parametrize("C,H,W", [(24, 4, 4), (6, 15, 20)])
def test_gauss_const_bwd(with_params, C, H, W):
    """GaussianPrior's per-channel constants: objective sum_b dl[b] logp_b with leaves z, bias, logs; dpar [B][4C]
    reduced with reduce_rows (stride 4C) as the training step does."""
    B, P = 3, H * W
    z, dl = rnd(B, C, P, seed=1), rnd(B, seed=2)
    bias, logs = rnd(2 * C, seed=3, scale=0.3), rnd(2 * C, seed=4, scale=0.1)
    dz, dpar, gp = Sink(B * C * P), Sink(B * 4 * C), Sink(4 * C)
    if with_params:
        N.gauss_const_bwd(dl.to(DEV), z.to(DEV), bias.to(DEV), logs.to(DEV), dz.t, dpar.t, B, C, P)
        N.reduce_rows(dpar.t, gp.t, B, 4 * C, 4 * C)
    else:
        N.gauss_const_bwd(dl.to(DEV), z.to(DEV), None, None, dz.t, None, B, C, P)
    torch.cuda.synchronize()
    zl = z.double().view(B, C, H, W).requires_grad_(True)
    bl, ll = bias.double().requires_grad_(True), logs.double().requires_grad_(True)
    lp = gauss_const_ref(zl, bl, ll) if with_params else gauss_logp(zl, 0.0 * zl.detach(), 0.0 * zl.detach())
    (lp * dl.double()).sum().backward()
    check("dz", dz.get(), zl.grad)
    if with_params:
        dpar.get()
        g = gp.get()
        check("dbias", g[:2 * C], bl.grad)
        check("dlogs", g[2 * C:], ll.grad)
    else:
        assert same_bits(dpar.buf.cpu(), dpar.before) and same_bits(gp.buf.cpu(), gp.before)


# ------------------------------------------------------------------------------------------------ col2im_add
@gpu
@pytest.mark.parametrize("B,Cin,H,W", [(3, 5, 5, 7), (4, 6, 1, 1), (8, 24, 64, 64)])
def test_col2im_add(B, Cin, H, W):
    """The adjoint of F.unfold(x, 3, padding=1) added into the first Cin channels of a pre-filled 2*Cin-channel
    gradient; 1x1 images have every tap but the centre outside, and 8x24x64x64 outputs exceed the 148*16 CTAs of 256
    threads the launch caps its grid at, so the grid-stride loop wraps."""
    P, M = H * W, B * H * W
    if H == 64:
        assert B * Cin * P > 148 * 16 * 256
    lda = 9 * Cin + 3
    da = rnd(M, lda, seed=1)
    dst = Sink(B * 2 * Cin * P, init=rnd(B, 2 * Cin, P, seed=2))
    N.col2im_add(da.to(DEV), lda, dst.t, 2 * Cin * P, B, Cin, H, W)
    torch.cuda.synchronize()
    got = dst.get((torch.arange(2 * Cin) < Cin).view(1, 2 * Cin, 1).expand(B, 2 * Cin, P)).view(B, 2 * Cin, P)
    before = dst.before[Sink.SLACK:Sink.SLACK + dst.n].view(B, 2 * Cin, P)
    xl = torch.zeros(B, Cin, H, W, dtype=torch.float64, requires_grad=True)
    (im2col_rows(xl) * da.double()[:, :9 * Cin]).sum().backward()
    check("dx", got[:, :Cin].double() - before[:, :Cin].double(), xl.grad.view(B, Cin, P))


# ------------------------------------------------------------------------------------------------ reduce_rows(2)
@gpu
@pytest.mark.parametrize("accumulate", [0, 1])
@pytest.mark.parametrize("n", [1, 31, 33, 1031])
@pytest.mark.parametrize("R", [1, 7, 9, 1000])
def test_reduce_rows(R, n, accumulate):
    stride = n + 5
    part = rnd(R, stride, seed=R + n).to(DEV)
    init = rnd(n, seed=7) if accumulate else None
    outs = []
    for _ in range(2):
        out = Sink(n, init=init)
        N.reduce_rows(part, out.t, R, n, stride, accumulate)
        torch.cuda.synchronize()
        outs.append(out.get())
    assert same_bits(outs[0], outs[1])
    want = part.cpu()[:, :n].double().sum(0) + (init.double() if accumulate else 0.0)
    check("out", outs[0], want)


@gpu
@pytest.mark.parametrize("n", [1, 31, 33, 1031])
@pytest.mark.parametrize("R", [1, 7, 9, 1000])
def test_reduce_rows2(R, n):
    n0, n1 = n, n // 2 + 1
    stride = n0 + n1 + 3
    part = rnd(R, stride, seed=R * n).to(DEV)
    outs = []
    for _ in range(2):
        o0, o1 = Sink(n0), Sink(n1)
        N.reduce_rows2(part, o0.t, o1.t, R, n0, n1, stride)
        torch.cuda.synchronize()
        outs.append((o0.get(), o1.get()))
    assert same_bits(outs[0][0], outs[1][0]) and same_bits(outs[0][1], outs[1][1])
    want = part.cpu()[:, :n0 + n1].double().sum(0)
    check("out0", outs[0][0], want[:n0])
    check("out1", outs[0][1], want[n0:])
