"""The coupling-network GEMMs (csrc/gemm_tc.cu, gemm_simt.cu, gemm_tn_tc.cu and gemm_tn_kernel in backward.cu), every
dispatch branch against an fp64 product of the values the kernel actually reads: the bf16-rounded operands, the decoded
hi + lo of split pairs, or fp32.

Every output is a guarded sink (kernel_refs.Sink): sentinel-filled with slack on both sides.  gemm_nt writes a strided
view [M, N] of a buffer [M + 2, ldd] with ldd > N, so the columns N..ldd and the rows past M must stay bit-identical.
Operand rows past M, rows past N of the weight operand and the padding columns K..lda / K..ldb hold NaN: none of it
may reach D.  gemm_tn's workspace is exactly ``gemm_tn_workspace(M, N1, N2)`` floats followed by a guard region that
must not change, and the self-re-arming tile counters of the in-kernel reduction must be zero after every call.

Each case names the branch it covers and asserts it: gemm_nt's plan through ``tc_nt_plan`` (csrc/tc_sched.h, compiled
here with g++; grid and work units confirmed on the GPU through nfdpm_gemm_debug), gemm_tn's path through the replica
in normalizing_flow._native (checked on the CPU against nfdpm_gemm_tn_workspace).  The replicas assume the default
NFDPM_TC_* / NFDPM_TN_MIN_KB knobs.  ``test_production_calls_are_covered`` records the GEMM calls of whole models and
fails on a branch no case here covers."""
import contextlib
import os
import subprocess
import tempfile

import pytest
import torch

from normalizing_flow import _native as N
import split_pairs as SP
from kernel_refs import DEV, WORST, Sink, check, check_bf16, report_worst, rnd, same_bits, split_words

gpu = pytest.mark.gpu
KNOBS = ("NFDPM_TC_BN", "NFDPM_TC_NARROW", "NFDPM_TC_SPLIT", "NFDPM_TC_DEEP", "NFDPM_TN_MIN_KB")
pytestmark = pytest.mark.skipif(any(os.environ.get(k) for k in KNOBS), reason="the plan replicas assume the default knobs")
HDR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                   "normalizing-flow-with-diffusion-prior-model_b200", "csrc")
_FMT = {"f32": torch.float32, "bf16": torch.bfloat16, "split": N.SPLIT}
_CODE = {"f32": N.F32, "bf16": N.BF16, "split": N.BF16X2}


@pytest.fixture(autouse=True)
def _report_worst(request):
    """Prints the worst value of each measure a test took (pytest -s)."""
    WORST.clear()
    yield
    report_worst(request.node.name)


# ------------------------------------------------------------------------------------------------ gemm_nt plan query
_PLAN_MAIN = r"""
#include <cstdio>
#include "tc_sched.h"
int main() {
  int M, N, K, f32, bf16, act, sms;
  while (scanf("%d %d %d %d %d %d %d", &M, &N, &K, &f32, &bf16, &act, &sms) == 7) {
    const nfdpm::TcNtPlan p = nfdpm::tc_nt_plan(M, N, K, f32, bf16, act, sms, 256, 74, 1, 1);
    printf("%d %d %d %d %d %d %d %d %d %d\n", p.BN, p.num_n, p.tiles, p.grid, p.split, p.plan.n_stages, p.plan.stage_bytes,
           p.plan.cstage_bytes, p.plan.cpw, p.smem);
  }
  return 0;
}
"""
_PLAN_KEYS = ("BN", "num_n", "tiles", "grid", "split", "n_stages", "stage_bytes", "cstage_bytes", "cpw", "smem")
_plan_exe = None


def nt_plans(queries):
    """tc_nt_plan for each (M, N, K, in, out, epi) with the default knobs on 148 SMs -> list of dicts."""
    global _plan_exe
    if _plan_exe is None:
        d = tempfile.mkdtemp(prefix="nfdpm_plan_")
        src, exe = os.path.join(d, "plan.cpp"), os.path.join(d, "plan")
        with open(src, "w") as f:
            f.write(_PLAN_MAIN)
        r = subprocess.run(["g++", "-std=c++17", "-O1", "-I", HDR, src, "-o", exe], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr[-3000:]
        _plan_exe = exe
    lines = "".join(f"{M} {Nn} {K * (2 if i == 'split' else 1)} {int(o == 'f32')} {int(o == 'bf16')} "
                    f"{int(e == N.EPI_ACTNORM_RELU)} 148\n" for M, Nn, K, i, o, e in queries)
    r = subprocess.run([_plan_exe], input=lines, capture_output=True, text=True, check=True)
    return [dict(zip(_PLAN_KEYS, map(int, ln.split()))) for ln in r.stdout.splitlines()]


def nt_branch(M, Nn, K, ind, out, epi, p=None):
    """The branch tuple of one gemm_nt call: what the launch plan decides (tensor core) or the CUDA-core tile width."""
    if ind == "f32":
        return ("simt", out, epi, 128 if Nn > 64 else 64, Nn % 4 != 0)
    p = p or nt_plans([(M, Nn, K, ind, out, epi)])[0]
    bn0 = 128 if out == "f32" else 256
    nblk0 = -(-Nn // bn0)
    cpb = 64 if out == "bf16" else 32
    unnarrowed = -(-Nn // 16) * 16 if nblk0 == 1 else -(-(-(-Nn // nblk0)) // cpb) * cpb
    return ("tc", ind, out, epi, p["num_n"] > 1, Nn % p["BN"] != 0, p["BN"] != unnarrowed, bool(p["split"]),
            "deep" if p["cpw"] == 1 else "classic")


@contextlib.contextmanager
def gemm_hook():
    """nfdpm_gemm_debug's per-CTA counters [sms][16] int64 for the launches inside the block.  The hook is reset to NULL
    (and the device synchronised) before the buffer can be freed: a hook left set makes later launches, graph replays
    included, write into freed memory."""
    sms = N.lib.nfdpm_sm_count()
    buf = torch.zeros(sms, 16, dtype=torch.int64, device=DEV)
    torch.cuda.synchronize()
    assert N.lib.nfdpm_gemm_debug(buf.data_ptr()) == 0
    try:
        yield buf
    finally:
        torch.cuda.synchronize()
        N.lib.nfdpm_gemm_debug(None)
        torch.cuda.synchronize()
        del buf


# ------------------------------------------------------------------------------------------------ operands
def operand(rows, k, ld, fmt, seed, scale=1.0, extra_rows=64):
    """A [rows + extra_rows, ld] operand whose first rows x k entries are random and whose padding columns and extra rows
    are NaN -> (device tensor in fmt, fp64 [rows, k] of the values the kernel reads)."""
    x = torch.full((rows + extra_rows, ld), float("nan"))
    x[:rows, :k] = rnd(rows, k, seed=seed, scale=scale)
    if fmt == "split":
        t = SP.encode(x)
        val = SP.value(t, rows + extra_rows, ld)[:rows, :k]
    elif fmt == "bf16":
        t = x.bfloat16()
        val = t[:rows, :k].double()
    else:
        t, val = x, x[:rows, :k].double()
    return t.to(DEV), val.to(DEV)


def check_out(name, got, ref, fmt, rows, cols):
    """got: the [rows, cols] logical output on the host (raw words for split pairs)."""
    if fmt == "f32":
        check(name, got, ref)
    elif fmt == "bf16":
        check_bf16(name, got, ref)
    else:
        hi, lo = SP.decode(got, rows, cols)
        check(name, hi.double() + lo.double(), ref)
        # hi is a nearest bf16 of hi + lo (= bf16(hi + lo) up to ties): |lo| <= half an ulp of hi
        _, e = torch.frexp(hi)
        assert bool((lo.abs() <= torch.ldexp(torch.ones_like(hi), e - 9)).all()), f"{name}: hi is not bf16(hi + lo)"


# ------------------------------------------------------------------------------------------------ gemm_nt, tcgen05
# (id, M, N, K, operands, output); every case runs with both epilogues and lda, ldb > K, ldd > N
NT_TC = [
    ("one_blk_n48_bf16_f32", 1000, 48, 128, "bf16", "f32"),
    ("one_blk_n112_zeroconv_split_f32", 3000, 112, 512, "split", "f32"),
    ("one_blk_n16_m77_single_kb_bf16_bf16", 77, 16, 64, "bf16", "bf16"),
    ("single_kb_split_split", 4096, 256, 32, "split", "split"),
    ("multi_partial_n432_f32_narrow_stopped", 2048, 432, 512, "bf16", "f32"),
    ("multi_partial_n432_split_f32", 2048, 432, 512, "split", "f32"),
    ("narrow_stopped_n432_bf16", 2048, 432, 512, "bf16", "bf16"),
    ("narrow_fires_m2048_n512", 2048, 512, 512, "bf16", "bf16"),
    ("narrow_fires_m2048_n512_split", 2048, 512, 512, "split", "split"),
    ("wide_zeroconv_n3456_split_f32", 300, 3456, 512, "split", "f32"),
    ("wide_zeroconv_n3456_bf16_partial", 300, 3456, 512, "bf16", "bf16"),
    ("split_on_512_tiles_deep", 32768, 512, 512, "bf16", "bf16"),
    ("split_on_split_pairs", 32768, 512, 512, "split", "split"),
    ("split_off_rem0", 18944, 512, 128, "bf16", "bf16"),
    ("split_off_2rem_gt_grid", 31744, 256, 128, "bf16", "bf16"),
    ("split_off_n_not_multiple_of_bn", 5120, 432, 256, "bf16", "f32"),
    ("deep_f32_out_stages", 32768, 512, 256, "bf16", "f32"),
    ("deep_split_f32_out", 8192, 512, 256, "split", "f32"),
    ("classic_kb_not_multiple_of_stages", 8192, 512, 320, "bf16", "bf16"),
    ("m_not_multiple_of_128_split_f32", 1000, 512, 256, "split", "f32"),
    ("m77_split_split", 77, 64, 96, "split", "split"),
    ("narrow_fires_bf16_f32", 2048, 256, 512, "bf16", "f32"),
    ("one_blk_n112_deep_split_f32", 32768, 112, 512, "split", "f32"),
    ("one_blk_n64_deep_bf16_f32", 32768, 64, 512, "bf16", "f32"),
    ("split_on_classic", 32768, 512, 128, "bf16", "bf16"),
    ("split_on_classic_split_pairs", 32768, 512, 64, "split", "split"),
    ("classic_one_wave_split_pairs", 8192, 512, 128, "split", "split"),
]
EPIS = [N.EPI_RAW, N.EPI_ACTNORM_RELU]
# the fused ActNorm epilogue supports N <= 2048
NT_TC_RUNS = [pytest.param(c, e, id=f"{c[0]}-{'raw' if e == N.EPI_RAW else 'actnorm_relu'}") for c in NT_TC for e in EPIS
              if e == N.EPI_RAW or c[2] <= 2048]


def run_nt(M, Nn, K, ind, out, epi, lda, ldb, ldd, d_off=0, seed=0, hook=False):
    """One guarded gemm_nt call -> (logical [M, N] host output, fp64 reference on the device, hook counters or None,
    the raw sink buffer)."""
    a, av = operand(M, K, lda, ind, seed + 1)
    b, bv = operand(Nn, K, ldb, ind, seed + 2, scale=0.1)
    es, eb = rnd(Nn, seed=seed + 3, scale=0.2).to(DEV), rnd(Nn, seed=seed + 4).to(DEV)
    rows = M + 2
    d = Sink(rows * ldd + d_off, _FMT[out])
    D = d.t[d_off:]
    with gemm_hook() if hook else contextlib.nullcontext() as h:
        N.gemm_nt(a, lda, b, ldb, D, ldd, M, Nn, K, epi, es, eb)
        counters = h.cpu() if hook else None
    mask = torch.zeros(rows, ldd, dtype=torch.bool)
    mask[:M, :Nn] = True
    if out == "split":
        mask = split_words(mask)
    written = torch.cat([torch.zeros(d_off, dtype=torch.bool), mask.reshape(-1)])
    got = d.get(written)[d_off:].view(rows, ldd)[:M, :Nn]
    ref = av @ bv.T
    if epi == N.EPI_ACTNORM_RELU:
        ref = torch.relu(torch.exp(es.double()) * (ref + eb.double()))
    return got, ref.cpu(), counters, d.buf.cpu()


@gpu
@pytest.mark.parametrize("case,epi", NT_TC_RUNS)
def test_gemm_nt_tensor_core(case, epi):
    name, M, Nn, K, ind, out = case
    lda, ldb = K + 32, K + 64
    ldd = Nn + 32
    p = nt_plans([(M, Nn, K, ind, out, epi)])[0]
    br = nt_branch(M, Nn, K, ind, out, epi, p)
    print(f"\n[plan] {name}: {p}")
    # the branch the case is named for
    want = {"one_blk": not br[4], "multi_partial": br[4] and br[5], "narrow_fires": br[6], "split_on": br[7],
            "single_kb": K * (2 if ind == "split" else 1) == 64, "deep": br[8] == "deep", "classic": br[8] == "classic",
            "m77": M < 128 and p["grid"] < 148, "m_not_multiple": M % 128 != 0}
    for key, ok in want.items():
        if key in name:
            assert ok, f"{name}: branch {key} not taken ({p})"
    nb0 = 128 if out == "f32" else 256
    if "narrow_stopped" in name:        # narrowing would fire on the tile count but N % (bn / 2) != 0 stops it
        assert (M + 127) // 128 * -(-Nn // nb0) <= 74 and Nn % (nb0 // 2) != 0 and not br[6]
    if "split_off" in name:
        assert p["tiles"] > p["grid"] and not p["split"]
    if "rem0" in name:
        assert p["tiles"] % p["grid"] == 0
    if "2rem_gt_grid" in name:
        assert 2 * (p["tiles"] % p["grid"]) > p["grid"]
    if "n_not_multiple_of_bn" in name:
        assert 2 * (p["tiles"] % p["grid"]) <= p["grid"] and Nn % p["BN"] != 0
    if "not_multiple_of_stages" in name:
        assert (K // 64) % p["n_stages"] != 0
    if name == "split_on_512_tiles_deep":
        assert p["tiles"] >= 3 * 148 and p["n_stages"] == 4
    if name == "deep_f32_out_stages":   # the ActNorm scratch takes one stage of the fp32-output deep ring
        assert p["BN"] == 128 and p["n_stages"] == (6 if epi == N.EPI_RAW else 5)
    got, ref, h, raw = run_nt(M, Nn, K, ind, out, epi, lda, ldb, ldd, seed=M % 97, hook=True)
    check_out(name, got, ref, out, M, Nn)
    # grid and units of work through the profiling hook: every CTA of the grid ran; the units are the tiles, plus one
    # more per tile of the split last round
    ctas = int((h[:, 0] != 0).sum())
    assert ctas == p["grid"] and bool((h[:ctas, 0] != 0).all()), (ctas, p)
    units = int(h[:, 10].sum())
    rem = p["tiles"] % p["grid"] if p["split"] else 0
    assert units == p["tiles"] + rem, (units, p)
    # repeated call: the same bits everywhere in the buffer
    raw2 = run_nt(M, Nn, K, ind, out, epi, lda, ldb, ldd, seed=M % 97)[3]
    assert same_bits(raw, raw2), f"{name}: a repeated call gave other bits"


def test_nt_cases_cover_every_operand_output_pair_and_both_plans():
    pairs = {(c[4], c[5]) for c in NT_TC}
    assert pairs == {("bf16", "f32"), ("bf16", "bf16"), ("split", "f32"), ("split", "split")}
    plans = nt_plans([(c[1], c[2], c[3], c[4], c[5], e) for c, e in (r.values for r in NT_TC_RUNS)])
    assert {p["cpw"] for p in plans} == {1, 2, 4} and {p["n_stages"] for p in plans} >= {3, 4, 5, 6}
    assert any(p["split"] for p in plans) and any(p["grid"] < 148 for p in plans)


# ------------------------------------------------------------------------------------------------ gemm_nt, CUDA core
# (id, M, N, K, output, D offset in elements, lda padding)
NT_SIMT = [
    ("bn64_n12", 300, 12, 64, "f32", 0, 16),
    ("bn64_n6_scalar_tail", 257, 6, 32, "f32", 0, 0),
    ("bn64_n40_bf16_out", 1000, 40, 64, "bf16", 0, 16),
    ("bn64_n6_bf16_scalar_tail", 130, 6, 16, "bf16", 0, 32),
    ("bn128_n112", 500, 112, 512, "f32", 0, 16),
    ("bn128_n130_scalar_tail", 200, 130, 96, "f32", 0, 0),
    ("bn128_n200_bf16_out", 129, 200, 64, "bf16", 0, 16),
    ("bn128_d_offset_4_bytes", 300, 72, 64, "f32", 1, 16),
    ("bn64_d_offset_bf16", 77, 24, 48, "bf16", 1, 0),
]


@gpu
@pytest.mark.parametrize("epi", EPIS, ids=["raw", "actnorm_relu"])
@pytest.mark.parametrize("case", NT_SIMT, ids=[c[0] for c in NT_SIMT])
def test_gemm_nt_cuda_core(case, epi):
    name, M, Nn, K, out, d_off, pad = case
    lda, ldb, ldd = K + pad, K + 8, (Nn + 7) // 8 * 8 + 8
    assert ("bn64" in name) == (Nn <= 64) and ("scalar_tail" in name) <= (Nn % 4 != 0) and ("offset" in name) == (d_off > 0)
    got, ref, _, raw = run_nt(M, Nn, K, "f32", out, epi, lda, ldb, ldd, d_off, seed=M % 89)
    check_out(name, got, ref, out, M, Nn)
    assert same_bits(raw, run_nt(M, Nn, K, "f32", out, epi, lda, ldb, ldd, d_off, seed=M % 89)[3])


# ------------------------------------------------------------------------------------------------ gemm_tn
def tn_kernel_dims(fmt, N1, N2):
    return (2 * ((N1 + 31) // 32 * 32), 2 * ((N2 + 31) // 32 * 32)) if fmt == "split" else (N1, N2)


def tn_workspace_replica(M, N1, N2):
    """nfdpm_gemm_tn_workspace: the largest of the CUDA-core, bf16 and split-pair path's slabs."""
    tiles = ((N1 + 127) // 128) * ((N2 + 127) // 128)
    splits = max(1, min((296 + tiles - 1) // tiles, (M + 255) // 256))
    s_tc = N.gemm_tn_tc_plan(M, N1, N2)[2]
    n1m, n2m = tn_kernel_dims("split", N1, N2)
    return max(max(splits, s_tc) * N1 * N2, N.gemm_tn_tc_plan(M, n1m, n2m)[2] * n1m * n2m)


def test_gemm_tn_replica_matches_the_workspace_query():
    """The plan replica behind gemm_tn_path / the launch count against the library's own workspace query (which runs
    without a GPU: 148 SMs), over a grid of shapes."""
    if N.lib.nfdpm_sm_count() not in (-1, 148):
        pytest.skip("the grid of shapes is sized for 148 SMs")
    for M in (1, 60, 64, 1000, 3000, 4100, 32768, 262144):
        for N1 in (12, 24, 112, 128, 200, 432, 512, 1536, 3456, 6912):
            for N2 in (16, 48, 64, 112, 256, 432, 512, 2560):
                assert N.gemm_tn_workspace(M, N1, N2) == tn_workspace_replica(M, N1, N2), (M, N1, N2)


def test_gemm_tn_launch_count_follows_the_path():
    assert N.gemm_tn_path(N.BF16, N.BF16, True, 256, 2048, 2560, True, N.TN_OUT_PLAIN) == ("tc", "reduce_rows")
    assert N.gemm_tn_path(N.BF16X2, N.BF16X2, True, 200, 3456, 512, True, N.TN_OUT_TAPS) == ("x3", "tn_reduce")
    assert N.gemm_tn_path(N.BF16, N.BF16, True, 2000, 128, 64, True, N.TN_OUT_PLAIN) == ("tc", "in_kernel")
    assert N.gemm_tn_path(N.F32, N.F32, True, 2000, 128, 64, True, N.TN_OUT_PLAIN) == ("simt", "reduce_rows")


# (id, M, N1, lda, N2, ldb, operands, out mode, out_c, fused_reduce, expected (gemm, reduction))
TN = [
    ("tc_bn64_partial_many_splits", 3000, 128, 136, 48, 64, "bf16", N.TN_OUT_PLAIN, 0, True, ("tc", "in_kernel")),
    ("tc_bn128_partial_n1_partial", 1000, 200, 208, 112, 128, "bf16", N.TN_OUT_PLAIN, 0, True, ("tc", "in_kernel")),
    ("tc_bn256_partial", 4100, 300, 304, 432, 448, "bf16", N.TN_OUT_PLAIN, 0, True, ("tc", "in_kernel")),
    ("tc_one_split_m60", 60, 512, 512, 256, 264, "bf16", N.TN_OUT_PLAIN, 0, True, ("tc", "in_kernel")),
    ("tc_unfused_reduce_rows", 2000, 128, 128, 64, 64, "bf16", N.TN_OUT_PLAIN, 0, False, ("tc", "reduce_rows")),
    ("tc_not_coresident_reduce_rows", 256, 2048, 2048, 2560, 2560, "bf16", N.TN_OUT_PLAIN, 0, True, ("tc", "reduce_rows")),
    ("tc_taps_ldp_gt_9c", 2000, 112, 128, 512, 512, "bf16", N.TN_OUT_TAPS, 12, True, ("tc", "in_kernel")),
    ("tc_strip_out_c_27", 3000, 512, 512, 32, 32, "bf16", N.TN_OUT_STRIP, 27, True, ("tc", "in_kernel")),
    ("x3_plain_in_kernel", 2000, 112, 128, 512, 512, "split", N.TN_OUT_PLAIN, 0, True, ("x3", "in_kernel")),
    ("x3_one_split_m60", 60, 96, 96, 64, 64, "split", N.TN_OUT_PLAIN, 0, True, ("x3", "in_kernel")),
    ("x3_taps_ldp_gt_9c", 1500, 112, 128, 512, 512, "split", N.TN_OUT_TAPS, 12, True, ("x3", "in_kernel")),
    ("x3_strip_out_c_27", 3000, 512, 512, 64, 64, "split", N.TN_OUT_STRIP, 27, True, ("x3", "in_kernel")),
    ("x3_taps_zeroconv_c384_tn_reduce", 200, 3456, 3456, 512, 512, "split", N.TN_OUT_TAPS, 384, True, ("x3", "tn_reduce")),
    ("x3_plain_tn_reduce", 200, 1536, 1536, 1024, 1024, "split", N.TN_OUT_PLAIN, 0, True, ("x3", "tn_reduce")),
    ("x3_strip_tn_reduce", 130, 3072, 3072, 480, 480, "split", N.TN_OUT_STRIP, 477, True, ("x3", "tn_reduce")),
    ("simt_f32_f32", 1500, 24, 32, 112, 112, "f32/f32", N.TN_OUT_PLAIN, 0, True, ("simt", "reduce_rows")),
    ("simt_f32_bf16", 700, 40, 48, 72, 80, "f32/bf16", N.TN_OUT_PLAIN, 0, True, ("simt", "reduce_rows")),
    ("simt_bf16_f32", 1100, 130, 136, 20, 24, "bf16/f32", N.TN_OUT_PLAIN, 0, False, ("simt", "reduce_rows")),
    ("simt_bf16_rejected_by_tc", 900, 64, 64, 40, 40, "bf16", N.TN_OUT_PLAIN, 0, True, ("simt", "reduce_rows")),
]
# an interleaved call of another shape between a case's two calls: a counter that fails to re-arm shows up there
_OTHER = ("other", 300, 256, 256, 64, 64, "bf16", N.TN_OUT_PLAIN, 0, True, ("tc", "in_kernel"))


def _tn_formats(fmt):
    return fmt.split("/") if "/" in fmt else (fmt, fmt)


def tn_branch(M, N1, N2, fa, fb, tc_ok, fused, mode):
    """(gemm, reduction, BN, several M splits, output mode); coverage asks for the output mode and the tiling separately."""
    gemm, red = N.gemm_tn_path(_CODE[fa], _CODE[fb], tc_ok, M, N1, N2, fused, mode)
    if gemm == "simt":
        return (gemm, red, 0, False, mode)
    bn, tiles, splits, _ = N.gemm_tn_tc_plan(M, *tn_kernel_dims(fa, N1, N2))
    return (gemm, red, bn, splits > 1, mode)


def _tn_parts(b):
    return {("tn_mode",) + b[:2] + b[4:], ("tn_tiling",) + b[:4]}


def run_tn(case, accumulate=False, old=None, d_align=0):
    """One guarded gemm_tn call -> (D host output, fp64 reference of D's layout, workspace buffer)."""
    name, M, N1, lda, N2, ldb, fmt, mode, out_c, fused, _ = case
    fa, fb = _tn_formats(fmt)
    a, av = operand(M, N1, lda, fa, 11)
    b, bv = operand(M, N2, ldb, fb, 12)
    ref = av.T @ bv
    if mode == N.TN_OUT_TAPS:               # n1 = tap*out_c + co -> [co][n2][tap]
        want = ref[:9 * out_c].reshape(9, out_c, N2).permute(1, 2, 0).reshape(-1)
    elif mode == N.TN_OUT_STRIP:
        want = ref[:, :out_c].reshape(-1)
    else:
        want = ref.reshape(-1)
    n_ws = N.gemm_tn_workspace(M, N1, N2)
    # guard: room for whatever a workspace sized for the plain operands or a missing row check could write past it
    # (the whole split-pair slabs; 128 slab rows)
    k1, k2 = tn_kernel_dims(fa, N1, N2)
    ws = Sink(n_ws, slack=(N.gemm_tn_tc_plan(M, k1, k2)[2] * k1 * k2 if fa == "split" else 0) + 128 * k2 + 64)
    d = Sink(want.numel() + d_align, init=None if old is None else torch.cat([torch.zeros(d_align), old]))
    D = d.t[d_align:]
    cnt = N._tn_counters(torch.device(DEV))
    l0 = N.launch_count
    N.gemm_tn(a, lda, b, ldb, D, M, N1, N2, ws.t, accumulate=accumulate, fused_reduce=fused, out_mode=mode, out_c=out_c)
    launches = N.launch_count - l0
    torch.cuda.synchronize()
    assert int(cnt.abs().sum()) == 0, f"{name}: tile counters not re-armed"
    ws.get()                                 # the guard around the workspace is untouched
    got = d.get(torch.cat([torch.zeros(d_align, dtype=torch.bool), torch.ones(want.numel(), dtype=torch.bool)]))
    return got[d_align:], want.cpu(), launches


@gpu
@pytest.mark.parametrize("case", TN, ids=[c[0] for c in TN])
def test_gemm_tn(case):
    name, M, N1, lda, N2, ldb, fmt, mode, out_c, fused, path = case
    fa, fb = _tn_formats(fmt)
    tc_ok = lda % 8 == 0 and ldb % 8 == 0 and N2 % 16 == 0
    br = tn_branch(M, N1, N2, fa, fb, tc_ok, fused, mode)
    assert br[:2] == path, (name, br)
    if "bn64" in name or "bn128" in name or "bn256" in name:
        assert f"bn{br[2]}" in name and N2 % br[2] != 0
    if "many_splits" in name:
        assert br[3]
    if "one_split" in name:
        assert not br[3] and M % 64 != 0
    if "ldp_gt_9c" in name:
        assert N1 > 9 * out_c
    if mode == N.TN_OUT_STRIP:
        assert out_c % 4 != 0
    got, want, launches = run_tn(case)
    check(name, got, want)
    assert launches == (1 if path[1] == "in_kernel" else 2), (name, launches)
    run_tn(_OTHER)
    got2 = run_tn(case)[0]
    assert same_bits(got, got2), f"{name}: a repeated call gave other bits"
    # accumulate: every path adds the old D to the finished slab sum (tn_reduce_item: after the slab loop;
    # reduce_rows_kernel: out + s), so the result is the fp32 sum of the plain result and the old D, bit for bit
    old = rnd(want.numel(), seed=5)
    acc = run_tn(case, accumulate=True, old=old)[0]
    assert same_bits(acc, got + old), f"{name}: accumulate is not D + the non-accumulating result"


@gpu
@pytest.mark.parametrize("fmt", ["split", "bf16"])
def test_gemm_tn_rejects_a_misaligned_plain_d_before_any_launch(fmt):
    """The tensor-core reduction stores float4 rows into a plain D: a D that is not 16-byte aligned is refused before
    any launch (D and the workspace untouched)."""
    M, N1, N2 = 500, 64, 64
    a, _ = operand(M, N1, 64, fmt, 1)
    b, _ = operand(M, N2, 64, fmt, 2)
    d = Sink(N1 * N2 + 1)
    ws = Sink(N.gemm_tn_workspace(M, N1, N2))
    l0 = N.launch_count
    with pytest.raises(RuntimeError, match="16-byte aligned"):
        N.gemm_tn(a, 64, b, 64, d.t[1:], M, N1, N2, ws.t)
    torch.cuda.synchronize()
    assert N.launch_count == l0
    d.get(torch.zeros(N1 * N2 + 1, dtype=torch.bool))
    ws.get(torch.zeros(ws.n, dtype=torch.bool))
    # the layout-changing outputs store scalars: an unaligned D is fine there
    got, want, _ = run_tn(("strip_unaligned", M, N1, 64, N2, 64, fmt, N.TN_OUT_STRIP, 27, True, None), d_align=1)
    check("strip_unaligned", got, want)


# ------------------------------------------------------------------------------------------------ production shapes
def _table_branches():
    nt = [(c[1], c[2], c[3], c[4], c[5], e) for c, e in (r.values for r in NT_TC_RUNS)]
    out = {nt_branch(*q, p) for q, p in zip(nt, nt_plans(nt))}
    out |= {nt_branch(c[1], c[2], c[3], "f32", c[4], e) for c in NT_SIMT for e in EPIS}
    for c in TN:
        fa, fb = _tn_formats(c[6])
        tc_ok = c[3] % 8 == 0 and c[5] % 8 == 0 and c[4] % 16 == 0
        out |= _tn_parts(tn_branch(c[1], c[2], c[4], fa, fb, tc_ok, c[9], c[7]))
    return out


_NAME = {torch.float32: "f32", torch.bfloat16: "bf16", N.SPLIT: "split"}


@gpu
def test_production_calls_are_covered(monkeypatch):
    """Every gemm_nt / gemm_tn call of the config-2 forward, inverse and training step, config-4 sampling and the L6
    wide-level forward and training step maps to a branch tuple some case above covers."""
    import normalizing_flow as nf
    from oracle import glow_oracle as O
    calls = []
    nt0, tn0 = N.gemm_nt, N.gemm_tn

    def nt(A, lda, Bw, ldb, D, ldd, M, Nn, K, epilogue=N.EPI_RAW, ep_scale=None, ep_bias=None):
        calls.append(("nt", M, Nn, K, _NAME[A.dtype], _NAME[D.dtype], epilogue))
        return nt0(A, lda, Bw, ldb, D, ldd, M, Nn, K, epilogue, ep_scale, ep_bias)

    def tn(A, lda, Bm, ldb, D, M, N1, N2, ws, accumulate=False, fused_reduce=True, out_mode=N.TN_OUT_PLAIN, out_c=0):
        calls.append(("tn", M, N1, N2, _NAME[A.dtype], _NAME[Bm.dtype], N.gemm_tn_tc_ok(A, lda, Bm, ldb, N2),
                      fused_reduce, out_mode))
        return tn0(A, lda, Bm, ldb, D, M, N1, N2, ws, accumulate, fused_reduce, out_mode, out_c)

    monkeypatch.setattr(N, "gemm_nt", nt)
    monkeypatch.setattr(N, "gemm_tn", tn)

    def model(c, L, K, B, S, seed):
        sd, psd = O.seeded_state(c, L, K, seed)
        flow = nf.Glow(c, L, K).to(DEV)
        flow.load_state_dict(sd)
        prior = nf.GaussianPrior(2 ** (L + 1) * c).to(DEV)
        prior.load_state_dict(psd)
        return flow, prior, O.seeded_input((B, c, S, S), seed + 1).to(DEV)

    def forward_inverse_train(flow, prior, x, S, inverse=True, sample=False):
        B = x.shape[0]
        with torch.no_grad():
            ld, lp = nf.initialize_with_zeros(2, B, DEV)
            zs, ld, lp = flow.transform(x, ld, lp)
            if inverse:
                flow.invert(zs)
            if sample:
                flow.invert([zs[-1]])
        flow.zero_grad(set_to_none=True)
        ld, lp = nf.initialize_with_zeros(2, B, DEV)
        zs, ld, lp = flow.transform(x, ld, lp)
        lp = lp + prior.compute_log_prob(zs[-1])
        nf.calculate_loss(ld + lp, 32.0, S * S * 3.0).backward()

    forward_inverse_train(*model(3, 3, 16, 128, 32, 3), 32)
    flow, prior, x = model(3, 5, 16, 8, 128, 5)
    with torch.no_grad():
        ld, lp = nf.initialize_with_zeros(2, 8, DEV)
        zs, _, _ = flow.transform(x, ld, lp)
        flow.invert([zs[-1]])
    forward_inverse_train(*model(3, 6, 2, 2, 64, 7), 64, inverse=False)
    torch.cuda.synchronize()
    assert calls, "no GEMM call recorded"
    covered = _table_branches()
    nt_calls = sorted({c for c in calls if c[0] == "nt"})
    branches = {}
    nt_tc = [c for c in nt_calls if c[4] != "f32"]
    for c, p in zip(nt_tc, nt_plans([c[1:] for c in nt_tc])):
        branches[c] = nt_branch(*c[1:], p)
    for c in nt_calls:
        if c[4] == "f32":
            branches[c] = nt_branch(*c[1:])
    for c in {c for c in calls if c[0] == "tn"}:
        _, M, N1, N2, fa, fb, tc_ok, fused, mode = c
        branches[c] = tn_branch(M, N1, N2, fa, fb, tc_ok, fused, mode)
    print(f"\n[production] {len(calls)} calls, {len(branches)} shapes, {len(set(branches.values()))} branch tuples")
    missing = {c: b for c, b in branches.items()
               if (_tn_parts(b) - covered if c[0] == "tn" else {b} - covered)}
    assert not missing, "branches no case covers:\n" + "\n".join(f"{c} -> {b}" for c, b in sorted(missing.items(), key=str))
