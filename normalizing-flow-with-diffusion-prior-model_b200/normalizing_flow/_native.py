"""ctypes binding of libnfdpm_b200.so (include/nfdpm_b200.h).

There is no fallback: if the shared library is missing or a kernel call fails this module raises.
Every wrapper enqueues on torch's *current* CUDA stream and passes raw device pointers; torch is used
only for memory and streams.
"""
from __future__ import annotations

import ctypes as C
import functools
import os
from typing import Optional

import torch

F32, F64, BF16, BF16X2 = 0, 1, 2, 3
EPI_RAW, EPI_ACTNORM_RELU = 0, 1

#: torch storage dtype of split bf16 pairs (NFDPM_BF16X2, include/nfdpm_b200.h): 4 bytes per LOGICAL element — a row of ld
#: logical columns is 2*ld bf16 (hi / lo planes interleaved in groups of 32).  torch has no such dtype; int32 buffers carry
#: the words and ``_dt`` maps them to the NFDPM_BF16X2 code.  Only the kernels interpret the contents.
SPLIT = torch.int32

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("NFDPM_B200_LIB", os.path.join(os.path.dirname(_HERE), "lib", "libnfdpm_b200.so"))


class MixItem(C.Structure):
    """struct nfdpm_mix_item (include/nfdpm_b200.h)."""
    _fields_ = [("weight", C.c_void_p), ("scale", C.c_void_p), ("bias", C.c_void_p), ("C", C.c_int32),
                ("pad_", C.c_int32), ("fwd_mt", C.c_void_p), ("fwd_beta", C.c_void_p), ("inv_mt", C.c_void_p),
                ("inv_beta", C.c_void_p), ("winv", C.c_void_p), ("logdet", C.c_void_p), ("lu_ws", C.c_void_p)]


class LatentPart(C.Structure):
    """struct nfdpm_latent_part (include/nfdpm_b200.h)."""
    _fields_ = [("ptr", C.c_void_p), ("C", C.c_int32), ("H", C.c_int32), ("W", C.c_int32), ("degree", C.c_int32),
                ("ch_offset", C.c_int32), ("ch_count", C.c_int32)]


class MixGradItem(C.Structure):
    """struct nfdpm_mix_grad_item (include/nfdpm_b200.h)."""
    _fields_ = [("part", C.c_void_p), ("B", C.c_int32), ("C", C.c_int32), ("weight", C.c_void_p), ("scale", C.c_void_p),
                ("bias", C.c_void_p), ("winv", C.c_void_p), ("dld_sum", C.c_void_p), ("P", C.c_float), ("pad_", C.c_int32),
                ("d_weight", C.c_void_p), ("d_scale", C.c_void_p), ("d_bias", C.c_void_p), ("scratch", C.c_void_p)]


def _load() -> C.CDLL:
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"libnfdpm_b200.so not found at {LIB_PATH}. Build it with `python -c 'import __graft_entry__ as g; "
            f"g.build()'` (nvcc, sm_100a). This package has no CPU or PyTorch fallback.")
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64, f32, u32 = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_uint32
    sig = {
        "nfdpm_version": ([], C.c_int),
        "nfdpm_last_error_string": ([], C.c_char_p),
        "nfdpm_sm_count": ([], C.c_int),
        "nfdpm_ld_tiles": ([i32], C.c_int),
        "nfdpm_mix_prepare": ([C.POINTER(MixItem), i32, vp], C.c_int),
        "nfdpm_channel_mix": ([vp, vp, vp, vp, i32, i32, i32, i64, i64, vp], C.c_int),
        "nfdpm_actnorm_apply": ([vp, vp, vp, vp, i32, i32, i32, i32, vp], C.c_int),
        "nfdpm_channel_stats": ([vp, i32, i32, i32, i32, i64, vp, vp, vp], C.c_int),
        "nfdpm_squeeze": ([vp, vp, i32, i32, i32, i32, i64, i64, vp], C.c_int),
        "nfdpm_unsqueeze": ([vp, vp, i32, i32, i32, i32, i64, i64, vp], C.c_int),
        "nfdpm_copy_channels": ([vp, vp, i32, i32, i32, i64, i64, vp], C.c_int),
        "nfdpm_im2col3x3": ([vp, vp, i32, i32, i32, i32, i32, i64, i64, vp], C.c_int),
        "nfdpm_pack_matrix": ([vp, vp, i32, i32, i32, i32, i64, i64, i64, i64, i32, vp], C.c_int),
        "nfdpm_gemm_nt": ([vp, i64, vp, i64, vp, i64, i32, i32, i32, i32, i32, i32, vp, vp, vp], C.c_int),
        "nfdpm_coupling_apply": ([vp, i64, vp, vp, vp, vp, vp, i32, i32, i32, i32, i64, i64, i32, vp], C.c_int),
        "nfdpm_split_prior_logp": ([vp, i64, vp, vp, vp, i64, vp, vp, i32, i32, i32, i32, vp], C.c_int),
        "nfdpm_split_prior_sample": ([vp, i64, vp, vp, vp, f32, vp, i64, i32, i32, i32, i32, vp], C.c_int),
        "nfdpm_gauss_logp_const": ([vp, vp, vp, vp, i32, i32, i32, vp], C.c_int),
        "nfdpm_gauss_sample_const": ([vp, vp, vp, f32, vp, i32, i32, i32, vp], C.c_int),
        "nfdpm_split_prior_sample_ex": ([vp, i64, vp, vp, vp, vp, u32, f32, vp, vp, vp, i64, i32, i32, i32, i32, vp], C.c_int),
        "nfdpm_gauss_sample_const_ex": ([vp, vp, u32, vp, vp, f32, vp, vp, vp, i32, i32, i32, vp], C.c_int),
        "nfdpm_rows_to_nchw": ([vp, i64, i32, vp, vp, vp, i32, i32, i32, vp], C.c_int),
        "nfdpm_nchw_to_rows": ([vp, vp, i32, i32, i32, i32, i64, i64, vp], C.c_int),
        "nfdpm_flow_boundary_smem": ([i32, i32, i32, i32, i32], C.c_size_t),
        "nfdpm_flow_boundary": ([vp, i64, i32, vp, i64, vp, vp, vp, vp, vp, vp, i64, vp, i32, i64, i32, i32, i32, i32,
                                 i32, vp], C.c_int),
        "nfdpm_coupling_bwd": ([vp, i64, vp, vp, i64, vp, i64, vp, vp, vp, i64, vp, i32, i64, vp, vp, vp, vp, vp, i32, i32,
                                i32, i32, vp], C.c_int),
        "nfdpm_coupling_inv_bwd": ([vp, i64, vp, i64, vp, i64, vp, vp, vp, i64, vp, i32, i64, vp, vp, vp, vp, vp, i32, i32,
                                    i32, i32, vp], C.c_int),
        "nfdpm_coupling_inv_bwd_ld": ([vp, i64, vp, vp, i64, vp, i64, vp, vp, vp, i64, vp, i32, i64, vp, vp, vp, vp, vp, i32,
                                       i32, i32, i32, vp], C.c_int),
        "nfdpm_coupling_bwd_tiles": ([i32, i32, i32], C.c_int),
        "nfdpm_mix_bwd_tiles": ([i32, i32, i32], C.c_int),
        "nfdpm_flow_boundary_stash": ([vp, i64, i32, vp, i64, vp, vp, vp, vp, vp, vp, i64, vp, i64, vp, i32, i64, i32, i32,
                                       i32, i32, vp], C.c_int),
        "nfdpm_flow_boundary_inv_stash": ([vp, i64, vp, i64, vp, vp, vp, vp, vp, i64, vp, i64, vp, i32, i64, i32, i32, i32, i32,
                                           vp], C.c_int),
        "nfdpm_flow_boundary_inv_stash_ld": ([vp, i64, vp, i64, vp, vp, vp, vp, vp, vp, i64, vp, i64, vp, i32, i64, i32, i32,
                                              i32, i32, vp], C.c_int),
        "nfdpm_actnorm_relu_bwd": ([vp, i32, i64, vp, i32, i64, vp, vp, i32, i64, vp, i32, i32, i32, vp], C.c_int),
        "nfdpm_reduce_rows2": ([vp, vp, vp, i32, i32, i32, i64, vp], C.c_int),
        "nfdpm_gemm3_boundary_ok": ([i32, i32, i32, i32, i32, i64], C.c_int),
        "nfdpm_gemm3_boundary": ([vp, i32, i64, vp, vp, i64, vp, i64, vp, vp, vp, vp, vp, vp, i64, vp, i64, vp, i32, i64, i32, i32,
                                  i32, i32, i32, i64, i32, vp], C.c_int),
        "nfdpm_gemm_debug": ([vp], C.c_int),
        "nfdpm_flow_boundary_debug": ([vp], C.c_int),
        "nfdpm_opt_chunk": ([], C.c_int),
        "nfdpm_pack_elems": ([], C.c_int),
        "nfdpm_pack_batch": ([vp, i32, i32, vp], C.c_int),
        "nfdpm_fused_clip_adam": ([vp, vp, i32, vp, vp, vp, vp, C.c_float, C.c_float, C.c_double, C.c_double, C.c_double,
                                   C.c_double, C.c_double, i32, vp], C.c_int),
        "nfdpm_reduce_rows": ([vp, vp, i32, i32, i64, i32, vp], C.c_int),
        "nfdpm_mix_bwd": ([vp, i64, vp, i64, vp, i64, vp, vp, i64, vp, i32, i32, i32, i32, vp], C.c_int),
        "nfdpm_mix_param_grad": ([C.POINTER(MixGradItem), i32, vp], C.c_int),
        "nfdpm_mix_inv_param_grad": ([C.POINTER(MixGradItem), i32, vp], C.c_int),
        "nfdpm_gemm_tn_workspace": ([i32, i32, i32, C.POINTER(C.c_int)], C.c_int64),
        "nfdpm_gemm_tn": ([vp, i32, i64, vp, i32, i64, vp, i64, i32, i32, i32, vp, i32, vp, i32, i32, vp], C.c_int),
        "nfdpm_split_prior_bwd": ([vp, vp, i64, vp, vp, vp, i64, vp, i64, vp, vp, i32, i32, i32, i32, vp], C.c_int),
        "nfdpm_gauss_const_bwd": ([vp, vp, vp, vp, vp, vp, i32, i32, i32, vp], C.c_int),
        "nfdpm_split_sample_bwd": ([vp, i64, vp, f32, vp, i64, vp, vp, vp, vp, i32, i32, i32, i32, vp], C.c_int),
        "nfdpm_split_sample_bwd_lp": ([vp, i64, vp, vp, f32, vp, i64, vp, vp, vp, vp, i32, i32, i32, i32, vp], C.c_int),
        "nfdpm_split_sample_bwd_ex": ([vp, i64, vp, f32, vp, vp, vp, i64, vp, vp, vp, vp, i32, i32, i32, i32, vp], C.c_int),
        "nfdpm_col2im_add": ([vp, i64, vp, i64, i32, i32, i32, i32, vp], C.c_int),
        "nfdpm_accumulate": ([vp, i32, vp, i32, i32, vp, vp, i32, vp], C.c_int),
        "nfdpm_flow_boundary_tiles": ([i32, i32, i32, i32, i32, i32, i32], C.c_int),
        "nfdpm_flow_boundary_tiled": ([vp, i64, i32, vp, i64, vp, vp, vp, vp, vp, vp, i64, vp, i64, vp, i32, i64, i32, i32,
                                       i32, i32, i32, i32, vp], C.c_int),
        "nfdpm_latent_format": ([C.POINTER(LatentPart), i32, vp, i32, i32, i32, i32, i32, vp], C.c_int),
        "nfdpm_postprocess_u8": ([vp, vp, i64, f32, f32, vp], C.c_int),
        "nfdpm_preprocess": ([vp, vp, vp, i64, i32, f32, vp], C.c_int),
    }
    for name, (args, res) in sig.items():
        fn = getattr(lib, name)   # AttributeError here == header / library mismatch: fail loudly
        fn.argtypes = args
        fn.restype = res
    return lib


lib = _load()

#: NVTX ranges per kernel family around every launch (NFDPM_NVTX=1; off by default: a range push/pop per launch costs host
#: time in the un-captured paths).  Families group the entry points the way DESIGN.md's kernel table does.
_FAMILIES = (("gemm", ("nfdpm_gemm_nt", "nfdpm_gemm_tn")),
             ("step_boundary", ("nfdpm_flow_boundary", "nfdpm_gemm3_boundary", "nfdpm_channel_mix", "nfdpm_coupling_apply",
                                "nfdpm_im2col3x3", "nfdpm_actnorm_apply", "nfdpm_squeeze", "nfdpm_unsqueeze", "nfdpm_copy_channels")),
             ("prior", ("nfdpm_split_prior", "nfdpm_gauss", "nfdpm_accumulate")),
             ("prepare", ("nfdpm_mix_prepare", "nfdpm_pack", "nfdpm_channel_stats", "nfdpm_rows_to_nchw", "nfdpm_nchw_to_rows")),
             ("backward", ("nfdpm_coupling_bwd", "nfdpm_coupling_inv_bwd", "nfdpm_mix_bwd", "nfdpm_mix_param_grad",
                           "nfdpm_mix_inv_param_grad", "nfdpm_split_sample_bwd", "nfdpm_flow_boundary_inv_stash",
                           "nfdpm_actnorm_relu_bwd", "nfdpm_reduce_rows",
                           "nfdpm_col2im_add")),
             ("optimizer", ("nfdpm_fused_clip_adam",)),
             ("formats", ("nfdpm_latent_format", "nfdpm_postprocess_u8", "nfdpm_preprocess")))


def _family(name: str) -> str:
    """The family of the longest listed prefix of ``name``."""
    best, fam_best = 0, "misc"
    for fam, prefixes in _FAMILIES:
        for p in prefixes:
            if name.startswith(p) and len(p) > best:
                best, fam_best = len(p), fam
    return fam_best


class _RangedLib:
    """The bound library with an NVTX range ("family:entry point") around every call."""

    def __init__(self, inner: C.CDLL):
        self._inner = inner

    def __getattr__(self, name: str):
        fn = getattr(self._inner, name)
        label = f"{_family(name)}:{name}"

        def call(*args):
            torch.cuda.nvtx.range_push(label)
            try:
                return fn(*args)
            finally:
                torch.cuda.nvtx.range_pop()
        setattr(self, name, call)
        return call


if os.environ.get("NFDPM_NVTX", "0") == "1":
    lib = _RangedLib(lib)
EXPORTS = ["nfdpm_version", "nfdpm_last_error_string", "nfdpm_sm_count", "nfdpm_ld_tiles", "nfdpm_mix_prepare",
           "nfdpm_channel_mix", "nfdpm_actnorm_apply", "nfdpm_channel_stats", "nfdpm_squeeze", "nfdpm_unsqueeze",
           "nfdpm_copy_channels", "nfdpm_im2col3x3", "nfdpm_pack_matrix", "nfdpm_gemm_nt", "nfdpm_coupling_apply",
           "nfdpm_split_prior_logp", "nfdpm_split_prior_sample", "nfdpm_gauss_logp_const",
           "nfdpm_gauss_sample_const", "nfdpm_accumulate", "nfdpm_rows_to_nchw", "nfdpm_nchw_to_rows",
           "nfdpm_flow_boundary_smem", "nfdpm_flow_boundary",
           "nfdpm_coupling_bwd", "nfdpm_actnorm_relu_bwd", "nfdpm_reduce_rows", "nfdpm_mix_bwd", "nfdpm_mix_param_grad",
           "nfdpm_gemm_tn_workspace", "nfdpm_gemm_tn", "nfdpm_split_prior_bwd", "nfdpm_gauss_const_bwd",
           "nfdpm_col2im_add", "nfdpm_flow_boundary_stash", "nfdpm_reduce_rows2",
           "nfdpm_opt_chunk", "nfdpm_fused_clip_adam", "nfdpm_pack_elems", "nfdpm_pack_batch",
           "nfdpm_gemm3_boundary_ok", "nfdpm_gemm3_boundary", "nfdpm_coupling_bwd_tiles", "nfdpm_mix_bwd_tiles", "nfdpm_gemm_debug", "nfdpm_flow_boundary_debug",
           "nfdpm_latent_format", "nfdpm_postprocess_u8", "nfdpm_preprocess",
           "nfdpm_flow_boundary_tiles", "nfdpm_flow_boundary_tiled",
           "nfdpm_coupling_inv_bwd", "nfdpm_mix_inv_param_grad", "nfdpm_split_sample_bwd", "nfdpm_flow_boundary_inv_stash",
           "nfdpm_coupling_inv_bwd_ld", "nfdpm_flow_boundary_inv_stash_ld", "nfdpm_split_sample_bwd_lp",
           "nfdpm_split_prior_sample_ex", "nfdpm_gauss_sample_const_ex", "nfdpm_split_sample_bwd_ex"]

#: number of kernels launched through this binding (bench.py reports it as ``gpu_launches``)
launch_count = 0


def _ok(rc: int, n_launch: int = 1) -> None:
    global launch_count
    if rc != 0:
        raise RuntimeError("libnfdpm_b200: " + lib.nfdpm_last_error_string().decode())
    launch_count += n_launch


def _p(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _st():
    return torch.cuda.current_stream().cuda_stream


def _dt(t: torch.Tensor) -> int:
    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.float64:
        return F64
    if t.dtype == torch.bfloat16:
        return BF16
    if t.dtype == SPLIT:
        return BF16X2
    raise TypeError(f"unsupported dtype {t.dtype}")


def require_cuda(t: torch.Tensor, what: str) -> None:
    if not t.is_cuda:
        raise RuntimeError(f"{what} must live on a CUDA device: this package runs only its sm_100a kernels and has "
                           f"no CPU fallback (got device {t.device}).")


def ld_tiles(P: int) -> int:
    return lib.nfdpm_ld_tiles(P)


def mix_prepare(items) -> None:
    arr = (MixItem * len(items))(*items)
    _ok(lib.nfdpm_mix_prepare(arr, len(items), _st()), (len(items) + 63) // 64)


def channel_mix(x, y, mt, beta, B, Cc, P, xbs, ybs) -> None:
    _ok(lib.nfdpm_channel_mix(_p(x), _p(y), _p(mt), _p(beta), B, Cc, P, xbs, ybs, _st()))


def actnorm_apply(x, y, scale, bias, B, Cc, P, inverse) -> None:
    _ok(lib.nfdpm_actnorm_apply(_p(x), _p(y), _p(scale), _p(bias), B, Cc, P, int(inverse), _st()))


def channel_stats(x, layout, B, Cc, P, xs, scale_out, bias_out) -> None:
    _ok(lib.nfdpm_channel_stats(_p(x), layout, B, Cc, P, xs, _p(scale_out), _p(bias_out), _st()))


def squeeze(x, y, B, Cc, H, W, xbs, ybs) -> None:
    _ok(lib.nfdpm_squeeze(_p(x), _p(y), B, Cc, H, W, xbs, ybs, _st()))


def unsqueeze(x, y, B, Cc, H, W, xbs, ybs) -> None:
    _ok(lib.nfdpm_unsqueeze(_p(x), _p(y), B, Cc, H, W, xbs, ybs, _st()))


def copy_channels(src, dst, B, Cn, P, sbs, dbs) -> None:
    _ok(lib.nfdpm_copy_channels(_p(src), _p(dst), B, Cn, P, sbs, dbs, _st()))


def im2col3x3(x, out, B, Cin, H, W, xbs, ld) -> None:
    _ok(lib.nfdpm_im2col3x3(_p(x), _p(out), _dt(out), B, Cin, H, W, xbs, ld, _st()))


def pack_matrix(src, out, na, nb, nk, sa, sb, sk, ld, rows_out) -> None:
    _ok(lib.nfdpm_pack_matrix(_p(src), _p(out), _dt(out), na, nb, nk, sa, sb, sk, ld, rows_out, _st()))


def gemm_nt(A, lda, Bw, ldb, D, ldd, M, N, K, epilogue=EPI_RAW, ep_scale=None, ep_bias=None) -> None:
    _ok(lib.nfdpm_gemm_nt(_p(A), lda, _p(Bw), ldb, _p(D), ldd, M, N, K, _dt(A), _dt(D), epilogue, _p(ep_scale),
                          _p(ep_bias), _st()))


def coupling_apply(pm, ldp, bias3, logs3, x, y, ld_part, B, Cc, H, W, xbs, ybs, inverse) -> None:
    _ok(lib.nfdpm_coupling_apply(_p(pm), ldp, _p(bias3), _p(logs3), _p(x), _p(y), _p(ld_part), B, Cc, H, W, xbs, ybs,
                                 int(inverse), _st()))


def split_prior_logp(h, ldh, bias, logs, x, xbs, z_out, logp_part, B, Cc, H, W) -> None:
    _ok(lib.nfdpm_split_prior_logp(_p(h), ldh, _p(bias), _p(logs), _p(x), xbs, _p(z_out), _p(logp_part), B, Cc, H, W,
                                   _st()))


def split_prior_sample(h, ldh, bias, logs, eps, temperature, y, ybs, B, Cc, H, W) -> None:
    _ok(lib.nfdpm_split_prior_sample(_p(h), ldh, _p(bias), _p(logs), _p(eps), float(temperature), _p(y), ybs, B, Cc,
                                     H, W, _st()))


#: draw site of GaussianPrior.sample in the seeded-draw contract (include/nfdpm_b200.h); a Split uses its level
PRIOR_STREAM = 0xFFFFFFFF


def split_prior_sample_ex(h, ldh, bias, logs, eps, seeds, stream_id, temperature, temp_b, eps_out, y, ybs, B, Cc, H,
                          W) -> None:
    """``split_prior_sample`` with a per-image temperature ``temp_b`` and/or seeded draws (``seeds``, ``stream_id``; the
    draws go to ``eps_out`` when given).  Exactly one of ``eps`` / ``seeds``."""
    _ok(lib.nfdpm_split_prior_sample_ex(_p(h), ldh, _p(bias), _p(logs), _p(eps), _p(seeds), int(stream_id),
                                        float(temperature), _p(temp_b), _p(eps_out), _p(y), ybs, B, Cc, H, W, _st()))


def gauss_sample_const_ex(eps, seeds, stream_id, bias, logs, temperature, temp_b, eps_out, out, B, Cc, P) -> None:
    _ok(lib.nfdpm_gauss_sample_const_ex(_p(eps), _p(seeds), int(stream_id), _p(bias), _p(logs), float(temperature),
                                        _p(temp_b), _p(eps_out), _p(out), B, Cc, P, _st()))


def gauss_logp_const(z, bias, logs, part, B, Cc, P) -> None:
    _ok(lib.nfdpm_gauss_logp_const(_p(z), _p(bias), _p(logs), _p(part), B, Cc, P, _st()))


def gauss_sample_const(eps, bias, logs, temperature, out, B, Cc, P) -> None:
    _ok(lib.nfdpm_gauss_sample_const(_p(eps), _p(bias), _p(logs), float(temperature), _p(out), B, Cc, P, _st()))


def accumulate(acc, part, R, B, cval=None, cmul=None, nc=0) -> None:
    _ok(lib.nfdpm_accumulate(_p(acc), _dt(acc), _p(part), R, B, _p(cval), _p(cmul), nc, _st()))


def rows_to_nchw(h, ldh, mode, p1, p2, out, B, Nc, P) -> None:
    _ok(lib.nfdpm_rows_to_nchw(_p(h), ldh, mode, _p(p1), _p(p2), _p(out), B, Nc, P, _st()))


def nchw_to_rows(x, out, B, Cc, P, xbs, ld) -> None:
    _ok(lib.nfdpm_nchw_to_rows(_p(x), _p(out), _dt(out), B, Cc, P, xbs, ld, _st()))


def flow_boundary_smem(Cc, H, W, coupling, mix) -> int:
    return int(lib.nfdpm_flow_boundary_smem(Cc, H, W, int(coupling), int(mix)))


def flow_boundary(src, src_bs, squeeze_in, pm, ldp, bias3, logs3, ld_part, mt, beta, y, y_bs, a1, lda1, B, Cc, H, W,
                  inverse) -> None:
    _ok(lib.nfdpm_flow_boundary(_p(src), src_bs, int(squeeze_in), _p(pm), ldp, _p(bias3), _p(logs3), _p(ld_part),
                                _p(mt), _p(beta), _p(y), y_bs, _p(a1), _dt(a1) if a1 is not None else F32, lda1, B, Cc,
                                H, W, int(inverse), _st()))






# ---------------------------------------------------------------------------------------------- backward
def coupling_bwd_tiles(Cc, H, W) -> int:
    return int(lib.nfdpm_coupling_bwd_tiles(Cc, H, W))


def mix_bwd_tiles(Cc, H, W) -> int:
    return int(lib.nfdpm_mix_bwd_tiles(Cc, H, W))


def coupling_bwd(dy, dy_bs, dld, u, u_bs, pm, ldp, bias3, logs3, du, du_bs, dpm, ld_dpm, dpar, B, Cc, H, W, dbias=None,
                 dlogs=None, dp_scratch=None) -> None:
    """With dbias/dlogs the kernel's last CTA reduces the per-image partials itself (no nfdpm_reduce_rows2 launch);
    images that do not fit one CTA (coupling_bwd_tiles > 1) need dp_scratch and a separate reduction of dpar."""
    cnt = _tn_counters(dy.device)[1023:] if dbias is not None else None
    _ok(lib.nfdpm_coupling_bwd(_p(dy), dy_bs, _p(dld), _p(u), u_bs, _p(pm), ldp, _p(bias3), _p(logs3), _p(du), du_bs,
                               _p(dpm), _dt(dpm), ld_dpm, _p(dpar), _p(dbias), _p(dlogs), _p(cnt), _p(dp_scratch), B, Cc,
                               H, W, _st()), 1 if dp_scratch is None else 2)


def coupling_inv_bwd(dx, dx_bs, y, y_bs, pm, ldp, bias3, logs3, dy, dy_bs, dpm, ld_dpm, dpar, B, Cc, H, W, dbias=None,
                     dlogs=None, dp_scratch=None) -> None:
    """Backward of the inverse coupling; reductions and tiling as in ``coupling_bwd``."""
    cnt = _tn_counters(dx.device)[1023:] if dbias is not None else None
    _ok(lib.nfdpm_coupling_inv_bwd(_p(dx), dx_bs, _p(y), y_bs, _p(pm), ldp, _p(bias3), _p(logs3), _p(dy), dy_bs, _p(dpm),
                                   _dt(dpm), ld_dpm, _p(dpar), _p(dbias), _p(dlogs), _p(cnt), _p(dp_scratch), B, Cc, H, W,
                                   _st()), 1 if dp_scratch is None else 2)


def coupling_inv_bwd_ld(dx, dx_bs, dld, y, y_bs, pm, ldp, bias3, logs3, dy, dy_bs, dpm, ld_dpm, dpar, B, Cc, H, W,
                        dbias=None, dlogs=None, dp_scratch=None) -> None:
    """``coupling_inv_bwd`` plus the gradient ``dld`` [B] (None: none) of the log-det the inverse accumulates."""
    cnt = _tn_counters(dx.device)[1023:] if dbias is not None else None
    _ok(lib.nfdpm_coupling_inv_bwd_ld(_p(dx), dx_bs, _p(dld), _p(y), y_bs, _p(pm), ldp, _p(bias3), _p(logs3), _p(dy), dy_bs,
                                      _p(dpm), _dt(dpm), ld_dpm, _p(dpar), _p(dbias), _p(dlogs), _p(cnt), _p(dp_scratch), B,
                                      Cc, H, W, _st()), 1 if dp_scratch is None else 2)


def flow_boundary_stash(src, src_bs, squeeze_in, pm, ldp, bias3, logs3, ld_part, mt, beta, y, y_bs, xs, xs_bs, a1, lda1,
                        B, Cc, H, W) -> None:
    _ok(lib.nfdpm_flow_boundary_stash(_p(src), src_bs, int(squeeze_in), _p(pm), ldp, _p(bias3), _p(logs3), _p(ld_part),
                                      _p(mt), _p(beta), _p(y), y_bs, _p(xs), xs_bs, _p(a1),
                                      _dt(a1) if a1 is not None else F32, lda1, B, Cc, H, W, _st()))


def flow_boundary_inv_stash(src, src_bs, pm, ldp, bias3, logs3, mt, beta, y, y_bs, xs, xs_bs, a1, lda1, B, Cc, H, W) -> None:
    _ok(lib.nfdpm_flow_boundary_inv_stash(_p(src), src_bs, _p(pm), ldp, _p(bias3), _p(logs3), _p(mt), _p(beta), _p(y), y_bs,
                                          _p(xs), xs_bs, _p(a1), _dt(a1) if a1 is not None else F32, lda1, B, Cc, H, W,
                                          _st()))


def flow_boundary_inv_stash_ld(src, src_bs, pm, ldp, bias3, logs3, ld_part, mt, beta, y, y_bs, xs, xs_bs, a1, lda1, B, Cc,
                               H, W) -> None:
    _ok(lib.nfdpm_flow_boundary_inv_stash_ld(_p(src), src_bs, _p(pm), ldp, _p(bias3), _p(logs3), _p(ld_part), _p(mt),
                                             _p(beta), _p(y), y_bs, _p(xs), xs_bs, _p(a1), _dt(a1) if a1 is not None else F32,
                                             lda1, B, Cc, H, W, _st()))


def actnorm_relu_bwd(dh, ld_dh, h, ld_h, scale, dpre, ld_o, part, M, Nn, rows_per_cta) -> None:
    _ok(lib.nfdpm_actnorm_relu_bwd(_p(dh), _dt(dh), ld_dh, _p(h), _dt(h), ld_h, _p(scale), _p(dpre), _dt(dpre), ld_o,
                                   _p(part), M, Nn, rows_per_cta, _st()))


def reduce_rows(part, out, R, n, stride, accumulate=False) -> None:
    _ok(lib.nfdpm_reduce_rows(_p(part), _p(out), R, n, stride, int(accumulate), _st()))


def reduce_rows2(part, out0, out1, R, n0, n1, stride) -> None:
    _ok(lib.nfdpm_reduce_rows2(_p(part), _p(out0), _p(out1), R, n0, n1, stride, _st()))


def mix_bwd(du, du_bs, da1, lda1, x, x_bs, mt, dx, dx_bs, part, B, Cc, H, W) -> None:
    _ok(lib.nfdpm_mix_bwd(_p(du), du_bs, _p(da1), lda1, _p(x), x_bs, _p(mt), _p(dx), dx_bs, _p(part), B, Cc, H, W, _st()))


def mix_param_grad(items) -> None:
    arr = (MixGradItem * len(items))(*items)
    _ok(lib.nfdpm_mix_param_grad(arr, len(items), _st()), (len(items) + 15) // 16)


def mix_inv_param_grad(items) -> None:
    arr = (MixGradItem * len(items))(*items)
    _ok(lib.nfdpm_mix_inv_param_grad(arr, len(items), _st()), (len(items) + 15) // 16)


def gemm_tn_workspace(M, N1, N2) -> int:
    return int(lib.nfdpm_gemm_tn_workspace(M, N1, N2, None))


_TN_COUNTERS = {}


def _tn_counters(dev: torch.device):
    """Zero-initialised, self-re-arming tile counters of the in-kernel split reduction (one set per device+stream)."""
    key = (dev.index, torch.cuda.current_stream(dev).cuda_stream)
    t = _TN_COUNTERS.get(key)
    if t is None:
        t = _TN_COUNTERS[key] = torch.zeros(1024, dtype=torch.int32, device=dev)
    return t


TN_OUT_PLAIN, TN_OUT_TAPS, TN_OUT_STRIP = 0, 1, 2


@functools.lru_cache(maxsize=None)
def _tn_sms() -> int:
    n = lib.nfdpm_sm_count()
    return n if n > 0 else 148          # gemm_tn_tc.cu sm_count(): 148 without a device


@functools.lru_cache(maxsize=None)
def gemm_tn_tc_plan(M, N1, N2):
    """gemm_tn_tc_plan (csrc/gemm_tn_tc.cu) for the kernel's dimensions (bf16 columns): (BN, tiles, splits,
    k-blocks per split)."""
    bn = 256 if N2 >= 256 else (N2 + 63) // 64 * 64
    tiles = ((N1 + 127) // 128) * ((N2 + bn - 1) // bn)
    num_kb = (M + 63) // 64
    min_kb = max(1, int(os.environ.get("NFDPM_TN_MIN_KB", "1") or 1))
    s = max(1, _tn_sms() // tiles)
    s = max(1, min(s, num_kb // min_kb))
    per = (num_kb + s - 1) // s
    return bn, tiles, (num_kb + per - 1) // per, per


@functools.lru_cache(maxsize=None)
def gemm_tn_path(a_dt, b_dt, tc_ok, M, N1, N2, counters, out_mode):
    """The kernels nfdpm_gemm_tn launches (csrc/backward.cu, gemm_tn_tc.cu): (GEMM, reduction).  GEMM: "x3" (tcgen05,
    split pairs), "tc" (tcgen05, bf16; tc_ok = gemm_tn_tc_ok) or "simt" (gemm_tn_kernel); reduction: "in_kernel" (the
    GEMM's CTAs sum their slabs, synchronised through the counters), "tn_reduce" (gemm_tn_reduce_kernel) or
    "reduce_rows" (reduce_rows_kernel)."""
    if a_dt == BF16X2 or b_dt == BF16X2:
        gemm, n1, n2 = "x3", 2 * ((N1 + 31) // 32 * 32), 2 * ((N2 + 31) // 32 * 32)
    elif a_dt == BF16 and b_dt == BF16 and tc_ok:
        gemm, n1, n2 = "tc", N1, N2
    else:
        return "simt", "reduce_rows"
    _, tiles, splits, _ = gemm_tn_tc_plan(M, n1, n2)
    coresident = not (tiles > 500 or tiles * splits > _tn_sms())
    if not coresident and (out_mode != TN_OUT_PLAIN or gemm == "x3"):
        return gemm, "tn_reduce"
    return gemm, "in_kernel" if coresident and counters else "reduce_rows"


def gemm_tn_tc_ok(A, lda, Bm, ldb, N2) -> bool:
    """gemm_tn_tc_ok (csrc/gemm_tn_tc.cu)."""
    return lda % 8 == 0 and ldb % 8 == 0 and N2 % 16 == 0 and A.data_ptr() % 16 == 0 and Bm.data_ptr() % 16 == 0


def gemm_tn(A, lda, Bm, ldb, D, M, N1, N2, ws, accumulate=False, fused_reduce=True, out_mode=TN_OUT_PLAIN, out_c=0) -> None:
    cnt = _tn_counters(A.device) if fused_reduce else None
    _, red = gemm_tn_path(_dt(A), _dt(Bm), gemm_tn_tc_ok(A, lda, Bm, ldb, N2), M, N1, N2, fused_reduce, out_mode)
    _ok(lib.nfdpm_gemm_tn(_p(A), _dt(A), lda, _p(Bm), _dt(Bm), ldb, _p(D), N2, M, N1, N2, _p(ws), int(accumulate),
                          _p(cnt), out_mode, out_c, _st()), 1 if red == "in_kernel" else 2)


def split_prior_bwd(dlp, h, ldh, bias, logs, x, xbs, dstate, dbs, dh, dpar, B, Cc, H, W) -> None:
    _ok(lib.nfdpm_split_prior_bwd(_p(dlp), _p(h), ldh, _p(bias), _p(logs), _p(x), xbs, _p(dstate), dbs, _p(dh), _p(dpar),
                                  B, Cc, H, W, _st()))


def gauss_const_bwd(dl, z, bias, logs, dz, dpar, B, Cc, P) -> None:
    _ok(lib.nfdpm_gauss_const_bwd(_p(dl), _p(z), _p(bias), _p(logs), _p(dz), _p(dpar), B, Cc, P, _st()))


def split_sample_bwd(dz, dz_bs, eps, temperature, h, ldh, bias, logs, dh, dpar, B, Cc, H, W) -> None:
    _ok(lib.nfdpm_split_sample_bwd(_p(dz), dz_bs, _p(eps), float(temperature), _p(h), ldh, _p(bias), _p(logs), _p(dh),
                                   _p(dpar), B, Cc, H, W, _st()))


def split_sample_bwd_lp(dz, dz_bs, dlp, eps, temperature, h, ldh, bias, logs, dh, dpar, B, Cc, H, W) -> None:
    _ok(lib.nfdpm_split_sample_bwd_lp(_p(dz), dz_bs, _p(dlp), _p(eps), float(temperature), _p(h), ldh, _p(bias), _p(logs),
                                      _p(dh), _p(dpar), B, Cc, H, W, _st()))


def split_sample_bwd_ex(dz, dz_bs, eps, temperature, temp_b, dlp, h, ldh, bias, logs, dh, dpar, B, Cc, H, W) -> None:
    _ok(lib.nfdpm_split_sample_bwd_ex(_p(dz), dz_bs, _p(eps), float(temperature), _p(temp_b), _p(dlp), _p(h), ldh, _p(bias),
                                      _p(logs), _p(dh), _p(dpar), B, Cc, H, W, _st()))


def col2im_add(da, lda, dstate, dbs, B, Cin, H, W) -> None:
    _ok(lib.nfdpm_col2im_add(_p(da), lda, _p(dstate), dbs, B, Cin, H, W, _st()))


def opt_chunk() -> int:
    return int(lib.nfdpm_opt_chunk())


def fused_clip_adam(refs, chunks, n_chunks, exp_avg, exp_avg_sq, partial, scal, clip_value, max_norm, lr, beta1, beta2, eps,
                    weight_decay, decoupled) -> None:
    _ok(lib.nfdpm_fused_clip_adam(_p(refs), _p(chunks), n_chunks, _p(exp_avg), _p(exp_avg_sq), _p(partial), _p(scal),
                                  clip_value, max_norm, lr, beta1, beta2, eps, weight_decay, int(decoupled), _st()), 3)


def pack_elems() -> int:
    return int(lib.nfdpm_pack_elems())


def pack_batch(jobs_dev, n_jobs, n_blocks) -> None:
    _ok(lib.nfdpm_pack_batch(_p(jobs_dev), n_jobs, n_blocks, _st()))


def gemm3_boundary_ok(B, Cc, H, W, K, ldp) -> bool:
    return bool(lib.nfdpm_gemm3_boundary_ok(B, Cc, H, W, K, ldp))


def gemm3_boundary(h2, ldh, w3p, pm_out, ld_pm_out, src, src_bs, bias3, logs3, ld_part, mt, beta, y, y_bs, xs, xs_bs, a1,
                   lda1, B, Cc, H, W, K, ldp, inverse) -> None:
    _ok(lib.nfdpm_gemm3_boundary(_p(h2), _dt(h2), ldh, _p(w3p), _p(pm_out), ld_pm_out, _p(src), src_bs, _p(bias3), _p(logs3),
                                 _p(ld_part), _p(mt), _p(beta), _p(y), y_bs, _p(xs), xs_bs, _p(a1),
                                 _dt(a1) if a1 is not None else F32, lda1, B, Cc, H, W, K, ldp, int(inverse), _st()))












def latent_format(parts, cat, B, Ct, Ht, Wt, to_cat: bool) -> None:
    """parts: list of (tensor [B,C,H,W] contiguous fp32, degree, ch_offset, ch_count)."""
    arr = (LatentPart * len(parts))()
    for i, (t, degree, off, cnt) in enumerate(parts):
        arr[i].ptr, arr[i].C, arr[i].H, arr[i].W = t.data_ptr(), t.shape[1], t.shape[2], t.shape[3]
        arr[i].degree, arr[i].ch_offset, arr[i].ch_count = degree, off, cnt
    _ok(lib.nfdpm_latent_format(arr, len(parts), _p(cat), B, Ct, Ht, Wt, int(to_cat), _st()))


def postprocess_u8(x, out, n_bins: float) -> None:
    _ok(lib.nfdpm_postprocess_u8(_p(x), _p(out), x.numel(), float(n_bins), float(256.0 / n_bins), _st()))


def preprocess(x, noise, y, n_bits: int, n_bins: float) -> None:
    _ok(lib.nfdpm_preprocess(_p(x), _p(noise), _p(y), x.numel(), int(n_bits), float(n_bins), _st()))


def flow_boundary_tiles(B, Cc, H, W, coupling, mix, want_a1) -> int:
    return int(lib.nfdpm_flow_boundary_tiles(B, Cc, H, W, int(coupling), int(mix), int(want_a1)))


def flow_boundary_tiled(src, src_bs, squeeze_in, pm, ldp, bias3, logs3, ld_part, mt, beta, y, y_bs, xs, xs_bs, a1, lda1,
                        B, Cc, H, W, inverse, tiles) -> None:
    _ok(lib.nfdpm_flow_boundary_tiled(_p(src), src_bs, int(squeeze_in), _p(pm), ldp, _p(bias3), _p(logs3), _p(ld_part),
                                      _p(mt), _p(beta), _p(y), y_bs, _p(xs), xs_bs, _p(a1),
                                      _dt(a1) if a1 is not None else F32, lda1, B, Cc, H, W, int(inverse), tiles, _st()))
