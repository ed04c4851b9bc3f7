"""ctypes binding of libdpb200.so (include/dpb200.h).  Fails loudly when the library is missing: the product
has no CPU or PyTorch-op fallback for the hot path."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdpb200.so")

i32, i64, f32, u64, vp = C.c_int32, C.c_int64, C.c_float, C.c_uint64, C.c_void_p


class ConvArgs(C.Structure):
    _fields_ = [(n, i32) for n in ("N", "H", "W", "C", "P", "Q", "K", "R", "S", "stride", "pad_t", "pad_l", "flags",
                                   "splits")] + [
        ("x", vp), ("ldx", i64), ("y", vp), ("ldy", i64), ("w", vp), ("w_tc_hi", vp), ("w_tc_lo", vp), ("bias", vp), ("rowadd", vp),
        ("ld_rowadd", i64), ("residual", vp), ("ld_res", i64), ("workspace", vp), ("amax_x", vp), ("amax_y", vp), ("amax_w", vp), ("amax_out", vp), ("bias_ws", vp)]


class WgradReduceArgs(C.Structure):
    _fields_ = [(n, i32) for n in ("K", "C", "R", "S", "splits")] + [
        ("workspace", vp), ("dw", vp), ("w", vp), ("score_out", vp), ("score_in", vp), ("bias_ws", vp), ("db", vp)]


class GemmArgs(C.Structure):
    _fields_ = [("M", i32), ("N", i32), ("Kd", i32), ("batch", i32),
                ("A", vp), ("a_rs", i64), ("a_cs", i64), ("a_bs", i64),
                ("B", vp), ("b_rs", i64), ("b_cs", i64), ("b_bs", i64),
                ("C", vp), ("ldc", i64), ("c_bs", i64), ("alpha", f32), ("accumulate", i32)]


class GemmNtArgs(C.Structure):
    _fields_ = [("batch", i32), ("H", i32), ("W", i32), ("Kg", i32), ("N", i32), ("A", vp), ("ld_a", i64), ("b_hi", vp),
                ("b_lo", vp), ("C", vp), ("ldc", i64), ("alpha", f32), ("amax_a", vp), ("amax_b", vp), ("amax_out", vp)]


class GnArgs(C.Structure):
    _fields_ = [("N", i32), ("HW", i32), ("C", i32), ("G", i32), ("eps", f32), ("silu", i32),
                ("x", vp), ("ldx", i64), ("y", vp), ("ldy", i64), ("gamma", vp), ("beta", vp), ("mean", vp),
                ("rstd", vp), ("dy", vp), ("lddy", i64), ("dx", vp), ("lddx", i64), ("dx_add", vp), ("ldadd", i64),
                ("dx_add2", vp), ("ldadd2", i64), ("dgamma", vp), ("dbeta", vp), ("workspace", vp),
                ("dropout_p", f32), ("dropout_seed", u64), ("dropout_seed_dev", vp), ("y_bf16", vp), ("ldyb", i64),
                ("amax_y", vp), ("amax_dx", vp), ("fin", vp)]


class ConvBf16Args(C.Structure):
    _fields_ = [(n, i32) for n in ("N", "H", "W", "C", "P", "Q", "K", "R", "S", "stride", "pad_t", "pad_l", "flags", "splits")] + [
        ("x_bf16", vp), ("ldx", i64), ("dy_bf16", vp), ("lddy", i64), ("out", vp), ("ld_out", i64), ("w_bf16", vp), ("bias", vp),
        ("rowadd", vp), ("ld_rowadd", i64), ("residual", vp), ("ld_res", i64), ("workspace", vp)]


class TaylorArgs(C.Structure):
    _fields_ = [("O", i32), ("I", i32), ("RS", i32), ("w", vp), ("dw", vp), ("out_signed", vp), ("out_abs", vp),
                ("out_sq", vp), ("in_signed", vp), ("in_abs", vp), ("in_sq", vp)]


class AdamArgs(C.Structure):
    _fields_ = [("n", i64), ("p", vp), ("g", vp), ("m", vp), ("v", vp), ("ema", vp), ("sumsq", vp),
                ("max_norm", C.c_double), ("lr", C.c_double), ("beta1", C.c_double), ("beta2", C.c_double),
                ("eps", C.c_double), ("ema_decay", C.c_double),
                ("step", i32), ("grad_scale", f32), ("step_scalars", vp)]


_SIGS = {
    "dp_version": (C.c_int, []),
    "dp_strerror": (C.c_char_p, [C.c_int]),
    "dp_last_cuda_error": (C.c_int, []),
    "dp_launch_count": (i64, []),
    "dp_tc_available": (C.c_int, []),
    "dp_tc_weight_row": (C.c_int, [C.c_int]),
    "dp_conv2d_fprop": (C.c_int, [C.POINTER(ConvArgs), vp]),
    "dp_conv2d_dgrad": (C.c_int, [C.POINTER(ConvArgs), vp]),
    "dp_conv2d_wgrad": (C.c_int, [C.POINTER(ConvArgs), vp]),
    "dp_conv_splitk_workspace_floats": (i64, [C.POINTER(ConvArgs), C.c_int]),
    "dp_conv_presplit_eligible": (C.c_int, [C.POINTER(ConvArgs)]),
    "dp_conv2d_wgrad_reduce": (C.c_int, [C.POINTER(WgradReduceArgs), vp]),
    "dp_pack_conv_weight": (C.c_int, [vp, i32, i32, i32, i32, vp, vp, vp]),
    "dp_pack_conv_weight_tc": (C.c_int, [vp, i32, i32, i32, i32, vp, vp, vp, vp, vp, vp]),
    "dp_amax": (C.c_int, [vp, i64, i64, i32, vp, vp]),
    "dp_zero_u32": (C.c_int, [vp, i64, vp]),
    "dp_bf16_available": (C.c_int, []),
    "dp_bf16_weight_row": (C.c_int, [C.c_int]),
    "dp_bf16_wgrad_ctile": (C.c_int, [C.c_int]),
    "dp_conv2d_fprop_bf16": (C.c_int, [C.POINTER(ConvBf16Args), vp]),
    "dp_conv2d_dgrad_bf16": (C.c_int, [C.POINTER(ConvBf16Args), vp]),
    "dp_conv2d_wgrad_bf16": (C.c_int, [C.POINTER(ConvBf16Args), vp]),
    "dp_conv_bf16_eligible": (C.c_int, [C.POINTER(ConvBf16Args), C.c_int]),
    "dp_cvt_bf16": (C.c_int, [vp, i64, i64, i32, vp, i64, vp]),
    "dp_pack_conv_weight_bf16": (C.c_int, [vp, i32, i32, i32, i32, vp, vp, vp]),
    "dp_gemm_batched": (C.c_int, [C.POINTER(GemmArgs), vp]),
    "dp_gemm_nt_tc": (C.c_int, [C.POINTER(GemmNtArgs), vp]),
    "dp_split_h3": (C.c_int, [vp, i64, i64, i32, i32, i32, i32, vp, vp, vp, vp]),
    "dp_transpose_batched": (C.c_int, [vp, vp, i32, i32, i32, vp]),
    "dp_softmax_fwd": (C.c_int, [vp, vp, i64, i32, vp]),
    "dp_softmax_bwd": (C.c_int, [vp, vp, vp, i64, i32, vp, vp]),
    "dp_groupnorm_workspace_bytes": (C.c_size_t, [i32, i32, i32, i32]),
    "dp_groupnorm_fwd": (C.c_int, [C.POINTER(GnArgs), vp]),
    "dp_groupnorm_fwd_split": (C.c_int, [C.POINTER(GnArgs), vp, i64, vp]),
    "dp_groupnorm_bwd": (C.c_int, [C.POINTER(GnArgs), vp]),
    "dp_groupnorm_bwd_param": (C.c_int, [C.POINTER(GnArgs), vp]),
    "dp_silu_fwd": (C.c_int, [vp, vp, i64, vp]),
    "dp_silu_bwd": (C.c_int, [vp, vp, vp, i64, i32, vp]),
    "dp_geglu_fwd": (C.c_int, [vp, i64, vp, i64, i64, i32, vp]),
    "dp_geglu_bwd": (C.c_int, [vp, i64, vp, i64, vp, i64, i64, i32, vp]),
    "dp_timestep_embedding": (C.c_int, [vp, vp, vp, i32, i32, i32, vp]),
    "dp_add_noise": (C.c_int, [vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i64, vp]),
    "dp_nchw_to_nhwc": (C.c_int, [vp, vp, i64, i32, i32, i32, i32, vp]),
    "dp_nhwc_to_nchw": (C.c_int, [vp, i64, vp, i32, i32, i32, i32, i32, vp]),
    "dp_mse_partials": (i64, [i64]),
    "dp_mse_loss_grad": (C.c_int, [vp, vp, vp, i64, f32, f32, vp, vp, vp]),
    "dp_upsample2x_fwd": (C.c_int, [vp, i64, vp, i64, i32, i32, i32, i32, vp]),
    "dp_upsample2x_bwd": (C.c_int, [vp, i64, vp, i64, i32, i32, i32, i32, i32, vp]),
    "dp_colsum": (C.c_int, [vp, i64, i64, i32, i64, vp, i64, i32, vp]),
    "dp_add_views": (C.c_int, [vp, i64, vp, i64, vp, i64, i64, i32, vp]),
    "dp_copy_rows": (C.c_int, [vp, i64, vp, i64, i64, i32, vp]),
    "dp_taylor_reduce": (C.c_int, [C.POINTER(TaylorArgs), vp]),
    "dp_sumsq_partials": (i64, [i64]),
    "dp_sumsq": (C.c_int, [vp, i64, vp, vp, vp]),
    "dp_adam_clip_ema": (C.c_int, [C.POINTER(AdamArgs), vp]),
    "dp_ddim_step": (C.c_int, [vp, vp, vp, vp, i64, f32, f32, f32, f32, f32, f32, vp]),
    "dp_scale": (C.c_int, [vp, i64, f32, vp]),
}
EXPORTS = tuple(_SIGS)

_lib = None


class DpError(RuntimeError):
    pass


def load():
    """Load (once) and return the ctypes handle; raises if libdpb200.so has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("DPB200_LIB", LIB_PATH)   # developer knob: A/B an alternative build of the same sources
    if not os.path.exists(path):
        raise DpError(
            f"diff_pruning_b200: {LIB_PATH} not found. Build it with `python -c 'import __graft_entry__ as g; "
            "g.build()'` (nvcc, sm_100a). There is no CPU / PyTorch fallback for the hot path.")
    lib = C.CDLL(path)
    for name, (res, args) in _SIGS.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib


def check(rc: int, what: str = ""):
    if rc != 0:
        lib = load()
        msg = lib.dp_strerror(rc).decode()
        extra = f" (cudaError {lib.dp_last_cuda_error()})" if rc == -4 else ""
        raise DpError(f"libdpb200 {what}: {msg}{extra}")
