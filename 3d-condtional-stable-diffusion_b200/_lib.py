"""ctypes binding of libb200dm.so (include/b200dm.h).  PyTorch tensors are only the device-memory
container: every call passes raw device pointers and the current CUDA stream.

There is no CPU fallback: importing works anywhere (so host logic can be unit-tested), but any
compute call without the library or without a GPU raises.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_lib = None
_HERE = os.path.dirname(os.path.abspath(__file__))
# Two builds of the same sources (build.py): bf16 storage (default; fp32 range) and fp16 storage (8x smaller storage
# rounding: the precision mode that meets the reference-fp32 chain tolerances, DESIGN.md section 2).  Selected once
# per process, before the first kernel call: set_precision("fp16") or B200DM_PRECISION=fp16.
_LIBS = {"bf16": os.path.join(_HERE, "libb200dm.so"), "fp16": os.path.join(_HERE, "libb200dm_f16.so")}
_precision = os.environ.get("B200DM_PRECISION", "bf16").lower()
if _precision not in _LIBS:
    raise ImportError(f"B200DM_PRECISION={_precision!r}: expected 'bf16' or 'fp16'")
_LIB_PATH = _LIBS[_precision]
ACT_DTYPE = torch.bfloat16 if _precision == "bf16" else torch.float16   # torch dtype of every 16-bit buffer


def storage(dtype=None):
    """Normalise a dtype argument: None or any 16-bit float type means 'the library's 16-bit storage type'."""
    return ACT_DTYPE if dtype in (None, torch.bfloat16, torch.float16) else dtype


def precision() -> str:
    return _precision


def set_precision(name: str):
    """Choose the storage build ('bf16' | 'fp16') for this process.  Must be called before the library is first used."""
    global _precision, _LIB_PATH, ACT_DTYPE
    name = name.lower()
    if name not in _LIBS:
        raise ValueError(f"precision {name!r}: expected 'bf16' or 'fp16'")
    if name == _precision:
        return
    if _lib is not None:
        raise B200dmError(f"libb200dm ({_precision}) is already loaded; the storage type is chosen once per process")
    _precision, _LIB_PATH = name, _LIBS[name]
    ACT_DTYPE = torch.bfloat16 if name == "bf16" else torch.float16

F32, BF16 = 0, 1
ERR_UNSUPPORTED = -3
ACT_NONE, ACT_SILU, ACT_RELU = 0, 1, 2
CONV_DIRECT, CONV_PARITY, CONV_BATCHED_GEMM = 0, 1, 2
ACT = {None: ACT_NONE, "none": ACT_NONE, "silu": ACT_SILU, "swish": ACT_SILU, "relu": ACT_RELU}


class B200dmError(RuntimeError):
    pass


class UpdateDesc(C.Structure):
    _fields_ = [("n_per_sample", C.c_int64), ("batch", C.c_int32), ("sampler", C.c_int32),
                ("beta", C.c_void_p), ("sqrt_alpha", C.c_void_p), ("alpha_bar", C.c_void_p),
                ("alpha_bar_prev", C.c_void_p), ("sqrt_alpha_bar", C.c_void_p), ("sqrt_alpha_bar_prev", C.c_void_p),
                ("sqrt_one_minus_alpha_bar", C.c_void_p), ("t_dev", C.c_void_p), ("t", C.c_int32), ("t_prev", C.c_int32),
                ("seed", C.c_uint64), ("sample_id0", C.c_int64), ("eps_dtype", C.c_int32), ("reserved", C.c_int32)]


class NormDesc(C.Structure):
    _fields_ = [("voxels", C.c_int64), ("batch", C.c_int32), ("c0", C.c_int32), ("c1", C.c_int32), ("kind", C.c_int32),
                ("groups", C.c_int32), ("act", C.c_int32), ("x_dtype", C.c_int32), ("y_dtype", C.c_int32)]


class VqDesc(C.Structure):
    _fields_ = [("n", C.c_int64), ("d", C.c_int32), ("k", C.c_int32), ("x_dtype", C.c_int32), ("q_dtype", C.c_int32)]


class NormExDesc(C.Structure):
    _fields_ = [("batch", C.c_int32), ("out_d", C.c_int32), ("out_h", C.c_int32), ("out_w", C.c_int32), ("c", C.c_int32),
                ("kind", C.c_int32), ("groups", C.c_int32), ("act", C.c_int32), ("post_act", C.c_int32), ("upsample", C.c_int32),
                ("x_dtype", C.c_int32), ("y_dtype", C.c_int32)]


class AttnDesc(C.Structure):
    _fields_ = [("batch", C.c_int32), ("lq", C.c_int32), ("lk", C.c_int32), ("d", C.c_int32), ("scale", C.c_float),
                ("reserved", C.c_int32 * 3)]


class ConvDesc(C.Structure):
    _fields_ = [("mode", C.c_int32), ("batch", C.c_int32), ("in_d", C.c_int32), ("in_h", C.c_int32), ("in_w", C.c_int32),
                ("c0", C.c_int32), ("c1", C.c_int32), ("c_out", C.c_int32), ("ksize", C.c_int32), ("stride", C.c_int32),
                ("act", C.c_int32), ("y_dtype", C.c_int32), ("chan_bias_rows", C.c_int32), ("use_halo", C.c_int32),
                ("reserved", C.c_int32 * 4)]  # reserved[0] = post_act, reserved[1] = transposed store


_SIGS = {
    "b200dm_version": (C.c_int, []),
    "b200dm_last_error": (C.c_char_p, []),
    "b200dm_storage_dtype": (C.c_char_p, []),
    "b200dm_device_info": (C.c_int, [C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "b200dm_ddpm_update": (C.c_int, [C.POINTER(UpdateDesc), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200dm_philox_normal": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_uint64, C.c_int64, C.c_int32, C.c_int32, C.c_void_p]),
    "b200dm_step_advance": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p]),
    "b200dm_step_advance_seq": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200dm_gather_rows_f32": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]),
    "b200dm_q_sample": (C.c_int, [C.c_void_p] * 5 + [C.c_int64, C.c_int32, C.c_uint64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200dm_noise_loss_workspace": (C.c_size_t, [C.c_int32]),
    "b200dm_noise_loss": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_double, C.c_uint64, C.c_int64,
                                    C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "b200dm_vq_distances": (C.c_int, [C.POINTER(VqDesc)] + [C.c_void_p] * 5),
    "b200dm_bn_fold": (C.c_int, [C.c_void_p] * 4 + [C.c_float, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200dm_gn_stats": (C.c_int, [C.POINTER(NormDesc), C.c_void_p, C.c_float, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "b200dm_gn_stats_workspace": (C.c_size_t, [C.POINTER(NormDesc)]),
    "b200dm_bn_stats_workspace": (C.c_size_t, [C.c_int32]),
    "b200dm_bn_stats": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_size_t, C.c_void_p]),
    "b200dm_norm_act_fwd": (C.c_int, [C.POINTER(NormDesc)] + [C.c_void_p] * 7),
    "b200dm_norm_act_ex": (C.c_int, [C.POINTER(NormExDesc)] + [C.c_void_p] * 8),
    "b200dm_stats_f32_workspace": (C.c_size_t, [C.c_int32]),
    "b200dm_stats_f32": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "b200dm_program_add_norm_act_ex": (C.c_int, [C.c_void_p, C.POINTER(NormExDesc)] + [C.c_void_p] * 7),
    "b200dm_program_add_stats_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_void_p, C.c_void_p, C.c_size_t]),
    "b200dm_layernorm_fwd": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_float, C.c_int32, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_void_p]),
    "b200dm_cast": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_int64, C.c_void_p]),
    "b200dm_vq_argmin_gather": (C.c_int, [C.POINTER(VqDesc)] + [C.c_void_p] * 7),
    "b200dm_vq_prepare": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "b200dm_vq_tc_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_int32]),
    "b200dm_vq_prepare_tc": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "b200dm_vq_argmin_gather_tc": (C.c_int, [C.POINTER(VqDesc)] + [C.c_void_p] * 9),
    "b200dm_dense_f32": (C.c_int, [C.c_void_p] * 4 + [C.c_int32, C.c_int32, C.c_int64, C.c_int32, C.c_int32, C.c_void_p]),
    "b200dm_softmax_rows": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_float, C.c_void_p]),
    "b200dm_conv_packed_weight_bytes": (C.c_size_t, [C.POINTER(ConvDesc)]),
    "b200dm_conv_pack_weights": (C.c_int, [C.POINTER(ConvDesc), C.c_void_p, C.c_int32, C.c_void_p]),
    "b200dm_conv_plan_create": (C.c_int, [C.POINTER(ConvDesc)] + [C.c_void_p] * 9 + [C.POINTER(C.c_void_p)]),
    "b200dm_conv_plan_run": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b200dm_conv_plan_destroy": (None, [C.c_void_p]),
    "b200dm_conv_plan_flops": (C.c_double, [C.c_void_p]),
    "b200dm_conv_plan_set_trace": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b200dm_conv_plan_set_out_affine": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200dm_conv_plan_set_fused_update": (C.c_int, [C.c_void_p, C.POINTER(UpdateDesc), C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200dm_conv_plan_set_shortcut": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200dm_conv_plan_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "b200dm_conv_plan_gn_partials_bytes": (C.c_size_t, [C.c_void_p, C.POINTER(C.c_int32)]),
    "b200dm_conv_plan_set_gn_partials": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "b200dm_gn_finalize": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int64, C.c_float, C.c_void_p, C.c_void_p]),
    "b200dm_program_add_gn_finalize": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int64, C.c_float, C.c_void_p]),
    "b200dm_attention_plan_create": (C.c_int, [C.POINTER(AttnDesc)] + [C.c_void_p] * 5 + [C.POINTER(C.c_void_p)]),
    "b200dm_attention_plan_run": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b200dm_attention_plan_destroy": (None, [C.c_void_p]),
    "b200dm_attention_plan_flops": (C.c_double, [C.c_void_p]),
    "b200dm_program_add_attention": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b200dm_debug_flag_read_reset": (C.c_int, [C.POINTER(C.c_int32)]),
    "b200dm_program_create": (C.c_int, [C.POINTER(C.c_void_p)]),
    "b200dm_program_destroy": (None, [C.c_void_p]),
    "b200dm_program_add_conv": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b200dm_program_add_norm_act": (C.c_int, [C.c_void_p, C.POINTER(NormDesc)] + [C.c_void_p] * 6),
    "b200dm_program_add_gn_stats": (C.c_int, [C.c_void_p, C.POINTER(NormDesc), C.c_void_p, C.c_float, C.c_void_p, C.c_void_p, C.c_size_t]),
    "b200dm_program_add_bn_stats": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_float,
                                              C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "b200dm_program_add_layernorm": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_float, C.c_int32, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]),
    "b200dm_program_add_softmax": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_float]),
    "b200dm_program_add_update": (C.c_int, [C.c_void_p, C.POINTER(UpdateDesc)] + [C.c_void_p] * 5),
    "b200dm_program_add_step_advance": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32]),
    "b200dm_program_set_lane": (C.c_int, [C.c_void_p, C.c_int32]),
    "b200dm_program_add_sync": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32]),
    "b200dm_program_run": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b200dm_program_num_launches": (C.c_int, [C.c_void_p]),
    "b200dm_program_num_ops": (C.c_int, [C.c_void_p]),
    "b200dm_program_run_timed": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_float), C.c_int32]),
}

EXPORTED_SYMBOLS = tuple(_SIGS)


def lib():
    """Load (once) and return the shared library; raise loudly if it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            raise B200dmError(f"{_LIB_PATH} is missing: run `python __graft_entry__.py build` (nvcc, sm_100a). "
                              "There is no CPU fallback.")
        l = C.CDLL(_LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(l, name)
            fn.restype, fn.argtypes = res, args
        got = l.b200dm_storage_dtype().decode()
        if got != _precision:
            raise B200dmError(f"{_LIB_PATH} stores {got}, expected {_precision}: rebuild (python __graft_entry__.py build)")
        _lib = l
    return _lib


def tuning_env(name: str, default: str) -> str:
    """Experiment switches (B200DM_CHAINS) are honoured only when B200DM_TUNING=1 is also set: a production process's environment
    cannot reconfigure the program by accident."""
    return os.environ.get(name, default) if os.environ.get("B200DM_TUNING") == "1" else default


def check(rc: int):
    if rc != 0:
        raise B200dmError(f"libb200dm error {rc}: {lib().b200dm_last_error().decode()}")


def require_gpu():
    if not torch.cuda.is_available():
        raise B200dmError("libb200dm needs a CUDA device (B200, sm_100a); there is no CPU fallback")


def ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def check_storage(*ts):
    """Raise when a 16-bit tensor is not the library's storage type: the kernels take raw pointers and would read bf16 bits as
    fp16 (or the reverse) without a word.  None and non-16-bit tensors pass."""
    for t in ts:
        if t is not None and t.dtype in (torch.bfloat16, torch.float16) and t.dtype != ACT_DTYPE:
            raise B200dmError(f"libb200dm ({_precision} build) stores {ACT_DTYPE}; got a {t.dtype} tensor")


def dt(t):
    if t.dtype == torch.float32:
        return F32
    if t.dtype == ACT_DTYPE:
        return BF16
    raise B200dmError(f"unsupported dtype {t.dtype}")


def debug_flag() -> int:
    f = C.c_int32(0)
    check(lib().b200dm_debug_flag_read_reset(C.byref(f)))
    return f.value
