"""ctypes binding of libphasegen.so (the C ABI declared in include/phasegen.h).

There is deliberately no fallback: if the shared library is missing, or the device is not
an sm_100 part, every entry point raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "..", "csrc", "libphasegen.so")

PG_CONV, PG_CONV_TRANSPOSE = 0, 1
PG_PREC_FP32_SIMT, PG_PREC_BF16X3, PG_PREC_BF16, PG_PREC_F16X3, PG_PREC_F16X2, PG_PREC_F16 = 0, 1, 2, 3, 4, 5
PG_DT_NONE, PG_DT_F32, PG_DT_BF16_SPLIT, PG_DT_BF16, PG_DT_F16_SPLIT, PG_DT_F16 = 0, 1, 2, 3, 4, 5
PG_FMT_BF16, PG_FMT_F16 = 0, 1
PG_STFT_LOGMAG, PG_STFT_REIM, PG_STFT_PROJECT, PG_STFT_PAIRS = 0, 1, 2, 3
PG_SPEC_POLAR_LOG, PG_SPEC_CARTESIAN, PG_SPEC_POLAR_MAG = 0, 1, 2
PG_EPI_RAW, PG_EPI_ACT, PG_EPI_NORM_ACT = 0, 1, 2
ABI_VERSION = 4

# "f16mix" is an executor-level name (phasegen/unet.py): fp16 planes everywhere, the three-product
# form on the small layers and the two-product form (fp16-rounded weights) on the three largest.
PRECISIONS = {"fp32_simt": PG_PREC_FP32_SIMT, "bf16x3": PG_PREC_BF16X3, "bf16": PG_PREC_BF16,
              "f16x3": PG_PREC_F16X3, "f16x2": PG_PREC_F16X2, "f16": PG_PREC_F16}


class ConvDesc(C.Structure):
    _fields_ = [(n, C.c_int) for n in (
        "kind", "B", "C_in", "C_out", "L_in", "L_out", "k", "stride", "pad",
        "in_rows", "in_ld", "out_rows", "out_ld", "precision",
        "taps_per_group", "tc_base_offset_mode", "tc_max_ctas", "max_clips_per_tile", "weights_mn_major", "tc_cta_pair",
        "tc_whole_clip")]


class GradSrc(C.Structure):
    _fields_ = [("g", C.c_void_p), ("ld", C.c_int), ("ch_off", C.c_int), ("slope", C.c_float)]


class ActDst(C.Structure):
    _fields_ = [("hi", C.c_void_p), ("lo", C.c_void_p), ("batch_stride", C.c_int64),
                ("ld", C.c_int), ("ch_off", C.c_int), ("dtype", C.c_int), ("slope", C.c_float),
                ("range_flag", C.c_void_p)]


class ConvEpilogue(C.Structure):
    _fields_ = [("mode", C.c_int), ("gamma", C.c_void_p), ("beta", C.c_void_p), ("eps", C.c_float),
                ("dst0", ActDst), ("dst1", ActDst), ("scale_shift", C.c_void_p)]


_P, _I, _F, _L = C.c_void_p, C.c_int, C.c_float, C.c_int64
_SIGNATURES = {
    "pg_last_error": (C.c_char_p, []),
    "pg_abi_version": (_I, []),
    "pg_check_device": (_I, [C.POINTER(_I)] * 3),
    "pg_stft_num_frames": (_I, [_I, _I]),
    "pg_stft": (_I, [_P, _I, _I, _I, _I, _P, _I, _P, _P, _P, _P, _L, _I, _P]),
    "pg_stft_project": (_I, [_P, _I, _I, _I, _I, _P, _P, _P, _P, _P]),
    "pg_stft_pairs": (_I, [_P, _I, _I, _I, _I, _P, _F, _F, _P, _P, _P]),
    "pg_istft": (_I, [_P, _P, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P, _I, _P]),
    "pg_peak_normalize": (_I, [_P, _P, _I, _I, _P]),
    "pg_stitch": (_I, [_P, _I, _I, _I, _I, _I, _P, _L, _P, _P]),
    "pg_pack_weight": (_I, [_P, _I, _I, _I, _I, _P, _P, _P, _I, _P]),
    "pg_conv_tc": (_I, [C.POINTER(ConvDesc), _P, _P, _P, _P, _P, _P, C.POINTER(ConvEpilogue), _P]),
    "pg_conv_epilogue_supported": (_I, [C.POINTER(ConvDesc), _I]),
    "pg_bn_running_update": (_I, [_P, _P, _P, _I, _F, _F, _P]),
    "pg_bn_from_running": (_I, [_P, _P, _P, _P, _F, _I, _I, _P, _P, _P]),
    "pg_conv_stat_parts": (_I, [C.POINTER(ConvDesc)]),
    "pg_conv_tc_plan": (_I, [C.POINTER(ConvDesc), C.POINTER(_I), _I]),
    "pg_conv_simt": (_I, [C.POINTER(ConvDesc), _P, _P, _P, _P]),
    "pg_channel_stats": (_I, [_P, _I, _I, _I, _I, _I, _P, _P]),
    "pg_bn_finalize": (_I, [_P, _I, _I, _I, _I, _P, _P, _F, _P, _P, _P]),
    "pg_bn_act": (_I, [_P, _I, _I, _I, _I, _I, _P, _I, C.POINTER(ActDst), C.POINTER(ActDst), _P]),
    "pg_transpose": (_I, [_P, _I, _I, _I, _L, _P, _P, _P, _L, _I, _I, _P, _P]),
    "pg_phase_loss": (_I, [_P, _P, _P, _L, _I, _F, _P, _P, _I, _P, _P]),
    "pg_bn_bwd": (_I, [_P, _I, _I, _I, _P, _P, _F, C.POINTER(GradSrc), C.POINTER(GradSrc), _P, _I, _P, _P, _P, _P, _P, _I, _I, _P]),
    "pg_wgrad_tc": (_I, [C.POINTER(ConvDesc), _P, _P, _P, _P, _I, _P, _I, _P]),
    "pg_wgrad_simt": (_I, [C.POINTER(ConvDesc), _P, _P, _I, _P, _P]),
    "pg_unpack_grad": (_I, [_P, _I, _I, _I, _I, _P, _P]),
    "pg_adam_step": (_I, [_P, _P, _I, _P, _P, _L, _F, _F, _F, _F, _I, _F, _P, _P, _P]),
    "pg_cast_split": (_I, [_P, _L, _P, _P, _I, _P, _P]),
    "pg_stft_ragged": (_I, [_P, _I, _I, _I, _I, _P, _I, _P, _P, _P, _P, _L, _I, _P, _P, _P]),
    "pg_conv_tc_ragged": (_I, [C.POINTER(ConvDesc), _P, _P, _P, _P, _P, _P, C.POINTER(ConvEpilogue), _P, _P]),
    "pg_bn_act_ragged": (_I, [_P, _I, _I, _I, _I, _I, _P, _I, C.POINTER(ActDst), C.POINTER(ActDst), _P, _P]),
    "pg_istft_ragged": (_I, [_P, _P, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P, _I, _P, _P, _P]),
    "pg_stft_packed": (_I, [_P, _L, _P, _I, _I, _I, _I, _P, _I, _P, _P, _P, _P, _L, _I, _P, _P]),
    "pg_peak_normalize_packed": (_I, [_P, _I, _L, _P, _P, _P, _L, _P]),
}
EXPORTS = tuple(_SIGNATURES)

_lib = None
launches = 0  # kernels launched through this binding (bench.py reports it as gpu_launches)


def load():
    global _lib
    if _lib is None:
        path = os.path.normpath(LIB_PATH)
        if not os.path.exists(path):
            raise RuntimeError(
                f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a). The phasegen path has no CPU fallback.")
        lib = C.CDLL(path)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


def last_error():
    return load().pg_last_error().decode("utf-8", "replace")


def call(name, *args, n_kernels=1):
    """Invoke an entry point; raise RuntimeError with the library's message on failure."""
    global launches
    rc = getattr(load(), name)(*args)
    if rc != 0:
        raise RuntimeError(f"{name} failed ({rc}): {last_error()}")
    launches += n_kernels
    return rc


_device_ok = {}


def require_device(device_index):
    """Raise unless the current CUDA device is an sm_100 part (checked once per device)."""
    if device_index not in _device_ok:
        sm, maj, mnr = _I(), _I(), _I()
        rc = load().pg_check_device(C.byref(sm), C.byref(maj), C.byref(mnr))
        if rc != 0:
            raise RuntimeError(f"phasegen: {last_error()}")
        _device_ok[device_index] = (sm.value, maj.value, mnr.value)
    return _device_ok[device_index]
