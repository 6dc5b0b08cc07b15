"""ctypes binding of libviettts_b200.so (the C ABI in include/viettts_b200.h).

The product path has NO fallback: if the library is missing or cannot be loaded,
importing the binding raises, and every failing call raises VttsError with the
library's message."""
from __future__ import annotations

import ctypes as C
from pathlib import Path

PKG = Path(__file__).resolve().parent
LIB_PATH = PKG / "libviettts_b200.so"

c_ctx = C.c_void_p
f32p = C.POINTER(C.c_float)
i32p = C.POINTER(C.c_int32)
u8p = C.POINTER(C.c_uint8)

# name -> (restype, argtypes); kept in sync with include/viettts_b200.h by tests/test_abi.py
SIGNATURES = {
    "vtts_version": (C.c_int, []),
    "vtts_create": (C.c_int, [C.c_int, C.POINTER(c_ctx)]),
    "vtts_destroy": (C.c_int, [c_ctx]),
    "vtts_last_error": (C.c_char_p, [c_ctx]),
    "vtts_device_info": (C.c_int, [c_ctx, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int64)]),
    "vtts_set_precision": (C.c_int, [c_ctx, C.c_int]),
    "vtts_get_precision": (C.c_int, [c_ctx]),
    "vtts_debug_conv": (C.c_int, [c_ctx, C.c_int, C.c_void_p, C.c_void_p, C.c_int]),
    "vtts_debug_conv_transpose": (C.c_int, [c_ctx, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                            C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "vtts_debug_tc_stats": (C.c_int, [c_ctx, C.c_int, C.c_void_p]),
    "vtts_debug_substages": (C.c_int, [c_ctx, C.c_int, C.c_void_p]),
    "vtts_debug_pair": (C.c_int, [c_ctx, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p]),
    "vtts_hifigan_blob_floats": (C.c_int64, []),
    "vtts_acoustic_blob_floats": (C.c_int64, []),
    "vtts_duration_blob_floats": (C.c_int64, []),
    "vtts_load_hifigan": (C.c_int, [c_ctx, C.c_void_p, C.c_int64]),
    "vtts_load_duration": (C.c_int, [c_ctx, C.c_void_p, C.c_int64]),
    "vtts_duration_forward": (C.c_int, [c_ctx, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "vtts_predict_duration_host": (C.c_int, [c_ctx, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "vtts_load_acoustic": (C.c_int, [c_ctx, C.c_void_p, C.c_int64]),
    "vtts_load_mel_filterbank": (C.c_int, [c_ctx, C.c_void_p, C.c_int, C.c_int]),
    "vtts_broadcast_weights": (C.c_int, [c_ctx, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "vtts_hifigan_forward": (C.c_int, [c_ctx, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "vtts_acoustic_forward": (C.c_int, [c_ctx, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_uint64,
                                        C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "vtts_melspec": (C.c_int, [c_ctx, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "vtts_debug_read": (C.c_int, [c_ctx, C.c_char_p, C.c_void_p, C.c_int64]),
    "vtts_mel2wave_host": (C.c_int, [c_ctx, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "vtts_predict_mel_host": (C.c_int, [c_ctx, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_uint64,
                                        C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "vtts_synthesize_host": (C.c_int, [c_ctx, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_uint64,
                                       C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "vtts_tts_host": (C.c_int, [c_ctx, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_int, C.c_uint64, C.c_int,
                                C.c_void_p, C.c_void_p, C.POINTER(C.c_int32), C.c_void_p]),
    "vtts_acoustic_teacher_forward": (C.c_int, [c_ctx, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                                C.c_int, C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "vtts_gta_host": (C.c_int, [c_ctx, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "vtts_melspec_host": (C.c_int, [c_ctx, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "vtts_launch_count": (C.c_int64, [c_ctx]),
    "vtts_last_stage_ms": (C.c_int, [c_ctx, C.c_int, C.POINTER(C.c_float)]),
}


class ConvGeometry(C.Structure):
    """vtts_conv_geometry"""
    _fields_ = [("B", C.c_int32), ("T_rows", C.c_int32), ("rows_out", C.c_int32), ("Cin", C.c_int32), ("Cout", C.c_int32),
                ("len", C.c_void_p), ("len_mul", C.c_int32), ("pre_mode", C.c_int32), ("pre_slope", C.c_float),
                ("post_act", C.c_int32)]


class ConvProblem(C.Structure):
    """vtts_conv_problem"""
    _fields_ = [(n, C.c_void_p) for n in ("x0", "x1", "x2", "w", "bias", "resid", "bn_mean", "bn_inv", "bn_off", "out")] + \
               [(n, C.c_int32) for n in ("k", "dil", "in_off", "out_stride", "out_off")]


class VttsError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libviettts_b200 error {code}: {msg}")
        self.code = code


_lib = None


def load() -> C.CDLL:
    """Load the shared library (once).  Raises if it has not been built: there is
    no CPU / PyTorch fallback behind this package."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -m viettts_b200.build` "
            "(or __graft_entry__.build()). viettts_b200 has no CPU fallback."
        )
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export the symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(ctx, rc: int) -> None:
    if rc != 0:
        msg = load().vtts_last_error(ctx)
        raise VttsError(rc, msg.decode() if msg else "?")
