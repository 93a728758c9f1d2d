"""ctypes binding of libpiper_b200.so (the C ABI declared in include/piper_b200.h).

The library is built in-tree by `__graft_entry__.build()` / `make -C piper_b200/csrc`.
There is no Python or CPU fallback: if the shared object is missing, importing any
engine entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpiper_b200.so")


class VoiceInfo(C.Structure):
    _fields_ = [(n, C.c_int32) for n in
                ("n_vocab", "hidden", "inter", "filter", "n_heads", "n_layers", "window", "resblock",
                 "n_upsamples", "hop", "up_initial", "device", "n_speakers", "gin")] + \
               [("n_params", C.c_int64), ("weight_bytes", C.c_int64)]


class Noise(C.Structure):
    _fields_ = [("eps_dp", C.POINTER(C.c_float)), ("eps_z", C.POINTER(C.c_float)),
                ("z_stride", C.c_int64), ("seed", C.c_uint64)]


# every symbol include/piper_b200.h declares: name -> (restype, argtypes)
_p = C.POINTER
SYMBOLS = {
    "pb200_voice_load": (C.c_int, [C.c_char_p, C.c_int, _p(C.c_void_p)]),
    "pb200_voice_load_ex": (C.c_int, [C.c_char_p, C.c_int, C.c_int32, _p(C.c_void_p)]),
    "pb200_voice_weight_buffers": (C.c_int, [C.c_void_p, _p(C.c_void_p), _p(C.c_int64)]),
    "pb200_voice_free": (None, [C.c_void_p]),
    "pb200_voice_get_info": (C.c_int, [C.c_void_p, _p(VoiceInfo)]),
    "pb200_voice_describe": (C.c_int, [C.c_char_p, C.c_char_p, C.c_int64]),
    "pb200_voice_pack": (C.c_int, [C.c_char_p, _p(C.c_float), _p(C.c_int64)]),
    "pb200_synthesize": (C.c_int, [C.c_void_p, _p(C.c_int64), C.c_int64, _p(C.c_float), _p(C.c_int64), _p(Noise),
                                   _p(_p(C.c_float)), _p(C.c_int64), _p(C.c_double)]),
    "pb200_synthesize_batch": (C.c_int, [C.c_void_p, _p(C.c_int64), _p(C.c_int64), C.c_int32, _p(C.c_float), _p(Noise),
                                         _p(C.c_int32), _p(_p(C.c_float)), _p(C.c_int64), _p(C.c_double)]),
    "pb200_synthesize_int16": (C.c_int, [C.c_void_p, _p(C.c_int64), _p(C.c_int64), C.c_int32, _p(C.c_float), _p(Noise),
                                         _p(_p(C.c_int16)), _p(C.c_int64), _p(C.c_double)]),
    "pb200_vocode": (C.c_int, [C.c_void_p, _p(C.c_float), C.c_int32, C.c_int64, _p(_p(C.c_float)), _p(C.c_double)]),
    "pb200_encode": (C.c_int, [C.c_void_p, _p(C.c_int64), C.c_int64, _p(C.c_float), _p(Noise), _p(_p(C.c_float)),
                               _p(C.c_int64), _p(C.c_double)]),
    "pb200_decode": (C.c_int, [C.c_void_p, _p(C.c_float), C.c_int32, C.c_int64, _p(_p(C.c_float)), _p(C.c_double)]),
    "pb200_stage": (C.c_int, [C.c_void_p, _p(C.c_int64), _p(C.c_int64), C.c_int32, _p(C.c_float), _p(Noise),
                              _p(C.c_int32)]),
    "pb200_run_staged": (C.c_int, [C.c_void_p, _p(C.c_int64), _p(C.c_float)]),
    "pb200_stage_times": (C.c_int, [C.c_void_p, _p(C.c_float)]),
    "pb200_set_profile": (C.c_int, [C.c_void_p, C.c_int32]),
    "pb200_profile_read": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int64]),
    "pb200_profile_read_launches": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int64]),
    "pb200_set_mma": (C.c_int, [C.c_void_p, C.c_int32]),
    "pb200_debug_conv1d": (C.c_int, [C.c_int32, _p(C.c_float), C.c_int32, C.c_int32, C.c_int32, _p(C.c_float),
                                     _p(C.c_float), C.c_int32, C.c_int32, C.c_int32, C.c_float, _p(C.c_float),
                                     _p(C.c_float)]),
    "pb200_debug_conv": (C.c_int, [C.c_int32, _p(C.c_int32), C.c_float, _p(C.c_float), _p(C.c_float), _p(C.c_float),
                                   _p(C.c_float), C.c_int32, _p(C.c_int32), C.c_int32, _p(C.c_float), _p(C.c_float),
                                   _p(C.c_float)]),
    "pb200_debug_mrf_pack": (C.c_int, [C.c_char_p, C.c_int32, C.c_int32, _p(C.c_int32), _p(C.c_uint8), _p(C.c_int64), _p(C.c_float),
                                       _p(C.c_int64)]),
    "pb200_release": (None, [C.c_void_p, C.c_void_p]),
    "pb200_set_speakers": (C.c_int, [C.c_void_p, _p(C.c_int64), C.c_int32]),
    "pb200_set_debug": (C.c_int, [C.c_void_p, C.c_int32]),
    "pb200_tap_shape": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int32, _p(C.c_int32), _p(C.c_int32)]),
    "pb200_tap_read": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int32, _p(C.c_float), C.c_int64]),
    "pb200_launch_count": (C.c_uint64, []),
    "pb200_last_error": (C.c_char_p, []),
    "pb200_version": (C.c_char_p, []),
}

_lib = None


def load() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(piper_b200 has no CPU / Python fallback)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


class PiperB200Error(RuntimeError):
    pass


def check(rc: int) -> None:
    if rc != 0:
        raise PiperB200Error(load().pb200_last_error().decode("utf-8", "replace"))
