"""Python host mirror of the engine's public call (the twin of `PiperVoice` in
/root/reference/src/python_run/piper/voice.py:20-185 for the ids -> audio half).

Everything here is a thin ctypes shim over the C ABI; arrays are numpy (host) buffers.
"""
from __future__ import annotations

import ctypes as C
import json
from typing import List, Optional, Sequence, Tuple

import numpy as np

from . import _lib
from ._lib import Noise, VoiceInfo, check


def _fptr(a: Optional[np.ndarray]):
    return a.ctypes.data_as(C.POINTER(C.c_float)) if a is not None else None


def describe(onnx_path: str) -> dict:
    """Host-only: inferred hyper-parameters + packed layout (no GPU needed)."""
    lib = _lib.load()
    buf = C.create_string_buffer(1 << 16)
    check(lib.pb200_voice_describe(onnx_path.encode(), buf, len(buf)))
    return json.loads(buf.value.decode())


def pack(onnx_path: str) -> np.ndarray:
    """Host-only: the packed fp32 weight blob exactly as it is uploaded to HBM."""
    lib = _lib.load()
    n = C.c_int64(0)
    check(lib.pb200_voice_pack(onnx_path.encode(), None, C.byref(n)))
    blob = np.empty(n.value, np.float32)
    check(lib.pb200_voice_pack(onnx_path.encode(), _fptr(blob), C.byref(n)))
    return blob


class Voice:
    def __init__(self, onnx_path: str, device: int = 0, upload: bool = True):
        self._lib = _lib.load()
        self._h = C.c_void_p()
        check(self._lib.pb200_voice_load_ex(onnx_path.encode(), device, 0 if upload else 1, C.byref(self._h)))
        self.device = device
        info = VoiceInfo()
        check(self._lib.pb200_voice_get_info(self._h, C.byref(info)))
        self.info = info
        self.hop = info.hop
        self.inter = info.inter
        self.path = onnx_path
        self._keep: list = []

    def close(self):
        if self._h:
            self._lib.pb200_voice_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ helpers
    def _noise(self, eps_dp, eps_z, seed) -> Tuple[Optional[Noise], list]:
        keep = []
        n = Noise()
        n.seed = int(seed)
        n.z_stride = 0
        if eps_dp is not None:
            a = np.ascontiguousarray(np.concatenate([np.asarray(e, np.float32).reshape(-1) for e in eps_dp]))
            keep.append(a)
            n.eps_dp = _fptr(a)
        if eps_z is not None:
            a = np.ascontiguousarray(np.asarray(eps_z, np.float32))
            assert a.ndim == 3 and a.shape[1] == self.inter, "eps_z must be [B][inter][z_stride]"
            keep.append(a)
            n.eps_z = _fptr(a)
            n.z_stride = a.shape[2]
        return n, keep

    @staticmethod
    def _ids(ids_list: Sequence[Sequence[int]]):
        lens = np.asarray([len(i) for i in ids_list], np.int64)
        cat = np.ascontiguousarray(np.concatenate([np.asarray(i, np.int64) for i in ids_list]))
        return cat, lens

    # ------------------------------------------------------------------ public
    def synthesize(self, ids: Sequence[int], scales=(0.667, 1.0, 0.8), eps_dp=None, eps_z=None, seed=0, sid=None):
        """One utterance through `pb200_synthesize` -> (fp32 waveform, infer_seconds)."""
        ids_a = np.ascontiguousarray(np.asarray(ids, np.int64))
        sc = np.asarray(scales, np.float32)
        n, keep = self._noise(None if eps_dp is None else [eps_dp],
                              None if eps_z is None else np.asarray(eps_z, np.float32)[None], seed)
        audio = C.POINTER(C.c_float)()
        ns = C.c_int64(0)
        sec = C.c_double(0)
        sid_c = None if sid is None else C.byref(C.c_int64(int(sid)))
        check(self._lib.pb200_synthesize(self._h, ids_a.ctypes.data_as(C.POINTER(C.c_int64)), len(ids_a), _fptr(sc),
                                         sid_c, C.byref(n), C.byref(audio), C.byref(ns), C.byref(sec)))
        out = np.ctypeslib.as_array(audio, shape=(ns.value,)).copy()
        return out, sec.value

    def synthesize_batch(self, ids_list, scales=(0.667, 1.0, 0.8), eps_dp=None, eps_z=None, seed=0,
                         w_ceil_override=None, copy=True):
        """B utterances -> (list of fp32 waveforms, infer_seconds)."""
        cat, lens = self._ids(ids_list)
        B = len(lens)
        sc = np.asarray(scales, np.float32)
        n, keep = self._noise(eps_dp, eps_z, seed)
        ov = None
        if w_ceil_override is not None:
            ov = np.ascontiguousarray(np.concatenate([np.asarray(w, np.int32) for w in w_ceil_override]))
        audio = C.POINTER(C.c_float)()
        ns = (C.c_int64 * B)()
        sec = C.c_double(0)
        check(self._lib.pb200_synthesize_batch(
            self._h, cat.ctypes.data_as(C.POINTER(C.c_int64)), lens.ctypes.data_as(C.POINTER(C.c_int64)), B, _fptr(sc),
            C.byref(n), ov.ctypes.data_as(C.POINTER(C.c_int32)) if ov is not None else None, C.byref(audio), ns,
            C.byref(sec)))
        counts = np.asarray(list(ns), np.int64)
        total = int(counts.sum())
        flat = np.ctypeslib.as_array(audio, shape=(total,))
        if not copy:
            return flat, counts, sec.value
        offs = np.concatenate([[0], np.cumsum(counts)])
        return [flat[offs[b]:offs[b + 1]].copy() for b in range(B)], sec.value

    def synthesize_int16(self, ids_list, scales=(0.667, 1.0, 0.8), eps_dp=None, eps_z=None, seed=0, copy=True):
        cat, lens = self._ids(ids_list)
        B = len(lens)
        sc = np.asarray(scales, np.float32)
        n, keep = self._noise(eps_dp, eps_z, seed)
        audio = C.POINTER(C.c_int16)()
        ns = (C.c_int64 * B)()
        sec = C.c_double(0)
        check(self._lib.pb200_synthesize_int16(
            self._h, cat.ctypes.data_as(C.POINTER(C.c_int64)), lens.ctypes.data_as(C.POINTER(C.c_int64)), B, _fptr(sc),
            C.byref(n), C.byref(audio), ns, C.byref(sec)))
        counts = np.asarray(list(ns), np.int64)
        flat = np.ctypeslib.as_array(audio, shape=(int(counts.sum()),))
        if not copy:
            return flat, counts, sec.value
        offs = np.concatenate([[0], np.cumsum(counts)])
        return [flat[offs[b]:offs[b + 1]].copy() for b in range(B)], sec.value

    def vocode(self, z: np.ndarray):
        """Generator only: z [B][inter][frames] -> ([B][frames*hop], infer_seconds)."""
        z = np.ascontiguousarray(np.asarray(z, np.float32))
        B, I, Fr = z.shape
        assert I == self.inter
        audio = C.POINTER(C.c_float)()
        sec = C.c_double(0)
        check(self._lib.pb200_vocode(self._h, _fptr(z), B, Fr, C.byref(audio), C.byref(sec)))
        return np.ctypeslib.as_array(audio, shape=(B, Fr * self.hop)).copy(), sec.value

    def encode(self, ids: Sequence[int], scales=(0.667, 1.0, 0.8), eps_dp=None, eps_z=None, seed=0) -> np.ndarray:
        """Encoder half of the streaming split: ids -> z_p [inter][frames]."""
        ids_a = np.ascontiguousarray(np.asarray(ids, np.int64))
        sc = np.asarray(scales, np.float32)
        n, keep = self._noise(None if eps_dp is None else [eps_dp],
                              None if eps_z is None else np.asarray(eps_z, np.float32)[None], seed)
        zp = C.POINTER(C.c_float)()
        fr = C.c_int64(0)
        sec = C.c_double(0)
        check(self._lib.pb200_encode(self._h, ids_a.ctypes.data_as(C.POINTER(C.c_int64)), len(ids_a), _fptr(sc),
                                     C.byref(n), C.byref(zp), C.byref(fr), C.byref(sec)))
        return np.ctypeslib.as_array(zp, shape=(self.inter, fr.value)).copy()

    def decode(self, z_p: np.ndarray):
        """Decoder half: flow reverse + generator on z_p [B][inter][frames] -> [B][frames*hop]."""
        z = np.ascontiguousarray(np.asarray(z_p, np.float32))
        if z.ndim == 2:
            z = z[None]
        B, I, Fr = z.shape
        assert I == self.inter
        audio = C.POINTER(C.c_float)()
        sec = C.c_double(0)
        check(self._lib.pb200_decode(self._h, _fptr(z), B, Fr, C.byref(audio), C.byref(sec)))
        return np.ctypeslib.as_array(audio, shape=(B, Fr * self.hop)).copy()

    def stage(self, ids_list, scales=(0.667, 1.0, 0.8), seed=0, w_ceil_override=None):
        cat, lens = self._ids(ids_list)
        sc = np.asarray(scales, np.float32)
        n, keep = self._noise(None, None, seed)
        ov = None
        if w_ceil_override is not None:
            ov = np.ascontiguousarray(np.concatenate([np.asarray(w, np.int32) for w in w_ceil_override]))
        check(self._lib.pb200_stage(self._h, cat.ctypes.data_as(C.POINTER(C.c_int64)),
                                    lens.ctypes.data_as(C.POINTER(C.c_int64)), len(lens), _fptr(sc), C.byref(n),
                                    ov.ctypes.data_as(C.POINTER(C.c_int32)) if ov is not None else None))

    def run_staged(self) -> Tuple[int, float]:
        total = C.c_int64(0)
        ms = C.c_float(0)
        check(self._lib.pb200_run_staged(self._h, C.byref(total), C.byref(ms)))
        return total.value, ms.value

    def stage_times(self) -> List[float]:
        ms = (C.c_float * 5)()
        check(self._lib.pb200_stage_times(self._h, ms))
        return list(ms)

    def weight_buffers(self):
        """(device pointer, bytes) of the fp32 weight blob (for the load-time NCCL broadcast)."""
        p = C.c_void_p()
        n = C.c_int64(0)
        check(self._lib.pb200_voice_weight_buffers(self._h, C.byref(p), C.byref(n)))
        return p.value, n.value

    def set_speakers(self, sids):
        """Speaker ids for the following calls (item b uses sids[min(b, len-1)]); empty -> speaker 0."""
        a = np.ascontiguousarray(np.asarray(list(sids), np.int64))
        check(self._lib.pb200_set_speakers(self._h, a.ctypes.data_as(C.POINTER(C.c_int64)), len(a)))

    def set_mma(self, mask: int):
        check(self._lib.pb200_set_mma(self._h, int(mask)))

    def set_profile(self, on: bool):
        check(self._lib.pb200_set_profile(self._h, 1 if on else 0))

    def profile(self) -> dict:
        buf = C.create_string_buffer(1 << 14)
        check(self._lib.pb200_profile_read(self._h, buf, len(buf)))
        return json.loads(buf.value.decode())

    def profile_launches(self) -> list:
        """Every conv launch of the last profiled call, in order (tag, us, shape, algorithmic bytes / FLOP)."""
        buf = C.create_string_buffer(1 << 19)
        check(self._lib.pb200_profile_read_launches(self._h, buf, len(buf)))
        return json.loads(buf.value.decode())

    def set_debug(self, on: bool):
        check(self._lib.pb200_set_debug(self._h, 1 if on else 0))

    def tap(self, name: str, b: int = 0) -> np.ndarray:
        ch, ln = C.c_int32(0), C.c_int32(0)
        check(self._lib.pb200_tap_shape(self._h, name.encode(), b, C.byref(ch), C.byref(ln)))
        buf = np.empty((ch.value, ln.value), np.float32)
        check(self._lib.pb200_tap_read(self._h, name.encode(), b, _fptr(buf), buf.size))
        return buf


def debug_conv1d(backend: int, x, w, bias=None, dil: int = 1, pre_slope: float = 0.0, resid=None) -> np.ndarray:
    """One same-padded Conv1d through the CUDA-core (0) or tensor-core (1) kernel (unit-test hook)."""
    x = np.ascontiguousarray(x, np.float32)
    w = np.ascontiguousarray(w, np.float32)
    B, ci, L = x.shape
    co, ci2, k = w.shape
    assert ci == ci2
    y = np.empty((B, co, L), np.float32)
    b = None if bias is None else np.ascontiguousarray(bias, np.float32)
    r = None if resid is None else np.ascontiguousarray(resid, np.float32)
    check(_lib.load().pb200_debug_conv1d(backend, _fptr(x), B, ci, L, _fptr(w), _fptr(b), co, k, dil, pre_slope,
                                         _fptr(r), _fptr(y)))
    return y


EPILOGUES = dict(BIAS=0, RELU=1, RES=2, GATE=3, WN=4, SUBFROM=5, UPSAMPLE=6, MRF=7)   # csrc/kernels.cuh Epilogue


def debug_conv(backend: int, x, w, lens, *, epi: str = "BIAS", bias=None, bias_item=None, dil: int = 1, pad=None,
               slope=None, y=None, y2=None, r=None, y_is_r: bool = False, split: int = 0, first: int = 0, up: int = 1,
               up_pad: int = 0, q_extra: int = 0, mrf: int = 0, mrf_n: int = 1, len_scale: int = 1, flat: bool = False,
               latency: bool = False):
    """One conv launch with a fused epilogue on a ragged batch, packed and launched as the engine does it (unit-test hook,
    pb200_debug_conv in include/piper_b200.h).  x, y, y2, r are [B][C][pitch], or [C][B][pitch] with flat=True; item b is
    valid on [0, lens[b] * len_scale).  w [rows][ci][k]; bias [rows]; bias_item [B][stride]; slope: leaky-relu before the
    conv (None: no pre-activation); pad defaults to dil * (k - 1) // 2.  y and y2 are in/out: the launch starts from copies
    of them, which come back whole as (y, y2) (None for a buffer not passed).  y_is_r: r is read from y, in place."""
    def f32(a):
        return None if a is None else np.ascontiguousarray(a, np.float32)
    x, w, r, bias, bias_item = f32(x), f32(w), f32(r), f32(bias), f32(bias_item)
    y = None if y is None else np.array(y, np.float32, order="C")
    y2 = None if y2 is None else np.array(y2, np.float32, order="C")
    lens = np.ascontiguousarray(lens, np.int32)
    rows, ci, k = w.shape
    ch = 0 if flat else 1                                  # index of the channel axis

    def dims(a):
        return (0, 0) if a is None else (a.shape[ch], a.shape[2])
    (_, cs_x), (C_y, cs_y), (C_y2, cs_y2), (C_r, cs_r) = dims(x), dims(y), dims(y2), dims(r)
    assert x.shape[ch] == ci and x.shape[1 - ch] == len(lens)
    desc = (C.c_int32 * 23)(ci, rows, k, dil, dil * (k - 1) // 2 if pad is None else pad, q_extra, 0 if slope is None else 1,
                            EPILOGUES[epi], split, first, up, up_pad, mrf, mrf_n, len_scale, cs_x, cs_y, cs_y2, cs_r,
                            C_y, C_y2, C_r, (1 if y_is_r else 0) | (2 if flat else 0) | (4 if latency else 0))
    check(_lib.load().pb200_debug_conv(backend, desc, 0.0 if slope is None else slope, _fptr(x), _fptr(w), _fptr(bias),
                                       _fptr(bias_item), 0 if bias_item is None else bias_item.shape[1],
                                       lens.ctypes.data_as(C.POINTER(C.c_int32)), len(lens), _fptr(y), _fptr(y2), _fptr(r)))
    return y, y2


def launch_count() -> int:
    return int(_lib.load().pb200_launch_count())
