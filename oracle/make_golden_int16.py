"""Mint tests/golden/int16_cpp.npz from the reference's own loops (oracle/_ref/libint16_ref.so = piper.cpp:411-431
compiled by oracle/build_ref.py) and from the reference's Python twin (python_run/piper/util.py:5-12, imported
read-only).  Build container only:  python -m oracle.build_ref && python -m oracle.make_golden_int16
Also mints tests/golden/reference/int16_seeded.npz (both on the seeded inputs of tests/test_oracle.py).
"""
from __future__ import annotations

import importlib.util
import os

import numpy as np

from oracle import int16_oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
UTIL = "/root/reference/src/python_run/piper/util.py"


def cases():
    rng = np.random.default_rng(20260922)
    c = {
        "zeros": np.zeros(64, np.float32),
        "below_floor": np.full(96, 0.001, np.float32) * rng.choice([-1, 1], 96).astype(np.float32),   # peak < 0.01 -> floor
        "at_floor": np.array([0.01, -0.01, 0.005, -0.0099999], np.float32),
        "single": np.array([0.37], np.float32),
        "neg_peak": np.concatenate([[-0.9], rng.uniform(-0.5, 0.5, 255)]).astype(np.float32),       # peak is negative
        "speech_like": (0.3 * rng.standard_normal(8192)).astype(np.float32).clip(-0.98, 0.98),
        "tanh_out": np.tanh(rng.standard_normal(4096) * 2).astype(np.float32),                       # saturating waveform
        "tiny_denormal": (rng.standard_normal(128) * 1e-39).astype(np.float32),
        "ramp": np.linspace(-1, 1, 4097, dtype=np.float32),
    }
    # products that land within an ulp of an integer / of the clamp edges
    k = np.arange(-32767, 32768, 257, dtype=np.float32)
    c["near_integers"] = np.concatenate([k / np.float32(32767.0), np.nextafter(k / np.float32(32767.0), np.float32(2)),
                                         np.nextafter(k / np.float32(32767.0), np.float32(-2))]).astype(np.float32)
    return c


def main():
    spec = importlib.util.spec_from_file_location("ref_piper_util", UTIL)
    util = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(util)
    out = {}
    for name, a in cases().items():
        out[f"{name}.in"] = a
        out[f"{name}.cpp"] = int16_oracle.float_to_int16_ref(a)
        out[f"{name}.py"] = util.audio_float_to_int16(a)
        print(f"{name}: n={a.size} cpp[:4]={out[f'{name}.cpp'][:4]} differs_from_python={int((out[f'{name}.cpp'] != out[f'{name}.py']).sum())}")
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "int16_cpp.npz"), **out)
    mint_seeded(util)


def seeded_cases(seed, spec):
    """The seeded inputs tests/test_oracle.py draws: (n, amplitude) pairs, tanh-shaped up to amplitude 1."""
    rng = np.random.default_rng(seed)
    return [(amp * np.tanh(rng.standard_normal(n))).astype(np.float32) if amp <= 1 else
            (amp * rng.standard_normal(n)).astype(np.float32) for n, amp in spec]


CPP_SEEDED = (11, ((1, 1.0), (7, 0.004), (1000, 0.5), (65536, 1.0), (4099, 3.0)))
PY_SEEDED = (12, ((3, 1.0), (500, 0.003), (30000, 0.7)))


def mint_seeded(util):
    """tests/golden/reference/int16_seeded.npz: the compiled loops and util.py on the tests' seeded inputs (at most 2048
    fixed, seeded sample positions of each)."""
    out = {}
    for tag, (seed, spec), fn in (("cpp", CPP_SEEDED, int16_oracle.float_to_int16_ref),
                                  ("py", PY_SEEDED, util.audio_float_to_int16)):
        for i, a in enumerate(seeded_cases(seed, spec)):
            idx = np.sort(np.random.default_rng(i).choice(a.size, min(a.size, 2048), replace=False)).astype(np.int32)
            out[f"{tag}{i}.idx"], out[f"{tag}{i}.val"] = idx, np.asarray(fn(a))[idx]
    os.makedirs(os.path.join(ROOT, "tests", "golden", "reference"), exist_ok=True)
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "reference", "int16_seeded.npz"), **out)


if __name__ == "__main__":
    main()
