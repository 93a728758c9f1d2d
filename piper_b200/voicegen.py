"""Seeded synthetic piper voices (`.onnx` + `.onnx.json`) on the exact medium / high /
x-low VITS architectures.

The released `en_US-lessac-medium` / `de_DE-thorsten-high` files are catalogue entries
only (`/root/reference/src/python_run/piper/voices.json`) and there is no network, so
the benchmark configs run random-init weights of the same architecture, written in
the same container layout the reference exporter produces
(`/root/reference/src/python/piper_train/export_onnx.py:51-101`; SURVEY.md App. B):
initializers as raw_data, the embedding table named `sid`, flow WN convs as anonymous
`onnx::Conv_N` tensors identified by their bias name, `exp(-dp.flows.0.logs)` as an
anonymous [2,1] Mul operand, Conv / ConvTranspose nodes carrying kernel / dilation /
pad / stride / group attributes.  The files carry only the nodes a loader needs
(Conv, ConvTranspose, Sub, Mul) — they are voice containers, not runnable ONNX graphs.

Architectures: quality presets of `/root/reference/src/python/piper_train/__main__.py:67-82`
and `vits/lightning.py:26-51`, `vits/config.py:44-56`.

Weight statistics are NOT the reference initialisers (those zero-init every flow
`post`/`proj`, making flows identities, and draw decoder weights from N(0, 0.01^2),
giving |o| ~ 2e-2 — a 1e-3 parity bar would be vacuous).  Draws here are
variance-preserving N(0, gain / fan_in) so that every stage is exercised and the
waveform has speech-like amplitude (rms ~ 0.2-0.4, no tanh saturation).
"""
from __future__ import annotations

import json
import math
import os
import tempfile
from typing import Dict, List, Tuple

import numpy as np

from . import onnx_wire

ARCHS: Dict[str, dict] = {
    "x-low": dict(hidden=96, inter=96, filter=384, heads=2, layers=6, resblock=2,
                  up_rates=(8, 8, 4), up_kernels=(16, 16, 8), up_initial=256,
                  rb_kernels=(3, 5, 7), rb_dilations=((1, 2), (2, 6), (3, 12)), sample_rate=16000),
    "medium": dict(hidden=192, inter=192, filter=768, heads=2, layers=6, resblock=2,
                   up_rates=(8, 8, 4), up_kernels=(16, 16, 8), up_initial=256,
                   rb_kernels=(3, 5, 7), rb_dilations=((1, 2), (2, 6), (3, 12)), sample_rate=22050),
    "high": dict(hidden=192, inter=192, filter=768, heads=2, layers=6, resblock=1,
                 up_rates=(8, 8, 2, 2), up_kernels=(16, 16, 4, 4), up_initial=512,
                 rb_kernels=(3, 7, 11), rb_dilations=((1, 3, 5), (1, 3, 5), (1, 3, 5)), sample_rate=22050),
    # small architecture for fast CPU-side tests (same topology, fewer channels)
    "tiny": dict(hidden=32, inter=32, filter=64, heads=2, layers=2, resblock=2,
                 up_rates=(8, 8, 4), up_kernels=(16, 16, 8), up_initial=64,
                 rb_kernels=(3, 5, 7), rb_dilations=((1, 2), (2, 6), (3, 12)), sample_rate=22050),
    # an exporter that keeps the initializers of the ConvFlow the reverse pass drops (dp.flows.1, models.py:110)
    "tiny-keepflow": dict(hidden=32, inter=32, filter=64, heads=2, layers=2, resblock=2,
                          up_rates=(8, 8, 4), up_kernels=(16, 16, 8), up_initial=64,
                          rb_kernels=(3, 5, 7), rb_dilations=((1, 2), (2, 6), (3, 12)), sample_rate=22050,
                          dp_flow_ids=(1, 3, 5, 7)),
    # multi-speaker variants (emb_g + dp.cond + WN cond_layer + dec.cond; gin 512 in piper: lightning.py:81-83)
    "tiny-ms": dict(hidden=32, inter=32, filter=64, heads=2, layers=2, resblock=2,
                    up_rates=(8, 8, 4), up_kernels=(16, 16, 8), up_initial=64,
                    rb_kernels=(3, 5, 7), rb_dilations=((1, 2), (2, 6), (3, 12)), sample_rate=22050,
                    n_speakers=5, gin=48),
    "medium-ms": dict(hidden=192, inter=192, filter=768, heads=2, layers=6, resblock=2,
                      up_rates=(8, 8, 4), up_kernels=(16, 16, 8), up_initial=256,
                      rb_kernels=(3, 5, 7), rb_dilations=((1, 2), (2, 6), (3, 12)), sample_rate=22050,
                      n_speakers=8, gin=512),
    "tiny-high": dict(hidden=32, inter=32, filter=64, heads=2, layers=2, resblock=1,
                      up_rates=(8, 8, 2, 2), up_kernels=(16, 16, 4, 4), up_initial=64,
                      rb_kernels=(3, 7, 11), rb_dilations=((1, 3, 5), (1, 3, 5), (1, 3, 5)),
                      sample_rate=22050),
}


class _Builder:
    def __init__(self, seed: int):
        self.rng = np.random.default_rng(seed)
        self.m = onnx_wire.Model(producer="pytorch", ir_version=8, opset=15)
        self.m.inputs = ["input", "input_lengths", "scales"]
        self.m.outputs = ["output"]
        self.anon = 9000
        self.t = 0

    def normal(self, shape, std) -> np.ndarray:
        return (self.rng.standard_normal(shape, dtype=np.float32) * np.float32(std)).astype(np.float32)

    def add(self, name: str, arr: np.ndarray) -> str:
        assert name not in self.m.initializers, name
        self.m.initializers[name] = np.ascontiguousarray(arr, dtype=np.float32)
        self.m.init_order.append(name)
        return name

    def tmp(self) -> str:
        self.t += 1
        return f"t{self.t}"

    def conv(self, prefix: str, cout: int, cin: int, k: int, *, std=None, gain=1.0, bias_std=0.02,
             dilation=1, pad=0, groups=1, anonymous=False, bias=True, transpose=False, stride=1):
        if transpose:
            shape = (cin, cout, k)
            fan_in = cin * k / stride
        else:
            shape = (cout, cin // groups, k)
            fan_in = (cin // groups) * k
        if std is None:
            std = math.sqrt(gain / fan_in)
        wname = prefix + ".weight"
        if anonymous:
            self.anon += 3
            wname = f"onnx::Conv_{self.anon}"
        self.add(wname, self.normal(shape, std))
        ins = [self.tmp(), wname]
        if bias:
            ins.append(self.add(prefix + ".bias", self.normal((cout,), bias_std)))
        node = onnx_wire.Node(op_type="ConvTranspose" if transpose else "Conv", name=f"Conv_{self.t}",
                              inputs=ins, outputs=[self.tmp()])
        node.ints = {"dilations": [dilation], "group": [groups], "kernel_shape": [k],
                     "pads": [pad, pad], "strides": [stride]}
        self.m.nodes.append(node)

    def layer_norm(self, prefix: str, c: int):
        self.add(prefix + ".gamma", 1.0 + self.normal((c,), 0.1))
        self.add(prefix + ".beta", self.normal((c,), 0.1))


def build(arch: str = "medium", seed: int = 1234, n_vocab: int = 256) -> onnx_wire.Model:
    cfg = ARCHS[arch]
    H, inter, Fc = cfg["hidden"], cfg["inter"], cfg["filter"]
    heads, dk = cfg["heads"], cfg["hidden"] // cfg["heads"]
    b = _Builder(seed)
    n_spk, gin = cfg.get("n_speakers", 1), cfg.get("gin", 0)
    if n_spk > 1:
        # a real `sid` graph input exists, so the exporter keeps the embedding tables' own names
        b.m.inputs = ["input", "input_lengths", "scales", "sid"]
        b.add("enc_p.emb.weight", b.normal((n_vocab, H), H ** -0.5))
        b.add("emb_g.weight", b.normal((n_spk, gin), 1.0))
    else:
        b.add("sid", b.normal((n_vocab, H), H ** -0.5))
    # ---- text encoder (attentions.py:60-74)
    for l in range(cfg["layers"]):
        p = f"enc_p.encoder.attn_layers.{l}"
        b.add(p + ".emb_rel_k", b.normal((1, 9, dk), dk ** -0.5))
        b.add(p + ".emb_rel_v", b.normal((1, 9, dk), dk ** -0.5))
        for c in ("conv_q", "conv_k", "conv_v", "conv_o"):
            b.conv(f"{p}.{c}", H, H, 1, gain=2.0 if c in ("conv_q", "conv_k") else 1.0)
    for l in range(cfg["layers"]):
        b.layer_norm(f"enc_p.encoder.norm_layers_1.{l}", H)
    for l in range(cfg["layers"]):
        p = f"enc_p.encoder.ffn_layers.{l}"
        b.conv(p + ".conv_1", Fc, H, 3, gain=2.0)
        b.conv(p + ".conv_2", H, Fc, 3, gain=1.0)
    for l in range(cfg["layers"]):
        b.layer_norm(f"enc_p.encoder.norm_layers_2.{l}", H)
    b.conv("enc_p.proj", 2 * inter, H, 1, gain=1.0)
    # prior log-std: centre around -0.7 so exp(logs_p) ~ 0.5 (speech-like prior spread)
    b.m.initializers["enc_p.proj.bias"][inter:] -= np.float32(0.7)
    b.m.initializers["enc_p.proj.weight"][inter:] *= np.float32(0.3)
    # ---- stochastic duration predictor (models.py:13-70)
    def dds(prefix):
        for i in range(3):
            b.conv(f"{prefix}.convs_sep.{i}", H, H, 3, dilation=3 ** i, pad=3 ** i, groups=H, gain=1.0)
        for i in range(3):
            b.conv(f"{prefix}.convs_1x1.{i}", H, H, 1, gain=1.0)
        for i in range(3):
            b.layer_norm(f"{prefix}.norms_1.{i}", H)
        for i in range(3):
            b.layer_norm(f"{prefix}.norms_2.{i}", H)
    b.add("dp.flows.0.m", np.array([[-0.3], [0.1]], np.float32))
    logs0 = np.array([[0.35], [-0.1]], np.float32)
    for f in cfg.get("dp_flow_ids", (3, 5, 7)):
        b.conv(f"dp.flows.{f}.pre", H, 1, 1, gain=1.0)
        dds(f"dp.flows.{f}.convs")
        b.conv(f"dp.flows.{f}.proj", 29, H, 1, std=0.05)
    b.conv("dp.pre", H, H, 1)
    if n_spk > 1:
        b.conv("dp.cond", H, gin, 1, gain=0.25)
    b.conv("dp.proj", H, H, 1)
    dds("dp.convs")
    # Sub(z, m) -> Mul(., exp(-logs)) : the only trace dp.flows.0.logs leaves in an export
    sub = onnx_wire.Node(op_type="Sub", name="Sub_ea", inputs=[b.tmp(), "dp.flows.0.m"], outputs=[b.tmp()])
    b.m.nodes.append(sub)
    mul_name = "onnx::Mul_7201"
    b.add(mul_name, np.exp(-logs0).astype(np.float32))
    b.m.nodes.append(onnx_wire.Node(op_type="Mul", name="Mul_ea", inputs=[sub.outputs[0], mul_name],
                                    outputs=[b.tmp()]))
    # ---- flow (models.py:212-254 ; modules.py:412-466)
    for f in (0, 2, 4, 6):
        p = f"flow.flows.{f}"
        b.conv(p + ".pre", H, inter // 2, 1)
        if n_spk > 1:   # weight-normed like the in/res_skip layers -> constant-folded to an anonymous tensor
            b.conv(f"{p}.enc.cond_layer", 2 * H * 4, gin, 1, anonymous=True, gain=0.25)
        for i in range(4):
            b.conv(f"{p}.enc.in_layers.{i}", 2 * H, H, 5, pad=2, anonymous=True, gain=2.0)
            b.conv(f"{p}.enc.res_skip_layers.{i}", 2 * H if i < 3 else H, H, 1, anonymous=True, gain=2.0)
        b.conv(p + ".post", inter // 2, H, 1, std=0.05)
    # ---- generator (models.py:299-368)
    C = cfg["up_initial"]
    b.conv("dec.conv_pre", C, inter, 7, pad=3)
    if n_spk > 1:
        b.conv("dec.cond", C, gin, 1, gain=0.25)
    nk = len(cfg["rb_kernels"])
    for i, (u, k) in enumerate(zip(cfg["up_rates"], cfg["up_kernels"])):
        b.conv(f"dec.ups.{i}", C // 2, C, k, transpose=True, stride=u, pad=(k - u) // 2, gain=2.0)
        C //= 2
        for j in range(nk):
            kk = cfg["rb_kernels"][j]
            rb = f"dec.resblocks.{i * nk + j}"
            for c, d in enumerate(cfg["rb_dilations"][j]):
                if cfg["resblock"] == 1:
                    b.conv(f"{rb}.convs1.{c}", C, C, kk, dilation=d, pad=d * (kk - 1) // 2, gain=1.0)
                    b.conv(f"{rb}.convs2.{c}", C, C, kk, pad=(kk - 1) // 2, gain=0.5)
                else:
                    b.conv(f"{rb}.convs.{c}", C, C, kk, dilation=d, pad=d * (kk - 1) // 2, gain=0.5)
    b.conv("dec.conv_post", 1, C, 7, pad=3, bias=False, gain=0.02)
    return b.m


def voice_config(arch: str, n_vocab: int = 256) -> dict:
    n_spk = ARCHS[arch].get("n_speakers", 1)
    """The `.onnx.json` twin (fields parsed at /root/reference/src/cpp/piper.cpp:47-214)."""
    symbols = ["_", "^", "$", " "] + [chr(0x61 + i) for i in range(26)] + [chr(0x250 + i) for i in range(96)]
    id_map = {s: [i] for i, s in enumerate(symbols[:n_vocab])}
    return {
        "audio": {"sample_rate": ARCHS[arch]["sample_rate"]},
        "espeak": {"voice": "en-us"},
        "inference": {"noise_scale": 0.667, "length_scale": 1, "noise_w": 0.8},
        "phoneme_type": "espeak",
        "phoneme_map": {},
        "phoneme_id_map": id_map,
        "num_symbols": n_vocab,
        "num_speakers": n_spk,
        "speaker_id_map": {f"speaker{i}": i for i in range(n_spk)} if n_spk > 1 else {},
    }


def write_voice(path: str, arch: str = "medium", seed: int = 1234, n_vocab: int = 256) -> str:
    """Write `<path>` (.onnx) and `<path>.json`; returns path.  Idempotent per (arch, seed)."""
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    tmp = path + f".tmp{os.getpid()}"
    onnx_wire.save(tmp, build(arch, seed, n_vocab))
    os.replace(tmp, path)
    with open(path + ".json", "w") as f:
        json.dump(voice_config(arch, n_vocab), f)
    return path


def cached_voice(arch: str = "medium", seed: int = 1234, root: str | None = None) -> str:
    # per user: the machine's temporary directory may be shared, and another user's cache is not writable
    root = root or os.environ.get("PIPER_B200_VOICE_CACHE",
                                  os.path.join(tempfile.gettempdir(), f"piper_b200_voices-{os.getuid()}"))
    path = os.path.join(root, f"synthetic-{arch}-s{seed}.onnx")
    if not (os.path.exists(path) and os.path.exists(path + ".json")):
        write_voice(path, arch, seed)
    return path


def benchmark_ids(n_phonemes: int = 128, seed: int = 1234, n_vocab: int = 256) -> np.ndarray:
    """`BOS, PAD, (p, PAD)*n, EOS` with p ~ U{3..n_vocab-1}  (SURVEY.md §8d config 2;
    layout of piper-phonemize `phonemes_to_ids`, ids from piper.hpp:44-47)."""
    rng = np.random.default_rng(seed)
    p = rng.integers(3, n_vocab, size=n_phonemes)
    ids = np.zeros(2 * n_phonemes + 3, np.int64)
    ids[0] = 1
    ids[2:-1:2] = p
    ids[-1] = 2
    return ids
