"""CPU tests: ONNX wire reader/writer, C++ loader/packer (through the C ABI, no GPU), host logic."""
import ctypes as C
import io
import json
import os
import re
import struct

import numpy as np
import pytest

from conftest import REAL_VOICE_CONFIG, ROOT, real_fixture_lines, real_voice_path
from piper_b200 import host, onnx_wire, voicegen


def test_wire_roundtrip(tmp_path):
    m = voicegen.build("tiny", seed=5)
    p = str(tmp_path / "v.onnx")
    onnx_wire.save(p, m)
    m2 = onnx_wire.load(p)
    assert m2.init_order == m.init_order
    for k in m.init_order:
        assert np.array_equal(m.initializers[k], m2.initializers[k]), k
    assert [(n.op_type, n.inputs, n.ints) for n in m.nodes] == [(n.op_type, n.inputs, n.ints) for n in m2.nodes]
    assert m2.opset == 15 and m2.inputs == ["input", "input_lengths", "scales"] and m2.outputs == ["output"]


def test_wire_reader_rejects_garbage(tmp_path):
    p = tmp_path / "bad.onnx"
    p.write_bytes(b"\x3a\xff\xff\xff\x0f" + b"\x00" * 8)
    with pytest.raises(Exception):
        onnx_wire.load(str(p))


@pytest.mark.parametrize("arch", ["tiny", "tiny-high"])
def test_cpp_loader_matches_oracle_loader(lib_built, arch):
    from oracle.voice_loader import load_voice
    from piper_b200 import engine
    path = voicegen.cached_voice(arch)
    spec, w, attrs = load_voice(path)
    d = engine.describe(path)
    for k in ("n_vocab", "hidden", "inter", "filter", "n_heads", "n_layers", "window", "ffn_kernel", "dds_layers",
              "spline_bins", "wn_layers", "wn_kernel", "wn_dilation_rate", "resblock", "up_initial", "hop",
              "dp_flows", "flow_layers", "up_rates", "up_kernels", "up_pads", "rb_kernels", "rb_dilations"):
        assert d[k] == getattr(spec, k), k
    blob = engine.pack(path)
    L = d["layers"]

    def packed(name):
        c = L[name]
        return blob[c["w"]:c["w"] + c["ci"] * c["k"] * c["rows_p"]].reshape(c["ci"], c["k"], c["rows_p"])[:, :, :c["rows"]], c

    got, c = packed("dec_pre")
    assert np.array_equal(got, np.transpose(w["dec.conv_pre.weight"], (1, 2, 0)))
    assert np.array_equal(blob[c["b"]:c["b"] + c["rows"]], w["dec.conv_pre.bias"])
    # WaveNet gate: rows interleaved (tanh_i, sigmoid_i); first executed coupling is the highest index, flipped
    f0 = spec.flow_layers[0]
    W = w[f"flow.flows.{f0}.enc.in_layers.0.weight"]
    H = W.shape[0] // 2
    Wg = np.empty_like(W)
    Wg[0::2], Wg[1::2] = W[:H], W[H:]
    got, _ = packed("flow0_in0")
    assert np.array_equal(got, np.transpose(Wg, (1, 2, 0)))
    got, _ = packed("flow0_pre")
    assert np.array_equal(got, np.transpose(w[f"flow.flows.{f0}.pre.weight"][:, ::-1], (1, 2, 0)))
    got, _ = packed("flow0_post")
    assert np.array_equal(got, np.transpose(w[f"flow.flows.{f0}.post.weight"][::-1], (1, 2, 0)))
    got, _ = packed("flow1_pre")
    assert np.array_equal(got, np.transpose(w[f"flow.flows.{spec.flow_layers[1]}.pre.weight"], (1, 2, 0)))
    # ConvTranspose lowering: rows = co*s + phase, taps reversed
    Wt = w["dec.ups.0.weight"]
    ci, co, k = Wt.shape
    s = spec.up_rates[0]
    m = k // s
    exp = np.zeros((ci, m, co * s), np.float32)
    for j in range(m):
        for phi in range(s):
            exp[:, j, phi::s] = Wt[:, :, phi + (m - 1 - j) * s]
    got, c = packed("up0")
    assert c["up"] == s and c["up_pad"] == spec.up_pads[0] and c["pad"] == m - 1
    assert np.array_equal(got, exp)
    assert abs(d["ea_scale"][0] - float(np.exp(-w["dp.flows.0.logs"][0, 0]))) < 1e-5


def test_cpp_loader_real_voice(lib_built):
    path = real_voice_path()
    if path is None:
        pytest.skip("reference test voice not staged")
    from piper_b200 import engine
    d = engine.describe(path)
    assert (d["n_vocab"], d["hidden"], d["inter"], d["filter"]) == (130, 96, 96, 384)
    assert d["dp_flows"] == [7, 5, 3] and d["flow_layers"] == [6, 4, 2, 0]
    assert d["up_rates"] == [8, 8, 4] and d["hop"] == 256 and d["resblock"] == 2
    assert d["rb_dilations"] == [[1, 2], [2, 6], [3, 12]]
    assert 4.9e6 < d["n_params"] < 5.1e6


def test_cpp_loader_multi_speaker(lib_built):
    from oracle.voice_loader import load_voice
    from piper_b200 import engine
    path = voicegen.cached_voice("tiny-ms")
    spec, w, _ = load_voice(path)
    d = engine.describe(path)
    H = spec.hidden
    assert (d["n_speakers"], d["gin"]) == (spec.n_speakers, spec.gin) == (5, 48)
    assert d["cond_rows"] == H + len(spec.flow_layers) * 2 * H * spec.wn_layers + spec.up_initial


def test_cpp_loader_errors(lib_built, tmp_path):
    from piper_b200 import engine
    from piper_b200._lib import PiperB200Error
    with pytest.raises(PiperB200Error, match="cannot open"):
        engine.describe(str(tmp_path / "missing.onnx"))
    bad = tmp_path / "bad.onnx"
    bad.write_bytes(b"not an onnx file at all")
    with pytest.raises(PiperB200Error):
        engine.describe(str(bad))
    # a voice with a tensor removed must be refused with a message naming it
    m = voicegen.build("tiny")
    del m.initializers["dec.conv_post.weight"]
    m.init_order.remove("dec.conv_post.weight")
    p = str(tmp_path / "broken.onnx")
    onnx_wire.save(p, m)
    with pytest.raises(PiperB200Error, match="dec.conv_post"):
        engine.describe(p)


def test_loader_drops_the_useless_vflow_even_if_the_file_keeps_it(lib_built):
    """models.py:110 drops self.flows[1] in the reverse pass; the stock exporter prunes its weights, another exporter may
    keep them - both loaders must still run ConvFlows 7, 5, 3 only."""
    from piper_b200 import engine
    from oracle.voice_loader import load_voice
    p = voicegen.cached_voice("tiny-keepflow")
    assert engine.describe(p)["dp_flows"] == [7, 5, 3]
    assert load_voice(p)[0].dp_flows == [7, 5, 3]


def test_cpp_loader_rejects_truncated_and_inconsistent_tensors(lib_built, tmp_path):
    """A tensor whose payload does not match its dims must be refused at load (ADVICE r1: heap over-read in the packer)."""
    from piper_b200 import engine
    from piper_b200._lib import PiperB200Error
    good = open(voicegen.cached_voice("tiny"), "rb").read()
    p = tmp_path / "trunc.onnx"
    for cut in (len(good) // 3, len(good) - 7):
        p.write_bytes(good[:cut])
        with pytest.raises(PiperB200Error):
            engine.describe(str(p))
    m = voicegen.build("tiny")
    name = "dec.conv_pre.weight"
    m.initializers[name] = m.initializers[name].reshape(-1)[:-3].copy()        # payload shorter than the conv's shape needs
    q = str(tmp_path / "short.onnx")
    onnx_wire.save(q, m)
    with pytest.raises(PiperB200Error):
        engine.describe(q)


def test_cabi_exports_every_declared_symbol(lib_built):
    header = open(os.path.join(ROOT, "include", "piper_b200.h")).read()
    declared = set(re.findall(r"\b(pb200_[a-z0-9_]+)\s*\(", header))
    from piper_b200 import _lib
    assert declared == set(_lib.SYMBOLS), declared ^ set(_lib.SYMBOLS)
    raw = C.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(raw, name), name
    assert b"sm_100a" in lib_built.pb200_version()


def test_no_cpu_fallback(lib_built):
    """Without a GPU the engine must fail loudly, never fall back."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from piper_b200 import engine
    from piper_b200._lib import PiperB200Error
    with pytest.raises(PiperB200Error, match="CUDA"):
        engine.Voice(voicegen.cached_voice("tiny"), 0)


# ------------------------------------------------------------------ host logic
def test_phonemes_to_ids_reproduces_reference_fixtures():
    lines = real_fixture_lines()
    cfg = host.VoiceConfig.load(REAL_VOICE_CONFIG)
    assert cfg.sample_rate == 16000 and cfg.num_speakers == 1
    for l in lines:
        assert host.phonemes_to_ids(l["phonemes"], cfg.phoneme_id_map) == l["phoneme_ids"]


def test_phonemes_to_ids_layouts_and_missing():
    id_map = {"_": [0], "^": [1], "$": [2], "a": [5], "b": [6, 7]}
    miss = {}
    assert host.phonemes_to_ids(["a", "?", "b"], id_map, missing=miss) == [1, 0, 5, 0, 6, 7, 0, 2]
    assert miss == {"?": 1}
    assert host.phonemes_to_ids(["a"], id_map, layout="python") == [1, 5, 0, 2]
    assert host.phonemes_to_ids([], id_map) == [1, 0, 2]


def test_int16_conversion_semantics():
    a = np.array([0.0, 0.5, -0.5, 0.25, -0.123456], np.float32)
    out = host.audio_float_to_int16(a)
    assert out.dtype == np.int16 and out[1] == 32767 and out[2] == -32767
    assert out[4] == int(np.trunc(np.float32(-0.123456) * (np.float32(32767.0) / np.float32(0.5))))
    # peak floor 0.01 (piper.cpp:411,423): silence is not amplified to full scale
    quiet = host.audio_float_to_int16(np.full(8, 0.001, np.float32))
    assert quiet.max() == int(0.001 * 32767.0 / 0.01)
    assert host.audio_float_to_int16(np.zeros(4, np.float32)).tolist() == [0, 0, 0, 0]


def test_wav_header_layout(tmp_path):
    h = host.wav_header(22050, 2, 1, 1000)
    assert len(h) == 44 and h[:4] == b"RIFF" and h[8:16] == b"WAVEfmt "
    chunk, = struct.unpack("<I", h[4:8])
    assert chunk == 2000 + 36
    rate, bps, align, bits = struct.unpack("<IIHH", h[24:36])
    assert (rate, bps, align, bits) == (22050, 44100, 2, 16)
    p = tmp_path / "a.wav"
    host.write_wav(str(p), np.arange(6000, dtype=np.int16), 16000)
    assert p.stat().st_size == 44 + 12000 >= 10000      # the reference's only assertion (src/cpp/test.cpp:52-55)
    import wave
    with wave.open(str(p)) as w:
        assert (w.getframerate(), w.getnchannels(), w.getsampwidth(), w.getnframes()) == (16000, 1, 2, 6000)


def test_shard_utterances_balanced_and_complete():
    lens = [381, 113, 193, 197, 151, 165, 307, 50, 900]
    for ws in (1, 2, 4, 8):
        plan = host.shard_utterances(lens, ws)
        assert sorted(i for p in plan for i in p) == list(range(len(lens)))
        loads = [sum(lens[i] for i in p) for p in plan]
        assert max(loads) - min(loads) <= max(lens)


def test_voicegen_is_deterministic(tmp_path):
    a = voicegen.build("tiny", seed=7)
    b = voicegen.build("tiny", seed=7)
    c = voicegen.build("tiny", seed=8)
    assert a.init_order == b.init_order
    assert all(np.array_equal(a.initializers[k], b.initializers[k]) for k in a.init_order)
    assert any(not np.array_equal(a.initializers[k], c.initializers[k]) for k in a.init_order)
    ids = voicegen.benchmark_ids(128)
    assert len(ids) == 259 and ids[0] == 1 and ids[-1] == 2 and (ids[1::2] == 0).all() and (ids[2:-1:2] >= 3).all()
    cfg = voicegen.voice_config("medium-ms")
    assert cfg["num_speakers"] == 8 and cfg["audio"]["sample_rate"] == 22050 and len(cfg["phoneme_id_map"]) > 100
