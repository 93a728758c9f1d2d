"""GPU parity tests: the CUDA engine, called through the C ABI, against the CPU oracle and the golden
fixtures minted from the reference source.  Tolerance (BASELINE.json north_star): waveform within
1e-3 max-abs fp32 on identical phoneme ids and injected noise; predicted durations exactly equal."""
import glob
import os

import numpy as np
import pytest

from conftest import GOLDEN, real_fixture_lines, real_voice_path
from piper_b200 import voicegen

pytestmark = pytest.mark.gpu
TOL = 1e-3


def _voice_path(tag):
    if tag.startswith("real:"):
        p = real_voice_path()
        if p is None:
            pytest.skip("reference test voice not staged (oracle/_ref/voice)")
        return p
    _, arch, seed = tag.split(":")
    return voicegen.cached_voice(arch, int(seed))


_cache = {}


def _pair(tag):
    """(engine voice, oracle) for a voice tag, cached per session."""
    if tag not in _cache:
        from oracle.voice_loader import load_voice
        from oracle.vits_oracle import Oracle
        from piper_b200 import engine
        path = _voice_path(tag)
        spec, w, attrs = load_voice(path)
        _cache[tag] = (engine.Voice(path, 0), Oracle(spec, w, attrs))
    return _cache[tag]


def _noise(inter, n_ids, seed, cols=None):
    rng = np.random.default_rng(seed)
    return (rng.standard_normal((2, n_ids)).astype(np.float32),
            rng.standard_normal((inter, cols or 6 * n_ids + 16)).astype(np.float32))


@pytest.mark.parametrize("name", sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN, "*.npz"))
                                        if not os.path.basename(p).startswith(("stream_", "int16_"))))
def test_engine_matches_reference_golden(name):
    g = np.load(os.path.join(GOLDEN, name + ".npz"))
    voice, _ = _pair(str(g["voice"]))
    voice.set_debug(True)
    audio, _ = voice.synthesize(g["ids"], g["scales"], g["eps_dp"] if "eps_dp" in g else None,
                                g["eps_z"] if "eps_z" in g else None, sid=int(g["sid"]) if "sid" in g else None)
    cum = voice.tap("cum")[0]
    voice.set_debug(False)
    w_ceil = np.diff(np.concatenate([[0], cum])).astype(np.int32)
    assert np.array_equal(w_ceil, g["w_ceil"])
    assert audio.shape == g["audio"].shape
    assert np.abs(audio - g["audio"]).max() <= TOL


@pytest.mark.parametrize("tag,n_ph", [("synthetic:tiny:1234", 20), ("synthetic:tiny-high:1234", 20),
                                      ("real:test_voice", 0), ("synthetic:medium:1234", 128),
                                      ("synthetic:high:1234", 64)])
def test_stage_by_stage_parity(tag, n_ph):
    voice, orc = _pair(tag)
    ids = real_fixture_lines()[5]["phoneme_ids"] if tag.startswith("real:") else voicegen.benchmark_ids(n_ph, seed=3)
    eps_dp, eps_z = _noise(orc.s.inter, len(ids), 77)
    scales = (0.667, 1.0, 0.8)
    dump = {}
    ref = orc.infer(ids, scales, eps_dp, eps_z, dump=dump)
    voice.set_debug(True)
    audio, _ = voice.synthesize(ids, scales, eps_dp, eps_z)
    taps = {k: voice.tap(k) for k in ["x", "stats", "logw", "cum", "z_p", "z"] +
            [f"stage{i}" for i in range(len(orc.s.up_rates))]}
    voice.set_debug(False)
    w_ceil = np.diff(np.concatenate([[0], taps["cum"][0]]))
    assert np.array_equal(w_ceil, dump["w_ceil"].numpy()), "durations must match exactly (ceil cliff)"
    I = orc.s.inter
    assert np.abs(taps["x"] - dump["x"].numpy()).max() <= TOL
    assert np.abs(taps["stats"][:I] - dump["m_p"].numpy()).max() <= TOL
    assert np.abs(taps["stats"][I:] - dump["logs_p"].numpy()).max() <= TOL
    assert np.abs(taps["logw"][0] - dump["logw"].numpy()).max() <= TOL
    assert np.abs(taps["z_p"] - dump["z_p"].numpy()).max() <= TOL
    for k in ["z"] + [f"stage{i}" for i in range(len(orc.s.up_rates))]:
        e = np.abs(taps[k] - dump[k].numpy()).max()
        assert e <= 2e-3, (k, e)          # pre-tanh activations have O(1-10) magnitude; waveform bar below
    assert audio.shape == ref.shape
    assert np.abs(audio - ref).max() <= TOL
    assert float(np.sqrt((ref ** 2).mean())) > 0.05, "vacuous parity: oracle waveform is near silent"


def test_ragged_batch_is_b_independent_utterances():
    """Batch semantics (SURVEY.md App. A.9): every item equals its own B = 1 oracle run."""
    voice, orc = _pair("synthetic:tiny:1234")
    rng = np.random.default_rng(5)
    lens = [3, 131, 17, 64, 1, 40]
    ids_list = [rng.integers(0, 256, n) for n in lens]
    zs = 400
    eps_dp = [rng.standard_normal((2, n)).astype(np.float32) for n in lens]
    eps_z = rng.standard_normal((len(lens), orc.s.inter, zs)).astype(np.float32)
    scales = (0.667, 1.1, 0.8)
    outs, _ = voice.synthesize_batch(ids_list, scales, eps_dp, eps_z)
    for b, ids in enumerate(ids_list):
        ref = orc.infer(ids, scales, eps_dp[b], eps_z[b])
        assert outs[b].shape == ref.shape, (b, outs[b].shape, ref.shape)
        assert np.abs(outs[b] - ref).max() <= TOL, b
    # and the batch composition does not change an item beyond accumulation-order noise
    solo, _ = voice.synthesize(ids_list[1], scales, eps_dp[1], eps_z[1])
    assert np.abs(solo - outs[1]).max() <= 2e-4


def test_vocoder_only():
    for tag, B, frames in (("synthetic:tiny:1234", 3, 50), ("synthetic:medium:1234", 2, 64)):
        voice, orc = _pair(tag)
        import torch
        rng = np.random.default_rng(1236)
        z = rng.standard_normal((B, orc.s.inter, frames)).astype(np.float32)
        out, _ = voice.vocode(z)
        assert out.shape == (B, frames * orc.s.hop)
        for b in range(B):
            ref = orc.generator(torch.from_numpy(z[b])).numpy()
            assert np.abs(out[b] - ref).max() <= TOL


def test_int16_epilogue_matches_reference_loops():
    """pb200_synthesize_int16 against the oracle of piper.cpp:411-431 (oracle/int16_oracle.py, pinned to the reference's
    compiled loops and golden) and, when it travelled, against those compiled loops themselves."""
    from oracle import int16_oracle
    voice, _ = _pair("synthetic:tiny:1234")
    ids_list = [voicegen.benchmark_ids(10, seed=1), voicegen.benchmark_ids(25, seed=2), voicegen.benchmark_ids(1, seed=3)]
    f32, _ = voice.synthesize_batch(ids_list, seed=42)
    i16, _ = voice.synthesize_int16(ids_list, seed=42)
    for a, q in zip(f32, i16):
        assert q.dtype == np.int16 and q.shape == a.shape
        assert np.array_equal(q, int16_oracle.float_to_int16_cpp(a))
        if int16_oracle.ref_lib() is not None:
            assert np.array_equal(q, int16_oracle.float_to_int16_ref(a))
        assert np.abs(q).max() >= 32766                               # peak-normalised (truncating cast)


def test_seeded_noise_is_deterministic_and_seed_dependent():
    voice, _ = _pair("synthetic:tiny:1234")
    ids = voicegen.benchmark_ids(30, seed=9)
    a, _ = voice.synthesize(ids, seed=123)
    b, _ = voice.synthesize(ids, seed=123)
    c, _ = voice.synthesize(ids, seed=124)
    assert np.array_equal(a, b)
    assert a.shape != c.shape or not np.array_equal(a, c)
    d, _ = voice.synthesize(ids, (0.0, 1.0, 0.0), seed=1)
    e, _ = voice.synthesize(ids, (0.0, 1.0, 0.0), seed=2)
    assert np.array_equal(d, e), "zero noise scales make the graph deterministic"


def test_edge_cases_and_overrides():
    voice, orc = _pair("synthetic:tiny:1234")
    for ids in ([1, 0, 2], [5]):
        ref = orc.infer(ids, (0.0, 1.0, 0.0))
        out, _ = voice.synthesize(ids, (0.0, 1.0, 0.0))
        assert out.shape == ref.shape and np.abs(out - ref).max() <= TOL
    ids = [1, 0, 7, 0, 2]
    for ov in ([1, 2, 3, 0, 1], [0, 0, 0, 0, 0], [0, 0, 0, 0, 9]):
        ref = orc.infer(ids, (0.0, 1.0, 0.0), w_ceil_override=ov)
        outs, _ = voice.synthesize_batch([ids], (0.0, 1.0, 0.0), w_ceil_override=[ov])
        assert outs[0].shape == ref.shape == (max(sum(ov), 1) * 256,)
        assert np.abs(outs[0] - ref).max() <= TOL
    # longest fixture of the reference is 2423 ids (etc/test_sentences/test_ne.jsonl): exercise that length
    rng = np.random.default_rng(8)
    long_ids = rng.integers(0, 256, 2423)
    eps_dp, eps_z = _noise(orc.s.inter, len(long_ids), 3, cols=8000)
    ref = orc.infer(long_ids, (0.667, 1.0, 0.8), eps_dp, eps_z)
    out, _ = voice.synthesize(long_ids, (0.667, 1.0, 0.8), eps_dp, eps_z)
    assert out.shape == ref.shape and np.abs(out - ref).max() <= TOL


def test_errors_are_reported_not_swallowed():
    from piper_b200._lib import PiperB200Error
    voice, _ = _pair("synthetic:tiny:1234")
    with pytest.raises(PiperB200Error, match="symbol table"):
        voice.synthesize([1, 0, 999, 0, 2])
    with pytest.raises(PiperB200Error, match="symbol table"):
        voice.synthesize([1, -4, 2])
    with pytest.raises(PiperB200Error, match="empty"):
        voice.synthesize_batch([[1, 2], []])
    eps_dp, eps_z = _noise(32, 40, 1, cols=4)
    with pytest.raises(PiperB200Error, match="eps_z"):
        voice.synthesize(voicegen.benchmark_ids(18, seed=4)[:40], (0.667, 1.0, 0.8), eps_dp, eps_z)


def test_full_size_properties_medium_batch32():
    """BASELINE.json config 3 (medium, 32 x 128 phonemes) through size-independent properties."""
    voice, orc = _pair("synthetic:medium:1234")
    ids_list = [voicegen.benchmark_ids(128, seed=1234 + b) for b in range(32)]
    outs, sec = voice.synthesize_batch(ids_list, seed=7)
    again, _ = voice.synthesize_batch(ids_list, seed=7)
    hop = orc.s.hop
    for a, b2 in zip(outs, again):
        assert np.array_equal(a, b2), "run-to-run determinism"
        assert len(a) % hop == 0 and np.isfinite(a).all() and np.abs(a).max() <= 1.0
    frames = np.array([len(a) // hop for a in outs])
    assert 1.5 * 259 < frames.mean() < 2.6 * 259, frames.mean()      # ~2 frames per id (SURVEY.md §8d config 2)
    # durations are produced before the prior noise is drawn: length_scale 2 with the same seed doubles
    # every ceil(w) up to the ceil itself:  sum ceil(2w) in [2*sum ceil(w) - T, 2*sum ceil(w)]
    outs2, _ = voice.synthesize_batch(ids_list[:4], (0.667, 2.0, 0.8), seed=7)
    for a, b2 in zip(outs[:4], outs2):
        fa, fb = len(a) // hop, len(b2) // hop
        assert 2 * fa - 259 <= fb <= 2 * fa
    # an item's waveform does not depend on its batch mates
    solo, _ = voice.synthesize_batch([ids_list[5]], seed=7)
    # (seeded noise is keyed by batch slot, so compare slot 0 against slot 0)
    first, _ = voice.synthesize_batch(ids_list[5:6] + ids_list[:3], seed=7)
    assert solo[0].shape == first[0].shape and np.abs(solo[0] - first[0]).max() <= 2e-4   # tile shapes differ with B
    # items of the FULL batch against the oracle with explicit noise (the batch-32 launch takes the persistent
    # tensor-core kernels, which a B = 1 call does not)
    rng = np.random.default_rng(21)
    eps_dp = [rng.standard_normal((2, 259)).astype(np.float32) for _ in range(32)]
    eps_z = rng.standard_normal((32, orc.s.inter, 1400)).astype(np.float32)
    outs3, _ = voice.synthesize_batch(ids_list, (0.667, 1.0, 0.8), eps_dp, eps_z)
    for b in (0, 13, 31):
        ref = orc.infer(ids_list[b], (0.667, 1.0, 0.8), eps_dp[b], eps_z[b])
        assert outs3[b].shape == ref.shape and np.abs(outs3[b] - ref).max() <= TOL, b
    out, _ = voice.synthesize(ids_list[0], (0.667, 1.0, 0.8), eps_dp[0], eps_z[0])
    assert np.abs(out - outs3[0]).max() <= 2e-4


def test_attention_short_last_tiles_on_the_tail_kernel():
    """40 utterances of 131 .. 147 ids: one full 128-query tile + 3 .. 19 rows, and 40 x 2 heads x 2 tiles = 160 tiles > 148
    SMs, so last tiles of <= 16 rows go to the key-parallel CUDA-core kernel (encoder.cu: rel_attention_tail_kernel) and the
    longer ones stay on the tensor cores (attentions.py:225-272 either way); items of both kinds against the oracle, and the
    encoder output tap of the whole batch is finite."""
    voice, orc = _pair("synthetic:medium:1234")
    ids_list = [voicegen.benchmark_ids(64 + (i % 9), seed=50 + i) for i in range(40)]
    assert {len(i) for i in ids_list} == set(range(131, 148, 2))
    rng = np.random.default_rng(3)
    eps_dp = [rng.standard_normal((2, len(i))).astype(np.float32) for i in ids_list]
    eps_z = rng.standard_normal((40, orc.s.inter, 6 * 147)).astype(np.float32)
    outs, _ = voice.synthesize_batch(ids_list, (0.667, 1.0, 0.8), eps_dp, eps_z)
    for b in (0, 5, 8, 26, 39):                          # 131, 141, 147, 147, 137 ids: tails of 3, 13, 19, 19, 9 rows
        ref = orc.infer(ids_list[b], (0.667, 1.0, 0.8), eps_dp[b], eps_z[b])
        assert outs[b].shape == ref.shape and np.abs(outs[b] - ref).max() <= TOL, (b, len(ids_list[b]))


def test_high_ragged_batch8_matches_per_item_oracle():
    """BASELINE.json configs[3]'s per-GPU share: the "high" preset (ResBlock1, 512-channel generator,
    piper_train/__main__.py:72-82), 8 ragged utterances of up to 128 phonemes in ONE batch launch, every item against its own
    B = 1 oracle run (SURVEY App. A.9), stage taps of the longest item included."""
    voice, orc = _pair("synthetic:high:1234")
    n_ph = [128, 96, 128, 57, 120, 33, 128, 101]
    ids_list = [voicegen.benchmark_ids(n, seed=40 + i) for i, n in enumerate(n_ph)]
    rng = np.random.default_rng(31)
    eps_dp = [rng.standard_normal((2, len(i))).astype(np.float32) for i in ids_list]
    eps_z = rng.standard_normal((len(ids_list), orc.s.inter, 6 * 259)).astype(np.float32)
    scales = (0.667, 1.0, 0.8)
    voice.set_debug(True)
    outs, _ = voice.synthesize_batch(ids_list, scales, eps_dp, eps_z)
    keys = ["z"] + [f"stage{i}" for i in range(len(orc.s.up_rates))]
    taps = {(k, b): voice.tap(k, b) for k in keys for b in (0, 3)}
    voice.set_debug(False)
    for b, ids in enumerate(ids_list):
        dump = {}
        ref = orc.infer(ids, scales, eps_dp[b], eps_z[b], dump=dump)
        assert outs[b].shape == ref.shape, (b, outs[b].shape, ref.shape)
        assert np.abs(outs[b] - ref).max() <= TOL, (b, float(np.abs(outs[b] - ref).max()))
        assert float(np.sqrt((ref ** 2).mean())) > 0.05
        if b in (0, 3):
            for k in keys:
                r = dump[k].numpy()
                assert taps[(k, b)].shape == r.shape and np.abs(taps[(k, b)] - r).max() <= 2e-3, (b, k)


def test_streaming_encode_decode_split():
    """pb200_encode / pb200_decode + the host chunker against the reference-minted streaming fixture and the oracle."""
    from piper_b200 import streaming
    g = np.load(os.path.join(GOLDEN, "stream_tiny.npz"))
    voice, orc = _pair(str(g["voice"]))
    z_p = voice.encode(g["ids"], g["scales"], g["eps_dp"], g["eps_z"])
    assert z_p.shape == g["z_p"].shape and np.abs(z_p - g["z_p"]).max() <= TOL
    st = streaming.SpeechStreamer(voice, int(g["chunk_size"]), int(g["chunk_padding"]))
    pieces = list(st.chunk(z_p))
    assert [len(p) for p in pieces] == g["piece_lens"].tolist()
    assert np.abs(np.concatenate(pieces) - g["audio"]).max() <= TOL
    # decode of the whole latent == the un-chunked synthesis
    whole = voice.decode(z_p)[0]
    full, _ = voice.synthesize(g["ids"], g["scales"], g["eps_dp"], g["eps_z"])
    assert whole.shape == full.shape and np.abs(whole - full).max() <= 2e-4
    # seeded end-to-end stream: pieces concatenate to a plausible utterance, first piece arrives chunk-sized
    ids = voicegen.benchmark_ids(60, seed=8)
    out = list(st.stream(ids, seed=5))
    assert len(out) >= 2 and len(out[0]) == 45 * orc.s.hop and all(np.isfinite(p).all() for p in out)
    pcm = list(st.stream_int16_bytes(ids, seed=5))
    assert len(pcm) == len(out) and all(len(b) == 2 * len(p) for b, p in zip(pcm, out))


def test_cpp_shim_test_program(tmp_path):
    """The reference's only automated test (src/cpp/test.cpp) restated against the piper.hpp-compatible shim."""
    import subprocess
    from conftest import ROOT
    exe = os.path.join(ROOT, "piper_b200", "test_piper")
    voice = real_voice_path()
    if voice is None or not os.path.exists(exe):
        pytest.skip("shim test program or reference voice not staged")
    sentences = os.path.join(GOLDEN, "reference", "test_en-us.jsonl")
    out = str(tmp_path / "shim_test.wav")
    r = subprocess.run([exe, voice, sentences, out, "1"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    assert "OK" in r.stdout and os.path.getsize(out) >= 10000
    import wave
    with wave.open(out) as w:
        assert w.getframerate() == 16000 and w.getnchannels() == 1 and w.getsampwidth() == 2
        assert w.getnframes() % 256 == 0 and 100 * 256 <= w.getnframes() <= 250 * 256   # ~150-170 frames for this line


@pytest.mark.parametrize("tag,n_ph", [("synthetic:tiny-ms:1234", 30), ("synthetic:medium-ms:1234", 64)])
def test_multi_speaker_conditioning(tag, n_ph):
    """SURVEY §8f rank 4: sid -> emb_g -> dp.cond, WN cond_layer (per layer slice), dec.cond."""
    voice, orc = _pair(tag)
    assert voice.info.n_speakers == orc.s.n_speakers > 1 and voice.info.gin == orc.s.gin
    ids = voicegen.benchmark_ids(n_ph, seed=12)
    eps_dp, eps_z = _noise(orc.s.inter, len(ids), 5)
    scales = (0.667, 1.0, 0.8)
    outs = {}
    for sid in (0, orc.s.n_speakers - 1):
        ref = orc.infer(ids, scales, eps_dp, eps_z, sid=sid)
        out, _ = voice.synthesize(ids, scales, eps_dp, eps_z, sid=sid)
        assert out.shape == ref.shape and np.abs(out - ref).max() <= TOL, sid
        outs[sid] = out
    a, b = outs.values()
    assert a.shape != b.shape or np.abs(a - b).max() > 1e-2, "speakers must actually differ"
    # batch with one speaker per item (and the streaming decode half sees the speaker too)
    sids = [1, 0, orc.s.n_speakers - 1]
    voice.set_speakers(sids)
    zs = 6 * len(ids) + 16
    rng = np.random.default_rng(9)
    eps_z3 = rng.standard_normal((3, orc.s.inter, zs)).astype(np.float32)
    eps_dp3 = [rng.standard_normal((2, len(ids))).astype(np.float32) for _ in range(3)]
    batch, _ = voice.synthesize_batch([ids] * 3, scales, eps_dp3, eps_z3)
    for bi, sid in enumerate(sids):
        ref = orc.infer(ids, scales, eps_dp3[bi], eps_z3[bi], sid=sid)
        assert batch[bi].shape == ref.shape and np.abs(batch[bi] - ref).max() <= TOL, (bi, sid)
    voice.set_speakers([])
    # sid = None means speaker 0 (include/piper_b200.h), whatever an earlier call used
    last = orc.s.n_speakers - 1
    voice.synthesize(ids, scales, eps_dp, eps_z, sid=last)
    again, _ = voice.synthesize(ids, scales, eps_dp, eps_z, sid=None)
    assert again.shape == outs[0].shape and np.array_equal(again, outs[0])
    from piper_b200._lib import PiperB200Error
    with pytest.raises(PiperB200Error, match="speaker id"):
        voice.synthesize(ids, sid=orc.s.n_speakers)
