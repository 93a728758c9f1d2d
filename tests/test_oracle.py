"""CPU tests that pin the oracle against the golden fixtures minted from the reference's own source."""
import glob
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN, real_fixture_lines, real_voice_path
from piper_b200 import voicegen


def _oracle_for(tag):
    from oracle.voice_loader import load_voice
    from oracle.vits_oracle import Oracle
    if tag.startswith("real:"):
        path = real_voice_path()
        if path is None:
            pytest.skip("reference test voice not staged")
    else:
        _, arch, seed = tag.split(":")
        path = voicegen.cached_voice(arch, int(seed))
    spec, w, attrs = load_voice(path)
    return Oracle(spec, w, attrs), w


@pytest.mark.parametrize("name", sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN, "*.npz"))
                                        if not os.path.basename(p).startswith(("stream_", "int16_"))))
def test_oracle_matches_golden(name):
    g = np.load(os.path.join(GOLDEN, name + ".npz"))
    orc, w = _oracle_for(str(g["voice"]))
    from oracle.make_golden import weights_digest
    assert weights_digest(w) == str(g["weights_sha256"]), "voice weights differ from the ones the golden was minted on"
    dump = {}
    o = orc.infer(g["ids"], g["scales"], g["eps_dp"] if "eps_dp" in g else None,
                  g["eps_z"] if "eps_z" in g else None, dump=dump, sid=int(g["sid"]) if "sid" in g else None)
    assert np.array_equal(dump["w_ceil"].numpy().astype(np.int32), g["w_ceil"])   # durations: exact
    assert o.shape == g["audio"].shape
    assert np.abs(dump["z"].numpy() - g["z"]).max() <= 1e-3
    assert np.abs(o - g["audio"]).max() <= 1e-3       # north_star tolerance, fp32 waveform


def test_oracle_matches_survey_anchors():
    """Frame counts / waveform statistics of all 7 en-us fixtures on the real voice (SURVEY.md App. C)."""
    lines = real_fixture_lines()
    orc, _ = _oracle_for("real:test_voice")
    anchors = json.load(open(os.path.join(GOLDEN, "real_enus_anchors.json")))
    for a in anchors[1:4]:
        dump = {}
        o = orc.infer(lines[a["index"]]["phoneme_ids"], (0.0, 1.0, 0.0), dump=dump)
        assert len(o) == a["frames"] * 256
        assert dump["w_ceil"].numpy().astype(int).tolist() == a["w_ceil"]
        assert abs(float(np.abs(o).max()) - a["max_abs"]) < 1e-3
        assert abs(float(np.abs(o).mean()) - a["mean_abs"]) < 1e-4
        assert np.abs(o[:3] - np.asarray(a["first3"], np.float32)).max() < 1e-3


def _sampled_err(g, key, a):
    """max |a - reference| over the fixed sample of the reference's output stored under `key`."""
    a = np.asarray(a)
    assert a.shape == tuple(g[f"{key}.shape"]), (key, a.shape)
    return float(np.abs(a.reshape(-1)[g[f"{key}.idx"]] - g[f"{key}.val"]).max())


@pytest.mark.parametrize("tag,n_ph,scales", [("real:test_voice", 0, (0.667, 1.0, 0.8)),
                                             ("synthetic:tiny:1234", 40, (0.667, 1.3, 0.8)),
                                             ("synthetic:tiny-high:1234", 12, (0.3, 0.8, 1.0)),
                                             ("synthetic:tiny-ms:1234", 25, (0.667, 1.0, 0.8))])
def test_oracle_matches_reference_source(tag, n_ph, scales):
    """Against SynthesizerTrn.infer of the reference's own PyTorch source, run on the same inputs by
    `python -m oracle.make_golden reference-checks` (tests/golden/reference/source_cases.npz)."""
    from oracle.make_golden import weights_digest
    g = np.load(os.path.join(GOLDEN, "reference", "source_cases.npz"))
    orc, w = _oracle_for(tag)
    assert weights_digest(w) == str(g[f"{tag}.weights_sha256"]), "voice weights differ from the ones the golden was minted on"
    if tag.startswith("real:"):
        ids = real_fixture_lines()[3]["phoneme_ids"]
    else:
        ids = voicegen.benchmark_ids(n_ph, seed=17)
    assert np.array_equal(np.asarray(ids, np.int64), g[f"{tag}.ids"])
    rng = np.random.default_rng(11)
    eps_dp = rng.standard_normal((2, len(ids))).astype(np.float32)
    eps_z = rng.standard_normal((orc.s.inter, 6 * len(ids))).astype(np.float32)
    sid = 2 if orc.s.n_speakers > 1 else None             # multi-speaker: emb_g / dp.cond / WN cond_layer / dec.cond
    dump = {}
    o = orc.infer(ids, scales, eps_dp, eps_z, dump=dump, sid=sid)
    assert np.array_equal(dump["w_ceil"].numpy(), g[f"{tag}.w_ceil"])
    assert _sampled_err(g, f"{tag}.z_p", dump["z_p"].numpy()) < 1e-4
    assert _sampled_err(g, f"{tag}.z", dump["z"].numpy()) < 1e-3
    assert _sampled_err(g, f"{tag}.o", o) < 1e-3


def test_oracle_edge_cases():
    """Shortest legal input (BOS, PAD, EOS), single id, and a duration override."""
    orc, _ = _oracle_for("synthetic:tiny:1234")
    o = orc.infer([1, 0, 2], (0.667, 1.0, 0.8))
    assert len(o) % 256 == 0 and len(o) >= 256 and np.isfinite(o).all()
    o1 = orc.infer([5], (0.0, 1.0, 0.0))
    assert len(o1) >= 256
    o2 = orc.infer([1, 0, 7, 0, 2], (0.0, 1.0, 0.0), w_ceil_override=[1, 2, 3, 0, 1])
    assert len(o2) == 7 * 256
    # all-zero durations: clamp_min(sum, 1) gives exactly one frame (models.py:704)
    o3 = orc.infer([1, 0, 2], (0.0, 1.0, 0.0), w_ceil_override=[0, 0, 0])
    assert len(o3) == 256


def test_streaming_chunks_match_golden():
    """Chunk plan + oracle decoder against the fixture minted with the reference's own chunk loop."""
    from piper_b200 import streaming
    g = np.load(os.path.join(GOLDEN, "stream_tiny.npz"))
    orc, _ = _oracle_for(str(g["voice"]))
    z_p = orc.encode(g["ids"], g["scales"], g["eps_dp"], g["eps_z"])
    assert np.abs(z_p - g["z_p"]).max() <= 1e-4

    class _V:
        hop = orc.s.hop
    st = streaming.SpeechStreamer(_V(), int(g["chunk_size"]), int(g["chunk_padding"]), reference_quirks=True)
    pieces = list(st.chunk(z_p, decode=orc.decode))
    assert [len(p) for p in pieces] == g["piece_lens"].tolist()
    assert np.abs(np.concatenate(pieces) - g["audio"]).max() <= 1e-3
    # without the reference's stale right-trim the last chunk keeps its tail: total = frames * hop
    full = list(streaming.SpeechStreamer(_V(), 45, 10, reference_quirks=False).chunk(z_p, decode=orc.decode))
    assert sum(len(p) for p in full) == z_p.shape[1] * orc.s.hop


def test_chunk_plan_properties():
    from piper_b200.streaming import plan_chunks
    assert plan_chunks(65) == [(0, 65, 0, 0)]                       # too short to stream
    for n in (66, 90, 135, 136, 161, 500):
        plan = plan_chunks(n, 45, 10, reference_quirks=False)
        kept = sum((hi - lo) - tl - tr for lo, hi, tl, tr in plan)
        assert kept == n and plan[0][0] == 0 and plan[-1][1] == n
        assert all(hi - lo <= 45 + 20 for lo, hi, _, _ in plan)


def test_streaming_matches_reference_chunk_loop():
    """Against the reference's own SpeechStreamer.chunk loop driving its PyTorch decoder on the same latent
    (tests/golden/reference/stream_chunk_loop.npz)."""
    from oracle.make_golden import weights_digest
    from piper_b200 import streaming
    g = np.load(os.path.join(GOLDEN, "reference", "stream_chunk_loop.npz"))
    orc, w = _oracle_for("synthetic:tiny:1234")
    assert weights_digest(w) == str(g["weights_sha256"])
    ids = voicegen.benchmark_ids(70, seed=5)
    z_p = orc.encode(ids, (0.667, 1.0, 0.8))
    assert _sampled_err(g, "z_p", z_p) <= 1e-5, "the latent the reference chunked differs"

    class _V:
        hop = orc.s.hop
    mine = list(streaming.SpeechStreamer(_V(), 45, 10, True).chunk(z_p, decode=orc.decode))
    assert [len(a) for a in mine] == g["piece_lens"].tolist()
    assert _sampled_err(g, "audio", np.concatenate(mine)) <= 1e-4


# ---- int16 peak normalisation (piper.cpp:411-431 / python_run/piper/util.py:5-12): the oracle pinned three ways

def _int16_golden():
    g = np.load(os.path.join(GOLDEN, "int16_cpp.npz"))
    return {k[:-3]: (g[k], g[k[:-3] + ".cpp"], g[k[:-3] + ".py"]) for k in g.files if k.endswith(".in")}


def test_int16_oracle_matches_reference_minted_golden():
    """tests/golden/int16_cpp.npz holds the outputs of the reference's own loops (compiled from piper.cpp:411-431)."""
    from oracle import int16_oracle
    from piper_b200 import host
    cases = _int16_golden()
    assert len(cases) >= 10
    for name, (a, cpp, py) in cases.items():
        assert np.array_equal(int16_oracle.float_to_int16_cpp(a), cpp), name
        assert np.array_equal(int16_oracle.float_to_int16_python(a), py), name
        assert np.array_equal(host.audio_float_to_int16(a), cpp), name            # the shim's Python mirror
        assert np.array_equal(host.audio_float_to_int16(a, "python"), py), name


def _int16_seeded(tag, seed, spec):
    from oracle.make_golden_int16 import seeded_cases
    g = np.load(os.path.join(GOLDEN, "reference", "int16_seeded.npz"))
    return [(a, g[f"{tag}{i}.idx"], g[f"{tag}{i}.val"]) for i, a in enumerate(seeded_cases(seed, spec))]


def test_int16_oracle_matches_compiled_reference_loops():
    """The reference's lines piper.cpp:411-431 compiled by oracle/build_ref.py, run on seeded inputs by
    oracle/make_golden_int16.py (tests/golden/reference/int16_seeded.npz)."""
    from oracle import int16_oracle
    from oracle.make_golden_int16 import CPP_SEEDED
    for a, idx, cpp in _int16_seeded("cpp", *CPP_SEEDED):
        assert np.array_equal(int16_oracle.float_to_int16_cpp(a)[idx], cpp), a.size


def test_int16_oracle_matches_reference_python_util():
    """python_run/piper/util.py:5-12 of the reference, run on seeded inputs by oracle/make_golden_int16.py."""
    from oracle import int16_oracle
    from oracle.make_golden_int16 import PY_SEEDED
    for a, idx, py in _int16_seeded("py", *PY_SEEDED):
        assert np.array_equal(int16_oracle.float_to_int16_python(a)[idx], py), a.size
