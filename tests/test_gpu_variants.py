"""GPU tests of the kernel variants behind the environment switches.  The defaults (persistent tensor-core conv kernel
for every dense layer, fp16x3 operands, tensor-map TMA, CUDA graphs, fused MRF stage, tensor-core attention) are what every
other GPU test runs; here the documented alternatives and fallbacks are kept honest: the other split precisions, the
per-row copies, the layer-wise MRF stage, the CUDA-core attention that takes the shapes the tensor-core attention
declines, programmatic dependent launch, both LayerNorm CTA widths, and graph replay against direct launches.
"""
import os

import numpy as np
import pytest

from piper_b200 import voicegen

pytestmark = pytest.mark.gpu
SCALES = (0.667, 1.0, 0.8)


def _noise(inter, n_ids, seed):
    rng = np.random.default_rng(seed)
    return rng.standard_normal((2, n_ids)).astype(np.float32), rng.standard_normal((inter, 6 * n_ids + 16)).astype(np.float32)


@pytest.mark.parametrize("arch,n_ph", [("tiny", 20), ("tiny-high", 20), ("medium", 64), ("high", 32)])
def test_fused_mrf_stage_matches_layerwise_and_oracle(arch, n_ph):
    """Engine mask bit 16 routes the 32-channel MRF stage through mrf_fused.cu: same taps as the layer-wise path (both
    are bf16x3) and the same waveform bar against the oracle."""
    from oracle.voice_loader import load_voice
    from oracle.vits_oracle import Oracle
    from piper_b200 import engine
    path = voicegen.cached_voice(arch)
    spec, w, attrs = load_voice(path)
    orc = Oracle(spec, w, attrs)
    ids = voicegen.benchmark_ids(n_ph, seed=3)
    eps_dp, eps_z = _noise(spec.inter, len(ids), 77)
    dump = {}
    ref = orc.infer(ids, SCALES, eps_dp, eps_z, dump=dump)
    v = engine.Voice(path, 0)
    try:
        stages = [i for i in range(len(spec.up_rates)) if dump[f"stage{i}"].shape[0] == 32]
        assert stages, "no 32-channel stage in this architecture"
        out = {}
        for mask in (15, 31):
            v.set_mma(mask)
            v.set_debug(True)
            audio, _ = v.synthesize(ids, SCALES, eps_dp, eps_z)
            out[mask] = (audio.copy(), {i: v.tap(f"stage{i}") for i in stages})
            v.set_debug(False)
        for i in stages:
            r = dump[f"stage{i}"].numpy()
            e_layer = np.abs(out[15][1][i] - r).max()
            e_fused = np.abs(out[31][1][i] - r).max()
            assert e_fused <= max(2e-4 * max(1.0, np.abs(r).max()), 2 * e_layer), (i, e_layer, e_fused)
        assert np.abs(out[31][0] - ref).max() <= 1e-3
        # taps off: the last stage runs with conv_post + tanh fused behind it (no stage output in HBM)
        v.set_mma(31)
        audio_tail, _ = v.synthesize(ids, SCALES, eps_dp, eps_z)
        assert audio_tail.shape == ref.shape and np.abs(audio_tail - ref).max() <= 1e-3
    finally:
        v.close()


def test_fused_mrf_ragged_batch():
    """Ragged batch through the fused stage: each item equals its own batch-1 run (utterance-edge zero padding)."""
    from piper_b200 import engine
    v = engine.Voice(voicegen.cached_voice("medium"), 0)
    try:
        v.set_mma(31)
        ids = [voicegen.benchmark_ids(n, seed=10 + n) for n in (5, 64, 23, 128, 1)]
        wavs, _ = v.synthesize_batch(ids, SCALES, seed=99)
        v.set_mma(15)
        wavs0, _ = v.synthesize_batch(ids, SCALES, seed=99)
        assert [len(a) for a in wavs] == [len(a) for a in wavs0]
        for a, b in zip(wavs, wavs0):
            assert np.abs(a - b).max() <= 2e-4
    finally:
        v.close()


_CHILD = r"""
import json, os, sys, tempfile
import numpy as np
sys.path.insert(0, {root!r})
from oracle.voice_loader import load_voice
from oracle.vits_oracle import Oracle
from piper_b200 import engine, voicegen
out = {{}}
for arch, n_ph, batch in (("tiny", 20, 1), ("medium", 64, 1), ("medium", 128, 32)):
    path = voicegen.cached_voice(arch)
    spec, w, attrs = load_voice(path)
    v = engine.Voice(path, 0)
    ids = [voicegen.benchmark_ids(n_ph, seed=3 + b) for b in range(batch)]
    rng = np.random.default_rng(77)
    eps_dp = [rng.standard_normal((2, len(i))).astype(np.float32) for i in ids]
    eps_z = [rng.standard_normal((spec.inter, 6 * len(i) + 16)).astype(np.float32) for i in ids]
    wavs, _ = v.synthesize_batch(ids, (0.667, 1.0, 0.8), eps_dp=eps_dp, eps_z=np.stack(eps_z))
    worst = 0.0
    for b in sorted(set([0, batch - 1])):
        # the oracle's answer is the same for every variant (cached per user: the temporary directory may be shared)
        cache = os.path.join(tempfile.gettempdir(), f"piper_b200_exp_ref-{{os.getuid()}}_{{arch}}_{{n_ph}}_{{batch}}_{{b}}.npy")
        if os.path.exists(cache):
            ref = np.load(cache)
        else:
            ref = Oracle(spec, w, attrs).infer(ids[b], (0.667, 1.0, 0.8), eps_dp[b], eps_z[b])
            np.save(cache + f".{{os.getpid()}}.npy", ref); os.replace(cache + f".{{os.getpid()}}.npy", cache)
        got = wavs[b]
        assert got.shape == ref.shape, (got.shape, ref.shape)
        worst = max(worst, float(np.abs(got - ref).max()))
    out[f"{{arch}}/{{batch}}"] = worst
    v.close()
print("RESULT " + json.dumps(out))
"""


@pytest.mark.parametrize("env", [{"PIPER_B200_ATT3": "0"},                                # CUDA-core attention for every shape
                                 {"PIPER_B200_PDL": "1"},                                 # programmatic dependent launch
                                 {"PIPER_B200_LN_WARPS": "24"},                           # 24-warp LayerNorm CTAs at every batch size
                                 {"PIPER_B200_V2_PREC": "std"},                           # bf16x3 generator, tf32x3 elsewhere
                                 {"PIPER_B200_V2_TM": "0"},                               # one bulk copy per channel row
                                 {"PIPER_B200_V2_MMA3": "1"},                             # three instructions per k-step
                                 {"PIPER_B200_GRAPH": "0"},
                                 {"PIPER_B200_FLAT": "0"},                                # [item][channel][pitch] activations, per-item tiles
                                 {"PIPER_B200_V2_ASTAT": "0", "PIPER_B200_ATT_TAIL": "0"},   # streaming operand ring for every layer; every query tile on the tensor cores
                                 {"PIPER_B200_ATT_TM": "0", "PIPER_B200_V2_CHAIN_K": "0"},   # per-row TMA in attention; two K-chains everywhere
                                 {"PIPER_B200_LN_WARPS": "8"},                            # 8-warp LayerNorm CTAs at every batch size
                                 {"PIPER_B200_MMA": "15"},                                # layer-wise MRF stage
                                 {"PIPER_B200_V2_PREC": "std", "PIPER_B200_V2_TM": "0", "PIPER_B200_GRAPH": "0", "PIPER_B200_MMA": "15"}])
def test_env_gated_variants_keep_parity(env):
    """Every non-default path keeps the 1e-3 waveform bar (the switches are read once per process, so each runs in a
    child process)."""
    import json, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    e = dict(os.environ, **env)
    r = subprocess.run([sys.executable, "-c", _CHILD.format(root=root)], capture_output=True, text=True, env=e, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("RESULT ")][-1]
    for k, err in json.loads(line[7:]).items():
        assert err <= 1e-3, (env, k, err)


_GRAPH_CHILD = r"""
import json, os, sys
import numpy as np
sys.path.insert(0, {root!r})
from piper_b200 import engine, voicegen
res = {{}}
for arch, n_ph, batch in (("tiny", 20, 3), ("medium", 128, 1), ("medium", 128, 32)):
    path = voicegen.cached_voice(arch)
    ids = [voicegen.benchmark_ids(n_ph - (b % 3), seed=3 + b) for b in range(batch)]
    outs = {{}}
    for mode in ("0", "1"):
        os.environ["PIPER_B200_GRAPH"] = mode
        v = engine.Voice(path, 0)
        runs = []
        # warm (direct), capture, replay, replay with another seed / length scale, and back
        for seed, ls in ((7, 1.0), (7, 1.0), (7, 1.0), (8, 1.0), (7, 1.3), (7, 1.0)):
            wavs, _ = v.synthesize_batch(ids, (0.667, ls, 0.8), seed=seed)
            runs.append(wavs)
        i16, _ = v.synthesize_int16(ids, (0.667, 1.0, 0.8), seed=7)
        outs[mode] = (runs, i16, engine.launch_count())
        v.close()
    g, d = outs["1"][0], outs["0"][0]
    worst = 0.0
    for r in range(len(g)):
        assert [len(a) for a in g[r]] == [len(a) for a in d[r]], (arch, batch, r)
        worst = max(worst, max(float(np.abs(a - b).max()) for a, b in zip(g[r], d[r])))
    # replays are deterministic, and per-call scalars are honoured by a replayed graph
    assert all(np.array_equal(a, b) for a, b in zip(g[1], g[2])) and all(np.array_equal(a, b) for a, b in zip(g[2], g[5]))
    assert any(not np.array_equal(a, b) for a, b in zip(g[2], g[3])), "seed ignored by the replayed graph"
    assert [len(a) for a in g[4]] != [len(a) for a in g[2]], "length_scale ignored by the replayed graph"
    assert all(np.array_equal(a, b) for a, b in zip(outs["1"][1], outs["0"][1])) or worst > 0
    res[f"{{arch}}/{{batch}}"] = worst
print("RESULT " + json.dumps(res))
"""


def test_cuda_graph_replay_matches_direct_launches():
    """PIPER_B200_GRAPH=1: the captured front / back graphs (shape buckets, per-call scalars in device memory) give the
    waveforms of the direct launch sequence."""
    import json, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", _GRAPH_CHILD.format(root=root)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("RESULT ")][-1]
    for k, err in json.loads(line[7:]).items():
        assert err <= 2e-4, (k, err)
