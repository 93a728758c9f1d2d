"""Mint the golden fixtures under tests/golden/ from the REFERENCE's own PyTorch model source.

Run in the build container only (needs /root/reference):  python -m oracle.make_golden
(`python -m oracle.make_golden reference-checks` mints tests/golden/reference/ only.)
Each fixture stores the inputs (phoneme ids, scales, injected noise) and the outputs of
`SynthesizerTrn.infer` (/root/reference/src/python/piper_train/vits/models.py:681-722) run on
CPU fp32 through oracle/ref_bridge.py: per-id frame counts, the latent z and the waveform.
The GPU box has no /root/reference; there these files are what pins the oracle (and the engine)
to the reference.
"""
from __future__ import annotations

import hashlib
import json
import os

import numpy as np

from oracle import ref_bridge
from oracle.voice_loader import load_voice
from piper_b200 import voicegen

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "tests", "golden")
REAL = "/root/reference/etc/test_voice.onnx"
FIXTURES = "/root/reference/etc/test_sentences/test_en-us.jsonl"


def weights_digest(w) -> str:
    h = hashlib.sha256()
    for k in sorted(w):
        h.update(k.encode())
        h.update(np.ascontiguousarray(w[k]).tobytes())
    return h.hexdigest()


def mint(name, voice_path, voice_tag, ids, scales, seed, sid=None):
    spec, w, _ = load_voice(voice_path)
    net = ref_bridge.build_reference_model(spec, w)
    ids = np.asarray(ids, np.int64)
    eps_dp = eps_z = None
    if seed is not None:
        rng = np.random.default_rng(seed)
        eps_dp = rng.standard_normal((2, len(ids))).astype(np.float32)
        eps_z = rng.standard_normal((spec.inter, 3 * len(ids))).astype(np.float32)
    r = ref_bridge.reference_infer(net, ids, scales, eps_dp, eps_z, sid=sid)
    if eps_z is not None:
        assert r["y_len"] <= eps_z.shape[1]
        eps_z = eps_z[:, : r["y_len"]].copy()
    out = dict(ids=ids, scales=np.asarray(scales, np.float32), w_ceil=r["w_ceil"].astype(np.int32),
               z=r["z"].astype(np.float32), audio=r["o"].astype(np.float32),
               voice=np.array(voice_tag), weights_sha256=np.array(weights_digest(w)))
    if eps_dp is not None:
        out.update(eps_dp=eps_dp, eps_z=eps_z)
    if sid is not None:
        out.update(sid=np.int64(sid))
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)
    print(f"{name}: ids={len(ids)} frames={r['y_len']} max|o|={np.abs(r['o']).max():.6f} "
          f"mean|o|={np.abs(r['o']).mean():.6f} o[0:3]={r['o'][:3]}")


def main():
    assert ref_bridge.available(), "needs /root/reference"
    os.makedirs(OUT, exist_ok=True)
    lines = [json.loads(l) for l in open(FIXTURES)]
    # real weights (x-low test voice), deterministic scales: SURVEY.md App. C anchors
    mint("real_enus1_det", REAL, "real:test_voice", lines[1]["phoneme_ids"], (0.0, 1.0, 0.0), None)
    mint("real_enus4_noise", REAL, "real:test_voice", lines[4]["phoneme_ids"], (0.667, 1.0, 0.8), 1235)
    # all 7 en-us lines: frame counts + waveform statistics only (small)
    spec, w, _ = load_voice(REAL)
    net = ref_bridge.build_reference_model(spec, w)
    anchors = []
    for i, l in enumerate(lines):
        r = ref_bridge.reference_infer(net, l["phoneme_ids"], (0.0, 1.0, 0.0))
        anchors.append(dict(index=i, n_ids=len(l["phoneme_ids"]), frames=r["y_len"],
                            max_abs=float(np.abs(r["o"]).max()), mean_abs=float(np.abs(r["o"]).mean()),
                            first3=[float(v) for v in r["o"][:3]], w_ceil=[int(v) for v in r["w_ceil"]]))
    with open(os.path.join(OUT, "real_enus_anchors.json"), "w") as f:
        json.dump(anchors, f)
    # synthetic voices (regenerated from their seed wherever the tests run)
    for arch, n_ph in (("tiny", 32), ("tiny-high", 32), ("medium", 24), ("high", 16)):
        path = voicegen.cached_voice(arch)
        mint(f"synthetic_{arch}", path, f"synthetic:{arch}:1234", voicegen.benchmark_ids(n_ph, seed=99),
             (0.667, 1.0, 0.8), 4321)
    mint("synthetic_tiny-ms_sid3", voicegen.cached_voice("tiny-ms"), "synthetic:tiny-ms:1234",
         voicegen.benchmark_ids(32, seed=99), (0.667, 1.0, 0.8), 4321, sid=3)
    mint_streaming()


def mint_streaming():
    """Chunked streaming golden: the reference's own chunk loop (infer_onnx_streaming.py:76-108) driving the
    reference PyTorch decoder on the reference encoder's z_p."""
    from oracle.vits_oracle import Oracle
    path = voicegen.cached_voice("tiny")
    spec, w, attrs = load_voice(path)
    net = ref_bridge.build_reference_model(spec, w)
    ids = voicegen.benchmark_ids(40, seed=2)
    rng = np.random.default_rng(3)
    eps_dp = rng.standard_normal((2, len(ids))).astype(np.float32)
    eps_z = rng.standard_normal((spec.inter, 6 * len(ids))).astype(np.float32)
    r = ref_bridge.reference_infer(net, ids, (0.667, 1.0, 0.8), eps_dp, eps_z)
    pieces = ref_bridge.reference_stream_chunks(net, r["z_p"], r["y_len"])
    np.savez_compressed(os.path.join(OUT, "stream_tiny.npz"), ids=ids, scales=np.asarray((0.667, 1.0, 0.8), np.float32),
                        eps_dp=eps_dp, eps_z=eps_z[:, : r["y_len"]].copy(), z_p=r["z_p"].astype(np.float32),
                        piece_lens=np.asarray([len(p) for p in pieces], np.int64),
                        audio=np.concatenate(pieces).astype(np.float32), chunk_size=np.int64(45),
                        chunk_padding=np.int64(10), voice=np.array("synthetic:tiny:1234"),
                        weights_sha256=np.array(weights_digest(w)))
    print("stream_tiny:", r["y_len"], "frames ->", [len(p) for p in pieces])


# The cases tests/test_oracle.py compares with the reference source (voice tag, phonemes, scales); their outputs are stored
# under tests/golden/reference/ so that the comparison runs without the reference tree.
SOURCE_CASES = [("real:test_voice", 0, (0.667, 1.0, 0.8)), ("synthetic:tiny:1234", 40, (0.667, 1.3, 0.8)),
                ("synthetic:tiny-high:1234", 12, (0.3, 0.8, 1.0)), ("synthetic:tiny-ms:1234", 25, (0.667, 1.0, 0.8))]
REF_OUT = os.path.join(OUT, "reference")
SAMPLES = 1024


def sample(out, key, a, seed):
    """Store the shape of `a` and a fixed seeded sample of its elements (flat indices and values) under `key`."""
    a = np.asarray(a, np.float32)
    idx = np.sort(np.random.default_rng(seed).choice(a.size, min(a.size, SAMPLES), replace=False)).astype(np.int32)
    out.update({f"{key}.shape": np.asarray(a.shape, np.int64), f"{key}.idx": idx, f"{key}.val": a.reshape(-1)[idx]})


def mint_reference_checks():
    """Outputs of the reference's own model source and streaming chunk loop for the inputs the tests draw, plus the
    test voice's config and its pre-phonemized en-us sentences (small text fixtures)."""
    import shutil
    from oracle.vits_oracle import Oracle
    assert ref_bridge.available(), "needs the reference source tree"
    os.makedirs(REF_OUT, exist_ok=True)
    shutil.copyfile(REAL + ".json", os.path.join(REF_OUT, "test_voice.onnx.json"))
    shutil.copyfile(FIXTURES, os.path.join(REF_OUT, "test_en-us.jsonl"))
    lines = [json.loads(l) for l in open(FIXTURES)]
    out = {}
    for i, (tag, n_ph, scales) in enumerate(SOURCE_CASES):
        path = REAL if tag.startswith("real:") else voicegen.cached_voice(tag.split(":")[1], int(tag.split(":")[2]))
        spec, w, _ = load_voice(path)
        net = ref_bridge.build_reference_model(spec, w)
        ids = lines[3]["phoneme_ids"] if tag.startswith("real:") else voicegen.benchmark_ids(n_ph, seed=17)
        rng = np.random.default_rng(11)
        eps_dp = rng.standard_normal((2, len(ids))).astype(np.float32)
        eps_z = rng.standard_normal((spec.inter, 6 * len(ids))).astype(np.float32)
        sid = 2 if spec.n_speakers > 1 else None
        r = ref_bridge.reference_infer(net, ids, scales, eps_dp, eps_z, sid=sid)
        out[f"{tag}.ids"] = np.asarray(ids, np.int64)
        out[f"{tag}.w_ceil"] = r["w_ceil"].astype(np.int32)
        out[f"{tag}.weights_sha256"] = np.array(weights_digest(w))
        for j, k in enumerate(("z_p", "z", "o")):
            sample(out, f"{tag}.{k}", r[k], 100 * i + j)
        print(f"{tag}: ids={len(ids)} frames={r['y_len']}")
    np.savez_compressed(os.path.join(REF_OUT, "source_cases.npz"), **out)

    # SpeechStreamer.chunk of the reference on the oracle's latent (tests/test_oracle.py draws the same input)
    path = voicegen.cached_voice("tiny")
    spec, w, attrs = load_voice(path)
    orc = Oracle(spec, w, attrs)
    net = ref_bridge.build_reference_model(spec, w)
    z_p = orc.encode(voicegen.benchmark_ids(70, seed=5), (0.667, 1.0, 0.8))
    pieces = ref_bridge.reference_stream_chunks(net, z_p, z_p.shape[1], 45, 10)
    out = dict(piece_lens=np.asarray([len(p) for p in pieces], np.int64), weights_sha256=np.array(weights_digest(w)))
    sample(out, "z_p", z_p, 1000)
    sample(out, "audio", np.concatenate(pieces), 1001)
    np.savez_compressed(os.path.join(REF_OUT, "stream_chunk_loop.npz"), **out)
    print("stream_chunk_loop:", [len(p) for p in pieces])


if __name__ == "__main__":
    import sys
    if sys.argv[1:] == ["reference-checks"]:
        mint_reference_checks()
    else:
        main()
