"""Every fused epilogue of both conv kernels on the GPU, launch by launch, against a float64 reference of the same op, and
the whole engine with its convolutions on the fp32 CUDA-core kernel against the CPU oracle.

Kernel level (engine.debug_conv): the CUDA-core kernel (back end 0, conv1d.cu) and the tensor-core kernel (conv_mma2.cu:
1 = bf16x3, 2 = tf32x3 with 2 K-chains, 5 = fp16x3, 6 = fp16x3 with 2 K-chains) on layer shapes the medium, high and tiny
presets launch.  Inputs are ragged batches with stale data (x40) past each item's length; y and y2 start from a sentinel
(or, in place, from the residual), and every element outside an item's valid output range must still hold it bit for bit,
gaps between items of the flat [channel][item][slot] layout included.

Engine level (Voice.set_mma): mask 0 puts every conv on the CUDA-core kernel, 16 keeps only the fused MRF stage, and 1, 2,
4, 8 move one family at a time to the tensor cores; waveform, stage taps and durations against the oracle with the bars of
test_gpu_parity.test_stage_by_stage_parity."""
import numpy as np
import pytest

from conftest import real_fixture_lines, real_voice_path
from piper_b200 import voicegen

pytestmark = pytest.mark.gpu

BACKENDS = [0, 1, 2, 5, 6]
SENTINEL = np.float32(7.25e7)
LENS = (1, 3, 130, 259)              # below one float4, not a multiple of 4, ragged tile ends


def _tol(backend):
    # the bars of test_gpu_conv_kernels: fp32 FFMA accumulation order / split-precision tensor-core products, relative to
    # max(1, |reference|)
    return 1e-4 if backend == 0 else 3e-4


def _ragged(ci, lens, seed, pitch=None):
    """x [B][ci][pitch]: N(0, 1) inside each item, stale data x40 past it; also the valid parts in float64."""
    rng = np.random.default_rng(seed)
    pitch = pitch or ((max(lens) + 3) & ~3) + 4          # the engine's slot: 16-byte rows plus a gap
    x = (rng.standard_normal((len(lens), ci, pitch)) * 40).astype(np.float32)
    for b, L in enumerate(lens):
        x[b, :, :L] = rng.standard_normal((ci, L)).astype(np.float32)
    return x, [x[b, :, :L].astype(np.float64) for b, L in enumerate(lens)]


def _weights(rows, ci, k, seed, bias_scale=1.0):
    rng = np.random.default_rng(seed + 1)
    w = (rng.standard_normal((rows, ci, k)) / np.sqrt(ci * k)).astype(np.float32)
    return w, (rng.standard_normal(rows) * bias_scale).astype(np.float32)


def _conv(xb, w, bias, dil, pad, slope):
    """float64 F.conv1d of one item (the un-lowered op), pre-activation included: [rows][L]."""
    import torch
    import torch.nn.functional as F
    xt = torch.from_numpy(xb)
    if slope is not None:
        xt = F.leaky_relu(xt, slope)
    b = None if bias is None else torch.from_numpy(bias.astype(np.float64))
    return F.conv1d(xt[None], torch.from_numpy(w.astype(np.float64)), b, dilation=dil, padding=pad)[0].numpy()


def _sigmoid(v):
    return 1.0 / (1.0 + np.exp(-v))


def _flat(a):
    """[B][C][pitch] <-> [C][B][pitch] (its own inverse)."""
    return None if a is None else np.ascontiguousarray(a.transpose(1, 0, 2))


def _launch(backend, x, w, lens, flat=False, y=None, y2=None, r=None, **kw):
    """engine.debug_conv on item-major host arrays; with flat=True the launch sees them in the flat layout."""
    from piper_b200 import engine
    f = _flat if flat else (lambda a: a)
    yo, y2o = engine.debug_conv(backend, f(x), w, lens, y=f(y), y2=f(y2), r=f(r), flat=flat, **kw)
    return f(yo), f(y2o)


def _check(got, init, want, valid, tol, what):
    """got / init [B][C][pitch]; want[b] = float64 reference of got[b, :C_b, :valid[b]].  Returns the error relative to
    max(1, |want|); asserts the bar, and that every element outside the valid ranges still holds `init` bit for bit."""
    inside = np.zeros(got.shape, bool)
    worst = 0.0
    for b, (wb, L) in enumerate(zip(want, valid)):
        assert wb.shape[1] == L, (what, b, wb.shape, L)
        inside[b, :wb.shape[0], :L] = True
        if L:
            err = float(np.abs(got[b, :wb.shape[0], :L] - wb).max()) / max(1.0, float(np.abs(wb).max()))
            assert err <= tol, (what, b, err)
            worst = max(worst, err)
    outside = ~inside
    bad = np.flatnonzero(got.view(np.uint32)[outside] != init.view(np.uint32)[outside])
    assert bad.size == 0, (what, "stored outside the valid range", bad.size, np.argwhere(outside)[bad[:4]].tolist())
    return worst


def _report(epi, backend, flat, err):
    print(f"\nEPILOGUE_ERR {epi} backend={backend} flat={int(flat)} err={err:.3e} bar={_tol(backend):.0e}")


# ---------------------------------------------------------------------------------------------------------------------
# plain epilogues: BIAS (+ per-item bias), RELU, RES, GATE (ci, rows, k, dil, epi, bias_item, flat)
PLAIN = [
    (192, 256, 7, 1, "BIAS", True, True),        # medium dec.pre + speaker conditioning
    (192, 512, 7, 1, "BIAS", True, False),       # high dec.pre
    (192, 192, 1, 1, "BIAS", True, True),        # duration predictor pre (+ dp.cond)
    (192, 768, 3, 1, "RELU", False, True),       # FFN first conv
    (768, 192, 3, 1, "RES", False, True),        # FFN second conv: 768-deep reduction
    (192, 192, 1, 1, "RES", False, True),        # attention output projection
    (192, 384, 5, 1, "GATE", False, True),       # flow WN in_layer
    (192, 384, 5, 1, "GATE", True, True),        # flow WN in_layer + cond_layer slice (multi-speaker)
    (32, 64, 5, 1, "GATE", True, True),          # tiny preset in_layer
]


@pytest.mark.parametrize("case", PLAIN, ids=lambda c: f"{c[4]}-{c[0]}x{c[1]}k{c[2]}" + ("-item" if c[5] else ""))
@pytest.mark.parametrize("backend", BACKENDS)
def test_plain_epilogues(lib_built, backend, case):
    ci, rows, k, dil, epi, with_item, flat_too = case
    lens = LENS
    B = len(lens)
    x, clean = _ragged(ci, lens, seed=ci + rows + k)
    w, bias = _weights(rows, ci, k, seed=rows)
    rng = np.random.default_rng(3)
    bias_item = (rng.standard_normal((B, rows + 16)) * 0.5).astype(np.float32) if with_item else None   # stride > rows
    C_y = rows // 2 if epi == "GATE" else rows
    r = rng.standard_normal((B, C_y, x.shape[2])).astype(np.float32) if epi == "RES" else None
    pad = dil * (k - 1) // 2
    want = []
    for b, L in enumerate(lens):
        v = _conv(clean[b], w, bias, dil, pad, None)
        if with_item:
            v = v + bias_item[b, :rows, None].astype(np.float64)
        if epi == "RELU":
            v = np.maximum(v, 0.0)
        elif epi == "RES":
            v = v + r[b, :, :L]
        elif epi == "GATE":
            v = np.tanh(v[0::2]) * _sigmoid(v[1::2])
        want.append(v)
    y0 = np.full((B, C_y, x.shape[2]), SENTINEL, np.float32)
    runs = {}
    for flat in (False, True) if flat_too else (False,):
        y, _ = _launch(backend, x, w, lens, flat=flat, epi=epi, bias=bias, bias_item=bias_item, dil=dil, y=y0, r=r)
        _report(epi + ("+item" if with_item else ""), backend, flat, _check(y, y0, want, lens, _tol(backend), (epi, flat)))
        runs[flat] = y
    if flat_too:                                         # flat launch == item-major launch, within the same bar
        for b, L in enumerate(lens):
            d = np.abs(runs[True][b, :, :L] - runs[False][b, :, :L]).max() if L else 0.0
            assert d <= _tol(backend) * max(1.0, float(np.abs(want[b]).max())), (b, d)


# ---------------------------------------------------------------------------------------------------------------------
# WaveNet res_skip (in place on the residual stream, skip sum into y2) and the coupling subtract, as engine.cu run_flow
@pytest.mark.parametrize("flat", [False, True])
@pytest.mark.parametrize("backend", BACKENDS)
def test_wn_res_skip_and_coupling_subtract_in_place(lib_built, backend, flat):
    H, half = 192, 96
    lens = LENS
    B = len(lens)
    acts, clean = _ragged(H, lens, seed=41)
    pitch = acts.shape[2]
    rng = np.random.default_rng(42)
    fh = rng.standard_normal((B, H, pitch)).astype(np.float32)           # the residual stream, updated in place
    skip = np.full((B, H, pitch), SENTINEL, np.float32)                  # the skip sum: first layer overwrites
    tol = _tol(backend)
    worst = 0.0
    # layer 0 (first = 1), layer 1 (first = 0: accumulates into the skip sum layer 0 left), last layer (split 0: skip only)
    for i, (rows, split, first) in enumerate(((2 * H, H, 1), (2 * H, H, 0), (H, 0, 0))):
        w, bias = _weights(rows, H, 1, seed=50 + i, bias_scale=0.1)
        v = [_conv(clean[b], w, bias, 1, 0, None) for b in range(B)]
        y_want = [fh[b, :, :L].astype(np.float64) + v[b][:split] for b, L in enumerate(lens)] if split else None
        s_want = [(0.0 if first else skip[b, :, :L].astype(np.float64)) + v[b][split:] for b, L in enumerate(lens)]
        fh_new, skip_new = _launch(backend, acts, w, lens, flat=flat, epi="WN", bias=bias, y=fh, y2=skip, y_is_r=True,
                                   split=split, first=first)
        if split:
            worst = max(worst, _check(fh_new, fh, y_want, lens, tol, ("WN residual", i)))
        else:
            assert np.array_equal(fh_new.view(np.uint32), fh.view(np.uint32)), "the last layer writes the skip sum only"
        worst = max(worst, _check(skip_new, skip, s_want, lens, tol, ("WN skip", i)))
        fh, skip = fh_new, skip_new
    _report("WN", backend, flat, worst)
    # coupling: x1 = x1 - post(skip sum)   (192 -> 96, 1x1, in place)
    w, bias = _weights(half, H, 1, seed=60)
    x1 = rng.standard_normal((B, half, pitch)).astype(np.float32)
    skip_c = [skip[b, :, :L].astype(np.float64) for b, L in enumerate(lens)]
    want = [x1[b, :, :L].astype(np.float64) - _conv(skip_c[b], w, bias, 1, 0, None) for b, L in enumerate(lens)]
    y, _ = _launch(backend, skip, w, lens, flat=flat, epi="SUBFROM", bias=bias, y=x1, y_is_r=True)
    _report("SUBFROM", backend, flat, _check(y, x1, want, lens, tol, "SUBFROM"))


# ---------------------------------------------------------------------------------------------------------------------
# ConvTranspose1d(k = 2 * stride, padding = stride / 2) lowered to stride-phase rows and a pixel-shuffle store, at the rate
# of its stage: (C_in, stride, kernel, len_scale) of the medium (x8 x8 x4) and high (x8 x8 x2 x2) generators
UPS = [(256, 8, 16, 1), (128, 8, 16, 8), (64, 4, 8, 64), (512, 8, 16, 1), (64, 2, 4, 128)]


def _lower_transpose(Wt, up):
    """ConvTranspose weights [C_in][C_out][ku] -> the engine's lowered Conv1d [C_out * up][C_in][ku / up] (voice.cc)."""
    ci, co, ku = Wt.shape
    m = ku // up
    w = np.zeros((co * up, ci, m), np.float32)
    for j in range(m):
        for phi in range(up):
            w[phi::up, :, j] = Wt[:, :, phi + (m - 1 - j) * up].T
    return w


@pytest.mark.parametrize("case", UPS, ids=lambda c: f"{c[0]}-s{c[1]}-k{c[2]}-rate{c[3]}")
@pytest.mark.parametrize("backend", BACKENDS)
def test_conv_transpose_upsample(lib_built, backend, case):
    import torch
    import torch.nn.functional as F
    ci, up, ku, rate = case
    co, m = ci // 2, ku // up
    frames = (1, 3, 7, 33) if rate > 1 else LENS
    lens_in = [f * rate for f in frames]
    x, clean = _ragged(ci, lens_in, seed=ci + up + rate)
    rng = np.random.default_rng(ci)
    Wt = (rng.standard_normal((ci, co, ku)) / np.sqrt(ci * 2)).astype(np.float32)
    bias_c = rng.standard_normal(co).astype(np.float32)
    pitch_out = x.shape[2] * up
    y0 = np.full((len(frames), co, pitch_out), SENTINEL, np.float32)
    y, _ = _launch(backend, x, _lower_transpose(Wt, up), frames, epi="UPSAMPLE", bias=np.repeat(bias_c, up), pad=m - 1,
                   slope=0.1, y=y0, up=up, up_pad=up // 2, q_extra=m - 1, len_scale=rate)
    want = []
    for b in range(len(frames)):
        ref = F.conv_transpose1d(F.leaky_relu(torch.from_numpy(clean[b]), 0.1)[None], torch.from_numpy(Wt.astype(np.float64)),
                                 torch.from_numpy(bias_c.astype(np.float64)), stride=up, padding=up // 2)[0].numpy()
        assert ref.shape[1] == lens_in[b] * up
        want.append(ref)
    _report("UPSAMPLE", backend, False, _check(y, y0, want, [L * up for L in lens_in], _tol(backend), case))


# ---------------------------------------------------------------------------------------------------------------------
# MRF: three resblock outputs into one accumulator, modes 0 -> 1 -> 2 (mrf_n = 3): y2 = v'; y2 += v'; y2 = (y2 + v') / 3
# with v' = conv(lrelu(x)) + x.  (channels, ((k, dil) per launch), len_scale, frames)
MRF = [
    (32, ((3, 1), (5, 6), (7, 12)), 256, (157, 150, 156, 155)),   # medium stage 3, ~40 k positions a item: many tiles per SM
    (32, ((3, 2), (5, 2), (7, 3)), 256, (1, 3, 2)),
    (64, ((3, 1), (5, 6), (7, 12)), 64, (1, 3, 7)),
    (128, ((3, 5), (7, 5), (11, 5)), 64, (1, 3, 5)),             # high stage 2 (ResBlock1 dilations)
    (128, ((11, 1), (11, 3), (11, 5)), 64, (2, 4)),
]


@pytest.mark.parametrize("case", MRF, ids=lambda c: f"{c[0]}ch-" + "-".join(f"k{k}d{d}" for k, d in c[1]) + f"-x{c[2]}-B{len(c[3])}")
@pytest.mark.parametrize("backend", BACKENDS)
def test_mrf_accumulation_modes(lib_built, backend, case):
    Cc, convs, rate, frames = case
    lens_in = [f * rate for f in frames]
    x, clean = _ragged(Cc, lens_in, seed=Cc + rate + len(frames))
    acc = np.full(x.shape, SENTINEL, np.float32)
    worst = 0.0
    for mode, (k, dil) in enumerate(convs):
        w, bias = _weights(Cc, Cc, k, seed=100 * k + dil)
        vp = [_conv(clean[b], w, bias, dil, dil * (k - 1) // 2, 0.1) + clean[b] for b in range(len(frames))]
        prev = [acc[b, :, :L].astype(np.float64) for b, L in enumerate(lens_in)]
        want = [vp[b] if mode == 0 else (prev[b] + vp[b] if mode == 1 else (prev[b] + vp[b]) / 3.0)
                for b in range(len(frames))]
        _, new = _launch(backend, x, w, frames, epi="MRF", bias=bias, dil=dil, slope=0.1, r=x, y2=acc, mrf=mode, mrf_n=3,
                         len_scale=rate)
        worst = max(worst, _check(new, acc, want, lens_in, _tol(backend), ("MRF", mode)))
        acc = new
    _report("MRF", backend, False, worst)


# ---------------------------------------------------------------------------------------------------------------------
# shapes the tensor-core plan declines run on the CUDA cores only (test_conv2_sim: the plan declines them)
DECLINED = [(192, 29, 1), (1, 192, 1), (100, 64, 3)]     # dp spline projection, dp pre of the 1-channel input, 100-ch conv


@pytest.mark.parametrize("case", DECLINED, ids=lambda c: f"{c[0]}x{c[1]}k{c[2]}")
def test_shapes_the_tensor_cores_decline(lib_built, case):
    from piper_b200._lib import PiperB200Error
    ci, rows, k = case
    lens = LENS
    x, clean = _ragged(ci, lens, seed=ci + rows)
    w, bias = _weights(rows, ci, k, seed=rows)
    y0 = np.full((len(lens), rows, x.shape[2]), SENTINEL, np.float32)
    want = [_conv(clean[b], w, bias, 1, (k - 1) // 2, None) for b in range(len(lens))]
    y, _ = _launch(0, x, w, lens, bias=bias, y=y0)
    _report("BIAS-declined", 0, False, _check(y, y0, want, lens, _tol(0), case))
    for backend in BACKENDS[1:]:
        with pytest.raises(PiperB200Error, match="not supported by the tensor-core conv"):
            _launch(backend, x, w, lens, bias=bias, y=y0)


def test_launches_the_engine_never_makes_are_errors(lib_built):
    from piper_b200._lib import PiperB200Error
    x, _ = _ragged(32, (5,), seed=1)
    w, bias = _weights(33, 32, 3, seed=1)
    y = np.zeros((1, 33, x.shape[2]), np.float32)
    for backend in (0, 5):
        with pytest.raises(PiperB200Error, match="GATE needs an even number of rows"):
            _launch(backend, x, w, (5,), epi="GATE", bias=bias, y=y)
        with pytest.raises(PiperB200Error, match="rows % up"):
            _launch(backend, x, w, (5,), epi="UPSAMPLE", bias=bias, y=y, up=2, up_pad=1)


def test_latency_plan(lib_built):
    """The two-chain latency plan the engine takes for small fp32-grade launches, on the flow in_layer shape."""
    ci, rows, k, lens = 192, 384, 5, (1, 3, 130)
    x, clean = _ragged(ci, lens, seed=7)
    w, bias = _weights(rows, ci, k, seed=7)
    y0 = np.full((len(lens), rows // 2, x.shape[2]), SENTINEL, np.float32)
    want = []
    for b in range(len(lens)):
        v = _conv(clean[b], w, bias, 1, 2, None)
        want.append(np.tanh(v[0::2]) * _sigmoid(v[1::2]))
    for flat in (False, True):
        y, _ = _launch(5, x, w, lens, flat=flat, epi="GATE", bias=bias, y=y0, latency=True)
        _report("GATE-latency", 5, flat, _check(y, y0, want, lens, _tol(5), flat))


# ---------------------------------------------------------------------------------------------------------------------
# the engine with its convolutions on the CUDA cores (and one family at a time on the tensor cores)
SCALES = (0.667, 1.0, 0.8)
_voices, _refs = {}, {}


def _voice(tag):
    if tag not in _voices:
        from oracle.voice_loader import load_voice
        from oracle.vits_oracle import Oracle
        from piper_b200 import engine
        if tag == "real":
            path = real_voice_path()
            if path is None:
                pytest.skip("reference test voice not staged (oracle/_ref/voice)")
        else:
            path = voicegen.cached_voice(tag)
        spec, w, attrs = load_voice(path)
        _voices[tag] = (engine.Voice(path, 0), Oracle(spec, w, attrs))
    return _voices[tag]


def _inputs(tag, batch, inter):
    if tag == "real":
        ids_list = [real_fixture_lines()[5]["phoneme_ids"]]
    else:
        n_ph = {1: (64,), 3: (48, 7, 29)}[batch]
        ids_list = [voicegen.benchmark_ids(n, seed=3 + i) for i, n in enumerate(n_ph)]
    rng = np.random.default_rng(77)
    eps_dp = [rng.standard_normal((2, len(i))).astype(np.float32) for i in ids_list]
    eps_z = rng.standard_normal((len(ids_list), inter, 6 * max(len(i) for i in ids_list) + 16)).astype(np.float32)
    return ids_list, eps_dp, eps_z


def _oracle(tag, batch, sids):
    """The oracle's answers per item (the same for every mask): (waveform, dump)."""
    key = (tag, batch, sids)
    if key not in _refs:
        _, orc = _voice(tag)
        ids_list, eps_dp, eps_z = _inputs(tag, batch, orc.s.inter)
        out = []
        for b, ids in enumerate(ids_list):
            dump = {}
            ref = orc.infer(ids, SCALES, eps_dp[b], eps_z[b], dump=dump, sid=None if sids is None else sids[b])
            out.append((ref, {k: v.numpy() for k, v in dump.items()}))
        _refs[key] = out
    return _refs[key]


def _engine_vs_oracle(tag, batch, mask, sids=None):
    voice, orc = _voice(tag)
    refs = _oracle(tag, batch, sids)
    ids_list, eps_dp, eps_z = _inputs(tag, batch, orc.s.inter)
    stages = [f"stage{i}" for i in range(len(orc.s.up_rates))]
    voice.set_mma(mask)
    voice.set_speakers(list(sids) if sids else [])
    voice.set_debug(True)
    try:
        wavs, _ = voice.synthesize_batch(ids_list, SCALES, eps_dp, eps_z)
        taps = [{k: voice.tap(k, b) for k in ["x", "stats", "logw", "cum", "z_p", "z"] + stages} for b in range(batch)]
    finally:
        voice.set_debug(False)
        voice.set_speakers([])
        voice.set_mma(31)
    I = orc.s.inter
    worst = 0.0
    for b, (ref, dump) in enumerate(refs):
        t = taps[b]
        w_ceil = np.diff(np.concatenate([[0], t["cum"][0]]))
        assert np.array_equal(w_ceil, dump["w_ceil"]), (b, "durations must match exactly (ceil cliff)")
        assert np.abs(t["x"] - dump["x"]).max() <= 1e-3, b
        assert np.abs(t["stats"][:I] - dump["m_p"]).max() <= 1e-3, b
        assert np.abs(t["stats"][I:] - dump["logs_p"]).max() <= 1e-3, b
        assert np.abs(t["logw"][0] - dump["logw"]).max() <= 1e-3, b
        assert np.abs(t["z_p"] - dump["z_p"]).max() <= 1e-3, b
        for k in ["z"] + stages:
            e = np.abs(t[k] - dump[k]).max()
            assert e <= 2e-3, (b, k, e)
        assert wavs[b].shape == ref.shape, (b, wavs[b].shape, ref.shape)
        err = float(np.abs(wavs[b] - ref).max())
        assert err <= 1e-3, (b, err)
        assert float(np.sqrt((ref ** 2).mean())) > 0.05, "vacuous parity: oracle waveform is near silent"
        worst = max(worst, err)
    print(f"\nENGINE_ERR {tag} B={batch} mask={mask} wave_err={worst:.3e}")


@pytest.mark.parametrize("batch", [1, 3])
@pytest.mark.parametrize("mask", [0, 16, 1, 2, 4, 8])
@pytest.mark.parametrize("arch", ["medium", "high"])
def test_engine_on_cuda_cores_matches_oracle(lib_built, arch, mask, batch):
    _engine_vs_oracle(arch, batch, mask)


def test_engine_on_cuda_cores_per_item_speakers(lib_built):
    _engine_vs_oracle("tiny-ms", 3, 0, sids=(1, 0, 4))


def test_real_voice_on_cuda_cores(lib_built):
    _engine_vs_oracle("real", 1, 0)
