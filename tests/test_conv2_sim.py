"""The experimental second-generation tensor-core convolution (piper_b200/csrc/conv2_body.inl: uniform-issue TMA warps,
stacked [W_hi ; W_lo] weights) run on the CPU model of the primitives (tests/sim) against torch, for every fused epilogue,
both split precisions, ragged batches, dilation, ConvTranspose lowering.  No GPU: checks logic, layouts and the barrier
protocol, not the hardware's asynchrony."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIM = os.path.join(ROOT, "tests", "sim", "libconv2_sim.so")
EPI = dict(BIAS=0, RELU=1, RES=2, GATE=3, WN=4, SUBFROM=5, UPSAMPLE=6, MRF=7)


@pytest.fixture(scope="module")
def sim():
    if not os.path.exists(SIM):
        subprocess.run(["make", "-C", os.path.join(ROOT, "piper_b200", "csrc"), "../../tests/sim/libconv2_sim.so"], check=True,
                       stdout=subprocess.DEVNULL)
    return C.CDLL(SIM)


def _fp(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_float))


def _run(sim, x, w, bias, lens, *, dil=1, pad=None, pre=0, slope=0.1, epi="BIAS", tf32=False, prec=None, chains=0, opts=0, r=None, y2_init=None, split=0,
         first=0, up=1, up_pad=0, mrf=0, mrf_n=3, q_extra=0, bias_item=None, grid=0, y_channels=None):
    B, ci, cs_x = x.shape
    rows, _, k = w.shape
    if pad is None:
        pad = (k - 1) // 2 * dil
    lens = np.asarray(lens, np.int32)
    C_y = y_channels if y_channels is not None else rows
    cs_y = cs_x * up
    y = np.full((B, C_y, cs_y), 7e7, np.float32)
    y2 = y2_init.copy() if y2_init is not None else np.full((B, max(rows - split, 1), cs_x), 7e7, np.float32)
    if prec is None:
        prec = 1 if tf32 else 0
    desc = (C.c_int32 * 26)(ci, rows, k, dil, pad, q_extra, pre, EPI[epi], split, first, up, up_pad, mrf, mrf_n, prec, 1,
                           cs_x, cs_y, y2.shape[2], 0 if r is None else r.shape[2], C_y, y2.shape[1],
                           0 if r is None else r.shape[1], grid, chains, opts)
    info = (C.c_int32 * 8)()
    err = C.create_string_buffer(512)
    rc = sim.conv2_sim_run(_fp(x), _fp(np.ascontiguousarray(w)), _fp(bias), _fp(bias_item), 0 if bias_item is None else bias_item.shape[1],
                           _fp(y), _fp(y2), _fp(r), lens.ctypes.data_as(C.POINTER(C.c_int32)), B, desc, C.c_float(slope),
                           int(lens.max()) + q_extra, info, err, len(err))
    assert rc == 0, err.value.decode()
    return y, y2, list(info)


def _ragged(B, ci, lens, seed, scale=1.0):
    rng = np.random.default_rng(seed)
    cs = (max(lens) + 3) & ~3
    x = rng.standard_normal((B, ci, cs)).astype(np.float32) * 40.0      # stale data past each item's length
    clean = []
    for b, L in enumerate(lens):
        v = rng.standard_normal((ci, L)).astype(np.float32) * scale
        x[b, :, :L] = v
        clean.append(torch.from_numpy(v))
    return x, clean


def _ref_conv(xb, w, bias, dil, pad, pre, slope):
    xt = F.leaky_relu(xb, slope) if pre else xb
    return F.conv1d(xt[None].double(), torch.from_numpy(w).double(), None if bias is None else torch.from_numpy(bias).double(),
                    dilation=dil, padding=pad)[0].float()


def _tol(tf32):
    return 2e-5 if tf32 else 3e-4      # relative to the output scale: tf32x3 keeps ~21 mantissa bits, bf16x3 ~16


@pytest.mark.parametrize("tf32", [False, True])
@pytest.mark.parametrize("ci,rows,k,dil,lens", [(32, 32, 7, 3, (300, 37, 129)),      # generator stage-3 shape, MT = 256
                                                 (64, 128, 3, 1, (140, 260)),         # n_tile = 128
                                                 (48, 96, 5, 2, (131,)),              # rows not a power of two
                                                 (192, 64, 1, 1, (259, 5)),           # 1x1, several channel chunks
                                                 (32, 16, 3, 1, (400, 130))])         # one 16-row chunk: half the epilogue warps idle
def test_plain_relu_and_residual_epilogues(sim, tf32, ci, rows, k, dil, lens):
    if tf32 and ci % 8:
        pytest.skip("tf32 needs ci % 8 == 0")
    B = len(lens)
    x, clean = _ragged(B, ci, lens, seed=ci + k)
    rng = np.random.default_rng(1)
    w = (rng.standard_normal((rows, ci, k)) / np.sqrt(ci * k)).astype(np.float32)
    bias = rng.standard_normal(rows).astype(np.float32)
    r = rng.standard_normal((B, rows, x.shape[2])).astype(np.float32)
    for epi, pre in (("BIAS", 0), ("RELU", 1), ("RES", 1), ("SUBFROM", 0)):
        y, _, info = _run(sim, x, w, bias, lens, dil=dil, pre=pre, epi=epi, tf32=tf32, r=r if epi in ("RES", "SUBFROM") else None,
                          grid=1 if rows == 16 else 3)      # one CTA: every TMEM set and ring slot gets reused
        for b, L in enumerate(lens):
            ref = _ref_conv(clean[b], w, bias, dil, (k - 1) // 2 * dil, pre, 0.1)
            if epi == "RELU":
                ref = torch.relu(ref)
            if epi == "RES":
                ref = ref + torch.from_numpy(r[b, :, :L])
            if epi == "SUBFROM":
                ref = torch.from_numpy(r[b, :, :L]) - ref
            e = float((torch.from_numpy(y[b, :, :L]) - ref).abs().max())
            assert e <= _tol(tf32) * max(1.0, float(ref.abs().max())), (epi, b, e, info)
            assert np.all(y[b, :, L:] == 7e7), "stored outside the utterance"


def test_wavenet_gate_and_res_skip(sim):
    """in_layer -> tanh*sigmoid gate (rows interleaved), then res_skip with in-place residual and skip accumulation."""
    H, lens = 64, (150, 61)
    B = len(lens)
    x, clean = _ragged(B, H, lens, seed=3)
    rng = np.random.default_rng(2)
    w = (rng.standard_normal((2 * H, H, 5)) / np.sqrt(H * 5)).astype(np.float32)
    bias = rng.standard_normal(2 * H).astype(np.float32) * 0.1
    cond = rng.standard_normal((B, 2 * H)).astype(np.float32) * 0.1            # per-item (speaker) bias
    y, _, info = _run(sim, x, w, bias, lens, epi="GATE", tf32=True, bias_item=cond, y_channels=H)
    for b, L in enumerate(lens):
        pre = _ref_conv(clean[b], w, bias, 1, 2, 0, 0.1) + torch.from_numpy(cond[b])[:, None]
        ref = torch.tanh(pre[0::2]) * torch.sigmoid(pre[1::2])
        assert float((torch.from_numpy(y[b, :, :L]) - ref).abs().max()) <= 2e-5, info
    # res_skip: rows < split update the residual stream (y = r + v), rows >= split accumulate into y2
    w2 = (rng.standard_normal((2 * H, H, 1)) / np.sqrt(H)).astype(np.float32)
    b2 = rng.standard_normal(2 * H).astype(np.float32) * 0.1
    r = rng.standard_normal((B, H, x.shape[2])).astype(np.float32)
    skip0 = rng.standard_normal((B, H, x.shape[2])).astype(np.float32)
    for first in (1, 0):
        y, y2, _ = _run(sim, x, w2, b2, lens, epi="WN", tf32=True, r=r, y2_init=skip0, split=H, first=first, y_channels=H)
        for b, L in enumerate(lens):
            v = _ref_conv(clean[b], w2, b2, 1, 0, 0, 0.1)
            assert float((torch.from_numpy(y[b, :, :L]) - (torch.from_numpy(r[b, :, :L]) + v[:H])).abs().max()) <= 2e-5
            want = v[H:] if first else torch.from_numpy(skip0[b, :, :L]) + v[H:]
            assert float((torch.from_numpy(y2[b, :, :L]) - want).abs().max()) <= 2e-5


@pytest.mark.parametrize("up,ku", [(8, 16), (4, 8), (2, 4)])
def test_conv_transpose_lowering(sim, up, ku):
    """ConvTranspose1d(k = 2 * stride, padding = stride / 2) as stride-phase rows + pixel-shuffle store (voice.cc lowering)."""
    ci, co, lens = 64, 32, (37, 140)
    B = len(lens)
    x, clean = _ragged(B, ci, lens, seed=up)
    rng = np.random.default_rng(4)
    Wt = (rng.standard_normal((ci, co, ku)) / np.sqrt(ci * 2)).astype(np.float32)
    bias_c = rng.standard_normal(co).astype(np.float32)
    m = ku // up
    w = np.zeros((co * up, ci, m), np.float32)                      # rows = co * up + phase, taps reversed
    for j in range(m):
        for phi in range(up):
            w[phi::up, :, j] = Wt[:, :, phi + (m - 1 - j) * up].T
    bias = np.repeat(bias_c, up)
    y, _, info = _run(sim, x, w, bias, lens, pad=m - 1, pre=1, epi="UPSAMPLE", up=up, up_pad=up // 2, q_extra=m - 1,
                      y_channels=co)
    for b, L in enumerate(lens):
        ref = F.conv_transpose1d(F.leaky_relu(clean[b], 0.1)[None].double(), torch.from_numpy(Wt).double(),
                                 torch.from_numpy(bias_c).double(), stride=up, padding=up // 2)[0].float()
        assert ref.shape[1] == L * up
        e = float((torch.from_numpy(y[b, :, :L * up]) - ref).abs().max())
        assert e <= 3e-4 * max(1.0, float(ref.abs().max())), (b, e, info)
        assert np.all(y[b, :, L * up:] == 7e7)


def test_mrf_accumulation_modes(sim):
    C_, lens = 32, (300, 90)
    B = len(lens)
    x, clean = _ragged(B, C_, lens, seed=9)
    rng = np.random.default_rng(5)
    w = (rng.standard_normal((C_, C_, 3)) / np.sqrt(C_ * 3)).astype(np.float32)
    bias = rng.standard_normal(C_).astype(np.float32)
    acc0 = rng.standard_normal((B, C_, x.shape[2])).astype(np.float32)
    for mode in (0, 1, 2):
        _, y2, _ = _run(sim, x, w, bias, lens, pre=1, epi="MRF", r=x, y2_init=acc0, mrf=mode, mrf_n=3)
        for b, L in enumerate(lens):
            v = _ref_conv(clean[b], w, bias, 1, 1, 1, 0.1) + clean[b]
            a0 = torch.from_numpy(acc0[b, :, :L])
            want = v if mode == 0 else (a0 + v if mode == 1 else (a0 + v) / 3)
            assert float((torch.from_numpy(y2[b, :, :L]) - want).abs().max()) <= 3e-4 * max(1.0, float(want.abs().max()))


def _piper_layer_shapes():
    """(ci, rows, k, dil, tf32) of every dense conv the engine sends to the tensor cores, for the three piper presets."""
    out = set()
    for H, F_ in ((96, 384), (192, 768)):                      # x-low | medium, high
        for ci, rows, k in ((H, 3 * H, 1), (H, H, 1), (H, F_, 3), (F_, H, 3), (H, 2 * H, 1)):
            out.add((ci, rows, k, 1, True))                    # text encoder
        out.add((H, H, 1, 1, True))                            # duration predictor 1x1
        for ci, rows, k in ((H // 2, H, 1), (H, 2 * H, 5), (H, 2 * H, 1), (H, H, 1), (H, H // 2, 1)):
            out.add((ci, rows, k, 1, True))                    # flow
        out.add((H, 256, 7, 1, False)); out.add((H, 512, 7, 1, False))     # conv_pre
    for C_, r, ku in ((256, 8, 16), (128, 8, 16), (64, 4, 8), (512, 8, 16), (128, 2, 4), (64, 2, 4)):
        out.add((C_, C_ // 2 * r, ku // r, 1, False))          # ConvTranspose lowered to stride-phase rows
    for C_ in (256, 128, 64, 32):
        for k, ds in ((3, (1, 2)), (5, (2, 6)), (7, (3, 12)), (3, (1, 3, 5)), (7, (1, 3, 5)), (11, (1, 3, 5))):
            for d in set(ds) | {1}:
                out.add((C_, C_, k, d, False))
    return sorted(out)


def _engine_plans(ci, k, tf32):
    """(prec, chains) the engine plans a layer with (engine.cu conv2_layer): fp16x3 by default - 1 chain for the
    generator; for the fp32-grade families 2 chains when ci * k >= 400 (1 otherwise) plus the 2-chain latency variant -
    and, under PIPER_B200_V2_PREC=std, bf16x3 with 1 chain for the generator and tf32x3 with 2 chains elsewhere."""
    if not tf32:
        return [(2, 1), (0, 1)]
    return sorted({(2, 2 if ci * k >= 400 else 1), (2, 2), (1, 2 if ci * k >= 400 else 1), (1, 2)})


def _check_plan(info, ci, rows, k, dil, prec, want_chains):
    ok, n_tile, n_tiles, mt, kc, stage_rows, raw_stride, t_slots, tmem_cols, chains, mh_stride, smem, w_bytes = list(info)
    assert ok, (ci, rows, k, dil, prec, want_chains)
    es, kstep = (4, 8) if prec == 1 else (2, 16)
    assert mt in (128, 256) and (mt == 128 or (prec != 1 and chains == 1))          # 256-row tiles: 1-chain bf16 / fp16 only
    assert n_tile * n_tiles == rows and n_tile % 16 == 0 and 2 * n_tile <= 256       # stacked instruction: N' = 2N <= 256
    assert chains == want_chains and mh_stride == chains * 2 * n_tile
    assert t_slots * (mt // 128) * mh_stride <= tmem_cols <= 512
    assert ci % kc == 0 and kc % kstep == 0
    assert stage_rows >= mt + (k - 1) * dil and stage_rows % 8 == 0 and raw_stride >= stage_rows + 4
    assert smem == 2 * kc * raw_stride * 4 + 2 * 2 * kc * stage_rows * es + 4 * kc * 2 * n_tile * es <= 196 * 1024
    assert (kc * raw_stride * 4) % 128 == 0 and (kc * stage_rows * es) % 128 == 0     # ring slots stay 128-byte aligned
    assert w_bytes == rows * k * ci * 2 * es


def test_plan_respects_hardware_limits_for_every_piper_layer(sim):
    sim.conv2_sim_plan.argtypes = [C.c_int] * 6 + [C.POINTER(C.c_longlong)]
    info = (C.c_longlong * 13)()
    for ci, rows, k, dil, tf32 in _piper_layer_shapes():
        sim.conv2_sim_plan(ci, rows, k, dil, int(tf32), 2 if tf32 else 1, info)
        _check_plan(info, ci, rows, k, dil, int(tf32), 2 if tf32 else 1)


def _engine_plans(ci, k, tf32):
    """(prec, chains) the engine plans a layer with (engine.cu conv2_layer): fp16x3 by default - 1 chain for the
    generator; for the fp32-grade families 2 chains when ci * k >= 400 (1 otherwise) plus the 2-chain latency variant -
    and, under PIPER_B200_V2_PREC=std, bf16x3 with 1 chain for the generator and tf32x3 with 2 chains elsewhere."""
    if not tf32:
        return [(2, 1), (0, 1)]
    return sorted({(2, 2 if ci * k >= 400 else 1), (2, 2), (1, 2 if ci * k >= 400 else 1), (1, 2)})


def test_tensor_core_plans_respect_hardware_limits(sim):
    """Every dense layer shape of the x-low / medium / high presets gets a tensor-core tiling that fits the SM for every
    precision and K-chain count the engine plans it with; shapes the plan declines stay on the CUDA-core kernel."""
    sim.conv2_sim_plan.argtypes = [C.c_int] * 6 + [C.POINTER(C.c_longlong)]
    info = (C.c_longlong * 13)()
    for ci, rows, k, dil, tf32 in _piper_layer_shapes():
        for prec, chains in _engine_plans(ci, k, tf32):
            sim.conv2_sim_plan(ci, rows, k, dil, prec, chains, info)
            _check_plan(info, ci, rows, k, dil, prec, chains)
    for ci, rows, k, dil in ((192, 29, 1, 1), (1, 192, 1, 1), (100, 64, 3, 1)):
        for tf32 in (False, True):
            for prec, chains in _engine_plans(ci, k, tf32):
                sim.conv2_sim_plan(ci, rows, k, dil, prec, chains, info)
                assert info[0] == 0, (ci, rows, k, dil, prec, chains)


@pytest.mark.parametrize("ci,rows,k,dil,tf32,epi", [(192, 384, 5, 1, True, "GATE"),     # flow in_layer: 128-wide tiles, one TMEM set
                                                     (768, 192, 3, 1, True, "BIAS"),     # FFN second conv: 24 channel chunks
                                                     (192, 256, 7, 1, False, "BIAS"),    # generator conv_pre
                                                     (128, 128, 7, 12, False, "RES")])   # widest halo of the medium generator
def test_real_layer_shapes(sim, ci, rows, k, dil, tf32, epi):
    lens = (150, 40)
    B = len(lens)
    x, clean = _ragged(B, ci, lens, seed=rows)
    rng = np.random.default_rng(7)
    w = (rng.standard_normal((rows, ci, k)) / np.sqrt(ci * k)).astype(np.float32)
    bias = rng.standard_normal(rows).astype(np.float32) * 0.1
    r = rng.standard_normal((B, rows, x.shape[2])).astype(np.float32)
    y, _, info = _run(sim, x, w, bias, lens, dil=dil, pre=1, epi=epi, tf32=tf32, r=r if epi == "RES" else None,
                      y_channels=rows // 2 if epi == "GATE" else None, grid=1)   # one CTA: rings and TMEM sets wrap
    for b, L in enumerate(lens):
        ref = _ref_conv(clean[b], w, bias, dil, (k - 1) // 2 * dil, 1, 0.1)
        if epi == "GATE":
            ref = torch.tanh(ref[0::2]) * torch.sigmoid(ref[1::2])
        if epi == "RES":
            ref = ref + torch.from_numpy(r[b, :, :L])
        e = float((torch.from_numpy(y[b, :, :L]) - ref).abs().max())
        assert e <= _tol(tf32) * max(1.0, float(ref.abs().max())), (b, e, info)


@pytest.mark.parametrize("ci,rows,k,dil,chains,lens", [(192, 384, 5, 1, 2, (150, 40)),      # flow in_layer with fp16 operands
                                                        (192, 192, 1, 1, 2, (259, 5)),      # encoder 1x1
                                                        (32, 32, 7, 12, 1, (300, 90)),      # generator stage 3
                                                        (768, 192, 3, 1, 2, (131,))])       # FFN second conv
def test_fp16x3_mode_has_tf32x3_class_accuracy(sim, ci, rows, k, dil, chains, lens):
    """PREC_F16: FP16 hi/lo operands (22 bits kept, K = 16 per instruction).  Same harness, tf32x3's tolerance."""
    B = len(lens)
    x, clean = _ragged(B, ci, lens, seed=k)
    rng = np.random.default_rng(11)
    w = (rng.standard_normal((rows, ci, k)) / np.sqrt(ci * k)).astype(np.float32)
    bias = rng.standard_normal(rows).astype(np.float32) * 0.1
    y, _, info = _run(sim, x, w, bias, lens, dil=dil, pre=1, prec=2, chains=chains, grid=1)
    assert info[5] == chains
    for b, L in enumerate(lens):
        ref = _ref_conv(clean[b], w, bias, dil, (k - 1) // 2 * dil, 1, 0.1)
        e = float((torch.from_numpy(y[b, :, :L]) - ref).abs().max())
        assert e <= 2e-5 * max(1.0, float(ref.abs().max())), (b, e, info)


def test_seeded_random_shapes(sim):
    """A small seeded sample of tools/conv2_fuzz.py (random shapes, precisions, epilogues, ragged batches, grid sizes)."""
    rng = np.random.default_rng(2024)
    done = 0
    while done < 10:
        prec = int(rng.integers(0, 3))
        ci = int(rng.choice([16, 32, 48, 64, 96, 128, 192]))
        rows = int(rng.choice([16, 32, 48, 64, 96, 128, 192, 384]))
        k = int(rng.choice([1, 3, 5, 7]))
        dil = int(rng.choice([1, 2, 3, 6])) if k > 1 else 1
        B = int(rng.integers(1, 4))
        lens = tuple(int(v) for v in rng.integers(1, 400, size=B))
        epi = str(rng.choice(["BIAS", "RES", "RELU"]))
        pre, chains, grid = int(rng.integers(0, 2)), int(rng.integers(1, 3)), int(rng.integers(1, 4))
        x, clean = _ragged(B, ci, lens, seed=done)
        w = (rng.standard_normal((rows, ci, k)) / np.sqrt(ci * k)).astype(np.float32)
        bias = rng.standard_normal(rows).astype(np.float32)
        r = rng.standard_normal((B, rows, x.shape[2])).astype(np.float32)
        y, _, info = _run(sim, x, w, bias, lens, dil=dil, pre=pre, epi=epi, prec=prec, chains=chains, r=r if epi == "RES" else None,
                          grid=grid)
        for b, L in enumerate(lens):
            ref = _ref_conv(clean[b], w, bias, dil, (k - 1) // 2 * dil, pre, 0.1)
            ref = torch.relu(ref) if epi == "RELU" else ref + torch.from_numpy(r[b, :, :L]) if epi == "RES" else ref
            e = float((torch.from_numpy(y[b, :, :L]) - ref).abs().max()) / max(1.0, float(ref.abs().max()))
            assert e <= (3e-4 if prec == 0 else 2e-5), (prec, ci, rows, k, dil, lens, epi, chains, grid, e, info)
            assert np.all(y[b, :, L:] == 7e7)
        done += 1


def test_tall_tiles_for_two_chain_layers(sim):
    """Plan option 1: 256-row tiles for a two-chain fp16 layer (flow in_layer shape): one TMEM set of 512 columns."""
    ci, rows, k, lens = 192, 384, 5, (300, 70)
    x, clean = _ragged(len(lens), ci, lens, seed=1)
    rng = np.random.default_rng(3)
    w = (rng.standard_normal((rows, ci, k)) / np.sqrt(ci * k)).astype(np.float32)
    bias = rng.standard_normal(rows).astype(np.float32) * 0.1
    y, _, info = _run(sim, x, w, bias, lens, epi="GATE", prec=2, chains=2, opts=1, grid=1, y_channels=rows // 2)
    assert info[2] == 256 and info[4] == 1 and info[5] == 2, info          # mt, TMEM sets, chains
    for b, L in enumerate(lens):
        pre = _ref_conv(clean[b], w, bias, 1, 2, 0, 0.1)
        ref = torch.tanh(pre[0::2]) * torch.sigmoid(pre[1::2])
        assert float((torch.from_numpy(y[b, :, :L]) - ref).abs().max()) <= 2e-5, info


@pytest.mark.parametrize("prec,ci,rows,k,dil,lens", [(0, 32, 32, 7, 12, (600, 37, 257)),     # 328-row window: two boxes per chunk
                                                      (0, 64, 64, 5, 6, (300, 9)),            # one box, 256-row tiles
                                                      (1, 192, 64, 5, 1, (259, 130)),         # tf32x3, several channel chunks
                                                      (2, 96, 192, 1, 1, (131, 4))])          # fp16x3 1x1 (flow pre)
def test_tensor_map_activation_loads(sim, prec, ci, rows, k, dil, lens):
    """opts bit 2: the activation window arrives as cp.async.bulk.tensor boxes (any start column, zero fill outside the
    tensor) instead of one bulk copy per channel row - same results as the per-row path, for negative window starts,
    windows that run past the pitch, and stale data past each utterance."""
    B = len(lens)
    x, clean = _ragged(B, ci, lens, seed=11 + ci)
    rng = np.random.default_rng(6)
    w = (rng.standard_normal((rows, ci, k)) / np.sqrt(ci * k)).astype(np.float32)
    bias = rng.standard_normal(rows).astype(np.float32)
    r = rng.standard_normal((B, rows, x.shape[2])).astype(np.float32)
    y_tm, _, info = _run(sim, x, w, bias, lens, dil=dil, pre=1, epi="RES", prec=prec, r=r, opts=4, grid=2)
    y_row, _, _ = _run(sim, x, w, bias, lens, dil=dil, pre=1, epi="RES", prec=prec, r=r, opts=0, grid=2)
    y_m3, _, _ = _run(sim, x, w, bias, lens, dil=dil, pre=1, epi="RES", prec=prec, r=r, opts=12, grid=2)   # + three-instruction k-step
    for b, L in enumerate(lens):
        assert np.array_equal(y_tm[b, :, :L], y_row[b, :, :L]), (b, info)       # same operands, same instruction order
        assert np.abs(y_m3[b, :, :L] - y_row[b, :, :L]).max() <= 1e-5 * max(1.0, np.abs(y_row[b, :, :L]).max()), (b, info)
        ref = _ref_conv(clean[b], w, bias, dil, (k - 1) // 2 * dil, 1, 0.1) + torch.from_numpy(r[b, :, :L])
        e = float((torch.from_numpy(y_tm[b, :, :L]) - ref).abs().max())
        assert e <= _tol(prec != 0) * max(1.0, float(ref.abs().max())), (b, e, info)
        assert np.all(y_tm[b, :, L:] == 7e7), "stored outside the utterance"


def test_tensor_map_conv_transpose_tail(sim):
    """ConvTranspose lowering in tensor-map mode: the tail tile past the input length loads a window that lies wholly
    outside the utterance (masked to zero by the converter)."""
    up, ku = 8, 16
    ci, co, lens = 64, 32, (256, 140)          # 256 = one full tile, so the q_extra tail is a tile of its own
    B = len(lens)
    x, clean = _ragged(B, ci, lens, seed=up)
    rng = np.random.default_rng(4)
    Wt = (rng.standard_normal((ci, co, ku)) / np.sqrt(ci * 2)).astype(np.float32)
    bias_c = rng.standard_normal(co).astype(np.float32)
    m = ku // up
    w = np.zeros((co * up, ci, m), np.float32)
    for j in range(m):
        for phi in range(up):
            w[phi::up, :, j] = Wt[:, :, phi + (m - 1 - j) * up].T
    bias = np.repeat(bias_c, up)
    y, _, info = _run(sim, x, w, bias, lens, pad=m - 1, pre=1, epi="UPSAMPLE", up=up, up_pad=up // 2, q_extra=m - 1,
                      y_channels=co, opts=4)
    for b, L in enumerate(lens):
        ref = F.conv_transpose1d(F.leaky_relu(clean[b], 0.1)[None].double(), torch.from_numpy(Wt).double(),
                                 torch.from_numpy(bias_c).double(), stride=up, padding=up // 2)[0].float()
        e = float((torch.from_numpy(y[b, :, :L * up]) - ref).abs().max())
        assert e <= 3e-4 * max(1.0, float(ref.abs().max())), (b, e, info)
        assert np.all(y[b, :, L * up:] == 7e7)


@pytest.mark.parametrize("prec,ci,rows,k,dil,epi,lens", [(2, 192, 64, 1, 1, "RES", (259, 259, 259)),      # equal lengths: 3 x 264 = 792 rows -> 7 tiles instead of 9
                                                          (2, 96, 192, 5, 1, "GATE", (131, 40, 259, 7)),   # halo across item boundaries, ragged
                                                          (1, 64, 128, 3, 1, "RELU", (100, 1, 128)),
                                                          (2, 192, 384, 1, 1, "WN", (70, 130))])
@pytest.mark.parametrize("astat", [0, 32])
def test_flat_mode_tiles_on_the_concatenated_time_axis(sim, prec, ci, rows, k, dil, epi, lens, astat):
    """opts bit 4: views laid out [channel][item][slot] and ONE launch item of length items x slot - a tile may cover the end
    of one utterance and the start of the next; rows in the gaps are neither read as data nor written."""
    B = len(lens)
    Tg = ((max(lens) + 3) & ~3) + 4                          # slot = pitch + gap >= the largest one-sided halo
    rng = np.random.default_rng(17)
    x = rng.standard_normal((ci, B, Tg)).astype(np.float32) * 40.0      # stale data in the gaps
    clean = []
    for b, L in enumerate(lens):
        v = rng.standard_normal((ci, L)).astype(np.float32)
        x[:, b, :L] = v
        clean.append(torch.from_numpy(v))
    w = (rng.standard_normal((rows, ci, k)) / np.sqrt(ci * k)).astype(np.float32)
    bias = rng.standard_normal(rows).astype(np.float32)
    pad = (k - 1) // 2 * dil
    C_y = rows // 2 if epi == "GATE" else (rows // 2 if epi == "WN" else rows)
    split = rows // 2 if epi == "WN" else 0
    y = np.full((C_y, B, Tg), 7e7, np.float32)
    r = rng.standard_normal((C_y, B, Tg)).astype(np.float32)
    y2 = rng.standard_normal((max(rows - split, 1), B, Tg)).astype(np.float32)
    y2_0 = y2.copy()
    if epi == "WN":
        y[...] = r                                           # in-place residual stream (y == r in the engine)
    lens_a = np.asarray(lens, np.int32)
    desc = (C.c_int32 * 26)(ci, rows, k, dil, pad, 0, 1 if epi == "RELU" else 0, EPI[epi], split, 0, 1, 0, 0, 3, prec, 1,
                           B * Tg, B * Tg, B * Tg, B * Tg, C_y, y2.shape[0], C_y, 2, 0, 16 | 4 | astat)
    info = (C.c_int32 * 8)()
    err = C.create_string_buffer(512)
    rc = sim.conv2_sim_run(_fp(x), _fp(np.ascontiguousarray(w)), _fp(bias), None, 0, _fp(y), _fp(y2), _fp(y if epi == "WN" else r),
                           lens_a.ctypes.data_as(C.POINTER(C.c_int32)), B, desc, C.c_float(0.1), int(lens_a.max()), info, err, len(err))
    assert rc == 0, err.value.decode()
    tol = (2e-5 if prec else 3e-4)
    for b, L in enumerate(lens):
        ref = _ref_conv(clean[b], w, bias, dil, pad, 1 if epi == "RELU" else 0, 0.1)
        if epi == "RES":
            want = ref + torch.from_numpy(r[:, b, :L])
        elif epi == "RELU":
            want = torch.relu(ref)
        elif epi == "GATE":
            want = torch.tanh(ref[0::2]) * torch.sigmoid(ref[1::2])
        else:                                                # WN, not the first layer: residual rows in place, skip rows accumulate
            want = torch.from_numpy(r[:, b, :L]) + ref[:split]
            skip = torch.from_numpy(y2_0[:, b, :L]) + ref[split:]
            assert float((torch.from_numpy(y2[:, b, :L]) - skip).abs().max()) <= tol * max(1.0, float(skip.abs().max())), (b, info[:])
            assert np.array_equal(y2[:, b, L:], y2_0[:, b, L:]), "skip sum written in the gap"
        e = float((torch.from_numpy(y[:, b, :L]) - want).abs().max())
        assert e <= tol * max(1.0, float(want.abs().max())), (epi, b, e, list(info))
        gap = y[:, b, L:]
        assert np.all(gap == (r[:, b, L:] if epi == "WN" else 7e7)), "stored in the gap between utterances"


@pytest.mark.parametrize("prec,ci,rows,k,dil,epi,lens,grid", [(2, 192, 576, 1, 1, "BIAS", (259, 130), 3),    # q|k|v: 5 output-row tiles per position, two chunks
                                                               (2, 64, 256, 5, 1, "RES", (300, 37), 2),        # one chunk (both ring slots alternate between positions)
                                                               (1, 96, 384, 3, 1, "RELU", (140,), 5),          # more CTAs than positions: groups split across CTAs
                                                               (2, 192, 384, 5, 1, "GATE", (131, 259), 4),
                                                               (2, 192, 768, 3, 1, "RELU", (259, 130, 40), 2),  # first FFN conv: 12 output-row tiles, 4 resident chunks, several groups per CTA
                                                               (2, 256, 512, 3, 1, "BIAS", (150,), 1)])         # 256 channels: the window does not fit, the default order runs
def test_a_stationary_tile_order(sim, prec, ci, rows, k, dil, epi, lens, grid):
    """opts bit 5: the output-row tiles of a position are consecutive tiles of one CTA; the activation window is loaded and
    converted once per position and stays in the operand ring (one slot per channel chunk) until the group's last tile -
    same numbers as the default order up to the summation order inside the tensor core (the chunk size is re-chosen so that
    the whole window fits), with and without the flat layout / tensor-map loads."""
    B = len(lens)
    x, clean = _ragged(B, ci, lens, seed=ci + rows)
    rng = np.random.default_rng(8)
    w = (rng.standard_normal((rows, ci, k)) / np.sqrt(ci * k)).astype(np.float32)
    bias = rng.standard_normal(rows).astype(np.float32)
    C_y = rows // 2 if epi == "GATE" else rows
    r = rng.standard_normal((B, C_y, x.shape[2])).astype(np.float32) if epi == "RES" else None
    kw = dict(dil=dil, pre=1 if epi == "RELU" else 0, epi=epi, prec=prec, r=r, grid=grid, y_channels=C_y)
    y_ref, _, _ = _run(sim, x, w, bias, lens, opts=0, **kw)
    for opts in (32, 32 | 4):
        y, _, info = _run(sim, x, w, bias, lens, opts=opts, **kw)
        for b, L in enumerate(lens):
            scale = max(1.0, float(np.abs(y_ref[b, :, :L]).max()))
            assert float(np.abs(y[b, :, :L] - y_ref[b, :, :L]).max()) <= 2e-6 * scale, (opts, b, info)
            assert np.all(y[b, :, L:] == 7e7)
    for b, L in enumerate(lens):                                  # and the default order is right in the first place
        ref = _ref_conv(clean[b], w, bias, dil, (k - 1) // 2 * dil, kw["pre"], 0.1)
        if epi == "RES":
            ref = ref + torch.from_numpy(r[b, :, :L])
        elif epi == "RELU":
            ref = torch.relu(ref)
        elif epi == "GATE":
            ref = torch.tanh(ref[0::2]) * torch.sigmoid(ref[1::2])
        e = float((torch.from_numpy(y_ref[b, :, :L]) - ref).abs().max())
        assert e <= _tol(prec != 0) * max(1.0, float(ref.abs().max())), (b, e)
