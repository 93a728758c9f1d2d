"""Analytical per-layer model of the headline step (medium voice, 32 utterances, T = 259 ids, T' ~ 509 frames) - runs on
the CPU, no GPU needed.  For every dense convolution it derives, from the tiling plan of the tensor-core kernel
(conv_mma2.cu, through tests/sim/libconv2_sim.so) and its stacked-weight scheme (A_hi x [W_hi;W_lo] + A_lo x W_hi, two
instructions per k-step):

  * t_hbm   - layer-wise algorithmic bytes (SURVEY 8d) / measured copy peak
  * t_mma   - tcgen05.mma issue time: instructions per tile x cost(N) (mma_cost below: the SS-form instruction is paced by
              reading its A (128 x 32 B) and B (N x 32 B) operands from shared memory at 128 B/clk)
  * t_w     - weight units streamed L2 -> shared memory per tile / ~42 B/clk/SM (6300 B/clk chip-wide)
  * t_tma   - issue time of the activation-row bulk copies by the TMA thread: rows per tile x ~20 cycles with uniform
              issue (PIPER_B200_V2_TM=0; tools/layer_report.py sets 0 for the tensor-map loads: one copy per channel chunk)
  * wave quantisation: tiles are dealt to 148 persistent CTAs, the slowest CTA sets the time

and prints them next to the measured per-family conv time of the final round-1 bench line (profiles/bench_r1_final.json,
the first-generation kernel, kept for reference).

usage: python tools/perf_model.py [--std]
  --std    bf16x3 for the generator and tf32x3 elsewhere (PIPER_B200_V2_PREC=std) instead of fp16x3 for every family
"""
import json, math, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HBM = 6572.2e9
CLK = 1.965e9
SMS = 148
L2_B_PER_CLK_SM = 6300.0 / SMS
F16 = "--std" not in sys.argv
TMA_CYC = 20.0                    # (tools/layer_report.py sets 0 for the tensor-map kernel: one copy per channel chunk)

B, T, TP = 32, 259, 509          # utterances, ids, frames per utterance (bench: 4 071 680 samples / 256 / 32 = 497..520)


def mma_cost(n):                  # cycles per tcgen05.mma, M = 128, K = 32 bytes
    # round 2, measured with the kernel's exact instruction stream (tools/probe/mma_probe.cu, profiles/r02_mma_probe_*.txt):
    # 64 / 49 / ~40 cycles at N = 128 / 64 / 32 = the larger of the tensor-pipe floor 128 N / 256 and the time its A
    # (128 x 32 B) and B (N x 32 B) operands take to leave shared memory at 128 B/clk.  (Round 1 fitted (4096 + 32 N) / 128 + 8
    # to a microbenchmark that included the issue loop.)
    return max(n / 2.0, 32.0 + n / 4.0)


_sim = None


def plan_v2(ci, rows, k, dil, prec, chains):
    """(n_tile, n_tiles, mt, kc) from the kernel's own planner."""
    global _sim
    import ctypes as C
    if _sim is None:
        _sim = C.CDLL(os.path.join(ROOT, "tests", "sim", "libconv2_sim.so"))
        _sim.conv2_sim_plan.argtypes = [C.c_int] * 6 + [C.POINTER(C.c_longlong)]
    info = (C.c_longlong * 13)()
    _sim.conv2_sim_plan(ci, rows, k, dil, prec, chains, info)
    assert info[0], (ci, rows, k, dil, prec, chains)
    return int(info[1]), int(info[2]), int(info[3]), int(info[4])


def layer(name, fam, ci, rows, k, dil, L, tf32, extra_rw=0.0, up=1):
    """L: output positions per utterance *before* the pixel shuffle (ConvT computes L_in positions x rows = co*stride)."""
    prec = 2 if F16 else (1 if tf32 else 0)
    n_tile, n_tiles, mt, kc = plan_v2(ci, rows, k, dil, prec, 2 if tf32 else 1)
    es = 4 if prec == 1 else 2
    kstep = 8 if es == 4 else 16
    tiles = math.ceil(L / mt) * B * n_tiles
    per_cta = math.ceil(tiles / SMS)
    per_k = mma_cost(2 * n_tile) + mma_cost(n_tile)   # A_hi x [W_hi;W_lo] (N doubled) + A_lo x W_hi
    mma_tile = (mt // 128) * (ci // kstep) * k * per_k
    w_tile = 2 * ci * k * n_tile * es
    t_mma = per_cta * mma_tile / CLK
    t_w = per_cta * w_tile / L2_B_PER_CLK_SM / CLK
    t_tma = per_cta * ci * TMA_CYC / CLK                 # one bulk copy per input-channel row and tile
    bytes_alg = 4.0 * B * (L * ci + L * rows) * (1 + extra_rw) + 4.0 * ci * k * rows
    flop = 2.0 * B * L * ci * rows * k
    return dict(name=name, fam=fam, n_tile=n_tile, n_tiles=n_tiles, mt=mt, tiles=tiles, per_cta=per_cta,
                waste=per_cta * SMS / tiles * (math.ceil(L / mt) * mt / L), t_hbm=bytes_alg / HBM, t_mma=t_mma, t_w=t_w, t_tma=t_tma,
                flop=flop, bytes=bytes_alg)


def medium():
    H, F, I = 192, 768, 192
    out = []
    for l in range(6):
        out += [layer(f"enc{l}.qkv", "enc.mma", H, 3 * H, 1, 1, T, True), layer(f"enc{l}.o", "enc.mma", H, H, 1, 1, T, True),
                layer(f"enc{l}.ffn1", "enc.mma", H, F, 3, 1, T, True), layer(f"enc{l}.ffn2", "enc.mma", F, H, 3, 1, T, True)]
    out.append(layer("enc.proj", "enc.mma", H, 2 * I, 1, 1, T, True))
    for f in range(4):
        out.append(layer(f"flow{f}.pre", "flow.mma", I // 2, H, 1, 1, TP, True))
        for l in range(4):
            out.append(layer(f"flow{f}.in{l}", "flow.mma", H, 2 * H, 5, 1, TP, True))
            out.append(layer(f"flow{f}.rs{l}", "flow.mma", H, 2 * H if l < 3 else H, 1, 1, TP, True))
        out.append(layer(f"flow{f}.post", "flow.mma", H, I // 2, 1, 1, TP, True))
    out.append(layer("dec.pre", "dec.pre.mma", I, 256, 7, 1, TP, False))
    C, L = 256, TP
    for s, (r, ku) in enumerate(((8, 16), (8, 16), (4, 8))):
        out.append(layer(f"dec.up{s}", "dec.up.mma", C, C // 2 * r, ku // r, 1, L, False))
        C, L = C // 2, L * r
        for j, (k, dils) in enumerate(((3, (1, 2)), (5, (2, 6)), (7, (3, 12)))):
            for i, d in enumerate(dils):
                # residual is the input itself; the last conv of resblocks 1 and 2 also read-modify-writes the MRF sum
                out.append(layer(f"dec.rb{s}.{j}.{i}", "dec.rb.mma", C, C, k, d, L, False))
    return out


if __name__ == "__main__":
    meas = {}
    p = os.path.join(ROOT, "profiles", "bench_r1_final.json")
    if os.path.exists(p):
        meas = {k: v["ms_per_step"] for k, v in json.load(open(p))["roofline"]["stages"].items()}
    rows = medium()
    print(f"{'layer':14s} {'N':>4s} {'nt':>2s} {'mt':>3s} {'tiles':>6s} {'/CTA':>4s} {'waste':>5s} | {'t_hbm':>7s} {'t_mma':>7s} {'t_w':>7s} {'t_tma':>7s} us")
    fam = {}
    for r in rows:
        print(f"{r['name']:14s} {r['n_tile']:4d} {r['n_tiles']:2d} {r['mt']:3d} {r['tiles']:6d} {r['per_cta']:4d} {r['waste']:5.2f} | "
              f"{r['t_hbm'] * 1e6:7.1f} {r['t_mma'] * 1e6:7.1f} {r['t_w'] * 1e6:7.1f} {r['t_tma'] * 1e6:7.1f}")
        f = fam.setdefault(r["fam"], dict(hbm=0.0, mma=0.0, w=0.0, bound=0.0, tma=0.0, all=0.0, n=0))
        f["hbm"] += r["t_hbm"]; f["mma"] += r["t_mma"]; f["w"] += r["t_w"]; f["tma"] += r["t_tma"]; f["n"] += 1
        f["bound"] += max(r["t_hbm"], r["t_mma"], r["t_w"])
        f["all"] += max(r["t_hbm"], r["t_mma"], r["t_w"], r["t_tma"])
    what = "tensor-core kernel, " + ("fp16x3 everywhere" if F16 else "bf16x3 / tf32x3") + ", stacked weights, uniform TMA issue"
    print(f"\nscheme: {what}")
    print(f"{'family':12s} {'launches':>8s} {'sum t_hbm':>10s} {'sum t_mma':>10s} {'sum t_w':>9s} {'sum t_tma':>10s} {'max w/o tma':>12s} {'max with tma':>13s} {'measured':>9s}  ms per step")
    for k, f in fam.items():
        print(f"{k:12s} {f['n']:8d} {f['hbm'] * 1e3:10.3f} {f['mma'] * 1e3:10.3f} {f['w'] * 1e3:9.3f} {f['tma'] * 1e3:10.3f} {f['bound'] * 1e3:12.3f} "
              f"{f['all'] * 1e3:13.3f} {meas.get(k, float('nan')):9.3f}")
    print("(measured = the round-1 kernel, for reference)")
