"""Per-launch report of the headline step (GPU): every conv launch's CUDA-event time (median of a few steps) next to the
analytical bounds of tools/perf_model.py for the same shape (HBM, tcgen05 issue, weight streaming).

usage: python tools/layer_report.py [--arch medium] [--batch 32] > gpurun_out/layer_report.txt   (JSON beside it)
With PIPER_B200_PROF_ROLES=1 each tensor-core launch also reports where its warp roles waited.
"""
import argparse, json, math, os, statistics, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np
import perf_model as pm
from piper_b200 import engine, voicegen

ap = argparse.ArgumentParser()
ap.add_argument("--arch", default="medium")
ap.add_argument("--batch", type=int, default=32)
ap.add_argument("--steps", type=int, default=5)
ap.add_argument("--from-json", default=None, help="re-print a saved gpurun_out/layer_report.json with the current model (no GPU)")
a = ap.parse_args()

if a.from_json:
    saved = json.load(open(a.from_json))
    runs = [[{k: r[k] for k in r if k not in ("n_tile", "n_tiles", "mt", "tiles", "t_hbm", "t_mma", "t_w", "t_tma", "bound")} for r in saved]]
    n, ms = 0, float("nan")
else:
  v = engine.Voice(voicegen.cached_voice(a.arch), 0)
  ids = [voicegen.benchmark_ids(128, seed=1234 + b) for b in range(a.batch)]
  v.stage(ids, (0.667, 1.0, 0.8), seed=4242)
  for _ in range(3):
      v.run_staged()
  v.set_profile(True)
  runs = []
  for _ in range(a.steps):
      n, ms = v.run_staged()
      runs.append(v.profile_launches())
  v.set_profile(False)
n_l = len(runs[0])
assert all(len(r) == n_l for r in runs)
pm.B = a.batch
# model the kernel that is actually running (default fp16x3 with tensor-map TMA)
pm.F16 = os.environ.get("PIPER_B200_V2_PREC", "f16") == "f16"
pm.TMA_CYC = 0.0 if os.environ.get("PIPER_B200_V2_TM", "1") != "0" else 20.0
rows = []
for i in range(n_l):
    r = dict(runs[0][i])
    r["us"] = statistics.median(x[i]["us"] for x in runs)
    if r["mma"] and r["tag"] != "dec.mrf":
        tf32 = not r["tag"].startswith("dec")
        L = r["len_sum"] / a.batch
        m = pm.layer(r["tag"], r["tag"], r["ci"], r["rows"], r["k"], r["dil"], L, tf32)
        # tiles follow the longest item; bytes follow the recorded algorithmic figure
        n_tile, n_tiles, mt = m["n_tile"], m["n_tiles"], m["mt"]
        tiles = math.ceil(r["max_len"] / mt) * a.batch * n_tiles
        scale = math.ceil(tiles / pm.SMS) / max(1, m["per_cta"])
        r.update(n_tile=n_tile, n_tiles=n_tiles, mt=mt, tiles=tiles, t_hbm=r["bytes"] / pm.HBM * 1e6,
                 t_mma=m["t_mma"] * scale * 1e6, t_w=m["t_w"] * scale * 1e6, t_tma=m["t_tma"] * scale * 1e6)
        r["bound"] = max(r["t_hbm"], r["t_mma"], r["t_w"], r["t_tma"])
    rows.append(r)
print(f"{a.arch}, {a.batch} utterances: " + (f"saved launch records of {a.from_json} re-modelled" if a.from_json else f"{n} samples in {ms:.3f} ms (profiled step)") + f", {n_l} conv launches")
print("bounds: t_hbm = algorithmic bytes / copy peak; t_mma = tcgen05 instructions x max(N/2, 32 + N/4) cycles (measured pacing, tools/perf_model.py); t_w = weight stream L2 -> SM; us/bound against the largest")
print(f"{'#':>3s} {'tag':8s} {'ci':>4s} {'rows':>5s} {'k':>2s} {'d':>2s} {'N':>4s} {'mt':>3s} {'tiles':>6s} | {'us':>7s} | {'t_hbm':>6s} {'t_mma':>6s} {'t_w':>6s} {'t_tma':>6s} | {'us/bound':>8s}")
fam = {}
for i, r in enumerate(rows):
    if r["mma"] and "bound" in r:
        print(f"{i:3d} {r['tag']:8s} {r['ci']:4d} {r['rows']:5d} {r['k']:2d} {r['dil']:2d} {r['n_tile']:4d} {r['mt']:3d} {r['tiles']:6d} | {r['us']:7.1f} | "
              f"{r['t_hbm']:6.1f} {r['t_mma']:6.1f} {r['t_w']:6.1f} {r['t_tma']:6.1f} | {r['us'] / r['bound']:8.2f}")
        if "roles" in r:   # PIPER_B200_PROF_ROLES=1: share of each role's loop spent waiting (conv2_body.inl, summed over CTAs)
            q = r["roles"]
            pc = lambda x, d: 100.0 * x / max(1, d)
            print(f"      roles: MMA waits accumulator-free {pc(q[0], q[3]):4.0f}%  operands {pc(q[1], q[3]):4.0f}%  weights {pc(q[2], q[3]):4.0f}% | "
                  f"epilogue waits accumulator {pc(q[4], q[5]):4.0f}% | converter waits raw {pc(q[6], q[8]):4.0f}%  free slot {pc(q[7], q[8]):4.0f}%")
        f = fam.setdefault(r["tag"], [0.0, 0.0, 0])
        f[0] += r["us"]; f[1] += r["bound"]; f[2] += 1
    else:
        what = "(fused MRF stage, k = taps)" if r["tag"] == "dec.mrf" else "(CUDA-core kernel)       "
        print(f"{i:3d} {r['tag']:8s} {r['ci']:4d} {r['rows']:5d} {r['k']:2d} {r['dil']:2d}   {what} | {r['us']:7.1f} |")
print("\nfamily    launches   measured ms   bound ms   ratio")
for k, (us, b, c) in fam.items():
    print(f"{k:9s} {c:8d} {us / 1e3:13.3f} {b / 1e3:10.3f} {us / b:7.2f}")
os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
if not a.from_json:
    json.dump(rows, open(os.path.join(ROOT, "gpurun_out", "layer_report.json"), "w"))
