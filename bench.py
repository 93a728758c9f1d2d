#!/usr/bin/env python
"""Benchmark of the hot path: phoneme ids -> fp32 waveform (VITS inference behind piper::synthesize).

    python bench.py --gpus N --steps K --warmup W [--config 2|3|4|5]   # this repo's CUDA engine
    python bench.py --impl reference --gpus N --steps K ...             # the reference's CPU path (oracle port)
    python bench.py ... --dump-outputs DIR                              # also write the last timed step's outputs

One "step" = one pass of the hot path over one batch of synthetic input.  `--config` selects the BASELINE.json
configuration (1-based, as SURVEY.md section 8d numbers them; default 3, the one the samples/sec metric is quoted on):

  3  medium architecture, 32 utterances x 128 phonemes (259 ids) per GPU, weak scaling         [default]
  2  medium architecture, batch = 1: latency, real-time factor, time to the first streamed chunk (replicas at N > 1)
  4  "high" architecture, 64 utterances x 128 phonemes in total, sharded over the N ranks (strong scaling)
  5  generator only (pb200_vocode): z ~ N(0,1) [B,192,256] -> [B,65536], B swept over {1,8,32,128}; GB/s per GPU

The real en_US-lessac-medium / de_DE-thorsten-high files are not available offline: the architectures are built with
seeded synthetic weights (piper_b200/voicegen.py, SURVEY.md section 8d).  Noise is drawn on the device (Philox), scales
are piper's defaults.  No data-path collective at any N; utterances are independent (piper.cpp:481-486).

The JSON line (rank 0) follows the driver contract; see DESIGN.md section 6 for every field.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np

METRIC = "audio_samples_per_sec_22050Hz"
N_PHONEMES = 128
SCALES = (0.667, 1.0, 0.8)
STAGES = ["text_encoder", "duration_predictor", "host_length_roundtrip", "expand_flow", "generator"]
# generator-only algorithmic work for 256 frames (SURVEY.md section 8d): (activation bytes per utterance, weight bytes, FLOP)
GEN_WORK = {"medium": (191.82e6, 6.65e6, 11.614e9), "high": (1037.50e6, 57.31e6, 157.416e9)}

CONFIGS = {
    2: dict(arch="medium", batch=1, scaling="weak", name="configs[1]: medium, batch=1 streaming (latency / RTF)"),
    3: dict(arch="medium", batch=32, scaling="weak", name="configs[2]: medium, batch=32 x 128-phoneme utterances per GPU"),
    4: dict(arch="high", batch=64, scaling="strong", name="configs[3]: high, batch=64 sharded over the GPUs"),
    5: dict(arch="medium", batch=128, scaling="weak", name="configs[4]: generator only, 256-frame batches, B sweep"),
}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=float(d["hbm_gbs"]), bf16_tflops=float(d.get("bf16_tflops_sustained", d["bf16_tflops"])),
                    source="measured (MEASURED_PEAKS.json; bf16 = sustained figure, kernels are timed inside a long step)")
    return dict(hbm_gbs=6650.0, bf16_tflops=1400.0, source="fallback (B200_PROFILING.md)")


def measure_pipe_peaks(torch):
    """TF32 tensor and FP32 FMA peaks with the MEASURED_PEAKS.json method (torch.matmul 8192^3, best of 5, CUDA events).
    Library GEMMs, run OUTSIDE every timed region: they only provide roofline denominators."""
    out = {}
    n = 8192
    a = torch.randn(n, n, device="cuda", dtype=torch.float32)
    b = torch.randn(n, n, device="cuda", dtype=torch.float32)
    for name, tf32 in (("tf32_tflops", True), ("fp32_fma_tflops", False)):
        torch.backends.cuda.matmul.allow_tf32 = tf32
        torch.matmul(a, b)
        best = float("inf")
        for _ in range(3 if not tf32 else 5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); torch.matmul(a, b); e1.record(); torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        out[name] = 2.0 * n ** 3 / (best * 1e-3) / 1e12
    torch.backends.cuda.matmul.allow_tf32 = False
    del a, b
    torch.cuda.empty_cache()
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device = device
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.device), "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def dist_env():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))


def workload_ids(cfg: dict, rank: int, world: int):
    """This rank's utterances.  Weak: `batch` per rank (distinct seeds per rank).  Strong: `batch` in total, dealt out
    round-robin (all 259 ids long, so the shards are balanced; host.shard_utterances does the length-aware deal)."""
    from piper_b200 import voicegen
    B = cfg["batch"]
    if cfg["scaling"] == "strong":
        return [voicegen.benchmark_ids(N_PHONEMES, seed=1234 + b) for b in range(B) if b % world == rank]
    return [voicegen.benchmark_ids(N_PHONEMES, seed=1234 + rank * B + b) for b in range(B)]


def workload_text(cfg: dict, world: int) -> str:
    arch, B = cfg["arch"], cfg["batch"]
    per = f"{B} x {N_PHONEMES}-phoneme utterances (259 ids) per GPU" if cfg["scaling"] == "weak" else \
          f"{B} x {N_PHONEMES}-phoneme utterances (259 ids) in total, {B // world if B % world == 0 else f'{B}/{world}'} per GPU"
    lay = {"medium": "en_US-lessac-medium", "high": "de_DE-thorsten-high"}[arch]
    return f"{arch} VITS ({lay} architecture, seeded synthetic weights), {per}, scales {SCALES}"


# ------------------------------------------------------------------------------------------------ CPU reference arm
def _oracle(arch):
    from oracle.voice_loader import load_voice
    from oracle.vits_oracle import Oracle
    from piper_b200 import voicegen
    spec, w, attrs = load_voice(voicegen.cached_voice(arch))
    return spec, Oracle(spec, w, attrs)


def pick_threads(orc, ids) -> int:
    """The torch CPU port does not scale to every core of a 128-thread host (small convs oversubscribe): find the
    per-process thread count with the best single-utterance latency on a short prefix."""
    import torch
    ncpu = os.cpu_count() or 1
    best, best_t = 1, float("inf")
    short = ids[:65]
    for c in sorted({c for c in (4, 8, 16, 32, 64, ncpu) if c <= ncpu}):
        torch.set_num_threads(c)
        orc.infer(short, SCALES)
        t = time.perf_counter()
        orc.infer(short, SCALES)
        dt = time.perf_counter() - t
        if dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    return best


def cpu_worker(args):
    """One CPU process of the reference arm: synthesise `--cpu-utts` utterances B = 1 (the only mode a reference caller
    uses, piper.cpp:352), print {"samples", "secs"}."""
    import torch
    torch.set_num_threads(args.cpu_threads)
    cfg = CONFIGS[args.config]
    spec, orc = _oracle(cfg["arch"])
    ids_list = workload_ids(dict(cfg, scaling="weak"), 0, 1)
    rng = np.random.default_rng(1235 + args.cpu_worker)
    def one(ids):
        if args.config == 5:                                              # generator only: z [192,256] -> 65536 samples
            import torch as _t
            return int(orc.generator(_t.from_numpy(rng.standard_normal((spec.inter, 256)).astype(np.float32))).numel())
        eps_dp = rng.standard_normal((2, len(ids))).astype(np.float32)
        eps_z = rng.standard_normal((spec.inter, 6 * len(ids))).astype(np.float32)
        return len(orc.infer(ids, SCALES, eps_dp, eps_z))
    one(ids_list[args.cpu_worker % len(ids_list)])                       # warm-up (untimed)
    print("READY", flush=True)
    sys.stdin.readline()                                                  # all workers start together
    t0 = time.perf_counter()
    n = sum(one(ids_list[(args.cpu_worker * args.cpu_utts + k) % len(ids_list)]) for k in range(args.cpu_utts))
    print(json.dumps({"samples": n, "secs": time.perf_counter() - t0}), flush=True)


def cpu_throughput(config: int, utts_per_proc: int, threads: int, procs: int):
    """Aggregate samples/s of `procs` concurrent oracle processes x `threads` threads (a throughput-fair use of the host:
    one process cannot use a 128-thread box).  Returns (samples/s, total utterances, wall seconds)."""
    ws = [subprocess.Popen([sys.executable, os.path.abspath(__file__), "--impl", "cpu-worker", "--config", str(config),
                            "--cpu-worker", str(i), "--cpu-utts", str(utts_per_proc), "--cpu-threads", str(threads)],
                           stdin=subprocess.PIPE, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
          for i in range(procs)]
    for w in ws:
        assert w.stdout.readline().strip() == "READY"
    t0 = time.perf_counter()
    for w in ws:
        w.stdin.write("go\n"); w.stdin.flush()
    res = [json.loads(w.stdout.readline()) for w in ws]
    wall = time.perf_counter() - t0
    for w in ws:
        w.wait()
    return sum(r["samples"] for r in res) / wall, utts_per_proc * procs, wall


def cpu_plan(cfg):
    """(threads per process, processes) for the host: the best single-process thread count, then as many processes as
    fit in the machine."""
    _, orc = _oracle(cfg["arch"])
    from piper_b200 import voicegen
    th = pick_threads(orc, voicegen.benchmark_ids(N_PHONEMES, seed=1234))
    return th, max(1, (os.cpu_count() or 1) // th)


def run_reference(args):
    """`--impl reference`: the reference's own CPU implementation of the path on the host cores.  onnxruntime is not in
    this image and the reference's PyTorch source cannot travel to the GPU box, so this is the oracle port
    (oracle/vits_oracle.py, pinned to that source), B = 1 calls, as many concurrent processes as the host holds."""
    rank, world, local = dist_env()
    if rank != 0:
        return
    cfg = CONFIGS[args.config]
    th, procs = cpu_plan(cfg)
    utts = 1 if cfg["arch"] == "high" else 2
    for _ in range(min(args.warmup, 1)):
        cpu_throughput(args.config, 1, th, procs)
    vals, wall = [], 0.0
    t_start = time.perf_counter()
    for _ in range(args.steps):
        v, n, w = cpu_throughput(args.config, utts, th, procs)
        vals.append(v); wall += w
        if time.perf_counter() - t_start > 150:       # bounded: the arm must end within a few minutes
            break
    v = statistics.median(vals)
    sample = (f"{utts} utterance(s) (259 ids) per process x {procs} concurrent processes x {th} threads per step, "
              f"{len(vals)} steps (median), B=1 calls; torch CPU fp32 oracle port of the reference graph (onnxruntime absent)")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "samples/s", "n_gpus": args.gpus,
        "steps": len(vals), "warmup": min(args.warmup, 1), "ms_per_step": wall / len(vals) * 1e3, "higher_is_better": True,
        "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_text(cfg, 1) + ", device Philox noise", "baseline_config": cfg["name"], "sample": sample},
        "cpu_baseline": {"value": v, "unit": "samples/s", "cores": th * procs, "threads_per_process": th, "processes": procs,
                         "kind": "port", "host_cpus": os.cpu_count(), "sample": sample},
        "e2e": {"value": v, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


# ------------------------------------------------------------------------------------------------ engine arm
DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(d: str, arrays: dict):
    """Write each array as `d/<name>.npy` (float32 or float64), at most DUMP_BYTES in all.  When the arrays do not fit, each
    one of more than 2^20 elements is replaced by a fixed seeded sample of its flattened elements, with the sampled flat
    positions in `d/<name>_index.npy`.  The inputs are seeded, so two builds can be compared file for file."""
    os.makedirs(d, exist_ok=True)
    big = {k for k, a in arrays.items() if a.size > 1 << 20}
    small_bytes = sum(a.nbytes for k, a in arrays.items() if k not in big) + 2048 * len(arrays)     # (.npy headers)
    big_bytes = sum(arrays[k].nbytes for k in big)
    for name, a in arrays.items():
        if name in big and small_bytes + big_bytes > DUMP_BYTES:
            k = int(a.size * (DUMP_BYTES - small_bytes) / big_bytes / (1 + 8 / a.itemsize))   # values + float64 positions
            idx = np.sort(np.random.default_rng(0).choice(a.size, k, replace=False))
            np.save(os.path.join(d, name + "_index.npy"), idx.astype(np.float64))
            a = a.reshape(-1)[idx]
        np.save(os.path.join(d, name + ".npy"), a)


class Dist:
    def __init__(self, torch):
        self.rank, self.world, self.local = dist_env()
        self.torch = torch
        self.dist = None
        torch.cuda.set_device(self.local)
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
            self.dist = dist

    def barrier(self):
        if self.dist:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def _red(self, x, op):
        if not self.dist:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=op)
        return float(t.item())

    def max(self, x):
        return self._red(x, self.dist.ReduceOp.MAX) if self.dist else x

    def sum(self, x):
        return self._red(x, self.dist.ReduceOp.SUM) if self.dist else x


# which pipe a conv family runs on (DESIGN.md section 3) and how many tensor-core passes one algorithmic FLOP costs there
def family_pipe(tag: str, mma: bool, prec: dict):
    if not mma:
        return "fp32_fma", 1
    fam = "generator" if tag.startswith("dec") else "front"
    p = prec[fam]
    return {"bf16x3": ("bf16", 3), "f16x3": ("bf16", 3), "tf32x3": ("tf32", 3)}[p]


def lib_sha16() -> str:
    from piper_b200 import _lib
    return hashlib.sha256(open(_lib.LIB_PATH, "rb").read()).hexdigest()[:16]


def kernel_src_sha16() -> str:
    """Hash of the sources that are compiled into libpiper_b200.so (piper_b200/csrc/*.{cu,cuh,inl,h,cc}, Makefile; not shim/)."""
    d = os.path.join(ROOT, "piper_b200", "csrc")
    h = hashlib.sha256()
    for name in sorted(os.listdir(d)):
        if name.endswith((".cu", ".cuh", ".inl", ".h", ".cc")) or name == "Makefile":
            h.update(name.encode())
            h.update(open(os.path.join(d, name), "rb").read())
    h.update(open(os.path.join(ROOT, "include", "piper_b200.h"), "rb").read())
    return h.hexdigest()[:16]


def conv_rooflines(voice, run, prof_steps, peaks, pipe_peaks, prec, config_id=3):
    """CUDA events around every conv launch (engine profile mode), aggregated per family; for each family the HBM
    fraction (algorithmic bytes) and the tensor/FMA-pipe fraction (algorithmic FLOP), and which one binds."""
    voice.set_profile(True)
    agg = {}
    for _ in range(prof_steps):
        run()
        for k, v in voice.profile().items():
            a = agg.setdefault(k, dict(launches=0, ms=0.0, bytes=0.0, flops=0.0))
            for f in a:
                a[f] += v[f]
    voice.set_profile(False)
    total_ms = sum(v["ms"] for v in agg.values())
    fams = {}
    for k, v in agg.items():
        mma = k.endswith(".mma")
        pipe, passes = family_pipe(k, mma, prec)
        pipe_peak = {"bf16": peaks["bf16_tflops"], "tf32": pipe_peaks["tf32_tflops"], "fp32_fma": pipe_peaks["fp32_fma_tflops"]}[pipe]
        gbs = v["bytes"] / (v["ms"] * 1e-3) / 1e9
        tfl = v["flops"] / (v["ms"] * 1e-3) / 1e12
        f_h, f_t = gbs / peaks["hbm_gbs"], tfl / pipe_peak
        # the binding resource is the one whose floor (work / peak) is larger; passes count the split-precision products
        t_h, t_t = v["bytes"] / peaks["hbm_gbs"], passes * v["flops"] / (pipe_peak * 1e3)
        fams[k] = {"launches_per_step": v["launches"] / prof_steps, "ms_per_step": v["ms"] / prof_steps, "gbs": gbs,
                   "tflops": tfl, "pipe": pipe, "passes": passes, "frac_hbm": f_h, "frac_pipe": f_t,
                   "frac_pipe_issued": f_t * passes, "bound": "hbm" if t_h >= t_t else "tensor",
                   "share_of_conv_time": v["ms"] / total_ms}
    dom = max(agg, key=lambda k: agg[k]["ms"])
    d, f = agg[dom], fams[dom]
    bound = f["bound"]
    roofline = {
        "kernel": dom, "bound": bound,
        "achieved": f["gbs"] if bound == "hbm" else f["tflops"] * f["passes"],
        "peak": peaks["hbm_gbs"] if bound == "hbm" else {"bf16": peaks["bf16_tflops"], "tf32": pipe_peaks["tf32_tflops"],
                                                          "fp32_fma": pipe_peaks["fp32_fma_tflops"]}[f["pipe"]],
        "unit": "GB/s" if bound == "hbm" else "TFLOP/s",
        "frac": f["frac_hbm"] if bound == "hbm" else f["frac_pipe_issued"],
        "frac_hbm": f["frac_hbm"], "frac_pipe": f["frac_pipe"],
        "traffic": None, "peak_source": peaks["source"], "pipe_peaks_measured_in_run": pipe_peaks,
        "avg_launch_us": d["ms"] / d["launches"] * 1e3, "launches_per_step": d["launches"] / prof_steps,
        "algorithmic_bytes_per_launch": d["bytes"] / d["launches"], "algorithmic_flop_per_launch": d["flops"] / d["launches"],
        "share_of_conv_time": d["ms"] / total_ms, "conv_ms_per_step": total_ms / prof_steps,
        "note": "achieved = algorithmic bytes (or FLOP x split-precision passes) / CUDA-event time of the family's launches; "
                "per-family fractions against both resources in `families`",
        "families": fams,
    }
    # dram__bytes per launch from an `ncu --set full` capture: only when it was taken on THIS build of the library
    tpath = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if os.path.exists(tpath):
        t = json.load(open(tpath))
        # (the library file's hash, or - a rebuild of the same sources need not be byte-identical - the hash of the sources
        # that go into it)
        same_build = t.get("lib_sha16") == lib_sha16() or (t.get("src_sha16") and t.get("src_sha16") == kernel_src_sha16())
        if same_build and t.get("config", 3) == config_id:      # (the capture is of one configuration's launches)
            roofline["traffic"] = t.get("families", {}).get(dom, {}).get("dram_bytes_per_launch")
            roofline["traffic_source"] = t.get("source")
    return roofline


def time_to_first_chunk(voice, ids, reps=7):
    """SpeechStreamer.stream (the reference's streaming loop, infer_onnx_streaming.py:76-124): wall time from the call to
    the first audio chunk on the host, and to the last."""
    from piper_b200 import streaming
    st = streaming.SpeechStreamer(voice, 45, 10)
    first, total, n_chunks = [], [], 0
    for r in range(reps + 2):
        t0 = time.perf_counter()
        t_first, n = None, 0
        for piece in st.stream(ids, SCALES, seed=1):
            if t_first is None:
                t_first = time.perf_counter() - t0
            n += 1
        if r >= 2:
            first.append(t_first); total.append(time.perf_counter() - t0); n_chunks = n
    return {"time_to_first_chunk_ms": statistics.median(first) * 1e3, "all_chunks_ms": statistics.median(total) * 1e3,
            "chunks": n_chunks, "chunk_frames": 45, "halo_frames": 10,
            "path": "SpeechStreamer.stream: pb200_encode once, pb200_decode per chunk (host z_p slices in, host audio out)"}


def batch1_latency(voice, ids, reps=10):
    one = [ids]
    for _ in range(3):
        voice.synthesize_batch(one, SCALES, seed=1, copy=False)
    lat, n1 = [], 0
    for _ in range(reps):
        t = time.perf_counter()
        flat, counts, _ = voice.synthesize_batch(one, SCALES, seed=1, copy=False)
        lat.append(time.perf_counter() - t); n1 = int(counts.sum())
    lat_s = statistics.median(lat)
    return {"latency_ms": lat_s * 1e3, "rtf": lat_s / (n1 / 22050.0), "samples": n1, "samples_per_s": n1 / lat_s,
            "stage_ms": dict(zip(STAGES, voice.stage_times()))}


def engine_precision() -> dict:
    """Split-precision scheme per family as the library is configured (DESIGN.md section 3)."""
    std = os.environ.get("PIPER_B200_V2_PREC", "f16") != "f16" or os.environ.get("PIPER_B200_V2", "2") == "0"
    return {"generator": "bf16x3", "front": "tf32x3"} if std else {"generator": "f16x3", "front": "f16x3"}


def run_engine(args):
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback for the engine arm)")
    D = Dist(torch)
    rank, world, local = D.rank, D.world, D.local
    cfg = CONFIGS[args.config]
    if args.config == 5:
        return run_generator_sweep(args, D, torch)
    from piper_b200 import engine, voicegen
    arch = cfg["arch"]
    if rank == 0:
        path = voicegen.cached_voice(arch)       # rank 0 writes the synthetic voice; others read it after the barrier
    D.barrier()
    path = voicegen.cached_voice(arch)
    if world > 1:
        from piper_b200 import dist as pdist
        voice = pdist.load_voice_broadcast(path, local, rank)     # weights: rank 0 uploads, NCCL broadcast to the rest
    else:
        voice = engine.Voice(path, local)
    ids_list = workload_ids(cfg, rank, world)
    B = len(ids_list)
    steps, warm = args.steps, max(args.warmup, 3)

    # ---------------- device-resident leg (`value`): inputs staged in HBM once, kernels only
    voice.stage(ids_list, SCALES, seed=4242)
    for _ in range(warm):
        voice.run_staged()
    sampler = ClockSampler(local)
    D.barrier()
    if rank == 0:
        sampler.start()
    launches0 = engine.launch_count()
    dev_ms, samples = 0.0, 0
    t0 = time.perf_counter()
    for _ in range(steps):
        n, ms = voice.run_staged()
        dev_ms += ms; samples += n
    D.barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    launches = (engine.launch_count() - launches0) / steps
    clocks = sampler.stop() if rank == 0 else None
    stage_ms = voice.stage_times()
    dev_ms_max = D.max(dev_ms)
    total_samples = D.sum(float(samples))
    value = total_samples / (dev_ms_max * 1e-3)

    # ---------------- end-to-end leg: the public call with HOST buffers, H2D + D2H inside the timed region
    # The reference-facing call returns what piper::synthesize returns: peak-normalised int16 samples (piper.cpp:411-431),
    # here produced on the GPU (pb200_synthesize_int16), so 2 bytes per sample cross PCIe.  The fp32 variant of the same
    # call (pb200_synthesize_batch, 4 bytes per sample) is timed beside it.
    # Both legs run the staged leg's inputs (same ids, scales and noise seed); what the last timed step of each returned
    # to its caller - the concatenated waveforms and the per-utterance sample counts - is what --dump-outputs writes.
    outputs = {}

    def e2e_leg(call, bytes_per_sample, name):
        for _ in range(3):
            call()
        D.barrier()
        t0 = time.perf_counter()
        n = 0
        for _ in range(steps):
            flat, counts, _ = call()
            n += int(counts.sum())
        D.barrier()
        secs = D.max(time.perf_counter() - t0)
        if args.dump_outputs:
            outputs[name] = flat.astype(np.float32)        # a copy: the library reuses its host buffer on the next call
            outputs["samples_per_utterance"] = counts.astype(np.float64)
        return D.sum(float(n)) / secs, secs, n // steps * bytes_per_sample
    e2e_value, e2e_s, d2h_audio = e2e_leg(lambda: voice.synthesize_int16(ids_list, SCALES, seed=4242, copy=False), 2,
                                          "audio_int16")
    e2e_f32, e2e_f32_s, d2h_f32 = e2e_leg(lambda: voice.synthesize_batch(ids_list, SCALES, seed=4242, copy=False), 4,
                                          "audio")
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, outputs)
    tp = (259 + 3) // 4 * 4
    h2d = B * tp * 4 + B * 4 + B * 8 + 24       # ids (int32, padded pitch) + lengths + output offsets + call parameters
    d2h = d2h_audio + B * 4                     # int16 audio + the per-item output lengths

    # ---------------- rooflines per conv family: CUDA events around every launch (profile mode), pipe-correct peaks
    peaks = measured_peaks()
    pipe_peaks = measure_pipe_peaks(torch) if (rank == 0 and not args.quick) else {"tf32_tflops": 1.0, "fp32_fma_tflops": 1.0}
    prec = engine_precision()
    roofline = conv_rooflines(voice, voice.run_staged, 2, peaks, pipe_peaks, prec, args.config)

    # ---------------- batch = 1 latency / real-time factor / time to first streamed chunk (BASELINE.json configs[1])
    b1 = batch1_latency(voice, ids_list[0])
    streaming = time_to_first_chunk(voice, ids_list[0]) if ((args.config == 2 or world == 1) and not args.quick) else None

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and not args.quick:
        th, procs = cpu_plan(cfg)
        utts = 1 if arch == "high" else 2
        v, n, secs = cpu_throughput(args.config, utts, th, procs)
        cpu_baseline = {"value": v, "unit": "samples/s", "cores": th * procs, "threads_per_process": th, "processes": procs,
                        "kind": "port", "host_cpus": os.cpu_count(),
                        "sample": f"{n} utterances (259 ids each) as {procs} concurrent B=1 processes x {th} threads, {secs:.1f} s wall; "
                                  "torch CPU fp32 oracle port of the reference graph (onnxruntime absent)"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "samples/s", "n_gpus": world, "steps": steps,
            "warmup": warm, "ms_per_step": dev_ms_max / steps, "higher_is_better": True,
            "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_text(cfg, world) + ", device Philox noise", "baseline_config": cfg["name"],
                       "batch_per_gpu": B, "ids_per_utterance": 259, "samples_per_step": total_samples / steps,
                       "l2": "working set (4 generator stage buffers of ~0.5 GB per step at batch 32) exceeds the 126 MB L2; no flush needed"
                             if B >= 8 else "batch 1: activations fit in L2, as they do for a real single-utterance caller",
                       "parallelism": f"dp{world} (utterances sharded, no data-path collective)",
                       "precision": f"fp32 I/O and accumulation; conv products on tcgen05 in split precision: generator {prec['generator']}, "
                                    f"flow / encoder / duration predictor {prec['front']}; parity <= 1e-3 vs the fp32 reference"},
            "wall_ms_per_step": wall_ms / steps,
            "stage_ms": dict(zip(STAGES, stage_ms)),
            "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_s / steps * 1e3,
                    "call": "pb200_synthesize_int16: host ids in, host int16 audio out (piper::synthesize's output, piper.cpp:411-431)",
                    "fp32_output": {"value": e2e_f32, "ms_per_step": e2e_f32_s / steps * 1e3, "d2h_bytes_per_step": d2h_f32 + B * 4,
                                    "call": "pb200_synthesize_batch: host fp32 audio out"}},
            "gpu_launches": launches,
            "clocks": clocks,
            "roofline": roofline,
            "cpu_baseline": cpu_baseline,
            "batch1": b1,
            "streaming": streaming,
        }
        if args.config == 2:
            line["rtf"] = b1["rtf"]
        print(json.dumps(line), flush=True)
    voice.close()
    if D.dist:
        D.dist.destroy_process_group()


def run_generator_sweep(args, D, torch):
    """configs[4]: the HiFi-GAN generator alone (pb200_vocode; the reference's harness is src/benchmark/benchmark_generator.py)
    on z ~ N(0,1) [B,192,256], B in {1,8,32,128}: device time of the generator (CUDA events inside the engine), e2e wall of
    the call (host z in, host audio out), algorithmic GB/s against the HBM peak and issued TFLOP/s against the tensor peak."""
    from piper_b200 import engine, voicegen
    rank, world, local = D.rank, D.world, D.local
    arch = args.arch
    if rank == 0:
        voicegen.cached_voice(arch)
    D.barrier()
    voice = engine.Voice(voicegen.cached_voice(arch), local)
    peaks = measured_peaks()
    act, wb, flop = GEN_WORK[arch]
    sweep, clocks = [], None
    for B in (1, 8, 32, 128):
        z = np.random.default_rng(1236 + rank).standard_normal((B, 192, 256)).astype(np.float32)
        for _ in range(max(args.warmup, 3)):
            voice.vocode(z)
        top = B == 128
        sampler = ClockSampler(local)
        D.barrier()
        if rank == 0 and top:
            sampler.start()
        dev_ms, t0 = 0.0, time.perf_counter()
        launches0 = engine.launch_count()
        for _ in range(args.steps):
            audio, _ = voice.vocode(z)
            dev_ms += voice.stage_times()[4]
        D.barrier()
        wall = D.max(time.perf_counter() - t0)
        launches = (engine.launch_count() - launches0) / args.steps
        if rank == 0 and top:
            clocks = sampler.stop()
            if args.dump_outputs:                        # the headline batch's waveforms [B, 65536] of the last step
                dump_outputs(args.dump_outputs, {"audio": audio})
        ms = D.max(dev_ms) / args.steps
        n = B * 256 * voice.hop
        gbs = (act * B + wb) / (ms * 1e-3) / 1e9
        tfl = flop * B / (ms * 1e-3) / 1e12
        t_h, t_t = (act * B + wb) / peaks["hbm_gbs"], 3 * flop * B / (peaks["bf16_tflops"] * 1e3)
        sweep.append({"B": B, "device_ms": ms, "samples_per_s": world * n / (ms * 1e-3), "e2e_samples_per_s": world * n * args.steps / wall,
                      "gbs_per_gpu": gbs, "frac_hbm": gbs / peaks["hbm_gbs"], "tflops_algorithmic_per_gpu": tfl,
                      "frac_tensor_issued": 3 * tfl / peaks["bf16_tflops"], "bound": "hbm" if t_h >= t_t else "tensor",
                      "launches": launches, "h2d_bytes": z.nbytes, "d2h_bytes": n * 4})
    if rank == 0:
        top = sweep[-1]
        bound = top["bound"]
        print(json.dumps({
            "metric": METRIC, "value": top["samples_per_s"], "unit": "samples/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": top["device_ms"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"generator only ({arch} decoder, seeded synthetic weights): z ~ N(0,1) [B,192,256] -> [B,65536], "
                                   f"B swept over 1/8/32/128 per GPU; headline = B 128", "baseline_config": CONFIGS[5]["name"],
                       "l2": "B >= 8 working sets exceed the 126 MB L2", "parallelism": f"dp{world} (replicas, no collective)",
                       "precision": "bf16x3 split precision on tcgen05, fp32 I/O"},
            "e2e": {"value": top["e2e_samples_per_s"], "unit": "samples/s", "h2d_bytes_per_step": top["h2d_bytes"],
                    "d2h_bytes_per_step": top["d2h_bytes"]},
            "gpu_launches": top["launches"], "clocks": clocks,
            "roofline": {"kernel": "generator (all launches of pb200_vocode)", "bound": bound,
                         "achieved": top["gbs_per_gpu"] if bound == "hbm" else 3 * top["tflops_algorithmic_per_gpu"],
                         "peak": peaks["hbm_gbs"] if bound == "hbm" else peaks["bf16_tflops"],
                         "unit": "GB/s" if bound == "hbm" else "TFLOP/s",
                         "frac": top["frac_hbm"] if bound == "hbm" else top["frac_tensor_issued"], "traffic": None,
                         "frac_hbm": top["frac_hbm"], "frac_tensor_issued": top["frac_tensor_issued"], "peak_source": peaks["source"]},
            "cpu_baseline": None, "sweep": sweep,
        }), flush=True)
    voice.close()
    if D.dist:
        D.dist.destroy_process_group()


def _claim_stdout():
    """Libraries (NCCL prints its version banner) write to fd 1; the driver wants exactly one JSON line there.
    Point fd 1 at stderr for the duration of the run and return a file object on the real stdout."""
    sys.stdout.flush()
    real = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    return real


def main():
    global print
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference", "cpu-worker"])
    ap.add_argument("--config", type=int, default=3, choices=sorted(CONFIGS))
    ap.add_argument("--arch", default="medium", choices=["medium", "high"], help="decoder of the generator sweep (config 5)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--quick", action="store_true", help="developer A/B runs: no pipe-peak measurement, streaming leg or CPU baseline")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed path returned in its last step to DIR/<name>.npy "
                    "(float32 / float64, at most 64 MB; seeded inputs, so runs of two builds compare output for output)")
    ap.add_argument("--cpu-worker", type=int, default=0)
    ap.add_argument("--cpu-utts", type=int, default=2)
    ap.add_argument("--cpu-threads", type=int, default=8)
    args = ap.parse_args()
    if args.impl == "cpu-worker":
        return cpu_worker(args)
    _real_stdout = _claim_stdout()
    _print = print

    def print(*a, **k):     # noqa: A001 - every print in this file goes to the real stdout
        k.setdefault("file", _real_stdout)
        _print(*a, **k)
        _real_stdout.flush()

    if args.impl == "reference":
        run_reference(args)
    else:
        run_engine(args)


if __name__ == "__main__":
    main()
