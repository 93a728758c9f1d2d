"""CPU emulation behind DESIGN.md §3 (no GPU needed; needs the real test voice, i.e. /root/reference or oracle/_ref).

Part 1 — which split-precision scheme does each layer family tolerate?  Products are formed exactly (fp64 accumulate)
from operands rounded like the tensor core sees them: single-pass TF32, bf16x3 (hi*hi + hi*lo + lo*hi), tf32x3.
Part 2 — the tensor core adds into its fp32 accumulator with truncation (round toward zero): emulate that per k-step
and evaluate the two mitigations against it (separate correction accumulator, K split into chains; conv2_body.inl keeps
a correction accumulator per K-chain).

Part 3 - FP16 operands: hi = fp16(x), lo = fp16(x - hi) keeps 22 mantissa bits at kind::f16's K = 16 per instruction,
i.e. tf32x3-class accuracy at bf16x3 cost (conv2_body.inl PREC_F16); with the accumulator truncation emulated as well.

usage: python tools/precision_study.py [part1|part2|part3|all]  > profiles/r01_precision_study.txt
"""
import json, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np, torch, torch.nn.functional as F
from oracle.voice_loader import load_voice
from oracle.vits_oracle import Oracle
from piper_b200 import voicegen

torch.set_num_threads(min(8, os.cpu_count() or 1))


def bf16(x): return x.to(torch.bfloat16).to(torch.float32)


def tf32(x):            # round to nearest (ties away), 10 explicit mantissa bits: cvt.rna.tf32.f32
    i = x.contiguous().view(torch.int32)
    return ((i + 0x1000) & ~0x1FFF).view(torch.float32)


def rz32(x64):          # fp64 -> fp32 with truncation toward zero (what the accumulator add does)
    f = x64.float()
    over = f.double().abs() > x64.abs()
    return torch.where(over, torch.nextafter(f, torch.zeros_like(f)), f)


class SplitOracle(Oracle):
    mode, scope = "bf16x3", ("dec.",)

    def conv(self, x, name, dilation=1, pad=0, groups=1):
        if groups != 1 or not name.startswith(self.scope):
            return super().conv(x, name, dilation, pad, groups)
        w, b = self.w[name + ".weight"], self.w.get(name + ".bias")
        cv = lambda a, ww: F.conv1d(a[None].double(), ww.double(), None, dilation=dilation, padding=pad)[0]
        r = {"bf16": bf16, "tf32": tf32}[self.mode[:4]]
        xh, wh = r(x), r(w)
        if self.mode.endswith("x1"):
            y = cv(xh, wh)
        else:
            xl, wl = r(x - xh), r(w - wh)
            y = cv(xh, wh) + cv(xh, wl) + cv(xl, wh)
        y = y.float()
        return y if b is None else y + b[:, None]


class RZOracle(Oracle):
    """tf32x3 with the accumulator truncation of the hardware, 8 channels per k-step, taps outer."""
    scope, sep_corr, chains = ("flow.",), False, 1

    def conv(self, x, name, dilation=1, pad=0, groups=1):
        if groups != 1 or not name.startswith(self.scope):
            return super().conv(x, name, dilation, pad, groups)
        w, b = self.w[name + ".weight"], self.w.get(name + ".bias")
        co, ci, k = w.shape
        xp = F.pad(x, (pad, pad))
        T = x.shape[1]
        xh, wh = tf32(xp), tf32(w)
        xl, wl = xp - xh, w - wh
        steps = [(j, kb) for j in range(k) for kb in range(0, ci, 8)]
        per_chain = -(-len(steps) // self.chains)
        total, acc, corr = torch.zeros(T, co), torch.zeros(T, co), torch.zeros(T, co)
        for s, (j, kb) in enumerate(steps):
            sl = slice(kb, kb + 8)
            a_h = xh[sl, j * dilation:j * dilation + T].t().double()
            a_l = xl[sl, j * dilation:j * dilation + T].t().double()
            w_h, w_l = wh[:, sl, j].double(), wl[:, sl, j].double()
            acc = rz32(acc.double() + a_h @ w_h.t())
            if self.sep_corr:
                corr = rz32(rz32(corr.double() + a_h @ w_l.t()).double() + a_l @ w_h.t())
            else:
                acc = rz32(rz32(acc.double() + a_h @ w_l.t()).double() + a_l @ w_h.t())
            if (s + 1) % per_chain == 0 or s == len(steps) - 1:
                total, acc = total + acc, torch.zeros(T, co)
        y = (total + corr).t().contiguous()
        return y if b is None else y + b[:, None]


def f16(x): return x.to(torch.float16).to(torch.float32)


class F16Oracle(Oracle):
    """hi*hi + hi*lo + lo*hi with FP16 operands, exact accumulation."""
    scope = ("flow.",)

    def conv(self, x, name, dilation=1, pad=0, groups=1):
        if groups != 1 or not name.startswith(self.scope):
            return super().conv(x, name, dilation, pad, groups)
        w, b = self.w[name + ".weight"], self.w.get(name + ".bias")
        cv = lambda a, ww: F.conv1d(a[None].double(), ww.double(), None, dilation=dilation, padding=pad)[0]
        xh, wh = f16(x), f16(w)
        xl, wl = f16(x - xh), f16(w - wh)
        y = (cv(xh, wh) + (cv(xh, wl) + cv(xl, wh))).float()
        return y if b is None else y + b[:, None]


class F16RZOracle(Oracle):
    """FP16 operands, 16 channels per k-step, truncating fp32 accumulation, one (main | correction) pair per K-chain."""
    scope, chains = ("flow.",), 2

    def conv(self, x, name, dilation=1, pad=0, groups=1):
        if groups != 1 or not name.startswith(self.scope):
            return super().conv(x, name, dilation, pad, groups)
        w, b = self.w[name + ".weight"], self.w.get(name + ".bias")
        co, ci, k = w.shape
        xp = F.pad(x, (pad, pad))
        T = x.shape[1]
        xh, wh = f16(xp), f16(w)
        xl, wl = f16(xp - xh), f16(w - wh)
        steps = [(j, kb) for j in range(k) for kb in range(0, ci, 16)]
        per_chain = -(-len(steps) // self.chains)
        total, acc, corr = torch.zeros(T, co), torch.zeros(T, co), torch.zeros(T, co)
        for s, (j, kb) in enumerate(steps):
            sl = slice(kb, kb + 16)
            a_h = xh[sl, j * dilation:j * dilation + T].t().double()
            a_l = xl[sl, j * dilation:j * dilation + T].t().double()
            w_h, w_l = wh[:, sl, j].double(), wl[:, sl, j].double()
            acc = rz32(acc.double() + a_h @ w_h.t())
            corr = rz32(rz32(corr.double() + a_h @ w_l.t()).double() + a_l @ w_h.t())
            if (s + 1) % per_chain == 0 or s == len(steps) - 1:
                total, acc, corr = total + acc + corr, torch.zeros(T, co), torch.zeros(T, co)
        y = total.t().contiguous()
        return y if b is None else y + b[:, None]


def real_voice():
    for p in ("/root/reference/etc/test_voice.onnx", os.path.join(ROOT, "oracle", "_ref", "voice", "test_voice.onnx")):
        if os.path.exists(p):
            return p, [json.loads(l) for l in open(os.path.join(os.path.dirname(p), "test_sentences", "test_en-us.jsonl")
                                                   if os.path.exists(os.path.join(os.path.dirname(p), "test_sentences"))
                                                   else os.path.join(os.path.dirname(p), "test_en-us.jsonl"))]
    raise SystemExit("real test voice not found")


def part1():
    path, lines = real_voice()
    cases = [("real x-low voice", path, lines[2]["phoneme_ids"]),
             ("synthetic medium", voicegen.cached_voice("medium"), voicegen.benchmark_ids(64))]
    for tag, p, ids in cases:
        s, w, a = load_voice(p)
        rng = np.random.default_rng(4)
        eps_dp = rng.standard_normal((2, len(ids))).astype(np.float32)
        eps_z = rng.standard_normal((s.inter, 6 * len(ids))).astype(np.float32)
        d0 = {}
        ref = Oracle(s, w, a).infer(ids, (0.667, 1, 0.8), eps_dp, eps_z, dump=d0)
        for scope in (("dec.",), ("flow.",), ("enc_p.",)):
            for mode in ("tf32x1", "bf16x3", "tf32x3"):
                o = SplitOracle(s, w, a)
                o.mode, o.scope = mode, scope
                d = {}
                out = o.infer(ids, (0.667, 1, 0.8), eps_dp, eps_z, dump=d)
                same = np.array_equal(d["w_ceil"].numpy(), d0["w_ceil"].numpy())
                err = float(np.abs(out - ref).max()) if out.shape == ref.shape else float("nan")
                print(f"{tag:18s} {scope[0]:7s} {mode:7s} durations_equal={same} max|audio err|={err:.3e}", flush=True)


def part2():
    path, lines = real_voice()
    ids = lines[4]["phoneme_ids"]
    s, w, a = load_voice(path)
    rng = np.random.default_rng(1235)
    eps_dp = rng.standard_normal((2, len(ids))).astype(np.float32)
    eps_z = rng.standard_normal((s.inter, 3 * len(ids))).astype(np.float32)
    d0 = {}
    ref = Oracle(s, w, a).infer(ids, (0.667, 1, 0.8), eps_dp, eps_z, dump=d0)
    for sep, chains in ((False, 1), (True, 1), (True, 2), (True, 3), (True, 8)):
        o = RZOracle(s, w, a)
        o.sep_corr, o.chains = sep, chains
        d = {}
        out = o.infer(ids, (0.667, 1, 0.8), eps_dp, eps_z, dump=d)
        print(f"real x-low voice, flow tf32x3 with RZ accumulation: separate_correction={sep} chains={chains} "
              f"max|audio err|={np.abs(out - ref).max():.3e} max|z err|={float((d['z'] - d0['z']).abs().max()):.3e}", flush=True)


def part3():
    path, lines = real_voice()
    cases = [("real x-low voice", path, lines[2]["phoneme_ids"]),
             ("synthetic medium", voicegen.cached_voice("medium"), voicegen.benchmark_ids(64))]
    for tag, p, ids in cases:
        s, w, a = load_voice(p)
        rng = np.random.default_rng(4)
        eps_dp = rng.standard_normal((2, len(ids))).astype(np.float32)
        eps_z = rng.standard_normal((s.inter, 6 * len(ids))).astype(np.float32)
        d0 = {}
        ref = Oracle(s, w, a).infer(ids, (0.667, 1, 0.8), eps_dp, eps_z, dump=d0)
        for scope in (("dec.",), ("flow.",), ("enc_p.",), ("dp.",)):
            o = F16Oracle(s, w, a)
            o.scope = scope
            d = {}
            out = o.infer(ids, (0.667, 1, 0.8), eps_dp, eps_z, dump=d)
            same = np.array_equal(d["w_ceil"].numpy(), d0["w_ceil"].numpy())
            err = float(np.abs(out - ref).max()) if out.shape == ref.shape else float("nan")
            print(f"{tag:18s} {scope[0]:7s} fp16x3  durations_equal={same} max|audio err|={err:.3e}", flush=True)
    ids = lines[4]["phoneme_ids"]
    s, w, a = load_voice(path)
    rng = np.random.default_rng(1235)
    eps_dp = rng.standard_normal((2, len(ids))).astype(np.float32)
    eps_z = rng.standard_normal((s.inter, 3 * len(ids))).astype(np.float32)
    ref = Oracle(s, w, a).infer(ids, (0.667, 1, 0.8), eps_dp, eps_z)
    for chains in (1, 2):
        o = F16RZOracle(s, w, a)
        o.chains = chains
        out = o.infer(ids, (0.667, 1, 0.8), eps_dp, eps_z)
        print(f"real x-low voice, flow fp16x3 (K = 16 per step) with RZ accumulation: chains={chains} "
              f"max|audio err|={np.abs(out - ref).max():.3e}", flush=True)


if __name__ == "__main__":
    what = sys.argv[1] if len(sys.argv) > 1 else "all"
    if what in ("part1", "all"):
        part1()
    if what in ("part2", "all"):
        part2()
    if what in ("part3", "all"):
        part3()
