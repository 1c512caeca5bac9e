"""Rate-adaptive reconciliation on the N = 10240 benchmark code (M = 5231, R0 = 0.489): for fp32 normalized min-sum (alpha = 0.8125)
and fp32 sum-product, modulated fraction delta = 0.1 and target efficiency f* in {1.1, 1.2}, per QBER point 0.03 ... 0.09:
the sweep's (p, s) split, the effective rate, FER (1 - keys-match ratio), mean iterations, the achieved efficiency
(M - p) / (n h2(q)) -- q the exact ratio over the n key bits -- and frames/s of qlb_run_trials_adapted, next to plain qlb_run_trials
(syndrome coding with all N bits, efficiency M / (N h2(q))) on the same code, rule and trial seeds. Frames/s are host wall time
around the call (keys drawn on the device, 8 B up and 5 B down per frame), after one warm-up call of each shape.

A second part times the kernels of one qlb_run_trials_adapted call with torch.profiler: key generation, fill, embed, syndrome,
decode and key extraction, so the cost of the rate adaptation itself is a measured figure.
usage: python scripts/rate_adaptive_sweep.py [--frames 65536] [--out rate_adaptive.md]
(the committed run: profiles/r06_rate_adaptive.md)"""
import argparse
import math
import subprocess
import sys
import time
from collections import defaultdict
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path[:0] = [str(ROOT), str(ROOT / "tests")]
from qkd_ldpc_b200 import capi, codes, workload  # noqa: E402
from test_rate_pattern import effective_rate, policy  # noqa: E402

GRID = [0.03, 0.04, 0.05, 0.06, 0.07, 0.08, 0.09]
RULES = [("min-sum a=0.8125", dict(min_sum_scale=0.8125)), ("fp32", {})]
DELTA, TARGETS, PATTERN_SEED, MAX_IT = 0.1, (1.1, 1.2), 5, 100


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name(0) + ", power limit not readable"


def h2(q):
    return -q * math.log2(q) - (1 - q) * math.log2(1 - q)


def timed(f):
    f()  # warm-up of this shape
    t0 = time.perf_counter()
    out = f()
    return out, time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=65536)
    ap.add_argument("--out", default="rate_adaptive.md")
    a = ap.parse_args()
    mat = codes.load_npz(codes.NORTH_STAR)
    code, ctx = capi.Code.from_graph(mat), capi.Context(0)
    seeds = workload.trial_seeds(777, a.frames)
    lines = [f"# Rate-adaptive reconciliation, N = {mat.n}, M = {mat.m}", "", f"card: {card()}", "",
             f"{a.frames} frames per point (trial seeds of Xoshiro256++(777) + point index), max_iterations {MAX_IT}, clamp 100, "
             f"delta = {DELTA}, pattern seed {PATTERN_SEED}. f = achieved efficiency; plain = qlb_run_trials with all N bits.", ""]
    for rule, kw in RULES:
        params = capi.make_params(32, MAX_IT, 100.0, True, **kw)
        for target in TARGETS:
            lines += [f"## {rule}, f* = {target}", "",
                      "| QBER | p | s | n | R | FER | mean it | f | frames/s | plain FER | plain mean it | plain f | plain frames/s |",
                      "|---|---|---|---|---|---|---|---|---|---|---|---|---|"]
            for pt, q in enumerate(GRID):
                p, s = policy(mat.n, mat.m, q, DELTA, target)
                n = mat.n - p - s
                cls = capi.rate_pattern(code, p, s, PATTERN_SEED)
                (it, res, ex), sec = timed(lambda: ctx.run_trials_adapted(code, params, cls, seeds, q, seed_offset=pt))
                (it0, res0, ex0), sec0 = timed(lambda: ctx.run_trials(code, params, seeds, q, seed_offset=pt))
                fer, fer0 = 1 - ((res >> 1) & 1).mean(), 1 - ((res0 >> 1) & 1).mean()
                lines.append(f"| {q:.2f} | {p} | {s} | {n} | {effective_rate(mat, p, s):.4f} | {fer:.4g} | {it.mean():.2f} | "
                             f"{(mat.m - p) / (n * h2(ex)):.3f} | {a.frames / sec:.4g} | {fer0:.4g} | {it0.mean():.2f} | "
                             f"{mat.m / (mat.n * h2(ex0)):.3f} | {a.frames / sec0:.4g} |")
                print(lines[-1], flush=True)
            lines.append("")

    # kernel times of one rate-adapted call (torch.profiler, CUDA activities; a run of its own after the timed sweep)
    from torch.profiler import ProfilerActivity, profile
    lines += ["## Kernel times of one qlb_run_trials_adapted call", ""]
    for rule, kw in RULES:
        params = capi.make_params(32, MAX_IT, 100.0, True, **kw)
        p, s = policy(mat.n, mat.m, 0.05, DELTA, 1.1)
        cls = capi.rate_pattern(code, p, s, PATTERN_SEED)
        ctx.run_trials_adapted(code, params, cls, seeds, 0.05)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            ctx.run_trials_adapted(code, params, cls, seeds, 0.05)
        us = defaultdict(float)
        for e in prof.events():
            if e.device_type.name == "CUDA":
                name = e.name.split("<")[0].split("(")[0].replace("void ", "").replace("qlb::", "")
                us[name] += e.device_time if hasattr(e, "device_time") else e.cuda_time
        total = sum(us.values())
        lines += [f"{rule}, QBER 0.05, p = {p}, s = {s}, {a.frames} frames: {total / 1e3:.3f} ms of kernels", "",
                  "| kernel | ms | share |", "|---|---|---|"]
        lines += [f"| {k} | {v / 1e3:.3f} | {v / total:.1%} |" for k, v in sorted(us.items(), key=lambda kv: -kv[1])]
        lines.append("")
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text("\n".join(lines) + "\n")
    print("\n".join(lines))


if __name__ == "__main__":
    main()
