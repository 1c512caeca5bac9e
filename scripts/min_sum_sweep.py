"""FER, mean iterations and device-resident speed of the fp32 normalized min-sum rule against fp64 and fp32-fast, on the
N = 10240 benchmark code with the reference's own frames (trial seeds from Xoshiro256++(777), offset by the point's index as
the sweep draws them, keys from the device generator), plus one N = 100 000 PEG point that runs through the streaming decoder.

Per variant and QBER point: FER (1 - keys-match ratio) with its Clopper-Pearson 95 % interval, mean iterations, frames/s and
frame-iterations/s of qlb_reconcile_device timed with CUDA events over `--reps` launches after one warm-up launch (keys stay
on the device), and the agreement with a CPU restatement on the first `--sample` frames: min-sum against the min-sum
restatement (tests/min_sum_restatement.c; every outcome must be equal), fp64 and fp32-fast against the fp64 restatement
(oracle/restatement).
usage: python scripts/min_sum_sweep.py [--frames 10000] [--sample 256] [--out min_sum_sweep.md]
(the committed run: profiles/r04_min_sum_sweep.md)"""
import argparse
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch
from scipy.stats import beta

ROOT = Path(__file__).resolve().parents[1]
sys.path[:0] = [str(ROOT), str(ROOT / "tests")]
from min_sum_restatement import MinSumRestatement  # noqa: E402
from oracle.bindings import Graph, Restatement  # noqa: E402
from qkd_ldpc_b200 import capi, codes, workload  # noqa: E402

GRID = [0.03, 0.04, 0.05, 0.06, 0.07, 0.08, 0.0825, 0.085, 0.0875, 0.09, 0.1, 0.11]
VARIANTS = [("fp64", dict(precision=64)), ("fp32-fast", dict(precision=32, fast_math=True))] + [
    (f"min-sum a={a:g}", dict(precision=32, min_sum_scale=a)) for a in (1.0, 0.875, 0.8125, 0.75, 0.625)]
MAX_IT = 100


def ci95(k, n):
    lo = 0.0 if k == 0 else beta.ppf(0.025, k, n - k + 1)
    hi = 1.0 if k == n else beta.ppf(0.975, k + 1, n - k)
    return lo, hi


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name(0) + ", power limit not readable"


def run_point(ctx, code, mat, g, orc, msr, name, kw, q, seeds, reps, sample):
    dev = torch.device("cuda", 0)
    frames = seeds.size
    p = capi.make_params(kw["precision"], MAX_IT, 100.0, True, fast_math=kw.get("fast_math", False),
                         min_sum_scale=kw.get("min_sum_scale"))
    d_seeds = torch.from_numpy(seeds.view(np.int64)).to(dev)
    d_a = torch.zeros((frames, code.words_n), dtype=torch.int32, device=dev)
    d_b = torch.zeros_like(d_a)
    torch.cuda.synchronize()
    ex = ctx.generate_device(mat.n, frames, d_seeds.data_ptr(), q, d_a.data_ptr(), d_b.data_ptr())
    d_lp = torch.full((frames,), workload.log_prior(ex), dtype=torch.float64, device=dev)
    d_it = torch.zeros(frames, dtype=torch.int32, device=dev)
    d_res = torch.zeros(frames, dtype=torch.uint8, device=dev)
    args = (code, p, frames, d_a.data_ptr(), d_b.data_ptr(), d_lp.data_ptr(), d_it.data_ptr(), d_res.data_ptr())
    ctx.reconcile_device(*args)  # warm-up
    ctx.synchronize()
    decoder = ctx.last_decoder
    ctx.timer_start()
    for _ in range(reps):
        ctx.reconcile_device(*args)
    ms = ctx.timer_stop()
    it = d_it.cpu().numpy().view(np.uint32).astype(np.int64)
    res = d_res.cpu().numpy()
    fails = int(frames - ((res >> 1) & 1).sum())
    s = seeds[:sample]
    if "min_sum_scale" in kw:
        want = msr.run_trials(g, q, s, kw["min_sum_scale"], threads=16, max_it=MAX_IT)
    else:
        want = orc.run_trials(g, q, s, threads=16, max_it=MAX_IT)
    same = (it[:sample] == want[:, 0]) & ((res[:sample] & 1) == want[:, 1]) & (((res[:sample] >> 1) & 1) == want[:, 2])
    sec = ms / 1e3 / reps
    return dict(variant=name, n=mat.n, q=q, frames=frames, fer=fails / frames, ci=ci95(fails, frames), mean_it=it.mean(),
                fps=frames / sec, fips=it.sum() / sec, agree=int(same.sum()), sample=int(s.size), decoder=decoder)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=10000)
    ap.add_argument("--sample", type=int, default=256)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--big-frames", type=int, default=2048)
    ap.add_argument("--out", default="min_sum_sweep.md")
    a = ap.parse_args()
    ctx = capi.Context(0)
    orc, msr = Restatement(), MinSumRestatement()
    who = card()
    rows = []
    t0 = time.time()
    mat = codes.load_npz(codes.NORTH_STAR)
    g = Graph(mat.n, mat.m, mat.row_ptr, mat.col_idx, mat.col_ptr, mat.row_idx)
    code = capi.Code.from_graph(mat)
    seeds = orc.trial_seeds(777, a.frames)
    for pt, q in enumerate(GRID):
        for name, kw in VARIANTS:
            rows.append(run_point(ctx, code, mat, g, orc, msr, name, kw, q, seeds + np.uint64(pt), a.reps, a.sample))
            print(rows[-1], flush=True)
    big = codes.load_npz("peg_n100000_m51080_cw3_seed666_bfs2000")
    gb = Graph(big.n, big.m, big.row_ptr, big.col_idx, big.col_ptr, big.row_idx)
    cb = capi.Code.from_graph(big)
    for name, kw in VARIANTS:
        rows.append(run_point(ctx, cb, big, gb, orc, msr, name, kw, 0.08, orc.trial_seeds(777, a.big_frames), a.reps, 16))
        print(rows[-1], flush=True)
    lines = [f"# fp32 normalized min-sum against fp64 and fp32-fast ({who}; nvidia-smi name, power limit, max SM clock)", "",
             f"Reference frames: seeds Xoshiro256++(777) + point index, keys from the device generator; max_it {MAX_IT}, clamp 100. "
             f"Speed: qlb_reconcile_device, CUDA events over {a.reps} launches after one warm-up; frame-iterations/s = executed "
             "iterations / time. Agreement: frames whose (iterations, syndromes_match, keys_match) equal the CPU restatement's "
             "(min-sum: tests/min_sum_restatement.c, exact by contract; fp64 / fp32-fast: the fp64 restatement).", "",
             "| N | QBER | variant | frames | FER | FER 95 % CI | mean it | frames/s | frame-it/s | agree | decoder |",
             "|---|---|---|---|---|---|---|---|---|---|---|"]
    for r in rows:
        lines.append(f"| {r['n']} | {r['q']:g} | {r['variant']} | {r['frames']} | {r['fer']:.4g} | [{r['ci'][0]:.3g}, {r['ci'][1]:.3g}] | "
                     f"{r['mean_it']:.2f} | {r['fps']:.4g} | {r['fips']:.4g} | {r['agree']}/{r['sample']} | {r['decoder']} |")
    lines += ["", f"Wall time {time.time() - t0:.0f} s."]
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text("\n".join(lines) + "\n")
    print("\n".join(lines))


if __name__ == "__main__":
    main()
