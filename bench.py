#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on BASELINE.json's config, one JSON line on stdout.

Metric   : decoded frames/s (and sifted-key Mbit/s = frames/s * N / 1e6) over the QBER sweep 0.03 ... 0.11 of the
           N=10240, M=5231, CW=3 code (configs[1]); FER per point reported beside it.
Frames   : the REFERENCE'S OWN frames -- trial k of sweep point pt is seeded with seeds[k] + pt, seeds = the raw draws of
           Xoshiro256PlusPlus(777) (src/simulation.cpp:222-228,247), and the keys are re-created on the GPU by the bit-exact
           generator (qlb_generate_device) before the timed region. The CPU sample (`cpu_baseline`) runs the reference's
           run_trial on the first trials of the same seeds, so `parity` counts frame-by-frame agreement on this very record.
A "step" : one pass of the hot path over one batch = the whole 9-point sweep, `--frames-per-point` frames per point
           per GPU (default 10 000, as configs[1]), every frame through the fused reconcile kernel
           (Alice syndrome + LLR init + sum-product decode with per-frame early termination + key compare).
dtype    : default --precision f64, the reference's own arithmetic and operation order (the headline is an fp64 / fp64
           comparison); f64fused (one-division fp64 rule), f32 and f32fast are `variants`, each with its own e2e and parity.
value    : whole-job frames/s with the packed keys already resident in HBM (device-timed, max over ranks).
e2e      : the same sweep through the C-ABI call a user makes (qlb_reconcile_batch_packed) with pinned HOST buffers:
           H2D of keys + QBERs and D2H of results inside the timed region.
roofline : the SM-resident kernels keep a frame's messages on the SM, so the roof that binds them is on the SM too: the primary
           figure is instruction issue (ncu-measured warp instructions per frame-iteration x the live frame-iterations/s against
           4 issue slots x SMs x the SM clock sampled under load); the fp64 pipe is given beside it. `algorithmic_hbm` is SURVEY.md
           8d's fixed figure (16 B fp32 / 32 B fp64 per edge-iteration against MEASURED_PEAKS.json's copy bandwidth) -- the number
           north_star's 60 % target refers to -- and `traffic` the DRAM bytes ncu measured for one launch of this bench's own
           shape. `variants.stream_*` are the truly HBM-bound design points (configs[3], N = 100 000 and 1 000 000).
strong   : configs[2]'s shape -- a FIXED total of trials per point sharded over the ranks, through qlb_run_trials (seeds up, keys
           generated on the GPU, results down), statistics from the all-reduced integer histogram.
cpu_baseline / --impl reference : the reference's own CPU implementation (oracle/_ref, the unmodified sources compiled in
           place) on the box's host cores, on a bounded sample of the same sweep.

Launch: `python bench.py --gpus 1 ...` or, for N > 1,
`python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...`
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

MAX_IT = 100
THR = 100.0
SIM_SEED = 777
BYTES_PER_EDGE_IT = {"f32": 16, "f32fast": 16, "f64": 32, "f64fused": 32}
PRECISIONS = ("f64", "f64fused", "f32", "f32fast")


def qber_grid():
    return [0.03 + 0.01 * j for j in range(9)]  # end-exclusive grid of src/simulation.cpp:55-61 for 0.03..0.12 step 0.01


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, iterations, flags):
    """--dump-outputs: what the last timed step returned, for comparing two builds output for output. iterations.npy and
    result_flags.npy (bit 0 syndromes match, bit 1 keys match) are float32 [QBER points x frames]; point_stats.npy is float64
    [points x sweep.PointStats]; frame_index.npy lists the frames kept. Above 64 MB the frames are a fixed, seeded sample."""
    from qkd_ldpc_b200 import sweep
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    points, frames = iterations.shape
    stats = np.zeros((points, MAX_IT + 5), np.float64)
    for pt in range(points):
        ps = sweep.PointStats(MAX_IT)
        ps.add(iterations[pt], flags[pt])
        stats[pt] = ps.vec
    keep = (DUMP_LIMIT_BYTES - stats.nbytes - 4096) // (2 * 4 * points + 8)
    idx = np.arange(frames) if frames <= keep else np.sort(np.random.default_rng(0).choice(frames, keep, replace=False))
    np.save(out / "iterations.npy", iterations[:, idx].astype(np.float32))
    np.save(out / "result_flags.npy", flags[:, idx].astype(np.float32))
    np.save(out / "frame_index.npy", idx.astype(np.float64))
    np.save(out / "point_stats.npy", stats)


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.tmp = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.gpu)], stdout=self.tmp, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.tmp.flush()
        rows = [r.split(",") for r in Path(self.tmp.name).read_text().splitlines() if r.count(",") >= 8]
        os.unlink(self.tmp.name)
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); pw.append(float(r[3]))
            except ValueError:
                continue
            for nm, v in zip(names, r[5:9]):
                if v.strip().lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "power_w_max": float(max(pw)),
                "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline
def cpu_reference_sweep(trials_per_point: int, threads: int, seed: int = 777):
    """The reference's CPU path on this host: run_trial (generate + QKD_LDPC_irregular) for `trials_per_point` trials
    at each of the 9 QBER points, `threads` host threads. Returns (kind, seconds, per-point out3 arrays)."""
    from oracle.bindings import REF_SO, Reference, Restatement
    from qkd_ldpc_b200 import codes
    mats = codes.materialize()
    grid = qber_grid()
    if REF_SO.exists():
        ref = Reference(max_it=MAX_IT, thr=THR, enable_thr=True, threads=threads)
        h = ref.load(mats[codes.NORTH_STAR], dense=False)
        seeds = ref.trial_seeds(seed, trials_per_point)
        run = lambda q, s: ref.run_trials(h, q, s, threads=threads)
        kind = "reference"
    else:
        from oracle.bindings import Graph
        orc = Restatement()
        m = codes.load_npz(codes.NORTH_STAR)
        g = Graph(m.n, m.m, m.row_ptr, m.col_idx, m.col_ptr, m.row_idx)
        seeds = orc.trial_seeds(seed, trials_per_point)
        run = lambda q, s: orc.run_trials(g, q, s, threads=threads)
        kind = "port"
    outs = []
    t0 = time.perf_counter()
    for pt, q in enumerate(grid):
        outs.append(run(q, seeds + np.uint64(pt)))  # trial seed = seeds[k] + curr_sim (src/simulation.cpp:247)
    return kind, time.perf_counter() - t0, outs


def cpu_tpp(args, cores):
    return args.cpu_trials_per_point or max(64, 8 * cores)  # ~4 s wall = ~60 core-seconds per sweep


def run_reference_arm(args, guard):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = os.cpu_count() or 1
    tpp = cpu_tpp(args, cores)
    grid = qber_grid()
    for _ in range(args.warmup):
        cpu_reference_sweep(max(1, tpp // 8), cores)
    times = []
    for _ in range(args.steps):
        kind, sec, outs = cpu_reference_sweep(tpp, cores)
        times.append(sec)
    frames = tpp * len(grid)
    sec = float(np.mean(times))
    value = frames / sec
    fer = [1.0 - float((o[:, 1] * o[:, 2]).mean()) for o in outs]
    sample = (f"each step = {tpp} trials per QBER point x {len(grid)} points = {frames} frames of the workload in `config` (trials 0..{tpp - 1} of every "
              f"point, seeds[k] + point), run_trial = key generation + reconciliation, {cores} host threads; frames/s does not depend on the trial count")
    line = {
        "impl": "reference", "metric": "decoded_frames_per_s", "value": value, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args.frames_per_point, args.precision),  # the workload both arms are quoted on
        "sample": sample, "frames_per_step": frames,
        "sifted_mbit_s": value * 10240 / 1e6,
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "per_qber": [{"qber": q, "fer": f} for q, f in zip(grid, fer)],
        "gpu_launches": 0,
    }
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, np.stack([o[:, 0] for o in outs]), np.stack([o[:, 1] | (o[:, 2] << np.uint64(1)) for o in outs]))
    guard.emit(line)
    return 0


def workload_config(frames_per_point, precision):
    return {
        "workload": "configs[1]: alist (N=10240,M=5231,R=0.49,CW=3,SEED=666) QBER sweep 0.03-0.11 (9 points), "
                    f"{frames_per_point} frames per point per GPU",
        "code": "N=10240 M=5231 E=30720 CW=3", "qber_grid": [round(q, 4) for q in qber_grid()],
        "frames_per_point_per_gpu": frames_per_point, "max_iterations": MAX_IT, "msg_threshold": THR,
        "precision": precision, "frames": f"the reference's own: trial seeds = Xoshiro256PlusPlus({SIM_SEED}) draws, seed + point index (src/simulation.cpp:222-228,247)",
        "parallelism": "trial-sharded (one process per GPU, no data-path collective); the 9 launches of a sweep alternate between two streams of the GPU",
        "l2_policy": "inputs larger than L2 (packed keys of one sweep > 126 MB) and a fresh key set per QBER point",
    }


# ---------------------------------------------------------------------------------------------------------------------
class StdoutGuard:
    """The contract is ONE JSON line on stdout: anything libraries print to fd 1 meanwhile (e.g. NCCL's version banner) is
    sent to stderr, and the line is written to the real stdout at the end."""

    def __init__(self):
        sys.stdout.flush()
        self.real = os.dup(1)
        os.dup2(2, 1)

    def emit(self, line: dict):
        sys.stdout.flush()
        os.write(self.real, (json.dumps(line) + "\n").encode())


def profile_constants():
    """ncu-measured per-launch constants of this round's build (profiles/traffic.json; captured with the bench's own launch shape)."""
    tp = ROOT / "profiles" / "traffic.json"
    try:
        return json.loads(tp.read_text())
    except Exception:
        return {}


def main():
    guard = StdoutGuard()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--frames-per-point", type=int, default=10000)
    ap.add_argument("--precision", default="f64", choices=list(PRECISIONS))
    ap.add_argument("--cpu-trials-per-point", type=int, default=0)
    ap.add_argument("--strong-frames-per-point", type=int, default=200000,
                    help="fixed TOTAL trials per QBER point of the strong-scaling block (configs[2] is 1 000 000)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-variants", action="store_true")
    ap.add_argument("--no-strong", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the per-frame outputs of the last timed step to DIR/*.npy (rank 0; the inputs are fixed by the seeds)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "b200":
        args.warmup = max(args.warmup, 3)

    if args.impl == "reference":
        return run_reference_arm(args, guard)

    import torch
    import torch.distributed as dist
    from qkd_ldpc_b200 import capi, codes, sweep, workload

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    mat = codes.load_npz(codes.NORTH_STAR)
    code = capi.Code.from_graph(mat)
    ctx = capi.Context(local_rank)
    grid = qber_grid()
    fpp = args.frames_per_point
    n, e = mat.n, mat.e
    prof = profile_constants()

    def params_for(prec):
        return capi.make_params(64 if prec.startswith("f64") else 32, MAX_IT, THR, True, fast_math=prec in ("f32fast", "f64fused"))

    # ---- the reference's frames, generated on the GPU before the timed region and resident in HBM ------------------------
    # rank r holds trials [r * fpp, (r + 1) * fpp) of every point; the keys of point pt come from seeds[k] + pt
    strong_total = 0 if args.no_strong else max(args.strong_frames_per_point, world)
    all_seeds = workload.trial_seeds(SIM_SEED, max(fpp * world, strong_total))
    my_seeds = np.ascontiguousarray(all_seeds[rank * fpp:(rank + 1) * fpp])
    d_seeds = torch.from_numpy(my_seeds.view(np.int64)).to(dev)
    keys = []
    for pt, q in enumerate(grid):
        a = torch.empty((fpp, code.words_n), dtype=torch.int32, device=dev)
        b = torch.empty((fpp, code.words_n), dtype=torch.int32, device=dev)
        qe = ctx.generate_device(n, fpp, d_seeds.data_ptr(), q, a.data_ptr(), b.data_ptr(), seed_offset=pt)
        lp = torch.full((fpp,), workload.log_prior(qe), dtype=torch.float64, device=dev)
        keys.append((a, b, lp, qe))
    ctx.synchronize()
    d_it = torch.zeros((len(grid), fpp), dtype=torch.int32, device=dev)
    d_res = torch.zeros((len(grid), fpp), dtype=torch.uint8, device=dev)
    h_it = torch.zeros((len(grid), fpp), dtype=torch.int32).pin_memory()
    h_res = torch.zeros((len(grid), fpp), dtype=torch.uint8).pin_memory()
    torch.cuda.synchronize()
    ext = torch.cuda.ExternalStream(ctx.stream, device=dev)
    # a second context (stream, frame queue) on the same GPU: the points of a sweep alternate between the two streams, so the
    # tail of one point's launch (SMs running out of frames) is filled by the next point's CTAs. Fork / join through events,
    # so that the CUDA events timed() records on ctx's stream still bracket everything.
    ctx_b = capi.Context(local_rank)
    ext_b = torch.cuda.ExternalStream(ctx_b.stream, device=dev)
    launch_order = sorted(range(len(grid)), key=lambda pt: -grid[pt])  # the long (non-converging) points first
    kernel_windows = []  # (start, end) event pairs around the 9 launches of each step, on the launching stream

    def sweep_step(prec, frames=fpp, collect=True):
        """One step on device-resident inputs: 9 launches over the two streams, then results -> host -> statistics."""
        p = params_for(prec)
        fork = torch.cuda.Event(enable_timing=True)
        fork.record(ext)
        ext_b.wait_event(fork)
        for i, pt in enumerate(launch_order):
            a, b, lp, _ = keys[pt]
            (ctx if i % 2 == 0 else ctx_b).reconcile_device(code, p, frames, a.data_ptr(), b.data_ptr(), lp.data_ptr(), d_it[pt].data_ptr(), d_res[pt].data_ptr())
        join = torch.cuda.Event()
        join.record(ext_b)
        ext.wait_event(join)
        done = torch.cuda.Event(enable_timing=True)
        done.record(ext)
        kernel_windows.append((fork, done))
        if not collect:
            return None
        with torch.cuda.stream(ext):
            h_it.copy_(d_it, non_blocking=True)
            h_res.copy_(d_res, non_blocking=True)
        ctx.synchronize()
        stats = np.zeros((len(grid), MAX_IT + 5), np.int64)
        for pt in range(len(grid)):
            ps = sweep.PointStats(MAX_IT)
            ps.add(h_it[pt, :frames].numpy(), h_res[pt, :frames].numpy())
            stats[pt] = ps.vec
        return sweep.allreduce_stats(stats, dev)  # the sweep's only collective (NCCL when world > 1)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """Device time of `steps` calls: CUDA events on the launching stream, bracketed by barrier + synchronize."""
        barrier()
        ctx.timer_start()
        t0 = time.perf_counter()
        out = None
        for _ in range(steps):
            out = fn()
        ms = ctx.timer_stop()
        barrier()
        wall = (time.perf_counter() - t0) * 1e3
        if world > 1:
            t = torch.tensor([ms, wall], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms, wall = float(t[0]), float(t[1])
        return ms, wall, out

    prec = args.precision
    for _ in range(args.warmup):
        sweep_step(prec)
    sampler = ClockSampler(local_rank)
    sampler.start()
    ctx.counters(reset=True)
    ctx_b.counters(reset=True)
    kernel_windows.clear()
    ms_total, wall_total, stats = timed(lambda: sweep_step(prec), args.steps)
    launches, frame_iters = (x + y for x, y in zip(ctx.counters(reset=True), ctx_b.counters(reset=True)))
    clocks = sampler.stop()
    kern_ms_step = sum(s0.elapsed_time(s1) for s0, s1 in kernel_windows) / args.steps  # the decode launches as the step runs them
    ms_step = ms_total / args.steps
    frames_step = fpp * len(grid) * world
    value = frames_step / (ms_step * 1e-3)
    results = [sweep.derive(stats[pt], MAX_IT) for pt in range(len(grid))]
    outcomes = {prec: (h_it.numpy().copy(), h_res.numpy().copy())}  # rank-local per-frame outcomes, for the parity block
    hbm_peak, peak_src = measured_peaks()
    sm_mhz = float(clocks.get("sm_mhz") or 0.0) if isinstance(clocks, dict) else 0.0

    # ---- per-point kernel durations (events tightly around each launch, one point at a time): explanatory ------------------
    def per_point(precision, frames):
        p = params_for(precision)
        out = []
        for pt in range(len(grid)):
            a, b, lp, _ = keys[pt]
            best = None
            for _ in range(2):
                ctx.timer_start()
                ctx.reconcile_device(code, p, frames, a.data_ptr(), b.data_ptr(), lp.data_ptr(), d_it[pt].data_ptr(), d_res[pt].data_ptr())
                ms = ctx.timer_stop()
                best = ms if best is None else min(best, ms)
            iters = int(d_it[pt, :frames].sum().item())
            ok = int(((d_res[pt, :frames] & 3) == 3).sum().item())
            out.append((best, iters, ok, frames))
        return out

    def kernel_name(precision):
        return ("qlb::decode_resident_f64_kernel" if precision.startswith("f64") else "qlb::decode_resident_f32_kernel") + \
               "<" + {"f64": "MathF64", "f64fused": "MathF64Fused", "f32": "RuleF32Accurate", "f32fast": "RuleF32Fast"}[precision] + ">"

    def roofs(precision, frame_it_per_s):
        """SM-side roofs from the ncu-measured instruction mix of this build + the algorithmic HBM figure of SURVEY 8d."""
        pc = prof.get(precision, {})
        out = {}
        wi, w64 = pc.get("warp_instructions_per_frame_iteration"), pc.get("fp64_warp_instructions_per_frame_iteration")
        if wi and sm_mhz > 0:
            peak = 4.0 * ctx.sm_count * sm_mhz * 1e6
            out["issue"] = {"bound": "issue", "unit": "G warp-instructions/s", "achieved": frame_it_per_s * wi / 1e9, "peak": peak / 1e9,
                            "frac": frame_it_per_s * wi / peak, "warp_instructions_per_frame_iteration": wi}
        if w64 and sm_mhz > 0:
            lanes = pc.get("fp64_lanes_per_sm_per_clock", 64)
            peak = lanes / 32.0 * ctx.sm_count * sm_mhz * 1e6
            out["fp64_pipe"] = {"bound": "fp64_pipe", "unit": "G warp-instructions/s", "achieved": frame_it_per_s * w64 / 1e9, "peak": peak / 1e9,
                                "frac": frame_it_per_s * w64 / peak, "fp64_warp_instructions_per_frame_iteration": w64,
                                "fp64_lanes_per_sm_per_clock": lanes}
        ach = frame_it_per_s * e * BYTES_PER_EDGE_IT[precision] / 1e9
        out["algorithmic_hbm"] = {"bound": "hbm (algorithmic bytes, SURVEY.md 8d)", "unit": "GB/s", "achieved": ach, "peak": hbm_peak, "frac": ach / hbm_peak,
                                  "algorithmic_bytes_per_edge_iteration": BYTES_PER_EDGE_IT[precision], "peak_source": peak_src}
        return out

    pp = per_point(prec, fpp)
    step_frame_it = int(frame_iters // args.steps)
    fi_per_s = step_frame_it / (kern_ms_step * 1e-3)  # frame-iterations/s of the decode launches inside the timed steps
    rf = roofs(prec, fi_per_s)
    sm_roofs = [rf[k] for k in ("issue", "fp64_pipe") if k in rf]
    primary = max(sm_roofs, key=lambda r: r["frac"]) if sm_roofs else rf["algorithmic_hbm"]
    pc = prof.get(prec, {})
    roofline = {
        "bound": primary["bound"], "achieved": primary["achieved"], "peak": primary["peak"], "unit": primary["unit"], "frac": primary["frac"],
        "traffic": pc.get("dram_bytes_per_launch"), "traffic_source": pc.get("capture"),
        "traffic_algorithmic_bytes_of_that_launch": pc.get("algorithmic_bytes_of_that_launch"),
        "kernel": kernel_name(prec) + " (fused reconcile: prior init + Alice syndrome + BP iterations + early termination + key compare)",
        "frame_iterations_per_s": fi_per_s, "edge_iterations_per_s": fi_per_s * e,
        "kernel_ms_per_step": kern_ms_step, "kernel_share_of_step": kern_ms_step / ms_step,
        "algorithmic_hbm": rf["algorithmic_hbm"], "secondary": [r for r in sm_roofs if r is not primary],
        "note": "SM-resident decoder: a frame's messages stay on the SM (fp32: all of them in shared memory; fp64: 92 % in shared memory + an "
                "L2-resident tail per CTA), so DRAM traffic (`traffic`, ncu) is far below the algorithmic bytes and the binding roof is on the SM. "
                "`frac` is the tighter of the two SM-side roofs: instruction issue = (ncu warp instructions per frame-iteration of this build) x "
                "(live frame-iterations/s) / (4 issue slots x SMs x SM clock under load), and the FP64 pipe = the same with the FP64 warp "
                "instructions against the DFMA rate measured on this GPU type (scripts/micro/fp64_peak.cu: 58 lanes per SM and clock). "
                "`algorithmic_hbm.frac` is SURVEY.md 8d's fixed figure, the one north_star's 60 % target is quoted on.",
    }
    per_qber = []
    for pt, q in enumerate(grid):
        ms_pt, iters, ok, fr = pp[pt]
        r = results[pt]
        per_qber.append({"qber": round(q, 4), "qber_exact": keys[pt][3], "frames_per_s": fr / (ms_pt * 1e-3),
                         "sifted_mbit_s": fr / (ms_pt * 1e-3) * n / 1e6, "mean_iterations": iters / fr, "fer": r.fer,
                         "mean_iterations_successful": r.mean,
                         "algorithmic_hbm_frac": iters * e * BYTES_PER_EDGE_IT[prec] / (ms_pt * 1e-3) / 1e9 / hbm_peak})

    # ---- end to end through the C-ABI with pinned host buffers -------------------------------------------------------
    h_keys = []
    for pt in range(len(grid)):
        a, b, lp, qe = keys[pt]
        h_keys.append((a.cpu().pin_memory(), b.cpu().pin_memory(), torch.full((fpp,), qe, dtype=torch.float64).pin_memory()))

    # Two host threads, each with a context (stream + staging buffers) of its own, take alternate QBER points -- what the C++
    # scheduler does with its two workers per GPU: one point's H2D / D2H copies run under the other point's decode. The calls
    # are the blocking C-ABI entry point; ctypes releases the GIL while they run.
    from concurrent.futures import ThreadPoolExecutor
    pool = ThreadPoolExecutor(max_workers=2)
    h2d = len(grid) * fpp * (2 * code.words_n * 4 + 8)
    d2h = len(grid) * fpp * 5

    def measure_e2e(precision, steps, warm):
        p_e2e = params_for(precision)

        def points(c, pts):
            for pt in pts:
                ha, hb, hq = h_keys[pt]
                c.reconcile_packed_ptrs(code, p_e2e, fpp, ha.data_ptr(), hb.data_ptr(), hq.data_ptr(), h_it[pt].data_ptr(), h_res[pt].data_ptr())

        def step():
            jobs = [pool.submit(points, ctx, launch_order[0::2]), pool.submit(points, ctx_b, launch_order[1::2])]
            for j in jobs:
                j.result()
            return float(h_it.sum())  # the step's result is read on the host

        for _ in range(warm):
            step()
        _, wall, _ = timed(step, steps)
        v = frames_step / (wall / steps * 1e-3)
        return {"value": v, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": wall / steps,
                "sifted_mbit_s": v * n / 1e6, "steps": steps,
                "api": "qlb_reconcile_batch_packed (pinned host buffers), two host threads / contexts per GPU taking alternate QBER points"}

    e2e = measure_e2e(prec, args.steps, max(1, args.warmup // 2))
    e2e_same = bool((h_it.numpy() == outcomes[prec][0]).all() and (h_res.numpy() == outcomes[prec][1]).all())
    e2e["same_outcomes_as_device_resident_run"] = e2e_same

    # ---- the other precisions (explanatory numbers, same JSON line): kernel-only, e2e and per-frame outcomes ----------------
    # every rank measures (the e2e timing is max over ranks; value = whole job), rank 0 reports
    variants = {}
    if not args.no_variants:
        for v in PRECISIONS:
            if v == prec:
                continue
            sweep_step(v, collect=False)  # warm
            ppv = per_point(v, fpp)
            outcomes[v] = (d_it.cpu().numpy().copy(), d_res.cpu().numpy().copy())
            kms = sum(x[0] for x in ppv)
            fiv = sum(x[1] for x in ppv) / (kms * 1e-3)
            ev = measure_e2e(v, 2, 1)
            rv = roofs(v, fiv)
            variants[v] = {"frames_per_point": fpp, "frames_per_s": fpp * len(grid) / (kms * 1e-3), "frame_iterations_per_s": fiv,
                           "timing": "sum of the 9 launches timed one at a time (no two-stream overlap), this rank",
                           "kernel": kernel_name(v), "algorithmic_hbm_frac": rv["algorithmic_hbm"]["frac"],
                           "roofs": {k: {kk: r[kk] for kk in ("achieved", "peak", "unit", "frac")} for k, r in rv.items()},
                           "traffic": prof.get(v, {}).get("dram_bytes_per_launch"),
                           "fer": [1.0 - x[2] / x[3] for x in ppv], "e2e": ev}

    # ---- strong scaling (configs[2]'s shape): a fixed total of trials per point, sharded over the ranks, qlb_run_trials ------
    strong = None
    if strong_total:
        lo, hi = sweep.shard_range(strong_total, rank, world)
        shard = np.ascontiguousarray(all_seeds[lo:hi])
        p_s = params_for(prec)
        s_it = [None] * len(grid)
        s_res = [None] * len(grid)

        def strong_points(c, pts):
            for pt in pts:
                s_it[pt], s_res[pt], _ = c.run_trials(code, p_s, shard, grid[pt], seed_offset=pt)

        def strong_step():
            jobs = [pool.submit(strong_points, ctx, launch_order[0::2]), pool.submit(strong_points, ctx_b, launch_order[1::2])]
            for j in jobs:
                j.result()
            st = np.zeros((len(grid), MAX_IT + 5), np.int64)
            for pt in range(len(grid)):
                ps = sweep.PointStats(MAX_IT)
                ps.add(s_it[pt], s_res[pt])
                st[pt] = ps.vec
            return sweep.allreduce_stats(st, dev)

        strong_points(ctx, [0]); strong_points(ctx_b, [1])  # warm (buffers of both contexts sized)
        _, s_wall, s_stats = timed(strong_step, 1)
        s_res_d = [sweep.derive(s_stats[pt], MAX_IT) for pt in range(len(grid))]
        assert all(r.n_trials == strong_total for r in s_res_d)
        strong = {"scaling": "strong", "total_frames_per_point": strong_total, "frames": strong_total * len(grid), "precision": prec,
                  "value": strong_total * len(grid) / (s_wall * 1e-3), "unit": "frames/s", "ms": s_wall,
                  "h2d_bytes": 8 * strong_total * len(grid), "d2h_bytes": 5 * strong_total * len(grid),
                  "fer": [r.fer for r in s_res_d], "mean_iterations_successful": [r.mean for r in s_res_d],
                  "api": "qlb_run_trials: trial seeds up, keys generated on the GPU (bit-exact generator), reconcile, 5 B per frame down; trials "
                         "sharded in contiguous blocks over the ranks, statistics derived from the all-reduced integer histogram",
                  "note": "configs[2] is this shape with 1 000 000 trials per point (--strong-frames-per-point 1000000; the C++ binary "
                          "qkd_ldpc_b200_sim runs it from config.json, profiles/)"}
        if rank == 0 and lo == 0:
            outcomes["strong:" + prec] = (np.stack([x[:fpp] for x in s_it]), np.stack([x[:fpp] for x in s_res]))

    # ---- the HBM-bound design points (configs[3]): N = 100 000 and 1 000 000 through the streaming decoders ------------------
    if not args.no_variants and rank == 0 and world == 1:
        def stream_case(name, big, fr, q_big, it_big, precision, reps, label):
            big_code = capi.Code.from_graph(big)
            sd = torch.from_numpy(workload.trial_seeds(4242, fr).view(np.int64)).to(dev)
            ba = torch.empty((fr, big_code.words_n), dtype=torch.int32, device=dev)
            bb = torch.empty((fr, big_code.words_n), dtype=torch.int32, device=dev)
            bq = ctx.generate_device(big.n, fr, sd.data_ptr(), q_big, ba.data_ptr(), bb.data_ptr())
            blp = torch.full((fr,), workload.log_prior(bq), dtype=torch.float64, device=dev)
            bit_ = torch.zeros(fr, dtype=torch.int32, device=dev)
            bres = torch.zeros(fr, dtype=torch.uint8, device=dev)
            ctx.synchronize()
            pbig = capi.make_params(64 if precision.startswith("f64") else 32, it_big, THR, True, fast_math=precision in ("f32fast", "f64fused"))
            best = None
            for _ in range(reps):
                ctx.timer_start()
                ctx.reconcile_device(big_code, pbig, fr, ba.data_ptr(), bb.data_ptr(), blp.data_ptr(), bit_.data_ptr(), bres.data_ptr())
                ms = ctx.timer_stop()
                best = ms if best is None else min(best, ms)
            its = int(bit_.sum().item())
            gbs = its * big.e * BYTES_PER_EDGE_IT[precision] / (best * 1e-3) / 1e9
            variants[name] = {"workload": label, "precision": precision, "frames": fr, "ms": best, "mean_iterations": its / fr,
                              "fer": 1.0 - float(((bres & 3) == 3).sum().item()) / fr,
                              "frame_iterations_per_s": its / (best * 1e-3), "edge_iterations_per_s": its * big.e / (best * 1e-3),
                              "achieved_GBps": gbs, "roofline_frac": gbs / hbm_peak, "bound": "hbm",
                              "kernels": "qlb::stream_{setup,init,check,update,bit,repack_*,finalize}_kernel<%s>" % ("StreamF64" if precision.startswith("f64") else "StreamF32"),
                              "traffic": prof.get(name, {}).get("dram_bytes_per_launch"),
                              "note": "whole call incl. set-up and result kernels, CUDA events on the launching stream, best of %d" % reps}
            del ba, bb, blp, bit_, bres, big_code
            torch.cuda.empty_cache()

        try:
            big = codes.peg_code(100000, 51080, 3, 666, bfs_limit=2000)  # committed copy under data/codes/
            lbl = "configs[3]: PEG N=100000 M=51080 CW=3 SEED=666"
            # nothing converges at QBER 0.10: 20 full iterations over 148 groups of 128 frames
            stream_case("stream_n100k", big, 18944, 0.10, 20, "f32fast", 5, lbl + ", 18944 frames, QBER 0.10, 20 iterations, fp32 fast rule")
            # a waterfall QBER: most frames converge around round 45, ~7 % run to 100 -- what the on-device frame compaction is
            # for (algorithmic bytes count only the rounds each frame needed)
            stream_case("stream_n100k_waterfall", big, 18944, 0.085, MAX_IT, "f32fast", 2, lbl + ", 18944 frames, QBER 0.085, max 100 iterations")
            stream_case("stream_n100k_f64", big, 9472, 0.10, 20, "f64", 3, lbl + ", 9472 frames, QBER 0.10, 20 iterations, fp64 reference order (fp64 streaming decoder)")
            stream_case("stream_n100k_f64fused", big, 9472, 0.10, 20, "f64fused", 3, lbl + ", 9472 frames, QBER 0.10, 20 iterations, fp64 fused-ratio rule (fp64 streaming decoder)")
            stream_case("stream_n100k_f64_waterfall", big, 9472, 0.085, MAX_IT, "f64", 1, lbl + ", 9472 frames, QBER 0.085, max 100 iterations, fp64 reference order")
            del big
            huge = codes.permutation_code(1_000_000, 510_800, 3, 666)
            lbl = "configs[3]: permutation code N=1000000 M=510800 CW=3 SEED=666"
            stream_case("stream_n1m", huge, 8192, 0.10, 12, "f32fast", 2, lbl + ", 8192 frames, QBER 0.10, 12 iterations, fp32 fast rule")
            stream_case("stream_n1m_f64", huge, 4096, 0.10, 12, "f64", 2, lbl + ", 4096 frames, QBER 0.10, 12 iterations, fp64 reference order (fp64 streaming decoder)")
            del huge
        except Exception as ex:  # the headline line must not depend on the side measurements
            variants["stream_error"] = {"error": str(ex)[:300]}
    if world > 1:
        dist.barrier()

    # ---- CPU baseline (rank 0, N = 1 only) + per-frame parity of every precision against it ----------------------------------
    cpu = None
    parity = None
    fer_parity = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        tpp = min(cpu_tpp(args, cores), fpp)
        kind, sec, outs = cpu_reference_sweep(tpp, cores, SIM_SEED)
        cpu_val = tpp * len(grid) / sec
        cpu = {"value": cpu_val, "unit": "frames/s", "cores": cores, "kind": kind, "seconds": sec,
               "sample": f"trials 0..{tpp - 1} of each of the {len(grid)} QBER points ({tpp * len(grid)} frames; run_trial: key generation + reconciliation), {cores} threads",
               "per_qber_fer": [1.0 - float((o[:, 1] * o[:, 2]).mean()) for o in outs],
               "per_qber_mean_iterations": [float(o[:, 0].mean()) for o in outs]}
        ref_it = np.stack([o[:, 0] for o in outs]).astype(np.int64)
        ref_fl = np.stack([o[:, 1] | (o[:, 2] << np.uint64(1)) for o in outs]).astype(np.int64)
        parity = {"reference": f"{kind}: the CPU sample above -- the same trials (same seeds, same keys) as frames 0..{tpp - 1} of every point of the GPU run",
                  "frames_compared": int(ref_it.size)}
        for v, (g_it, g_res) in outcomes.items():
            same_fl = (g_res[:, :tpp].astype(np.int64) & 3) == ref_fl
            same_it = g_it[:, :tpp].astype(np.int64) == ref_it
            parity[v] = {"frames_compared": int(ref_it.size), "identical_flags": int(same_fl.sum()), "identical_iterations": int(same_it.sum()),
                         "identical_flags_and_iterations": int((same_fl & same_it).sum())}
        fer_parity = []
        for pt in range(len(grid)):
            k_ref = int(tpp - (outs[pt][:, 1] * outs[pt][:, 2]).sum())
            lo_, hi_ = sweep.binomial_ci95(k_ref, tpp)
            fer_parity.append({"qber": round(grid[pt], 4), "fer_gpu": results[pt].fer, "fer_ref": k_ref / tpp, "ref_ci95": [lo_, hi_],
                               "inside": bool(lo_ <= results[pt].fer <= hi_)})

    if rank == 0:
        line = {
            "metric": "decoded_frames_per_s", "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64" if prec.startswith("f64") else "f32", "data": "synthetic",
            "config": workload_config(fpp, prec),
            "sifted_mbit_s": value * n / 1e6,
            "frame_iterations_per_step": step_frame_it * world if world == 1 else None, "wall_ms_per_step": wall_total / args.steps,
            "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu, "clocks": clocks,
            "parity": parity, "per_qber": per_qber, "fer_parity_vs_cpu_sample": fer_parity, "strong": strong, "variants": variants,
        }
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, *outcomes[prec])
        guard.emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
