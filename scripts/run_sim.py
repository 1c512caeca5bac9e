"""Runs qkd_ldpc_b200_sim (the reference's main() counterpart) on the N=10240 code in a scratch directory.
usage: run_sim.py <trials> <precision 64|32|32fast> [gpus]"""
import json, shutil, subprocess, sys, tempfile, time
from pathlib import Path
sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from qkd_ldpc_b200 import build, codes
trials = int(sys.argv[1]); prec = sys.argv[2]
gpus = int(sys.argv[3]) if len(sys.argv) > 3 else 0
cfg = {"threads_number": 16, "trials_number": trials, "use_config_simulation_seed": True, "simulation_seed": 777, "interactive_mode": False,
       "sum_product_max_iterations": 100, "use_dense_matrices": False, "trace_qkd_ldpc": False, "trace_sum_product": False,
       "trace_sum_product_llr": False, "enable_sum_product_msg_llr_threshold": True, "sum_product_msg_llr_threshold": 100.0,
       "code_rate_QBER_parameters": [{"code_rate": 0.5, "QBER_begin": 0.03, "QBER_end": 0.12, "QBER_step": 0.01}],
       "device_precision": 64 if prec == "64" else 32, "device_fp32_fast_math": prec == "32fast",
       "device_gpus": gpus, "device_batch_frames": 16384}
d = Path(tempfile.mkdtemp())
(d / "config.json").write_text(json.dumps(cfg))
(d / "alist_sparse_matrices").mkdir()
shutil.copy(codes.materialize()[codes.NORTH_STAR], d / "alist_sparse_matrices")
t = time.perf_counter()
p = subprocess.run([str(build.SIM_PATH), str(d)], capture_output=True, text=True)
dt = time.perf_counter() - t
print(p.stdout.strip().splitlines()[-1] if p.stdout.strip() else "", p.stderr.strip())
print(f"wall {dt:.2f} s for {trials*9} frames -> {trials*9/dt:.0f} frames/s (precision {prec}, gpus {gpus or 'all'})")
print(sorted((d / "results").glob("*.csv"))[0].read_text())
