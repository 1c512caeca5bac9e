"""The host-side C++ mirror of the reference API (qkd_ldpc_b200/host): loaders, key generator and config handling on
the CPU; the config.json-driven sweep against the reference's own CSV output on the GPU."""
import json
import shutil
import subprocess
from pathlib import Path

import numpy as np
import pytest

from conftest import GOLD, NS, ROOT
from qkd_ldpc_b200 import build, codes

SIM = build.SIM_PATH


@pytest.fixture(scope="module")
def sim():
    build.build_all()
    assert SIM.exists()
    return SIM


def run(sim, *args, cwd=None, check=True):
    p = subprocess.run([str(sim), *map(str, args)], capture_output=True, text=True, cwd=cwd)
    if check:
        assert p.returncode == 0, p.stderr
    return p


def parse_dump(text):
    lines = text.strip().splitlines()
    n, m, mbw, mcw, reg = map(int, lines[0].split())
    bit_lists = [list(map(int, ln.split()))[1:] for ln in lines[1:1 + n]]
    check_lists = [list(map(int, ln.split()))[1:] for ln in lines[1 + n:1 + n + m]]
    return n, m, mbw, mcw, bool(reg), bit_lists, check_lists


@pytest.mark.parametrize("name", ["dense_n6_m4", "dense_n7_m3", "dense_n10_m5", NS])
def test_cpp_loaders_match_reference_matrices(sim, matrices, name):
    """read_dense_matrix / read_sparse_alist_matrix produce the H_matrix the reference's loaders produced (data/codes/*.npz
    hold the reference's own output)."""
    mat = matrices[name]
    path = codes.materialize()[name]
    n, m, mbw, mcw, reg, bit_lists, check_lists = parse_dump(run(sim, "--dump-matrix", "dense" if name.startswith("dense") else "alist", path).stdout)
    assert (n, m, reg) == (mat.n, mat.m, mat.is_regular)
    assert (mbw, mcw) == (mat.max_bit_w, mat.max_check_w)
    assert sum(bit_lists, []) == mat.row_idx.tolist() and sum(check_lists, []) == mat.col_idx.tolist()
    assert [len(b) for b in bit_lists] == np.diff(mat.col_ptr).tolist()


def test_cpp_loader_errors(sim, tmp_path):
    bad = tmp_path / "bad.txt"
    bad.write_text("1 0 2\n0 1 1\n")
    p = run(sim, "--dump-matrix", "dense", bad, check=False)
    assert p.returncode != 0 and "can only take values" in p.stderr
    bad.write_text("1 1 1\n0 0 0\n")
    p = run(sim, "--dump-matrix", "dense", bad, check=False)
    assert p.returncode != 0 and "Row '2' weight cannot be equal to or less than zero" in p.stderr
    bad.write_text("3 2\n2 2\n1 1 2\n2 2\n1 0\n2 0\n1 0\n1 3\n2 3\n")      # column 3 lists one entry, declares two
    p = run(sim, "--dump-matrix", "alist", bad, check=False)
    assert p.returncode != 0 and "does not match the weight" in p.stderr
    p = run(sim, "--dump-matrix", "alist", tmp_path / "missing.txt", check=False)
    assert p.returncode != 0 and "Failed to open file" in p.stderr


def test_cpp_generator_matches_oracle(sim, oracle):
    """Same seeds -> same Alice/Bob keys as the (reference-pinned) oracle generator, including the shuffle."""
    assert run(sim, "--seeds", 777, 3).stdout.split() == [str(v) for v in oracle.trial_seeds(777, 3)]
    for seed, n, q in [(int(oracle.trial_seeds(777, 1)[0]), 10240, 0.03), (12345, 7, 0.25), (99, 33, 0.5), (5, 64, 0.01)]:
        out = run(sim, "--gen", seed, n, q).stdout.split()
        a, b, exact = oracle.generate(seed, n, q)
        assert float(out[0]) == exact
        assert out[1] == "".join(map(str, a)) and out[2] == "".join(map(str, b))


def base_cfg(**kw):
    cfg = {"threads_number": 8, "trials_number": 64, "use_config_simulation_seed": True, "simulation_seed": 777,
           "interactive_mode": False, "sum_product_max_iterations": 100, "use_dense_matrices": False, "trace_qkd_ldpc": False,
           "trace_sum_product": False, "trace_sum_product_llr": False, "enable_sum_product_msg_llr_threshold": True,
           "sum_product_msg_llr_threshold": 100.0,
           "code_rate_QBER_parameters": [{"code_rate": 0.5, "QBER_begin": 0.03, "QBER_end": 0.12, "QBER_step": 0.01}]}
    cfg.update(kw)
    return cfg


def make_dir(tmp_path, cfg, name, dense):
    (tmp_path / "config.json").write_text(json.dumps(cfg))
    sub = tmp_path / ("dense_matrices" if dense else "alist_sparse_matrices")
    sub.mkdir()
    shutil.copy(codes.materialize()[name], sub)
    return tmp_path


def test_cpp_config_validation(sim, tmp_path):
    d = make_dir(tmp_path, base_cfg(trials_number=0), NS, False)
    p = run(sim, d, check=False)
    assert p.returncode != 0 and "Number of trials must be >= 1!" in p.stderr
    (d / "config.json").write_text(json.dumps(base_cfg(code_rate_QBER_parameters=[{"code_rate": 0.5, "QBER_begin": 0.2, "QBER_end": 0.1, "QBER_step": 0.01}])))
    p = run(sim, d, check=False)
    assert p.returncode != 0 and "Invalid QBER begin or end parameters" in p.stderr
    (d / "config.json").write_text(json.dumps(base_cfg(code_rate_QBER_parameters=[{"code_rate": 0.3, "QBER_begin": 0.03, "QBER_end": 0.12, "QBER_step": 0.01}])))
    p = run(sim, d, check=False)
    assert p.returncode != 0 and "QBER range based on code rate" in p.stderr
    (d / "config.json").unlink()
    p = run(sim, d, check=False)
    assert p.returncode != 0 and "Configuration file not found" in p.stderr


def test_cpp_matrix_warnings(sim, tmp_path, lib):
    """An alist file with an unsorted list loads (as in the reference) but is flagged; the device layout then rejects it
    because the reference's positional routing would misroute on it."""
    mat = codes.load_npz("dense_n7_m3")
    bad = tmp_path / "alist_sparse_matrices"
    bad.mkdir()
    codes.write_alist(mat, bad / "h.txt")
    lines = (bad / "h.txt").read_text().splitlines()
    parts = lines[4 + 6].split()            # bit 7 is in checks 1 2 3: swap two entries
    parts[0], parts[1] = parts[1], parts[0]
    lines[4 + 6] = " ".join(parts)
    (bad / "h.txt").write_text("\n".join(lines) + "\n")
    (tmp_path / "config.json").write_text(json.dumps(base_cfg(trials_number=4, code_rate_QBER_parameters=[
        {"code_rate": 0.58, "QBER_begin": 0.15, "QBER_end": 0.35, "QBER_step": 0.1}])))
    p = run(sim, tmp_path, check=False)
    assert "not sorted ascending" in p.stderr
    assert p.returncode != 0


def test_cpp_no_gpu_fails_loudly(sim, tmp_path, lib):
    if lib.qlb_device_count() > 0:
        pytest.skip("a GPU is present")
    d = make_dir(tmp_path, base_cfg(trials_number=4), NS, False)
    p = run(sim, d, check=False)
    assert p.returncode != 0 and "no CPU decoder" in p.stderr


@pytest.mark.gpu
def test_sweep_csv_equals_reference_north_star(sim, tmp_path):
    """config.json -> CSV on the N=10240 code, 64 trials x 9 QBER points: byte-identical to the CSV written by the
    reference's own main() (tests/golden/sweep_n10240_t64_seed777.csv), fp64 messages; keys drawn on the GPU from the
    trial seeds."""
    d = make_dir(tmp_path, base_cfg(), NS, False)
    run(sim, d)
    out = sorted((d / "results").glob("ldpc*.csv"))
    assert len(out) == 1 and out[0].name == "ldpc(trial_num=64,max_sum_prod_iters=100,seed=777).csv"
    assert out[0].read_text() == (GOLD / "sweep_n10240_t64_seed777.csv").read_text()
    # the side report (never mixed into the reference-format CSV): throughput, efficiency f = (1-R)/h2(q), leakage = M
    rep = [ln.split(";") for ln in sorted((d / "results").glob("throughput*.csv"))[0].read_text().splitlines()]
    assert rep[0][:6] == ["SIM", "MATRIX_FILENAME", "M", "N", "QBER", "FRAMES"] and len(rep) == 10
    import math
    q = float(rep[1][4]); h2 = -q * math.log2(q) - (1 - q) * math.log2(1 - q)
    assert abs(float(rep[1][11]) - (5231 / 10240) / h2) < 1e-3 and rep[1][12] == "5231" and rep[1][5] == "64" and float(rep[1][7]) > 0


@pytest.mark.gpu
def test_sweep_csv_equals_reference_dense_n7(sim, tmp_path):
    """BASELINE.json configs[0]: dense (N=7,K=4,M=3) through config.json, 1000 trials, two QBER points."""
    cfg = base_cfg(trials_number=1000, use_dense_matrices=True, device_batch_frames=256,
                   code_rate_QBER_parameters=[{"code_rate": 0.58, "QBER_begin": 0.15, "QBER_end": 0.35, "QBER_step": 0.1}])
    d = make_dir(tmp_path, cfg, "dense_n7_m3", True)
    run(sim, d)
    out = sorted((d / "results").glob("ldpc*.csv"))
    assert out[0].read_text() == (GOLD / "sweep_dense_n7_t1000_seed777.csv").read_text()
    # a second run must not overwrite: the reference de-duplicates the file name
    run(sim, d)
    assert len(sorted((d / "results").glob("ldpc*.csv"))) == 2
    assert not list((d / "results").glob("*.partial.csv")), "progress files are removed once the sweep has completed"


@pytest.mark.gpu
def test_sweep_fp32_and_forced_allreduce(sim, tmp_path):
    """fp32 fast path through config.json (same FER / ratios on this grid; iteration means within a few percent), with the
    NCCL statistics all-reduce forced on the single GPU (config key device_force_allreduce)."""
    d = make_dir(tmp_path, base_cfg(device_precision=32, device_fp32_fast_math=True, device_force_allreduce=True), NS, False)
    run(sim, d)
    got = [ln.split(";") for ln in sorted((d / "results").glob("ldpc*.csv"))[0].read_text().splitlines()[1:]]
    want = [ln.split(";") for ln in (GOLD / "sweep_n10240_t64_seed777.csv").read_text().splitlines()[1:]]
    for g, w in zip(got, want):
        assert g[:7] == w[:7] and g[11:] == w[11:], (g, w)          # identity columns, success ratios, FER
        assert abs(float(g[7]) - float(w[7])) <= 0.05 * float(w[7]) + 1e-9


@pytest.mark.gpu
def test_key_too_small_error(sim, tmp_path):
    cfg = base_cfg(use_dense_matrices=True, trials_number=4,
                   code_rate_QBER_parameters=[{"code_rate": 0.58, "QBER_begin": 0.05, "QBER_end": 0.1, "QBER_step": 0.05}])
    d = make_dir(tmp_path, cfg, "dense_n7_m3", True)
    p = run(sim, d, check=False)
    assert p.returncode != 0 and "Key size '7' is too small for QBER." in p.stderr


# (N, M, max bit weight, max check weight, regular, bit lists, check lists) of the 3 x 2 code the alist cases below spell out
H_3X2 = (3, 2, 2, 2, False, [[0], [1], [0, 1]], [[0, 2], [1, 2]])
MALFORMED = {  # name -> (kind, file text, the reference's outcome); every branch of its loaders (src/array_and_matrix_operations.cpp:109-421)
    # The outcome is the error message the reference's loader throws ("{path}" = the file's path) or the matrix it loads; the
    # host loaders matched every one of them when the reference's loaders were compiled beside them.
    "alist_three_lines": ("alist", "3 2\n2 2\n1 1 2\n", "Insufficient data in the file: {path}"),
    "alist_header_three_numbers": ("alist", "3 2 1\n2 2\n1 1 2\n2 2\n1 0\n2 0\n1 2\n1 3\n2 3\n",
                                   "File format does not match the alist format: {path}"),
    "alist_second_line_one_number": ("alist", "3 2\n2\n1 1 2\n2 2\n1 0\n2 0\n1 2\n1 3\n2 3\n",
                                     "File format does not match the alist format: {path}"),
    "alist_too_few_lines": ("alist", "3 2\n2 2\n1 1 2\n2 2\n1 0\n2 0\n1 2\n1 3\n", "Insufficient data in the file: {path}"),
    "alist_n_mismatch": ("alist", "4 2\n2 2\n1 1 2\n2 2\n1 0\n2 0\n1 2\n1 3\n2 3\n",
                         "Number of columns '4' is not the same as the length of the third line '3'. File: {path}"),
    "alist_m_mismatch": ("alist", "3 3\n2 2\n1 1 2\n2 2\n1 0\n2 0\n1 2\n1 3\n2 3\n",
                         "Number of rows '3' is not the same as the length of the fourth line '2'. File: {path}"),
    "alist_bit_weight_mismatch": ("alist", "3 2\n2 2\n1 1 2\n2 2\n1 0\n2 0\n1 0\n1 3\n2 3\n",
                                  "Number of non-zero elements '1' in the line '7' does not match the weight in the third line '2'. File: {path}"),
    "alist_check_weight_mismatch": ("alist", "3 2\n2 2\n1 1 2\n2 2\n1 0\n2 0\n1 2\n1 3 2\n2 3\n",
                                    "Number of non-zero elements '3' in the line '8' does not match the weight in the fourth line '2'. File: {path}"),
    "alist_token_ends_row": ("alist", "3 2\n2 2\n1 1 2\n2 2\n1 0\n2 x 0\n1 2\n1 3\n2 3\n", H_3X2),
    "alist_no_final_newline_ok": ("alist", "3 2\n2 2\n1 1 2\n2 2\n1 0\n2 0\n1 2\n1 3\n2 3", H_3X2),
    "alist_crlf_and_padding_ok": ("alist", "3 2\r\n2 2\r\n1 1 2\r\n2 2\r\n1 0\r\n2 0\r\n1 2\r\n1 3\r\n2 3\r\n\r\n", H_3X2),
    "alist_leading_zero_entry": ("alist", "3 2\n2 2\n1 1 2\n2 2\n1 0\n2 0\n0 1 2\n1 3\n2 3\n",
                                 (3, 2, 2, 2, False, [[0], [1], [-1, 0]], [[0, 2], [1, 2]])),
    "empty": ("alist", "", "File is empty or cannot be read properly: {path}"),
    "dense_bad_value": ("dense", "1 0 2\n0 1 1\n", "Parity check matrix can only take values 0 or 1."),
    "dense_ragged": ("dense", "1 0 1\n0 1\n", "Different lengths of rows in a matrix. File: {path}"),
    "dense_zero_column": ("dense", "1 0 1\n1 0 1\n", "Column '2' weight cannot be equal to or less than zero. File: {path}"),
    "dense_zero_row": ("dense", "1 1 1\n0 0 0\n", "Row '2' weight cannot be equal to or less than zero. File: {path}"),
    "dense_token_ends_row": ("dense", "1 1 1\n0 1 a 1\n", "Different lengths of rows in a matrix. File: {path}"),
    "dense_empty": ("dense", "", "File is empty or cannot be read properly: {path}"),
    "dense_blank_last_line": ("dense", "1 1 0\n0 1 1\n\n", "Different lengths of rows in a matrix. File: {path}"),
}


@pytest.mark.parametrize("case", sorted(MALFORMED))
def test_cpp_loader_behaviour_equals_reference(sim, tmp_path, case):
    """The flat (CSR / CSC emitting) loaders accept and reject exactly what the reference's loaders do, with the same message;
    when the file loads, both produce the same adjacency lists."""
    kind, text, want = MALFORMED[case]
    path = tmp_path / f"{case}.txt"
    path.write_text(text, newline="")
    ours = run(sim, "--dump-matrix", kind, path, check=False)
    if isinstance(want, str):
        want = want.format(path=path)
        assert ours.returncode != 0, (case, "the reference rejects this file:", want)
        assert want in ours.stderr, (case, want, ours.stderr)
        return
    assert ours.returncode == 0, (case, ours.stderr)
    assert parse_dump(ours.stdout) == want


def test_cpp_alist_load_one_million(sim, tmp_path):
    """SURVEY 8f-2: the N = 1 000 000 alist (3 M edges, 45 MB of text) goes from the file into flat CSR / CSC arrays in one pass;
    the adjacency the loader produces is checked against the generator's through position-weighted checksums, and the load
    time is printed (0.28 s here; the line-by-line istringstream form of round 1 took 1.4-1.6 s on the same file)."""
    n, m = 1_000_000, 510_800
    mat = codes.permutation_code(n, m, 3, 666)
    path = tmp_path / "n1m.alist"
    codes.write_alist(mat, path)
    out = run(sim, "--time-load", "alist", path).stdout.split()
    seconds, (gn, gm, edges, sum_bits, sum_checks) = float(out[0]), map(int, out[1:])
    assert (gn, gm, edges) == (n, m, mat.e)
    col = np.repeat(np.arange(n, dtype=np.uint64) + np.uint64(1), np.diff(mat.col_ptr))
    row = np.repeat(np.arange(m, dtype=np.uint64), np.diff(mat.row_ptr))
    assert sum_bits == int((mat.row_idx.astype(np.uint64) * col).sum()) and sum_checks == int(((mat.col_idx.astype(np.uint64) + np.uint64(1)) * row).sum())
    print(f"N=1M alist load: {seconds:.2f} s")
    assert seconds < 5.0


@pytest.mark.gpu
def test_sweep_csv_equals_reference_three_matrices(sim, tmp_path):
    """A directory with the three shipped dense matrices -- one of them regular, so its frames go through QKD_LDPC_regular
    (src/qkd_ldpc_algorithm.cpp:347-396) -- and three rate presets: six sweep points numbered across the matrices, the
    trial seeds offset by the global point number (src/simulation.cpp:231-247). Byte-identical to the CSV of the reference's own
    main() (tests/golden/make_multi_matrix.py). The point numbers -- hence the seeds -- follow the directory iteration order, which
    is the file system's: when this machine lists the files in another order than the one the golden file was made on, the test
    says so instead of comparing different sweeps."""
    PRESETS = [{"code_rate": 0.34, "QBER_begin": 0.17, "QBER_end": 0.51, "QBER_step": 0.17},  # as in tests/golden/make_multi_matrix.py
               {"code_rate": 0.5, "QBER_begin": 0.1, "QBER_end": 0.3, "QBER_step": 0.1},
               {"code_rate": 0.58, "QBER_begin": 0.15, "QBER_end": 0.35, "QBER_step": 0.1}]
    cfg = base_cfg(trials_number=500, use_dense_matrices=True, device_batch_frames=128, code_rate_QBER_parameters=PRESETS)
    (tmp_path / "config.json").write_text(json.dumps(cfg))
    sub = tmp_path / "dense_matrices"
    sub.mkdir()
    for name in ("dense_n6_m4", "dense_n7_m3", "dense_n10_m5"):
        shutil.copy(codes.materialize()[name], sub)
    run(sim, tmp_path)
    got = sorted((tmp_path / "results").glob("ldpc*.csv"))[0].read_text()
    want = (GOLD / "sweep_dense_three_matrices_t500_seed777.csv").read_text()

    def order(csv):
        names = []
        for ln in csv.splitlines()[1:]:
            if ln.split(";")[1] not in names:
                names.append(ln.split(";")[1])
        return names
    if order(got) != order(want):
        pytest.skip(f"this file system lists the matrices as {order(got)}, the golden run had {order(want)}")
    assert got == want
