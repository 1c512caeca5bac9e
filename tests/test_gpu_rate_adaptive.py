"""Rate-adaptive reconciliation (qlb_reconcile_adapted_packed, qlb_run_trials_adapted) on the GPU. A rate-adapted batch is decoded
by the unchanged decoders in sum-product mode, so each case restates the frame assembly in numpy (test_rate_pattern.assemble),
decodes those LLRs and that syndrome with a CPU restatement, and requires the GPU to give the same iterations, both flags and every
decoded key bit on every frame. Each case names the decoder it expects (qlb_ctx_last_decoder)."""
import functools
import json
import shutil
import subprocess

import numpy as np
import pytest

from conftest import NS
from min_sum_restatement import MinSumRestatement
from qkd_ldpc_b200 import build, capi, codes
from test_gpu_codes import graph_of
from test_gpu_decoder_paths import assert_decoder, code_of
from test_rate_pattern import assemble, effective_rate, fill_bits, policy, restated_pattern

pytestmark = pytest.mark.gpu
MAX_IT = 40
ALPHA = 0.8125
THR = 100.0
PEG100K = "peg_n100000_m51080_cw3_seed666_bfs2000"


@pytest.fixture(scope="module")
def msr():
    return MinSumRestatement()


@functools.lru_cache(maxsize=None)
def code_for(key):
    if key == "peg_n100000":
        mat = codes.load_npz(PEG100K)
        return mat, graph_of(mat), capi.Code.from_graph(mat)
    return code_of(key)


def frames_of(ctx, mat, cls, seeds, q):
    """n-bit keys from the device generator, fill bits from numpy, the exact QBER over the n key bits"""
    n, n_fill = int((cls == capi.POS_KEY).sum()), int((cls != capi.POS_KEY).sum())
    a, b, ex = ctx.generate(n, seeds, q)
    rng = np.random.default_rng([int(seeds[0]) & 0xFFFFFFFF, n])
    fill = (rng.random((seeds.size, n_fill)) < 0.5).astype(np.int32)
    return a, b, fill, ex


def restated_outcomes(decode, mat, cls, a, b, fill, ex, thr=THR):
    """per frame: (iterations, syndrome flag, keys flag, decoded key bits) of the CPU decode of the restated assembly"""
    n = int((cls == capi.POS_KEY).sum())
    key_pos = np.flatnonzero(cls == capi.POS_KEY)
    A, B = capi.unpack_bits(a, n), capi.unpack_bits(b, n)
    out = []
    for f in range(A.shape[0]):
        llr, syn = assemble(mat, cls, A[f], B[f], fill[f], ex, thr)
        it, ok, bits = decode(llr, syn)
        out.append((it, ok, bool((bits[key_pos] == A[f]).all()), bits[key_pos]))
    return out


def assert_equal(case, want, it, res, dec, n):
    D = capi.unpack_bits(dec, n)
    for f, (w_it, w_ok, w_keys, w_bits) in enumerate(want):
        assert (int(it[f]), bool(res[f] & 1), bool(res[f] & 2)) == (w_it, w_ok, w_keys), (case, f, it[f], res[f], w_it, w_ok, w_keys)
        assert (D[f] == w_bits).all(), (case, f)


def fill_packed(cls, fill):
    n_fill = int((cls != capi.POS_KEY).sum())
    return capi.pack_bits(fill, n_fill) if n_fill else None


# ---- min-sum: every decoder family against the restatement ---------------------------------------------------------------------
MS_CASES = [
    ("north_star", {}, 0.04, "resident_f32minsum bw=3"),
    ("perm3_n1024", {"tier": 0}, 0.02, "generic f32minsum tier=0 shape=8"),
    ("perm3_n1024", {"tier": 1}, 0.02, "generic f32minsum tier=1 shape=8"),
    ("ladder_n4096", {"tier": 2}, 0.02, "generic f32minsum tier=2 shape=0"),
    ("ladder_n4096", {"tier": 3}, 0.02, "stream_f32 vec=4 bw=3"),
    ("perm3_n4001", {}, 0.04, "stream_f32 vec=4 bw=3"),   # N % 32 != 0
    ("peg_n100000", {}, 0.04, "stream_f32"),
]


def splits(mat, seed):
    """(p, s) pairs: none, shortening only, puncturing only, both; n = N - p - s is not a multiple of 32 in the last three"""
    avail = restated_pattern(mat, mat.n, 0, seed)
    p = min(mat.n // 20, avail - 1) | 1
    s = (mat.n // 25) | 1
    return [(0, 0), (0, s), (p, 0), (p, s)]


@pytest.mark.parametrize("key,kw,q,expect", MS_CASES, ids=[f"{c[0]}-{c[3].split()[0]}-{'-'.join(f'{k}={v}' for k, v in c[1].items())}" for c in MS_CASES])
def test_min_sum_matches_restatement(ctx, oracle, msr, key, kw, q, expect):
    mat, g, code = code_for(key)
    frames = 16 if mat.n > 20000 else 48
    params = capi.make_params(32, MAX_IT, THR, True, min_sum_scale=ALPHA, **kw)
    reconciled = 0
    for k, (p, s) in enumerate(splits(mat, 11)):
        cls = capi.rate_pattern(code, p, s, 11)
        n = mat.n - p - s
        seeds = oracle.trial_seeds(1200 + k, frames)
        a, b, fill, ex = frames_of(ctx, mat, cls, seeds, q)
        it, res, dec = ctx.reconcile_adapted(code, params, cls, a, b, fill_packed(cls, fill), ex)
        assert_decoder(ctx, expect, (key, p, s))
        want = restated_outcomes(lambda llr, syn: msr.sum_product(g, llr, syn, ALPHA, max_it=MAX_IT, thr=THR), mat, cls, a, b, fill, ex)
        assert_equal((key, kw, p, s), want, it, res, dec, n)
        reconciled += sum(w[2] for w in want)
    assert reconciled > 0, "no frame reconciled: the case checks nothing but failures"


@pytest.mark.parametrize("key,kw", [("north_star", {}), ("ladder_n4096", {"tier": 3}), ("perm3_n4001", {})])
def test_run_trials_adapted_keys_and_fill(ctx, oracle, msr, key, kw):
    """Keys are qlb_generate_batch_packed's at n bits, fill is the numpy stream of ~(seed + offset); outcomes equal the restatement."""
    mat, g, code = code_for(key)
    p, s = splits(mat, 3)[3]
    cls = capi.rate_pattern(code, p, s, 3)
    n = mat.n - p - s
    seeds, offset, q = oracle.trial_seeds(4545, 40), 5, 0.05
    params = capi.make_params(32, MAX_IT, THR, True, min_sum_scale=ALPHA, **kw)
    it, res, ex = ctx.run_trials_adapted(code, params, cls, seeds, q, seed_offset=offset)
    a, b, ex_g = ctx.generate(n, seeds, q, seed_offset=offset)
    assert ex == ex_g == int(n * q) / n
    fill = np.stack([fill_bits(x, offset, p + s) for x in seeds])
    it2, res2, _ = ctx.reconcile_adapted(code, params, cls, a, b, capi.pack_bits(fill, p + s), ex)
    assert (it == it2).all() and (res == res2).all()
    want = restated_outcomes(lambda llr, syn: msr.sum_product(g, llr, syn, ALPHA, max_it=MAX_IT, thr=THR), mat, cls, a, b, fill, ex)
    assert [(int(i), bool(r & 1), bool(r & 2)) for i, r in zip(it, res)] == [w[:3] for w in want]


# ---- fp64 and fp64 fused: shortening only, against the oracle ------------------------------------------------------------------------
@pytest.mark.parametrize("fused", [False, True])
@pytest.mark.parametrize("key,kw,expect", [("north_star", {}, "resident_f64"), ("perm3_n1024", {"tier": 0}, "generic f64")])
def test_fp64_shortening_matches_oracle(ctx, oracle, key, kw, expect, fused):
    mat, g, code = code_for(key)
    q = 0.06 if key == "north_star" else 0.05
    params = capi.make_params(64, MAX_IT, THR, True, fast_math=fused, **kw)
    for s in (0, mat.n // 16 + 3):
        cls = capi.rate_pattern(code, 0, s, 21)
        seeds = oracle.trial_seeds(77 + s, 32)
        a, b, fill, ex = frames_of(ctx, mat, cls, seeds, q)
        it, res, dec = ctx.reconcile_adapted(code, params, cls, a, b, fill_packed(cls, fill), ex)
        assert_decoder(ctx, expect, (key, s, fused))
        want = restated_outcomes(lambda llr, syn: oracle.sum_product(g, llr, syn, max_it=MAX_IT, thr=THR), mat, cls, a, b, fill, ex)
        assert_equal((key, s, fused), want, it, res, dec, mat.n - s)
    cls = capi.rate_pattern(code, 8, 0, 21)
    a, b, fill, ex = frames_of(ctx, mat, cls, oracle.trial_seeds(5, 4), q)
    with pytest.raises(capi.QlbError) as e:
        ctx.reconcile_adapted(code, params, cls, a, b, fill_packed(cls, fill), ex)
    assert e.value.code == 3 and ("fp64 fused" if fused else "fp64 divides") in e.value.message


# ---- fp32 accurate with puncturing --------------------------------------------------------------------------------------------------
def test_fp32_puncturing_resident_equals_streaming(ctx, oracle):
    mat, g, code = code_for("north_star")
    p, s = policy(mat.n, mat.m, 0.05, 0.1, 1.1)
    cls = capi.rate_pattern(code, p, s, 5)
    seeds = oracle.trial_seeds(31, 1024)
    a, b, fill, ex = frames_of(ctx, mat, cls, seeds, 0.05)
    fp = fill_packed(cls, fill)
    it, res, dec = ctx.reconcile_adapted(code, capi.make_params(32, 100, THR, True), cls, a, b, fp, ex)
    assert_decoder(ctx, "resident_f32 bw=3", "resident")
    it_s, res_s, dec_s = ctx.reconcile_adapted(code, capi.make_params(32, 100, THR, True, tier=3), cls, a, b, fp, ex)
    assert_decoder(ctx, "stream_f32", "stream")
    assert (it == it_s).all() and (res == res_s).all() and (dec == dec_s).all()
    n = mat.n - p - s
    keys_equal = (capi.unpack_bits(dec, n) == capi.unpack_bits(a, n)).all(axis=1)
    assert (keys_equal == ((res & 2) != 0)).all()


def test_fp32_all_frames_converge_at_q003_p1024(ctx, oracle):
    """q = 0.03, delta = 0.1, f* = 1.1: the policy punctures all 1 024 modulated positions, R = 0.54."""
    mat, g, code = code_for("north_star")
    p, s = policy(mat.n, mat.m, 0.03, 0.1, 1.1)
    assert (p, s) == (1024, 0) and round(effective_rate(mat, p, s), 2) == 0.54
    cls = capi.rate_pattern(code, p, s, 5)
    it, res, ex = ctx.run_trials_adapted(code, capi.make_params(32, 100, THR, True), cls, oracle.trial_seeds(777, 1024), 0.03)
    assert ctx.last_decoder.startswith("resident_f32 bw=3")
    assert (res == 3).all(), (np.flatnonzero(res != 3)[:16], np.bincount(it))


# ---- errors and corners -------------------------------------------------------------------------------------------------------------
def test_errors(ctx, oracle):
    mat, g, code = code_for("perm3_n1024")
    ms = capi.make_params(32, MAX_IT, THR, True, min_sum_scale=ALPHA)
    cls = capi.rate_pattern(code, 10, 20, 1)
    n = mat.n - 30
    a, b, fill, ex = frames_of(ctx, mat, cls, oracle.trial_seeds(9, 4), 0.05)
    fp = capi.pack_bits(fill, 30)

    def error_of(f):
        with pytest.raises(capi.QlbError) as e:
            f()
        return e.value.code, e.value.message

    rc, msg = error_of(lambda: ctx.reconcile_adapted(code, ms, cls, a, b, fp, 0.0))
    assert rc == 4 and f"Key size '{n}' is too small for QBER." in msg
    rc, msg = error_of(lambda: ctx.run_trials_adapted(code, ms, cls, oracle.trial_seeds(9, 4), 0.5 / n))
    assert rc == 4 and f"Key size '{n}'" in msg
    rc, msg = error_of(lambda: ctx.reconcile_adapted(code, capi.make_params(32, MAX_IT, THR, False, min_sum_scale=ALPHA), cls, a, b, fp, ex))
    assert rc == 1 and "enable_threshold" in msg
    rc, msg = error_of(lambda: ctx.reconcile_adapted(code, capi.make_params(32, MAX_IT, THR, True, fast_math=True), cls, a, b, fp, ex))
    assert rc == 3 and "fp32 fast math" in msg
    bad = cls.copy()
    bad[17] = 3
    rc, msg = error_of(lambda: ctx.run_trials_adapted(code, ms, bad, oracle.trial_seeds(9, 4), 0.05))
    assert rc == 1 and "pos_class[17] = 3" in msg
    rc, msg = error_of(lambda: ctx.run_trials_adapted(code, ms, np.full(mat.n, capi.POS_SHORTENED, np.uint8), oracle.trial_seeds(9, 4), 0.05))
    assert rc == 1 and "no key position" in msg
    # shortening only with the clamp off is refused too; no modulation at all is plain syndrome coding and needs no clamp
    sh = capi.rate_pattern(code, 0, 5, 1)
    rc, _ = error_of(lambda: ctx.run_trials_adapted(code, capi.make_params(32, MAX_IT, THR, False), sh, oracle.trial_seeds(9, 4), 0.05))
    assert rc == 1
    it, res, ex0 = ctx.run_trials_adapted(code, capi.make_params(64, MAX_IT, THR, False), np.zeros(mat.n, np.uint8), oracle.trial_seeds(9, 8), 0.05)
    it_r, res_r, ex_r = ctx.run_trials(code, capi.make_params(64, MAX_IT, THR, False), oracle.trial_seeds(9, 8), 0.05)
    assert ex0 == ex_r and (it == it_r).all() and (res == res_r).all()


# ---- the C++ sweep ------------------------------------------------------------------------------------------------------------------
GRID = [0.03, 0.04, 0.05, 0.06, 0.07, 0.08, 0.09, 0.1, 0.11]


def _sweep(tmp_path, **kw):
    cfg = {"threads_number": 8, "trials_number": 64, "use_config_simulation_seed": True, "simulation_seed": 777,
           "interactive_mode": False, "sum_product_max_iterations": 100, "use_dense_matrices": False, "trace_qkd_ldpc": False,
           "trace_sum_product": False, "trace_sum_product_llr": False, "enable_sum_product_msg_llr_threshold": True,
           "sum_product_msg_llr_threshold": 100.0, "device_precision": 32,
           "code_rate_QBER_parameters": [{"code_rate": 0.5, "QBER_begin": 0.03, "QBER_end": 0.12, "QBER_step": 0.01}]}
    cfg.update(kw)
    (tmp_path / "config.json").write_text(json.dumps(cfg))
    (tmp_path / "alist_sparse_matrices").mkdir()
    shutil.copy(codes.materialize()[NS], tmp_path / "alist_sparse_matrices")
    p = subprocess.run([str(build.SIM_PATH), str(tmp_path)], capture_output=True, text=True)
    assert p.returncode == 0, p.stderr
    csv = sorted((tmp_path / "results").glob("ldpc*.csv"))[0].read_text().splitlines()
    side = sorted((tmp_path / "results").glob("throughput*.csv"))[0].read_text().splitlines()
    return csv, side


OLD_SIDE_HEADER = ("SIM;MATRIX_FILENAME;M;N;QBER;FRAMES;SECONDS;FRAMES_PER_S;SIFTED_MBIT_PER_S;FRAME_ITERATIONS;MEAN_ITERATIONS;"
                   "EFFICIENCY_F;LEAKED_BITS_PER_FRAME;GPUS;PRECISION")


def test_cpp_sweep_with_rate_adaptation(ctx, oracle, tmp_path):
    build.build_all()
    mat, g, code = code_for("north_star")
    ra = {"modulated_fraction": 0.1, "target_efficiency": 1.2, "pattern_seed": 5}
    csv, side = _sweep(tmp_path, device_rate_adaptation=ra, device_fp32_min_sum_scale=ALPHA)
    assert csv[0].count(";") == 13 and side[0] == OLD_SIDE_HEADER + ";PUNCTURED;SHORTENED;KEY_BITS;EFFECTIVE_RATE"
    rows, srows = [r.split(";") for r in csv[1:]], [r.split(";") for r in side[1:]]
    assert len(rows) == len(GRID) == len(srows)
    seeds = oracle.trial_seeds(777, 64)
    params = capi.make_params(32, 100, THR, True, min_sum_scale=ALPHA)
    for pt, (row, srow, q) in enumerate(zip(rows, srows, GRID)):
        p, s = policy(mat.n, mat.m, q, 0.1, 1.2)
        n = mat.n - p - s
        assert float(row[6]) == pytest.approx(int(n * q) / n, rel=1e-5)
        cls = capi.rate_pattern(code, p, s, 5)
        it, res, _ = ctx.run_trials_adapted(code, params, cls, seeds, q, seed_offset=pt)
        out3 = np.stack([it, res & 1, (res >> 1) & 1], axis=1).astype(np.uint64)
        st = oracle.point_stats(out3, 100)
        want = [st["mean"], st["std_dev"], st["min"], st["max"], st["ratio_sp"], st["ratio_ldpc"], 1.0 - st["ratio_ldpc"]]
        assert np.allclose([float(x) for x in row[7:14]], want, rtol=1e-5, atol=1e-6), (q, row, want)
        assert [int(x) for x in srow[15:18]] == [p, s, n] and int(srow[12]) == mat.m - p
        h2 = -float(srow[4]) * np.log2(float(srow[4])) - (1 - float(srow[4])) * np.log2(1 - float(srow[4]))
        assert float(srow[11]) == pytest.approx((mat.m - p) / (n * h2), rel=1e-5)
        assert float(srow[18]) == pytest.approx(effective_rate(mat, p, s), rel=1e-5)


def test_cpp_sweep_without_key_keeps_its_files(tmp_path):
    """Without the key the side file keeps its 15 columns, N key bits and M leaked bits (the reference-format CSV is held
    byte-identical to the reference's by test_host_cpp.py)."""
    build.build_all()
    mat = codes.load_npz(NS)
    csv, side = _sweep(tmp_path, trials_number=16)
    assert side[0] == OLD_SIDE_HEADER and all(r.count(";") == 14 for r in side)
    for r in side[1:]:
        f = r.split(";")
        q = float(f[4])
        h2 = -q * np.log2(q) - (1 - q) * np.log2(1 - q)
        assert int(f[12]) == mat.m and float(f[11]) == pytest.approx(mat.m / mat.n / h2, rel=1e-5)
