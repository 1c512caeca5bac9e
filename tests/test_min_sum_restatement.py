"""The CPU restatement of the fp32 normalized min-sum rule (min_sum_restatement.c) against an independent numpy float32
restatement, the rule's parameters in the Python binding, and the sweep config key. No GPU needed.

The numpy form below is written from the rule's definition in include/qkd_ldpc_b200.h on its own: edge routing through
index tables instead of arrival counters, vectorised per check weight, the other-edge minimum by deleting a column."""
import json

import numpy as np
import pytest

from min_sum_restatement import MinSumRestatement
from oracle.bindings import Graph
from qkd_ldpc_b200 import build, capi, codes
from conftest import GOLD, NS

INF32 = np.float32(np.inf)


@pytest.fixture(scope="module")
def msr():
    return MinSumRestatement()


def graph_of(mat):
    return Graph(mat.n, mat.m, mat.row_ptr, mat.col_idx, mat.col_ptr, mat.row_idx)


CODES = {
    "dense_n7": lambda: codes.load_npz("dense_n7_m3"),
    "peg_n96": lambda: codes.read_alist(GOLD / "trace" / "peg_n96_m48.alist"),
    "perm3_n1024": lambda: codes.permutation_code(1024, 512, 3, 1024),
}


def np_min_sum(mat, prior, lsb0, syndrome, max_it, cap, scale):
    """(iterations, syndromes_match, bits) of the min-sum decode from fp32 priors, numpy float32 throughout."""
    n, m = mat.n, mat.m
    row_ptr, col_idx = np.asarray(mat.row_ptr), np.asarray(mat.col_idx)
    col_ptr, row_idx = np.asarray(mat.col_ptr), np.asarray(mat.row_idx)
    e = col_idx.size
    chk_of = np.repeat(np.arange(m), np.diff(row_ptr))  # check of each check-major edge
    # check-major edge p = (check j, bit b) -> bit-major position of the same edge (the code's two halves list the same edges)
    to_bit = np.empty(e, np.int64)
    pos = col_ptr[:-1].copy()
    for p in range(e):
        b = col_idx[p]
        to_bit[p] = pos[b]
        pos[b] += 1
    assert (row_idx[to_bit] == chk_of).all()
    bw = np.diff(col_ptr)
    cap = np.float32(cap)
    scale = np.float32(scale)
    prior = np.asarray(prior, np.float32)
    b2c = (prior[col_idx].view(np.uint32) & np.uint32(0xFFFFFFFE)) | np.asarray(lsb0, np.uint32)[col_idx]
    syn = np.asarray(syndrome, np.uint32)
    wts = np.diff(row_ptr)
    groups = [(w, np.flatnonzero(wts == w)) for w in np.unique(wts) if w > 0]
    bits = np.zeros(n, np.int32)
    for it in range(max_it):
        c2b_cm = np.zeros(e, np.float32)  # check-major
        for w, js in groups:
            idx = row_ptr[js][:, None] + np.arange(w)[None, :]
            u = b2c[idx]
            x = np.bitwise_xor.reduce(u, axis=1) ^ (syn[js] << np.uint32(31))
            a = u & np.uint32(0x7FFFFFFF)
            for k in range(w):
                rest = np.delete(a, k, axis=1)
                mu = rest.min(axis=1) if w > 1 else np.full(len(js), 0x7F800000, np.uint32)
                with np.errstate(invalid="ignore", over="ignore"):
                    mag = np.fmin(scale * mu.view(np.float32), cap)
                out = ((x ^ u[:, k]) & np.uint32(0x80000000)) | mag.view(np.uint32)
                c2b_cm[idx[:, k]] = out.view(np.float32)
        c2b = np.empty(e, np.float32)
        c2b[to_bit] = c2b_cm
        total = prior.copy()
        with np.errstate(invalid="ignore", over="ignore"):
            for a in range(bw.max()):
                has = bw > a
                total[has] = total[has] + c2b[col_ptr[:-1][has] + a]
            z = total <= 0
            bits = z.astype(np.int32)
            v = total[col_idx] - c2b_cm  # edge p: the total of its bit minus what its check sent
            v = np.fmin(np.fmax(v, -cap), cap)
        b2c = (v.view(np.uint32) & np.uint32(0xFFFFFFFE)) | z[col_idx].astype(np.uint32)
        par = np.zeros(m, np.uint32)
        np.bitwise_xor.at(par, chk_of, z[col_idx].astype(np.uint32))
        if (par == syn).all():
            return it + 1, True, bits
    return max_it, False, bits


def llr_sets(n, rng):
    """name -> LLR vector (float64), the special values the rule has to carry"""
    base = rng.normal(2.0, 2.5, n)
    sets = {"random": base, "zero": np.zeros(n), "random_with_zeros": np.where(rng.random(n) < 0.2, 0.0, base)}
    inf = base.copy()
    inf[rng.choice(n, max(1, n // 8), replace=False)] = np.inf
    inf[rng.choice(n, max(1, n // 8), replace=False)] = -np.inf
    sets["pm_inf"] = inf
    nan = base.copy()
    nan[rng.choice(n, max(1, n // 10), replace=False)] = np.nan
    sets["nan"] = nan
    sets["subnormal"] = np.where(rng.random(n) < 0.3, 1e-40, base)
    return sets


def np_prior_of_llr(llr):
    p = np.asarray(llr, np.float64).astype(np.float32)
    p[np.isnan(p)] = np.uint32(0x7FFFFFFF).view(np.float32)
    return p


@pytest.mark.parametrize("key", list(CODES))
@pytest.mark.parametrize("scale", [1.0, 0.75, 0.5])
@pytest.mark.parametrize("clamp", [True, False])
def test_sum_product_entry_equals_numpy(msr, key, scale, clamp):
    mat = CODES[key]()
    g = graph_of(mat)
    rng = np.random.default_rng([len(key), int(scale * 4), int(clamp), mat.n])
    thr, max_it = 6.0, 12
    cap = np.float32(thr) if clamp else INF32
    for name, llr in llr_sets(mat.n, rng).items():
        bits_true = (rng.random(mat.n) < 0.5).astype(np.int32)
        syn = np.zeros(mat.m, np.int32)
        for j in range(mat.m):
            syn[j] = bits_true[mat.col_idx[mat.row_ptr[j]:mat.row_ptr[j + 1]]].sum() & 1
        llr = np.where(bits_true == 1, -llr, llr)
        it, ok, bits = msr.sum_product(g, llr, syn, scale, max_it=max_it, thr=thr, enable_thr=clamp)
        w_it, w_ok, w_bits = np_min_sum(mat, np_prior_of_llr(llr), np.zeros(mat.n, np.int32), syn, max_it, cap, scale)
        assert (it, ok) == (w_it, w_ok), (key, name, scale, clamp)
        assert (bits == w_bits).all(), (key, name, scale, clamp)


@pytest.mark.parametrize("key", list(CODES))
@pytest.mark.parametrize("scale", [1.0, 0.75, 0.5])
def test_reconcile_entry_equals_numpy(msr, oracle, key, scale):
    mat = CODES[key]()
    g = graph_of(mat)
    q = 0.3 if mat.n < 100 else 0.06
    for seed in oracle.trial_seeds(31, 6):
        a, b, ex = oracle.generate(int(seed), mat.n, q)
        it, ok, keys, syn, dec = msr.qkd_ldpc(g, a, b, ex, scale, max_it=30)
        assert (syn == oracle.syndrome(g, a)).all()
        lp = np.float32(np.log((1.0 - ex) / ex))
        prior = np.where(b == 1, -lp, lp).astype(np.float32)
        w_it, w_ok, w_bits = np_min_sum(mat, prior, a, syn, 30, np.float32(100.0), scale)
        assert (it, ok) == (w_it, w_ok) and (dec == w_bits).all() and keys == bool((dec == a).all())


def test_run_trials_equals_reconcile(msr, oracle):
    mat = CODES["perm3_n1024"]()
    g = graph_of(mat)
    seeds = oracle.trial_seeds(777, 24)
    out3, dec = msr.run_trials(g, 0.07, seeds, 0.75, threads=4, max_it=40, want_decoded=True)
    for k, s in enumerate(seeds):
        a, b, ex = oracle.generate(int(s), mat.n, 0.07)
        it, ok, keys, _, d = msr.qkd_ldpc(g, a, b, ex, 0.75, max_it=40)
        assert tuple(out3[k]) == (it, ok, keys) and (dec[k] == d).all()


def test_hand_worked_check():
    """One check over three bits, syndrome 0, LLRs (2, -0.5, 3), alpha = 0.75, clamp off. The first messages are the priors
    (bit 0 already clear). The check's sign X = 1 (one negative message); the least other magnitudes are 0.5, 2, 0.5, scaled
    0.375, 1.5, 0.375, so the check sends -0.375, +1.5, -0.375. Totals 1.625, 1.0, 2.625: all decide 0, the check is
    satisfied after one iteration and bit 1's error is corrected."""
    mat = codes.Matrix.from_lists(3, [[0, 1, 2]], [[0], [0], [0]], "one_check")
    g = graph_of(mat)
    it, ok, bits = MinSumRestatement().sum_product(g, np.array([2.0, -0.5, 3.0]), np.zeros(1, np.int32), 0.75, max_it=5,
                                                   enable_thr=False)
    assert (it, ok) == (1, True) and bits.tolist() == [0, 0, 0]
    # with alpha = 0.5 the check sends +1.0 to bit 1: total 0.5, still 0; with a clamp at 0.25 it sends +0.25: total -0.25, bit 1 decides 1
    it, ok, bits = MinSumRestatement().sum_product(g, np.array([2.0, -0.5, 3.0]), np.zeros(1, np.int32), 0.5, max_it=1,
                                                   thr=0.25, enable_thr=True)
    assert (it, ok) == (1, False) and bits.tolist() == [0, 1, 0]


def test_make_params_writes_flag_and_scale():
    p = capi.make_params(32, 50, 20.0, True, min_sum_scale=0.75)
    assert p.flags & capi.FLAG_F32_MIN_SUM and not p.flags & capi.FLAG_F32_FAST_MATH
    assert p.min_sum_scale == 0.75 and p.precision == 32
    q = capi.make_params(32, 50, 20.0, True, min_sum_scale=1.0, tier=2)
    assert q.flags == capi.FLAG_F32_MIN_SUM | (3 << 8) and q.min_sum_scale == 1.0
    r = capi.make_params(32, 50, 20.0, True)
    assert r.flags == 0 and r.min_sum_scale == 0.0
    # same 40-byte layout: the scale sits where `reserved` was
    import ctypes
    assert ctypes.sizeof(capi.DecodeParams) == 40 and capi.DecodeParams.min_sum_scale.offset == 36


@pytest.fixture(scope="module")
def sim():
    build.build_all()
    return build.SIM_PATH


def _base_cfg(**kw):
    cfg = {"threads_number": 8, "trials_number": 4, "use_config_simulation_seed": True, "simulation_seed": 777,
           "interactive_mode": False, "sum_product_max_iterations": 100, "use_dense_matrices": False, "trace_qkd_ldpc": False,
           "trace_sum_product": False, "trace_sum_product_llr": False, "enable_sum_product_msg_llr_threshold": True,
           "sum_product_msg_llr_threshold": 100.0,
           "code_rate_QBER_parameters": [{"code_rate": 0.5, "QBER_begin": 0.03, "QBER_end": 0.05, "QBER_step": 0.01}]}
    cfg.update(kw)
    return cfg


REJECTED = [
    ({"device_precision": 32, "device_fp32_min_sum_scale": 1.5}, "must be 0 (off) or in (0, 1]"),
    ({"device_precision": 32, "device_fp32_min_sum_scale": -0.5}, "must be 0 (off) or in (0, 1]"),
    ({"device_fp32_min_sum_scale": 0.75}, "needs device_precision 32"),
    ({"device_precision": 64, "device_fp32_min_sum_scale": 0.75}, "needs device_precision 32"),
    ({"device_precision": 32, "device_fp32_fast_math": True, "device_fp32_min_sum_scale": 0.75}, "no device_fp32_fast_math"),
    ({"device_precision": 32, "device_fp32_min_sum_scale": "0.75"}, "type must be number"),
]


@pytest.mark.parametrize("keys,msg", REJECTED)
def test_config_key_rejections(sim, tmp_path, keys, msg):
    import subprocess
    import shutil
    (tmp_path / "config.json").write_text(json.dumps(_base_cfg(**keys)))
    sub = tmp_path / "alist_sparse_matrices"
    sub.mkdir()
    shutil.copy(codes.materialize()[NS], sub)
    p = subprocess.run([str(sim), str(tmp_path)], capture_output=True, text=True)
    assert p.returncode != 0 and msg in p.stderr, p.stderr


@pytest.mark.parametrize("keys", [{"device_precision": 32, "device_fp32_min_sum_scale": 0.75},
                                  {"device_precision": 32, "device_fp32_min_sum_scale": 1},
                                  {"device_precision": 64, "device_fp32_min_sum_scale": 0},
                                  {"device_precision": 32, "device_fp32_fast_math": True, "device_fp32_min_sum_scale": 0.0}])
def test_config_key_accepted(sim, tmp_path, lib, keys):
    """Valid settings pass the config reader: without a GPU the run then stops at the device, not at the config."""
    import subprocess
    import shutil
    if lib.qlb_device_count() > 0:
        pytest.skip("a GPU is present: the accepted key runs a sweep in test_gpu_min_sum.py")
    (tmp_path / "config.json").write_text(json.dumps(_base_cfg(**keys)))
    sub = tmp_path / "alist_sparse_matrices"
    sub.mkdir()
    shutil.copy(codes.materialize()[NS], sub)
    p = subprocess.run([str(sim), str(tmp_path)], capture_output=True, text=True)
    assert p.returncode != 0 and "no CPU decoder" in p.stderr and "device_fp32_min_sum_scale" not in p.stderr, p.stderr
