"""Rate-adaptive reconciliation on the host, no GPU: qlb_rate_pattern against a numpy restatement of the untainted walk, the
sweep's (punctured, shortened) policy and the device_rate_adaptation config key. The restatements here (pattern, frame
assembly, fill stream) are also what test_gpu_rate_adaptive.py holds the device to."""
import json
import math
import re
import shutil
import subprocess

import numpy as np
import pytest

from conftest import GOLD, NS
from qkd_ldpc_b200 import build, capi, codes, workload

_M64 = (1 << 64) - 1


def restated_pattern(mat, p, s, seed):
    """-> class array, or the number of untainted positions when the walk finds fewer than p."""
    r = workload.trial_seeds(seed, mat.n)
    order = np.lexsort((np.arange(mat.n), r))  # by (r_j, j)
    tainted = np.zeros(mat.m, bool)
    cls = np.zeros(mat.n, np.uint8)
    found = 0
    for i in order:
        if found == p:
            break
        checks = mat.row_idx[mat.col_ptr[i]:mat.col_ptr[i + 1]]
        if not tainted[checks].any():
            cls[i] = capi.POS_PUNCTURED
            tainted[checks] = True
            found += 1
    if found < p:
        return found
    cls[[i for i in order if cls[i] == capi.POS_KEY][:s]] = capi.POS_SHORTENED
    return cls


def fill_bits(seed, offset, count):
    """Fill bit k of a run-trials frame: the top bit of the k-th output of Xoshiro256PlusPlus(~(seed + offset))."""
    return (workload.trial_seeds(~(int(seed) + int(offset)) & _M64, count) >> np.uint64(63)).astype(np.int32)


def assemble(mat, cls, alice_key, bob_key, fill, q_exact, thr):
    """One frame's LLR row and target syndrome, restated from the header's definition (n-bit keys, (p+s)-bit fill, unpacked)."""
    key_pos, fill_pos = np.flatnonzero(cls == capi.POS_KEY), np.flatnonzero(cls != capi.POS_KEY)
    lp = math.log((1.0 - q_exact) / q_exact)
    llr = np.zeros(mat.n)
    word = np.zeros(mat.n, np.int32)
    llr[key_pos] = np.where(bob_key == 1, -lp, lp)
    word[key_pos] = alice_key
    word[fill_pos] = fill
    short = cls == capi.POS_SHORTENED
    llr[short] = np.where(word[short] == 1, -thr, thr)  # punctured positions keep +0.0
    chk_of = np.repeat(np.arange(mat.m), np.diff(mat.row_ptr))
    syn = np.zeros(mat.m, np.int32)
    np.bitwise_xor.at(syn, chk_of, word[mat.col_idx])
    return llr, syn


def effective_rate(mat, p, s):
    return (mat.n - mat.m - s) / (mat.n - p - s)


def _codes():
    return {"dense_n7": codes.load_npz("dense_n7_m3"), "peg_n96": codes.read_alist(GOLD / "trace" / "peg_n96_m48.alist"),
            "north_star": codes.load_npz(NS)}


@pytest.fixture(scope="module")
def dev_code():
    mats = _codes()
    return {k: (m, capi.Code.from_graph(m)) for k, m in mats.items()}


def _untainted(mat, seed):
    return restated_pattern(mat, mat.n, 0, seed)  # the walk never finds N: this is the count


@pytest.mark.parametrize("key", ["dense_n7", "peg_n96", "north_star"])
def test_pattern_equals_restatement(dev_code, key):
    mat, code = dev_code[key]
    for seed in (0, 1, 12345, 2**64 - 1):
        avail = _untainted(mat, seed)
        assert 1 <= avail < mat.n
        for p in sorted({0, 1, avail // 2, avail}):
            for s in sorted({0, 1, (mat.n - p) // 3, mat.n - p - 1}):
                want = restated_pattern(mat, p, s, seed)
                got = capi.rate_pattern(code, p, s, seed)
                assert (got == want).all(), (key, seed, p, s)
                assert (got == capi.POS_PUNCTURED).sum() == p and (got == capi.POS_SHORTENED).sum() == s


@pytest.mark.parametrize("key", ["dense_n7", "peg_n96", "north_star"])
def test_pattern_untainted_and_prefix_compatible(dev_code, key):
    mat, code = dev_code[key]
    seed = 666
    avail = _untainted(mat, seed)
    prev = None
    for p in np.unique(np.linspace(0, avail, 6).astype(int)):
        punct = capi.rate_pattern(code, int(p), 0, seed) == capi.POS_PUNCTURED
        # every check has at most one punctured bit
        chk_of = np.repeat(np.arange(mat.m), np.diff(mat.row_ptr))
        assert np.bincount(chk_of[punct[mat.col_idx]], minlength=mat.m).max(initial=0) <= 1
        if prev is not None:
            assert (punct[prev]).all(), "the punctured set of a smaller p is a prefix of the larger one"
        prev = punct


def test_north_star_has_room_for_delta_tenth(dev_code):
    mat, _ = dev_code["north_star"]
    counts = [_untainted(mat, seed) for seed in range(5)]
    assert min(counts) >= 1024, counts


@pytest.mark.parametrize("key", ["dense_n7", "peg_n96", "north_star"])
def test_pattern_errors(dev_code, key):
    mat, code = dev_code[key]
    seed = 7
    avail = _untainted(mat, seed)
    with pytest.raises(capi.QlbError) as e:
        capi.rate_pattern(code, avail + 1, 0, seed)
    assert e.value.code == 3 and re.search(rf"\b{avail}\b", e.value.message), e.value.message
    for p, s in ((-1, 0), (0, -1), (0, mat.n), (1, mat.n - 1)):
        with pytest.raises(capi.QlbError) as e:
            capi.rate_pattern(code, p, s, seed)
        assert e.value.code == 1, (p, s)


def test_effective_rate_of_the_issue_example():
    mat = codes.load_npz(NS)
    assert round(effective_rate(mat, 1024, 0), 2) == 0.54


# ---- the sweep's policy ------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def sim():
    build.build_all()
    return build.SIM_PATH


def policy(n, m, q, delta, f):
    h2 = -q * math.log2(q) - (1 - q) * math.log2(1 - q)
    d = round(delta * n)
    s = min(max(round((1 - m / n - (1 - f * h2) * (1 - delta)) * n), 0), d)
    return d - s, s


def test_rate_split_worked_example(sim):
    """N = 10 240, M = 5 231, delta = 0.1, f* = 1.1. At q = 0.09: h2 = 0.43647, sigma = 0.48916 - 0.51988 * 0.9 = 0.02127,
    s = round(217.7) = 218 and p = 1024 - 218 = 806. At q = 0.03 sigma < 0: all 1 024 positions are punctured."""
    def split(q, delta=0.1, f=1.1, n=10240, m=5231):
        out = subprocess.run([str(sim), "--rate-split", str(n), str(m), repr(q), repr(delta), repr(f)], capture_output=True, text=True, check=True)
        return tuple(map(int, out.stdout.split()))
    assert split(0.09) == (806, 218)
    assert split(0.03) == (1024, 0)
    assert split(0.05, delta=0.0) == (0, 0)
    for q in (0.03, 0.05, 0.07, 0.085, 0.09):
        for f in (1.1, 1.2, 1.5):
            assert split(q, f=f) == policy(10240, 5231, q, 0.1, f), (q, f)
    # the split hits the target: R = 1 - f h2(q) up to the rounding of s, when 0 < s < D
    p, s = split(0.09)
    h2 = -0.09 * math.log2(0.09) - 0.91 * math.log2(0.91)
    assert abs((10240 - 5231 - s) / (10240 - p - s) - (1 - 1.1 * h2)) < 1.0 / (10240 - 1024)


# ---- the config key ----------------------------------------------------------------------------------------------------------
def _cfg(**kw):
    cfg = {"threads_number": 8, "trials_number": 4, "use_config_simulation_seed": True, "simulation_seed": 777,
           "interactive_mode": False, "sum_product_max_iterations": 100, "use_dense_matrices": False, "trace_qkd_ldpc": False,
           "trace_sum_product": False, "trace_sum_product_llr": False, "enable_sum_product_msg_llr_threshold": True,
           "sum_product_msg_llr_threshold": 100.0,
           "code_rate_QBER_parameters": [{"code_rate": 0.5, "QBER_begin": 0.03, "QBER_end": 0.05, "QBER_step": 0.01}]}
    cfg.update(kw)
    return cfg


def _ra(delta=0.1, f=1.1, seed=5):
    return {"modulated_fraction": delta, "target_efficiency": f, "pattern_seed": seed}


def _run(sim, tmp_path, cfg):
    (tmp_path / "config.json").write_text(json.dumps(cfg))
    sub = tmp_path / "alist_sparse_matrices"
    sub.mkdir()
    shutil.copy(codes.materialize()[NS], sub)
    return subprocess.run([str(sim), str(tmp_path)], capture_output=True, text=True)


REJECTED = [
    ({"device_rate_adaptation": _ra(delta=1.0)}, "0 <= fraction < 1"),
    ({"device_rate_adaptation": _ra(delta=-0.1)}, "0 <= fraction < 1"),
    ({"device_rate_adaptation": _ra(f=0.0)}, "target_efficiency must be > 0"),
    ({"device_rate_adaptation": _ra(f=-1.0)}, "target_efficiency must be > 0"),
    ({"device_rate_adaptation": {"modulated_fraction": 0.1, "target_efficiency": 1.1}}, "key 'pattern_seed' not found"),
    ({"device_rate_adaptation": _ra(), "trace_qkd_ldpc": True}, "without interactive_mode and traces"),
    ({"device_rate_adaptation": _ra(), "trace_sum_product_llr": True}, "without interactive_mode and traces"),
    ({"device_rate_adaptation": _ra(), "interactive_mode": True}, "without interactive_mode and traces"),
    # q = 0.03 ... 0.05 at delta = 0.1, f* = 1.1 punctures: fp64 and fp32 fast math cannot
    ({"device_rate_adaptation": _ra()}, "puncturing needs device_precision 32"),
    ({"device_rate_adaptation": _ra(), "device_precision": 32, "device_fp32_fast_math": True}, "puncturing needs device_precision 32"),
    # f* = 3 shortens every modulated position: with the clamp off there is no finite prior for them
    ({"device_rate_adaptation": _ra(f=3.0), "device_precision": 32, "enable_sum_product_msg_llr_threshold": False},
     "shortening needs enable_sum_product_msg_llr_threshold"),
    # more punctured positions than the untainted walk finds (delta = 0.5 of N = 10 240)
    ({"device_rate_adaptation": _ra(delta=0.5), "device_precision": 32}, "untainted walk of this seed finds"),
]


@pytest.mark.parametrize("keys,msg", REJECTED)
def test_config_key_rejections(sim, tmp_path, keys, msg):
    p = _run(sim, tmp_path, _cfg(**keys))
    assert p.returncode != 0 and msg in p.stderr, p.stderr


@pytest.mark.parametrize("keys", [{"device_rate_adaptation": _ra(), "device_precision": 32},
                                  {"device_rate_adaptation": _ra(), "device_precision": 32, "device_fp32_min_sum_scale": 0.8125},
                                  {"device_rate_adaptation": _ra(f=3.0)},  # shortening only: fp64 takes it
                                  {"device_rate_adaptation": _ra(delta=0.0)},
                                  {"device_rate_adaptation": _ra(seed=2**64 - 1), "device_precision": 32}])
def test_config_key_accepted(sim, tmp_path, lib, keys):
    """Valid settings pass the config reader and the pattern set-up: without a GPU the run then stops at the device."""
    if lib.qlb_device_count() > 0:
        pytest.skip("a GPU is present: the accepted key runs a sweep in test_gpu_rate_adaptive.py")
    p = _run(sim, tmp_path, _cfg(**keys))
    assert p.returncode != 0 and "no CPU decoder" in p.stderr and "device_rate_adaptation" not in p.stderr, p.stderr
