"""fp32 normalized min-sum (QLB_FLAG_F32_MIN_SUM) on every decoder that runs it, against the CPU restatement
(min_sum_restatement.c): iterations, both flags, every decoded bit (failed frames included) and Alice's syndromes must be equal
on every frame. Each case names the decoder it expects (qlb_ctx_last_decoder). Codes come from test_gpu_decoder_paths.py, plus an
irregular code (bit weights 2, 3, 4 and 6) for the any-weight paths."""
import functools
import json
import shutil
import subprocess

import numpy as np
import pytest

from min_sum_restatement import MinSumRestatement
from qkd_ldpc_b200 import build, capi, codes, workload
from test_gpu_codes import graph_of
from test_gpu_decoder_paths import BUILDERS, QBERS, assert_decoder, code_of
from conftest import NS

pytestmark = pytest.mark.gpu
MAX_IT = 40
SCALES = (1.0, 0.75)


@pytest.fixture(scope="module")
def msr():
    return MinSumRestatement()


def irregular_code(n=2048, m=1280, seed=99):
    """Bit weights 2 / 3 / 4 / 6, each bit on distinct random checks; check weights at most 16."""
    rng = np.random.default_rng(seed)
    bw = rng.choice([2, 3, 4, 6], size=n, p=[0.3, 0.4, 0.2, 0.1])
    bit_lists = [sorted(rng.choice(m, w, replace=False).tolist()) for w in bw]
    check_lists = [[] for _ in range(m)]
    for i, r in enumerate(bit_lists):
        for c in r:
            check_lists[c].append(i)
    return codes.Matrix.from_lists(n, check_lists, bit_lists, f"irregular_n{n}_seed{seed}")


@functools.lru_cache(maxsize=None)
def code_for(key):
    if key in BUILDERS:
        return code_of(key)
    mat = irregular_code()
    return mat, graph_of(mat), capi.Code.from_graph(mat)


QB = dict(QBERS, ladder_n4096=(0.03, 0.05), north_star=(0.05, 0.08), irreg_n2048=(0.02, 0.05), perm3_n1024=(0.03, 0.07))


def params(scale, **kw):
    kw.setdefault("max_iterations", MAX_IT)
    return capi.make_params(32, kw.pop("max_iterations"), kw.pop("threshold", 100.0), kw.pop("enable_threshold", True),
                            min_sum_scale=scale, **kw)


def want_trials(msr, oracle, g, seeds, q, scale, **kw):
    """restatement outcomes (iterations, flags, decoded bits, Alice's syndromes) of the reference's frames"""
    out3, dec = msr.run_trials(g, q, seeds, scale, threads=8, max_it=kw.get("max_it", MAX_IT), thr=kw.get("thr", 100.0),
                               enable_thr=kw.get("enable_thr", True), want_decoded=True)
    syn = None
    if kw.get("want_syn", True):
        syn = np.stack([oracle.syndrome(g, oracle.generate(int(s), g.n, q)[0]) for s in seeds])
    return out3, dec, syn


def assert_equal_outcomes(case, mat, want, it, res, dec_packed, syn_packed=None):
    out3, wdec, wsyn = want
    assert (it == out3[:, 0]).all(), (case, np.flatnonzero(it != out3[:, 0])[:8])
    assert ((res & 1) == out3[:, 1]).all() and (((res >> 1) & 1) == out3[:, 2]).all(), case
    assert (capi.unpack_bits(dec_packed, mat.n) == wdec).all(), case
    if syn_packed is not None:
        assert (capi.unpack_bits(syn_packed, mat.m) == wsyn).all(), case


# ---- a. every path: reconcile (packed and unpacked) and run-trials entries, two QBERs, alpha = 1 and 0.75 ----------------------
CASES = [
    ("perm2_n4096", {}, 96, "resident_f32minsum bw=2"),
    ("ladder_n4096", {}, 96, "resident_f32minsum bw=3"),
    ("perm4_n4096", {}, 96, "resident_f32minsum bw=4"),
    ("north_star", {}, 96, "resident_f32minsum bw=3"),
    ("perm3_n1024", {"tier": 0}, 96, "generic f32minsum tier=0 shape=8"),
    ("perm3_n1024", {"tier": 1}, 96, "generic f32minsum tier=1 shape=8"),
    ("ladder_n4096", {"tier": 0}, 96, "generic f32minsum tier=0 shape=16"),
    ("ladder_n4096", {"tier": 1}, 96, "generic f32minsum tier=1 shape=16"),
    ("ladder_n4096", {"tier": 2}, 96, "generic f32minsum tier=2 shape=0"),
    ("irreg_n2048", {"tier": 0}, 96, "generic f32minsum tier=0 shape=0"),
    ("irreg_n2048", {"tier": 2}, 96, "generic f32minsum tier=2 shape=0"),
    ("perm3_n10000", {}, 96, "stream_f32 vec=4 bw=3"),
    ("perm3_n4001", {}, 24, "stream_f32 vec=1 bw=3"),
    ("perm2_n4096", {"tier": 3}, 96, "stream_f32 vec=4 bw=2"),
    ("perm4_n4096", {"tier": 3}, 24, "stream_f32 vec=1 bw=4"),
    ("ladder_n4096", {"tier": 3}, 96, "stream_f32 vec=4 bw=3"),
    ("irreg_n2048", {}, 96, "stream_f32 vec=4 bw=any"),
    ("irreg_n2048", {}, 24, "stream_f32 vec=1 bw=any"),
]


def _case_id(c):
    return f"{c[0]}-{c[2]}-" + "-".join(f"{k}={v}" for k, v in c[1].items())


def test_irregular_code_shape():
    mat = irregular_code()
    assert sorted(set(np.diff(mat.col_ptr).tolist())) == [2, 3, 4, 6] and np.diff(mat.row_ptr).max() <= 16


@pytest.mark.parametrize("key,kw,frames,expect", CASES, ids=[_case_id(c) for c in CASES])
def test_min_sum_path_matches_restatement(ctx, oracle, msr, key, kw, frames, expect):
    mat, g, code = code_for(key)
    for pt, q in enumerate(QB[key]):
        seeds = oracle.trial_seeds(808 + pt, frames)
        a, b, ex = ctx.generate(mat.n, seeds, q)
        for scale in SCALES:
            case = (key, kw, q, scale)
            want = want_trials(msr, oracle, g, seeds, q, scale)
            p = params(scale, **kw)
            it, res, dec, syn = ctx.reconcile_packed(code, p, a, b, np.full(frames, ex), want_decoded=True, want_syndrome=True)
            assert_decoder(ctx, expect, case)
            assert_equal_outcomes(case, mat, want, it, res, dec, syn)
            # unpacked host entry, first 8 frames
            A, B = capi.unpack_bits(a[:8], mat.n), capi.unpack_bits(b[:8], mat.n)
            it_u, res_u, dec_u, syn_u = ctx.reconcile(code, p, A, B, ex, want_decoded=True, want_syndrome=True)
            assert (it_u == it[:8]).all() and (res_u == res[:8]).all() and (dec_u == want[1][:8]).all() and (syn_u == want[2][:8]).all()
            # run-trials entry: keys drawn on the device from the same seeds
            it_t, res_t, ex_t = ctx.run_trials(code, p, seeds, q)
            assert ex_t == ex and (it_t == it).all() and (res_t == res).all(), case


# ---- b. sum-product entry: zero, +-inf and NaN LLRs, clamp on and off -----------------------------------------------------------
SP_PATHS = [("ladder_n4096", {}, "resident_f32minsum bw=3"), ("ladder_n4096", {"tier": 0}, "generic f32minsum tier=0 shape=16"),
            ("ladder_n4096", {"tier": 2}, "generic f32minsum tier=2 shape=0"), ("ladder_n4096", {"tier": 3}, "stream_f32 vec=1 bw=3"),
            ("irreg_n2048", {}, "stream_f32 vec=1 bw=any"), ("irreg_n2048", {"tier": 1}, "generic f32minsum tier=1 shape=0")]


def llr_frames(mat, rng, frames=12):
    bits = (rng.random((frames, mat.n)) < 0.5).astype(np.int32)
    llr = rng.normal(2.5, 2.0, (frames, mat.n))
    kinds = ["random", "zeros", "inf", "nan", "all_zero", "subnormal"]
    for f in range(frames):
        kind = kinds[f % len(kinds)]
        if kind == "zeros":
            llr[f, rng.random(mat.n) < 0.2] = 0.0
        elif kind == "inf":
            llr[f, rng.random(mat.n) < 0.1] = np.inf
            llr[f, rng.random(mat.n) < 0.05] = -np.inf
        elif kind == "nan":
            llr[f, rng.random(mat.n) < 0.05] = np.nan
        elif kind == "all_zero":
            llr[f] = 0.0
        elif kind == "subnormal":
            llr[f, rng.random(mat.n) < 0.3] = 1e-40
    llr = np.where(bits == 1, -llr, llr)
    chk_of = np.repeat(np.arange(mat.m), np.diff(mat.row_ptr))
    syn = np.zeros((frames, mat.m), np.int32)
    for f in range(frames):
        np.bitwise_xor.at(syn[f], chk_of, bits[f][mat.col_idx])
    return llr, syn


@pytest.mark.parametrize("key,kw,expect", SP_PATHS, ids=[f"{k}-{e.split()[0]}-{'-'.join(map(str, kw.values()))}" for k, kw, e in SP_PATHS])
@pytest.mark.parametrize("clamp", [True, False])
def test_sum_product_entry_special_llrs(ctx, msr, key, kw, expect, clamp):
    mat, g, code = code_for(key)
    rng = np.random.default_rng([mat.n, int(clamp), len(kw)])
    llr, syn = llr_frames(mat, rng)
    for scale in SCALES:
        p = params(scale, threshold=8.0, enable_threshold=clamp, **kw)
        it, res, bits = ctx.sum_product(code, p, llr, syn)
        assert_decoder(ctx, expect, (key, kw, clamp))
        for f in range(llr.shape[0]):
            w_it, w_ok, w_bits = msr.sum_product(g, llr[f], syn[f], scale, max_it=MAX_IT, thr=8.0, enable_thr=clamp)
            assert (it[f], bool(res[f] & 1)) == (w_it, w_ok), (key, kw, clamp, scale, f)
            assert (bits[f] == w_bits).all(), (key, kw, clamp, scale, f)


# ---- c. corners ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kw,expect", [({}, "resident_f32minsum bw=3"), ({"tier": 1}, "generic f32minsum tier=1 shape=16"),
                                       ({"tier": 3}, "stream_f32 vec=4 bw=3")])
def test_clamp_off_ladder_reconcile(ctx, oracle, msr, kw, expect):
    """Weight-1 checks send +inf with the clamp off; min-sum has one definition for what follows, so every path still agrees."""
    mat, g, code = code_for("ladder_n4096")
    seeds = oracle.trial_seeds(4242, 64)
    for q in (0.03, 0.05):
        a, b, ex = ctx.generate(mat.n, seeds, q)
        for scale in SCALES:
            want = want_trials(msr, oracle, g, seeds, q, scale, enable_thr=False)
            it, res, dec, syn = ctx.reconcile_packed(code, params(scale, enable_threshold=False, **kw), a, b, np.full(64, ex),
                                                     want_decoded=True, want_syndrome=True)
            assert_decoder(ctx, expect, kw)
            assert_equal_outcomes((kw, q, scale), mat, want, it, res, dec, syn)


@pytest.mark.parametrize("key,kw", [("perm3_n1024", {}), ("perm3_n1024", {"tier": 2}), ("perm3_n4001", {})])
def test_qber_half(ctx, oracle, msr, key, kw):
    """QBER 0.5: the log prior is 0, every prior is +-0 and the sign of a zero matters to the check's XOR."""
    mat, g, code = code_for(key)
    seeds = oracle.trial_seeds(55, 40)
    a, b, ex = ctx.generate(mat.n, seeds, 0.5)
    want = want_trials(msr, oracle, g, seeds, 0.5, 0.75, max_it=10)
    it, res, dec, syn = ctx.reconcile_packed(code, params(0.75, max_iterations=10, **kw), a, b, np.full(40, ex), want_decoded=True,
                                             want_syndrome=True)
    assert_equal_outcomes((key, kw), mat, want, it, res, dec, syn)


@pytest.mark.parametrize("kw", [{"stream_max_bundles": 1}, {"stream_no_repack": True}, {"stream_max_bundles": 2, "stream_no_repack": True}, {}])
def test_stream_waves_and_repacks(ctx, oracle, msr, kw):
    mat, g, code = code_for("perm3_n10000")
    frames, q = 1100, 0.08
    seeds = oracle.trial_seeds(9090, frames)
    a, b, ex = ctx.generate(mat.n, seeds, q)
    want = want_trials(msr, oracle, g, seeds, q, 0.75)
    it, res, dec, syn = ctx.reconcile_packed(code, params(0.75, **kw), a, b, np.full(frames, ex), want_decoded=True, want_syndrome=True)
    used = assert_decoder(ctx, "stream_f32 vec=4 bw=3", kw)
    if kw.get("stream_max_bundles"):
        assert "waves=1 " not in used, used
    assert ("repack=0" in used) == bool(kw.get("stream_no_repack")), used
    assert_equal_outcomes(kw, mat, want, it, res, dec, syn)


@pytest.mark.parametrize("key,kw,expect", [("north_star", {}, "resident_f32minsum"), ("perm3_n10000", {}, "stream_f32"),
                                            ("perm3_n1024", {"tier": 0}, "generic f32minsum")])
def test_batch_slices(ctx, oracle, msr, key, kw, expect):
    """A frame's outcome does not depend on the batch it is decoded in: slices of 1, 31, 33 and 129 frames."""
    mat, g, code = code_for(key)
    q = QB[key][1]
    seeds = oracle.trial_seeds(3131, 194)
    a, b, ex = ctx.generate(mat.n, seeds, q)
    want = want_trials(msr, oracle, g, seeds, q, 0.75)
    lo = 0
    for size in (1, 31, 33, 129):
        sl = slice(lo, lo + size)
        it, res, dec, syn = ctx.reconcile_packed(code, params(0.75, **kw), a[sl], b[sl], np.full(size, ex), want_decoded=True,
                                                 want_syndrome=True)
        assert_decoder(ctx, expect, (key, size))
        assert_equal_outcomes((key, size), mat, tuple(w[sl] for w in want), it, res, dec, syn)
        lo += size


@pytest.mark.parametrize("key,threads", [("north_star", (320, 512, 768, 1024)), ("ladder_n4096", (128, 256, 608, 1024))])
def test_block_threads(ctx, oracle, msr, key, threads):
    mat, g, code = code_for(key)
    q = QB[key][1]
    seeds = oracle.trial_seeds(6161, 148)
    a, b, ex = ctx.generate(mat.n, seeds, q)
    want = want_trials(msr, oracle, g, seeds, q, 0.75)
    for t in threads:
        it, res, dec, syn = ctx.reconcile_packed(code, params(0.75, block_threads=t), a, b, np.full(148, ex), want_decoded=True,
                                                 want_syndrome=True)
        assert f"threads={t}" in assert_decoder(ctx, "resident_f32minsum bw=3", t)
        assert_equal_outcomes((key, t), mat, want, it, res, dec, syn)


@pytest.mark.parametrize("key", ["north_star", "perm3_n10000"])
def test_device_entry(ctx, oracle, msr, key):
    """qlb_reconcile_device with device buffers and the caller's log prior equals the restatement."""
    import torch
    mat, g, code = code_for(key)
    frames, q = 200, QB[key][1]
    dev = torch.device("cuda", 0)
    seeds = oracle.trial_seeds(7070, frames)
    a, b, ex = ctx.generate(mat.n, seeds, q)
    want = want_trials(msr, oracle, g, seeds, q, 0.75)
    d_a = torch.from_numpy(a.view(np.int32)).to(dev)
    d_b = torch.from_numpy(b.view(np.int32)).to(dev)
    d_lp = torch.full((frames,), workload.log_prior(ex), dtype=torch.float64, device=dev)
    d_it = torch.zeros(frames, dtype=torch.int32, device=dev)
    d_res = torch.zeros(frames, dtype=torch.uint8, device=dev)
    d_dec = torch.zeros_like(d_a)
    d_syn = torch.zeros((frames, code.words_m), dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    ctx.reconcile_device(code, params(0.75), frames, d_a.data_ptr(), d_b.data_ptr(), d_lp.data_ptr(), d_it.data_ptr(),
                         d_res.data_ptr(), d_dec.data_ptr(), d_syn.data_ptr())
    ctx.synchronize()
    assert_equal_outcomes(key, mat, want, d_it.cpu().numpy().view(np.uint32), d_res.cpu().numpy(), d_dec.cpu().numpy().view(np.uint32),
                          d_syn.cpu().numpy().view(np.uint32))


REJECT = [
    dict(precision=64, flags=capi.FLAG_F32_MIN_SUM, scale=0.75),                                   # fp64
    dict(precision=32, flags=capi.FLAG_F32_MIN_SUM | capi.FLAG_F32_FAST_MATH, scale=0.75),         # with the fast rule
    dict(precision=32, flags=capi.FLAG_F32_MIN_SUM, scale=0.0),
    dict(precision=32, flags=capi.FLAG_F32_MIN_SUM, scale=-0.5),
    dict(precision=32, flags=capi.FLAG_F32_MIN_SUM, scale=1.0000001),
    dict(precision=32, flags=capi.FLAG_F32_MIN_SUM, scale=float("nan")),
    dict(precision=32, flags=capi.FLAG_F32_MIN_SUM, scale=float("inf")),
    dict(precision=32, flags=0, scale=0.75),                                                       # a scale without the flag
    dict(precision=64, flags=0, scale=0.5),
    dict(precision=32, flags=0, scale=float("nan")),
]


@pytest.mark.parametrize("bad", REJECT)
def test_parameter_rejections(ctx, oracle, bad):
    mat, g, code = code_for("perm3_n1024")
    a, b, ex = ctx.generate(mat.n, oracle.trial_seeds(1, 4), 0.05)
    p = capi.make_params(bad["precision"], 10, 100.0, True)
    p.flags, p.min_sum_scale = bad["flags"], bad["scale"]
    with pytest.raises(capi.QlbError) as e:
        ctx.reconcile_packed(code, p, a, b, np.full(4, ex))
    assert e.value.code == 1, e.value.message
    with pytest.raises(capi.QlbError) as e:
        ctx.sum_product(code, p, np.ones((1, mat.n)), np.zeros((1, mat.m), np.int32))
    assert e.value.code == 1
    with pytest.raises(capi.QlbError) as e:
        ctx.run_trials(code, p, oracle.trial_seeds(1, 4), 0.05)
    assert e.value.code == 1
    # the boundary value is accepted
    ctx.reconcile_packed(code, capi.make_params(32, 10, 100.0, True, min_sum_scale=1.0), a, b, np.full(4, ex))


# ---- d. a campaign on the benchmark code and the C++ sweep -----------------------------------------------------------------------
GRID = [0.03, 0.04, 0.05, 0.06, 0.07, 0.08, 0.09, 0.1, 0.11]


def test_campaign_north_star(ctx, oracle, msr):
    """9 QBER points x 512 reference frames (seeds of simulation seed 777, offset by the point's index, as the sweep draws them)."""
    mat, g, code = code_for("north_star")
    seeds = oracle.trial_seeds(777, 512)
    for pt, q in enumerate(GRID):
        s = seeds + np.uint64(pt)
        out3 = msr.run_trials(g, q, s, 0.75, threads=8, max_it=100)
        it, res, _ = ctx.run_trials(code, capi.make_params(32, 100, 100.0, True, min_sum_scale=0.75), s, q)
        assert ctx.last_decoder.startswith("resident_f32minsum bw=3")
        assert (it == out3[:, 0]).all() and ((res & 1) == out3[:, 1]).all() and (((res >> 1) & 1) == out3[:, 2]).all(), q


def test_cpp_sweep_with_min_sum_key(ctx, oracle, msr, tmp_path):
    build.build_all()
    cfg = {"threads_number": 8, "trials_number": 64, "use_config_simulation_seed": True, "simulation_seed": 777,
           "interactive_mode": False, "sum_product_max_iterations": 100, "use_dense_matrices": False, "trace_qkd_ldpc": False,
           "trace_sum_product": False, "trace_sum_product_llr": False, "enable_sum_product_msg_llr_threshold": True,
           "sum_product_msg_llr_threshold": 100.0, "device_precision": 32, "device_fp32_min_sum_scale": 0.75,
           "code_rate_QBER_parameters": [{"code_rate": 0.5, "QBER_begin": 0.03, "QBER_end": 0.12, "QBER_step": 0.01}]}
    (tmp_path / "config.json").write_text(json.dumps(cfg))
    (tmp_path / "alist_sparse_matrices").mkdir()
    shutil.copy(codes.materialize()[NS], tmp_path / "alist_sparse_matrices")
    p = subprocess.run([str(build.SIM_PATH), str(tmp_path)], capture_output=True, text=True)
    assert p.returncode == 0, p.stderr
    rows = [ln.split(";") for ln in sorted((tmp_path / "results").glob("ldpc*.csv"))[0].read_text().splitlines()[1:]]
    side = sorted((tmp_path / "results").glob("throughput*.csv"))[0].read_text()
    assert "fp32-min-sum" in side
    mat, g, _ = code_for("north_star")
    seeds = oracle.trial_seeds(777, 64)
    assert len(rows) == len(GRID)
    for pt, (row, q) in enumerate(zip(rows, GRID)):
        out3 = msr.run_trials(g, q, seeds + np.uint64(pt), 0.75, threads=8, max_it=100)
        st = oracle.point_stats(out3, 100)
        want = [st["mean"], st["std_dev"], st["min"], st["max"], st["ratio_sp"], st["ratio_ldpc"], 1.0 - st["ratio_ldpc"]]
        got = [float(x) for x in row[7:14]]
        assert np.allclose(got, want, rtol=1e-5, atol=1e-6), (q, got, want)
