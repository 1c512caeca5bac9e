"""The streaming decoder (qlb_stream_split.cuh) at the batch sizes it is benchmarked at, against exact references.

Paths that depend only on the batch size, each crossed on purpose and checked to be crossed:
  - a repack with more than kRepackStage = 4 096 live frames: the message move runs a second staging chunk;
  - a wave of kMaxRepackGroups = 256 groups repacks (full s_cnt scan and s_old stage); at 313 groups repacking is off;
  - more groups than the setup and finalize grids (2 x SMs): one CTA handles a second group;
  - waves with repacks in each wave, the last wave smaller and ending in a partial group;
  - N = 100 000 (e >= 65 535: the large-code layout) in bundles of 4 groups with repacks.
A. N = 10 240, streaming forced with the tier-3 hook: every frame equals the SM-resident kernel of the same rule (which equals the
   reference: test_gpu_codes.py, test_gpu_min_sum.py).
B. N = 100 000, the default routes: fp64 against the generic fp64 kernel in the all-global tier on every frame and the oracle on a
   sample; fp32 against itself without repacks, in waves and in slices, and the oracle's flags; min-sum against the restatement.
Each case prints its decoder string, its repack schedule (restated from the iteration counts) and the device memory its context
holds. The context is this module's own and is closed at the end, so the scratch of these batches is not kept for the session."""
import os
import re
from types import SimpleNamespace

import numpy as np
import pytest

from min_sum_restatement import MinSumRestatement
from qkd_ldpc_b200 import capi, codes
from test_gpu_codes import graph_of
from test_gpu_decoder_paths import assert_decoder, code_of

pytestmark = pytest.mark.gpu
MAX_IT = 60
THREADS = os.cpu_count() or 8
STAGE = 4096  # kRepackStage: message values staged per chunk of a repack


@pytest.fixture(scope="module")
def sctx():
    import torch
    torch.cuda.init()
    c = capi.Context(0)
    c.free0 = torch.cuda.mem_get_info(0)[0]
    yield c
    c.close()


@pytest.fixture(scope="module")
def msr():
    return MinSumRestatement()


def held_gb(ctx):
    """device memory taken since the context was created (its grow-only scratch, mostly), GB"""
    import torch
    return (ctx.free0 - torch.cuda.mem_get_info(0)[0]) / 1e9


# ---- helpers ----------------------------------------------------------------------------------------------------------------------
def mixed_batch(ctx, oracle, n, classes, seed):
    """classes: [(qber, count)]. Keys of class k are drawn on the device from oracle.trial_seeds(seed + k, count); the batch is then
    permuted by a seeded generator, so that every group holds frames of every class. Per frame: seed, class QBER, exact QBER."""
    a, b, q, s, qc = [], [], [], [], []
    for k, (qber, cnt) in enumerate(classes):
        seeds = oracle.trial_seeds(seed + k, cnt)
        ak, bk, ex = ctx.generate(n, seeds, qber)
        a.append(ak); b.append(bk); q.append(np.full(cnt, ex)); s.append(seeds); qc.append(np.full(cnt, qber))
    perm = np.random.default_rng(seed).permutation(sum(c for _, c in classes))
    return SimpleNamespace(n=n, a=np.ascontiguousarray(np.concatenate(a)[perm]), b=np.ascontiguousarray(np.concatenate(b)[perm]),
                           q=np.concatenate(q)[perm], seed=np.concatenate(s)[perm], qclass=np.concatenate(qc)[perm])


def repack_schedule(iterations, G, groups_per_wave, max_it, pct=65, lag=0):
    """stream_repack_plan_kernel's decisions, restated from the per-frame iteration counts of a decode.
    Frame f starts in group f // G, column f % G (stream_setup_kernel); a wave holds `groups_per_wave` groups. stream_update_kernel(r)
    retires the frames whose iteration count is r, so after round r the live frames are those with iterations > r (failed frames
    report max_it). lag = 1 restates with iterations > r - 1 instead, to show that a claim does not hang on the round convention.
    Attempts at rounds 4 <= r < max_it with r % 4 == 2; go when 100 live <= pct * live_groups * G and ceil(live / G) < live_groups.
    A repack keeps the live frames' (group, column) order and packs them from column 0.
    Returns [(wave, round, live, groups_before, groups_after)]."""
    it = np.asarray(iterations).astype(np.int64)
    per_wave = groups_per_wave * G
    out = []
    for w, f0 in enumerate(range(0, len(it), per_wave)):
        wit = it[f0:f0 + per_wave]
        ng = (len(wit) + G - 1) // G
        if ng > 256 or ng < 2:
            continue
        pos = np.arange(len(wit))  # column id of each frame in this wave
        for r in range(4, max_it):
            if r % 4 != 2:
                continue
            live = wit > r - lag
            n_live = int(live.sum())
            live_groups = len(np.unique(pos[live] // G))
            if n_live and 100 * n_live <= pct * live_groups * G and (n_live + G - 1) // G < live_groups:
                out.append((w, r, n_live, live_groups, (n_live + G - 1) // G))
                pos = np.where(live, np.cumsum(live) - 1, -1)
    return out


def both_schedules(it, G, per_wave):
    """the schedule under the kernel's round convention and under r - 1"""
    return repack_schedule(it, G, per_wave, MAX_IT), repack_schedule(it, G, per_wave, MAX_IT, lag=1)


def parse_decoder(s):
    """{'vec', 'bw', 'bundle', 'waves', 'repack'} of a streaming decoder string (ctx.last_decoder)"""
    d = dict(re.findall(r"(\w+)=(\w+)", s))
    return {k: (int(d[k]) if d[k].isdigit() else d[k]) for k in ("vec", "bw", "bundle", "waves", "repack") if k in d}


def assert_shape(ctx, prefix, case, **want):
    s = assert_decoder(ctx, prefix, case)
    got = parse_decoder(s)
    for k, v in want.items():
        msg = (case, s) if k != "waves" or v != 1 else (case, s, "waves > 1: the device was short of free memory")
        assert got.get(k) == v, msg
    return s


def assert_same(case, bt, G, got, want, frames=None):
    """iterations, flags, decoded words and syndrome words of `got` equal `want` on every frame, compared as packed uint32"""
    frames = np.arange(len(got[0])) if frames is None else np.asarray(frames)
    bad = got[0] != want[0]
    bad |= got[1] != want[1]
    for x, y in zip(got[2:], want[2:]):
        if x is not None and y is not None:
            bad |= (x != y).any(axis=1)
    if bad.any():
        k = np.flatnonzero(bad)[:8]
        rows = [dict(frame=int(frames[i]), qber=float(bt.qclass[frames[i]]), group=int(frames[i]) // G, it=int(got[0][i]),
                     want_it=int(want[0][i]), res=int(got[1][i]), want_res=int(want[1][i])) for i in k]
        raise AssertionError(f"{case}: {int(bad.sum())} of {len(bad)} frames differ; first: {rows}")


def report(case, ctx, sched):
    print(f"\n{case}: {ctx.last_decoder}; context holds {held_gb(ctx):.2f} GB")
    for w, r, live, before, after in sched:
        print(f"  wave {w} round {r}: live {live}, groups {before} -> {after}")


def sample_frames(rng, pick):
    """pick = [(mask, count)]: `count` frames drawn from each mask in turn, none drawn twice; sorted"""
    taken = np.zeros(len(pick[0][0]), bool)
    for mask, cnt in pick:
        idx = np.flatnonzero(mask & ~taken)
        taken[rng.choice(idx, min(cnt, idx.size), replace=False)] = True
    return np.flatnonzero(taken)


def decode_slices(ctx, code, p, bt, idx, prefix, size=32):
    """idx decoded in slices of `size` frames: (it, res, dec, syn) of those frames; every slice takes the 32-frame form of `prefix`"""
    parts = []
    for lo in range(0, len(idx), size):
        sl = idx[lo:lo + size]
        parts.append(ctx.reconcile_packed(code, p, bt.a[sl], bt.b[sl], bt.q[sl], want_decoded=True, want_syndrome=True))
        assert_shape(ctx, prefix, ("slice", lo), vec=1, bundle=1, repack=0)
    return tuple(np.concatenate([x[k] for x in parts]) for k in range(4))


# ---- A. N = 10 240, the tier-3 hook, every frame against the resident kernel of the rule --------------------------------------
# rule -> (precision, make_params keywords, stream decoder prefix, resident decoder prefix)
RULES = {
    "fp32": (32, {}, "stream_f32 vec=4 bw=3", "resident_f32 "),
    "fp32fast": (32, {"fast_math": True}, "stream_f32 vec=4 bw=3", "resident_f32fast "),
    "minsum": (32, {"min_sum_scale": 0.75}, "stream_f32 vec=4 bw=3", "resident_f32minsum "),
    "fp64": (64, {}, "stream_f64 vec=2 bw=3", "resident_f64 "),
    "fp64fused": (64, {"fast_math": True}, "stream_f64 vec=2 bw=3", "resident_f64fused "),
}
# case -> (frames at G = 128, frames at G = 64, stream_max_bundles)
CASES = {
    "second_chunk": (9216, 9216, 0),
    "full_wave": (32768, 16384, 0),
    "over_limit": (40000, 20000, 0),
    "waves": (40000, 20000, 64),
}
# ~45 % converge within 5 rounds, the rest converge late or fail: ~55 % of the columns are live at round 6
MIX10K = ((0.03, 0.45), (0.075, 0.1375), (0.08, 0.1375), (0.085, 0.1375), (0.09, 0.1375))
_batches = {}
_refs = {}


def batch10k(ctx, oracle, frames):
    if frames not in _batches:
        mat = code_of("north_star")[0]
        counts = [int(round(f * frames)) for _, f in MIX10K]
        counts[0] += frames - sum(counts)
        _batches[frames] = mixed_batch(ctx, oracle, mat.n, [(q, c) for (q, _), c in zip(MIX10K, counts)], 10240 + frames)
    return _batches[frames]


def params(rule, **kw):
    precision, extra = RULES[rule][0], dict(RULES[rule][1])
    extra.update(kw)
    return capi.make_params(precision, MAX_IT, 100.0, True, **extra)


@pytest.mark.parametrize("case", list(CASES))
@pytest.mark.parametrize("rule", list(RULES))
def test_stream_at_scale_equals_resident(sctx, oracle, rule, case):
    mat, _, code = code_of("north_star")
    fp32 = RULES[rule][0] == 32
    G = 128 if fp32 else 64
    frames, max_bundles = CASES[case][0 if fp32 else 1], CASES[case][2]
    bt = batch10k(sctx, oracle, frames)
    if (rule, frames) not in _refs:
        _refs.clear()  # one reference at a time on the host (the cases of one batch run one after another)
        _refs[rule, frames] = sctx.reconcile_packed(code, params(rule), bt.a, bt.b, bt.q, want_decoded=True, want_syndrome=True)
        assert_decoder(sctx, RULES[rule][3], (rule, "resident"))
    want = _refs[rule, frames]
    got = sctx.reconcile_packed(code, params(rule, tier=3, stream_max_bundles=max_bundles), bt.a, bt.b, bt.q, want_decoded=True,
                                want_syndrome=True)
    groups = (frames + G - 1) // G
    bundles = (groups + 3) // 4
    if case == "waves":
        waves = (bundles + max_bundles - 1) // max_bundles
        per_wave = (bundles + waves - 1) // waves * 4
        assert waves == 2 and groups - per_wave < per_wave and frames % G, (groups, per_wave)  # a smaller last wave, a partial group
        shape = dict(waves=2, repack=1)
    else:
        per_wave = groups
        shape = dict(waves=1, repack=int(groups <= 256))
    s = assert_shape(sctx, RULES[rule][2], (rule, case), bundle=4, **shape)
    sched, sched_lag = both_schedules(got[0], G, per_wave)
    report(f"{rule} {case} ({frames} frames, {groups} groups)", sctx, sched)
    assert_same((rule, case, s), bt, G, got, want)
    assert 0 < int((got[1] & 1).sum()) < frames  # the batch mixes converging and failing frames
    if case == "over_limit":
        assert groups > 256 and groups > 2 * sctx.sm_count, (groups, sctx.sm_count)
    for sc in (sched, sched_lag):
        first = {}
        for w, r, live, before, after in sc:
            first.setdefault(w, (r, live, before))
        if case == "waves":
            assert sorted(first) == [0, 1] and all(v[1] > STAGE for v in first.values()), sc
        elif case != "over_limit":
            assert 0 in first and first[0][1] > STAGE and first[0][2] == groups, sc  # the first repack: every group, 2 chunks
    if case == "second_chunk":
        # 256 frames decoded in slices of 32 (one group each, no repack): failed ones, ones that converged after round 6, others
        it, res = got[0], got[1]
        idx = sample_frames(np.random.default_rng(frames), [((res & 1) == 0, 64), (((res & 1) == 1) & (it > 6), 64), (it > 0, 128)])
        assert idx.size == 256 and ((res[idx] & 1) == 0).sum() >= 64 and (((res[idx] & 1) == 1) & (it[idx] > 6)).sum() >= 64
        sl = decode_slices(sctx, code, params(rule, tier=3), bt, idx, f"stream_f{RULES[rule][0]}")
        assert_same((rule, "slices"), bt, G, sl, tuple(x[idx] for x in got), frames=idx)


# ---- B. N = 100 000, the default routes at the benchmark's shape ----------------------------------------------------------------
MIX100K = ((0.03, 3440), (0.075, 1188), (0.08, 1188), (0.085, 1188), (0.09, 1188))  # 8 192 frames, ~58 % live at round 6


def big():
    if "big" not in _batches:
        mat = codes.peg_code(100000, 51080, 3, 666, bfs_limit=2000)
        _batches["big"] = (mat, graph_of(mat), capi.Code.from_graph(mat))
    return _batches["big"]


def batch100k(ctx, oracle):
    if "b100k" not in _batches:
        _batches["b100k"] = mixed_batch(ctx, oracle, 100000, MIX100K, 100000)
    return _batches["b100k"]


def assert_big_repack(got, G):
    groups = (len(got[0]) + G - 1) // G
    sched, sched_lag = both_schedules(got[0], G, groups)
    for sc in (sched, sched_lag):
        assert any(live > STAGE for _, _, live, _, _ in sc), sc
    return sched


def reference_outcomes(run_trials, oracle, g, bt, idx):
    """(iterations, result bytes, packed decoded words, packed syndrome words) of frames idx from a CPU reference's run_trials,
    called per class with the frames' seeds"""
    out3, dec = np.zeros((idx.size, 3), np.uint64), np.zeros((idx.size, bt.n), np.int32)
    for q in np.unique(bt.qclass[idx]):
        sel = np.flatnonzero(bt.qclass[idx] == q)
        out3[sel], dec[sel] = run_trials(g, float(q), bt.seed[idx[sel]], threads=THREADS, max_it=MAX_IT, want_decoded=True)
    syn = capi.pack_bits(np.stack([oracle.syndrome(g, x) for x in capi.unpack_bits(bt.a[idx], bt.n)]), g.m)
    return out3[:, 0].astype(np.uint32), (out3[:, 1] | (out3[:, 2] << 1)).astype(np.uint8), capi.pack_bits(dec, bt.n), syn


@pytest.mark.parametrize("fused", [False, True])
def test_n100k_fp64_default_route(sctx, oracle, fused):
    mat, g, code = big()
    bt = batch100k(sctx, oracle)
    p = capi.make_params(64, MAX_IT, 100.0, True, fast_math=fused)
    got = sctx.reconcile_packed(code, p, bt.a, bt.b, bt.q, want_decoded=True, want_syndrome=True)
    s = assert_shape(sctx, "stream_f64 vec=2 bw=3", fused, bundle=4, waves=1, repack=1)
    report(f"N=100000 fp64 fused={fused}", sctx, assert_big_repack(got, 64))
    ref = sctx.reconcile_packed(code, capi.make_params(64, MAX_IT, 100.0, True, fast_math=fused, tier=2), bt.a, bt.b, bt.q,
                                want_decoded=True, want_syndrome=True)
    assert_decoder(sctx, "generic f64" + ("fused" if fused else "") + " tier=2 shape=0", fused)
    assert_same((fused, s), bt, 64, got, ref)
    if fused:
        return  # the fused rule is not the reference's; the generic kernel above is its exact reference
    # the oracle on a stratified sample: failed frames, frames that converged after the first repack, first / middle / last bundle
    it, res = got[0], got[1]
    first_round = repack_schedule(it, 64, 128, MAX_IT)[0][1]
    f = np.arange(len(it))
    bundle = f // 256
    idx = sample_frames(np.random.default_rng(5), [((res & 1) == 0, 10), (((res & 1) == 1) & (it > first_round), 10),
                                                   (bundle == 0, 10), (bundle == 16, 10), (bundle == 31, 10)])
    assert idx.size == 50 and ((res[idx] & 1) == 0).sum() >= 10 and (((res[idx] & 1) == 1) & (it[idx] > first_round)).sum() >= 10
    want = reference_outcomes(oracle.run_trials, oracle, g, bt, idx)
    assert_same(("oracle", s), bt, 64, tuple(x[idx] for x in got), want, frames=idx)


@pytest.mark.parametrize("fast", [False, True])
def test_n100k_fp32_default_route(sctx, oracle, fast):
    mat, g, code = big()
    bt = batch100k(sctx, oracle)
    p = lambda **kw: capi.make_params(32, MAX_IT, 100.0, True, fast_math=fast, **kw)
    got = sctx.reconcile_packed(code, p(), bt.a, bt.b, bt.q, want_decoded=True, want_syndrome=True)
    s = assert_shape(sctx, "stream_f32 vec=4 bw=3", fast, bundle=4, waves=1, repack=1)
    report(f"N=100000 fp32 fast={fast}", sctx, assert_big_repack(got, 128))
    nr = sctx.reconcile_packed(code, p(stream_no_repack=True), bt.a, bt.b, bt.q, want_decoded=True, want_syndrome=True)
    assert_shape(sctx, "stream_f32 vec=4 bw=3", (fast, "no repack"), bundle=4, repack=0)
    assert_same((fast, "no repack"), bt, 128, got, nr)
    wv = sctx.reconcile_packed(code, p(stream_max_bundles=4), bt.a, bt.b, bt.q, want_decoded=True, want_syndrome=True)
    assert_shape(sctx, "stream_f32 vec=4 bw=3", (fast, "waves"), bundle=4, waves=4, repack=1)
    assert_same((fast, "waves"), bt, 128, got, wv)
    it, res = got[0], got[1]
    idx = sample_frames(np.random.default_rng(7), [((res & 1) == 0, 64), (it > 6, 64), (it > 0, 128)])
    assert idx.size == 256
    sl = decode_slices(sctx, code, p(), bt, idx, "stream_f32")
    assert_same((fast, "slices"), bt, 128, sl, tuple(x[idx] for x in got), frames=idx)
    # no exact fp32 reference at this length: flags against the oracle, keys where both converged
    ix = idx[::5]
    w_it, w_res, w_dec, w_syn = reference_outcomes(oracle.run_trials, oracle, g, bt, ix)
    assert (got[3][ix] == w_syn).all()
    same = (res[ix] & 3) == w_res
    assert same.mean() >= 0.9, (fast, same.mean())
    ok = same & ((w_res & 1) == 1)
    assert (got[2][ix][ok] == w_dec[ok]).all()


def test_n100k_min_sum_equals_restatement(sctx, oracle, msr):
    mat, g, code = big()
    bt = batch100k(sctx, oracle)
    p = lambda **kw: capi.make_params(32, MAX_IT, 100.0, True, min_sum_scale=0.75, **kw)
    got = sctx.reconcile_packed(code, p(), bt.a, bt.b, bt.q, want_decoded=True, want_syndrome=True)
    s = assert_shape(sctx, "stream_f32 vec=4 bw=3", "min-sum", bundle=4, waves=1, repack=1)
    report("N=100000 min-sum 0.75", sctx, assert_big_repack(got, 128))
    nr = sctx.reconcile_packed(code, p(stream_no_repack=True), bt.a, bt.b, bt.q, want_decoded=True, want_syndrome=True)
    assert_shape(sctx, "stream_f32 vec=4 bw=3", "min-sum no repack", bundle=4, repack=0)
    assert_same(("min-sum", "no repack"), bt, 128, got, nr)
    it, res = got[0], got[1]
    idx = sample_frames(np.random.default_rng(9), [((res & 1) == 0, 32), (((res & 1) == 1) & (it > 10), 32), (it > 0, 64)])
    assert idx.size == 128 and ((res[idx] & 1) == 0).sum() >= 32 and (((res[idx] & 1) == 1) & (it[idx] > 10)).sum() >= 32
    want = reference_outcomes(lambda g_, q, seeds, **kw: msr.run_trials(g_, q, seeds, 0.75, **kw), oracle, g, bt, idx)
    assert_same(("min-sum restatement", s), bt, 128, tuple(x[idx] for x in got), want, frames=idx)
