"""BASELINE.json configs[3] and configs[4] as parity cases: seeded PEG codes of other rates (R = 0.3 ... 0.8 at N = 10240,
check weights 4 ... 16) and of larger block length (N = 100 000, messages in global scratch), against the oracle."""
import numpy as np
import pytest

from qkd_ldpc_b200 import capi, codes

pytestmark = pytest.mark.gpu


def graph_of(mat):
    from oracle.bindings import Graph
    return Graph(mat.n, mat.m, mat.row_ptr, mat.col_idx, mat.col_ptr, mat.row_idx)


def frames_for(oracle, n, q, seeds):
    ab = [oracle.generate(int(s), n, q) for s in seeds]
    return np.stack([x[0] for x in ab]), np.stack([x[1] for x in ab]), np.array([x[2] for x in ab])


@pytest.mark.parametrize("m,qs", [(7168, (0.10, 0.13, 0.17)), (5231, (0.06, 0.085)), (3072, (0.03, 0.045, 0.06)), (2048, (0.012, 0.02, 0.03))])
def test_multi_rate_codes_match_oracle(ctx, oracle, m, qs):
    n = 10240
    mat = codes.peg_code(n, m, 3, 666)
    g, code = graph_of(mat), capi.Code.from_graph(mat)
    seeds = oracle.trial_seeds(4242, 12)
    seen = set()
    for pt, q in enumerate(qs):
        s = seeds + np.uint64(pt)
        want, wdec = oracle.run_trials(g, q, s, threads=8, want_decoded=True)
        A, B, Q = frames_for(oracle, n, q, s)
        it, res, dec, _ = ctx.reconcile_packed(code, capi.make_params(64, 100, 100.0, True), capi.pack_bits(A), capi.pack_bits(B), Q)
        assert (it == want[:, 0]).all(), (m, q, it, want[:, 0])
        assert ((res & 1) == want[:, 1]).all() and (((res >> 1) & 1) == want[:, 2]).all()
        assert (capi.unpack_bits(dec, n) == wdec).all()
        seen.update(want[:, 1].tolist())
        for fast in (False, True):
            it32, res32, dec32, _ = ctx.reconcile_packed(code, capi.make_params(32, 100, 100.0, True, fast_math=fast), capi.pack_bits(A), capi.pack_bits(B), Q)
            same = ((res32 & 1) == want[:, 1]) & (((res32 >> 1) & 1) == want[:, 2])
            assert same.mean() >= 0.9, (m, q, fast, same)
            ok = (want[:, 1] == 1) & same
            assert (capi.unpack_bits(dec32, n)[ok] == wdec[ok]).all()
    assert seen == {0, 1}, "the QBER points must straddle the code's threshold"


def test_large_block_length_matches_oracle(ctx, oracle):
    """N = 100 000 (E = 300 000, 300 000 message slots): both precisions go to the streaming decoder, which takes every fp64 code
    with 65 535 or more slots; three frames take its 32-frame-group form (vec=1, one bundle of one group, no repack)."""
    n, m = 100000, 51080
    mat = codes.peg_code(n, m, 3, 666, bfs_limit=2000)
    g, code = graph_of(mat), capi.Code.from_graph(mat)
    seeds = oracle.trial_seeds(99, 3)
    for q, mi in ((0.05, 100), (0.10, 12)):
        want, wdec = oracle.run_trials(g, q, seeds, threads=3, max_it=mi, want_decoded=True)
        A, B, Q = frames_for(oracle, n, q, seeds)
        for precision in (64, 32):
            it, res, dec, syn = ctx.reconcile_packed(code, capi.make_params(precision, mi, 100.0, True), capi.pack_bits(A), capi.pack_bits(B), Q,
                                                     want_syndrome=True)
            assert ctx.last_decoder.startswith(f"stream_f{precision} vec=1 bw=3 bundle=1 waves=1"), ctx.last_decoder
            want_syn = np.stack([oracle.syndrome(g, a) for a in A])
            assert (capi.unpack_bits(syn, m) == want_syn).all()
            assert ((res & 1) == want[:, 1]).all() and (((res >> 1) & 1) == want[:, 2]).all()
            if precision == 64:
                assert (it == want[:, 0]).all()
                assert (capi.unpack_bits(dec, n) == wdec).all()


@pytest.mark.parametrize("norepack", [False, True])
def test_streaming_kernel_equals_resident_kernel(ctx, oracle, norepack):
    """The frame-interleaved HBM-streaming decoder (forced with the tier-3 test hook) runs the same node arithmetic as the
    SM-resident kernel: iterations, flags and decoded keys must be identical, for a ragged batch (300 frames = 2 groups + 44)
    mixing QBER points, in both fp32 rules -- with and without the on-device compaction of the live frames
    (qlb_decode_params.stream_no_repack; the mixed-QBER batch below triggers several repacks)."""
    mat = codes.load_npz(codes.NORTH_STAR)
    code = capi.Code.from_graph(mat)
    seeds = oracle.trial_seeds(31337, 300)
    qs = [0.03, 0.07, 0.085, 0.09]
    A, B, Q = [], [], []
    for k, s in enumerate(seeds):
        a, b, ex = oracle.generate(int(s), mat.n, qs[k % 4])
        A.append(a); B.append(b); Q.append(ex)
    A, B, Q = capi.pack_bits(np.stack(A)), capi.pack_bits(np.stack(B)), np.array(Q)
    for fast in (True, False):
        r = ctx.reconcile_packed(code, capi.make_params(32, 60, 100.0, True, fast_math=fast), A, B, Q, want_syndrome=True)
        s = ctx.reconcile_packed(code, capi.make_params(32, 60, 100.0, True, fast_math=fast, tier=3, stream_no_repack=norepack), A, B, Q, want_syndrome=True)
        assert (r[0] == s[0]).all(), np.flatnonzero(r[0] != s[0])
        assert (r[1] == s[1]).all() and (r[2] == s[2]).all() and (r[3] == s[3]).all()
    # and the sum-product entry (arbitrary LLRs + target syndromes) through the streaming kernel
    g = graph_of(mat)
    bob = capi.unpack_bits(B[:5], mat.n); alice = capi.unpack_bits(A[:5], mat.n)
    llr = np.where(bob != 0, -1.0, 1.0) * np.log((1 - Q[:5]) / Q[:5])[:, None]
    syn = np.stack([oracle.syndrome(g, a) for a in alice])
    it_r, res_r, bits_r = ctx.sum_product(code, capi.make_params(32, 60, 100.0, True, fast_math=True), llr, syn)
    it_s, res_s, bits_s = ctx.sum_product(code, capi.make_params(32, 60, 100.0, True, fast_math=True, tier=3), llr, syn)
    assert (it_r == it_s).all() and (res_r == res_s).all() and (bits_r == bits_s).all()
    # a batch of <= 32 frames takes the 32-frame-group instantiation
    r = ctx.reconcile_packed(code, capi.make_params(32, 60, 100.0, True, fast_math=True), A[:21], B[:21], Q[:21], want_syndrome=True)
    s = ctx.reconcile_packed(code, capi.make_params(32, 60, 100.0, True, fast_math=True, tier=3), A[:21], B[:21], Q[:21], want_syndrome=True)
    assert all((x == y).all() for x, y in zip(r, s))


def assert_several_repacks(iterations, G, max_it):
    """the streaming decoder repacked at least twice: restated from the iteration counts, under the kernel's round convention
    and under r - 1 (test_gpu_stream_scale.repack_schedule)"""
    from test_gpu_stream_scale import repack_schedule
    groups = (len(iterations) + G - 1) // G
    for lag in (0, 1):
        sched = repack_schedule(iterations, G, groups, max_it, lag=lag)
        assert len(sched) >= 2, sched


def test_streaming_compaction_many_groups(ctx, oracle):
    """1 100 frames of the N=10240 code (9 groups = 3 bundles of 4, the last one partial and ragged) drawn by the on-device
    reference generator at QBERs that converge at very different rounds: the streaming decoder repacks the live frames
    several times on the way (and retires whole bundles); iterations, flags, decoded keys and syndromes must stay
    bit-identical to the SM-resident kernel, which decodes every frame on its own."""
    mat = codes.load_npz(codes.NORTH_STAR)
    code = capi.Code.from_graph(mat)
    A, B, Q = [], [], []
    for pt, (q, cnt) in enumerate(((0.03, 300), (0.06, 250), (0.08, 250), (0.085, 200), (0.0875, 60), (0.09, 40))):
        seeds = oracle.trial_seeds(4242 + pt, cnt)
        a, b, ex = ctx.generate(mat.n, seeds, q)
        A.append(a); B.append(b); Q.append(np.full(cnt, ex))
    A, B, Q = np.concatenate(A), np.concatenate(B), np.concatenate(Q)
    perm = np.random.default_rng(7).permutation(len(Q))  # every group holds frames of every kind
    A, B, Q = np.ascontiguousarray(A[perm]), np.ascontiguousarray(B[perm]), Q[perm]
    p_res = capi.make_params(32, 100, 100.0, True, fast_math=True)
    p_str = capi.make_params(32, 100, 100.0, True, fast_math=True, tier=3)
    r = ctx.reconcile_packed(code, p_res, A, B, Q, want_syndrome=True)
    s = ctx.reconcile_packed(code, p_str, A, B, Q, want_syndrome=True)
    assert (r[0] == s[0]).all(), np.flatnonzero(r[0] != s[0])[:10]
    assert (r[1] == s[1]).all() and (r[2] == s[2]).all() and (r[3] == s[3]).all()
    assert 0 < int((r[1] & 1).sum()) < len(Q)  # the batch really mixes converging and failing frames
    assert ctx.last_decoder.startswith("stream_f32 vec=4 bw=3 bundle=4 waves=1 repack=1"), ctx.last_decoder
    assert_several_repacks(s[0], 128, 100)
    # sum-product entry (LLRs + target syndromes, no keys) through the same repacks; the priors are products here, which every
    # fp32 kernel rounds on their own (__fmul_rn) -- a contraction into the first sum would make the chaotic, non-converging
    # frames end on different last decisions in different kernels
    g = graph_of(mat)
    k = 200
    bob = capi.unpack_bits(B[:k], mat.n)
    llr = np.where(bob != 0, -1.0, 1.0) * np.log((1 - Q[:k]) / Q[:k])[:, None]
    syn = capi.unpack_bits(r[3][:k], mat.m)
    it_r, res_r, bits_r = ctx.sum_product(code, p_res, llr, syn)
    it_s, res_s, bits_s = ctx.sum_product(code, p_str, llr, syn)
    assert (it_r == it_s).all() and (res_r == res_s).all() and (bits_r == bits_s).all()


def test_streaming_decoder_in_waves(ctx, oracle):
    """When device memory cannot hold every frame group the batch is decoded in waves (here forced: at most 2 bundles = 8 groups
    per wave for 2 500 frames = 20 groups -> 3 waves): per-wave state is re-used, frames are addressed through the wave's
    frame map. Must equal the resident kernel frame by frame."""
    mat = codes.load_npz(codes.NORTH_STAR)
    code = capi.Code.from_graph(mat)
    A, B, Q = [], [], []
    for pt, (q, cnt) in enumerate(((0.04, 900), (0.075, 800), (0.085, 500), (0.095, 300))):
        a, b, ex = ctx.generate(mat.n, oracle.trial_seeds(900 + pt, cnt), q)
        A.append(a); B.append(b); Q.append(np.full(cnt, ex))
    A, B, Q = np.concatenate(A), np.concatenate(B), np.concatenate(Q)
    perm = np.random.default_rng(11).permutation(len(Q))
    A, B, Q = np.ascontiguousarray(A[perm]), np.ascontiguousarray(B[perm]), Q[perm]
    r = ctx.reconcile_packed(code, capi.make_params(32, 50, 100.0, True, fast_math=True), A, B, Q, want_syndrome=True)
    s = ctx.reconcile_packed(code, capi.make_params(32, 50, 100.0, True, fast_math=True, tier=3, stream_max_bundles=2), A, B, Q, want_syndrome=True)
    assert all((x == y).all() for x, y in zip(r, s))


def test_streaming_kernel_large_block_length(ctx, oracle):
    """N = 100 000 in fp32 goes through the streaming kernel by default; flags must equal the fp64 oracle's."""
    n, m = 100000, 51080
    mat = codes.peg_code(n, m, 3, 666, bfs_limit=2000)
    g, code = graph_of(mat), capi.Code.from_graph(mat)
    seeds = oracle.trial_seeds(99, 3)
    for q, mi in ((0.05, 100), (0.10, 12)):
        want, wdec = oracle.run_trials(g, q, seeds, threads=3, max_it=mi, want_decoded=True)
        A, B, Q = frames_for(oracle, n, q, seeds)
        for fast in (True, False):
            it, res, dec, syn = ctx.reconcile_packed(code, capi.make_params(32, mi, 100.0, True, fast_math=fast), capi.pack_bits(A), capi.pack_bits(B), Q,
                                                     want_syndrome=True)
            assert (capi.unpack_bits(syn, m) == np.stack([oracle.syndrome(g, a) for a in A])).all()
            assert ((res & 1) == want[:, 1]).all() and (((res >> 1) & 1) == want[:, 2]).all()
            ok = want[:, 1] == 1
            assert (capi.unpack_bits(dec, n)[ok] == wdec[ok]).all()
            assert (np.abs(it.astype(int) - want[:, 0].astype(int)) <= 1).all()


def test_block_length_one_million(ctx, oracle):
    """BASELINE.json configs[3] at N = 1 000 000 (E = 3 000 000; seeded permutation code, codes.permutation_code): three frames --
    two that converge (QBER 0.05, 8 rounds) and one that runs into max_it = 12 (QBER 0.10) -- against the fp64 oracle. fp64: the
    large-frame fp64 decoder, iterations / flags / every decoded bit equal; fp32 (both rules): the streaming decoder, flags equal,
    decoded key equal on the converged frames, iteration counts within one round. The device key generator runs at this length too."""
    n, m = 1_000_000, 510_800
    mat = codes.permutation_code(n, m, 3, 666)
    g, code = graph_of(mat), capi.Code.from_graph(mat)
    seeds = oracle.trial_seeds(99, 2)
    for q, mi, sd in ((0.05, 12, seeds), (0.10, 12, seeds[:1])):
        want, wdec = oracle.run_trials(g, q, sd, threads=2, max_it=mi, want_decoded=True)
        A, B, Q = frames_for(oracle, n, q, sd)
        ga, gb, gq = ctx.generate(n, sd, q)
        assert gq == Q[0] and (capi.unpack_bits(ga, n) == A).all() and (capi.unpack_bits(gb, n) == B).all()
        want_syn = np.stack([oracle.syndrome(g, a) for a in A])
        for precision, fast in ((64, False), (64, True), (32, False), (32, True)):
            it, res, dec, syn = ctx.reconcile_packed(code, capi.make_params(precision, mi, 100.0, True, fast_math=fast), ga, gb, Q, want_syndrome=True)
            assert (capi.unpack_bits(syn, m) == want_syn).all()
            assert ((res & 1) == want[:, 1]).all() and (((res >> 1) & 1) == want[:, 2]).all(), (q, precision, fast)
            if precision == 64:
                assert (it == want[:, 0]).all(), (q, fast, it, want[:, 0])
                assert (capi.unpack_bits(dec, n) == wdec).all()
            else:
                ok = want[:, 1] == 1
                assert (capi.unpack_bits(dec, n)[ok] == wdec[ok]).all()
                assert (np.abs(it.astype(int) - want[:, 0].astype(int)) <= 1).all()


@pytest.mark.parametrize("fused", [False, True])
def test_streaming_fp64_equals_resident_kernel(ctx, oracle, fused):
    """The fp64 streaming decoder (64-frame groups, the reference's check rule, parity from the packed decisions) forced with the
    tier-3 hook on the N=10240 code: iterations, flags, every decoded bit (failed frames included) and syndromes must equal the
    fp64 SM-resident kernel's -- which equals the reference on the campaign -- for 700 mixed-QBER frames (11 groups = 3 bundles,
    the last ragged; several repacks), without repacks, in waves, for a <= 32-frame batch, with the clamp off (NaN semantics)
    and through the sum-product entry."""
    mat = codes.load_npz(codes.NORTH_STAR)
    code = capi.Code.from_graph(mat)
    A, B, Q = [], [], []
    for pt, (q, cnt) in enumerate(((0.03, 200), (0.06, 150), (0.08, 150), (0.085, 120), (0.0875, 50), (0.09, 30))):
        a, b, ex = ctx.generate(mat.n, oracle.trial_seeds(5150 + pt, cnt), q)
        A.append(a); B.append(b); Q.append(np.full(cnt, ex))
    A, B, Q = np.concatenate(A), np.concatenate(B), np.concatenate(Q)
    perm = np.random.default_rng(3).permutation(len(Q))
    A, B, Q = np.ascontiguousarray(A[perm]), np.ascontiguousarray(B[perm]), Q[perm]
    r = ctx.reconcile_packed(code, capi.make_params(64, 100, 100.0, True, fast_math=fused), A, B, Q, want_decoded=True, want_syndrome=True)
    assert 0 < int((r[1] & 1).sum()) < len(Q)
    for kw in ({}, {"stream_no_repack": True}, {"stream_max_bundles": 1}):
        s = ctx.reconcile_packed(code, capi.make_params(64, 100, 100.0, True, fast_math=fused, tier=3, **kw), A, B, Q, want_decoded=True, want_syndrome=True)
        assert (r[0] == s[0]).all(), (kw, np.flatnonzero(r[0] != s[0])[:10])
        assert all((x == y).all() for x, y in zip(r[1:], s[1:])), kw
        if not kw:
            assert ctx.last_decoder.startswith("stream_f64 vec=2 bw=3 bundle=4 waves=1 repack=1"), ctx.last_decoder
            assert_several_repacks(s[0], 64, 100)
    # <= 32 frames: the 32-frame-group instantiation; and the clamp off (saturated products -> inf -> NaN totals, :508-524)
    for thr_on in (True, False):
        r21 = ctx.reconcile_packed(code, capi.make_params(64, 40, 100.0, thr_on, fast_math=fused), A[:21], B[:21], Q[:21], want_decoded=True, want_syndrome=True)
        s21 = ctx.reconcile_packed(code, capi.make_params(64, 40, 100.0, thr_on, fast_math=fused, tier=3), A[:21], B[:21], Q[:21], want_decoded=True, want_syndrome=True)
        assert all((x == y).all() for x, y in zip(r21, s21)), thr_on
    r100 = ctx.reconcile_packed(code, capi.make_params(64, 40, 100.0, False, fast_math=fused), A[:100], B[:100], Q[:100], want_decoded=True)
    s100 = ctx.reconcile_packed(code, capi.make_params(64, 40, 100.0, False, fast_math=fused, tier=3), A[:100], B[:100], Q[:100], want_decoded=True)
    assert all((x == y).all() for x, y in zip(r100[:3], s100[:3]))
    # the sum-product entry: arbitrary LLRs + target syndromes
    k = 90
    bob = capi.unpack_bits(B[:k], mat.n)
    rng = np.random.default_rng(17)
    llr = np.where(bob != 0, -1.0, 1.0) * np.log((1 - Q[:k]) / Q[:k])[:, None] * rng.uniform(0.6, 1.4, size=bob.shape)
    syn = capi.unpack_bits(r[3][:k], mat.m)
    it_r, res_r, bits_r = ctx.sum_product(code, capi.make_params(64, 60, 100.0, True, fast_math=fused), llr, syn)
    it_s, res_s, bits_s = ctx.sum_product(code, capi.make_params(64, 60, 100.0, True, fast_math=fused, tier=3), llr, syn)
    assert (it_r == it_s).all() and (res_r == res_s).all() and (bits_r == bits_s).all()


@pytest.mark.parametrize("dv", [2, 4])
def test_streaming_other_bit_weights(ctx, oracle, dv):
    """Column weights 2 and 4 through the streaming decoder (template instantiations of the bit pass) on a permutation code of
    N = 4 096: fp64 must equal the oracle on iterations, flags and decoded bits; fp32 must equal the generic fp32 kernel's flags."""
    n, m = 4096, 2048
    mat = codes.permutation_code(n, m, dv, 4321)
    g, code = graph_of(mat), capi.Code.from_graph(mat)
    for q in ((0.01, 0.02) if dv == 2 else (0.04, 0.09)):
        seeds = oracle.trial_seeds(2024 + dv, 150)
        want, wdec = oracle.run_trials(g, q, seeds, threads=8, max_it=30, want_decoded=True)
        a, b, ex = ctx.generate(n, seeds, q)
        Q = np.full(len(seeds), ex)
        for fused in (False, True):
            it, res, dec, syn = ctx.reconcile_packed(code, capi.make_params(64, 30, 100.0, True, fast_math=fused, tier=3), a, b, Q, want_decoded=True,
                                                     want_syndrome=True)
            assert ((res & 1) == want[:, 1]).all() and (((res >> 1) & 1) == want[:, 2]).all(), (dv, q, fused)
            assert (it == want[:, 0]).all(), (dv, q, fused, np.flatnonzero(it != want[:, 0])[:8])
            assert (capi.unpack_bits(dec, n) == wdec).all()
        for fast in (False, True):
            gen = ctx.reconcile_packed(code, capi.make_params(32, 30, 100.0, True, fast_math=fast, tier=2), a, b, Q)
            st = ctx.reconcile_packed(code, capi.make_params(32, 30, 100.0, True, fast_math=fast, tier=3), a, b, Q)
            assert ((gen[1] & 3) == (st[1] & 3)).mean() >= 0.98, (dv, q, fast)
            assert (np.abs(gen[0].astype(int) - st[0].astype(int)) <= 1).mean() >= 0.95


def test_high_rate_code_check_weight_80(ctx, oracle):
    """config.json's code_rate 0.95 preset at column weight 4 means check weight 80 (ADVICE r1: the layout used to stop at 64). A
    permutation code N = 4 000, M = 200: fp64 must equal the oracle frame by frame (generic kernel, two-pass rule over 80 edges),
    fp32 must agree on the flags."""
    n, m = 4000, 200
    mat = codes.permutation_code(n, m, 4, 99)
    assert int(np.diff(mat.row_ptr).max()) == 80
    g, code = graph_of(mat), capi.Code.from_graph(mat)
    seeds = oracle.trial_seeds(5, 64)
    seen = set()
    for q in (0.002, 0.004):
        want, wdec = oracle.run_trials(g, q, seeds, threads=8, max_it=30, want_decoded=True)
        a, b, ex = ctx.generate(n, seeds, q)
        Q = np.full(len(seeds), ex)
        seen |= set(want[:, 1].tolist())
        for fused in (False, True):
            it, res, dec, syn = ctx.reconcile_packed(code, capi.make_params(64, 30, 100.0, True, fast_math=fused), a, b, Q, want_decoded=True, want_syndrome=True)
            assert (capi.unpack_bits(syn, m) == np.stack([oracle.syndrome(g, x) for x in capi.unpack_bits(a, n)])).all()
            assert ((res & 1) == want[:, 1]).all() and (((res >> 1) & 1) == want[:, 2]).all() and (it == want[:, 0]).all(), (q, fused)
            assert (capi.unpack_bits(dec, n) == wdec).all()
        it, res, _, _ = ctx.reconcile_packed(code, capi.make_params(32, 30, 100.0, True), a, b, Q)
        assert ((res & 3) == (want[:, 1] | (want[:, 2] << 1))).mean() >= 0.9
    assert seen == {0, 1}


def irregular_code(n, m, seed):
    """A seeded code with column weights 2 / 3 / 4 / 6 (40 / 35 / 15 / 10 %) and near-equal check weights: every bit draws its
    checks from a shuffled pool in which each check appears equally often; duplicates inside a bit are re-drawn."""
    rng = np.random.default_rng(seed)
    w = rng.choice([2, 3, 4, 6], size=n, p=[0.40, 0.35, 0.15, 0.10])
    e = int(w.sum())
    pool = np.resize(rng.permutation(m), e)
    rng.shuffle(pool)
    h = np.zeros((m, n), np.uint8)
    at = 0
    for i in range(n):
        picks = set()
        for c in pool[at:at + w[i]]:
            c = int(c)
            while c in picks:
                c = int(rng.integers(m))
            picks.add(c)
        at += w[i]
        h[sorted(picks), i] = 1
    assert (h.sum(1) >= 2).all()
    return codes.Matrix.from_dense(h, f"irregular_n{n}_m{m}_seed{seed}")


def test_streaming_irregular_bit_weights(ctx, oracle):
    """Irregular column weights (2 / 3 / 4 / 6) through the streaming decoder's any-weight bit pass (forced with the tier-3 hook;
    N = 2 048, check weights <= 16): fp64, both rules, must equal the oracle frame by frame -- iterations, flags, every decoded bit,
    syndromes -- on 200 frames that straddle the code's threshold, through repacks and in the <= 32-frame form; fp32 must agree
    with the generic fp32 kernel on the flags."""
    n, m = 2048, 1024
    mat = irregular_code(n, m, 12)
    assert mat.max_check_w <= 16 and len(set(np.diff(mat.col_ptr).tolist())) >= 3
    g, code = graph_of(mat), capi.Code.from_graph(mat)
    seeds = oracle.trial_seeds(77, 200)
    seen = set()
    for q in (0.02, 0.08, 0.10):
        want, wdec = oracle.run_trials(g, q, seeds, threads=8, max_it=40, want_decoded=True)
        seen |= set(want[:, 1].tolist())
        a, b, ex = ctx.generate(n, seeds, q)
        Q = np.full(len(seeds), ex)
        want_syn = np.stack([oracle.syndrome(g, x) for x in capi.unpack_bits(a, n)])
        for fused in (False, True):
            for cnt in (200, 20):
                it, res, dec, syn = ctx.reconcile_packed(code, capi.make_params(64, 40, 100.0, True, fast_math=fused, tier=3), a[:cnt], b[:cnt], Q[:cnt],
                                                         want_decoded=True, want_syndrome=True)
                assert (capi.unpack_bits(syn, m) == want_syn[:cnt]).all()
                assert ((res & 1) == want[:cnt, 1]).all() and (((res >> 1) & 1) == want[:cnt, 2]).all(), (q, fused, cnt)
                assert (it == want[:cnt, 0]).all(), (q, fused, cnt, np.flatnonzero(it != want[:cnt, 0])[:8])
                assert (capi.unpack_bits(dec, n) == wdec[:cnt]).all()
        for fast in (False, True):
            gen = ctx.reconcile_packed(code, capi.make_params(32, 40, 100.0, True, fast_math=fast, tier=2), a, b, Q)
            st = ctx.reconcile_packed(code, capi.make_params(32, 40, 100.0, True, fast_math=fast, tier=3), a, b, Q)
            assert ((gen[1] & 3) == (st[1] & 3)).mean() >= 0.97, (q, fast)
    assert seen == {0, 1}
