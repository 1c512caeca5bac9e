"""The trust chain of the parity tests, on the CPU: Restatement (oracle/restatement, plain C) == the reference's own outputs,
recorded from the unmodified reference sources into the committed golden fixtures (tests/golden/make_*.py)."""
import numpy as np
import pytest

from conftest import GOLD, NS


@pytest.fixture(scope="module")
def campaign():
    z = np.load(GOLD / "campaign_n10240.npz")
    return {k: z[k] for k in z.files}


def test_campaign_fixture_shape(campaign):
    """12 points x 4096 frames of the reference's own run_trial outcomes (tests/golden/make_campaign.py)."""
    per = int(campaign["frames_per_point"])
    assert campaign["iterations"].shape == (12, per) and campaign["flags"].shape == (12, per)
    assert np.allclose(campaign["qber"][:9], [0.03 + 0.01 * j for j in range(9)]) and campaign["seed_offset"][:9].tolist() == list(range(9))
    ok = campaign["flags"] & 1
    assert ok[:5].all() and not ok[7:9].any()           # 0.03 ... 0.07 always converge, 0.10 / 0.11 never
    assert 0 < ok[10].sum() < per                        # the waterfall points straddle
    assert ((campaign["flags"] >> 1) & 1 <= ok).all()    # keys can only match when the syndromes do
    assert (campaign["iterations"][ok == 0] == int(campaign["max_it"])).all()


def test_restatement_equals_fixture(oracle, graphs, campaign):
    """The plain-C restatement reproduces the reference's outcomes on the first frames of every campaign point."""
    g = graphs[NS]
    seeds = oracle.trial_seeds(int(campaign["simulation_seed"]), 12)
    for pt in range(12):
        k = 12 if campaign["qber"][pt] < 0.0825 else 4  # failing frames cost 100 iterations each
        out = oracle.run_trials(g, float(campaign["qber"][pt]), seeds[:k] + campaign["seed_offset"][pt], threads=4)
        assert (out[:, 0] == campaign["iterations"][pt, :k]).all(), pt
        assert ((out[:, 1] | (out[:, 2] << 1)) == campaign["flags"][pt, :k]).all(), pt


def test_reference_equals_fixture_and_restatement(oracle, graphs, campaign):
    """The reference's trial seeds (Xoshiro256PlusPlus(777), src/simulation.cpp:222-228) and key generator
    (src/array_and_matrix_operations.cpp:424-460), as recorded in frames_n10240.npz, against the restatement: same seeds ->
    same exact QBER, same Alice and Bob keys. The run_trial outcomes of the same seeds are pinned by test_restatement_equals_fixture."""
    g = graphs[NS]
    z = np.load(GOLD / "frames_n10240.npz")
    seeds = oracle.trial_seeds(int(campaign["simulation_seed"]), 8)
    assert set(z["seed"].tolist()) <= set(seeds.tolist())
    for q, seed, ex, a_packed, b_packed in zip(z["q_req"], z["seed"], z["q_exact"], z["alice"], z["bob"]):
        a, b, ex2 = oracle.generate(int(seed), g.n, float(q))
        assert ex2 == ex, (q, seed)
        assert (a == np.unpackbits(a_packed, bitorder="little")[:g.n]).all() and (b == np.unpackbits(b_packed, bitorder="little")[:g.n]).all(), (q, seed)


@pytest.mark.parametrize("name", ["dense_n6_m4", "dense_n7_m3", "dense_n10_m5"])
def test_reference_regular_and_irregular_entries_on_small_codes(oracle, graphs, name):
    """QKD_LDPC_regular (src/qkd_ldpc_algorithm.cpp:347-396) and QKD_LDPC_irregular (:398-447) of the reference itself, as
    recorded in small_codes.npz (every Alice x every single-bit error), against the restatement: iterations, flags, syndrome
    and decoded key; on the regular N=6 code both entries were recorded, so the two must also agree."""
    g = graphs[name]
    bits = lambda v, w: np.array([(int(v) >> i) & 1 for i in range(w)], np.int32)
    for av, epos, variant, it, sm, km, dv, sv in np.load(GOLD / "small_codes.npz")[name]:
        a = bits(av, g.n)
        b = a.copy(); b[epos] ^= 1
        got = oracle.qkd_ldpc(g, a, b, 1.0 / g.n)
        assert got[:3] == (it, bool(sm), bool(km)), (name, av, epos, variant, got[:3], (it, sm, km))
        assert (got[3] == bits(sv, g.m)).all() and (got[4] == bits(dv, g.n)).all(), (name, av, epos, variant)
