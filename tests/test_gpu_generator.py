"""The device key generator (generate_keys_kernel, csrc/qlb_generate.cuh) against the reference's generator as the pinned
restatement states it (oracle.generate: the full N-entry shuffle, so it also checks the kernel's K-prefix shortcut), in every
state tier, CTA shape and slice the launcher (qlb_generate_device) can choose, and on the Lemire redraw path.

Every frame the library decodes in qlb_run_trials, the C++ sweep and bench.py comes from this kernel, so each case compares Alice,
Bob and the exact QBER with the oracle, checks that Alice and Bob differ in exactly K = floor(N q) bits and that the padding bits
of the last word are zero.

The launcher keeps each trial's K-entry shuffle prefix in shared memory when 64, else 32, trials' prefixes fit the block budget
(the device's opt-in shared memory minus 1 KB), and in global memory with 128 threads per CTA otherwise, in slices of at most
2^30 bytes of prefixes (one launch each). Positions are uint16_t up to N = 65 536, uint32_t above. Each case computes that choice
from torch's view of the device (plan()), picks q = (K + 0.5) / N so the host's floor(N q) lands on the intended K, and confirms
under torch.profiler that the kernel ran as claimed: template arguments, block size, dynamic shared memory, grid and the number of
launches.
"""
import json
import os
import re
import tempfile
from collections import namedtuple

import numpy as np
import pytest
import torch

from generator_replay import GeneratorReplay
from qkd_ldpc_b200 import capi

pytestmark = pytest.mark.gpu

MASK64 = (1 << 64) - 1
SLICE_BYTES = 1 << 30
FRAME_COUNTS = (1, 31, 33, 65, 129)  # the last CTA partial at 32, 64 and 128 threads
NS = "n10240_m5231_cw3_seed666"
PEG = "peg_n100000_m51080_cw3_seed666_bfs2000"

Plan = namedtuple("Plan", "pos shared threads smem slice")


def plan(n, k):
    """qlb_generate_device's choice for an n-bit key with k flipped positions: position bytes, shared or global state, threads per
    CTA, dynamic shared memory per CTA and frames per launch (None: every frame in one launch)."""
    pos = 2 if n <= 65536 else 4
    state = k * pos
    budget = torch.cuda.get_device_properties(0).shared_memory_per_block_optin - 1024
    threads = 64 if 64 * state <= budget else 32
    if threads * state <= budget:
        return Plan(pos, True, threads, threads * state, None)
    return Plan(pos, False, 128, 0, max(1, SLICE_BYTES // state))


def tier_k(pos, edge):
    """The largest K of a tier, and the first K past it: edge = (64 | 32, 0 | 1)."""
    budget = torch.cuda.get_device_properties(0).shared_memory_per_block_optin - 1024
    threads, past = edge
    return budget // (threads * pos) + past


def q_for(n, k):
    q = (k + 0.5) / n
    assert int(n * q) == k
    return q


def expected_launches(p, frame_counts):
    out = []
    for c in frame_counts:
        sl = p.slice or c
        out += [dict(pos=p.pos, shared=p.shared, block=p.threads, grid=-(-min(sl, c - f0) // p.threads), smem=p.smem)
                for f0 in range(0, c, sl)]
    return out


_KERNEL = re.compile(r"generate_keys_kernel<unsigned (short|int), (true|false|1|0)>")


@pytest.fixture(scope="module")
def gctx():
    """A context of this file's own, so the global-state scratch of the N = 10^6 cases (about 1 GB) is freed with it."""
    c = capi.Context(0)
    yield c
    c.close()
    torch.cuda.empty_cache()


@pytest.fixture(scope="module")
def replay():
    return GeneratorReplay()


def profiled(fn):
    """fn() under torch.profiler -> (fn's result, every generate_keys_kernel launch in order: position bytes, shared state, block
    size, grid size, shared memory)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as fh:
            events = json.load(fh)["traceEvents"]
    launches = []
    for e in sorted((e for e in events if e.get("cat") == "kernel" and "generate_keys_kernel" in e.get("name", "")),
                    key=lambda e: e["ts"]):
        m = _KERNEL.search(e["name"])
        assert m, e["name"]
        args = e["args"]
        launches.append(dict(pos=2 if m[1] == "short" else 4, shared=m[2] in ("true", "1"), block=args["block"][0],
                             grid=args["grid"][0], smem=args["shared memory"]))
    return out, launches


def padding_of(n):
    pad = np.zeros((n + 31) // 32, np.uint32)
    if n % 32:
        pad[-1] = np.uint32((0xFFFFFFFF << (n % 32)) & 0xFFFFFFFF)
    return pad


def check_structure(n, q, a, b, exact):
    """Exact QBER floor(n q) / n, zero padding, Alice and Bob apart in exactly K bits -- on every frame of the call."""
    k = int(n * q)
    assert exact == k / n, (n, q, exact)
    assert a.shape == b.shape == (a.shape[0], (n + 31) // 32)
    pad = padding_of(n)
    assert not (a & pad).any() and not (b & pad).any(), (n, q)
    flips = np.bitwise_count(a ^ b).sum(axis=1, dtype=np.int64)
    assert (flips == k).all(), (n, q, np.flatnonzero(flips != k)[:8])


def check_oracle(oracle, n, q, seeds, a, b, exact, frames=None, offset=0):
    """Frames `frames` (default all) of a call over `seeds` equal the oracle's keys of seed + offset (mod 2^64)."""
    for f in range(len(seeds)) if frames is None else frames:
        wa, wb, wq = oracle.generate((int(seeds[f]) + offset) & MASK64, n, q)
        assert wq == exact, (n, q, f)
        assert (a[f] == capi.pack_bits(wa)[0]).all(), ("alice", n, q, f)
        assert (b[f] == capi.pack_bits(wb)[0]).all(), ("bob", n, q, f)


# ---- 1. tiers: K on both sides of each shared-memory threshold, partial last CTAs --------------------------------------------------
TIER_CASES = [(n, edge) for n in (65536, 100001) for edge in ((64, 0), (64, 1), (32, 0), (32, 1))]


@pytest.mark.parametrize("n,edge", TIER_CASES, ids=[f"n{n}-k{'past' if e[1] else 'last'}{e[0]}" for n, e in TIER_CASES])
def test_state_tier_edges(gctx, oracle, n, edge):
    """n = 65 536 (uint16_t positions, Alice in uint4 stores) and n = 100 001 (uint32_t positions, odd n: the pair loop runs on odd
    i through the 32- to 64-bit division switch at (i+1)(i+2) > 2^32): the last K that fits 64 trials' prefixes in shared memory,
    the first that does not (32 threads), the last that fits 32 trials' and the first that goes to global memory (128 threads).
    Frame counts 1, 31, 33, 65, 129 in calls of their own; every frame against the oracle."""
    pos = 2 if n <= 65536 else 4
    k = tier_k(pos, edge)
    q = q_for(n, k)
    p = plan(n, k)
    want_tier = {(64, 0): (True, 64), (64, 1): (True, 32), (32, 0): (True, 32), (32, 1): (False, 128)}[edge]
    assert (p.shared, p.threads) == want_tier and p.pos == pos
    seeds = oracle.trial_seeds(4100 + k, max(FRAME_COUNTS))
    calls, launches = profiled(lambda: [gctx.generate(n, seeds[:c], q) for c in FRAME_COUNTS])
    assert launches == expected_launches(p, FRAME_COUNTS), (n, k, launches)
    full = calls[-1]
    check_structure(n, q, *full)
    check_oracle(oracle, n, q, seeds, *full)
    for c, (a, b, exact) in zip(FRAME_COUNTS, calls):
        assert exact == full[2] and (a == full[0][:c]).all() and (b == full[1][:c]).all(), (n, k, c)


# ---- 2. shapes: N around the uint16_t / uint32_t boundary, the uint4 Alice path with uint32_t state, K > N / 2, K = N - 1 ----------
SHAPES = [(65535, 0.02), (65535, 0.2), (65536, 0.01), (65536, 0.2), (65537, 0.01), (65537, 0.3), (100001, 0.005), (100001, 0.05),
          (131072, 0.005), (131072, 0.3), (10**6, 0.45), (10**6, 0.9), (10240, float(np.nextafter(1.0, 0.0))), (100, 0.29)]


@pytest.mark.parametrize("n,q", SHAPES, ids=[f"n{n}-q{q!r}" for n, q in SHAPES])
def test_shapes(gctx, oracle, n, q):
    """33 frames (a partial last CTA at every block size) at key lengths either side of the uint16_t / uint32_t boundary, odd n
    above it, n = 131 072 (Alice's uint4 stores with uint32_t positions), n = 10^6 with K > n / 2, q just below 1 (K = n - 1) and
    q = 0.29 at n = 100, where n q = 28.999... in double, so K = 28 and the exact QBER is 28 / 100 as the reference forms it."""
    k = int(n * q)
    if q > 0.99:
        assert k == n - 1
    if n == 100:
        assert k == 28
    p = plan(n, k)
    seeds = oracle.trial_seeds(4200 + n % 997, 33)
    (a, b, exact), launches = profiled(lambda: gctx.generate(n, seeds, q))
    assert launches == expected_launches(p, [33]), (n, q, launches)
    check_structure(n, q, a, b, exact)
    check_oracle(oracle, n, q, seeds, a, b, exact)


# ---- 3. slices of global-state frames ----------------------------------------------------------------------------------------------
def test_global_state_slices(gctx, oracle):
    """n = 10^6, q = 0.9: 3.6 MB of prefix per trial, so a launch takes at most 2^30 / 3.6 MB = 298 frames. 650 frames in one call
    are 3 launches, the last one short; each reads its seeds and writes its keys at the slice's frame offset. Every frame must equal
    the same seed's frame from calls of at most one slice that place it elsewhere in the batch (windows starting half a slice in),
    frames 0, slice - 1, slice, slice + 1, 2 slice and the last one the oracle and a one-frame call."""
    n, q = 10**6, 0.9
    k = int(n * q)
    p = plan(n, k)
    assert not p.shared and p.slice < 325
    frames = 650
    assert -(-frames // p.slice) >= 3 and frames % p.slice
    seeds = oracle.trial_seeds(4300, frames)
    (a, b, exact), launches = profiled(lambda: gctx.generate(n, seeds, q))
    assert launches == expected_launches(p, [frames]), launches
    assert len(launches) == -(-frames // p.slice)
    check_structure(n, q, a, b, exact)
    half = p.slice // 2
    edges = list(range(half, frames, p.slice))
    for lo, hi in zip([0] + edges, edges + [frames]):
        wa, wb, wq = gctx.generate(n, seeds[lo:hi], q)
        assert wq == exact and (wa == a[lo:hi]).all() and (wb == b[lo:hi]).all(), (lo, hi)
    picks = [0, p.slice - 1, p.slice, p.slice + 1, 2 * p.slice, frames - 1]
    check_oracle(oracle, n, q, seeds, a, b, exact, frames=picks)
    for f in picks:
        wa, wb, _ = gctx.generate(n, seeds[f:f + 1], q)
        assert (wa[0] == a[f]).all() and (wb[0] == b[f]).all(), f


# ---- 4. Lemire redraws -------------------------------------------------------------------------------------------------------------
# Seeds whose shuffle at n = 10^6 rejects one draw, and where (the first position i of the pair): trials 88, 92, 630, 843 and 1931
# of simulation seed 4 (tests/generator_replay.py's scan: 11 of its first 2 000 trials redraw), and two raw seeds found by an
# earlier scan. Trial 0 of simulation seed 4 draws no redraw (the control).
REDRAWS = {11679853522669457157: [455374], 10162179824987653725: [983062], 5414213607530400652: [735780],
           16286656810267357581: [910948], 14032007756207970399: [328568], 4964135871473638144: [590766],
           16691737426576479127: [975168], 12535900630535485233: []}


def test_lemire_redraws(gctx, oracle, replay):
    """The replay finds each seed's redraws where recorded; at q = 0.9 (K = 900 000) and at q = 0.45 (K = 450 000) redraws fall
    below K for some seeds (the prefix swap) and at or above it for others (the write into the prefix), and the device keys equal
    the oracle's."""
    n = 10**6
    seeds = np.array(list(REDRAWS), np.uint64)
    for s, want in REDRAWS.items():
        assert replay.redraws(s, n) == want, s
    for q in (0.9, 0.45):
        k = int(n * q)
        at = [i for r in REDRAWS.values() for i in r]
        assert any(i < k for i in at) and any(i >= k for i in at), q
        p = plan(n, k)
        (a, b, exact), launches = profiled(lambda: gctx.generate(n, seeds, q))
        assert launches == expected_launches(p, [len(seeds)]), launches
        check_structure(n, q, a, b, exact)
        check_oracle(oracle, n, q, seeds, a, b, exact)


# ---- 5. seed offsets and the device entry --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,k", [(10240, 300), (100001, 1809)], ids=["shared-u16", "global-u32"])
def test_seed_offset_wraps(gctx, oracle, n, k):
    """seed + seed_offset wraps modulo 2^64 as the reference's uint64_t addition does, in shared and global state."""
    q = q_for(n, k)
    p = plan(n, k)
    seeds = oracle.trial_seeds(4400, 65)
    for off in (MASK64, (1 << 63) + 12345, MASK64 - int(seeds.min()) + 1):
        assert any(int(s) + off > MASK64 for s in seeds)
        (a, b, exact), launches = profiled(lambda: gctx.generate(n, seeds, q, seed_offset=off))
        assert launches == expected_launches(p, [len(seeds)]), launches
        check_structure(n, q, a, b, exact)
        check_oracle(oracle, n, q, seeds, a, b, exact, offset=off)


def test_device_entry_equals_host_entry(gctx, oracle):
    """qlb_generate_device on caller-owned device buffers equals qlb_generate_batch_packed at a global-state point with slices
    (n = 10^6, q = 0.45: 1.8 MB per prefix, 596 frames per launch; 700 frames make two launches) and a wrapping seed offset."""
    n, q, frames, off = 10**6, 0.45, 700, MASK64 - 3
    p = plan(n, int(n * q))
    assert not p.shared and p.slice < frames
    seeds = oracle.trial_seeds(4500, frames)
    dev = torch.device("cuda", gctx.device)
    words = (n + 31) // 32
    d_seeds = torch.from_numpy(seeds.view(np.int64)).to(dev)
    d_a = torch.full((frames, words), -1, dtype=torch.int32, device=dev)
    d_b = torch.full_like(d_a, -1)
    torch.cuda.synchronize()

    def run():
        ex = gctx.generate_device(n, frames, d_seeds.data_ptr(), q, d_a.data_ptr(), d_b.data_ptr(), seed_offset=off)
        gctx.synchronize()
        return ex

    ex, launches = profiled(run)
    assert launches == expected_launches(p, [frames]), launches
    a, b = d_a.cpu().numpy().view(np.uint32), d_b.cpu().numpy().view(np.uint32)
    del d_seeds, d_a, d_b
    ha, hb, hex_ = gctx.generate(n, seeds, q, seed_offset=off)
    assert ex == hex_ and (a == ha).all() and (b == hb).all()
    check_structure(n, q, a, b, ex)
    check_oracle(oracle, n, q, seeds, a, b, ex, frames=[0, p.slice - 1, p.slice, frames - 1], offset=off)


# ---- 6. end to end: qlb_run_trials at the tiers no other test reaches --------------------------------------------------------------
E2E = [(PEG, 0.01, (4, True, 32)), (PEG, 0.05, (4, False, 128)), (NS, 0.18, (2, True, 32))]
E2E_MAX_IT = 10


@pytest.mark.parametrize("key,q,tier", E2E, ids=["peg100k-q0.01", "peg100k-q0.05", "n10240-q0.18"])
def test_run_trials_at_new_tiers(gctx, dev_codes, graphs, oracle, key, q, tier):
    """qlb_run_trials (keys drawn on the device, fp64 decode, max_it 10) equals the oracle's run_trial frame by frame -- iterations
    and both flags -- on the N = 100 000 PEG code with uint32_t state in shared memory at 32 threads (q = 0.01) and in global memory
    (q = 0.05), and on the N = 10 240 code with uint16_t state at 32 threads (q = 0.18)."""
    g, code = graphs[key], dev_codes[key]
    p = plan(g.n, int(g.n * q))
    assert (p.pos, p.shared, p.threads) == tier
    seeds = oracle.trial_seeds(4600, 65)
    params = capi.make_params(64, E2E_MAX_IT, 100.0, True)
    (it, res, exact), launches = profiled(lambda: gctx.run_trials(code, params, seeds, q, seed_offset=7))
    assert launches == expected_launches(p, [len(seeds)]), launches
    want = oracle.run_trials(g, q, seeds + np.uint64(7), threads=8, max_it=E2E_MAX_IT)
    assert exact == int(g.n * q) / g.n
    assert (it == want[:, 0]).all(), (key, q, np.flatnonzero(it != want[:, 0])[:8])
    assert ((res & 1) == want[:, 1]).all() and (((res >> 1) & 1) == want[:, 2]).all(), (key, q)
