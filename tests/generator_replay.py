"""TEST INFRASTRUCTURE ONLY: ctypes binding of generator_replay.c, which replays one key generation's random stream and reports
the shuffle's Lemire redraws.

The library is compiled on first use into a temporary directory (the tree may be read-only), together with the pinned
restatement's sp_oracle.c for the PRNG.

Run as a script, it repeats the scan that chose the redraw seeds of tests/test_gpu_generator.py: the first 2 000 trial seeds of
simulation seed 4 at n = 10^6, and for every seed with a redraw its raw value and the redraw positions (11 of the 2 000 redraw,
each once; about 10 s).
"""
from __future__ import annotations

import ctypes as C
import hashlib
import subprocess
import tempfile
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent
SOURCES = [HERE / "generator_replay.c", ROOT / "oracle" / "restatement" / "sp_oracle.c"]
HEADERS = [ROOT / "oracle" / "restatement" / "sp_oracle.h", ROOT / "oracle" / "restatement" / "sp_decode_body.inc"]

_u64p = np.ctypeslib.ndpointer(dtype=np.uint64, flags="C_CONTIGUOUS")


def build() -> Path:
    digest = hashlib.sha256(b"".join(p.read_bytes() for p in SOURCES + HEADERS)).hexdigest()[:16]
    out = Path(tempfile.gettempdir()) / f"qlb_generator_replay_{digest}.so"
    if not out.exists():
        tmp = out.with_suffix(f".{np.random.randint(1 << 30)}.tmp")
        subprocess.run(["gcc", "-std=c11", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-pthread", "-o", str(tmp),
                        *map(str, SOURCES), "-lm"], check=True, capture_output=True)
        tmp.replace(out)
    return out


class GeneratorReplay:
    def __init__(self):
        lib = C.CDLL(str(build()))
        lib.gr_redraws.restype = C.c_uint64
        lib.gr_redraws.argtypes = [C.c_uint64, C.c_uint64, _u64p, C.c_uint64]
        self.lib = lib

    def redraws(self, seed: int, n: int, cap: int = 16) -> list[int]:
        """The first position i of the pair (i, i+1) of every rejected shuffle draw of an n-bit key from `seed`, in order."""
        pos = np.zeros(cap, np.uint64)
        count = int(self.lib.gr_redraws(int(seed) & 0xFFFFFFFFFFFFFFFF, int(n), pos, cap))
        if count == 0xFFFFFFFFFFFFFFFF:
            raise ValueError(f"n = {n}: the shuffle draws one position per draw, not pairs")
        if count > cap:
            raise ValueError(f"{count} redraws, more than cap = {cap}")
        return [int(x) for x in pos[:count]]


def scan(n=1_000_000, simulation_seed=4, count=2000):
    """-> [(trial index, raw seed, redraw positions)] for the trials of `simulation_seed` whose shuffle redraws."""
    from oracle.bindings import Restatement
    rep = GeneratorReplay()
    seeds = Restatement().trial_seeds(simulation_seed, count)
    return [(k, int(s), r) for k, s in enumerate(seeds) if (r := rep.redraws(int(s), n))]


if __name__ == "__main__":
    import sys
    sys.path.insert(0, str(ROOT))
    for k, s, r in scan():
        print(f"trial {k:5d}  seed {s:20d}  redraws at {r}")
