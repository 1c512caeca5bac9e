"""The fp64 check rule as the resident decoder runs it (qlb_test_f64_math op 6: MathF64::check_fast for W = 3 ... 8) against
f64_rule_restatement.c, a C restatement of the rule's operation sequence: every outgoing message bit for bit (NaN against NaN)."""
import ctypes as C
import hashlib
import subprocess
import tempfile
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SRC = Path(__file__).resolve().parent / "f64_rule_restatement.c"
_f64p = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")


def restatement():
    digest = hashlib.sha256(SRC.read_bytes()).hexdigest()[:16]
    out = Path(tempfile.gettempdir()) / f"qlb_f64_rule_restatement_{digest}.so"
    if not out.exists():
        tmp = out.with_suffix(f".{np.random.randint(1 << 30)}.tmp")
        subprocess.run(["gcc", "-std=c11", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-o", str(tmp), str(SRC), "-lm"],
                       check=True, capture_output=True)
        tmp.replace(out)
    lib = C.CDLL(str(out))
    lib.f64_rule_records.restype = None
    lib.f64_rule_records.argtypes = [C.c_long, _f64p, _f64p, _f64p]
    return lib


def records(rng, n, thr_eff):
    """n checks of random weight 3 ... 8: messages of decoder-like magnitudes, a share of them replaced by special values"""
    a = rng.standard_normal((n, 8)) * rng.choice([0.5, 3.0, 10.0, 40.0], (n, 1))
    specials = np.array([0.0, -0.0, 5e-324, -5e-324, 2.2e-308, -1e-310, np.nan, 100.0, -100.0, 37.0, -37.4, 38.5, -39.0, 40.0,
                         np.inf, -np.inf, 1e-17, -3e-9, 700.0, 1e300])
    pick = rng.random((n, 8)) < 0.04
    a[pick] = rng.choice(specials, pick.sum())
    near = rng.random((n, 8)) < 0.05  # around the magnitude where tanh(m / 2) rounds to 1
    a[near] = rng.uniform(36.0, 40.0, near.sum()) * rng.choice([-1.0, 1.0], near.sum())
    b = np.zeros((n, 8))
    b[:, 0] = rng.integers(3, 9, n)
    b[:, 1] = rng.integers(0, 2, n)
    b[:, 2] = thr_eff
    return np.ascontiguousarray(a), np.ascontiguousarray(b)


@pytest.mark.parametrize("thr_eff", [100.0, 20.0, 1000.0, np.inf], ids=["clamp100", "clamp20", "clamp1000", "no_clamp"])
def test_check_rule_bit_exact(ctx, thr_eff):
    lib = restatement()
    rng = np.random.default_rng(int(thr_eff) if np.isfinite(thr_eff) else 7)
    n = 1_000_000 if thr_eff == 100.0 else 250_000
    a, b = records(rng, n, thr_eff)
    got = ctx.f64_math(6, a.ravel(), b.ravel()).reshape(n, 8)
    want = np.zeros_like(a)
    lib.f64_rule_records(n, a, b, want)
    used = np.arange(8)[None, :] < b[:, :1]
    same = (got.view(np.uint64) == want.view(np.uint64)) | (np.isnan(got) & np.isnan(want))
    bad = np.argwhere(used & ~same)
    assert bad.size == 0, (len(bad), [(a[i].tolist(), b[i, :3].tolist(), got[i, j], want[i, j]) for i, j in bad[:3]])
    assert (got[~used] == 0).all()
