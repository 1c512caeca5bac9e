"""TEST INFRASTRUCTURE ONLY: ctypes binding of min_sum_restatement.c, the CPU restatement of the fp32 min-sum decoder.

The library is compiled on first use into a temporary directory (the tree may be read-only), together with the pinned
restatement's sp_oracle.c for key generation and the syndrome. Graphs are oracle.bindings.Graph objects.
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
SOURCES = [HERE / "min_sum_restatement.c", ROOT / "oracle" / "restatement" / "sp_oracle.c"]
HEADERS = [ROOT / "oracle" / "restatement" / "sp_oracle.h", ROOT / "oracle" / "restatement" / "sp_decode_body.inc"]

_i32p = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
_u64p = np.ctypeslib.ndpointer(dtype=np.uint64, flags="C_CONTIGUOUS")
_f64p = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")


class _SP(C.Structure):
    _fields_ = [("iterations_num", C.c_uint64), ("syndromes_match", C.c_int32)]


class _LDPC(C.Structure):
    _fields_ = [("sp_res", _SP), ("keys_match", C.c_int32)]


def build() -> Path:
    digest = hashlib.sha256(b"".join(p.read_bytes() for p in SOURCES + HEADERS)).hexdigest()[:16]
    out = Path(tempfile.gettempdir()) / f"qlb_min_sum_restatement_{digest}.so"
    if not out.exists():
        tmp = out.with_suffix(f".{np.random.randint(1 << 30)}.tmp")
        subprocess.run(["gcc", "-std=c11", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fopenmp", "-pthread",
                        "-o", str(tmp), *map(str, SOURCES), "-lm"], check=True, capture_output=True)
        tmp.replace(out)
    return out


class MinSumRestatement:
    def __init__(self):
        lib = C.CDLL(str(build()))
        lib.msr_sum_product.restype = _SP
        lib.msr_sum_product.argtypes = [C.c_void_p, _f64p, _i32p, C.c_uint64, C.c_int, C.c_double, C.c_float, _i32p]
        lib.msr_qkd_ldpc.restype = _LDPC
        lib.msr_qkd_ldpc.argtypes = [C.c_void_p, _i32p, _i32p, C.c_double, C.c_uint64, C.c_int, C.c_double, C.c_float,
                                     _i32p, _i32p]
        lib.msr_run_trials.restype = C.c_int
        lib.msr_run_trials.argtypes = [C.c_void_p, C.c_double, _u64p, C.c_uint64, C.c_int, C.c_uint64, C.c_int, C.c_double,
                                       C.c_float, _u64p, C.c_void_p]
        self.lib = lib

    def sum_product(self, g, llr, syndrome, scale, max_it=100, thr=100.0, enable_thr=True):
        """-> (iterations, syndromes_match, bits)"""
        out = np.zeros(g.n, np.int32)
        r = self.lib.msr_sum_product(C.byref(g._c), np.ascontiguousarray(llr, np.float64),
                                     np.ascontiguousarray(syndrome, np.int32), max_it, int(enable_thr), thr, scale, out)
        return int(r.iterations_num), bool(r.syndromes_match), out

    def qkd_ldpc(self, g, alice, bob, qber, scale, max_it=100, thr=100.0, enable_thr=True):
        """-> (iterations, syndromes_match, keys_match, alice_syndrome, decoded)"""
        syn, dec = np.zeros(g.m, np.int32), np.zeros(g.n, np.int32)
        r = self.lib.msr_qkd_ldpc(C.byref(g._c), np.ascontiguousarray(alice, np.int32), np.ascontiguousarray(bob, np.int32),
                                  qber, max_it, int(enable_thr), thr, scale, syn, dec)
        return int(r.sp_res.iterations_num), bool(r.sp_res.syndromes_match), bool(r.keys_match), syn, dec

    def run_trials(self, g, qber, seeds, scale, threads=8, max_it=100, thr=100.0, enable_thr=True, want_decoded=False):
        """-> out3 [count][3] = (iterations, syndromes_match, keys_match)[, decoded [count][n]]"""
        seeds = np.ascontiguousarray(seeds, np.uint64)
        out3 = np.zeros(3 * seeds.size, np.uint64)
        dec = np.zeros((seeds.size, g.n), np.int32) if want_decoded else None
        rc = self.lib.msr_run_trials(C.byref(g._c), qber, seeds, seeds.size, threads, max_it, int(enable_thr), thr, scale,
                                     out3, dec.ctypes.data if want_decoded else None)
        if rc != 0:
            raise RuntimeError(f"Key size '{g.n}' is too small for QBER.")
        out3 = out3.reshape(-1, 3)
        return (out3, dec) if want_decoded else out3
