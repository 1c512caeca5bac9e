"""ctypes binding of libqkdldpc_b200.so -- a thin, typed mirror of include/qkd_ldpc_b200.h.

There is no CPU implementation behind these classes: a missing library or a missing GPU raises.
"""
from __future__ import annotations

import os
import ctypes as C
from pathlib import Path

import numpy as np

from . import build as _build

QLB_OK = 0
PRECISION_F64 = 64
PRECISION_F32 = 32
FLAG_F32_FAST_MATH = 1
FLAG_F64_FUSED_RATIO = 2
RES_SYNDROMES_MATCH = 1
RES_KEYS_MATCH = 2

EXPORTS = [
    "qlb_version", "qlb_last_error", "qlb_device_count",
    "qlb_code_create", "qlb_code_destroy", "qlb_code_n", "qlb_code_m", "qlb_code_edges", "qlb_code_words_n",
    "qlb_code_words_m", "qlb_code_max_bit_weight", "qlb_code_max_check_weight", "qlb_code_slots", "qlb_code_layout",
    "qlb_code_gather_wavefronts",
    "qlb_ctx_create", "qlb_ctx_destroy", "qlb_ctx_device", "qlb_ctx_sm_count", "qlb_ctx_stream", "qlb_ctx_last_decoder", "qlb_ctx_synchronize",
    "qlb_ctx_counters", "qlb_ctx_timer_start", "qlb_ctx_timer_stop",
    "qlb_syndrome_batch", "qlb_syndrome_batch_packed", "qlb_sum_product_batch", "qlb_sum_product_trace",
    "qlb_reconcile_batch", "qlb_reconcile_batch_packed", "qlb_reconcile_device", "qlb_stats_allreduce", "qlb_stats_comm_prepare",
    "qlb_generate_batch_packed", "qlb_generate_device", "qlb_run_trials", "qlb_test_f64_math",
]


class QlbError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"[qlb {code}] {message}")
        self.code = code
        self.message = message


class DecodeParams(C.Structure):
    _fields_ = [
        ("precision", C.c_int32),
        ("max_iterations", C.c_int32),
        ("enable_threshold", C.c_int32),
        ("flags", C.c_int32),
        ("threshold", C.c_double),
        ("stream_max_bundles", C.c_int32),
        ("stream_no_repack", C.c_int32),
        ("block_threads", C.c_int32),
        ("reserved", C.c_int32),
    ]


_lib = None


def load_library(path: Path | None = None) -> C.CDLL:
    """Loads (building first if the .so is absent) the C-ABI library. Raises if it cannot be had."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = Path(path) if path else Path(os.environ.get("QLB_LIBRARY") or _build.LIB_PATH)  # QLB_LIBRARY: kernel-tuning experiments
    if not p.exists():
        _build.build_library()
    lib = C.CDLL(str(p))
    vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
    lib.qlb_version.restype = C.c_int
    lib.qlb_last_error.restype = C.c_char_p
    lib.qlb_device_count.restype = C.c_int
    lib.qlb_code_create.argtypes = [i32, i32, vp, vp, vp, vp, C.POINTER(vp)]
    lib.qlb_code_destroy.argtypes = [vp]
    lib.qlb_code_destroy.restype = None
    for f in ("qlb_code_n", "qlb_code_m", "qlb_code_edges", "qlb_code_words_n", "qlb_code_words_m",
              "qlb_code_max_bit_weight", "qlb_code_max_check_weight", "qlb_code_slots"):
        getattr(lib, f).argtypes = [vp]
        getattr(lib, f).restype = i32
    lib.qlb_code_layout.argtypes = [vp, vp, vp, vp]
    lib.qlb_code_gather_wavefronts.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    lib.qlb_ctx_create.argtypes = [C.c_int, C.POINTER(vp)]
    lib.qlb_ctx_destroy.argtypes = [vp]
    lib.qlb_ctx_destroy.restype = None
    lib.qlb_ctx_device.argtypes = [vp]
    lib.qlb_ctx_sm_count.argtypes = [vp]
    lib.qlb_ctx_stream.argtypes = [vp]
    lib.qlb_ctx_stream.restype = vp
    lib.qlb_ctx_last_decoder.argtypes = [vp]
    lib.qlb_ctx_last_decoder.restype = C.c_char_p
    lib.qlb_ctx_synchronize.argtypes = [vp]
    lib.qlb_ctx_counters.argtypes = [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.c_int]
    lib.qlb_ctx_timer_start.argtypes = [vp]
    lib.qlb_ctx_timer_stop.argtypes = [vp, C.POINTER(C.c_float)]
    pp = C.POINTER(DecodeParams)
    lib.qlb_syndrome_batch.argtypes = [vp, vp, i64, vp, vp]
    lib.qlb_syndrome_batch_packed.argtypes = [vp, vp, i64, vp, vp]
    lib.qlb_sum_product_batch.argtypes = [vp, vp, pp, i64, vp, vp, vp, vp, vp]
    lib.qlb_sum_product_trace.argtypes = [vp, vp, pp, vp, vp, i32, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.qlb_reconcile_batch.argtypes = [vp, vp, pp, i64, vp, vp, vp, vp, vp, vp, vp]
    lib.qlb_reconcile_batch_packed.argtypes = [vp, vp, pp, i64, vp, vp, vp, vp, vp, vp, vp]
    lib.qlb_reconcile_device.argtypes = [vp, vp, pp, i64, vp, vp, vp, vp, vp, vp, vp]
    lib.qlb_stats_allreduce.argtypes = [C.POINTER(vp), C.c_int, C.POINTER(vp), C.c_size_t]
    dp = C.POINTER(C.c_double)
    lib.qlb_generate_batch_packed.argtypes = [vp, i32, i64, vp, C.c_uint64, C.c_double, vp, vp, dp]
    lib.qlb_generate_device.argtypes = [vp, i32, i64, vp, C.c_uint64, C.c_double, vp, vp, dp]
    lib.qlb_run_trials.argtypes = [vp, vp, pp, i64, vp, C.c_uint64, C.c_double, vp, vp, dp]
    lib.qlb_test_f64_math.argtypes = [vp, C.c_int, i64, vp, vp, vp]
    if path is None:
        _lib = lib
    return lib


def _check(lib, rc: int):
    if rc != QLB_OK:
        raise QlbError(rc, lib.qlb_last_error().decode(errors="replace"))


def _ptr(a):
    if a is None:
        return None
    if isinstance(a, int):
        return a
    return a.ctypes.data


def make_params(precision=64, max_iterations=100, threshold=100.0, enable_threshold=True, fast_math=False, tier=None,
                stream_max_bundles=0, stream_no_repack=False, block_threads=0):
    if fast_math:  # the cheaper check rule of either precision
        flags = FLAG_F32_FAST_MATH if int(precision) == 32 else FLAG_F64_FUSED_RATIO
    else:
        flags = 0
    if tier is not None:
        flags |= (int(tier) + 1) << 8  # QLB_FLAG_TEST_TIER: force a slower storage tier
    return DecodeParams(int(precision), int(max_iterations), int(bool(enable_threshold)), flags, float(threshold),
                        int(stream_max_bundles), int(bool(stream_no_repack)), int(block_threads), 0)


def pack_bits(bits, n=None) -> np.ndarray:
    """[F][n] 0/1 -> [F][ceil(n/32)] uint32, bit i at word i//32, position i%32."""
    b = np.asarray(bits)
    if b.ndim == 1:
        b = b[None, :]
    n = b.shape[1] if n is None else n
    words = (n + 31) // 32
    pad = np.zeros((b.shape[0], words * 32), np.uint8)
    pad[:, :n] = b[:, :n] & 1
    return np.ascontiguousarray(np.packbits(pad, axis=1, bitorder="little").view(np.uint32))


def unpack_bits(words, n) -> np.ndarray:
    w = np.ascontiguousarray(words, dtype=np.uint32)
    if w.ndim == 1:
        w = w[None, :]
    return np.unpackbits(w.view(np.uint8), axis=1, bitorder="little")[:, :n].astype(np.int32)


class Code:
    """A parity-check matrix prepared for the device (qlb_code)."""

    def __init__(self, n, m, row_ptr, col_idx, col_ptr, row_idx, lib=None):
        self.lib = lib or load_library()
        self._arrays = [np.ascontiguousarray(a, np.int32) for a in (row_ptr, col_idx, col_ptr, row_idx)]
        h = C.c_void_p()
        _check(self.lib, self.lib.qlb_code_create(int(n), int(m), *[a.ctypes.data for a in self._arrays], C.byref(h)))
        self.handle = h
        self.n, self.m = self.lib.qlb_code_n(h), self.lib.qlb_code_m(h)
        self.e = self.lib.qlb_code_edges(h)
        self.words_n, self.words_m = self.lib.qlb_code_words_n(h), self.lib.qlb_code_words_m(h)
        self.max_bit_w = self.lib.qlb_code_max_bit_weight(h)
        self.max_check_w = self.lib.qlb_code_max_check_weight(h)
        self.slots = self.lib.qlb_code_slots(h)

    @classmethod
    def from_graph(cls, g, lib=None):
        """g: any object with n, m, row_ptr, col_idx, col_ptr, row_idx."""
        return cls(g.n, g.m, g.row_ptr, g.col_idx, g.col_ptr, g.row_idx, lib=lib)

    def layout(self):
        slot_of_edge = np.zeros(self.e, np.uint32)
        bit_slots = np.zeros((self.max_bit_w, self.n), np.uint32)
        check_order = np.zeros(self.m, np.uint32)
        _check(self.lib, self.lib.qlb_code_layout(self.handle, _ptr(slot_of_edge), _ptr(bit_slots), _ptr(check_order)))
        return slot_of_edge, bit_slots, check_order

    def gather_wavefronts(self):
        a, b = C.c_double(), C.c_double()
        _check(self.lib, self.lib.qlb_code_gather_wavefronts(self.handle, C.byref(a), C.byref(b)))
        return a.value, b.value

    def close(self):
        if getattr(self, "handle", None):
            self.lib.qlb_code_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Context:
    """One GPU (qlb_ctx). Raises QlbError when no sm_100-class device is present -- there is no CPU fallback."""

    def __init__(self, device: int = 0, lib=None):
        self.lib = lib or load_library()
        h = C.c_void_p()
        _check(self.lib, self.lib.qlb_ctx_create(int(device), C.byref(h)))
        self.handle = h
        self.device = device
        self.sm_count = self.lib.qlb_ctx_sm_count(h)

    @property
    def stream(self) -> int:
        return int(self.lib.qlb_ctx_stream(self.handle) or 0)

    @property
    def last_decoder(self) -> str:
        """The decoder the last decode on this context launched (qlb_ctx_last_decoder)."""
        return self.lib.qlb_ctx_last_decoder(self.handle).decode()

    def synchronize(self):
        _check(self.lib, self.lib.qlb_ctx_synchronize(self.handle))

    def counters(self, reset=False):
        a, b = C.c_uint64(), C.c_uint64()
        _check(self.lib, self.lib.qlb_ctx_counters(self.handle, C.byref(a), C.byref(b), int(reset)))
        return a.value, b.value

    def timer_start(self):
        _check(self.lib, self.lib.qlb_ctx_timer_start(self.handle))

    def timer_stop(self) -> float:
        ms = C.c_float()
        _check(self.lib, self.lib.qlb_ctx_timer_stop(self.handle, C.byref(ms)))
        return ms.value

    # ---- reference-convention (one int per bit) entry points ----------------------------------------------------
    def syndrome(self, code: Code, bits):
        bits = np.ascontiguousarray(np.atleast_2d(bits), np.int32)
        out = np.zeros((bits.shape[0], code.m), np.int32)
        _check(self.lib, self.lib.qlb_syndrome_batch(self.handle, code.handle, bits.shape[0], _ptr(bits), _ptr(out)))
        return out

    def syndrome_packed(self, code: Code, bits_packed):
        bp = np.ascontiguousarray(np.atleast_2d(bits_packed), np.uint32)
        out = np.zeros((bp.shape[0], code.words_m), np.uint32)
        _check(self.lib, self.lib.qlb_syndrome_batch_packed(self.handle, code.handle, bp.shape[0], _ptr(bp), _ptr(out)))
        return out

    def sum_product(self, code: Code, params: DecodeParams, llr, syndrome, want_bits=True):
        llr = np.ascontiguousarray(np.atleast_2d(llr), np.float64)
        syn = np.ascontiguousarray(np.atleast_2d(syndrome), np.int32)
        f = llr.shape[0]
        bits = np.zeros((f, code.n), np.int32) if want_bits else None
        it = np.zeros(f, np.uint32)
        res = np.zeros(f, np.uint8)
        _check(self.lib, self.lib.qlb_sum_product_batch(self.handle, code.handle, C.byref(params), f, _ptr(llr), _ptr(syn),
                                                        _ptr(bits), _ptr(it), _ptr(res)))
        return it, res, bits

    def sum_product_trace(self, code: Code, params: DecodeParams, llr, syndrome, capacity: int):
        """One fp64 frame with the reference's TRACE_SUM_PRODUCT intermediates per iteration.
        Returns dict(E, L, z, s, M, bits, iterations, result); E/M are [capacity][edges] in the reference's row order."""
        llr = np.ascontiguousarray(llr, np.float64).reshape(code.n)
        syn = np.ascontiguousarray(syndrome, np.int32).reshape(code.m)
        cap = min(int(capacity), int(params.max_iterations))
        e = np.zeros((cap, code.e), np.float64)
        m = np.zeros((cap, code.e), np.float64)
        tot = np.zeros((cap, code.n), np.float64)
        z = np.zeros((cap, code.n), np.int32)
        s = np.zeros((cap, code.m), np.int32)
        bits = np.zeros(code.n, np.int32)
        it = np.zeros(1, np.uint32)
        res = np.zeros(1, np.uint8)
        _check(self.lib, self.lib.qlb_sum_product_trace(self.handle, code.handle, C.byref(params), _ptr(llr), _ptr(syn), cap,
                                                        _ptr(e), _ptr(tot), _ptr(z), _ptr(s), _ptr(m), _ptr(bits), _ptr(it), _ptr(res)))
        return dict(E=e, L=tot, z=z, s=s, M=m, bits=bits, iterations=int(it[0]), result=int(res[0]))

    def reconcile(self, code: Code, params: DecodeParams, alice, bob, qber, want_decoded=True, want_syndrome=False):
        alice = np.ascontiguousarray(np.atleast_2d(alice), np.int32)
        bob = np.ascontiguousarray(np.atleast_2d(bob), np.int32)
        f = alice.shape[0]
        q = np.ascontiguousarray(np.broadcast_to(np.asarray(qber, np.float64), (f,)))
        it, res = np.zeros(f, np.uint32), np.zeros(f, np.uint8)
        dec = np.zeros((f, code.n), np.int32) if want_decoded else None
        syn = np.zeros((f, code.m), np.int32) if want_syndrome else None
        _check(self.lib, self.lib.qlb_reconcile_batch(self.handle, code.handle, C.byref(params), f, _ptr(alice), _ptr(bob),
                                                      _ptr(q), _ptr(it), _ptr(res), _ptr(dec), _ptr(syn)))
        return it, res, dec, syn

    # ---- packed host buffers ------------------------------------------------------------------------------------
    def reconcile_packed(self, code: Code, params: DecodeParams, alice_packed, bob_packed, qber, want_decoded=True,
                         want_syndrome=False, out=None):
        ap = np.ascontiguousarray(np.atleast_2d(alice_packed), np.uint32)
        bp = np.ascontiguousarray(np.atleast_2d(bob_packed), np.uint32)
        f = ap.shape[0]
        q = np.ascontiguousarray(np.broadcast_to(np.asarray(qber, np.float64), (f,)))
        it, res = np.zeros(f, np.uint32), np.zeros(f, np.uint8)
        dec = np.zeros((f, code.words_n), np.uint32) if want_decoded else None
        syn = np.zeros((f, code.words_m), np.uint32) if want_syndrome else None
        _check(self.lib, self.lib.qlb_reconcile_batch_packed(self.handle, code.handle, C.byref(params), f, _ptr(ap), _ptr(bp),
                                                             _ptr(q), _ptr(it), _ptr(res), _ptr(dec), _ptr(syn)))
        return it, res, dec, syn

    def reconcile_packed_ptrs(self, code: Code, params: DecodeParams, n_frames, alice_ptr, bob_ptr, qber_ptr, it_ptr, res_ptr,
                              dec_ptr=None, syn_ptr=None):
        """Raw host pointers (e.g. pinned torch tensors' data_ptr())."""
        _check(self.lib, self.lib.qlb_reconcile_batch_packed(self.handle, code.handle, C.byref(params), int(n_frames), alice_ptr,
                                                             bob_ptr, qber_ptr, it_ptr, res_ptr, dec_ptr, syn_ptr))

    # ---- device-resident buffers (raw device pointers, e.g. torch tensors' data_ptr()) -----------------------------
    def reconcile_device(self, code: Code, params: DecodeParams, n_frames, d_alice, d_bob, d_log_prior, d_iterations, d_result,
                         d_decoded=None, d_syndrome=None):
        _check(self.lib, self.lib.qlb_reconcile_device(self.handle, code.handle, C.byref(params), int(n_frames), d_alice, d_bob,
                                                       d_log_prior, d_iterations, d_result, d_decoded, d_syndrome))

    # ---- on-device key generation (bit-exact with the reference's generator) -------------------------------------------
    def generate(self, n_bits, seeds, qber, seed_offset=0):
        seeds = np.ascontiguousarray(seeds, np.uint64)
        words = (n_bits + 31) // 32
        a = np.zeros((seeds.size, words), np.uint32)
        b = np.zeros((seeds.size, words), np.uint32)
        exact = C.c_double()
        _check(self.lib, self.lib.qlb_generate_batch_packed(self.handle, int(n_bits), seeds.size, _ptr(seeds), int(seed_offset), float(qber),
                                                            _ptr(a), _ptr(b), C.byref(exact)))
        return a, b, exact.value

    def generate_device(self, n_bits, n_frames, d_seeds, qber, d_alice, d_bob, seed_offset=0):
        exact = C.c_double()
        _check(self.lib, self.lib.qlb_generate_device(self.handle, int(n_bits), int(n_frames), d_seeds, int(seed_offset), float(qber),
                                                      d_alice, d_bob, C.byref(exact)))
        return exact.value

    def run_trials(self, code: Code, params: DecodeParams, seeds, qber, seed_offset=0):
        seeds = np.ascontiguousarray(seeds, np.uint64)
        it, res = np.zeros(seeds.size, np.uint32), np.zeros(seeds.size, np.uint8)
        exact = C.c_double()
        _check(self.lib, self.lib.qlb_run_trials(self.handle, code.handle, C.byref(params), seeds.size, _ptr(seeds), int(seed_offset),
                                                 float(qber), _ptr(it), _ptr(res), C.byref(exact)))
        return it, res, exact.value

    def f64_math(self, op: int, a, b=None):
        """Test probe: element-wise fp64 building blocks of the check rule (qlb_test_f64_math)."""
        a = np.ascontiguousarray(a, np.float64)
        b = None if b is None else np.ascontiguousarray(b, np.float64)
        out = np.zeros_like(a)
        _check(self.lib, self.lib.qlb_test_f64_math(self.handle, int(op), a.size, _ptr(a), _ptr(b), _ptr(out)))
        return out

    def stats_allreduce(self, vectors, others=()):
        """In-process NCCL sum of uint64 statistics over this context and `others` (one vector per context)."""
        ctxs = [self, *others]
        vecs = [np.ascontiguousarray(v, np.uint64) for v in vectors]
        assert len(vecs) == len(ctxs)
        cs = (C.c_void_p * len(ctxs))(*[c.handle for c in ctxs])
        ps = (C.c_void_p * len(ctxs))(*[v.ctypes.data for v in vecs])
        _check(self.lib, self.lib.qlb_stats_allreduce(cs, len(ctxs), ps, vecs[0].size))
        return vecs

    def close(self):
        if getattr(self, "handle", None):
            self.lib.qlb_ctx_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
