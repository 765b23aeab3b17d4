"""ctypes access to oracle/libgmoracle.so (the plain-C restatement of the
reference search).  TEST INFRASTRUCTURE: imported only by tests/, by
__graft_entry__.smoke() and by bench.py's cpu_baseline / --impl reference legs.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_DIR = _HERE
HDR_BYTES = 32   # sizeof(gm_hit_hdr_t)
EL_BYTES = 8     # sizeof(gm_hit_el_t)


class Stats(C.Structure):
    _fields_ = [("n_starts", C.c_uint64), ("n_pair_evals", C.c_uint64),
                ("n_chk_seq", C.c_uint64), ("n_regex_steps", C.c_uint64),
                ("n_candidates", C.c_uint64)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        path = os.path.join(ORACLE_DIR, "libgmoracle.so")
        if not os.path.exists(path):
            raise RuntimeError("oracle/libgmoracle.so missing: run `make -C oracle port`")
        _lib = C.CDLL(path)
        _lib.gmo_scan_db.restype = C.c_int64
        _lib.gmo_scan_db.argtypes = [C.c_char_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                     C.c_void_p, C.c_size_t, C.POINTER(Stats)]
        _lib.gmo_scan_db_range.restype = C.c_int64
        _lib.gmo_scan_db_range.argtypes = [C.c_char_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_int64,
                                           C.c_void_p, C.c_size_t, C.POINTER(Stats)]
        _lib.gmo_hit_stride.restype = C.c_size_t
        _lib.gmo_hit_stride.argtypes = [C.c_char_p]
    return _lib


def plan_n_descr(plan: bytes) -> int:
    return int(np.frombuffer(plan, dtype=np.int32, count=3)[2])


def hit_dtype(n_descr: int) -> np.dtype:
    return np.dtype([("rec", "<u4"), ("szero", "<u4"), ("seq", "<u4"), ("comp", "u1"), ("pad", "u1", 3),
                     ("lctx_off", "<i4"), ("lctx_len", "<i4"), ("rctx_off", "<i4"), ("rctx_len", "<i4"),
                     ("el", [("off", "<i4"), ("len", "<i2"), ("mpr", "i1"), ("mm", "i1")], n_descr)])


def scan_db(plan: bytes, seq: np.ndarray, rec_off: np.ndarray, both: bool, cap_hits: int = 1 << 20,
            f_range: tuple[int, int] | None = None):
    """Run the oracle over a database.  Returns (hits structured array in the
    reference's enumeration order, Stats).  f_range = (lo, hi): only the starts whose
    5' end lies at a forward position in [lo, hi) of each record (a complementary-strand
    start owns forward position slen - 1 - szero)."""
    L = lib()
    n_descr = plan_n_descr(plan)
    dt = hit_dtype(n_descr)
    assert dt.itemsize == L.gmo_hit_stride(plan), (dt.itemsize, L.gmo_hit_stride(plan))
    seq = np.ascontiguousarray(seq, dtype=np.uint8)
    rec_off = np.ascontiguousarray(rec_off, dtype=np.int64)
    st = Stats()
    while True:
        out = np.zeros(cap_hits, dtype=dt)
        if f_range is None:
            n = L.gmo_scan_db(plan, seq.ctypes.data, rec_off.ctypes.data, len(rec_off) - 1, int(both),
                              out.ctypes.data, out.nbytes, C.byref(st))
        else:
            n = L.gmo_scan_db_range(plan, seq.ctypes.data, rec_off.ctypes.data, len(rec_off) - 1, int(both),
                                    int(f_range[0]), int(f_range[1]), out.ctypes.data, out.nbytes, C.byref(st))
        if n < 0:
            raise RuntimeError("oracle scan failed (bad plan?)")
        if n <= cap_hits:
            return out[:n], st
        cap_hits = int(n)
        st = Stats()
