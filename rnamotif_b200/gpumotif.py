"""ctypes binding of libgpumotif.so (C ABI: include/gpumotif.h) -- the B200
descriptor search that stands in for rnamotif's RM_fm_init / RM_find_motif
(reference: src/rnamot.h:347-349, src/find_motif.c:109-207).

There is no CPU path here: if the CUDA library is missing or no sm_100a device
is visible, construction fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GPUMOTIF_LIB") or os.path.join(_HERE, "csrc", "libgpumotif.so")

PLAN_BYTES = 32152


class ScanStats(C.Structure):
    _fields_ = [("kernel_ms", C.c_double), ("pack_ms", C.c_double), ("h2d_ms", C.c_double),
                ("d2h_ms", C.c_double), ("sort_ms", C.c_double),
                ("n_starts", C.c_uint64), ("n_strand_nt", C.c_uint64), ("n_hits", C.c_uint64),
                ("n_launches", C.c_uint32), ("n_retries", C.c_uint32),
                ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64),
                ("filter_ms", C.c_double), ("n_survivors", C.c_uint64),
                ("n_filter_launches", C.c_uint32), ("pad_", C.c_uint32),
                ("n_score_rejected", C.c_uint64)]


class GpuMotifError(RuntimeError):
    pass


_lib = None

EXPORTS = ["gm_last_error", "gm_version", "gm_device_count", "gm_host_alloc", "gm_host_free", "gm_ctx_create", "gm_ctx_destroy",
           "gm_plan_check", "gm_plan_describe", "gm_db_upload_chars", "gm_db_upload_chars_hostpack", "gm_host_pack", "gm_db_set_device_chars", "gm_db_upload_fastn",
           "gm_db_upload_2bit", "gm_db_upload_fastn_bgzf", "gm_db_upload_fastq", "gm_db_upload_fastq_bgzf", "gm_db_get_text",
           "gm_db_records", "gm_db_get_chars", "gm_db_total_nt", "gm_hit_windows",
           "gm_scan", "gm_scan_launch", "gm_scan_finish", "gm_hits", "gm_stats",
           "gm_set_hit_capacity", "gm_set_tile", "gm_stream", "gm_prune_hits", "gm_order_hits",
           "gm_ctx_set_score", "gm_score_prescreen", "gm_rmfmt"]


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise GpuMotifError(f"{LIB_PATH} missing: run `make -C rnamotif_b200/csrc` "
                                "(or __graft_entry__.build()); there is no CPU fallback")
        L = C.CDLL(LIB_PATH)
        L.gm_last_error.restype = C.c_char_p
        L.gm_version.restype = C.c_char_p
        L.gm_ctx_create.argtypes = [C.POINTER(C.c_void_p), C.c_char_p, C.c_int]
        L.gm_ctx_destroy.argtypes = [C.c_void_p]
        L.gm_ctx_destroy.restype = None
        L.gm_plan_check.argtypes = [C.c_char_p]
        L.gm_plan_describe.argtypes = [C.c_char_p, C.c_char_p, C.c_size_t]
        L.gm_db_upload_chars.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        L.gm_db_upload_chars_hostpack.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        L.gm_host_pack.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int]
        L.gm_db_set_device_chars.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        L.gm_db_upload_fastn.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
        L.gm_db_upload_2bit.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                                        C.c_int64]
        L.gm_db_upload_fastn_bgzf.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
        L.gm_db_upload_fastq.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
        L.gm_db_upload_fastq_bgzf.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
        L.gm_db_get_text.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p]
        L.gm_db_records.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_int)]
        L.gm_hit_windows.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]
        L.gm_db_get_chars.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p]
        L.gm_db_total_nt.argtypes = [C.c_void_p]
        L.gm_db_total_nt.restype = C.c_int64
        L.gm_scan.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_int]
        L.gm_scan_launch.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_int]
        L.gm_scan_finish.argtypes = [C.c_void_p]
        L.gm_hits.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]
        L.gm_stats.argtypes = [C.c_void_p, C.POINTER(ScanStats)]
        L.gm_set_hit_capacity.argtypes = [C.c_void_p, C.c_size_t]
        L.gm_set_tile.argtypes = [C.c_void_p, C.c_int]
        L.gm_stream.argtypes = [C.c_void_p]
        L.gm_stream.restype = C.c_void_p
        L.gm_ctx_set_score.argtypes = [C.c_void_p, C.c_char_p]
        L.gm_score_prescreen.argtypes = [C.c_char_p, C.c_char_p, C.c_void_p, C.c_char_p, C.c_int]
        L.gm_prune_hits.argtypes = [C.c_char_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p, C.c_void_p]
        L.gm_order_hits.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_int, C.c_void_p]
        _lib = L
    return _lib


def prune_hits(plan: bytes, hits: np.ndarray, group=None) -> np.ndarray:
    """rmprune (src/rmprune.c) over a candidate array in enumeration order:
    boolean mask of the hits rmprune keeps.  `group[i]` = block (locus) of hit i,
    default: its record.  Host code, needs no device."""
    hits = np.ascontiguousarray(hits)
    keep = np.ones(len(hits), dtype=np.uint8)
    g = None if group is None else np.ascontiguousarray(group, dtype=np.int32)
    rc = lib().gm_prune_hits(plan, hits.ctypes.data if len(hits) else None, len(hits), hits.dtype.itemsize,
                             None if g is None else g.ctypes.data, keep.ctypes.data)
    if rc != 0:
        raise GpuMotifError("gm_prune_hits: " + _err())
    return keep.astype(bool)


def order_hits(hits: np.ndarray, name_rank, rec_off, score=None) -> np.ndarray:
    """rmfmt's ordering (src/rmfmt.c:240-262) over a candidate array: permutation
    putting the hits in the order rmfmt prints them (score descending if given,
    then name rank, strand, printed position, length).  Host code."""
    hits = np.ascontiguousarray(hits)
    nd = hits.dtype["el"].shape[0]
    nr = np.ascontiguousarray(name_rank, dtype=np.int32)
    ro = np.ascontiguousarray(rec_off, dtype=np.int64)
    sc = None if score is None else np.ascontiguousarray(score, dtype=np.float64)
    perm = np.zeros(len(hits), dtype=np.uint32)
    rc = lib().gm_order_hits(hits.ctypes.data if len(hits) else None, len(hits), hits.dtype.itemsize, nd,
                             None if sc is None else sc.ctypes.data, nr.ctypes.data, ro.ctypes.data, len(ro) - 1,
                             perm.ctypes.data)
    if rc != 0:
        raise GpuMotifError("gm_order_hits: " + _err())
    return perm


def _err():
    return lib().gm_last_error().decode("utf-8", "replace")


def plan_describe(plan: bytes) -> str:
    """What the library derives from a plan (per-search table, level-0 filter,
    look-ahead targets, probes) as text.  Host side, needs no device."""
    buf = C.create_string_buffer(1 << 16)
    if lib().gm_plan_describe(plan, buf, len(buf)) != 0:
        raise GpuMotifError("gm_plan_describe: " + _err())
    return buf.value.decode()


def plan_field(plan: bytes, idx: int) -> int:
    """int32 field `idx` of the gm_plan_t header (2 n_descr, 3 n_searches,
    4 dminlen, 5 dmaxlen, 6 windowsize, 7 strict_helices, 8 chk_both_strs)."""
    return int(np.frombuffer(plan, dtype=np.int32, count=16)[idx])


def hit_dtype(n_descr: int) -> np.dtype:
    return np.dtype([("rec", "<u4"), ("szero", "<u4"), ("seq", "<u4"), ("comp", "u1"), ("pad", "u1", 3),
                     ("lctx_off", "<i4"), ("lctx_len", "<i4"), ("rctx_off", "<i4"), ("rctx_len", "<i4"),
                     ("el", [("off", "<i4"), ("len", "<i2"), ("mpr", "i1"), ("mm", "i1")], n_descr)])


def plan_check(plan: bytes) -> str | None:
    """Host-side validation only (no device needed).  None if the plan is
    acceptable, else the reason."""
    if len(plan) != PLAN_BYTES:
        return f"plan has {len(plan)} bytes, expected {PLAN_BYTES}"
    return None if lib().gm_plan_check(plan) == 0 else _err()


class MotifSearch:
    """One descriptor on one GPU.  Mirrors the reference seam: construction is
    RM_fm_init, `find_motif` is the record loop's pair of RM_find_motif calls
    over a batch of records."""

    def __init__(self, plan: bytes, device: int = 0):
        if len(plan) != PLAN_BYTES:
            raise GpuMotifError(f"plan has {len(plan)} bytes, expected {PLAN_BYTES}")
        self._plan = bytes(plan)
        self.n_descr = plan_field(plan, 2)
        self.chk_both_strs = bool(plan_field(plan, 8))
        self._ctx = C.c_void_p()
        if lib().gm_ctx_create(C.byref(self._ctx), self._plan, device) != 0:
            self._ctx = None
            raise GpuMotifError("gm_ctx_create: " + _err())
        self._keep = None

    def close(self):
        if getattr(self, "_ctx", None):
            lib().gm_ctx_destroy(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc, what):
        if rc != 0:
            raise GpuMotifError(f"{what}: {_err()}")

    def set_score(self, score: bytes | None):
        """gm_ctx_set_score: the flattened MAIN score program (include/gpumotif_score.h);
        the sink then drops the candidates it rejects.  None switches it off."""
        self._score = bytes(score) if score is not None else None
        self._ck(lib().gm_ctx_set_score(self._ctx, self._score), "gm_ctx_set_score")

    def set_tile(self, n: int):
        self._ck(lib().gm_set_tile(self._ctx, n), "gm_set_tile")

    def set_hit_capacity(self, n: int):
        self._ck(lib().gm_set_hit_capacity(self._ctx, n), "gm_set_hit_capacity")

    def upload(self, seq, rec_off):
        """seq: uint8 array of sequence characters (host), rec_off: int64 offsets."""
        seq = np.ascontiguousarray(seq, dtype=np.uint8)
        rec_off = np.ascontiguousarray(rec_off, dtype=np.int64)
        self._keep = seq  # the upload is asynchronous: keep the buffer alive until the next scan
        self._ck(lib().gm_db_upload_chars(self._ctx, seq.ctypes.data, rec_off.ctypes.data, len(rec_off) - 1),
                 "gm_db_upload_chars")

    def upload_ptr(self, host_ptr: int, rec_off, host_pack=False):
        """gm_db_upload_chars from a raw host pointer; host_pack=True: gm_db_upload_chars_hostpack
        (4-bit codes made by a host thread team, half the bytes over PCIe)."""
        rec_off = np.ascontiguousarray(rec_off, dtype=np.int64)
        if host_pack:
            self._ck(lib().gm_db_upload_chars_hostpack(self._ctx, host_ptr, rec_off.ctypes.data, len(rec_off) - 1),
                     "gm_db_upload_chars_hostpack")
            return
        self._ck(lib().gm_db_upload_chars(self._ctx, host_ptr, rec_off.ctypes.data, len(rec_off) - 1),
                 "gm_db_upload_chars")

    def upload_hostpack(self, seq, rec_off):
        """gm_db_upload_chars_hostpack over a uint8 array (pinned or pageable)."""
        seq = np.ascontiguousarray(seq, dtype=np.uint8)
        self._keep = seq  # packing runs on until the next scan has been launched
        self.upload_ptr(seq.ctypes.data, rec_off, host_pack=True)

    def set_device_chars(self, dev_ptr: int, rec_off):
        rec_off = np.ascontiguousarray(rec_off, dtype=np.int64)
        self._ck(lib().gm_db_set_device_chars(self._ctx, dev_ptr, rec_off.ctypes.data, len(rec_off) - 1),
                 "gm_db_set_device_chars")

    def upload_fastn(self, text):
        """gm_db_upload_fastn: `text` = FASTA as it sits in the file (bytes or a uint8
        array); the reader of src/dbutil.c:42-128 runs on the device."""
        if isinstance(text, (bytes, bytearray, memoryview)):
            text = np.frombuffer(text, dtype=np.uint8)
        text = np.ascontiguousarray(text, dtype=np.uint8)
        self._keep = text
        self._ck(lib().gm_db_upload_fastn(self._ctx, text.ctypes.data, text.size), "gm_db_upload_fastn")

    def upload_fastn_ptr(self, host_ptr: int, n_bytes: int):
        self._ck(lib().gm_db_upload_fastn(self._ctx, host_ptr, n_bytes), "gm_db_upload_fastn")

    def upload_2bit(self, tb, first: int = 0, last: int | None = None):
        """gm_db_upload_2bit: records [first, last) of a parsed .2bit file (twobit.read_2bit),
        its bytes passed as they are -- a quarter of a byte per nucleotide over PCIe.  Read
        the file into pinned memory (read_2bit's `out`) for an asynchronous upload."""
        rec_off, dna_off, nblk = tb.tables(first, last)
        data = np.ascontiguousarray(tb.data, dtype=np.uint8)
        self._keep = data  # the upload is asynchronous: keep the buffer alive until the next scan
        self.upload_2bit_ptr(data.ctypes.data, data.size, dna_off, rec_off, nblk)

    def upload_2bit_ptr(self, host_ptr: int, n_bytes: int, dna_off, rec_off, nblk=None):
        """gm_db_upload_2bit from a raw host pointer: record r's packed bases at byte dna_off[r],
        nblk = flat [start, end) N ranges in rec_off coordinates."""
        dna_off = np.ascontiguousarray(dna_off, dtype=np.int64)
        rec_off = np.ascontiguousarray(rec_off, dtype=np.int64)
        nblk = np.zeros(0, dtype=np.int64) if nblk is None else np.ascontiguousarray(nblk, dtype=np.int64)
        self._ck(lib().gm_db_upload_2bit(self._ctx, host_ptr, n_bytes, dna_off.ctypes.data, rec_off.ctypes.data,
                                         len(rec_off) - 1, nblk.ctypes.data if nblk.size else None, nblk.size // 2),
                 "gm_db_upload_2bit")

    def upload_fastn_bgzf(self, buf):
        """gm_db_upload_fastn_bgzf: `buf` = a BGZF-compressed FASTA file's bytes (bytes or a uint8
        array, pinned or pageable); the members are inflated and read on the device.  Returns when
        the record table is known, so `buf` may be reused."""
        if isinstance(buf, (bytes, bytearray, memoryview)):
            buf = np.frombuffer(buf, dtype=np.uint8)
        buf = np.ascontiguousarray(buf, dtype=np.uint8)
        self.upload_fastn_bgzf_ptr(buf.ctypes.data, buf.size)

    def upload_fastn_bgzf_ptr(self, host_ptr: int, n_bytes: int):
        self._ck(lib().gm_db_upload_fastn_bgzf(self._ctx, host_ptr, n_bytes), "gm_db_upload_fastn_bgzf")

    def upload_fastq(self, text):
        """gm_db_upload_fastq: `text` = four-line FASTQ as it sits in the file (bytes or a uint8
        array); the reads are taken out and the format is checked on the device."""
        if isinstance(text, (bytes, bytearray, memoryview)):
            text = np.frombuffer(text, dtype=np.uint8)
        text = np.ascontiguousarray(text, dtype=np.uint8)
        self._keep = text
        self.upload_fastq_ptr(text.ctypes.data, text.size)

    def upload_fastq_ptr(self, host_ptr: int, n_bytes: int):
        self._ck(lib().gm_db_upload_fastq(self._ctx, host_ptr, n_bytes), "gm_db_upload_fastq")

    def upload_fastq_bgzf(self, buf):
        """gm_db_upload_fastq_bgzf: `buf` = a BGZF-compressed FASTQ file's bytes (bytes or a uint8
        array, pinned or pageable); the members are inflated and read on the device.  Returns when
        the record table is known, so `buf` may be reused."""
        if isinstance(buf, (bytes, bytearray, memoryview)):
            buf = np.frombuffer(buf, dtype=np.uint8)
        buf = np.ascontiguousarray(buf, dtype=np.uint8)
        self.upload_fastq_bgzf_ptr(buf.ctypes.data, buf.size)

    def upload_fastq_bgzf_ptr(self, host_ptr: int, n_bytes: int):
        self._ck(lib().gm_db_upload_fastq_bgzf(self._ctx, host_ptr, n_bytes), "gm_db_upload_fastq_bgzf")

    def get_text(self, off: int = 0, n: int | None = None) -> bytes:
        """gm_db_get_text: bytes [off, off + n) of the FASTA or FASTQ text of the last upload_fastn,
        upload_fastn_bgzf, upload_fastq or upload_fastq_bgzf (n = None: to the end)."""
        if n is None:
            _, hdr = self.records()
            n = (int(hdr[-1]) if hdr is not None else 0) - off
        out = np.empty(max(n, 1), dtype=np.uint8)
        self._ck(lib().gm_db_get_text(self._ctx, off, n, out.ctypes.data), "gm_db_get_text")
        return out[:n].tobytes()

    def records(self):
        """(rec_off, hdr_off) of the uploaded batch; hdr_off is None unless it came
        through upload_fastn, upload_fastn_bgzf, upload_fastq or upload_fastq_bgzf."""
        ro, ho, n = C.c_void_p(), C.c_void_p(), C.c_int()
        self._ck(lib().gm_db_records(self._ctx, C.byref(ro), C.byref(ho), C.byref(n)), "gm_db_records")
        m = n.value + 1
        rec = np.frombuffer((C.c_int64 * m).from_address(ro.value), dtype=np.int64).copy()
        hdr = np.frombuffer((C.c_int64 * m).from_address(ho.value), dtype=np.int64).copy() if ho.value else None
        return rec, hdr

    def get_chars(self, off: int = 0, n: int | None = None):
        """gm_db_get_chars: the uploaded characters (lower case, u -> t) as a uint8 array."""
        if n is None:
            n = self.total_nt - off
        out = np.empty(max(n, 0), dtype=np.uint8)
        self._ck(lib().gm_db_get_chars(self._ctx, off, n, out.ctypes.data), "gm_db_get_chars")
        return out

    def hit_windows(self, lead: int = 0, trail: int = 0):
        """gm_hit_windows: uint8 array [n_hits, stride]; row i = the searched strand from
        offset szero_i - lead on, as fm_sbuf would hold it."""
        p, st = C.c_void_p(), C.c_size_t()
        self._ck(lib().gm_hit_windows(self._ctx, lead, trail, C.byref(p), C.byref(st)), "gm_hit_windows")
        n = C.c_size_t()
        self._ck(lib().gm_hits(self._ctx, None, C.byref(n), None), "gm_hits")
        if n.value == 0:
            return np.zeros((0, st.value), dtype=np.uint8)
        buf = (C.c_uint8 * (n.value * st.value)).from_address(p.value)
        return np.frombuffer(buf, dtype=np.uint8).reshape(n.value, st.value).copy()

    @property
    def total_nt(self) -> int:
        return int(lib().gm_db_total_nt(self._ctx))

    def scan(self, g_begin: int = 0, g_end: int | None = None, strands: int | None = None, copy: bool = True):
        """gm_scan.  Returns the candidates (a copy; with copy=False a view of the
        library's host buffer that is valid until the next scan)."""
        if g_end is None:
            g_end = self.total_nt
        if strands is None:
            strands = 2 if self.chk_both_strs else 1
        self._ck(lib().gm_scan(self._ctx, g_begin, g_end, strands), "gm_scan")
        return self.hits(copy)

    def scan_launch(self, g_begin: int = 0, g_end: int | None = None, strands: int | None = None):
        if g_end is None:
            g_end = self.total_nt
        if strands is None:
            strands = 2 if self.chk_both_strs else 1
        self._ck(lib().gm_scan_launch(self._ctx, g_begin, g_end, strands), "gm_scan_launch")

    def scan_finish(self):
        self._ck(lib().gm_scan_finish(self._ctx), "gm_scan_finish")

    def hits(self, copy: bool = True):
        p, n, st = C.c_void_p(), C.c_size_t(), C.c_size_t()
        self._ck(lib().gm_hits(self._ctx, C.byref(p), C.byref(n), C.byref(st)), "gm_hits")
        dt = hit_dtype(self.n_descr)
        assert dt.itemsize == st.value
        if n.value == 0:
            return np.zeros(0, dtype=dt)
        buf = (C.c_uint8 * (n.value * st.value)).from_address(p.value)
        a = np.frombuffer(buf, dtype=dt)
        return a.copy() if copy else a

    def stats(self) -> ScanStats:
        s = ScanStats()
        self._ck(lib().gm_stats(self._ctx, C.byref(s)), "gm_stats")
        return s

    @property
    def stream(self) -> int:
        return int(lib().gm_stream(self._ctx) or 0)

    # reference-named entry: both strands of every record of a batch
    def find_motif(self, seq, rec_off):
        self.upload(seq, rec_off)
        return self.scan()


def host_pack(seq, n_threads=0):
    """gm_host_pack: uint8 characters -> 4-bit codes, two per byte (host code, no device)."""
    seq = np.ascontiguousarray(seq, dtype=np.uint8)
    out = np.zeros((seq.size + 1) // 2, dtype=np.uint8)
    if lib().gm_host_pack(seq.ctypes.data, seq.size, out.ctypes.data, n_threads) != 0:
        raise GpuMotifError("gm_host_pack failed")
    return out
