"""Searches and read-backs past 2^31 and 2^32 nucleotides, and on one record at the length cap.

Global positions are int64 in the library and positions inside a strand are int, so a record may
hold up to 0x7ffffff0 nucleotides (check_records, gpumotif.cu) and a batch is bounded by device
memory only.  A 32-bit truncation at a boundary between the two, or an int sum that passes 2^31
near the end of a record at the cap, shows only on inputs this big.

The reference is the oracle on pieces.  A candidate whose 5' end lies at strand offset szero reads
its window [szero, szero + W) (W = min(dmaxlen, windowsize)), up to the longest context on either
side of it, one more position for the strict-helix checks, and the record end wherever that clips
the window.  So the oracle over a piece [P0, P1) of a record, taken as a record of its own, gives
exactly the full record's candidates whose 5' end lies at a forward position in [lo, hi), provided
lo - P0 and P1 - hi are at least W + 2 maxctx + 2 or the piece reaches the record's end on that
side.  piece_reference() searches only the piece's starts in [lo, hi) (oracle_port.scan_db's
f_range) and shifts the candidates back into the record's coordinates; test_piece_reference pins
that down on the CPU against whole-record oracle runs.

Every probe region holds the golden database (synth.golden_db) glued into one record and cycled;
the bulk between the regions is random and is never read on the host.  Every check compares the
device with piece_reference, with the characters put into the regions, or with the host's score
pre-screen, and every probe must give candidates for every plan.
"""
import ctypes as C

import numpy as np
import pytest

from rnamotif_b200 import gpumotif, synth
from oracle import oracle_port
import helpers

CAP = 0x7ffffff0          # the longest record the uploads take
PROBE = 1 << 18           # nucleotides per probe scan: more than the golden record, so every probe holds all of it
MARGIN = 1 << 14          # known characters beyond a probe: > W + 2 maxctx + 2 and > the hit windows' reach
LEAD, TRAIL = 40, 3000    # hit windows: TRAIL runs past the record ends at the end probes

ELOOP_PROBE = 2048        # descr.eloop's probes: its 6 000-nt windows make the oracle take ~1 ms a start

CTX_PLAN = "score.1.strict+ctx4000"  # at the cap only
PLANS = ["trna", "pk1", "qu+tr", "ire", "score.1", "descr.eloop", "trna@fused", "trna@split"]


def load_plan(name):
    """A golden plan, or score.1.strict with both contexts 4 000 nt long (int32 fields 116 and 120 of
    gm_plan_t: 14 header ints, searches[100], then lctx and rctx as present, minlen, maxlen, regex)."""
    if name == "descr.eloop":
        return helpers.load_extra_plan(name)
    if name != CTX_PLAN:
        return helpers.load_plan(name)
    plan = bytearray(helpers.load_plan("score.1.strict"))
    f = np.frombuffer(plan, dtype=np.int32)
    assert f[114] == 1 and f[118] == 1, "score.1.strict has both contexts"
    f[116] = f[120] = 4000
    return bytes(plan)


def margin(plan):
    f = np.frombuffer(plan, dtype=np.int32, count=122)
    w = min(int(f[5]), int(f[6]))
    maxctx = max(int(f[116]) if f[114] else 0, int(f[120]) if f[118] else 0)
    return w + 2 * maxctx + 2


# mk_rcmp (src/rnamot.c:193-216) over characters as fm_sbuf holds them
_RCMP = np.full(256, ord("n"), dtype=np.uint8)
for _a, _b in zip(b"acgt", b"tgca"):
    _RCMP[_a] = _b
_RCMP[0] = 0
# what a .2bit file keeps of a letter (twobit.write_2bit, twobit.to_chars): acgt in lower case, u as t, the rest n
_AS_2BIT = np.full(256, ord("n"), dtype=np.uint8)
for _ch in b"acgt":
    _AS_2BIT[_ch] = _AS_2BIT[_ch - 32] = _ch
_AS_2BIT[ord("u")] = _AS_2BIT[ord("U")] = ord("t")
# what fm_sbuf holds of a letter (src/dbutil.c:105-111): lower case, u as t
_FOLD = np.arange(256, dtype=np.uint8) | 0x20
_FOLD[ord("u")] = _FOLD[ord("U")] = ord("t")
_FOLD[0] = 0
_CODE2 = np.zeros(256, dtype=np.uint8)  # t and n: 0
for _ch, _c in zip(b"cag", (1, 2, 3)):
    _CODE2[_ch] = _c


def golden_record():
    """synth.golden_db() glued into one record."""
    return synth.golden_db()[1]


def piece_reference(plan, chars, rec_start, rec_end, P0, P1, lo, hi, rec=0):
    """The oracle's candidates of record `rec` = [rec_start, rec_end) (batch coordinates) whose 5' end
    lies at a forward position in [lo, hi), in enumeration order, from the oracle over the piece
    chars = the record's characters [P0, P1) alone.  A comp-strand start owns forward position
    slen - 1 - szero (gm_scan's range contract)."""
    m = margin(plan)
    assert rec_start <= P0 <= lo <= hi <= P1 <= rec_end and len(chars) == P1 - P0
    assert P0 == rec_start or lo - P0 >= m, f"piece starts {lo - P0} nt before the range, needs {m}"
    assert P1 == rec_end or P1 - hi >= m, f"piece ends {P1 - hi} nt after the range, needs {m}"
    both = bool(gpumotif.plan_field(plan, 8))
    h, _ = oracle_port.scan_db(plan, chars, np.array([0, P1 - P0], dtype=np.int64), both, f_range=(lo - P0, hi - P0))
    h = h.copy()
    fwd = h["comp"] == 0
    shift = np.where(fwd, P0 - rec_start, rec_end - P1).astype(np.int64)
    h["szero"] = (h["szero"].astype(np.int64) + shift).astype(np.uint32)
    off = h["el"]["off"]
    off += shift[:, None].astype(np.int32)
    h["el"]["off"] = off
    for f in ("lctx_off", "rctx_off"):
        h[f] = np.where(h[f] >= 0, h[f] + shift, h[f]).astype(np.int32)
    h["rec"] = rec
    return h


def _filter(hits, rec_off, lo, hi):
    """The candidates of a batch-wide stream whose 5' end lies at a forward position in [lo, hi)."""
    rs = rec_off[hits["rec"].astype(np.int64)]
    slen = rec_off[hits["rec"].astype(np.int64) + 1] - rs
    sz = hits["szero"].astype(np.int64)
    pos = rs + np.where(hits["comp"] == 0, sz, slen - 1 - sz)
    return hits[(pos >= lo) & (pos < hi)]


# ------------------------------------------------------------------ CPU: the reduction itself

CPU_PLANS = helpers.golden_names() + ["extra.ctx_seq+ctx4000", CTX_PLAN]


def _cpu_plan(name):
    if name == "extra.ctx_seq+ctx4000":
        plan = bytearray(helpers.load_plan("extra.ctx_seq"))
        f = np.frombuffer(plan, dtype=np.int32)
        f[116] = f[120] = 4000
        return bytes(plan)
    return load_plan(name)


@pytest.mark.parametrize("name", CPU_PLANS)
def test_piece_reference(name):
    """Pieces cut mid-record, at the record's start and at its end give the whole record's candidates
    (the oracle over the whole record, every start, kept where the 5' end lies in the range)."""
    plan = _cpu_plan(name)
    assert gpumotif.plan_check(plan) is None
    seq = golden_record()
    n = len(seq)
    both = bool(gpumotif.plan_field(plan, 8))
    full, _ = oracle_port.scan_db(plan, seq, np.array([0, n], dtype=np.int64), both)
    rec_off = np.array([0, n], dtype=np.int64)
    m = margin(plan)
    for lo, hi, P0, P1 in [(n // 4, 3 * n // 4, n // 4 - m, 3 * n // 4 + m),      # mid-record
                           (0, n // 3, 0, n // 3 + m),                            # at the record start
                           (2 * n // 3, n, 2 * n // 3 - m, n)]:                   # at the record end
        P0, P1 = max(P0, 0), min(P1, n)
        got = piece_reference(plan, seq[P0:P1], 0, n, P0, P1, lo, hi)
        helpers.assert_same_hits(got, _filter(full, rec_off, lo, hi), f"{name}: piece [{P0}, {P1}) for [{lo}, {hi})")


# ------------------------------------------------------------------ GPU: the batches

class TwoBitBatch:
    """A 2-bit batch in host memory: records of `sizes` nucleotides, each on bytes of its own, random
    bases except in `regions` -- [g0, g1) ranges in batch coordinates, each inside one record -- which
    hold the golden record cycled (as a .2bit file keeps it), with N blocks where that has other
    letters and over the `n_runs` ranges.  chars(a, b) are the characters the device must give back
    over a range inside the regions."""

    def __init__(self, sizes, regions, n_runs=(), seed=0, shifts=None):
        sizes = np.asarray(sizes, dtype=np.int64)
        self.rec_off = np.zeros(len(sizes) + 1, dtype=np.int64)
        np.cumsum(sizes, out=self.rec_off[1:])
        nb = (sizes + 3) // 4
        self.dna_off = np.zeros(len(sizes), dtype=np.int64)
        np.cumsum(nb[:-1], out=self.dna_off[1:])
        rng = np.random.default_rng(seed)
        self.data = rng.integers(0, 256, size=int(nb.sum()) + 8, dtype=np.uint8)
        gold = _AS_2BIT[golden_record()]
        self.starts, self.parts, nblk = [], [], []
        for i, (g0, g1) in enumerate(sorted(regions)):
            r = int(np.searchsorted(self.rec_off, g0, side="right")) - 1
            rs, re = int(self.rec_off[r]), int(self.rec_off[r + 1])
            assert rs <= g0 < g1 <= re
            g0 = rs + (g0 - rs) // 4 * 4                        # whole bytes of the record
            g1 = min(re, rs + (g1 - rs + 3) // 4 * 4)
            shift = 7919 * i if shifts is None else shifts[i]  # where in the golden record the region starts
            s = gold[(np.arange(g1 - g0) + shift) % len(gold)]
            for a, b in n_runs:
                if a < g1 and b > g0:
                    s[max(a, g0) - g0:min(b, g1) - g0] = ord("n")
            c = _CODE2[s]
            c = np.concatenate([c, np.zeros(-len(c) % 4, dtype=np.uint8)]).reshape(-1, 4)
            b0 = int(self.dna_off[r]) + (g0 - rs) // 4
            self.data[b0:b0 + len(c)] = (c[:, 0] << 6) | (c[:, 1] << 4) | (c[:, 2] << 2) | c[:, 3]
            d = np.diff(np.concatenate([[0], (s == ord("n")).astype(np.int8), [0]]))
            for a, b in zip(np.nonzero(d == 1)[0], np.nonzero(d == -1)[0]):
                nblk += [g0 + int(a), g0 + int(b)]
            self.starts.append(g0)
            self.parts.append(s)
        self.nblk = np.array(nblk, dtype=np.int64)
        self.ends = np.array([a + len(p) for a, p in zip(self.starts, self.parts)], dtype=np.int64)
        self.starts = np.array(self.starts, dtype=np.int64)
        self.total_nt = int(self.rec_off[-1])
        self.fold = np.arange(256, dtype=np.uint8)  # the regions hold decoded characters already

    def chars_at(self, g):
        g = np.asarray(g, dtype=np.int64)
        k = np.searchsorted(self.starts, g, side="right") - 1
        assert (k >= 0).all() and (g < self.ends[np.maximum(k, 0)]).all(), "a position outside the known regions"
        out = np.empty(len(g), dtype=np.uint8)
        for j in np.unique(k):
            sel = k == j
            out[sel] = self.parts[j][g[sel] - self.starts[j]]
        return out

    def chars(self, a, b):
        return self.chars_at(np.arange(a, b, dtype=np.int64))

    def upload(self, ms, rec_off=None, dna_off=None):
        ms.upload_2bit_ptr(self.data.ctypes.data, self.data.size, self.dna_off if dna_off is None else dna_off,
                           self.rec_off if rec_off is None else rec_off, self.nblk)


def _record(rec_off, lo, hi):
    r = int(np.searchsorted(rec_off, lo, side="right")) - 1
    assert rec_off[r] <= lo < hi <= rec_off[r + 1], "a probe lies inside one record"
    return r, int(rec_off[r]), int(rec_off[r + 1])


def _need_device(n_bytes):
    import torch
    free, _ = torch.cuda.mem_get_info()
    if free < n_bytes:
        pytest.skip(f"needs {n_bytes / 2**30:.1f} GiB of free device memory, {free / 2**30:.1f} GiB free")


_REF = {}


def probe_reference(key, name, plan, batch, rec_off, lo, hi):
    """piece_reference for probe [lo, hi) of `batch` under the record table rec_off (cached per key)."""
    k = (key, name, lo, hi)
    if k not in _REF:
        r, rs, re = _record(rec_off, lo, hi)
        P0, P1 = max(rs, lo - MARGIN), min(re, hi + MARGIN)
        _REF[k] = piece_reference(plan, batch.chars(P0, P1), rs, re, P0, P1, lo, hi, rec=r)
    return _REF[k]


def expected_starts(plan, rec_off, lo, hi, strands):
    """(start, strand) pairs a scan of [lo, hi) searches: szero in [0, slen - dminlen] on each strand."""
    _, rs, re = _record(rec_off, lo, hi)
    dm = gpumotif.plan_field(plan, 4)
    n = max(0, min(hi, re - dm + 1) - max(lo, rs))
    if strands > 1:
        n += max(0, min(hi, re) - max(lo, rs + dm - 1))
    return n


def expected_windows(hits, batch, rec_off, lead, stride):
    out = np.zeros((len(hits), stride), dtype=np.uint8)
    for i in range(len(hits)):
        r = int(hits["rec"][i])
        rs, slen = int(rec_off[r]), int(rec_off[r + 1] - rec_off[r])
        p = int(hits["szero"][i]) - lead + np.arange(stride, dtype=np.int64)
        ok = (p >= 0) & (p < slen)
        if hits["comp"][i]:
            out[i, ok] = _RCMP[batch.fold[batch.chars_at(rs + slen - 1 - p[ok])]]
        else:
            out[i, ok] = batch.fold[batch.chars_at(rs + p[ok])]
    return out


def prescreen(plan, score, hits, batch, rec_off, lo, hi):
    """gm_score_prescreen on the host over each candidate of probe [lo, hi): the full record's slen, and
    sbuf = the piece's strand characters less the piece's strand offset (gm_hit_windows' trick)."""
    L = gpumotif.lib()
    _, rs, re = _record(rec_off, lo, hi)
    P0, P1 = max(rs, lo - MARGIN), min(re, hi + MARGIN)
    fwd = batch.chars(P0, P1)
    strands = [np.ascontiguousarray(fwd), np.ascontiguousarray(_RCMP[fwd[::-1]])]
    base = [P0 - rs, re - P1]
    rej = np.zeros(len(hits), dtype=bool)
    for i in range(len(hits)):
        c = int(hits["comp"][i])
        rej[i] = bool(L.gm_score_prescreen(plan, score, hits[i:i + 1].ctypes.data,
                                           C.c_char_p(strands[c].ctypes.data - base[c]), re - rs))
    return rej


def check_probes(ms, name, plan, batch, key, probes, rec_off=None, windows=True):
    """Range scans of every probe against piece_reference, with their start counts and hit windows."""
    rec_off = batch.rec_off if rec_off is None else rec_off
    strands = 2 if gpumotif.plan_field(plan, 8) else 1
    got = {}
    for lo, hi in probes:
        what = f"{name}: [{lo}, {hi})"
        ref = probe_reference(key, name, plan, batch, rec_off, lo, hi)
        hits = ms.scan(lo, hi)
        helpers.assert_same_hits(hits, ref, what)
        assert len(ref) > 0, f"{what}: the probe gives no candidates"
        assert ms.stats().n_starts == expected_starts(plan, rec_off, lo, hi, strands), what
        if windows:
            w = ms.hit_windows(LEAD, TRAIL)
            assert w.shape[0] == len(hits) and w.shape[1] >= LEAD + TRAIL + 1
            exp = expected_windows(hits, batch, rec_off, LEAD, w.shape[1])
            bad = np.nonzero((w != exp).any(axis=1))[0]
            assert bad.size == 0, f"{what}: hit window {bad[:1]} differs from the characters put there"
        got[(lo, hi)] = hits
    return got


def check_score(plan, batch, key, probes, rec_off=None):
    """score.1 with its score program: the kept candidates are the piece reference's less the ones the
    host pre-screen rejects, and n_score_rejected counts the difference."""
    rec_off = batch.rec_off if rec_off is None else rec_off
    score = helpers.load_score("score.1")
    ms = gpumotif.MotifSearch(plan)
    ms.set_score(score)
    batch.upload(ms, rec_off)
    for lo, hi in probes:
        ref = probe_reference(key, "score.1", plan, batch, rec_off, lo, hi)
        rej = prescreen(plan, score, ref, batch, rec_off, lo, hi)
        kept = ms.scan(lo, hi)
        helpers.assert_same_hits(kept, ref[~rej], f"score.1 pre-screen: [{lo}, {hi})")
        assert ms.stats().n_score_rejected == int(rej.sum())
    ms.close()


def _probes_around(places, rec_off, n=PROBE):
    """A probe of n nucleotides on each side of each place that lies inside a record."""
    out = []
    for c in places:
        for lo, hi in ((c - n, c), (c, c + n)):
            r = int(np.searchsorted(rec_off, lo, side="right")) - 1
            if 0 <= lo and hi <= rec_off[-1] and rec_off[r] <= lo and hi <= rec_off[r + 1]:
                out.append((lo, hi))
    return out


def _regions(probes, rec_off):
    """The probes widened by MARGIN and cut at record ends."""
    out = []
    for lo, hi in probes:
        r, rs, re = _record(rec_off, lo, hi)
        out.append((max(rs, lo - MARGIN), min(re, hi + MARGIN)))
    out.sort()
    merged = []
    for a, b in out:
        if merged and a <= merged[-1][1] and _record(rec_off, a, b)[0] == _record(rec_off, *merged[-1])[0]:
            merged[-1] = (merged[-1][0], max(b, merged[-1][1]))
        else:
            merged.append((a, b))
    return merged


# ------------------------------------------------------------------ leg A: a 2-bit genome past 2^32

G31, G32 = 1 << 31, 1 << 32
# R1 ends exactly at 2^31; R1 + R2 joined (second record table) span it; R3 spans 2^32 with N blocks
# across it; R4 starts at an odd position past 2^32; R5 ends at total_nt
A_SIZES = [1_200_000_000, G31 - 1_200_000_000, 1_100_000_000, G32 + 50_000_001 - (G31 + 1_100_000_000),
           30_000_000, 25_032_703]
A_NRUNS = [(G32 - 700, G32 + 900), (G32 + 3001, G32 + 3050)]


@pytest.fixture(scope="module")
def leg_a():
    rec_off = np.concatenate([[0], np.cumsum(A_SIZES)]).astype(np.int64)
    places = [G31, G32, int(rec_off[4]), int(rec_off[-1])]
    probes = _probes_around(places, rec_off)
    batch = TwoBitBatch(A_SIZES, _regions(probes, rec_off), A_NRUNS, seed=1)
    assert batch.total_nt > G32 + 100_000_000 and rec_off[4] % 2 == 1 and rec_off[2] == G31
    return batch, probes, places


def _open(name, monkeypatch):
    """name = plan[@path]: a context for the plan, on the fused or worklist path if one is named."""
    base, _, path = name.partition("@")
    if path:
        monkeypatch.setenv("GPUMOTIF_PATH", path)
    else:
        monkeypatch.delenv("GPUMOTIF_PATH", raising=False)
    plan = load_plan(base)
    return base, plan, gpumotif.MotifSearch(plan)


def _plan_probes(base, places, rec_off):
    """The probes a plan is checked on: descr.eloop's are the ELOOP_PROBE nucleotides next to each place."""
    return _probes_around(places, rec_off, ELOOP_PROBE if base == "descr.eloop" else PROBE)


@pytest.mark.gpu
@pytest.mark.parametrize("name", PLANS)
def test_2bit_past_2_32(name, leg_a, monkeypatch):
    _need_device(4 << 30)
    batch, _, places = leg_a
    base, plan, ms = _open(name, monkeypatch)
    probes = _plan_probes(base, places, batch.rec_off)
    try:
        batch.upload(ms)
        if name == "score.1":
            # the first scan of the upload streams the chunks in: the whole batch, once
            whole = ms.scan()
        got = check_probes(ms, base, plan, batch, "A", probes)
        if name == "score.1":
            for (lo, hi), hits in got.items():
                helpers.assert_same_hits(_filter(whole, batch.rec_off, lo, hi), hits, f"whole-batch scan in [{lo}, {hi})")
        # characters across 2^32 (an N block straddles it) and at R4's odd start
        for a, n in ((G32 - 1000, 2500), (int(batch.rec_off[4]) - 3, 11), (batch.total_nt - 7, 7)):
            assert ms.get_chars(a, n).tobytes() == batch.chars(a, a + n).tobytes(), f"get_chars({a}, {n})"
        # R1 and R2 as one record across 2^31: the same bytes, another record table
        if base in ("trna", "score.1"):
            joined = np.delete(batch.rec_off, 2)
            batch.upload(ms, joined, np.delete(batch.dna_off, 2))
            check_probes(ms, base, plan, batch, "A-joined", [(G31 - PROBE, G31 + PROBE)], joined)
    finally:
        ms.close()


@pytest.mark.gpu
def test_2bit_past_2_32_score_prescreen(leg_a):
    _need_device(4 << 30)
    batch, probes, _ = leg_a
    check_score(load_plan("score.1"), batch, "A", probes)


@pytest.mark.gpu
def test_assemble_past_2_32(leg_a):
    """gm_db_assemble with blocks past 2^31 and 2^32: across 2^32 inside R3, 1-nt blocks, minus records."""
    _need_device(4 << 30)
    batch, _, _ = leg_a
    r4 = int(batch.rec_off[4])
    blk = np.array([G31 + 1000, G31 + 4000,          # past 2^31, R2
                    G32 - 90000, G32 + 90001,        # across 2^32 inside R3 (and its N blocks)
                    G32 + 11, G32 + 12,              # one nucleotide
                    r4, r4 + 1,                      # R4's first nucleotide (odd position)
                    r4 + 5, r4 + 3333,
                    batch.total_nt - 2000, batch.total_nt], dtype=np.int64).reshape(-1, 2)
    recs = [[0, 1], [1, 2, 3], [4], [5, 1], [2], [3, 4]]
    strand = np.array([0, 1, 0, 1, 1, 0], dtype=np.uint8)
    flat = np.concatenate([blk[k] for rec in recs for k in rec])
    rec_blk = np.concatenate([[0], np.cumsum([len(rec) for rec in recs])]).astype(np.int64)
    parts = []
    for r, rec in enumerate(recs):
        s = np.concatenate([batch.chars(*blk[k]) for k in rec])
        parts.append(_RCMP[s[::-1]] if strand[r] else s)
    chars = np.concatenate(parts)
    rec_off = np.concatenate([[0], np.cumsum([len(p) for p in parts])]).astype(np.int64)
    for name in ("trna", "score.1"):
        plan = load_plan(name)
        ms = gpumotif.MotifSearch(plan)
        batch.upload(ms)
        ms.assemble(flat, rec_blk, strand)
        assert ms.get_chars().tobytes() == chars.tobytes()
        ref, _ = oracle_port.scan_db(plan, chars, rec_off, bool(gpumotif.plan_field(plan, 8)))
        helpers.assert_same_hits(ms.scan(), ref, f"{name}: assembled from blocks past 2^31 and 2^32")
        assert len(ref) > 0, f"{name}: the assembled batch gives no candidates"
        ms.close()


# ------------------------------------------------------------------ leg B: characters on the device past 2^31

class DeviceCharBatch(TwoBitBatch):
    """Characters in device memory (a torch tensor handed over with gm_db_set_device_chars): random acgt,
    except in `regions`, which hold the golden record's letters as they are -- IUPAC codes, upper case
    and u included."""

    def __init__(self, sizes, regions):
        import torch
        sizes = np.asarray(sizes, dtype=np.int64)
        self.rec_off = np.zeros(len(sizes) + 1, dtype=np.int64)
        np.cumsum(sizes, out=self.rec_off[1:])
        self.total_nt = int(self.rec_off[-1])
        self.fold = _FOLD
        dev = torch.device("cuda", 0)
        self.seq = torch.empty(self.total_nt, dtype=torch.uint8, device=dev)
        lut = torch.tensor(list(b"acgt"), dtype=torch.uint8, device=dev)
        gen = torch.Generator(device=dev).manual_seed(3)
        step = 1 << 26
        for a in range(0, self.total_nt, step):
            k = min(step, self.total_nt - a)
            self.seq[a:a + k] = lut[torch.randint(0, 4, (k,), device=dev, generator=gen)]
        gold = golden_record()
        self.starts, self.parts = [], []
        for i, (g0, g1) in enumerate(sorted(regions)):
            s = gold[(np.arange(g1 - g0) + 7919 * i) % len(gold)]
            self.seq[g0:g1] = torch.from_numpy(s).to(dev)
            self.starts.append(g0)
            self.parts.append(s)
        torch.cuda.synchronize()
        self.ends = np.array([a + len(p) for a, p in zip(self.starts, self.parts)], dtype=np.int64)
        self.starts = np.array(self.starts, dtype=np.int64)

    def upload(self, ms, rec_off=None):
        ms.set_device_chars(self.seq.data_ptr(), self.rec_off if rec_off is None else rec_off)


# R1 spans 2^31; the batch ends 16 Mi past it
B_SIZES = [1_000_000_000, G31 + (16 << 20) - 1_000_000_000]


@pytest.mark.gpu
def test_device_chars_past_2_31(monkeypatch):
    _need_device(5 << 30)
    rec_off = np.concatenate([[0], np.cumsum(B_SIZES)]).astype(np.int64)
    places = [G31, int(rec_off[-1])]
    batch = DeviceCharBatch(B_SIZES, _regions(_probes_around(places, rec_off), rec_off))
    gold = golden_record()
    assert (gold != _FOLD[gold]).any() and (gold == ord("u")).any(), "the regions hold upper case and u"
    try:
        for name in PLANS:
            base, plan, ms = _open(name, monkeypatch)
            try:
                batch.upload(ms)
                check_probes(ms, base, plan, batch, "B", _plan_probes(base, places, rec_off))
                for a, n in ((G31 - 1000, 2500), (batch.total_nt - 9, 9)):
                    assert ms.get_chars(a, n).tobytes() == _FOLD[batch.chars(a, a + n)].tobytes(), f"get_chars({a}, {n})"
            finally:
                ms.close()
    finally:
        del batch.seq


# ------------------------------------------------------------------ leg C: one record at the cap

def _cap_shifts(regions):
    """Where leg C's two regions start in the golden record: so that a forward candidate of CTX_PLAN has
    its right context start 2 000 nt before the record end, and a complementary-strand one 2 000 nt after
    the record start (its right context runs towards the record start).  Both contexts are clipped there."""
    gold = _AS_2BIT[golden_record()]
    n = len(gold)
    h, _ = oracle_port.scan_db(load_plan(CTX_PLAN), gold, np.array([0, n], dtype=np.int64), True)
    h = h[(h["rctx_off"] > 8000) & (h["rctx_off"] < n - 8000)]  # away from the seam of the cycle
    r_f = int(h["rctx_off"][h["comp"] == 0][0])
    r_c = int(h["rctx_off"][h["comp"] == 1][0])
    (a0, a1), (b0, b1) = regions
    assert a0 == 0 and b1 == CAP
    return [(n - 1 - r_c - 2000) % n, (r_f + 2000 - (b1 - b0)) % n]


@pytest.fixture(scope="module")
def leg_c():
    rec_off = np.array([0, CAP], dtype=np.int64)
    probes = [(0, PROBE), (CAP - PROBE, CAP)]
    regions = _regions(probes, rec_off)
    return TwoBitBatch([CAP], regions, seed=2, shifts=_cap_shifts(regions)), probes


@pytest.mark.gpu
@pytest.mark.parametrize("name", PLANS + [CTX_PLAN])
def test_record_at_the_cap(name, leg_c, monkeypatch):
    _need_device(2 << 30)
    batch, probes = leg_c
    base, plan, ms = _open(name, monkeypatch)
    if base == "descr.eloop":
        # its windows and hit windows run past both strands' ends here: szero + 6 000 passes 2^31 - 1
        probes = [(0, ELOOP_PROBE), (CAP - ELOOP_PROBE, CAP)]
    try:
        batch.upload(ms)
        got = check_probes(ms, base, plan, batch, "C", probes)
        if base == CTX_PLAN:
            # right contexts clipped by the strand's end: the forward strand at the record end, the
            # complementary one at the record start; roff + 4000 passes 2^31 - 1 for these
            for comp, (lo, hi) in ((0, probes[1]), (1, probes[0])):
                h = got[(lo, hi)]
                h = h[h["comp"] == comp]
                assert (h["rctx_off"].astype(np.int64) + 4000 > (1 << 31) - 1).any(), \
                    f"strand {comp}: no candidate whose right context reaches the record end"
        assert ms.get_chars(0, 100).tobytes() == batch.chars(0, 100).tobytes()
        assert ms.get_chars(CAP - 100, 100).tobytes() == batch.chars(CAP - 100, CAP).tobytes()
        if base == "trna" and name == base:
            # one nucleotide more is refused, and the batch held stays as it was
            with pytest.raises(gpumotif.GpuMotifError, match="longer than 2"):
                ms.upload_2bit_ptr(batch.data.ctypes.data, batch.data.size, batch.dna_off,
                                   np.array([0, CAP + 1], dtype=np.int64), batch.nblk)
            assert ms.total_nt == CAP
            check_probes(ms, base, plan, batch, "C", probes, windows=False)
    finally:
        ms.close()


@pytest.mark.gpu
def test_record_at_the_cap_score_prescreen(leg_c):
    _need_device(2 << 30)
    batch, probes = leg_c
    check_score(load_plan("score.1"), batch, "C", probes)


# ------------------------------------------------------------------ leg D: FASTA text past 2^31 bytes

class FastaBatch(TwoBitBatch):
    """A FASTA text in host memory: records of `lengths` nucleotides in 60-column lines under the given
    header lines, random acgt except at the nucleotides of `regions` (batch coordinates), which hold the
    golden record's letters as they are.  hdr_off and rec_off are what the device's reader must find."""

    def __init__(self, headers, lengths, regions, seed=4):
        lengths = np.asarray(lengths, dtype=np.int64)
        self.rec_off = np.zeros(len(lengths) + 1, dtype=np.int64)
        np.cumsum(lengths, out=self.rec_off[1:])
        self.total_nt = int(self.rec_off[-1])
        self.fold = _FOLD
        self.headers = [h.encode() for h in headers]
        body = lengths + (lengths + 59) // 60                  # every line ends in '\n'
        sizes = np.array([len(h) + 1 for h in self.headers], dtype=np.int64) + body
        self.hdr_off = np.zeros(len(lengths) + 1, dtype=np.int64)
        np.cumsum(sizes, out=self.hdr_off[1:])
        self.body_off = self.hdr_off[:-1] + [len(h) + 1 for h in self.headers]
        n = int(self.hdr_off[-1])
        self.text = np.empty(n, dtype=np.uint8)
        rng = np.random.default_rng(seed)
        lut = np.frombuffer(b"acgt", dtype=np.uint8)
        step = 1 << 26
        for a in range(0, n, step):
            k = min(step, n - a)
            self.text[a:a + k] = lut[np.frombuffer(rng.bytes(k), dtype=np.uint8) & 3]
        for r, h in enumerate(self.headers):
            a = int(self.hdr_off[r])
            self.text[a:a + len(h) + 1] = np.frombuffer(h + b"\n", dtype=np.uint8)
            L, b0 = int(lengths[r]), int(self.body_off[r])
            self.text[b0 + 60 + 61 * np.arange(L // 60, dtype=np.int64)] = ord("\n")
            if L % 60:
                self.text[b0 + 61 * (L // 60) + L % 60] = ord("\n")
        gold = golden_record()
        self.starts, self.parts = [], []
        for i, (g0, g1) in enumerate(sorted(regions)):
            s = gold[(np.arange(g1 - g0) + 7919 * i) % len(gold)]
            self.text[self.text_pos(np.arange(g0, g1, dtype=np.int64))] = s
            self.starts.append(g0)
            self.parts.append(s)
        self.ends = np.array([a + len(p) for a, p in zip(self.starts, self.parts)], dtype=np.int64)
        self.starts = np.array(self.starts, dtype=np.int64)

    def text_pos(self, g):
        """Byte offsets in the text of nucleotides g (batch coordinates)."""
        r = np.searchsorted(self.rec_off, g, side="right") - 1
        p = g - self.rec_off[r]
        return self.body_off[r] + p + p // 60

    def upload(self, ms, rec_off=None):
        assert rec_off is None
        ms.upload_fastn(self.text)


G31B = 1 << 31
D_HEADERS = [">r0 below 2^31 bytes", ">r1 its lines cross byte 2^31", ">r2 header past byte 2^31, spans nucleotide 2^31",
             ">r3 last record, a short last line"]


@pytest.fixture(scope="module")
def leg_d():
    # r1 ends 4 MiB past byte 2^31, so r2's and r3's headers lie past it; r2 holds nucleotide 2^31
    l0 = 1_000_000_000
    t0 = len(D_HEADERS[0]) + 1 + l0 + (l0 + 59) // 60 + len(D_HEADERS[1]) + 1
    l1 = (G31B + (4 << 20) - t0) * 60 // 61
    lengths = [l0, l1, 60_000_001, 999_999]
    rec_off = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
    places = [int(rec_off[2]), G31, int(rec_off[-1])]
    batch = FastaBatch(D_HEADERS, lengths, _regions(_probes_around(places, rec_off), rec_off))
    assert batch.hdr_off[2] > G31B and batch.text.size > G31B + (32 << 20) and rec_off[2] < G31 < rec_off[3]
    return batch, places


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["trna", "score.1"])
def test_fasta_text_past_2_31_bytes(name, leg_d, monkeypatch):
    _need_device(6 << 30)
    batch, places = leg_d
    base, plan, ms = _open(name, monkeypatch)
    try:
        batch.upload(ms)
        rec, hdr = ms.records()
        assert rec.tolist() == batch.rec_off.tolist()
        assert hdr.tolist() == batch.hdr_off.tolist()
        for r in (2, 3):
            h = batch.headers[r]
            assert ms.get_text(int(batch.hdr_off[r]), len(h) + 1) == h + b"\n", f"header of record {r}"
        check_probes(ms, base, plan, batch, "D", _plan_probes(base, places, batch.rec_off))
        for a, n in ((G31 - 1000, 2500), (batch.total_nt - 9, 9)):
            assert ms.get_chars(a, n).tobytes() == _FOLD[batch.chars(a, a + n)].tobytes(), f"get_chars({a}, {n})"
    finally:
        ms.close()
