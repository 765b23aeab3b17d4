"""GPU: the FASTQ uploads (gm_db_upload_fastq / gm_db_upload_fastq_bgzf, MotifSearch.upload_fastq and
upload_fastq_bgzf, include/gpumotif.h).

The database is seeded reads of 0 to 400 nt (synth.random_reads: planted stem-loops, 'N' and '.'
calls), written by fastq.write_fastq with quality strings that start with '@' or '+' now and then,
so records and lines straddle many of the reader's 16 KB segments.  Everything is checked against
the oracle over fastq.parse_fastq's reads and against the character upload of the same reads: the
candidate streams, what the caller reads back, sequences of uploads, shards, the starts a scan
counts, and the refusals -- on the host before the previous batch is touched, and on the device,
naming the first failing record, after which the context holds no database."""
import concurrent.futures
import gzip
import re
import struct

import numpy as np
import pytest

from rnamotif_b200 import bgzf, fastn, fastq, gpumotif, synth
from oracle import oracle_port
import helpers
import shard

pytestmark = pytest.mark.gpu

NAMES = ["trna", "ire", "score.1", "pk1", "qu+tr"]
N_READS = 50000
# pk1's oracle takes minutes over 50 000 reads: it is checked on the first 5 000
ORACLE_READS = {"pk1": 5000}


def make_reads(n_reads=N_READS, seed=2026, crlf=False):
    rng = np.random.default_rng(seed)
    lengths = rng.integers(0, 401, size=n_reads)
    ids, seq, off = synth.random_reads(seed, lengths)
    qual = []
    for r in range(n_reads):
        q = rng.integers(33, 74, size=int(lengths[r]), dtype=np.uint8)
        if len(q) and r % 5 == 0:
            q[0] = ord("@") if r % 2 else ord("+")  # quality strings that look like header lines
        qual.append(q.tobytes())
    return fastq.write_fastq([f"{i} sample=7 run=3" for i in ids], seq, off, qual, crlf)


@pytest.fixture(scope="module")
def db():
    text = make_reads()
    ids, seq, off, hdr = fastq.parse_fastq(text)
    return text, bgzf.write_bgzf(text), seq, off, hdr


@pytest.fixture(scope="module")
def refs(db):
    """The oracle's candidates per descriptor, computed side by side (the oracle releases the GIL)."""
    text, _, seq, off, _ = db

    def one(name):
        plan = helpers.load_plan(name)
        n = ORACLE_READS.get(name, N_READS)
        return oracle_port.scan_db(plan, seq[:off[n]], off[:n + 1], bool(gpumotif.plan_field(plan, 8)))[0]

    with concurrent.futures.ThreadPoolExecutor(len(NAMES)) as ex:
        return dict(zip(NAMES, ex.map(one, NAMES)))


def subset(text, seq, off, hdr, name):
    """The FASTQ text, reads and offsets of the first ORACLE_READS[name] records."""
    n = ORACLE_READS.get(name, N_READS)
    return text[:hdr[n]], seq[:off[n]], off[:n + 1]


def pinned(b):
    import torch
    t = torch.empty(len(b), dtype=torch.uint8, pin_memory=True)
    t.numpy()[:] = np.frombuffer(b, dtype=np.uint8)
    return t


@pytest.mark.parametrize("memory", ["pageable", "pinned"])
@pytest.mark.parametrize("chunk", ["default", "16384"])
@pytest.mark.parametrize("name", NAMES)
def test_fastq_upload_matches_oracle_and_character_upload(name, chunk, memory, db, refs, monkeypatch):
    if chunk != "default":
        monkeypatch.setenv("GPUMOTIF_CHUNK_NT", chunk)  # many chunks of the pack and of the BGZF copy
    text, seq, off = subset(*db[0:1], *db[2:], name)
    gz = db[1] if len(text) == len(db[0]) else bgzf.write_bgzf(text)
    ref = refs[name]
    ms = gpumotif.MotifSearch(helpers.load_plan(name))
    if memory == "pinned":
        t, g = pinned(text), pinned(gz)
        ms.upload_fastq_ptr(t.data_ptr(), len(text))
        by_fastq = ms.scan()
        ms.upload_fastq_bgzf_ptr(g.data_ptr(), len(gz))
    else:
        ms.upload_fastq(text)
        by_fastq = ms.scan()
        ms.upload_fastq_bgzf(gz)
    by_bgzf = ms.scan()
    again = ms.scan()
    ms.upload(seq, off)
    by_chars = ms.scan()
    ms.close()
    helpers.assert_same_hits(by_chars, ref, f"{name}: character upload")
    helpers.assert_same_hits(by_fastq, ref, f"{name}: FASTQ upload ({chunk}, {memory})")
    helpers.assert_same_hits(by_bgzf, ref, f"{name}: BGZF FASTQ upload ({chunk}, {memory})")
    helpers.assert_same_hits(again, ref, f"{name}: BGZF FASTQ upload, rescan")
    assert len(ref) > 0 or name == "ire"


@pytest.mark.parametrize("name", ["trna", "score.1"])
def test_what_comes_back(name, db, monkeypatch):
    monkeypatch.setenv("GPUMOTIF_CHUNK_NT", "16384")
    text, gz, seq, off, hdr = db
    ms = gpumotif.MotifSearch(helpers.load_plan(name))
    ms.upload(seq, off)
    ms.scan()
    win_c = ms.hit_windows(40, 500)
    for up in (ms.upload_fastq, ms.upload_fastq_bgzf):
        up(text if up == ms.upload_fastq else gz)
        hits = ms.scan()
        rec, hd = ms.records()
        assert (rec == off).all() and (hd == hdr).all() and ms.total_nt == off[-1]
        assert ms.get_text() == text
        names = [ms.get_text(int(hd[r]), int(text.index(b"\n", hd[r]) - hd[r])) for r in range(len(hd) - 1)]
        assert names == [text[hd[r]:text.index(b"\n", hd[r])] for r in range(len(hd) - 1)]
        assert names[7] == b"@read7 sample=7 run=3"
        win = ms.hit_windows(40, 500)
        assert len(hits) > 0 and win.shape == win_c.shape and (win == win_c).all()
        assert ms.get_chars().tobytes() == seq.tobytes()
    ms.close()


def test_crlf_and_no_last_newline(db):
    text, gz, seq, off, hdr = db
    crlf = make_reads(3000, seed=9, crlf=True)
    plain = make_reads(3000, seed=9)
    ms = gpumotif.MotifSearch(helpers.load_plan("trna"))
    ms.upload_fastq(plain)
    want = ms.scan()
    rec_p, _ = ms.records()
    for what, t in (("CR LF", crlf), ("CR LF, no last line end", crlf[:-2]), ("no last newline", plain[:-1])):
        for up in (ms.upload_fastq, lambda b: ms.upload_fastq_bgzf(bgzf.write_bgzf(b, block=777))):
            up(t)
            rec, hd = ms.records()
            assert (rec == rec_p).all() and (hd == fastq.parse_fastq(t)[3]).all(), what
            helpers.assert_same_hits(ms.scan(), want, what)
    ms.close()


def test_sequences_of_uploads_and_shards(db, refs, monkeypatch):
    monkeypatch.setenv("GPUMOTIF_CHUNK_NT", "16384")
    text, gz, seq, off, hdr = db
    ref = refs["trna"]
    # the same reads as FASTA, where '.' is not a letter: 'x' is, and packs to the same code 0
    fseq = seq.copy()
    fseq[fseq == ord(".")] = ord("x")
    fasta = b"".join(b">r%d\n%s\n" % (r, fseq[off[r]:off[r + 1]].tobytes()) for r in range(len(off) - 1))
    assert (fastn.parse_fastn(fasta)[3] == off).all()
    ms = gpumotif.MotifSearch(helpers.load_plan("trna"))
    ms.upload_fastq(text)
    a = ms.scan()
    ms.upload_fastn(fasta)
    b = ms.scan()
    ms.upload_fastq_bgzf(gz)
    c = ms.scan()
    ms.upload(seq, off)
    d = ms.scan()
    with pytest.raises(gpumotif.GpuMotifError, match="gm_db_upload_fastq"):
        ms.get_text(0, 10)  # refused after a character upload
    ms.close()
    for what, h in (("FASTQ", a), ("BGZF FASTQ after FASTA", c), ("characters after BGZF FASTQ", d)):
        helpers.assert_same_hits(h, ref, what)
    helpers.assert_same_hits(b, ref, "FASTA after FASTQ")
    for up in ("fastq", "bgzf"):
        parts = []
        for lo, hi in shard.shard_ranges(int(off[-1]), 3):
            m = gpumotif.MotifSearch(helpers.load_plan("trna"))
            m.upload_fastq(text) if up == "fastq" else m.upload_fastq_bgzf(gz)
            parts.append(m.scan(lo, hi))
            m.close()
        helpers.assert_same_hits(shard.merge_hits(parts), ref, f"three shards of one {up} upload")


def sieve_starts(rec_off, lo, hi, strands, dm):
    """The starts a sieve-path scan of [lo, hi) counts, one record at a time."""
    ns = 0
    for r in range(len(rec_off) - 1):
        a, b = max(rec_off[r], lo), min(rec_off[r + 1], hi)
        if b <= a:
            continue
        o, slen = rec_off[r], rec_off[r + 1] - rec_off[r]
        ns += max(0, min(b, o + slen - dm + 1) - a)
        if strands > 1:
            ns += max(0, b - max(a, o + dm - 1))
    return ns


@pytest.mark.parametrize("name", ["trna"])  # the sieve path counts its starts on the host
def test_starts_counted_per_range(name, db):
    text, gz, seq, off, hdr = db
    plan = helpers.load_plan(name)
    dm, both = gpumotif.plan_field(plan, 4), gpumotif.plan_field(plan, 8)
    ro = [int(x) for x in off[:2001]]
    n = ro[-1]
    ms = gpumotif.MotifSearch(plan)
    ms.upload(seq[:n], off[:2001])
    rng = np.random.default_rng(4)
    ranges = [(0, n), (0, 0), (0, 1), (n - 1, n), (ro[10], ro[11]), (ro[10] + 1, ro[12] - 1), (ro[5], ro[5] + 3)]
    ranges += [tuple(sorted(int(x) for x in rng.integers(0, n + 1, size=2))) for _ in range(12)]
    for lo, hi in ranges:
        ms.scan(lo, hi)
        st = ms.stats()
        assert st.n_starts == sieve_starts(ro, lo, hi, 2 if both else 1, dm), (name, lo, hi)
    ms.close()


# ---- refusals ------------------------------------------------------------------------------------

def test_host_refusals_leave_the_previous_batch(db, refs):
    text, gz, seq, off, hdr = db
    ref = refs["trna"]
    ms = gpumotif.MotifSearch(helpers.load_plan("trna"))
    ms.upload_fastq(text)
    helpers.assert_same_hits(ms.scan(), ref, "before the refusals")
    for what, call, msg in (("no '@'", lambda: ms.upload_fastq(b"ACGT\n" + text), "does not begin with '@'"),
                            ("NULL", lambda: ms.upload_fastq_ptr(0, 10), "text is NULL"),
                            ("too long", lambda: ms.upload_fastq_ptr(1, (1 << 40) + 1), "text too long"),
                            ("plain gzip", lambda: ms.upload_fastq_bgzf(gzip.compress(text[:1000])),
                             "not BGZF"),
                            ("NULL gz", lambda: ms.upload_fastq_bgzf_ptr(0, 10), "gz is NULL")):
        with pytest.raises(gpumotif.GpuMotifError, match=msg):
            call()
        helpers.assert_same_hits(ms.scan(), ref, f"the previous upload after refusing {what}")
        assert (ms.records()[1] == hdr).all(), what
    ms.close()


def device_error_cases(text, hdr):
    """(what, text, record, message) -- each mutation of the reads' text the device refuses."""
    lines = text.split(b"\n")

    def edit(fn):
        ls = list(lines)
        fn(ls)
        return b"\n".join(ls)

    def rec_line(ls, r, k, v):
        ls[4 * r + k] = v

    cut = int(hdr[20001])
    return [
        ("'@' line", edit(lambda ls: rec_line(ls, 20000, 0, b"read20000")), 20000, "line 80001 does not start with '@'"),
        ("'+' line", edit(lambda ls: rec_line(ls, 31234, 2, b"-")), 31234, "line 124939 does not start with '+'"),
        ("multi-line", edit(lambda ls: ls.insert(4 * 40000 + 2, b"ACGT")), 40000, "does not start with '+'"),
        ("quality length", edit(lambda ls: rec_line(ls, 777, 3, ls[4 * 777 + 3] + b"I")), 777,
         "quality string is not as long as its read"),
        ("short last record", text + b"@extra\nACGT\n", 50000, "fewer than four lines"),
        ("two lines cut off", text[:cut] + b"@x\nAC\n+\nII\n@y\nAC\n", 20002, "fewer than four lines"),
        ("first of two", edit(lambda ls: (rec_line(ls, 45000, 2, b"x"), rec_line(ls, 12345, 3, ls[4 * 12345 + 3] + b"II"))), 12345,
         "quality string"),
    ]


def test_device_errors_name_the_record_and_drop_the_database(db, refs):
    text, gz, seq, off, hdr = db
    ref = refs["trna"]
    ms = gpumotif.MotifSearch(helpers.load_plan("trna"))
    for what, bad, rec, msg in device_error_cases(text, hdr):
        with pytest.raises(fastq.FastqError, match=re.escape(msg)) as e:
            fastq.parse_fastq(bad)
        assert e.value.record == rec, what
        want = f"FASTQ record {rec} at byte {e.value.offset}: "
        for up in (ms.upload_fastq, lambda b: ms.upload_fastq_bgzf(bgzf.write_bgzf(b))):
            ms.upload_fastq(text)
            ms.scan()
            with pytest.raises(gpumotif.GpuMotifError, match=want) as g:
                up(bad)
            assert str(e.value) in str(g.value), what
            assert ms.total_nt == 0, what
            for call in (lambda: ms.scan(0, 0), lambda: ms.records(), lambda: ms.get_chars(0, 1),
                         lambda: ms.get_text(0, 1), lambda: ms.hit_windows()):
                with pytest.raises(gpumotif.GpuMotifError, match="no database uploaded"):
                    call()
        ms.upload_fastq(text)
        helpers.assert_same_hits(ms.scan(), ref, f"the upload after a {what} error")
    with pytest.raises(gpumotif.GpuMotifError, match="does not begin with '@'"):
        ms.upload_fastq_bgzf(bgzf.write_bgzf(b"\n" + text))
    ms.close()


def test_bytes_over_the_link_and_empty_uploads(db):
    text, gz, seq, off, hdr = db
    ms = gpumotif.MotifSearch(helpers.load_plan("trna"))
    ms.upload_fastq(text)
    ms.scan()
    assert ms.stats().h2d_bytes == len(text)
    ms.upload_fastq_bgzf(gz)
    ms.scan()
    n_mem, p = 0, 0
    while p < len(gz):
        p += struct.unpack_from("<H", gz, p + 16)[0] + 1
        n_mem += 1
    assert ms.stats().h2d_bytes == len(gz) + 32 * n_mem
    for t in (b"", bgzf.EOF_BLOCK):
        (ms.upload_fastq if t == b"" else ms.upload_fastq_bgzf)(t)
        assert ms.total_nt == 0 and len(ms.scan()) == 0 and ms.get_text() == b""
        rec, hd = ms.records()
        assert list(rec) == [0] and list(hd) == [0]
    ms.close()
