"""GPU: low-quality masking of the FASTQ uploads (gm_ctx_set_min_quality, MotifSearch.set_min_quality,
include/gpumotif.h).

The database is seeded reads of 0 to 400 nt (synth.random_reads) as four-line FASTQ whose quality
strings are mostly Q30-Q40 with one base in eight between Q0 and Q29, and start with '@' (Q31) or
'+' (Q10) now and then, so records and quality strings straddle the reader's 16 KB segments.  At
each threshold the candidate stream of a masked upload must equal the oracle's over
fastq.parse_fastq(text, min_qual)'s reads, the unmasked upload of the same text with the masked
read bytes written as 'n', and the character upload of the masked reads."""
import concurrent.futures
import re

import numpy as np
import pytest

from rnamotif_b200 import bgzf, fastq, gpumotif, synth, twobit
from oracle import oracle_port
import helpers

pytestmark = pytest.mark.gpu

NAMES = ["trna", "ire", "score.1", "pk1", "qu+tr"]
N_READS = 20000
ORACLE_READS = {"pk1": 2000}  # pk1's oracle is slow: it is checked on the first 2 000 reads
THRESHOLDS = [20, 33]


def make_reads(n_reads=N_READS, seed=2027):
    """(ids, seq, off, qual): the reads as synth.random_reads gives them, one quality string each"""
    rng = np.random.default_rng(seed)
    lengths = rng.integers(0, 401, size=n_reads)
    ids, seq, off = synth.random_reads(seed, lengths)
    qual = []
    for r in range(n_reads):
        n = int(lengths[r])
        q = np.where(rng.random(n) < 0.125, rng.integers(33, 63, size=n), rng.integers(63, 74, size=n)).astype(np.uint8)
        if n and r % 5 == 0:
            q[0] = ord("@") if r % 2 else ord("+")  # quality strings that look like header lines
        qual.append(q.tobytes())
    return [f"{i} sample=7" for i in ids], seq, off, qual


def rewritten(seq, qual, min_qual):
    """The read bytes with every low-quality one replaced by 'n' (what the masked upload must read)"""
    s = seq.copy()
    s[np.frombuffer(b"".join(qual), dtype=np.uint8) < 33 + min_qual] = ord("n")
    return s


@pytest.fixture(scope="module")
def db():
    ids, seq, off, qual = make_reads()
    text = fastq.write_fastq(ids, seq, off, qual)
    masked = {}
    for mq in THRESHOLDS:
        m = fastq.parse_fastq(text, mq)
        assert (m[2] == off).all()
        hand = rewritten(seq, qual, mq)
        assert (m[1] == fastq._LOWER[hand]).all()
        # the text with the masked read bytes written as 'n', uploaded with masking off
        masked[mq] = (m[1], fastq.write_fastq(ids, hand, off, qual))
    return text, off, qual, masked


@pytest.fixture(scope="module")
def refs(db):
    """The oracle's candidates per (descriptor, threshold), over parse_fastq's masked reads."""
    text, off, _, masked = db

    def one(key):
        name, mq = key
        plan = helpers.load_plan(name)
        n = ORACLE_READS.get(name, N_READS)
        return oracle_port.scan_db(plan, masked[mq][0][:off[n]], off[:n + 1], bool(gpumotif.plan_field(plan, 8)))[0]

    keys = [(name, mq) for name in NAMES for mq in THRESHOLDS]
    with concurrent.futures.ThreadPoolExecutor(len(keys)) as ex:
        return dict(zip(keys, ex.map(one, keys)))


def pinned(b):
    import torch
    t = torch.empty(len(b), dtype=torch.uint8, pin_memory=True)
    t.numpy()[:] = np.frombuffer(b, dtype=np.uint8)
    return t


@pytest.mark.parametrize("memory", ["pageable", "pinned"])
@pytest.mark.parametrize("chunk", ["default", "16384"])
@pytest.mark.parametrize("name", NAMES)
def test_masked_upload_matches_oracle_rewritten_text_and_characters(name, chunk, memory, db, refs, monkeypatch):
    if chunk != "default":
        monkeypatch.setenv("GPUMOTIF_CHUNK_NT", chunk)
    text, off, _, masked = db
    n = ORACLE_READS.get(name, N_READS)
    hdr = fastq.parse_fastq(text)[3]
    text, off = text[:hdr[n]], off[:n + 1]
    texts = (("FASTQ", text), ("BGZF", bgzf.write_bgzf(text)), ("BGZF block 777", bgzf.write_bgzf(text, block=777)))
    ms = gpumotif.MotifSearch(helpers.load_plan(name))
    for mq in THRESHOLDS:
        ref = refs[(name, mq)]
        seq_m, text_m = masked[mq]
        text_m = text_m[:len(text)]  # the rewritten text has the same layout
        ms.set_min_quality(mq)
        got = {}
        for what, data in texts:
            up = ms.upload_fastq_ptr if what == "FASTQ" else ms.upload_fastq_bgzf_ptr
            if memory == "pinned":
                buf = pinned(data)
                up(buf.data_ptr(), len(data))
            else:
                a = np.frombuffer(data, dtype=np.uint8)
                up(a.ctypes.data, a.size)
            got[what] = ms.scan()
        ms.set_min_quality(0)
        ms.upload_fastq(text_m)
        got["rewritten text, masking off"] = ms.scan()
        ms.set_min_quality(mq)
        ms.upload(seq_m[:off[-1]], off)
        got["characters of the masked reads"] = ms.scan()
        for what, h in got.items():
            helpers.assert_same_hits(h, ref, f"{name} at Q{mq}: {what} ({chunk}, {memory})")
        if mq == THRESHOLDS[0]:
            assert len(ref) > 0 or name == "ire"
    ms.close()


@pytest.mark.parametrize("name", ["trna", "score.1"])
def test_what_comes_back(name, db, monkeypatch):
    monkeypatch.setenv("GPUMOTIF_CHUNK_NT", "16384")
    text, off, _, masked = db
    seq_m, _ = masked[20]
    gz = bgzf.write_bgzf(text, block=777)
    ms = gpumotif.MotifSearch(helpers.load_plan(name))
    ms.upload_fastq(text)
    ms.scan()
    rec0, hdr0 = ms.records()
    h2d = {"FASTQ": ms.stats().h2d_bytes}
    ms.upload_fastq_bgzf(gz)
    ms.scan()
    h2d["BGZF"] = ms.stats().h2d_bytes
    ms.upload(seq_m, off)
    ms.scan()
    win_c = ms.hit_windows(40, 500)
    ms.set_min_quality(20)
    for what, up in (("FASTQ", lambda: ms.upload_fastq(text)), ("BGZF", lambda: ms.upload_fastq_bgzf(gz))):
        up()
        hits = ms.scan()
        rec, hd = ms.records()
        assert (rec == rec0).all() and (hd == hdr0).all() and ms.total_nt == off[-1], what
        assert ms.stats().h2d_bytes == h2d[what], what
        assert ms.get_text() == text, what
        assert ms.get_chars().tobytes() == seq_m.tobytes(), what
        win = ms.hit_windows(40, 500)
        assert len(hits) > 0 and win.shape == win_c.shape and (win == win_c).all(), what
    ms.close()


def test_the_setting(db, refs):
    text, off, qual, masked = db
    ids = [str(r) for r in range(len(off) - 1)]
    plan = helpers.load_plan("trna")
    lib = gpumotif.lib()
    assert lib.gm_ctx_set_min_quality(None, 20, 33) != 0 and "NULL" in gpumotif._err()
    ms = gpumotif.MotifSearch(plan)
    ms.upload_fastq(text)
    plain = ms.scan()
    plain_chars = ms.get_chars()
    # 0 is never having set it
    ms.set_min_quality(30, 64)
    ms.set_min_quality(0)
    ms.upload_fastq(text)
    assert ms.scan().tobytes() == plain.tobytes() and ms.get_chars().tobytes() == plain_chars.tobytes()
    # the database held does not change until the next upload
    ms.set_min_quality(20)
    assert ms.scan().tobytes() == plain.tobytes() and ms.get_chars().tobytes() == plain_chars.tobytes()
    ms.upload_fastq(text)
    helpers.assert_same_hits(ms.scan(), refs[("trna", 20)], "the upload after the setting")
    masked20 = ms.get_chars()
    assert masked20.tobytes() == masked[20][0].tobytes()
    ms.set_min_quality(0)
    helpers.assert_same_hits(ms.scan(), refs[("trna", 20)], "switched off after the upload")
    # refused arguments leave the setting as it was
    ms.set_min_quality(20)
    for mq, qo in ((-1, 33), (94, 33), (63, 64), (20, 32), (20, 34), (20, 0)):
        with pytest.raises(gpumotif.GpuMotifError, match="gm_ctx_set_min_quality"):
            ms.set_min_quality(mq, qo)
    ms.upload_fastq(text)
    assert ms.get_chars().tobytes() == masked20.tobytes()
    # the FASTA, character and 2-bit uploads ignore it
    seq = plain_chars.copy()
    fseq = seq.copy()
    fseq[fseq == ord(".")] = ord("x")  # '.' is not a FASTA letter; 'x' is, and packs to the same code
    fasta = b"".join(b">r%d\n%s\n" % (r, fseq[off[r]:off[r + 1]].tobytes()) for r in range(len(off) - 1))
    tb = twobit.read_2bit(twobit.write_2bit(ids, seq, off))
    for what, up in (("FASTA", lambda: ms.upload_fastn(fasta)), ("BGZF FASTA", lambda: ms.upload_fastn_bgzf(bgzf.write_bgzf(fasta))),
                     ("characters", lambda: ms.upload(seq, off)), ("2-bit", lambda: ms.upload_2bit(tb))):
        ms.set_min_quality(0)
        up()
        want = ms.scan()
        ms.set_min_quality(20)
        up()
        assert ms.scan().tobytes() == want.tobytes(), what
    # a threshold that masks every base (every quality byte is below 33 + 93)
    ms.set_min_quality(93)
    ms.upload_fastq(text)
    assert set(ms.get_chars().tobytes()) == {ord("n")}
    assert len(ms.scan()) == 0
    ms.close()
    ms = gpumotif.MotifSearch(helpers.load_plan("score.1"))
    ms.set_min_quality(62, 64)  # every byte is below 64 + 62 = 126, and none below 64 is allowed: refused
    with pytest.raises(gpumotif.GpuMotifError, match=r"quality byte \d+ is outside \[64, 126\]"):
        ms.upload_fastq(text)
    ms.set_min_quality(93)
    ms.upload_fastq_bgzf(bgzf.write_bgzf(text))
    assert len(ms.scan()) == 0 and set(ms.get_chars().tobytes()) == {ord("n")}
    ms.close()


def range_error_cases(text):
    """(what, text) -- quality bytes out of range, alone and behind an earlier format error"""
    lines = text.split(b"\n")

    def edit(fn):
        ls = list(lines)
        fn(ls)
        return b"\n".join(ls)

    def put(ls, r, k, i, v):
        s = bytearray(ls[4 * r + k])
        s[i] = v
        ls[4 * r + k] = bytes(s)

    def longer(r0, n):
        return next(r for r in range(r0, N_READS) if len(lines[4 * r + 3]) > n)

    long_rec = longer(7000, 300)
    return [
        ("a space", edit(lambda ls: put(ls, longer(7000, 0), 3, 0, 32))),
        ("DEL at the end of a long string", edit(lambda ls: put(ls, long_rec, 3, -1, 127))),
        ("a high byte, two records", edit(lambda ls: (put(ls, long_rec, 3, 5, 200), put(ls, longer(15000, 0), 3, 0, 31)))),
        ("behind a format error", edit(lambda ls: (ls.__setitem__(4 * 3000 + 2, b"-"), put(ls, long_rec, 3, 1, 0)))),
        ("a format error behind it", edit(lambda ls: (ls.__setitem__(4 * 15000 + 2, b"-"), put(ls, long_rec, 3, 1, 0)))),
    ]


def test_range_refusals_name_the_record_and_drop_the_database(db, refs):
    text, off, _, _ = db
    ms = gpumotif.MotifSearch(helpers.load_plan("trna"))
    for what, bad in range_error_cases(text):
        with pytest.raises(fastq.FastqError) as e:
            fastq.parse_fastq(bad, 20)
        rec = e.value.record
        want = f"FASTQ record {rec} at byte {e.value.offset}: "
        for up in (ms.upload_fastq, lambda b: ms.upload_fastq_bgzf(bgzf.write_bgzf(b, block=777))):
            ms.set_min_quality(20)
            ms.upload_fastq(text)
            ms.scan()
            with pytest.raises(gpumotif.GpuMotifError, match=re.escape(want)) as g:
                up(bad)
            assert str(e.value) in str(g.value), what
            assert ms.total_nt == 0, what
            with pytest.raises(gpumotif.GpuMotifError, match="no database uploaded"):
                ms.records()
            if "format" not in what:
                ms.set_min_quality(0)
                up(bad)  # accepted with masking off
                assert ms.total_nt == off[-1], what
        ms.set_min_quality(20)
        ms.upload_fastq(text)
        helpers.assert_same_hits(ms.scan(), refs[("trna", 20)], f"the upload after a {what} refusal")
    ms.close()
