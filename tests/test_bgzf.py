"""GPU: the BGZF upload (gm_db_upload_fastn_bgzf / MotifSearch.upload_fastn_bgzf, include/gpumotif.h).

It is defined as gm_db_upload_fastn of the decompressed text, so everything here is checked against
that upload and against the oracle over fastn.parse_fastn of the text.  The FASTA has ragged records
of 0 to 150 001 nt, mixed case, N runs, 60-column and irregular lines, so header lines and records
straddle members.  Also: what the caller reads back, zlib's levels and strategies, member sizes,
empty members, concatenated files, the GenBank sample against the reference's stored candidate
streams, sequences of uploads, shards, and the refusals -- on the host before the previous batch is
touched, and on the device after inflating, after which the context holds no database."""
import gzip
import json
import os
import struct
import zlib

import numpy as np
import pytest

from rnamotif_b200 import bgzf, fastn, gpumotif, synth
from oracle import oracle_port
import helpers
import shard

pytestmark = pytest.mark.gpu

NAMES = ["trna", "ire", "score.1", "pk1", "qu+tr"]


def make_text(seed=43):
    rng = np.random.default_rng(seed)
    lengths = [0, 1, 3, 5] + list(rng.integers(0, 6000, size=30)) + [150001, 120, 0, 40, 7000]
    ids, seq, off = synth.random_records(seed, lengths, planted=True)
    up = rng.random(len(seq)) < 0.2
    seq[up] -= 32  # mixed case
    for r in range(4, len(lengths)):
        a, b = int(off[r]), int(off[r + 1])
        if b - a > 50:
            k = int(rng.integers(1, 40))
            p = int(rng.integers(a, b - k))
            seq[p:p + k] = ord("N")
    out = []
    for r, sid in enumerate(ids):
        out.append(b">%s record %d of the BGZF test\n" % (sid.encode(), r))
        s = seq[off[r]:off[r + 1]].tobytes()
        k = 0
        while k < len(s):
            w = 60 if r % 3 else int(rng.integers(1, 300))  # 60-column and irregular lines
            out.append(s[k:k + w] + (b"\n\n" if rng.random() < 0.02 else b"\n"))
            k += w
    return b"".join(out)


@pytest.fixture(scope="module")
def db():
    text = make_text()
    _, _, seq, off = fastn.parse_fastn(text)
    return text, bgzf.write_bgzf(text), seq, off


_REF = {}


def reference(name, seq, off):
    if name not in _REF:
        plan = helpers.load_plan(name)
        _REF[name] = oracle_port.scan_db(plan, seq, off, bool(gpumotif.plan_field(plan, 8)))[0]
    return _REF[name]


def pinned(b):
    import torch
    t = torch.empty(len(b), dtype=torch.uint8, pin_memory=True)
    t.numpy()[:] = np.frombuffer(b, dtype=np.uint8)
    return t


@pytest.mark.parametrize("memory", ["pageable", "pinned"])
@pytest.mark.parametrize("chunk", ["default", "16384"])
@pytest.mark.parametrize("name", NAMES)
def test_bgzf_upload_matches_oracle_and_text_upload(name, chunk, memory, db, monkeypatch):
    if chunk != "default":
        monkeypatch.setenv("GPUMOTIF_CHUNK_NT", chunk)  # chunks of 16 KiB of compressed bytes: many of them
    text, gz, seq, off = db
    ref = reference(name, seq, off)
    ms = gpumotif.MotifSearch(helpers.load_plan(name))
    ms.upload_fastn(text)
    by_text = ms.scan()
    if memory == "pinned":
        t = pinned(gz)
        ms.upload_fastn_bgzf_ptr(t.data_ptr(), len(gz))
    else:
        ms.upload_fastn_bgzf(gz)
    first = ms.scan()
    again = ms.scan()
    ms.close()
    helpers.assert_same_hits(by_text, ref, f"{name}: text upload")
    helpers.assert_same_hits(first, ref, f"{name}: BGZF upload ({chunk}, {memory})")
    helpers.assert_same_hits(again, ref, f"{name}: BGZF upload, rescan")
    assert len(ref) > 0 or name in ("ire", "qu+tr")


@pytest.mark.parametrize("name", ["trna", "score.1"])
def test_what_the_caller_reads_back(name, db, monkeypatch):
    monkeypatch.setenv("GPUMOTIF_CHUNK_NT", "16384")
    text, gz, seq, off = db
    ms = gpumotif.MotifSearch(helpers.load_plan(name))
    ms.upload_fastn(text)
    ms.scan()
    rec_t, hdr_t = ms.records()
    txt_t = ms.get_text()
    win_t = ms.hit_windows(40, 5000)
    ch_t = ms.get_chars()
    ms.upload_fastn_bgzf(gz)
    hits = ms.scan()
    rec_b, hdr_b = ms.records()
    txt_b = ms.get_text()
    part = ms.get_text(1000, 777)
    win_b = ms.hit_windows(40, 5000)
    ch_b = ms.get_chars()
    total = ms.total_nt
    ms.close()
    assert len(hits) > 0
    assert (rec_b == rec_t).all() and (hdr_b == hdr_t).all() and hdr_b[-1] == len(text)
    assert (rec_b == off).all() and total == off[-1]
    assert txt_b == txt_t == text and part == text[1000:1777]
    assert win_b.shape == win_t.shape and (win_b == win_t).all()
    assert ch_b.tobytes() == ch_t.tobytes() == seq.tobytes()


def variants(text):
    small = text[:3000]
    def co(lv, st=zlib.Z_DEFAULT_STRATEGY, block=0xff00, data=text):
        return bgzf.write_bgzf(data, lv, block, st)
    return {
        "level 0": (co(0), text), "level 1": (co(1), text), "level 9": (co(9), text),
        "huffman only": (co(6, zlib.Z_HUFFMAN_ONLY), text), "rle": (co(6, zlib.Z_RLE), text),
        "fixed": (co(6, zlib.Z_FIXED), text),
        "1-byte members": (co(6, block=1, data=small), small), "100-byte members": (co(6, block=100), text),
        "4 KiB members": (co(6, block=4096), text), "64 KiB members": (co(6, block=65536), text),
        "empty members": (bgzf.EOF_BLOCK + bgzf.write_bgzf(text[:7000], eof=False) + bgzf.EOF_BLOCK * 3
                          + bgzf.write_bgzf(text[7000:]), text),
        "two files": (bgzf.write_bgzf(text[:123456]) + bgzf.write_bgzf(text[123456:]), text),
        "no EOF block": (bgzf.write_bgzf(text, eof=False), text),
    }


def test_compression_variants(db, monkeypatch):
    monkeypatch.setenv("GPUMOTIF_CHUNK_NT", "16384")
    text, gz, seq, off = db
    ms = gpumotif.MotifSearch(helpers.load_plan("trna"))
    for what, (g, want) in variants(text).items():
        assert gzip.decompress(g) == want, what
        ms.upload_fastn_bgzf(g)
        assert ms.get_text() == want, what
        rec, hdr = ms.records()
        assert (rec == fastn.parse_fastn(want)[3]).all() and hdr[-1] == len(want), what
    ms.close()


def test_empty_uploads(db):
    text, gz, seq, off = db
    ms = gpumotif.MotifSearch(helpers.load_plan("trna"))
    for g in (b"", bgzf.EOF_BLOCK, bgzf.EOF_BLOCK * 2):
        ms.upload_fastn_bgzf(g)
        assert ms.total_nt == 0 and len(ms.scan()) == 0 and ms.get_text() == b""
        rec, hdr = ms.records()
        assert list(rec) == [0] and list(hdr) == [0]
    ms.close()


# ---- the GenBank sample, recompressed ------------------------------------------------------------

GBRNA = os.path.join(helpers.GOLDEN, "gbrna")
STREAMS = json.load(open(os.path.join(GBRNA, "streams.json")))


def assert_stream(hits, want, what):
    """The check of tests/test_gpu_stdout.py: count and digest of the reference's candidate stream."""
    assert len(hits) == want["n"], f"{what}: {len(hits)} candidates, the reference {want['n']}"
    if want["n"]:
        head, els = helpers.hits_to_rows(hits)
        got = helpers.stream_md5(head, els, helpers.ctx_rows(hits) if want["context"] else None)
        assert got == want["md5"], f"{what}: candidate stream differs from the reference's"


def gbrna_plain_gzip():
    with open(os.path.join(GBRNA, "sample.fastn.gz"), "rb") as fh:
        return fh.read()


@pytest.fixture(scope="module")
def gbrna_bgzf():
    return bgzf.write_bgzf(gzip.decompress(gbrna_plain_gzip()))


@pytest.mark.parametrize("name", sorted(STREAMS))
def test_gbrna_sample_as_bgzf_equals_reference_stream(name, gbrna_bgzf):
    ms = gpumotif.MotifSearch(helpers.load_plan(name))
    ms.upload_fastn_bgzf(gbrna_bgzf)
    assert_stream(ms.scan(), STREAMS[name], name)
    ms.close()


# ---- sequences of uploads, shards ----------------------------------------------------------------

def test_sequences_of_uploads(db, monkeypatch):
    monkeypatch.setenv("GPUMOTIF_CHUNK_NT", "16384")
    text, gz, seq, off = db
    ref = reference("trna", seq, off)
    ms = gpumotif.MotifSearch(helpers.load_plan("trna"))
    ms.upload_fastn_bgzf(gz)
    a = ms.scan()
    b = ms.find_motif(seq, off)
    ms.upload_fastn_bgzf(bgzf.write_bgzf(text, level=1, block=3000))
    c = ms.scan()
    _, hdr_c = ms.records()
    ms.upload_fastn(text)
    d = ms.scan()
    ms.find_motif(seq, off)
    with pytest.raises(gpumotif.GpuMotifError, match="not gm_db_upload_fastn"):
        ms.get_text(0, 10)  # refused after a character upload
    ms.close()
    for what, h in (("BGZF", a), ("characters after BGZF", b), ("BGZF after characters", c), ("text after BGZF", d)):
        helpers.assert_same_hits(h, ref, what)
    assert hdr_c[-1] == len(text)


@pytest.mark.parametrize("name", ["trna", "score.1"])
def test_shards_of_one_bgzf_upload(name, db, monkeypatch):
    monkeypatch.setenv("GPUMOTIF_CHUNK_NT", "16384")
    text, gz, seq, off = db
    parts = []
    for lo, hi in shard.shard_ranges(int(off[-1]), 3):
        ms = gpumotif.MotifSearch(helpers.load_plan(name))
        ms.upload_fastn_bgzf(gz)
        parts.append(ms.scan(lo, hi))
        ms.close()
    helpers.assert_same_hits(shard.merge_hits(parts), reference(name, seq, off), f"{name}: three shards")


# ---- refusals ------------------------------------------------------------------------------------

def members(buf):
    out, p = [], 0
    while p < len(buf):
        size = struct.unpack_from("<H", buf, p + 16)[0] + 1
        out.append((p, size))
        p += size
    return out


def test_host_refusals_leave_the_previous_batch(db):
    text, gz, seq, off = db
    ref = reference("trna", seq, off)
    ms_ = members(gz)
    p_last, size_last = ms_[-2]  # the last data member (the EOF block follows)
    big = bytearray(gz)
    struct.pack_into("<I", big, p_last + size_last - 4, 65537)
    past = bytearray(gz)
    struct.pack_into("<H", past, ms_[-1][0] + 16, 200)  # the EOF block's BSIZE runs past the end
    cases = [("plain gzip", gbrna_plain_gzip(), "not BGZF: recompress with bgzip"),
             ("truncated last member", gz[:p_last + size_last - 3], "runs past"),
             ("BSIZE past the end", bytes(past), "runs past"),
             ("ISIZE over 65536", bytes(big), "ISIZE 65537 over 65536"),
             ("bytes left over", gz + b"\x1f\x8b\x08", "left over")]
    ms = gpumotif.MotifSearch(helpers.load_plan("trna"))
    ms.upload_fastn_bgzf(gz)
    helpers.assert_same_hits(ms.scan(), ref, "before the refusals")
    for what, g, msg in cases:
        with pytest.raises(gpumotif.GpuMotifError, match=msg):
            ms.upload_fastn_bgzf(g)
        helpers.assert_same_hits(ms.scan(), ref, f"the previous upload after refusing {what}")
    ms.close()


def device_error_cases(text, gz):
    ms_ = members(gz)
    k = 3
    p, size = ms_[k]
    crc = bytearray(gz)
    crc[p + size - 8] ^= 0x40                   # a flipped CRC byte: the data inflates, the CRC differs
    isz = bytearray(gz)
    struct.pack_into("<I", isz, p + size - 4, struct.unpack_from("<I", gz, p + size - 4)[0] - 1)  # output longer than ISIZE
    bad = bytearray(gz)
    bad[p + 18] |= 0x06                         # the first block's type becomes 3
    return [("CRC", bytes(crc), f"member {k} at byte {p}: CRC-32 mismatch"),
            ("ISIZE", bytes(isz), f"member {k} at byte {p}: output longer than ISIZE"),
            ("deflate", bytes(bad), f"member {k} at byte {p}: bad block type"),
            ("no '>'", bgzf.write_bgzf(b"acgt\n" + text), "does not begin with '>'")]


def test_device_errors_name_the_member_and_drop_the_database(db):
    text, gz, seq, off = db
    ref = reference("trna", seq, off)
    ms = gpumotif.MotifSearch(helpers.load_plan("trna"))
    for what, g, msg in device_error_cases(text, gz):
        ms.upload_fastn_bgzf(gz)
        ms.scan()
        with pytest.raises(gpumotif.GpuMotifError, match=msg):
            ms.upload_fastn_bgzf(g)
        for call in (lambda: ms.scan(0, 0), lambda: ms.get_chars(0, 1), lambda: ms.get_text(0, 1),
                     lambda: ms.hit_windows()):
            with pytest.raises(gpumotif.GpuMotifError, match="no database uploaded"):
                call()
        ms.upload_fastn_bgzf(gz)
        helpers.assert_same_hits(ms.scan(), ref, f"the upload after a {what} error")
    ms.close()


@pytest.mark.parametrize("name", ["trna"])
def test_bytes_over_the_link(name, db):
    text, gz, seq, off = db
    ms = gpumotif.MotifSearch(helpers.load_plan(name))
    ms.upload_fastn_bgzf(gz)
    ms.scan()
    st = ms.stats()
    ms.close()
    assert st.h2d_bytes == len(gz) + 32 * len(members(gz))
