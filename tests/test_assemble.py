"""GPU: records assembled on the device from blocks of the held batch (gm_db_assemble /
MotifSearch.assemble, include/gpumotif.h).

The genome is synthetic: mixed case, IUPAC and non-IUPAC letters, N runs, empty and tiny records and
one of 150 001 nt.  The transcripts are seeded BED12 lines (synth.random_transcripts: both strands,
1-nt exons, shared and overlapping exons, non-coding lines, lines at chromosome ends).  After every
source upload -- characters from pageable and pinned memory, host-packed, device characters, FASTA,
BGZF FASTA and 2-bit -- the candidates after assemble must equal the oracle's over
Assembly.assemble_chars and the character upload's of those characters, with the default chunks and
with 16 Knt chunks.  Also: rescans, shards, the score pre-screen, one strand, the characters handed
back, assembling an assembled batch, an upload after an assembly, empty tables, the bytes over the
link, and every refusal leaving the held batch as it was."""
import numpy as np
import pytest

from rnamotif_b200 import bed, bgzf, gpumotif, synth, twobit
from oracle import oracle_port
import helpers
import shard

pytestmark = pytest.mark.gpu

NAMES = ["trna", "ire", "score.1", "pk1", "qu+tr"]
SOURCES = ["chars", "pinned", "hostpack", "device", "fastn", "bgzf", "2bit"]


@pytest.fixture(scope="module")
def genome():
    rng = np.random.default_rng(43)
    lengths = [0, 1, 3, 5] + list(rng.integers(0, 6000, size=30)) + [150001, 120, 40, 2, 7000]
    ids, seq, off = synth.random_records(43, lengths, planted=True, iupac_rate=0.01)
    up = rng.random(len(seq)) < 0.2
    seq[up] = np.frombuffer(bytes(seq[up]).upper(), dtype=np.uint8)
    for r in range(4, len(lengths)):
        a, b = int(off[r]), int(off[r + 1])
        if b - a > 50:
            k = int(rng.integers(1, 40))
            p = int(rng.integers(a, b - k))
            seq[p:p + k] = ord("N")
    tb = twobit.read_2bit(twobit.write_2bit(ids, seq, off))
    fasta = b"".join(b">" + i.encode() + b" synthetic record %d\n" % r + seq[off[r]:off[r + 1]].tobytes() + b"\n"
                     for r, i in enumerate(ids))
    text = synth.random_transcripts(8, ids, np.diff(off), 400, exon=40, first=60, last=150, intron=300, utr5=30,
                                    utr3=80, p_one=0.05, p_edge=0.05)
    asm = bed.read_bed(text, ids, off)
    return ids, seq, off, tb, fasta, asm


def held_chars(genome, source):
    """The characters the held batch reads as after `source`: the 2-bit file holds only a c g t n"""
    ids, seq, off, tb, fasta, asm = genome
    return twobit.to_chars(tb) if source == "2bit" else seq


_REF = {}


def reference(name, genome, source):
    kind = "2bit" if source == "2bit" else "chars"
    if (name, kind) not in _REF:
        chars, ro = genome[5].assemble_chars(held_chars(genome, source), genome[2])
        plan = helpers.load_plan(name)
        _REF[name, kind] = chars, ro, oracle_port.scan_db(plan, chars, ro, bool(gpumotif.plan_field(plan, 8)))[0]
    return _REF[name, kind]


def upload(ms, genome, source):
    """The source upload; returns what must stay alive until the next scan"""
    import torch
    ids, seq, off, tb, fasta, asm = genome
    if source == "chars":
        ms.upload(seq, off)
    elif source == "pinned":
        buf = torch.from_numpy(seq).pin_memory()
        ms.upload_ptr(buf.data_ptr(), off)  # asynchronous: assemble waits for the copy
        return buf
    elif source == "hostpack":
        ms.upload_hostpack(seq, off)
    elif source == "device":
        d = torch.from_numpy(seq).cuda()
        torch.cuda.synchronize()
        ms.set_device_chars(d.data_ptr(), off)
        return d
    elif source == "fastn":
        ms.upload_fastn(fasta)
    elif source == "bgzf":
        ms.upload_fastn_bgzf(bgzf.write_bgzf(fasta, block=7777))
    else:
        ms.upload_2bit(tb)
    return None


@pytest.mark.parametrize("chunk", ["default", "16384"])
@pytest.mark.parametrize("source", SOURCES)
@pytest.mark.parametrize("name", NAMES)
def test_assembled_candidates_match_oracle_and_character_upload(name, source, chunk, genome, monkeypatch):
    if chunk != "default":
        monkeypatch.setenv("GPUMOTIF_CHUNK_NT", chunk)
    chars, ro, ref = reference(name, genome, source)
    ms = gpumotif.MotifSearch(helpers.load_plan(name))
    keep = upload(ms, genome, source)
    ms.assemble_bed(genome[5])
    rec, hdr = ms.records()
    assert rec.tolist() == ro.tolist() and hdr is None and ms.total_nt == int(ro[-1])
    first = ms.scan()
    again = ms.scan()
    by_chars = ms.find_motif(chars, ro)
    ms.close()
    del keep
    helpers.assert_same_hits(first, ref, f"{name}: assembled after {source} ({chunk})")
    helpers.assert_same_hits(again, ref, f"{name}: rescan")
    helpers.assert_same_hits(by_chars, ref, f"{name}: character upload of assemble_chars")
    assert len(ref) > 0 or name in ("ire", "qu+tr")


@pytest.mark.parametrize("name", ["trna", "score.1"])
@pytest.mark.parametrize("source", ["chars", "2bit"])
def test_shards_of_one_assembled_batch(name, source, genome, monkeypatch):
    monkeypatch.setenv("GPUMOTIF_CHUNK_NT", "16384")
    chars, ro, ref = reference(name, genome, source)
    parts = []
    for lo, hi in shard.shard_ranges(int(ro[-1]), 3):
        ms = gpumotif.MotifSearch(helpers.load_plan(name))
        upload(ms, genome, source)
        ms.assemble_bed(genome[5])
        parts.append(ms.scan(lo, hi))
        ms.close()
    helpers.assert_same_hits(shard.merge_hits(parts), ref, f"{name}: three shards of one assembled batch")


def test_score_prescreen_and_one_strand(genome):
    chars, ro, ref = reference("score.1", genome, "chars")
    score = helpers.load_score("score.1")
    ms = gpumotif.MotifSearch(helpers.load_plan("score.1"))
    ms.set_score(score)
    want = ms.find_motif(chars, ro)
    rej = ms.stats().n_score_rejected
    want1 = ms.scan(strands=1)
    upload(ms, genome, "2bit")
    ms.assemble_bed(genome[5])
    got = ms.scan()
    got_rej = ms.stats().n_score_rejected
    got1 = ms.scan(strands=1)
    ms.close()
    helpers.assert_same_hits(got, want, "score.1 with the pre-screen")
    assert got_rej == rej and (rej > 0 or len(want) == len(ref))
    helpers.assert_same_hits(got1, want1, "score.1, sense strand only")
    assert (got1["comp"] == 0).all()


@pytest.mark.parametrize("source", ["chars", "device", "fastn", "2bit"])
def test_characters_back_equal_the_character_uploads(source, genome, monkeypatch):
    monkeypatch.setenv("GPUMOTIF_CHUNK_NT", "16384")
    chars, ro, ref = reference("trna", genome, source)
    ms = gpumotif.MotifSearch(helpers.load_plan("trna"))
    ms.find_motif(chars, ro)
    w_want, c_want = ms.hit_windows(40, 3000), ms.get_chars()
    keep = upload(ms, genome, source)
    ms.assemble_bed(genome[5])
    ms.scan()
    w_got, c_got = ms.hit_windows(40, 3000), ms.get_chars()
    part = ms.get_chars(7, 12345)
    with pytest.raises(gpumotif.GpuMotifError, match="no FASTA or FASTQ text"):
        ms.get_text(0, 1)
    ms.close()
    del keep
    assert len(w_want) > 0 and w_got.shape == w_want.shape and (w_got == w_want).all()
    assert c_got.tobytes() == c_want.tobytes() == chars.tobytes()
    assert part.tobytes() == chars[7:7 + 12345].tobytes()


def test_no_characters_after_a_host_packed_source(genome):
    chars, ro, ref = reference("trna", genome, "chars")
    ms = gpumotif.MotifSearch(helpers.load_plan("trna"))
    upload(ms, genome, "hostpack")
    ms.assemble_bed(genome[5])
    helpers.assert_same_hits(ms.scan(), ref, "assembled after a host-packed upload")
    for call in (lambda: ms.hit_windows(3, 4), lambda: ms.get_chars(0, 10)):
        with pytest.raises(gpumotif.GpuMotifError, match="no characters"):
            call()
    ms.close()


def random_assembly(rng, rec_off, n_rec):
    """Blocks in any order, overlapping, repeated and empty, over the batch rec_off, random strands"""
    blk, rec_blk = [], [0]
    for _ in range(n_rec):
        for _ in range(int(rng.integers(0, 6))):
            r = int(rng.integers(0, len(rec_off) - 1))
            a, b = int(rec_off[r]), int(rec_off[r + 1])
            s = int(rng.integers(a, b + 1))
            e = int(rng.integers(s, min(b, s + 400) + 1))
            blk += [(s, e)] * (1 + (rng.random() < 0.1))
        rec_blk.append(len(blk))
    strand = rng.integers(0, 2, size=n_rec).astype(np.uint8)
    return bed.Assembly(np.array(blk, dtype=np.int64).reshape(-1), rec_blk, strand, [""] * n_rec, rec_off)


@pytest.mark.parametrize("source", ["chars", "2bit"])
def test_assembling_an_assembled_batch_and_uploading_after(source, genome, monkeypatch):
    monkeypatch.setenv("GPUMOTIF_CHUNK_NT", "16384")
    ids, seq, off, tb, fasta, asm = genome
    chars, ro, ref = reference("trna", genome, source)
    second = random_assembly(np.random.default_rng(3), ro, 300)
    chars2, ro2 = second.assemble_chars(chars, ro)
    plan = helpers.load_plan("trna")
    ref2, _ = oracle_port.scan_db(plan, chars2, ro2, True)
    ms = gpumotif.MotifSearch(plan)
    upload(ms, genome, source)
    ms.assemble_bed(asm)
    ms.scan()
    ms.assemble_bed(second)
    assert ms.records()[0].tolist() == ro2.tolist()
    got = ms.scan()
    c_got = ms.get_chars()
    ms.upload(seq, off)  # an upload after an assembly
    after = ms.scan()
    ms.close()
    helpers.assert_same_hits(got, ref2, "an assembled batch assembled again")
    assert c_got.tobytes() == chars2.tobytes()
    assert len(ref2) > 0
    helpers.assert_same_hits(after, oracle_port.scan_db(plan, seq, off, True)[0], "an upload after an assembly")


def test_empty_tables_and_bytes_over_the_link(genome):
    ids, seq, off, tb, fasta, asm = genome
    ms = gpumotif.MotifSearch(helpers.load_plan("trna"))
    ms.upload(seq, off)
    ms.assemble(np.zeros(0, np.int64), [0], [])
    assert ms.records()[0].tolist() == [0] and ms.total_nt == 0 and len(ms.scan()) == 0
    ms.upload(seq, off)
    ms.assemble([5, 5, 9, 9], [0, 0, 2, 2], [1, 0, 1])  # empty blocks, empty records
    assert ms.records()[0].tolist() == [0, 0, 0, 0] and len(ms.scan()) == 0
    ms.upload(seq, off)
    ms.assemble_bed(asm)
    ms.scan()
    st = ms.stats()
    ms.close()
    n_seg = int(((asm.blk[1::2] - asm.blk[0::2]) > 0).sum())
    assert st.h2d_bytes == 8 * len(asm.rec_blk) + 8 * (2 * n_seg + 1)


def refusals(off):
    big = int(np.argmax(np.diff(off)))
    a, b = int(off[big]), int(off[big + 1])
    n = int(off[-1])
    ok = [a, a + 10]
    return [
        ("a NULL block table", (None, 1, [0, 1], [0], 1), "bad assembly table"),
        ("a NULL strand table", (ok, 1, [0, 1], None, 1), "bad assembly table"),
        ("n_rec < 0", (ok, 1, [0], [0], -1), "bad assembly table"),
        ("rec_blk[0] != 0", (ok, 1, [1, 1], [0], 1), r"rec_blk\[0\] must be 0"),
        ("rec_blk descending", (ok + ok, 2, [0, 2, 1], [0, 0], 2), "not ascending at 1"),
        ("rec_blk[n_rec] != n_blk", (ok + ok, 2, [0, 1], [0], 1), r"rec_blk\[1\] = 1, not n_blk = 2"),
        ("a block ending before it starts", ([a + 5, a + 4], 1, [0, 1], [0], 1), r"block 0 \[.*\) ends before it starts"),
        ("a block past the end", (ok + [n - 3, n + 1], 2, [0, 2], [0], 1), r"block 1 \[.*\) outside the .* held"),
        ("a negative block", ([-1, 3], 1, [0, 1], [0], 1), "outside"),
        ("a block across a record end", (ok + [b - 3, b + 2], 2, [0, 2], [1], 1),
         f"block 1 .* crosses the end of held record {big} "),
        ("a strand byte of 2", (ok, 1, [0, 1], [2], 1), r"strand\[0\] = 2"),
        ("a record over 2^31", ([a, b] * 15000, 15000, [0, 15000], [0], 1), "record 0 longer than 2"),
    ]


def raw_assemble(ms, blk, n_blk, rec_blk, strand, n_rec):
    arr = lambda x, t: None if x is None else np.ascontiguousarray(x, dtype=t)
    blk, rec_blk, strand = arr(blk, np.int64), arr(rec_blk, np.int64), arr(strand, np.uint8)
    ptr = lambda x: None if x is None else x.ctypes.data
    rc = gpumotif.lib().gm_db_assemble(ms._ctx, ptr(blk), n_blk, ptr(rec_blk), ptr(strand), n_rec)
    if rc != 0:
        raise gpumotif.GpuMotifError("gm_db_assemble: " + gpumotif._err())


def test_refusals_leave_the_held_batch(genome):
    ids, seq, off, tb, fasta, asm = genome
    plan = helpers.load_plan("trna")
    ref, _ = oracle_port.scan_db(plan, seq, off, True)
    ms = gpumotif.MotifSearch(plan)
    with pytest.raises(gpumotif.GpuMotifError, match="no database uploaded"):
        ms.assemble_bed(asm)
    ms.upload(seq, off)
    first = ms.scan()
    for what, args, msg in refusals(off):
        with pytest.raises(gpumotif.GpuMotifError, match=msg):
            raw_assemble(ms, *args)
        rec, hdr = ms.records()
        assert rec.tolist() == off.tolist() and ms.total_nt == int(off[-1]), what
        helpers.assert_same_hits(ms.hits(), first, f"candidates after refusing {what}")
    ms.scan_launch()
    with pytest.raises(gpumotif.GpuMotifError, match="a scan is in flight"):
        ms.assemble_bed(asm)
    ms.scan_finish()
    helpers.assert_same_hits(ms.hits(), ref, "the scan in flight during the refusal")
    assert ms.records()[0].tolist() == off.tolist()
    ms.close()
