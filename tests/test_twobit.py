"""GPU: the 2-bit upload (gm_db_upload_2bit / MotifSearch.upload_2bit, include/gpumotif.h).

The database is a .2bit file written by twobit.write_2bit: ragged records with N runs (at record
starts and ends, adjacent across a boundary), records that are N throughout, records of 0, 1, 3
and 5 nucleotides and one of 150 001.  The candidate stream after the 2-bit upload must equal the
oracle's over twobit.to_chars() and the character upload's of those characters -- with the default
chunks and with 16 Knt chunks (boundaries inside a byte and a record), from pinned and pageable
memory, always from the file's own bytes (the record headers between the records go along).
Also: sequences of uploads on one context, three shards of one upload, the score pre-screen, the
characters handed back (hit windows, get_chars), the bytes over the link, and refused tables."""
import numpy as np
import pytest

from rnamotif_b200 import gpumotif, synth, twobit
from oracle import oracle_port
import helpers
import shard

NAMES = ["trna", "ire", "score.1", "pk1", "qu+tr"]  # lite and full, helix, literal and chain sieves, two-stage plans


def make_db(seed=41):
    rng = np.random.default_rng(seed)
    lengths = [0, 1, 3, 5] + list(rng.integers(0, 6000, size=30)) + [150001, 120, 40, 2, 7000]
    ids, seq, off = synth.random_records(seed, lengths, planted=True)
    up = rng.random(len(seq)) < 0.2
    seq[up] -= 32  # mixed case: the search folds it
    for r in range(4, len(lengths)):
        a, b = int(off[r]), int(off[r + 1])
        if b - a > 50:
            k = int(rng.integers(1, 40))
            p = int(rng.integers(a, b - k))
            seq[p:p + k] = ord("N")
    seq[off[5]:off[5] + 9] = ord("n")          # at a record start
    seq[off[7] - 4:off[7]] = ord("N")          # at a record end ...
    seq[off[7]:off[7] + 6] = ord("N")          # ... and the next one's start: adjacent across the boundary
    big = lengths.index(150001)
    seq[off[big + 1]:off[big + 2]] = ord("n")  # records that are N throughout (120 and 40 nt)
    seq[off[big + 2]:off[big + 3]] = ord("N")
    f = twobit.write_2bit(ids, seq, off)
    tb = twobit.read_2bit(f)
    rec_off, _, _ = tb.tables()
    return f, tb, twobit.to_chars(tb), rec_off


@pytest.fixture(scope="module")
def db():
    return make_db()


_REF = {}


def reference(name, chars, rec_off):
    if name not in _REF:
        plan = helpers.load_plan(name)
        _REF[name] = oracle_port.scan_db(plan, chars, rec_off, bool(gpumotif.plan_field(plan, 8)))[0]
    return _REF[name]


def pinned_2bit(f):
    import torch
    buf = torch.empty(len(f), dtype=torch.uint8, pin_memory=True)
    return buf, twobit.read_2bit(f, out=buf.numpy())


@pytest.mark.gpu
@pytest.mark.parametrize("memory", ["pageable", "pinned"])
@pytest.mark.parametrize("chunk", ["default", "16384"])
@pytest.mark.parametrize("name", NAMES)
def test_2bit_upload_matches_oracle_and_character_upload(name, chunk, memory, db, monkeypatch):
    if chunk != "default":
        monkeypatch.setenv("GPUMOTIF_CHUNK_NT", chunk)  # many chunks: boundaries fall inside bytes and records
    f, tb, chars, rec_off = db
    ref = reference(name, chars, rec_off)
    keep = None
    if memory == "pinned":
        keep, tb = pinned_2bit(f)
    ms = gpumotif.MotifSearch(helpers.load_plan(name))
    by_chars = ms.find_motif(chars, rec_off)
    ms.upload_2bit(tb)
    first = ms.scan()
    again = ms.scan()                       # rescan of the same upload
    ms.close()
    del keep
    helpers.assert_same_hits(by_chars, ref, f"{name}: character upload")
    helpers.assert_same_hits(first, ref, f"{name}: 2-bit upload ({chunk}, {memory})")
    helpers.assert_same_hits(again, ref, f"{name}: 2-bit upload, rescan")
    assert len(ref) > 0 or name in ("ire", "qu+tr")  # ire's motif is rare: none in a database this small


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", ["default", "16384"])
def test_sequences_of_uploads(chunk, db, monkeypatch):
    if chunk != "default":
        monkeypatch.setenv("GPUMOTIF_CHUNK_NT", chunk)
    f, tb, chars, rec_off = db
    name = "trna"
    plan = helpers.load_plan(name)
    ref = reference(name, chars, rec_off)
    ms = gpumotif.MotifSearch(plan)
    ms.upload_2bit(tb)
    big = ms.scan()
    ms.upload_2bit(tb, 0, 6)                # a smaller batch over a larger one
    small = ms.scan()
    ms.upload_2bit(tb, 30, 36)              # a slice from the middle of the file
    mid = ms.scan()
    back = ms.find_motif(chars, rec_off)    # characters -> 2-bit -> characters on one context
    ms.upload_2bit(tb)
    again = ms.scan()
    ms.close()
    helpers.assert_same_hits(big, ref, "2-bit upload")
    n6 = int(rec_off[6])
    both = bool(gpumotif.plan_field(plan, 8))
    ref_small, _ = oracle_port.scan_db(plan, chars[:n6], rec_off[:7], both)
    helpers.assert_same_hits(small, ref_small, "smaller 2-bit batch")
    ref_mid, _ = oracle_port.scan_db(plan, chars[rec_off[30]:rec_off[36]], rec_off[30:37] - rec_off[30], both)
    helpers.assert_same_hits(mid, ref_mid, "2-bit slice of records 30..35")
    helpers.assert_same_hits(back, ref, "character upload after a 2-bit one")
    helpers.assert_same_hits(again, ref, "2-bit upload after a character one")


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["trna", "score.1"])
def test_shards_of_one_2bit_upload(name, db, monkeypatch):
    monkeypatch.setenv("GPUMOTIF_CHUNK_NT", "16384")
    f, tb, chars, rec_off = db
    plan = helpers.load_plan(name)
    ref = reference(name, chars, rec_off)
    parts = []
    for lo, hi in shard.shard_ranges(int(rec_off[-1]), 3):
        ms = gpumotif.MotifSearch(plan)
        ms.upload_2bit(tb)
        parts.append(ms.scan(lo, hi))
        ms.close()
    helpers.assert_same_hits(shard.merge_hits(parts), ref, f"{name}: three shards of one 2-bit upload")


@pytest.mark.gpu
def test_score_prescreen_after_2bit_upload(db):
    f, tb, chars, rec_off = db
    score = helpers.load_score("score.1")
    assert score is not None and helpers.score_present(score)
    ms = gpumotif.MotifSearch(helpers.load_plan("score.1"))
    ms.set_score(score)
    by_chars = ms.find_motif(chars, rec_off)
    rej_chars = ms.stats().n_score_rejected
    ms.upload_2bit(tb)
    by_2bit = ms.scan()
    rej_2bit = ms.stats().n_score_rejected
    ms.close()
    helpers.assert_same_hits(by_2bit, by_chars, "score.1 with the pre-screen")
    assert rej_2bit == rej_chars
    assert rej_chars > 0 or len(by_chars) == len(reference("score.1", chars, rec_off))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["trna", "score.1"])
def test_characters_back_after_2bit_upload(name, db, monkeypatch):
    monkeypatch.setenv("GPUMOTIF_CHUNK_NT", "16384")
    f, tb, chars, rec_off = db
    ms = gpumotif.MotifSearch(helpers.load_plan(name))
    ms.find_motif(chars, rec_off)
    w_chars = ms.hit_windows(40, 5000)      # windows run past record ends on both strands
    c_chars = ms.get_chars()
    part_chars = ms.get_chars(7, 12345)
    ms.upload_2bit(tb)
    hits = ms.scan()
    w_2bit = ms.hit_windows(40, 5000)
    c_2bit = ms.get_chars()
    part_2bit = ms.get_chars(7, 12345)
    ms.close()
    assert len(hits) > 0 and (hits["comp"] == 1).any()
    assert w_2bit.shape == w_chars.shape and (w_2bit == w_chars).all()
    assert c_2bit.tobytes() == c_chars.tobytes() == chars.tobytes()
    assert part_2bit.tobytes() == part_chars.tobytes()


@pytest.mark.gpu
def test_bytes_over_the_link(db):
    f, tb, chars, rec_off = db
    n_rec = len(rec_off) - 1
    _, dna_off, nblk = tb.tables()
    n_nblk = len(nblk) // 2
    total = int(rec_off[-1])
    span = int(dna_off[-1] + (tb.sizes[-1] + 3) // 4 - dna_off[0])
    packed = int(((tb.sizes + 3) // 4).sum())
    headers = span - packed  # the record headers between the records' bases
    ms = gpumotif.MotifSearch(helpers.load_plan("trna"))
    ms.upload_2bit(tb)
    ms.scan()
    st = ms.stats()
    ms.close()
    assert st.h2d_bytes == span + 8 * (n_rec + 1) + 8 * n_rec + 16 * n_nblk
    # a quarter byte per nucleotide, plus the headers, the records' last partial bytes and the tables
    assert st.h2d_bytes <= total / 4 + headers + 0.75 * n_rec + 8 * (2 * n_rec + 2 * n_nblk + 2)


@pytest.mark.gpu
def test_bad_tables_are_refused_and_the_context_stays_usable(db):
    f, tb, chars, rec_off = db
    _, dna_off, nblk = tb.tables()
    data = np.ascontiguousarray(tb.data)
    ref = reference("trna", chars, rec_off)
    ms = gpumotif.MotifSearch(helpers.load_plan("trna"))
    ms.upload_2bit(tb)
    ms.scan()
    down = dna_off.copy()
    down[10], down[11] = down[11], down[10]
    over = nblk.copy()
    over[2] = over[1] - 1  # the second range starts inside the first
    past = dna_off.copy()
    past[-1] = data.size - 1
    back = nblk.copy()
    back[1] = back[0] - 1
    cases = [("descending dna_off", down, nblk, "not ascending"), ("overlapping N ranges", dna_off, over, "overlaps"),
             ("dna_off past n_bytes", past, nblk, "run past"), ("an N range ending before its start", dna_off, back, "ends before")]
    for what, d, nb, msg in cases:
        with pytest.raises(gpumotif.GpuMotifError, match=msg):
            ms.upload_2bit_ptr(data.ctypes.data, data.size, d, rec_off, nb)
        helpers.assert_same_hits(ms.scan(), ref, f"the previous upload after refusing {what}")
    ms.upload_2bit(tb)
    helpers.assert_same_hits(ms.scan(), ref, "a 2-bit upload after the refusals")
    ms.close()


@pytest.mark.gpu
def test_compact_buffer_without_headers(db):
    """The raw-pointer form over bases packed back to back (no file around them)."""
    f, tb, chars, rec_off = db
    _, dna_off, nblk = tb.tables()
    nb = (tb.sizes + 3) // 4
    compact = np.concatenate([tb.data[o:o + k] for o, k in zip(dna_off, nb)])
    coff = np.concatenate([[0], np.cumsum(nb)[:-1]]).astype(np.int64)
    ms = gpumotif.MotifSearch(helpers.load_plan("trna"))
    ms.upload_2bit_ptr(compact.ctypes.data, compact.size, coff, rec_off, nblk)
    hits = ms.scan()
    st = ms.stats()
    ms.close()
    helpers.assert_same_hits(hits, reference("trna", chars, rec_off), "compact 2-bit buffer")
    assert st.h2d_bytes == compact.size + 8 * (2 * len(nb) + 1) + 8 * len(nblk)
