"""CPU: the BED reader (rnamotif_b200/bed.py) that builds gm_db_assemble's tables, its host reference
(Assembly.assemble_chars) and position map (Assembly.to_source), the seeded BED12 writer
(synth.random_transcripts), and the 16-nucleotide gather of the device's assembly
(rnamotif_b200/csrc/gm_assemble.h, built for the host by tests/csrc/assemble_check.cpp with
AddressSanitizer and UndefinedBehaviorSanitizer) against its per-nucleotide definition."""
import os
import subprocess

import numpy as np
import pytest

from rnamotif_b200 import bed, synth
import helpers

NAMES = ["chrA", "chrB", "chrC"]
OFF = np.array([0, 100, 100, 160], dtype=np.int64)  # chrB is empty
COMP = {ord("a"): ord("t"), ord("c"): ord("g"), ord("g"): ord("c"), ord("t"): ord("a")}


def tables(a):
    return a.blk.tolist(), a.rec_blk.tolist(), a.strand.tolist(), a.names


def test_bed3_bed6_bed12_lines():
    text = ("track name=x\nbrowser position chrA:1-10\n# comment\n\n"
            "chrA\t10\t20\n"
            "chrC 5 9 r6 0 -\n"
            "chrC\t0\t60\tr6dot\t0\t.\n"
            "chrA\t30\t90\ttx\t0\t+\t35\t80\t0\t3\t10,5,20,\t0,20,40,\n"
            "chrA\t30\t90\ttxm\t0\t-\t30\t30\t0\t2\t1,1\t0,59\n"
            "chrA\t0\t0\tempty\n")
    a = bed.read_bed(text, NAMES, OFF)
    assert tables(a) == ([10, 20, 105, 109, 100, 160, 30, 40, 50, 55, 70, 90, 30, 31, 89, 90, 0, 0], [0, 1, 2, 3, 6, 8, 9],
                         [0, 1, 0, 0, 1, 0], ["chrA:10-20", "r6", "r6dot", "tx", "txm", "empty"])
    assert a.rec_off_new().tolist() == [0, 10, 14, 74, 109, 111, 111]
    assert bed.read_bed(text.encode(), NAMES, OFF).blk.tolist() == a.blk.tolist()


def test_parts_of_one_coding_line_on_each_strand():
    for s in "+-":
        line = f"chrA\t30\t90\ttx\t0\t{s}\t35\t80\t0\t3\t10,5,20,\t0,20,40,\n"
        part = {p: bed.read_bed(line, NAMES, OFF, p).blk.tolist() for p in bed.PARTS}
        assert part["exons"] == [30, 40, 50, 55, 70, 90]
        assert part["cds"] == [35, 40, 50, 55, 70, 80]
        low, high = [30, 35], [80, 90]
        assert (part["utr5"], part["utr3"]) == ((low, high) if s == "+" else (high, low))
    # thickStart == thickEnd: no cds and no UTRs, but a record for the line all the same
    for p in ("cds", "utr5", "utr3"):
        a = bed.read_bed("chrA\t30\t90\tnc\t0\t-\t50\t50\t0\t1\t60,\t0,\n", NAMES, OFF, p)
        assert len(a) == 1 and a.rec_blk.tolist() == [0, 0]
    # no thick columns: all of it is cds
    assert bed.read_bed("chrA 3 9 x 0 -\n", NAMES, OFF, "cds").blk.tolist() == [3, 9]
    assert bed.read_bed("chrA 3 9 x 0 -\n", NAMES, OFF, "utr3").blk.tolist() == []
    with pytest.raises(ValueError):
        bed.read_bed("", NAMES, OFF, "introns")


@pytest.mark.parametrize("line,msg", [
    ("chrZ\t0\t10", "unknown chromosome 'chrZ'"),
    ("chrA\t0\t101", "chromEnd 101 past the end of chrA"),
    ("chrB\t0\t1", "past the end of chrB"),
    ("chrA\t10\t5", "do not make a range"),
    ("chrA\t0", "fewer than 3 columns"),
    ("chrA\tx\t5", "not an integer"),
    ("chrA\t0\t50\tt\t0\t+\t0\t50\t0\t2\t10,10,\t20,0,", "block 1 at 0 is out of order or overlaps block 0"),
    ("chrA\t0\t50\tt\t0\t+\t0\t50\t0\t2\t10,10,\t0,5,", "block 1 at 5 is out of order or overlaps"),
    ("chrA\t10\t50\tt\t0\t+\t0\t50\t0\t2\t10,11,\t0,30,", r"block 1 \[40, 51\) outside \[10, 50\)"),
    ("chrA\t10\t50\tt\t0\t+\t0\t50\t0\t1\t10,\t-1,", "block 0 .* outside"),
    ("chrA\t0\t50\tt\t0\t+\t0\t50\t0\t3\t10,10,\t0,20,", "blockCount 3 with 2 sizes and 2 starts"),
    ("chrA\t0\t50\tt\t0\t+\t0\t50\t0\t2\t10,10,\t0,", "blockCount 2 with 2 sizes and 1 starts"),
    ("chrA\t0\t50\tt\t0\t+\t0\t50\t0\t2\t10,x,\t0,20,", "not a list of integers"),
])
def test_bed_errors_name_the_line(line, msg):
    with pytest.raises(bed.BedError, match=msg) as e:
        bed.read_bed("# header\nchrA\t0\t5\n" + line + "\n", NAMES, OFF)
    assert e.value.line == 3 and str(e.value).startswith("BED line 3: ")


def per_base(text, names, rec_off, chars, part):
    """The assembled records from the definition: every exonic base of a line, kept by a per-base test
    of `part`, in ascending order; on '-' reversed and complemented (a c g t n)."""
    fold = bed._FOLD[np.asarray(chars, dtype=np.uint8)]
    out, offs = [], [0]
    for raw in text.splitlines():
        f = raw.split()
        c = names.index(f[0])
        cs, ts, te = int(f[1]), int(f[6]), int(f[7])
        minus = f[5] == "-"
        bases = sorted({cs + int(s) + i for s, z in zip(f[11].rstrip(",").split(","), f[10].rstrip(",").split(","))
                        for i in range(int(z))})
        keep = {
            "exons": lambda p: True,
            "cds": lambda p: ts <= p < te,
            "utr5": lambda p: ts < te and (p < ts if not minus else p >= te),
            "utr3": lambda p: ts < te and (p >= te if not minus else p < ts),
        }[part]
        s = [int(fold[rec_off[c] + p]) for p in bases if keep(p)]
        if minus:
            s = [COMP.get(x, ord("n")) for x in s[::-1]]
        out += s
        offs.append(len(out))
    return np.array(out, dtype=np.uint8), np.array(offs, dtype=np.int64)


@pytest.fixture(scope="module")
def genome():
    ids, seq, off = synth.random_records(23, [3000, 0, 1, 2500, 700, 4000], iupac_rate=0.05)
    up = np.random.default_rng(1).random(len(seq)) < 0.3
    seq[up] = np.frombuffer(bytes(seq[up]).upper(), dtype=np.uint8)
    text = synth.random_transcripts(4, ids, np.diff(off), 300, exon=40, first=60, last=120, intron=150, utr5=30,
                                    utr3=60, p_one=0.1, p_edge=0.05)
    return ids, seq, off, text


@pytest.mark.parametrize("part", bed.PARTS)
def test_assemble_chars_matches_per_base_definition(part, genome):
    ids, seq, off, text = genome
    a = bed.read_bed(text, ids, off, part)
    got, ro = a.assemble_chars(seq, off)
    want, wro = per_base(text, ids, off, seq, part)
    assert ro.tolist() == wro.tolist()
    assert got.tobytes() == want.tobytes()
    assert len(a) == len(text.splitlines()) and a.names == [ln.split()[3] for ln in text.splitlines()]


@pytest.mark.parametrize("part", ["exons", "utr5"])
def test_to_source_round_trips(part, genome):
    ids, seq, off, text = genome
    a = bed.read_bed(text, ids, off, part)
    chars, ro = a.assemble_chars(seq, off)
    rec = np.repeat(np.arange(len(a)), np.diff(ro))
    pos = np.arange(len(chars)) - ro[rec]
    held, at = a.to_source(rec, pos)
    src = bed._FOLD[seq[off[held] + at]]
    minus = a.strand[rec] == 1
    comp = bed._COMP[src]
    assert (np.where(minus, comp, src) == chars).all()
    assert ((at >= 0) & (at < off[held + 1] - off[held])).all()
    with pytest.raises(IndexError):
        a.to_source([0], [int(ro[1] - ro[0])])


def test_assemble_chars_refuses_another_record_table(genome):
    ids, seq, off, text = genome
    with pytest.raises(ValueError, match="record table"):
        bed.read_bed(text, ids, off).assemble_chars(seq, off + 1)


def test_random_transcripts_cover_what_they_promise(genome):
    ids, seq, off, text = genome
    sizes = np.diff(off)
    lines = [ln.split("\t") for ln in text.splitlines()]
    assert text == synth.random_transcripts(4, ids, sizes, 300, exon=40, first=60, last=120, intron=150, utr5=30,
                                            utr3=60, p_one=0.1, p_edge=0.05)  # seeded
    strands = {f[5] for f in lines}
    assert strands == {"+", "-"}
    exons = [[(int(f[1]) + int(s), int(f[1]) + int(s) + int(z)) for s, z in zip(f[11].rstrip(",").split(","),
                                                                                 f[10].rstrip(",").split(","))]
             for f in lines]
    flat = [e for ex in exons for e in ex]
    assert any(len(ex) > 3 for ex, f in zip(exons, lines) if f[5] == "-")
    assert any(e - s == 1 for s, e in flat)
    assert {s % 2 for s, e in flat} == {0, 1}
    assert len(flat) > len(set(flat))  # exons shared across isoforms
    by_start, by_end = {}, {}
    for s, e in flat:
        by_start.setdefault(s, set()).add(e)
        by_end.setdefault(e, set()).add(s)
    # overlapping, not equal: an isoform's exon with one end moved
    assert any(len(v) > 1 for v in by_start.values()) and any(len(v) > 1 for v in by_end.values())
    assert any(f[6] == f[7] for f in lines) and any(f[6] != f[7] for f in lines)
    assert any(int(f[1]) == 0 for f in lines)
    assert any(int(f[2]) == sizes[ids.index(f[0])] for f in lines)
    bed.read_bed(text, ids, off)  # and every line is valid


@pytest.fixture(scope="module")
def checker(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("assemble") / "assemble_check")
    subprocess.run(["g++", "-O1", "-g", "-std=c++17", "-fsanitize=address,undefined", "-fno-sanitize-recover=all",
                    "-I", os.path.join(helpers.ROOT, "rnamotif_b200", "csrc"),
                    os.path.join(helpers.HERE, "csrc", "assemble_check.cpp"), "-o", exe], check=True)
    return exe


def test_sixteen_nucleotide_gather_matches_per_nucleotide_definition(checker):
    env = dict(os.environ, ASAN_OPTIONS="detect_leaks=0")
    r = subprocess.run([checker], capture_output=True, text=True, env=env)
    assert r.returncode == 0 and r.stdout.strip() == "ok", r.stdout + r.stderr
