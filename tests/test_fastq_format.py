"""CPU: the FASTQ reference reader and writer (rnamotif_b200/fastq.py), the seeded reads of
synth.random_reads, and the FASTQ reader's scan operator (rnamotif_b200/csrc/gm_fastq.h, built for
the host by tests/csrc/fastq_check.cpp with AddressSanitizer and UndefinedBehaviorSanitizer).

The operator and the kernels' sixteen-byte classifier must equal the per-byte definition for every
entry phase, over FASTQ texts and random texts cut at random points, between '\\r' and '\\n' and
at the start of every line."""
import os
import re
import subprocess

import numpy as np
import pytest

from rnamotif_b200 import fastq, synth
import helpers


def test_writer_against_hand_written_bytes():
    seq = np.frombuffer(b"ACGTnacgu.", dtype=np.uint8)
    off = np.array([0, 4, 4, 10])
    assert fastq.write_fastq(["r1", "r2 desc", "r3"], seq, off, qual=[b"IIII", b"", b"@+!#$%"]) == (
        b"@r1\nACGT\n+\nIIII\n"
        b"@r2 desc\n\n+\n\n"
        b"@r3\nnacgu.\n+\n@+!#$%\n")
    assert fastq.write_fastq(["a"], seq, [0, 2], crlf=True) == b"@a\r\nAC\r\n+\r\nII\r\n"
    assert fastq.write_fastq([], seq, [0]) == b""


def test_parser_on_hand_written_bytes():
    text = (b"@r1 first read\nACGU\n+r1 first read\n@+II\n"
            b"@r2\n\n+\n\n"
            b"@r3\r\nnA.g\r\n+\r\n+@@I\r\n"
            b"@r4\nT\n+\nI")
    ids, seq, off, hdr = fastq.parse_fastq(text)
    assert ids == ["r1", "r2", "r3", "r4"]
    assert seq.tobytes() == b"acgtna.gt"
    assert list(off) == [0, 4, 4, 8, 9]
    assert list(hdr) == [0, text.index(b"@r2"), text.index(b"@r3"), text.index(b"@r4"), len(text)]
    assert fastq.parse_fastq(b"")[3].tolist() == [0]


def reads(seed=5, n=300, crlf=False, weird_qual=True):
    rng = np.random.default_rng(seed)
    lengths = rng.integers(0, 401, size=n)
    lengths[:4] = [0, 1, 0, 150]
    ids, seq, off = synth.random_reads(seed, lengths)
    qual = []
    for r in range(n):
        q = rng.integers(33, 74, size=int(lengths[r]), dtype=np.uint8)
        if weird_qual and len(q) and r % 3 == 0:
            q[0] = ord("@") if r % 2 else ord("+")  # quality strings that look like header lines
        qual.append(q.tobytes())
    return ids, seq, off, qual, fastq.write_fastq(ids, seq, off, qual, crlf)


@pytest.mark.parametrize("crlf", [False, True])
@pytest.mark.parametrize("last_newline", [True, False])
def test_round_trip(crlf, last_newline):
    ids, seq, off, qual, text = reads(crlf=crlf)
    if not last_newline:
        text = text[:-2] if crlf else text[:-1]
    ids2, seq2, off2, hdr2 = fastq.parse_fastq(text)
    assert ids2 == ids and (off2 == off).all()
    assert seq2.tobytes() == fastq._LOWER[seq].tobytes()
    assert b"." in seq2.tobytes() and b"n" in seq2.tobytes()
    assert all(text[h:h + 1] == b"@" for h in hdr2[:-1]) and hdr2[-1] == len(text)
    assert fastq.write_fastq(ids2, seq2, off2, qual, crlf) == fastq.write_fastq(ids, fastq._LOWER[seq], off, qual, crlf)


def test_seeded_reads_are_seeded():
    a = synth.random_reads(7, [150] * 1000)
    b = synth.random_reads(7, [150] * 1000)
    c = synth.random_reads(8, [150] * 1000)
    assert (a[1] == b[1]).all() and not (a[1] == c[1]).all()
    assert a[2][-1] == 150000 and a[0][:2] == ["read0", "read1"]


def refusal_cases():
    """(what, text, record, message) for every refusal; record None = refused on the host."""
    good = b"@a\nACGT\n+\nIIII\n@b\nAC\n+\nII\n"
    b_at = good.index(b"@b")
    return [
        ("no '@' first", b"ACGT\n" + good, None, "does not begin with '@'"),
        ("line 4k not '@'", good.replace(b"@b", b"b"), 1, "line 5 does not start with '@'"),
        ("line 4k+2 not '+'", good.replace(b"AC\n+\nII", b"AC\n-\nII"), 1, "line 7 does not start with '+'"),
        ("multi-line read", b"@a\nACGT\nACGT\n+\nIIIIIIII\n", 0, "line 3 does not start with '+'"),
        ("quality too short", good.replace(b"IIII", b"III"), 0, "quality string is not as long"),
        ("quality too long", good[:-1] + b"I\n", 1, "quality string is not as long"),
        ("two lines", good + b"@c\nAC\n", 2, "fewer than four lines"),
        ("three lines", good + b"@c\nAC\n+\n", 2, "fewer than four lines"),
        ("one line", good + b"@c", 2, "fewer than four lines"),
        ("blank line after", good + b"\n", 2, "line 9 does not start with '@'"),
        ("empty '+' line", good.replace(b"AC\n+\nII", b"AC\n\nII"), 1, "line 7 does not start with '+'"),
        ("CR before CR LF", good[:-4] + b"\nII\r\r\n", 1, "quality string is not as long"),
    ], good


def test_every_refusal():
    cases, good = refusal_cases()
    at = {0: 0, 1: good.index(b"@b"), 2: len(good)}  # where each record's '@' is (or should be)
    for what, text, rec, msg in cases:
        with pytest.raises(fastq.FastqError, match=re.escape(msg)) as e:
            fastq.parse_fastq(text)
        assert e.value.record == rec, what
        if rec is not None:
            assert e.value.offset == at[rec], what
            assert f"record {rec} at byte {at[rec]}:" in str(e.value), what


def test_the_first_failing_record_is_named():
    ids, seq, off, qual, text = reads(n=50, weird_qual=False)
    _, _, _, hdr = fastq.parse_fastq(text)
    lines = text.split(b"\n")
    lines[4 * 30 + 2] = b"x"   # record 30's '+' line
    lines[4 * 12 + 3] += b"I"  # record 12's quality string
    with pytest.raises(fastq.FastqError, match=f"record 12 at byte {hdr[12]}:"):
        fastq.parse_fastq(b"\n".join(lines))


def test_trimmed_length():
    assert [fastq.trimmed_length(t) for t in (b"", b"\n", b"@\r\n", b"@\n\n", b"@\r", b"@a")] == [0, 0, 1, 2, 1, 2]


@pytest.fixture(scope="module")
def checker(tmp_path_factory):
    d = tmp_path_factory.mktemp("fastq")
    exe = str(d / "fastq_check")
    subprocess.run(["g++", "-O1", "-g", "-std=c++17", "-fsanitize=address,undefined", "-fno-sanitize-recover=all",
                    "-I", os.path.join(helpers.ROOT, "rnamotif_b200", "csrc"),
                    os.path.join(helpers.HERE, "csrc", "fastq_check.cpp"), "-o", exe], check=True)
    return exe, d


def test_scan_operator_matches_per_byte_definition(checker):
    exe, d = checker
    files = []
    for crlf in (False, True):
        *_, text = reads(seed=11, n=120, crlf=crlf)
        p = d / f"reads_{int(crlf)}.fq"
        p.write_bytes(text)
        files.append(str(p))
    cases, _ = refusal_cases()
    p = d / "refused.fq"  # texts the reader refuses are summarised all the same
    p.write_bytes(b"".join(t for _, t, _, _ in cases))
    files.append(str(p))
    env = dict(os.environ, ASAN_OPTIONS="detect_leaks=0")
    r = subprocess.run([exe] + files, capture_output=True, text=True, env=env)
    assert r.returncode == 0 and r.stdout.strip() == "ok", r.stdout + r.stderr
