"""CPU: low-quality masking of the FASTQ uploads (gm_ctx_set_min_quality) -- the reference,
fastq.parse_fastq(min_qual=...), on hand-written bytes, and the masking kernel's sixteen-byte compare
(rnamotif_b200/csrc/gm_fastq.h, built for the host by tests/csrc/fastq_mask_check.cpp with
AddressSanitizer and UndefinedBehaviorSanitizer) against its per-byte definition."""
import os
import re
import subprocess

import numpy as np
import pytest

from rnamotif_b200 import fastq
import helpers


def seq_of(text, **kw):
    return fastq.parse_fastq(text, **kw)[1].tobytes()


def test_threshold_is_inclusive():
    # '5' = Q20 at offset 33: kept at min_qual 20, masked at 21; '4' = Q19 is masked at 20
    text = b"@r\nACGUN.\n+\n545!I5\n"
    assert seq_of(text) == b"acgtn."
    assert seq_of(text, min_qual=20) == b"angnn."
    assert seq_of(text, min_qual=21) == b"nnnnnn"
    assert seq_of(text, min_qual=1) == b"acgnn."  # '!' = Q0
    assert seq_of(text, min_qual=93) == b"nnnnnn"
    assert seq_of(text, min_qual=0) == seq_of(text)


def test_defaults_return_what_they_returned():
    text = (b"@r1 first read\nACGU\n+r1 first read\n@+II\n"
            b"@r2\n\n+\n\n"
            b"@r3\r\nnA.g\r\n+\r\n+@@I\r\n"
            b"@r4\nT\n+\nI")
    a, b = fastq.parse_fastq(text), fastq.parse_fastq(text, 0, 64)
    for x, y in zip(a[1:], b[1:]):
        assert (x == y).all()
    assert a[0] == b[0] == ["r1", "r2", "r3", "r4"]
    # Q0 bytes below offset 64 are not refused with masking off
    assert seq_of(b"@r\nAC\n+\n!!\n", qual_offset=64) == b"ac"


def test_crlf_empty_reads_and_no_last_line_end():
    text = (b"@r1\r\nACGT\r\n+\r\n#I#I\r\n"
            b"@r2\r\n\r\n+\r\n\r\n"
            b"@r3\r\nGG\r\n+\r\nI#")
    ids, seq, off, hdr = fastq.parse_fastq(text, min_qual=20)
    assert seq.tobytes() == b"ncntgn" and list(off) == [0, 4, 4, 6]
    assert list(hdr) == [0, text.index(b"@r2"), text.index(b"@r3"), len(text)]
    assert seq_of(text[:-1] + b"I\r\n", min_qual=20) == b"ncntgg"
    # the '\r' before a '\n' is no quality byte, and one that ends the text is cut with the line end
    assert seq_of(b"@r\nAC\n+\nI#\r", min_qual=20) == b"an"


def test_offset_64():
    text = b"@r\nACGTA\n+\n@ST^h\n"  # Q0, Q19, Q20, Q30, Q40 at offset 64
    assert seq_of(text, min_qual=20, qual_offset=64) == b"nngta"
    assert seq_of(text, min_qual=62, qual_offset=64) == b"nnnnn"


def test_arguments():
    for mq, off in ((-1, 33), (94, 33), (63, 64), (20, 32), (20, 0)):
        with pytest.raises(ValueError):
            fastq.parse_fastq(b"", mq, off)
    assert fastq.parse_fastq(b"", 93, 33)[3].tolist() == [0]
    assert fastq.parse_fastq(b"", 62, 64)[3].tolist() == [0]


def range_cases():
    """(what, text, min_qual, qual_offset, record, message); the texts whose message is a quality
    byte's are accepted with masking off"""
    good = b"@a\nACGT\n+\nIIII\n@b\nAC\n+\nII\n@c\nGG\n+\nII\n"
    return [
        ("Phred+33 read as 64", good.replace(b"@b\nAC\n+\nII", b"@b\nAC\n+\nI5"), 20, 64, 1,
         "quality byte 53 is outside [64, 126]"),
        ("space", good.replace(b"IIII", b"II I"), 1, 33, 0, "quality byte 32 is outside [33, 126]"),
        ("DEL", good.replace(b"@c\nGG\n+\nII", b"@c\nGG\n+\nI\x7f"), 1, 33, 2, "quality byte 127 is outside [33, 126]"),
        ("high byte", good.replace(b"IIII", b"\xffIII"), 30, 33, 0, "quality byte 255 is outside [33, 126]"),
        ("the first bad byte of the record", good.replace(b"IIII", b"I\x80 I"), 30, 33, 0,
         "quality byte 128 is outside [33, 126]"),
        ("the first record", good.replace(b"IIII", b"II I").replace(b"@c\nGG\n+\nII", b"@c\nGG\n+\n\x01I"), 1, 33, 0,
         "quality byte 32"),
        ("a format error in an earlier record first", good.replace(b"@b\nAC\n+\nII", b"@b\nAC\n-\nII")
         .replace(b"@c\nGG\n+\nII", b"@c\nGG\n+\n I"), 1, 33, 1, "line 7 does not start with '+'"),
        ("a format error in the same record first", good.replace(b"@b\nAC\n+\nII", b"@b\nAC\n+\n I I"), 1, 33, 1,
         "quality string is not as long as its read"),
        ("a format error ('@' missing) in the same record", good.replace(b"@b\nAC\n+\nII", b"b\nAC\n+\n I"), 1, 33, 1,
         "line 5 does not start with '@'"),
        ("the range error in an earlier record first", good.replace(b"IIII", b"I I ")
         .replace(b"@c\nGG\n+\nII", b"@c\nGG\n+\nIII"), 1, 33, 0, "quality byte 32"),
        ("a later format error", good.replace(b"IIII", b"I I ").replace(b"@b\nAC", b"b\nAC"), 1, 33, 0,
         "quality byte 32"),
        ("CR LF", good.replace(b"\n", b"\r\n").replace(b"IIII", b"III\x7f"), 1, 33, 0, "quality byte 127"),
    ], good


def test_range_refusals():
    cases, good = range_cases()
    at = {r: good.index(b"@" + bytes([ord("a") + r])) for r in range(3)}
    for what, text, mq, off, rec, msg in cases:
        with pytest.raises(fastq.FastqError, match=re.escape(msg)) as e:
            fastq.parse_fastq(text, mq, off)
        assert e.value.record == rec, what
        assert e.value.offset == at[rec], what
        assert f"FASTQ record {rec} at byte {at[rec]}: " in str(e.value), what
        if "format" not in what and "earlier" not in what:
            fastq.parse_fastq(text)


@pytest.fixture(scope="module")
def checker(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("fastq_mask") / "fastq_mask_check")
    subprocess.run(["g++", "-O1", "-g", "-std=c++17", "-fsanitize=address,undefined", "-fno-sanitize-recover=all",
                    "-I", os.path.join(helpers.ROOT, "rnamotif_b200", "csrc"),
                    os.path.join(helpers.HERE, "csrc", "fastq_mask_check.cpp"), "-o", exe], check=True)
    return exe


def test_sixteen_byte_compare_matches_per_byte_definition(checker):
    env = dict(os.environ, ASAN_OPTIONS="detect_leaks=0")
    r = subprocess.run([checker], capture_output=True, text=True, env=env)
    assert r.returncode == 0 and r.stdout.strip() == "ok", r.stdout + r.stderr
