"""CPU: the .2bit reader and writer (rnamotif_b200/twobit.py) and the 16-nucleotide expansion of the
device's 2-bit upload (rnamotif_b200/csrc/gm_twobit.h, compiled for the host).

The writer is checked against bytes written out from the format's definition, not only by a round
trip; the round trips cover ragged and empty records, N runs at record ends and across record
boundaries, mixed case, both byte orders and both versions, and the GenBank sample records."""
import os
import struct
import subprocess

import numpy as np
import pytest

from rnamotif_b200 import twobit, synth
import helpers

# one record "s" = ACGTA, little-endian, version 0
ACGTA = bytes.fromhex("4327411A" "00000000" "01000000" "00000000"
                      "01" "73" "16000000"
                      "05000000" "00000000" "00000000" "00000000"
                      "9C80")


def fold(seq):
    """What to_chars must give back: lower case, u -> t, anything but a/c/g/t/u -> n."""
    s = np.asarray(seq, dtype=np.uint8) | 0x20
    s = np.where(s == ord("u"), ord("t"), s).astype(np.uint8)
    ok = np.isin(s, np.frombuffer(b"acgt", dtype=np.uint8))
    return np.where(ok, s, ord("n")).astype(np.uint8)


def roundtrip(ids, seq, off, **kw):
    tb = twobit.read_2bit(twobit.write_2bit(ids, seq, off, **kw))
    assert tb.names == list(ids)
    assert (tb.sizes == np.diff(off)).all()
    got = twobit.to_chars(tb)
    want = fold(seq)
    assert got.tobytes() == want.tobytes()
    return tb


def test_golden_bytes_acgta():
    assert twobit.write_2bit(["s"], b"ACGTA", [0, 5]) == ACGTA
    tb = twobit.read_2bit(ACGTA)
    assert tb.names == ["s"] and list(tb.sizes) == [5] and list(tb.dna_off) == [38] and tb.version == 0
    assert twobit.to_chars(tb).tobytes() == b"acgta"


def test_golden_packed_bytes():
    for s, byte in ((b"TCAG", 0x1B), (b"GGGG", 0xFF)):
        f = twobit.write_2bit(["x"], s, [0, 4])
        assert f[-1] == byte and len(f) == 16 + 1 + 1 + 4 + 16 + 1
        assert twobit.to_chars(twobit.read_2bit(f)).tobytes() == s.lower()


def test_big_endian_and_version_1_headers():
    f = twobit.write_2bit(["s"], b"ACGTA", [0, 5], byteswap=True)
    assert f[:4] == bytes.fromhex("1A412743") and f[16:22] == b"\x01s\x00\x00\x00\x16"
    assert twobit.read_2bit(f).byteswapped
    f1 = twobit.write_2bit(["s"], b"ACGTA", [0, 5], version=1)
    assert f1[4:8] == b"\x01\x00\x00\x00" and f1[18:26] == struct.pack("<Q", 26)
    assert twobit.to_chars(twobit.read_2bit(f1)).tobytes() == b"acgta"


@pytest.mark.parametrize("byteswap", [False, True])
@pytest.mark.parametrize("version", [0, 1])
def test_roundtrip_ragged_records(byteswap, version):
    rng = np.random.default_rng(5 + version + 2 * byteswap)
    lengths = list(range(10)) + [150001] + list(rng.integers(0, 40, size=30))
    ids, seq, off = synth.random_records(9, lengths, planted=True, iupac_rate=0.01)
    # mixed case
    up = rng.random(len(seq)) < 0.3
    seq[up] = np.frombuffer(bytes(seq[up]).upper(), dtype=np.uint8)
    # N runs at record starts and ends, a record that is N throughout, runs adjacent across a boundary
    seq[off[10]:off[10] + 7] = ord("N")
    seq[off[11] - 5:off[11]] = ord("n")
    seq[off[11]:off[11] + 3] = ord("N")
    seq[off[9]:off[10]] = ord("n")
    tb = roundtrip(ids, seq, off, byteswap=byteswap, version=version)
    assert tb.byteswapped == byteswap and tb.version == version
    # the N ranges of the whole file and of a slice, in concatenation coordinates
    for first, last in ((0, len(ids)), (9, 12)):
        rec_off, dna_off, nblk = tb.tables(first, last)
        chars = twobit.to_chars(tb, first, last)
        isn = np.zeros(len(chars), dtype=bool)
        for a, b in nblk.reshape(-1, 2):
            isn[a:b] = True
        assert (isn == (chars == ord("n"))).all()
        assert (np.diff(nblk) >= 0).all()  # sorted and disjoint: starts and ends interleave ascending
        assert rec_off[-1] == len(chars) and (dna_off == tb.dna_off[first:last]).all()


def test_mask_blocks_are_lower_case_runs():
    tb = twobit.read_2bit(twobit.write_2bit(["a", "b"], b"acGTnnACgt" + b"AAAA", [0, 10, 14]))
    assert list(tb.mask_idx) == [0, 3, 3]
    assert list(tb.mask_start) == [0, 4, 8] and list(tb.mask_size) == [2, 2, 2]
    assert list(tb.nblk_start) == [4] and list(tb.nblk_size) == [2]


def test_roundtrip_gbrna_sample():
    ids, _, seq, off = helpers.gbrna_sample()
    roundtrip(ids, seq, off)


def test_read_from_path_into_given_buffer(tmp_path):
    ids, seq, off = synth.random_records(3, [1000, 0, 77], iupac_rate=0.01)
    f = twobit.write_2bit(ids, seq, off)
    p = tmp_path / "x.2bit"
    p.write_bytes(f)
    out = np.zeros(len(f) + 100, dtype=np.uint8)
    tb = twobit.read_2bit(str(p), out=out)
    assert tb.data.ctypes.data == out.ctypes.data and tb.data.size == len(f)
    assert twobit.to_chars(tb).tobytes() == fold(seq).tobytes()
    with pytest.raises(ValueError):
        twobit.read_2bit(str(p), out=np.zeros(10, dtype=np.uint8))


def test_truncation_anywhere_is_refused():
    ids, seq, off = synth.random_records(4, [9, 0, 13], iupac_rate=0.2)
    for f in (ACGTA, twobit.write_2bit(ids, seq, off), twobit.write_2bit(ids, seq, off, byteswap=True, version=1)):
        for cut in range(len(f)):
            with pytest.raises(twobit.TwoBitError, match="truncated|outside"):
                twobit.read_2bit(f[:cut])


def test_malformed_files_are_refused():
    with pytest.raises(twobit.TwoBitError, match="signature"):
        twobit.read_2bit(b"\x00" * 40)
    bad = bytearray(ACGTA)
    bad[4] = 2
    with pytest.raises(twobit.TwoBitError, match="version 2"):
        twobit.read_2bit(bytes(bad))
    bad = bytearray(ACGTA)
    bad[18:22] = struct.pack("<I", 4000)
    with pytest.raises(twobit.TwoBitError, match="offset 4000 outside"):
        twobit.read_2bit(bytes(bad))
    # one record "s" of 12 nt with two N blocks at record offset 22: dnaSize, count, starts, sizes
    f = twobit.write_2bit(["s"], b"nnaacgtnnacg", [0, 12])
    assert struct.unpack_from("<5I", f, 22) == (12, 2, 0, 7, 2)
    outside = bytearray(f)
    struct.pack_into("<I", outside, 42, 6)  # second block's size: [7, 13)
    with pytest.raises(twobit.TwoBitError, match="N block 1 .* outside the record"):
        twobit.read_2bit(bytes(outside))
    unsorted = bytearray(f)
    struct.pack_into("<II", unsorted, 30, 7, 0)  # starts 7, 0
    with pytest.raises(twobit.TwoBitError, match="out of order or overlaps"):
        twobit.read_2bit(bytes(unsorted))
    overlap = bytearray(f)
    struct.pack_into("<I", overlap, 34, 1)  # [0, 2) and [1, 3)
    with pytest.raises(twobit.TwoBitError, match="out of order or overlaps"):
        twobit.read_2bit(bytes(overlap))


def test_expansion_header_matches_per_nucleotide_definition(tmp_path):
    exe = str(tmp_path / "twobit_check")
    subprocess.run(["g++", "-O2", "-std=c++17", "-I", os.path.join(helpers.ROOT, "rnamotif_b200", "csrc"),
                    os.path.join(helpers.HERE, "csrc", "twobit_check.cpp"), "-o", exe], check=True)
    out = subprocess.run([exe], check=True, capture_output=True, text=True).stdout
    assert out.strip() == "ok", out


def test_no_source_names_a_batched_copy():
    """Uploads copy with cudaMemcpyAsync only."""
    csrc = os.path.join(helpers.ROOT, "rnamotif_b200", "csrc")
    banned = "Memcpy" + "Batch"
    for name in os.listdir(csrc):
        if name.endswith((".cu", ".cuh", ".h", ".cpp", ".inc")):
            with open(os.path.join(csrc, name), encoding="utf-8", errors="replace") as fh:
                text = fh.read()
            assert banned not in text and ("Memcpy3D" + "Batch") not in text, name
