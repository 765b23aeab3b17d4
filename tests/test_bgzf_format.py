"""CPU: the DEFLATE decoder of the BGZF upload (rnamotif_b200/csrc/gm_inflate.h, built for the host
by tests/csrc/inflate_check.cpp) and the BGZF writer (rnamotif_b200/bgzf.py).

The decoder's output and CRC-32 must equal zlib's over FASTA text, random bytes, runs and long
repeats, compressed at several levels and with every zlib strategy, in members of 1 byte to 64 KiB.
Built with AddressSanitizer and UndefinedBehaviorSanitizer, with every stream and output buffer
allocated to its exact size, it must also survive every truncation of three streams, about 20 000
bit flips and byte overwrites, and hand-built hostile streams: each returns an error, or, where the
mutated stream is still valid DEFLATE, exactly what zlib decodes from it, and nothing is read or
written out of bounds."""
import gzip
import os
import struct
import subprocess
import zlib

import numpy as np
import pytest

from rnamotif_b200 import bgzf
import helpers

# gm_inflate.h's status codes
OK, BLOCK_TYPE, STORED_LEN, CODE, REPEAT, SYMBOL, DISTANCE, OVERFLOW, UNDERFLOW, OVERRUN = range(10)

LEVELS = [(0, zlib.Z_DEFAULT_STRATEGY), (1, zlib.Z_DEFAULT_STRATEGY), (6, zlib.Z_DEFAULT_STRATEGY),
          (9, zlib.Z_DEFAULT_STRATEGY), (6, zlib.Z_FILTERED), (6, zlib.Z_HUFFMAN_ONLY), (6, zlib.Z_RLE),
          (6, zlib.Z_FIXED)]
MEMBER_SIZES = [1, 100, 0xff00, 65536]


def gbrna_text():
    with gzip.open(os.path.join(helpers.GOLDEN, "gbrna", "sample.fastn.gz"), "rb") as fh:
        return fh.read()


def synthetic_fasta(seed=3, n_rec=40):
    """Mixed case, N runs, empty records, blank lines, irregular and 60-column lines, CR LF."""
    rng = np.random.default_rng(seed)
    out = []
    for r in range(n_rec):
        out.append(b">rec%d some definition %d\n" % (r, rng.integers(1 << 30)))
        n = int(rng.choice([0, 1, 59, 60, 61, 1000, int(rng.integers(0, 20000))]))
        s = bytearray(rng.choice(np.frombuffer(b"acgtACGTuUn", dtype=np.uint8), size=n).tobytes())
        if n > 100:
            p = int(rng.integers(0, n - 50))
            s[p:p + 50] = b"N" * 50
        k = 0
        while k < n:
            w = 60 if rng.random() < 0.7 else int(rng.integers(0, 200))
            out.append(bytes(s[k:k + w]) + (b"\r\n" if rng.random() < 0.05 else b"\n"))
            if rng.random() < 0.05:
                out.append(b"\n")
            k += max(w, 1)
    return b"".join(out)


def period_32k():
    """A 40 KB input of period 32 768: zlib's matches reach as far back as its window lets them."""
    r = np.random.default_rng(9).integers(0, 256, size=32768, dtype=np.uint8).tobytes()
    return r + r[:8192]


INPUTS = {
    "gbrna": gbrna_text,
    "synthetic_fasta": synthetic_fasta,
    "random": lambda: np.random.default_rng(5).integers(0, 256, size=150000, dtype=np.uint8).tobytes(),
    "one_byte_65536": lambda: b"a" * 65536,
    "period_32k": period_32k,
    "empty": lambda: b"",
}


def deflate(data, level=6, strategy=zlib.Z_DEFAULT_STRATEGY):
    co = zlib.compressobj(level, zlib.DEFLATED, -15, 8, strategy)
    return co.compress(data) + co.flush()


# ---- a DEFLATE bit writer for the hand-built streams ---------------------------------------------

class BitWriter:
    def __init__(self):
        self.v, self.n = 0, 0

    def bits(self, v, k):  # k bits, least significant first
        self.v |= (v & ((1 << k) - 1)) << self.n
        self.n += k
        return self

    def code(self, c, k):  # a Huffman code: most significant bit first
        return self.bits(int(format(c, f"0{k}b")[::-1], 2), k)

    def bytes(self):
        return self.v.to_bytes((self.n + 7) // 8, "little")

    # fixed Huffman codes (RFC 1951 3.2.6)
    def lit(self, s):
        if s < 144:
            return self.code(0x30 + s, 8)
        if s < 256:
            return self.code(0x190 + s - 144, 9)
        if s < 280:
            return self.code(s - 256, 7)
        return self.code(0xC0 + s - 280, 8)

    LBASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258]
    LEXT = [0] * 8 + [1] * 4 + [2] * 4 + [3] * 4 + [4] * 4 + [5] * 4 + [0]
    DBASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073,
             4097, 6145, 8193, 12289, 16385, 24577]
    DEXT = [0, 0, 0, 0] + [k // 2 for k in range(2, 28)]

    def match(self, length, dist):
        s = max(i for i, b in enumerate(self.LBASE) if b <= length) if length < 258 else 28
        self.lit(257 + s).bits(length - self.LBASE[s], self.LEXT[s])
        d = max(i for i, b in enumerate(self.DBASE) if b <= dist)
        return self.code(d, 5).bits(dist - self.DBASE[d], self.DEXT[d])


def fixed(body, final=1):
    w = BitWriter().bits(final, 1).bits(1, 2)
    body(w)
    return w.lit(256).bytes()


def dynamic_header(hlit, hdist, clens):
    """BFINAL=1, BTYPE=2, HLIT, HDIST and the code-length code's lengths in transmission order."""
    w = BitWriter().bits(1, 1).bits(2, 2).bits(hlit - 257, 5).bits(hdist - 1, 5).bits(len(clens) - 4, 4)
    for c in clens:
        w.bits(c, 3)
    return w


def hand_built():
    """(name, stream, isize, expected status, expected output or None)"""
    cases = []
    cases.append(("block type 3", BitWriter().bits(1, 1).bits(3, 2).bits(0, 16).bytes(), 0, BLOCK_TYPE, None))
    cases.append(("stored LEN != ~NLEN", bytes([1]) + struct.pack("<HH", 3, 0x1234) + b"abc", 3, STORED_LEN, None))
    cases.append(("stored, valid", bytes([1]) + struct.pack("<HH", 3, 0xfffc) + b"abc", 3, OK, b"abc"))
    cases.append(("stored, LEN past the input", bytes([1]) + struct.pack("<HH", 9, 0xfff6) + b"abc", 9, OVERRUN, None))
    # code-length code: order 16 17 18 0 8 7 9 6 10 5 11 4 12 3 13 2 14 1 15
    cases.append(("over-subscribed code-length code", dynamic_header(257, 1, [1] * 19).bits(0, 32).bytes(), 0, CODE, None))
    cases.append(("incomplete code-length code", dynamic_header(257, 1, [1, 0, 0, 0]).bits(0, 32).bytes(), 0, CODE, None))
    # symbols 16 and 0 of length 1: 0 -> code 0, 16 -> code 1; a repeat of nothing
    cases.append(("repeat code 16 first", dynamic_header(257, 1, [1, 0, 0, 1]).code(1, 1).bits(0, 2).bits(0, 32).bytes(),
                  0, REPEAT, None))
    # 18 and 0 of length 1: 0 -> 0, 18 -> 1; 138 + 138 zeros > 258 lengths
    w = dynamic_header(257, 1, [0, 0, 1, 1])
    w.code(1, 1).bits(127, 7).code(1, 1).bits(127, 7).bits(0, 32)
    cases.append(("lengths past HLIT + HDIST", w.bytes(), 0, REPEAT, None))
    cases.append(("HLIT 287", dynamic_header(287, 1, [1] * 19).bits(0, 32).bytes(), 0, CODE, None))
    cases.append(("symbol 286", fixed(lambda w: w.lit(286)), 0, SYMBOL, None))
    cases.append(("symbol 287", fixed(lambda w: w.lit(97).lit(287)), 1, SYMBOL, None))
    for d in (30, 31):
        cases.append((f"distance symbol {d}", fixed(lambda w, d=d: w.lit(97).lit(257).code(d, 5)), 4, SYMBOL, None))
    cases.append(("distance before the output start", fixed(lambda w: w.lit(97).match(3, 2)), 4, DISTANCE, None))
    cases.append(("distance 1 at the output start", fixed(lambda w: w.match(3, 1)), 3, DISTANCE, None))
    ten = fixed(lambda w: [w.lit(c) for c in b"abcdefghij"])
    cases.append(("output longer than ISIZE", ten, 5, OVERFLOW, None))
    cases.append(("match past ISIZE", fixed(lambda w: w.lit(97).match(10, 1)), 5, OVERFLOW, None))
    cases.append(("output shorter than ISIZE", ten, 20, UNDERFLOW, None))
    cases.append(("no final block", BitWriter().bits(0, 1).bits(1, 2).lit(256).bytes(), 0, OVERRUN, None))
    cases.append(("empty input", b"", 0, OVERRUN, None))
    cases.append(("fixed, empty", fixed(lambda w: None), 0, OK, b""))
    cases.append(("fixed, ten literals", ten, 10, OK, b"abcdefghij"))
    # the farthest match DEFLATE allows: distance 32 768, length 258 (zlib's encoder stops short of it)
    r = np.random.default_rng(2).integers(0, 256, size=32768, dtype=np.uint8).tobytes()
    far = fixed(lambda w: ([w.lit(c) for c in r], w.match(258, 32768)))
    cases.append(("distance 32768, length 258", far, 32768 + 258, OK, r + r[:258]))
    return cases


# ---- the host build --------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def checker(tmp_path_factory):
    d = tmp_path_factory.mktemp("inflate")
    exe = str(d / "inflate_check")
    subprocess.run(["g++", "-O1", "-g", "-std=c++17", "-fsanitize=address,undefined", "-fno-sanitize-recover=all",
                    "-fno-omit-frame-pointer", "-I", os.path.join(helpers.ROOT, "rnamotif_b200", "csrc"),
                    os.path.join(helpers.HERE, "csrc", "inflate_check.cpp"), "-o", exe], check=True)

    def run(streams):
        """streams: [(deflate bytes, isize)] -> [(status, output, crc)]"""
        corpus, out = str(d / "corpus.bin"), str(d / "out.bin")
        with open(corpus, "wb") as fh:
            for s, isize in streams:
                fh.write(struct.pack("<II", len(s), isize))
                fh.write(s)
        env = dict(os.environ, ASAN_OPTIONS="detect_leaks=1:abort_on_error=0", UBSAN_OPTIONS="print_stacktrace=1")
        r = subprocess.run([exe, corpus, out], capture_output=True, text=True, env=env)
        assert r.returncode == 0 and not r.stderr, r.stderr[-4000:]
        assert int(r.stdout) == len(streams)
        res, raw, p = [], open(out, "rb").read(), 0
        for _ in streams:
            st, n, crc = struct.unpack_from("<III", raw, p)
            res.append((st, raw[p + 12:p + 12 + n], crc))
            p += 12 + n
        return res
    return run


def zlib_inflate(s):
    """zlib's raw inflate of s, or None where zlib finds it invalid or unfinished."""
    d = zlib.decompressobj(-15)
    try:
        out = d.decompress(s)
    except zlib.error:
        return None
    return out if d.eof else None


@pytest.mark.parametrize("name", sorted(INPUTS))
def test_output_and_crc_equal_zlib(name, checker):
    data = INPUTS[name]()
    streams, want = [], []
    for level, strategy in LEVELS:
        for m in MEMBER_SIZES:
            # members of 1 and 100 bytes: the first few hundred, the rest are alike
            limit = {1: 300, 100: 200}.get(m, len(data))
            pieces = [data[o:o + m] for o in range(0, min(len(data), limit * m), m)] or [b""]
            for p in pieces:
                streams.append((deflate(p, level, strategy), len(p)))
                want.append(p)
    got = checker(streams)
    for k, ((st, out, crc), w) in enumerate(zip(got, want)):
        assert st == OK, f"{name}: stream {k}: status {st}"
        assert out == w, f"{name}: stream {k}: output differs from zlib's"
        assert crc == zlib.crc32(w), f"{name}: stream {k}: CRC-32 differs from zlib's"


def hostile_bases():
    text = gbrna_text()
    return [(deflate(text[:4000], 6), 4000),                          # dynamic Huffman
            (deflate(text[5000:7000], 6, zlib.Z_FIXED), 2000),         # fixed Huffman
            (deflate(text[9000:9300], 0), 300)]                        # stored


def check_hostile(streams, got):
    for (s, isize), (st, out, crc) in zip(streams, got):
        assert len(out) <= isize
        if st == OK:  # still valid DEFLATE: then exactly zlib's output, and all of it
            z = zlib_inflate(s)
            assert z is not None and z == out and len(out) == isize, f"accepted a stream zlib decodes otherwise: {s.hex()}"
        assert crc == zlib.crc32(out)


def test_every_truncation(checker):
    streams = [(s[:cut], isize) for s, isize in hostile_bases() for cut in range(len(s))]
    got = checker(streams)
    check_hostile(streams, got)
    assert all(st != OK for st, _, _ in got)


def test_bit_flips_and_byte_overwrites(checker):
    rng = np.random.default_rng(17)
    streams = []
    for s, isize in hostile_bases():
        for _ in range(3400):
            b = bytearray(s)
            b[int(rng.integers(len(b)))] ^= 1 << int(rng.integers(8))
            streams.append((bytes(b), isize))
        for _ in range(3400):
            b = bytearray(s)
            for _ in range(int(rng.integers(1, 4))):
                b[int(rng.integers(len(b)))] = int(rng.integers(256))
            streams.append((bytes(b), isize))
    got = checker(streams)
    check_hostile(streams, got)
    # both outcomes occur: errors, and mutations (mostly of stored bytes) that stay valid DEFLATE
    assert 0 < sum(st != OK for st, _, _ in got) < len(streams)


def test_hand_built_streams(checker):
    cases = hand_built()
    got = checker([(s, isize) for _, s, isize, _, _ in cases])
    for (name, s, isize, want_st, want_out), (st, out, crc) in zip(cases, got):
        assert st == want_st, f"{name}: status {st}, expected {want_st}"
        if want_out is not None:
            assert out == want_out and zlib_inflate(s) == want_out, name
    check_hostile([(s, isize) for _, s, isize, _, _ in cases], got)


def test_members_of_the_device_error_tests_decode_to_errors_here(checker):
    """The corrupted files tests/test_bgzf.py sends to the device: this build finds the same faults."""
    import test_bgzf
    text = test_bgzf.make_text()
    for what, g, _ in test_bgzf.device_error_cases(text, bgzf.write_bgzf(text)):
        ms = members(g)
        got = checker([(g[p + 18:p + size - 8], isize) for p, size, isize, _ in ms])
        bad = [k for k, ((st, out, crc), (_, _, _, want_crc)) in enumerate(zip(got, ms)) if st != OK or crc != want_crc]
        if what == "no '>'":
            assert bad == [] and got[0][1][:1] != b">"
        else:
            assert bad == [3], what
            st = got[3][0]
            assert st == {"CRC": OK, "ISIZE": OVERFLOW, "deflate": BLOCK_TYPE}[what], what


# ---- bgzf.py ----------------------------------------------------------------------------------------

def members(buf):
    """[(offset, BSIZE + 1, ISIZE, CRC)] of a BGZF file, from its headers."""
    out, p = [], 0
    while p < len(buf):
        assert buf[p:p + 4] == b"\x1f\x8b\x08\x04" and buf[p + 10:p + 12] == b"\x06\x00" and buf[p + 12:p + 16] == b"BC\x02\x00"
        size = struct.unpack_from("<H", buf, p + 16)[0] + 1
        crc, isize = struct.unpack_from("<II", buf, p + size - 8)
        out.append((p, size, isize, crc))
        p += size
    assert p == len(buf)
    return out


def test_eof_block_is_the_specifications():
    assert bgzf.EOF_BLOCK == bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")
    assert bgzf.write_bgzf(b"") == bgzf.EOF_BLOCK
    assert gzip.decompress(bgzf.EOF_BLOCK) == b""


@pytest.mark.parametrize("name", sorted(INPUTS))
def test_write_bgzf_round_trip_and_member_fields(name):
    data = INPUTS[name]()
    for level, strategy in LEVELS:
        for m in (100, 0xff00, 65536):
            try:
                f = bgzf.write_bgzf(data, level=level, block=m, strategy=strategy)
            except ValueError:
                # 64 KiB in stored blocks (level 0, or data zlib cannot compress) do not fit a member
                assert m == 65536 and (level == 0 or name == "random")
                continue
            assert gzip.decompress(f) == data
            ms = members(f)
            assert ms[-1] == (len(f) - 28, 28, 0, 0)
            o = 0
            for p, size, isize, crc in ms[:-1]:
                assert isize == min(m, len(data) - o) and crc == zlib.crc32(data[o:o + isize])
                assert zlib_inflate(f[p + 18:p + size - 8]) == data[o:o + isize]
                o += isize
            assert o == len(data)
    assert bgzf.write_bgzf(data, eof=False) == bgzf.write_bgzf(data)[:-28]
