"""UCSC .2bit files (the format genomes are distributed in): reader, decoder and writer.

Layout (all integers 32-bit in the file's byte order, which the signature tells):

    header   signature 0x1A412743, version (0, or 1: 64-bit offsets in the index),
             sequence count, reserved
    index    per sequence: name length (1 byte), name, offset of its record
    record   dnaSize, nBlockCount, nBlockStarts[], nBlockSizes[], maskBlockCount,
             maskBlockStarts[], maskBlockSizes[], reserved, then the packed bases:
             T=0 C=1 A=2 G=3, four to a byte, the first in the two most significant bits

N blocks are runs that read N (their packed bases are T); mask blocks are lower-case
runs, which the search does not need (it folds case).

read_2bit() parses the headers and blocks and never walks the packed bases: those go to
the device as they are (gpumotif.MotifSearch.upload_2bit).  to_chars() decodes on the
host, as fm_sbuf would hold the records (lower case, n in N blocks).  write_2bit() is
the inverse of faToTwoBit's packing for the tests.
"""
from __future__ import annotations

import os
import struct

import numpy as np

SIGNATURE = 0x1A412743


class TwoBitError(ValueError):
    pass


class TwoBit:
    """A parsed .2bit file.  `data` is the file's bytes (uint8); record r has `sizes[r]`
    nucleotides packed from byte `dna_off[r]` of `data`; its N blocks are
    nblk_start/nblk_size[nblk_idx[r]:nblk_idx[r+1]] (record coordinates), its mask
    blocks likewise (mask_*)."""

    def __init__(self, data, names, sizes, dna_off, nblk_idx, nblk_start, nblk_size, mask_idx, mask_start, mask_size,
                 byteswapped, version):
        self.data = data
        self.names = names
        self.sizes = sizes
        self.dna_off = dna_off
        self.nblk_idx, self.nblk_start, self.nblk_size = nblk_idx, nblk_start, nblk_size
        self.mask_idx, self.mask_start, self.mask_size = mask_idx, mask_start, mask_size
        self.byteswapped = byteswapped
        self.version = version

    def __len__(self):
        return len(self.names)

    def tables(self, first: int = 0, last: int | None = None):
        """(rec_off, dna_off, nblk) of records [first, last) as gm_db_upload_2bit takes them:
        rec_off[0..n] over the concatenation, byte offsets into `data`, and the N blocks as
        flat [start, end) pairs shifted by their record's rec_off."""
        last = len(self) if last is None else last
        if not 0 <= first <= last <= len(self):
            raise IndexError(f"records [{first}, {last}) outside the {len(self)} of the file")
        sizes = self.sizes[first:last]
        rec_off = np.zeros(len(sizes) + 1, dtype=np.int64)
        np.cumsum(sizes, out=rec_off[1:])
        a, b = int(self.nblk_idx[first]), int(self.nblk_idx[last])
        rec_of_blk = np.repeat(np.arange(last - first), np.diff(self.nblk_idx[first:last + 1]))
        starts = self.nblk_start[a:b] + rec_off[rec_of_blk]
        nblk = np.empty(2 * (b - a), dtype=np.int64)
        nblk[0::2] = starts
        nblk[1::2] = starts + self.nblk_size[a:b]
        return rec_off, np.ascontiguousarray(self.dna_off[first:last], dtype=np.int64), nblk


def _read_file(path, out):
    size = os.path.getsize(path)
    if out is None:
        buf = np.empty(size, dtype=np.uint8)
    else:
        if not isinstance(out, np.ndarray) or out.dtype != np.uint8 or out.ndim != 1 or not out.flags.c_contiguous:
            raise TypeError("out must be a contiguous one-dimensional uint8 array")
        if out.size < size:
            raise ValueError(f"out holds {out.size} bytes, the file has {size}")
        buf = out[:size]
    mv = memoryview(buf)
    with open(path, "rb") as fh:
        got = 0
        while got < size:
            k = fh.readinto(mv[got:])
            if not k:
                raise TwoBitError(f"{path}: file shrank while being read ({got} of {size} bytes)")
            got += k
    return buf


def read_2bit(path_or_bytes, out=None) -> TwoBit:
    """Parse a .2bit file (a path, or its bytes).  `out`: a uint8 array to read the file
    into (e.g. a pinned torch tensor's numpy view, so the upload is asynchronous); the
    returned TwoBit's `data` is a view of it.  Raises TwoBitError naming the problem."""
    if isinstance(path_or_bytes, (str, os.PathLike)):
        data = _read_file(path_or_bytes, out)
    else:
        src = np.frombuffer(path_or_bytes, dtype=np.uint8) if not isinstance(path_or_bytes, np.ndarray) \
            else np.ascontiguousarray(path_or_bytes, dtype=np.uint8).reshape(-1)
        if out is not None:
            if out.size < src.size:
                raise ValueError(f"out holds {out.size} bytes, the file has {src.size}")
            out[:src.size] = src
            src = out[:src.size]
        data = src
    raw = memoryview(data)
    n = data.size

    def need(pos, k, what):
        if pos + k > n:
            raise TwoBitError(f"truncated file: {what} needs bytes [{pos}, {pos + k}), the file has {n}")

    need(0, 16, "the header")
    sig_le = struct.unpack_from("<I", raw, 0)[0]
    if sig_le == SIGNATURE:
        e = "<"
    elif struct.unpack_from(">I", raw, 0)[0] == SIGNATURE:
        e = ">"
    else:
        raise TwoBitError(f"bad signature 0x{sig_le:08x} (a .2bit file starts with 0x{SIGNATURE:08x} in either byte order)")
    version, count, _ = struct.unpack_from(e + "III", raw, 4)
    if version not in (0, 1):
        raise TwoBitError(f"unknown .2bit version {version} (0 and 1 are defined)")
    ofmt, osz = (e + "I", 4) if version == 0 else (e + "Q", 8)
    names, offs = [], []
    pos = 16
    for i in range(count):
        need(pos, 1, f"the name length of index entry {i}")
        ln = raw[pos]
        need(pos + 1, ln, f"the name of index entry {i}")
        names.append(bytes(raw[pos + 1:pos + 1 + ln]).decode("latin-1"))
        pos += 1 + ln
        need(pos, osz, f"the offset of index entry {i}")
        offs.append(struct.unpack_from(ofmt, raw, pos)[0])
        pos += osz
    u4 = np.dtype(e + "u4")
    sizes = np.zeros(count, dtype=np.int64)
    dna_off = np.zeros(count, dtype=np.int64)
    blocks = {"N": ([0], [], []), "mask": ([0], [], [])}
    for i, o in enumerate(offs):
        rec = f"record {i} ({names[i]!r})"
        if o >= n:
            raise TwoBitError(f"{rec}: offset {o} outside the file of {n} bytes")
        need(o, 8, f"{rec}'s dnaSize and N block count")
        size, nb = struct.unpack_from(e + "II", raw, o)
        p = o + 8
        for kind, cnt in (("N", nb), ("mask", None)):
            if cnt is None:
                need(p, 4, f"{rec}'s mask block count")
                cnt = struct.unpack_from(e + "I", raw, p)[0]
                p += 4
            need(p, 8 * cnt, f"{rec}'s {cnt} {kind} blocks")
            st = np.frombuffer(data, dtype=u4, count=cnt, offset=p).astype(np.int64)
            sz = np.frombuffer(data, dtype=u4, count=cnt, offset=p + 4 * cnt).astype(np.int64)
            p += 8 * cnt
            if cnt:
                if (st + sz > size).any():
                    k = int(np.nonzero(st + sz > size)[0][0])
                    raise TwoBitError(f"{rec}: {kind} block {k} [{st[k]}, {st[k] + sz[k]}) outside the record's {size} nucleotides")
                bad = np.nonzero(st[1:] < st[:-1] + sz[:-1])[0]
                if bad.size:
                    k = int(bad[0]) + 1
                    raise TwoBitError(f"{rec}: {kind} block {k} at {st[k]} is out of order or overlaps block {k - 1} "
                                      f"[{st[k - 1]}, {st[k - 1] + sz[k - 1]})")
            idx, sts, szs = blocks[kind]
            idx.append(idx[-1] + cnt)
            sts.append(st)
            szs.append(sz)
        need(p, 4, f"{rec}'s reserved word")
        p += 4
        need(p, (size + 3) // 4, f"{rec}'s {size} packed bases")
        sizes[i] = size
        dna_off[i] = p

    def flat(kind):
        idx, sts, szs = blocks[kind]
        cat = (lambda a: np.concatenate(a) if a else np.zeros(0, dtype=np.int64))
        return np.asarray(idx, dtype=np.int64), cat(sts), cat(szs)

    return TwoBit(data, names, sizes, dna_off, *flat("N"), *flat("mask"), byteswapped=(e == ">"), version=version)


# byte -> its four bases, first base from the two most significant bits
_DECODE4 = np.frombuffer(b"tcag", dtype=np.uint8)[
    (np.arange(256)[:, None] >> np.array([6, 4, 2, 0])[None, :]) & 3].astype(np.uint8)


def to_chars(tb: TwoBit, first: int = 0, last: int | None = None) -> np.ndarray:
    """Records [first, last) decoded and concatenated as uint8 characters: lower case,
    n in N blocks (what fm_sbuf holds for them)."""
    last = len(tb) if last is None else last
    parts = []
    for r in range(first, last):
        size, o = int(tb.sizes[r]), int(tb.dna_off[r])
        s = _DECODE4[tb.data[o:o + (size + 3) // 4]].reshape(-1)[:size].copy()
        for k in range(int(tb.nblk_idx[r]), int(tb.nblk_idx[r + 1])):
            a = int(tb.nblk_start[k])
            s[a:a + int(tb.nblk_size[k])] = ord("n")
        parts.append(s)
    return np.concatenate(parts) if parts else np.zeros(0, dtype=np.uint8)


def _runs(mask):
    """(starts, sizes) of the runs of True in a boolean array."""
    d = np.diff(np.concatenate([[0], mask.astype(np.int8), [0]]))
    starts = np.nonzero(d == 1)[0]
    return starts, np.nonzero(d == -1)[0] - starts


_CODE2 = np.zeros(256, dtype=np.uint8)  # T (and anything that becomes N) = 0
for _ch, _c in (("c", 1), ("a", 2), ("g", 3)):
    _CODE2[ord(_ch)] = _CODE2[ord(_ch.upper())] = _c
_ACGTU = np.zeros(256, dtype=bool)
for _ch in "acgtuACGTU":
    _ACGTU[ord(_ch)] = True


def write_2bit(ids, seq, rec_off, byteswap: bool = False, version: int = 0) -> bytes:
    """A .2bit file of the records seq[rec_off[r]:rec_off[r+1]] named ids[r], as faToTwoBit
    writes it: letters other than a/c/g/t/u become N (N blocks), lower-case runs become
    mask blocks.  byteswap: big-endian integers; version 1: 64-bit index offsets."""
    if version not in (0, 1):
        raise ValueError("version must be 0 or 1")
    seq = np.frombuffer(seq, dtype=np.uint8) if isinstance(seq, (bytes, bytearray)) else np.asarray(seq, dtype=np.uint8)
    rec_off = np.asarray(rec_off, dtype=np.int64)
    e = ">" if byteswap else "<"
    names = [i.encode("latin-1") for i in ids]
    if len(names) != len(rec_off) - 1:
        raise ValueError("one id per record")
    if any(len(nm) > 255 for nm in names):
        raise ValueError("names are at most 255 bytes")
    bodies = []
    for r in range(len(names)):
        s = seq[rec_off[r]:rec_off[r + 1]]
        ns, nz = _runs(~_ACGTU[s])
        ms, mz = _runs((s >= ord("a")) & (s <= ord("z")))
        c = _CODE2[s]
        c = np.concatenate([c, np.zeros((-len(c)) % 4, dtype=np.uint8)]).reshape(-1, 4)
        packed = ((c[:, 0] << 6) | (c[:, 1] << 4) | (c[:, 2] << 2) | c[:, 3]).astype(np.uint8)
        u4 = np.dtype(e + "u4")
        bodies.append(b"".join([
            struct.pack(e + "II", len(s), len(ns)), ns.astype(u4).tobytes(), nz.astype(u4).tobytes(),
            struct.pack(e + "I", len(ms)), ms.astype(u4).tobytes(), mz.astype(u4).tobytes(),
            struct.pack(e + "I", 0), packed.tobytes()]))
    osz = 4 if version == 0 else 8
    pos = 16 + sum(1 + len(nm) + osz for nm in names)
    index = []
    for nm, body in zip(names, bodies):
        if version == 0 and pos >= 1 << 32:
            raise ValueError("file too large for version 0 (use version=1)")
        index.append(struct.pack("B", len(nm)) + nm + struct.pack(e + ("I" if version == 0 else "Q"), pos))
        pos += len(body)
    return b"".join([struct.pack(e + "IIII", SIGNATURE, version, len(names), 0)] + index + bodies)
