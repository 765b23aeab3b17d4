"""Four-line FASTQ: the reference reader and writer for MotifSearch.upload_fastq.

The format (include/gpumotif.h, gm_db_upload_fastq): every record is four lines -- '@' + id and
description, the read, '+' (anything may follow), the quality string.  A line's role is its index
mod 4, never its first byte.  Every byte of a read line but a trailing '\\r' is one nucleotide.
Lines end in '\\n' or '\\r\\n'; the line end after the last line is optional.  parse_fastq raises
FastqError for each input the device reader refuses, with the record it names.  With a minimum base
quality (gm_ctx_set_min_quality) it masks low-quality bases as n and refuses quality bytes outside
[qual_offset, 126], as the device does.
"""
from __future__ import annotations

import numpy as np

_LOWER = np.arange(256, dtype=np.uint8)
for _c in range(ord("A"), ord("Z") + 1):
    _LOWER[_c] = _c + 32
_LOWER[ord("U")] = ord("t")
_LOWER[ord("u")] = ord("t")


class FastqError(ValueError):
    """A refused input: `record` and `offset` (of its '@') name the first failing record, or are
    None for a refusal of the whole text."""

    def __init__(self, msg, record=None, offset=None):
        super().__init__(msg)
        self.record, self.offset = record, offset


def trimmed_length(data: bytes) -> int:
    """The text without the line end after its last line ('\\n', '\\r\\n' or '\\r')."""
    n = len(data)
    if n and data[n - 1:n] == b"\n":
        n -= 1
    if n and data[n - 1:n] == b"\r":
        n -= 1
    return n


def parse_fastq(data: bytes, min_qual: int = 0, qual_offset: int = 33):
    """Return (ids, seq, rec_off, hdr_off): ids = each record's id (the first blank-delimited
    token after '@'), seq = the reads' characters concatenated as uint8 (lower case, u -> t, as
    MotifSearch.get_chars reads them back), rec_off = n+1 int64 offsets into seq, hdr_off = n+1
    int64 offsets of each record's '@' in `data` (hdr_off[n] = len(data)).  min_qual > 0: every
    base whose quality byte q has q - qual_offset < min_qual is n in seq, and a record with a
    quality byte outside [qual_offset, 126] is refused (after its own format checks)."""
    if qual_offset not in (33, 64) or not 0 <= min_qual <= 126 - qual_offset:
        raise ValueError(f"min_qual {min_qual}, qual_offset {qual_offset}: offset 33 or 64, min_qual in [0, 126 - offset]")
    data = bytes(data)
    if data and data[:1] != b"@":
        raise FastqError("FASTQ text does not begin with '@'")
    n = trimmed_length(data)
    ids, reads, quals, offs, hdrs = [], [], [], [0], []
    if n:
        lines, starts, p = [], [], 0
        while True:
            e = data.find(b"\n", p, n)
            if e < 0:
                e = n
            body = data[p:e]
            if body.endswith(b"\r") and e < n:
                body = body[:-1]  # a '\r' before the '\n'
            lines.append(body)
            starts.append(p)
            if e == n:
                break
            p = e + 1
        total = 0
        for r in range(0, (len(lines) + 3) // 4):
            k, at = 4 * r, starts[4 * r]
            rec = lines[k:k + 4]
            if not rec[0].startswith(b"@"):
                raise FastqError(f"FASTQ record {r} at byte {at}: line {k + 1} does not start with '@'", r, at)
            if len(rec) > 2 and not rec[2].startswith(b"+"):
                raise FastqError(f"FASTQ record {r} at byte {at}: line {k + 3} does not start with '+' "
                                 "(only four-line FASTQ is accepted)", r, at)
            if len(rec) < 4:
                raise FastqError(f"FASTQ record {r} at byte {at}: the last record has fewer than four lines", r, at)
            if len(rec[1]) != len(rec[3]):
                raise FastqError(f"FASTQ record {r} at byte {at}: its quality string is not as long as its read", r, at)
            if min_qual > 0:
                q = np.frombuffer(rec[3], dtype=np.uint8)
                out = np.flatnonzero((q < qual_offset) | (q > 126))
                if out.size:
                    raise FastqError(f"FASTQ record {r} at byte {at}: quality byte {q[out[0]]} is outside "
                                     f"[{qual_offset}, 126]", r, at)
                quals.append(rec[3])
            parts = rec[0][1:].split(None, 1)
            ids.append(parts[0].decode("latin-1") if parts else "")
            reads.append(rec[1])
            total += len(rec[1])
            offs.append(total)
            hdrs.append(at)
    hdrs.append(len(data))
    seq = _LOWER[np.frombuffer(b"".join(reads), dtype=np.uint8)]
    if min_qual > 0:
        seq[np.frombuffer(b"".join(quals), dtype=np.uint8) < qual_offset + min_qual] = ord("n")
    return ids, seq, np.asarray(offs, dtype=np.int64), np.asarray(hdrs, dtype=np.int64)


def write_fastq(ids, seq, rec_off, qual=None, crlf: bool = False) -> bytes:
    """Four-line FASTQ of records ids[r] / seq[rec_off[r]:rec_off[r+1]]: '@id', the read, '+', the
    quality string (qual: one bytes per record, default 'I' for every base), every line ended by
    '\\n' (crlf: '\\r\\n')."""
    seq = np.asarray(seq, dtype=np.uint8)
    nl = b"\r\n" if crlf else b"\n"
    out = []
    for r, sid in enumerate(ids):
        s = seq[rec_off[r]:rec_off[r + 1]].tobytes()
        q = b"I" * len(s) if qual is None else bytes(qual[r])
        sid = sid.encode("latin-1") if isinstance(sid, str) else bytes(sid)
        out += [b"@", sid, nl, s, nl, b"+", nl, q, nl]
    return b"".join(out)
