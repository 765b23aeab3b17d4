"""BED annotation -> the block tables of gm_db_assemble (gpumotif.MotifSearch.assemble_bed).

A BED line names a region of an uploaded genome: BED3/BED6 one block [chromStart, chromEnd), BED12
the exons (blockCount, blockSizes, blockStarts relative to chromStart).  Strand '-' makes the
record the reverse complement (the transcript as it is read 5' to 3'); '+', '.' or no strand column
is the plus strand.  `part` picks what of the exons becomes the record:

    exons   the spliced transcript
    cds     the exonic bases in [thickStart, thickEnd)
    utr5    strand-aware: the exonic bases below thickStart on '+', at or above thickEnd on '-'
    utr3    the other side: at or above thickEnd on '+', below thickStart on '-'

A line with thickStart == thickEnd (non-coding) has an empty cds and empty UTRs; a line without the
thick columns has thickStart = chromStart and thickEnd = chromEnd.  A line with nothing in the part
gives an empty record, so record r is always BED line r.

Assembly.assemble_chars is the host reference of what the device builds, and Assembly.to_source maps
a position of an assembled record back to the genome.
"""
from __future__ import annotations

import numpy as np

PARTS = ("exons", "cds", "utr5", "utr3")


class BedError(ValueError):
    def __init__(self, line: int, msg: str):
        super().__init__(f"BED line {line}: {msg}")
        self.line = line


# fm_sbuf's characters (src/dbutil.c:105-111): letters folded to lower case, u -> t
_FOLD = np.arange(256, dtype=np.uint8)
_FOLD[ord("A"):ord("Z") + 1] += 32
_FOLD[ord("u")] = _FOLD[ord("U")] = ord("t")
# mk_rcmp's complement of a folded character (src/rnamot.c:193-216): a <-> t, c <-> g, else n
_COMP = np.full(256, ord("n"), dtype=np.uint8)
for _a, _b in zip(b"acgt", b"tgca"):
    _COMP[_a] = _b
_COMP = _COMP[_FOLD]


class Assembly:
    """gm_db_assemble's tables: blk (flat [start, end) pairs in the held batch's rec_off coordinates),
    rec_blk (n_rec + 1 entries), strand (uint8, 1 = minus) and one name per record; rec_off is the
    held batch's record table the blocks refer to."""

    def __init__(self, blk, rec_blk, strand, names, rec_off):
        self.blk = np.ascontiguousarray(blk, dtype=np.int64).reshape(-1)
        self.rec_blk = np.ascontiguousarray(rec_blk, dtype=np.int64)
        self.strand = np.ascontiguousarray(strand, dtype=np.uint8)
        self.names = list(names)
        self.rec_off = np.ascontiguousarray(rec_off, dtype=np.int64)

    def __len__(self):
        return len(self.rec_blk) - 1

    def _starts(self):
        """(cum, rec_start): each block's offset in the concatenation of all blocks (plus order), n_blk + 1
        entries, and each record's first entry in it, n_rec + 1 entries"""
        cum = np.zeros(len(self.blk) // 2 + 1, dtype=np.int64)
        np.cumsum(self.blk[1::2] - self.blk[0::2], out=cum[1:])
        return cum, cum[self.rec_blk]

    def rec_off_new(self) -> np.ndarray:
        """The assembled batch's record table."""
        _, rs = self._starts()
        return rs - rs[0]

    def to_source(self, rec, pos):
        """Position `pos` of assembled record `rec` (forward strand of that record, vectorised) -> (held
        record, offset in it)."""
        rec = np.asarray(rec, dtype=np.int64)
        pos = np.asarray(pos, dtype=np.int64)
        cum, rs = self._starts()
        length = rs[rec + 1] - rs[rec]
        if ((pos < 0) | (pos >= length)).any():
            raise IndexError("position outside its assembled record")
        c = rs[rec] + np.where(self.strand[rec] == 1, length - 1 - pos, pos)
        k = np.searchsorted(cum, c, side="right") - 1
        g = self.blk[2 * k] + (c - cum[k])
        held = np.searchsorted(self.rec_off, g, side="right") - 1
        return held, g - self.rec_off[held]

    def assemble_chars(self, chars, rec_off=None):
        """The assembled records as fm_sbuf would hold them, built on the host from the held batch's
        characters: (uint8 characters, rec_off).  Plus records fold case and read u as t; minus records
        are mk_rcmp of their blocks (a c g t n)."""
        chars = np.asarray(chars, dtype=np.uint8)
        if rec_off is not None and not np.array_equal(np.asarray(rec_off, dtype=np.int64), self.rec_off):
            raise ValueError("rec_off is not the record table the blocks refer to")
        b = self.blk.reshape(-1, 2)
        pieces = []
        for r in range(len(self)):
            k0, k1 = int(self.rec_blk[r]), int(self.rec_blk[r + 1])
            if self.strand[r]:
                pieces += [_COMP[chars[s:e][::-1]] for s, e in b[k0:k1][::-1]]
            else:
                pieces += [chars[s:e] for s, e in b[k0:k1]]
        out = np.concatenate(pieces) if pieces else np.zeros(0, dtype=np.uint8)
        return _FOLD[out], self.rec_off_new()


def _ints(field: str, line: int, what: str):
    try:
        return [int(x) for x in field.rstrip(",").split(",")] if field.rstrip(",") else []
    except ValueError:
        raise BedError(line, f"{what} {field!r} is not a list of integers") from None


def _clip(exons, lo, hi):
    """the exons' bases in [lo, hi)"""
    return [(max(s, lo), min(e, hi)) for s, e in exons if min(e, hi) > max(s, lo)]


def read_bed(text, names, rec_off, part: str = "exons") -> Assembly:
    """Parse BED text (str or bytes) against the held batch: `names` = its record names in upload order
    (TwoBit.names, or the first word of each FASTA definition line), `rec_off` = its record table.
    Skips track, browser, '#' and blank lines.  Raises BedError naming the line (1-based) for an unknown
    chromosome, an end past the chromosome, blocks out of order or overlapping, blocks outside
    [chromStart, chromEnd) or a wrong block count."""
    if part not in PARTS:
        raise ValueError(f"part must be one of {PARTS}")
    if isinstance(text, (bytes, bytearray)):
        text = text.decode("latin-1")
    rec_off = np.asarray(rec_off, dtype=np.int64)
    index = {}
    for i, nm in enumerate(names):
        index.setdefault(nm, i)
    blk, rec_blk, strand, out_names = [], [0], [], []
    for ln, raw in enumerate(text.splitlines(), 1):
        f = raw.split()
        if not f or f[0].startswith("#") or f[0] in ("track", "browser"):
            continue
        if len(f) < 3:
            raise BedError(ln, "fewer than 3 columns")
        if f[0] not in index:
            raise BedError(ln, f"unknown chromosome {f[0]!r}")
        chrom = index[f[0]]
        size = int(rec_off[chrom + 1] - rec_off[chrom])
        try:
            cs, ce = int(f[1]), int(f[2])
            ts, te = (int(f[6]), int(f[7])) if len(f) >= 8 else (cs, ce)
        except ValueError:
            raise BedError(ln, "a coordinate is not an integer") from None
        if cs < 0 or ce < cs:
            raise BedError(ln, f"chromStart {cs} and chromEnd {ce} do not make a range")
        if ce > size:
            raise BedError(ln, f"chromEnd {ce} past the end of {f[0]} ({size} nt)")
        minus = len(f) >= 6 and f[5] == "-"
        if len(f) >= 12:
            n = _ints(f[9], ln, "blockCount")
            sizes, starts = _ints(f[10], ln, "blockSizes"), _ints(f[11], ln, "blockStarts")
            if len(n) != 1 or len(sizes) != n[0] or len(starts) != n[0]:
                raise BedError(ln, f"blockCount {f[9]} with {len(sizes)} sizes and {len(starts)} starts")
            exons = []
            for k, (s, z) in enumerate(zip(starts, sizes)):
                if s < 0 or z < 0 or cs + s + z > ce:
                    raise BedError(ln, f"block {k} [{cs + s}, {cs + s + z}) outside [{cs}, {ce})")
                if exons and cs + s < exons[-1][1]:
                    raise BedError(ln, f"block {k} at {cs + s} is out of order or overlaps block {k - 1}")
                exons.append((cs + s, cs + s + z))
        else:
            exons = [(cs, ce)]
        if part == "cds":
            exons = _clip(exons, ts, te) if ts < te else []
        elif part != "exons":
            low = (part == "utr5") != minus  # utr5 on '+' and utr3 on '-' lie below thickStart
            exons = [] if ts >= te else _clip(exons, cs, ts) if low else _clip(exons, te, ce)
        o = int(rec_off[chrom])
        blk += [(o + s, o + e) for s, e in exons]
        rec_blk.append(len(blk))
        strand.append(1 if minus else 0)
        out_names.append(f[3] if len(f) >= 4 else f"{f[0]}:{cs}-{ce}")
    flat = np.array(blk, dtype=np.int64).reshape(-1)
    return Assembly(flat, np.array(rec_blk, dtype=np.int64), np.array(strand, dtype=np.uint8), out_names, rec_off)
