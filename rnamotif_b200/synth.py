"""Deterministic synthetic sequence databases (numpy default_rng, i.i.d. uniform
acgt as in SURVEY.md section 8d), optionally with planted stem-loops and a
sprinkle of IUPAC / upper-case / 'u' letters so that small inputs still
exercise helices, the comp-strand 'n' mapping and case folding."""
from __future__ import annotations

import numpy as np

_ACGT = np.frombuffer(b"acgt", dtype=np.uint8)
_COMP = {ord("a"): ord("t"), ord("c"): ord("g"), ord("g"): ord("c"), ord("t"): ord("a")}


def random_records(seed: int, lengths, planted: bool = False, iupac_rate: float = 0.0):
    """Returns (ids, seq uint8 (characters), rec_off int64)."""
    rng = np.random.default_rng(seed)
    chunks, offs, ids = [], [0], []
    for i, n in enumerate(lengths):
        s = _ACGT[rng.integers(0, 4, size=int(n))].copy()
        if planted and n >= 40:
            # stem-loops: copy the reverse complement of a stretch a little downstream
            for _ in range(max(1, int(n) // 120)):
                stem = int(rng.integers(3, 11))
                loop = int(rng.integers(3, 13))
                if 2 * stem + loop + 2 >= n:
                    continue
                p = int(rng.integers(0, n - (2 * stem + loop)))
                left = s[p:p + stem]
                rc = np.array([_COMP[int(c)] for c in left[::-1]], dtype=np.uint8)
                # a G:U wobble now and then
                if stem > 4 and rng.random() < 0.3:
                    k = int(rng.integers(0, stem))
                    if rc[k] == ord("c"):
                        rc[k] = ord("t")
                s[p + stem + loop:p + 2 * stem + loop] = rc
        if iupac_rate > 0 and n > 0:
            m = rng.random(int(n)) < iupac_rate
            alt = np.frombuffer(b"nrywskmbdhvNAGCTuUx", dtype=np.uint8)
            s[m] = alt[rng.integers(0, len(alt), size=int(m.sum()))]
        chunks.append(s)
        offs.append(offs[-1] + int(n))
        ids.append("syn%06d" % i)
    seq = np.concatenate(chunks) if chunks else np.zeros(0, dtype=np.uint8)
    return ids, seq, np.asarray(offs, dtype=np.int64)


def write_fastn(path: str, ids, seq: np.ndarray, rec_off: np.ndarray, width: int = 70):
    with open(path, "wb") as fh:
        for i, sid in enumerate(ids):
            fh.write(b">" + sid.encode() + b" synthetic record %d\n" % i)
            s = seq[rec_off[i]:rec_off[i + 1]].tobytes()
            for k in range(0, len(s), width):
                fh.write(s[k:k + width] + b"\n")


GOLDEN_LENGTHS = [5, 0, 21, 22, 45, 46, 62, 63, 64, 94, 95, 96, 101, 118, 119, 200, 333, 1000, 2047, 2048,
                  2049, 4100, 6000, 9000, 12000, 20000, 30011, 50000, 60000]


def golden_db():
    """The database the committed golden candidate streams were produced on."""
    return random_records(20261018, GOLDEN_LENGTHS, planted=True, iupac_rate=0.004)


_COMP_TABLE = np.arange(256, dtype=np.uint8)
for _a, _b in _COMP.items():
    _COMP_TABLE[_a] = _b


def random_reads(seed: int, lengths, stem_every: int = 120, n_rate: float = 0.002, dot_rate: float = 0.0005):
    """Seeded sequencing reads: i.i.d. acgt, with a stem-loop planted every `stem_every` nt on average
    (stems of 3..10 nt, loops of 3..12, placed over the concatenation so that some straddle reads)
    and no-calls -- 'N' at n_rate and '.' at dot_rate.  Vectorised, so that a profile can draw
    1 Gnt.  Returns (ids, seq uint8 (characters), rec_off int64)."""
    rng = np.random.default_rng(seed)
    lengths = np.asarray(lengths, dtype=np.int64)
    off = np.zeros(len(lengths) + 1, dtype=np.int64)
    np.cumsum(lengths, out=off[1:])
    n = int(off[-1])
    seq = _ACGT[rng.integers(0, 4, size=n, dtype=np.uint8)]
    if stem_every > 0 and n > 40:
        per = 1 << 22  # stems per batch (bounds the index arrays)
        todo = n // stem_every
        while todo > 0:
            k = min(todo, per)
            todo -= k
            stem = int(rng.integers(3, 11))
            loop = int(rng.integers(3, 13))
            span = 2 * stem + loop
            p = rng.integers(0, n - span, size=k)
            j = np.arange(stem)
            left = seq[p[:, None] + j]
            seq[p[:, None] + span - 1 - j] = _COMP_TABLE[left]
    for ch, rate in ((ord("N"), n_rate), (ord("."), dot_rate)):
        if rate > 0 and n > 0:
            seq[rng.integers(0, n, size=rng.binomial(n, rate))] = ch
    ids = ["read%d" % i for i in range(len(lengths))]
    return ids, seq, off


def random_transcripts(seed: int, names, sizes, n: int, exon: float = 130, first: float = 250, last: float = 900,
                       intron: float = 1500, utr5: float = 150, utr3: float = 700, max_exons: int = 16,
                       isoforms: int = 3, coding: float = 0.8, p_one: float = 0.03, p_edge: float = 0.03) -> str:
    """Seeded BED12 lines: n transcripts over chromosomes `names` of `sizes` nt, about `isoforms` per gene.
    Exon, intron and UTR lengths are log-normal around the given medians (the defaults are those of a
    human annotation: internal exons ~130 nt, first and last exons longer, 5' UTRs ~150, 3' UTRs ~700).
    What the lines include:
      - one- and multi-exon transcripts on both strands, exons at odd and even offsets, and 1-nt
        exons (share p_one);
      - isoforms of a gene that share exons (exon skipping) and overlap them (an exon end moved);
      - thick ranges inside the exons, a `coding` share of lines; the rest have thickStart == thickEnd;
      - genes that start at 0 or end at the chromosome's end (share p_edge each)."""
    import random
    rng = random.Random(seed)
    sizes = [int(s) for s in sizes]
    chroms = [i for i, s in enumerate(sizes) if s > 0]
    weights = [sizes[i] for i in chroms]

    def draw(median):
        return max(1, int(rng.lognormvariate(np.log(median), 0.8)))

    lines = []
    while len(lines) < n:
        c = rng.choices(chroms, weights)[0]
        size = sizes[c]
        m = min(max_exons, 1 + int(rng.expovariate(1 / 6)))
        ex = [draw(first)] + [draw(exon) for _ in range(m - 2)] + ([draw(last)] if m > 1 else [])
        ex = [1 if rng.random() < p_one else z for z in ex]
        gaps = [draw(intron) for _ in range(m - 1)]
        while len(ex) > 1 and sum(ex) + sum(gaps) > size:
            ex.pop()
            gaps.pop()
        ex[0] = min(ex[0], size)
        span = sum(ex) + sum(gaps)
        u = rng.random()
        g0 = 0 if u < p_edge else size - span if u < 2 * p_edge else rng.randrange(0, size - span + 1)
        gene = []
        p = g0
        for k, z in enumerate(ex):
            gene.append((p, p + z))
            p += z + (gaps[k] if k < len(gaps) else 0)
        minus = rng.random() < 0.5
        for _ in range(1 + rng.randrange(isoforms)):
            if len(lines) >= n:
                break
            # exon skipping: the internal exons are kept with probability 0.8; an exon end moved now and then
            keep = [s_e for k, s_e in enumerate(gene) if k in (0, len(gene) - 1) or rng.random() < 0.8]
            tx = []
            for k, (s, e) in enumerate(keep):
                if e - s > 2 and rng.random() < 0.15:
                    if k < len(keep) - 1:
                        e -= rng.randrange(1, e - s)
                    else:
                        s += rng.randrange(1, e - s)
                tx.append((s, e))
            cs, ce = tx[0][0], tx[-1][1]
            ln = sum(e - s for s, e in tx)
            ts = te = cs
            if rng.random() < coding and ln > 3:
                # the UTRs as exonic lengths from either end, 5' on the transcript's own strand
                a, b = draw(utr5), draw(utr3)
                if minus:
                    a, b = b, a
                if a + b >= ln:
                    a, b = rng.randrange(0, ln // 2), rng.randrange(0, ln // 2)
                ts, te = _exonic(tx, a), _exonic(tx, ln - b)
            lines.append("\t".join(map(str, [names[c], cs, ce, "tx%d" % len(lines), 0, "-" if minus else "+", ts, te, 0,
                                             len(tx), "".join("%d," % (e - s) for s, e in tx),
                                             "".join("%d," % (s - cs) for s, e in tx)])))
    return "".join(line + "\n" for line in lines)


def _exonic(exons, k):
    """The chromosome position of exonic base k of ascending exons (k = their length: the last end)."""
    for s, e in exons:
        if k < e - s:
            return s + k
        k -= e - s
    return exons[-1][1]
