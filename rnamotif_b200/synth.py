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
