"""gm_prune_hits (rmprune over the binary candidate stream, SURVEY section 8 f4)
against the reference's own rmprune run on the reference's own output.

CPU only: candidates come from the oracle port (the same records the device
returns), the expected verdicts from oracle/_ref/rnamotif | oracle/_ref/rmprune
over the reference's test database.  Descriptors are those whose every
candidate is printed (no REJECT in the score section), so that hit i of the
candidate stream is hit i of rnamotif's output."""
import gzip
import os
import subprocess

import numpy as np
import pytest

from oracle import oracle_port
from rnamotif_b200 import fastn, gpumotif
import helpers

REF = helpers.REF
DATA = os.path.join(REF, "data", "test")
have = all(os.path.exists(p) for p in (os.path.join(REF, "rnamotif"), os.path.join(REF, "rmprune"),
                                        os.path.join(DATA, "gbrna.111.0.fastn"), gpumotif.LIB_PATH))


def hit_lines(text: bytes):
    """[(def line, hit line)] of an rnamotif / rmprune output"""
    lines = text.split(b"\n")
    out = []
    i = 0
    while i < len(lines):
        if lines[i].startswith(b">"):
            out.append((lines[i], lines[i + 1]))
            i += 2
        else:
            i += 1
    return out


@pytest.mark.skipif(not have, reason="oracle/_ref (reference rnamotif + rmprune + test database) not built")
@pytest.mark.parametrize("name", ["trna", "pk1", "qu+tr", "pk_j1+2", "nanlin"])
def test_prune_matches_reference_rmprune(name):
    env = dict(os.environ, EFNDATA=os.path.join(REF, "data", "efndata"))
    raw = subprocess.run([os.path.join(REF, "rnamotif"), "-descr", name + ".descr", "gbrna.111.0.fastn"],
                         cwd=DATA, env=env, capture_output=True, timeout=600, check=True).stdout
    pruned = subprocess.run([os.path.join(REF, "rmprune")], input=raw, cwd=DATA, capture_output=True,
                            timeout=600, check=True).stdout
    all_hits, kept = hit_lines(raw), hit_lines(pruned)

    plan = helpers.load_plan(name)
    ids, defs, seq, off = fastn.read_fastn(os.path.join(DATA, "gbrna.111.0.fastn"))
    both = bool(gpumotif.plan_field(plan, 8))
    cands, _ = oracle_port.scan_db(plan, seq, off, both)
    assert len(cands) == len(all_hits), "descriptor prints every candidate: counts must agree"

    # rmprune's blocks are runs of hits with the same locus name up to the first '.'
    names = [i.split(".")[0] for i in ids]
    uniq = {n: k for k, n in enumerate(dict.fromkeys(names))}
    group = np.array([uniq[names[r]] for r in cands["rec"]], dtype=np.int32)
    keep = gpumotif.prune_hits(plan, cands, group)

    # rmprune keeps the order: walk both lists
    expect = np.zeros(len(all_hits), dtype=bool)
    j = 0
    for i, h in enumerate(all_hits):
        if j < len(kept) and kept[j] == h:
            expect[i] = True
            j += 1
    assert j == len(kept), "every line rmprune kept must be found, in order"
    diff = np.nonzero(keep != expect)[0]
    assert diff.size == 0, f"{name}: {diff.size} verdicts differ, first at hit {diff[0]}: {all_hits[diff[0]][1][:80]!r}"
    if name == "trna":
        assert (~keep).sum() > 100, "trna over gbrna has hundreds of unzipped helices to drop"


def locus(name: str) -> str:
    """rmfmt -l: what follows the last '|' of the id, or what lies between the last
    two if the id ends in '|' (src/rmfmt.c:190-214)"""
    if "|" not in name:
        return name
    parts = name.split("|")
    if parts[-1] != "":
        return parts[-1]
    return parts[-2] if len(parts) >= 3 else name[:-1]


@pytest.mark.parametrize("name", ["efn", "trna"])
def test_order_matches_reference_rmfmt(name):
    """gm_order_hits against `rnamotif | rmfmt -l` (efn: real scores, every candidate
    printed; trna: all scores equal) over records sampled from the reference's
    test database, both outputs stored under tests/golden/gbrna/.  sort(1) breaks ties
    in every key by comparing whole lines, the library keeps enumeration order there,
    so the comparison is on the key tuples of the two orders (identical sequences)
    and on the lines as a set."""
    gbrna = os.path.join(helpers.GOLDEN, "gbrna")
    with gzip.open(os.path.join(gbrna, name + ".rnamotif.gz"), "rb") as fh:
        raw = fh.read()
    with gzip.open(os.path.join(gbrna, name + ".rmfmt_l.gz"), "rb") as fh:
        fmt = fh.read()
    all_hits = hit_lines(raw)
    ref_rows = [l.split() for l in fmt.decode("latin-1").split("\n") if l and not l.startswith("#")]
    assert len(ref_rows) == len(all_hits)

    plan = helpers.load_plan(name)
    ids, defs, seq, off = helpers.gbrna_sample()
    cands, _ = oracle_port.scan_db(plan, seq, off, bool(gpumotif.plan_field(plan, 8)))
    assert len(cands) == len(all_hits)
    scores = np.array([float(h[1].split()[1]) for h in all_hits])
    loci = [locus(i) for i in ids]
    rank = {n: k for k, n in enumerate(sorted(set(loci), key=lambda s: s.encode("latin-1")))}
    name_rank = np.array([rank[loci[r]] for r in cands["rec"]], dtype=np.int32)
    perm = gpumotif.order_hits(cands, name_rank, off, scores)
    assert sorted(perm.tolist()) == list(range(len(cands)))

    def key_of_row(row):      # name score comp pos len ...
        return (float(row[1]), row[0], int(row[2]), int(row[3]), int(row[4]))

    mine = []
    for i in perm:
        f = all_hits[i][1].decode("latin-1").split()
        mine.append((float(f[1]), locus(f[0]), int(f[2]), int(f[3]), int(f[4])))
    assert mine == [key_of_row(r) for r in ref_rows]
