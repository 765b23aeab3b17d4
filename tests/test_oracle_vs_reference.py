"""CPU: the oracle port against the instrumented REFERENCE binary (rnamotif_cand -O0,
oracle/cand_hook.c) on real GenBank records sampled from the reference's
test/gbrna.111.0.fastn -- upper case, IUPAC letters, N runs, records shorter than
the motif.  The records and the reference's candidate streams are stored under
tests/golden/gbrna/ (make_gbrna.py regenerates them from a reference build)."""
import os

import numpy as np
import pytest

from oracle import oracle_port
import helpers

GBRNA = os.path.join(helpers.GOLDEN, "gbrna")


@pytest.fixture(scope="module")
def sample():
    return helpers.gbrna_sample()


@pytest.mark.parametrize("name,flags", [
    ("trna", []), ("pk1", []), ("qu+tr", []), ("pk_j1+2", []), ("nanlin", []),
    ("trna.strict", ["-sh", "-context", "-Dctx_maxlen=5"]),
    ("score.1.strict", ["-sh", "-context", "-Dctx_maxlen=5"]),
])
def test_oracle_port_equals_reference_binary(name, flags, sample):
    """`flags`: the reference's command line the stored stream was made with."""
    plan = helpers.load_plan(name)
    hdr = np.frombuffer(plan, dtype=np.int32, count=9)
    assert bool(hdr[7]) == ("-sh" in flags), "plan and reference run disagree on -sh"
    ids, defs, seq, off = sample
    both = bool(hdr[8])
    hits, _ = oracle_port.scan_db(plan, seq, off, both)
    head, els = helpers.hits_to_rows(hits)
    ref = np.load(os.path.join(GBRNA, "cands.npz"))[name]
    nd = oracle_port.plan_n_descr(plan)
    assert len(head) == len(ref)
    if len(ref):
        assert (head == ref[:, :3]).all()
        assert (els == ref[:, 5:5 + 4 * nd]).all()
