"""GPU: what the context holds after an upload fails or replaces a batch (include/gpumotif.h, the
database calls).  Input an upload refuses leaves the previous batch as it was; a failure after the
upload has started leaves no database; an upload forgets the last scan's candidates.  Every case
checks the host-side values (records(), total_nt, hits()) before it scans, so no kernel ever runs
against a record table the device buffers do not match."""
import numpy as np
import pytest

from rnamotif_b200 import gpumotif, synth
from oracle import oracle_port
import helpers

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def db():
    rng = np.random.default_rng(5)
    lengths = list(rng.integers(0, 6000, size=24)) + [40001]
    ids, seq, off = synth.random_records(17, lengths, planted=True)
    plan = helpers.load_plan("trna")
    ref, _ = oracle_port.scan_db(plan, seq, off, True)
    k = 6  # the small batch: the first k records
    small_seq, small_off = seq[:int(off[k])].copy(), off[:k + 1].copy()
    small_ref, _ = oracle_port.scan_db(plan, small_seq, small_off, True)
    assert len(ref) > 0 and len(small_ref) > 0
    return plan, seq, off, ref, small_seq, small_off, small_ref


def assert_holds(ms, off):
    rec, hdr = ms.records()
    assert rec.tolist() == off.tolist() and hdr is None
    assert ms.total_nt == int(off[-1])


@pytest.mark.parametrize("kind", ["chars", "hostpack", "device"])
def test_null_pointer_with_a_larger_table_keeps_the_previous_batch(kind, db):
    import torch
    plan, seq, off, ref, small_seq, small_off, small_ref = db
    ms = gpumotif.MotifSearch(plan)
    if kind == "chars":
        ms.upload(small_seq, small_off)
        again = lambda: ms.upload_ptr(0, off)
    elif kind == "hostpack":
        ms.upload_hostpack(small_seq, small_off)
        again = lambda: ms.upload_ptr(0, off, host_pack=True)
    else:
        d_small = torch.from_numpy(small_seq).cuda()
        torch.cuda.synchronize()  # the library's streams do not wait for torch's
        ms.set_device_chars(d_small.data_ptr(), small_off)
        again = lambda: ms.set_device_chars(0, off)
    with pytest.raises(gpumotif.GpuMotifError, match="is NULL"):
        again()
    assert_holds(ms, small_off)
    helpers.assert_same_hits(ms.scan(), small_ref, f"{kind}: the small batch after a refused NULL pointer")
    ms.close()


def test_failure_after_the_batch_is_touched_leaves_no_database(db):
    import torch
    plan, seq, off, ref, small_seq, small_off, small_ref = db
    ms = gpumotif.MotifSearch(plan)
    ms.upload(small_seq, small_off)
    assert_holds(ms, small_off)
    # ~4e12 nt: the table passes every check, but the packed buffer alone would take about 2 TB, so the
    # upload fails in cudaMalloc after it has started (no kernel is launched)
    d_chars = torch.zeros(16, dtype=torch.uint8, device="cuda")
    huge = np.arange(1901, dtype=np.int64) * 0x7ffffff0
    with pytest.raises(gpumotif.GpuMotifError, match="cudaMalloc"):
        ms.set_device_chars(d_chars.data_ptr(), huge)
    with pytest.raises(gpumotif.GpuMotifError, match="no database uploaded"):
        ms.records()
    assert ms.total_nt == 0
    for call in (lambda: ms.scan(0, 0), lambda: ms.get_chars(0, 1), lambda: ms.hit_windows()):
        with pytest.raises(gpumotif.GpuMotifError, match="no database uploaded"):
            call()
    # the failed allocation is not reported again by the next upload's kernel launch checks
    ms.upload(seq, off)
    assert_holds(ms, off)
    helpers.assert_same_hits(ms.scan(), ref, "the upload after a failed allocation")
    ms.close()


def test_an_upload_forgets_the_last_scans_candidates(db):
    plan, seq, off, ref, small_seq, small_off, small_ref = db
    ms = gpumotif.MotifSearch(plan)
    ms.upload(seq, off)
    first = ms.scan()
    assert len(first) > 0
    ms.upload(seq, off)
    assert len(ms.hits()) == 0
    assert ms.hit_windows(3, 4).shape[0] == 0
    helpers.assert_same_hits(ms.scan(), first, "the rescan after the second upload")
    helpers.assert_same_hits(first, ref, "the first scan")
    ms.close()
