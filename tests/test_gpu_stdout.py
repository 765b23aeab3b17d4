"""-m gpu: byte-identical rnamotif stdout.  rnamotif_gpu (reference front end +
score/efn/printer on the host, search in libgpumotif) against
  (a) the committed md5 of the reference binary's raw stdout for each of the
      24 `make test` command lines (tests/golden/make_test_md5.json; the same
      runs pass the reference's test/*.chk goldens, oracle/check_goldens.sh), and
  (b) the reference binary itself (oracle/_ref/rnamotif), run side by side.
Needs the prebuilt programs and test inputs under oracle/_ref/ and
rnamotif_b200/host/_build/, built from the reference's sources; they skip without them.
The tests at the end of the file check the library's side of the same command lines
against the reference's stored outputs and need neither."""
import hashlib
import json
import os
import subprocess

import numpy as np
import pytest

import helpers
import shard

pytestmark = pytest.mark.gpu

GPU_BIN = os.path.join(helpers.ROOT, "rnamotif_b200", "host", "_build", "rnamotif_gpu")
REF_BIN = os.path.join(helpers.REF, "rnamotif")
DATA = os.path.join(helpers.REF, "data")
MD5 = json.load(open(os.path.join(helpers.GOLDEN, "make_test_md5.json")))

have = os.path.exists(GPU_BIN) and os.path.exists(os.path.join(DATA, "test", "gbrna.111.0.fastn"))


def run(binary, name, extra_env=None):
    flags = ["-sh", "-context", "-Dctx_maxlen=5"] if name.endswith(".strict") else []
    env = dict(os.environ, EFNDATA=os.path.join(DATA, "efndata"))
    env.update(extra_env or {})
    r = subprocess.run([binary, *flags, "-descr", name + ".descr", "gbrna.111.0.fastn"],
                       cwd=os.path.join(DATA, "test"), env=env, capture_output=True, timeout=1200)
    assert r.returncode == 0, r.stderr.decode(errors="replace")[-2000:]
    return r.stdout


@pytest.mark.skipif(not have, reason="oracle/_ref or rnamotif_gpu not built")
@pytest.mark.parametrize("name", sorted(MD5))
def test_make_test_stdout_md5(name):
    out = run(GPU_BIN, name)
    assert hashlib.md5(out).hexdigest() == MD5[name]["md5"], f"{name}: stdout differs from the reference"


@pytest.mark.skipif(not (have and os.path.exists(REF_BIN)), reason="reference binary not built")
@pytest.mark.parametrize("name", ["trna", "pk1", "qu+tr.strict", "getbest"])
def test_stdout_equals_reference_binary_small_batches(name):
    # small batches: records split across many uploads, score state carried across
    out = run(GPU_BIN, name, {"GPUMOTIF_BATCH_NT": "300000"})
    ref = run(REF_BIN, name)
    assert out == ref


@pytest.mark.skipif(not have, reason="oracle/_ref or rnamotif_gpu not built")
@pytest.mark.parametrize("name", ["trna", "getbest", "pk1.strict"])
def test_stdout_with_sharded_scan(name):
    """The host driver's in-process sharding (GPUMOTIF_DEVICES): the batch is cut
    into ranges of start positions, one context each, and the candidate lists are
    merged before the (stateful) score replay.  Two contexts on device 0 exercise
    the same code as two GPUs; with more than one GPU visible use them."""
    import torch
    devs = "0,1,0" if torch.cuda.device_count() > 1 else "0,0,0"
    out = run(GPU_BIN, name, {"GPUMOTIF_DEVICES": devs, "GPUMOTIF_BATCH_NT": "1000000"})
    assert hashlib.md5(out).hexdigest() == MD5[name]["md5"]


PRUNE_BIN = os.path.join(helpers.REF, "rmprune")


@pytest.mark.skipif(not (have and os.path.exists(REF_BIN) and os.path.exists(PRUNE_BIN)),
                    reason="reference binaries (rnamotif, rmprune) not built")
@pytest.mark.parametrize("name", ["trna", "score.1"])
def test_prune_option_equals_rnamotif_piped_through_rmprune(name):
    """GPUMOTIF_PRUNE=1 (gm_prune_hits on the accepted hits' records, SURVEY 8 f4) prints
    byte for byte what `rnamotif ... | rmprune` prints.  The host side of this is also
    checked without a GPU in tests/test_host_driver_cpu.py."""
    ref = run(REF_BIN, name)
    want = subprocess.run([PRUNE_BIN], input=ref, capture_output=True, timeout=600, check=True).stdout
    got = run(GPU_BIN, name, {"GPUMOTIF_PRUNE": "1"})
    assert got == want


RMFMT = os.path.join(helpers.REF, "rmfmt")


@pytest.mark.skipif(not (have and os.path.exists(RMFMT)), reason="oracle/_ref (rmfmt, test data) or rnamotif_gpu not built")
@pytest.mark.parametrize("name", sorted(MD5))
def test_make_test_chk_goldens(name):
    """The reference's own `make test` (test/Makefile:30-245): rnamotif ... | rmfmt -l
    diffed against test/<name>.chk -- with rnamotif_gpu in rnamotif's place and the
    reference's rmfmt and .chk files as they are."""
    out = run(GPU_BIN, name)
    fmt = subprocess.run([RMFMT, "-l"], input=out, capture_output=True, timeout=600, cwd=os.path.join(DATA, "test"))
    assert fmt.returncode == 0, fmt.stderr.decode(errors="replace")[-500:]
    with open(os.path.join(DATA, "test", name + ".chk"), "rb") as fh:
        assert fmt.stdout == fh.read(), f"{name}: differs from the reference's {name}.chk"


@pytest.mark.skipif(not have, reason="oracle/_ref (test data) or rnamotif_gpu not built")
@pytest.mark.parametrize("name", sorted(MD5))
def test_fmt_option_chk_goldens(name):
    """GPUMOTIF_FMT=l: rnamotif_gpu prints what `rnamotif ... | rmfmt -l` prints (gm_rmfmt):
    the reference's 24 .chk files with no reference program in the pipe."""
    out = run(GPU_BIN, name, {"GPUMOTIF_FMT": "l"})
    with open(os.path.join(DATA, "test", name + ".chk"), "rb") as fh:
        assert out == fh.read(), f"{name}: differs from the reference's {name}.chk"


# ---- the library on the device against the reference's stored outputs ----------------------
# Records sampled from the reference's test database and what the reference printed over them
# (tests/golden/gbrna/, make_gbrna.py): the digest of rnamotif_cand -O0's candidate stream for
# every `make test` command line, the same of the candidates RM_score accepts, rnamotif's stdout
# and that stdout through `rmfmt -l`.  They need no reference build.

GBRNA = os.path.join(helpers.GOLDEN, "gbrna")
STREAMS = json.load(open(os.path.join(GBRNA, "streams.json")))
PURE_SCORE = {"score.1", "score.2", "mp.ends"}  # score programs that only filter (tests/test_score_prescreen.py)


def _base(name):
    return name[:-len(".strict")] if name.endswith(".strict") else name


SCORED = [n for n in sorted(MD5) if helpers.load_score(_base(n)) is not None
          and helpers.score_present(helpers.load_score(_base(n)))]


@pytest.fixture(scope="module")
def sample():
    ids, defs, seq, off = helpers.gbrna_sample()
    return seq, off


def assert_stream(hits, want, what):
    assert len(hits) == want["n"], f"{what}: {len(hits)} candidates, the reference {want['n']}"
    if want["n"]:
        head, els = helpers.hits_to_rows(hits)
        got = helpers.stream_md5(head, els, helpers.ctx_rows(hits) if want["context"] else None)
        assert got == want["md5"], f"{what}: candidate stream differs from the reference's"


@pytest.mark.parametrize("name", sorted(MD5))
def test_device_stream_equals_reference_on_gbrna_sample(name, sample):
    """One upload of every sampled record: the candidate stream is the reference's, and it
    is not empty for any command line that prints hits over the whole database."""
    from rnamotif_b200 import gpumotif
    want = STREAMS[name]
    assert want["n"] > 0 or MD5[name]["hits"] == 0, f"{name}: the sample holds none of its hits"
    ms = gpumotif.MotifSearch(helpers.load_plan(name))
    assert_stream(ms.find_motif(*sample), want, name)
    ms.close()


@pytest.mark.parametrize("name", ["trna", "pk1", "qu+tr.strict", "getbest"])
def test_device_small_uploads_equal_reference_stream(name, sample):
    """The records over many uploads of one context (at most 30 knt each), the candidate
    lists of the uploads concatenated in order, record numbers offset by each upload's first."""
    from rnamotif_b200 import gpumotif
    seq, off = sample
    ms = gpumotif.MotifSearch(helpers.load_plan(name))
    parts, a, n_rec = [], 0, len(off) - 1
    while a < n_rec:
        b = a + 1
        while b < n_rec and off[b + 1] - off[a] <= 30000:
            b += 1
        ms.upload(seq[off[a]:off[b]], off[a:b + 1] - off[a])
        h = ms.scan()
        h["rec"] += np.uint32(a)
        parts.append(h)
        a = b
    ms.close()
    assert len(parts) > 5
    assert_stream(np.concatenate(parts), STREAMS[name], name)


@pytest.mark.parametrize("name", ["trna", "getbest", "pk1.strict"])
def test_device_range_shards_merged_equal_reference_stream(name, sample):
    """The batch cut into three ranges of start positions, one context each (on two GPUs
    where there are), the candidate lists merged into enumeration order (tests/shard.py)."""
    import torch
    from rnamotif_b200 import gpumotif
    seq, off = sample
    devs = [0, 1, 0] if torch.cuda.device_count() > 1 else [0, 0, 0]
    plan = helpers.load_plan(name)
    parts = []
    for dev, (lo, hi) in zip(devs, shard.shard_ranges(int(off[-1]), len(devs))):
        ms = gpumotif.MotifSearch(plan, device=dev)
        ms.upload(seq, off)
        parts.append(ms.scan(lo, hi))
        ms.close()
    assert_stream(shard.merge_hits(parts), STREAMS[name], name)


@pytest.mark.parametrize("name", SCORED)
def test_device_prescreen_against_reference_verdicts_on_gbrna_sample(name, sample):
    """The score section's pre-screen on the device: it never drops a candidate the reference
    accepts, and for programs that only filter it keeps exactly the accepted ones."""
    from rnamotif_b200 import gpumotif
    want = STREAMS[name]
    ms = gpumotif.MotifSearch(helpers.load_plan(name))
    ms.set_score(helpers.load_score(_base(name)))
    kept = ms.find_motif(*sample)
    st = ms.stats()
    ms.close()
    assert len(kept) + st.n_score_rejected == want["n"]
    if _base(name) in PURE_SCORE:
        assert_stream(kept, want["accepted"], name + " (accepted)")
    else:
        assert len(kept) >= want["accepted"]["n"]


@pytest.mark.parametrize("name", sorted(MD5))
def test_gm_rmfmt_prints_what_rmfmt_l_printed(name, tmp_path):
    """gm_rmfmt (GPUMOTIF_FMT=l): from rnamotif's stdout, what `rmfmt -l` printed from it."""
    import ctypes as C
    import ctypes.util
    import gzip
    from rnamotif_b200 import gpumotif

    def stored(what):
        with gzip.open(os.path.join(GBRNA, f"{name}.{what}.gz"), "rb") as fh:
            return fh.read()

    L = gpumotif.lib()
    L.gm_rmfmt.argtypes = [C.c_char_p, C.c_size_t, C.c_int, C.c_void_p]
    libc = C.CDLL(ctypes.util.find_library("c"))
    libc.fopen.restype = C.c_void_p
    libc.fopen.argtypes = [C.c_char_p, C.c_char_p]
    libc.fclose.argtypes = [C.c_void_p]
    raw = stored("rnamotif")
    path = str(tmp_path / "fmt.out")
    fp = libc.fopen(path.encode(), b"w")
    assert fp
    rc = L.gm_rmfmt(raw, len(raw), 1, fp)
    assert libc.fclose(fp) == 0
    assert rc == 0, L.gm_last_error()
    assert open(path, "rb").read() == stored("rmfmt_l"), f"{name}: differs from `rmfmt -l`"
