#!/usr/bin/env python3
"""Regenerate tests/golden/gbrna/ from the REFERENCE build (oracle/_ref: `make -C oracle ref`).

The reference's own programs run over a sample of its test database (test/gbrna.111.0.fastn:
real GenBank records with upper case, IUPAC letters, N runs and records shorter than the
motifs): its first 400 records and, for every `make test` command line that none of them
gives a hit, the first EXTRA records past them on which the reference accepts or holds
a candidate of that command line.  What they print over the sample is stored here:

  sample.fastn.gz          the sampled records, in the database's order
  streams.json             per command line of the reference's `make test`: the candidate
                           stream of rnamotif_cand -O0 (oracle/cand_hook.c), run as
                           tests/golden/make_golden.py runs it (malloc_ff.so preloaded): its
                           length, helpers.stream_md5 and whether it carries context fields;
                           the same of the candidates RM_score accepts (`accepted`)
  cands.npz                the whole stream (one int row per candidate) of the command lines in
                           ORACLE_NAMES
  <name>.rnamotif.gz       the stdout of `rnamotif [flags] -descr <name>.descr`
  <name>.rmfmt_l.gz        the same piped through `rmfmt -l`

tests/test_oracle_vs_reference.py, tests/test_prune.py and tests/test_gpu_stdout.py compare
against them.
"""
import gzip
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(HERE)))
REF = os.path.join(ROOT, "oracle", "_ref")
DATA = os.path.join(REF, "data", "test")
DUMP = os.path.join(ROOT, "rnamotif_b200", "host", "_build", "rm_plan_dump")
N_RECORDS = 400
EXTRA = 2
STRICT = ["-sh", "-context", "-Dctx_maxlen=5"]
MAKE_TEST = [b + s for b in ("bulge", "efn", "getbest", "mp.ends", "nanlin", "pk1", "pk_j1+2", "qu+tr", "score.1",
                               "score.2", "sprintf", "trna") for s in ("", ".strict")]


ORACLE_NAMES = ["trna", "pk1", "qu+tr", "pk_j1+2", "nanlin", "trna.strict", "score.1.strict"]


def flags_of(name):
    return STRICT if name.endswith(".strict") else []


def records(data):
    """byte ranges of the records of a FASTA text"""
    starts = [0] + [i + 1 for i in range(len(data) - 1) if data[i] == 0x0A and data[i + 1] == 0x3E]
    return list(zip(starts, starts[1:] + [len(data)]))


def cand_stream(name, db, env, tmp):
    """rnamotif_cand -O0's candidate stream of one command line over `db`: int32 rows"""
    cf = os.path.join(tmp, name + ".cand")
    subprocess.run([os.path.join(REF, "rnamotif_cand"), "-O0", *flags_of(name), "-descr", name + ".descr", db],
                   cwd=DATA, check=True, capture_output=True,
                   env=dict(env, GM_CAND_FILE=cf, LD_PRELOAD=os.path.join(REF, "malloc_ff.so")))
    rows = [ln.split() for ln in open(cf)] if os.path.exists(cf) else []  # no file: no candidate
    os.unlink(cf) if os.path.exists(cf) else None
    return np.array(rows, dtype=np.int32).reshape(len(rows), -1) if rows else np.zeros((0, 0), np.int32)


def digest(helpers, a):
    nd = int(a[0, 4]) if len(a) else 0
    ctx = a.shape[1] > 5 + 4 * nd
    return {"n": len(a), "context": bool(ctx),
            "md5": helpers.stream_md5(a[:, :3], a[:, 5:5 + 4 * nd], a[:, 5 + 4 * nd:] if ctx else None) if len(a) else None}


def main():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import helpers
    env = dict(os.environ, EFNDATA=os.path.join(REF, "data", "efndata"), LC_ALL="C")
    full = os.path.join(DATA, "gbrna.111.0.fastn")
    data = open(full, "rb").read()
    recs = records(data)
    with tempfile.TemporaryDirectory() as tmp:
        pick = set(range(N_RECORDS))
        for name in MAKE_TEST:
            a = cand_stream(name, full, env, tmp)
            hit_recs = sorted({int(r) for r in a[a[:, 3] != 0, 0]}) if len(a) else []
            if hit_recs and not any(r < N_RECORDS for r in hit_recs):
                pick.update([r for r in hit_recs if r >= N_RECORDS][:EXTRA])
        sample = b"".join(data[recs[r][0]:recs[r][1]] for r in sorted(pick))
        db = os.path.join(tmp, "sample.fastn")
        open(db, "wb").write(sample)
        with gzip.GzipFile(os.path.join(HERE, "sample.fastn.gz"), "wb", 9, mtime=0) as fh:
            fh.write(sample)
        streams, cands = {}, {}
        for name in MAKE_TEST:
            if os.path.exists(DUMP):  # the committed plan must be what the reference's front end makes
                plan_file = os.path.join(tmp, name + ".plan")
                subprocess.run([DUMP, *flags_of(name), "-descr", name + ".descr"], cwd=DATA, check=True,
                               capture_output=True, env=dict(env, GM_PLAN_OUT=plan_file))
                assert open(plan_file, "rb").read() == helpers.load_plan(name), f"{name}: committed plan is stale"
            a = cands[name] = cand_stream(name, db, env, tmp)
            streams[name] = dict(digest(helpers, a), accepted=digest(helpers, a[a[:, 3] == 2] if len(a) else a))
        with open(os.path.join(HERE, "streams.json"), "w") as fh:
            json.dump(streams, fh, indent=1, sort_keys=True)
        np.savez_compressed(os.path.join(HERE, "cands.npz"), **{k: cands[k] for k in ORACLE_NAMES})
        for name in MAKE_TEST:
            raw = subprocess.run([os.path.join(REF, "rnamotif"), *flags_of(name), "-descr", name + ".descr", db],
                                 cwd=DATA, env=env, check=True, capture_output=True).stdout
            fmt = subprocess.run([os.path.join(REF, "rmfmt"), "-l"], input=raw, cwd=DATA, env=env, check=True,
                                 capture_output=True).stdout
            for suffix, text in (("rnamotif", raw), ("rmfmt_l", fmt)):
                with gzip.GzipFile(os.path.join(HERE, f"{name}.{suffix}.gz"), "wb", 9, mtime=0) as fh:
                    fh.write(text)


if __name__ == "__main__":
    main()
