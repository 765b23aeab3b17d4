"""Shared helpers for the parity tests."""
import gzip
import json
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLDEN = os.path.join(HERE, "golden")
REF = os.path.join(ROOT, "oracle", "_ref")


def manifest():
    with open(os.path.join(GOLDEN, "manifest.json")) as fh:
        return [e for e in json.load(fh)["entries"] if "skipped" not in e]


def golden_names():
    return [e["name"] for e in manifest()]


def load_plan(name: str) -> bytes:
    with gzip.open(os.path.join(GOLDEN, "plans", name + ".plan.gz"), "rb") as fh:
        return fh.read()


def load_extra_plan(name: str):
    """Plans without a committed candidate stream (tools/make_bench_plans.sh)."""
    path = os.path.join(GOLDEN, "plans_extra", name + ".plan.gz")
    if not os.path.exists(path):
        return None
    with gzip.open(path, "rb") as fh:
        return fh.read()


def load_score(name: str):
    """The MAIN score program as the device's pre-screen takes it (include/gpumotif_score.h;
    tools/make_bench_plans.sh), or None."""
    path = os.path.join(GOLDEN, "scores", name + ".score.gz")
    if not os.path.exists(path):
        return None
    with gzip.open(path, "rb") as fh:
        return fh.read()


def score_present(score: bytes) -> bool:
    return int(np.frombuffer(score, dtype=np.int32, count=1)[0]) != 0


def load_cands(name: str):
    z = np.load(os.path.join(GOLDEN, "cands", name + ".npz"))
    return z["head"], z["els"], z["ctx"]


def hits_to_rows(hits):
    """structured hits -> (head[n,3] = rec comp szero, els[n, 4*nd]) int32"""
    n = len(hits)
    nd = hits.dtype["el"].shape[0]
    head = np.stack([hits["rec"].astype(np.int64), hits["comp"].astype(np.int64),
                     hits["szero"].astype(np.int64)], axis=1).astype(np.int32) if n else np.zeros((0, 3), np.int32)
    els = np.zeros((n, nd, 4), dtype=np.int32)
    if n:
        els[:, :, 0] = hits["el"]["off"]
        els[:, :, 1] = hits["el"]["len"]
        els[:, :, 2] = hits["el"]["mpr"]
        els[:, :, 3] = hits["el"]["mm"]
    return head, els.reshape(n, nd * 4)


def ctx_rows(hits):
    n = len(hits)
    if not n:
        return np.zeros((0, 4), np.int32)
    return np.stack([hits["lctx_off"], hits["lctx_len"], hits["rctx_off"], hits["rctx_len"]], axis=1).astype(np.int32)


def gbrna_sample():
    """(ids, defs, seq, rec_off) of the records sampled from the reference's test database
    (tests/golden/gbrna/make_gbrna.py)."""
    from rnamotif_b200 import fastn
    with gzip.open(os.path.join(GOLDEN, "gbrna", "sample.fastn.gz"), "rb") as fh:
        return fastn.parse_fastn(fh.read())


def stream_md5(head, els, ctx=None):
    """md5 of a candidate stream in enumeration order: per candidate rec comp szero, the
    {off len mispairs mismatches} of every element and, if given, the context fields, as
    int32.  The same digest of the reference's stream is stored in tests/golden/gbrna/."""
    import hashlib
    cols = [np.asarray(head, dtype=np.int32), np.asarray(els, dtype=np.int32)]
    if ctx is not None:
        cols.append(np.asarray(ctx, dtype=np.int32))
    n = len(cols[0])
    return hashlib.md5(np.ascontiguousarray(np.concatenate([c.reshape(n, -1) for c in cols], axis=1)).tobytes()).hexdigest()


def assert_same_hits(a, b, what=""):
    ha, ea = hits_to_rows(a)
    hb, eb = hits_to_rows(b)
    assert len(ha) == len(hb), f"{what}: {len(ha)} vs {len(hb)} candidates"
    if len(ha) == 0:
        return
    bad = np.nonzero((ha != hb).any(axis=1) | (ea != eb).any(axis=1))[0]
    assert bad.size == 0, f"{what}: first difference at candidate {bad[0]}: {ha[bad[0]]} {ea[bad[0]]} vs {hb[bad[0]]} {eb[bad[0]]}"
    assert (a["seq"] == b["seq"]).all(), f"{what}: DFS ranks differ"
    assert (ctx_rows(a) == ctx_rows(b)).all(), f"{what}: context fields differ"
