#!/usr/bin/env python3
"""End-to-end rate from pinned host memory of FASTA text uploaded as it is and compressed as BGZF:

    text      gm_db_upload_fastn         the text, about 1.02 B/nt
    bgzf6     gm_db_upload_fastn_bgzf    the text as bgzip writes it (level 6), inflated on the device
    bgzf1     gm_db_upload_fastn_bgzf    the same at level 1
    2bit      gm_db_upload_2bit          the records as a .2bit file, 0.25 B/nt

For trna, ire, score.1, pk1 and qu+tr over 1024 x 1 Mnt uniform acgt records as 60-column FASTA, a
step is one upload + gm_scan (candidates sorted in host memory), timed by the host clock around a
device synchronise; the upload call alone is timed too (the FASTA uploads return once the record
table is known: after the copy, the inflate and the device reader; the pack runs on).  Compression
happens before any timing.  The legs run in one process, alternating step by step after a warm-up;
the resident rate (database already packed on the device) is given beside them.  The candidate
arrays of all legs and the resident run must be byte-equal, else the script fails.  ire and
score.1 run with their score pre-screen on, as bench.py's configs do.

    python profiles/bgzf_e2e.py --out DIR [--steps 10] [--warmup 2] [--mnt 1024]

writes DIR/bgzf_e2e.json with the card's name, power limit and SM clock, queried in the same run.
"""
import argparse
import concurrent.futures
import gzip
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from rnamotif_b200 import bgzf, gpumotif, twobit  # noqa: E402

PLAN_DIR = os.path.join(ROOT, "rnamotif_b200", "plans")
WORKLOADS = ["trna", "ire", "score.1", "pk1", "qu+tr"]
LEGS = ["text", "bgzf6", "bgzf1", "2bit"]


def load(name, kind):
    path = os.path.join(PLAN_DIR, f"{name}.{kind}.gz")
    if not os.path.exists(path):
        return None
    with gzip.open(path, "rb") as fh:
        b = fh.read()
    if kind == "score" and not int(np.frombuffer(b, dtype=np.int32, count=1)[0]):
        return None
    return b


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm,temperature.gpu"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                             check=True, capture_output=True, text=True).stdout.strip()
    except (OSError, subprocess.CalledProcessError) as e:
        return {"error": str(e)}
    return dict(zip(q.split(","), [v.strip() for v in out.split(",")]))


def fasta(chars, rec_off, width=60):
    """60-column FASTA of the records (numpy, no per-line Python loop)."""
    parts = []
    for r in range(len(rec_off) - 1):
        s = chars[rec_off[r]:rec_off[r + 1]]
        n = len(s)
        full = n // width * width
        body = np.concatenate([s[:full].reshape(-1, width), np.full((full // width, 1), 10, np.uint8)], axis=1).ravel()
        tail = np.concatenate([s[full:], [10]]).astype(np.uint8) if n > full else np.zeros(0, np.uint8)
        parts += [np.frombuffer(b">syn%06d\n" % r, dtype=np.uint8), body, tail]
    return np.concatenate(parts)


def compress(text, level, threads):
    """BGZF at `level`, members of 0xff00 bytes compressed in parallel (zlib releases the GIL)."""
    piece = 0xff00 * 256
    with concurrent.futures.ThreadPoolExecutor(threads) as ex:
        out = list(ex.map(lambda o: bgzf.write_bgzf(text[o:o + piece], level=level, eof=False), range(0, len(text), piece)))
    return b"".join(out) + bgzf.EOF_BLOCK


def pinned(b):
    import torch
    t = torch.empty(len(b), dtype=torch.uint8, pin_memory=True)
    t.numpy()[:] = np.frombuffer(b, dtype=np.uint8)
    return t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--mnt", type=int, default=1024, help="records of 1 Mnt")
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bgzf_e2e.py: no CUDA device; libgpumotif has no CPU path")
    os.makedirs(args.out, exist_ok=True)

    n_rec = args.mnt
    rec_off = np.concatenate([[0], np.cumsum([1_000_000] * n_rec)]).astype(np.int64)
    total = int(rec_off[-1])
    lut = torch.tensor(list(b"acgt"), dtype=torch.uint8, device="cuda")
    g = torch.Generator(device="cuda")
    g.manual_seed(1001)
    d_chars = lut[torch.randint(0, 4, (total,), generator=g, device="cuda")]
    chars = d_chars.cpu().numpy()
    t0 = time.perf_counter()
    text = fasta(chars, rec_off)
    h_text = pinned(text.tobytes())
    threads = len(os.sched_getaffinity(0))
    gz = {}
    for lv in (6, 1):
        gz[lv] = pinned(compress(memoryview(text), lv, threads))
    f = twobit.write_2bit(["syn%06d" % r for r in range(n_rec)], chars, rec_off)
    h_2bit = pinned(f)
    tb = twobit.read_2bit(f)
    del f, text, chars
    t_prep = time.perf_counter() - t0
    _, dna_off, nblk = tb.tables()

    res = {"card_before": card(), "database": f"{n_rec} x 1000000 nt uniform acgt (seed 1001) as 60-column FASTA, "
                                              f"{total} nt, text {h_text.numel()} bytes, BGZF level 6 {gz[6].numel()} "
                                              f"bytes, level 1 {gz[1].numel()} bytes, .2bit {h_2bit.numel()} bytes",
           "steps": args.steps, "warmup": args.warmup, "timing": "host clock around upload + gm_scan (which ends in a "
           "device synchronise and leaves the sorted candidates in host memory), legs alternating step by step; "
           "upload_ms: the upload call alone", "cpus": threads, "prep_s": t_prep, "workloads": []}
    ok_all = True
    for name in args.workloads.split(","):
        plan, score = load(name, "plan"), load(name, "score")
        strands = 2 if int(np.frombuffer(plan, dtype=np.int32, count=9)[8]) else 1
        ms = gpumotif.MotifSearch(plan)
        if score is not None:
            ms.set_score(score)
        legs = {
            "text": lambda: ms.upload_fastn_ptr(h_text.data_ptr(), h_text.numel()),
            "bgzf6": lambda: ms.upload_fastn_bgzf_ptr(gz[6].data_ptr(), gz[6].numel()),
            "bgzf1": lambda: ms.upload_fastn_bgzf_ptr(gz[1].data_ptr(), gz[1].numel()),
            "2bit": lambda: ms.upload_2bit_ptr(h_2bit.data_ptr(), h_2bit.numel(), dna_off, rec_off, nblk),
        }
        times = {k: [] for k in legs}
        t_up = {k: [] for k in legs}
        h2d = {}
        hits = {}

        def step(leg):
            torch.cuda.synchronize()
            t = time.perf_counter()
            legs[leg]()
            tu = time.perf_counter() - t
            ms.scan(0, total, strands, copy=False)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t
            h2d[leg] = int(ms.stats().h2d_bytes)
            return dt, tu

        for i in range(args.warmup + args.steps):
            for leg in legs:
                dt, tu = step(leg)
                if i >= args.warmup:
                    times[leg].append(dt)
                    t_up[leg].append(tu)
        for leg in legs:
            step(leg)
            hits[leg] = ms.hits(copy=True)
        ms.set_device_chars(d_chars.data_ptr(), rec_off)
        ms.scan(0, total, strands, copy=False)
        t_res = []
        for _ in range(args.steps):
            torch.cuda.synchronize()
            t = time.perf_counter()
            ms.scan(0, total, strands, copy=False)
            torch.cuda.synchronize()
            t_res.append(time.perf_counter() - t)
        hits["resident"] = ms.hits(copy=True)
        ms.close()
        ref = hits["resident"].tobytes()
        same = {k: v.tobytes() == ref for k, v in hits.items()}
        ok_all = ok_all and all(same.values())
        work = float(total) * strands
        entry = {"workload": name, "strands": strands, "score_prescreen": score is not None,
                 "candidates": int(len(hits["resident"])), "candidates_byte_equal": same,
                 "resident": {"G_strand_nt_s": work / np.median(t_res) / 1e9, "ms_per_step": 1e3 * float(np.median(t_res))}}
        for leg in legs:
            med = float(np.median(times[leg]))
            entry[leg] = {"G_strand_nt_s": work / med / 1e9, "ms_per_step": 1e3 * med,
                          "ms_per_step_min_max": [1e3 * min(times[leg]), 1e3 * max(times[leg])],
                          "upload_ms": 1e3 * float(np.median(t_up[leg])),
                          "h2d_bytes_per_step": h2d[leg], "h2d_bytes_per_nt": h2d[leg] / total}
        entry["card_after"] = card()
        res["workloads"].append(entry)
        print(json.dumps({k: entry[k] for k in ("workload", "candidates", "candidates_byte_equal")} |
                         {k: round(entry[k]["G_strand_nt_s"], 1) for k in ["resident"] + LEGS} |
                         {k + "_upload_ms": round(entry[k]["upload_ms"], 2) for k in LEGS}), flush=True)
    res["ok"] = ok_all
    with open(os.path.join(args.out, "bgzf_e2e.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    if not ok_all:
        raise SystemExit("bgzf_e2e.py: the candidate arrays differ between the legs")


if __name__ == "__main__":
    main()
