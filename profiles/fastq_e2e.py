#!/usr/bin/env python3
"""End-to-end rate from pinned host memory of sequencing reads uploaded as characters, as FASTQ text and
as BGZF-compressed FASTQ:

    chars     gm_db_upload_chars         the reads' characters, parsed on the host beforehand (1 B/nt)
    fastq     gm_db_upload_fastq         the FASTQ text as it sits in the file, read on the device
    bgzf6     gm_db_upload_fastq_bgzf    the text as bgzip writes it (level 6), inflated on the device
    bgzf1     gm_db_upload_fastq_bgzf    the same at level 1

The database is about 1 Gnt of 150-nt reads from synth.random_reads (seed 150: planted stem-loops,
'N' and '.' calls) in four-line FASTQ with Illumina-binned quality strings.  For trna, ire, score.1,
pk1 and qu+tr a step is one upload + gm_scan (candidates sorted in host memory), timed by the host
clock around a device synchronise; the upload call alone is timed too.  Compression happens before
any timing.  The legs run in one process, alternating step by step after a warm-up.  Beside them:
  resident         the reads already packed on the device (gm_db_set_device_chars), scan only
  resident_1mnt    the same characters cut into 1 Mnt records: what millions of short records cost
                   the search itself
  small_scan_ms    a scan of the first 1 Mnt of the reads (host work per scan over the whole record
                   table shows here)
The candidate arrays of all legs and the resident run must be byte-equal, else the script fails.
ire and score.1 run with their score pre-screen on, as bench.py's configs do.

--min-qual Q adds three legs with low-quality masking (gm_ctx_set_min_quality, offset 33) at Q,
alternating with the others:
    chars_q   gm_db_upload_chars         the reads with every base of quality below Q written as n
                                         on the host
    fastq_q   gm_db_upload_fastq         the FASTQ text, masked on the device
    bgzf6_q   gm_db_upload_fastq_bgzf    the level-6 BGZF text, masked on the device
whose candidate arrays must be byte-equal to each other (fastq_q and bgzf6_q to chars_q), else the
script fails.  Comparing upload_ms of fastq with fastq_q, and of bgzf6 with bgzf6_q, gives what the
masking pass costs the upload call.

    python profiles/fastq_e2e.py --out DIR [--steps 5] [--warmup 1] [--mnt 1000] [--min-qual Q]

writes DIR/fastq_e2e.json (with --min-qual: DIR/fastq_mask_e2e.json) with the card's name, power
limit and SM clock, queried in the same run.
"""
import argparse
import concurrent.futures
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

from rnamotif_b200 import bgzf, fastq, gpumotif, synth  # noqa: E402
from bgzf_e2e import card, load, pinned, WORKLOADS  # noqa: E402

LEGS = ["chars", "fastq", "bgzf6", "bgzf1"]
MASKED_LEGS = ["chars_q", "fastq_q", "bgzf6_q"]
READ = 150
ID_DIGITS = 9


def fastq_text(seq, n_reads, qual):
    """Four-line FASTQ of n_reads reads of READ nt: '@read%09d', the read, '+', the quality string
    (numpy, no per-record Python loop; equal to fastq.write_fastq, checked on a prefix)."""
    head = 1 + 4 + ID_DIGITS + 1
    width = head + READ + 3 + READ + 1
    rows = np.empty((n_reads, width), dtype=np.uint8)
    rows[:, 0:5] = np.frombuffer(b"@read", dtype=np.uint8)
    r = np.arange(n_reads, dtype=np.int64)
    for k in range(ID_DIGITS):
        rows[:, 5 + ID_DIGITS - 1 - k] = ord("0") + (r // 10 ** k) % 10
    rows[:, head - 1] = 10
    rows[:, head:head + READ] = seq.reshape(n_reads, READ)
    rows[:, head + READ:head + READ + 3] = np.frombuffer(b"\n+\n", dtype=np.uint8)
    rows[:, head + READ + 3:width - 1] = qual.reshape(n_reads, READ)
    rows[:, width - 1] = 10
    return rows.reshape(-1)


def compress(text, level, threads):
    """BGZF at `level`, members of 0xff00 bytes compressed in parallel (zlib releases the GIL)."""
    piece = 0xff00 * 256
    with concurrent.futures.ThreadPoolExecutor(threads) as ex:
        out = list(ex.map(lambda o: bgzf.write_bgzf(text[o:o + piece], level=level, eof=False), range(0, len(text), piece)))
    return b"".join(out) + bgzf.EOF_BLOCK


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--mnt", type=int, default=1000, help="Mnt of reads")
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--min-qual", type=int, default=0, help="add the masked legs at this minimum base quality")
    args = ap.parse_args()
    if not 0 <= args.min_qual <= 93:
        raise SystemExit("fastq_e2e.py: --min-qual must be in [0, 93]")
    legs_run = LEGS + (MASKED_LEGS if args.min_qual else [])
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("fastq_e2e.py: no CUDA device; libgpumotif has no CPU path")
    os.makedirs(args.out, exist_ok=True)

    t0 = time.perf_counter()
    n_reads = args.mnt * 1_000_000 // READ
    ids, seq, rec_off = synth.random_reads(150, np.full(n_reads, READ))
    total = int(rec_off[-1])
    # Illumina-binned quality values (the four bins of recent instruments)
    g = torch.Generator(device="cuda")
    g.manual_seed(150)
    bins = torch.tensor(list(b"#,:F"), dtype=torch.uint8, device="cuda")
    probs = torch.tensor([0.02, 0.03, 0.10, 0.85], device="cuda")
    qual = bins[torch.multinomial(probs, total, replacement=True, generator=g)].cpu().numpy()
    text = fastq_text(seq, n_reads, qual)
    k = 1000
    assert text[:k * (len(text) // n_reads)].tobytes() == fastq.write_fastq(
        ["read%09d" % i for i in range(k)], seq, rec_off[:k + 1], [qual[i * READ:(i + 1) * READ] for i in range(k)])
    assert (fastq.parse_fastq(text[:k * (len(text) // n_reads)].tobytes())[2] == rec_off[:k + 1]).all()
    h_chars = pinned(seq.tobytes())
    if args.min_qual:
        seq_q = seq.copy()
        seq_q[qual < 33 + args.min_qual] = ord("n")
        masked_share = float((qual < 33 + args.min_qual).mean())
        h_chars_q = pinned(seq_q.tobytes())
        del seq_q
    h_text = pinned(text.tobytes())
    threads = len(os.sched_getaffinity(0))
    gz = {lv: pinned(compress(memoryview(text), lv, threads)) for lv in (6, 1)}
    d_chars = torch.from_numpy(seq).cuda()
    del text, qual, ids
    t_prep = time.perf_counter() - t0
    mnt_off = np.arange(0, total + 1, 1_000_000, dtype=np.int64)
    if mnt_off[-1] != total:
        mnt_off = np.append(mnt_off, total)

    res = {"card_before": card(),
           "database": f"{n_reads} reads of {READ} nt (synth.random_reads seed 150), {total} nt, FASTQ text "
                       f"{h_text.numel()} bytes, BGZF level 6 {gz[6].numel()} bytes, level 1 {gz[1].numel()} bytes",
           "steps": args.steps, "warmup": args.warmup, "timing": "host clock around upload + gm_scan (which ends in a "
           "device synchronise and leaves the sorted candidates in host memory), legs alternating step by step; "
           "upload_ms: the upload call alone", "cpus": threads, "prep_s": t_prep, "workloads": []}
    if args.min_qual:
        res["min_qual"] = {"min_qual": args.min_qual, "qual_offset": 33, "bases_masked": masked_share}
    ok_all = True
    for name in args.workloads.split(","):
        plan, score = load(name, "plan"), load(name, "score")
        strands = 2 if int(np.frombuffer(plan, dtype=np.int32, count=9)[8]) else 1
        ms = gpumotif.MotifSearch(plan)
        if score is not None:
            ms.set_score(score)
        legs = {
            "chars": lambda: ms.upload_ptr(h_chars.data_ptr(), rec_off),
            "fastq": lambda: ms.upload_fastq_ptr(h_text.data_ptr(), h_text.numel()),
            "bgzf6": lambda: ms.upload_fastq_bgzf_ptr(gz[6].data_ptr(), gz[6].numel()),
            "bgzf1": lambda: ms.upload_fastq_bgzf_ptr(gz[1].data_ptr(), gz[1].numel()),
        }
        if args.min_qual:
            legs |= {
                "chars_q": lambda: ms.upload_ptr(h_chars_q.data_ptr(), rec_off),
                "fastq_q": legs["fastq"],
                "bgzf6_q": legs["bgzf6"],
            }
        times = {k: [] for k in legs}
        t_up = {k: [] for k in legs}
        h2d, hits = {}, {}

        def step(leg):
            if args.min_qual:
                ms.set_min_quality(args.min_qual if leg in MASKED_LEGS else 0)
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

        def resident(off):
            ms.set_device_chars(d_chars.data_ptr(), off)
            ms.scan(0, total, strands, copy=False)
            t_res = []
            for _ in range(args.steps):
                torch.cuda.synchronize()
                t = time.perf_counter()
                ms.scan(0, total, strands, copy=False)
                torch.cuda.synchronize()
                t_res.append(time.perf_counter() - t)
            return float(np.median(t_res))

        t_1m = resident(mnt_off)
        t_res = resident(rec_off)
        hits["resident"] = ms.hits(copy=True)
        t_small = []
        for _ in range(20):
            t = time.perf_counter()
            ms.scan(0, 1_000_000, strands, copy=False)
            t_small.append(time.perf_counter() - t)
        ms.close()
        ref = hits["resident"].tobytes()
        same = {k: v.tobytes() == ref for k, v in hits.items() if k not in MASKED_LEGS}
        if args.min_qual:
            ref_q = hits["chars_q"].tobytes()
            same |= {k: hits[k].tobytes() == ref_q for k in MASKED_LEGS[1:]}
        ok_all = ok_all and all(same.values())
        work = float(total) * strands
        entry = {"workload": name, "strands": strands, "score_prescreen": score is not None,
                 "candidates": int(len(hits["resident"])), "candidates_byte_equal": same,
                 "resident": {"G_strand_nt_s": work / t_res / 1e9, "ms_per_step": 1e3 * t_res},
                 "resident_1mnt": {"G_strand_nt_s": work / t_1m / 1e9, "ms_per_step": 1e3 * t_1m},
                 "small_scan_ms": 1e3 * float(np.median(t_small))}
        if args.min_qual:
            entry["candidates_masked"] = int(len(hits["chars_q"]))
        for leg in legs:
            med = float(np.median(times[leg]))
            entry[leg] = {"G_strand_nt_s": work / med / 1e9, "ms_per_step": 1e3 * med,
                          "ms_per_step_min_max": [1e3 * min(times[leg]), 1e3 * max(times[leg])],
                          "upload_ms": 1e3 * float(np.median(t_up[leg])),
                          "h2d_bytes_per_step": h2d[leg], "h2d_bytes_per_nt": h2d[leg] / total}
        entry["card_after"] = card()
        res["workloads"].append(entry)
        print(json.dumps({k: entry[k] for k in ("workload", "candidates", "candidates_byte_equal", "small_scan_ms")} |
                         {k: round(entry[k]["G_strand_nt_s"], 1) for k in ["resident", "resident_1mnt"] + legs_run} |
                         {k + "_upload_ms": round(entry[k]["upload_ms"], 2) for k in legs_run}), flush=True)
    res["ok"] = ok_all
    with open(os.path.join(args.out, "fastq_mask_e2e.json" if args.min_qual else "fastq_e2e.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    if not ok_all:
        raise SystemExit("fastq_e2e.py: the candidate arrays differ between the legs")


if __name__ == "__main__":
    main()
