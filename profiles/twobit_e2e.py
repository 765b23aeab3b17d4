#!/usr/bin/env python3
"""End-to-end rate from pinned host memory of the three ways a database reaches the device:

    chars     gm_db_upload_chars            1 B/nt, packed to 4-bit codes on the device
    hostpack  gm_db_upload_chars_hostpack   a host thread team packs (a share of) every chunk
    2bit      gm_db_upload_2bit             a .2bit file's bytes as read from disk, 0.25 B/nt

For trna, ire, score.1, pk1 and qu+tr over 1024 x 1 Mnt uniform acgt records (so the .2bit file is
exact: no N blocks), a step is one upload + gm_scan (candidates sorted in host memory), timed by the
host clock around a device synchronise.  The three legs run in one process, alternating step by
step after a warm-up; the resident rate (database already packed on the device) is given beside
them.  The candidate arrays of the three legs and the resident run must be byte-equal, else the
script fails.  ire and score.1 run with their score pre-screen on, as bench.py's configs do.

    python profiles/twobit_e2e.py --out DIR [--steps 10] [--warmup 2] [--mnt 1024]

writes DIR/twobit_e2e.json with the card's name, power limit and SM clock, queried in the same run.
"""
import argparse
import gzip
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from rnamotif_b200 import gpumotif, twobit  # noqa: E402

PLAN_DIR = os.path.join(ROOT, "rnamotif_b200", "plans")
WORKLOADS = ["trna", "ire", "score.1", "pk1", "qu+tr"]


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
        raise SystemExit("twobit_e2e.py: no CUDA device; libgpumotif has no CPU path")
    os.makedirs(args.out, exist_ok=True)

    # the database: uniform acgt made on the device (seeded), characters to pinned host memory,
    # and the same records as a .2bit file read into pinned memory
    n_rec = args.mnt
    n_rec_nt = [1_000_000] * n_rec
    rec_off = np.concatenate([[0], np.cumsum(n_rec_nt)]).astype(np.int64)
    total = int(rec_off[-1])
    lut = torch.tensor(list(b"acgt"), dtype=torch.uint8, device="cuda")
    g = torch.Generator(device="cuda")
    g.manual_seed(1001)
    d_chars = lut[torch.randint(0, 4, (total,), generator=g, device="cuda")]
    h_chars = torch.empty(total, dtype=torch.uint8, pin_memory=True)
    h_chars.copy_(d_chars)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    f = twobit.write_2bit(["syn%06d" % r for r in range(n_rec)], h_chars.numpy(), rec_off)
    h_2bit = torch.empty(len(f), dtype=torch.uint8, pin_memory=True)
    tb = twobit.read_2bit(f, out=h_2bit.numpy())
    del f
    t_file = time.perf_counter() - t0
    rec2, dna_off, nblk = tb.tables()
    assert (rec2 == rec_off).all() and len(nblk) == 0

    res = {"card_before": card(), "database": f"{n_rec} x {n_rec_nt[0]} nt uniform acgt (seed 1001), "
                                              f"{total} nt, .2bit file {tb.data.size} bytes",
           "steps": args.steps, "warmup": args.warmup, "timing": "host clock around upload + gm_scan (which ends in a "
           "device synchronise and leaves the sorted candidates in host memory), legs alternating step by step",
           "pack_threads": os.environ.get("GPUMOTIF_PACK_THREADS", "default (CPUs of the process, at most 16)"),
           "cpus": len(os.sched_getaffinity(0)), "file_build_s": t_file, "workloads": []}
    ok_all = True
    for name in args.workloads.split(","):
        plan, score = load(name, "plan"), load(name, "score")
        strands = 2 if int(np.frombuffer(plan, dtype=np.int32, count=9)[8]) else 1
        ms = gpumotif.MotifSearch(plan)
        if score is not None:
            ms.set_score(score)
        legs = {
            "chars": lambda: ms.upload_ptr(h_chars.data_ptr(), rec_off),
            "hostpack": lambda: ms.upload_ptr(h_chars.data_ptr(), rec_off, host_pack=True),
            "2bit": lambda: ms.upload_2bit_ptr(h_2bit.data_ptr(), tb.data.size, dna_off, rec_off, nblk),
        }
        times = {k: [] for k in legs}
        h2d = {}
        hits = {}

        def step(leg):
            torch.cuda.synchronize()
            t = time.perf_counter()
            legs[leg]()
            ms.scan(0, total, strands, copy=False)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t
            h2d[leg] = int(ms.stats().h2d_bytes)
            return dt

        for i in range(args.warmup + args.steps):
            for leg in legs:
                dt = step(leg)
                if i >= args.warmup:
                    times[leg].append(dt)
        for leg in legs:
            step(leg)
            hits[leg] = ms.hits(copy=True)
        # resident: the characters already on the device, packed there once
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
                          "h2d_bytes_per_step": h2d[leg]}
        entry["card_after"] = card()
        res["workloads"].append(entry)
        print(json.dumps({k: entry[k] for k in ("workload", "candidates", "candidates_byte_equal")} |
                         {k: round(entry[k]["G_strand_nt_s"], 1) for k in ("resident", "chars", "hostpack", "2bit")}),
              flush=True)
    res["ok"] = ok_all
    with open(os.path.join(args.out, "twobit_e2e.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    if not ok_all:
        raise SystemExit("twobit_e2e.py: the candidate arrays differ between the legs")


if __name__ == "__main__":
    main()
