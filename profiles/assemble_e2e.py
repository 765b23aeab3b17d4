#!/usr/bin/env python3
"""Spliced transcripts of an uploaded genome, built on the device (gm_db_assemble) or on the host.

The genome is 1 Gnt of uniform acgt (seeded, made on the device) in eight chromosome-sized records,
written as a .2bit file and read into pinned memory.  The transcripts are seeded BED12 lines from
synth.random_transcripts with its defaults, which follow a human annotation's exon, intron and UTR
sizes; `exons` of every line is assembled.  Two legs, alternating step by step after a warm-up:

    device  gm_db_upload_2bit (not timed), then gm_db_assemble to a device synchronise (host clock)
    host    Assembly.assemble_chars over the genome's characters, copied into pinned memory, then
            gm_db_upload_chars from there to a device synchronise (host clock, both parts)

The gather's kernel time is taken apart in a torch.profiler pass of its own over one more call (CUDA
activities: the gm_assemble_kernel launches and the block table's copy).  Then trna, ire, score.1,
pk1 and qu+tr scan the assembled batch: the first scan after the call (it streams the chunks in) and
`steps` rescans.  ire and score.1 run with their score pre-screen on, as bench.py's configs do.  The
candidate arrays after the device leg and after the host leg must be byte-equal, else the script
fails.

    python profiles/assemble_e2e.py --out DIR [--steps 5] [--warmup 1] [--transcripts 150000]

writes DIR/assemble_e2e.json with the card's name, power limit and SM clock, queried in the same run.
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

from rnamotif_b200 import bed, gpumotif, synth, twobit  # noqa: E402

PLAN_DIR = os.path.join(ROOT, "rnamotif_b200", "plans")
WORKLOADS = ["trna", "ire", "score.1", "pk1", "qu+tr"]
CHROM_MNT = [200, 180, 160, 140, 120, 100, 80, 44]  # 1 024 Mnt


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


def med(v):
    return 1e3 * float(np.median(v))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--transcripts", type=int, default=150000)
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("assemble_e2e.py: no CUDA device; libgpumotif has no CPU path")
    os.makedirs(args.out, exist_ok=True)

    sizes = [m * 1_000_000 for m in CHROM_MNT]
    names = ["chr%d" % (i + 1) for i in range(len(sizes))]
    rec_off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    total = int(rec_off[-1])
    lut = torch.tensor(list(b"acgt"), dtype=torch.uint8, device="cuda")
    g = torch.Generator(device="cuda")
    g.manual_seed(1003)
    h_chars = torch.empty(total, dtype=torch.uint8, pin_memory=True)
    h_chars.copy_(lut[torch.randint(0, 4, (total,), generator=g, device="cuda")])
    torch.cuda.synchronize()
    chars = h_chars.numpy()
    f = twobit.write_2bit(names, chars, rec_off)
    h_2bit = torch.empty(len(f), dtype=torch.uint8, pin_memory=True)
    tb = twobit.read_2bit(f, out=h_2bit.numpy())
    del f
    _, dna_off, nblk = tb.tables()

    t0 = time.perf_counter()
    text = synth.random_transcripts(2026, names, sizes, args.transcripts)
    t_bed = time.perf_counter() - t0
    t0 = time.perf_counter()
    asm = bed.read_bed(text, names, rec_off)
    t_read = time.perf_counter() - t0
    ro = asm.rec_off_new()
    n_asm = int(ro[-1])
    lens = asm.blk[1::2] - asm.blk[0::2]
    print(f"{len(asm)} transcripts, {len(lens)} exons (median {int(np.median(lens))} nt), assembled {n_asm} nt", flush=True)
    h_asm = torch.empty(n_asm, dtype=torch.uint8, pin_memory=True)

    res = {"card_before": card(),
           "genome": f"{len(sizes)} records of {CHROM_MNT} Mnt uniform acgt (seed 1003), {total} nt, .2bit file "
                     f"{tb.data.size} bytes in pinned memory",
           "transcripts": len(asm), "exons": int(len(lens)), "exon_nt_median": int(np.median(lens)),
           "transcript_nt_median": int(np.median(np.diff(ro))), "assembled_nt": n_asm,
           "minus_share": float(asm.strand.mean()), "bed_write_s": t_bed, "bed_read_s": t_read,
           "steps": args.steps, "warmup": args.warmup,
           "timing": "host clock to a device synchronise; device and host legs alternate step by step"}

    ms = gpumotif.MotifSearch(load("trna", "plan"))
    times = {"device_call": [], "host_assemble_chars": [], "host_upload": []}
    for i in range(args.warmup + args.steps):
        ms.upload_2bit_ptr(h_2bit.data_ptr(), tb.data.size, dna_off, rec_off, nblk)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ms.assemble_bed(asm)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        a_chars, a_ro = asm.assemble_chars(chars, rec_off)
        h_asm.numpy()[:] = a_chars
        t2 = time.perf_counter()
        ms.upload_ptr(h_asm.data_ptr(), a_ro)
        torch.cuda.synchronize()
        t3 = time.perf_counter()
        if i >= args.warmup:
            times["device_call"].append(t1 - t0)
            times["host_assemble_chars"].append(t2 - t1)
            times["host_upload"].append(t3 - t2)
    host_total = [a + b for a, b in zip(times["host_assemble_chars"], times["host_upload"])]
    res["device_call_ms"] = med(times["device_call"])
    res["device_call_ms_min_max"] = [1e3 * min(times["device_call"]), 1e3 * max(times["device_call"])]
    res["host_assemble_chars_ms"] = med(times["host_assemble_chars"])
    res["host_upload_chars_ms"] = med(times["host_upload"])
    res["host_total_ms"] = med(host_total)

    # the gather's kernels and the table copy, apart, in a profiler pass of their own
    from torch.profiler import ProfilerActivity, profile
    ms.upload_2bit_ptr(h_2bit.data_ptr(), tb.data.size, dna_off, rec_off, nblk)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ms.assemble_bed(asm)
        torch.cuda.synchronize()
    kern, copy, n_kern = 0.0, 0.0, 0
    for e in prof.events():
        t = e.device_time_total
        if "gm_assemble_kernel" in e.name:
            kern += t
            n_kern += 1
        elif "Memcpy HtoD" in e.name:
            copy += t
    st = ms.stats()
    res["gather_kernel_ms"] = kern / 1e3
    res["gather_kernel_launches"] = n_kern
    res["table_copy_ms"] = copy / 1e3
    res["h2d_bytes"] = int(st.h2d_bytes)
    ms.close()
    print(json.dumps({k: res[k] for k in ("device_call_ms", "gather_kernel_ms", "table_copy_ms", "host_assemble_chars_ms",
                                          "host_upload_chars_ms")}), flush=True)

    ok_all = True
    res["workloads"] = []
    for name in args.workloads.split(","):
        plan, score = load(name, "plan"), load(name, "score")
        strands = 2 if int(np.frombuffer(plan, dtype=np.int32, count=9)[8]) else 1
        ms = gpumotif.MotifSearch(plan)
        if score is not None:
            ms.set_score(score)
        ms.upload_2bit_ptr(h_2bit.data_ptr(), tb.data.size, dna_off, rec_off, nblk)
        ms.assemble_bed(asm)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ms.scan(0, n_asm, strands, copy=False)
        t_first = time.perf_counter() - t0
        t_res = []
        for _ in range(args.steps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ms.scan(0, n_asm, strands, copy=False)
            torch.cuda.synchronize()
            t_res.append(time.perf_counter() - t0)
        dev = ms.hits(copy=True)
        ms.upload_ptr(h_asm.data_ptr(), a_ro)
        host = ms.scan(0, n_asm, strands)
        ms.close()
        same = dev.tobytes() == host.tobytes()
        ok_all = ok_all and same
        work = float(n_asm) * strands
        entry = {"workload": name, "strands": strands, "score_prescreen": score is not None, "candidates": int(len(dev)),
                 "candidates_byte_equal": same, "first_scan_ms": 1e3 * t_first, "scan_ms": med(t_res),
                 "G_strand_nt_s": work / float(np.median(t_res)) / 1e9, "card_after": card()}
        res["workloads"].append(entry)
        print(json.dumps({k: entry[k] for k in ("workload", "candidates", "candidates_byte_equal", "scan_ms")} |
                         {"G_strand_nt_s": round(entry["G_strand_nt_s"], 1)}), flush=True)
    res["ok"] = ok_all
    with open(os.path.join(args.out, "assemble_e2e.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    if not ok_all:
        raise SystemExit("assemble_e2e.py: the candidate arrays differ between the device and host legs")


if __name__ == "__main__":
    main()
