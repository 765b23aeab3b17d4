#!/usr/bin/env python3
"""bench.py -- throughput of the descriptor search, in strand-nucleotides
scanned per second (BASELINE.json: "Gnt/s scanned (both strands) per
descriptor at 1/2/4/8 B200; hits bit-exact").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl gpumotif|reference]
                    [--descr trna] [--mnt 1024] [--configs all|none|a,b,..] [--dump-outputs DIR]

A step is one pass of the hot path over one batch: every start offset on the
searched strands of a synthetic database (i.i.d. uniform acgt, SURVEY.md 8d).
One process per GPU; ranks own disjoint databases (weak scaling); no collective
on the data path.

The headline (`value`, `e2e`, `roofline`, ...) is BASELINE.json's target config:
test/trna.descr over 1 024 x 1 Mnt per GPU.  `per_config` carries the other
configs of BASELINE.json at their named sizes -- ire and score.1 (1 Gnt),
trna.general (syn_ecoli: 465 x 11.8 knt + one 5.49 Mnt record), pk1 and pk_j1+2
(1 Gnt per GPU), qu+tr (2 Gnt per GPU) -- each with

  value   kernels + candidate ordering + gather, packed database RESIDENT in HBM
  e2e     the same call made with HOST buffers (pinned characters): H2D copy,
          device pack, search, candidates back on the host -- every step
  parity  checked OUTSIDE the timed regions: the candidate stream of a prefix
          against the oracle (oracle/, CPU), and the full-size candidate arrays of
          the resident run, the end-to-end run (chunk-streamed upload, deferred
          enumeration) and a run through a second context with small segments and
          another tile size -- byte for byte.  A mismatch fails the bench.

Timed with CUDA events on the library's stream, max over ranks.

--impl reference times the reference's own CPU implementation (the binary built
from its sources, oracle/_ref/rnamotif, else the oracle port) on the host cores.
"""
import argparse
import gzip
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "strand-nt scanned per second (both strands)"
UNIT = "G strand-nt/s"
REF_DIR = os.path.join(ROOT, "oracle", "_ref")
PLAN_DIR = os.path.join(ROOT, "rnamotif_b200", "plans")

# BASELINE.json configs 2-5 (config 1's descriptor at the target's size is the headline).
# name -> (plan, record lengths per GPU, seed, prefix records checked against the oracle)
ECOLI = [11_800] * 465 + [5_490_000]
CONFIGS = {
    "ire": ("ire", [1_000_000] * 1000, 1001, 16),
    "score.1": ("score.1", [1_000_000] * 1000, 1001, 16),
    "trna.general": ("trna.general", ECOLI, 1003, len(ECOLI)),
    "pk1": ("pk1", [1_000_000] * 1000, 1004, 8),
    "pk_j1+2": ("pk_j1+2", [1_000_000] * 1000, 1004, 16),
    "qu+tr": ("qu+tr", [1_000_000] * 2000, 1005, 16),
}
# descriptor file of each plan below the reference's tree (for the CPU arm)
DESCR_FILE = {"trna.general": os.path.join("descr", "trna.general.descr")}  # (oracle/Makefile copies it from Ecoli.trna.example/)


def load_plan(name):
    """Flattened plans of the benchmark descriptors, produced by the reference's own
    front end (tools/make_bench_plans.sh -> rnamotif_b200/host rm_plan_dump)."""
    path = os.path.join(PLAN_DIR, name + ".plan.gz")
    if not os.path.exists(path):  # ad-hoc profiling runs (--descr descr.quad ...): the test corpus' plans
        path = os.path.join(ROOT, "tests", "golden", "plans", name + ".plan.gz")
    with gzip.open(path, "rb") as fh:
        return fh.read()


def load_score(name):
    """The descriptor's MAIN score program for the device's pre-screen (gm_ctx_set_score), or None."""
    path = os.path.join(PLAN_DIR, name + ".score.gz")
    if not os.path.exists(path):
        return None
    with gzip.open(path, "rb") as fh:
        sc = fh.read()
    return sc if int(np.frombuffer(sc, dtype=np.int32, count=1)[0]) else None


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured"
    return {"hbm_gbs": 6650.0}, "fallback"


def plan_strands(plan):
    return 2 if int(np.frombuffer(plan, dtype=np.int32, count=9)[8]) else 1


# ------------------------------------------------------------------ CPU arm

def _write_sample(path, n_records, rec_nt, seed):
    from rnamotif_b200 import synth
    ids, seq, off = synth.random_records(seed, [rec_nt] * n_records)
    synth.write_fastn(path, ids, seq, off)
    return int(off[-1])


def cpu_reference_run(descr, procs, rec_per_proc, rec_nt, seed=1001):
    """Time the reference CPU implementation over `procs` files of
    rec_per_proc x rec_nt nucleotides, one process per file (what mrnamotif
    does over MPI, src/mrnamotif.c:884-921).  Returns (strand_nt, seconds, kind)."""
    ref_bin = os.path.join(REF_DIR, "rnamotif")
    descr_file = os.path.join(REF_DIR, "data", DESCR_FILE.get(descr, os.path.join("test", descr + ".descr")))
    plan = load_plan(descr)
    strands = plan_strands(plan)
    with tempfile.TemporaryDirectory() as tmp:
        files, total = [], 0
        for p in range(procs):
            f = os.path.join(tmp, "part%03d.fastn" % p)
            total += _write_sample(f, rec_per_proc, rec_nt, seed + p)
            files.append(f)
        if os.path.exists(ref_bin) and os.path.exists(descr_file):
            env = dict(os.environ, EFNDATA=os.path.join(REF_DIR, "data", "efndata"))
            t0 = time.perf_counter()
            ps = [subprocess.Popen([ref_bin, "-descr", os.path.basename(descr_file), f],
                                   cwd=os.path.dirname(descr_file), env=env,
                                   stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL) for f in files]
            rcs = [p.wait() for p in ps]
            dt = time.perf_counter() - t0
            if any(rcs):
                raise RuntimeError("reference rnamotif failed: %r" % rcs)
            return total * strands, dt, "reference"
        # the reference binary did not travel: time the plain-C port instead
        from rnamotif_b200 import fastn
        from oracle import oracle_port
        dbs = [fastn.read_fastn(f) for f in files]

        def work(db):
            oracle_port.scan_db(plan, db[2], db[3], strands == 2)

        t0 = time.perf_counter()
        th = [threading.Thread(target=work, args=(db,)) for db in dbs]  # ctypes releases the GIL
        [t.start() for t in th]
        [t.join() for t in th]
        dt = time.perf_counter() - t0
        return total * strands, dt, "port"


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    procs = max(1, cores)
    # ~1.3 M strand-nt/s/core for trna: 4 x 1 Mnt per process ~ 6 s per step
    rec_per_proc, rec_nt = 4, 1_000_000
    times, work, kind = [], 0, "reference"
    for i in range(args.warmup + args.steps):
        w, dt, kind = cpu_reference_run(args.descr, procs, rec_per_proc, rec_nt, seed=1001 + 97 * i)
        if i >= args.warmup:
            times.append(dt)
            work += w
    total_t = sum(times)
    val = work / total_t / 1e9
    sample = f"{procs} processes x {rec_per_proc} x {rec_nt} nt synthetic acgt per step, default flags (-O2.5 prefilter on)"
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total_t / max(args.steps, 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": f"test/{args.descr}.descr over synthetic uniform acgt, 1 Mnt records, both strands",
                   "sample": sample},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": procs, "kind": kind, "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------ GPU arm

class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag = index, False
        self.sm, self.reasons, self.sm_max = [], set(), None

    def run(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.sm_max = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            names = {
                pynvml.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                pynvml.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                pynvml.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                pynvml.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
            }
            while not self.stop_flag:
                self.sm.append(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                r = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
                time.sleep(0.1)
        except Exception as e:  # clocks are evidence, not a dependency
            self.reasons.add("unavailable:" + type(e).__name__)

    def summary(self):
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.sm_max,
                "reasons": sorted(self.reasons)}


class Bench:
    """Buffers shared by all workloads of a run (device characters, pinned host
    characters), timing helpers, and the measurement of one (plan, database)."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist, self.args = torch, dist, args
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; libgpumotif has no CPU path")
        try:
            self.ncpu = len(os.sched_getaffinity(0))
        except AttributeError:
            self.ncpu = os.cpu_count() or 1
        self.numa_node = numa_bind(self.local)
        torch.cuda.set_device(self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
        self.cap = 0
        self.d_chars = self.h_chars = None
        # host threads of the packed upload: this rank's share of the CPUs (gpumotif reads the variable)
        ncpu = self.ncpu
        self.pack_threads = int(os.environ.get("GPUMOTIF_PACK_THREADS", max(1, min(16, ncpu // max(1, int(os.environ.get("LOCAL_WORLD_SIZE", self.world)))))))
        os.environ["GPUMOTIF_PACK_THREADS"] = str(self.pack_threads)
        self.lut = torch.tensor(list(b"acgt"), dtype=torch.uint8, device="cuda")

    def database(self, lengths, seed):
        """Synthetic database of this rank: uniform acgt characters generated on the
        device (seeded per rank), copied once to pinned host memory for the e2e leg."""
        torch = self.torch
        rec_off = np.concatenate([[0], np.cumsum(np.asarray(lengths, dtype=np.int64))]).astype(np.int64)
        total = int(rec_off[-1])
        if total > self.cap:
            self.d_chars = self.h_chars = None
            self.cap = total
            self.d_chars = torch.empty(total, dtype=torch.uint8, device="cuda")
            self.h_chars = torch.empty(total, dtype=torch.uint8, pin_memory=True)
        g = torch.Generator(device="cuda")
        g.manual_seed(seed + self.rank)
        for o in range(0, total, 1 << 27):
            n = min(1 << 27, total - o)
            self.d_chars[o:o + n] = self.lut[torch.randint(0, 4, (n,), generator=g, device="cuda")]
        self.h_chars[:total].copy_(self.d_chars[:total])
        torch.cuda.synchronize()
        return rec_off, total

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def timed(self, stream, fn, steps):
        torch = self.torch
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            fn()
        e1.record(stream)
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        self.barrier()
        return float(t.item())

    def all_ok(self, ok):
        """AND of a per-rank verdict over the ranks."""
        if self.world == 1:
            return bool(ok)
        t = self.torch.tensor([1 if ok else 0], dtype=self.torch.int32, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MIN)
        return bool(t.item())

    # --------------------------------------------------------------------------------
    def measure(self, plan, rec_off, total, steps, warmup, clocks=False, prefix_recs=0, tile=0, score=None):
        """Resident and end-to-end throughput of one plan over the database in the
        shared buffers; parity checks outside the timed regions.  Returns a dict."""
        from rnamotif_b200 import gpumotif
        torch, world = self.torch, self.world
        strands = plan_strands(plan)
        ms = gpumotif.MotifSearch(plan, device=self.local)
        if tile:
            ms.set_tile(tile)
        if score is not None:
            ms.set_score(score)  # candidates the score section rejects outright are dropped at the sink
        stream = torch.cuda.ExternalStream(ms.stream, device=torch.device("cuda", self.local))
        res = {"strands": strands, "n_descr": ms.n_descr}

        # ---- resident leg -----------------------------------------------------
        ms.set_device_chars(self.d_chars.data_ptr(), rec_off)
        acc = {"kernel_ms": [], "filter_ms": [], "launches": 0, "filter_launches": 0, "survivors": 0, "hits": 0,
               "score_rejected": 0}

        def step_resident():
            ms.scan(0, total, strands, copy=False)
            st = ms.stats()
            acc["kernel_ms"].append(st.kernel_ms)
            acc["filter_ms"].append(st.filter_ms)
            acc["launches"] += st.n_launches
            acc["filter_launches"] += st.n_filter_launches
            acc["survivors"] = st.n_survivors
            acc["hits"] = st.n_hits
            acc["score_rejected"] = st.n_score_rejected

        for _ in range(warmup):
            step_resident()
        acc["kernel_ms"].clear()
        acc["filter_ms"].clear()
        acc["launches"] = acc["filter_launches"] = 0
        sampler = None
        if clocks:
            sampler = ClockSampler(self.local)
            sampler.start()
        t_res = self.timed(stream, step_resident, steps)
        if sampler is not None:
            sampler.stop_flag = True
            sampler.join(timeout=2)
            res["clocks"] = sampler.summary()
        hits_res = ms.hits(copy=True)

        # ---- end-to-end leg: host characters in, candidates out, every step --------
        # Two ways over PCIe, both timed, the faster one reported (`e2e.upload`), the other kept
        # in `e2e.other_uploads`: the characters as they are (1 B per nucleotide, packed on the device), or
        # gm_db_upload_chars_hostpack: a host thread team packs a share of every chunk inside the timed
        # region (0.5 B per nucleotide) while the rest crosses as characters.
        def e2e_leg(host_pack):
            info = {}

            def step_e2e():
                ms.upload_ptr(self.h_chars.data_ptr(), rec_off, host_pack=host_pack)
                ms.scan(0, total, strands, copy=False)  # candidates are in host memory (library buffer)
                st = ms.stats()
                info.update(h2d=st.h2d_bytes, d2h=st.d2h_bytes,
                            phases=dict(h2d_ms=st.h2d_ms, pack_ms=st.pack_ms, kernel_ms=st.kernel_ms,
                                        d2h_ms=st.d2h_ms, sort_ms=st.sort_ms))

            for _ in range(max(1, min(warmup, 2))):
                step_e2e()
            t = self.timed(stream, step_e2e, steps)
            return t, info, ms.hits(copy=True)

        legs = {}
        for mode in self.args.upload.split(","):
            legs[mode] = e2e_leg(mode == "hostpack")
        best = min(legs, key=lambda m: legs[m][0])
        t_e2e, e2e_info, hits_e2e = legs[best]
        same_legs = all(len(v[2]) == len(hits_e2e) and v[2].tobytes() == hits_e2e.tobytes() for v in legs.values())
        res["upload"] = {"chars": "characters (1 B/nt), packed on the device",
                         "hostpack": "a share of every chunk packed to 4-bit codes by %d host threads inside the timed "
                                     "region, the rest sent as characters beside it (gm_db_upload_chars_hostpack)"
                         % self.pack_threads}[best]
        res["other_uploads"] = {m: {"ms_per_step": v[0] / steps, "h2d_bytes_per_step": int(v[1]["h2d"])}
                                for m, v in legs.items() if m != best}

        work = float(total) * strands * world  # strand-nt per step, all ranks
        res.update(value=work * steps / (t_res / 1e3) / 1e9, ms_per_step=t_res / steps,
                   e2e_value=work * steps / (t_e2e / 1e3) / 1e9, e2e_ms_per_step=t_e2e / steps,
                   h2d=int(e2e_info["h2d"]), d2h=int(e2e_info["d2h"]), phases=e2e_info["phases"],
                   t_res=t_res, acc=acc, total=total, candidates=int(acc["hits"]))

        # ---- parity, outside the timed regions -----------------------------------------
        par = {"full_candidates": int(len(hits_res))}
        same = same_legs and len(hits_res) == len(hits_e2e) and hits_res.tobytes() == hits_e2e.tobytes()
        # a second context: small worklist segments (several filter/enumeration launch
        # pairs, no deferred enumeration) and another tile size
        os.environ["GPUMOTIF_SEG_NT"] = str(48 << 20)
        try:
            ms2 = gpumotif.MotifSearch(plan, device=self.local)
        finally:
            del os.environ["GPUMOTIF_SEG_NT"]
        ms2.set_tile(416)
        if score is not None:
            ms2.set_score(score)
        ms2.set_device_chars(self.d_chars.data_ptr(), rec_off)
        hits_alt = ms2.scan(0, total, strands, copy=True)
        same = same and len(hits_alt) == len(hits_res) and hits_alt.tobytes() == hits_res.tobytes()
        par["full_equal_across_paths"] = self.all_ok(same)
        if prefix_recs > 0 and self.rank == 0:
            n_pre = min(prefix_recs, len(rec_off) - 1)
            pre_nt = int(rec_off[n_pre])
            ms2.set_score(None)  # the oracle enumerates every candidate
            hits_pre = ms2.scan(0, pre_nt, strands, copy=True)
            ok, n_ref, W = oracle_check(plan, self.h_chars[:pre_nt].numpy(), rec_off[:n_pre + 1], strands, hits_pre)
            par.update(prefix_nt=pre_nt, prefix_candidates=int(n_ref), prefix_equal_oracle=bool(ok))
            res["pair_evals_per_strand_nt"] = W
        ms2.close()
        if self.world > 1:
            self.dist.barrier()
        res["parity"] = par
        res["hits"] = hits_res
        ms.close()
        return res


def oracle_check(plan, chars, rec_off, strands, gpu_hits):
    """The oracle (oracle/, plain C, CPU) over the same records, on all host cores
    (records dealt out to threads; ctypes releases the GIL).  Returns (equal,
    candidates of the oracle, pair-rule evaluations per start)."""
    from oracle import oracle_port
    n_rec = len(rec_off) - 1
    order = sorted(range(n_rec), key=lambda r: -(rec_off[r + 1] - rec_off[r]))
    n_thr = max(1, min(os.cpu_count() or 1, n_rec))
    groups = [[] for _ in range(n_thr)]
    load = [0] * n_thr
    for r in order:  # longest first onto the least loaded thread
        k = load.index(min(load))
        groups[k].append(r)
        load[k] += int(rec_off[r + 1] - rec_off[r])
    out = {}
    evals = [0, 0]
    lock = threading.Lock()

    def work(recs):
        for r in recs:
            seq = np.ascontiguousarray(chars[rec_off[r]:rec_off[r + 1]])
            h, st = oracle_port.scan_db(plan, seq, np.array([0, len(seq)], dtype=np.int64), strands == 2,
                                        cap_hits=1 << 14)
            h = h.copy()
            h["rec"] = r
            with lock:
                out[r] = h
                evals[0] += st.n_pair_evals
                evals[1] += st.n_starts

    th = [threading.Thread(target=work, args=(g,)) for g in groups if g]
    [t.start() for t in th]
    [t.join() for t in th]
    parts = [out[r] for r in range(n_rec) if len(out[r])]
    ref = np.concatenate(parts) if parts else gpu_hits[:0]
    ok = len(ref) == len(gpu_hits)
    if ok and len(ref):
        for f in ("rec", "szero", "seq", "comp", "lctx_off", "lctx_len", "rctx_off", "rctx_len"):
            ok = ok and bool((ref[f] == gpu_hits[f]).all())
        for f in ("off", "len", "mpr", "mm"):
            ok = ok and bool((ref["el"][f] == gpu_hits["el"][f]).all())
    return ok, len(ref), evals[0] / max(evals[1], 1)


def dominant_kernel(res, steps, n_descr):
    """Which kernel dominates a measured step, its per-launch duration (CUDA events the
    library records around its launches) and its algorithmic bytes per launch."""
    acc, total, t_res = res["acc"], res["total"], res["t_res"]
    k_sum, f_sum = float(np.sum(acc["kernel_ms"])), float(np.sum(acc["filter_ms"]))
    fl, gl = acc["filter_launches"], acc["launches"]
    per_step_fl = max(fl / steps, 1)
    if fl > 0 and f_sum < 0.5 * k_sum:
        name = "gm_dfs_kernel<FULL> (enumeration of the filter's survivors)"
        ms = (k_sum - f_sum) / fl
        alg = acc["survivors"] / per_step_fl * (32 + 64) + acc["hits"] * (32 + 8 * n_descr) / per_step_fl
        share = (k_sum - f_sum) / t_res
    elif fl > 0:
        name = "gm_filter_kernel<PF> (level-0 sieve / prefilter of the worklist path)"
        ms = f_sum / fl
        alg = total * steps / fl * 0.5 + acc["survivors"] / per_step_fl * 32
        share = f_sum / t_res
    else:
        name = "gm_search_kernel<0,FULL,PF> (fused filter + enumeration)"
        ms = k_sum / steps / max(gl / steps, 1)
        alg = total * steps / max(gl, 1) * 0.5 + acc["hits"] * (32 + 8 * n_descr) / max(gl / steps, 1)
        share = k_sum / t_res
    return name, ms, alg, share, k_sum / steps, (f_sum / steps if fl > 0 else None)


def write_fasta(path, n_rec, rec_nt, seed, width=70):
    """n_rec x rec_nt uniform acgt, `width` per line, ids syn%06d (SURVEY.md 8d)."""
    rng = np.random.default_rng(seed)
    lut = np.frombuffer(b"acgt", dtype=np.uint8)
    full, rest = divmod(rec_nt, width)
    with open(path, "wb") as fh:
        for r in range(n_rec):
            fh.write(b">syn%06d synthetic record %d\n" % (r, r))
            a = np.empty((full, width + 1), dtype=np.uint8)
            a[:, :width] = lut[rng.integers(0, 4, size=(full, width), dtype=np.uint8)]
            a[:, width] = 10
            a.tofile(fh)
            if rest:
                fh.write(lut[rng.integers(0, 4, size=rest, dtype=np.uint8)].tobytes() + b"\n")
    return n_rec * rec_nt


DUMP_BYTES = 64_000_000
NPY_HEADER_RESERVE = 4096  # the .npy headers of one workload's 13 files (128 bytes each)


def dump_hits(out_dir, workload, hits, budget):
    """The candidates of the last timed resident step of one workload, one float64 array per
    field of the hit record (integers, all exact in float64), as out_dir/<workload>.<field>.npy.
    `rows` holds the indices of the written candidates: all of them when the files fit in
    `budget` bytes, else a fixed, seeded sample in enumeration order."""
    nd = hits.dtype["el"].shape[0]
    row_bytes = 8 * (1 + 8 + 4 * nd)
    n = len(hits)
    cap = max(0, (budget - NPY_HEADER_RESERVE) // row_bytes)
    rows = np.arange(n) if n <= cap else np.sort(np.random.default_rng(0).choice(n, size=cap, replace=False))
    h = hits[rows]
    cols = {"rows": rows}
    for f in ("rec", "szero", "seq", "comp", "lctx_off", "lctx_len", "rctx_off", "rctx_len"):
        cols[f] = h[f]
    for f in ("off", "len", "mpr", "mm"):
        cols["el_" + f] = h["el"][f].reshape(len(h), nd)
    os.makedirs(out_dir, exist_ok=True)
    for f, a in cols.items():
        np.save(os.path.join(out_dir, f"{workload}.{f}.npy"), np.asarray(a, dtype=np.float64))


def _pipeline_rate(summary):
    """G strand-nt/s of the driver's read / search / replay pipeline alone (its own timer, between CUDA
    start-up + context creation and tear-down), from the GPUMOTIF_STATS summary line."""
    import re
    m = re.search(r"pipeline [0-9.]+ s \(([0-9.]+) G strand-nt/s", summary or "")
    return float(m.group(1)) if m else None


def numa_bind(local_rank):
    """Run this rank on the CPUs of its GPU's NUMA node before any pinned buffer is allocated (pinned
    pages land on the node of the allocating thread; eight ranks reading one node's memory was round 1's
    end-to-end limiter at 8 GPUs).  Quietly does nothing where the platform does not tell (numa_node -1)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        idx = int(vis.split(",")[local_rank]) if vis and vis.split(",")[local_rank].strip().isdigit() else local_rank
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(idx)).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]  # nvml prints an eight-digit domain, sysfs four
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return node
    except Exception:
        pass
    return None


def binary_leg(descr, mnt, prefix_mnt):
    """The drop-in program itself: rnamotif_b200/host/_build/rnamotif_gpu (the
    reference's front end, score program and printer around libgpumotif) over a FASTA
    FILE, wall clock from exec to exit, stdout to a file -- beside the reference binary
    on a prefix of the same file, outputs compared byte for byte."""
    exe = os.path.join(ROOT, "rnamotif_b200", "host", "_build", "rnamotif_gpu")
    ref_bin = os.path.join(REF_DIR, "rnamotif")
    dfile = os.path.join(REF_DIR, "data", DESCR_FILE.get(descr, os.path.join("test", descr + ".descr")))
    if not (os.path.exists(exe) and os.path.exists(dfile)):
        return {"unavailable": "rnamotif_gpu or the descriptor file was not built into this tree"}
    strands = plan_strands(load_plan(descr))
    base = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else None
    env = dict(os.environ, EFNDATA=os.path.join(REF_DIR, "data", "efndata"), GPUMOTIF_STATS="1")
    out = {}
    with tempfile.TemporaryDirectory(dir=base) as tmp:
        big, pre = os.path.join(tmp, "syn.fastn"), os.path.join(tmp, "prefix.fastn")
        nt = write_fasta(big, mnt, 1_000_000, 1001)
        write_fasta(pre, prefix_mnt, 1_000_000, 1001)  # same generator and seed: the first records of `big`
        cwd = os.path.dirname(dfile)

        def run(cmd, path, dest):
            t0 = time.perf_counter()
            with open(dest, "wb") as fh:
                r = subprocess.run([cmd, "-descr", os.path.basename(dfile), path], cwd=cwd, env=env, stdout=fh,
                                   stderr=subprocess.PIPE)
            return time.perf_counter() - t0, r

        run(exe, pre, os.path.join(tmp, "warm.out"))  # page cache, CUDA driver warm-up
        dt, r = run(exe, big, os.path.join(tmp, "big.out"))
        if r.returncode != 0:
            return {"error": r.stderr.decode(errors="replace")[-400:]}
        summary = [ln for ln in r.stderr.decode(errors="replace").splitlines() if "wall" in ln]
        out.update(value=nt * strands / dt / 1e9, unit=UNIT, wall_s=dt, file_mnt=mnt,
                   file_bytes=os.path.getsize(big), stdout_bytes=os.path.getsize(os.path.join(tmp, "big.out")),
                   driver_summary=summary[-1] if summary else None,
                   pipeline_value=_pipeline_rate(summary[-1]) if summary else None,
                   what="wall clock of `rnamotif_gpu -descr %s.descr FILE` from exec to exit (CUDA start-up, file read, "
                        "search, score + print of every candidate, stdout to a file on tmpfs)" % descr)
        dtg, rg = run(exe, pre, os.path.join(tmp, "pre_gpu.out"))
        if os.path.exists(ref_bin):
            dtr, rr = run(ref_bin, pre, os.path.join(tmp, "pre_ref.out"))
            same = open(os.path.join(tmp, "pre_gpu.out"), "rb").read() == open(os.path.join(tmp, "pre_ref.out"), "rb").read()
            out["prefix"] = {"mnt": prefix_mnt, "stdout_equal_reference": bool(same and rg.returncode == 0 and rr.returncode == 0),
                             "stdout_bytes": os.path.getsize(os.path.join(tmp, "pre_ref.out")),
                             "reference_wall_s": dtr, "rnamotif_gpu_wall_s": dtg,
                             "reference_value": prefix_mnt * 1e6 * strands / dtr / 1e9}
        else:
            out["prefix"] = {"unavailable": "oracle/_ref/rnamotif did not travel"}
    return out


def run_gpu_arm(args):
    B = Bench(args)
    rank, world = B.rank, B.world
    pk, which = peaks()
    names = [] if args.configs == "none" else (list(CONFIGS) if args.configs == "all" else args.configs.split(","))
    dump_budget = DUMP_BYTES // (1 + len(names))

    # ---- headline: BASELINE.json's target config ----------------------------------
    plan = load_plan(args.descr)
    rec_off, total = B.database([1_000_000] * max(1, args.mnt), 1001)
    res = B.measure(plan, rec_off, total, args.steps, args.warmup, clocks=True,
                    prefix_recs=(16 if not args.no_parity else 0), tile=args.tile)
    if args.dump_outputs and rank == 0:
        dump_hits(args.dump_outputs, args.descr, res["hits"], dump_budget)
    name, dom_ms, alg, share, k_ms, f_ms = dominant_kernel(res, args.steps, res["n_descr"])
    line = None
    if rank == 0:
        achieved = alg / (dom_ms / 1e3) / 1e9
        traffic = None
        issue_ncu = None
        tj = os.path.join(ROOT, "profiles", "r2_sieve_kernel.json")
        if os.path.exists(tj):
            t = json.load(open(tj))
            if t.get("workload") == {"descr": args.descr, "mnt": args.mnt}:
                traffic = t["dram_bytes_read"] + t["dram_bytes_write"]  # bytes per launch, ncu
                issue_ncu = t.get("issue")
        sm_clk = (res["clocks"]["sm_mhz"] or 1965.0) * 1e6
        lane_peak = 148 * 128 * sm_clk
        W = res.get("pair_evals_per_strand_nt")
        line = {
            "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": f"test/{args.descr}.descr over syn_{args.mnt}M: {args.mnt} x 1 Mnt uniform acgt per GPU, "
                                   f"{res['strands']} strand(s)",
                       "l2": "input (packed) larger than L2" if total / 2 > 126e6
                       else "input smaller than L2; each step re-reads it after the hit gather",
                       "candidates_per_step_rank0": res["candidates"]},
            "e2e": {"value": res["e2e_value"], "unit": UNIT, "h2d_bytes_per_step": res["h2d"],
                    "d2h_bytes_per_step": res["d2h"], "ms_per_step": res["e2e_ms_per_step"],
                    "upload": res["upload"], "other_uploads": res["other_uploads"],
                    "phases_ms_last_step": res["phases"]},
            "gpu_launches": int(res["acc"]["launches"]),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": pk["hbm_gbs"], "unit": "GB/s",
                         "frac": achieved / pk["hbm_gbs"], "traffic": traffic, "algorithmic_bytes": alg,
                         "peak_source": which, "kernel": name, "kernel_ms": dom_ms, "kernel_share_of_step": share,
                         "all_kernels_ms_per_step": k_ms,
                         "note": "the search is integer-issue bound, not HBM bound (SURVEY.md F8); see issue and profiles/"},
            "parity": res["parity"],
            "clocks": res["clocks"],
            "host": {"cpus": B.ncpu, "numa_node_bound": B.numa_node, "pack_threads": B.pack_threads},
        }
        if W is not None:
            line["issue"] = {"pair_evals_per_strand_nt": W,
                             "pair_evals_per_s": W * total * res["strands"] / (k_ms / 1e3),
                             "int_lane_peak_per_s": lane_peak,
                             "frac_of_lane_peak": W * total * res["strands"] / (k_ms / 1e3) / lane_peak,
                             "ncu": issue_ncu,
                             "note": "the reference's pair-rule evaluations per strand-nt (oracle count on the parity prefix) x "
                                     "measured strand-nt/s = algorithm-level rate; `ncu` = issue-slot utilisation of the "
                                     "dominant kernel from the committed capture (profiles/r2_sieve_kernel.json)"}

    # ---- the other configs of BASELINE.json ------------------------------------------
    per_config = []
    for cname in names:
        pname, lengths, seed, pre = CONFIGS[cname]
        cplan = load_plan(pname)
        c_off, c_total = B.database(lengths, seed)
        r = B.measure(cplan, c_off, c_total, args.cfg_steps, args.cfg_warmup,
                      prefix_recs=(pre if not args.no_parity else 0), score=load_score(pname))
        if rank != 0:
            continue
        if args.dump_outputs:
            dump_hits(args.dump_outputs, cname, r["hits"], dump_budget)
        kname, kms, kalg, kshare, kk_ms, kf_ms = dominant_kernel(r, args.cfg_steps, r["n_descr"])
        entry = {
            "config": cname, "workload": f"{pname}.descr over {len(lengths)} records, {c_total / 1e6:.1f} Mnt per GPU "
                                         f"(seed {seed}), {r['strands']} strand(s)",
            "value": r["value"], "unit": UNIT, "ms_per_step": r["ms_per_step"],
            "e2e": {"value": r["e2e_value"], "ms_per_step": r["e2e_ms_per_step"], "h2d_bytes_per_step": r["h2d"],
                    "d2h_bytes_per_step": r["d2h"], "upload": r["upload"], "other_uploads": r["other_uploads"]},
            "steps": args.cfg_steps, "warmup": args.cfg_warmup,
            "candidates_per_step_rank0": r["candidates"], "survivors_of_level0_rank0": int(r["acc"]["survivors"]),
            "score_prescreen": ({"on": True, "rejected_on_device_per_step_rank0": int(r["acc"].get("score_rejected", 0))}
                                if load_score(pname) is not None else {"on": False}),
            "kernel": kname, "kernel_ms": kms, "kernel_share_of_step": kshare,
            "kernels_ms_per_step": kk_ms, "filter_ms_per_step": kf_ms,
            "hbm_frac": kalg / (kms / 1e3) / 1e9 / pk["hbm_gbs"],
            "parity": r["parity"],
        }
        W = r.get("pair_evals_per_strand_nt")
        if W is not None:
            lane_peak = 148 * 128 * 1965.0e6
            entry["useful_work"] = {"pair_evals_per_strand_nt": W,
                                    "frac_of_lane_peak": W * c_total * r["strands"] / (kk_ms / 1e3) / lane_peak}
        per_config.append(entry)

    if rank == 0:
        if per_config:
            line["per_config"] = per_config
        bad = [e["config"] for e in per_config if not all(v for k, v in e["parity"].items() if k.endswith("equal_oracle") or k.startswith("full_equal"))]
        hp = line["parity"]
        if not hp.get("full_equal_across_paths", True) or not hp.get("prefix_equal_oracle", True):
            bad.append(args.descr)
        if world == 1 and not args.no_cpu:
            w, dt, kind = cpu_reference_run(args.descr, 1, 16, 1_000_000)
            line["cpu_baseline"] = {"value": w / dt / 1e9, "unit": UNIT, "cores": 1, "kind": kind,
                                    "sample": "16 x 1 Mnt synthetic acgt, one process, default flags"}
        if world == 1 and not args.no_binary:
            line["binary"] = binary_leg(args.descr, args.binary_mnt, 8)
            if line["binary"].get("prefix", {}).get("stdout_equal_reference") is False:
                bad.append("rnamotif_gpu stdout")
        print(json.dumps(line), flush=True)
        if bad:
            print("bench.py: PARITY FAILED for " + ", ".join(bad), file=sys.stderr)
    if world > 1:
        B.dist.destroy_process_group()
    if rank == 0 and bad:
        sys.exit(3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="gpumotif", choices=["gpumotif", "reference"])
    ap.add_argument("--descr", default="trna")
    ap.add_argument("--mnt", type=int, default=1024, help="Mnt of synthetic sequence per GPU (headline)")
    ap.add_argument("--configs", default="all", help="per_config block: all, none, or a comma list of "
                    + ",".join(CONFIGS))
    ap.add_argument("--cfg-steps", type=int, default=None, help="timed steps of each per_config workload (default: --steps)")
    ap.add_argument("--cfg-warmup", type=int, default=3)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle prefix checks")
    ap.add_argument("--no-binary", action="store_true", help="skip the rnamotif_gpu program leg")
    ap.add_argument("--binary-mnt", type=int, default=1024, help="Mnt of the FASTA file the program leg reads")
    ap.add_argument("--upload", default="chars,hostpack", help="e2e leg: chars, hostpack, or both (the faster is reported)")
    ap.add_argument("--tile", type=int, default=0, help="starts per tile (0 = library default)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the candidates of each workload's last timed step (rank 0) as DIR/<workload>.<field>.npy "
                         "(float64, at most 64 MB in all; a seeded sample of the rows beyond that)")
    args = ap.parse_args()
    if args.cfg_steps is None:
        args.cfg_steps = args.steps
    if args.steps < 1 or args.cfg_steps < 1:
        ap.error("--steps and --cfg-steps must be at least 1")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
