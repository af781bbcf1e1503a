#!/usr/bin/env python
"""bench.py — throughput of the nohuman hot path (kraken2-style classification
+ keep/drop) on B200.

    python bench.py --gpus N --steps K --warmup W            # this repo (CUDA)
    python bench.py --impl reference --gpus N ...            # CPU arm (no CUDA library loaded)
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's calls as DIR/*.npy

Workload = BASELINE.json configs[1]: 10 M synthetic 2x150 bp read pairs, 50 %
sampled from the genome the table was built from ("human-derived"), --conf 0.5,
against a synthetic kraken2-format table sized like HPRC.r2 (configs[3]:
2^31 cells = 8 GiB, load 0.7).  One step = those 10 M pairs per GPU = ten
launches of 1 M pairs over ten different batches.  `value` is measured with
the batches resident in HBM; `e2e` goes through nh_classify_batch with pinned
HOST buffers (H2D + D2H inside the timed region).

Outside the headline timing the line also carries
  parity_vs_oracle   every rank classifies one common batch on ITS replica of the
                     table; mismatches against the CPU oracle are summed over ranks
  workloads          configs[2] (ONT-like long reads, keep-human) and configs[4]
                     (read-length sweep 100 bp - 50 kb), each with Gbp/s, lookups/s,
                     fraction of the measured table-request ceiling and an oracle
                     parity sample of >= 20 Mbp, at whatever N the run has
  roofline_probe     the probe's own access pattern measured alone on the same table

The reference arm times the CPU implementation of the same path — the oracle's
restatement of kraken2's classifier (kraken2 itself is not installable offline)
— on the host cores.  It builds the same table and samples the same reads with
the CPU twin of the generator (oracle/k2_synth.c) and never imports torch or
loads libnohuman_gpu.so.  oracle/ is touched ONLY in cpu_baseline(), the parity
checks and the reference arm.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

READ_LEN = 150
CONF = 0.5
METRIC = "classified+filtered throughput (Gbp/s)"
UNIT = "Gbp/s"
GENOME_SEED = 0x5EED
COMMON_SEED = 424242  # the batch every rank classifies for the parity check


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--capacity-log2", type=int, default=31, help="hash table cells = 2^this")
    ap.add_argument("--pairs-per-launch", type=int, default=1_000_000, help="read pairs per kernel launch")
    ap.add_argument("--launches-per-step", type=int, default=10, help="launches (different batches) per step and GPU")
    ap.add_argument("--ref-pairs-per-step", type=int, default=0,
                    help="reference arm: pairs per step (0 = sized for ~1 s per step)")
    ap.add_argument("--workload-mbases", type=int, default=150, help="bases per GPU of each `workloads` entry")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-packed", default="auto", help="packed e2e shapes 'workers x pack threads' (0 = cores / workers), "
                    "comma separated; the best one is reported, all are listed")
    ap.add_argument("--no-workloads", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the calls and keep mask of the last timed step to DIR/*.npy "
                         "(a fixed sample if they exceed 64 MB), so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the CUDA path only")
    return args


def workload_config(args):
    """What is measured; identical in both arms."""
    capacity = 1 << args.capacity_log2
    return {
        "workload": "BASELINE configs[1]: 10M 2x150 bp paired-end reads per step, 50% genome-derived, --conf 0.5, "
                    "against configs[3]'s synthetic HPRC.r2-sized kraken2 table",
        "pairs_per_step_per_gpu": args.pairs_per_launch * args.launches_per_step,
        "pairs_per_launch": args.pairs_per_launch, "launches_per_step": args.launches_per_step,
        "read_len": READ_LEN, "confidence": CONF, "table_cells": capacity,
        "table_gib": round(capacity * 4 / 2 ** 30, 2), "table_target_load": 0.7, "k": 35, "l": 31,
        "read_sampler": "50% from the table's synthetic genome (first 2*table_cells bases), 0.5% substitutions, "
                        "1% of reads with an N, insert 350+-50; same bytes on GPU and CPU generators",
        "l2_policy": "inputs larger than L2: ten different 300 MB batches per step + random probes over the 8 GiB table",
    }


def read_span(capacity):
    """Reads are sampled from this prefix of the synthetic genome: known to both arms without building
    the table (a table at load 0.7 always covers more than 2 bases per cell)."""
    return 2 * capacity


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed regions.  The
    sampler runs from before warm-up to the end of the bench; `mark()` brackets
    the timed regions and only samples whose timestamp falls inside one count."""

    FIELDS = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []
        self.windows = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}",
                 "--format=csv,noheader,nounits", "-lms", "25"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def mark(self):
        import datetime
        self.windows.append([datetime.datetime.now(), None])
        return len(self.windows) - 1

    def close(self, tok):
        import datetime
        self.windows[tok][1] = datetime.datetime.now()

    def stop(self):
        import datetime
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi not sampled on this rank"]}
        time.sleep(0.1)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        rows = []
        for ln in self.lines:
            parts = [x.strip() for x in ln.split(",")]
            if len(parts) < 8:
                continue
            try:
                ts = datetime.datetime.strptime(parts[0], "%Y/%m/%d %H:%M:%S.%f")
                rows.append((ts, float(parts[1]), float(parts[2]), float(parts[3]), parts[4:8]))
            except ValueError:
                continue
        inside = [r for r in rows if any(w0 <= r[0] <= (w1 or r[0]) for w0, w1 in self.windows)]
        reasons = set()
        for r in inside:
            for nm, v in zip(self.NAMES, r[4]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm = [r[1] for r in inside]
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": inside[0][2] if inside else (rows[0][2] if rows else None),
                "power_w_max": max((r[3] for r in inside), default=None),
                "reasons": sorted(reasons), "samples": len(sm), "samples_total": len(rows),
                "window": "timed regions (device-resident steps and e2e steps)"}


class DevPtr:
    """Zero-copy torch view of a raw device pointer (for NCCL broadcast of the table)."""

    def __init__(self, ptr: int, nbytes: int):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False),
                                         "version": 3, "strides": None}


# ---------------------------------------------------------------------------------------------
# workload shapes (shared by the GPU generator and its CPU twin)

def pair_offsets(n_pairs):
    return (np.arange(2 * n_pairs + 1, dtype=np.int64) * READ_LEN)


READS_PE = dict(human_frac=0.5, sub_rate=0.005, ins_rate=0.0, del_rate=0.0, n_rate=0.01, paired=True,
                insert_mean=350.0, insert_sd=50.0)


def ont_lengths(rng, total_bases, n50=10_000, lo=200, hi=100_000):
    """log-normal read lengths whose length-weighted median (N50) is ~10 kb, clipped to [200, 100k]"""
    sigma = 0.9
    mu = np.log(n50) - sigma * sigma
    out = []
    acc = 0
    while acc < total_bases:
        L = np.clip(np.exp(rng.normal(mu, sigma, size=4096)).astype(np.int64), lo, hi)
        out.append(L)
        acc += int(L.sum())
    L = np.concatenate(out)
    n = int(np.searchsorted(np.cumsum(L), total_bases)) + 1
    L = L[:n]
    L[0] = hi  # the longest read the config allows is always present
    return L


def workload_list(args):
    """BASELINE configs[2] and configs[4].  (name, lengths or read length, sampler arguments, conf, keep_human, paired)"""
    e = 0.05 / 3
    ont = dict(human_frac=0.5, sub_rate=e, ins_rate=e, del_rate=e, n_rate=0.01, paired=False)
    ill = dict(human_frac=0.5, sub_rate=0.005, ins_rate=0.0, del_rate=0.0, n_rate=0.01, paired=False)
    w = [("configs[2] ONT N50~10kb <=100kb 5% error keep-human", "ont", ont, 0.0, True, False)]
    for L in (100, 250, 300, 500, 1000, 10_000, 50_000):
        w.append((f"configs[4] sweep {L} bp single-end", L, ont if L >= 1000 else ill, 0.0, True, False))
    return w


def workload_offsets(shape, total_bases, seed):
    if shape == "ont":
        L = ont_lengths(np.random.default_rng(seed), total_bases)
    else:
        n = max(64, total_bases // int(shape))
        L = np.full(n, int(shape), np.int64)
    off = np.zeros(len(L) + 1, np.int64)
    np.cumsum(L, out=off[1:])
    return off


DUMP_BYTES = 64_000_000
DUMP_SAMPLE = 1 << 21
DUMP_SEED = 20240601


def dump_outputs(out_dir, call, keep):
    """Writes one step's results (the launches' outputs concatenated in batch order) as call.npy (external taxid,
    float64: exact for every 32-bit id) and keep.npy (0/1, float32).  Above DUMP_BYTES only a fixed seeded sample
    of positions is written, with those positions in index.npy."""
    os.makedirs(out_dir, exist_ok=True)
    n = len(call)
    if n * 12 > DUMP_BYTES:
        idx = np.sort(np.random.default_rng(DUMP_SEED).choice(n, size=min(n, DUMP_SAMPLE), replace=False))
        call, keep = call[idx], keep[idx]
        np.save(os.path.join(out_dir, "index.npy"), idx.astype(np.float64))
    np.save(os.path.join(out_dir, "call.npy"), call.astype(np.uint32).astype(np.float64))
    np.save(os.path.join(out_dir, "keep.npy"), keep.astype(np.float32))


# ---------------------------------------------------------------------------------------------
# CPU side (oracle): the only functions that touch oracle/

def oracle_db_from_cells(cells, opts_b, taxo_b, hdr):
    from oracle import k2oracle
    import ctypes as C
    import tempfile
    d = tempfile.mkdtemp(prefix="nh_bench_db_")
    with open(os.path.join(d, "opts.k2d"), "wb") as f:
        f.write(opts_b)
    with open(os.path.join(d, "taxo.k2d"), "wb") as f:
        f.write(taxo_b)
    L = k2oracle.lib()
    opts, tax = k2oracle.IndexOptions(), k2oracle.Taxonomy()
    assert L.k2o_load_opts(os.path.join(d, "opts.k2d").encode(), C.byref(opts)) == 0
    assert L.k2o_load_taxonomy(os.path.join(d, "taxo.k2d").encode(), C.byref(tax)) == 0
    return k2oracle.OracleDb.from_arrays(opts, tax, cells, hdr[0], hdr[1], hdr[3])


def cpu_timed_sample(odb, bases, offsets, target_s, cores):
    """Oracle classification of a bounded prefix of (bases, offsets): ~target_s seconds of CPU work."""
    n_pairs_all = (len(offsets) - 1) // 2

    def run(n_pairs):
        o = offsets[:2 * n_pairs + 1]
        t0 = time.perf_counter()
        r = odb.classify_batch(bases[:int(o[-1])], o, paired=True, threads=cores)
        return time.perf_counter() - t0, r

    probe_n = min(n_pairs_all, 20000)
    t, _ = run(probe_n)
    rate = probe_n / max(t, 1e-6)
    n = int(min(n_pairs_all, max(probe_n, rate * target_s)))
    t, r = run(n)
    passes = 1
    if n == n_pairs_all and t < 0.6 * target_s:  # the whole batch is faster than the budget: repeat it
        extra = int(min(30, max(1, round(target_s / max(t, 1e-3)) - 1)))
        for _ in range(extra):
            t += run(n)[0]
        passes += extra
    return {"pairs": n, "passes": passes, "seconds": t, "gbp_s": passes * n * 2 * READ_LEN / t / 1e9,
            "reads_s": passes * 2 * n / t, "cores": cores, "result": r}


# ---------------------------------------------------------------------------------------------

def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return 0 if rank != 0 else reference_arm(args)

    import torch
    import torch.distributed as dist
    from nohuman_b200 import Database, Session, synth
    from nohuman_b200 import dist as nhd

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback exists)")
    torch.cuda.set_device(local_rank)
    dev = local_rank
    use_dist = world > 1
    if use_dist:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if use_dist:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if not use_dist:
            return float(x)
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        if not use_dist:
            return int(x)
        t = torch.tensor([int(x)], dtype=torch.int64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return int(t.item())

    # ---------------- database: built on rank 0, replicated over NCCL/NVLink ----------------
    capacity = 1 << args.capacity_log2
    span = read_span(capacity)
    t_build0 = time.perf_counter()
    sdb = None
    cells = hdr = opts_b = taxo_b = None
    if rank == 0:
        sdb = synth.build_synthetic_db(capacity, device=dev, genome_seed=GENOME_SEED)
        assert sdb.genome_bases >= span, (sdb.genome_bases, span)
        opts_b, taxo_b = sdb.opts, sdb.taxo
        hdr = sdb.hash_header()
        db = sdb.db
    t_build = time.perf_counter() - t_build0
    keep_alive = None
    t_bcast = 0.0
    if use_dist:
        t0 = time.perf_counter()
        if rank == 0:
            cells = torch.as_tensor(DevPtr(sdb.db.device_cells_ptr(), nhd.padded_cells(capacity) * 4), device="cuda")
        cells, hdr, opts_b, taxo_b = nhd.broadcast_table(cells, hdr, opts_b, taxo_b, torch.device("cuda", dev))
        torch.cuda.synchronize()
        t_bcast = time.perf_counter() - t0
        if rank != 0:
            keep_alive = cells
            db = Database.from_memory(opts_b, taxo_b, hdr, cells.data_ptr(), device=dev, cells_on_device=True)
    # every replica must hold the bytes rank 0 built: 64-bit word sum of the cell array, compared on all ranks
    dcells = torch.as_tensor(DevPtr(db.device_cells_ptr(), capacity * 4), device="cuda")
    checksum = int(dcells.view(torch.int64).sum().item())
    replicas_equal = True
    if use_dist:
        sums = [None] * world
        dist.all_gather_object(sums, checksum)
        replicas_equal = all(s == sums[0] for s in sums)
    del dcells

    n_pairs = args.pairs_per_launch
    n_seqs = 2 * n_pairs
    total = n_seqs * READ_LEN
    d_off = torch.from_numpy(pair_offsets(n_pairs)).cuda()

    def make_pe_batch(seed):
        d_bases = torch.zeros(total + 64, dtype=torch.uint8, device="cuda")
        synth.synth_reads(dev, d_bases.data_ptr(), d_off.data_ptr(), n_seqs, GENOME_SEED, span, seed=seed,
                          stream=torch.cuda.current_stream().cuda_stream, **READS_PE)
        return d_bases

    n_launch = args.launches_per_step
    bufs = [make_pe_batch(1000 * (rank + 1) + b) for b in range(n_launch)]
    torch.cuda.synchronize()

    # ---------------- device-resident timing (`value`) ----------------
    sess = Session(db, confidence=CONF, paired=True, max_batch_bases=total + 4096, max_batch_seqs=n_seqs)
    # one output pair per batch: after the timed loop they hold what the last step computed
    d_calls = [torch.empty(n_pairs, dtype=torch.int32, device="cuda") for _ in range(n_launch)]
    d_keeps = [torch.empty(n_pairs, dtype=torch.uint8, device="cuda") for _ in range(n_launch)]
    d_call, d_keep = d_calls[0], d_keeps[0]
    ext = torch.cuda.ExternalStream(sess.stream)

    def launch(i):
        b = i % n_launch
        sess.classify_device(bufs[b].data_ptr(), d_off.data_ptr(), n_seqs, total, d_calls[b].data_ptr(),
                             d_keeps[b].data_ptr())
        return sess.sync()

    sampler = ClockSampler(dev)
    if rank == 0:  # one nvidia-smi poller per run is enough; rank 0's GPU is the one reported
        sampler.start()
    for i in range(args.warmup * n_launch):
        st = launch(i)

    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    stage = {"plan": 0.0, "stream_classify": 0.0, "probe": 0.0, "score_deferred": 0.0}
    lookups = sectors = launches = classified = 0
    fused_form = 0
    barrier()
    tok = sampler.mark()
    torch.cuda.cudart().cudaProfilerStart()  # `ncu --profile-from-start off` sees the timed steps only
    ev0.record(ext)
    for i in range(args.steps * n_launch):
        st = launch(i)
        stage["plan"] += st.ms_plan
        stage["stream_classify"] += st.ms_minimizer
        stage["probe"] += st.ms_probe
        stage["score_deferred"] += st.ms_score
        lookups += st.n_lookups
        sectors += st.n_sector_reads
        launches += st.gpu_launches
        classified += st.n_classified
        fused_form = int(st.fused_kernel)
    ev1.record(ext)
    barrier()
    torch.cuda.cudart().cudaProfilerStop()
    sampler.close(tok)
    ms_total = max_over_ranks(ev0.elapsed_time(ev1))
    ms_step = ms_total / args.steps
    n_timed = args.steps * n_launch
    gbp_s = world * n_pairs * 2 * READ_LEN * n_timed / (ms_total * 1e-3) / 1e9
    reads_s = world * n_seqs * n_timed / (ms_total * 1e-3)
    if fused_form != 2:  # warp-per-tile kernels (NH_LEGACY_KERNELS=1): the stages are separate kernels
        stage = {"plan": stage["plan"], "minimizer": stage["stream_classify"], "probe": stage["probe"],
                 "score": stage["score_deferred"]}
    else:
        del stage["probe"]
    for kname in stage:
        stage[kname] /= n_timed
    lk_per_launch = lookups / n_timed
    sec_per_launch = sectors / n_timed
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, torch.cat(d_calls).cpu().numpy(), torch.cat(d_keeps).cpu().numpy())

    # ---------------- e2e through the C ABI with host buffers ----------------
    e2e = None
    if not args.no_e2e:
        e2e = run_e2e(args, torch, dist if use_dist else None, db, bufs, d_off, n_pairs, n_seqs, total, world, sampler)
    clocks = sampler.stop()

    # ---------------- the probe's access pattern alone: the ceiling the kernel is held to ----------------
    probe_kernel = "stream_classify" if fused_form == 2 else "probe"
    ms_probe_kernel = stage[probe_kernel]
    roofline_probe = None
    if rank == 0:
        spill = sec_per_launch / lk_per_launch - 1.0 if sectors and lk_per_launch else 0.41
        variants = []
        # every pattern is run at several numbers of requests in flight (blocks of 256 threads per SM x chains per
        # thread); its best launch is what counts
        shapes = ((1, 1), (2, 1), (3, 1), (4, 1), (8, 1), (3, 2), (8, 2), (3, 4), (8, 4))
        for name, lanes, p, win in (("independent random sectors", 1, 0.0, 0),
                                    ("probe chains: adjacent sector after the first arrived, p = table's spill rate", 1, spill, 0),
                                    ("probe chains fetched like k_stream_classify does (cp.async by lane pairs into shared memory)",
                                     0, spill, 0),
                                    ("2 lanes per lookup (64-byte block), p = 0.24", 2, 0.24, 0),
                                    ("4 lanes per lookup (128-byte line), p = 0.12", 4, 0.12, 0),
                                    ("probe chains, every SM confined to its own 64 MiB window (not reachable by a hash table)",
                                     1, spill, 64 << 20)):
            best = None
            for bps, depth in shapes:
                if lanes == 0 and depth == 4:
                    continue
                ipc = max(16, 4096 // (bps * depth))  # every launch issues ~150 M requests: 4-5 ms
                items_s, req_s = db.probe_pattern(lanes=lanes, p_continue=p, sm_window_bytes=win, items_per_chain=ipc,
                                                  iters=4, depth=depth, blocks_per_sm=bps)
                if best is None or items_s > best[0]:
                    best = (items_s, req_s, bps, depth)
            variants.append({"pattern": name, "lanes": lanes, "p_continue": round(p, 4), "sm_window_bytes": win,
                             "lookups_per_s": round(best[0], 1), "requests_per_s": round(best[1], 1),
                             "best_blocks_per_sm": best[2], "best_chains_per_thread": best[3]})
        uniform = [v for v in variants if v["sm_window_bytes"] == 0]
        peak_req = max(v["requests_per_s"] for v in variants)
        peak_lk = max(v["lookups_per_s"] for v in variants if v["p_continue"] > 0)
        uni_req = max(v["requests_per_s"] for v in uniform)
        uni_lk = max(v["lookups_per_s"] for v in uniform if v["p_continue"] > 0)
        k_lk = lk_per_launch / (ms_probe_kernel * 1e-3)
        k_req = (sec_per_launch if sectors else lk_per_launch) / (ms_probe_kernel * 1e-3)
        roofline_probe = {
            "kernel": "k_" + probe_kernel, "lookups_per_s": round(k_lk, 1), "table_requests_per_s": round(k_req, 1),
            "sectors_per_lookup": round(sec_per_launch / lk_per_launch, 4) if sectors else None,
            "achieved_sector_gbs": round(k_req * 32.0 / 1e9, 1),
            "peak_requests_per_s": peak_req, "peak_lookups_per_s": peak_lk,
            "random_sector_peak_gbs": round(peak_req * 32.0 / 1e9, 1),
            "frac_by_requests": round(k_req / peak_req, 4), "frac_by_lookups": round(k_lk / peak_lk, 4),
            "frac_of_random_sector_peak": round(k_req / peak_req, 4),
            "uniform_random_peak_requests_per_s": uni_req, "uniform_random_peak_lookups_per_s": uni_lk,
            "frac_of_uniform_random_requests": round(k_req / uni_req, 4),
            "frac_of_uniform_random_lookups": round(k_lk / uni_lk, 4),
            "patterns": variants,
            "note": "every pattern runs alone on the same table in the same process, at 9 numbers of requests in flight, best "
                    "launch kept.  peak_* = best over ALL patterns, including the one that confines every SM to its own 64 MiB "
                    "window (perfect page locality; a hash table cannot produce it); uniform_random_* = best over the patterns "
                    "with uniformly random addresses, which is what hashing k-mers produces - the fused kernel runs at that "
                    "rate (a fraction slightly above 1 is the spread between a continuous microbenchmark and the kernel's "
                    "bursts of 32 requests per warp).  sectors_per_lookup counts every 32-byte request of the kernel, table "
                    "sectors and miss-filter records alike: with the filter a lookup needs fewer of them than the table's "
                    "probe chains alone (cpu_baseline.oracle_sectors_per_lookup), and the patterns are run at the kernel's "
                    "own continuation rate",
        }

    # ---------------- parity: every rank, its own replica, one common batch ----------------
    odb = None
    host_cells = None
    parity = None
    if not args.no_parity:
        common = make_pe_batch(COMMON_SEED)
        torch.cuda.synchronize()
        want = torch.zeros(n_pairs, dtype=torch.int32, device="cuda")
        n_check = n_pairs
        if rank == 0:
            host_cells = sdb.download_cells()
            odb = oracle_db_from_cells(host_cells, opts_b, taxo_b, hdr)
            odb.confidence = CONF
            h_bases = common[:total].cpu().numpy()
            r = odb.classify_batch(h_bases, pair_offsets(n_pairs).astype(np.uint64), paired=True)
            want.copy_(torch.from_numpy(r["ext"].astype(np.int32)))
        if use_dist:
            dist.broadcast(want, 0)
        sess.classify_device(common.data_ptr(), d_off.data_ptr(), n_seqs, total, d_call.data_ptr(), d_keep.data_ptr())
        sess.sync()
        mism = int((d_call != want).sum().item())
        keep_bad = int((d_keep != (want == 0).to(torch.uint8)).sum().item())
        parity = {"ranks_checked": sum_over_ranks(1), "pairs_checked_per_rank": n_check,
                  "mismatches": sum_over_ranks(mism), "keep_mask_mismatches": sum_over_ranks(keep_bad),
                  "replica_checksums_equal": bool(replicas_equal),
                  "how": "each rank classifies the same seeded 1M-pair batch against its own replica; expected calls from "
                         "the CPU oracle on rank 0, broadcast; counts summed over ranks"}
        del common
    sess.close()
    del bufs
    torch.cuda.empty_cache()

    # ---------------- BASELINE configs[2] and configs[4], at this N ----------------
    workloads = None
    if not args.no_workloads:
        peak_lk = roofline_probe["uniform_random_peak_lookups_per_s"] if roofline_probe else None
        peak_req = roofline_probe["uniform_random_peak_requests_per_s"] if roofline_probe else None
        if use_dist:
            t = torch.tensor([peak_lk or 0.0, peak_req or 0.0], dtype=torch.float64, device="cuda")
            dist.broadcast(t, 0)
            peak_lk, peak_req = (float(x) or None for x in t.tolist())
        workloads = run_workloads(args, torch, dist if use_dist else None, db, synth, Session, odb, span, rank, world,
                                  dev, peak_lk, peak_req, max_over_ranks, sum_over_ranks)

    if rank != 0:
        if use_dist:
            dist.barrier()
            dist.destroy_process_group()
        return 0

    # ---------------- roofline of the dominant kernel ----------------
    peak, peak_src = peaks()
    if fused_form == 2:
        # one kernel: 1 B/base read + one 32 B sector per lookup + 5 B/unit of results (SURVEY §8d)
        alg = {"stream_classify": total * 1.0 + lk_per_launch * 32.0 + n_pairs * 5.0, "score_deferred": 0.0, "plan": n_seqs * 8.0}
    else:
        alg = {"minimizer": total * 1.0 + lk_per_launch * 10.0, "probe": lk_per_launch * 32.0,
               "score": lk_per_launch * 6.0 + n_pairs * 5.0, "plan": n_seqs * 8.0}
    dom = max(stage, key=lambda k_: stage[k_])
    traffic_tab = {}
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        with open(tpath) as f:
            tj = json.load(f)
        w = tj.get("workload", {})
        if w.get("pairs_per_launch") == n_pairs and w.get("table_cells") == capacity and w.get("read_len") == READ_LEN:
            traffic_tab = tj
    ach = alg[dom] / (stage[dom] * 1e-3) / 1e9 if stage[dom] > 0 else 0.0
    roofline = {"kernel": "k_" + dom, "bound": "hbm", "achieved": round(ach, 1), "peak": peak, "unit": "GB/s",
                "frac": round(ach / peak, 4), "traffic": traffic_tab.get("k_" + dom, {}).get("dram_bytes_per_launch"),
                "peak_source": peak_src, "ms_per_launch": round(stage[dom], 4),
                "algorithmic_bytes_per_launch": int(alg[dom]),
                "note": "per launch of 1M pairs; the HBM streaming peak is the denominator the contract asks for, "
                        "roofline_probe holds the request-rate ceiling that actually binds"}

    cfg = workload_config(args)
    out = {
        "metric": METRIC, "value": round(gbp_s, 3), "unit": UNIT, "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_step, 4),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64",
        "data": "synthetic", "config": cfg,
        "run": {"table_load": round(hdr[1] / capacity, 4), "genome_bases": int(sdb.genome_bases),
                "db_build_s": round(t_build, 2), "db_broadcast_s": round(t_bcast, 2),
                "parallelism": f"dp{world} (read batches sharded, table replicated via NCCL broadcast)",
                "miss_filter": {"bytes": int(db.info.filter_bytes), "mode": int(os.environ.get("NH_FILTER_MODE", "3")),
                                "what": "one 32-byte record per block of 32 table cells (occupancy + Bloom bits of the keys stored "
                                        "in the block), built on the device when the table is opened; units whose last lookups "
                                        "all missed ask it before the table, so a lookup that misses costs one request instead of 1.65 "
                                        "(DESIGN.md §2)"}},
        "reads_per_s": round(reads_s, 1),
        "stage_ms_per_launch": {k_: round(v, 4) for k_, v in stage.items()},
        "lookups_per_launch": int(lk_per_launch),
        "kernel_path": {0: "warp-per-tile", 2: "streaming (k_stream_classify)"}.get(fused_form, str(fused_form)),
        "classified_frac": round(classified / (n_timed * n_pairs), 4),
        "gpu_launches": int(launches),
        "clocks": clocks, "roofline": roofline, "roofline_probe": roofline_probe,
    }
    if e2e:
        out["e2e"] = e2e
    if parity:
        out["parity_vs_oracle"] = parity
    if workloads is not None:
        out["workloads"] = workloads

    if world == 1 and not args.no_cpu_baseline:
        if odb is None:
            host_cells = sdb.download_cells()
            odb = oracle_db_from_cells(host_cells, opts_b, taxo_b, hdr)
        odb.confidence = CONF
        b0 = torch.zeros(total + 64, dtype=torch.uint8, device="cuda")
        synth.synth_reads(dev, b0.data_ptr(), d_off.data_ptr(), n_seqs, GENOME_SEED, span, seed=1000, **READS_PE)
        torch.cuda.synchronize()
        cb = cpu_timed_sample(odb, b0[:total].cpu().numpy(), pair_offsets(n_pairs).astype(np.uint64), 12.0,
                              os.cpu_count() or 1)
        out["cpu_baseline"] = {
            "value": round(cb["gbp_s"], 5), "unit": UNIT, "cores": cb["cores"], "kind": "port",
            "sample": f"first {cb['pairs']} pairs of one launch's batch x {cb['passes']} passes, {cb['seconds']:.1f} s, "
                      "kraken2 restatement (upstream binary unavailable offline), OpenMP",
            "reads_per_s": round(cb["reads_s"], 1),
            "oracle_lookups_per_pair": round(cb["result"]["lookups"] / cb["pairs"], 2),
            "oracle_sectors_per_lookup": round(cb["result"]["sectors"] / max(1, cb["result"]["lookups"]), 3),
        }
    print(json.dumps(out))
    if use_dist:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def run_e2e(args, torch, dist, db, bufs, d_off, n_pairs, n_seqs, total, world, sampler=None):
    """Same metric through the C ABI with pinned HOST buffers holding ASCII reads: every launch copies its input
    H2D and its calls + keep mask D2H.  Two sessions on two host threads overlap one launch's copies with the
    other's kernel.  A step is again launches_per_step launches.

    Two transfer formats for the same ASCII host buffers: "ascii" = nh_classify_batch (1 byte per base over
    PCIe, no host core involved); "packed" = nh_classify_batch_pack (the host cores pack INSIDE the timed region,
    0.43 byte per base crosses PCIe), run with several sessions on as many host threads so that the cores keep
    packing while other sessions' copies and kernels run.  Packing needs the host's cores and memory bandwidth,
    so it is measured at N = 1 only (one process per host); `e2e` is the better of the two."""
    from nohuman_b200 import Session
    shapes = []
    cores = os.cpu_count() or 16
    spec = args.e2e_packed
    if spec == "auto":  # twice as many packer threads as cores, spread over sessions that take turns sleeping on their copies and kernels
        a, b = min(12, max(2, cores // 2)), min(12, max(2, cores * 3 // 8))
        spec = f"{a}x{max(1, 2 * cores // a)},{b}x{max(1, 2 * cores // b + 1)},{b}x{max(1, 3 * cores // (2 * b))}"
    for item in spec.split(","):
        w, t = item.lower().split("x")
        shapes.append((max(1, int(w)), int(t) if int(t) > 0 else max(1, (os.cpu_count() or 2) // max(1, int(w)))))
    n_workers = max([2] + [w for w, _ in shapes]) if world == 1 else 2
    n_host = min(4, len(bufs))  # distinct pinned host batches (1.3 GB), cycled
    sessions = [Session(db, confidence=CONF, paired=True, max_batch_bases=total + 4096,
                        max_batch_seqs=n_seqs) for _ in range(n_workers)]
    host = []
    ho = torch.empty(n_seqs + 1, dtype=torch.int64).pin_memory()
    ho.copy_(d_off)
    for b in bufs[:n_host]:
        hb = torch.empty(total, dtype=torch.uint8).pin_memory()
        hb.copy_(b[:total])
        host.append(hb)
    outs = [(torch.empty(n_pairs, dtype=torch.int32).pin_memory(), torch.empty(n_pairs, dtype=torch.uint8).pin_memory())
            for _ in range(n_workers)]
    units = n_seqs * ((READ_LEN + 31) // 32)
    torch.cuda.synchronize()
    n_launch = args.launches_per_step
    steps = args.steps
    cur = {"workers": 2, "pack_threads": max(1, (os.cpu_count() or 2) // 2)}

    def worker(fmt, w, n):
        hc, hk = outs[w]
        nw, pack_threads = cur["workers"], cur["pack_threads"]
        for i in range(n):
            hb = host[(w + nw * i) % n_host]
            if fmt == "ascii":
                sessions[w].classify_raw(hb.data_ptr(), ho.data_ptr(), n_seqs, hc.data_ptr(), hk.data_ptr())
            else:
                sessions[w].classify_pack_raw(hb.data_ptr(), ho.data_ptr(), n_seqs, pack_threads, hc.data_ptr(), hk.data_ptr())

    def run(fmt, n_total):
        nw = cur["workers"]
        ths = [threading.Thread(target=worker, args=(fmt, w, n_total // nw + (1 if w < n_total % nw else 0)))
               for w in range(nw)]
        for t in ths:
            t.start()
        for t in ths:
            t.join()

    def timed(fmt):
        run(fmt, max(args.warmup, 1) * cur["workers"] * 2)
        if dist:
            dist.barrier()
        torch.cuda.synchronize()
        tok = sampler.mark() if sampler else None
        t0 = time.perf_counter()
        run(fmt, steps * n_launch)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if sampler:
            sampler.close(tok)
        if dist:
            t = torch.tensor([dt], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        # outside the timed region: the first host batch once more through the same entry point, so that the formats
        # are compared on the same reads whatever batch a worker happened to finish on
        worker(fmt, 0, 1)
        calls = torch.cat([outs[0][0].clone(), outs[0][1].clone().to(torch.int32)])
        h2d = (total + (n_seqs + 1) * 8) if fmt == "ascii" else (units * 12 + n_seqs * 4)
        return {"value": round(world * steps * n_launch * n_pairs * 2 * READ_LEN / dt / 1e9, 3), "unit": UNIT,
                "h2d_bytes_per_step": int(n_launch * h2d), "d2h_bytes_per_step": int(n_launch * n_pairs * 5),
                "ms_per_step": round(dt / steps * 1e3, 4), "steps": steps}, calls

    res_a, calls_a = timed("ascii")
    res_a["input_format"] = "ASCII, 1 byte per base (nh_classify_batch)"
    formats = {"ascii": res_a}
    best = res_a
    if world == 1:
        # nh_classify_batch_pack at several thread shapes (session threads x packing threads per session);
        # the best one that reproduces the ASCII calls counts
        res_p, sweep = None, []
        for nw, pt in shapes:
            cur["workers"], cur["pack_threads"] = nw, pt
            r, calls_p = timed("packed")
            r["session_threads"], r["pack_threads_per_session_thread"] = nw, pt
            r["same_calls_as_ascii"] = bool(torch.equal(calls_a, calls_p))
            sweep.append({"session_threads": nw, "pack_threads": pt, "value": r["value"]})
            if res_p is None or (r["same_calls_as_ascii"] and r["value"] > res_p["value"]):
                res_p = r
        res_p["input_format"] = ("ASCII host buffers handed to nh_classify_batch_pack: packed by the host cores INSIDE the timed region "
                                 "(AVX2, 2-bit codes + validity bits), 0.43 byte per base over PCIe")
        if len(sweep) > 1:
            res_p["shapes_tried"] = sweep
        formats["packed"] = res_p
        if res_p["value"] > best["value"] and res_p["same_calls_as_ascii"]:
            best = res_p
        cur["workers"] = 2
    for s in sessions:
        s.close()
    out = dict(best)
    out["api"] = (f"host buffers (pinned ASCII), {best.get('session_threads', 2)} sessions on as many host threads, "
                  f"{n_host} distinct host batches cycled")
    out["formats"] = formats
    out["note"] = ("packing costs host cores (tools/pack_bench.cc: 8 Gbases/s per core, 86-103 on 16) while one PCIe link moves 52 Gbases/s "
                   "of ASCII without using a core; with more than one rank per host the ASCII path is measured (DESIGN.md §4c)")
    return out


def run_workloads(args, torch, dist, db, synth, Session, odb, span, rank, world, dev, peak_lk, peak_req, max_over_ranks,
                  sum_over_ranks):
    """BASELINE configs[2] / configs[4]: device-resident timing of every shape on every rank's own batch, plus an
    oracle parity sample of >= 20 Mbp that all ranks classify on their own replica."""
    rows = []
    total_target = args.workload_mbases * 1_000_000
    for name, shape, sampler_args, conf, keep_human, paired in workload_list(args):
        off = workload_offsets(shape, total_target, seed=7)  # same lengths on every rank, different reads
        n = len(off) - 1
        total = int(off[-1])
        d_off = torch.from_numpy(off).cuda()
        d_bases = torch.zeros(total + 64, dtype=torch.uint8, device="cuda")
        synth.synth_reads(dev, d_bases.data_ptr(), d_off.data_ptr(), n, GENOME_SEED, span, seed=9000 + 17 * rank, **sampler_args)
        # the parity sample: a prefix of >= 20 Mbp of a batch seeded the same on every rank
        n_s = min(n, int(np.searchsorted(off, 20_000_000)) + 1)
        s_total = int(off[n_s])
        d_sample = torch.zeros(s_total + 64, dtype=torch.uint8, device="cuda")
        synth.synth_reads(dev, d_sample.data_ptr(), d_off.data_ptr(), n_s, GENOME_SEED, span, seed=COMMON_SEED, **sampler_args)
        torch.cuda.synchronize()
        d_call = torch.empty(n, dtype=torch.int32, device="cuda")
        d_keep = torch.empty(n, dtype=torch.uint8, device="cuda")
        want = torch.zeros(n_s, dtype=torch.int32, device="cuda")
        have_oracle = torch.tensor([1 if odb is not None else 0], dtype=torch.int32, device="cuda")
        if rank == 0 and odb is not None:
            odb.confidence = conf
            r = odb.classify_batch(d_sample[:s_total].cpu().numpy(), off[:n_s + 1].astype(np.uint64), paired=paired)
            want.copy_(torch.from_numpy(r["ext"].astype(np.int32)))
        if dist:
            dist.broadcast(want, 0)
            dist.broadcast(have_oracle, 0)
        with Session(db, confidence=conf, keep_human=keep_human, paired=paired, max_batch_bases=total + 4096,
                     max_batch_seqs=n) as sess:
            ext = torch.cuda.ExternalStream(sess.stream)
            sess.classify_device(d_sample.data_ptr(), d_off.data_ptr(), n_s, s_total, d_call.data_ptr(), d_keep.data_ptr())
            sess.sync()
            mism = int((d_call[:n_s] != want).sum().item()) if int(have_oracle.item()) else -1
            keep_bad = int((d_keep[:n_s] != (want != 0).to(torch.uint8)).sum().item()) if keep_human else 0
            for _ in range(2):
                sess.classify_device(d_bases.data_ptr(), d_off.data_ptr(), n, total, d_call.data_ptr(), d_keep.data_ptr())
                st = sess.sync()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            if dist:
                dist.barrier()
            torch.cuda.synchronize()
            reps = 4
            fused = 0.0
            e0.record(ext)
            for _ in range(reps):
                sess.classify_device(d_bases.data_ptr(), d_off.data_ptr(), n, total, d_call.data_ptr(), d_keep.data_ptr())
                st = sess.sync()
                fused += st.ms_minimizer
            e1.record(ext)
            torch.cuda.synchronize()
            ms = max_over_ranks(e0.elapsed_time(e1) / reps)
            ms_fused = max_over_ranks(fused / reps)
        lk = int(st.n_lookups)
        sec = int(st.n_sector_reads)
        row = {"workload": name, "reads_per_gpu": n, "bases_per_gpu": total, "ms_per_launch": round(ms, 4),
               "gbp_s": round(world * total / ms / 1e6, 2), "reads_per_s": round(world * n / ms * 1e3, 1),
               "lookups_per_s": round(world * lk / ms_fused * 1e3, 1),
               "sectors_per_lookup": round(sec / lk, 4) if lk and sec else None,
               "table_requests_per_s": round(world * sec / ms_fused * 1e3, 1),
               "frac_of_uniform_random_requests": round(sec / (ms_fused * 1e-3) / peak_req, 4) if peak_req and sec else None,
               "frac_of_uniform_random_lookups": round(lk / (ms_fused * 1e-3) / peak_lk, 4) if peak_lk else None,
               "stage_ms": {"plan": round(st.ms_plan, 4), "stream_classify": round(st.ms_minimizer, 4),
                            "score_deferred": round(st.ms_score, 4)},
               "classified_frac": round(st.n_classified / n, 4),
               "parity_vs_oracle": {"sample_reads": n_s, "sample_bases": s_total, "ranks_checked": sum_over_ranks(1),
                                    "mismatches": sum_over_ranks(max(mism, 0)) if mism >= 0 else None,
                                    "keep_mask_mismatches": sum_over_ranks(keep_bad)}}
        rows.append(row)
        del d_bases, d_sample, d_call, d_keep, d_off, want
        torch.cuda.empty_cache()
    return rows


def reference_arm(args):
    """CPU implementation of the path on the host cores: the oracle port of kraken2's classifier
    (kraken2 itself is not installable offline), on the same workload.  No torch, no CUDA library:
    the table and the reads come from the generator's CPU twin (oracle/k2_synth.c)."""
    from oracle import k2synth
    capacity = 1 << args.capacity_log2
    cores = os.cpu_count() or 1
    t0 = time.perf_counter()
    odb, meta = k2synth.build_synthetic_db(capacity, genome_seed=GENOME_SEED, threads=cores)
    t_build = time.perf_counter() - t0
    odb.confidence = CONF
    span = read_span(capacity)
    n_pairs = args.pairs_per_launch
    off = pair_offsets(n_pairs).astype(np.uint64)
    bases = k2synth.synth_reads(off, GENOME_SEED, span, seed=1000, threads=cores, **READS_PE)  # rank 0's first batch
    probe = cpu_timed_sample(odb, bases, off, 1.0, cores)
    n = args.ref_pairs_per_step or probe["pairs"]
    n = min(n, n_pairs)
    o = off[:2 * n + 1]
    bb = bases[:int(o[-1])]
    for _ in range(max(1, min(args.warmup, 2))):
        odb.classify_batch(bb, o, paired=True, threads=cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        odb.classify_batch(bb, o, paired=True, threads=cores)
    dt = time.perf_counter() - t0
    gbp_s = args.steps * n * 2 * READ_LEN / dt / 1e9
    out = {
        "impl": "reference", "metric": METRIC, "value": round(gbp_s, 5), "unit": UNIT,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(dt / args.steps * 1e3, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64", "data": "synthetic", "config": workload_config(args),
        "run": {"table_load": round(meta["hash_header"][1] / capacity, 4), "genome_bases": meta["genome_bases"],
                "db_build_s": round(t_build, 2), "table_built_by": "oracle/k2_synth.c on the host cores"},
        "reads_per_s": round(args.steps * 2 * n / dt, 1),
        "cpu_baseline": {"value": round(gbp_s, 5), "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{n} pairs per step (a bounded sample of the 10M-pair step) x {args.steps} steps; kraken2 "
                                   "restatement (upstream binary unavailable offline), OpenMP on all host cores"},
        "e2e": {"value": round(gbp_s, 5), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out))
    return 0


if __name__ == "__main__":
    sys.exit(main())
