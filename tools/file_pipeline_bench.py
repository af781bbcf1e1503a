#!/usr/bin/env python
"""BASELINE configs[1] as the user runs it: `nohuman -t T --conf 0.5 r_1.fq.gz r_2.fq.gz` on N pairs of 2x150 bp
FASTQ (50 % genome-derived), gzip in / gzip out, against the synthetic HPRC.r2-sized table, on 1..N GPUs of the box.
Wall clock of the whole CLI process and of the pipeline alone, busy seconds per host stage, and a check of the
OUTPUT BYTES against what the CPU oracle says must be kept.

    python tools/file_pipeline_bench.py [--pairs 10000000] [--threads 16[,4...]] [--capacity-log2 31] [--gpus 1]
                                        [--gpu-gzip]

--threads takes a comma-separated list: every variant runs at each count.  --gpu-gzip deflates the gzip
output on the GPU (nohuman --gpu-gzip) instead of on the host threads.
"""
import argparse
import hashlib
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def fastq_array(seqs2d: np.ndarray, mate: int) -> np.ndarray:
    n, L = seqs2d.shape
    hdr = np.frombuffer(b"@r000000000/%d\n" % mate, np.uint8).copy()
    rec = np.empty((n, len(hdr) + L + 3 + L + 1), np.uint8)
    rec[:, :len(hdr)] = hdr
    idx = np.arange(n)
    for d in range(9):
        rec[:, 2 + 8 - d] = 48 + (idx // 10 ** d) % 10
    o = len(hdr)
    rec[:, o:o + L] = seqs2d
    rec[:, o + L:o + L + 3] = np.frombuffer(b"\n+\n", np.uint8)
    rec[:, o + L + 3:o + 2 * L + 3] = ord("I")
    rec[:, -1] = ord("\n")
    return rec


def sha_of_stream(cmd):
    h = hashlib.sha256()
    p = subprocess.Popen(cmd, stdout=subprocess.PIPE)
    n = 0
    while True:
        b = p.stdout.read(1 << 24)
        if not b:
            break
        h.update(b)
        n += len(b)
    assert p.wait() == 0, cmd
    return h.hexdigest(), n


def sha_of_rows(rec2d, keep):
    h = hashlib.sha256()
    n = 0
    for lo in range(0, len(rec2d), 1 << 18):
        blk = rec2d[lo:lo + (1 << 18)][keep[lo:lo + (1 << 18)]]
        h.update(blk.tobytes())
        n += blk.size
    return h.hexdigest(), n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=10_000_000)
    ap.add_argument("--threads", default=str(os.cpu_count() or 16))
    ap.add_argument("--capacity-log2", type=int, default=31)
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--variants", default="gz-gz,bgz-gz,plain-plain,gz-plain,bgz-plain,plain-gz")
    ap.add_argument("--tmp", default=None)
    ap.add_argument("--gpu-gzip", action="store_true")
    args = ap.parse_args()
    thread_counts = [int(t) for t in args.threads.split(",")]
    import torch
    from nohuman_b200 import synth
    from oracle import k2oracle  # the checker of the output bytes; not in any timed region
    torch.cuda.set_device(0)
    capacity = 1 << args.capacity_log2
    sdb = synth.build_synthetic_db(capacity, device=0)
    d = tempfile.mkdtemp(prefix="nh_filebench_", dir=args.tmp)
    db_dir = os.path.join(d, "db")
    t0 = time.perf_counter()
    sdb.save(db_dir)
    t_save = time.perf_counter() - t0
    n_seqs, L = 2 * args.pairs, 150
    seqs = np.empty((n_seqs, L), np.uint8)
    step = 2_000_000  # sequences per generator launch
    for lo in range(0, n_seqs, step):
        m = min(step, n_seqs - lo)
        d_off = torch.arange(m + 1, dtype=torch.int64, device="cuda") * L
        d_bases = torch.zeros(m * L + 64, dtype=torch.uint8, device="cuda")
        synth.synth_reads(0, d_bases.data_ptr(), d_off.data_ptr(), m, sdb.genome_seed, 2 * capacity, seed=3 + lo,
                          paired=True, n_rate=0.01)
        torch.cuda.synchronize()
        seqs[lo:lo + m] = d_bases[:m * L].cpu().numpy().reshape(m, L)
    # what must come out: the pairs the oracle leaves unclassified at --conf 0.5
    import ctypes as C
    odb = k2oracle.OracleDb.load(db_dir)
    odb.confidence = 0.5
    t0 = time.perf_counter()
    want = odb.classify_batch(seqs.reshape(-1), (np.arange(n_seqs + 1, dtype=np.uint64) * L), paired=True)
    t_oracle = time.perf_counter() - t0
    keep = want["ext"] == 0
    sdb.db.close()
    del odb
    torch.cuda.empty_cache()
    rec1, rec2 = fastq_array(seqs[0::2], 1), fastq_array(seqs[1::2], 2)
    del seqs
    exp1, exp2 = sha_of_rows(rec1, keep), sha_of_rows(rec2, keep)
    p1, p2 = os.path.join(d, "s_1.fq"), os.path.join(d, "s_2.fq")
    rec1.tofile(p1)
    rec2.tofile(p2)
    del rec1, rec2
    zs = [subprocess.Popen(["gzip", "-k", "-1", p]) for p in (p1, p2)]  # ordinary single-member gzip, both files at once
    assert all(z.wait() == 0 for z in zs)
    variants = args.variants.split(",")
    b1, b2 = os.path.join(d, "b_1.fq.gz"), os.path.join(d, "b_2.fq.gz")
    if any(v.startswith("bgz") for v in variants):
        # blocked gzip (BGZF: what bgzip / bcl2fastq / this library write) of the same reads, made with the host-only hook
        from nohuman_b200.api import rewrite_files
        rewrite_files(np.ones(args.pairs, np.uint8), np.zeros(args.pairs, np.uint32), p1, b1, p2, b2, out_format="g",
                      threads=max(thread_counts))
    cli = os.path.join(ROOT, "nohuman_b200", "bin", "nohuman")
    rows = []
    gbp = args.pairs * 2 * L / 1e9
    ins = {"plain": (p1, p2), "gz": (p1 + ".gz", p2 + ".gz"), "bgz": (b1, b2)}
    for v, threads in [(v, t) for t in thread_counts for v in variants]:
        vin, vout = v.split("-")
        a, b = ins[vin]
        fmt = "g" if vout == "gz" else "u"
        o1, o2 = os.path.join(d, "o1"), os.path.join(d, "o2")
        t0 = time.perf_counter()
        r = subprocess.run([cli, "-v", "--db", db_dir, "-t", str(threads), "--conf", "0.5", "-F", fmt, "-o", o1, "-O", o2,
                            "--gpus", str(args.gpus), *(["--gpu-gzip"] if args.gpu_gzip else []), a, b],
                           capture_output=True, text=True)
        dt = time.perf_counter() - t0
        assert r.returncode == 0, r.stderr
        dbg = [ln.split("] ", 1)[1] for ln in r.stderr.splitlines() if "DEBUG" in ln]
        line = [ln for ln in r.stderr.splitlines() if "classified as human" in ln][0].split("] ", 1)[1]
        pipe_s = float([x for x in dbg if " s, " in x and "Mbp" in x][0].split(" s")[0])
        load_s = float([x for x in dbg if x.startswith("database load")][0].split()[2])
        busy = [x for x in dbg if x.startswith("busy seconds")][0]
        stages = {m.group(1): float(m.group(2)) for m in re.finditer(r"(inflate|parse|stage|classify|serialise|compress|write) ([0-9.]+)", busy)}
        got1 = sha_of_stream(["gzip", "-dc", o1] if fmt == "g" else ["cat", o1])
        got2 = sha_of_stream(["gzip", "-dc", o2] if fmt == "g" else ["cat", o2])
        rows.append({"variant": f"{vin} in, {vout} out" + (" (configs[1])" if v == "gz-gz" else ""), "gpus": args.gpus,
                     "threads": threads, "gpu_gzip": bool(args.gpu_gzip and fmt == "g"),
                     "seconds": round(dt, 2), "gbp_s": round(gbp / dt, 3),
                     "pipeline_seconds": pipe_s, "pipeline_gbp_s": round(gbp / pipe_s, 3), "database_load_seconds": load_s,
                     "busy_seconds_per_stage": stages,
                     "stage_occupancy": {k_: round(v_ / pipe_s, 2) for k_, v_ in stages.items()},
                     "out_bytes": os.path.getsize(o1) + os.path.getsize(o2), "summary": line,
                     "output_matches_oracle": bool(got1 == exp1 and got2 == exp2),
                     "kept_pairs_expected": int(keep.sum())})
        print(json.dumps(rows[-1]), file=sys.stderr)
    print(json.dumps({"pairs": args.pairs, "threads": thread_counts, "host_cores": os.cpu_count(), "gpus": args.gpus,
                      "table_cells": capacity, "db_save_seconds": round(t_save, 1), "oracle_seconds_all_cores": round(t_oracle, 1),
                      "note": "seconds = whole CLI process (CUDA context + database load + pipeline); stage_occupancy = busy seconds "
                              "of the stage summed over its threads / pipeline seconds (a value of 7 means seven threads' worth)",
                      "rows": rows}, indent=1))
    import shutil
    shutil.rmtree(d, ignore_errors=True)


if __name__ == "__main__":
    main()
