#!/usr/bin/env python
"""GPU database build (nh_build_db, kraken2-build --build) on a seeded synthetic library shaped like a human
pangenome: --haplotypes records of chromosome length (--gbp in all), each a copy of one base sequence with
--snp-rate substitutions and runs of N, written as FASTA (80 bases a line) both plain and gzip (level 1,
one file per record), with matching nodes.dmp / names.dmp / seqid2taxid.map.  Prints one JSON line per
library form, after the card's name and power limit:

- library_gbp_s: library bases over the build's wall clock (taxonomy + estimate + insert + write);
- seconds per phase (nh_build_stats_t), and insert_gbp_s / estimate_gbp_s for the two library passes;
- estimate against size: the capacity pass's estimate of distinct minimizers, and the occupied cells of the
  table the same build wrote (distinct minimizers, less the rare pairs kraken2 merges on a shared compacted key);
- the oracle's sequential CPU build (oracle/k2_oracle.c, k2o_build_add_sequence) on a 1/--oracle-div subset of
  the library: one process per host core, each building its own table from its share of the subset, so the
  aggregate rate is an upper bound for a threaded CPU build of the same code.

    python tools/build_db_bench.py [--gbp 4] [--haplotypes 24] [--device 0] [--json out.jsonl]
"""
import argparse
import gzip
import json
import multiprocessing as mp
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ACGT = np.frombuffer(b"ACGT", np.uint8)


def card(device):
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(device), "--query-gpu=name,power.limit",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=60).stdout.strip()
        name, power = [x.strip() for x in q.split(",")]
        return name, power
    except Exception as e:  # the numbers stand without it, but say so
        return f"unknown ({e})", "unknown"


def haplotype(base, i, snp_rate, seed):
    rng = np.random.default_rng(seed + 1000 + i)
    s = base.copy()
    n = len(s)
    pos = rng.integers(0, n, size=int(n * snp_rate))
    s[pos] = ACGT[rng.integers(0, 4, size=len(pos))]
    for _ in range(20):  # assembly gaps
        a = int(rng.integers(0, n - 200_000))
        s[a:a + int(rng.integers(1_000, 100_000))] = ord("N")
    return s


def fasta_bytes(name, s, width=80):
    pad = (-len(s)) % width
    body = np.concatenate([s, np.full(pad, ord("\n"), np.uint8)]).reshape(-1, width)
    body = np.hstack([body, np.full((len(body), 1), ord("\n"), np.uint8)]).tobytes()
    if pad:
        body = body[: len(body) - pad - 1] + b"\n"
    return f">{name} synthetic haplotype\n".encode() + body


def gzip_file(args):
    src, dst = args
    with open(src, "rb") as f, gzip.open(dst, "wb", compresslevel=1) as g:
        shutil.copyfileobj(f, g, 16 << 20)
    return dst


def write_library(d, gbp, n_hap, snp_rate, seed):
    from nohuman_b200 import synth
    nodes, leaves = synth.human_pangenome_taxonomy(n_super=6, n_hap_per_super=(n_hap + 5) // 6)
    leaves = leaves[:n_hap]
    with open(os.path.join(d, "nodes.dmp"), "w") as f:
        for n in nodes:
            f.write(f"{n.ext_id}\t|\t{n.parent_ext_id}\t|\t{n.rank}\t|\t\t|\n")
    with open(os.path.join(d, "names.dmp"), "w") as f:
        for n in nodes:
            f.write(f"{n.ext_id}\t|\t{n.name}\t|\t\t|\tscientific name\t|\n")
    hap_len = int(gbp * 1e9 / n_hap)
    base = ACGT[np.random.default_rng(seed).integers(0, 4, size=hap_len, dtype=np.uint8)]
    plain = []
    with open(os.path.join(d, "seqid2taxid.map"), "w") as m:
        for i in range(n_hap):
            name = f"hap{i:02d}"
            m.write(f"{name}\t{leaves[i]}\n")
            p = os.path.join(d, f"{name}.fna")
            with open(p, "wb") as f:
                f.write(fasta_bytes(name, haplotype(base, i, snp_rate, seed)))
            plain.append(p)
    with mp.Pool(min(len(plain), os.cpu_count() or 1)) as pool:
        gz = pool.map(gzip_file, [(p, p + ".gz") for p in plain])
    return plain, gz, hap_len


def oracle_share(args):
    """seconds of the oracle's sequential build of bases [start, start + n) of one haplotype file"""
    path, start, n = args
    from oracle import k2oracle as K
    from nohuman_b200 import synth
    nodes, leaves = synth.human_pangenome_taxonomy()
    tax = [K.TaxSpec(x.ext_id, x.parent_ext_id, x.name, x.rank) for x in nodes]
    with open(path, "rb") as f:
        hdr = len(f.readline())
        f.seek(hdr + (start // 80) * 81)
        seq = f.read(n + n // 80 + 162).replace(b"\n", b"")[start % 80:start % 80 + n]
    t0 = time.perf_counter()
    K.OracleDb.build([(leaves[0], seq)], tax, capacity=max(1024, int(n / 3 / 0.7)))
    return time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gbp", type=float, default=4.0)
    ap.add_argument("--haplotypes", type=int, default=24)
    ap.add_argument("--snp-rate", type=float, default=0.001)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--threads", type=int, default=os.cpu_count() or 1)
    ap.add_argument("--oracle-div", type=int, default=50)
    ap.add_argument("--json", default=None)
    ap.add_argument("--workdir", default=None, help="where the library is written (default: a temporary directory)")
    a = ap.parse_args()
    name, power = card(a.device)
    head = dict(card=name, power_limit=power, gbp=a.gbp, haplotypes=a.haplotypes, host_cores=os.cpu_count())
    print(json.dumps(head), flush=True)
    out = open(a.json, "a") if a.json else None
    if out:
        out.write(json.dumps(head) + "\n")
    from nohuman_b200 import api
    work = tempfile.mkdtemp(prefix="nh_build_bench_", dir=a.workdir)
    try:
        t0 = time.perf_counter()
        plain, gz, hap_len = write_library(work, a.gbp, a.haplotypes, a.snp_rate, a.seed)
        lib_s = time.perf_counter() - t0
        for form, files in (("plain", plain), ("gzip", gz)):
            db = os.path.join(work, f"db_{form}")
            t0 = time.perf_counter()
            st = api.build_db(files, os.path.join(work, "nodes.dmp"), os.path.join(work, "names.dmp"),
                              os.path.join(work, "seqid2taxid.map"), db, threads=a.threads, device=a.device)
            wall = time.perf_counter() - t0
            phases = st.s_taxonomy + st.s_estimate + st.s_insert + st.s_write
            rec = dict(card=name, power_limit=power, form=form, files=len(files), gbp=st.bases / 1e9,
                       library_gbp_s=st.bases / 1e9 / phases, wall_s=wall, seconds=dict(
                           taxonomy=st.s_taxonomy, estimate=st.s_estimate, insert=st.s_insert, write=st.s_write),
                       estimate_gbp_s=st.bases / 1e9 / st.s_estimate, insert_gbp_s=st.bases / 1e9 / st.s_insert,
                       estimate=st.estimate, size=st.size, estimate_over_size=st.estimate / max(st.size, 1),
                       capacity=st.capacity, minimizers=st.minimizers, sequences=st.sequences,
                       library_write_s=lib_s)
            print(json.dumps(rec), flush=True)
            if out:
                out.write(json.dumps(rec) + "\n")
            shutil.rmtree(db)
        # the oracle on a 1/oracle_div subset, one process per core over disjoint shares
        sub = min(int(a.gbp * 1e9 / a.oracle_div), hap_len)
        cores = os.cpu_count() or 1
        share = -(-sub // cores)
        with mp.Pool(cores) as pool:
            secs = pool.map(oracle_share, [(plain[0], i * share, min(share, sub - i * share)) for i in range(cores)
                                           if i * share < sub])
        rec = dict(card=name, power_limit=power, form="oracle_cpu", gbp=sub / 1e9, processes=len(secs),
                   library_gbp_s=sub / 1e9 / max(secs), slowest_process_s=max(secs))
        print(json.dumps(rec), flush=True)
        if out:
            out.write(json.dumps(rec) + "\n")
    finally:
        shutil.rmtree(work, ignore_errors=True)


if __name__ == "__main__":
    main()
