#!/usr/bin/env python
"""GPU DUST masking (nh_dust_mask / nh_dust_fasta, the dustmasker shim) on a seeded library shaped like a human
pangenome: tools/build_db_bench.py's haplotypes (--gbp in all over --haplotypes records, --snp-rate
substitutions, runs of N), with microsatellites (units of 1-6 bases, 20-300 bases, 3 % substitutions) and
homopolymers spliced in at --lc-per-mbp sites per Mbp, as a FASTA file plain and `gzip -1`.  Prints one JSON
line per measurement, after the card's name and power limit:

- kernel: nh_bench_dust's device time of the kernels on --kernel-mbp of the library already on the device
  (more than the 126 MB L2), as Gbases/s;
- file: nh_dust_fasta host to host (FASTA out, to a file in the same temporary directory), plain and gzip,
  with the fraction of bases masked;
- oracle_cpu: the CPU restatement of sdust (tests/native/dust_oracle.c) on a 1/--oracle-div subset cut into 1 Mbp
  records, OpenMP over the records on every host core.

    python tools/dust_bench.py [--gbp 2] [--device 0] [--json out.jsonl]
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tools"), os.path.join(ROOT, "tests")]

import build_db_bench as bb  # noqa: E402
import dust_inputs as di  # noqa: E402
import dust_oracle  # noqa: E402


def write_library(path, gbp, n_hap, snp_rate, lc_per_mbp, seed):
    hap_len = int(gbp * 1e9 / n_hap)
    base = bb.ACGT[np.random.default_rng(seed).integers(0, 4, size=hap_len, dtype=np.uint8)]
    sample = None
    with open(path, "wb") as f:
        for i in range(n_hap):
            s = di.splice_low_complexity(np.random.default_rng(seed + 2000 + i),
                                         bb.haplotype(base, i, snp_rate, seed), per_mbp=lc_per_mbp)
            f.write(bb.fasta_bytes(f"hap{i:02d}", s))
            if sample is None:
                sample = s
    return sample


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gbp", type=float, default=2.0)
    ap.add_argument("--haplotypes", type=int, default=16)
    ap.add_argument("--snp-rate", type=float, default=0.001)
    ap.add_argument("--lc-per-mbp", type=int, default=200)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--kernel-mbp", type=int, default=100)
    ap.add_argument("--oracle-div", type=int, default=10)
    ap.add_argument("--json", default=None)
    ap.add_argument("--workdir", default=None, help="where the library is written (default: a temporary directory)")
    a = ap.parse_args()
    name, power = bb.card(a.device)
    out = open(a.json, "a") if a.json else None

    def emit(rec):
        rec = dict(card=name, power_limit=power, **rec)
        print(json.dumps(rec), flush=True)
        if out:
            out.write(json.dumps(rec) + "\n")

    emit(dict(gbp=a.gbp, haplotypes=a.haplotypes, lc_per_mbp=a.lc_per_mbp, host_cores=os.cpu_count()))
    from nohuman_b200 import api
    work = tempfile.mkdtemp(prefix="nh_dust_bench_", dir=a.workdir)
    try:
        plain = os.path.join(work, "lib.fna")
        t0 = time.perf_counter()
        sample = write_library(plain, a.gbp, a.haplotypes, a.snp_rate, a.lc_per_mbp, a.seed)
        gz = plain + ".gz"
        subprocess.check_call(f"gzip -1 -c '{plain}' > '{gz}'", shell=True)
        emit(dict(form="library", write_s=time.perf_counter() - t0, plain_bytes=os.path.getsize(plain),
                  gzip_bytes=os.path.getsize(gz)))

        n = min(len(sample), a.kernel_mbp * 1_000_000)
        recs = [sample[i:i + 1_000_000].tobytes() for i in range(0, n, 1_000_000)]
        secs = api.dust_kernel_seconds(recs, a.device, iters=5)
        emit(dict(form="kernel", gbases=n / 1e9, seconds=secs, kernel_gbases_s=n / 1e9 / secs))

        for form, src in (("plain", plain), ("gzip", gz)):
            dst = os.path.join(work, "masked.fna")
            t0 = time.perf_counter()
            st = api.dust_fasta(src, dst, fmt="fasta", threads=os.cpu_count() or 1, device=a.device)
            wall = time.perf_counter() - t0
            emit(dict(form=form, gbases=st.bases / 1e9, wall_s=wall, gbases_s=st.bases / 1e9 / wall,
                      masked_fraction=st.masked / max(st.bases, 1), intervals=st.intervals, sequences=st.sequences))
            os.unlink(dst)

        sub = sample[: min(len(sample), int(a.gbp * 1e9 / a.oracle_div))]
        offs = np.arange(0, len(sub) + 1, 1_000_000, dtype=np.uint64)
        if offs[-1] != len(sub):
            offs = np.append(offs, np.uint64(len(sub)))
        t0 = time.perf_counter()
        dust_oracle.dust_mask_batch(sub, offs)
        s = time.perf_counter() - t0
        emit(dict(form="oracle_cpu", gbases=len(sub) / 1e9, seconds=s, gbases_s=len(sub) / 1e9 / s,
                  threads=os.cpu_count()))
    finally:
        shutil.rmtree(work, ignore_errors=True)


if __name__ == "__main__":
    main()
