#!/usr/bin/env python
"""GPU BGZF compression (nh_bgzf_compress) against zlib level 6 on the same 0xff00-byte members, for two
seeded FASTQ corpora laid out as the file pipeline writes kept reads: the synthetic reads (qualities all
`I`) and the same reads with uniformly random Phred 2..41 qualities.  Prints one JSON line:

- kernel_gb_s: input bytes over device time of the three kernels for one batch already on the device
  (CUDA events, mean over launches that span at least --min-kernel-seconds);
- host_gb_s: input bytes over the wall clock of nh_bgzf_compress on --gb of input, host memory to host
  memory (staging into pinned memory, copies, kernels);
- ratio_vs_zlib6: GPU bytes / zlib level 6 bytes, both with BGZF framing, over --ratio-mib of input
  (zlib's side runs on one host thread);
- the card's name and power limit, which belong with every number above.

    python tools/gzip_bench.py [--gb 1.0] [--batch-mib 256] [--ratio-mib 64] [--device 0]
"""
import argparse
import json
import os
import subprocess
import sys
import time
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CUT = 0xFF00


def card(device):
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(device), "--query-gpu=name,power.limit",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=60).stdout.strip()
        name, power = [x.strip() for x in q.split(",")]
        return name, power
    except Exception as e:  # the numbers stand without it, but say so
        return f"unknown ({e})", "unknown"


def zlib6_bytes(data):
    n = 0
    for i in range(0, len(data), CUT):
        z = zlib.compressobj(6, zlib.DEFLATED, -15)
        n += len(z.compress(data[i:i + CUT]) + z.flush()) + 26
    return n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gb", type=float, default=1.0, help="input for the host-to-host timing")
    ap.add_argument("--batch-mib", type=int, default=256, help="input per launch for the kernel timing")
    ap.add_argument("--min-kernel-seconds", type=float, default=0.5)
    ap.add_argument("--ratio-mib", type=int, default=64)
    ap.add_argument("--device", type=int, default=0)
    args = ap.parse_args()
    from nohuman_b200 import _ffi
    from nohuman_b200 import synth
    from nohuman_b200.api import bgzf_compress, bgzf_kernel_seconds
    if _ffi.lib().nh_device_count() < 1:
        sys.exit("gzip_bench needs a CUDA device")
    name, power = card(args.device)
    n_host = int(args.gb * 1e9)
    res = {"card": name, "power_limit": power, "host_bytes": n_host, "kernel_batch_bytes": args.batch_mib << 20,
           "ratio_bytes": args.ratio_mib << 20, "corpora": {}}
    for label, rq in (("synthetic_reads", False), ("random_phred_2_41", True)):
        data = synth.fastq_corpus(n_host, seed=7, random_quals=rq)
        batch = data[:args.batch_mib << 20]
        one = bgzf_kernel_seconds(batch, args.device, iters=1)
        iters = max(3, int(args.min_kernel_seconds / max(one, 1e-6)) + 1)
        k_s = bgzf_kernel_seconds(batch, args.device, iters=iters)
        bgzf_compress(data[:64 << 20], args.device)  # warm-up: module load, first allocations
        t0 = time.perf_counter()
        out = bgzf_compress(data, args.device)
        h_s = time.perf_counter() - t0
        r = data[:args.ratio_mib << 20]
        gpu_r = len(bgzf_compress(r, args.device))
        zl_r = zlib6_bytes(r)
        res["corpora"][label] = {
            "kernel_seconds_per_batch": round(k_s, 6), "kernel_launches_timed": iters,
            "kernel_gb_s": round(len(batch) / k_s / 1e9, 2),
            "host_seconds": round(h_s, 3), "host_gb_s": round(n_host / h_s / 1e9, 3),
            "compressed_fraction": round(len(out) / n_host, 4),
            "gpu_bytes": gpu_r, "zlib6_bytes": zl_r, "ratio_vs_zlib6": round(gpu_r / zl_r, 4),
        }
        del data, out
    print(json.dumps(res))


if __name__ == "__main__":
    main()
