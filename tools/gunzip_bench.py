#!/usr/bin/env python
"""GPU gzip decompression (nh_gunzip) against one zlib thread on the same files.  The inputs are about --gb of
seeded FASTQ laid out as the file pipeline reads it (synth.fastq_corpus: qualities all `I`, and uniformly random
Phred 2..41), each compressed as ONE ordinary gzip member at levels 1 and 6 (the `gzip` program), plus a
member-heavy file: the random-quality reads cut into members of --member-kib of input.  Prints one JSON line:

- kernel_gb_s: inflated bytes over the device time of the kernels (nh_bench_gunzip: CUDA events around the
  launches, input already on the device, no output copy), mean of --iters runs after a warm-up;
- host_gb_s: inflated bytes over the wall clock of nh_gunzip, host memory to host memory (reads into pinned
  staging, copies, kernels, copy back), best of --iters;
- zlib_gb_s: inflated bytes over the wall clock of zlib.decompress on one thread, best of --iters;
- device_seconds_per_phase: where the device time of the host-to-host run goes (CUDA events): finding block
  starts, the first decode of every chunk, repairs and spills, the 32 KiB history chain, markers + CRC32;
- sweep: host_gb_s of the level-1 constant-quality file over chunk and window sizes;
- the card's name and power limit, which belong with every number above.

    python tools/gunzip_bench.py [--gb 1.0] [--iters 3] [--device 0] [--sweep-mib 512]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card(device):
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(device), "--query-gpu=name,power.limit",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=60).stdout.strip()
        name, power = [x.strip() for x in q.split(",")]
        return name, power
    except Exception as e:  # the numbers stand without it, but say so
        return f"unknown ({e})", "unknown"


def gunzip_into(blob, out, device, chunk=0, window=0):
    """nh_debug_gunzip into a buffer of the known output size: (wall clock of the call, its counts)"""
    from nohuman_b200 import _ffi
    got = C.c_size_t()
    counts = (C.c_uint64 * len(_ffi.GUNZIP_COUNTS))()
    t0 = time.perf_counter()
    _ffi.check(_ffi.lib().nh_debug_gunzip(device, blob, len(blob), out.ctypes.data, len(out), C.byref(got), chunk, window,
                                          0, counts))
    dt = time.perf_counter() - t0
    assert got.value == len(out)
    return dt, dict(zip(_ffi.GUNZIP_COUNTS, counts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gb", type=float, default=1.0)
    ap.add_argument("--iters", type=int, default=3)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--member-kib", type=int, default=64)
    ap.add_argument("--sweep-mib", type=int, default=512, help="inflated size of the file the sweep runs on")
    ap.add_argument("--sweep-chunks", default="8,16,32,64", help="KiB")
    ap.add_argument("--sweep-windows", default="4,16,64", help="MiB")
    args = ap.parse_args()
    from nohuman_b200 import _ffi, synth
    from nohuman_b200.api import gunzip_kernel_seconds
    if _ffi.lib().nh_device_count() < 1:
        sys.exit("gunzip_bench needs a CUDA device")
    name, power = card(args.device)
    print(json.dumps({"card": name, "power_limit": power}), file=sys.stderr)
    n = int(args.gb * 1e9)
    d = tempfile.mkdtemp(prefix="nh_gunzip_bench_")
    plain = {"synthetic_reads": synth.fastq_corpus(n, seed=7), "random_phred_2_41": synth.fastq_corpus(n, seed=7, random_quals=True)}
    files, procs = {}, []
    for label, data in plain.items():
        p = os.path.join(d, label)
        with open(p, "wb") as f:
            f.write(data)
        for level in (1, 6):
            out = open(f"{p}.{level}.gz", "wb")
            procs.append((subprocess.Popen(["gzip", f"-{level}", "-c", p], stdout=out), out))
            files[f"{label}_gzip{level}"] = (f"{p}.{level}.gz", label)
    for pr, out in procs:
        assert pr.wait() == 0
        out.close()
    cut = args.member_kib << 10
    rq = plain["random_phred_2_41"]
    members = b"".join(zlib.compress(rq[i:i + cut], 6, wbits=31) for i in range(0, len(rq), cut))
    res = {"card": name, "power_limit": power, "inflated_bytes": n, "iters": args.iters, "files": {}}
    for label, (path, src) in list(files.items()) + [(f"random_phred_2_41_members_{args.member_kib}kib", (None, "random_phred_2_41"))]:
        blob = open(path, "rb").read() if path else members
        want = plain[src]
        out = np.empty(len(want), np.uint8)
        gunzip_into(blob, out, args.device)  # warm-up: module load, first allocations
        host, counts = min(gunzip_into(blob, out, args.device) for _ in range(args.iters))
        assert out.tobytes() == want
        kern = gunzip_kernel_seconds(blob, args.device, iters=args.iters)
        zl = []
        for _ in range(args.iters):
            t0 = time.perf_counter()
            z = zlib.decompressobj(31)
            got = z.decompress(blob)
            while z.unused_data:  # every member, as gzip -dc does
                rest = z.unused_data
                z = zlib.decompressobj(31)
                got += z.decompress(rest)
            zl.append(time.perf_counter() - t0)
        assert len(got) == len(want)
        res["files"][label] = {"compressed_bytes": len(blob), "kernel_seconds": round(kern, 4), "kernel_gb_s": round(n / kern / 1e9, 2),
                               "host_seconds": round(host, 4), "host_gb_s": round(n / host / 1e9, 3),
                               "zlib_seconds": round(min(zl), 4), "zlib_gb_s": round(n / min(zl) / 1e9, 3),
                               "host_vs_zlib": round(min(zl) / host, 2),
                               "device_seconds_per_phase": {k[3:]: round(v / 1e9, 4) for k, v in counts.items() if k.startswith("ns_")},
                               "windows": counts["windows"], "chunks": counts["chunks"], "repaired": counts["repaired"],
                               "overflowed": counts["overflowed"]}
        print(json.dumps({label: res["files"][label]}), file=sys.stderr)
    # chunk x window sweep on the level-1 constant-quality file
    sweep_n = min(n, args.sweep_mib << 20)
    blob = zlib.compress(plain["synthetic_reads"][:sweep_n], 1, wbits=31)
    out = np.empty(sweep_n, np.uint8)
    res["sweep"] = {"file": "synthetic_reads, zlib level 1", "inflated_bytes": sweep_n, "host_gb_s": {}}
    for ck in [int(x) for x in args.sweep_chunks.split(",")]:
        for wm in [int(x) for x in args.sweep_windows.split(",")]:
            t = min(gunzip_into(blob, out, args.device, ck << 10, wm << 20)[0] for _ in range(args.iters))
            res["sweep"]["host_gb_s"][f"chunk {ck} KiB, window {wm} MiB"] = round(sweep_n / t / 1e9, 3)
    import shutil
    shutil.rmtree(d, ignore_errors=True)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
