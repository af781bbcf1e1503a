#!/usr/bin/env python
"""GPU taxon counts (nh_bench_taxon_counts, behind nh_db_inspect and the kraken2-inspect shim) on tables filled on
the device from a seed: capacities of 2^31 and 2^33 cells (8 and 32 GiB), taxonomies of 30, 40 000 and 500 000
nodes (a root and its children; value_bits the smallest that holds them), load 0.7, and two value distributions:
95 % of the occupied cells in one taxon, and uniform.  The tables are torch tensors adopted by
Database.from_memory(cells_on_device=True) (built with NH_FILTER=0: no miss filter, which inspection does not use),
so nothing large is written to disk.  Prints one JSON line per measurement, after the card's name and power limit:

- kernel: the device time of one counting pass (CUDA events, mean of --iters after a warm-up) and the bytes it
  reads (4 x capacity) over that time, next to the 7.7 TB/s HBM3e data-sheet figure; the path the kernel took
  (shared-memory bins up to the opt-in shared-memory size / 4 nodes, global counters above); the counts are
  checked against a chunked torch.bincount on the device.  numpy_s is np.bincount over a host copy of the first
  --numpy-cells cells (bin 0 dropped, out-of-range values split off), timed on the host as the reference point.
- command: `kraken2-inspect --db DIR` on a --disk-cells table written to a temporary directory: its wall time, and
  the same work through the API split into nh_db_open and nh_db_inspect.

    python tools/inspect_bench.py [--device 0] [--iters 5] [--json out.jsonl]
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
sys.path[:0] = [ROOT, os.path.join(ROOT, "tools")]

import build_db_bench as bb  # noqa: E402

HBM_TB_S = 7.7  # HGX B200 data sheet, one GPU
CHUNK = 1 << 28


def value_bits(nodes):
    vb = 1
    while (1 << vb) < nodes:
        vb += 1
    return vb


def star_taxonomy(nodes):
    from nohuman_b200 import synth
    tax = [synth.TaxNode(1, 1, "root", "no rank")]
    tax += [synth.TaxNode(1000 + i, 1, f"taxon {i}", "species") for i in range(nodes - 2)]
    return synth.taxonomy_image(tax)[0]


def fill(t, cap, nodes, dist, seed):
    """cells = random key bits | value, 30 % empty; value 1 for 95 % of the occupied cells (skew95) or uniform"""
    import torch
    vb = value_bits(nodes)
    g = torch.Generator(device=t.device)
    g.manual_seed(seed)
    for s in range(0, cap, CHUNK):
        n = min(CHUNK, cap - s)
        v = torch.randint(1, nodes, (n,), device=t.device, generator=g)
        if dist == "skew95":
            v = torch.where(torch.rand(n, device=t.device, generator=g) < 0.95, torch.ones_like(v), v)
        c = (torch.randint(0, 1 << (32 - vb), (n,), device=t.device, generator=g) << vb) | v
        c[torch.rand(n, device=t.device, generator=g) < 0.3] = 0
        t[s:s + n] = torch.where(c >= 1 << 31, c - (1 << 32), c).to(torch.int32)
        del v, c
    t[cap:] = 0


def device_counts(t, cap, nodes):
    """(counts, occupied, out_of_range) by torch.bincount over chunks: the check, not the measurement"""
    import torch
    mask = (1 << value_bits(nodes)) - 1
    counts = torch.zeros(1 << value_bits(nodes), dtype=torch.int64, device=t.device)
    for s in range(0, cap, CHUNK):
        v = t[s:min(cap, s + CHUNK)].to(torch.int64) & mask
        counts += torch.bincount(v, minlength=mask + 1)
    c = counts.cpu().numpy()
    want = c[:nodes].copy()
    want[0] = 0  # empty cells and cells with value 0 are not counted
    return want, int(c[1:].sum()), int(c[nodes:].sum())


def numpy_seconds(t, cells, nodes):
    """np.bincount over a host copy of the first `cells` cells, chunk by chunk: host seconds (copies not timed)"""
    mask = np.uint32((1 << value_bits(nodes)) - 1)
    secs = 0.0
    for s in range(0, cells, CHUNK):
        h = t[s:min(cells, s + CHUNK)].cpu().numpy().view(np.uint32)
        t0 = time.perf_counter()
        v = h & mask
        occupied = np.count_nonzero(v)
        out_of_range = np.count_nonzero(v >= nodes)
        counts = np.bincount(v[v < nodes], minlength=nodes)
        counts[0] = 0
        secs += time.perf_counter() - t0
        del occupied, out_of_range, counts
    return secs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--capacities", default="31,33", help="log2 of the table capacities in cells")
    ap.add_argument("--nodes", default="30,40000,500000")
    ap.add_argument("--numpy-cells", type=int, default=1 << 31)
    ap.add_argument("--disk-cells", type=int, default=1 << 28)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    os.environ["NH_FILTER"] = "0"
    import torch
    from nohuman_b200 import Database, synth
    name, power = bb.card(a.device)
    out = open(a.json, "a") if a.json else None

    def emit(rec):
        rec = dict(card=name, power_limit=power, **rec)
        print(json.dumps(rec), flush=True)
        if out:
            out.write(json.dumps(rec) + "\n")
            out.flush()

    dev = torch.device("cuda", a.device)
    torch.cuda.set_device(dev)
    optin = torch.cuda.get_device_properties(dev).shared_memory_per_block_optin
    opts = synth.opts_image()
    taxo = {n: star_taxonomy(n) for n in (int(x) for x in a.nodes.split(","))}
    for lc in (int(x) for x in a.capacities.split(",")):
        cap = 1 << lc
        t = torch.empty((cap + 31) // 32 * 32, dtype=torch.int32, device=dev)
        for nodes in taxo:
            for dist in ("skew95", "uniform"):
                fill(t, cap, nodes, dist, a.seed + lc * 7 + nodes)
                want, occupied, oor = device_counts(t, cap, nodes)
                vb = value_bits(nodes)
                db = Database.from_memory(opts, taxo[nodes], [cap, occupied, 32 - vb, vb], t.data_ptr(), a.device,
                                          cells_on_device=True)
                try:
                    got, got_occ, got_oor = db.taxon_counts()
                    assert np.array_equal(got, want.astype(np.uint64)) and (got_occ, got_oor) == (occupied, oor)
                    secs = db.taxon_counts_kernel_seconds(a.iters)
                finally:
                    db.close()
                n_np = min(cap, a.numpy_cells)
                np_s = numpy_seconds(t, n_np, nodes)
                emit(dict(form="kernel", capacity=cap, nodes=nodes, dist=dist, value_bits=vb,
                          path="shared" if nodes <= optin // 4 else "global", occupied=occupied, iters=a.iters,
                          kernel_s=secs, bytes=4 * cap, gb_s=4 * cap / secs / 1e9, datasheet_tb_s=HBM_TB_S,
                          of_datasheet=4 * cap / secs / (HBM_TB_S * 1e12), numpy_cells=n_np, numpy_s=np_s,
                          numpy_gb_s=4 * n_np / np_s / 1e9))
        del t
        torch.cuda.empty_cache()

    # the whole command on a table on disk, as a user runs it (the miss filter is built on open)
    os.environ.pop("NH_FILTER", None)
    nodes, cap = 30, a.disk_cells
    work = tempfile.mkdtemp(prefix="nh_inspect_bench_")
    try:
        t = torch.empty((cap + 31) // 32 * 32, dtype=torch.int32, device=dev)
        fill(t, cap, nodes, "skew95", a.seed)
        _, occupied, _ = device_counts(t, cap, nodes)
        vb = value_bits(nodes)
        with open(os.path.join(work, "hash.k2d"), "wb") as f:
            f.write(np.array([cap, occupied, 32 - vb, vb], np.uint64).tobytes())
            t[:cap].cpu().numpy().tofile(f)
        del t
        torch.cuda.empty_cache()
        with open(os.path.join(work, "opts.k2d"), "wb") as f:
            f.write(opts)
        with open(os.path.join(work, "taxo.k2d"), "wb") as f:
            f.write(taxo[nodes])
        shim = os.path.join(ROOT, "nohuman_b200", "bin", "kraken2-inspect")
        t0 = time.perf_counter()
        r = subprocess.run([shim, "--db", work, "--gpu", str(a.device)], capture_output=True, text=True)
        wall = time.perf_counter() - t0
        assert r.returncode == 0, r.stderr
        t0 = time.perf_counter()
        db = Database.open(work, a.device)
        open_s = time.perf_counter() - t0
        t0 = time.perf_counter()
        db.inspect(os.path.join(work, "report.txt"))
        inspect_s = time.perf_counter() - t0
        db.close()
        emit(dict(form="command", capacity=cap, nodes=nodes, dist="skew95", file_bytes=32 + 4 * cap,
                  kraken2_inspect_wall_s=wall, report_lines=len(r.stdout.splitlines()), api_db_open_s=open_s,
                  api_inspect_s=inspect_s))
    finally:
        shutil.rmtree(work, ignore_errors=True)


if __name__ == "__main__":
    main()
