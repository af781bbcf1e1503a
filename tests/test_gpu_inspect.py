"""kraken2-inspect on the GPU: nh_db_taxon_counts against np.bincount over the hash.k2d cells, nh_db_inspect's
header and report against restatements of kraken2's, the damage checks, the `kraken2-inspect` shim after a
`kraken2-build --build`, and a real kraken2-inspect when one is on $PATH."""
import os
import shutil
import struct
import subprocess
import zlib

import numpy as np
import pytest

import build_inputs as bi
import synth
from test_gpu_files import py_report

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "nohuman_b200", "bin")
SHIM = os.path.join(BIN, "kraken2-inspect")


def nh_synth():
    from nohuman_b200 import synth as s
    return s


def numpy_counts(cells, value_bits, node_count):
    """np.bincount(cells & mask) with bin 0 dropped and the values >= node_count split off"""
    v = np.asarray(cells, np.uint32) & np.uint32((1 << value_bits) - 1)
    inside = v[v < node_count]
    counts = np.bincount(inside, minlength=node_count).astype(np.uint64)
    counts[0] = 0
    return counts, int(np.count_nonzero(v)), int(np.count_nonzero(v >= node_count))


def read_db(path):
    hdr = np.fromfile(os.path.join(path, "hash.k2d"), np.uint64, 4)
    cells = np.fromfile(os.path.join(path, "hash.k2d"), np.uint32, offset=32)
    return hdr, cells


def star_taxonomy(n_nodes):
    """root (taxid 1) with n_nodes - 2 species under it"""
    nodes = [nh_synth().TaxNode(1, 1, "root", "no rank")]
    nodes += [nh_synth().TaxNode(1000 + i, 1, f"taxon {i}", "species") for i in range(n_nodes - 2)]
    img, _ = nh_synth().taxonomy_image(nodes)
    return img


def crafted_db(cells, n_nodes, value_bits, min_hash=0):
    from nohuman_b200 import Database
    _, occupied, _ = numpy_counts(cells, value_bits, n_nodes)
    hdr = [len(cells), occupied, 32 - value_bits, value_bits]
    return Database.from_memory(nh_synth().opts_image(min_hash=min_hash), star_taxonomy(n_nodes), hdr, cells)


def random_cells(rng, capacity, value_bits, values, empty=0.3):
    keys = rng.integers(0, 1 << (32 - value_bits), capacity, dtype=np.uint64).astype(np.uint32) << np.uint32(value_bits)
    cells = keys | np.asarray(values, np.uint32)
    cells[rng.random(capacity) < empty] = 0
    return cells


def case_cells(name):
    """(cells, node_count, value_bits) of a crafted table"""
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    cap = 1 << 20
    if name == "one_taxon":
        return random_cells(rng, cap, 5, 7, empty=0), 23, 5
    if name == "uniform":
        return random_cells(rng, cap, 5, rng.integers(1, 23, cap)), 23, 5
    if name == "skewed":
        v = np.where(rng.random(cap) < 0.95, 3, rng.integers(1, 23, cap))
        return random_cells(rng, cap, 5, v), 23, 5
    if name == "key_bits_value_zero":
        c = random_cells(rng, cap, 12, rng.integers(1, 3000, cap))
        zero = rng.random(cap) < 0.4
        c[zero] = (rng.integers(1, 1 << 20, int(zero.sum()), dtype=np.uint64).astype(np.uint32) << np.uint32(12))
        return c, 3000, 12
    if name == "out_of_range":
        c = random_cells(rng, cap, 5, rng.integers(1, 23, cap))
        idx = rng.choice(cap, 1000, replace=False)
        c[idx] = (c[idx] & ~np.uint32(31)) | rng.integers(23, 32, 1000).astype(np.uint32)
        return c, 23, 5
    if name == "odd_capacity":
        cap = (1 << 20) + 13
        c = random_cells(rng, cap, 5, rng.integers(1, 23, cap))
        c[-13:] = np.arange(1, 14, dtype=np.uint32) | np.uint32(0xFFFFFFE0)
        return c, 23, 5
    if name == "value_bits_12":
        return random_cells(rng, cap, 12, rng.integers(1, 4096, cap)), 4096, 12
    if name == "two_nodes":
        return random_cells(rng, cap, 1, 1, empty=0.5), 2, 1
    if name == "150k_nodes":
        return random_cells(rng, cap, 18, rng.integers(1, 150_000, cap)), 150_000, 18
    raise KeyError(name)


CASES = ["one_taxon", "uniform", "skewed", "key_bits_value_zero", "out_of_range", "odd_capacity", "value_bits_12",
         "two_nodes", "150k_nodes"]


@pytest.mark.parametrize("path", ["default", "global"])
@pytest.mark.parametrize("name", CASES)
def test_crafted_counts(name, path, monkeypatch):
    if path == "global":
        monkeypatch.setenv("NH_TEST_INSPECT_SHARED_BINS", "1")
    cells, n_nodes, vb = case_cells(name)
    want = numpy_counts(cells, vb, n_nodes)
    with crafted_db(cells, n_nodes, vb) as db:
        counts, occ, oor = db.taxon_counts()
    assert np.array_equal(counts, want[0]) and (occ, oor) == want[1:]
    if name == "out_of_range":
        assert oor > 0
    if name == "one_taxon":
        assert counts[7] == len(cells) == occ


def test_23_nodes_with_8_shared_bins(monkeypatch):
    """a taxonomy above the (lowered) shared-memory bound takes the global path"""
    monkeypatch.setenv("NH_TEST_INSPECT_SHARED_BINS", "8")
    cells, n_nodes, vb = case_cells("skewed")
    with crafted_db(cells, n_nodes, vb) as db:
        got = db.taxon_counts()
    want = numpy_counts(cells, vb, n_nodes)
    assert np.array_equal(got[0], want[0]) and got[1:] == want[1:]


def test_small_db_counts(small_db, gpu_db):
    hdr, cells = read_db(small_db.path)
    counts, occ, oor = gpu_db.taxon_counts()
    want = numpy_counts(cells, int(hdr[3]), int(gpu_db.info.node_count))
    assert np.array_equal(counts, want[0]) and (occ, oor) == want[1:]
    assert occ == int(hdr[1]) and oor == 0
    assert gpu_db.taxon_counts_kernel_seconds(3) > 0


def test_past_2_32_cells():
    """taxon 1 in every cell of a 2^32 + 2^27 + 13-cell table, other values at 2^32 - 1, 2^32 and the last cell"""
    import torch
    from nohuman_b200 import Database
    free, _ = torch.cuda.mem_get_info(0)
    if free < 24 << 30:
        pytest.skip(f"needs 24 GiB of free device memory, {free >> 30} GiB free")
    cap = (1 << 32) + (1 << 27) + 13
    t = torch.zeros((cap + 31) // 32 * 32, dtype=torch.int32, device="cuda")
    t[:cap] = 1
    planted = {(1 << 32) - 1: 2, 1 << 32: 3, cap - 1: 4}
    for i, v in planted.items():
        t[i] = v
    torch.cuda.synchronize()
    hdr = [cap, cap, 27, 5]
    db = Database.from_memory(nh_synth().opts_image(), star_taxonomy(23), hdr, t.data_ptr(), cells_on_device=True)
    try:
        for path in ("default", "global"):
            if path == "global":
                os.environ["NH_TEST_INSPECT_SHARED_BINS"] = "1"
            try:
                counts, occ, oor = db.taxon_counts()
            finally:
                os.environ.pop("NH_TEST_INSPECT_SHARED_BINS", None)
            want = np.zeros(23, np.uint64)
            want[1] = cap - 3
            want[2:5] = 1
            assert np.array_equal(counts, want), path
            assert occ == cap and oor == 0 and int(counts[1]) > 1 << 32
    finally:
        db.close()
        del t
        torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------------------------
# the report

def header_lines(info):
    l = int(info.l)
    lines = [f"# Database options: nucleotide db, k = {int(info.k)}, l = {l}",
             "# Spaced mask = " + format(int(info.spaced_seed_mask), f"0{2 * l}b")[-2 * l:],
             "# Toggle mask = " + format(int(info.toggle_mask), "064b"),
             f"# Total taxonomy nodes: {int(info.node_count)}",
             f"# Table size: {int(info.size)}",
             f"# Table capacity: {int(info.capacity)}"]
    if int(info.minimum_acceptable_hash_value):
        lines.append(f"# Min clear hash value = {int(info.minimum_acceptable_hash_value)}")
    return "".join(s + "\n" for s in lines)


def py_report_zero(db, direct):
    """py_report with --report-zero-counts: the unclassified line and every node, zero counts too"""
    import ctypes as C
    par, ext = db.parents().tolist(), db.external_ids().tolist()
    n = len(par)
    names = [C.string_at(db.tax.name_data + db.tax.nodes[i].name_offset).decode() if i else "" for i in range(n)]
    ranks = [C.string_at(db.tax.rank_data + db.tax.nodes[i].rank_offset).decode() if i else "" for i in range(n)]
    clade = [int(x) for x in direct]
    for i in range(n - 1, 1, -1):
        clade[par[i]] += clade[i]
    total = clade[1]
    kids = [[] for _ in range(n)]
    for i in range(2, n):
        kids[par[i]].append(i)
    fmt = lambda cl, d, rk, tid, name, depth: "%6.2f\t%d\t%d\t%s\t%d\t%s%s\n" % (100.0 * cl / total, cl, d, rk, tid, "  " * depth, name)
    out = [fmt(0, 0, "U", 0, "unclassified", 0)]
    codes = {"superkingdom": "D", "kingdom": "K", "phylum": "P", "class": "C", "order": "O", "family": "F", "genus": "G", "species": "S"}

    def dfs(t, code, rdepth, depth):
        if ranks[t] in codes:
            code, rdepth = codes[ranks[t]], 0
        else:
            rdepth += 1
        out.append(fmt(clade[t], int(direct[t]), code + (str(rdepth) if rdepth else ""), ext[t], names[t], depth))
        for c in sorted(kids[t], key=lambda x: -clade[x]):
            dfs(c, code, rdepth, depth + 1)
    dfs(1, "R", -1, 0)
    return "".join(out)


@pytest.fixture(scope="module")
def small_counts(small_db):
    hdr, cells = read_db(small_db.path)
    return numpy_counts(cells, int(hdr[3]), len(small_db.parents()))[0]


def test_report_matches_restatement(small_db, gpu_db, small_counts, tmp_path):
    out = tmp_path / "inspect.txt"
    gpu_db.inspect(out)
    text = out.read_text()
    head = header_lines(gpu_db.info)
    assert text.startswith(head)
    body = text[len(head):]
    calls = np.repeat(np.arange(len(small_counts)), small_counts.astype(np.int64))
    assert body == py_report(small_db, calls, int(small_counts.sum()))
    root = [ln for ln in body.splitlines() if ln.split("\t")[3] == "R"]
    assert len(root) == 1 and int(root[0].split("\t")[1]) == int(gpu_db.info.size)
    assert not any(ln.split("\t")[3] == "U" for ln in body.splitlines())


def test_skip_counts_writes_the_header_only(gpu_db, tmp_path):
    out = tmp_path / "h.txt"
    gpu_db.inspect(out, skip_counts=True)
    assert out.read_text() == header_lines(gpu_db.info)


def test_zero_counts_lists_every_node(small_db, gpu_db, small_counts, tmp_path):
    out = tmp_path / "z.txt"
    gpu_db.inspect(out, zero_counts=True)
    body = out.read_text()[len(header_lines(gpu_db.info)):]
    assert body == py_report_zero(small_db, small_counts)
    assert len(body.splitlines()) == len(small_counts)  # every node but 0, and the unclassified line


def test_min_clear_hash_value_line(tmp_path):
    cells, n_nodes, vb = case_cells("uniform")
    with crafted_db(cells, n_nodes, vb, min_hash=1 << 60) as db:
        out = tmp_path / "m.txt"
        db.inspect(out, skip_counts=True)
        text = out.read_text()
        assert text == header_lines(db.info) and f"# Min clear hash value = {1 << 60}\n" in text


def test_shim_on_small_db(small_db, gpu_db, tmp_path):
    r = subprocess.run([SHIM, "--db", small_db.path, "--threads", "4", "--memory-mapping", "--gpu", "0"],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    out = tmp_path / "api.txt"
    gpu_db.inspect(out)
    assert r.stdout == out.read_text()


# ---------------------------------------------------------------------------------------------------------------
# damage

@pytest.fixture(params=["out_of_range", "size_off_by_one"])
def damaged(request, small_db, tmp_path):
    d = str(tmp_path / "db")
    shutil.copytree(small_db.path, d)
    hp = os.path.join(d, "hash.k2d")
    hdr, cells = read_db(d)
    vb, n_nodes = int(hdr[3]), len(small_db.parents())
    mask = np.uint32((1 << vb) - 1)
    if request.param == "out_of_range":
        occupied = np.flatnonzero(cells & mask)[[5, 500, -1]]
        cells[occupied] = (cells[occupied] & ~mask) | np.uint32(n_nodes)
        with open(hp, "r+b") as f:
            f.seek(32)
            f.write(cells.tobytes())
        msg = f"3 cells hold taxon ids >= node_count {n_nodes}"
    else:
        with open(hp, "r+b") as f:
            f.seek(8)
            f.write(struct.pack("<Q", int(hdr[1]) + 1))
        msg = f"occupied cells {int(hdr[1])} != header size {int(hdr[1]) + 1}"
    return d, cells, vb, n_nodes, msg


def test_damaged_table_is_reported(damaged, tmp_path):
    from nohuman_b200 import Database, NhError, _ffi
    d, cells, vb, n_nodes, msg = damaged
    r = subprocess.run([SHIM, "--db", d], capture_output=True, text=True)
    assert r.returncode == 1 and r.stdout == ""
    assert msg in r.stderr
    out = tmp_path / "never.txt"
    with Database.open(d, 0) as db:
        with pytest.raises(NhError) as ei:
            db.inspect(out)
        assert ei.value.code == _ffi.NH_ERR_IO and msg in ei.value.message
        assert not out.exists()
        counts, occ, oor = db.taxon_counts()
    want = numpy_counts(cells, vb, n_nodes)
    assert np.array_equal(counts, want[0]) and (occ, oor) == want[1:]


# ---------------------------------------------------------------------------------------------------------------
# end to end: kraken2-build --build, then kraken2-inspect

def ancestors(tid, parent):
    out = [tid]
    while tid != 1:
        tid = parent[tid]
        out.append(tid)
    return out


@pytest.fixture(scope="module")
def built_cfg1(tmp_path_factory):
    d = str(tmp_path_factory.mktemp("inspect_build"))
    genomes = synth.cfg1_genomes(seed=1, scale=1.0)
    files, mp, _ = bi.write_library(os.path.join(d, "library"), genomes)
    bi.write_dmp(os.path.join(d, "taxonomy"))
    shutil.move(mp, os.path.join(d, "seqid2taxid.map"))
    r = subprocess.run([os.path.join(BIN, "kraken2-build"), "--build", "--db", d, "--threads", "4"],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return d, [t for t, _ in genomes]


def test_build_then_inspect(built_cfg1):
    from nohuman_b200 import Database
    d, lib_taxa = built_cfg1
    r = subprocess.run([SHIM, "--db", d], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    lines = r.stdout.splitlines()
    head = [ln for ln in lines if ln.startswith("#")]
    body = [ln.split("\t") for ln in lines if not ln.startswith("#")]
    hdr, cells = read_db(d)
    assert f"# Table size: {int(hdr[1])}" in head and f"# Table capacity: {int(hdr[0])}" in head
    assert head[0] == "# Database options: nucleotide db, k = 35, l = 31"
    root = [f for f in body if f[3] == "R"]
    assert len(root) == 1 and int(root[0][1]) == int(hdr[1])
    parent = {t[0]: t[1] for t in synth.TAXONOMY_CFG1}
    allowed = set(lib_taxa)
    for a in lib_taxa:
        for b in lib_taxa:
            anc_a = ancestors(a, parent)
            allowed.add(next(t for t in ancestors(b, parent) if t in anc_a))
    direct = {int(f[4]) for f in body if int(f[2]) > 0}
    assert direct and direct <= allowed, direct - allowed
    assert set(lib_taxa) <= direct
    with Database.open(d, 0) as db:
        counts, occ, oor = db.taxon_counts()
    want = numpy_counts(cells, int(hdr[3]), len(counts))
    assert np.array_equal(counts, want[0]) and (occ, oor) == want[1:]
    assert sum(int(f[2]) for f in body) == occ == int(hdr[1])


# ---------------------------------------------------------------------------------------------------------------
# upstream

def real_kraken2_inspect():
    exe = shutil.which("kraken2-inspect")
    if not exe or os.path.realpath(os.path.dirname(exe)) == os.path.realpath(BIN):
        return None
    return exe


@pytest.mark.skipif(real_kraken2_inspect() is None, reason="no upstream kraken2-inspect on PATH (its output stays unpinned)")
def test_shim_matches_real_kraken2_inspect(small_db):
    outs = []
    for exe in (real_kraken2_inspect(), SHIM):
        r = subprocess.run([exe, "--db", small_db.path], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        outs.append(r.stdout)
    assert outs[0] == outs[1]
