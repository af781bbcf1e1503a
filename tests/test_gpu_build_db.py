"""nh_build_db (kraken2-build --build on the GPU) against the oracle's sequential build of the same library:
the cfg1 genomes written as FASTA files (plain, gzip, bzip2; wrapped; lowercase, N and x runs; one record
without a map entry) with NCBI-style taxonomy dumps that include unmarked taxa."""
import glob
import os
import shutil
import subprocess

import numpy as np
import pytest

import build_inputs as bi
import synth

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "nohuman_b200", "bin")


def fmix64(x: np.ndarray) -> np.ndarray:
    x = x.astype(np.uint64)
    x ^= x >> np.uint64(33)
    x *= np.uint64(0xFF51AFD7ED558CCD)
    x ^= x >> np.uint64(33)
    x *= np.uint64(0xC4CEB9FE1A85EC53)
    x ^= x >> np.uint64(33)
    return x


@pytest.fixture(scope="module")
def lib(oracle, tmp_path_factory):
    d = str(tmp_path_factory.mktemp("build_lib"))
    genomes = synth.cfg1_genomes(seed=1, scale=1.0)
    files, mp, records = bi.write_library(os.path.join(d, "library"), genomes)
    nodes, names = bi.write_dmp(os.path.join(d, "taxonomy"))
    mk = bi.marked([t for t, _ in genomes])
    _, ts = bi.oracle_taxonomy(oracle, mk)
    mapped = [(t, s) for t, s in records if t is not None]
    odb = oracle.OracleDb.build(mapped, ts)
    odir = os.path.join(d, "oracle_db")
    odb.save(odir)
    parts = []
    for _, s in mapped:
        mins, amb = oracle.scan_positions(odb.opts, s)
        parts.append(np.unique(mins[amb == 0]))
    distinct = np.unique(np.concatenate(parts))
    return dict(dir=d, files=files, map=mp, nodes=nodes, names=names, genomes=genomes, odb=odb, odir=odir,
                distinct=distinct, records=records)


def build(lib, out, **kw):
    from nohuman_b200 import api
    return api.build_db(lib["files"], lib["nodes"], lib["names"], lib["map"], out, **kw)


@pytest.fixture(scope="module")
def built(lib, tmp_path_factory):
    out = str(tmp_path_factory.mktemp("gpu_db"))
    st = build(lib, out, capacity=int(lib["odb"].cht.capacity))
    return out, st


def header(path):
    return np.fromfile(os.path.join(path, "hash.k2d"), np.uint64, 4)


def test_seed_has_no_compacted_key_meeting(lib):
    """No two distinct library minimizers share a compacted key inside one run of occupied cells, so the
    table's content cannot depend on insertion order (linear probing fills the same cells in any order)."""
    cht = lib["odb"].cht
    cap, vb = int(cht.capacity), int(cht.value_bits)
    cells = lib["odb"].cells()
    assert int(cht.size) == len(lib["distinct"])
    occ = (cells & np.uint32((1 << vb) - 1)) != 0
    run = np.cumsum(~occ)
    if occ[0] and occ[-1]:  # the run that wraps around the end
        run[run == run[-1]] = run[0]
    h = fmix64(lib["distinct"])
    home = (h % np.uint64(cap)).astype(np.int64)
    ckey = h >> np.uint64(32 + vb)
    pairs = np.stack([ckey, run[home].astype(np.uint64)], axis=1)
    assert len(np.unique(pairs, axis=0)) == len(pairs)


def test_files_and_stats_match_the_oracle_build(lib, built):
    out, st = built
    assert open(os.path.join(out, "opts.k2d"), "rb").read() == open(os.path.join(lib["odir"], "opts.k2d"), "rb").read()
    assert open(os.path.join(out, "taxo.k2d"), "rb").read() == open(os.path.join(lib["odir"], "taxo.k2d"), "rb").read()
    assert list(header(out)) == list(header(lib["odir"]))
    assert st.skipped == 1
    assert st.sequences == sum(t is not None for t, _ in lib["records"])
    assert st.bases == sum(len(s) for t, s in lib["records"] if t is not None)
    assert st.size == lib["odb"].cht.size and st.capacity == lib["odb"].cht.capacity and st.estimate == 0
    assert not glob.glob(os.path.join(out, "*.tmp"))


def probe(db_dir, keys):
    from nohuman_b200 import Database, Session
    with Database.open(db_dir, 0) as db, Session(db, max_batch_bases=1 << 20) as s:
        return s.debug_probe(keys)


def absent_keys(lib, n=1_000_000):
    rng = np.random.default_rng(11)
    k = rng.integers(0, 2 ** 63, size=n, dtype=np.uint64) * np.uint64(2) + np.uint64(1)
    return k[~np.isin(k, lib["distinct"])]


def test_lookups_equal_the_oracle_table(lib, built):
    keys = np.concatenate([lib["distinct"], absent_keys(lib)])
    got = probe(built[0], keys)
    want = probe(lib["odir"], keys)
    assert np.array_equal(got, want)
    nd = len(lib["distinct"])
    assert (got[:nd] != 0).all()
    sample = np.random.default_rng(3).choice(nd, 20000, replace=False)
    assert [lib["odb"].get(int(lib["distinct"][i])) for i in sample] == got[sample].tolist()


def test_small_batches_split_records_and_give_the_same_lookups(lib, tmp_path):
    out = str(tmp_path / "db")
    st = build(lib, out, capacity=int(lib["odb"].cht.capacity), batch_bases=256 * 1024)
    assert st.size == lib["odb"].cht.size
    assert np.array_equal(probe(out, lib["distinct"]), probe(lib["odir"], lib["distinct"]))


def gpu_classify(db_dir, bases, offsets, paired, conf):
    from nohuman_b200 import Database, Session
    n_units = (len(offsets) - 1) // (2 if paired else 1)
    with Database.open(db_dir, 0) as db, Session(db, confidence=conf, paired=paired,
                                                 max_batch_bases=int(offsets[-1]) + 4096,
                                                 max_batch_seqs=len(offsets)) as s:
        call, _, _ = s.classify(bases, offsets)
        internal, tk, hg = s.debug_last_batch(n_units)
    return call, internal, tk, hg


@pytest.mark.parametrize("paired,conf", [(False, 0.0), (False, 0.5), (True, 0.0), (True, 0.5)])
def test_classification_on_the_gpu_built_db(lib, built, oracle, paired, conf):
    reads = synth.illumina_reads(lib["genomes"], 4000, paired=paired, seed=21 + paired)
    bases, offsets = synth.pack(reads)
    _, internal, tk, hg = gpu_classify(built[0], bases, offsets, paired, conf)
    odb = lib["odb"]
    odb.confidence = conf
    want = odb.classify_batch(bases, offsets, paired=paired)
    assert np.array_equal(internal, want["call"])
    assert np.array_equal(tk, want["total_kmers"])
    assert np.array_equal(hg, want["hit_groups"])
    gdb = oracle.OracleDb.load(built[0])  # the oracle reads the GPU-written table
    gdb.confidence = conf
    again = gdb.classify_batch(bases, offsets, paired=paired)
    for f in ("call", "total_kmers", "hit_groups"):
        assert np.array_equal(again[f], want[f]), f


def test_estimated_capacity(lib, tmp_path):
    a = build(lib, str(tmp_path / "a"))
    b = build(lib, str(tmp_path / "b"), batch_bases=1 << 20)
    n = len(lib["distinct"])
    assert abs(a.estimate - n) <= 0.1 * n, (a.estimate, n)
    # the sample is exact: the distinct minimizers whose hash has low bits 0..3, times 1024 / 4
    assert a.estimate == exact_estimate(lib)
    assert a.estimate_rescans == 0 and a.estimate_slots == 1 << 20  # the default set never grows here
    assert a.capacity == int(np.ceil((a.estimate + 8192) / 0.7))
    assert (a.estimate, a.capacity) == (b.estimate, b.capacity)
    assert list(header(str(tmp_path / "a")))[:1] == [a.capacity]


def exact_estimate(lib):
    """the capacity pass's estimate, computed from the library's distinct minimizers"""
    return int(((fmix64(lib["distinct"]) & np.uint64(1023)) < 4).sum()) * 256


@pytest.mark.parametrize("batch_bases", [0, 256 * 1024])
def test_estimate_set_growth_and_rescans(lib, tmp_path, monkeypatch, batch_bases):
    """A set started at 64 slots has to double about ten times: by scanning an overfilled batch again into a
    set twice the size, and (with many small batches) by doubling at half load between batches."""
    monkeypatch.setenv("NH_TEST_ESTIMATE_SLOTS", "64")
    st = build(lib, str(tmp_path / "db"), batch_bases=batch_bases)
    assert st.estimate == exact_estimate(lib)
    assert st.capacity == int(np.ceil((st.estimate + 8192) / 0.7))
    doublings = int(st.estimate_slots).bit_length() - 1 - 6
    assert st.estimate_slots >= 2 * st.estimate // 256
    assert st.estimate_rescans >= 1
    assert doublings > st.estimate_rescans  # at least one doubling at half load between or after batches
    if batch_bases:
        assert np.array_equal(probe(str(tmp_path / "db"), lib["distinct"][::7]),
                              probe(lib["odir"], lib["distinct"][::7]))


def test_failed_rename_removes_the_renamed_files(lib, tmp_path):
    """taxo.k2d is renamed last; a directory in its place makes that rename fail after the other two."""
    from nohuman_b200 import NhError
    from nohuman_b200._ffi import NH_ERR_IO
    out = tmp_path / "db"
    (out / "taxo.k2d").mkdir(parents=True)
    with pytest.raises(NhError) as ei:
        build(lib, str(out), capacity=int(lib["odb"].cht.capacity))
    assert ei.value.code == NH_ERR_IO and "cannot rename" in ei.value.message
    assert sorted(os.listdir(out)) == ["taxo.k2d"] and os.path.isdir(out / "taxo.k2d")


def test_truncated_gzip_is_an_io_error(lib, tmp_path):
    from nohuman_b200 import NhError
    from nohuman_b200._ffi import NH_ERR_IO
    gz = [f for f in lib["files"] if f.endswith(".gz")][0]
    data = open(gz, "rb").read()
    bad = str(tmp_path / "bad.fna.gz")
    open(bad, "wb").write(data[: len(data) // 2])
    files = [bad if f == gz else f for f in lib["files"]]
    out = str(tmp_path / "db")
    from nohuman_b200 import api
    with pytest.raises(NhError) as ei:
        api.build_db(files, lib["nodes"], lib["names"], lib["map"], out, capacity=int(lib["odb"].cht.capacity))
    assert ei.value.code == NH_ERR_IO
    assert not glob.glob(os.path.join(out, "*.k2d*"))


def test_too_small_capacity_is_table_full(lib, tmp_path):
    from nohuman_b200 import NhError
    from nohuman_b200._ffi import NH_ERR_CAPACITY
    out = str(tmp_path / "db")
    with pytest.raises(NhError) as ei:
        build(lib, out, capacity=100_000)
    assert ei.value.code == NH_ERR_CAPACITY and "table full" in ei.value.message
    assert not glob.glob(os.path.join(out, "*.k2d*"))


def test_kraken2_build_then_nohuman(lib, tmp_path):
    d = str(tmp_path / "db")
    os.makedirs(os.path.join(d, "library"))
    for f in lib["files"]:
        shutil.copy(f, os.path.join(d, "library"))
    shutil.copytree(os.path.join(lib["dir"], "taxonomy"), os.path.join(d, "taxonomy"))
    shutil.copy(lib["map"], os.path.join(d, "seqid2taxid.map"))
    r = subprocess.run([os.path.join(BIN, "kraken2-build"), "--build", "--db", d, "--threads", "4"],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert "Estimated" in r.stderr and "skipped" in r.stderr
    reads = synth.illumina_reads(lib["genomes"], 3000, seed=5)
    fq = str(tmp_path / "r.fq")
    synth.write_fastq(fq, reads)
    outs = []
    for db in (d, lib["odir"]):
        o = str(tmp_path / f"out_{len(outs)}.fq")
        r = subprocess.run([os.path.join(BIN, "nohuman"), "--db", db, "-t", "2", "-o", o, fq],
                           capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        outs.append(open(o, "rb").read())
    assert outs[0] == outs[1] and len(outs[0]) > 0
