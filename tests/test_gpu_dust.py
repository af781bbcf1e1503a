"""DUST masking on the GPU (nh_dust_mask, nh_dust_fasta, the dustmasker shim), byte for byte against the
CPU restatement of sdust (tests/native/dust_oracle.c), and a kraken2 database built from a library masked on
the GPU, against the oracle's build of the same library masked on the CPU."""
import bz2
import gzip
import os
import random
import shutil
import subprocess

import numpy as np
import pytest

import build_inputs as bi
import dust_inputs as di
import dust_oracle as do
import synth

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "nohuman_b200", "bin")
# a microsatellite spliced into the human genome of the end-to-end library.  Its period is over 5, so a read of it
# has several minimizers; a read of a dinucleotide or homopolymer run has one (every k-mer's window of l-mers
# spans all its phases), which is one hit group, and kraken2 never calls such a read with any database
REPEAT = b"TTAGGG" * 70


def gpu(seqs, window=64, level=20):
    from nohuman_b200 import api
    return api.dust_mask(seqs, window, level)


@pytest.fixture(scope="module")
def big():
    """cfg1 genomes with low-complexity stretches spliced in, cut into 1 Mbp records, plus seeded host-generator
    records and longer spliced random records: more than 50 Mbp in all"""
    rng = np.random.default_rng(5)
    recs = []
    for _, g in synth.cfg1_genomes(seed=1, scale=1.0):
        s = di.splice_low_complexity(rng, g, per_mbp=2000)
        recs += [bytes(s[i:i + 1_000_000]) for i in range(0, len(s), 1_000_000)]
    for i in range(36):
        s = di.splice_low_complexity(rng, synth.random_genome(rng, 1_000_000), per_mbp=1000)
        s[rng.integers(0, len(s), 2000)] = ord("N")
        recs.append(bytes(s))
    r = random.Random(7)
    recs += [di.gen(r, r.randint(3, 3000)) for _ in range(2000)]
    assert sum(map(len, recs)) > 50_000_000
    return recs


@pytest.mark.parametrize("window,level", [(64, 20), (33, 10), (16, 40), (64, 255), (4, 1)])
def test_large_inputs_equal_the_restatement(big, window, level):
    want = do.dust_mask(big, window, level)
    assert gpu(big, window, level) == want
    if (window, level) == (64, 20):
        frac = sum(c >= ord("a") for w in want[-2000:] for c in w) / sum(map(len, big[-2000:]))
        assert frac > 0.2


@pytest.mark.parametrize("chunk", ["64", "65", "127", "1000"])
def test_chunk_size_does_not_change_the_mask(monkeypatch, chunk):
    """small chunks put chunk borders inside repeats: every interval longer than a chunk straddles one"""
    r = random.Random(int(chunk))
    seqs = [di.gen(r, r.randint(3, 5000)) for _ in range(400)] + [b"ACGT" * 3000, b"A" * 700 + b"CAG" * 500]
    want = gpu(seqs)
    assert want == do.dust_mask(seqs)
    monkeypatch.setenv("NH_TEST_DUST_CHUNK", chunk)
    for w, t in ((64, 20), (20, 15)):
        assert gpu(seqs, w, t) == do.dust_mask(seqs, w, t)


def test_awkward_records():
    r = random.Random(3)
    seqs = [b"", b"A", b"AC", b"ACG", b"N" * 500, b"nnnn", b"", b"AAAAAAA", b"x" * 10 + b"aaaaaaa" + b"-" * 3]
    seqs += [di.gen(r, r.randint(0, 12)) for _ in range(100_000)]
    assert gpu(seqs) == do.dust_mask(seqs)
    assert gpu([]) == []


def test_out_of_range_parameters_are_refused():
    from nohuman_b200 import NhError
    from nohuman_b200._ffi import NH_ERR_INVALID
    for w, t in ((3, 20), (65, 20), (64, 0), (64, 256)):
        with pytest.raises(NhError) as ei:
            gpu([b"ACGT"], w, t)
        assert ei.value.code == NH_ERR_INVALID


def write_fasta(path, records, kind):
    body = b"".join(b">" + h + b"\n" + bi.wrap(s, 70) if s else b">" + h + b"\n" for h, s in records)
    if kind == "gz":
        body = gzip.compress(body)
    elif kind == "bz2":
        body = bz2.compress(body)
    elif kind == "bgzf":
        body = b"".join(bgzf_member(body[i:i + 0xff00]) for i in range(0, len(body), 0xff00)) + bgzf_member(b"")
    with open(path, "wb") as f:
        f.write(body)
    return path


def bgzf_member(data):
    import struct
    import zlib
    c = zlib.compressobj(6, zlib.DEFLATED, -15)
    cd = c.compress(data) + c.flush()
    hdr = b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff\x06\x00BC\x02\x00" + struct.pack("<H", len(cd) + 25)
    return hdr + cd + struct.pack("<II", zlib.crc32(data), len(data))


@pytest.fixture(scope="module")
def records():
    r = random.Random(11)
    rng = np.random.default_rng(11)
    recs = [(b"long one with a description\ttab", bytes(di.splice_low_complexity(rng, synth.random_genome(rng, 700_000),
                                                                               per_mbp=3000)))]
    recs += [(b"r%d" % i, di.gen(r, r.randint(0, 2000))) for i in range(300)]
    recs += [(b"empty", b""), (b"ns", b"N" * 100)]
    return recs


@pytest.mark.parametrize("kind", ["plain", "gz", "bgzf", "bz2"])
@pytest.mark.parametrize("fmt", ["fasta", "interval"])
def test_dust_fasta_equals_the_restatement(tmp_path, records, kind, fmt):
    from nohuman_b200 import api
    src = write_fasta(str(tmp_path / f"in.fa.{kind}"), records, kind)
    masked = do.dust_mask([s for _, s in records])
    want = di.render([(h, m) for (h, _), m in zip(records, masked)], fmt)
    out = str(tmp_path / "out.txt")
    st = api.dust_fasta(src, out, fmt=fmt, threads=4)
    assert open(out, "rb").read() == want
    assert st.sequences == len(records) and st.bases == sum(len(s) for _, s in records)
    assert st.masked == sum(c >= ord("a") for m in masked for c in m)
    assert st.intervals == sum(len(di.intervals(m)) for m in masked)


@pytest.mark.parametrize("fmt", ["fasta", "interval"])
def test_record_longer_than_a_batch(tmp_path, records, fmt):
    """64 KiB batches cut the 700 kbp record into pieces; the output equals the default batch's"""
    from nohuman_b200 import api
    src = write_fasta(str(tmp_path / "in.fa"), records, "plain")
    outs = []
    for bb in (0, 64 * 1024, 8192 + 63):
        out = str(tmp_path / f"out{bb}.txt")
        api.dust_fasta(src, out, fmt=fmt, batch_bases=bb)
        outs.append(open(out, "rb").read())
    masked = do.dust_mask([s for _, s in records])
    assert outs[0] == outs[1] == outs[2] == di.render([(h, m) for (h, _), m in zip(records, masked)], fmt)


def test_truncated_gzip_fails_and_leaves_no_output(tmp_path, records):
    from nohuman_b200 import NhError, api
    from nohuman_b200._ffi import NH_ERR_IO
    src = write_fasta(str(tmp_path / "in.fa.gz"), records, "gz")
    data = open(src, "rb").read()
    open(src, "wb").write(data[: len(data) // 2])
    out = tmp_path / "out.fa"
    with pytest.raises(NhError) as ei:
        api.dust_fasta(src, str(out))
    assert ei.value.code == NH_ERR_IO
    assert not out.exists()
    r = subprocess.run([os.path.join(BIN, "dustmasker"), "-in", src, "-out", str(out), "-outfmt", "fasta"],
                       capture_output=True, text=True)
    assert r.returncode != 0 and len(r.stderr.strip().splitlines()) == 1
    assert not out.exists()


def test_dustmasker_shim_default_is_interval_to_stdout(tmp_path, records):
    src = write_fasta(str(tmp_path / "in.fa"), records[:50], "plain")
    r = subprocess.run([os.path.join(BIN, "dustmasker"), "-in", src], capture_output=True)
    assert r.returncode == 0, r.stderr
    masked = do.dust_mask([s for _, s in records[:50]])
    assert r.stdout == di.render([(h, m) for (h, _), m in zip(records[:50], masked)], "interval")


# ---- end to end: mask a library the way kraken2-build --add-to-library does, then build on it ----

@pytest.fixture(scope="module")
def e2e(oracle, tmp_path_factory):
    d = str(tmp_path_factory.mktemp("dust_e2e"))
    rng = np.random.default_rng(9)
    genomes = []
    for i, (tid, g) in enumerate(synth.cfg1_genomes(seed=1, scale=0.2)):
        if i == 0:  # only the human genome carries microsatellites, among them the stretch the reads cover
            g = di.splice_low_complexity(rng, g, per_mbp=500)
            g[5000:5000 + len(REPEAT)] = np.frombuffer(REPEAT, np.uint8)
        genomes.append((tid, g))
    files, mp, recs = bi.write_library(os.path.join(d, "raw"), genomes)
    nodes, names = bi.write_dmp(os.path.join(d, "taxonomy"))
    _, ts = bi.oracle_taxonomy(oracle, bi.marked([t for t, _ in genomes]))
    mapped = [(t, s) for t, s in recs if t is not None]
    odb_raw = oracle.OracleDb.build(mapped, ts)
    masked = do.dust_mask([s for _, s in mapped])
    masked = [(t, bytes(c if c < ord("a") else ord("x") for c in m)) for (t, _), m in zip(mapped, masked)]
    odb = oracle.OracleDb.build(masked, ts)
    raw_dir, odir = os.path.join(d, "oracle_raw"), os.path.join(d, "oracle_masked")
    odb_raw.save(raw_dir)
    odb.save(odir)
    parts = [np.unique(m[a == 0]) for m, a in (oracle.scan_positions(odb.opts, s) for _, s in masked)]
    return dict(dir=d, files=files, map=mp, nodes=nodes, names=names, odb=odb, odir=odir, raw_dir=raw_dir,
                distinct=np.unique(np.concatenate(parts)))


@pytest.fixture(scope="module")
def masked_db(e2e):
    """dustmasker -in F -outfmt fasta | sed -e '/^>/!s/[a-z]/x/g' > DIR/library/F, then kraken2-build --build"""
    d = os.path.join(e2e["dir"], "db")
    os.makedirs(os.path.join(d, "library"))
    env = dict(os.environ, PATH=BIN + os.pathsep + os.environ.get("PATH", ""))
    for f in e2e["files"]:
        name = os.path.basename(f).replace(".gz", "").replace(".bz2", "")
        cmd = f"dustmasker -in '{f}' -outfmt fasta | sed -e '/^>/!s/[a-z]/x/g' > '{os.path.join(d, 'library', name)}'"
        r = subprocess.run(["bash", "-o", "pipefail", "-c", cmd], env=env, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
    shutil.copytree(os.path.join(e2e["dir"], "taxonomy"), os.path.join(d, "taxonomy"))
    shutil.copy(e2e["map"], os.path.join(d, "seqid2taxid.map"))
    r = subprocess.run(["kraken2-build", "--build", "--db", d, "--threads", "4"], env=env, capture_output=True,
                       text=True)
    assert r.returncode == 0, r.stderr
    return d


def probe(db_dir, keys):
    from nohuman_b200 import Database, Session
    with Database.open(db_dir, 0) as db, Session(db, max_batch_bases=1 << 20) as s:
        return s.debug_probe(keys)


def test_masked_build_equals_the_oracle_build(e2e, masked_db):
    for f in ("opts.k2d", "taxo.k2d"):
        assert open(os.path.join(masked_db, f), "rb").read() == open(os.path.join(e2e["odir"], f), "rb").read()
    h = np.fromfile(os.path.join(masked_db, "hash.k2d"), np.uint64, 4)
    want = np.fromfile(os.path.join(e2e["odir"], "hash.k2d"), np.uint64, 4)
    assert list(h[1:]) == list(want[1:])  # size, key and value bits; the capacity here is estimated
    rng = np.random.default_rng(12)
    absent = rng.integers(0, 2 ** 63, size=300_000, dtype=np.uint64) * np.uint64(2) + np.uint64(1)
    keys = np.concatenate([e2e["distinct"], absent[~np.isin(absent, e2e["distinct"])]])
    got = probe(masked_db, keys)
    assert np.array_equal(got, probe(e2e["odir"], keys))
    assert (got[:len(e2e["distinct"])] != 0).all()


def test_masked_microsatellite_reads_are_no_longer_human(masked_db, e2e):
    from nohuman_b200 import Database, Session
    reads = [REPEAT[i:i + 150] for i in range(0, len(REPEAT) - 150, 2)]
    bases, offsets = synth.pack([np.frombuffer(r, np.uint8) for r in reads])
    calls = []
    for d in (e2e["raw_dir"], masked_db):
        with Database.open(d, 0) as db, Session(db, max_batch_bases=1 << 20) as s:
            calls.append(s.classify(bases, offsets)[0])
    assert (calls[0] == 9606).all()
    assert (calls[1] == 0).all()
