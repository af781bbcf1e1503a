"""BGZF compression on the GPU (nh_bgzf_compress, Session(gpu_gzip=True), nohuman --gpu-gzip): every member
is a valid gzip member with the BGZF framing the zlib path writes, the same input gives the same bytes
whatever the batch, and the file pipeline writes the same records as with zlib."""
import gzip
import os
import struct
import subprocess
import zlib

import numpy as np
import pytest

import synth

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "nohuman_b200", "bin", "nohuman")
CUT = 0xFF00
MIB = 1 << 20
SIZES = [0, 1, 2, 3, 257, 258, 259, 65279, 65280, 65281, MIB, MIB + 1]
CONTENTS = ["zeros", "random", "fastq", "fastq_random_quals", "far_repeats"]


def content(kind, n, seed=0):
    from nohuman_b200 import synth as nhsynth
    rng = np.random.default_rng(seed + n)
    if kind == "zeros":
        return bytes(n)
    if kind == "random":
        return rng.integers(0, 256, n, dtype=np.uint8).tobytes()
    if kind == "fastq":
        return nhsynth.fastq_corpus(n, seed=seed)
    if kind == "fastq_random_quals":
        return nhsynth.fastq_corpus(n, seed=seed, random_quals=True)
    # text whose only long matches lie 32 767, 32 768 and 32 769 bytes back: the last one is out of reach
    a = np.frombuffer(b"abcdefghijklmnopqrstuvwxyz .,", np.uint8)[rng.integers(0, 29, n)].copy()
    for k, d in enumerate((32767, 32768, 32769)):
        lo = 1000 + 400 * k
        if lo + d + 300 <= n:
            a[lo + d:lo + d + 300] = a[lo:lo + 300]
    return a.tobytes()


def members(out):
    """(BSIZE, CRC, ISIZE, deflate stream) of each member, checking the BGZF header on the way."""
    got, at = [], 0
    while at < len(out):
        hdr = out[at:at + 18]
        assert hdr[:4] == b"\x1f\x8b\x08\x04" and hdr[10:16] == b"\x06\x00BC\x02\x00", hdr
        bsize = struct.unpack("<H", hdr[16:18])[0] + 1
        assert bsize <= 65536
        m = out[at:at + bsize]
        assert len(m) == bsize
        crc, isize = struct.unpack("<II", m[-8:])
        got.append((bsize, crc, isize, m[18:-8]))
        at += bsize
    return got


def check_framing(data, out, tmp_path=None):
    assert gzip.decompress(out) == data
    ms = members(out)
    assert [m[2] for m in ms] == [min(CUT, len(data) - i) for i in range(0, len(data), CUT)]
    for (bsize, crc, isize, stream), i in zip(ms, range(0, len(data), CUT)):
        piece = data[i:i + CUT]
        assert crc == zlib.crc32(piece)
        d = zlib.decompressobj(-15)
        assert d.decompress(stream) == piece
        assert d.eof and d.unused_data == b""  # the deflate stream ends exactly at the trailer
    if tmp_path is not None and data:
        p = tmp_path / "x.gz"
        p.write_bytes(out)
        subprocess.run(["gzip", "-t", str(p)], check=True)
    return ms


@pytest.mark.parametrize("kind", CONTENTS)
@pytest.mark.parametrize("size", SIZES)
def test_round_trip_and_framing(kind, size, tmp_path):
    from nohuman_b200.api import bgzf_compress
    data = content(kind, size)
    out = bgzf_compress(data)
    ms = check_framing(data, out, tmp_path)
    assert len(out) <= -(-size // CUT) * 65536
    if kind == "random":  # stored fallback: never larger than a stored block
        assert all(m[0] <= 65311 for m in ms)
        assert all(m[3][0] & 7 == 1 for m in ms if m[2] >= 64)  # BFINAL, BTYPE 0
    if kind in ("zeros", "fastq") and size >= 65280:
        assert ms[0][3][0] & 7 == 5  # BFINAL, BTYPE 2: dynamic Huffman codes


def test_matches_at_window_edge():
    """A repeat 32 768 bytes back is used; one 32 769 back cannot be."""
    from nohuman_b200.api import bgzf_compress
    rng = np.random.default_rng(5)
    a = rng.integers(0, 256, 65280, dtype=np.uint8)
    near, far = a.copy(), a.copy()
    near[40000:42000] = near[40000 - 32768:42000 - 32768]
    far[40000:42000] = far[40000 - 32769:42000 - 32769]
    sn, sf = bgzf_compress(near.tobytes()), bgzf_compress(far.tobytes())
    check_framing(near.tobytes(), sn)
    check_framing(far.tobytes(), sf)
    assert len(sf) == 18 + 5 + 65280 + 8  # stored: nothing to match within reach
    assert len(sn) < len(sf) - 1500


def test_deterministic_and_independent_of_batch():
    from nohuman_b200.api import bgzf_compress
    data = content("fastq_random_quals", 4 * MIB + 1, seed=3)
    out = bgzf_compress(data)
    assert bgzf_compress(data) == out
    # blocks of whole members one call each, and single members one call each, give the same bytes.
    # nh_bgzf_compress cuts members at multiples of 0xff00 of its input, so the blocks here are 16 members
    # long rather than 1 MiB; the pipeline's 1 MiB blocks, each ending in a short member and several to a
    # round, are compared across thread counts (and so across batch compositions) in test_run_files_gpu_gzip.
    blk = 16 * CUT
    assert b"".join(bgzf_compress(data[i:i + blk]) for i in range(0, len(data), blk)) == out
    ms = members(out)
    at = 0
    for k, m in enumerate(ms):
        if k % 7 == 0 or k == len(ms) - 1:
            assert bgzf_compress(data[k * CUT:(k + 1) * CUT]) == out[at:at + m[0]]
        at += m[0]


def test_second_gpu_gives_the_same_bytes():
    from nohuman_b200 import _ffi
    from nohuman_b200.api import bgzf_compress
    if _ffi.lib().nh_device_count() < 2:
        pytest.skip("needs two GPUs")
    data = content("fastq", 3 * MIB + 5, seed=9)
    assert bgzf_compress(data, device=1) == bgzf_compress(data, device=0)


@pytest.mark.parametrize("random_quals", [False, True])
def test_ratio_against_zlib_level_6(random_quals):
    from nohuman_b200 import synth as nhsynth
    from nohuman_b200.api import bgzf_compress
    data = nhsynth.fastq_corpus(64 * MIB, seed=11, random_quals=random_quals)
    gpu = len(bgzf_compress(data))
    host = 0
    for i in range(0, len(data), CUT):
        z = zlib.compressobj(6, zlib.DEFLATED, -15)
        host += len(z.compress(data[i:i + CUT]) + z.flush()) + 26
    ratio = gpu / host
    print(f"GPU members / zlib level 6 members ({'random' if random_quals else 'constant'} qualities): "
          f"{gpu} / {host} = {ratio:.4f}")
    assert ratio <= 1.10


# ---- the file pipeline -------------------------------------------------------------------------------


def fastq_text(seqs, prefix, suffix=""):
    rng = np.random.default_rng(len(seqs))
    out = bytearray()
    for i, s in enumerate(seqs):
        q = (rng.integers(2, 42, len(s)) + 33).astype(np.uint8).tobytes()
        out += f"@{prefix}{i}{suffix} len={len(s)}\n".encode() + bytes(s) + b"\n+\n" + q + b"\n"
    return bytes(out)


@pytest.fixture(scope="module")
def reads(small_db, tmp_path_factory):
    d = tmp_path_factory.mktemp("gzfq")
    se = synth.illumina_reads(small_db.genomes, 12000, 150, seed=51, n_rate=0.02)
    pe = synth.illumina_reads(small_db.genomes, 9000, 150, seed=52, paired=True)
    paths = {"se": str(d / "se.fq"), "m1": str(d / "p_1.fq.gz"), "m2": str(d / "p_2.fq.gz")}
    with open(paths["se"], "wb") as f:
        f.write(fastq_text(se, "r"))
    with open(paths["m1"], "wb") as f:
        f.write(gzip.compress(fastq_text(pe[0::2], "p", "/1")))
    with open(paths["m2"], "wb") as f:
        f.write(gzip.compress(fastq_text(pe[1::2], "p", "/2")))
    return paths


def run(gpu_db, reads, tmp_path, tag, paired, keep_human, threads, gpu_gzip):
    from nohuman_b200 import Session
    o1, o2 = str(tmp_path / f"{tag}_1.gz"), str(tmp_path / f"{tag}_2.gz")
    with Session(gpu_db, threads=threads, keep_human=keep_human, gpu_gzip=gpu_gzip) as s:
        if paired:
            st = s.run_files(reads["m1"], o1, reads["m2"], o2, out_format="g")
        else:
            st = s.run_files(reads["se"], o1, out_format="g")
    outs = [open(o1, "rb").read()] + ([open(o2, "rb").read()] if paired else [])
    return st, outs, [o1, o2] if paired else [o1]


@pytest.mark.parametrize("paired,keep_human", [(False, False), (True, False), (True, True)],
                         ids=["single", "paired", "paired-keep-human"])
def test_run_files_gpu_gzip(gpu_db, reads, tmp_path, paired, keep_human):
    from nohuman_b200.api import rewrite_files
    _, ref, _ = run(gpu_db, reads, tmp_path, "zlib", paired, keep_human, 8, False)
    st1, g1, paths = run(gpu_db, reads, tmp_path, "gpu1", paired, keep_human, 1, True)
    st8, g8, _ = run(gpu_db, reads, tmp_path, "gpu8", paired, keep_human, 8, True)
    assert st1.threads_compress == 1 and st8.threads_compress == 1
    assert g1 == g8  # the same bytes whatever -t is
    for z, g in zip(ref, g1):
        plain = gzip.decompress(g)
        assert plain == gzip.decompress(z)
        assert len(plain) > 100_000
        assert g.endswith(bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000"))
        # 1 MiB output blocks, each cut at 0xff00 bytes
        ms = members(g[:-28])
        cuts = [min(CUT, min(MIB, len(plain) - b) - i) for b in range(0, len(plain), MIB)
                for i in range(0, min(MIB, len(plain) - b), CUT)]
        assert [m[2] for m in ms] == cuts
        at = 0
        for bsize, crc, isize, stream in ms:
            piece = plain[at:at + isize]
            assert zlib.decompress(stream, -15) == piece and crc == zlib.crc32(piece)
            at += isize
    # read back by the parallel BGZF reader (threads > 1), every record kept as is
    n = gzip.decompress(g1[0]).count(b"\n") // 4
    back = [str(tmp_path / "back_1.fq"), str(tmp_path / "back_2.fq")]
    rewrite_files(np.ones(n, np.uint8), np.zeros(n, np.uint32), paths[0], back[0],
                  paths[1] if paired else None, back[1] if paired else None, out_format="u", tag_classified=False,
                  threads=8)
    for g, b in zip(g1, back):
        assert open(b, "rb").read() == gzip.decompress(g)


def test_run_files_multi_gpu_gzip(small_db, reads, tmp_path):
    from nohuman_b200 import Database, Session, _ffi
    from nohuman_b200.api import run_files_multi
    if _ffi.lib().nh_device_count() < 2:
        pytest.skip("needs two GPUs")
    dbs = Database.open_multi(small_db.path, [0, 1])
    try:
        outs = {}
        for k, ds in (("one", dbs[:1]), ("two", dbs)):
            sessions = [Session(d, threads=4, gpu_gzip=True) for d in ds]
            o1, o2 = str(tmp_path / f"{k}_1.gz"), str(tmp_path / f"{k}_2.gz")
            st = run_files_multi(sessions, reads["m1"], o1, reads["m2"], o2, out_format="g")
            assert st.threads_compress == len(ds)
            outs[k] = (open(o1, "rb").read(), open(o2, "rb").read())
            for s in sessions:
                s.close()
        assert outs["one"] == outs["two"]
    finally:
        for d in dbs:
            d.close()


def test_cli_gpu_gzip_paired(small_db, reads, tmp_path):
    got = {}
    for flag in ([], ["--gpu-gzip"]):
        o1, o2 = str(tmp_path / f"c{len(flag)}_1.gz"), str(tmp_path / f"c{len(flag)}_2.gz")
        r = subprocess.run([CLI, "--db", small_db.path, "-t", "4", "-F", "g", *flag, "-o", o1, "-O", o2,
                            reads["m1"], reads["m2"]], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        got[len(flag)] = (open(o1, "rb").read(), open(o2, "rb").read())
    assert got[0] != got[1]  # zlib and the GPU encoder choose different codes ...
    for z, g in zip(got[0], got[1]):
        assert gzip.decompress(g) == gzip.decompress(z)  # ... for the same records
