"""Host logic of the file API (reader -> ordered writer -> block compressor),
driven through the C ABI with caller-supplied decisions (nh_debug_rewrite_files),
so it runs without a GPU.  Expected bytes are written here from the kraken2
output rules (SURVEY.md A.6): header\\nseq\\n+\\nquals\\n, trailing whitespace
stripped, FASTA joined, classified records tagged " kraken:taxid|N"."""
import bz2
import gzip
import lzma
import os
import shutil
import subprocess

import numpy as np
import pytest

import synth
from nohuman_b200 import NhError
from nohuman_b200.api import rewrite_files


def make_records(n, seed, fasta=False, messy=False):
    rng = np.random.default_rng(seed)
    recs = []
    for i in range(n):
        L = int(rng.integers(1, 400))
        seq = bytes(synth.random_genome(rng, L))
        qual = bytes(rng.integers(33, 74, size=L, dtype=np.uint8))
        hdr = (b">" if fasta else b"@") + f"read{i} extra=words {i * 7}".encode()
        recs.append((hdr, seq, qual))
    return recs


def write_input(path, recs, fasta=False, messy=False, comp=None):
    out = bytearray()
    for i, (h, s, q) in enumerate(recs):
        if fasta:
            out += h + (b"  \r\n" if messy else b"\n")
            w = 60 if messy else max(1, len(s))
            for k in range(0, len(s), w):
                out += s[k:k + w] + b"\n"
        else:
            out += h + (b" \t\r\n" if messy and i % 3 == 0 else b"\n")
            out += s + (b"\r\n" if messy and i % 5 == 0 else b"\n")
            out += (b"+" + h[1:] if messy and i % 2 == 0 else b"+") + b"\n"
            out += q + b"\n"
    data = bytes(out)
    if comp == "gz":
        data = gzip.compress(data)
    elif comp == "bz2":
        data = bz2.compress(data)
    with open(path, "wb") as f:
        f.write(data)


def expected(recs, keep, call, fasta=False, tag=True):
    out = bytearray()
    for (h, s, q), k, c in zip(recs, keep, call):
        if not k:
            continue
        hh = h.rstrip()
        if c and tag:
            hh += b" kraken:taxid|%d" % c
        out += hh + b"\n" + s + b"\n"
        if not fasta:
            out += b"+\n" + q + b"\n"
    return bytes(out)


def read_output(path, fmt):
    raw = open(path, "rb").read()
    if fmt == "g":
        assert raw[:2] == b"\x1f\x8b"
        # gzip -dc reads concatenated members in one pass; gzip.decompress copies the rest of the input once per
        # member, which takes minutes on outputs of thousands of members
        return subprocess.run(["gzip", "-dc", str(path)], check=True, capture_output=True).stdout
    if fmt == "b":
        assert raw[:3] == b"BZh"
        return bz2.decompress(raw)
    if fmt == "x":
        assert raw[:6] == b"\xfd7zXZ\x00"
        return lzma.decompress(raw)
    if fmt == "z":
        assert raw[:4] == b"\x28\xb5\x2f\xfd"
        import ctypes as C
        z = C.CDLL("libzstd.so.1")
        z.ZSTD_decompressStream  # present
        # frame-by-frame with the simple API
        z.ZSTD_findFrameCompressedSize.restype = C.c_size_t
        z.ZSTD_findFrameCompressedSize.argtypes = [C.c_char_p, C.c_size_t]
        z.ZSTD_getFrameContentSize.restype = C.c_ulonglong
        z.ZSTD_getFrameContentSize.argtypes = [C.c_char_p, C.c_size_t]
        z.ZSTD_decompress.restype = C.c_size_t
        z.ZSTD_decompress.argtypes = [C.c_char_p, C.c_size_t, C.c_char_p, C.c_size_t]
        out, pos = bytearray(), 0
        while pos < len(raw):
            chunk = raw[pos:]
            n = z.ZSTD_findFrameCompressedSize(chunk, len(chunk))
            size = z.ZSTD_getFrameContentSize(chunk, n)
            buf = C.create_string_buffer(size)
            got = z.ZSTD_decompress(buf, size, chunk, n)
            assert got == size
            out += buf.raw[:size]
            pos += n
        return bytes(out)
    return raw


@pytest.mark.parametrize("fmt,n,threads", [
    *(pytest.param(fmt, 5000, 3, id=fmt) for fmt in ["u", "g", "b", "x", "z"]),
    # one compressor thread keeps the writer behind the classifier.  The writer stalls once the block writer
    # holds 64 blocks of 1 MiB (about 5 batches of 65536 records at half of them kept); the 19 batches here
    # are enough for 8 more to wait in the hand-off, so its window fills and must still keep the order
    pytest.param("g", 1_200_000, 1, id="g-slow-writer"),
])
def test_single_end_formats(tmp_path, fmt, n, threads):
    if fmt == "b" and not shutil.which("bzip2") or fmt == "x" and not shutil.which("xz"):
        pytest.skip("compressor CLI missing")
    recs = make_records(n, seed=1)
    rng = np.random.default_rng(2)
    keep = rng.integers(0, 2, size=len(recs), dtype=np.uint8)
    call = np.where(keep == 0, 9606, 0).astype(np.uint32)  # default mode: kept == unclassified
    inp, out = tmp_path / "in.fq", tmp_path / f"out.{fmt}"
    write_input(inp, recs)
    st = rewrite_files(keep, call, inp, out, out_format=fmt, threads=threads)
    assert (st.total, st.classified, st.unclassified) == (n, int((call != 0).sum()), int((call == 0).sum()))
    assert st.bases == sum(len(s) for _, s, _ in recs)
    assert read_output(out, fmt) == expected(recs, keep, call)


@pytest.mark.parametrize("comp", [None, "gz", "bz2"])
def test_paired_keep_human_tags_and_messy_input(tmp_path, comp):
    n = 70000  # more than one reader chunk (65536 records)
    r1, r2 = make_records(n, seed=3), make_records(n, seed=4)
    rng = np.random.default_rng(5)
    call = np.where(rng.random(n) < 0.5, 9606, 0).astype(np.uint32)
    call[::11] = np.where(call[::11] != 0, 131567, 0)
    keep = (call != 0).astype(np.uint8)  # -H: kept == classified
    ext = {None: "", "gz": ".gz", "bz2": ".bz2"}[comp]
    i1, i2 = tmp_path / f"a_1.fq{ext}", tmp_path / f"a_2.fq{ext}"
    write_input(i1, r1, messy=True, comp=comp)
    write_input(i2, r2, messy=True, comp=comp)
    o1, o2 = tmp_path / "o1.fq.gz", tmp_path / "o2.fq.gz"
    st = rewrite_files(keep, call, i1, o1, i2, o2, out_format="g", threads=4)
    assert st.total == n and st.classified == int(keep.sum())
    assert read_output(o1, "g") == expected(r1, keep, call)
    assert read_output(o2, "g") == expected(r2, keep, call)
    # the gzip output is multi-member (one member per block) and plain gunzip reads it
    assert subprocess.run(["gzip", "-t", str(o1)]).returncode == 0
    assert open(o1, "rb").read().count(b"\x1f\x8b\x08") >= 2


def test_fasta_multiline_is_joined(tmp_path):
    recs = make_records(300, seed=6, fasta=True)
    keep = np.ones(len(recs), np.uint8)
    call = np.zeros(len(recs), np.uint32)
    inp, out = tmp_path / "in.fa", tmp_path / "out.fq"
    write_input(inp, recs, fasta=True, messy=True)
    rewrite_files(keep, call, inp, out)
    assert open(out, "rb").read() == expected(recs, keep, call, fasta=True)


def test_paired_stops_at_shorter_file_and_empty_input(tmp_path):
    r1, r2 = make_records(100, seed=7), make_records(60, seed=8)
    i1, i2 = tmp_path / "x_1.fq", tmp_path / "x_2.fq"
    write_input(i1, r1)
    write_input(i2, r2)
    keep = np.ones(100, np.uint8)
    call = np.zeros(100, np.uint32)
    o1, o2 = tmp_path / "o1.fq", tmp_path / "o2.fq"
    st = rewrite_files(keep, call, i1, o1, i2, o2)
    assert st.total == 60
    assert open(o1, "rb").read() == expected(r1[:60], keep, call)
    assert open(o2, "rb").read() == expected(r2, keep, call)
    # empty input: zero records, empty output, no error
    e = tmp_path / "empty.fq"
    e.write_bytes(b"")
    st = rewrite_files(keep, call, e, tmp_path / "oe.fq")
    assert st.total == 0 and os.path.getsize(tmp_path / "oe.fq") == 0


def test_errors(tmp_path):
    keep, call = np.ones(4, np.uint8), np.zeros(4, np.uint32)
    with pytest.raises(NhError) as ei:
        rewrite_files(keep, call, tmp_path / "missing.fq", tmp_path / "o.fq")
    assert "cannot open" in ei.value.message
    bad = tmp_path / "bad.txt"
    bad.write_bytes(b"hello world\n")
    with pytest.raises(NhError) as ei:
        rewrite_files(keep, call, bad, tmp_path / "o.fq")
    assert "format not recognised" in ei.value.message
    xz = tmp_path / "in.fq.xz"
    xz.write_bytes(lzma.compress(b"@r\nACGT\n+\nIIII\n"))
    with pytest.raises(NhError) as ei:
        rewrite_files(keep, call, xz, tmp_path / "o.fq")
    assert "xz-compressed input is not supported" in ei.value.message
    ok = tmp_path / "ok.fq"
    ok.write_bytes(b"@r\nACGT\n+\nIIII\n")
    with pytest.raises(NhError):
        rewrite_files(keep, call, ok, tmp_path / "o.fq", out_format="q")


def test_unusual_but_valid_endings(tmp_path):
    """no trailing newline, blank line at the end, a record cut off in the middle: no hang, no crash;
    what was read completely is written (kraken2's reader stops at the first empty header line)"""
    keep, call = np.ones(8, np.uint8), np.zeros(8, np.uint32)
    a = tmp_path / "nonl.fq"
    a.write_bytes(b"@r1\nACGT\n+\nIIII\n@r2\nGGCC\n+\nJJJJ")  # no final newline
    st = rewrite_files(keep, call, a, tmp_path / "o1.fq")
    assert st.total == 2 and open(tmp_path / "o1.fq", "rb").read() == b"@r1\nACGT\n+\nIIII\n@r2\nGGCC\n+\nJJJJ\n"
    b = tmp_path / "blank.fq"
    b.write_bytes(b"@r1\nACGT\n+\nIIII\n\n\n")
    st = rewrite_files(keep, call, b, tmp_path / "o2.fq")
    assert st.total == 1
    c = tmp_path / "cut.fq"
    c.write_bytes(b"@r1\nACGT\n+\nIIII\n@r2\nGG")  # truncated second record: sequence only
    st = rewrite_files(keep, call, c, tmp_path / "o3.fq")
    assert st.total == 2  # kraken2 also hands the partial record on; its quality string is empty
    assert open(tmp_path / "o3.fq", "rb").read() == b"@r1\nACGT\n+\nIIII\n@r2\nGG\n+\n\n"
    d = tmp_path / "lower.fa"
    d.write_bytes(b">s1 desc\nacgtn\nACGT\n>s2\n\n>s3\nTT\n")
    st = rewrite_files(keep, call, d, tmp_path / "o4.fa")
    assert st.total == 3
    assert open(tmp_path / "o4.fa", "rb").read() == b">s1 desc\nacgtnACGT\n>s2\n\n>s3\nTT\n"


def test_gzip_output_is_bgzf_and_is_read_back_in_parallel(tmp_path):
    """gzip output = BGZF (members <= 64 KiB with a 'BC' size subfield + bgzip's EOF marker); such input
    (bgzip, bcl2fastq, our own output) is inflated by several threads and must give identical records"""
    check_bgzf_round_trip(tmp_path, 30000, write_threads=4)


def test_bgzf_round_trip_fills_the_reader_and_writer_windows(tmp_path):
    """The same with more than 64 MiB per file: the writer holds at most 64 blocks of 1 MiB and the parallel
    reader at most 64 tasks of 16 members, so both windows fill up and must still keep the order."""
    n = 170_000  # about 73 MB of FASTQ per file: more than 64 x 16 members, more than 64 blocks
    check_bgzf_round_trip(tmp_path, n, write_threads=8, min_members=64 * 16)


def check_bgzf_round_trip(tmp_path, n, write_threads, min_members=50):
    import struct
    import zlib
    r1, r2 = make_records(n, seed=11), make_records(n, seed=12)
    keep, call = np.ones(n, np.uint8), np.zeros(n, np.uint32)
    i1, i2 = tmp_path / "p_1.fq", tmp_path / "p_2.fq"
    write_input(i1, r1)
    write_input(i2, r2)
    g1, g2 = tmp_path / "g_1.fq.gz", tmp_path / "g_2.fq.gz"
    rewrite_files(keep, call, i1, g1, i2, g2, out_format="g", threads=write_threads)
    raw = open(g1, "rb").read()
    assert raw[:4] == b"\x1f\x8b\x08\x04" and raw[12:16] == b"BC\x02\x00"
    assert raw.endswith(bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000"))
    # walk the members by their announced sizes
    pos, members, total = 0, 0, 0
    while pos < len(raw):
        bsize = struct.unpack_from("<H", raw, pos + 16)[0] + 1
        isize = struct.unpack_from("<I", raw, pos + bsize - 4)[0]
        assert isize <= 0xFF00 and bsize <= 65536
        assert len(zlib.decompress(raw[pos + 18:pos + bsize - 8], wbits=-15)) == isize
        total += isize
        members += 1
        pos += bsize
    assert pos == len(raw) and members > min_members and total == len(expected(r1, keep, call))
    assert read_output(g1, "g") == expected(r1, keep, call)
    assert subprocess.run(["gzip", "-t", str(g1)]).returncode == 0
    # read it back with 8 threads (parallel member inflate) and with 1 (zlib's gzread): same bytes
    for threads in (8, 1):
        o1, o2 = tmp_path / f"back{threads}_1.fq", tmp_path / f"back{threads}_2.fq"
        st = rewrite_files(keep, call, g1, o1, g2, o2, out_format="u", threads=threads)
        assert st.total == n
        assert open(o1, "rb").read() == expected(r1, keep, call)
        assert open(o2, "rb").read() == expected(r2, keep, call)
    # a damaged member is an error, not silence
    bad = bytearray(raw)
    bad[len(bad) // 2] ^= 0x55
    b1 = tmp_path / "bad_1.fq.gz"
    b1.write_bytes(bytes(bad))
    with pytest.raises(NhError):
        rewrite_files(keep, call, b1, tmp_path / "x1.fq", g2, tmp_path / "x2.fq", threads=8)


def test_truncated_compressed_input_is_an_error(tmp_path):
    """A .fq.gz / .fq.bz2 / blocked .gz cut in the middle must fail the run (zlib's gzread hands back the
    bytes it has and only sets Z_BUF_ERROR; kraken2 + the reference would silently drop the rest)."""
    n = 20000
    recs = make_records(n, seed=21)
    keep, call = np.ones(n, np.uint8), np.zeros(n, np.uint32)
    plain = tmp_path / "t.fq"
    write_input(plain, recs)
    raw = open(plain, "rb").read()
    for name, data in (("t.fq.gz", gzip.compress(raw)), ("t.fq.bz2", bz2.compress(raw))):
        whole = tmp_path / name
        whole.write_bytes(data)
        st = rewrite_files(keep, call, whole, tmp_path / "ok.fq", threads=4)
        assert st.total == n
        cut = tmp_path / ("cut_" + name)
        cut.write_bytes(data[:len(data) // 2])
        with pytest.raises(NhError) as ei:
            rewrite_files(keep, call, cut, tmp_path / "o.fq", threads=4)
        assert "truncated or corrupt" in ei.value.message
    # blocked gzip, cut inside a member and between members
    bg = tmp_path / "t.bgz.gz"
    rewrite_files(keep, call, plain, bg, out_format="g", threads=4)
    data = open(bg, "rb").read()
    cut = tmp_path / "cut.bgz.gz"
    cut.write_bytes(data[:len(data) // 2])
    with pytest.raises(NhError):
        rewrite_files(keep, call, cut, tmp_path / "o.fq", threads=4)
    # a gzip stream with trailing garbage after a complete member is read like gzread reads it
    tg = tmp_path / "garbage.fq.gz"
    tg.write_bytes(gzip.compress(raw) + b"\x00" * 100)
    assert rewrite_files(keep, call, tg, tmp_path / "o2.fq", threads=1).total == n
    # concatenated members (cat a.gz b.gz)
    half = raw.index(b"\n@read10000 ") + 1
    cat = tmp_path / "cat.fq.gz"
    cat.write_bytes(gzip.compress(raw[:half]) + gzip.compress(raw[half:]))
    assert rewrite_files(keep, call, cat, tmp_path / "o3.fq", threads=1).total == n
    assert open(tmp_path / "o3.fq", "rb").read() == expected(recs, keep, call)


def test_blocked_gzip_followed_by_plain_members(tmp_path):
    """`cat blocked.gz plain.gz`: the first member selects the parallel reader, later members have no BC
    subfield; zlib and kraken2 read such a file, so must we.  A member announcing more than 64 KiB is refused."""
    import struct
    n = 6000
    recs = make_records(n, seed=22)
    keep, call = np.ones(n, np.uint8), np.zeros(n, np.uint32)
    plain = tmp_path / "m.fq"
    write_input(plain, recs)
    raw = open(plain, "rb").read()
    half = raw.index(b"\n@read3000 ") + 1
    (tmp_path / "h1.fq").write_bytes(raw[:half])
    rewrite_files(keep, call, tmp_path / "h1.fq", tmp_path / "h1.gz", out_format="g", threads=2)
    blocked = open(tmp_path / "h1.gz", "rb").read()
    blocked = blocked[:-28]  # without bgzip's empty end marker
    mixed = tmp_path / "mixed.fq.gz"
    mixed.write_bytes(blocked + gzip.compress(raw[half:]))
    st = rewrite_files(keep, call, mixed, tmp_path / "o.fq", threads=4)
    assert st.total == n and open(tmp_path / "o.fq", "rb").read() == expected(recs, keep, call)
    # forged ISIZE: a member that claims 1 GiB
    forged = bytearray(blocked)
    bsize = struct.unpack_from("<H", forged, 16)[0] + 1
    struct.pack_into("<I", forged, bsize - 4, 1 << 30)
    bad = tmp_path / "forged.fq.gz"
    bad.write_bytes(bytes(forged))
    with pytest.raises(NhError):
        rewrite_files(keep, call, bad, tmp_path / "o2.fq", threads=4)


def test_codec_parameters_follow_the_reference(tmp_path):
    """src/compression.rs:203-212 bzip2 level default (6), :256-268 zstd frames carry the content checksum."""
    n = 3000
    recs = make_records(n, seed=23)
    keep, call = np.ones(n, np.uint8), np.zeros(n, np.uint32)
    inp = tmp_path / "c.fq"
    write_input(inp, recs)
    if shutil.which("bzip2"):
        rewrite_files(keep, call, inp, tmp_path / "o.bz2", out_format="b")
        assert open(tmp_path / "o.bz2", "rb").read(4) == b"BZh6"
    rewrite_files(keep, call, inp, tmp_path / "o.zst", out_format="z", threads=2)
    raw = open(tmp_path / "o.zst", "rb").read()
    assert raw[:4] == b"\x28\xb5\x2f\xfd"
    assert raw[4] & 0x04, "Content_Checksum_flag of the frame header descriptor"
    assert read_output(tmp_path / "o.zst", "z") == expected(recs, keep, call)


def test_long_reads_cut_chunks_by_bases_and_mates_stay_together(tmp_path):
    """Chunks end after 65536 records OR ~48 Mbp of the first file; the second file follows the first
    file's cuts, so pairs stay aligned when the mates' lengths differ wildly."""
    rng = np.random.default_rng(24)
    n = 130
    r1, r2 = [], []
    for i in range(n):
        L1 = int(rng.integers(400_000, 1_200_000))  # ~100 Mbp in total: several chunks
        L2 = int(rng.integers(1, 300))
        s1 = bytes(synth.random_genome(rng, L1))
        s2 = bytes(synth.random_genome(rng, L2))
        r1.append((f"@long{i}/1".encode(), s1, b"I" * L1))
        r2.append((f"@long{i}/2".encode(), s2, b"J" * L2))
    i1, i2 = tmp_path / "l_1.fq", tmp_path / "l_2.fq"
    write_input(i1, r1)
    write_input(i2, r2)
    keep = (np.arange(n) % 3 != 0).astype(np.uint8)
    call = np.where(keep == 0, 9606, 0).astype(np.uint32)
    o1, o2 = tmp_path / "o_1.fq", tmp_path / "o_2.fq"
    st = rewrite_files(keep, call, i1, o1, i2, o2, threads=2)
    assert st.total == n
    assert open(o1, "rb").read() == expected(r1, keep, call)
    assert open(o2, "rb").read() == expected(r2, keep, call)


def test_pack_reads_matches_the_scalar_definition():
    """nh_pack_reads (host, AVX2 when available): 2-bit codes with the first base in the top bits, validity bits LSB
    first, every sequence on a unit of 32 bases, padding invalid; the same for 1 and many threads."""
    from nohuman_b200.api import pack_reads, packed_units
    rng = np.random.default_rng(1)
    lens = np.concatenate([rng.integers(0, 300, size=3000), [0, 1, 31, 32, 33, 64, 4097]])
    off = np.zeros(len(lens) + 1, np.uint64)
    off[1:] = np.cumsum(lens)
    alpha = np.frombuffer(b"ACGTacgtNnRY\x00-", np.uint8)
    p = np.array([.2, .2, .2, .2, .03, .03, .03, .03, .02, .01, .01, .01, .005, .005])
    bases = alpha[rng.choice(len(alpha), size=int(off[-1]), p=p / p.sum())]
    code_of = np.full(256, 255, np.uint8)
    for i, ch in enumerate(b"ACGT"):
        code_of[ch] = code_of[ch | 0x20] = i
    units = (lens + 31) // 32
    want_poff = np.zeros(len(lens) + 1, np.uint32)
    want_poff[1:] = np.cumsum(units)
    assert packed_units(off) == int(units.sum())
    ref = None
    for thr in (1, 5):
        codes, valid, poff = pack_reads(bases, off, thr)
        np.testing.assert_array_equal(poff, want_poff)
        # unpack everything back to per-base (code, valid) and compare with the definition
        nu = int(units.sum())
        c4 = codes[:nu * 8]
        per_base_code = np.stack([(c4 >> 6) & 3, (c4 >> 4) & 3, (c4 >> 2) & 3, c4 & 3], axis=1).reshape(-1)
        per_base_valid = ((valid[:nu, None] >> np.arange(32, dtype=np.uint32)[None, :]) & 1).reshape(-1).astype(bool)
        for s in (0, 1, 17, 2999, len(lens) - 1, len(lens) - 3):
            pass
        pos = np.concatenate([np.arange(int(want_poff[s]) * 32, int(want_poff[s]) * 32 + int(lens[s])) for s in range(len(lens))])
        want_code = code_of[bases]
        ok = want_code != 255
        np.testing.assert_array_equal(per_base_valid[pos], ok)
        np.testing.assert_array_equal(per_base_code[pos][ok], want_code[ok])
        inside = np.zeros(nu * 32, bool)
        inside[pos] = True
        assert not per_base_valid[~inside].any()  # padding is invalid
        if ref is None:
            ref = (codes.copy(), valid.copy())
        else:
            np.testing.assert_array_equal(codes, ref[0])
            np.testing.assert_array_equal(valid, ref[1])
