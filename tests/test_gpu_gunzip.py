"""GPU gzip decompression (nh_gunzip / nh_debug_gunzip): every output byte equal to what zlib gives, over
contents, writers, sizes, member layouts, chunk and window sizes, window ends at every byte of block headers and
codes, the repair and overflow paths, and every error zlib reports."""
import gzip
import random
import struct
import subprocess
import zlib

import pytest

pytestmark = pytest.mark.gpu

C_SMALL = 4096      # chunk bytes for the tests: many chunks per window at small sizes
W_SMALL = 1 << 16   # window bytes


def need_gpu():
    from nohuman_b200 import _ffi
    if _ffi.lib().nh_device_count() < 1:
        pytest.skip("no CUDA device")


@pytest.fixture(autouse=True)
def _gpu():
    need_gpu()


def ref(data):
    """what gzip -dc / gzread give: every member, trailing non-member bytes ignored"""
    out, d = [], data
    while d and d[0] == 0x1F:
        z = zlib.decompressobj(31)
        out.append(z.decompress(d))
        if not z.eof:
            raise ValueError("truncated")
        d = z.unused_data
    return b"".join(out)


def gz(data, level=6, strategy=zlib.Z_DEFAULT_STRATEGY, flushes=(), flush=zlib.Z_SYNC_FLUSH):
    c = zlib.compressobj(level, zlib.DEFLATED, 31, 8, strategy)
    parts, at = [], 0
    for f in sorted(flushes):
        parts.append(c.compress(data[at:f]))
        parts.append(c.flush(flush))
        at = f
    parts.append(c.compress(data[at:]))
    parts.append(c.flush())
    return b"".join(parts)


def inflate(blob, chunk=C_SMALL, window=W_SMALL, flags=0):
    from nohuman_b200.api import debug_gunzip
    return debug_gunzip(blob, chunk=chunk, window=window, flags=flags)


def check(blob, expect=None, **kw):
    got, counts = inflate(blob, **kw)
    want = ref(blob) if expect is None else expect
    assert len(got) == len(want)
    assert got == want
    return counts


def fastq(n_bytes, qualities="random", seed=1):
    from nohuman_b200.synth import fastq_corpus
    return fastq_corpus(n_bytes, seed=seed, random_quals=qualities == "random")


@pytest.fixture(scope="module")
def corpora():
    rng = random.Random(7)
    return {
        "fastq_const": fastq(1_000_000, "constant"),
        "fastq_random": fastq(1_000_000, "random"),
        "random": rng.randbytes(300_000),
        "zeros": bytes(3_000_000),
    }


@pytest.mark.parametrize("kind", ["fastq_const", "fastq_random", "random"])
@pytest.mark.parametrize("level", [1, 6, 9])
def test_contents_and_levels(corpora, kind, level):
    check(gzip.compress(corpora[kind], level))


def test_zeros_take_the_overflow_path(corpora):
    counts = check(gzip.compress(corpora["zeros"]))
    assert counts["overflowed"] > 0


@pytest.mark.parametrize("period", [32767, 32768, 32769])
def test_repeats_at_the_window_distance(period):
    rng = random.Random(period)
    unit = rng.randbytes(period)
    data = unit * 6 + unit[: period // 3]
    for chunk, window in ((C_SMALL, W_SMALL), (8192, 3 * 8192), (32768, 1 << 20)):
        check(gzip.compress(data, 6), chunk=chunk, window=window)


@pytest.mark.parametrize("strategy", [zlib.Z_FIXED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE, zlib.Z_FILTERED])
def test_zlib_strategies(corpora, strategy):
    check(gz(corpora["fastq_random"][:200_000], 6, strategy))


@pytest.mark.parametrize("flush", [zlib.Z_SYNC_FLUSH, zlib.Z_FULL_FLUSH])
def test_flush_points(corpora, flush):
    data = corpora["fastq_const"][:150_000]
    pts = list(range(1, len(data), 9973)) + [4096, 4097, 65536]
    check(gz(data, 6, flushes=pts, flush=flush))


def test_gzip_cli_level1(corpora, tmp_path):
    p = tmp_path / "x"
    p.write_bytes(corpora["fastq_random"])
    r = subprocess.run(["gzip", "-1", "-c", str(p)], capture_output=True)
    if r.returncode != 0:
        pytest.skip("no gzip program")
    check(r.stdout)


@pytest.mark.parametrize("size", [0, 1, C_SMALL - 1, C_SMALL, C_SMALL + 1, 5 * W_SMALL + 17])
def test_sizes(corpora, size):
    data = (corpora["fastq_random"] * 4)[:size]
    for level in (1, 6):
        check(gzip.compress(data, level))


def test_repair_path_gives_the_same_bytes(corpora):
    blob = gzip.compress(corpora["fastq_random"], 6)
    a, ca = inflate(blob)
    b, cb = inflate(blob, flags=1)
    assert a == b == ref(blob)
    assert cb["repaired"] > 0 and cb["repaired"] >= ca["repaired"]


def test_chunk_and_window_sizes_agree(corpora):
    blob = gzip.compress(corpora["fastq_const"] + corpora["random"][:50_000] + corpora["fastq_random"], 1)
    want = ref(blob)
    for chunk, window in ((2048, 1 << 17), (C_SMALL, W_SMALL), (16384, 1 << 18), (0, 0)):
        got, counts = inflate(blob, chunk=chunk, window=window)
        assert got == want, (chunk, window)
    assert inflate(blob)[0] == inflate(blob)[0]


def test_default_entry_point(corpora):
    from nohuman_b200.api import gunzip
    blob = gzip.compress(corpora["fastq_const"])
    assert gunzip(blob) == corpora["fastq_const"]


# ---- members ----

def member(data, level=6, mtime=0, name=None, comment=None, extra=None, hcrc=False):
    flg = (4 if extra is not None else 0) | (8 if name else 0) | (16 if comment else 0) | (2 if hcrc else 0)
    h = bytearray(b"\x1f\x8b\x08" + bytes([flg]) + struct.pack("<I", mtime) + b"\x00\x03")
    if extra is not None:
        h += struct.pack("<H", len(extra)) + extra
    if name:
        h += name + b"\x00"
    if comment:
        h += comment + b"\x00"
    if hcrc:
        h += struct.pack("<H", zlib.crc32(bytes(h)) & 0xFFFF)
    c = zlib.compressobj(level, zlib.DEFLATED, -15)
    body = c.compress(data) + c.flush()
    return bytes(h) + body + struct.pack("<II", zlib.crc32(data), len(data) & 0xFFFFFFFF)


def test_two_members(corpora):
    a, b = corpora["fastq_const"][:70_000], corpora["fastq_random"][:90_000]
    counts = check(member(a) + member(b), a + b)
    assert counts["members"] == 2


def test_many_tiny_members():
    rng = random.Random(3)
    parts = [rng.randbytes(rng.randrange(0, 40)) for _ in range(1000)]
    counts = check(b"".join(member(p) for p in parts), b"".join(parts))
    assert counts["members"] == 1000


def test_header_fields_and_empty_member(corpora):
    d = corpora["fastq_random"][:40_000]
    blob = (member(d[:10_000], extra=b"AB\x02\x00xy", name=b"reads.fq", comment=b"a comment", hcrc=True) + member(b"")
            + member(d[10_000:], name=b"x" * 5000) + member(b"", hcrc=True))
    counts = check(blob, d)
    assert counts["members"] == 4


def test_member_edges_inside_chunks_and_on_window_edges(corpora):
    d = corpora["fastq_random"]
    for cut in (C_SMALL * 3, W_SMALL - 5, W_SMALL, W_SMALL + 3):
        first = member(d[:50_000])
        # pad the first member with a stored prefix so that the second starts near `cut` compressed bytes
        filler = random.Random(cut).randbytes(max(0, cut - len(first) - 30))
        blob = member(filler, level=0) + member(d[:50_000]) + member(d[50_000:120_000])
        check(blob, filler + d[:120_000])


# ---- errors: the same outcome as GzipStream ----

def expect_io(blob, **kw):
    from nohuman_b200 import NhError, _ffi
    with pytest.raises(NhError) as ei:
        inflate(blob, **kw)
    assert ei.value.code == _ffi.NH_ERR_IO, ei.value.message


def test_truncation(corpora):
    blob = gzip.compress(corpora["fastq_random"][:100_000])
    for n in (1, 5, 9, 20, len(blob) // 2, len(blob) - 9, len(blob) - 4, len(blob) - 1):
        expect_io(blob[:n])


def test_wrong_crc_and_isize(corpora):
    blob = bytearray(gzip.compress(corpora["fastq_const"][:100_000]))
    bad = bytearray(blob)
    bad[-8] ^= 1
    expect_io(bytes(bad))
    bad = bytearray(blob)
    bad[-4] ^= 1
    expect_io(bytes(bad))


def test_distance_too_far_back():
    # fixed-Huffman block: literal 'a', then a match of length 3 at distance 2 (only 1 byte exists)
    bits = []

    def put(v, n, rev=False):
        if rev:
            v = int(format(v, f"0{n}b")[::-1], 2)
        for i in range(n):
            bits.append((v >> i) & 1)
    put(1, 1)
    put(1, 2)
    put(0x30 + ord("a"), 8, rev=True)   # literal 'a' (8-bit code 00110000 + 97)
    put(1, 7, rev=True)                 # length code 257 (3), 7-bit code 0000001
    put(1, 5, rev=True)                 # distance code 1 (distance 2)
    put(0, 7, rev=True)                 # end of block
    while len(bits) % 8:
        bits.append(0)
    body = bytes(sum(bits[i + j] << j for j in range(8)) for i in range(0, len(bits), 8))
    blob = b"\x1f\x8b\x08\x00\x00\x00\x00\x00\x00\x03" + body + struct.pack("<II", 0, 4)
    with pytest.raises(zlib.error):
        zlib.decompress(blob, 31)
    expect_io(blob)
    # the same distance inside a second member reaches back into the first: still too far
    expect_io(gzip.compress(b"hello world") + blob)


def test_trailing_bytes(corpora):
    d = corpora["fastq_const"][:50_000]
    blob = gzip.compress(d)
    check(blob + bytes(100), d)            # zeros: ignored as gzread ignores them
    check(blob + b"garbage", d)
    expect_io(blob + b"\x1f")              # a new member that is not one
    expect_io(blob + b"\x1f\x8b\x08")
    expect_io(blob + b"\x1fxyzxyzxyzxyz")


def test_not_gzip():
    expect_io(b"")
    expect_io(b"@read\nACGT\n+\nIIII\n")
    expect_io(b"\x1f\x8b\x09\x00" + bytes(20))



# ---- window ends at every byte of block headers and codes ----

def small_blocks(data, level=6):
    """a stream of many dynamic blocks: memLevel 1 ends a block every 127 symbols, so a header or a code
    lies under almost every byte"""
    c = zlib.compressobj(level, zlib.DEFLATED, 31, 1)
    return c.compress(data) + c.flush()


def test_window_ends_at_every_byte(corpora):
    blob = small_blocks(corpora["fastq_random"][:60_000])
    want = ref(blob)
    assert len(blob) > 8192
    for window in range(3000, 3400):  # the first window ends at `window`, later ones wherever the carry puts them
        got, counts = inflate(blob, chunk=1024, window=window)
        assert got == want, window
        assert counts["windows"] > 1


def test_truncation_at_every_byte(corpora):
    from nohuman_b200 import NhError, _ffi
    blob = small_blocks(corpora["fastq_const"][:40_000])
    for n in range(len(blob) // 2, len(blob) // 2 + 300):
        for window in (1024, 1 << 16):
            with pytest.raises(NhError) as ei:
                inflate(blob[:n], chunk=1024, window=window)
            assert ei.value.code == _ffi.NH_ERR_IO, (n, window, ei.value.message)
