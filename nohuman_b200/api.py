"""Host-side face of the hot path, mirroring how the reference drives kraken2.

The reference (mbhall88/nohuman) assembles a kraken2 argv and blocks on the
child process (src/main.rs:210-270, src/lib.rs:22-48).  `Database` is its
`--db` (validated like src/lib.rs:119-141), `Session` carries `--confidence`,
`--paired` and the classified/unclassified-out polarity (src/main.rs:259-265),
and `Session.classify` is the work kraken2 does per batch of reads.  All
computation happens in libnohuman_gpu.so (CUDA, sm_100a).
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _ffi
from ._ffi import (GUNZIP_COUNTS, NH_ERR_CAPACITY, BatchStats, DbInfo, Files, NhError, Params, RunStats, check,
                   lib)


def parse_confidence_score(text: str) -> float:
    """parse_confidence_score (src/lib.rs:145-151) plus the f32 -> string ->
    double round trip of src/main.rs:213: nohuman parses the value as f32,
    hands kraken2 its shortest decimal form, and kraken2 re-parses a double."""
    try:
        f32 = np.float32(float(text))
    except ValueError as e:  # same wording as the reference's error
        raise ValueError("Confidence score must be a number") from e
    if not (0.0 <= float(f32) <= 1.0):
        raise ValueError("Confidence score must be in the closed interval [0, 1]")
    return float(np.format_float_positional(f32, unique=True, trim="0"))


def make_files(in1, out1, in2=None, out2=None, out_format="u", tag_classified=True) -> Files:
    f = Files()
    f.in1 = str(in1).encode()
    f.in2 = str(in2).encode() if in2 is not None else None
    f.out1 = str(out1).encode()
    f.out2 = str(out2).encode() if out2 is not None else None
    f.out_format = ord(out_format)
    f.tag_classified = int(tag_classified)
    return f


def run_files_multi(sessions, in1, out1, in2=None, out2=None, out_format="u", tag_classified=True) -> RunStats:
    """nh_run_files over several sessions (one per GPU, database replicated): batches are
    dealt to the GPUs, output order is input order."""
    f = make_files(in1, out1, in2, out2, out_format, tag_classified)
    arr = (C.c_void_p * len(sessions))(*[s._h for s in sessions])
    st = RunStats()
    check(lib().nh_run_files_multi(arr, len(sessions), C.byref(f), C.byref(st)))
    return st


def rewrite_files(keep: np.ndarray, call_ext: np.ndarray, in1, out1, in2=None, out2=None,
                  out_format="u", tag_classified=True, threads=2) -> RunStats:
    """Host-logic test hook (no GPU): the file pipeline with decisions supplied by the caller."""
    keep = np.ascontiguousarray(keep, dtype=np.uint8)
    call_ext = np.ascontiguousarray(call_ext, dtype=np.uint32)
    f = make_files(in1, out1, in2, out2, out_format, tag_classified)
    st = RunStats()
    check(lib().nh_debug_rewrite_files(C.byref(f), keep.ctypes.data, call_ext.ctypes.data, len(keep),
                                       threads, C.byref(st)))
    return st


def packed_units(offsets: np.ndarray) -> int:
    offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
    n = C.c_uint64()
    check(lib().nh_packed_units(offsets.ctypes.data, len(offsets) - 1, C.byref(n)))
    return int(n.value)


def pack_reads(bases: np.ndarray, offsets: np.ndarray, threads: int = 1):
    """ASCII -> (codes u8[units*8], valid u32[units], poff u32[n_seqs+1]) on the host (nh_pack_reads, no GPU needed)."""
    bases = np.ascontiguousarray(bases, dtype=np.uint8)
    offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
    units = packed_units(offsets)
    codes = np.zeros(units * 8 + 16, np.uint8)
    valid = np.zeros(units + 4, np.uint32)
    poff = np.zeros(len(offsets), np.uint32)
    check(lib().nh_pack_reads(bases.ctypes.data, offsets.ctypes.data, len(offsets) - 1, codes.ctypes.data, valid.ctypes.data,
                              poff.ctypes.data, threads))
    return codes, valid, poff


BGZF_INPUT = 0xFF00  # input bytes per BGZF member


def bgzf_compress(data: bytes, device: int = 0) -> bytes:
    """BGZF members of `data` (0xff00 input bytes each, no end-of-file member), deflated on `device`
    (nh_bgzf_compress).  gzip.decompress() reads the result."""
    n = len(data)
    cap = -(-n // BGZF_INPUT) * 65536
    out = np.empty(max(cap, 1), np.uint8)  # not zero-filled: only the bytes written are read back
    got = C.c_size_t()
    check(lib().nh_bgzf_compress(int(device), data, n, out.ctypes.data, cap, C.byref(got)))
    return C.string_at(out.ctypes.data, got.value)


def bgzf_kernel_seconds(data: bytes, device: int = 0, iters: int = 10) -> float:
    """Device time of the BGZF kernels for `data` in one batch (nh_bench_bgzf), mean of `iters` launches."""
    t = C.c_double()
    check(lib().nh_bench_bgzf(int(device), data, len(data), int(iters), C.byref(t)))
    return t.value


def debug_gunzip(data: bytes, device: int = 0, chunk: int = 0, window: int = 0, flags: int = 0):
    """(inflated bytes, counts) of the gzip stream `data` inflated on `device` with the given chunk and window
    sizes in compressed bytes (0: the defaults) and nh_debug_gunzip flags; counts maps _ffi.GUNZIP_COUNTS to
    what ran."""
    n = len(data)
    counts = (C.c_uint64 * len(GUNZIP_COUNTS))()
    got = C.c_size_t()
    cap = 4 * n + 65536  # FASTQ inflates about 4x; a larger stream is inflated again into the size it reported
    for _ in range(2):
        out = np.empty(cap, np.uint8)
        rc = lib().nh_debug_gunzip(int(device), data, n, out.ctypes.data, cap, C.byref(got), int(chunk), int(window),
                                   int(flags), counts)
        if rc != NH_ERR_CAPACITY or got.value <= cap:
            break
        cap = got.value
    check(rc)
    return C.string_at(out.ctypes.data, got.value), dict(zip(GUNZIP_COUNTS, counts))


def gunzip(data: bytes, device: int = 0) -> bytes:
    """What `gzip -dc` gives for `data`, inflated on `device` (nh_gunzip): every member, trailing bytes that
    do not start a member ignored.  NhError NH_ERR_IO for a corrupt or truncated stream."""
    return debug_gunzip(data, device)[0]


def gunzip_kernel_seconds(data: bytes, device: int = 0, iters: int = 3) -> float:
    """Device time of nh_gunzip's kernels for the gzip stream `data` (nh_bench_gunzip), mean of `iters` runs."""
    t = C.c_double()
    check(lib().nh_bench_gunzip(int(device), data, len(data), int(iters), C.byref(t)))
    return t.value


class Database:
    """A kraken2 database (hash.k2d / opts.k2d / taxo.k2d) resident in HBM."""

    def __init__(self, handle: int):
        self._h = C.c_void_p(handle)

    @classmethod
    def open(cls, db_dir: str, device: int = 0) -> "Database":
        h = C.c_void_p()
        check(lib().nh_db_open(str(db_dir).encode(), device, C.byref(h)))
        return cls(h.value)

    @classmethod
    def open_multi(cls, db_dir: str, devices: list[int]) -> list["Database"]:
        """One disk read, one replica per device (NCCL broadcast, or a peer-copy tree): nh_db_open_multi."""
        ids = (C.c_int * len(devices))(*devices)
        hs = (C.c_void_p * len(devices))()
        check(lib().nh_db_open_multi(str(db_dir).encode(), ids, len(devices), hs))
        return [cls(h) for h in hs]

    @classmethod
    def from_memory(cls, opts: bytes, taxo: bytes, hash_header, cells, device: int = 0,
                    cells_on_device: bool = False) -> "Database":
        """cells: numpy uint32 array (host) or an int device pointer."""
        hdr = (C.c_uint64 * 4)(*[int(x) for x in hash_header])
        h = C.c_void_p()
        keep = None
        if cells_on_device:
            ptr = C.c_void_p(int(cells))
        else:
            keep = np.ascontiguousarray(cells, dtype=np.uint32)
            ptr = C.c_void_p(keep.ctypes.data)
        check(lib().nh_db_open_memory(opts, len(opts), taxo, len(taxo), hdr, ptr,
                                      int(cells_on_device), device, C.byref(h)))
        return cls(h.value)

    def clone(self, device: int) -> "Database":
        """Replica on another GPU of this process (peer copy)."""
        h = C.c_void_p()
        check(lib().nh_db_clone(self._h, device, C.byref(h)))
        return Database(h.value)

    @property
    def info(self) -> DbInfo:
        out = DbInfo()
        check(lib().nh_db_info(self._h, C.byref(out)))
        return out

    def device_cells_ptr(self) -> int:
        return int(lib().nh_db_device_cells(self._h) or 0)

    def random_gather_gbs(self, n_reads: int = 1 << 26, iters: int = 3) -> float:
        out = C.c_double()
        check(lib().nh_bench_random_gather(self._h, n_reads, iters, C.byref(out)))
        return out.value

    def probe_pattern(self, lanes: int = 1, p_continue: float = 0.41, sm_window_bytes: int = 0,
                      items_per_chain: int = 64, iters: int = 3, depth: int = 4,
                      blocks_per_sm: int = 8) -> tuple[float, float]:
        """(lookups/s, table requests/s) of the probe's access pattern alone (nh_bench_probe_pattern)."""
        a, b = C.c_double(), C.c_double()
        check(lib().nh_bench_probe_pattern(self._h, lanes, depth, blocks_per_sm, p_continue, sm_window_bytes,
                                           items_per_chain, iters, C.byref(a), C.byref(b)))
        return a.value, b.value

    def close(self) -> None:
        if self._h:
            lib().nh_db_close(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()


class Session:
    """One classification stream: parameters + device buffers + CUDA stream."""

    def __init__(self, db: Database, confidence: float = 0.0, paired: bool = False,
                 keep_human: bool = False, minimum_hit_groups: int = 2, threads: int = 1,
                 max_batch_bases: int = 0, max_batch_seqs: int = 0, emit_runs: bool = False,
                 gpu_gzip: bool = False):
        p = Params()
        p.confidence = float(confidence)
        p.minimum_hit_groups = int(minimum_hit_groups)
        p.paired = int(paired)
        p.keep_human = int(keep_human)
        p.threads = int(threads)
        p.max_batch_bases = int(max_batch_bases)
        p.max_batch_seqs = int(max_batch_seqs)
        p.emit_runs = int(emit_runs)
        p.gpu_gzip = int(gpu_gzip)  # gzip output of run_files / run_files_multi deflated on the GPU
        self.paired = bool(paired)
        self.db = db
        self._h = C.c_void_p()
        check(lib().nh_session_create(db._h, C.byref(p), C.byref(self._h)))

    # -- host buffers in, host results out (H2D/D2H inside the call) --
    def classify(self, bases: np.ndarray, offsets: np.ndarray, out_call: np.ndarray | None = None,
                 out_keep: np.ndarray | None = None):
        bases = np.ascontiguousarray(bases, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        n_seqs = len(offsets) - 1
        n_units = n_seqs // 2 if self.paired else n_seqs
        call = out_call if out_call is not None else np.empty(n_units, np.uint32)
        keep = out_keep if out_keep is not None else np.empty(n_units, np.uint8)
        st = BatchStats()
        check(lib().nh_classify_batch(self._h, bases.ctypes.data, offsets.ctypes.data, n_seqs,
                                      call.ctypes.data, keep.ctypes.data, C.byref(st)))
        return call, keep, st

    def classify_raw(self, bases_ptr: int, offsets_ptr: int, n_seqs: int, call_ptr: int,
                     keep_ptr: int) -> BatchStats:
        """Same call on raw host addresses (e.g. pinned torch tensors)."""
        st = BatchStats()
        check(lib().nh_classify_batch(self._h, bases_ptr, offsets_ptr, n_seqs, call_ptr, keep_ptr,
                                      C.byref(st)))
        return st

    # -- packed transfer format (2-bit codes + validity bits, 0.4 B/base over PCIe) ---------
    def classify_packed(self, bases: np.ndarray, offsets: np.ndarray, threads: int = 1):
        """pack_reads on the host, then nh_classify_batch_packed; same results as classify()."""
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        codes, valid, poff = pack_reads(bases, offsets, threads)
        n_seqs = len(offsets) - 1
        n_units = n_seqs // 2 if self.paired else n_seqs
        call = np.zeros(n_units, np.uint32)
        keep = np.zeros(n_units, np.uint8)
        st = BatchStats()
        check(lib().nh_classify_batch_packed(self._h, codes.ctypes.data, valid.ctypes.data, poff.ctypes.data,
                                             offsets.ctypes.data, n_seqs, call.ctypes.data, keep.ctypes.data, C.byref(st)))
        return call, keep, st

    def classify_packed_raw(self, codes_ptr: int, valid_ptr: int, poff_ptr: int, offsets_ptr: int, n_seqs: int,
                            call_ptr: int, keep_ptr: int) -> BatchStats:
        st = BatchStats()
        check(lib().nh_classify_batch_packed(self._h, codes_ptr, valid_ptr, poff_ptr, offsets_ptr, n_seqs, call_ptr,
                                             keep_ptr, C.byref(st)))
        return st

    def classify_pack(self, bases: np.ndarray, offsets: np.ndarray, threads: int = 1):
        """nh_classify_batch_pack: ASCII in, packed by the session's pool of `threads` host threads into
        pinned planes, sent in the packed format; same results as classify()."""
        bases = np.ascontiguousarray(bases, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        n_seqs = len(offsets) - 1
        n_units = n_seqs // 2 if self.paired else n_seqs
        call = np.zeros(n_units, np.uint32)
        keep = np.zeros(n_units, np.uint8)
        st = BatchStats()
        check(lib().nh_classify_batch_pack(self._h, bases.ctypes.data, offsets.ctypes.data, n_seqs, int(threads),
                                           call.ctypes.data, keep.ctypes.data, C.byref(st)))
        return call, keep, st

    def classify_pack_raw(self, bases_ptr: int, offsets_ptr: int, n_seqs: int, threads: int, call_ptr: int,
                          keep_ptr: int) -> BatchStats:
        st = BatchStats()
        check(lib().nh_classify_batch_pack(self._h, bases_ptr, offsets_ptr, n_seqs, int(threads), call_ptr, keep_ptr,
                                           C.byref(st)))
        return st

    # -- device-resident (asynchronous on the session stream) ---------
    def classify_device(self, d_bases: int, d_offsets: int, n_seqs: int, total_bases: int,
                        d_out_call: int, d_out_keep: int) -> None:
        check(lib().nh_classify_batch_device(self._h, d_bases, d_offsets, n_seqs, total_bases,
                                             d_out_call, d_out_keep))

    def last_batch_runs(self, n_seqs: int, capacity: int):
        """(seq_first_run[n_seqs+1], run_taxon_ext, run_len) of the batch just classified."""
        first = np.zeros(n_seqs + 1, np.uint32)
        ext = np.zeros(max(capacity, 1), np.uint32)
        ln = np.zeros(max(capacity, 1), np.uint16)
        n = C.c_uint64()
        check(lib().nh_last_batch_runs(self._h, n_seqs, first.ctypes.data, ext.ctypes.data, ln.ctypes.data,
                                       capacity, C.byref(n)))
        return first, ext[:n.value], ln[:n.value]

    def sync(self) -> BatchStats:
        st = BatchStats()
        check(lib().nh_session_sync(self._h, C.byref(st)))
        return st

    # -- file API: what `kraken.run(&kraken_cmd)` + compress() do in the reference --
    def run_files(self, in1: str, out1: str, in2: str | None = None, out2: str | None = None,
                  out_format: str = "u", tag_classified: bool = True) -> RunStats:
        """src/main.rs:270 + :340-368 in one call: classify in1[/in2], write the kept
        records (final, compressed per out_format u/g/b/x/z) to out1[/out2] in input order."""
        f = make_files(in1, out1, in2, out2, out_format, tag_classified)
        st = RunStats()
        check(lib().nh_run_files(self._h, C.byref(f), C.byref(st)))
        return st

    @property
    def stream(self) -> int:
        return int(lib().nh_session_stream(self._h) or 0)

    # -- per-stage entry points used by the parity tests --------------
    def debug_minimizers(self, bases: np.ndarray, offsets: np.ndarray):
        bases = np.ascontiguousarray(bases, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        n_seqs = len(offsets) - 1
        k = int(self.db.info.k)
        lens = np.diff(offsets).astype(np.int64)
        npos = np.maximum(lens - k + 1, 0).astype(np.uint64)
        pos_off = np.zeros(n_seqs + 1, np.uint64)
        np.cumsum(npos, out=pos_off[1:])
        total = int(pos_off[-1])
        mins = np.zeros(total + 1, np.uint64)
        amb = np.zeros(total + 1, np.uint8)
        check(lib().nh_debug_minimizers(self._h, bases.ctypes.data, offsets.ctypes.data, n_seqs,
                                        pos_off.ctypes.data, mins.ctypes.data, amb.ctypes.data))
        return mins[:total], amb[:total], pos_off

    def debug_probe(self, keys: np.ndarray) -> np.ndarray:
        keys = np.ascontiguousarray(keys, dtype=np.uint64)
        out = np.zeros(len(keys), np.uint32)
        check(lib().nh_debug_probe(self._h, keys.ctypes.data, len(keys), out.ctypes.data))
        return out

    def debug_last_batch(self, n_units: int):
        call = np.zeros(n_units, np.uint32)
        tk = np.zeros(n_units, np.uint32)
        hg = np.zeros(n_units, np.uint32)
        check(lib().nh_debug_last_batch(self._h, call.ctypes.data, tk.ctypes.data, hg.ctypes.data,
                                        n_units))
        return call, tk, hg

    def close(self) -> None:
        if self._h:
            lib().nh_session_destroy(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()


__all__ = ["Database", "Session", "NhError", "BatchStats", "DbInfo", "parse_confidence_score"]
