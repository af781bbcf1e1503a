"""Synthetic kraken2-format databases and reads, generated on the GPU
(include/nohuman_synth.h).  Tooling for bench.py and smoke(): the HPRC
databases nohuman downloads (reference config.toml:1-19) are unavailable
offline.  File images follow SURVEY.md Appendix B byte for byte, so the
resulting directory is an ordinary kraken2 database.
"""
from __future__ import annotations

import ctypes as C
import os
import struct
from dataclasses import dataclass

import numpy as np

from . import _ffi
from ._ffi import check, lib
from .api import Database

DEFAULT_TOGGLE_MASK = 0xE37E28C4271B5A2D


class SynthDbParams(C.Structure):
    _fields_ = [
        ("capacity", C.c_uint64), ("target_load", C.c_double), ("genome_seed", C.c_uint64),
        ("block_bases", C.c_uint64), ("overlap_frac", C.c_double), ("max_genome_bases", C.c_uint64),
    ]


class SynthReadsParams(C.Structure):
    _fields_ = [
        ("seed", C.c_uint64), ("genome_seed", C.c_uint64), ("genome_bases", C.c_uint64),
        ("human_frac", C.c_double), ("sub_rate", C.c_double), ("ins_rate", C.c_double),
        ("del_rate", C.c_double), ("n_rate", C.c_double), ("paired", C.c_int32),
        ("reserved", C.c_int32), ("insert_mean", C.c_double), ("insert_sd", C.c_double),
    ]


_vp, _u64, _i32 = C.c_void_p, C.c_uint64, C.c_int
_SYNTH_SYMBOLS = {
    "nh_synth_build_db": (_i32, [_vp, C.c_size_t, _vp, C.c_size_t, _vp, _i32,
                                 C.POINTER(SynthDbParams), _i32, C.POINTER(_vp), C.POINTER(_u64)]),
    "nh_db_download_cells": (_i32, [_vp, _vp]),
    "nh_synth_reads": (_i32, [_i32, _vp, _vp, _u64, C.POINTER(SynthReadsParams), _vp]),
    "nh_synth_genome": (_i32, [_i32, _u64, _u64, _u64, _vp]),
}
_bound = False


def _lib():
    global _bound
    L = lib()
    if not _bound:
        for name, (res, args) in _SYNTH_SYMBOLS.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _bound = True
    return L


def spaced_seed_mask(l: int = 31, spaces: int = 7) -> int:
    """kraken2-build's seed template '1'*(l-2s) + '01'*s, each bit doubled (SURVEY A.1)."""
    tmpl = "1" * (l - 2 * spaces) + "01" * spaces
    return int("".join("11" if c == "1" else "00" for c in tmpl), 2)


def opts_image(k: int = 35, l: int = 31, spaces: int = 7, toggle: int = DEFAULT_TOGGLE_MASK,
               min_hash: int = 0) -> bytes:
    """opts.k2d: struct IndexOptions, 64 bytes (SURVEY Appendix B)."""
    ssm = spaced_seed_mask(l, spaces) if spaces else 0
    return struct.pack("<QQQQB7xQiii4x", k, l, ssm, toggle, 1, min_hash, 1, 0, 0)


@dataclass
class TaxNode:
    ext_id: int
    parent_ext_id: int
    name: str = ""
    rank: str = ""


def taxonomy_image(nodes: list[TaxNode]):
    """taxo.k2d image with kraken2's BFS numbering (root = 1, parent < child).
    Returns (bytes, {ext_id: internal_id})."""
    by_parent: dict[int, list[TaxNode]] = {}
    root = None
    for n in nodes:
        if n.parent_ext_id == n.ext_id or n.parent_ext_id == 0:
            root = n
        else:
            by_parent.setdefault(n.parent_ext_id, []).append(n)
    assert root is not None, "taxonomy needs a root"
    order = [root]
    internal = {root.ext_id: 1}
    recs = [None, dict(parent=0, first_child=0, child_count=0, node=root)]
    i = 0
    while i < len(order):
        cur = order[i]
        cid = internal[cur.ext_id]
        for ch in by_parent.get(cur.ext_id, []):
            nid = len(recs)
            internal[ch.ext_id] = nid
            if recs[cid]["child_count"] == 0:
                recs[cid]["first_child"] = nid
            recs[cid]["child_count"] += 1
            recs.append(dict(parent=cid, first_child=0, child_count=0, node=ch))
            order.append(ch)
        i += 1
    names, ranks = bytearray(), bytearray()
    body = bytearray(struct.pack("<7Q", 0, 0, 0, 0, 0, 0, 0))
    for r in recs[1:]:
        n = r["node"]
        body += struct.pack("<7Q", r["parent"], r["first_child"], r["child_count"], len(names),
                            len(ranks), n.ext_id, 0)
        names += n.name.encode() + b"\0"
        ranks += n.rank.encode() + b"\0"
    img = b"K2TAXDAT" + struct.pack("<QQQ", len(recs), len(names), len(ranks)) + bytes(body) \
        + bytes(names) + bytes(ranks)
    return img, internal


def human_pangenome_taxonomy(n_super: int = 5, n_hap_per_super: int = 4):
    """Human lineage down to Homo sapiens, then synthetic population /
    haplotype nodes (HPRC-like: a few dozen nodes).  Returns (nodes, leaf_ext_ids)."""
    lineage = [
        (1, 1, "root", "no rank"), (131567, 1, "cellular organisms", "no rank"),
        (2759, 131567, "Eukaryota", "superkingdom"), (33154, 2759, "Opisthokonta", "clade"),
        (33208, 33154, "Metazoa", "kingdom"), (7711, 33208, "Chordata", "phylum"),
        (40674, 7711, "Mammalia", "class"), (9443, 40674, "Primates", "order"),
        (9604, 9443, "Hominidae", "family"), (9605, 9604, "Homo", "genus"),
        (9606, 9605, "Homo sapiens", "species"),
    ]
    nodes = [TaxNode(*t) for t in lineage]
    leaves = []
    for s in range(n_super):
        sid = 9000001 + s
        nodes.append(TaxNode(sid, 9606, f"synthetic superpopulation {s}", "subspecies"))
        for h in range(n_hap_per_super):
            hid = 9100001 + s * 100 + h
            nodes.append(TaxNode(hid, sid, f"synthetic haplotype {s}.{h}", "strain"))
            leaves.append(hid)
    return nodes, leaves


@dataclass
class SynthDb:
    db: Database
    opts: bytes
    taxo: bytes
    internal: dict
    genome_seed: int
    genome_bases: int

    def download_cells(self) -> np.ndarray:
        info = self.db.info
        out = np.empty(int(info.capacity), np.uint32)
        check(_lib().nh_db_download_cells(self.db._h, out.ctypes.data))
        return out

    def hash_header(self):
        i = self.db.info
        return [int(i.capacity), int(i.size), int(i.key_bits), int(i.value_bits)]

    def save(self, db_dir: str) -> None:
        os.makedirs(db_dir, exist_ok=True)
        with open(os.path.join(db_dir, "opts.k2d"), "wb") as f:
            f.write(self.opts)
        with open(os.path.join(db_dir, "taxo.k2d"), "wb") as f:
            f.write(self.taxo)
        with open(os.path.join(db_dir, "hash.k2d"), "wb") as f:
            f.write(struct.pack("<4Q", *self.hash_header()))
            self.download_cells().tofile(f)


def build_synthetic_db(capacity: int, device: int = 0, target_load: float = 0.7,
                       genome_seed: int = 0x5EED, block_bases: int = 1 << 20,
                       overlap_frac: float = 0.1, max_genome_bases: int = 0, k: int = 35,
                       l: int = 31, spaces: int = 7, n_super: int = 5,
                       n_hap_per_super: int = 4) -> SynthDb:
    nodes, leaves = human_pangenome_taxonomy(n_super, n_hap_per_super)
    taxo, internal = taxonomy_image(nodes)
    opts = opts_image(k, l, spaces)
    leaf_ids = np.array([internal[x] for x in leaves], np.uint32)
    p = SynthDbParams(capacity, target_load, genome_seed, block_bases, overlap_frac,
                      max_genome_bases)
    h = C.c_void_p()
    gb = C.c_uint64()
    check(_lib().nh_synth_build_db(opts, len(opts), taxo, len(taxo), leaf_ids.ctypes.data,
                                   len(leaf_ids), C.byref(p), device, C.byref(h), C.byref(gb)))
    return SynthDb(Database(h.value), opts, taxo, internal, genome_seed, gb.value)


def synth_reads(device: int, d_bases: int, d_offsets: int, n_seqs: int, genome_seed: int,
                genome_bases: int, seed: int = 1, human_frac: float = 0.5, sub_rate: float = 0.005,
                ins_rate: float = 0.0, del_rate: float = 0.0, n_rate: float = 0.01,
                paired: bool = False, insert_mean: float = 350.0, insert_sd: float = 50.0,
                stream: int = 0) -> None:
    p = SynthReadsParams(seed, genome_seed, genome_bases, human_frac, sub_rate, ins_rate, del_rate,
                         n_rate, int(paired), 0, insert_mean, insert_sd)
    check(_lib().nh_synth_reads(device, d_bases, d_offsets, n_seqs, C.byref(p), stream))


def synth_genome(device: int, genome_seed: int, start: int, n: int) -> np.ndarray:
    out = np.empty(n, np.uint8)
    check(_lib().nh_synth_genome(device, genome_seed, start, n, out.ctypes.data))
    return out


def fastq_corpus(n_bytes: int, seed: int = 0, random_quals: bool = False, read_len: int = 150) -> bytes:
    """Seeded FASTQ text of n_bytes (the last record cut short), laid out as the file pipeline writes kept
    reads: `@r<9-digit id>/1` headers, bases from ACGT with 1 % N, `+`, and qualities that are all `I` as
    in tools/file_pipeline_bench.py, or uniformly random Phred 2..41 (random_quals).  The corpus of the
    GPU gzip ratio checks and of tools/gzip_bench.py."""
    rng = np.random.default_rng(seed)
    hdr_len = len(b"@r000000000/1\n")
    rec_len = hdr_len + 2 * read_len + 4
    n = max(1, -(-n_bytes // rec_len))
    rec = np.empty((n, rec_len), np.uint8)
    rec[:, :hdr_len] = np.frombuffer(b"@r000000000/1\n", np.uint8)
    idx = np.arange(n)
    for d in range(9):
        rec[:, 2 + 8 - d] = 48 + (idx // 10 ** d) % 10
    seq = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, size=(n, read_len))]
    seq[rng.random((n, read_len)) < 0.01] = ord("N")
    o = hdr_len
    rec[:, o:o + read_len] = seq
    rec[:, o + read_len:o + read_len + 3] = np.frombuffer(b"\n+\n", np.uint8)
    q = rec[:, o + read_len + 3:o + 2 * read_len + 3]
    q[:] = rng.integers(33 + 2, 33 + 42, size=q.shape) if random_quals else ord("I")
    rec[:, -1] = ord("\n")
    return rec.tobytes()[:n_bytes]
