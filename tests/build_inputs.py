"""Inputs for the database-build tests: NCBI-style taxonomy dumps, seqid2taxid maps and FASTA libraries
written from the cfg1 taxonomy and genomes of synth.py, and the oracle's taxonomy over the same marked nodes."""
from __future__ import annotations

import bz2
import ctypes as C
import gzip
import os

import numpy as np

import synth

# taxa that no map entry uses: a whole unmarked branch (archaea), an unmarked sibling genus and species
UNMARKED = [
    (2157, 131567, "Archaea", "superkingdom"),
    (28890, 2157, "Methanobacteriota", "phylum"),
    (9596, 9604, "Pan", "genus"),
    (9598, 9596, "Pan troglodytes", "species"),
    (1280, 1386, "Staphylococcus aureus", "species"),
]


def write_dmp(d, taxa=None, extra=UNMARKED, seed=0):
    """nodes.dmp / names.dmp in NCBI's layout, lines shuffled, several name classes per taxon."""
    taxa = list(taxa or synth.TAXONOMY_CFG1) + list(extra)
    rng = np.random.default_rng(seed)
    order = rng.permutation(len(taxa))
    nodes, names = [], []
    for i in order:
        tid, parent, name, rank = taxa[i]
        nodes.append(f"{tid}\t|\t{parent}\t|\t{rank}\t|\tXX\t|\t0\t|\t1\t|\t11\t|\t1\t|\t0\t|\t1\t|\t0\t|\t0\t|\t\t|\n")
        names.append(f"{tid}\t|\t{name} (synonym)\t|\t\t|\tsynonym\t|\n")
        names.append(f"{tid}\t|\t{name}\t|\t\t|\tscientific name\t|\n")
        names.append(f"{tid}\t|\t{name.lower()}\t|\t{name} <common>\t|\tgenbank common name\t|\n")
    os.makedirs(d, exist_ok=True)
    with open(os.path.join(d, "nodes.dmp"), "w") as f:
        f.writelines(nodes)
    with open(os.path.join(d, "names.dmp"), "w") as f:
        f.writelines(names)
    return os.path.join(d, "nodes.dmp"), os.path.join(d, "names.dmp")


def marked(map_taxids, taxa=None):
    """The map's taxids and all their ancestors."""
    parent = {t[0]: t[1] for t in (list(taxa or synth.TAXONOMY_CFG1) + UNMARKED)}
    out = set()
    for t in map_taxids:
        while t not in out:
            out.add(t)
            if t == 1:
                break
            t = parent[t]
    return out


def oracle_taxonomy(oracle, marked_ids, taxa=None):
    """k2o_taxonomy_build over the marked nodes given in ascending taxid (so children come in that order)."""
    info = {t[0]: t for t in (list(taxa or synth.TAXONOMY_CFG1) + UNMARKED)}
    ts = [oracle.TaxSpec(*info[t]) for t in sorted(marked_ids)]
    L = oracle.lib()
    tax = oracle.Taxonomy()
    n = len(ts)
    ext = (C.c_uint64 * n)(*[t.ext_id for t in ts])
    par = (C.c_uint64 * n)(*[t.parent_ext_id for t in ts])
    nm = (C.c_char_p * n)(*[t.name.encode() for t in ts])
    rk = (C.c_char_p * n)(*[t.rank.encode() for t in ts])
    assert L.k2o_taxonomy_build(C.byref(tax), n, ext, par, nm, rk) == 0
    return tax, ts


def oracle_taxo_bytes(oracle, tax, tmp) -> bytes:
    p = os.path.join(tmp, "oracle_taxo.k2d")
    assert oracle.lib().k2o_save_taxonomy(p.encode(), C.byref(tax)) == 0
    return open(p, "rb").read()


def wrap(seq: bytes, width: int) -> bytes:
    return b"\n".join(seq[i:i + width] for i in range(0, len(seq), width)) + b"\n"


def mask_runs(rng, seq: np.ndarray) -> np.ndarray:
    """Lowercase runs, N runs and dustmasker-style x runs."""
    s = seq.copy()
    n = len(s)
    for ch, count in ((None, 6), (ord("N"), 4), (ord("x"), 4)):
        for _ in range(count):
            a = int(rng.integers(0, max(1, n - 400)))
            b = a + int(rng.integers(20, 400))
            if ch is None:
                s[a:b] = s[a:b] | 0x20
            else:
                s[a:b] = ch
    return s


def write_library(d, genomes, seed=7):
    """The cfg1 genomes as a library of several files: plain, gzip and bzip2; multi-record; wrapped at 60 and
    80; lowercase, N and x runs; one record without a map entry.  Returns (files, map path, records) where
    records is [(taxid or None, sequence bytes)] in library order."""
    rng = np.random.default_rng(seed)
    os.makedirs(d, exist_ok=True)
    recs = []  # (file index, seqid, taxid, bytes)
    for gi, (tid, g) in enumerate(genomes):
        s = mask_runs(rng, g)
        if gi == 0:  # the human chromosome as one record
            recs.append((0, f"chr_{tid}_a", tid, bytes(s)))
        else:  # bacteria cut into two records (chromosome + "plasmid")
            cut = len(s) * 3 // 4
            recs.append((gi, f"seq{gi}_chrom", tid, bytes(s[:cut])))
            recs.append((gi, f"seq{gi}_plasmid", tid, bytes(s[cut:])))
    junk = bytes(synth.random_genome(rng, 5000))
    recs.append((1, "unmapped_contig", None, junk))
    kinds = ["plain", "gz", "bz2", "plain"]
    files = []
    for fi in range(len(genomes)):
        body = b"".join(b">" + sid.encode() + b" some description\n" + wrap(s, 60 if fi % 2 else 80)
                        for f, sid, _, s in recs if f == fi)
        kind = kinds[fi % len(kinds)]
        name = os.path.join(d, f"lib{fi}.fna" + {"plain": "", "gz": ".gz", "bz2": ".bz2"}[kind])
        with open(name, "wb") as f:
            f.write({"plain": lambda b: b, "gz": gzip.compress, "bz2": bz2.compress}[kind](body))
        files.append(name)
    mp = os.path.join(d, "seqid2taxid.map")
    with open(mp, "w") as f:
        for _, sid, tid, _ in recs:
            if tid is not None:
                f.write(f"{sid}\t{tid}\n")
    order = [(tid, s) for fi in range(len(genomes)) for f, _, tid, s in recs if f == fi]
    return files, mp, order
