"""Inputs and references for the DUST masking tests: seeded sequences mixing short repeat units with
substitutions, random stretches, N runs and lowercase runs; a brute-force enumeration of the definition of
the mask (DESIGN.md §4f); low-complexity stretches spliced into genomes; and dustmasker's two output forms
rendered from a masked sequence."""
from __future__ import annotations

import random

import numpy as np

CODE = {c: i for i, c in enumerate("ACGT")}


def gen(rng: random.Random, n: int) -> bytes:
    out = []
    while len(out) < n:
        k = rng.random()
        if k < 0.3:
            out += rng.choices("ACGT", k=rng.randint(1, 40))
        elif k < 0.8:
            u = "".join(rng.choices("ACGT", k=rng.randint(1, 6)))
            rep = (u * 80)[: rng.randint(5, 120)]
            out += [ch if rng.random() > 0.05 else rng.choice("ACGT") for ch in rep]
        elif k < 0.9:
            out += ["N"] * rng.randint(1, 3)
        else:
            out += list("acgt"[rng.randint(0, 3)] * rng.randint(1, 10))
    return "".join(out[:n]).encode()


def runs(seq: bytes):
    """(first base, triplet codes) of every run of A/C/G/T (either case) with at least one triplet"""
    s = seq.upper()
    i = 0
    while i < len(s):
        if chr(s[i]) not in CODE:
            i += 1
            continue
        j = i
        while j < len(s) and chr(s[j]) in CODE:
            j += 1
        if j - i >= 3:
            b = np.array([CODE[chr(c)] for c in s[i:j]], np.int64)
            yield i, b[:-2] * 16 + b[1:-1] * 4 + b[2:]
        i = j


def brute(seq: bytes, window: int = 64, level: int = 20) -> bytes:
    """The definition, enumerated: every triplet interval x = [a, a + L] with L <= window - 3 is scored; x is
    perfect when it is suspicious (10 r > T L) and no proper sub-interval of it with l >= 1 scores higher,
    compared by cross-multiplication.  The best score over the sub-intervals of [a, a + L] is carried up from
    length L - 1 (those of [a, a + L - 1] and [a + 1, a + L])."""
    mask = np.zeros(len(seq), bool)
    for st, tri in runs(seq):
        n = len(tri)
        cnt = np.zeros((n, 64), np.int64)
        cnt[np.arange(n), tri] = 1
        r = np.zeros(n, np.int64)
        best_r, best_l = None, None
        for L in range(1, min(window - 3, n - 1) + 1):
            m = n - L  # starts a = 0 .. m-1
            t_new = tri[L:L + m]
            r = r[:m] + cnt[np.arange(m), t_new]
            cnt = cnt[:m]
            cnt[np.arange(m), t_new] += 1
            susp = 10 * r > level * L
            if L == 1:
                perfect = susp
                best_r, best_l = r.copy(), np.ones(m, np.int64)
            else:
                ar, al = best_r[:m], best_l[:m]  # [a, a + L - 1]
                br, bl = best_r[1:m + 1], best_l[1:m + 1]  # [a + 1, a + L]
                sub_r = np.where(ar * bl >= br * al, ar, br)
                sub_l = np.where(ar * bl >= br * al, al, bl)
                perfect = susp & (sub_r * L <= r * sub_l)
                take = r * sub_l > sub_r * L
                best_r, best_l = np.where(take, r, sub_r), np.where(take, L, sub_l)
            for a in np.nonzero(perfect)[0]:
                mask[st + a: st + a + L + 3] = True
    out = bytearray(seq.upper())
    for i in np.nonzero(mask)[0]:
        out[i] |= 0x20
    return bytes(out)


KNOWN = [(b"AAAAAA", b"AAAAAA"), (b"AAAAAAA", b"aaaaaaa"), (b"ACGT" * 20, b"acgt" * 20), (b"CA" * 5, b"CA" * 5)]


def splice_low_complexity(rng: np.random.Generator, seq: np.ndarray, per_mbp: int = 400) -> np.ndarray:
    """Microsatellites (units of 1-6 bases, 20-300 bases long, 3 % substitutions) and homopolymers spliced
    into a copy of seq at `per_mbp` sites per million bases."""
    s = seq.copy()
    n = len(s)
    acgt = np.frombuffer(b"ACGT", np.uint8)
    for _ in range(max(1, n * per_mbp // 1_000_000)):
        ln = int(rng.integers(20, 300))
        if n <= ln:
            break
        a = int(rng.integers(0, n - ln))
        unit = acgt[rng.integers(0, 4, size=int(rng.integers(1, 7)))]
        rep = np.resize(unit, ln)
        sub = rng.random(ln) < 0.03
        rep[sub] = acgt[rng.integers(0, 4, size=int(sub.sum()))]
        s[a:a + ln] = rep
    return s


def intervals(masked: bytes):
    """(start, end) of every maximal run of lower-case (masked) bases, 0-based and inclusive"""
    lo = np.frombuffer(masked, np.uint8) >= ord("a")
    d = np.diff(np.concatenate([[0], lo.astype(np.int8), [0]]))
    return list(zip(np.nonzero(d == 1)[0].tolist(), (np.nonzero(d == -1)[0] - 1).tolist()))


def render(records, fmt: str) -> bytes:
    """dustmasker's output for [(header line without '>', masked sequence)]: FASTA wrapped at 60, or interval
    lines "start - end" under each header"""
    out = []
    for h, m in records:
        out.append(b">" + h + b"\n")
        if fmt == "fasta":
            out += [m[i:i + 60] + b"\n" for i in range(0, len(m), 60)]
        else:
            out += [f"{a} - {b}\n".encode() for a, b in intervals(m)]
    return b"".join(out)
