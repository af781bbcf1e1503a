"""Probe chains at the hash table's edges, on tables whose every lookup is placed by design.

kraken2 walks a chain of occupied cells from a key's home cell `hash % capacity` to the first cell that is empty or
holds the key's compacted key, with 64-bit indices and no limit on the distance.  The kernels walk it by 32-byte
sectors (and, with the miss filter, by 32-cell filter records), count sectors and records in narrow fields and keep
sector indices in 32 bits.  Naturally built tables at load 0.7 never reach those limits, so this module builds the
tables itself:

  * `fmix64_inv` inverts kraken2's MurmurHash3 finaliser, so that a key can be made for a chosen home cell; keys for
    homes that need not be exact are drawn forwards.  A key is a masked minimizer (spaced-seed bits zero, below
    4^l) whose toggled value is small, and a 35-base read whose only k-mer position has that minimizer carries it:
    `oracle.scan_positions` decides whether a read does.
  * A `Table` is sparse: runs of *blocker* cells (valid taxa, compacted keys from a small pool that holds 0 and
    all-ones) with planted cells at chosen depths, and decoys that share a planted key's compacted key after its
    slot and before its home (kraken2 returns the first match).  The oracle answers from the same cells.
  * Reads are classified with minimum_hit_groups 1 and confidence 0, so that a one-k-mer read's call is exactly
    its lookup's taxon.

The tables:
  1. capacity 2^22 + 13 (partial last sector and filter block) with one run of 1.25 M occupied cells that wraps
     from the table's end to cell 0, keys planted at depths 0-40, at powers of two, and around the streaming
     kernel's old visit caps (262 128 cells: 32 766 sectors, 524 280: 65 535 sectors, 1 048 512: 32 766 filter
     records), homes in the partial last sector and block, and keys past the run's end (true misses);
  2. capacity 2^32 + 2^27 + 13 (17.7 GB of cells, 4.4 GB of miss filter): homes above 2^32, chains across cell 2^32
     (sector 2^29, filter block 2^27), chains that wrap from the partial last sector to cell 0, and a control set
     below 2^31.  It needs about 26 GB of free device memory and is skipped with the reason otherwise.
The boundary between the streaming and the warp-per-tile kernels at 2^35 - 8 cells (a 128 GiB table) is out of
scope here."""
import os

import numpy as np
import pytest

import synth

gpu = pytest.mark.gpu
U = np.uint64
MASK64 = (1 << 64) - 1
FMIX_C1, FMIX_C2 = 0xFF51AFD7ED558CCD, 0xC4CEB9FE1A85EC53
FMIX_C1_INV, FMIX_C2_INV = pow(FMIX_C1, -1, 1 << 64), pow(FMIX_C2, -1, 1 << 64)
SENTINEL = (1 << 64) - 3  # oracle taxa at or above this are ambiguous positions
ACGT = np.frombuffer(b"ACGT", np.uint8)

# the streaming kernel's old visit caps, in cells: 32 766 sectors, 65 535 sectors, 32 766 filter records
CAPS = {"filter_sectors": 0x7FFE * 8, "sectors": 0xFFFF * 8, "filter_records": 0x7FFE * 32}

SMALL_CAP = (1 << 22) + 13
SMALL_RUN_START = SMALL_CAP - 600_000
SMALL_RUN_LEN = 1_250_000
BIG_CAP = (1 << 32) + (1 << 27) + 13
BIG_FREE_BYTES = 26 << 30


# ---------------------------------------------------------------------------------------------------------------
# the toolkit

def fmix64(x):
    x = np.atleast_1d(np.asarray(x, dtype=np.uint64)).copy()
    x ^= x >> U(33)
    x *= U(FMIX_C1)
    x ^= x >> U(33)
    x *= U(FMIX_C2)
    x ^= x >> U(33)
    return x


def fmix64_inv(h):
    """x ^= x >> 33 undoes itself (33 > 64 / 2); each multiply is undone by its constant's inverse mod 2^64"""
    x = np.atleast_1d(np.asarray(h, dtype=np.uint64)).copy()
    x ^= x >> U(33)
    x *= U(FMIX_C2_INV)
    x ^= x >> U(33)
    x *= U(FMIX_C1_INV)
    x ^= x >> U(33)
    return x


def filter_bits(ck):
    """nh_filter_hash: the miss filter's bit in each of its four partitions (64, 64, 64 and 32 bits)"""
    h = (np.asarray(ck, np.uint64) * U(0x9E3779B1)) & U(0xFFFFFFFF)
    h ^= h >> U(15)
    h = (h * U(0x85EBCA77)) & U(0xFFFFFFFF)
    h ^= h >> U(13)
    return h & U(63), (h >> U(6)) & U(63), (h >> U(12)) & U(63), (h >> U(18)) & U(31)


class KeyMaker:
    """Masked minimizers of the database's options and 35-base reads that carry them."""

    def __init__(self, oracle, opts, rng):
        self.oracle, self.opts, self.rng = oracle, opts, rng
        self.k, self.l = int(opts.k), int(opts.l)
        self.lmask = (1 << (2 * self.l)) - 1
        self.seed = int(opts.spaced_seed_mask) or self.lmask
        self.toggle = int(opts.toggle_mask) & self.lmask

    def valid(self, K):
        return (np.asarray(K, np.uint64) & U(~self.seed & MASK64)) == 0

    def rank(self, K):
        """the toggled value the window minimum compares: small wins"""
        return (np.asarray(K, np.uint64) ^ U(self.toggle)) & U(self.seed)

    def forward(self, n):
        """n valid keys with small toggled values, homes wherever fmix64 puts them"""
        r = self.rng.integers(0, 1 << 40, n, dtype=np.uint64)
        return np.unique((U(self.toggle) ^ r) & U(self.seed))

    def at_home(self, home, capacity, want=24):
        """valid keys K with fmix64(K) % capacity == home, the smallest toggled values first"""
        qmax = (MASK64 - home) // capacity
        out = np.zeros(0, np.uint64)
        for _ in range(40):
            q = self.rng.integers(0, qmax + 1, 1 << 18, dtype=np.uint64)
            K = fmix64_inv(U(home) + q * U(capacity))
            out = np.concatenate([out, K[self.valid(K)]])
            if len(out) >= want:
                break
        return out[np.argsort(self.rank(out), kind="stable")]

    def read(self, K, tries=24):
        """35 bases whose only k-mer position has minimizer K, or None"""
        K = int(K)
        free = ~self.seed & self.lmask
        for _ in range(tries):
            j = int(self.rng.integers(0, self.k - self.l + 1))
            v = K | (int(self.rng.integers(0, 1 << 62)) & free)
            codes = np.array([(v >> (2 * (self.l - 1 - i))) & 3 for i in range(self.l)], np.int64)
            seq = np.concatenate([ACGT[self.rng.integers(0, 4, j)], ACGT[codes],
                                  ACGT[self.rng.integers(0, 4, self.k - self.l - j)]])
            mins, amb = self.oracle.scan_positions(self.opts, bytes(seq))
            if len(mins) == 1 and amb[0] == 0 and int(mins[0]) == K:
                return seq
        return None


class Table:
    """A sparse kraken2 cell array: runs of blocker cells, planted keys, decoys.  Later writes win."""

    def __init__(self, capacity, value_bits, n_nodes, keymaker, rng):
        self.cap, self.vb, self.n_nodes = capacity, value_bits, n_nodes
        self.km, self.rng = keymaker, rng
        ckmax = (1 << (32 - value_bits)) - 1
        pool = {0, ckmax}
        while len(pool) < 8:
            pool.add(int(rng.integers(1, ckmax)))
        self.pool = np.array(sorted(pool), np.uint64)
        self.pool_bits = [set(b.tolist()) for b in filter_bits(self.pool)]
        self.used_ck = set(pool)
        self._idx, self._val = [], []
        self.busy = set()    # cells of short chains
        self.runs = []       # (start, length) of long runs
        self.slots = set()   # planted and decoy cells
        self.keys = []       # dict(K, home, ck, depth (None: miss), taxon, seq, tag)
        self.size = 0
        self._dense = None

    # -- cells
    def _write(self, idx, val):
        self._idx.append(np.asarray(idx, np.uint64) % U(self.cap))
        self._val.append(np.asarray(val, np.uint32))
        self._sorted = None

    def fill(self, start, length):
        """length blocker cells from start on (wrapping): valid taxa, compacted keys from the pool"""
        if length <= 0:
            return
        idx = (U(start) + np.arange(length, dtype=np.uint64)) % U(self.cap)
        ck = self.pool[self.rng.integers(0, len(self.pool), length)]
        tx = self.rng.integers(1, self.n_nodes, length).astype(np.uint64)
        self._write(idx, ((ck << U(self.vb)) | tx).astype(np.uint32))

    def finish(self):
        idx = np.concatenate(self._idx)[::-1]
        val = np.concatenate(self._val)[::-1]
        u, first = np.unique(idx, return_index=True)  # the last write of every cell
        self._sorted = (u, val[first])
        self.size = len(u)
        return self

    def get(self, idx):
        idx = np.asarray(idx, np.uint64)
        if self._dense is not None:
            return self._dense[idx]
        u, v = self._sorted
        pos = np.minimum(np.searchsorted(u, idx), len(u) - 1)
        return np.where(u[pos] == idx, v[pos], 0).astype(np.uint32)

    def dense(self, out=None):
        u, v = self._sorted
        out = np.zeros(self.cap, np.uint32) if out is None else out
        out[u] = v
        self._dense = out
        return out

    def walk(self, K, limit):
        """(depth, value) of the first cell from K's home that is empty or holds its compacted key, within limit"""
        h = int(fmix64(K)[0])
        home, ck = h % self.cap, h >> (32 + self.vb)
        step = 1 << 16
        for base in range(0, limit, step):
            n = min(step, limit - base)
            c = self.get((U(home + base) + np.arange(n, dtype=np.uint64)) % U(self.cap))
            term = ((c & np.uint32((1 << self.vb) - 1)) == 0) | ((c >> np.uint32(self.vb)) == ck)
            if term.any():
                j = int(np.argmax(term))
                return base + j, int(c[j] & ((1 << self.vb) - 1))
        return None, None

    # -- keys
    def home_ck(self, K):
        h = fmix64(K)
        return (h % U(self.cap)).astype(np.int64), (h >> U(32 + self.vb)).astype(np.int64)

    def usable(self, K, ck):
        """a fresh compacted key that the pool's filter bits do not cover (so that runs of blockers are no
        false positives of the miss filter for it), and a read that carries K"""
        if ck in self.used_ck:
            return None
        bits = [int(b[0]) for b in filter_bits(np.array([ck], np.uint64))]
        if all(b in s for b, s in zip(bits, self.pool_bits)):
            return None
        return self.km.read(K)

    def free(self, a, n):
        """cells a - 1 .. a + n free of short chains and long runs"""
        for s, ln in self.runs:
            if (a - 1 - s) % self.cap < ln or (s - (a - 1)) % self.cap < n + 2:
                return False
        return not any(((a + i) % self.cap) in self.busy for i in range(-1, n + 1))

    def plant(self, K, seq, depth, tag, taxon=None):
        home, ck = (int(x[0]) for x in self.home_ck(K))
        taxon = int(self.rng.integers(1, self.n_nodes)) if taxon is None else taxon
        self.used_ck.add(ck)
        if depth is not None:
            slot = (home + depth) % self.cap
            assert slot not in self.slots
            self.slots.add(slot)
            self._write([slot], [(ck << self.vb) | taxon])
        self.keys.append(dict(K=int(K), home=home, ck=ck, depth=depth, taxon=taxon if depth is not None else 0,
                              seq=seq, tag=tag))
        return self.keys[-1]

    def plant_short(self, K, depth, tag, lo, hi):
        """K in a chain of its own: depth blockers from its home, then K; None if it does not fit in [lo, hi)"""
        home, ck = (int(x[0]) for x in self.home_ck(K))
        if not (lo <= home and home + depth + 1 < hi) or not self.free(home, depth + 1):
            return None
        seq = self.usable(K, ck)
        if seq is None:
            return None
        self.busy.update(range(home, home + depth + 1))
        self.fill(home, depth)
        return self.plant(K, seq, depth, tag)

    def decoy(self, key, cell):
        """a cell with key's compacted key and another taxon, off the key's chain"""
        cell %= self.cap
        if cell in self.slots:
            return False
        other = 1 + (key["taxon"] % (self.n_nodes - 1))
        self.slots.add(cell)
        self._write([cell], [(key["ck"] << self.vb) | other])
        return True


def _run_offset(cell, start, cap):
    return (cell - start) % cap


def _sweep(km, table, targets, lo_hi, tag, n_cand=1 << 19):
    """For each (depth, tag) in targets, a forward key whose home h satisfies lo_hi(h, depth)."""
    cand = km.forward(n_cand)
    homes, cks = table.home_ck(cand)
    order = table.rng.permutation(len(cand))
    used = set()
    out = []
    for depth, t in targets:
        for i in order:
            if i in used or not lo_hi(int(homes[i]), depth):
                continue
            slot = (int(homes[i]) + depth) % table.cap if depth is not None else None
            if slot is not None and slot in table.slots:
                continue
            seq = table.usable(cand[i], int(cks[i]))
            if seq is None:
                used.add(i)
                continue
            used.add(i)
            out.append(table.plant(cand[i], seq, depth, t))
            break
        else:
            raise AssertionError(f"no key for {tag} depth {depth}")
    return out


def _exact(km, table, homes_depths, tag):
    """keys whose homes are exact: made with fmix64_inv"""
    out = []
    for home, depth in homes_depths:
        while (home + depth) % table.cap in table.slots:  # neighbouring homes: the next free slot
            depth += 1
        for K in km.at_home(home, table.cap):
            ck = int(table.home_ck(K)[1][0])
            seq = table.usable(K, ck)
            if seq is not None:
                out.append(table.plant(K, seq, depth, tag))
                break
        else:
            raise AssertionError(f"no key for home {home}")
    return out


def build_small(oracle, opts, n_nodes, value_bits, seed):
    """Table 1: capacity 2^22 + 13 and one run of 1.25 M occupied cells across the table's end."""
    rng = np.random.default_rng(seed)
    km = KeyMaker(oracle, opts, rng)
    cap, rs, rl = SMALL_CAP, SMALL_RUN_START, SMALL_RUN_LEN
    t = Table(cap, value_bits, n_nodes, km, rng)
    t.fill(rs, rl)
    t.runs.append((rs, rl))
    depths = list(range(41)) + [1 << p for p in range(6, 21)]
    for c in CAPS.values():
        depths += [c + d for d in range(-24, 25, 3)]
    targets = [(d, "run") for d in depths]

    def in_run(h, d):
        return _run_offset(h, rs, cap) + d + 64 < rl

    # homes in the partial last sector (5 cells), the partial last filter block (13 cells), and just before them
    edge = [cap - 1, cap - 2, cap - 5, cap - 6, cap - 13, cap - 14]
    edge_depths = [0, 1, 4, 5, 12, 13, 40, 1000, CAPS["filter_sectors"] + 9, CAPS["sectors"] + 9]
    keys = _exact(km, t, [(h, d) for h in edge for d in edge_depths[(edge.index(h) % 3)::3]], "edge")
    keys += _sweep(km, t, targets, in_run, "run")
    # true misses: homes near the run's end, and homes whose walk to the run's end passes every cap
    keys += _sweep(km, t, [(None, "miss_end")] * 12,
                   lambda h, d: rl - 3000 <= _run_offset(h, rs, cap) < rl, "miss_end")
    keys += _sweep(km, t, [(None, "miss_far")] * 6,
                   lambda h, d: _run_offset(h, rs, cap) < rl - CAPS["filter_records"] - 4000, "miss_far")
    # first match wins: decoys after the slot and before the home
    for i, k in enumerate(keys):
        if k["depth"] is None or i % 3:
            continue
        after = (k["home"] + k["depth"] + 1 + int(rng.integers(0, 30))) % cap
        if _run_offset(after, rs, cap) < rl:
            t.decoy(k, after)
        if _run_offset(k["home"], rs, cap) >= 1:
            t.decoy(k, k["home"] - 1)
    # ordinary hits in short chains of their own, away from the run
    hits = []
    cand = km.forward(1 << 14)
    for K in cand:
        k = t.plant_short(K, int(rng.integers(0, 4)), "hit", rs + rl - cap + 1000, rs - 1000)
        if k is not None:
            hits.append(k)
        if len(hits) == 48:
            break
    t.finish()
    return t, keys, hits


def build_big(oracle, opts, n_nodes, value_bits, seed):
    """Table 2: capacity 2^32 + 2^27 + 13."""
    rng = np.random.default_rng(seed)
    km = KeyMaker(oracle, opts, rng)
    cap = BIG_CAP
    t = Table(cap, value_bits, n_nodes, km, rng)
    keys = []
    # across cell 2^32 = sector 2^29 = filter block 2^27: homes below it, slots at and after it
    cross0 = (1 << 32) - 2048
    t.fill(cross0, 4096)
    t.runs.append((cross0, 4096))
    below = [1, 2, 3, 7, 8, 9, 31, 32, 33, 40, 1000]
    keys += _exact(km, t, [((1 << 32) - x, x + j * 300 + i) for i, x in enumerate(below) for j in range(4)], "cross")
    # from the partial last sector and block to cell 0
    wrap0 = cap - 2048
    t.fill(wrap0, 4096)
    t.runs.append((wrap0, 4096))
    ends = [1, 2, 5, 6, 13, 14, 40]
    keys += _exact(km, t, [(cap - x, x + j * 300 + i) for i, x in enumerate(ends) for j in range(4)], "wrap")
    keys += _exact(km, t, [(cap - 40, 3), (cap - 13, 7), (cap - 14, 12)], "end")
    # homes spread over [2^32, capacity), and a control set below 2^31, each in a chain of its own
    cand = km.forward(1 << 18)
    homes, _ = t.home_ck(cand)
    for lo, hi, n, tag in (((1 << 32) + 4096, cap - 4096, 2500, "high"), (4096, 1 << 31, 300, "low")):
        pick = cand[(homes >= lo) & (homes < hi)]
        got = 0
        for i, K in enumerate(pick):
            depth = int(rng.integers(0, 41)) if i % 10 else int(rng.integers(41, 300))
            if i % 25 == 24:  # a miss: blockers from the home on, then an empty cell
                home, ck = (int(x[0]) for x in t.home_ck(K))
                if home + depth + 1 < hi and t.free(home, depth + 1):
                    seq = t.usable(K, ck)
                    if seq is not None:
                        t.busy.update(range(home, home + depth + 1))
                        t.fill(home, depth)
                        keys.append(t.plant(K, seq, None, tag + "_miss"))
                continue
            k = t.plant_short(K, depth, tag, lo, hi)
            if k is not None:
                keys.append(k)
                got += 1
            if got == n:
                break
    t.finish()
    return t, keys


def reads_for(keys, hits):
    """one 35-base read per key, then [ordinary hit] N*64 [key] for the keys of long chains"""
    seqs = [k["seq"] for k in keys]
    gap = np.full(64, ord("N"), np.uint8)
    multi = [k for k in keys if k["depth"] is None or k["depth"] >= 200 or k["tag"] in ("edge", "wrap", "cross")]
    for i, k in enumerate(multi):
        seqs.append(np.concatenate([hits[i % len(hits)]["seq"], gap, k["seq"]]))
    return seqs


def reach(t, keys):
    """what the planted keys exercise, counted from the design"""
    out = {"keys": len(keys), "misses": sum(k["depth"] is None for k in keys)}
    planted = [k for k in keys if k["depth"] is not None]
    out["homes_at_or_above_2^32"] = sum(k["home"] >= 1 << 32 for k in keys)
    out["chains_crossing_2^32"] = sum(k["home"] < 1 << 32 <= k["home"] + k["depth"] for k in planted)
    out["chains_crossing_the_wrap"] = sum(k["home"] + k["depth"] >= t.cap for k in planted)
    for name, c in CAPS.items():
        out[f"beyond_{name}_{c}"] = sum(k["depth"] > c for k in planted)
    return out


# ---------------------------------------------------------------------------------------------------------------
# the databases' images

@pytest.fixture(scope="module")
def base(oracle, tmp_path_factory):
    """cfg1 taxonomy (24 nodes: value_bits 5, the least the miss filter accepts) and kraken2's default options"""
    tax = [oracle.TaxSpec(*r) for r in synth.TAXONOMY_CFG1]
    db = oracle.OracleDb.build([], tax, capacity=8)
    d = str(tmp_path_factory.mktemp("edges_base"))
    db.save(d)
    with open(os.path.join(d, "opts.k2d"), "rb") as f:
        opts_b = f.read()
    with open(os.path.join(d, "taxo.k2d"), "rb") as f:
        taxo_b = f.read()
    assert int(db.cht.value_bits) == 5
    return db, opts_b, taxo_b


_SMALL = {}


def small(oracle, base, vb):
    if vb not in _SMALL:
        db = base[0]
        t, keys, hits = build_small(oracle, db.opts, int(db.tax.node_count), vb, seed=100 + vb)
        _SMALL[vb] = (t, keys, hits)
    return _SMALL[vb]


def _oracle_on(oracle, base, t, cells):
    o = oracle.OracleDb.from_arrays(base[0].opts, base[0].tax, cells, t.cap, t.size, t.vb)
    o.min_hit_groups, o.confidence = 1, 0.0
    return o


# ---------------------------------------------------------------------------------------------------------------
# CPU: the toolkit holds

def test_fmix64_inv_inverts_fmix64(oracle):
    rng = np.random.default_rng(1)
    x = np.concatenate([rng.integers(0, MASK64, 4096, dtype=np.uint64, endpoint=True),
                        np.array([0, 1, MASK64, 1 << 63, (1 << 62) - 1], np.uint64)])
    np.testing.assert_array_equal(fmix64_inv(fmix64(x)), x)
    np.testing.assert_array_equal(fmix64(fmix64_inv(x)), x)
    for v in x[:64].tolist() + [0, MASK64]:
        assert int(fmix64(v)[0]) == oracle.fmix64(v)


@pytest.mark.parametrize("vb", [5, 12])
def test_small_table_design(oracle, base, vb):
    """every read carries its key; every key's home, compacted key and depth are as designed; the oracle finds
    each planted taxon and misses past the run's end"""
    t, keys, hits = small(oracle, base, vb)
    opts = base[0].opts
    for k in keys + hits:
        mins, amb = oracle.scan_positions(opts, bytes(k["seq"]))
        assert len(mins) == 1 and amb[0] == 0 and int(mins[0]) == k["K"]
        h = oracle.fmix64(k["K"])
        assert (h % t.cap, h >> (32 + vb)) == (k["home"], k["ck"])
    for k in keys + hits:
        limit = (k["depth"] if k["depth"] is not None else SMALL_RUN_LEN) + 2
        depth, val = t.walk(k["K"], limit)
        if k["depth"] is None:
            assert val == 0 and depth is not None, k["tag"]
        else:
            assert (depth, val) == (k["depth"], k["taxon"]), (k["tag"], k["depth"])
    o = _oracle_on(oracle, base, t, t.dense())
    for k in keys + hits:
        assert o.get(k["K"]) == k["taxon"], (k["tag"], k["depth"])
    r = reach(t, keys)
    assert r["chains_crossing_the_wrap"] >= 20
    assert r["misses"] >= 18
    for name, c in CAPS.items():
        assert r[f"beyond_{name}_{c}"] >= (8 if c == CAPS["filter_records"] else 20), (name, r)
    # decoys: same compacted key after the slot or before the home
    assert len(t.slots) >= len([k for k in keys if k["depth"] is not None]) + 40
    # blockers with compacted keys 0 and all-ones sit on the run
    run = t.get((U(SMALL_RUN_START) + np.arange(100_000, dtype=np.uint64)) % U(t.cap))
    assert (run & np.uint32((1 << vb) - 1)).all()
    cks = set((run >> np.uint32(vb)).tolist())
    assert {0, (1 << (32 - vb)) - 1} <= cks


def test_big_table_design(oracle, base):
    """The 2^32 + 2^27 + 13 design, checked on its sparse cells (the dense 17.7 GB array is made on the GPU
    machine only)."""
    t, keys = _big(oracle, base)
    opts = base[0].opts
    for k in keys[::7] + [k for k in keys if k["tag"] in ("cross", "wrap", "end")]:
        mins, amb = oracle.scan_positions(opts, bytes(k["seq"]))
        assert len(mins) == 1 and amb[0] == 0 and int(mins[0]) == k["K"]
        h = oracle.fmix64(k["K"])
        assert (h % t.cap, h >> 37) == (k["home"], k["ck"])
    for k in keys:
        depth, val = t.walk(k["K"], (k["depth"] if k["depth"] is not None else 400) + 2)
        if k["depth"] is None:
            assert val == 0
        else:
            assert (depth, val) == (k["depth"], k["taxon"]), (k["tag"], k["home"], k["depth"])
    r = reach(t, keys)
    assert r["homes_at_or_above_2^32"] >= 2500
    assert r["chains_crossing_2^32"] >= 40
    assert r["chains_crossing_the_wrap"] >= 25
    assert sum(k["home"] < 1 << 31 for k in keys) >= 250
    assert sum(k["home"] >= (1 << 32) and k["depth"] is None for k in keys) >= 50


_BIG = {}


def _big(oracle, base):
    if "t" not in _BIG:
        db = base[0]
        _BIG["t"] = build_big(oracle, db.opts, int(db.tax.node_count), 5, seed=7)
    return _BIG["t"]


# ---------------------------------------------------------------------------------------------------------------
# GPU

def _device_classify(sess, bases, offsets, n_units):
    import torch
    d_bases = torch.from_numpy(np.concatenate([bases, np.zeros(64, np.uint8)])).cuda()
    d_off = torch.from_numpy(offsets.astype(np.int64)).cuda()
    d_call = torch.full((max(n_units, 1),), -1, dtype=torch.int32, device="cuda")
    d_keep = torch.full((max(n_units, 1),), 7, dtype=torch.uint8, device="cuda")
    sess.classify_device(d_bases.data_ptr(), d_off.data_ptr(), len(offsets) - 1, int(offsets[-1]),
                         d_call.data_ptr(), d_keep.data_ptr())
    sess.sync()
    return d_call.cpu().numpy().view(np.uint32)[:n_units]


def _rle(taxa, ext_ids):
    out = []
    for x in taxa:
        if x >= SENTINEL:
            continue
        e = int(ext_ids[x])
        if out and out[-1][0] == e:
            out[-1][1] += 1
        else:
            out.append([e, 1])
    return out


def _failures(want, call, dbg, what):
    """the reads whose call, total_kmers or hit_groups differ from the oracle's, with their keys' designs"""
    icall, tk, hg = dbg if dbg is not None else (None, None, None)
    bad = call != want["ext"]
    if dbg is not None:
        bad |= (icall != want["call"]) | (tk != want["total_kmers"]) | (hg != want["hit_groups"])
    return [(what, int(i)) for i in np.flatnonzero(bad)]


def _describe(bad, labels):
    return "; ".join(f"{w} read {i} ({labels[i]})" for w, i in bad[:40]) + (f" ... {len(bad)} in all" if len(bad) > 40
                                                                            else "")


def _run_entry_points(gdb, o, t, keys, seqs, labels, want, switch, monkeypatch, emit=True):
    from nohuman_b200 import Session
    for var in ("NH_FILTER_MODE", "NH_LEGACY_KERNELS"):
        monkeypatch.delenv(var, raising=False)
    if switch.startswith("filter"):
        monkeypatch.setenv("NH_FILTER_MODE", switch[-1])
    elif switch == "legacy":
        monkeypatch.setenv("NH_LEGACY_KERNELS", "1")
    fused = switch != "legacy"
    bases, offsets = synth.pack(seqs)
    n = len(seqs)
    cap = dict(max_batch_bases=len(bases) + 4096, max_batch_seqs=n + 2)
    bad = []
    with Session(gdb, confidence=0.0, minimum_hit_groups=1, **cap) as sess:
        call, keep, st = sess.classify(bases, offsets)
        assert st.fused_kernel == (2 if fused else 0)
        bad += _failures(want, call, sess.debug_last_batch(n), "classify")
        np.testing.assert_array_equal(keep, (want["ext"] == 0).astype(np.uint8))
        bad += _failures(want, _device_classify(sess, bases, offsets, n), None, "classify_device")
        if fused:
            call, _, _ = sess.classify_packed(bases, offsets, threads=3)
            bad += _failures(want, call, sess.debug_last_batch(n), "classify_packed")
            for threads in (1, 5):
                call, _, _ = sess.classify_pack(bases, offsets, threads=threads)
                bad += _failures(want, call, sess.debug_last_batch(n), f"classify_pack/{threads}")
        ks = np.array([k["K"] for k in keys], np.uint64)
        got = sess.debug_probe(ks)
        exp = np.array([k["taxon"] for k in keys], np.uint32)
        np.testing.assert_array_equal(exp, [o.get(int(K)) for K in ks])
        bad += [("debug_probe", int(i)) for i in np.flatnonzero(got != exp)]
    if emit and not switch.startswith("filter"):
        ext_ids = o.external_ids()
        with Session(gdb, confidence=0.0, minimum_hit_groups=1, emit_runs=True, **cap) as sess:
            call, _, st = sess.classify(bases, offsets)
            assert st.fused_kernel == (2 if fused else 0)
            bad += _failures(want, call, sess.debug_last_batch(n), "emit_runs classify")
            first, ext, ln = sess.last_batch_runs(n, int(offsets[-1]))
        for i in range(n):
            runs = [[int(ext[j]), int(ln[j])] for j in range(int(first[i]), int(first[i + 1]))]
            merged = []
            for e, c in runs:
                if merged and merged[-1][0] == e:
                    merged[-1][1] += c
                else:
                    merged.append([e, c])
            if merged != _rle(o.classify_one(bytes(seqs[i]), want_taxa=True)["taxa"], ext_ids):
                bad.append(("emit_runs per lookup", i))
    return bad


def _labels(keys, seqs):
    lab = [f"{k['tag']} home {k['home']} depth {k['depth']}" for k in keys]
    long = [k for k in keys if k["depth"] is None or k["depth"] >= 200 or k["tag"] in ("edge", "wrap", "cross")]
    lab += [f"hit + {k['tag']} home {k['home']} depth {k['depth']}" for k in long]
    assert len(lab) == len(seqs)
    return lab


SMALL_SWITCHES = ["plain", "filter0", "filter1", "filter2", "filter3", "legacy"]


@gpu
@pytest.mark.parametrize("switch", SMALL_SWITCHES)
@pytest.mark.parametrize("vb", [5, 12])
def test_long_runs_on_a_small_table(oracle, base, vb, switch, monkeypatch):
    """Chains up to 1.1 M cells long, across the table's end, around every old visit cap: every entry point and
    filter policy against the oracle, per read and (emit_runs) per lookup."""
    from nohuman_b200 import Database
    t, keys, hits = small(oracle, base, vb)
    cells = t.dense()
    o = _oracle_on(oracle, base, t, cells)
    seqs = reads_for(keys, hits)
    labels = _labels(keys, seqs)
    bases, offsets = synth.pack(seqs)
    want = o.classify_batch(bases, offsets)
    assert (want["call"][:len(keys)] == [k["taxon"] for k in keys]).all()
    r = reach(t, keys)
    print(f"\nreach small vb={vb}: {r}")
    assert r["beyond_filter_records_1048512"] >= 8 and r["chains_crossing_the_wrap"] >= 20
    with Database.from_memory(base[1], base[2], (t.cap, t.size, 32 - vb, vb), cells, device=0) as gdb:
        assert int(gdb.info.capacity) == SMALL_CAP and int(gdb.info.value_bits) == vb
        assert gdb.info.filter_bytes == ((SMALL_CAP + 31) // 32) * 32
        bad = _run_entry_points(gdb, o, t, keys, seqs, labels, want, switch, monkeypatch)
    assert not bad, _describe(bad, labels)


def _big_memory_or_skip():
    import torch
    free, _ = torch.cuda.mem_get_info()
    if free < BIG_FREE_BYTES:
        pytest.skip(f"the 2^32 + 2^27 + 13 cell table needs about 26 GB of free device memory, {free / 2**30:.1f} "
                    "GiB are free (the device is shared)")


@pytest.fixture(scope="module")
def big_world(oracle, base):
    """the dense host image of table 2 (np.zeros: only the planted pages are ever written) and the oracle on it"""
    _big_memory_or_skip()
    t, keys = _big(oracle, base)
    try:
        cells = np.zeros(t.cap, np.uint32)
    except MemoryError:
        pytest.skip("no host memory for a 17.7 GB image of the table")
    t.dense(cells)
    o = _oracle_on(oracle, base, t, cells)
    hits = [k for k in keys if k["tag"] == "low" and k["depth"] is not None][:48]
    seqs = reads_for(keys, hits)
    bases, offsets = synth.pack(seqs)
    want = o.classify_batch(bases, offsets)
    assert (want["call"][:len(keys)] == [k["taxon"] for k in keys]).all()
    yield t, keys, cells, o, seqs, want
    del o
    del cells


BIG_SWITCHES = ["plain", "filter0", "filter1", "filter2", "legacy"]


@gpu
def test_table_past_2_to_the_32_cells(oracle, base, big_world, monkeypatch):
    """Homes above cell 2^32, filter records past byte 4 GiB, chains across cell 2^32 and across the wrap from the
    partial last sector: every entry point and filter policy against the oracle; then the same table adopted from
    a device copy."""
    import torch
    from nohuman_b200 import Database
    _big_memory_or_skip()
    t, keys, cells, o, seqs, want = big_world
    labels = _labels(keys, seqs)
    r = reach(t, keys)
    print(f"\nreach big: {r}")
    assert r["homes_at_or_above_2^32"] >= 2500 and r["chains_crossing_2^32"] >= 40
    assert r["chains_crossing_the_wrap"] >= 25
    bad = []
    with Database.from_memory(base[1], base[2], (t.cap, t.size, 27, 5), cells, device=0) as gdb:
        assert int(gdb.info.capacity) == BIG_CAP
        assert gdb.info.filter_bytes == ((BIG_CAP + 31) // 32) * 32 > 1 << 32
        for switch in BIG_SWITCHES:
            bad += [(f"{switch} {w}", i) for w, i in
                    _run_entry_points(gdb, o, t, keys, seqs, labels, want, switch, monkeypatch,
                                      emit=switch in ("plain", "legacy"))]
    assert not bad, _describe(bad, labels)
    # the same table adopted from a torch allocation that only the planted cells were copied into
    free, _ = torch.cuda.mem_get_info()
    if free < BIG_FREE_BYTES:
        return
    u, v = t._sorted
    words = ((t.cap + 31) // 32) * 32
    dev = torch.zeros(words, dtype=torch.int32, device="cuda")
    dev[torch.from_numpy(u.astype(np.int64)).cuda()] = torch.from_numpy(v.view(np.int32)).cuda()
    torch.cuda.synchronize()
    try:
        with Database.from_memory(base[1], base[2], (t.cap, t.size, 27, 5), dev.data_ptr(), device=0,
                                  cells_on_device=True) as gdb:
            bad = [("adopted " + w, i) for w, i in
                   _run_entry_points(gdb, o, t, keys, seqs, labels, want, "plain", monkeypatch, emit=False)]
    finally:
        del dev
        torch.cuda.empty_cache()
    assert not bad, _describe(bad, labels)
