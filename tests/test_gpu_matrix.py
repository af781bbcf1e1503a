"""Every streaming-kernel instantiation, entry point and scoring boundary against the oracle.

The dispatch in nh_launch_stream picks one of the k_stream_classify instantiations that
nh_kernels_init registers from the database (k / l / revcom_version), the entry point (ASCII,
packed, per-position debug), emit_runs and the miss-filter policy.  This module runs each of them,
the warp-per-tile kernels and the three scoring kernels on inputs where a subtly wrong kernel gives
a different per-unit answer than the CPU oracle:
  1. an instantiation x entry-point x switch matrix on five databases (plus a CPU guard that every
     registered instantiation has a parity case listed in COVERED),
  2. minimum_hit_groups and confidence values that sit exactly on a scoring edge,
  3. units with exactly 8/9, 64/65 and 16384/16385 distinct taxa, and taxonomies of exactly
     8192 / 8193 nodes (NH_SMEM_PARENT_MAX),
  4. one session fed batches of changing shape through every entry point, and two sessions on one
     database in flight at once.
Oracle answers are computed once per (database, batch, paired, confidence, minimum_hit_groups)."""
import os
import re

import numpy as np
import pytest

import synth

gpu = pytest.mark.gpu
JUNK = b"NnRY-.\0*"
SENTINEL = (1 << 64) - 3  # oracle taxa at or above this are ambiguous / skipped positions

# ---------------------------------------------------------------------------------------------
# instantiation -> the parity cases that run it.  <W, KL, DBG, REV0, EMIT, PACKED, FILTER>
F, T = False, True
COVERED = {
    (5, 1, F, F, F, F, 0): ["test_entry_points[default-filter0]", "test_entry_points[smalltax-plain]"],
    (5, 1, F, F, T, F, 0): ["test_entry_points[default-plain]", "test_entry_points[smalltax-plain]"],
    (5, 0, F, F, F, F, 0): ["test_entry_points[k25-plain]"],
    (5, 0, F, T, F, F, 0): ["test_entry_points[rev0-plain]"],
    (5, 0, T, F, F, F, 0): ["test_entry_points[default-plain]", "test_entry_points[rev0-plain]"],
    (5, 0, F, F, T, F, 0): ["test_entry_points[k25-plain]", "test_entry_points[k25-lane_taxa_1]"],
    (5, 0, F, T, T, F, 0): ["test_entry_points[rev0-plain]", "test_entry_points[rev0-lane_taxa_1]"],
    (5, 1, F, F, F, T, 0): ["test_entry_points[default-filter0]", "test_entry_points[smalltax-plain]"],
    (5, 0, F, F, F, T, 0): ["test_entry_points[k25-plain]", "test_entry_points[k25-lane_taxa_1]"],
    (5, 0, F, T, F, T, 0): ["test_entry_points[rev0-plain]", "test_entry_points[rev0-lane_taxa_1]"],
    (5, 1, F, F, F, F, 1): ["test_entry_points[default-filter1]"],
    (5, 1, F, F, F, F, 2): ["test_entry_points[default-filter2]"],
    (5, 1, F, F, F, F, 3): ["test_entry_points[default-filter3]", "test_entry_points[default-plain]"],
    (5, 1, F, F, F, T, 1): ["test_entry_points[default-filter1]"],
    (5, 1, F, F, F, T, 2): ["test_entry_points[default-filter2]"],
    (5, 1, F, F, F, T, 3): ["test_entry_points[default-filter3]", "test_entry_points[default-plain]"],
}

DB_NAMES = ["default", "rev0", "k25", "k31", "smalltax"]
SWITCHES = {
    "plain": {},
    "filter0": {"NH_FILTER_MODE": "0"},
    "filter1": {"NH_FILTER_MODE": "1"},
    "filter2": {"NH_FILTER_MODE": "2"},
    "filter3": {"NH_FILTER_MODE": "3"},
    "lane_taxa_1": {"NH_TEST_LANE_TAXA": "1"},   # every unit with a hit overflows into k_score_big
    "tile_pos_64": {"NH_FUSED_TILE_POS": "64"},  # long units are deferred to k_score
    "legacy": {"NH_LEGACY_KERNELS": "1"},        # warp-per-tile kernels
}
ENTRY_CASES = [(d, s) for d in DB_NAMES for s in ("plain", "lane_taxa_1", "tile_pos_64", "legacy")]
ENTRY_CASES += [("default", f"filter{m}") for m in range(4)]


def _parse_registered(src: str):
    out = []
    for m in re.finditer(r"NH_SET_SMEM\(\(k_stream_classify<([^>]*)>\)", src):
        args = [a.strip() for a in m.group(1).split(",")]
        out.append(tuple(int(a) if a.isdigit() else a == "true" for a in args))
    return out


def test_every_registered_instantiation_has_a_parity_case():
    """CPU-only: whoever registers another k_stream_classify specialisation adds its case to COVERED."""
    src_path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                            "nohuman_b200", "csrc", "nh_kernels.cu")
    with open(src_path) as f:
        registered = _parse_registered(f.read())
    assert len(registered) >= 16
    missing = [r for r in registered if r not in COVERED]
    assert not missing, f"registered instantiations without a parity case in COVERED: {missing}"
    stale = [c for c in COVERED if c not in registered]
    assert not stale, f"COVERED lists instantiations nh_kernels_init no longer registers: {stale}"
    ids = {f"test_entry_points[{d}-{s}]" for d, s in ENTRY_CASES}
    for inst, tests in COVERED.items():
        assert tests, inst
        for t in tests:
            assert t.split("[")[0] in globals(), t
            assert "[" not in t or t in ids, t


# ---------------------------------------------------------------------------------------------
# databases and batches

SMALL_TAXONOMY = [(1, 1, "root", "no rank"), (131567, 1, "cellular organisms", "no rank"),
                  (2759, 131567, "Eukaryota", "superkingdom"), (9606, 2759, "Homo sapiens", "species"),
                  (2, 131567, "Bacteria", "superkingdom"), (561, 2, "Escherichia", "genus"),
                  (562, 561, "Escherichia coli", "species"), (564, 561, "Escherichia fergusonii", "species"),
                  (1423, 2, "Bacillus subtilis", "species")]
DB_OPTS = {
    "default": (dict(), 1),
    "rev0": (dict(), 0),
    "k25": (dict(k=25, l=21, spaces=3), 1),
    "k31": (dict(k=31, l=31, spaces=0), 1),
    "smalltax": (dict(), 1),
}


def _adversarial(genomes, k, seed):
    """2x150 bp pairs with N runs, lower case and junk bytes; three-taxon chimeras; empty reads and
    reads of length 1, k-1, k, k+1; lengths at the borders of 508- and 252-position tiles; ONT reads."""
    rng = np.random.default_rng(seed)
    g = dict(genomes)
    seqs = synth.illumina_reads(genomes, 300, 150, seed=seed, paired=True, n_rate=0.3)
    for i in range(0, len(seqs), 5):
        r = seqs[i].copy()
        r[20:20 + int(rng.integers(1, 12))] = ord("N")
        r[60:90] |= 0x20
        r[int(rng.integers(95, 150))] = JUNK[i % len(JUNK)]
        seqs[i] = r
    for i in range(40):
        seqs.append(np.concatenate([g[9606][i * 40:i * 40 + 75], g[562][i * 30:i * 30 + 75], g[1423][i * 20:i * 20 + 90]]))
    src = g[9606]
    for L in (0, 1, k - 1, k, k + 1, 0):
        o = int(rng.integers(0, len(src) - L - 1))
        seqs.append(src[o:o + L].copy())
    for tp, tiles in ((508, (1, 2, 3, 32)), (252, (1, 2, 33))):
        for nt in tiles:
            for d in (-1, 0, 1):
                L = nt * tp + k - 1 + d
                o = int(rng.integers(0, len(src) - L - 1))
                seqs.append(src[o:o + L].copy())
    seqs += synth.ont_reads(genomes, 6, seed=seed + 1, n50=6000, max_len=20_000)
    r = g[562][500:1400].copy()
    r[100:140] = ord("N"); r[300] = ord("n"); r[400:600] |= 0x20; r[700] = 0; r[701] = ord("*")
    seqs.append(r)
    if len(seqs) % 2:
        seqs.append(seqs[3][:100].copy())
    return seqs


def _long_reads(genomes, seed):
    return synth.ont_reads(genomes, 24, seed=seed, n50=3000, max_len=12_000, min_len=1200)


def _rle(taxa, ext_ids):
    """oracle positions without the ambiguous ones, run-length encoded on the external id"""
    out = []
    for t in taxa:
        if t >= SENTINEL:
            continue
        e = int(ext_ids[t])
        if out and out[-1][0] == e:
            out[-1][1] += 1
        else:
            out.append([e, 1])
    return out


class World:
    def __init__(self, oracle, tmp):
        self.oracle, self.tmp = oracle, tmp
        self.dbs, self.paths, self.gdbs, self.batches, self._want, self._runs = {}, {}, {}, {}, {}, {}

    def db(self, name):
        if name not in self.dbs:
            o = self.oracle
            kw, rev = DB_OPTS[name]
            opts = o.default_options(**kw)
            opts.revcom_version = rev
            genomes = synth.cfg1_genomes(seed=3, scale=0.004)
            rows = SMALL_TAXONOMY if name == "smalltax" else synth.TAXONOMY_CFG1
            db = o.OracleDb.build([(t, bytes(gg)) for t, gg in genomes], [o.TaxSpec(*t) for t in rows], opts=opts)
            db.genomes = genomes
            path = str(self.tmp / name)
            db.save(path)
            self.dbs[name], self.paths[name] = db, path
        return self.dbs[name]

    def gdb(self, name):
        if name not in self.gdbs:
            from nohuman_b200 import Database
            self.db(name)
            self.gdbs[name] = Database.open(self.paths[name], 0)
        return self.gdbs[name]

    def batch(self, dbname, kind):
        key = (dbname, kind)
        if key not in self.batches:
            db = self.db(dbname)
            k = int(db.opts.k)
            if kind == "adv":
                seqs = _adversarial(db.genomes, k, seed=61)
            elif kind == "long":
                seqs = _long_reads(db.genomes, seed=62)
            elif kind == "pairs":
                seqs = synth.illumina_reads(db.genomes, 500, 150, seed=63, paired=True, n_rate=0.2)
            elif kind == "one":
                seqs = [db.genomes[1][1][1000:1180].copy()]
            elif kind == "onepair":
                seqs = [db.genomes[1][1][1000:1150].copy(), synth.revcomp(db.genomes[1][1][1200:1350])]
            else:
                raise KeyError(kind)
            self.batches[key] = (seqs,) + synth.pack(seqs)
        return self.batches[key]

    def want(self, dbname, kind, paired, conf, mhg=2):
        key = (dbname, kind, paired, float(conf), mhg)
        if key not in self._want:
            db = self.db(dbname)
            _, bases, offsets = self.batch(dbname, kind)
            db.confidence, db.min_hit_groups = float(conf), mhg
            self._want[key] = db.classify_batch(bases, offsets, paired=paired)
            db.confidence, db.min_hit_groups = 0.0, 2
        return self._want[key]

    def runs(self, dbname, kind):
        key = (dbname, kind)
        if key not in self._runs:
            db = self.db(dbname)
            seqs = self.batch(dbname, kind)[0]
            ext_ids = db.external_ids()
            self._runs[key] = [_rle(db.classify_one(bytes(s), want_taxa=True)["taxa"], ext_ids) for s in seqs]
        return self._runs[key]

    def close(self):
        for g in self.gdbs.values():
            g.close()


@pytest.fixture(scope="module")
def world(oracle, tmp_path_factory):
    w = World(oracle, tmp_path_factory.mktemp("matrix_dbs"))
    yield w
    w.close()


def _assert_units(want, call, dbg=None, err=""):
    np.testing.assert_array_equal(call, want["ext"], err_msg=err + " ext call")
    if dbg is not None:
        icall, tk, hg = dbg
        np.testing.assert_array_equal(tk, want["total_kmers"], err_msg=err + " total_kmers")
        np.testing.assert_array_equal(hg, want["hit_groups"], err_msg=err + " hit_groups")
        np.testing.assert_array_equal(icall, want["call"], err_msg=err + " call")


def _device_classify(sess, bases, offsets, n_units):
    """classify_device on torch buffers; (call, keep) on the host.  No debug arrays on this path."""
    import torch
    n_seqs = len(offsets) - 1
    d_bases = torch.from_numpy(np.concatenate([bases, np.zeros(64, np.uint8)])).cuda()
    d_off = torch.from_numpy(offsets.astype(np.int64)).cuda()
    d_call = torch.full((max(n_units, 1),), -1, dtype=torch.int32, device="cuda")
    d_keep = torch.full((max(n_units, 1),), 7, dtype=torch.uint8, device="cuda")
    sess.classify_device(d_bases.data_ptr(), d_off.data_ptr(), n_seqs, int(offsets[-1]), d_call.data_ptr(),
                         d_keep.data_ptr())
    sess.sync()
    return d_call.cpu().numpy().view(np.uint32)[:n_units], d_keep.cpu().numpy()[:n_units]


def _is_unsupported(fn):
    from nohuman_b200 import NhError
    from nohuman_b200._ffi import NH_ERR_UNSUPPORTED
    with pytest.raises(NhError) as ei:
        fn()
    assert ei.value.code == NH_ERR_UNSUPPORTED, ei.value


# ---------------------------------------------------------------------------------------------
# 1. instantiation x entry point x switch

@gpu
@pytest.mark.parametrize("dbname,switch", ENTRY_CASES, ids=[f"{d}-{s}" for d, s in ENTRY_CASES])
def test_entry_points(world, oracle, dbname, switch, monkeypatch):
    """classify, classify_device, classify_packed (3 threads), classify_pack (1 and 5 threads) and an
    emit_runs session (classify + last_batch_runs), single-end and paired, on one adversarial batch."""
    from nohuman_b200 import Session
    for var, val in SWITCHES[switch].items():
        monkeypatch.setenv(var, val)
    db, gdb = world.db(dbname), world.gdb(dbname)
    info = gdb.info
    kw, rev = DB_OPTS[dbname]
    assert (int(info.k), int(info.l), int(info.revcom_version)) == (kw.get("k", 35), kw.get("l", 31), rev)
    assert int(info.node_count) == int(db.tax.node_count)
    if dbname == "smalltax":
        assert int(info.value_bits) == 4 and info.filter_bytes == 0  # too few value bits for the miss filter
    elif dbname == "k31":
        assert info.filter_bytes == 0  # window of 1: warp-per-tile kernels, no filter
    else:
        assert info.filter_bytes > 0
    fused = dbname != "k31" and switch != "legacy"
    seqs, bases, offsets = world.batch(dbname, "adv")
    cap = dict(max_batch_bases=len(bases) + 4096)
    for paired, conf in ((False, 0.0), (True, 0.1)):
        want = world.want(dbname, "adv", paired, conf)
        assert (want["call"] != 0).mean() > 0.2 and len(set(want["ext"].tolist())) >= 4
        n_units = len(want["ext"])
        tag = f"{dbname}/{switch}/paired={paired}"
        with Session(gdb, confidence=conf, paired=paired, **cap) as sess:
            call, keep, st = sess.classify(bases, offsets)
            _assert_units(want, call, sess.debug_last_batch(n_units), tag + " classify")
            np.testing.assert_array_equal(keep, (want["ext"] == 0).astype(np.uint8))
            assert st.fused_kernel == (2 if fused else 0)
            assert st.n_classified == int((want["call"] != 0).sum())
            dcall, dkeep = _device_classify(sess, bases, offsets, n_units)
            _assert_units(want, dcall, None, tag + " classify_device")
            np.testing.assert_array_equal(dkeep, (want["ext"] == 0).astype(np.uint8))
            if not fused:
                _is_unsupported(lambda: sess.classify_packed(bases, offsets, threads=3))
                _is_unsupported(lambda: sess.classify_pack(bases, offsets, threads=1))
            else:
                call, keep, st = sess.classify_packed(bases, offsets, threads=3)
                _assert_units(want, call, sess.debug_last_batch(n_units), tag + " classify_packed")
                assert st.fused_kernel == 2
                for threads in (1, 5):
                    call, keep, st = sess.classify_pack(bases, offsets, threads=threads)
                    _assert_units(want, call, sess.debug_last_batch(n_units), tag + f" classify_pack/{threads}")
                    np.testing.assert_array_equal(keep, (want["ext"] == 0).astype(np.uint8))
            if switch == "plain" and not paired:
                # nh_debug_minimizers: the per-position debug instantiation
                n = 80
                mins, amb, pos_off = sess.debug_minimizers(bases[:int(offsets[n])], offsets[:n + 1])
                for i in range(n):
                    wm, wa = oracle.scan_positions(db.opts, bytes(seqs[i]))
                    lo, hi = int(pos_off[i]), int(pos_off[i + 1])
                    np.testing.assert_array_equal(amb[lo:hi], wa, err_msg=f"{tag} ambiguity seq {i}")
                    np.testing.assert_array_equal(mins[lo:hi][wa == 0], wm[wa == 0], err_msg=f"{tag} minimizer seq {i}")
        if switch.startswith("filter"):
            continue  # emit_runs never takes the filter instantiations
        with Session(gdb, confidence=conf, paired=paired, emit_runs=True, **cap) as sess:
            call, keep, st = sess.classify(bases, offsets)
            _assert_units(want, call, sess.debug_last_batch(n_units), tag + " emit_runs classify")
            assert st.fused_kernel == (2 if fused else 0)
            first, ext, ln = sess.last_batch_runs(len(seqs), int(offsets[-1]))
            _is_unsupported(lambda: sess.classify_packed(bases, offsets, threads=3))
            _is_unsupported(lambda: sess.classify_pack(bases, offsets, threads=2))
        runs = world.runs(dbname, "adv")
        for i in range(len(seqs)):
            got = []
            for j in range(int(first[i]), int(first[i + 1])):
                if got and got[-1][0] == int(ext[j]):
                    got[-1][1] += int(ln[j])
                else:
                    got.append([int(ext[j]), int(ln[j])])
            assert got == runs[i], f"{tag} hit runs of sequence {i} (length {len(seqs[i])})"


@gpu
def test_device_entry_rejects_misaligned_bases(world):
    """The streaming kernel stages bases with 16-byte asynchronous copies: d_bases must be aligned."""
    import torch
    from nohuman_b200 import NhError, Session
    from nohuman_b200._ffi import NH_ERR_INVALID
    _, bases, offsets = world.batch("default", "pairs")
    d_bases = torch.from_numpy(np.concatenate([np.zeros(16, np.uint8), bases])).cuda()
    d_off = torch.from_numpy(offsets.astype(np.int64)).cuda()
    d_call = torch.zeros(len(offsets), dtype=torch.int32, device="cuda")
    d_keep = torch.zeros(len(offsets), dtype=torch.uint8, device="cuda")
    with Session(world.gdb("default"), max_batch_bases=len(bases) + 4096) as sess:
        for shift in (1, 8, 15):
            with pytest.raises(NhError) as ei:
                sess.classify_device(d_bases.data_ptr() + shift, d_off.data_ptr(), len(offsets) - 1, len(bases),
                                     d_call.data_ptr(), d_keep.data_ptr())
            assert ei.value.code == NH_ERR_INVALID
        # the same session still works on an aligned copy
        sess.classify_device(d_bases.data_ptr() + 16, d_off.data_ptr(), len(offsets) - 1, len(bases),
                             d_call.data_ptr(), d_keep.data_ptr())
        sess.sync()
    want = world.want("default", "pairs", False, 0.0)
    np.testing.assert_array_equal(d_call.cpu().numpy().view(np.uint32)[:len(want["ext"])], want["ext"])


# ---------------------------------------------------------------------------------------------
# 2. scoring boundaries: the four scoring sites are the in-warp scorer of the streaming kernel,
#    k_score (deferred units), k_score_big (overflowed units) and the warp-per-tile k_score.

SITES = {"in_warp": {}, "k_score": None, "k_score_big": {"NH_TEST_LANE_TAXA": "1"},
         "legacy": {"NH_LEGACY_KERNELS": "1"}}


def _site_env(monkeypatch, site, k_score_tile):
    for var in ("NH_TEST_LANE_TAXA", "NH_LEGACY_KERNELS", "NH_FUSED_TILE_POS", "NH_FILTER_MODE"):
        monkeypatch.delenv(var, raising=False)
    env = SITES[site] if site != "k_score" else {"NH_FUSED_TILE_POS": str(k_score_tile)}
    for var, val in env.items():
        monkeypatch.setenv(var, val)


def _sparse_reads(genomes, n, length, rng):
    """random sequence carrying 0..4 short genome pieces: units with 0..~5 hit groups"""
    out = []
    for i in range(n):
        r = synth.random_genome(rng, length)
        for _ in range(i % 5):
            gname, gseq = genomes[int(rng.integers(0, len(genomes)))]
            w = int(rng.integers(36, 44))
            o = int(rng.integers(0, len(gseq) - w))
            p = int(rng.integers(0, length - w))
            r[p:p + w] = gseq[o:o + w]
        out.append(r)
    return out


@pytest.fixture(scope="module")
def scoring_batches(world):
    db = world.db("default")
    rng = np.random.default_rng(71)
    seqs = []
    for i in range(1500):  # 150 bp reads with 1..5 % substitutions: max scores spread over 0..116
        g = db.genomes[i % 4][1]
        o = int(rng.integers(0, len(g) - 151))
        seqs.append(synth.mutate(rng, g[o:o + 150], 0.01 + 0.04 * rng.random()))
    seqs += _sparse_reads(db.genomes, 500, 150, rng)
    fixed = seqs  # every read 150 bp: T = 116 single-end, 232 per pair
    longs = _sparse_reads(db.genomes, 150, 2300, rng)  # > 32 tiles of 64 positions: deferred to k_score
    longs += [synth.mutate(rng, db.genomes[0][1][i * 97:i * 97 + 2300], 0.04) for i in range(50)]
    return fixed, fixed + longs


@gpu
@pytest.mark.parametrize("site", list(SITES))
def test_minimum_hit_groups_at_every_scoring_site(world, scoring_batches, site, monkeypatch):
    from nohuman_b200 import Session
    _site_env(monkeypatch, site, 64)
    db, gdb = world.db("default"), world.gdb("default")
    seqs = scoring_batches[1]
    bases, offsets = synth.pack(seqs)
    wants = {}
    for paired in (False, True):
        for mhg in (0, 1, 2, 3, 10):
            db.min_hit_groups, db.confidence = mhg, 0.0
            want = wants[paired, mhg] = db.classify_batch(bases, offsets, paired=paired)
            db.min_hit_groups, db.confidence = 2, 0.0
            with Session(gdb, confidence=0.0, paired=paired, minimum_hit_groups=mhg,
                         max_batch_bases=len(bases) + 4096) as sess:
                call, keep, st = sess.classify(bases, offsets)
                _assert_units(want, call, sess.debug_last_batch(len(call)), f"{site} mhg={mhg} paired={paired}")
                assert st.fused_kernel == (0 if site == "legacy" else 2)
        # teeth: units on the edge between 2 and 3 groups, and hit_groups spread over the edge values
        assert (wants[paired, 2]["call"] != wants[paired, 3]["call"]).sum() >= 5
        assert (wants[paired, 0]["call"] != wants[paired, 1]["call"]).sum() == 0  # a call needs a hit
        assert (wants[paired, 1]["call"] != wants[paired, 2]["call"]).sum() >= 3
        hg = wants[paired, 2]["hit_groups"]
        assert all((hg == v).sum() >= 3 for v in (1, 2, 3, 9, 10))


def _edge_confidences(db, bases, offsets, paired, T):
    """Confidences on the edges of required = ceil(conf * T), picked by search: for every j whose
    boundary moves a call (the oracle's calls at required j and j + 1 differ), c = j / T, its two
    neighbouring doubles, and the last double whose required score is still j plus the next one.
    Returns {conf: required} for a set that holds products c * T that are not exactly j in double and
    confidences where a float32 product has another ceil than the double one and changes a call."""
    calls = {}
    for r in range(1, T + 2):
        db.confidence = (r - 0.5) / T  # ceil() of this is r in any rounding
        calls[r] = db.classify_batch(bases, offsets, paired=paired)["call"]
    db.confidence = 0.0
    moves = [j for j in range(1, T + 1) if (calls[j] != calls[j + 1]).any()]
    inexact, slips, exact = [], [], []
    for j in moves:
        c = j / T
        for v in (float(np.nextafter(c, 0)), c, float(np.nextafter(c, 1))):
            r64, r32 = int(np.ceil(v * T)), int(np.ceil(np.float32(v) * np.float32(T)))
            if r32 != r64 and 1 <= r32 <= T + 1 and (calls[r32] != calls[r64]).any():
                slips.append(j)
        (inexact if c * T != j else exact).append(j)
    js = sorted(set(inexact[:3] + slips[::max(1, len(slips) // 4)][:4] + exact[::max(1, len(exact) // 2)][:2]))
    assert inexact and slips, (inexact, slips)
    out = {}
    for j in js:
        c = j / T
        b = c  # the largest double whose required score is j
        while np.ceil(b * T) > j:
            b = float(np.nextafter(b, 0))
        while np.ceil(float(np.nextafter(b, 1)) * T) <= j:
            b = float(np.nextafter(b, 1))
        for v in (float(np.nextafter(c, 0)), c, float(np.nextafter(c, 1)), b, float(np.nextafter(b, 1))):
            out[v] = int(np.ceil(v * T))
        assert out[b] == j and out[float(np.nextafter(b, 1))] == j + 1
    return out, calls


@gpu
@pytest.mark.parametrize("site", list(SITES))
def test_confidence_on_the_rounding_edge(world, scoring_batches, site, monkeypatch):
    """required = ceil(conf * total_kmers) in IEEE double, as kraken2 and the oracle compute it."""
    from nohuman_b200 import Session
    _site_env(monkeypatch, site, 20)  # 20: 116-position units of 6 tiles, 1 in 8 crosses a group border
    db, gdb = world.db("default"), world.gdb("default")
    bases, offsets = synth.pack(scoring_batches[0])
    for paired, T in ((False, 116), (True, 232)):
        key = ("edges", paired)
        if key not in world._want:
            world._want[key] = _edge_confidences(db, bases, offsets, paired, T)
        confs, calls = world._want[key]
        for v, required in confs.items():
            db.confidence = v
            want = db.classify_batch(bases, offsets, paired=paired)
            db.confidence = 0.0
            assert (want["total_kmers"] == T).all()
            np.testing.assert_array_equal(want["call"], calls[required])
            with Session(gdb, confidence=v, paired=paired, max_batch_bases=len(bases) + 4096) as sess:
                call, keep, st = sess.classify(bases, offsets)
                _assert_units(want, call, sess.debug_last_batch(len(call)), f"{site} conf={v!r} paired={paired}")
                assert st.fused_kernel == (0 if site == "legacy" else 2)


# ---------------------------------------------------------------------------------------------
# 3. table and taxonomy boundaries

N_LEAVES = 16_500
LEAF_BP = 60
PIECE_BP = 45  # a non-dominant leaf contributes 11 k-mers, the dominant one its whole 26


@pytest.fixture(scope="module")
def many_leaves(oracle, tmp_path_factory):
    """16 500 leaf taxa under one clade, a random 60 bp genome each; only leaves whose every k-mer
    classifies to the leaf itself (no minimizer shared with another leaf) are used in reads."""
    rng = np.random.default_rng(41)
    tax = [oracle.TaxSpec(1, 1, "root", "no rank"), oracle.TaxSpec(2, 1, "clade", "no rank")]
    tax += [oracle.TaxSpec(100 + i, 2, f"leaf{i}", "species") for i in range(N_LEAVES)]
    genomes = [(100 + i, synth.random_genome(rng, LEAF_BP)) for i in range(N_LEAVES)]
    db = oracle.OracleDb.build([(t, bytes(g)) for t, g in genomes], tax, capacity=2_000_003)
    path = str(tmp_path_factory.mktemp("many_leaves"))
    db.save(path)
    clean = []
    for t, g in genomes:
        internal = db.internal_id(t)
        taxa = db.classify_one(bytes(g), want_taxa=True)["taxa"]
        if taxa and all(x == internal for x in taxa):
            clean.append((t, internal, g))
    assert len(clean) >= 16_420
    db.clean = clean
    db.path = path
    from nohuman_b200 import Database
    gdb = Database.open(path, 0)
    yield db, gdb
    gdb.close()


def _leaf_read(clean, n, start, dominant_last, pad=0):
    """n distinct leaves: one dominant (whole genome), n - 1 pieces; N between them keeps k-mers within a leaf"""
    sep = np.array([ord("N")], np.uint8)
    dom = clean[start][2]
    others = [clean[start + 1 + i][2][:PIECE_BP] for i in range(n - 1)]
    parts = others + [dom] if dominant_last else [dom] + others
    out = [np.full(pad, ord("N"), np.uint8)] if pad else []
    for p in parts:
        out += [p, sep]
    return np.concatenate(out[:-1]), {clean[start + i][1] for i in range(n)}


LEAF_COUNTS = [7, 8, 9, 63, 64, 65, 16_383, 16_384, 16_385]
PLACEMENTS = {
    "in_warp": ("single", {}),                           # one tile up to 9 leaves; larger units overflow
    "k_score": ("padded", {"NH_FUSED_TILE_POS": "64"}),  # N prefix: more than 32 tiles, deferred to k_score
    "paired": ("paired", {}),                            # leaves split between the mates
    "legacy": ("single", {"NH_LEGACY_KERNELS": "1"}),
}
_LEAF_CACHE = {}


def _leaf_units(db, kind):
    """(units as lists of mates, hit count per unit, oracle answer at confidence 0) for one input shape.
    Every unit's distinct taxa are confirmed with the oracle: exactly n leaves, none folded into the clade."""
    if kind in _LEAF_CACHE:
        return _LEAF_CACHE[kind]
    pad = 33 * 64 + 40 if kind == "padded" else 0
    units, hits = [], []
    for i, n in enumerate(LEAF_COUNTS):
        for last in (False, True):
            r, taxa = _leaf_read(db.clean, n, 2 * i + last, last, pad)
            if kind == "paired":  # the first n // 2 leaves in mate 1, the rest in mate 2
                cut = int(np.flatnonzero(r == ord("N"))[n // 2 - 1])
                units.append([r[:cut], r[cut + 1:]])
            else:
                units.append([r])
            res = db.classify_one(*[bytes(m) for m in units[-1]], want_taxa=True)
            got = {t for t in res["taxa"] if 0 < t < SENTINEL}
            assert got == taxa and len(got) == n
            hits.append(sum(1 for t in res["taxa"] if 0 < t < SENTINEL))
    seqs = [m for u in units for m in u]
    bases, offsets = synth.pack(seqs)
    db.confidence = 0.0
    want = db.classify_batch(bases, offsets, paired=kind == "paired")
    dominant = [db.clean[2 * i + last][0] for i in range(len(LEAF_COUNTS)) for last in (False, True)]
    np.testing.assert_array_equal(want["ext"], dominant)
    _LEAF_CACHE[kind] = (units, hits, want, bases, offsets)
    return _LEAF_CACHE[kind]


@gpu
@pytest.mark.parametrize("placement", list(PLACEMENTS))
def test_units_on_taxon_table_edges(many_leaves, placement, monkeypatch):
    """Units with exactly 8/9 (in-warp lane tables), 64/65 (k_score) and 16384/16385 (k_score_big, then the
    database's global table) distinct taxa.  At confidence 0 the dominant leaf wins (placed first and last);
    at the confidence whose required score is the unit's total hit count only the clade's sum over every
    table slot reaches it, so losing any one slot changes the call."""
    from nohuman_b200 import Session
    db, gdb = many_leaves
    kind, env = PLACEMENTS[placement]
    paired = kind == "paired"
    for var, val in env.items():
        monkeypatch.setenv(var, val)
    units, hits, want, bases, offsets = _leaf_units(db, kind)
    cap = dict(max_batch_bases=len(bases) + 4096, max_batch_seqs=len(offsets) + 2)
    with Session(gdb, confidence=0.0, paired=paired, **cap) as sess:
        call, keep, st = sess.classify(bases, offsets)
        _assert_units(want, call, sess.debug_last_batch(len(call)), f"{placement} conf=0")
    clade = db.internal_id(2)
    # one unit per session at the confidence that requires every hit: only the clade's sum reaches it
    for u, (mates, h) in enumerate(zip(units, hits)):
        ub, uo = synth.pack(mates)
        conf = (h - 0.5) / int(want["total_kmers"][u])
        key = (kind, "edge", u)
        if key not in _LEAF_CACHE:
            db.confidence = conf
            _LEAF_CACHE[key] = db.classify_batch(ub, uo, paired=paired)
            db.confidence = 0.0
        w1 = _LEAF_CACHE[key]
        assert int(w1["call"][0]) == clade
        with Session(gdb, confidence=conf, paired=paired, max_batch_bases=len(ub) + 4096) as sess:
            call, keep, st = sess.classify(ub, uo)
            _assert_units(w1, call, sess.debug_last_batch(1), f"{placement} unit {u} all-hits confidence")


def _bushy_taxonomy(oracle, n_specs, seed):
    rng = np.random.default_rng(seed)
    tax = [oracle.TaxSpec(1, 1, "root", "no rank")]
    ids = [1]
    for i in range(2, n_specs + 1):
        parent = ids[int(rng.integers(max(0, len(ids) - 40), len(ids)))]  # deep, bushy tree
        tax.append(oracle.TaxSpec(i, parent, f"n{i}", "no rank"))
        ids.append(i)
    return tax, rng


@gpu
@pytest.mark.parametrize("node_count", [8192, 8193])
def test_taxonomy_on_the_shared_memory_parent_edge(oracle, tmp_path, node_count, monkeypatch):
    """NH_SMEM_PARENT_MAX = 8192 nodes: the last taxonomy whose parent array is staged in shared memory
    by the streaming kernel and k_score<true>, and the first that is read through L2 (k_score<false>)."""
    from nohuman_b200 import Database, Session
    tax, rng = _bushy_taxonomy(oracle, node_count - 1, seed=node_count)
    leaves = [int(x) for x in rng.choice(np.arange(node_count - 3000, node_count), size=24, replace=False)]
    genomes = [(t, synth.random_genome(rng, 6000)) for t in leaves]
    shared = synth.random_genome(rng, 1500)
    for _, g in genomes[::2]:
        g[2000:3500] = shared  # LCA values deep and high in the tree
    db = oracle.OracleDb.build([(t, bytes(g)) for t, g in genomes], tax)
    path = str(tmp_path / "tax")
    db.save(path)
    seqs = synth.illumina_reads(genomes, 600, 150, seed=8, paired=True, n_rate=0.1)
    seqs += synth.ont_reads(genomes, 16, seed=9, n50=2500, max_len=5000)
    bases, offsets = synth.pack(seqs)
    with Database.open(path, 0) as gdb:
        assert int(gdb.info.node_count) == node_count == int(db.tax.node_count)
        for env in ({}, {"NH_FUSED_TILE_POS": "64"}, {"NH_TEST_LANE_TAXA": "1"}, {"NH_LEGACY_KERNELS": "1"}):
            for var in ("NH_FUSED_TILE_POS", "NH_TEST_LANE_TAXA", "NH_LEGACY_KERNELS"):
                monkeypatch.delenv(var, raising=False)
            for var, val in env.items():
                monkeypatch.setenv(var, val)
            for paired, conf in ((False, 0.05), (True, 0.5)):
                db.confidence = conf
                want = db.classify_batch(bases, offsets, paired=paired)
                with Session(gdb, confidence=conf, paired=paired, max_batch_bases=len(bases) + 4096) as sess:
                    call, keep, st = sess.classify(bases, offsets)
                    _assert_units(want, call, sess.debug_last_batch(len(call)), f"{env} paired={paired}")
                assert len(set(want["call"].tolist())) > 10
                depth = []
                for c in set(want["call"].tolist()) - {0}:
                    d, x = 0, c
                    while x > 1:
                        x, d = db.tax.nodes[x].parent_id, d + 1
                    depth.append(d)
                assert max(depth) >= 20  # calls deep in the tree walk long parent chains


# ---------------------------------------------------------------------------------------------
# 4. one session, many batches

@gpu
@pytest.mark.parametrize("paired", [False, True], ids=["single", "paired"])
@pytest.mark.parametrize("dbname", DB_NAMES)
def test_one_session_many_batches(world, dbname, paired):
    """long reads (tile 252, per-tile plan), 2x150 pairs (tile 508), an empty batch, the pairs packed, a
    one-sequence (one-pair) batch, classify_device, then long reads through classify_pack: every step against
    the oracle and against a fresh session's answer."""
    from nohuman_b200 import Session
    gdb = world.gdb(dbname)
    fused = dbname != "k31"
    conf = 0.1
    cap = dict(max_batch_bases=1 << 22, max_batch_seqs=1 << 12)
    steps = [("long", "classify"), ("pairs", "classify"), (None, "empty"), ("pairs", "packed"),
             ("onepair" if paired else "one", "classify"), ("pairs", "device"), ("long", "pack")]
    _, lb, lo = world.batch(dbname, "long")
    assert int(lo[-1]) // (len(lo) - 1) > 1000
    with Session(gdb, confidence=conf, paired=paired, **cap) as sess:
        for kind, entry in steps:
            tag = f"{dbname} paired={paired} {kind}/{entry}"
            if entry == "empty":
                call, keep, st = sess.classify(np.zeros(0, np.uint8), np.zeros(1, np.uint64))
                assert len(call) == 0 and st.n_units == 0
                continue
            _, bases, offsets = world.batch(dbname, kind)
            want = world.want(dbname, kind, paired, conf)
            n_units = len(want["ext"])

            def run(s):
                if entry == "classify":
                    c, _, _ = s.classify(bases, offsets)
                    return c, s.debug_last_batch(n_units)
                if entry == "device":
                    return _device_classify(s, bases, offsets, n_units)[0], None
                if entry == "packed":
                    c, _, _ = s.classify_packed(bases, offsets, threads=3)
                else:
                    c, _, _ = s.classify_pack(bases, offsets, threads=5)
                return c, s.debug_last_batch(n_units)

            if entry in ("packed", "pack") and not fused:
                _is_unsupported(lambda: run(sess))
                continue
            call, dbg = run(sess)
            _assert_units(want, call, dbg, tag)
            with Session(gdb, confidence=conf, paired=paired, **cap) as fresh:
                fcall, fdbg = run(fresh)
            np.testing.assert_array_equal(call, fcall, err_msg=tag + " fresh session")
            if dbg is not None:
                for a, b in zip(dbg, fdbg):
                    np.testing.assert_array_equal(a, b, err_msg=tag + " fresh session")


@gpu
def test_two_sessions_share_the_huge_table(many_leaves):
    """Two sessions on one database, both enqueued before either syncs, each with a unit of more than 16 384
    distinct taxa: k_score_big's global table and its lock belong to the database."""
    import torch
    from nohuman_b200 import Session
    db, gdb = many_leaves
    rng = np.random.default_rng(5)
    batches = []
    for s in range(2):
        r, taxa = _leaf_read(db.clean, 16_385 + s, 11 * s, bool(s))
        shorts = [db.clean[int(i)][2] for i in rng.integers(0, len(db.clean), 300)]
        seqs = shorts[:150] + [r] + shorts[150:] + [r[::-1].copy()]
        batches.append(synth.pack(seqs))
    confs = (0.0, 0.3)
    bufs = []
    sessions = [Session(gdb, confidence=confs[s], max_batch_bases=len(batches[s][0]) + 4096) for s in range(2)]
    try:
        for s, (bases, offsets) in enumerate(batches):
            n = len(offsets) - 1
            d_bases = torch.from_numpy(np.concatenate([bases, np.zeros(64, np.uint8)])).cuda()
            d_off = torch.from_numpy(offsets.astype(np.int64)).cuda()
            d_call = torch.full((n,), -1, dtype=torch.int32, device="cuda")
            d_keep = torch.zeros(n, dtype=torch.uint8, device="cuda")
            torch.cuda.synchronize()
            bufs.append((d_bases, d_off, d_call, d_keep))
        for s, (bases, offsets) in enumerate(batches):
            d_bases, d_off, d_call, d_keep = bufs[s]
            sessions[s].classify_device(d_bases.data_ptr(), d_off.data_ptr(), len(offsets) - 1, len(bases),
                                        d_call.data_ptr(), d_keep.data_ptr())
        for s in (1, 0):
            sessions[s].sync()
    finally:
        for sess in sessions:
            sess.close()
    for s, (bases, offsets) in enumerate(batches):
        db.confidence = confs[s]
        want = db.classify_batch(bases, offsets)
        db.confidence = 0.0
        assert want["hit_groups"][150] > 16_384
        np.testing.assert_array_equal(bufs[s][2].cpu().numpy().view(np.uint32), want["ext"], err_msg=f"session {s}")
