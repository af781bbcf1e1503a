"""Loading a database: every constructor checks hash.k2d / opts.k2d / taxo.k2d before any device work, and every
constructor that succeeds yields the same database.

The malformed-input cases need no GPU: the library rejects them before it looks for a device, with the same code and
message on a machine with or without one."""
import ctypes as C
import os
import shutil
import struct

import numpy as np
import pytest

import synth

NODE = 56  # bytes per taxo.k2d node record: parent, first child, child count, name, rank, external id, godparent


def _cut(key, length):
    def mutate(f):
        del f[key][length:]
    return mutate


def _put(key, offset, fmt, *values):
    def mutate(f):
        struct.pack_into(fmt, f[key], offset, *values)
    return mutate


def _node(i):
    return 32 + NODE * i


def _truncate_taxo(f):
    n = struct.unpack_from("<Q", f["taxo"], 8)[0]
    del f["taxo"][_node(n) - 1:]


def _grow_hash(f):
    f["hash"] += bytes(4)


def _capacity_zero(f):
    _put("hash", 0, "<Q", 0)(f)
    del f["hash"][32:]  # so that open's file-size check passes and the header check is what fails


# (id, mutation of the {"opts", "taxo", "hash"} images, NH_ERR_* name, message substring, checked by open only)
CASES = [
    ("opts_short", _cut("opts", 31), "NH_ERR_IO", "opts.k2d too short", False),
    ("taxo_bad_magic", _put("taxo", 0, "8s", b"K2TAXDAX"), "NH_ERR_IO", "taxo.k2d: bad magic", False),
    ("taxo_truncated", _truncate_taxo, "NH_ERR_IO", "taxo.k2d: truncated", False),
    ("parent_not_below_child", _put("taxo", _node(3), "<Q", 3), "NH_ERR_UNSUPPORTED", "node 3 has parent 3", False),
    ("external_id_over_32_bits", _put("taxo", _node(2) + 40, "<Q", 1 << 32), "NH_ERR_UNSUPPORTED",
     "external id 4294967296 does not fit 32 bits", False),
    ("hash_short_header", _cut("hash", 20), "NH_ERR_IO", "hash.k2d: short header", True),
    ("hash_size_mismatch", _grow_hash, "NH_ERR_IO", "!= 32 + 4*capacity", True),
    ("key_plus_value_bits", _put("hash", 16, "<QQ", 13, 18), "NH_ERR_IO", "key_bits 13 + value_bits 18 != 32", False),
    ("capacity_zero", _capacity_zero, "NH_ERR_IO", "hash.k2d: bad capacity", False),
    ("protein_db", _put("opts", 32, "<B", 0), "NH_ERR_UNSUPPORTED", "protein databases are not supported", False),
    ("l_zero", _put("opts", 0, "<QQ", 35, 0), "NH_ERR_UNSUPPORTED", "unsupported k=35 l=0", False),
    ("l_over_31", _put("opts", 0, "<QQ", 35, 32), "NH_ERR_UNSUPPORTED", "unsupported k=35 l=32", False),
    ("k_below_l", _put("opts", 0, "<QQ", 30, 31), "NH_ERR_UNSUPPORTED", "unsupported k=30 l=31", False),
    ("window_over_32", _put("opts", 0, "<QQ", 63, 31), "NH_ERR_UNSUPPORTED", "minimizer window k-l+1=33 exceeds 32",
     False),
    ("nodes_over_value_bits", _put("hash", 16, "<QQ", 28, 4), "NH_ERR_IO", "more nodes than value_bits can address",
     False),
]

PARAMS = [pytest.param(c, entry, id=f"{c[0]}-{entry}") for c in CASES for entry in ("open", "from_memory")
          if entry == "open" or not c[4]]


def _read_files(path):
    out = {}
    for key in ("opts", "taxo", "hash"):
        with open(os.path.join(path, f"{key}.k2d"), "rb") as fh:
            out[key] = bytearray(fh.read())
    return out


@pytest.fixture
def corrupt_db(small_db, tmp_path):
    """A fresh copy of small_db; returns (dir, files) for the test to corrupt and write back."""
    d = tmp_path / "db"
    shutil.copytree(small_db.path, d)
    return str(d), _read_files(str(d))


def _write_files(d, files):
    for key, data in files.items():
        with open(os.path.join(d, f"{key}.k2d"), "wb") as fh:
            fh.write(data)


def _construct(entry, d, files, cells):
    from nohuman_b200 import Database
    if entry == "open":
        _write_files(d, files)
        return Database.open(d, 0)
    header = struct.unpack_from("<4Q", files["hash"])
    return Database.from_memory(bytes(files["opts"]), bytes(files["taxo"]), header, cells, device=0)


@pytest.mark.parametrize("case,entry", PARAMS)
def test_malformed_database_is_rejected(corrupt_db, case, entry):
    from nohuman_b200 import NhError, _ffi
    _, mutate, code, message, _ = case
    d, files = corrupt_db
    cells = np.frombuffer(bytes(files["hash"][32:]), np.uint32)
    mutate(files)
    with pytest.raises(NhError) as ei:
        _construct(entry, d, files, cells).close()
    assert ei.value.code == getattr(_ffi, code), ei.value.message
    assert message in ei.value.message


@pytest.mark.parametrize("entry", ["open", "from_memory"])
def test_intact_copy_passes_the_checks(corrupt_db, entry):
    """The control of the cases above: without corruption the copy fails only for want of a GPU, or opens."""
    from nohuman_b200 import NhError, _ffi
    d, files = corrupt_db
    cells = np.frombuffer(bytes(files["hash"][32:]), np.uint32)
    if _ffi.lib().nh_device_count() > 0:
        db = _construct(entry, d, files, cells)
        assert int(db.info.capacity) == len(cells)
        db.close()
        return
    with pytest.raises(NhError) as ei:
        _construct(entry, d, files, cells)
    assert ei.value.code == _ffi.NH_ERR_CUDA and "no CPU path" in ei.value.message


# ---------------------------------------------------------------------------------------------------------------
# every constructor yields the same database


def _n_devices():
    from nohuman_b200 import _ffi
    return _ffi.lib().nh_device_count()


def _info(db):
    i = db.info
    return {f: getattr(i, f) for f, _ in type(i)._fields_ if f not in ("device", "replicated_by")}


def _cells(db):
    from nohuman_b200 import _ffi
    out = np.empty(int(db.info.capacity), np.uint32)
    assert _ffi.lib().nh_db_download_cells(db._h, C.c_void_p(out.ctypes.data)) == 0
    return out


def _calls(db, bases, offsets):
    from nohuman_b200 import Session
    with Session(db, confidence=0.1) as s:
        call, keep, _ = s.classify(bases, offsets)
    return call, keep


def _check_same(ref, db, ref_cells, batch, want):
    assert _info(db) == _info(ref)  # filter_bytes included
    np.testing.assert_array_equal(_cells(db), ref_cells)
    call, keep = _calls(db, *batch)
    np.testing.assert_array_equal(call, want[0])
    np.testing.assert_array_equal(keep, want[1])


@pytest.fixture(scope="module")
def batch(small_db):
    return synth.pack(synth.illumina_reads(small_db.genomes, 800, 150, seed=31))


@pytest.mark.gpu
def test_every_constructor_builds_the_same_database(small_db, batch):
    from nohuman_b200 import Database
    files = _read_files(small_db.path)
    header = struct.unpack_from("<4Q", files["hash"])
    host_cells = np.frombuffer(bytes(files["hash"][32:]), np.uint32)
    ref = Database.open(small_db.path, 0)
    made = []
    try:
        ref_cells = _cells(ref)
        np.testing.assert_array_equal(ref_cells, host_cells)
        assert ref.info.filter_bytes > 0 and ref.info.replicated_by == 0
        want = _calls(ref, *batch)
        small_db.confidence = 0.1
        np.testing.assert_array_equal(want[0], small_db.classify_batch(*batch)["ext"])
        made.append(Database.from_memory(bytes(files["opts"]), bytes(files["taxo"]), header, host_cells, device=0))
        made.append(Database.from_memory(bytes(files["opts"]), bytes(files["taxo"]), header, ref.device_cells_ptr(),
                                         device=0, cells_on_device=True))
        assert made[-1].device_cells_ptr() == ref.device_cells_ptr()
        made.append(ref.clone(0))
        made += Database.open_multi(small_db.path, [0])
        for db in made:
            assert db.info.device == 0 and db.info.replicated_by == 0
            _check_same(ref, db, ref_cells, batch, want)
    finally:
        for db in made:  # the adopting handle goes before the one that owns its cells
            db.close()
        ref.close()


@pytest.mark.gpu
@pytest.mark.parametrize("how", ["auto", "p2p"])
def test_replicas_are_the_same_database(small_db, batch, how, monkeypatch):
    if _n_devices() < 2:
        pytest.skip("needs two CUDA devices")
    from nohuman_b200 import Database
    if how == "p2p":
        monkeypatch.setenv("NH_DB_REPLICATE", "p2p")
    dbs = Database.open_multi(small_db.path, [0, 1])
    try:
        ref_cells = _cells(dbs[0])
        want = _calls(dbs[0], *batch)
        assert dbs[1].info.device == 1 and dbs[1].info.replicated_by == (2 if how == "p2p" else dbs[1].info.replicated_by)
        assert dbs[1].info.replicated_by in (1, 2)
        _check_same(dbs[0], dbs[1], ref_cells, batch, want)
    finally:
        for db in dbs:
            db.close()
