"""kraken2-inspect without a GPU: the shim's argument handling, the inspect flags against the header, and
NH_ERR_CUDA (not a crash) from the inspect entry points on a machine without a device."""
import ctypes as C
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHIM = os.path.join(ROOT, "nohuman_b200", "bin", "kraken2-inspect")


def no_device():
    from nohuman_b200 import _ffi
    return _ffi.lib().nh_device_count() == 0


@pytest.mark.parametrize("args,word", [(["--use-mpa-style", "--db", "x"], "--use-mpa-style"),
                                       (["--db", "x", "--print-optstring"], "--print-optstring"),
                                       (["-x", "--db", "x"], "-x"),
                                       (["--db", "x", "extra"], "extra"),
                                       (["--db"], "--db"),
                                       ([], "--db DIR is required"),
                                       (["--skip-counts", "--threads", "4"], "--db DIR is required")])
def test_shim_refuses(tmp_path, args, word):
    r = subprocess.run([SHIM, *args], capture_output=True, text=True, cwd=tmp_path)
    assert r.returncode == 64, r.stderr
    lines = r.stderr.strip().splitlines()
    assert len(lines) == 1 and word in lines[0], r.stderr
    assert r.stdout == "" and os.listdir(tmp_path) == []


def test_missing_database_exits_1(tmp_path):
    r = subprocess.run([SHIM, "--db", str(tmp_path / "none"), "--threads", "2", "--memory-mapping"],
                       capture_output=True, text=True)
    assert r.returncode == 1 and r.stdout == ""
    assert "hash.k2d" in r.stderr and len(r.stderr.strip().splitlines()) == 1


def test_flags_match_the_header():
    from nohuman_b200 import _ffi
    src = open(os.path.join(ROOT, "include", "nohuman_gpu.h")).read()
    defs = dict(re.findall(r"#define (NH_INSPECT_\w+) (\d+)", src))
    assert {k: int(v) for k, v in defs.items()} == {"NH_INSPECT_SKIP_COUNTS": _ffi.NH_INSPECT_SKIP_COUNTS,
                                                     "NH_INSPECT_ZERO_COUNTS": _ffi.NH_INSPECT_ZERO_COUNTS}


def test_entry_points_without_device_fail_with_nh_err_cuda():
    if not no_device():
        pytest.skip("a CUDA device is present")
    from nohuman_b200 import _ffi
    L = _ffi.lib()
    counts = (C.c_uint64 * 4)()
    occ, oor = C.c_uint64(), C.c_uint64()
    t = C.c_double()
    assert L.nh_db_taxon_counts(None, counts, 4, C.byref(occ), C.byref(oor)) == _ffi.NH_ERR_CUDA
    assert b"no CUDA device" in L.nh_last_error()
    assert L.nh_db_inspect(None, None, 0) == _ffi.NH_ERR_CUDA
    assert L.nh_bench_taxon_counts(None, 3, C.byref(t)) == _ffi.NH_ERR_CUDA


def test_shim_without_device_fails(small_db):
    if not no_device():
        pytest.skip("a CUDA device is present")
    r = subprocess.run([SHIM, "--db", small_db.path], capture_output=True, text=True)
    assert r.returncode == 1 and r.stdout == ""
    assert "no CPU path" in r.stderr
