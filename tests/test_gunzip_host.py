"""GPU gzip decompression surface that needs no GPU: nh_gunzip argument checks, and NH_ERR_CUDA without a
device, as every compute entry point."""
import ctypes as C
import gzip

import pytest


def gunzip_rc(data, out_cap, null_in=False, null_len=False, null_out=False):
    from nohuman_b200 import _ffi
    out = C.create_string_buffer(max(out_cap, 1))
    got = C.c_size_t(123)
    rc = _ffi.lib().nh_gunzip(0, None if null_in else data, len(data), None if null_out else out, out_cap,
                              None if null_len else C.byref(got))
    return rc


def test_gunzip_argument_checks():
    from nohuman_b200 import _ffi
    blob = gzip.compress(b"x" * 100)
    assert gunzip_rc(blob, 1000, null_in=True) == _ffi.NH_ERR_INVALID
    assert gunzip_rc(blob, 1000, null_len=True) == _ffi.NH_ERR_INVALID
    assert gunzip_rc(blob, 1000, null_out=True) == _ffi.NH_ERR_INVALID
    counts = (C.c_uint64 * len(_ffi.GUNZIP_COUNTS))()
    got = C.c_size_t()
    out = C.create_string_buffer(1000)
    # unknown test flags
    assert _ffi.lib().nh_debug_gunzip(0, blob, len(blob), out, 1000, C.byref(got), 0, 0, 2, counts) == _ffi.NH_ERR_INVALID
    t = C.c_double()
    assert _ffi.lib().nh_bench_gunzip(0, blob, len(blob), 0, C.byref(t)) == _ffi.NH_ERR_INVALID
    assert _ffi.lib().nh_bench_gunzip(0, None, 0, 1, C.byref(t)) == _ffi.NH_ERR_INVALID


def test_gunzip_without_gpu():
    from nohuman_b200 import NhError, _ffi
    from nohuman_b200.api import gunzip
    if _ffi.lib().nh_device_count() > 0:
        pytest.skip("a CUDA device is present")
    assert gunzip_rc(gzip.compress(b"abc"), 100) == _ffi.NH_ERR_CUDA
    with pytest.raises(NhError) as ei:
        gunzip(gzip.compress(b"abc"))
    assert ei.value.code == _ffi.NH_ERR_CUDA
    assert "no CPU path" in ei.value.message

