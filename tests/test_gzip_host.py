"""GPU gzip surface that needs no GPU: nh_bgzf_compress argument checks (and NH_ERR_CUDA without a
device, as every compute entry point), and the CLI's --gpu-gzip switch."""
import ctypes as C
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "nohuman_b200", "bin", "nohuman")


def compress(data, out_cap, null_in=False):
    from nohuman_b200 import _ffi
    out = C.create_string_buffer(max(out_cap, 1))
    got = C.c_size_t(123)
    rc = _ffi.lib().nh_bgzf_compress(0, None if null_in else data, len(data), out, out_cap, C.byref(got))
    return rc, got.value


def test_bgzf_compress_argument_checks():
    from nohuman_b200 import _ffi
    assert compress(b"x" * 10, 65536, null_in=True)[0] == _ffi.NH_ERR_INVALID
    assert compress(b"x" * 0xFF00, 65535)[0] == _ffi.NH_ERR_CAPACITY
    assert compress(b"x" * (0xFF00 + 1), 65536)[0] == _ffi.NH_ERR_CAPACITY


def test_bgzf_compress_without_gpu():
    from nohuman_b200 import NhError, _ffi
    from nohuman_b200.api import bgzf_compress
    if _ffi.lib().nh_device_count() > 0:
        pytest.skip("a CUDA device is present")
    assert compress(b"x" * 100, 65536)[0] == _ffi.NH_ERR_CUDA
    with pytest.raises(NhError) as ei:
        bgzf_compress(b"abc")
    assert ei.value.code == _ffi.NH_ERR_CUDA
    assert "no CPU path" in ei.value.message


def test_session_params_carry_gpu_gzip():
    from nohuman_b200 import _ffi
    p = _ffi.Params()
    p.gpu_gzip = 1
    assert _ffi.Params.gpu_gzip.offset == C.sizeof(_ffi.Params) - 4


def plan(args, tmp_path):
    db = tmp_path / "db"
    db.mkdir()
    for n in ("hash.k2d", "opts.k2d", "taxo.k2d"):
        (db / n).write_bytes(b"")
    fq = tmp_path / "r.fq"
    fq.write_bytes(b"@r\nACGT\n+\nIIII\n")
    r = subprocess.run([CLI, "--plan", "--db", str(db), *args, str(fq)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return dict(line.split("=", 1) for line in r.stdout.splitlines() if "=" in line)


def test_cli_gpu_gzip_flag(tmp_path):
    if not os.path.exists(CLI):
        from nohuman_b200 import build
        build.build()
    assert plan(["-F", "g"], tmp_path)["gpu_gzip"] == "0"
    (tmp_path / "db").rename(tmp_path / "db0")
    kv = plan(["-F", "g", "--gpu-gzip"], tmp_path)
    assert kv["gpu_gzip"] == "1" and kv["format"] == "g"
    r = subprocess.run([CLI, "--help"], capture_output=True, text=True)
    assert "--gpu-gzip" in r.stdout
