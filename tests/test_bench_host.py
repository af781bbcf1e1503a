"""bench.py on the CPU: the reference arm runs without torch and without the CUDA library and prints the
same `config` the GPU arm would; the workload shapes are what BASELINE.json names."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_is_cpu_only_and_shares_the_config():
    code = r'''
import sys, json
sys.argv = ["bench.py", "--impl", "reference", "--capacity-log2", "18", "--steps", "2", "--warmup", "1", "--pairs-per-launch", "4000"]
sys.path.insert(0, %r)
import bench
bench.main()
maps = open("/proc/self/maps").read()
print(json.dumps({"torch": "torch" in sys.modules, "gpu_lib": "libnohuman_gpu" in maps, "cudart": "libcudart" in maps,
                  "oracle": "libk2oracle" in maps}), file=sys.stderr)
''' % ROOT
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
    loaded = json.loads(r.stderr.strip().splitlines()[-1])
    assert loaded == {"torch": False, "gpu_lib": False, "cudart": False, "oracle": True}
    assert line["impl"] == "reference" and line["gpu_launches"] == 0 and line["value"] > 0
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["cpu_baseline"]["kind"] == "port"
    assert 0.69 < line["run"]["table_load"] < 0.72
    sys.path.insert(0, ROOT)
    import bench
    saved = sys.argv
    try:
        sys.argv = ["bench.py", "--capacity-log2", "18", "--pairs-per-launch", "4000"]
        ours = bench.workload_config(bench.parse_args())
    finally:
        sys.argv = saved
    assert ours == line["config"]  # the driver's same_config check


def test_dump_outputs_is_bounded_and_repeatable(tmp_path):
    sys.path.insert(0, ROOT)
    import bench
    rng = np.random.default_rng(3)
    small = rng.choice(np.array([0, 9606, 9100404], np.int32), size=1000)
    bench.dump_outputs(str(tmp_path / "s"), small, (small == 0).astype(np.uint8))
    assert sorted(os.listdir(tmp_path / "s")) == ["call.npy", "keep.npy"]
    call = np.load(tmp_path / "s" / "call.npy")
    assert call.dtype == np.float64 and np.array_equal(call, small)
    assert np.load(tmp_path / "s" / "keep.npy").dtype == np.float32
    big = rng.integers(0, 1 << 31, size=10_000_000, dtype=np.int64).astype(np.int32)  # one default step: 10 x 1M pairs
    keep = (big & 1).astype(np.uint8)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), big, keep)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["call.npy", "index.npy", "keep.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64_000_000
    for f in files:
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f))
    idx = np.load(tmp_path / "a" / "index.npy").astype(np.int64)
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "call.npy"), big[idx].astype(np.uint32))
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "keep.npy"), keep[idx])


def test_steps_must_be_positive(monkeypatch):
    sys.path.insert(0, ROOT)
    import bench
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "0"])
    with pytest.raises(SystemExit):
        bench.parse_args()
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "3", "--dump-outputs", "d"])
    args = bench.parse_args()
    assert args.steps == 3 and args.dump_outputs == "d"


def test_workload_shapes():
    sys.path.insert(0, ROOT)
    import bench
    L = bench.ont_lengths(np.random.default_rng(7), 150_000_000)
    s = np.sort(L)[::-1]
    n50 = s[np.searchsorted(np.cumsum(s), s.sum() / 2)]
    assert 8_000 < n50 < 12_500 and L.max() == 100_000 and L.min() >= 200 and 150_000_000 <= L.sum() < 150_200_000
    names = [w[0] for w in bench.workload_list(None)]
    assert names[0].startswith("configs[2]") and sum(n.startswith("configs[4]") for n in names) == 7
    off = bench.workload_offsets(300, 150_000_000, 7)
    assert (np.diff(off) == 300).all() and off[-1] == 150_000_000
