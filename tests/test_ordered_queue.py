"""nohuman_b200/csrc/nh_ordered.h (the ordered work queue behind the file pipeline's BGZF reader, block
writer and classifier hand-off) built on the host with ThreadSanitizer and driven by
tests/native/ordered_check.cc: pop order equals entry order under several pushers and workers with random
delays, the window bound, batch takes, claimed and done entries, close() draining and stop() releasing
blocked calls."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_ordered_queue_under_thread_sanitizer(tmp_path):
    exe = str(tmp_path / "ordered_check")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-g", "-fsanitize=thread", "-pthread", "-o", exe,
                           os.path.join(ROOT, "tests", "native", "ordered_check.cc")])
    # a broken queue shows as a hang as often as a failed check
    out = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0 and out.stdout.strip() == "OK", out.stdout + out.stderr
    assert "ThreadSanitizer" not in out.stderr, out.stderr
