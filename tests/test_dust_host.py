"""DUST masking without a GPU: the CPU restatement of sdust (tests/native/dust_oracle.c) against a
brute-force enumeration of the definition (DESIGN.md §4f), the ABI mirrors of the DUST structures, the
`dustmasker` shim's argument handling, the kraken2-build shim's pointer to it, and a real dustmasker when
one is on $PATH."""
import ctypes as C
import os
import random
import shutil
import subprocess

import pytest

import dust_inputs as di
import dust_oracle as do

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INCLUDE = os.path.join(ROOT, "include")
BIN = os.path.join(ROOT, "nohuman_b200", "bin")
SHIM = os.path.join(BIN, "dustmasker")


@pytest.fixture(scope="module")
def seqs():
    rng = random.Random(20261022)
    return [di.gen(rng, rng.randint(3, 300)) for _ in range(300)]


def test_known_answers():
    for seq, want in di.KNOWN:
        assert di.brute(seq) == want
        assert do.dust_mask([seq]) == [want]


@pytest.mark.parametrize("window", [64, 33, 16, 8])
@pytest.mark.parametrize("level", [10, 20, 40])
def test_restatement_is_the_definition(seqs, window, level):
    got = do.dust_mask(seqs, window, level)
    for s, g in zip(seqs, got):
        assert g == di.brute(s, window, level), s
    if (window, level) == (64, 20):
        assert sum(c >= ord("a") for g in got for c in g) > 10_000  # the set masks plenty


def test_restatement_refuses_out_of_range():
    for w, t in ((3, 20), (65, 20), (64, 0), (64, 256)):
        with pytest.raises(ValueError):
            do.dust_mask([b"ACGT"], w, t)


def test_dust_structs_match_the_header(tmp_path):
    from nohuman_b200 import _ffi
    prog = ('#include <stdio.h>\n#include "nohuman_gpu.h"\n'
            'int main(void){printf("%zu %zu\\n", sizeof(nh_dust_params_t), sizeof(nh_dust_stats_t));return 0;}\n')
    (tmp_path / "s.c").write_text(prog)
    subprocess.check_call(["gcc", "-I", INCLUDE, "-o", str(tmp_path / "s"), str(tmp_path / "s.c")])
    sizes = [int(x) for x in subprocess.check_output([str(tmp_path / "s")]).split()]
    assert sizes == [C.sizeof(_ffi.DustParams), C.sizeof(_ffi.DustStats)]


@pytest.mark.parametrize("args,word", [(["-in", "x.fa", "-linker", "2"], "-linker"),
                                       (["-in", "x.fa", "-outfmt", "acclist"], "acclist"),
                                       (["-in", "x.fa", "-window", "65"], "-window 65"),
                                       (["-in", "x.fa", "-level", "0"], "-level 0"),
                                       (["-in"], "-in")])
def test_dustmasker_refuses(tmp_path, args, word):
    r = subprocess.run([SHIM, *args], capture_output=True, text=True, cwd=tmp_path)
    assert r.returncode != 0
    lines = r.stderr.strip().splitlines()
    assert len(lines) == 1 and word in lines[0], r.stderr
    assert os.listdir(tmp_path) == []


def no_device():
    from nohuman_b200 import _ffi
    return _ffi.lib().nh_device_count() == 0


def test_dustmasker_without_device_fails_and_writes_nothing(tmp_path):
    if not no_device():
        pytest.skip("a CUDA device is present")
    fa = tmp_path / "in.fa"
    fa.write_bytes(b">a\n" + b"CA" * 50 + b"\n")
    out = tmp_path / "out.fa"
    r = subprocess.run([SHIM, "-in", str(fa), "-out", str(out), "-outfmt", "fasta"], capture_output=True, text=True)
    assert r.returncode != 0 and "no CUDA device" in r.stderr
    assert not out.exists()


def test_add_to_library_names_the_dustmasker_route(tmp_path):
    r = subprocess.run([os.path.join(BIN, "kraken2-build"), "--add-to-library", "x.fna", "--db", str(tmp_path)],
                       capture_output=True, text=True)
    lines = r.stderr.strip().splitlines()
    assert r.returncode != 0 and len(lines) == 1
    assert "not supported" in lines[0] and "dustmasker -in F -outfmt fasta" in lines[0]
    assert "nohuman_b200/bin/dustmasker" in lines[0]


def real_dustmasker():
    exe = shutil.which("dustmasker")
    if not exe or os.path.realpath(exe) == os.path.realpath(SHIM):
        return None
    try:
        v = subprocess.run([exe, "-version"], capture_output=True, text=True, timeout=20).stdout
    except Exception:
        return None
    return exe if "dustmasker" in v else None


@pytest.mark.skipif(real_dustmasker() is None, reason="no NCBI dustmasker on PATH (its output stays unpinned)")
def test_shim_matches_real_dustmasker(tmp_path, seqs):
    fa = tmp_path / "in.fa"
    fa.write_bytes(b"".join(b">s%d\n" % i + s + b"\n" for i, s in enumerate(seqs)))
    outs = []
    for exe in (real_dustmasker(), SHIM):
        o = tmp_path / f"out{len(outs)}.txt"
        r = subprocess.run([exe, "-in", str(fa), "-out", str(o), "-outfmt", "interval"], capture_output=True, text=True)
        if r.returncode != 0 and exe == SHIM and no_device():
            pytest.skip("the shim needs a CUDA device")
        assert r.returncode == 0, r.stderr
        outs.append(o.read_bytes())
    assert outs[0] == outs[1]
