"""Database build without a GPU: nh_build_taxonomy against the oracle's taxonomy builder, its errors, the
ABI mirrors of the build structures, and the kraken2-build shim's host side."""
import ctypes as C
import glob
import os
import subprocess

import pytest

import build_inputs as bi
import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INCLUDE = os.path.join(ROOT, "include")
SHIM = os.path.join(ROOT, "nohuman_b200", "bin", "kraken2-build")

MAP_TAXIDS = [562, 9606, 564]


def write_map(path, entries):
    with open(path, "w") as f:
        for sid, tid in entries:
            f.write(f"{sid}\t{tid}\n")
    return path


def test_taxonomy_is_the_oracles_image(oracle, tmp_path):
    from nohuman_b200 import api
    nodes, names = bi.write_dmp(str(tmp_path), seed=3)
    mp = write_map(str(tmp_path / "seqid2taxid.map"), [(f"s{i}", t) for i, t in enumerate(MAP_TAXIDS)])
    out = str(tmp_path / "taxo.k2d")
    n = api.build_taxonomy(nodes, names, mp, out)
    mk = bi.marked(MAP_TAXIDS)
    tax, _ = bi.oracle_taxonomy(oracle, mk)
    want = bi.oracle_taxo_bytes(oracle, tax, str(tmp_path))
    assert open(out, "rb").read() == want
    assert n == len(mk) + 1 == tax.node_count


def test_marked_set_is_map_taxids_and_ancestors(oracle, tmp_path):
    from nohuman_b200 import api
    nodes, names = bi.write_dmp(str(tmp_path), seed=5)
    for taxids in ([1423], [562, 564], [9606, 1423, 562]):
        mp = write_map(str(tmp_path / "m.map"), [(f"x{i}", t) for i, t in enumerate(taxids)])
        out = str(tmp_path / "t.k2d")
        api.build_taxonomy(nodes, names, mp, out)
        got = oracle.Taxonomy()
        assert oracle.lib().k2o_load_taxonomy(out.encode(), C.byref(got)) == 0
        ext = {got.nodes[i].external_id for i in range(1, got.node_count)}
        assert ext == bi.marked(taxids)
        assert not ext & {t[0] for t in bi.UNMARKED}
        for i in range(2, got.node_count):  # parent < child, root first
            assert got.nodes[i].parent_id < i
        assert got.nodes[1].external_id == 1


def _error(tmp_path, nodes_lines=None, names_lines=None, map_lines=None):
    from nohuman_b200 import NhError, api
    from nohuman_b200._ffi import NH_ERR_IO
    nodes, names = bi.write_dmp(str(tmp_path))
    if nodes_lines is not None:
        with open(nodes, "a") as f:
            f.writelines(nodes_lines)
    if names_lines is not None:
        with open(names, "a") as f:
            f.writelines(names_lines)
    mp = str(tmp_path / "seqid2taxid.map")
    with open(mp, "w") as f:
        f.writelines(map_lines if map_lines is not None else ["a\t562\n"])
    with pytest.raises(NhError) as ei:
        api.build_taxonomy(nodes, names, mp, str(tmp_path / "taxo.k2d"))
    assert ei.value.code == NH_ERR_IO
    return ei.value.message


def test_taxonomy_errors_name_file_and_line(tmp_path):
    n_nodes = len(synth.TAXONOMY_CFG1) + len(bi.UNMARKED)
    m = _error(tmp_path, map_lines=["a\t562\n", "b\t424242\n"])
    assert "seqid2taxid.map:2:" in m and "424242 is not in nodes.dmp" in m
    m = _error(tmp_path, nodes_lines=["77\t|\t78\t|\tgenus\t|\n", "78\t|\t77\t|\tgenus\t|\n"], map_lines=["c\t77\n"])
    assert "nodes.dmp:" in m and "parent cycle" in m
    assert f"nodes.dmp:{n_nodes + 1}:" in m or f"nodes.dmp:{n_nodes + 2}:" in m
    m = _error(tmp_path, nodes_lines=["90\t|\t91\t|\tgenus\t|\n"], map_lines=["a\t562\n", "d\t90\n"])
    assert f"nodes.dmp:{n_nodes + 1}:" in m and "does not reach taxid 1" in m
    m = _error(tmp_path, nodes_lines=["92\t|\t92\t|\tgenus\t|\n"], map_lines=["d\t92\n"])
    assert "does not reach taxid 1" in m and "is itself" in m
    m = _error(tmp_path, nodes_lines=["93 92 genus\n"])
    assert f"nodes.dmp:{n_nodes + 1}: malformed nodes.dmp line" in m
    m = _error(tmp_path, names_lines=["abc\t|\tname\t|\t\t|\tscientific name\t|\n"])
    assert f"names.dmp:{3 * n_nodes + 1}: malformed names.dmp line" in m
    m = _error(tmp_path, map_lines=["a\t562\n", "\n", "b\tnotanumber\n"])
    assert "seqid2taxid.map:3: malformed seqid2taxid line" in m


def test_build_structs_match_the_header(tmp_path):
    from nohuman_b200 import _ffi
    prog = ('#include <stdio.h>\n#include "nohuman_gpu.h"\n'
            'int main(void){printf("%zu %zu\\n", sizeof(nh_build_params_t), sizeof(nh_build_stats_t));return 0;}\n')
    (tmp_path / "s.c").write_text(prog)
    subprocess.check_call(["gcc", "-I", INCLUDE, "-o", str(tmp_path / "s"), str(tmp_path / "s.c")])
    sizes = [int(x) for x in subprocess.check_output([str(tmp_path / "s")]).split()]
    assert sizes == [C.sizeof(_ffi.BuildParams), C.sizeof(_ffi.BuildStats)]


def stage_db_dir(d, with_map=True, prelim=None):
    """kraken2-build's layout: DIR/taxonomy/{nodes,names}.dmp, DIR/library/**, DIR/seqid2taxid.map."""
    bi.write_dmp(os.path.join(d, "taxonomy"))
    lib = os.path.join(d, "library", "added")
    os.makedirs(lib)
    with open(os.path.join(lib, "a.fna"), "w") as f:
        f.write(">kraken:taxid|562|s1 x\n" + "ACGT" * 30 + "\n")
    if with_map:
        write_map(os.path.join(d, "seqid2taxid.map"), [("kraken:taxid|562|s1", 562)])
    if prelim is not None:
        with open(os.path.join(lib, "prelim_map_abc.txt"), "w") as f:
            f.writelines(prelim)


def no_device():
    from nohuman_b200 import _ffi
    return _ffi.lib().nh_device_count() == 0


def test_kraken2_build_without_device_fails_and_writes_nothing(tmp_path):
    assert os.access(SHIM, os.X_OK)
    if not no_device():
        pytest.skip("a CUDA device is present")
    d = str(tmp_path / "db")
    stage_db_dir(d)
    r = subprocess.run([SHIM, "--build", "--db", d, "--threads", "2"], capture_output=True, text=True)
    assert r.returncode != 0
    assert "no CUDA device" in r.stderr
    assert not glob.glob(os.path.join(d, "**", "*.k2d*"), recursive=True)


@pytest.mark.parametrize("flag", [["--download-taxonomy"], ["--download-library", "bacteria"],
                                  ["--add-to-library", "x.fna"], ["--standard"], ["--special", "greengenes"],
                                  ["--clean"]])
def test_kraken2_build_unsupported_modes(tmp_path, flag):
    r = subprocess.run([SHIM, *flag, "--db", str(tmp_path)], capture_output=True, text=True)
    assert r.returncode != 0
    lines = r.stderr.strip().splitlines()
    assert len(lines) == 1 and "not supported" in lines[0] and flag[0] in lines[0]


def test_kraken2_build_writes_map_from_prelim_taxid_lines(tmp_path):
    d = str(tmp_path / "db")
    stage_db_dir(d, with_map=False, prelim=["TAXID\tkraken:taxid|562|s1\t562\n", "TAXID\tother\t9606\n"])
    r = subprocess.run([SHIM, "--build", "--db", d], capture_output=True, text=True)
    assert open(os.path.join(d, "seqid2taxid.map")).read() == "kraken:taxid|562|s1\t562\nother\t9606\n"
    if no_device():
        assert r.returncode != 0 and "no CUDA device" in r.stderr


def test_kraken2_build_refuses_accnum_lines(tmp_path):
    d = str(tmp_path / "db")
    stage_db_dir(d, with_map=False, prelim=["TAXID\ts1\t562\n", "ACCNUM\ts2\tNC_000913.3\n"])
    r = subprocess.run([SHIM, "--build", "--db", d], capture_output=True, text=True)
    assert r.returncode != 0 and "accession2taxid" in r.stderr
    assert not os.path.exists(os.path.join(d, "seqid2taxid.map"))
