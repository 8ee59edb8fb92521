"""CPU tests of the per-cell matrix writer (nb_write_cell_matrix: the 10x v3 layout Seurat's Read10X and scanpy's
read_10x_mtx load) and of the `nimble` CLI's --cell-matrix / --no-rows checks.  None of these reaches the GPU."""
import gzip
import os
import subprocess

import numpy as np
import pytest
import scipy.io

import nimble_aligner_b200 as nb

LIB = os.path.join(os.path.dirname(__file__), "golden", "ref", "libraries", "basic.json")
CLI = os.path.join(os.path.dirname(nb.SO_PATH), "nimble")


@pytest.fixture(scope="module")
def lib():
    return nb.Library.from_json(LIB)


def counts(rows, callsets):
    """rows: [(cell, callset, umis, reads)] in (cell, callset) order; callsets: lists of group indices."""
    off = np.concatenate([[0], np.cumsum([len(c) for c in callsets])]).astype(np.uint64)
    r = np.array(rows, dtype=np.int64).reshape(-1, 4)
    return dict(row_cell=r[:, 0], row_callset=r[:, 1], row_umis=r[:, 2], row_reads=r[:, 3], callset_off=off,
                callset_items=np.array([g for c in callsets for g in c], dtype=np.uint32), n_scopes=7)


def gz_lines(path):
    return gzip.open(path, "rt").read().split("\n")[:-1]


def test_matrix_layout_and_values(tmp_path, lib):
    names = lib.group_names()                       # A02-0 A02-1 A02-2 A02-LC KIR2DL-4
    callsets = [[0], [0, 3], [4]]
    rows = [(0, 0, 2, 5), (0, 2, 1, 1), (2, 1, 3, 9), (2, 2, 1, 2), (3, 0, 1, 1)]
    barcodes = ["AAAC-1", "AAAG-1", "CCCT-1", "GGGA-1"]
    d = tmp_path / "m"                              # created by the writer
    nb.write_cell_matrix(d, lib, counts(rows, callsets), barcodes)
    assert sorted(os.listdir(d)) == ["barcodes.tsv.gz", "features.tsv.gz", "matrix.mtx.gz", "reads.mtx.gz"]
    umis, reads = scipy.io.mmread(str(d / "matrix.mtx.gz")), scipy.io.mmread(str(d / "reads.mtx.gz"))
    assert umis.shape == reads.shape == (3, 4)
    want_u, want_r = np.zeros((3, 4), np.int64), np.zeros((3, 4), np.int64)
    for c, s, u, r in rows:
        want_u[s, c], want_r[s, c] = u, r
    assert np.array_equal(umis.toarray(), want_u) and np.array_equal(reads.toarray(), want_r)
    lines = gz_lines(d / "matrix.mtx.gz")
    assert lines[0] == "%%MatrixMarket matrix coordinate integer general" and lines[1] == "3 4 5"
    assert lines[2:] == ["%d %d %d" % (s + 1, c + 1, u) for c, s, u, _ in rows]      # sorted by barcode, then feature
    assert gz_lines(d / "reads.mtx.gz")[2:] == ["%d %d %d" % (s + 1, c + 1, r) for c, s, _, r in rows]
    feats = [",".join(names[g] for g in cs) for cs in callsets]
    assert gz_lines(d / "features.tsv.gz") == ["%s\t%s\tGene Expression" % (f, f) for f in feats]
    assert gz_lines(d / "barcodes.tsv.gz") == barcodes
    for f in os.listdir(d):
        raw = open(d / f, "rb").read()
        assert raw[:4] == b"\x1f\x8b\x08\x00" and raw[4:8] == b"\0\0\0\0", f    # no FNAME flag, mtime 0
    # the same counts give the same bytes; an existing directory is written into
    before = {f: open(d / f, "rb").read() for f in os.listdir(d)}
    nb.write_cell_matrix(d, lib, counts(rows, callsets), barcodes)
    assert {f: open(d / f, "rb").read() for f in os.listdir(d)} == before


def test_empty_matrix(tmp_path, lib):
    d = tmp_path / "e"
    nb.write_cell_matrix(d, lib, counts([], []), ["AAAC-1", "CCCT-1"])
    assert gz_lines(d / "matrix.mtx.gz") == ["%%MatrixMarket matrix coordinate integer general", "0 2 0"]
    assert gz_lines(d / "reads.mtx.gz") == ["%%MatrixMarket matrix coordinate integer general", "0 2 0"]
    assert gzip.open(d / "features.tsv.gz").read() == b"" and gz_lines(d / "barcodes.tsv.gz") == ["AAAC-1", "CCCT-1"]
    d2 = tmp_path / "e2"
    nb.write_cell_matrix(d2, lib, counts([], []), [])
    assert gz_lines(d2 / "matrix.mtx.gz")[1] == "0 0 0" and gzip.open(d2 / "barcodes.tsv.gz").read() == b""


@pytest.mark.parametrize("rows,callsets,nbc,msg", [
    ([(0, 1, 1, 1), (0, 0, 1, 1)], [[0], [1]], 1, "not sorted"),
    ([(0, 0, 1, 1), (0, 0, 1, 1)], [[0]], 1, "not sorted"),
    ([(1, 0, 1, 1)], [[0]], 1, "outside"),
    ([(0, 1, 1, 1)], [[0]], 1, "outside"),
    ([(0, 0, 1, 1)], [[9]], 1, "not a group"),
])
def test_bad_counts_are_rejected(tmp_path, lib, rows, callsets, nbc, msg):
    with pytest.raises(nb.NbError, match=msg):
        nb.write_cell_matrix(tmp_path / "x", lib, counts(rows, callsets), ["C%d" % i for i in range(nbc)])


def test_missing_parent_directory_is_an_io_error(tmp_path, lib):
    with pytest.raises(nb.NbError) as e:
        nb.write_cell_matrix(tmp_path / "no" / "such", lib, counts([], []), [])
    assert e.value.code == -2


def run(*args):
    p = subprocess.run([CLI, *args], capture_output=True, text=True)
    return p.returncode, p.stdout + p.stderr


@pytest.mark.parametrize("args,msg", [
    (("-r", "a.json", "b.json", "-o", "a.tsv.gz", "b.tsv.gz", "-i", "x.bam", "--cell-matrix", "m1"), "one directory per reference library"),
    (("-r", "a.json", "-o", "a.tsv.gz", "-i", "x.bam", "--cell-matrix", "m1", "m2"), "one directory per reference library"),
    (("-r", "a.json", "-o", "a.tsv.gz", "-i", "x.bam", "--cell-matrix", "m1", "--no-rows"), "leave out --output"),
    (("-r", "a.json", "-i", "x.bam", "--no-rows"), "needs --cell-matrix"),
    (("-r", "a.json", "-o", "a.tsv", "-i", "a.fastq", "--cell-matrix", "m1"), "need a BAM input"),
    (("-r", "a.json", "-i", "a.fastq.gz", "--cell-matrix", "m1", "--no-rows"), "need a BAM input"),
])
def test_cli_cell_matrix_arguments(tmp_path, args, msg):
    assert os.path.exists(CLI)
    rc, out = run(*args)
    assert rc == 101 and msg in out, (rc, out)
    rc, out = run("--help")
    assert rc == 0 and "--cell-matrix" in out and "--no-rows" in out
