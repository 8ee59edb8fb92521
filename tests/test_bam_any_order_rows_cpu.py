"""CPU tests of the TSV.gz rows of BAM mode in any record order (`nimble --any-order -o`, process_bam(..., output_paths,
any_order=True)): the argument checks that accept the rows mode and the combinations that stay refused."""
import os
import subprocess

import pytest

import nimble_aligner_b200 as nb

LIB = os.path.join(os.path.dirname(__file__), "golden", "ref", "libraries", "basic.json")
CLI = os.path.join(os.path.dirname(nb.SO_PATH), "nimble")


def run(tmp_path, *extra):
    return subprocess.run([CLI, "-r", LIB, "-i", str(tmp_path / "missing.bam"), "--any-order"] + list(extra), capture_output=True, text=True, cwd=tmp_path)


@pytest.mark.parametrize("extra", [["-o", "x.tsv.gz"], ["-o", "x.tsv.gz", "--device-budget", "8G"]])
def test_cli_accepts_rows_in_any_order(tmp_path, extra):
    # past the argument checks the run starts and fails on the missing input or device, not with an argument error
    p = run(tmp_path, *extra)
    assert p.returncode == 101 and "Processing as BAM file" in p.stdout, p.stdout + p.stderr
    assert not p.stderr.startswith("error:"), p.stderr


@pytest.mark.parametrize("extra,msg", [
    (["-o", "x.tsv.gz", "--cell-matrix", "m"], "run the two modes separately"),      # rows and matrix in one run
    (["--cell-matrix", "m"], "run the two modes separately"),
    (["-o", "x.tsv.gz", "-p"], "-p"),                                                 # mate pairing
    (["-o", "x.tsv.gz", "--no-rows"], "--no-rows"),                                    # --no-rows without --cell-matrix
    (["--no-rows"], "--no-rows"),
])
def test_cli_still_refuses(tmp_path, extra, msg):
    p = run(tmp_path, *extra)
    assert p.returncode == 101 and msg in p.stderr, p.stderr
    assert not os.path.exists(tmp_path / "m") and not os.path.exists(tmp_path / "x.tsv.gz")


def test_cli_refuses_rows_in_any_order_on_fastq(tmp_path):
    fq = tmp_path / "r.fastq"
    fq.write_text("@a\nACGT\n+\nIIII\n")
    p = subprocess.run([CLI, "-r", LIB, "-i", str(fq), "--any-order", "-o", "x.tsv.gz"], capture_output=True, text=True, cwd=tmp_path)
    assert p.returncode == 101 and "--any-order" in p.stderr
    assert not os.path.exists(tmp_path / "x.tsv.gz")


def test_help_mentions_rows_in_any_order():
    out = subprocess.run([CLI, "--help"], capture_output=True, text=True, check=True).stdout
    assert "TSV.gz rows in any order" in out


def test_python_passes_the_argument_checks_and_refuses_the_rest(tmp_path):
    out = str(tmp_path / "o.tsv.gz")
    with pytest.raises(nb.NbError) as e:
        nb.process_bam(str(tmp_path / "missing.bam"), [LIB], [out], any_order=True)
    assert e.value.code != -1                                                          # past the checks: the run itself fails
    for kw in (dict(matrix_dirs=[str(tmp_path / "m")]), dict(force_bam_paired=True)):
        with pytest.raises(nb.NbError) as e:
            nb.process_bam(str(tmp_path / "x.bam"), [LIB], [out], any_order=True, **kw)
        assert e.value.code == -1
    with pytest.raises(nb.NbError) as e:
        nb.process_bam(str(tmp_path / "x.bam"), [LIB], [out], any_order=True, matrix_dirs=[str(tmp_path / "m")])
    assert "separately" in str(e.value)
    for outs in ([], [out, out + "2"]):                                                 # one output per library
        with pytest.raises(nb.NbError) as e:
            nb.process_bam(str(tmp_path / "x.bam"), [LIB], outs, any_order=True)
        assert e.value.code == -1 and "one output path per reference library" in str(e.value)
    for bad in (0, -1, 1.5, "1G", True):
        with pytest.raises(nb.NbError) as e:
            nb.process_bam(str(tmp_path / "x.bam"), [LIB], [out], any_order=True, device_budget=bad)
        assert e.value.code == -1
    assert not os.path.exists(tmp_path / "m")
