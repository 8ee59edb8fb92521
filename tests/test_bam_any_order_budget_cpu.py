"""CPU tests of the device-memory budget of BAM mode in any record order (`nimble --any-order --device-budget SIZE`,
process_bam(..., any_order=True, device_budget=...)): the argument checks, all refused before any device work, and the
UMI bucket that splits the passes against a restatement in Python."""
import os
import subprocess

import pytest

import nimble_aligner_b200 as nb

LIB = os.path.join(os.path.dirname(__file__), "golden", "ref", "libraries", "basic.json")
CLI = os.path.join(os.path.dirname(nb.SO_PATH), "nimble")
ANY = ["--any-order", "--cell-matrix", "m", "--no-rows"]
MALFORMED = "--device-budget needs a positive number of bytes"


def run(tmp_path, *extra):
    return subprocess.run([CLI, "-r", LIB, "-i", str(tmp_path / "missing.bam")] + list(extra), capture_output=True, text=True, cwd=tmp_path)


def test_cli_refuses_a_budget_without_any_order(tmp_path):
    p = run(tmp_path, "--cell-matrix", "m", "--no-rows", "--device-budget", "1G")
    assert p.returncode == 101 and "--device-budget needs --any-order" in p.stderr, p.stderr
    assert not os.path.exists(tmp_path / "m")


@pytest.mark.parametrize("value", ["", "0", "-1", "12Q", "1.5G", "1g", "G", "12KB", "99999999999999999999", "17179869184G"])
def test_cli_refuses_malformed_budgets(tmp_path, value):
    p = run(tmp_path, *ANY, "--device-budget", value)
    assert p.returncode == 101 and MALFORMED in p.stderr, p.stderr
    assert not os.path.exists(tmp_path / "m")


@pytest.mark.parametrize("value", ["1", "4096", "64K", "3M", "2G", "16777215G"])
def test_cli_parses_sizes(tmp_path, value):
    # a well-formed size passes the parser and is then refused for the missing --any-order, before any device work
    p = run(tmp_path, "--cell-matrix", "m", "--no-rows", "--device-budget", value)
    assert p.returncode == 101 and MALFORMED not in p.stderr and "--device-budget needs --any-order" in p.stderr, p.stderr


def test_cli_refuses_a_missing_value(tmp_path):
    p = run(tmp_path, *ANY, "--device-budget")
    assert p.returncode == 101 and "--device-budget" in p.stderr


def test_help_lists_the_budget():
    out = subprocess.run([CLI, "--help"], capture_output=True, text=True, check=True).stdout
    assert "--device-budget" in out and "K/M/G" in out


def test_python_refuses_a_budget_without_any_order_or_out_of_range(tmp_path):
    for kw in (dict(device_budget=1 << 20), dict(device_budget=1 << 20, matrix_dirs=[str(tmp_path / "m")])):
        with pytest.raises(nb.NbError) as e:
            nb.process_bam(str(tmp_path / "x.bam"), [LIB], None, **kw)
        assert e.value.code == -1 and "any_order" in str(e.value)
    for bad in (0, -1, 1.5, "1G", True):
        with pytest.raises(nb.NbError) as e:
            nb.process_bam(str(tmp_path / "x.bam"), [LIB], None, matrix_dirs=[str(tmp_path / "m")], any_order=True, device_budget=bad)
        assert e.value.code == -1
        with pytest.raises(nb.NbError):
            nb.bam_dump_scopes_any_order(str(tmp_path / "x.bam"), str(tmp_path / "d.tsv"), device_budget=bad)
    assert not os.path.exists(tmp_path / "m") and not os.path.exists(tmp_path / "d.tsv")


def pack_umi(s):
    """bam_group.hpp pack_umi: A C G N T as 1..5, first character in bits 62..60, 3 bits each"""
    k = 0
    for i, c in enumerate(s):
        k |= "ACGNT".index(c) + 1 << (60 - 3 * i)
    return k


def bucket(umi):
    """the top 16 bits of the splitmix64 finalizer of the packed UMI"""
    m = (1 << 64) - 1
    k = pack_umi(umi)
    k ^= k >> 30; k = (k * 0xBF58476D1CE4E5B9) & m
    k ^= k >> 27; k = (k * 0x94D049BB133111EB) & m
    k ^= k >> 31
    return k >> 48


def test_umi_bucket_matches_the_restatement():
    umis = ["A", "T", "N", "ACGT", "TTTTTTTTTTTT", "AAAAAAAAAA", "TGTGTGTGTGTG", "CCCCAAAATTTT", "ACGTACGTACGTACGTACGTA", "NNNNNNNNNNNNNNNN"]
    umis += ["".join("ACGNT"[(i * 7 + j * 3) % 5] for j in range(1 + i % 21)) for i in range(200)]
    got = [nb.any_order_umi_bucket(u) for u in umis]
    assert got == [bucket(u) for u in umis]
    assert len(set(got)) > 100 and all(0 <= b < 65536 for b in got)
    assert bucket("A") == nb.any_order_umi_bucket("A") and pack_umi("A") == 1 << 60
    for bad in ("", "ACGT-ACGT", "A" * 22):
        with pytest.raises(nb.NbError) as e:
            nb.any_order_umi_bucket(bad)
        assert e.value.code == -5
