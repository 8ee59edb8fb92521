"""CPU tests of bulk BAM mode (`nimble --bulk`, process_bam(..., bulk=True)): the argument checks, and the Python restatement
tests/bulk_ref.py on hand-made records."""
import os
import subprocess

import pytest

import nimble_aligner_b200 as nb
from tests import bulk_ref
from tests.bulk_ref import PAIRED, READ1, READ2, REVERSE, SECONDARY, SUPPLEMENTARY, Rec

LIB = os.path.join(os.path.dirname(__file__), "golden", "ref", "libraries", "basic.json")
CLI = os.path.join(os.path.dirname(nb.SO_PATH), "nimble")


def run(tmp_path, inp, *extra):
    return subprocess.run([CLI, "-r", LIB, "-i", str(inp), "--bulk"] + list(extra), capture_output=True, text=True, cwd=tmp_path)


def test_cli_accepts_bulk(tmp_path):
    # past the argument checks the run starts and fails on the missing input or device, not with an argument error
    p = run(tmp_path, tmp_path / "missing.bam", "-o", "x.tsv", "-t", "40:0.9")
    assert p.returncode == 101 and "Processing as BAM file" in p.stdout, p.stdout + p.stderr
    assert not p.stderr.startswith("error:"), p.stderr


@pytest.mark.parametrize("extra,msg", [
    (["-o", "x.tsv", "--cell-matrix", "m"], "--cell-matrix"),
    (["--cell-matrix", "m", "--no-rows"], "--no-rows"),
    (["-o", "x.tsv", "--no-rows"], "--no-rows"),
    (["-o", "x.tsv", "--any-order"], "--any-order"),
    (["-o", "x.tsv", "-p"], "-p"),
    (["-o", "x.tsv", "--device-budget", "8G"], "--device-budget"),
    (["-o", "x.tsv", "-t", "40:0.9,40:0.9"], "trim options"),            # -t keeps its count check
])
def test_cli_refuses(tmp_path, extra, msg):
    p = run(tmp_path, tmp_path / "missing.bam", *extra)
    assert p.returncode == 101 and msg in p.stderr, p.stderr
    assert not os.path.exists(tmp_path / "m") and not os.path.exists(tmp_path / "x.tsv")


@pytest.mark.parametrize("name", ["r.fastq", "r.fastq.gz"])
def test_cli_refuses_fastq_input(tmp_path, name):
    fq = tmp_path / name
    fq.write_bytes(b"@a\nACGT\n+\nIIII\n")
    p = run(tmp_path, fq, "-o", "x.tsv")
    assert p.returncode == 101 and "--bulk needs a BAM input" in p.stderr, p.stderr
    assert not os.path.exists(tmp_path / "x.tsv")


def test_help_lists_bulk():
    out = subprocess.run([CLI, "--help"], capture_output=True, text=True, check=True).stdout
    assert "--bulk" in out


def test_python_refusals(tmp_path):
    out = str(tmp_path / "o.tsv")
    with pytest.raises(nb.NbError) as e:
        nb.process_bam(str(tmp_path / "missing.bam"), [LIB], [out], bulk=True)
    assert e.value.code != -1                                              # past the checks: the run itself fails
    for kw in (dict(matrix_dirs=[str(tmp_path / "m")]), dict(any_order=True), dict(force_bam_paired=True), dict(device_budget=1 << 30)):
        with pytest.raises(nb.NbError) as e:
            nb.process_bam(str(tmp_path / "x.bam"), [LIB], [out], bulk=True, **kw)
        assert e.value.code == -1
    for outs in (None, [], [out, out + "2"]):
        with pytest.raises(nb.NbError) as e:
            nb.process_bam(str(tmp_path / "x.bam"), [LIB], outs, bulk=True)
        assert e.value.code == -1 and "one output path per reference library" in str(e.value)
    assert not os.path.exists(tmp_path / "m") and not os.path.exists(out)


P1, P2 = PAIRED | READ1, PAIRED | READ2


def test_ref_kept_and_dropped():
    recs = [
        Rec("a", P1, "ACGT"), Rec("a", P2 | REVERSE, "GGTT"),                    # a pair
        Rec("a", P1 | SECONDARY, "TTTT"), Rec("a", P2 | SUPPLEMENTARY, ""),      # not kept (SEQ * allowed there)
        Rec("b", P1, "AAAA"),                                                     # singleton
        Rec("c", P1, "CCCC"), Rec("c", P1, "CCCA"),                               # two READ1s
        Rec("d", PAIRED, "GGGG"), Rec("d", P2, "GGGA"),                           # READ_OTHER
        Rec("e", PAIRED | READ1 | READ2, "TTTA"), Rec("e", P2, "TTTC"),           # both bits
        Rec("f", P1, "ACGA"), Rec("f", P2, "ACGC"), Rec("f", P2, "ACGG"),         # three records
        Rec("g", P2 | 0x200 | 0x400 | 0x4, "CATG"), Rec("g", P1 | 0x4, "GTAC"),   # QC-fail, duplicate, unmapped: kept; R2 before R1
    ]
    assert [i for i, _ in bulk_ref.kept(recs)] == [0, 1, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15]
    paired, ps = bulk_ref.pairs(recs)
    assert paired and ps == [(0, 1), (15, 14)]
    assert bulk_ref.dump_lines(recs) == ["0\t1\t4\t4\t0\t4", "15\t14\t4\t4\t0\t0"]


def test_ref_names_compare_exactly():
    long_a, long_b = "x" * 253 + "a", "x" * 253 + "b"
    recs = [Rec(long_a, P1, "A"), Rec(long_b, P2, "C"), Rec(long_b, P1, "G"), Rec(long_a, P2, "T"),
            Rec("ab", P1, "AC"), Rec("a", P2, "GT"), Rec("abc", P2, "TT")]
    assert bulk_ref.pairs(recs) == (True, [(0, 3), (2, 1)])


def test_ref_reverse_with_iupac():
    r = Rec("n", P2 | REVERSE, "ACGTNRYM=")
    assert bulk_ref.fastq_text(r) == "=KRYNACGT"
    assert bulk_ref.fastq_mode(bulk_ref.fastq_text(r)) == "AAAAAACGT"    # non-ACGT stays A after the complement, unlike BAM mode's T
    f = Rec("n", P1, "ACGTNRYM=")
    assert bulk_ref.fastq_mode(bulk_ref.fastq_text(f)) == "ACGTAAAAA"


def test_ref_single_end_and_refusals(tmp_path):
    recs = [Rec("s1", 0, "ACGT"), Rec("s2", REVERSE, "AACC"), Rec("s3", SECONDARY, "GG"), Rec("s1", 0, "TTTT")]
    assert bulk_ref.pairs(recs) == (False, [(0, None), (1, None), (3, None)])
    assert bulk_ref.dump_lines(recs) == ["0\t-\t4\t-\t0\t-", "1\t-\t4\t-\t4\t-", "3\t-\t4\t-\t0\t-"]
    paths = bulk_ref.write_fastqs(recs, tmp_path)
    assert len(paths) == 1 and open(paths[0]).read() == "@s1\nACGT\n+\nIIII\n@s2\nGGTT\n+\nIIII\n@s1\nTTTT\n+\nIIII\n"
    with pytest.raises(bulk_ref.Refused, match="record 1 is paired and record 0 is not"):
        bulk_ref.pairs([Rec("a", 0, "A"), Rec("a", P1, "C")])
    with pytest.raises(bulk_ref.Refused, match="record 1 has no SEQ"):
        bulk_ref.pairs([Rec("a", P1, "A"), Rec("b", P1, "")])
    assert bulk_ref.pairs([Rec("a", SECONDARY, "")]) == (False, [])
