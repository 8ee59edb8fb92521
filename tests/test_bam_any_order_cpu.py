"""CPU tests of BAM mode in any record order: the `nimble --any-order` argument checks (all refused before any device work)
and the definition of the scopes, tests/any_order_ref.groups_any_order, on small hand-made record lists."""
import os
import subprocess

import pytest

import nimble_aligner_b200 as nb
from oracle import bam_ref
from synth import bamio
from tests import any_order_ref

LIB = os.path.join(os.path.dirname(__file__), "golden", "ref", "libraries", "basic.json")
CLI = os.path.join(os.path.dirname(nb.SO_PATH), "nimble")


@pytest.mark.parametrize("extra", [
    ["--cell-matrix", "m"],                                   # without --no-rows
    ["--no-rows"],                                            # without --cell-matrix
    ["--cell-matrix", "m", "-o", "o.tsv.gz"],                 # TSV rows
    ["--cell-matrix", "m", "--no-rows", "-o", "o.tsv.gz"],
    ["--cell-matrix", "m", "--no-rows", "-p"],                # mate pairing
])
def test_cli_refuses_any_order_combinations(tmp_path, extra):
    p = subprocess.run([CLI, "-r", LIB, "-i", str(tmp_path / "missing.bam"), "--any-order"] + extra, capture_output=True, text=True, cwd=tmp_path)
    assert p.returncode == 101, p.stdout + p.stderr
    assert not os.path.exists(tmp_path / "m") and not os.path.exists(tmp_path / "o.tsv.gz")


def test_cli_refuses_any_order_on_fastq(tmp_path):
    fq = tmp_path / "r.fastq"
    fq.write_text("@a\nACGT\n+\nIIII\n")
    p = subprocess.run([CLI, "-r", LIB, "-i", str(fq), "--any-order", "--cell-matrix", "m", "--no-rows"], capture_output=True, text=True, cwd=tmp_path)
    assert p.returncode == 101 and "--any-order" in p.stderr
    assert not os.path.exists(tmp_path / "m")


def test_help_lists_any_order():
    out = subprocess.run([CLI, "--help"], capture_output=True, text=True, check=True).stdout
    assert "--any-order" in out


def test_python_refuses_rows_pairing_and_missing_dirs(tmp_path):
    for kw in (dict(matrix_dirs=[str(tmp_path / "m")], force_bam_paired=True), dict(matrix_dirs=None)):
        with pytest.raises(nb.NbError) as e:
            nb.process_bam(str(tmp_path / "x.bam"), [LIB], None, any_order=True, **kw)
        assert e.value.code == -1
    with pytest.raises(nb.NbError) as e:
        nb.process_bam(str(tmp_path / "x.bam"), [LIB], [str(tmp_path / "o.tsv.gz")], matrix_dirs=[str(tmp_path / "m")], any_order=True)
    assert e.value.code == -1


def rec(name, flag, cb=None, ub=None, ur=None, seq="ACGTACGTAC"):
    tags = [(t, "Z", v) for t, v in (("CB", cb), ("UB", ub), ("UR", ur)) if v is not None]
    raw = bamio.encode_record(name, flag, seq, bytes([30] * len(seq)), tags)
    r = bam_ref.Record(raw[4:])
    return r


def ordinals(recs):
    for i, r in enumerate(recs):
        r.ordinal = i
    return recs


def scopes(groups):
    """-> [[(ordinal, skip_align), ...] per scope], items in order (sequence slot, mate slot, ...)"""
    return [[(it["ordinal"], it["f"][37]) for it in g] for g in groups]


def test_groups_any_order_sorts_filters_and_pairs():
    recs = ordinals([
        rec("a", 0, "CCCC-1", "TTT"),           # 0
        rec("b", 0, "AAAA-1", "GGG"),           # 1
        rec("n", 0, None, "GGG"),               # 2 no CB: skipped
        rec("w", 0, "AAAA-1", "AAAAAAAAAA"),    # 3 whitelisted UMI: skipped
        rec("c", 0, "AAAA-2", "GGG"),           # 4 same UMI, same CB[..len-2] as 1: same scope, after it
        rec("d", 0, "BBBB-1", "GGG", ur="X"),   # 5 UB wins over UR; a second CB under GGG: a scope of its own
        rec("e", 0, "CCCC-1", None, ur="TTT"),  # 6 UR when UB is missing: joins record 0
    ])
    got = scopes(any_order_ref.groups_any_order(recs))
    T, F = "TRUE", "FALSE"
    # unpaired records get a SKIP_ALIGN dummy; is_first is false, so the dummy takes the sequence slot
    assert got == [[(1, T), (1, F), (4, T), (4, F)], [(5, T), (5, F)], [(0, T), (0, F), (6, T), (6, F)]]


def test_groups_any_order_pairs_mates_and_keeps_the_filter_paired_quirk():
    recs = ordinals([
        rec("m", 1 | 128, "AAAA-1", "CCC"),     # 0 last in template
        rec("u", 0, "AAAA-1", "CCC"),           # 1
        rec("m", 1 | 64, "AAAA-1", "CCC"),      # 2 first in template
        rec("q", 1 | 64, "AAAA-1", "GGG"),      # 3 paired record ...
        rec("q", 0, "AAAA-1", "GGG"),           # 4 ... next to an unpaired one with the same name
        rec("z", 1, "AAAA-1", "GGG"),           # 5 a lone paired record: dropped
    ])
    got = scopes(any_order_ref.groups_any_order(recs))
    T, F = "TRUE", "FALSE"
    # CCC: m(0), u(1), u-dummy, m(2) in ordinal order: m(0) and u differ -> m(0) dropped; u + dummy pair; m(2) alone dropped.
    # GGG: q(3) + q(4) pair (q(3) is first in template), then q(4)'s dummy and z are left alone.
    assert got == [[(1, T), (1, F)], [(3, F), (4, F)]]


def test_groups_any_order_edge_inputs():
    assert any_order_ref.groups_any_order([]) == []
    assert any_order_ref.groups_any_order(ordinals([rec("n", 0, None, "GGG"), rec("w", 0, "A-1", "AAAAAAAAAA")])) == []
    with pytest.raises(RuntimeError, match="Could not read UMI"):
        any_order_ref.groups_any_order(ordinals([rec("x", 0, "A-1")]))
    # one record: still a scope (the sentinel keeps it from being the dropped last group)
    assert scopes(any_order_ref.groups_any_order(ordinals([rec("x", 0, "A-1", "GGG")]))) == [[(0, "TRUE"), (0, "FALSE")]]
    # clone keeps the ordinal
    r = ordinals([rec("x", 0, "A-1", "GGG")])[0]
    assert r.clone().ordinal == 0


def test_ordinal_reader_groups_equal_the_oracles(tmp_path):
    """tests/any_order_ref.py restates the oracle's grouped reader only to keep each record's ordinal: on a make_bam file its
    groups are the oracle's groups_of item for item, and every item's ordinal names the record it came from."""
    import synth
    from tests.bamcases import make_bam
    L = synth.SynthLibrary(seed=1234, n_fam=20, n_all=5)
    bam = make_bam(str(tmp_path / "t.bam"), L, n_groups=200, paired_fraction=0.3)
    recs = any_order_ref.read_bam(bam)
    want = bam_ref.groups_of(bam_ref.read_bam(bam))
    got = any_order_ref._groups_of(recs)
    strip = lambda gs: [[{k: v for k, v in it.items() if k != "ordinal"} for it in g] for g in gs]   # noqa: E731
    assert strip(got) == want and len(want) > 100
    assert all(recs[it["ordinal"]].qname == it["f"][0] for g in got for it in g)
