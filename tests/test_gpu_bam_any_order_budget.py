"""GPU tests of BAM mode in any record order under a device-memory budget (nb_process_bam_cells_any_order_budget,
`nimble --any-order --device-budget SIZE`).  The budgets are small against the test files, never against the device: they
are what forces the passes.  Every budgeted run must write the bytes of the unbudgeted run, and the unbudgeted run is held
against the oracle."""
import collections
import gzip
import os
import re
import subprocess

import numpy as np
import pytest

import nimble_aligner_b200 as nb
from oracle import bam_ref
from synth import bamio
from tests import any_order_ref
from tests.bamcases import make_bam
from tests.test_gpu_bam_any_order import edge_units, enc, oracle_any_order, shuffled
from tests.test_gpu_cell_matrix import CLI, files, library, read_matrix

pytestmark = pytest.mark.gpu

STATS = re.compile(r"store (\d+) bytes, grouping (\d+) bytes.*?(?:, budget (\d+) bytes, passes (\d+), evictions (\d+), peak device bytes (\d+), windows per pass (\S+))?$")


def cli_run(bam, libs, out_dirs, budget=None, cores=4, window_kb=None, chem="unstranded", trim=None):
    """the CLI with NB_BAM_STATS=1 -> the stats fields of its nb_process_bam_any_order line"""
    env = dict(os.environ, NB_BAM_STATS="1")
    env.pop("NB_BAM_WINDOW_KB", None)
    if window_kb:
        env["NB_BAM_WINDOW_KB"] = str(window_kb)
    args = [CLI] + [a for lib in libs for a in ("-r", lib)] + ["-i", bam, "-c", str(cores), "--strand_filter", chem, "--any-order", "--no-rows", "--cell-matrix"] + list(out_dirs)
    args += (["-t", trim] if trim else []) + (["--device-budget", str(budget)] if budget else [])
    p = subprocess.run(args, capture_output=True, text=True, env=env)
    assert p.returncode == 0, p.stderr
    line = [l for l in p.stderr.split("\n") if l.startswith("nb_process_bam_any_order:")]
    assert len(line) == 1, p.stderr
    m = STATS.search(line[0])
    assert m, line[0]
    st = dict(store=int(m.group(1)), grouping=int(m.group(2)), line=line[0])
    if budget:
        assert m.group(3), line[0]
        st.update(budget=int(m.group(3)), passes=int(m.group(4)), evictions=int(m.group(5)), peak=int(m.group(6)), windows=m.group(7).split("/"))
        assert st["budget"] == budget and len(st["windows"]) == st["passes"]
        assert st["peak"] <= budget, line[0]
    else:
        assert m.group(3) is None, line[0]                                             # the unbudgeted line keeps its format
    return st


@pytest.mark.parametrize("chem,trim", [("unstranded", None), ("fiveprime", "30:0.5"), ("threeprime", None)])
def test_budgeted_passes_write_the_unbudgeted_bytes(tmp_path, chem, trim):
    L, obj, lib_json = library(tmp_path)
    src = make_bam(str(tmp_path / "g.bam"), L, n_groups=1500, seed=21)
    bam = shuffled(src, str(tmp_path / "s.bam"), seed=3)
    assert len(gzip.open(bam, "rb").read()) > 8 * 64 * 1024                            # many 64 KB windows
    ref = str(tmp_path / "ref")
    nb.process_bam(bam, [lib_json], None, strand_filter=chem, trim=trim, num_cores=4, matrix_dirs=[ref], any_order=True)
    feats, bcs, got = read_matrix(ref)
    want_bcs, want = oracle_any_order(obj, chem, trim, bam)
    assert got == want and bcs == want_bcs and len(bcs) > 100
    base = cli_run(bam, [lib_json], [str(tmp_path / "u")], chem=chem, trim=trim)
    assert files(str(tmp_path / "u")) == files(ref)
    need = base["store"] + base["grouping"]
    for div, min_passes in ((3, 2), (8, 4), (16, 8)):
        budget = need // div
        d = str(tmp_path / ("b%d" % div))
        st = cli_run(bam, [lib_json], [d], budget=budget, window_kb=64, chem=chem, trim=trim)
        assert st["passes"] >= min_passes and st["evictions"] >= 1, st["line"]
        assert files(d) == files(ref), st["line"]
    # the Python call writes the CLI's bytes
    dp = str(tmp_path / "py")
    nb.process_bam(bam, [lib_json], None, strand_filter=chem, trim=trim, num_cores=4, matrix_dirs=[dp], any_order=True, device_budget=need // 8)
    assert files(dp) == files(ref)


def test_a_budget_well_above_the_need_takes_one_pass(tmp_path):
    L, obj, lib_json = library(tmp_path)
    bam = shuffled(make_bam(str(tmp_path / "g.bam"), L, n_groups=600, seed=5), str(tmp_path / "s.bam"), seed=4)
    base = cli_run(bam, [lib_json], [str(tmp_path / "u")])
    for budget in (4 * (base["store"] + base["grouping"]), 1 << 40):
        d = str(tmp_path / ("b%d" % budget))
        st = cli_run(bam, [lib_json], [d], budget=budget, window_kb=64)
        assert st["passes"] == 1 and st["evictions"] == 0, st["line"]
        assert files(d) == files(str(tmp_path / "u"))


def umi_of(rec):
    return bam_ref.SortedBamReader.umi_of(rec)


def clipped(rec):
    seq, qual = rec.seq, rec.qual
    x, y = 0, len(seq)
    if len(seq) == 124:
        if rec.flag & 16:
            y = 111
        else:
            x = 13
    return seq[x:y], qual[x:y].hex()


# The compaction moves the store through one scratch tile.  None: the tile the budget leaves (one tile for files this
# small); small caps make the byte runs and the per-record arrays cross many tile boundaries, at unaligned offsets.
@pytest.mark.parametrize("tile", [None, "4096", "1000"])
def test_dumped_scopes_and_store_contents_equal_the_single_pass(tmp_path, monkeypatch, tile):
    L, obj, lib_json = library(tmp_path)
    src = make_bam(str(tmp_path / "g.bam"), L, n_groups=600, tso_fraction=0.3)
    bam = shuffled(src, str(tmp_path / "s.bam"), seed=11, extra_units=edge_units(np.random.default_rng(3)))
    one, many = tmp_path / "one.tsv", tmp_path / "many.tsv"
    nb.bam_dump_scopes_any_order(bam, one, num_cores=4)
    base = cli_run(bam, [lib_json], [str(tmp_path / "u")])
    monkeypatch.setenv("NB_BAM_WINDOW_KB", "64")
    if tile:
        monkeypatch.setenv("NB_BAM_COMPACT_TILE_BYTES", tile)
    nb.bam_dump_scopes_any_order(bam, many, num_cores=4, device_budget=max((base["store"] + base["grouping"]) // 2, 2 << 20))
    single = [l.split("\t") for l in one.read_text().split("\n")[:-1]]
    multi = [l.split("\t") for l in many.read_text().split("\n")[:-1]]
    assert all(len(l) == 13 for l in multi)
    # the pair lines (cell, ordinals, flags, lengths) are the single pass's, as a multiset
    assert collections.Counter(tuple(l[1:]) for l in single) == collections.Counter(tuple(l[2:9]) for l in multi)
    recs = any_order_ref.read_bam(bam)
    # every scope lies in one pass, and the passes take the UMI buckets in increasing order
    pass_of, bucket_of = {}, {}
    for l in multi:
        pass_of.setdefault(l[1], set()).add(int(l[0]))
        bucket_of[l[1]] = nb.any_order_umi_bucket(umi_of(recs[int(l[3])]))
    assert all(len(p) == 1 for p in pass_of.values())
    order = sorted(pass_of, key=lambda s: bucket_of[s])
    passes = [next(iter(pass_of[s])) for s in order]
    assert passes == sorted(passes) and passes[-1] >= 1, "expected several passes"
    # each slot's bases and quals, read back from the store after the compactions, are the record's in the file
    for l in multi:
        for o, b, q in ((int(l[3]), l[9], l[10]), (int(l[4]), l[11], l[12])):
            assert (b, q) == clipped(recs[o]), (l[:9], o)
    assert max(collections.Counter(l[1] for l in multi).values()) >= 5000              # the big scope came through whole


@pytest.mark.parametrize("tile", ["4096", "1000"])
def test_small_compaction_tiles_write_the_unbudgeted_bytes(tmp_path, monkeypatch, tile):
    L, obj, lib_json = library(tmp_path)
    bam = shuffled(make_bam(str(tmp_path / "g.bam"), L, n_groups=1500, seed=21, tso_fraction=0.3), str(tmp_path / "s.bam"), seed=3)
    ref = str(tmp_path / "ref")
    nb.process_bam(bam, [lib_json], None, num_cores=4, matrix_dirs=[ref], any_order=True)
    want_bcs, want = oracle_any_order(obj, "unstranded", None, bam)
    _, bcs, got = read_matrix(ref)
    assert got == want and bcs == want_bcs
    base = cli_run(bam, [lib_json], [str(tmp_path / "u")])
    monkeypatch.setenv("NB_BAM_COMPACT_TILE_BYTES", tile)
    for div in (4, 12):
        d = str(tmp_path / ("b%d" % div))
        st = cli_run(bam, [lib_json], [d], budget=(base["store"] + base["grouping"]) // div, window_kb=64)
        assert st["passes"] >= 2 and st["evictions"] >= 1, st["line"]
        assert files(d) == files(ref), st["line"]


def test_a_budget_below_one_bucket_fails_and_names_both_numbers(tmp_path):
    L, obj, lib_json = library(tmp_path)
    src = make_bam(str(tmp_path / "g.bam"), L, n_groups=100)
    bam = shuffled(src, str(tmp_path / "s.bam"), seed=2, extra_units=edge_units(np.random.default_rng(3)))
    budget = 1 << 20                                                                   # the 5000-record scope's bucket needs more
    with pytest.raises(nb.NbError) as e:
        nb.process_bam(bam, [lib_json], None, num_cores=4, matrix_dirs=[str(tmp_path / "m")], any_order=True, device_budget=budget)
    msg = str(e.value)
    assert e.value.code == -6 and str(budget) in msg, msg
    need = [int(x) for x in re.findall(r"needs (\d+) bytes", msg)]
    assert need and need[0] > budget, msg
    assert "UMI bucket %d" % nb.any_order_umi_bucket("TGTGTGTGTGTG") in msg, msg


def test_budgeted_runs_are_deterministic_across_threads_and_windows(tmp_path, monkeypatch):
    L, obj, lib_json = library(tmp_path)
    bam = shuffled(make_bam(str(tmp_path / "g.bam"), L, n_groups=1500, seed=77), str(tmp_path / "s.bam"), seed=5)
    ref = str(tmp_path / "ref")
    nb.process_bam(bam, [lib_json], None, num_cores=4, matrix_dirs=[ref], any_order=True)
    base = cli_run(bam, [lib_json], [str(tmp_path / "u")])
    budget = (base["store"] + base["grouping"]) // 6
    for cores in (1, 4, 16):
        for window in (None, "64", "200"):
            monkeypatch.delenv("NB_BAM_WINDOW_KB", raising=False)
            if window:
                monkeypatch.setenv("NB_BAM_WINDOW_KB", window)
            d = str(tmp_path / ("c%d_%s" % (cores, window)))
            nb.process_bam(bam, [lib_json], None, num_cores=cores, matrix_dirs=[d], any_order=True, device_budget=budget)
            assert files(d) == files(ref), (cores, window)


def test_two_libraries_all_skipped_and_one_bucket_under_a_budget(tmp_path):
    L, obj, lib_a = library(tmp_path)
    _, obj_b, lib_b = library(tmp_path, seed=1234, group_on="", name="lib_b.json")
    bam = shuffled(make_bam(str(tmp_path / "g.bam"), L, n_groups=800), str(tmp_path / "s.bam"), seed=9)
    ua, ub = str(tmp_path / "ua"), str(tmp_path / "ub")
    base = cli_run(bam, [lib_a, lib_b], [ua, ub])
    da, db = str(tmp_path / "a"), str(tmp_path / "b")
    st = cli_run(bam, [lib_a, lib_b], [da, db], budget=(base["store"] + base["grouping"]) // 5, window_kb=64)
    assert st["passes"] >= 2 and files(da) == files(ua) and files(db) == files(ub)
    for o, d in ((obj, da), (obj_b, db)):
        want_bcs, want = oracle_any_order(o, "unstranded", None, bam)
        _, bcs, got = read_matrix(d)
        assert bcs == want_bcs and got == want
    # every record skipped
    skipped = str(tmp_path / "skipped.bam")
    bamio.write_bam(skipped, [enc("n%d" % i, 0, "ACGT" * 20, [("UB", "Z", "ACGTACGTACGT")]) for i in range(5)] +
                    [enc("w%d" % i, 0, "ACGT" * 20, [("CB", "Z", "ACGT-1"), ("UB", "Z", "AAAAAAAAAA")]) for i in range(5)])
    de, dw = str(tmp_path / "empty"), str(tmp_path / "written")
    nb.process_bam(skipped, [lib_a], None, num_cores=2, matrix_dirs=[de], any_order=True, device_budget=1 << 16)
    nb.process_bam(skipped, [lib_a], None, num_cores=2, matrix_dirs=[dw], any_order=True)
    assert files(de) == files(dw)
    # every kept record in one bucket: one UMI, many cells
    rng = np.random.default_rng(8)
    seqs = [r.seq for r in any_order_ref.read_bam(bam)[:400]]
    one = [enc("o%d" % i, 16 if i % 5 == 0 else 0, seqs[i], [("CB", "Z", "%016d-1" % (i % 37)), ("UB", "Z", "CATCATCATCAT")]) for i in range(400)]
    ob = str(tmp_path / "one.bam")
    bamio.write_bam(ob, [one[i] for i in rng.permutation(len(one))], block_bytes=4000)
    du, dbud = str(tmp_path / "one_u"), str(tmp_path / "one_b")
    base = cli_run(ob, [lib_a], [du])
    st = cli_run(ob, [lib_a], [dbud], budget=2 * (base["store"] + base["grouping"]) + (1 << 20), window_kb=64)
    assert st["passes"] == 1 and files(dbud) == files(du)
    want_bcs, want = oracle_any_order(obj, "unstranded", None, ob)
    _, bcs, got = read_matrix(du)
    assert bcs == want_bcs and got == want and len(bcs) > 10
