"""GPU tests of BAM mode in any record order (nb_process_bam_cells_any_order, `nimble --any-order`).

Every BAM is built by tests.bamcases.make_bam and rewritten as a shuffled twin: units (single records, or adjacent mate
pairs) in random order, so groups interleave across the whole file and the no-CB / AAAAAAAAAA records are scattered
among them.  The matrix of the new mode on the twin must equal groups_any_order (tests/any_order_ref.py) -> the oracle's align_groups rolled up by
cell, and the existing matrix-only run on G = the kept records in (UMI, CB) order followed by a sentinel scope."""
import collections
import gzip
import os
import subprocess

import numpy as np
import pytest

import nimble_aligner_b200 as nb
import oracle as orc
from oracle import bam_ref
from synth import bamio
from tests import any_order_ref
from tests.bamcases import make_bam
from tests.test_gpu_cell_matrix import CLI, files, library, read_matrix

pytestmark = pytest.mark.gpu


def raw_records(path):
    raw = gzip.open(path, "rb").read()
    l_text = int.from_bytes(raw[4:8], "little"); p = 8 + l_text
    n_ref = int.from_bytes(raw[p:p + 4], "little"); p += 4
    for _ in range(n_ref):
        p += 4 + int.from_bytes(raw[p:p + 4], "little") + 4
    recs = []
    while p < len(raw):
        n = int.from_bytes(raw[p:p + 4], "little"); recs.append(raw[p:p + 4 + n]); p += 4 + n
    return recs


def units_of(recs):
    """single records, or adjacent records with the same name (mate pairs)"""
    out, i = [], 0
    while i < len(recs):
        if i + 1 < len(recs) and bam_ref.Record(recs[i][4:]).qname == bam_ref.Record(recs[i + 1][4:]).qname:
            out.append(recs[i:i + 2]); i += 2
        else:
            out.append(recs[i:i + 1]); i += 1
    return out


def shuffled(src, dst, seed=7, extra_units=()):
    units = units_of(raw_records(src)) + [list(u) for u in extra_units]
    rng = np.random.default_rng(seed)
    order = rng.permutation(len(units))
    bamio.write_bam(dst, [r for i in order for r in units[i]], block_bytes=20000)
    return dst


def sorted_plus_sentinel(src, dst):
    """G: the kept records of src, stably sorted by (UMI, CB), then one scope with a UMI no record has"""
    kept = []
    for raw in raw_records(src):
        r = bam_ref.Record(raw[4:])
        cb = r.aux_string("CB")
        if cb is None:
            continue
        umi = bam_ref.SortedBamReader.umi_of(r)
        if umi != "AAAAAAAAAA":
            kept.append(((umi, cb), raw))
    kept.sort(key=lambda x: x[0])
    sentinel = bamio.encode_record("sentinel", 0, "ACGT" * 20, bytes([30] * 80), [("CB", "Z", "SENTINEL-1"), ("UB", "Z", "N" * 16)])
    bamio.write_bam(dst, [raw for _, raw in kept] + [sentinel], block_bytes=20000)
    return dst


def oracle_any_order(obj, chem, trim, bam):
    """-> (barcodes in order of the first kept record with that CB, {(feature, barcode): (umis, reads)})"""
    ocfg, oref = orc.parse_reference_library(obj, chem)
    if trim:
        ocfg["trim_target_length"], ocfg["trim_strictness"] = int(trim.split(":")[0]), float(trim.split(":")[1])
    recs = any_order_ref.read_bam(bam)
    groups = any_order_ref.groups_any_order(recs)
    want = bam_ref.align_groups(orc.Oracle(ocfg, oref), groups)
    cells = collections.defaultdict(lambda: [0, 0]); used = set()
    for g, w in zip(groups, want):
        cell = g[0]["f"][33]
        used.add(cell)
        for cs, n in w["rows"]:
            e = cells[(",".join(cs), cell)]
            e[0] += 1; e[1] += n
    first = {}
    for r in recs:
        cb = r.aux_string("CB")
        if cb is not None and cb in used and cb not in first and bam_ref.SortedBamReader.umi_of(r) != "AAAAAAAAAA":
            first[cb] = r.ordinal
    return sorted(used, key=first.get), {k: tuple(v) for k, v in cells.items()}


@pytest.mark.parametrize("chem,trim", [("unstranded", None), ("fiveprime", "30:0.5"), ("threeprime", None)])
def test_any_order_matches_oracle_and_the_presorted_driver(tmp_path, chem, trim):
    L, obj, lib_json = library(tmp_path)
    src = make_bam(str(tmp_path / "g.bam"), L, n_groups=400)
    bam = shuffled(src, str(tmp_path / "s.bam"))
    d, dg = str(tmp_path / "m"), str(tmp_path / "mg")
    nb.process_bam(bam, [lib_json], None, strand_filter=chem, trim=trim, num_cores=4, matrix_dirs=[d], any_order=True)
    feats, bcs, got = read_matrix(d)
    want_bcs, want = oracle_any_order(obj, chem, trim, bam)
    assert got == want and len(got) > 50
    assert bcs == want_bcs and len(bcs) > 50                                           # first appearance in the shuffled file
    G = sorted_plus_sentinel(bam, str(tmp_path / "G.bam"))
    nb.process_bam(G, [lib_json], None, strand_filter=chem, trim=trim, num_cores=4, matrix_dirs=[dg])
    feats_g, bcs_g, got_g = read_matrix(dg)
    assert got_g == got and feats_g == feats and set(bcs_g) == set(bcs)
    # the CLI writes the same bytes
    args = [CLI, "-r", lib_json, "-i", bam, "-c", "4", "--strand_filter", chem, "--any-order", "--no-rows", "--cell-matrix", str(tmp_path / "cli")]
    subprocess.check_call(args + (["-t", trim] if trim else []), stdout=subprocess.DEVNULL)
    assert files(str(tmp_path / "cli")) == files(d)


def enc(name, flag, seq, tags, **kw):
    return bamio.encode_record(name, flag, seq, bytes([20 + i % 20 for i in range(len(seq))]), tags, **kw)


def edge_units(rng):
    nt = lambda n: "".join("ACGT"[i] for i in rng.integers(0, 4, n))   # noqa: E731
    tag = lambda cb, umi: [("CB", "Z", cb), ("UB", "Z", umi)]           # noqa: E731
    u = []
    # CBs X-1 and X-2 under one UMI: one scope, cell X-1
    for i, cb in enumerate(["ACGTACGTACGTACGT-2", "ACGTACGTACGTACGT-1", "ACGTACGTACGTACGT-2"]):
        u.append([enc("x%d" % i, 0, nt(91), tag(cb, "CCCCAAAATTTT"))])
    # two different CBs under one UMI: two scopes
    for i, cb in enumerate(["TTTTGGGGCCCCAAAA-1", "GGGGTTTTAAAACCCC-1", "TTTTGGGGCCCCAAAA-1"]):
        u.append([enc("y%d" % i, 16 if i == 1 else 0, nt(124), tag(cb, "GGGGAAAACCCC"))])
    # a secondary record that shares its primary's name; REVERSE and 124-base records
    u.append([enc("sec", 0, nt(124), tag("CATGCATGCATGCATG-1", "TTTTCCCCAAAA")), enc("sec", 256 | 16, nt(124), tag("CATGCATGCATGCATG-1", "TTTTCCCCAAAA"))])
    u.append([enc("rev", 16, nt(124), tag("CATGCATGCATGCATG-1", "TTTTCCCCAAAA"))])
    # a paired record next to an unpaired one with the same name (filter_paired_reads pairs them)
    u.append([enc("quirk", 1 | 64, nt(91), tag("GATCGATCGATCGATC-1", "ACACACACACAC")), enc("quirk", 0, nt(91), tag("GATCGATCGATCGATC-1", "ACACACACACAC"))])
    # one scope of 5000 records
    for i in range(5000):
        u.append([enc("big%05d" % i, 16 if i % 3 == 0 else 0, nt(124 if i % 7 == 0 else 60), tag("AAAACCCCGGGGTTTT-1", "TGTGTGTGTGTG"))])
    return u


def test_dumped_scopes_equal_the_oracle_on_edge_cases(tmp_path):
    L, obj, lib_json = library(tmp_path)
    src = make_bam(str(tmp_path / "g.bam"), L, n_groups=200, tso_fraction=0.3)
    bam = shuffled(src, str(tmp_path / "s.bam"), seed=11, extra_units=edge_units(np.random.default_rng(3)))
    out = tmp_path / "dump.tsv"
    nb.bam_dump_scopes_any_order(bam, out, num_cores=4)
    got = [tuple(l.split("\t")) for l in out.read_text().split("\n")[:-1]]
    groups = any_order_ref.groups_any_order(any_order_ref.read_bam(bam))
    want = []
    fl = lambda it: (1 if it["f"][37] == "TRUE" else 0) | (2 if it["f"][2] == "true" else 0)   # noqa: E731
    for gi, g in enumerate(groups):
        for j in range(0, len(g) - 1, 2):
            a, b = g[j], g[j + 1]
            want.append(tuple(str(x) for x in (gi, g[0]["f"][33], a["ordinal"], b["ordinal"], fl(a), fl(b), len(a["seq"]), len(b["seq"]))))
    assert got == want
    sizes = collections.Counter(l[0] for l in got)
    assert max(sizes.values()) >= 5000                                                 # the big scope (a dummy mate per record)
    cells = {l[1] for l in got}
    assert "ACGTACGTACGTACGT-1" in cells and "ACGTACGTACGTACGT-2" not in cells
    assert {"TTTTGGGGCCCCAAAA-1", "GGGGTTTTAAAACCCC-1"} <= cells
    assert any(l[4] == "0" and l[5] == "0" for l in got)                               # the quirk: a real pair of two records


def test_any_order_is_deterministic_across_threads_and_windows(tmp_path, monkeypatch):
    L, obj, lib_json = library(tmp_path)
    src = make_bam(str(tmp_path / "g.bam"), L, n_groups=1500, seed=77)
    bam = shuffled(src, str(tmp_path / "s.bam"), seed=5)
    runs = {}
    for name, cores, window in (("c1", 1, None), ("c8", 8, None), ("w64", 8, "64")):
        if window:
            monkeypatch.setenv("NB_BAM_WINDOW_KB", window)
        nb.process_bam(bam, [lib_json], None, num_cores=cores, matrix_dirs=[str(tmp_path / name)], any_order=True)
        monkeypatch.delenv("NB_BAM_WINDOW_KB", raising=False)
        runs[name] = files(str(tmp_path / name))
    assert runs["c1"] == runs["c8"] == runs["w64"]
    assert len(gzip.open(bam, "rb").read()) > 4 * 64 * 1024                            # several windows
    monkeypatch.setenv("NB_BAM_WINDOW_KB", "64")
    monkeypatch.setenv("NB_BAM_STATS", "1")
    p = subprocess.run([CLI, "-r", lib_json, "-i", bam, "-c", "8", "--any-order", "--no-rows", "--cell-matrix", str(tmp_path / "st")], capture_output=True, text=True, env=dict(os.environ))
    assert p.returncode == 0, p.stderr
    line = [l for l in p.stderr.split("\n") if l.startswith("nb_process_bam_any_order:")]
    assert len(line) == 1 and "store" in line[0] and "peak RSS" in line[0]
    assert files(str(tmp_path / "st")) == runs["c1"]


def test_two_libraries_grouped_input_and_all_skipped(tmp_path):
    L, obj, lib_a = library(tmp_path)
    _, obj_b, lib_b = library(tmp_path, seed=1234, group_on="", name="lib_b.json")
    src = make_bam(str(tmp_path / "g.bam"), L, n_groups=300)
    bam = shuffled(src, str(tmp_path / "s.bam"), seed=9)
    da, db = str(tmp_path / "a"), str(tmp_path / "b")
    nb.process_bam(bam, [lib_a, lib_b], None, num_cores=4, matrix_dirs=[da, db], any_order=True)
    fa, ba, ga = read_matrix(da)
    fb, bb, gb = read_matrix(db)
    assert ba == bb and fa != fb
    for o, got in ((obj, ga), (obj_b, gb)):
        want_bcs, want = oracle_any_order(o, "unstranded", None, bam)
        assert ba == want_bcs and got == want
    # an already-grouped file (make_bam itself)
    dg = str(tmp_path / "grouped")
    nb.process_bam(src, [lib_a], None, num_cores=4, matrix_dirs=[dg], any_order=True)
    _, bg, gg = read_matrix(dg)
    want_bcs, want = oracle_any_order(obj, "unstranded", None, src)
    assert bg == want_bcs and gg == want
    # every record skipped: the empty matrix nb_write_cell_matrix writes for no rows
    skipped = str(tmp_path / "skipped.bam")
    bamio.write_bam(skipped, [enc("n%d" % i, 0, "ACGT" * 20, [("UB", "Z", "ACGTACGTACGT")]) for i in range(5)] +
                    [enc("w%d" % i, 0, "ACGT" * 20, [("CB", "Z", "ACGT-1"), ("UB", "Z", "AAAAAAAAAA")]) for i in range(5)])
    de, dw = str(tmp_path / "empty"), str(tmp_path / "written")
    nb.process_bam(skipped, [lib_a], None, num_cores=2, matrix_dirs=[de], any_order=True)
    empty = dict(row_cell=[], row_callset=[], row_umis=[], row_reads=[], callset_off=[0], callset_items=[], n_scopes=0)
    nb.write_cell_matrix(dw, nb.Library.from_json(lib_a), empty, [])
    assert files(de) == files(dw)


def test_refusals(tmp_path):
    L, obj, lib_json = library(tmp_path)
    src = make_bam(str(tmp_path / "g.bam"), L, n_groups=40)
    base = raw_records(src)
    cases = {
        "empty_ub": ([("CB", "Z", "ACGTACGTACGTACGT-1"), ("UR", "Z", "ACGTACGTACGT"), ("UB", "Z", "")], -5, "empty UMI"),
        "unpackable": ([("CB", "Z", "ACGTACGTACGTACGT-1"), ("UB", "Z", "ACGT-ACGT")], -5, "ACGT-ACGT"),
        "no_umi": ([("CB", "Z", "ACGTACGTACGTACGT-1")], -3, "Could not read UMI"),
    }
    for name, (tags, code, msg) in cases.items():
        bam = str(tmp_path / (name + ".bam"))
        bamio.write_bam(bam, base[:len(base) // 2] + [enc("bad", 0, "ACGT" * 20, tags)] + base[len(base) // 2:], block_bytes=20000)
        with pytest.raises(nb.NbError) as e:
            nb.process_bam(bam, [lib_json], None, matrix_dirs=[str(tmp_path / name)], any_order=True)
        assert e.value.code == code and msg in str(e.value), str(e.value)
    with pytest.raises(nb.NbError) as e:
        nb.process_bam(src, [lib_json], None, matrix_dirs=[str(tmp_path / "p")], force_bam_paired=True, any_order=True)
    assert e.value.code == -1
    with pytest.raises(nb.NbError) as e:
        nb.process_bam(src, [lib_json], [str(tmp_path / "o.tsv.gz")], matrix_dirs=[str(tmp_path / "o")], any_order=True)
    assert e.value.code == -1
