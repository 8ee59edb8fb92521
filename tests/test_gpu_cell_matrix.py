"""GPU tests of the per-cell count matrix of BAM mode (nb_cells_*, nb_process_bam_cells, `nimble --cell-matrix`).

The matrix is a projection of the TSV.gz the BAM driver writes: for a cell (the full CB of a scope's first record) and a
callset, umis = scopes of that cell with a row for the callset, reads = the sum of those rows' nimble_score.  It is checked
against the CPU oracle's per-scope counts (independent of the device TSV), against the TSV of the same run, across runs
(rows-free, thread counts, window sizes, the whole-file fallback) and at the C ABI over several scoped batches."""
import collections
import gzip
import json
import os
import subprocess

import numpy as np
import pytest
import scipy.io

import nimble_aligner_b200 as nb
import oracle as orc
import synth
from oracle import bam_ref
from synth import bamio
from tests.bamcases import make_bam

pytestmark = pytest.mark.gpu

CLI = os.path.join(os.path.dirname(nb.SO_PATH), "nimble")
FILES = ["barcodes.tsv.gz", "features.tsv.gz", "matrix.mtx.gz", "reads.mtx.gz"]


def library(tmp_path, seed=1234, group_on="family", name="lib.json"):
    L = synth.SynthLibrary(seed=seed, n_fam=40, n_all=5, group_on=group_on, num_mismatches=1)
    obj = L.to_json_obj()
    path = tmp_path / name
    path.write_text(json.dumps(obj))
    return L, obj, str(path)


def read_matrix(d):
    """-> (features, barcodes, {(feature, barcode): (umis, reads)}); both .mtx files list the same coordinates in the same order."""
    feats = [l.split("\t") for l in gzip.open(os.path.join(d, "features.tsv.gz"), "rt").read().split("\n")[:-1]]
    assert all(len(f) == 3 and f[0] == f[1] and f[2] == "Gene Expression" for f in feats)
    feats = [f[0] for f in feats]
    bcs = gzip.open(os.path.join(d, "barcodes.tsv.gz"), "rt").read().split("\n")[:-1]
    mu = gzip.open(os.path.join(d, "matrix.mtx.gz"), "rt").read().split("\n")[:-1]
    mr = gzip.open(os.path.join(d, "reads.mtx.gz"), "rt").read().split("\n")[:-1]
    assert mu[0] == mr[0] == "%%MatrixMarket matrix coordinate integer general" and mu[1] == mr[1] == "%d %d %d" % (len(feats), len(bcs), len(mu) - 2)
    cu = [tuple(int(x) for x in l.split()) for l in mu[2:]]
    cr = [tuple(int(x) for x in l.split()) for l in mr[2:]]
    assert [c[:2] for c in cu] == [c[:2] for c in cr]
    assert [(c[1], c[0]) for c in cu] == sorted(set((c[1], c[0]) for c in cu))          # by barcode, then feature, no duplicates
    assert all(c[2] > 0 for c in cu) and all(c[2] >= u[2] for c, u in zip(cr, cu))
    assert feats == sorted(set(feats), key=lambda s: s.split(","))                      # Vec<String> Ord
    m = scipy.io.mmread(os.path.join(d, "matrix.mtx.gz"))
    assert m.shape == (len(feats), len(bcs)) and int(m.sum()) == sum(c[2] for c in cu)
    used = set(c[0] for c in cu)
    assert used == set(range(1, len(feats) + 1))                                        # every feature has an entry
    return feats, bcs, {(feats[a - 1], bcs[b - 1]): (u, r[2]) for (a, b, u), r in zip(cu, cr)}


def files(d):
    return {f: open(os.path.join(d, f), "rb").read() for f in FILES}


def oracle_cells(obj, chem, trim, bam, force_paired):
    """-> (first-appearance barcodes, {(feature, barcode): (umis, reads)}) from the oracle's per-scope rows."""
    ocfg, oref = orc.parse_reference_library(obj, chem)
    if trim:
        ocfg["trim_target_length"], ocfg["trim_strictness"] = int(trim.split(":")[0]), float(trim.split(":")[1])
    groups = bam_ref.groups_of(bam_ref.read_bam(bam), force_paired)
    want = bam_ref.align_groups(orc.Oracle(ocfg, oref), groups)
    bcs, cells = [], collections.defaultdict(lambda: [0, 0])
    for g, w in zip(groups, want):
        if not g:
            continue
        cell = g[0]["f"][33]
        if cell not in bcs:
            bcs.append(cell)
        for cs, n in w["rows"]:
            e = cells[(",".join(cs), cell)]
            e[0] += 1; e[1] += n
    return bcs, {k: tuple(v) for k, v in cells.items()}


def tsv_projection(path):
    """The TSV.gz's rows projected onto (feature, r2_CB): (count rows, sum of nimble_score); zero rows contribute nothing."""
    lines = gzip.open(path, "rt", encoding="latin1").read().split("\n")[:-1]
    hdr = lines[0].split("\t"); cb = hdr.index("r2_CB")
    out = collections.defaultdict(lambda: [0, 0])
    for l in lines[1:]:
        f = l.split("\t")
        if f[0]:
            e = out[(f[0], f[cb])]
            e[0] += 1; e[1] += int(f[1])
    return {k: tuple(v) for k, v in out.items()}


@pytest.mark.parametrize("chem,force_paired,trim", [("unstranded", False, None), ("fiveprime", False, "30:0.5"), ("threeprime", False, None), ("unstranded", True, None)])
def test_matrix_matches_oracle_tsv_and_rows_free_run(tmp_path, chem, force_paired, trim):
    L, obj, lib_json = library(tmp_path)
    bam = make_bam(str(tmp_path / "t.bam"), L, n_groups=400, paired_fraction=0.3 if force_paired else 0.15)
    kw = dict(strand_filter=chem, trim=trim, num_cores=4, force_bam_paired=force_paired)
    tsv, tsv0, d, d2 = tmp_path / "o.tsv.gz", tmp_path / "plain.tsv.gz", str(tmp_path / "m"), str(tmp_path / "m2")
    nb.process_bam(bam, [lib_json], [str(tsv)], matrix_dirs=[d], **kw)
    nb.process_bam(bam, [lib_json], [str(tsv0)], **kw)
    # 1. against the oracle
    feats, bcs, got = read_matrix(d)
    want_bcs, want = oracle_cells(obj, chem, trim, bam, force_paired)
    assert bcs == want_bcs and len(bcs) > 50
    assert got == want and len(got) > 50
    # 2. the TSV of the same run is nb_process_bam's, and the matrix is its projection
    assert gzip.open(tsv, "rb").read() == gzip.open(tsv0, "rb").read()
    assert tsv_projection(tsv) == got
    # 3. rows-free: the same matrix files and no TSV
    before = set(os.listdir(tmp_path))
    nb.process_bam(bam, [lib_json], None, matrix_dirs=[d2], **kw)
    assert files(d2) == files(d)
    assert set(os.listdir(tmp_path)) - before == {"m2"}
    # 7. the CLI writes the same files, with and without the rows
    for extra, sub in ((["-o", str(tmp_path / "cli.tsv.gz")], "c1"), (["--no-rows"], "c2")):
        args = [CLI, "-r", lib_json, "-i", bam, "-c", "4", "--strand_filter", chem, "--cell-matrix", str(tmp_path / sub)] + extra
        subprocess.check_call(args + (["-t", trim] if trim else []) + (["-p"] if force_paired else []), stdout=subprocess.DEVNULL)
        assert files(str(tmp_path / sub)) == files(d)
    assert gzip.open(tmp_path / "cli.tsv.gz", "rb").read() == gzip.open(tsv, "rb").read()


def with_empty_ub(src, dst):
    """`src` with one more record whose UB:Z is empty (a kept record without a UMI string: the driver reads the whole file
    again with the serial readers), placed between two UMI runs."""
    raw = gzip.open(src, "rb").read()
    l_text = int.from_bytes(raw[4:8], "little"); p = 8 + l_text
    n_ref = int.from_bytes(raw[p:p + 4], "little"); p += 4
    for _ in range(n_ref):
        p += 4 + int.from_bytes(raw[p:p + 4], "little") + 4
    recs = []
    while p < len(raw):
        n = int.from_bytes(raw[p:p + 4], "little"); recs.append(raw[p:p + 4 + n]); p += 4 + n
    at = len(recs) // 2
    while b"UBZ" in recs[at] and recs[at].split(b"UBZ")[1][:12] == recs[at - 1].split(b"UBZ")[1][:12]:
        at += 1
    extra = bamio.encode_record("empty_ub", 0, "ACGT" * 22 + "ACG", bytes([36] * 91), [("CB", "Z", "ACGTACGTACGTACGT-1"), ("UR", "Z", "ACGTACGTACGT"), ("UB", "Z", "")])
    bamio.write_bam(dst, recs[:at] + [extra] + recs[at:], block_bytes=20000)
    return dst


def test_matrix_is_deterministic_across_threads_windows_and_the_whole_file_fallback(tmp_path, monkeypatch):
    L, obj, lib_json = library(tmp_path)
    bam = make_bam(str(tmp_path / "t.bam"), L, n_groups=1500, seed=77)
    runs = {}
    for name, cores, window in (("c1", 1, None), ("c8", 8, None), ("w64", 8, "64")):
        if window:
            monkeypatch.setenv("NB_BAM_WINDOW_KB", window)
        nb.process_bam(bam, [lib_json], None, num_cores=cores, matrix_dirs=[str(tmp_path / name)])
        monkeypatch.delenv("NB_BAM_WINDOW_KB", raising=False)
        runs[name] = files(str(tmp_path / name))
    assert runs["c1"] == runs["c8"] == runs["w64"]
    assert os.path.getsize(bam) > 4 * 64 * 1024 // 4                                       # several windows
    # the whole-file fallback starts over: its matrix must count every scope once
    fb = with_empty_ub(bam, str(tmp_path / "fb.bam"))
    monkeypatch.setenv("NB_BAM_WINDOW_KB", "64")
    monkeypatch.setenv("NB_BAM_STATS", "1")
    tsv = tmp_path / "fb.tsv.gz"
    p = subprocess.run([CLI, "-r", lib_json, "-o", str(tsv), "-i", fb, "-c", "8", "--cell-matrix", str(tmp_path / "fb")], capture_output=True, text=True, env=dict(os.environ))
    assert p.returncode == 0, p.stderr
    assert "whole-file fallback" in p.stderr
    monkeypatch.delenv("NB_BAM_WINDOW_KB")
    monkeypatch.delenv("NB_BAM_STATS")
    nb.process_bam(fb, [lib_json], None, num_cores=1, matrix_dirs=[str(tmp_path / "fb1")])
    assert files(str(tmp_path / "fb")) == files(str(tmp_path / "fb1"))
    feats, bcs, got = read_matrix(str(tmp_path / "fb"))
    assert tsv_projection(tsv) == got
    want_bcs, want = oracle_cells(obj, "unstranded", None, fb, False)
    assert bcs == want_bcs and got == want


def test_two_libraries_share_the_barcodes(tmp_path):
    L, obj, lib_a = library(tmp_path)
    _, obj_b, lib_b = library(tmp_path, seed=1234, group_on="", name="lib_b.json")    # same sequences, one group per transcript
    bam = make_bam(str(tmp_path / "t.bam"), L, n_groups=300)
    da, db = str(tmp_path / "a"), str(tmp_path / "b")
    nb.process_bam(bam, [lib_a, lib_b], None, num_cores=4, matrix_dirs=[da, db])
    fa, ba, ga = read_matrix(da)
    fb, bb, gb = read_matrix(db)
    assert ba == bb and fa != fb
    for o, got in ((obj, ga), (obj_b, gb)):
        want_bcs, want = oracle_cells(o, "unstranded", None, bam, False)
        assert ba == want_bcs and got == want


def test_cells_abi_over_batches_with_resets_and_rehashes():
    """Three scoped batches with nb_counts_reset between them (dense callset ids renumbered every time), cells recurring across
    batches, a per-cell table of 64 slots that has to grow: nb_cells_finalize equals the oracle's per-scope rows rolled up by
    cell on the host."""
    L = synth.SynthLibrary(seed=1234, n_fam=40, n_all=5, group_on="family", num_mismatches=1)
    obj = L.to_json_obj()
    lib = nb.Library.from_text(json.dumps(obj), "unstranded")
    ix = nb.build_index(lib, 2, device=0)
    ocfg, oref = orc.parse_reference_library(obj, "unstranded")
    o = orc.Oracle(ocfg, oref)
    names = lib.group_names()
    ctx = nb.Context(ix, lib, device=0, cell_slots=64)
    rng = np.random.default_rng(5)
    want = collections.defaultdict(lambda: [0, 0])
    dicts, n_scopes = [], 0
    for bi, (first, ng, seed) in enumerate(((0, 60, 11), (60, 400, 12), (460, 150, 13))):
        u = synth.umi_reads(L, first, ng, seed=seed, threads=4)
        n = u["n_reads"]
        scope = np.repeat(np.arange(ng, dtype=np.uint32), u["sizes"])
        scope_off = np.concatenate([[0], np.cumsum(u["sizes"], dtype=np.uint64)]).astype(np.uint64)
        ones, zeros = np.ones(n, dtype=np.uint8), np.zeros(n, dtype=np.uint8)
        cell_of_scope = rng.integers(0, 25, ng).astype(np.uint32)
        ctx.align_batch(u["bases"], u["off"], u["bases"], u["off"], q1=u["qual"], q2=u["qual"], flags1=ones * nb.FLAG_SKIP_ALIGN, flags2=zeros,
                        scope_id=scope, max_read_len=91)
        raw = ctx.counts_raw()
        dicts.append([tuple(raw["callset_items"][int(raw["callset_off"][i]):int(raw["callset_off"][i + 1])]) for i in range(len(raw["callset_off"]) - 1)])
        with pytest.raises(nb.NbError):
            ctx.cells_roll(cell_of_scope[: ng // 2])                                     # fewer cells than scopes
        ctx.cells_roll(cell_of_scope)
        with pytest.raises(nb.NbError):
            ctx.cells_roll(cell_of_scope)                                                # a batch rolls once
        n_scopes += ng
        ref = o.run(u["bases"], u["off"], u["bases"], u["off"], q1=u["qual"], q2=u["qual"], skip1=ones, skip2=zeros, scope_off=scope_off, threads=4, want_records=False)
        for si, rows in enumerate(ref["scopes"]):
            for cs, c in rows:
                e = want[(int(cell_of_scope[si]), tuple(cs))]
                e[0] += 1; e[1] += int(c)
        ctx.reset()
    assert dicts[0] != dicts[1] != dicts[2]                                              # renumbered between batches
    got = ctx.cells_finalize()
    callsets = [tuple(names[g] for g in got["callset_items"][int(got["callset_off"][i]):int(got["callset_off"][i + 1])]) for i in range(len(got["callset_off"]) - 1)]
    assert callsets == sorted(set(callsets), key=list)
    keys = list(zip(got["row_cell"].tolist(), got["row_callset"].tolist()))
    assert keys == sorted(set(keys))
    table = {(c, callsets[s]): (u, r) for (c, s), u, r in zip(keys, got["row_umis"].tolist(), got["row_reads"].tolist())}
    assert table == {k: tuple(v) for k, v in want.items()} and len(table) > 100
    assert got["n_scopes"] == n_scopes
    assert len(set(c for c, _ in want)) == 25                                            # cells recur across batches
    ctx.cells_reset()
    e = ctx.cells_finalize()
    assert len(e["row_cell"]) == 0 and len(e["callset_off"]) == 1
    ctx.align_batch(u["bases"], u["off"], u["bases"], u["off"], q1=u["qual"], q2=u["qual"], flags1=ones * nb.FLAG_SKIP_ALIGN, flags2=zeros, scope_id=scope, max_read_len=91)
    ctx.counts_raw()
    with pytest.raises(nb.NbError) as err:
        ctx.cells_roll(np.full(ng, 0xFFFFFFFF, dtype=np.uint32))                         # cell ids stop below 2^32 - 1
    assert err.value.code == -5
