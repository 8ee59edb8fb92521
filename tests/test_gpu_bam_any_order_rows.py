"""GPU tests of the TSV.gz rows of BAM mode in any record order (nb_process_bam_rows_any_order, `nimble --any-order -o`).

The rows are defined against G = the kept records of the file stably sorted by (UMI, CB), followed by a sentinel scope
(tests.test_gpu_bam_any_order.sorted_plus_sentinel): decompressed, they must be the bytes the grouped driver (nb_process_bam)
writes on G.  The gzip member layout may differ.  Under a budget of P passes the data lines are G's, pass by pass: the same
lines once both files are stably sorted by the UMI bucket."""
import gzip
import os
import re
import subprocess

import numpy as np
import pytest

import nimble_aligner_b200 as nb
import oracle as orc
from oracle import bam_ref
from synth import bamio
from tests import any_order_ref
from tests.bamcases import make_bam
from tests.test_gpu_bam_any_order import edge_units, enc, raw_records, shuffled, sorted_plus_sentinel, units_of
from tests.test_gpu_cell_matrix import CLI, library

pytestmark = pytest.mark.gpu

STATS = re.compile(r"store (\d+) bytes, grouping (\d+) bytes.*?(?:, budget (\d+) bytes, passes (\d+), evictions (\d+), peak device bytes (\d+), windows per pass (\S+))?$")
ROWS = re.compile(r", rows (\d+), row bytes (\d+), row chunks (\d+) \(at most (\d+) per batch\), metadata (\d+) bytes")


def gunzip(path):
    return gzip.open(path, "rb").read()


def grouped_on_G(bam, libs, tmp_path, name="G", **kw):
    """decompressed rows of the grouped driver on G, one per library"""
    G = sorted_plus_sentinel(bam, str(tmp_path / (name + ".bam")))
    outs = [str(tmp_path / ("%s_%d.tsv.gz" % (name, i))) for i in range(len(libs))]
    nb.process_bam(G, libs, outs, num_cores=4, **kw)
    return [gunzip(o) for o in outs]


def cli_rows(bam, libs, outs, budget=None, cores=4, window_kb=None, rows_kb=None, tile=None, chem="unstranded", trim=None, matrix=False):
    """the CLI with NB_BAM_STATS=1 -> the fields of its nb_process_bam_any_order line"""
    env = dict(os.environ, NB_BAM_STATS="1")
    for k, v in (("NB_BAM_WINDOW_KB", window_kb), ("NB_BAM_ROWS_BUFFER_KB", rows_kb), ("NB_BAM_COMPACT_TILE_BYTES", tile)):
        env.pop(k, None)
        if v:
            env[k] = str(v)
    args = [CLI] + [a for lib in libs for a in ("-r", lib)] + ["-i", bam, "-c", str(cores), "--strand_filter", chem, "--any-order"]
    args += (["--no-rows", "--cell-matrix"] if matrix else ["-o"]) + list(outs)
    args += (["-t", trim] if trim else []) + (["--device-budget", str(budget)] if budget else [])
    p = subprocess.run(args, capture_output=True, text=True, env=env)
    assert p.returncode == 0, p.stderr
    line = [l for l in p.stderr.split("\n") if l.startswith("nb_process_bam_any_order:")]
    assert len(line) == 1, p.stderr
    m = STATS.search(line[0])
    assert m, line[0]
    st = dict(store=int(m.group(1)), grouping=int(m.group(2)), line=line[0])
    if budget:
        st.update(passes=int(m.group(4)), evictions=int(m.group(5)), peak=int(m.group(6)))
    r = ROWS.search(line[0])
    assert (r is None) == matrix, line[0]
    if r:
        st.update(rows=int(r.group(1)), row_bytes=int(r.group(2)), chunks=int(r.group(3)), max_chunks=int(r.group(4)), metadata=int(r.group(5)))
    return st


def check_projection(text, bam, obj, chem, trim):
    """the checks tests/test_gpu_bam.py applies to the grouped driver, with the any-order scopes in place of the file's groups"""
    lines = text.decode("latin1").split("\n")
    assert lines[-1] == ""
    lines = lines[:-1]
    ocfg, oref = orc.parse_reference_library(obj, chem)
    if trim:
        ocfg["trim_target_length"], ocfg["trim_strictness"] = int(trim.split(":")[0]), float(trim.split(":")[1])
    groups = any_order_ref.groups_any_order(any_order_ref.read_bam(bam))
    want = bam_ref.align_groups(orc.Oracle(ocfg, oref), groups)
    assert sum(1 for w in want if w["rows"]) > 20
    assert lines[0] == bam_ref.header_line()
    hdr = lines[0].split("\t")
    col = {n: i for i, n in enumerate(hdr)}
    got = []   # runs of rows with one (UMI, CB[..-2]), in file order
    for l in lines[1:]:
        f = l.split("\t")
        assert len(f) == len(hdr)
        key = (f[col["r2_UB"]] or f[col["r2_UR"]], f[col["r2_CB"]][:-2])
        if not got or got[-1][0] != key:
            got.append((key, []))
        got[-1][1].append(f)
    exp = [(w["key"], g, w) for g, w in zip(groups, want) if w["rows"]]
    assert [k for k, _ in got] == [k for k, _, _ in exp]
    for (key, rows), (_, g, w) in zip(got, exp):
        nonzero = sorted((r[0], int(r[1])) for r in rows if r[0] != "")
        assert nonzero == sorted((",".join(cs), n) for cs, n in w["rows"]), key
        assert sum(1 for r in rows if r[0] == "") == w["n_zero_rows"], key
        by_q = {p["qname"]: p for p in w["pairs"]}
        for r in rows:
            q = r[col["r2_QNAME"]]
            p = by_q[q]
            assert r[col["r2_filter_forward"]] == orc.REASONS[p["fr1"]] and r[col["r1_filter_forward"]] == orc.REASONS[p["fr2"]], (key, q)
            assert int(r[col["r2_forward_score"]]) == p["score1"] and int(r[col["r1_forward_score"]]) == p["score2"]
            assert r[col["triage_reason"]] == orc.REASONS[p["triage"]]
            if r[0] != "":
                assert p["callset"] is not None and ",".join(p["callset"]) == r[0]
            j = [i for i, it in enumerate(g) if it["f"][0] == q]
            seq_slot, mate_slot = g[j[0]], g[j[1]]
            assert "\t".join(r[2:38]) == bam_ref.data_values(mate_slot["f"]) and "\t".join(r[38:74]) == bam_ref.data_values(seq_slot["f"])


@pytest.mark.parametrize("chem,trim", [("unstranded", None), ("fiveprime", "30:0.5"), ("threeprime", None)])
def test_rows_equal_the_grouped_driver_on_G_and_the_oracle(tmp_path, chem, trim):
    L, obj, lib_json = library(tmp_path)
    src = make_bam(str(tmp_path / "g.bam"), L, n_groups=400)
    bam = shuffled(src, str(tmp_path / "s.bam"))
    out = str(tmp_path / "o.tsv.gz")
    nb.process_bam(bam, [lib_json], [out], strand_filter=chem, trim=trim, num_cores=4, any_order=True)
    got = gunzip(out)
    assert got == grouped_on_G(bam, [lib_json], tmp_path, strand_filter=chem, trim=trim)[0]
    assert got.count(b"\n") > 100
    check_projection(got, bam, obj, chem, trim)
    st = cli_rows(bam, [lib_json], [str(tmp_path / "cli.tsv.gz")], chem=chem, trim=trim)
    assert gunzip(str(tmp_path / "cli.tsv.gz")) == got
    assert st["rows"] == got.count(b"\n") - 1 and st["row_bytes"] == len(got) - len(got.split(b"\n")[0]) - 1


def with_qn(src, dst):
    """src with a QN string aux (field 0 of the rows) on every record: consecutive units share one, so scopes hold pairs
    with the same field 0, and every fifth one contains a tab"""
    units = units_of(raw_records(src))
    out = []
    for k, u in enumerate(units):
        qn = ("f0-%d" % (k // 2) + ("\tx" if k % 5 == 0 else "")).encode() + b"\0"
        for raw in u:
            body = raw[4:] + b"QNZ" + qn
            out.append(len(body).to_bytes(4, "little") + body)
    bamio.write_bam(dst, out, block_bytes=20000)
    return dst


def test_edge_cases_equal_G(tmp_path):
    L, obj, lib_json = library(tmp_path)
    src = make_bam(str(tmp_path / "g.bam"), L, n_groups=200, tso_fraction=0.3)
    bam = shuffled(with_qn(src, str(tmp_path / "qn.bam")), str(tmp_path / "s.bam"), seed=11, extra_units=edge_units(np.random.default_rng(3)))
    out = str(tmp_path / "o.tsv.gz")
    nb.process_bam(bam, [lib_json], [out], num_cores=4, any_order=True)
    got = gunzip(out)
    assert got == grouped_on_G(bam, [lib_json], tmp_path)[0]
    assert got.count(b"\n") > 100 and b"\tx\t" in got                                 # rows whose field 0 holds a tab


def test_threads_windows_and_row_chunks_give_the_same_bytes(tmp_path):
    L, obj, lib_json = library(tmp_path)
    src = make_bam(str(tmp_path / "g.bam"), L, n_groups=1500, seed=77)
    bam = shuffled(src, str(tmp_path / "s.bam"), seed=5)
    runs = {}
    for name, cores, window, rows_kb in (("c1", 1, None, None), ("c8", 8, None, None), ("w64", 8, 64, None), ("chunks", 8, 64, 16)):
        st = cli_rows(bam, [lib_json], [str(tmp_path / (name + ".tsv.gz"))], cores=cores, window_kb=window, rows_kb=rows_kb)
        runs[name] = gunzip(str(tmp_path / (name + ".tsv.gz")))
        if name == "chunks":
            assert st["max_chunks"] >= 3, st["line"]                                        # several row chunks in one batch
    assert runs["c1"] == runs["c8"] == runs["w64"] == runs["chunks"]
    assert runs["c1"] == grouped_on_G(bam, [lib_json], tmp_path)[0]


def test_two_libraries_and_all_skipped(tmp_path):
    L, obj, lib_a = library(tmp_path)
    _, obj_b, lib_b = library(tmp_path, seed=1234, group_on="", name="lib_b.json")
    src = make_bam(str(tmp_path / "g.bam"), L, n_groups=300)
    bam = shuffled(src, str(tmp_path / "s.bam"), seed=9)
    oa, ob = str(tmp_path / "a.tsv.gz"), str(tmp_path / "b.tsv.gz")
    nb.process_bam(bam, [lib_a, lib_b], [oa, ob], num_cores=4, any_order=True)
    ga, gb = grouped_on_G(bam, [lib_a, lib_b], tmp_path)
    assert gunzip(oa) == ga and gunzip(ob) == gb and ga != gb
    skipped = str(tmp_path / "skipped.bam")
    bamio.write_bam(skipped, [enc("n%d" % i, 0, "ACGT" * 20, [("UB", "Z", "ACGTACGTACGT")]) for i in range(5)] +
                    [enc("w%d" % i, 0, "ACGT" * 20, [("CB", "Z", "ACGT-1"), ("UB", "Z", "AAAAAAAAAA")]) for i in range(5)])
    e, w = str(tmp_path / "e.tsv.gz"), str(tmp_path / "w.tsv.gz")
    nb.process_bam(skipped, [lib_a], [e], num_cores=2, any_order=True)
    nb.process_bam(skipped, [lib_a], [w], num_cores=2)
    assert open(e, "rb").read() == open(w, "rb").read() and gunzip(e) == b""


def by_bucket(text):
    """header, then the data lines stably sorted by the UMI bucket of r2_UB (else r2_UR)"""
    lines = text.split(b"\n")[:-1]
    hdr = lines[0].decode().split("\t")
    ub, ur = hdr.index("r2_UB"), hdr.index("r2_UR")
    def bucket(l):
        f = l.split(b"\t")
        return nb.any_order_umi_bucket((f[ub] or f[ur]).decode())
    return lines[0], sorted(lines[1:], key=bucket)


def test_budgeted_passes_write_the_lines_of_the_unbudgeted_run(tmp_path):
    L, obj, lib_json = library(tmp_path)
    src = make_bam(str(tmp_path / "g.bam"), L, n_groups=1500, seed=31)
    bam = shuffled(src, str(tmp_path / "s.bam"), seed=4)
    rows_kb = 32   # the row buffer is counted under the budget: small, so that the store decides the passes
    # 64 KB windows: the store already holds records when a window lowers hi, so the passes compact it (evictions), moving
    # the metadata text and its offsets with the rest; small compaction tiles make those moves cross many tile boundaries
    base = cli_rows(bam, [lib_json], [str(tmp_path / "u.tsv.gz")], rows_kb=rows_kb, window_kb=64)
    unb = gunzip(str(tmp_path / "u.tsv.gz"))
    assert unb == grouped_on_G(bam, [lib_json], tmp_path)[0]
    need = base["store"] + base["grouping"]
    want = by_bucket(unb)
    for div, passes, tile in ((3, 2, None), (8, 4, 4096), (16, 8, 64)):
        out = str(tmp_path / ("b%d.tsv.gz" % div))
        st = cli_rows(bam, [lib_json], [out], budget=need // div, rows_kb=rows_kb, window_kb=64, tile=tile)
        assert st["passes"] >= passes and st["evictions"] >= 1 and st["peak"] <= need // div, st["line"]
        got = gunzip(out)
        assert got.split(b"\n")[0] == unb.split(b"\n")[0] and by_bucket(got) == want, div
    big = cli_rows(bam, [lib_json], [str(tmp_path / "big.tsv.gz")], budget=64 * need, rows_kb=rows_kb, window_kb=64)
    assert big["passes"] == 1 and big["evictions"] == 0 and gunzip(str(tmp_path / "big.tsv.gz")) == unb
    with pytest.raises(nb.NbError) as e:
        nb.process_bam(bam, [lib_json], [str(tmp_path / "small.tsv.gz")], num_cores=4, any_order=True, device_budget=1 << 16)
    need_named = [int(x) for x in re.findall(r"needs (\d+) bytes", str(e.value))]
    assert need_named and need_named[0] > 1 << 16, str(e.value)


def test_matrix_only_runs_stage_no_metadata(tmp_path):
    L, obj, lib_json = library(tmp_path)
    src = make_bam(str(tmp_path / "g.bam"), L, n_groups=400)
    bam = shuffled(src, str(tmp_path / "s.bam"))
    rows = cli_rows(bam, [lib_json], [str(tmp_path / "o.tsv.gz")])
    mat = cli_rows(bam, [lib_json], [str(tmp_path / "m")], matrix=True)
    assert rows["metadata"] > 0 and mat["store"] == rows["store"] - rows["metadata"]
    assert "rows" not in mat["line"].split("peak RSS")[1]
