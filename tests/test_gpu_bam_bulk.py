"""GPU tests of bulk BAM mode (nb_process_bam_bulk, `nimble --bulk`): a BAM without cell barcodes in any record order gives
exactly the TSV bytes FASTQ mode (nb_process_fastq) writes on the FASTQs the BAM stands for (tests/bulk_ref.py), and the
device's pairs equal the restatement's pair for pair (nb_bam_dump_pairs_bulk)."""
import json
import os
import re
import subprocess

import numpy as np
import pytest

import nimble_aligner_b200 as nb
import oracle as orc
import synth
from synth import bamio
from tests import bulk_ref
from tests.bulk_ref import PAIRED, READ1, READ2, REVERSE, SECONDARY, SUPPLEMENTARY

pytestmark = pytest.mark.gpu

CLI = os.path.join(os.path.dirname(nb.SO_PATH), "nimble")
P1, P2 = PAIRED | READ1, PAIRED | READ2
_RC = str.maketrans("ACGTN", "TGCAN")
STATS = re.compile(r"nb_process_bam_bulk: (\d+) records, (\d+) kept, (paired|single-end), (\d+) pairs, dropped (\d+) singletons, (\d+) unsplit .*?, (\d+) in templates of 3\+, (\d+) batches")


def library(tmp_path, name="lib.json", seed=1234, **cfg):
    L = synth.SynthLibrary(seed=seed, n_fam=40, n_all=5, group_on="family", **cfg)
    obj = L.to_json_obj()
    (tmp_path / name).write_text(json.dumps(obj))
    return L, obj, str(tmp_path / name)


def reads(L, n, paired=True):
    r1, o1, r2, o2 = synth.pairs(L, 0, n, paired=paired)
    def txt(r, o):
        return [bytes(r[int(o[i]):int(o[i + 1])]).decode() for i in range(n)]
    return (r1, o1, r2, o2), txt(r1, o1), (txt(r2, o2) if paired else None)


def pair_records(s1, s2, prefix="p", r1_reverse=()):
    """R1 forward (or REVERSE, stored reverse-complemented), R2 stored REVERSE as an aligner stores it"""
    recs = []
    for i, (a, b) in enumerate(zip(s1, s2)):
        rev1 = i in r1_reverse
        recs.append(bulk_ref.Rec("%s%d" % (prefix, i), P1 | (REVERSE if rev1 else 0), a[::-1].translate(_RC) if rev1 else a))
        recs.append(bulk_ref.Rec("%s%d" % (prefix, i), P2 | REVERSE, b[::-1].translate(_RC)))
    return recs


def write(path, recs, order=None, pos=None):
    idx = range(len(recs)) if order is None else order
    bamio.write_bam(str(path), [bamio.encode_record(recs[i].qname, recs[i].flag, recs[i].seq, b"\x28" * len(recs[i].seq),
                                                    refid=0 if pos is not None else -1, pos=int(pos[i]) if pos is not None else -1) for i in idx], level=1)
    return str(path), [recs[i] for i in idx]


def bulk_tsv(bam, libs, tmp_path, name="bulk", chem="unstranded", cores=4):
    outs = [str(tmp_path / ("%s_%d.tsv" % (name, k))) for k in range(len(libs))]
    nb.process_bam(bam, libs, outs, strand_filter=chem, num_cores=cores, bulk=True)
    return [open(o, "rb").read() for o in outs]


def fastq_tsv(recs, libs, tmp_path, name="fq", chem="unstranded"):
    fqs = bulk_ref.write_fastqs(recs, tmp_path, name)
    outs = [str(tmp_path / ("%s_%d.tsv" % (name, k))) for k in range(len(libs))]
    nb.process_fastq(fqs, libs, outs, strand_filter=chem, num_cores=4)
    return [open(o, "rb").read() for o in outs]


def dump(bam, tmp_path, cores=4):
    p = tmp_path / "dump.txt"
    nb.bam_dump_pairs_bulk(bam, str(p), num_cores=cores)
    return p.read_text().split("\n")[:-1]


def cli(bam, libs, outs, cores=4, env_extra=None):
    env = dict(os.environ, NB_BAM_STATS="1")
    env.update(env_extra or {})
    args = [CLI] + [a for lib in libs for a in ("-r", lib)] + ["-i", bam, "--bulk", "-c", str(cores), "-o"] + list(outs)
    p = subprocess.run(args, capture_output=True, text=True, env=env)
    assert p.returncode == 0, p.stderr
    m = STATS.search(p.stderr)
    assert m, p.stderr
    return dict(records=int(m.group(1)), kept=int(m.group(2)), paired=m.group(3) == "paired", pairs=int(m.group(4)), singletons=int(m.group(5)),
                unsplit=int(m.group(6)), multi=int(m.group(7)), batches=int(m.group(8)))


@pytest.fixture(scope="module")
def paired_file(tmp_path_factory):
    tmp = tmp_path_factory.mktemp("bulk")
    L = synth.SynthLibrary(seed=1234, n_fam=40, n_all=5)
    arrays, s1, s2 = reads(L, 4000)
    recs = pair_records(s1, s2, r1_reverse=set(range(0, 4000, 7)))
    rng = np.random.default_rng(5)
    bam, ordered = write(tmp / "shuffled.bam", recs, rng.permutation(len(recs)))
    return tmp, arrays, recs, bam, ordered


@pytest.mark.parametrize("chem", ["unstranded", "fiveprime", "threeprime", "none"])
@pytest.mark.parametrize("mm", [0, 2])
def test_paired_equals_fastq_driver_and_oracle(tmp_path, paired_file, chem, mm):
    _, (r1, o1, r2, o2), recs, bam, ordered = paired_file
    _, obj, lib = library(tmp_path, num_mismatches=mm)
    got = bulk_tsv(bam, [lib], tmp_path, chem=chem)[0]
    assert got == fastq_tsv(ordered, [lib], tmp_path, chem=chem)[0]
    ocfg, oref = orc.parse_reference_library(obj, chem)
    ref = orc.Oracle(ocfg, oref).run(r1, o1, r2, o2, want_records=False)["scopes"][0]
    want = "feature\tscore\n" + "".join("\t".join(cs) + "\t%d\n" % n for cs, n in ref)
    assert got.decode() == want and len(ref) > 10


def test_record_order_does_not_matter(tmp_path, paired_file):
    tmp, _, recs, bam, _ = paired_file
    _, _, lib = library(tmp_path)
    want = bulk_tsv(bam, [lib], tmp_path, name="shuffled")[0]
    collated, _ = write(tmp_path / "collated.bam", recs)                              # name-collated: mates next to each other
    rng = np.random.default_rng(9)
    pos = rng.integers(0, 10 ** 7, len(recs))
    coord, _ = write(tmp_path / "coord.bam", recs, np.argsort(pos, kind="stable"), pos)
    assert bulk_tsv(collated, [lib], tmp_path, name="collated")[0] == want
    assert bulk_tsv(coord, [lib], tmp_path, name="coord")[0] == want


def edge_records(L):
    """the edge cases of bulk mode next to ordinary pairs"""
    _, s1, s2 = reads(L, 600)
    recs = pair_records(s1[:400], s2[:400], r1_reverse=set(range(0, 400, 3)))
    R = bulk_ref.Rec
    # N and IUPAC codes in both orientations (R1 forward, R2 REVERSE; and the other way round)
    for i, (a, b) in enumerate(zip(s1[400:440], s2[400:440])):
        a = a[:10] + "NRYKM" + a[15:60] + "=SWBDHV" + a[67:]
        b = b[:20] + "NNNN" + b[24:]
        rev1 = i % 2 == 1
        recs.append(R("iupac%d" % i, P1 | (REVERSE if rev1 else 0), a[::-1].translate(str.maketrans("ACGTMRWSYKVHDBN=", "TGCAKYWSRMBDHVN=")) if rev1 else a))
        recs.append(R("iupac%d" % i, P2 | (0 if rev1 else REVERSE), b if rev1 else b[::-1].translate(_RC)))
    # 124-base reads (no TSO clip), both orientations
    for i, (a, b) in enumerate(zip(s1[440:470], s2[440:470])):
        recs.append(R("len124_%d" % i, P1 | (REVERSE if i % 2 else 0), a[:124]))
        recs.append(R("len124_%d" % i, P2 | (0 if i % 2 else REVERSE), b[:124]))
    # names differing in the last byte, prefixes of one another, 254-byte names
    for i, (a, b) in enumerate(zip(s1[470:500], s2[470:500])):
        stem = ("L" * 249 + "%04d" % i) if i % 3 == 0 else ("q" * (1 + i % 5))
        recs.append(R(stem + "a", P1, a)); recs.append(R(stem + "b", P2 | REVERSE, b[::-1].translate(_RC)))   # two singletons
        recs.append(R(stem[:-1] if len(stem) > 1 else stem + "zz", P1, a)); recs.append(R(stem + "a", P2, b))   # prefix singleton; stem+a becomes a pair
    # secondaries and supplementaries, with and without SEQ; QC-fail and duplicates (kept)
    for i, (a, b) in enumerate(zip(s1[500:540], s2[500:540])):
        recs.append(R("sec%d" % i, P1 | (SECONDARY if i % 2 else SUPPLEMENTARY), "" if i % 4 < 2 else a))
        recs.append(R("qc%d" % i, P1 | 0x200, a)); recs.append(R("qc%d" % i, P2 | 0x400 | REVERSE, b[::-1].translate(_RC)))
        recs.append(R("sec%d" % i, P2 | SECONDARY, "" if i % 3 else b))
    # singletons, READ_OTHER / both-bits records, three-record templates
    for i, (a, b) in enumerate(zip(s1[540:600], s2[540:600])):
        k = i % 4
        if k == 0:
            recs.append(R("single%d" % i, P2, b))
        elif k == 1:
            recs.append(R("other%d" % i, PAIRED, a)); recs.append(R("other%d" % i, P2, b))
        elif k == 2:
            recs.append(R("both%d" % i, PAIRED | READ1 | READ2, a)); recs.append(R("both%d" % i, P2, b))
        else:
            recs.append(R("three%d" % i, P1, a)); recs.append(R("three%d" % i, P2, b)); recs.append(R("three%d" % i, P2 | REVERSE, b))
    return recs


@pytest.fixture(scope="module")
def edge_file(tmp_path_factory):
    tmp = tmp_path_factory.mktemp("bulk_edge")
    L = synth.SynthLibrary(seed=1234, n_fam=40, n_all=5)
    recs = edge_records(L)
    rng = np.random.default_rng(3)
    bam, ordered = write(tmp / "edge.bam", recs, rng.permutation(len(recs)))
    return bam, ordered


@pytest.mark.parametrize("bits", [None, "4"])
def test_edge_cases_pair_for_pair(tmp_path, edge_file, monkeypatch, bits):
    bam, ordered = edge_file
    if bits:
        monkeypatch.setenv("NB_BULK_NAME_HASH_BITS", bits)                                  # runs of ~100 equal keys: the warp path
    want = bulk_ref.dump_lines(ordered)
    assert len(want) > 450
    assert dump(bam, tmp_path) == want
    _, _, lib = library(tmp_path)
    assert bulk_tsv(bam, [lib], tmp_path)[0] == fastq_tsv(ordered, [lib], tmp_path)[0]


def test_stats_count_the_drops(tmp_path, edge_file):
    bam, ordered = edge_file
    _, _, lib = library(tmp_path)
    st = cli(bam, [lib], [str(tmp_path / "o.tsv")])
    kept = bulk_ref.kept(ordered)
    assert st["records"] == len(ordered) and st["kept"] == len(kept) and st["paired"]
    assert st["pairs"] == len(bulk_ref.pairs(ordered)[1]) and st["batches"] == 1
    sizes = {}
    for _, r in kept:
        sizes[r.qname] = sizes.get(r.qname, 0) + 1
    assert st["singletons"] == sum(1 for n in sizes.values() if n == 1)
    assert st["multi"] == sum(n for n in sizes.values() if n > 2) > 0
    assert st["unsplit"] == 2 * sum(1 for n in sizes.values() if n == 2) - 2 * st["pairs"] > 0


def test_batches_threads_and_windows(tmp_path, paired_file):
    tmp, _, recs, bam, _ = paired_file
    _, _, lib = library(tmp_path)
    base = tmp_path / "base.tsv"
    st = cli(bam, [lib], [str(base)])
    assert st["pairs"] == 4000 and st["batches"] == 1
    want = base.read_bytes()
    for k, env in enumerate([dict(NB_BULK_BATCH_PAIRS="450"), dict(NB_BAM_WINDOW_KB="64")]):
        o = tmp_path / ("e%d.tsv" % k)
        st = cli(bam, [lib], [str(o)], env_extra=env)
        assert o.read_bytes() == want, env
        if "NB_BULK_BATCH_PAIRS" in env:
            assert st["batches"] >= 8
    for cores in (1, 4, 16):
        assert bulk_tsv(bam, [lib], tmp_path, name="c%d" % cores, cores=cores)[0] == want


def test_single_end_two_libraries_cli_equals_python(tmp_path):
    L = synth.SynthLibrary(seed=1234, n_fam=40, n_all=5)
    (r1, o1, _, _), s1, _ = reads(L, 3000, paired=False)
    R = bulk_ref.Rec
    recs = [R("s%d" % i, REVERSE if i % 2 else 0, s[::-1].translate(_RC) if i % 2 else s) for i, s in enumerate(s1)]
    recs += [R("sec", SECONDARY, ""), R("sup", SUPPLEMENTARY, s1[0])]
    rng = np.random.default_rng(11)
    bam, ordered = write(tmp_path / "single.bam", recs, rng.permutation(len(recs)))
    assert bulk_ref.pairs(ordered)[0] is False
    assert dump(bam, tmp_path) == bulk_ref.dump_lines(ordered)
    _, obj_a, lib_a = library(tmp_path, "a.json")
    _, _, lib_b = library(tmp_path, "b.json", num_mismatches=2)
    got = bulk_tsv(bam, [lib_a, lib_b], tmp_path)
    assert got == fastq_tsv(ordered, [lib_a, lib_b], tmp_path)
    ocfg, oref = orc.parse_reference_library(obj_a, "unstranded")
    ref = orc.Oracle(ocfg, oref).run(r1, o1, None, None, want_records=False)["scopes"][0]
    assert got[0].decode() == "feature\tscore\n" + "".join("\t".join(cs) + "\t%d\n" % n for cs, n in ref)
    outs = [str(tmp_path / "cli_a.tsv"), str(tmp_path / "cli_b.tsv")]
    st = cli(bam, [lib_a, lib_b], outs)
    assert not st["paired"] and st["pairs"] == 3000
    assert [open(o, "rb").read() for o in outs] == got
    # appended like the FASTQ writer: a second run adds the rows without a second header
    nb.process_bam(bam, [lib_a], [outs[0]], bulk=True)
    assert open(outs[0], "rb").read() == got[0] + got[0][len(b"feature\tscore\n"):]


def test_empty_and_refusals(tmp_path):
    _, _, lib = library(tmp_path)
    R = bulk_ref.Rec
    empty, _ = write(tmp_path / "empty.bam", [R("x", P1 | SECONDARY, "ACGT")])
    assert bulk_tsv(empty, [lib], tmp_path)[0] == fastq_tsv([], [lib], tmp_path, name="empty")[0]
    cases = [
        ([R("a", P1, "ACGT"), R("b", 0, "ACGT")], "record 0 of .* is paired and record 1 is not"),
        ([R("a", P1, "ACGT"), R("a", P2, "")], "record 1 of .* has no SEQ"),
        ([R("a", P1, "A" * 1100), R("a", P2, "ACGT")], "longer than 1024"),
    ]
    for k, (recs, msg) in enumerate(cases):
        bam, _ = write(tmp_path / ("bad%d.bam" % k), recs)
        out = tmp_path / ("bad%d.tsv" % k)
        with pytest.raises(nb.NbError) as e:
            nb.process_bam(bam, [lib], [str(out)], bulk=True)
        assert e.value.code == -5 and re.search(msg, str(e.value)), str(e.value)
        assert not out.exists()
    # a long read that is dropped (a singleton) is not read at all, as it is in no FASTQ
    ok, ordered = write(tmp_path / "long_single.bam", [R("a", P1, "A" * 1100)] + pair_records(["ACGT" * 20], ["TTGA" * 20]))
    assert bulk_tsv(ok, [lib], tmp_path)[0] == fastq_tsv(ordered, [lib], tmp_path, name="long")[0]
