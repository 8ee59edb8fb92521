"""GPU tests of the sample manifest (nb_process_samples, process_samples, `nimble --samples`): every (sample, library) TSV
of a manifest run is byte for byte what the single run of that sample writes to that path (nb_process_fastq for FASTQ
samples, nb_process_bam_bulk for bulk BAM samples), including append mode, empty inputs and a failure in the middle."""
import json
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import nimble_aligner_b200 as nb
import synth
from tests import bulk_ref
from tests.bulk_ref import PAIRED, READ1, READ2, REVERSE, SECONDARY
from synth import bamio

pytestmark = pytest.mark.gpu

CLI = os.path.join(os.path.dirname(nb.SO_PATH), "nimble")
P1, P2 = PAIRED | READ1, PAIRED | READ2
_RC = str.maketrans("ACGTN", "TGCAN")
SAMPLE_LINE = re.compile(r"nb_process_samples: sample (\S+): (\d+) pairs")


def library(d, name, seed, **cfg):
    L = synth.SynthLibrary(seed=seed, n_fam=40, n_all=5, group_on="family", **cfg)
    path = os.path.join(str(d), name)
    with open(path, "w") as f:
        json.dump(L.to_json_obj(), f)
    return L, path


def write_reads(L, d, stem, n, first=0, paired=True, gz=False):
    r1, o1, r2, o2 = synth.pairs(L, first, n, paired=paired, threads=8)
    ext = "fastq.gz" if gz else "fastq"
    paths = [os.path.join(str(d), "%s_%d.%s" % (stem, m, ext)) for m in ((1, 2) if paired else (1,))]
    synth.write_fastq(paths[0], r1, o1, 1)
    if paired:
        synth.write_fastq(paths[1], r2, o2, 2)
    return paths


@pytest.fixture(scope="module")
def fastq_set(tmp_path_factory):
    """paired plain, paired .gz, single-end, an empty pair, 200 k pairs then 3 pairs, and the same reads under two names"""
    d = tmp_path_factory.mktemp("samples_fq")
    L = synth.SynthLibrary(seed=1234, n_fam=40, n_all=5)
    empty = [str(d / "empty_1.fastq"), str(d / "empty_2.fastq")]
    for p in empty:
        open(p, "w").close()
    plain = write_reads(L, d, "plain", 3000)
    samples = [
        ("plain", plain),
        ("gz", write_reads(L, d, "gz", 2500, first=5000, gz=True)),
        ("single", write_reads(L, d, "single", 2000, first=9000, paired=False)),
        ("empty", empty),
        ("big", write_reads(L, d, "big", 200_000, first=20_000)),
        ("tiny", write_reads(L, d, "tiny", 3, first=400_000)),
        ("plain.again", plain),
    ]
    return d, samples


def write_manifest(path, samples, comments=True):
    with open(path, "w") as f:
        if comments:
            f.write("# a cohort\n\n")
        for name, ins in samples:
            f.write("\t".join([name] + list(ins)) + "\n")
    return str(path)


def single_fastq(ins, libs, out_dir, name, chem="unstranded", cores=4):
    os.makedirs(out_dir, exist_ok=True)
    outs = [os.path.join(out_dir, "%s.%d.tsv" % (name, k)) for k in range(len(libs))]
    nb.process_fastq(ins, libs, outs, strand_filter=chem, num_cores=cores)
    return [open(o, "rb").read() for o in outs]


def read_outs(dirs, name):
    return [open(os.path.join(d, name + ".tsv"), "rb").read() for d in dirs]


@pytest.mark.parametrize("mm,chem", [(0, "unstranded"), (2, "unstranded"), (0, "fiveprime"), (2, "threeprime")])
def test_fastq_manifest_equals_single_runs(tmp_path, fastq_set, mm, chem):
    _, samples = fastq_set
    _, lib_a = library(tmp_path, "a.json", 1234, num_mismatches=mm)
    _, lib_b = library(tmp_path, "b.json", 77, num_mismatches=2 - mm)
    dirs = [str(tmp_path / "out_a"), str(tmp_path / "out_b")]
    nb.process_samples(write_manifest(tmp_path / "m.tsv", samples), [lib_a, lib_b], dirs, strand_filter=chem, num_cores=4)
    for name, ins in samples:
        want = single_fastq(ins, [lib_a, lib_b], str(tmp_path / "single"), name, chem)
        assert read_outs(dirs, name) == want, name
    assert read_outs(dirs, "empty")[0] == b"feature\tscore\n"
    assert read_outs(dirs, "plain") == read_outs(dirs, "plain.again")
    assert read_outs(dirs, "big")[0].count(b"\n") > 10 and read_outs(dirs, "tiny")[0].startswith(b"feature\tscore\n")
    assert sorted(os.listdir(dirs[0])) == sorted(n + ".tsv" for n, _ in samples)


def test_position_in_manifest_does_not_matter(tmp_path, fastq_set):
    d, samples = fastq_set
    _, lib = library(tmp_path, "a.json", 1234)
    S = dict(samples)
    L = synth.SynthLibrary(seed=1234, n_fam=40, n_all=5)
    fill = [("f%02d" % i, write_reads(L, tmp_path, "f%02d" % i, 50 + 37 * i, first=600_000 + 1000 * i, paired=i % 3 != 0)) for i in range(18)]
    order = [("first", S["gz"])] + fill + [("twentieth", S["gz"])]
    dirs = [str(tmp_path / "out")]
    nb.process_samples(write_manifest(tmp_path / "m.tsv", order), [lib], dirs)
    assert read_outs(dirs, "first") == read_outs(dirs, "twentieth")
    assert read_outs(dirs, "f07") == single_fastq(dict(fill)["f07"], [lib], str(tmp_path / "single"), "f07")


def test_existing_files_are_appended(tmp_path, fastq_set):
    _, samples = fastq_set
    S = dict(samples)
    _, lib = library(tmp_path, "a.json", 1234)
    out, single = tmp_path / "out", tmp_path / "single"
    os.makedirs(out); os.makedirs(single)
    for d in (out, single):
        (d / "plain.tsv").write_bytes(b"feature\tscore\nold\t1\n")   # appended without a header
        (d / "gz.tsv").write_bytes(b"")                               # empty: the header is written
    pick = [("plain", S["plain"]), ("gz", S["gz"]), ("single", S["single"])]
    nb.process_samples(pick, [lib], [str(out)])
    for name, ins in pick:
        nb.process_fastq(ins, [lib], [str(single / (name + ".tsv"))], num_cores=4)
        assert (out / (name + ".tsv")).read_bytes() == (single / (name + ".tsv")).read_bytes(), name
    assert (out / "plain.tsv").read_bytes().startswith(b"feature\tscore\nold\t1\n") and (out / "plain.tsv").read_bytes().count(b"feature") == 1


def test_cli_equals_python_and_threads_do_not_matter(tmp_path, fastq_set):
    _, samples = fastq_set
    pick = [s for s in samples if s[0] in ("plain", "gz", "single", "empty", "tiny")]
    _, lib_a = library(tmp_path, "a.json", 1234)
    _, lib_b = library(tmp_path, "b.json", 77, num_mismatches=2)
    m = write_manifest(tmp_path / "m.tsv", pick)
    py = [str(tmp_path / "py_a"), str(tmp_path / "py_b")]
    nb.process_samples(m, [lib_a, lib_b], py, num_cores=4)
    for cores in (1, 4, 16):
        dirs = [str(tmp_path / ("c%d_a" % cores)), str(tmp_path / ("c%d_b" % cores))]
        p = subprocess.run([CLI, "--samples", m, "-r", lib_a, "-r", lib_b, "-o"] + dirs + ["-c", str(cores)], capture_output=True, text=True,
                           env=dict(os.environ, NB_FASTQ_STATS="1"))
        assert p.returncode == 0, p.stderr
        assert "nb_process_samples: setup" in p.stderr
        seen = {x.group(1): int(x.group(2)) for x in SAMPLE_LINE.finditer(p.stderr)}
        assert seen == {"plain": 3000, "gz": 2500, "single": 2000, "empty": 0, "tiny": 3}, p.stderr
        assert "nb_process_fastq:" not in p.stderr
        for name, _ in pick:
            assert read_outs(dirs, name) == read_outs(py, name), (cores, name)


# ---------------------------------------------------------------------------------------------------------------- bulk
def pair_records(s1, s2, prefix):
    recs = []
    for i, (a, b) in enumerate(zip(s1, s2)):
        recs.append(bulk_ref.Rec("%s%d" % (prefix, i), P1, a))
        recs.append(bulk_ref.Rec("%s%d" % (prefix, i), P2 | REVERSE, b[::-1].translate(_RC)))
    return recs


def write_bam(path, recs, order=None):
    idx = range(len(recs)) if order is None else order
    bamio.write_bam(str(path), [bamio.encode_record(recs[i].qname, recs[i].flag, recs[i].seq, b"\x28" * len(recs[i].seq)) for i in idx], level=1)
    return str(path)


def texts(L, n, first, paired=True):
    r1, o1, r2, o2 = synth.pairs(L, first, n, paired=paired)
    t = lambda r, o: [bytes(r[int(o[i]):int(o[i + 1])]).decode() for i in range(n)]
    return t(r1, o1), (t(r2, o2) if paired else None)


@pytest.fixture(scope="module")
def bam_set(tmp_path_factory):
    """a shuffled paired BAM, a name-collated one, a single-end one and one without kept records"""
    d = tmp_path_factory.mktemp("samples_bam")
    L = synth.SynthLibrary(seed=1234, n_fam=40, n_all=5)
    rng = np.random.default_rng(5)
    s1, s2 = texts(L, 4000, 0)
    recs = pair_records(s1, s2, "p")
    c1, c2 = texts(L, 1500, 10_000)
    se, _ = texts(L, 2500, 20_000, paired=False)
    single = [bulk_ref.Rec("s%d" % i, REVERSE if i % 2 else 0, s[::-1].translate(_RC) if i % 2 else s) for i, s in enumerate(se)]
    return d, [
        ("shuffled", write_bam(d / "shuffled.bam", recs, rng.permutation(len(recs)))),
        ("collated", write_bam(d / "collated.bam", pair_records(c1, c2, "c"))),
        ("single", write_bam(d / "single.bam", single, rng.permutation(len(single)))),
        ("nothing_kept", write_bam(d / "nothing.bam", [bulk_ref.Rec("x", P1 | SECONDARY, "ACGT")])),
    ]


def single_bulk(bam, libs, out_dir, name, cores=4):
    os.makedirs(out_dir, exist_ok=True)
    outs = [os.path.join(out_dir, "%s.%d.tsv" % (name, k)) for k in range(len(libs))]
    nb.process_bam(bam, libs, outs, num_cores=cores, bulk=True)
    return [open(o, "rb").read() for o in outs]


def test_bulk_manifest_equals_single_runs(tmp_path, bam_set):
    _, samples = bam_set
    _, lib_a = library(tmp_path, "a.json", 1234)
    _, lib_b = library(tmp_path, "b.json", 77, num_mismatches=2)
    dirs = [str(tmp_path / "out_a"), str(tmp_path / "out_b")]
    m = write_manifest(tmp_path / "m.tsv", [(n, [b]) for n, b in samples])
    nb.process_samples(m, [lib_a, lib_b], dirs, num_cores=4, bulk=True)
    for name, bam in samples:
        assert read_outs(dirs, name) == single_bulk(bam, [lib_a, lib_b], str(tmp_path / "single"), name), name
    assert read_outs(dirs, "nothing_kept") == [b"feature\tscore\n"] * 2
    assert read_outs(dirs, "shuffled")[0].count(b"\n") > 10
    # the CLI writes the same bytes, with one setup line and one line per sample
    cdirs = [str(tmp_path / "cli_a"), str(tmp_path / "cli_b")]
    p = subprocess.run([CLI, "--samples", m, "--bulk", "-r", lib_a, "-r", lib_b, "-o"] + cdirs + ["-c", "8"], capture_output=True, text=True,
                       env=dict(os.environ, NB_BAM_STATS="1"))
    assert p.returncode == 0, p.stderr
    assert "nb_process_samples: setup" in p.stderr and len(re.findall(r"nb_process_samples: sample \S+: \d+ records, \d+ pairs", p.stderr)) == 4, p.stderr
    for name, _ in samples:
        assert read_outs(cdirs, name) == read_outs(dirs, name), name


# ---------------------------------------------------------------------------------------------------------------- a failure mid-run
def expect_failure(run):
    with pytest.raises(nb.NbError) as e:
        run()
    return e.value.code, str(e.value).split(": ", 1)[1]   # "nimble_b200 error <code>: <message>"


def check_mid_run_failure(tmp_path, samples, libs, bulk, single):
    """samples: five (name, inputs), the third bad.  The code is the single run's, the message is the single run's behind
    the sample's name and line; samples 1-2 are complete, sample 3 leaves what its single run leaves, 4-5 are untouched."""
    m = str(tmp_path / "m.tsv")
    with open(m, "w") as f:
        f.write("# five samples\n\n")
        for name, ins in samples:
            f.write("\t".join([name] + ins) + "\n")
    dirs = [str(tmp_path / "out_a"), str(tmp_path / "out_b")]
    bad_name, bad_ins = samples[2]
    s_code, s_msg = expect_failure(lambda: single(bad_ins, libs, str(tmp_path / "single_bad"), bad_name))
    code, msg = expect_failure(lambda: nb.process_samples(m, libs, dirs, num_cores=4, bulk=bulk))
    assert code == s_code and msg == "sample %s (line 5): %s" % (bad_name, s_msg), (code, msg, s_code, s_msg)
    for name, ins in samples[:2]:
        assert read_outs(dirs, name) == single(ins, libs, str(tmp_path / "single"), name), name
    left = sorted(f for f in os.listdir(str(tmp_path / "single_bad")))
    assert sorted(os.listdir(dirs[0]) + os.listdir(dirs[1])) == sorted([samples[0][0] + ".tsv"] * 2 + [samples[1][0] + ".tsv"] * 2 +
                                                                       [bad_name + ".tsv" for f in left])
    # the CLI: exit 101 and the same message
    shutil.rmtree(dirs[0]); shutil.rmtree(dirs[1])
    p = subprocess.run([CLI, "--samples", m, "-r", libs[0], "-r", libs[1], "-o"] + dirs + ["-c", "4"] + (["--bulk"] if bulk else []), capture_output=True, text=True)
    assert p.returncode == 101 and p.stderr.rstrip("\n").split("\n")[-1] == msg, p.stderr
    assert sorted(os.listdir(dirs[0])) == sorted([samples[0][0] + ".tsv", samples[1][0] + ".tsv"])


def test_fastq_failure_mid_run(tmp_path, fastq_set):
    _, S = fastq_set
    S = dict(S)
    L = synth.SynthLibrary(seed=1234, n_fam=40, n_all=5)
    r1 = write_reads(L, tmp_path, "u", 500, first=800_000)[0]
    r2 = write_reads(L, tmp_path, "v", 499, first=900_000)[1]             # one record short
    _, lib_a = library(tmp_path, "a.json", 1234)
    _, lib_b = library(tmp_path, "b.json", 77)
    samples = [("one", S["plain"]), ("two", S["single"]), ("unequal", [r1, r2]), ("four", S["gz"]), ("five", S["tiny"])]
    check_mid_run_failure(tmp_path, samples, [lib_a, lib_b], False, single_fastq)


def test_bulk_failure_mid_run(tmp_path, bam_set):
    _, S = bam_set
    S = dict(S)
    mixed = write_bam(tmp_path / "mixed.bam", [bulk_ref.Rec("a", P1, "ACGT" * 20), bulk_ref.Rec("a", P2, "TTGA" * 20), bulk_ref.Rec("b", 0, "ACGT" * 20)])
    _, lib_a = library(tmp_path, "a.json", 1234)
    _, lib_b = library(tmp_path, "b.json", 77)
    samples = [("one", [S["shuffled"]]), ("two", [S["single"]]), ("mixed", [mixed]), ("four", [S["collated"]]), ("five", [S["nothing_kept"]])]
    check_mid_run_failure(tmp_path, samples, [lib_a, lib_b], True, lambda ins, libs, d, n: single_bulk(ins[0], libs, d, n))
