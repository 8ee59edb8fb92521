"""CPU tests of the sample manifest (`nimble --samples`, process_samples, nb_process_samples): the manifest rules, the CLI
refusals, the checks made before any device work, and the Python argument checks.  A run that passes every check fails
afterwards on a library that does not exist, before any device is touched."""
import os
import subprocess

import pytest

import nimble_aligner_b200 as nb

LIB = os.path.join(os.path.dirname(__file__), "golden", "ref", "libraries", "basic.json")
CLI = os.path.join(os.path.dirname(nb.SO_PATH), "nimble")
FQ = b"@a\nACGT\n+\nIIII\n"


@pytest.fixture
def inputs(tmp_path):
    for n in ("a_1.fastq", "a_2.fastq", "b.FASTQ"):
        (tmp_path / n).write_bytes(FQ)
    (tmp_path / "c.fastq.gz").write_bytes(b"")
    (tmp_path / "x.bam").write_bytes(b"")
    (tmp_path / "y.bam").write_bytes(b"")
    return tmp_path


def manifest(tmp_path, text, name="m.tsv"):
    (tmp_path / name).write_text(text)
    return str(tmp_path / name)


def cli(tmp_path, args, env_extra=None):
    env = dict(os.environ)
    env.pop("NB_DEVICES", None)
    env.update(env_extra or {})
    return subprocess.run([CLI] + args, capture_output=True, text=True, cwd=tmp_path, env=env)


GOOD = "# cohort\n\na\ta_1.fastq\ta_2.fastq\n  \nb\tb.FASTQ\n#c\tnot\ta sample\nc.1_x-Y\tc.fastq.gz\r\n"


def test_manifest_comments_and_blank_lines(inputs):
    assert nb.read_manifest(manifest(inputs, GOOD)) == [("a", ["a_1.fastq", "a_2.fastq"], 3), ("b", ["b.FASTQ"], 5), ("c.1_x-Y", ["c.fastq.gz"], 7)]


def test_cli_accepts_manifest(inputs):
    # past every check: the output directories exist, and the run fails on the missing library (no device touched)
    p = cli(inputs, ["--samples", manifest(inputs, GOOD), "-r", "missing.json", "-o", "out", "-c", "4", "-f", "fiveprime"])
    assert p.returncode == 101 and "Processing 3 FASTQ samples" in p.stdout, p.stdout + p.stderr
    assert not p.stderr.startswith("error:") and "sample" not in p.stderr, p.stderr
    assert os.path.isdir(inputs / "out") and os.listdir(inputs / "out") == []


def test_python_accepts_manifest_and_list(inputs, monkeypatch):
    monkeypatch.chdir(inputs)
    for samples in (manifest(inputs, GOOD), [("a", ["a_1.fastq", "a_2.fastq"]), ("b", ("b.FASTQ",))]):
        with pytest.raises(nb.NbError) as e:
            nb.process_samples(samples, ["missing.json"], ["out"])
        assert e.value.code not in (0, -1) and "sample" not in str(e.value), str(e.value)   # the missing library, after the checks
    assert os.path.isdir(inputs / "out")


BAD = [
    ("a\ta_1.fastq\n#\nb\n", 3, "found 1 column"),
    ("a\ta_1.fastq\ta_2.fastq\ta_1.fastq\n", 1, "found 4 column"),
    ("a\t\ta_1.fastq\n", 1, "empty column"),
    ("a\ta_1.fastq\n\na\tb.FASTQ\n", 3, "'a' is already used on line 1"),
    ("a/b\ta_1.fastq\n", 1, "must match"),
    ("..\ta_1.fastq\n", 1, "must match"),
    (".\ta_1.fastq\n", 1, "must match"),
    ("a b\ta_1.fastq\n", 1, "must match"),
]


@pytest.mark.parametrize("text,line,msg", BAD)
def test_manifest_syntax_and_names_refused_by_line(inputs, text, line, msg):
    m = manifest(inputs, text)
    p = cli(inputs, ["--samples", m, "-r", LIB, "-o", "out"])
    assert p.returncode == 101 and ("m.tsv line %d: " % line) in p.stderr and msg in p.stderr, p.stderr
    with pytest.raises(nb.NbError) as e:
        nb.process_samples(m, [LIB], [str(inputs / "out")])
    assert e.value.code == -1 and ("m.tsv line %d: " % line) in str(e.value) and msg in str(e.value), str(e.value)
    assert not os.path.exists(inputs / "out")


def test_empty_manifest_refused(inputs):
    m = manifest(inputs, "# nothing\n\n")
    p = cli(inputs, ["--samples", m, "-r", LIB, "-o", "out"])
    assert p.returncode == 101 and "has no samples" in p.stderr, p.stderr
    with pytest.raises(nb.NbError) as e:
        nb.process_samples(m, [LIB], [str(inputs / "out")])
    assert e.value.code == -1 and "has no samples" in str(e.value)
    assert not os.path.exists(inputs / "out")


KINDS = [
    ("a\ta_1.fastq\n# bams need --bulk\nx\tx.bam\n", False, "sample x (line 3): x.bam is a BAM"),                    # mixed kinds
    ("x\tx.bam\n", False, "sample x (line 1): x.bam is a BAM"),                                                       # a BAM without --bulk
    ("x\tx.bam\ny\ty.bam\nb\tb.FASTQ\n", True, "sample b (line 3): a bulk sample has exactly one .bam input"),       # FASTQ with --bulk
    ("x\tx.bam\ty.bam\n", True, "sample x (line 1): a bulk sample has exactly one .bam input"),
    ("a\ta_1.fastq\tx.txt\n", False, "sample a (line 1): unsupported file format of x.txt"),
]


@pytest.mark.parametrize("text,bulk,msg", KINDS)
def test_input_kinds_refused_by_line(inputs, monkeypatch, text, bulk, msg):
    m = manifest(inputs, text)
    p = cli(inputs, ["--samples", m, "-r", LIB, "-o", "out"] + (["--bulk"] if bulk else []))
    assert p.returncode == 101 and p.stderr.startswith(msg), p.stderr
    monkeypatch.chdir(inputs)
    with pytest.raises(nb.NbError) as e:
        nb.process_samples(m, [LIB], ["out"], bulk=bulk)
    assert e.value.code == -1 and msg in str(e.value), str(e.value)
    assert not os.path.exists(inputs / "out")


@pytest.mark.parametrize("bulk", [False, True])
def test_missing_input_on_last_line_refused_before_any_output(inputs, monkeypatch, bulk):
    rows = ["s%03d\t%s\n" % (i, "x.bam" if bulk else "a_1.fastq\ta_2.fastq") for i in range(299)]
    m = manifest(inputs, "".join(rows) + ("last\t%s\n" % ("gone.bam" if bulk else "a_1.fastq\tgone.fastq")))
    p = cli(inputs, ["--samples", m, "-r", LIB, "-r", LIB, "-o", "out1", "out2"] + (["--bulk"] if bulk else []))
    assert p.returncode == 101 and p.stderr.startswith("sample last (line 300): could not open gone."), p.stderr
    monkeypatch.chdir(inputs)
    with pytest.raises(nb.NbError) as e:
        nb.process_samples(m, [LIB, LIB], ["out1", "out2"], bulk=bulk)
    assert e.value.code == -2 and "sample last (line 300): could not open gone." in str(e.value), str(e.value)
    assert not os.path.exists(inputs / "out1") and not os.path.exists(inputs / "out2")


def test_output_directory_needs_its_parent(inputs):
    p = cli(inputs, ["--samples", manifest(inputs, "a\ta_1.fastq\n"), "-r", LIB, "-r", LIB, "-o", "ok", "no/such/dir"])
    assert p.returncode == 101 and "could not create output directory no/such/dir" in p.stderr, p.stderr
    (inputs / "file").write_text("")
    p = cli(inputs, ["--samples", "m.tsv", "-r", LIB, "-o", "file"])
    assert p.returncode == 101 and "output directory file is not a directory" in p.stderr, p.stderr


@pytest.mark.parametrize("extra,msg", [
    (["-i", "a_1.fastq"], "leave out --input"),
    (["--cell-matrix", "m"], "--cell-matrix"),
    (["--cell-matrix", "m", "--no-rows"], "--no-rows"),
    (["--any-order"], "--any-order"),
    (["-p"], "-p"),
    (["--device-budget", "8G"], "--device-budget"),
    (["--bulk", "-p"], "-p"),
    (["-d", "0,1"], "samples run on one GPU"),
    (["-r", LIB], "one --output directory per --reference library"),        # 2 -r, 1 -o
    (["-t", "40:0.9,40:0.9"], "trim options"),                               # -t keeps its count check
])
def test_cli_refuses(inputs, extra, msg):
    m = manifest(inputs, "a\ta_1.fastq\n")
    p = cli(inputs, ["--samples", m, "-r", LIB, "-o", "out"] + extra)
    assert p.returncode == 101 and msg in p.stderr, p.stderr
    assert not os.path.exists(inputs / "out") and not os.path.exists(inputs / "m")


def test_cli_refuses_several_devices_from_env(inputs):
    p = cli(inputs, ["--samples", manifest(inputs, "a\ta_1.fastq\n"), "-r", LIB, "-o", "out"], env_extra={"NB_DEVICES": "0,1"})
    assert p.returncode == 101 and "samples run on one GPU" in p.stderr, p.stderr
    assert not os.path.exists(inputs / "out")


def test_cli_needs_outputs_and_a_readable_manifest(inputs):
    p = cli(inputs, ["--samples", manifest(inputs, "a\ta_1.fastq\n"), "-r", LIB])
    assert p.returncode == 101 and "one --output directory per --reference library" in p.stderr, p.stderr
    p = cli(inputs, ["--samples", "nope.tsv", "-r", LIB, "-o", "out"])
    assert p.returncode == 101 and "could not read the sample manifest nope.tsv" in p.stderr, p.stderr
    assert not os.path.exists(inputs / "out")


def test_python_argument_checks(inputs, monkeypatch):
    monkeypatch.chdir(inputs)
    ok = [("a", ["a_1.fastq"])]
    cases = [
        ([], [LIB], ["out"], {}),
        ([("a",)], [LIB], ["out"], {}),
        ([("a", "a_1.fastq")], [LIB], ["out"], {}),                                  # inputs not a list
        ([("a", [])], [LIB], ["out"], {}),
        ([("a", ["a_1.fastq", "a_2.fastq", "a_1.fastq"])], [LIB], ["out"], {}),
        ([(1, ["a_1.fastq"])], [LIB], ["out"], {}),
        (ok, [], ["out"], {}),
        (ok, [LIB], [], {}),
        (ok, [LIB], "out", {}),
        (ok, [LIB, LIB], ["out"], {}),
        (ok, [LIB], ["out"], dict(strand_filter="sideways")),
        (str(inputs / "nope.tsv"), [LIB], ["out"], {}),
        ([("a/b", ["a_1.fastq"])], [LIB], ["out"], {}),                              # name checks of nb_process_samples, before any device work
        ([("a", ["a_1.fastq"]), ("a", ["b.FASTQ"])], [LIB], ["out"], {}),
        ([("x", ["x.bam"])], [LIB], ["out"], {}),
    ]
    for samples, refs, outs, kw in cases:
        with pytest.raises(nb.NbError) as e:
            nb.process_samples(samples, refs, outs, **kw)
        assert e.value.code == -1, (samples, refs, outs, kw, str(e.value))
    assert not os.path.exists(inputs / "out")


def test_help_lists_samples():
    out = subprocess.run([CLI, "--help"], capture_output=True, text=True, check=True).stdout
    assert "--samples <file>" in out
