#!/usr/bin/env python
"""BAM mode with and without the per-cell matrix, on the C3-shaped synthetic BAM of bench_bam.py (single-end 91 bp records,
CB/UB tags, 8000 cells): three runs of nb_process_bam_cells, alternated and repeated in one process so that they share the
machine's state — rows only (the TSV.gz, as nb_process_bam), rows + matrix, matrix only (no rows stage).  Prints one JSON
line: records/s per mode (best of the repeats), the NB_BAM_STATS phase times of each mode's best run, and the card's name and
power limit read in the same call."""
import argparse, json, os, re, subprocess, sys, tempfile, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import nimble_aligner_b200 as nb
import synth

PHASES = {"windows": r"windows \(read\+inflate\+group, overlapped\) ([\d.]+)s", "fill": r"batch fill ([\d.]+)s",
          "device": r"device align\+finalize ([\d.]+)s", "rows": r"rows\+gzip\+write ([\d.]+)s", "cell_roll": r"cell roll ([\d.]+)s",
          "cell_finalize_write": r"cell finalize\+matrix write ([\d.]+)s", "total": r"total ([\d.]+)s", "peak_rss_mb": r"peak RSS (\d+) MB"}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip().split("\n")[0]
        name, power, clock = [x.strip() for x in q.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:   # the numbers below still stand; the card is then unnamed
        return {"gpu": None, "error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--groups", type=int, default=1_250_000, help="UMI groups (about 4 records each)")
    ap.add_argument("--repeat", type=int, default=3)
    a = ap.parse_args()
    cores = os.cpu_count() or 1
    L = synth.SynthLibrary(seed=1234, n_fam=200, n_all=5, group_on="", trim_target_length=40, trim_strictness=0.9)
    tmp = tempfile.mkdtemp(prefix="nb_bam_matrix_")
    lib_path = os.path.join(tmp, "lib.json"); json.dump(L.to_json_obj(), open(lib_path, "w"))
    u = synth.umi_reads(L, 0, a.groups, seed=2345, threads=cores)
    bam = os.path.join(tmp, "c3.bam"); size = synth.write_umi_bam(bam, u, threads=cores)
    n = u["n_reads"]; del u
    exe = os.path.join(os.path.dirname(os.path.abspath(nb.__file__)), "nimble")
    modes = {"rows": ["-o", os.path.join(tmp, "out.tsv.gz")],
             "rows_and_matrix": ["-o", os.path.join(tmp, "out.tsv.gz"), "--cell-matrix", os.path.join(tmp, "m_rows")],
             "matrix_only": ["--no-rows", "--cell-matrix", os.path.join(tmp, "m_only")]}
    env = dict(os.environ, NB_BAM_STATS="1")
    best, walls = {}, {m: [] for m in modes}
    for _ in range(a.repeat):
        for mode, extra in modes.items():   # alternated: a drift of the machine touches every mode alike
            t = time.time()
            pr = subprocess.run([exe, "-r", lib_path, "-i", bam, "-c", str(cores)] + extra, check=True, stdout=subprocess.DEVNULL, stderr=subprocess.PIPE, text=True, env=env)
            dt = time.time() - t
            line = [l for l in pr.stderr.split("\n") if l.startswith("nb_process_bam:")][-1]
            ph = {k: float(m.group(1)) for k, rx in PHASES.items() for m in [re.search(rx, line)] if m}
            walls[mode].append(round(dt, 3))
            if mode not in best or dt < best[mode]["seconds"]:
                best[mode] = {"seconds": dt, "records_per_s": n / dt, "phases_s": ph}
    for mode in modes:
        best[mode]["all_seconds"] = walls[mode]   # the spread of the repeats
    res = {"workload": "C3-shaped BAM: %d single-end 91 bp records in %d (UMI,CB) groups, 8000 cells, 1k-transcript library; %.0f MB BAM; `nimble` CLI per run" % (n, a.groups, size / 1e6),
           "host_threads": cores, "repeat": a.repeat, "modes": best}
    files = {m: sorted(os.listdir(os.path.join(tmp, d))) for m, d in (("rows_and_matrix", "m_rows"), ("matrix_only", "m_only"))}
    same = all(open(os.path.join(tmp, "m_rows", f), "rb").read() == open(os.path.join(tmp, "m_only", f), "rb").read() for f in files["matrix_only"])
    res["matrix_files_identical"] = same and files["rows_and_matrix"] == files["matrix_only"]
    res["card"] = card()
    print(json.dumps(res))
    import shutil; shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
