#!/usr/bin/env python
"""BAM mode in any record order under a device-memory budget, on the shuffled C3-shaped file of bench_bam_any_order.py
(single-end 91 bp records, CB/UB tags, 8000 cells, records randomly permuted).  `nimble --any-order --no-rows
--cell-matrix` runs unbudgeted first; its peak device bytes (store + grouping arrays of the NB_BAM_STATS line) sets the
budgets of the next runs: 1/2, 1/4 and 1/8 of it (`--device-budget`).  Prints one JSON line: per run the wall time,
passes, evictions, peak device bytes and the windows time of each pass, matrices_equal (every budgeted matrix directory
byte-identical to the unbudgeted one) and the card's name and power limit read in the same call."""
import argparse, json, os, re, shutil, subprocess, sys, tempfile, time
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import numpy as np
import bench_bam_any_order as bo
import nimble_aligner_b200 as nb
import synth


def files(d):
    return {f: open(os.path.join(d, f), "rb").read() for f in sorted(os.listdir(d))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--groups", type=int, default=5_000_000, help="UMI groups (about 4 records each)")
    a = ap.parse_args()
    cores = os.cpu_count() or 1
    L = 91
    lib = synth.SynthLibrary(seed=1234, n_fam=200, n_all=5, group_on="", trim_target_length=40, trim_strictness=0.9)
    tmp = tempfile.mkdtemp(prefix="nb_bam_any_order_budget_")
    lib_path = os.path.join(tmp, "lib.json"); json.dump(lib.to_json_obj(), open(lib_path, "w"))
    u = synth.umi_reads(lib, 0, a.groups, seed=2345, threads=cores)
    n = u["n_reads"]
    perm = np.random.default_rng(99).permutation(n)       # the shuffled file of bench_bam_any_order.py
    s = bo.with_order(u, perm, L)
    shuffled = os.path.join(tmp, "shuffled.bam"); size_s = synth.write_umi_bam(shuffled, s, threads=cores); del s, u
    exe = os.path.join(os.path.dirname(os.path.abspath(nb.__file__)), "nimble")
    env = dict(os.environ, NB_BAM_STATS="1")

    def run(name, budget):
        out = os.path.join(tmp, name)
        t = time.time()
        pr = subprocess.run([exe, "-r", lib_path, "-i", shuffled, "-c", str(cores), "--any-order", "--no-rows", "--cell-matrix", out] + (["--device-budget", str(budget)] if budget else []),
                            check=True, stdout=subprocess.DEVNULL, stderr=subprocess.PIPE, text=True, env=env)
        dt = time.time() - t
        line = [l for l in pr.stderr.split("\n") if l.startswith("nb_process_bam_any_order:")][-1]
        num = lambda rx: int(re.search(rx, line).group(1))   # noqa: E731
        r = {"budget": budget, "seconds": round(dt, 3), "store_bytes": num(r"store (\d+) bytes"), "grouping_bytes": num(r"grouping (\d+) bytes"),
             "windows_s": float(re.search(r"windows \(read\+inflate\+stage\+upload\) ([\d.]+)s", line).group(1))}
        if budget:
            r.update(passes=num(r"passes (\d+)"), evictions=num(r"evictions (\d+)"), peak_device_bytes=num(r"peak device bytes (\d+)"),
                     windows_per_pass_s=[float(x.rstrip("s")) for x in re.search(r"windows per pass (\S+)", line).group(1).split("/")])
        else:
            r.update(passes=1, evictions=0, peak_device_bytes=r["store_bytes"] + r["grouping_bytes"])
        return r, files(out)

    base, ref = run("unbudgeted", 0)
    runs, equal = [base], True
    for div in (2, 4, 8):
        r, got = run("budget_1_%d" % div, base["peak_device_bytes"] // div)
        runs.append(r); equal = equal and got == ref
    res = {"workload": "C3-shaped BAM in any record order: %d single-end 91 bp records in %d (UMI,CB) groups, 8000 cells, randomly permuted, %.0f MB; `nimble --any-order --no-rows --cell-matrix [--device-budget B]`" % (n, a.groups, size_s / 1e6),
           "host_threads": cores, "runs": runs, "matrices_equal": equal, "card": bo.card()}
    print(json.dumps(res))
    shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
