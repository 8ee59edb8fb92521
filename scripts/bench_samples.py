#!/usr/bin/env python
"""A cohort through one `nimble --samples` run against one `nimble` process per sample, for FASTQ and bulk BAM samples,
with and without --index-cache, in one call:
  manifest    `nimble --samples m.tsv -r lib -o dir [--bulk]`: setup once, then sample after sample
  separate    `nimble -i r1 r2 -r lib -o dir/<name>.tsv` (or `--bulk -i x.bam`) for each sample: setup every time
The samples are C2-shaped pairs (150 bp, 1k-transcript library), --pairs per sample, written as plain FASTQ R1/R2 and as a
BAM in shuffled record order (bench_bam_bulk.py's writer).  --distinct sets of pairs are generated and the N sample names
cycle through them, so that a large cohort does not need N sets of files on disk; every run reads from the page cache
alike.  --separate K runs only the first K samples as separate processes (default: all N) and reports their mean; the
JSON then names the N-sample figure an extrapolation.  The cached arms run after one warm-up run has written the cache.
Arms are alternated --repeat times.  Every TSV is asserted equal to the separate run of the same pairs, and the FASTQ and
bulk TSVs to each other.  One JSON line: wall times, the manifest runs' setup line and per-sample phases (NB_FASTQ_STATS /
NB_BAM_STATS), and the card's name and power limit read in the same call."""
import argparse, json, os, re, shutil, subprocess, sys, tempfile, time
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench_bam_any_order as bo
import bench_bam_bulk as bb
import nimble_aligner_b200 as nb
import synth

SETUP = re.compile(r"nb_process_samples: setup ([\d.]+) s")
FQ_SAMPLE = re.compile(r"nb_process_samples: sample \S+: (\d+) pairs, parse\+align ([\d.]+) s, finalize\+tsv ([\d.]+) s")
BULK_SAMPLE = re.compile(r"nb_process_samples: sample \S+: \d+ records, (\d+) pairs, windows ([\d.]+) s, pairing ([\d.]+) s, align\+finalize\+tsv ([\d.]+) s")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=32)
    ap.add_argument("--pairs", type=int, default=1_000_000)
    ap.add_argument("--repeat", type=int, default=1)
    ap.add_argument("--distinct", type=int, default=4)
    ap.add_argument("--separate", type=int, default=0)
    a = ap.parse_args()
    N, D = a.samples, max(1, min(a.distinct, a.samples))
    K = min(N, max(a.separate, D)) if a.separate > 0 else N   # (at least one run of every distinct set: the reference bytes)
    cores = os.cpu_count() or 1
    exe = os.path.join(os.path.dirname(os.path.abspath(nb.__file__)), "nimble")
    lib = synth.SynthLibrary(seed=1234, n_fam=200, n_all=5)
    tmp = tempfile.mkdtemp(prefix="nb_samples_")
    try:
        lib_path = os.path.join(tmp, "lib.json"); json.dump(lib.to_json_obj(), open(lib_path, "w"))
        fq, bam = [], []
        for d in range(D):
            r1, o1, r2, o2 = synth.pairs(lib, d * a.pairs, a.pairs, threads=cores)
            f = [os.path.join(tmp, "d%d_%d.fastq" % (d, m)) for m in (1, 2)]
            synth.write_fastq(f[0], r1, o1, 1); synth.write_fastq(f[1], r2, o2, 2)
            b = os.path.join(tmp, "d%d.bam" % d); bb.write_bam(b, (r1, o1, r2, o2), a.pairs, 99 + d, cores)
            fq.append(f); bam.append(b); del r1, r2
        names = ["s%04d" % i for i in range(N)]
        inputs = {"fastq": [fq[i % D] for i in range(N)], "bulk": [[bam[i % D]] for i in range(N)]}
        manifests = {}
        for kind in inputs:
            manifests[kind] = os.path.join(tmp, kind + ".tsv")
            with open(manifests[kind], "w") as f:
                for n, ins in zip(names, inputs[kind]):
                    f.write("\t".join([n] + ins) + "\n")
        cache = os.path.join(tmp, "cache")
        env = dict(os.environ, NB_BAM_STATS="1", NB_FASTQ_STATS="1")
        env.pop("NB_INDEX_CACHE", None)

        def cached(c):
            return ["--index-cache", cache] if c else []

        def manifest_run(kind, c):
            out = os.path.join(tmp, "m_%s_%d" % (kind, c)); shutil.rmtree(out, ignore_errors=True)
            t = time.time()
            pr = subprocess.run([exe, "--samples", manifests[kind], "-r", lib_path, "-o", out, "-c", str(cores)] + (["--bulk"] if kind == "bulk" else []) + cached(c),
                                check=True, stdout=subprocess.DEVNULL, stderr=subprocess.PIPE, text=True, env=env)
            dt = time.time() - t
            rx = FQ_SAMPLE if kind == "fastq" else BULK_SAMPLE
            per = [tuple(float(x) for x in m.groups()) for m in rx.finditer(pr.stderr)]
            assert len(per) == N, pr.stderr[-2000:]
            cols = ["parse_align", "finalize_tsv"] if kind == "fastq" else ["windows", "pairing", "align_finalize_tsv"]
            ph = {"setup": float(SETUP.search(pr.stderr).group(1)), "pairs_per_sample": per[0][0]}
            ph.update({c + "_total": round(sum(p[k + 1] for p in per), 3) for k, c in enumerate(cols)})
            ph.update({c + "_mean": round(sum(p[k + 1] for p in per) / N, 4) for k, c in enumerate(cols)})
            return dt, ph, out

        def separate_run(kind, c):
            out = os.path.join(tmp, "s_%s_%d" % (kind, c)); shutil.rmtree(out, ignore_errors=True); os.makedirs(out)
            t = time.time()
            for n, ins in zip(names[:K], inputs[kind][:K]):
                subprocess.run([exe, "-r", lib_path, "-i"] + ins + ["-o", os.path.join(out, n + ".tsv"), "-c", str(cores)] + (["--bulk"] if kind == "bulk" else []) + cached(c),
                               check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, env=env)
            return time.time() - t, out

        subprocess.run([exe, "-r", lib_path, "-i"] + fq[0] + ["-o", os.path.join(tmp, "warm.tsv")] + cached(True), check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, env=env)
        walls, phases, outs = {}, {}, {}
        for _ in range(a.repeat):   # alternated: a drift of the machine touches every arm alike
            for c in (False, True):
                for kind in ("fastq", "bulk"):
                    key = "%s%s" % (kind, "_index_cache" if c else "")
                    dt, ph, out = manifest_run(kind, c)
                    walls.setdefault(key + "_manifest", []).append(round(dt, 3)); phases.setdefault(key, []).append(ph); outs[key + "_manifest"] = out
                    dt, out = separate_run(kind, c)
                    walls.setdefault(key + "_separate", []).append(round(dt, 3)); outs[key + "_separate"] = out
        want = [open(os.path.join(outs["fastq_separate"], n + ".tsv"), "rb").read() for n in names[:min(K, D)]]
        for key, out in outs.items():
            for i, n in enumerate(names if key.endswith("_manifest") else names[:K]):
                assert open(os.path.join(out, n + ".tsv"), "rb").read() == want[i % D], (key, n)
        runs = {}
        for key in phases:
            m, s = min(walls[key + "_manifest"]), min(walls[key + "_separate"])
            runs[key] = {"manifest_seconds": m, "manifest_all_seconds": walls[key + "_manifest"], "manifest_phases": min(phases[key], key=lambda p: p["setup"]),
                         "separate_seconds_measured": s, "separate_all_seconds": walls[key + "_separate"], "separate_runs_measured": K,
                         "separate_mean_seconds_per_run": round(s / K, 4),
                         ("separate_seconds" if K == N else "separate_seconds_extrapolated"): round(s / K * N, 3),
                         "speedup_manifest_vs_separate": round(s / K * N / m, 3)}
        res = {"workload": "%d samples x %d C2-shaped pairs of 150 bp (%d distinct sets of pairs), 1k-transcript library; FASTQ %.0f MB plain and BAM (shuffled, no CB) %.0f MB per sample"
                           % (N, a.pairs, D, sum(os.path.getsize(f) for f in fq[0]) / 1e6, os.path.getsize(bam[0]) / 1e6),
               "host_threads": cores, "repeat": a.repeat, "runs": runs, "tsv_equal": True, "card": bo.card()}
        print(json.dumps(res))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
