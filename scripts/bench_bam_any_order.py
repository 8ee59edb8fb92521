#!/usr/bin/env python
"""BAM mode in any record order against the grouped matrix-only run, on the C3-shaped synthetic BAM of bench_bam_matrix.py
(single-end 91 bp records, CB/UB tags, 8000 cells).  Two files hold the same records:
  grouped   the shuffled file's records stably sorted by (UMI, CB) plus one sentinel record with a UMI of its own at the end: the file G
            for which `nimble --no-rows --cell-matrix` and `nimble --any-order` must give the same matrix (the grouped
            reader never sends the last group; synthetic UMIs of different groups collide, so the generator's own group
            order is not a valid grouped file)
  shuffled  the records in random order (the umi_reads arrays permuted before synth.write_umi_bam)
The two runs are alternated --repeat times in one process.  Prints one JSON line: wall times (best and all), the
NB_BAM_STATS phases of each mode's best run, the device store bytes, peak RSS, matrices_equal (the two matrices compared as
{(feature, barcode): (umis, reads)}) and the card's name and power limit read in the same call."""
import argparse, gzip, json, os, re, shutil, subprocess, sys, tempfile, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import nimble_aligner_b200 as nb
import synth

GROUPED = {"windows": r"windows \(read\+inflate\+group, overlapped\) ([\d.]+)s", "fill": r"batch fill ([\d.]+)s",
           "device": r"device align\+finalize ([\d.]+)s", "cell_roll": r"cell roll ([\d.]+)s",
           "cell_finalize_write": r"cell finalize\+matrix write ([\d.]+)s", "total": r"total ([\d.]+)s", "peak_rss_mb": r"peak RSS (\d+) MB"}
ANY = {"setup": r"setup ([\d.]+)s", "windows": r"windows \(read\+inflate\+stage\+upload\) ([\d.]+)s", "upload_wait": r"upload wait ([\d.]+)s",
       "key_sort_scope": r"key\+sort\+scope build ([\d.]+)s", "device": r"device align\+finalize ([\d.]+)s", "cell_roll": r"cell roll ([\d.]+)s",
       "cell_finalize_write": r"cell finalize\+matrix write ([\d.]+)s", "total": r"total ([\d.]+)s", "store_bytes": r"store (\d+) bytes",
       "grouping_bytes": r"grouping (\d+) bytes", "peak_rss_mb": r"peak RSS (\d+) MB", "records": r"(\d+) records", "scopes": r"(\d+) scopes",
       "pairs": r"(\d+) pairs"}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip().split("\n")[0]
        name, power, clock = [x.strip() for x in q.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:   # the numbers below still stand; the card is then unnamed
        return {"gpu": None, "error": str(e)}


def sort_key(v, n):
    """synth_write_bam writes character i of a tag as "ACGT"[(v >> 2i) & 3]: the integer that sorts like the string"""
    k = np.zeros_like(v)
    for i in range(n):
        k = (k << np.uint64(2)) | ((v >> np.uint64(2 * i)) & np.uint64(3))
    return k


def tag_values(ids, mult):
    with np.errstate(over="ignore"):
        return (ids.astype(np.uint64) * np.uint64(mult)) >> np.uint64(8)


def with_order(u, order, L):
    n = len(order)
    out = dict(u)
    out["bases"] = np.concatenate([u["bases"][: u["n_reads"] * L].reshape(-1, L)[order].ravel(), np.zeros(64, np.uint8)])
    out["qual"] = np.concatenate([u["qual"][: u["n_reads"] * L].reshape(-1, L)[order].ravel(), np.zeros(64, np.uint8)])
    out["cell"] = np.ascontiguousarray(u["cell"][order]); out["scope"] = np.ascontiguousarray(u["scope"][order]); out["n_reads"] = n
    return out


def matrix(d):
    feats = [l.split("\t")[0] for l in gzip.open(os.path.join(d, "features.tsv.gz"), "rt").read().split("\n")[:-1]]
    bcs = gzip.open(os.path.join(d, "barcodes.tsv.gz"), "rt").read().split("\n")[:-1]
    mu = gzip.open(os.path.join(d, "matrix.mtx.gz"), "rt").read().split("\n")[2:-1]
    mr = gzip.open(os.path.join(d, "reads.mtx.gz"), "rt").read().split("\n")[2:-1]
    out = {}
    for a, b in zip(mu, mr):
        f, c, n = (int(x) for x in a.split()); out[(feats[f - 1], bcs[c - 1])] = (n, int(b.split()[2]))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--groups", type=int, default=5_000_000, help="UMI groups (about 4 records each)")
    ap.add_argument("--repeat", type=int, default=3)
    a = ap.parse_args()
    cores = os.cpu_count() or 1
    L = 91
    lib = synth.SynthLibrary(seed=1234, n_fam=200, n_all=5, group_on="", trim_target_length=40, trim_strictness=0.9)
    tmp = tempfile.mkdtemp(prefix="nb_bam_any_order_")
    lib_path = os.path.join(tmp, "lib.json"); json.dump(lib.to_json_obj(), open(lib_path, "w"))
    u = synth.umi_reads(lib, 0, a.groups, seed=2345, threads=cores)
    n = u["n_reads"]
    umi = sort_key(tag_values(u["scope"], 0x9E3779B97F4A7C15), 12); cbk = sort_key(tag_values(u["cell"], 0xD1B54A32D192ED03), 16)
    perm = np.random.default_rng(99).permutation(n)       # the shuffled file's record order
    # G is the stable sort of the SHUFFLED file: inside a scope the order decides which of two pairs with the same bases (and
    # different quals, so possibly different trims) the read_key de-duplication keeps
    order = perm[np.lexsort((cbk[perm], umi[perm]))]
    g = with_order(u, order, L)
    sentinel = a.groups                                   # a group id whose UMI differs from the last sorted one
    while sort_key(tag_values(np.array([sentinel], np.uint64), 0x9E3779B97F4A7C15), 12)[0] == umi[order[-1]]:
        sentinel += 1
    g["bases"] = np.concatenate([g["bases"][: n * L], g["bases"][n * L - L: n * L], np.zeros(64, np.uint8)])
    g["qual"] = np.concatenate([g["qual"][: n * L], g["qual"][n * L - L: n * L], np.zeros(64, np.uint8)])
    g["cell"] = np.append(g["cell"], np.uint32(0)); g["scope"] = np.append(g["scope"], np.uint32(sentinel)); g["n_reads"] = n + 1
    grouped = os.path.join(tmp, "grouped.bam"); size_g = synth.write_umi_bam(grouped, g, threads=cores); del g
    s = with_order(u, perm, L)
    shuffled = os.path.join(tmp, "shuffled.bam"); size_s = synth.write_umi_bam(shuffled, s, threads=cores); del s, u
    exe = os.path.join(os.path.dirname(os.path.abspath(nb.__file__)), "nimble")
    modes = {"grouped_matrix_only": (grouped, [], "nb_process_bam:", GROUPED), "any_order_shuffled": (shuffled, ["--any-order"], "nb_process_bam_any_order:", ANY)}
    env = dict(os.environ, NB_BAM_STATS="1")
    best, walls = {}, {m: [] for m in modes}
    for _ in range(a.repeat):
        for mode, (path, extra, prefix, rx) in modes.items():   # alternated: a drift of the machine touches both modes alike
            out = os.path.join(tmp, mode)
            t = time.time()
            pr = subprocess.run([exe, "-r", lib_path, "-i", path, "-c", str(cores), "--no-rows", "--cell-matrix", out] + extra, check=True, stdout=subprocess.DEVNULL, stderr=subprocess.PIPE, text=True, env=env)
            dt = time.time() - t
            line = [l for l in pr.stderr.split("\n") if l.startswith(prefix)][-1]
            ph = {k: float(m.group(1)) for k, r in rx.items() for m in [re.search(r, line)] if m}
            walls[mode].append(round(dt, 3))
            if mode not in best or dt < best[mode]["seconds"]:
                best[mode] = {"seconds": round(dt, 3), "records_per_s": n / dt, "phases": ph}
    for mode in modes:
        best[mode]["all_seconds"] = walls[mode]
    m_g, m_a = matrix(os.path.join(tmp, "grouped_matrix_only")), matrix(os.path.join(tmp, "any_order_shuffled"))
    res = {"workload": "C3-shaped BAM: %d single-end 91 bp records in %d (UMI,CB) groups, 8000 cells, 1k-transcript library; grouped (sorted by UMI, CB, + 1 sentinel record) %.0f MB, shuffled %.0f MB; `nimble --no-rows --cell-matrix` per run" % (n, a.groups, size_g / 1e6, size_s / 1e6),
           "host_threads": cores, "repeat": a.repeat, "modes": best,
           "store_bytes": best["any_order_shuffled"]["phases"].get("store_bytes"), "peak_rss_mb": {m: best[m]["phases"].get("peak_rss_mb") for m in modes},
           "matrices_equal": m_g == m_a, "matrix_entries": len(m_a),
           "slowdown_any_order_vs_grouped": round(best["any_order_shuffled"]["seconds"] / best["grouped_matrix_only"]["seconds"], 3)}
    res["card"] = card()
    print(json.dumps(res))
    shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
