#!/usr/bin/env python
"""TSV.gz rows of BAM mode in any record order against the grouped rows run, on the C3-shaped files of bench_bam_any_order.py
(single-end 91 bp records, CB/UB tags, 8000 cells): the shuffled file and G (its records stably sorted by (UMI, CB) plus one
sentinel record).  Runs, alternated --repeat times in one call:
  any_order         `nimble --any-order -o` on the shuffled file
  grouped           `nimble -o` on G (the sort by UB the any-order rows make unnecessary is not timed)
  budget_1_2/1_4    `nimble --any-order -o --device-budget B` at 1/2 and 1/4 of the unbudgeted run's peak device bytes
Prints one JSON line: wall times, the NB_BAM_STATS phases of each run's best repeat, store / metadata / row-buffer / peak
device bytes, peak RSS, rows_equal (the unbudgeted any-order rows decompress to the grouped run's bytes, and every budgeted
file holds the same lines: the same header and the same multiset of data lines by per-line CRC-32) and the card's name and
power limit read in the same call.  The metadata text bytes per record are M(r)'s bytes over the kept records of the
unbudgeted run (its NB_BAM_STATS "metadata text"); the metadata store bytes are the device arrays with their growth slack.
The unbudgeted peak is that run's device peak (every allocation of the store, grouping and row stage)."""
import argparse, concurrent.futures, json, os, re, shutil, subprocess, sys, tempfile, time, zlib
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import bench_bam_any_order as bo
import nimble_aligner_b200 as nb
import synth

ANY = dict(bo.ANY, rows=r", rows (\d+)", row_bytes=r"row bytes (\d+)", row_chunks=r"row chunks (\d+)", metadata_bytes=r"metadata (\d+) bytes", metadata_text_bytes=r"metadata text (\d+) bytes", device_peak_bytes=r"device peak (\d+) bytes",
           metadata_formatting=r"metadata formatting ([\d.]+)s", row_buffer_bytes=r"row buffer (\d+) bytes", device_row_build=r"device row build ([\d.]+)s",
           deflate_write=r"deflate\+write ([\d.]+)s", kept=r"(\d+) kept", passes=r"passes (\d+)", peak_device_bytes=r"peak device bytes (\d+)")
GROUPED = dict(bo.GROUPED, rows_gzip_write=r"rows\+gzip\+write ([\d.]+)s")


def digest(path):
    """one pass over a .gz file (any member layout): CRC-32 and length of the decompressed bytes, the header line, and an
    order-free digest of the data lines (count, sum and xor of per-line CRC-32s) for files that hold the same lines"""
    d = zlib.decompressobj(16 + zlib.MAX_WBITS); crc, n, rest, head, cnt, sm, xr = 0, 0, b"", None, 0, 0, 0
    with open(path, "rb") as f:
        while True:
            buf = f.read(1 << 24)
            if not buf:
                break
            while buf:
                out = d.decompress(buf); buf = d.unused_data
                if buf:
                    d = zlib.decompressobj(16 + zlib.MAX_WBITS)   # next gzip member
                crc = zlib.crc32(out, crc); n += len(out)
                parts = (rest + out).split(b"\n"); rest = parts.pop()
                if head is None and parts:
                    head = parts.pop(0)
                for p in parts:
                    c = zlib.crc32(p); cnt += 1; sm += c; xr ^= c
    return {"crc": crc, "bytes": n, "header": zlib.crc32(head or b""), "lines": (cnt, sm, xr)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--groups", type=int, default=5_000_000, help="UMI groups (about 4 records each)")
    ap.add_argument("--repeat", type=int, default=1)
    a = ap.parse_args()
    cores = os.cpu_count() or 1
    L = 91
    lib = synth.SynthLibrary(seed=1234, n_fam=200, n_all=5, group_on="", trim_target_length=40, trim_strictness=0.9)
    tmp = tempfile.mkdtemp(prefix="nb_bam_any_order_rows_")
    lib_path = os.path.join(tmp, "lib.json"); json.dump(lib.to_json_obj(), open(lib_path, "w"))
    u = synth.umi_reads(lib, 0, a.groups, seed=2345, threads=cores)
    n = u["n_reads"]
    umi = bo.sort_key(bo.tag_values(u["scope"], 0x9E3779B97F4A7C15), 12); cbk = bo.sort_key(bo.tag_values(u["cell"], 0xD1B54A32D192ED03), 16)
    perm = np.random.default_rng(99).permutation(n)       # the files of bench_bam_any_order.py
    order = perm[np.lexsort((cbk[perm], umi[perm]))]
    g = bo.with_order(u, order, L)
    sentinel = a.groups
    while bo.sort_key(bo.tag_values(np.array([sentinel], np.uint64), 0x9E3779B97F4A7C15), 12)[0] == umi[order[-1]]:
        sentinel += 1
    g["bases"] = np.concatenate([g["bases"][: n * L], g["bases"][n * L - L: n * L], np.zeros(64, np.uint8)])
    g["qual"] = np.concatenate([g["qual"][: n * L], g["qual"][n * L - L: n * L], np.zeros(64, np.uint8)])
    g["cell"] = np.append(g["cell"], np.uint32(0)); g["scope"] = np.append(g["scope"], np.uint32(sentinel)); g["n_reads"] = n + 1
    # G's records keep the names they have in the shuffled file (record perm[k] is named r<k> there): field 0 is in the rows
    pos = np.empty(n, np.uint64); pos[perm] = np.arange(n, dtype=np.uint64)
    names = np.append(pos[order], np.uint64(n))   # the sentinel: a name of its own
    grouped = os.path.join(tmp, "grouped.bam"); size_g = synth.write_umi_bam(grouped, g, threads=cores, name_ids=names); del g
    s = bo.with_order(u, perm, L)
    shuffled = os.path.join(tmp, "shuffled.bam"); size_s = synth.write_umi_bam(shuffled, s, threads=cores); del s, u
    exe = os.path.join(os.path.dirname(os.path.abspath(nb.__file__)), "nimble")
    env = dict(os.environ, NB_BAM_STATS="1")

    def run(name, path, extra, prefix, rx):
        out = os.path.join(tmp, name + ".tsv.gz")
        t = time.time()
        pr = subprocess.run([exe, "-r", lib_path, "-i", path, "-c", str(cores), "-o", out] + extra, check=True, stdout=subprocess.DEVNULL, stderr=subprocess.PIPE, text=True, env=env)
        dt = time.time() - t
        line = [l for l in pr.stderr.split("\n") if l.startswith(prefix)][-1]
        return round(dt, 3), {k: float(m.group(1)) for k, r in rx.items() for m in [re.search(r, line)] if m}, out

    best, walls, outs = {}, {}, {}
    def keep(name, dt, ph, out):
        walls.setdefault(name, []).append(dt); outs[name] = out
        if name not in best or dt < best[name]["seconds"]:
            best[name] = {"seconds": dt, "records_per_s": n / dt, "phases": ph}
    peak = None
    for _ in range(a.repeat):   # alternated: a drift of the machine touches every run alike
        keep("any_order", *run("any_order", shuffled, ["--any-order"], "nb_process_bam_any_order:", ANY))
        keep("grouped", *run("grouped", grouped, [], "nb_process_bam:", GROUPED))
        ph = best["any_order"]["phases"]
        peak = peak or int(ph["device_peak_bytes"])
        for div in (2, 4):
            keep("budget_1_%d" % div, *run("budget_1_%d" % div, shuffled, ["--any-order", "--device-budget", str(peak // div)], "nb_process_bam_any_order:", ANY))
    for k in best:
        best[k]["all_seconds"] = walls[k]
    with concurrent.futures.ProcessPoolExecutor(4) as ex:
        dg = dict(zip(outs, ex.map(digest, [outs[k] for k in outs])))
    equal = (dg["any_order"]["crc"], dg["any_order"]["bytes"]) == (dg["grouped"]["crc"], dg["grouped"]["bytes"])
    lines_equal = all((dg[k]["header"], dg[k]["lines"]) == (dg["any_order"]["header"], dg["any_order"]["lines"]) for k in ("budget_1_2", "budget_1_4"))
    ph = best["any_order"]["phases"]
    res = {"workload": "C3-shaped BAM: %d single-end 91 bp records in %d (UMI,CB) groups, 8000 cells, 1k-transcript library; G (sorted by UMI, CB, + 1 sentinel record) %.0f MB, shuffled %.0f MB; `nimble -o` rows" % (n, a.groups, size_g / 1e6, size_s / 1e6),
           "host_threads": cores, "repeat": a.repeat, "runs": best, "unbudgeted_peak_device_bytes": peak,
           "store_bytes": ph.get("store_bytes"), "metadata_store_bytes": ph.get("metadata_bytes"), "row_buffer_bytes": ph.get("row_buffer_bytes"),
           "metadata_text_bytes": ph.get("metadata_text_bytes"), "metadata_text_bytes_per_kept_record": round(ph["metadata_text_bytes"] / ph["kept"], 1) if ph.get("kept") else None,
           "peak_rss_mb": {k: best[k]["phases"].get("peak_rss_mb") for k in best},
           "rows_equal": equal, "budgeted_lines_equal": lines_equal, "decompressed_bytes": dg["any_order"]["bytes"],
           "speedup_any_order_vs_grouped": round(best["grouped"]["seconds"] / best["any_order"]["seconds"], 3), "card": bo.card()}
    print(json.dumps(res))
    shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
