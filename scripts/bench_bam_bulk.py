#!/usr/bin/env python
"""Bulk BAM mode against the FASTQ driver on the same C2-shaped pairs (150 bp, 1k-transcript library), in one call:
  fastq      `nimble -i r1.fastq r2.fastq` (plain text)
  fastq_gz   `nimble -i r1.fastq.gz r2.fastq.gz`
  bulk       `nimble --bulk -i x.bam`, the pairs as a BAM in shuffled record order (R2 stored REVERSE, as an aligner stores
             it; no cell barcodes)
alternated --repeat times.  Asserts that the three TSVs are equal, and prints one JSON line: wall times, the NB_BAM_STATS
phases of the best bulk run, the NB_FASTQ_STATS line of the best FASTQ runs, and the card's name and power limit read in
the same call."""
import argparse, json, multiprocessing, os, re, shutil, struct, subprocess, sys, tempfile, time, zlib
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import bench_bam_any_order as bo
import nimble_aligner_b200 as nb
import synth
from synth import bamio

BULK = dict(records=r"(\d+) records", kept=r"(\d+) kept", pairs=r"(\d+) pairs", batches=r"(\d+) batches", windows=r"windows \(read\+inflate\+stage\+upload\) ([\d.]+)s",
            upload_wait=r"upload wait ([\d.]+)s", key_sort_pairing=r"key\+sort\+pairing ([\d.]+)s", align_finalize=r"align\+finalize ([\d.]+)s",
            total=r"total ([\d.]+)s", store_bytes=r"store (\d+) bytes", peak_rss_mb=r"peak RSS (\d+) MB")
FASTQ = dict(parse_align=r"parse\+align ([\d.]+) s", finalize_tsv=r"finalize\+tsv ([\d.]+) s", reads_per_s=r"([\d.]+) M reads/s")

_CODE = np.zeros(256, np.uint8)
for _i, _c in enumerate("=ACMGRSVTWYHKDBN"):
    _CODE[ord(_c)] = _i
_COMP = np.arange(256, dtype=np.uint8)
for _a, _b in zip(b"ACGT", b"TGCA"):
    _COMP[_a] = _b


_PAIRS = None   # (r1, o1, r2, o2), inherited by the forked encoders


def _encode(ks):
    """records ks (2p = R1 of pair p, 2p + 1 = its R2) in this order -> BGZF blocks (60000 raw bytes each, the last one
    possibly shorter: the blocks of consecutive jobs concatenate into one stream)"""
    r1, o1, r2, o2 = _PAIRS
    out = bytearray()
    for k in ks:
        p, side = int(k) >> 1, int(k) & 1
        r, o = (r2, o2) if side else (r1, o1)
        s = r[int(o[p]):int(o[p + 1])]
        if side:
            s = _COMP[s[::-1]]                                     # R2 stored REVERSE
        c = _CODE[s]
        if len(c) & 1:
            c = np.append(c, 0)
        name = b"p%d\0" % p
        body = struct.pack("<iiBBHHHIiii", -1, -1, len(name), 255, 4680, 0, 0x1 | (0x90 if side else 0x40), len(s), -1, -1, 0)
        body += name + ((c[0::2] << 4) | c[1::2]).astype(np.uint8).tobytes() + b"\x28" * len(s)
        out += struct.pack("<I", len(body)) + body
    return b"".join(bamio._bgzf_block(bytes(out[i:i + 60000]), 1) for i in range(0, len(out), 60000))


def write_bam(path, pairs, n_pairs, seed, cores):
    global _PAIRS
    _PAIRS = pairs
    order = np.random.default_rng(seed).permutation(2 * n_pairs)
    text = b"@HD\tVN:1.6\tSO:unsorted\n"
    hdr = b"BAM\1" + struct.pack("<I", len(text)) + text + struct.pack("<I", 0)
    jobs = [order[i:i + 100000] for i in range(0, len(order), 100000)]
    with open(path, "wb") as f, multiprocessing.get_context("fork").Pool(cores) as pool:
        f.write(bamio._bgzf_block(hdr, 1))
        for blocks in pool.imap(_encode, jobs):
            f.write(blocks)
        f.write(bamio._bgzf_block(b"", 1))
    return os.path.getsize(path)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=2_000_000)
    ap.add_argument("--repeat", type=int, default=1)
    a = ap.parse_args()
    cores = os.cpu_count() or 1
    lib = synth.SynthLibrary(seed=1234, n_fam=200, n_all=5)
    tmp = tempfile.mkdtemp(prefix="nb_bam_bulk_")
    try:
        lib_path = os.path.join(tmp, "lib.json"); json.dump(lib.to_json_obj(), open(lib_path, "w"))
        r1, o1, r2, o2 = synth.pairs(lib, 0, a.pairs, threads=cores)
        files = {}
        for ext in ("fastq", "fastq.gz"):
            files[ext] = [os.path.join(tmp, "r%d.%s" % (m, ext)) for m in (1, 2)]
            synth.write_fastq(files[ext][0], r1, o1, 1); synth.write_fastq(files[ext][1], r2, o2, 2)
        bam = os.path.join(tmp, "shuffled.bam"); bam_size = write_bam(bam, (r1, o1, r2, o2), a.pairs, 99, cores); del r1, r2
        exe = os.path.join(os.path.dirname(os.path.abspath(nb.__file__)), "nimble")
        env = dict(os.environ, NB_BAM_STATS="1", NB_FASTQ_STATS="1")

        def run(name, inputs, extra, prefix, rx):
            out = os.path.join(tmp, name + ".tsv")
            if os.path.exists(out):
                os.remove(out)
            t = time.time()
            pr = subprocess.run([exe, "-r", lib_path, "-i"] + inputs + ["-c", str(cores), "-o", out] + extra, check=True, stdout=subprocess.DEVNULL, stderr=subprocess.PIPE, text=True, env=env)
            dt = time.time() - t
            line = [l for l in pr.stderr.split("\n") if l.startswith(prefix)][-1]
            return round(dt, 3), {k: float(m.group(1)) for k, r in rx.items() for m in [re.search(r, line)] if m}, open(out, "rb").read()

        best, walls, tsv = {}, {}, {}
        for _ in range(a.repeat):   # alternated: a drift of the machine touches every run alike
            for name, inputs, extra, prefix, rx in (("fastq", files["fastq"], [], "nb_process_fastq:", FASTQ), ("fastq_gz", files["fastq.gz"], [], "nb_process_fastq:", FASTQ),
                                                    ("bulk", [bam], ["--bulk"], "nb_process_bam_bulk:", BULK)):
                dt, ph, out = run(name, inputs, extra, prefix, rx)
                walls.setdefault(name, []).append(dt); tsv[name] = out
                if name not in best or dt < best[name]["seconds"]:
                    best[name] = {"seconds": dt, "pairs_per_s": a.pairs / dt, "phases": ph}
        assert tsv["bulk"] == tsv["fastq"] == tsv["fastq_gz"], "the TSVs differ"
        for k in best:
            best[k]["all_seconds"] = walls[k]
        res = {"workload": "C2-shaped: %d pairs of 150 bp, 1k-transcript library; BAM (shuffled, no CB) %.0f MB, FASTQ %.0f MB plain, %.0f MB gz" %
                           (a.pairs, bam_size / 1e6, sum(os.path.getsize(f) for f in files["fastq"]) / 1e6, sum(os.path.getsize(f) for f in files["fastq.gz"]) / 1e6),
               "host_threads": cores, "repeat": a.repeat, "runs": best, "tsv_equal": True,
               "speedup_bulk_vs_fastq_gz": round(best["fastq_gz"]["seconds"] / best["bulk"]["seconds"], 3),
               "speedup_bulk_vs_fastq": round(best["fastq"]["seconds"] / best["bulk"]["seconds"], 3), "card": bo.card()}
        print(json.dumps(res))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
