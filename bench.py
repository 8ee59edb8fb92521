#!/usr/bin/env python
"""bench.py — aligned reads/sec of the nimble-aligner hot path on B200 (BASELINE.json metric), with the GPU counts
checked against the CPU oracle inside the same run ("bit-exact counts vs CPU ref").

Top-level line = workload C2 (BASELINE.json configs[1]): synthetic 1k-transcript family library (200 families x 5
alleles, seed 1234) and 10 M 2x150 bp read pairs per GPU, FASTQ-mode semantics (one whole-run aggregation scope, counts
over unique read pairs).  A "step" is one complete pass of the hot path (pack -> seed-and-walk map -> pair/orientation
-> de-duplicate -> callset histogram -> counts on the host) over that input.

  value         reads/s with the ASCII reads already resident in HBM (device-timed, CUDA events on the launching stream)
  e2e           reads/s through the C ABI with pinned HOST buffers: H2D copies and the D2H of the counts inside the timed
                region; `of_h2d_ceiling` = the H2D rate it ran at / the box's measured pinned-copy ceiling
  roofline      map stage (k_seed + k_walk, the dominant kernels): algorithmic bytes per launch / mean launch time
                (CUDA events inside the library); C2's index is L2-resident, so the roof is the L2 record-gather
                bandwidth measured live on this GPU (nb_measure_gather); C4's is HBM (MEASURED_PEAKS.json)
  cpu_baseline  the CPU oracle with the reference's cost structure on a bounded sample, all host cores
  parity_checked  GPU counts == oracle counts on a prefix of the same seeded stream (asserted; the run fails otherwise)

Block `c5` (configs[4]: the mismatch-tolerance sweep on the C2 library and reads, with the count merge at N > 1): the points of
the sweep (num_mismatches 0 / 1 / 2) the top-level line does not cover, timed on the same device-resident inputs, each
with its own parity check (N = 1: counts and work counters == oracle on a prefix; N > 1: merged counts of a small sharded job
== oracle == one GPU over the union).
Blocks `c4` (configs[3] shape: library whose index is far larger than L2, single-end 150 bp, HBM-bound probes; N=1
only) and `c3` (configs[2] shape: 10x-style single-end 91 bp records with quals in (UMI, CB) scopes, MAXINFO trim,
dummy mates, per-cell count table; every N, scopes sharded over ranks) carry the same keys for their workloads.

`--impl reference` times the oracle (reference cost structure: string-keyed maps, linear unmap, per-read maxinfo tables)
with all host threads on C2 and, in its `c3` / `c4` blocks, on those workloads.
N > 1 (torchrun): reads shard over ranks, index replicated; key records are routed to their owning GPU inside k_pair
over NVLink and the count tables are merged with NCCL.  Weak scaling: 10 M pairs per GPU.  A verification pass (untimed)
checks the merged result of a small sharded job against the oracle and against one GPU over the union of the shards.
"""
import argparse
import ctypes as C
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "aligned reads/sec per box, bit-exact counts vs CPU ref"
UNIT = "reads/s"
SEED = 1234
READ_LEN = 150
DTYPE = "u8/u64 integer (f64 thresholds)"


def algorithmic_bytes_per_read(work, n_reads_total, read_len=READ_LEN):
    """DESIGN.md 'Roofline': bytes the map stage must touch per read = packed read words + 16 B per hash probe + 32 B
    node record and c_v/4 unitig bytes per visited unitig + 4 B per colour id touched + 32 B result record."""
    packed = 8 * ((read_len + 31) // 32)
    tot = packed * n_reads_total + 16 * work["probes"] + 32 * work["nodes"] + work["bases"] / 4.0 + 4 * work["colour_elems"] + 32 * n_reads_total
    return tot / n_reads_total


class ClockSampler:
    """Polls NVML (same counters as the nvidia-smi clocks line of B200_PROFILING.md) every ~2 ms from a thread, so that
    even a sub-second timed region gets samples DURING it."""
    REASONS = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40, "hw_power_brake": 0x80}

    def __init__(self, gpu_index):
        self.gpu, self.rows, self.stop_flag, self.thread, self.h = gpu_index, [], False, None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        except Exception:
            self.h = None

    def _poll(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.rows.append((time.time(), sm, rs))
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self.h is not None:
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()

    def stop(self, t0=None, t1=None):
        self.stop_flag = True
        if self.thread:
            self.thread.join(timeout=1.0)
        rows = [r for r in self.rows if (t0 is None or r[0] >= t0) and (t1 is None or r[0] <= t1)]
        mx = None
        try:
            mx = float(self.nv.nvmlDeviceGetMaxClockInfo(self.h, self.nv.NVML_CLOCK_SM))
        except Exception:
            pass
        reasons = set()
        for _, _, rs in rows:
            for name, bit in self.REASONS.items():
                if rs & bit:
                    reasons.add(name)
        return {"sm_mhz": float(np.median([r[1] for r in rows])) if rows else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(rows)}


# ---------------------------------------------------------------------------------------------- workloads
def c2_library(mismatches=0):
    import synth
    return synth.SynthLibrary(seed=SEED, n_fam=200, n_all=5, group_on="", num_mismatches=mismatches)


def c3_library():
    import synth
    return synth.SynthLibrary(seed=SEED, n_fam=200, n_all=5, group_on="", trim_target_length=40, trim_strictness=0.9)


def c4_library(families):
    import synth
    return synth.SynthLibrary(seed=3456, n_fam=families, n_all=5, group_on="")


def c3_prefix(u, m_records):
    """First whole (UMI, CB) scopes of a C3 shard covering about m_records records -> (n_records, scope_off uint64)."""
    ends = np.cumsum(u["sizes"].astype(np.int64))
    g = int(np.searchsorted(ends, m_records, side="left")) + 1
    g = min(g, len(ends))
    return int(ends[g - 1]), np.concatenate([[0], ends[:g]]).astype(np.uint64)


def c3_oracle_cells(ref, u, scope_off):
    """Oracle per-scope counts -> the per-cell table {(cell, callset): count} (sum over the cell's scopes)."""
    out = {}
    for si, rows in enumerate(ref["scopes"]):
        cell = int(u["cell"][int(scope_off[si])])
        for cs, c in rows:
            k = (cell, tuple(cs))
            out[k] = out.get(k, 0) + int(c)
    return out


# ---------------------------------------------------------------------------------------------- reference (CPU) arm
def run_reference(args):
    """CPU arm: the oracle with the reference's cost structure on bounded samples, all host threads (rank 0 only)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle as orc
    import synth
    cores = os.cpu_count() or 1
    L = c2_library(args.mismatches)
    ocfg, oref = orc.parse_reference_library(L.to_json_obj(), "unstranded")
    o = orc.Oracle(ocfg, oref, faithful_cost=True)
    n = args.ref_pairs
    r1, o1, r2, o2 = synth.pairs(L, 0, n, seed=SEED, threads=cores)
    for _ in range(args.warmup):
        o.run(r1, o1[:n // 8 + 1], r2, o2[:n // 8 + 1], threads=cores, shard_single=True, want_records=False)
    t0 = time.time()
    for _ in range(args.steps):
        o.run(r1, o1, r2, o2, threads=cores, shard_single=True, want_records=False)
    dt = (time.time() - t0) / args.steps
    v = 2 * n / dt
    sample = "%d of the 10M C2 pairs per step (pairs 0..%d of the same seeded stream), %d threads over contiguous shards" % (n, n, cores)
    out = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": DTYPE,
           "data": "synthetic", "config": {"workload": "C2: 1k-transcript family library x 2x150 bp pairs, FASTQ-mode scope", "sample_pairs": n, "num_mismatches": args.mismatches},
           "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
           "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    blocks = [b for b in args.blocks.split(",") if b]
    if "c3" in blocks:
        out["c3"] = cpu_c3(args, orc, synth, cores)
    if "c4" in blocks:
        out["c4"] = cpu_c4(args, orc, synth, cores, None)
    emit_json(out)


def cpu_c3(args, orc, synth, cores):
    L = c3_library()
    ocfg, oref = orc.parse_reference_library(L.to_json_obj(), "unstranded")
    o = orc.Oracle(ocfg, oref, faithful_cost=True)
    u = synth.umi_reads(L, 0, max(1, args.c3_ref_records // 4), seed=2345, threads=cores)
    m, scope_off = c3_prefix(u, args.c3_ref_records)
    ones, zeros = np.ones(m, dtype=np.uint8), np.zeros(m, dtype=np.uint8)
    t0 = time.time()
    o.run(u["bases"], u["off"][: m + 1], u["bases"], u["off"][: m + 1], q1=u["qual"], q2=u["qual"], skip1=ones, skip2=zeros, scope_off=scope_off, threads=cores, want_records=False)
    dt = time.time() - t0
    return {"value": m / dt, "unit": "reads/s", "cores": cores, "kind": "port",
            "sample": "%d records in %d (UMI,CB) scopes of the C3 stream, oracle with the reference's cost structure (per-read maxinfo tables), scopes over %d threads" % (m, len(scope_off) - 1, cores)}


def cpu_c4(args, orc, synth, cores, prebuilt):
    """prebuilt: (L, oracle) from the GPU arm's parity leg (the 40k-transcript oracle index takes most of a minute)."""
    if prebuilt is None:
        L = c4_library(args.c4_families)
        ocfg, oref = orc.parse_reference_library(L.to_json_obj(), "unstranded")
        o = orc.Oracle(ocfg, oref, faithful_cost=True)
    else:
        L, o = prebuilt
        o.faithful_cost = True
        o.set_config()
    m = args.c4_ref_reads
    r1, o1, _, _ = synth.pairs(L, 0, m, seed=3456, paired=False, threads=cores)
    t0 = time.time()
    o.run(r1, o1, threads=cores, shard_single=True, want_records=False)
    dt = time.time() - t0
    return {"value": m / dt, "unit": "reads/s", "cores": cores, "kind": "port",
            "sample": "%d single-end 150 bp reads of the C4 stream on the %d-transcript library, oracle with the reference's cost structure (linear unmap over %d rows), %d threads" % (m, 5 * L.n_fam, 10 * L.n_fam, cores)}


_JSON_OUT = None


def guard_stdout():
    """stdout carries exactly one JSON line: everything else that any library prints there (NCCL's version banner,
    torchrun notices of child ranks) is sent to stderr; emit_json writes to the saved descriptor."""
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit_json(obj):
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(obj) + "\n")
    out.flush()


def log(*a):
    print(*a, file=sys.stderr, flush=True)


DUMP_BYTES = 64 << 20


def dump_outputs(path, arrays):
    """Writes each array as <path>/<name>.npy in float64 (the counts and indices here are exact in it).  An array longer
    than its even share of DUMP_BYTES is cut to a sample at fixed, seeded positions, so runs with the same arguments stay
    comparable element for element."""
    os.makedirs(path, exist_ok=True)
    share = (DUMP_BYTES // max(1, len(arrays)) - 128) // 8   # elements per file; 128 bytes of .npy header each
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float64).reshape(-1)
        if a.size > share:
            a = a[np.sort(np.random.default_rng(SEED).choice(a.size, share, replace=False))]
        np.save(os.path.join(path, name + ".npy"), a)


# ---------------------------------------------------------------------------------------------- GPU arm helpers
class Env:
    pass


def timed(env, fn, steps):
    """K steps bracketed by barrier + synchronize on both sides; device time from CUDA events on the launching stream, max
    with the wall clock (a step ends with host work after its last kernel), max over ranks."""
    torch, dist = env.torch, env.dist
    if env.world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0 = time.time()
    e0.record()
    out = None
    for _ in range(steps):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    if env.world > 1:
        dist.barrier()
    ms = max(e0.elapsed_time(e1), 0.0)
    wall = (time.time() - w0) * 1e3
    ms = max(ms, wall)
    if env.world > 1:
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return ms / steps, out


def whole_counts(ctx, raw):
    d = ctx.decode_counts(raw)
    if "dense_counts" in raw:
        return {tuple(cs): int(c) for cs, c in zip(d["callsets"], raw["dense_counts"].tolist()) if c}
    return {tuple(cs): int(c) for _, cs, c in d["rows"]}


def hbm_peak():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (stream copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def static_traffic(key):
    """DRAM bytes per map-stage launch from the tracked ncu capture (profiles/k_map_traffic.json): a static figure from a
    profiler run of the same command, not something this un-profiled run can measure."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "k_map_traffic.json")))
        e = t.get(key)
        if isinstance(e, dict):
            return e.get("dram_bytes_per_launch"), "static, from profiles/%s" % e.get("source", "k_map_traffic.json")
        if key == "c2" and "dram_bytes_per_launch" in t:
            return t["dram_bytes_per_launch"], "static, from profiles/%s" % t.get("source", "k_map_traffic.json")
    except Exception:
        pass
    return None, None


def roofline(bound, peak, peak_src, bpr, ks, ms_step, steps, work, m_reads, traffic_key):
    launch_ms = ks["map_ms"] / max(1, ks["map_launches"])
    rpl = ks["map_reads"] / max(1, ks["map_launches"])
    achieved = bpr * rpl / (launch_ms / 1e3) / 1e9
    traffic, tsrc = static_traffic(traffic_key)
    return {"bound": bound, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_source": tsrc,
            "kernel": "map stage = k_seed + k_walk (one launch pair per chunk; CUDA events bracket the pair on the launching stream)", "peak_source": peak_src,
            "algorithmic_bytes_per_read": bpr, "reads_per_launch": rpl, "launch_ms": launch_ms, "kernel_share_of_step": ks["map_ms"] / (ms_step * steps),
            "work_per_read": {k: work[k] / float(m_reads) for k in ("probes", "nodes", "bases", "colour_elems")}}


# ---------------------------------------------------------------------------------------------- C4 block (N = 1)
def run_c4(env, args):
    nb, synth, torch = env.nb, env.synth, env.torch
    import oracle as orc
    cores = env.cores
    t0 = time.time()
    L = c4_library(args.c4_families)
    obj = L.to_json_obj()
    lib = nb.Library.from_text(json.dumps(obj), "unstranded")
    t1 = time.time()
    ix = nb.build_index(lib, cores, device=env.local_rank)   # K5: the CUDA index builder
    t2 = time.time()
    st = ix.stats()
    n = args.c4_reads
    o1 = np.zeros(n + 1, dtype=np.uint64)
    synth.lib().synth_pair_offsets(3456, 0, n, READ_LEN, 0.1, o1.ctypes.data, None, cores)
    h1 = torch.empty(int(o1[-1]) + 64, dtype=torch.uint8).pin_memory()
    synth.pairs(L, 0, n, seed=3456, paired=False, threads=cores, out=(h1.numpy(), None))
    ho1 = torch.from_numpy(o1.astype(np.int64)).pin_memory()
    d1, do1 = h1.cuda(), ho1.cuda()
    opts = dict(max_batch_pairs=args.chunk, callset_slots=1 << 22, agg_slots=1 << 23)
    ctx = nb.Context(ix, lib, device=env.local_rank, stream=env.stream, **opts)

    def step_device():
        ctx.reset()
        ctx.align_batch(d1, do1, n_pairs=n, max_read_len=READ_LEN, location=nb.NB_MEM_DEVICE)
        return ctx.counts_raw()

    def step_host():
        ctx.reset()
        b = nb.Batch(n, nb.NB_MEM_HOST, READ_LEN, h1.data_ptr(), ho1.data_ptr(), None, None, None, None, None, None, None, None)
        nb._ck(nb.lib().nb_align_batch(ctx.h, C.byref(b), None, None))
        return ctx.counts_raw()

    for _ in range(args.warmup):
        step_device()
    ctx.kernel_stats(reset=True)
    ms_dev, raw_dev = timed(env, step_device, args.steps)
    ks = ctx.kernel_stats(reset=True)
    step_host()
    ms_host, raw_host = timed(env, step_host, args.steps)
    cd, ch = whole_counts(ctx, raw_dev), whole_counts(ctx, raw_host)
    assert cd == ch, "C4: host-fed and device-resident runs disagree"
    h2d = int(o1[-1]) + 8 * (n + 1)
    out = {"workload": "C4-shaped: synthetic %d-transcript family library (%d x 5, seed 3456; %d k-mers, index %.0f MB on the device >> 126 MB L2) x %d single-end 150 bp reads, FASTQ-mode whole-run scope"
                       % (5 * args.c4_families, args.c4_families, st["n_kmers"], st["device_bytes"] / 1e6, n),
           "value": n / (ms_dev / 1e3), "unit": UNIT, "ms_per_step": ms_dev, "steps": args.steps, "warmup": args.warmup,
           "e2e": {"value": n / (ms_host / 1e3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 36 * len(cd) + 192, "ms_per_step": ms_host,
                   "h2d_gbs": h2d / (ms_host / 1e3) / 1e9, "of_h2d_ceiling": (h2d / (ms_host / 1e3) / 1e9) / env.h2d_ceiling if env.h2d_ceiling else None},
           "index_device_mb": st["device_bytes"] / 1e6, "library_parse_s": t1 - t0, "index_build_gpu_s": t2 - t1,
           "unique_read_keys": int(raw_dev["n_unique_keys"]), "callsets_counted": len(cd), "gpu_launches": ks["launches"]}
    if not args.no_cpu_baseline:
        # ---- parity: the oracle (own index, own walk) on a prefix of the same stream; its work counters feed the roofline
        m = min(args.parity_reads, n)
        t3 = time.time()
        ocfg, oref = orc.parse_reference_library(obj, "unstranded")
        o = orc.Oracle(ocfg, oref)
        t4 = time.time()
        ref = o.run(h1.numpy(), o1[: m + 1], threads=cores, want_records=False)
        pctx = nb.Context(ix, lib, device=env.local_rank, stream=env.stream, count_work=1, **opts)
        pctx.align_batch(h1.numpy(), o1[: m + 1], max_read_len=READ_LEN)
        got = sorted((tuple(cs), int(k)) for _, cs, k in pctx.counts()["rows"])
        want = sorted((tuple(cs), int(k)) for cs, k in ref["scopes"][0])
        assert got == want, "C4: GPU counts differ from the oracle's on the first %d reads" % m
        w = pctx.work_counters()
        assert all(w[k] == ref["work"][k] for k in ("probes", "nodes", "bases")), "C4: device work counters differ from the oracle's: %s vs %s" % (w, ref["work"])
        pctx.close()
        out["parity_checked"] = True
        out["parity"] = "GPU counts == oracle counts (%d callsets) and probe / unitig / base work counters equal on the first %d reads; oracle index build %.0f s" % (len(want), m, t4 - t3)
        bpr = algorithmic_bytes_per_read(ref["work"], m)
        peak, src = hbm_peak()
        out["roofline"] = roofline("hbm", peak, src, bpr, ks, ms_dev, args.steps, ref["work"], m, "c4")
        out["roofline"]["hbm_gather_roof_gbs"] = env.gather_hbm
        out["roofline"]["note"] = "index traffic is random 32-byte buckets / 64-byte walk records: the HBM record-gather roof measured on this GPU (nb_measure_gather, 2 GB table) is quoted beside the stream peak"
        out["cpu_baseline"] = cpu_c4(args, orc, synth, cores, (L, o))
    ctx.close()
    return out


# ---------------------------------------------------------------------------------------------- C3 block (every N)
def run_c3(env, args):
    nb, synth, torch, dist = env.nb, env.synth, env.torch, env.dist
    import oracle as orc
    cores, rank, world = env.cores, env.rank, env.world
    L = c3_library()
    obj = L.to_json_obj()
    lib = nb.Library.from_text(json.dumps(obj), "unstranded")
    ix = nb.build_index(lib, cores, device=env.local_rank)
    groups = args.c3_records // 4
    u = synth.umi_reads(L, rank * groups, groups, seed=2345, threads=cores)   # weak scaling: every rank takes its own run of (UMI, CB) groups
    n = u["n_reads"]
    n_cells = 8000
    pin = lambda x: torch.from_numpy(x).pin_memory()
    bases, qual, off = pin(u["bases"]), pin(u["qual"]), pin(u["off"].astype(np.int64))
    scope, cell = pin(u["scope"].astype(np.int32)), pin(u["cell"].astype(np.int32))
    f1, f2 = pin(np.full(n, nb.FLAG_SKIP_ALIGN, dtype=np.uint8)), pin(np.zeros(n, dtype=np.uint8))
    dv = [t.cuda() for t in (bases, qual, off, scope, cell, f1, f2)]
    ctx = nb.Context(ix, lib, device=env.local_rank, stream=env.stream, max_batch_pairs=args.chunk, agg_slots=1 << 24)
    # device-resident scoped batches must fit max_batch_pairs: cut at scope boundaries on the host
    cuts, sc = [0], u["scope"]
    while cuts[-1] < n:
        p1 = min(n, cuts[-1] + args.chunk)
        while p1 < n and p1 > cuts[-1] + 1 and sc[p1] == sc[p1 - 1]:
            p1 -= 1
        cuts.append(p1)
    if world > 1:
        from nimble_aligner_b200.multigpu import lib_comm
        lib_comm(ctx, nb, torch, dist, rank, world)

    def finish():
        # the row columns (5 M rows here) are read as views of the library's pinned buffer, as a C host would: they stay valid
        # until the next finalize, so every use below happens before the next step
        if world > 1:   # nb_merge_scoped_sharded: dictionaries all-gathered, per-cell tables summed by one dense reduce-scatter: every rank ends with (and reads back) the rows of its own range of cells
            return ctx.merge_scoped(n_cells, copy=False, sharded=True)
        return ctx.counts_raw(copy=False)

    def step_device():
        ctx.reset()
        db, dq, do, dsc, dce, df1, df2 = dv
        for a, b_ in zip(cuts[:-1], cuts[1:]):
            bt = nb.Batch(b_ - a, nb.NB_MEM_DEVICE, 91, db.data_ptr(), do.data_ptr() + 8 * a, db.data_ptr(), do.data_ptr() + 8 * a, dq.data_ptr(), dq.data_ptr(),
                          df1.data_ptr() + a, df2.data_ptr() + a, dsc.data_ptr() + 4 * a, dce.data_ptr() + 4 * a)
            nb._ck(nb.lib().nb_align_batch(ctx.h, C.byref(bt), None, None))
        return finish()

    def step_host():
        ctx.reset()
        bt = nb.Batch(n, nb.NB_MEM_HOST, 91, bases.data_ptr(), off.data_ptr(), bases.data_ptr(), off.data_ptr(), qual.data_ptr(), qual.data_ptr(),
                      f1.data_ptr(), f2.data_ptr(), scope.data_ptr(), cell.data_ptr())
        nb._ck(nb.lib().nb_align_batch(ctx.h, C.byref(bt), None, None))
        return finish()

    def table(raw):
        return (raw["row_scope"].astype(np.int64), raw["row_callset"].astype(np.int64), raw["row_count"].astype(np.int64))

    for _ in range(max(1, args.warmup - 1)):
        step_device()
    ctx.kernel_stats(reset=True)
    ms_dev, raw_dev = timed(env, step_device, args.steps)
    td = table(raw_dev)          # (copies: the views die with the next finalize)
    ks = ctx.kernel_stats(reset=True)
    step_host()
    ms_host, raw_host = timed(env, step_host, args.steps)
    th = table(raw_host)
    n_rows_job, n_pairs_job = int(len(td[0])), int(td[2].sum())
    if world > 1:   # the job's table is the union of the ranks' shards
        tt = torch.tensor([n_rows_job, n_pairs_job], device="cuda", dtype=torch.int64)
        dist.all_reduce(tt)
        n_rows_job, n_pairs_job = int(tt[0].item()), int(tt[1].item())
    if rank != 0:
        ctx.close()
        return None
    assert all(np.array_equal(a, b) for a, b in zip(td, th)), "C3: host-fed and device-resident runs disagree"
    total = n * world
    h2d = int(u["off"][-1]) * 2 + n * (8 + 4 + 4 + 2)
    out = {"workload": "C3-shaped: %d 10x-style single-end 91 bp records with raw Phred quals per GPU in %d (UMI,CB) scopes (dummy mates, MAXINFO trim 40:0.9), %d cells, 1k-transcript library; per-cell count table%s"
                       % (n, len(u["sizes"]), n_cells, (", scopes sharded over %d ranks and the tables merged by nb_merge_scoped_sharded (NCCL all-gather + dense reduce-scatter inside the library; every rank reads back its own range of cells)" % world) if world > 1 else ""),
           "value": total / (ms_dev / 1e3), "unit": UNIT, "ms_per_step": ms_dev, "steps": args.steps, "n_gpus": world, "records_per_step": total,
           "e2e": {"value": total / (ms_host / 1e3), "unit": UNIT, "h2d_bytes_per_step": h2d * world, "d2h_bytes_per_step": 16 * n_rows_job + 192 * world, "ms_per_step": ms_host,
                   "h2d_gbs": h2d * world / (ms_host / 1e3) / 1e9, "of_h2d_ceiling": (h2d / (ms_host / 1e3) / 1e9) / env.h2d_ceiling if env.h2d_ceiling else None},
           "count_rows": n_rows_job, "counted_pairs": n_pairs_job, "gpu_launches": ks["launches"],
           "k_map_ms_per_launch": ks["map_ms"] / max(1, ks["map_launches"]), "k_map_reads_per_launch": ks["map_reads"] / max(1, ks["map_launches"])}
    if not args.no_cpu_baseline:
        # ---- parity: per-cell table of the first scopes vs the oracle (string-level restatement of get_calls per scope)
        m, scope_off = c3_prefix(u, args.parity_reads)
        ocfg, oref = orc.parse_reference_library(obj, "unstranded")
        o = orc.Oracle(ocfg, oref)
        ones, zeros = np.ones(m, dtype=np.uint8), np.zeros(m, dtype=np.uint8)
        ref = o.run(u["bases"], u["off"][: m + 1], u["bases"], u["off"][: m + 1], q1=u["qual"], q2=u["qual"], skip1=ones, skip2=zeros, scope_off=scope_off, threads=cores, want_records=False)
        want = c3_oracle_cells(ref, u, scope_off)
        pctx = nb.Context(ix, lib, device=env.local_rank, stream=env.stream, max_batch_pairs=args.chunk, count_work=1)
        pctx.align_batch(u["bases"], u["off"][: m + 1], u["bases"], u["off"][: m + 1], q1=u["qual"], q2=u["qual"], flags1=f1.numpy()[:m], flags2=f2.numpy()[:m],
                         scope_id=u["scope"][:m], cell_id=u["cell"][:m], max_read_len=91)
        got = {(int(c), tuple(cs)): int(k) for c, cs, k in pctx.counts()["rows"]}
        assert got == want, "C3: GPU per-cell counts differ from the oracle's on the first %d records" % m
        w = pctx.work_counters()
        pctx.close()
        out["parity_checked"] = True
        out["parity"] = "GPU per-cell table == oracle (%d (cell, callset) rows) on the first %d records / %d scopes of rank 0's shard" % (len(want), m, len(scope_off) - 1)
        # the skipped dummy mates never reach the map stage's probe / walk work: bytes per MAPPED read, launches count both slots
        bpr = algorithmic_bytes_per_read(ref["work"], m, 91) + 91     # + the quality bytes k_trim streams
        out["roofline"] = roofline("l2", env.gather_l2, "measured live: nb_measure_gather over a 47 MB table at 32-byte records (L2-resident index)", bpr,
                                   dict(ks, map_reads=ks["map_reads"] / 2), ms_dev, args.steps, ref["work"], m, "c3")
        out["cpu_baseline"] = cpu_c3(args, orc, synth, cores)
    ctx.close()
    return out


def verify_sharded(env, args, job, counts_of, L, obj, lib, ix, n, mm=0):
    """N > 1 (untimed): a small sharded job through the same merge path must equal (a) the oracle over the union of the
    mini-shards and (b) one GPU over that union.  Every rank takes pairs [0, m) of ITS shard with its real global pair orders,
    so ownership, routing and "later duplicate wins" are exercised across ranks.  Returns the note (rank 0) or None."""
    nb, synth, rank, world, cores = env.nb, env.synth, env.rank, env.world, env.cores
    m = max(1000, args.parity_reads // world)
    mini, _u = job(m, False)
    mini = counts_of(mini)
    if rank != 0:
        return None
    import oracle as orc
    parts1, parts2, offs1, offs2 = [], [], [np.zeros(1, dtype=np.uint64)], [np.zeros(1, dtype=np.uint64)]
    for r in range(world):   # rank r's first m pairs = pairs [r*n, r*n + m) of the seeded stream
        a1, b1, a2, b2 = synth.pairs(L, r * n, m, seed=SEED, threads=cores)
        parts1.append(a1[: int(b1[-1])]); parts2.append(a2[: int(b2[-1])])
        offs1.append(b1[1:] + offs1[-1][-1]); offs2.append(b2[1:] + offs2[-1][-1])
    v1, v2 = np.concatenate(parts1 + [np.zeros(64, np.uint8)]), np.concatenate(parts2 + [np.zeros(64, np.uint8)])
    vo1, vo2 = np.concatenate(offs1).astype(np.uint64), np.concatenate(offs2).astype(np.uint64)
    ocfg, oref = orc.parse_reference_library(obj, "unstranded")
    ref = orc.Oracle(ocfg, oref).run(v1, vo1, v2, vo2, threads=cores, want_records=False)
    want = {tuple(cs): int(c) for cs, c in ref["scopes"][0]}
    vctx = nb.Context(ix, lib, device=env.local_rank, max_batch_pairs=args.chunk)
    vctx.align_batch(v1, vo1, v2, vo2, max_read_len=READ_LEN)
    one = {tuple(cs): int(c) for _, cs, c in vctx.counts()["rows"]}
    vctx.close()
    assert one == want, "single-GPU counts over the union of the mini-shards differ from the oracle's (num_mismatches %d)" % mm
    assert mini == want, "%d-GPU merged counts differ from the oracle's over the union of the mini-shards (num_mismatches %d)" % (world, mm)
    note = "%d-GPU merged counts == oracle == one GPU over the union of %d pairs per rank (%d callsets)" % (world, m, len(want))
    log("verify (num_mismatches %d): %s" % (mm, note))
    return note


# ---------------------------------------------------------------------------------------------- C5 block (every N)
def run_c5(env, args, sh):
    """BASELINE.json configs[4]: the mismatch-tolerance sweep on the C2 library and reads, with the count merge at N > 1.  The
    top-level line is one point of the sweep (--mismatches, default 0); this block adds the other two on the same inputs:
    device-resident jobs timed like the top level, and the same parity checks (N = 1: GPU counts and work counters == oracle on
    a prefix; N > 1: merged counts of a small sharded job == oracle == one GPU over the union)."""
    nb, synth, torch, dist, rank, world = env.nb, env.synth, env.torch, env.dist, env.rank, env.world
    from nimble_aligner_b200.multigpu import lib_comm
    n, out = sh["n"], {"workload": "C5: mismatch sweep on the C2 library and reads (same %d pairs per GPU per step, inputs resident in HBM)%s" % (sh["n"], ", merged by nb_merge_whole_run" if world > 1 else ""),
                       "unit": UNIT, "sweep": {}}
    for mm in (0, 1, 2):
        if mm == args.mismatches:
            continue
        L = c2_library(mm)
        obj = L.to_json_obj()
        lib = nb.Library.from_text(json.dumps(obj), "unstranded")
        ctx = nb.Context(sh["ix"], lib, device=env.local_rank, stream=env.stream, max_batch_pairs=args.chunk)
        if world > 1:
            lib_comm(ctx, nb, torch, dist, rank, world)
            try:
                ctx.route_setup((n + n // 2) // world + 4096, sh["pair_base"])
            except nb.NbError as e:
                ctx.close()
                out["skipped"] = "peer routing unavailable (%s)" % e
                return out

        def job(pairs, dev, ctx=ctx):
            ctx.reset()
            if dev:
                ctx.align_batch(sh["d1"], sh["do1"], sh["d2"], sh["do2"], n_pairs=pairs, max_read_len=READ_LEN, location=nb.NB_MEM_DEVICE)
            else:
                b = nb.Batch(pairs, nb.NB_MEM_HOST, READ_LEN, sh["h1"].data_ptr(), sh["ho1"].data_ptr(), sh["h2"].data_ptr(), sh["ho2"].data_ptr(), None, None, None, None, None, None)
                nb._ck(nb.lib().nb_align_batch(ctx.h, C.byref(b), None, None))
            raw = ctx.merge_whole_run() if world > 1 else ctx.counts_raw()
            return raw, raw["n_unique_keys"]
        for _ in range(2):
            job(n, True)
        ctx.kernel_stats(reset=True)
        ms, (raw, uniq) = timed(env, lambda: job(n, True), args.steps)
        ks = ctx.kernel_stats(reset=True)
        e = {"value": 2 * n * world / (ms / 1e3), "ms_per_step": ms, "unique_pair_keys": int(uniq), "k_map_ms_per_launch": ks["map_ms"] / max(1, ks["map_launches"])}
        if not args.no_cpu_baseline and not (world > 1 and args.no_verify):
            if world == 1:
                import oracle as orc
                ocfg, oref = orc.parse_reference_library(obj, "unstranded")
                mp = min(args.parity_reads, n)
                ref = orc.Oracle(ocfg, oref).run(sh["h1"].numpy(), sh["o1"][: mp + 1], sh["h2"].numpy(), sh["o2"][: mp + 1], threads=env.cores, want_records=False)
                want = {tuple(cs): int(c) for cs, c in ref["scopes"][0]}
                pctx = nb.Context(sh["ix"], lib, device=env.local_rank, stream=env.stream, max_batch_pairs=args.chunk, count_work=1)
                pctx.align_batch(sh["h1"].numpy(), sh["o1"][: mp + 1], sh["h2"].numpy(), sh["o2"][: mp + 1], max_read_len=READ_LEN)
                got = {tuple(cs): int(c) for _, cs, c in pctx.counts()["rows"]}
                assert got == want, "C5: GPU counts differ from the oracle's at num_mismatches %d" % mm
                w = pctx.work_counters()
                assert all(w[k] == ref["work"][k] for k in ("probes", "nodes", "bases")), "C5: device work counters differ from the oracle's at num_mismatches %d" % mm
                pctx.close()
                e["parity_checked"] = True
                e["parity"] = "GPU counts == oracle counts (%d callsets) and work counters equal on the first %d pairs" % (len(want), mp)
            else:
                note = verify_sharded(env, args, job, lambda r, ctx=ctx: whole_counts(ctx, r), L, obj, lib, sh["ix"], n, mm)
                if note:
                    e["parity_checked"] = True
                    e["parity"] = note
        ctx.close()
        out["sweep"]["mm%d" % mm] = e
    return out


# ---------------------------------------------------------------------------------------------- main (C2 + blocks)
def main():
    guard_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--pairs", type=int, default=10_000_000, help="read pairs per GPU per step (C2: 10M)")
    ap.add_argument("--ref-pairs", type=int, default=2_000_000, help="pairs per step of the CPU reference arm / cpu_baseline sample")
    ap.add_argument("--parity-reads", type=int, default=200_000, help="prefix (pairs for C2, reads / records for C4 / C3) on which GPU counts are asserted equal to the oracle's")
    ap.add_argument("--chunk", type=int, default=1 << 20)
    ap.add_argument("--blocks", default="c5,c3,c4", help="extra workload blocks in the JSON line (c5: the other points of the mismatch sweep; c4: N=1 only)")
    ap.add_argument("--c4-families", type=int, default=8000, help="C4 library: families x 5 alleles (8000 -> 40k transcripts, 1.9 GB index; 40000 = BASELINE's full 200k)")
    ap.add_argument("--c4-reads", type=int, default=8_000_000)
    ap.add_argument("--c4-ref-reads", type=int, default=400_000)
    ap.add_argument("--c3-records", type=int, default=20_000_000, help="C3 records per GPU per step (about; whole (UMI,CB) groups)")
    ap.add_argument("--c3-ref-records", type=int, default=2_000_000)
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the oracle legs (parity + cpu_baseline + roofline): kernel tuning runs only")
    ap.add_argument("--no-verify", action="store_true", help="N>1: skip the verification pass")
    ap.add_argument("--verify", action="store_true", help="N>1: ALSO check the full-size merged counts against one GPU over the union of all shards (slow)")
    ap.add_argument("--merge", default="lib", choices=["lib", "py-p2p", "py-nccl"], help="N>1: merge inside the library over NCCL with key records routed inside k_pair (default); py-*: round 1's host-driven choreography (routed / NCCL all-to-all)")
    ap.add_argument("--mismatches", type=int, default=0, help="num_mismatches of the library config (C5 sweeps 0/1/2)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the counts the top-level timed job returned in its "
                    "last step as DIR/<name>.npy (float64), to compare two builds on the same seeded inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the GPU arm computed (--impl b200)")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = max(args.warmup, 1)
    if args.impl == "reference":
        return run_reference(args)

    rank, world, local_rank = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
    numa_cpus = None
    if world > 1:   # one rank per GPU: keep each rank's pinned batches on its GPU's NUMA node (N=1 stays unbound: its cpu_baseline leg uses every core)
        from nimble_aligner_b200.multigpu import bind_to_gpu_numa_node
        numa_cpus = bind_to_gpu_numa_node(local_rank)
    import torch
    import torch.distributed as dist
    import nimble_aligner_b200 as nb
    import synth
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", "WARN"):
            os.environ.pop("NCCL_DEBUG")             # at these two levels NCCL prints its version banner on stdout
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    n = args.pairs
    cores = max(1, (os.cpu_count() or 1) // max(1, world))
    env = Env()
    env.nb, env.synth, env.torch, env.dist, env.rank, env.world, env.local_rank, env.cores = nb, synth, torch, dist, rank, world, local_rank, cores
    # ---- roofs of this box, measured live (diagnostics of the library, nothing on the data path): L2 / HBM record gather, H2D ceiling
    env.gather_l2 = nb.measure_gather(47 << 20, 32, device=local_rank)
    env.gather_hbm = nb.measure_gather(2 << 30, 32, device=local_rank) if world == 1 else None
    env.h2d_ceiling = nb.measure_h2d([local_rank], 256 << 20, 6)[1]
    blocks = [b for b in args.blocks.split(",") if b]
    L = c2_library(args.mismatches)
    obj = L.to_json_obj()
    lib = nb.Library.from_text(json.dumps(obj), "unstranded")
    t0 = time.time()
    ix = nb.build_index(lib, cores)
    index_build_s = time.time() - t0
    # one explicit CUDA stream shared by torch (events, NCCL ordering) and the library (kernels, D2H); the legacy default
    # stream has handle 0, which nb_ctx_create reads as "create your own"
    tstream = torch.cuda.Stream()
    torch.cuda.set_stream(tstream)
    stream = tstream.cuda_stream
    assert stream != 0
    env.stream = stream
    ctx = nb.Context(ix, lib, device=local_rank, stream=stream, max_batch_pairs=args.chunk)
    # ---- inputs: this rank's shard of the seeded stream, in pinned host memory and resident in HBM
    pair_base = rank * n
    o1 = np.zeros(n + 1, dtype=np.uint64); o2 = np.zeros(n + 1, dtype=np.uint64)
    synth.lib().synth_pair_offsets(SEED, pair_base, n, READ_LEN, 0.1, o1.ctypes.data, o2.ctypes.data, cores)
    h1 = torch.empty(int(o1[-1]) + 64, dtype=torch.uint8).pin_memory(); h2 = torch.empty(int(o2[-1]) + 64, dtype=torch.uint8).pin_memory()
    synth.pairs(L, pair_base, n, seed=SEED, threads=cores, out=(h1.numpy(), h2.numpy()))
    ho1, ho2 = torch.from_numpy(o1.astype(np.int64)).pin_memory(), torch.from_numpy(o2.astype(np.int64)).pin_memory()
    d1, d2, do1, do2 = h1.cuda(), h2.cuda(), ho1.cuda(), ho2.cuda()
    n_reads = 2 * n

    from nimble_aligner_b200.multigpu import merge_across_ranks, DeviceShard, setup_routes, lib_comm
    # N>1, default: the merge runs inside the library (nb_merge_whole_run: NCCL called from C++ on the context's stream, key
    # records routed inside k_pair over NVLink).  --merge py-p2p / py-nccl keep round 1's Python choreography for A/B.
    in_lib = routed = False
    if world > 1 and args.merge == "lib":
        lib_comm(ctx, nb, torch, dist, rank, world)
        try:
            ctx.route_setup((n + n // 2) // world + 4096, pair_base)
            in_lib = routed = True
        except nb.NbError as e:   # no NVLink / IPC between the processes: every rank fails together
            log("rank %d: in-library merge unavailable (%s); falling back to the NCCL all-to-all driven from the host" % (rank, e))
    if world > 1 and not in_lib:
        routed = args.merge != "py-nccl" and setup_routes(ctx, torch, dist, rank, world, "cuda", pair_base, (n + n // 2) // world + 4096)
    shard = DeviceShard(ctx, nb, torch, pair_base, n, routed=routed) if world > 1 and not in_lib else None   # merge buffers are allocated once, outside the job

    def job(pairs, dev):
        """one whole job over this rank's first `pairs` pairs: device-resident or host-fed input"""
        ctx.reset()
        if dev:
            ctx.align_batch(d1, do1, d2, do2, n_pairs=pairs, max_read_len=READ_LEN, location=nb.NB_MEM_DEVICE)
        else:
            b = nb.Batch(pairs, nb.NB_MEM_HOST, READ_LEN, h1.data_ptr(), ho1.data_ptr(), h2.data_ptr(), ho2.data_ptr(), None, None, None, None, None, None)
            nb._ck(nb.lib().nb_align_batch(ctx.h, C.byref(b), None, None))
        if in_lib:
            raw = ctx.merge_whole_run()  # nb_merge_whole_run: every rank ends with the whole job's counts
            return raw, raw["n_unique_keys"]
        if world > 1:
            return merge_across_ranks(shard, torch, dist, rank, world, "cuda", routed=routed)
        raw = ctx.counts_raw()          # nb_counts_finalize: the job's result (group indices + counts) on the host
        return raw, raw["n_unique_keys"]

    for _ in range(args.warmup):
        job(n, True)
    ctx.kernel_stats(reset=True)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    tw0 = time.time()
    ms_dev, (counts_dev, uniq_dev) = timed(env, lambda: job(n, True), args.steps)
    raw_dev = counts_dev
    tw1 = time.time()
    ks = ctx.kernel_stats(reset=True)
    clocks = sampler.stop(tw0, tw1) if rank == 0 else None
    job(n, False)
    ms_host, (counts_host, uniq_host) = timed(env, lambda: job(n, False), args.steps)
    # ---- the same job with the reads shipped 2-bit packed (NB_SEQ_2BIT: the boundary score::call really has — DnaStrings —
    # and a quarter of the PCIe bytes); packing happens outside the timed region, as a host that holds packed reads would have it
    p1 = torch.empty((int(o1[-1]) + 3) // 4 + 64, dtype=torch.uint8).pin_memory(); p2 = torch.empty((int(o2[-1]) + 3) // 4 + 64, dtype=torch.uint8).pin_memory()
    synth.encode_2bit(h1.numpy(), int(o1[-1]), p1.numpy(), cores); synth.encode_2bit(h2.numpy(), int(o2[-1]), p2.numpy(), cores)

    def job_packed():
        ctx.reset()
        b = nb.Batch(n, nb.NB_MEM_HOST, READ_LEN, p1.data_ptr(), ho1.data_ptr(), p2.data_ptr(), ho2.data_ptr(), None, None, None, None, None, None, nb.NB_SEQ_2BIT, 0, None, None)
        nb._ck(nb.lib().nb_align_batch(ctx.h, C.byref(b), None, None))
        if in_lib:
            raw = ctx.merge_whole_run()
            return raw, raw["n_unique_keys"]
        if world > 1:
            return merge_across_ranks(shard, torch, dist, rank, world, "cuda", routed=routed)
        raw = ctx.counts_raw()
        return raw, raw["n_unique_keys"]
    job_packed()
    ms_packed, (counts_packed, uniq_packed) = timed(env, job_packed, args.steps)
    counts_packed = whole_counts(ctx, counts_packed)
    counts_dev, counts_host = whole_counts(ctx, counts_dev), whole_counts(ctx, counts_host)
    assert counts_packed == counts_host and uniq_packed == uniq_host, "2-bit packed and ASCII host-fed runs disagree"
    if counts_host != counts_dev:
        diff = [(k, counts_dev.get(k), counts_host.get(k)) for k in set(counts_dev) | set(counts_host) if counts_dev.get(k) != counts_host.get(k)]
        log("rank %d: %d callsets differ (dev total %d, host total %d, %d vs %d callsets); e.g. %s" % (rank, len(diff), sum(counts_dev.values()), sum(counts_host.values()), len(counts_dev), len(counts_host), diff[:3]))
    assert counts_host == counts_dev, "host-fed and device-resident runs disagree"
    assert sum(counts_dev.values()) <= uniq_dev <= n * world, "count table inconsistent with the number of unique read_keys"

    # ---- verification pass at N>1 (untimed)
    verify_note = None
    if world > 1 and not args.no_verify:
        verify_note = verify_sharded(env, args, job, lambda r: whole_counts(ctx, r), L, obj, lib, ix, n, args.mismatches)
    if args.verify and world > 1 and rank == 0:
        # the merged multi-GPU counts must equal one GPU processing the union of all ranks' shards
        vo1 = np.zeros(n * world + 1, dtype=np.uint64); vo2 = np.zeros(n * world + 1, dtype=np.uint64)
        synth.lib().synth_pair_offsets(SEED, 0, n * world, READ_LEN, 0.1, vo1.ctypes.data, vo2.ctypes.data, cores)
        v1 = np.empty(int(vo1[-1]) + 64, dtype=np.uint8); v2 = np.empty(int(vo2[-1]) + 64, dtype=np.uint8)
        synth.pairs(L, 0, n * world, seed=SEED, threads=cores, out=(v1, v2))
        vctx = nb.Context(ix, lib, device=local_rank, max_batch_pairs=args.chunk)
        vctx.align_batch(v1, vo1, v2, vo2, max_read_len=READ_LEN)
        union = {tuple(cs): int(c) for _, cs, c in vctx.counts()["rows"]}
        vctx.close()
        assert union == counts_dev, "multi-GPU merge differs from the single-GPU result over the union of shards"
        log("verify: %d-GPU merged counts == single-GPU counts over the union (%d callsets)" % (world, len(union)))

    out = None
    if rank == 0:
        value = n_reads * world / (ms_dev / 1e3)
        e2e = n_reads * world / (ms_host / 1e3)
        h2d = int(o1[-1]) + int(o2[-1]) + 2 * 8 * (n + 1)
        d2h = 16 * len(counts_dev) + (2 + 16) * 4 * len(counts_dev) + 2 * 96   # compacted count rows + callset rows + counters read by nb_counts_finalize
        h2d_gbs = h2d / (ms_host / 1e3) / 1e9
        out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_dev,
               "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": DTYPE, "data": "synthetic",
               "config": {"workload": "C2: synthetic 1k-transcript family library (200x5, seed 1234) x %d 2x150 bp pairs per GPU, FASTQ-mode whole-run scope" % n,
                          "num_mismatches": args.mismatches, "merge": (("nb_merge_whole_run inside the library (NCCL from C++ on the context's stream; " if in_lib else "host-driven (") + ("k_pair stores key records into their owners' inboxes over NVLink)" if routed else "nccl all-to-all at job end)")) if world > 1 else "none (one GPU)",
                          "numa_bind": ("each rank bound to the %d CPUs local to its GPU" % numa_cpus) if numa_cpus else "none",
                          "pairs_per_gpu": n, "reads_per_step": n_reads * world, "chunk_pairs": args.chunk, "l2": "inputs (%.1f GB ASCII per step) exceed the 126 MB L2" % ((int(o1[-1]) + int(o2[-1])) / 1e9),
                          "index_device_mb": ix.stats()["device_bytes"] / 1e6, "index_build_s": index_build_s, "unique_pair_keys": int(uniq_dev), "callsets_counted": len(counts_dev)},
               "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": h2d * world, "d2h_bytes_per_step": d2h, "ms_per_step": ms_host, "h2d_gbs_per_gpu": h2d_gbs,
                       "h2d_ceiling_gbs_per_gpu": env.h2d_ceiling, "of_h2d_ceiling": h2d_gbs / env.h2d_ceiling if env.h2d_ceiling else None,
                       "encoding": "ASCII bases (1 byte per base), the reference's FASTQ boundary"},
               "e2e_packed": {"value": n_reads * world / (ms_packed / 1e3), "unit": UNIT, "ms_per_step": ms_packed, "encoding": "NB_SEQ_2BIT (2 bits per base, offsets in bases)",
                              "h2d_bytes_per_step": ((int(o1[-1]) + 3) // 4 + (int(o2[-1]) + 3) // 4 + 2 * 8 * (n + 1)) * world, "d2h_bytes_per_step": d2h,
                              "h2d_gbs_per_gpu": ((int(o1[-1]) + 3) // 4 + (int(o2[-1]) + 3) // 4 + 2 * 8 * (n + 1)) / (ms_packed / 1e3) / 1e9,
                              "parity": "counts and unique-key count identical to the ASCII host-fed run of the same step (asserted)"},
               "gpu_launches": ks["launches"], "clocks": clocks,
               "k_map_ms_per_launch": ks["map_ms"] / max(1, ks["map_launches"]), "k_map_reads_per_launch": ks["map_reads"] / max(1, ks["map_launches"]),
               "roofs_measured_live": {"l2_gather_gbs_47MB_rec32": env.gather_l2, "hbm_gather_gbs_2GB_rec32": env.gather_hbm, "h2d_pinned_gbs": env.h2d_ceiling}}
        if verify_note:
            out["parity_checked"] = True
            out["parity"] = verify_note
    # ---- cpu baseline + parity + roofline (rank 0, N=1 only)
    if world == 1 and not args.no_cpu_baseline:
        import oracle as orc
        ocfg, oref = orc.parse_reference_library(obj, "unstranded")
        # parity: oracle (single whole-run scope, like src/process/fastq.rs) vs the GPU on the first pairs of the same stream
        mp = min(args.parity_reads, n)
        ref = orc.Oracle(ocfg, oref).run(h1.numpy(), o1[: mp + 1], h2.numpy(), o2[: mp + 1], threads=cores, want_records=False)
        want = {tuple(cs): int(c) for cs, c in ref["scopes"][0]}
        pctx = nb.Context(ix, lib, device=local_rank, stream=stream, max_batch_pairs=args.chunk, count_work=1)
        pctx.align_batch(h1.numpy(), o1[: mp + 1], h2.numpy(), o2[: mp + 1], max_read_len=READ_LEN)
        got = {tuple(cs): int(c) for _, cs, c in pctx.counts()["rows"]}
        assert got == want, "C2: GPU counts differ from the oracle's on the first %d pairs" % mp
        w = pctx.work_counters()
        assert all(w[k] == ref["work"][k] for k in ("probes", "nodes", "bases")), "C2: device work counters differ from the oracle's: %s vs %s" % (w, ref["work"])
        pctx.close()
        out["parity_checked"] = True
        out["parity"] = "GPU counts == oracle counts (%d callsets) and probe / unitig / base work counters equal on the first %d pairs of the step's stream" % (len(want), mp)
        o = orc.Oracle(ocfg, oref, faithful_cost=True)
        m = min(args.ref_pairs, n)
        t0 = time.time()
        cref = o.run(h1.numpy(), o1[: m + 1], h2.numpy(), o2[: m + 1], threads=cores, shard_single=True, want_records=False)
        dt = time.time() - t0
        out["cpu_baseline"] = {"value": 2 * m / dt, "unit": UNIT, "cores": cores, "kind": "port",
                               "sample": "first %d of the step's %d pairs, oracle with the reference's cost structure, %d threads over contiguous shards" % (m, n, cores)}
        bpr = algorithmic_bytes_per_read(cref["work"], 2 * m)
        out["roofline"] = roofline("l2", env.gather_l2, "measured live: nb_measure_gather over a 47 MB table at 32-byte records (the index is L2-resident: %.0f MB)" % (ix.stats()["device_bytes"] / 1e6),
                                   bpr, ks, ms_dev, args.steps, cref["work"], 2 * m, "c2")
        hp, hsrc = hbm_peak()
        out["roofline"]["frac_of_hbm_stream_peak"] = out["roofline"]["achieved"] / hp
        out["roofline"]["hbm_stream_peak"] = hp
    c5 = None
    if "c5" in blocks:
        t0 = time.time()
        c5 = run_c5(env, args, dict(n=n, ix=ix, pair_base=pair_base, d1=d1, d2=d2, do1=do1, do2=do2, h1=h1, h2=h2, ho1=ho1, ho2=ho2, o1=o1, o2=o2))
        if rank == 0:
            c5["sweep"]["mm%d" % args.mismatches] = {"value": out["value"], "ms_per_step": out["ms_per_step"], "k_map_ms_per_launch": out["k_map_ms_per_launch"], "parity_checked": out.get("parity_checked", False), "note": "the top-level line"}
            c5["block_wall_s"] = time.time() - t0
            out["c5"] = c5
    ctx.close()
    del d1, d2, do1, do2, h1, h2, p1, p2
    torch.cuda.empty_cache()
    if "c4" in blocks and world == 1:
        t0 = time.time()
        c4 = run_c4(env, args)
        c4["block_wall_s"] = time.time() - t0
        out["c4"] = c4
    if "c3" in blocks:
        t0 = time.time()
        c3 = run_c3(env, args)
        if rank == 0:
            c3["block_wall_s"] = time.time() - t0
            out["c3"] = c3
    if rank == 0:
        if args.dump_outputs:
            # slot_to_callset maps dictionary slots (where colliding callsets land depends on the order threads insert them)
            # for per-pair records this job does not ask for; everything else is ordered by callset content
            dump_outputs(args.dump_outputs, {k: v for k, v in raw_dev.items() if k != "slot_to_callset"})
        emit_json(out)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
