"""Host side of the multi-GPU whole-run merge (SURVEY.md §8e): what a C++ host would do with NCCL between the C-ABI
calls, written once against a small shard interface so that the same choreography runs over NCCL with device shards
(bench.py) and over gloo with a host model of the tables (tests/test_multirank_cpu.py, world_size 2, no GPU).

Reads shard over ranks; counts are over unique read_keys of the whole run (src/align.rs:576-579, 685), so key records
must meet on one rank: every key has an owner (a slice of its 128-bit value mod world).  Four collectives:
  (1) all_gather of the per-rank sizes (callset rows, key records per owner),
  (2) all_gather of the callset dictionary rows, after which every rank holds the same dictionary,
  (3) one all_to_all of the key records {key_lo, key_hi, global pair order, callset tag}; each rank re-imports its
      partition with the "later duplicate wins" rule and folds it,
  (4) one all_reduce of the dense per-callset counts (+ the unique-key count in the last element).
With peer routing (setup_routes, nb_route_*) step (3) disappears: k_pair stores every record whose key another rank
owns into that rank's inbox over NVLink while the alignment runs, and each rank merges its inbox locally.

A shard provides:
  callsets_export() -> np.uint32 [k, cw] rows {slot, len, tag_lo, tag_hi, items[gcap]}
  keys_export_partitioned(world) -> (records int64 [n, 4] on the shard's device, grouped by owner; counts per owner)
  callsets_import(rows np.uint32 [m, cw]);  keys_import(records int64 [m, 4] on the device)
  recv_buffer(n) -> int64 [>= n, 4] on the device;  finalize() -> dict(callset_off, row_callset, row_count, n_unique_keys, ...)
"""
import ctypes as C
import os
import sys
import time

import numpy as np


def bind_to_gpu_numa_node(local_rank):
    """Restricts this process to the CPUs NVML reports as local to its GPU, before any pinned buffer is allocated, so that
    the pinned batches live on the GPU's own NUMA node (first touch) and H2D copies do not cross the socket link — with
    eight ranks feeding eight GPUs the host fabric, not PCIe, is the limit.  No-op on a single-node host, when NVML or
    the affinity call is unavailable, or with NB_NO_NUMA_BIND=1.  Returns the number of CPUs bound to, or None."""
    if os.environ.get("NB_NO_NUMA_BIND"):
        return None
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, ((os.cpu_count() or 1) + 63) // 64)
        cpus = {64 * i + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1}
        allowed = os.sched_getaffinity(0)
        cpus &= allowed
        if len(cpus) >= 2 and cpus != allowed:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception as e:   # no NVML, no permission, cpuset mismatch: stay unbound
        print("numa bind skipped: %s" % e, file=sys.stderr)
    return None


def lib_comm(ctx, nb, torch, dist, rank, world):
    """Gives the context its own NCCL communicator (nb_comm_init_rank): rank 0 creates the unique id through the library,
    the process group that launched the job carries it to the other ranks.  After this the merges run inside the library
    (nb_route_setup, nb_merge_whole_run, nb_merge_scoped); this module is only their caller."""
    uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
    if rank == 0:
        uid.copy_(torch.from_numpy(nb.comm_unique_id()))
    dist.broadcast(uid, 0)
    ctx.comm_init_rank(uid.cpu().numpy(), world, rank)


def setup_routes(ctx, torch, dist, rank, world, device, pair_base, records_per_peer):
    """Peer routing (nb_route_*, include/nimble_b200.h): every rank creates its inbox, the CUDA IPC handles travel by
    all_gather, every rank opens its peers' inboxes.  Returns False — on every rank — when any rank could not (no NVLink
    / IPC between the processes); the caller then keeps the exchange of merge_across_ranks(routed=False)."""
    handle = ctx.route_create(world, records_per_peer)
    allh = torch.empty((world, 64), dtype=torch.uint8, device=device)
    dist.all_gather_into_tensor(allh.view(-1), torch.from_numpy(handle.copy()).to(device))
    ok = 1
    try:
        ctx.route_attach_ipc(world, rank, allh.cpu().numpy(), pair_base)
    except RuntimeError as e:
        print("rank %d: peer routing unavailable (%s)" % (rank, e), file=sys.stderr)
        ok = 0
    flag = torch.tensor([ok], dtype=torch.int32, device=device)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if int(flag.item()) == 0:
        if ok:
            ctx.route_detach()
        return False
    return True


_ROUTED_CAP = [4096]   # rows per rank in the routed merge's dictionary block (grows by doubling, alike on every rank)


def merge_across_ranks(shard, torch, dist, rank, world, device, routed=False):
    """routed=True: the key records already travelled during the alignment (k_pair stored them into their owners' inboxes
    over NVLink); what is left is (1) sizes — also the barrier after which every peer's last batch is known to be done —
    (2) dictionaries, the local merge of the inbox (shard.route_import) and (4) the count all_reduce."""
    stats = os.environ.get("NB_MERGE_STATS") and rank == 0
    marks = []

    def mark(name):
        if stats:
            if device != "cpu":
                torch.cuda.synchronize()
            marks.append((name, time.time()))
    mark("start")
    rows = shard.callsets_export()
    k, cw = rows.shape
    mark("callsets_export")
    if not routed:
        rec, cnt = shard.keys_export_partitioned(world)
        mark("keys_export_partitioned")
    if routed:
        # (1)+(2) in one collective: a fixed-capacity block per rank {k, sent[world], rows[cap]}; the capacity is a ratchet
        # every rank raises alike (all ranks see all k) when a dictionary outgrows it.  The collective is also the barrier
        # after which every peer's last k_pair — and with it every record bound for this rank's inbox — is complete.
        sent = np.asarray(shard.route_sent(), dtype=np.int64)
        hdr = 1 + 2 * world          # k, then sent[] as (lo, hi) int32 halves
        cap = _ROUTED_CAP[0]
        while True:
            head = np.zeros(hdr, dtype=np.int32)
            head[0] = k
            head[1:] = sent.astype(np.int64).view(np.int32)
            blk = torch.zeros(hdr + cap * cw, dtype=torch.int32, device=device)
            body = np.ascontiguousarray(rows).view(np.int32).reshape(-1) if 0 < k <= cap else np.zeros(0, dtype=np.int32)
            blk[: hdr + body.size] = torch.from_numpy(np.concatenate([head, body])).to(device)
            allblk = torch.empty((world, hdr + cap * cw), dtype=torch.int32, device=device)
            dist.all_gather_into_tensor(allblk.view(-1), blk)
            on_dev = device != "cpu" and hasattr(shard, "callsets_import_device")
            hb = (allblk[:, :hdr].contiguous() if on_dev else allblk).cpu().numpy()   # device shards: only the headers come to the host
            szs = hb[:, 0].tolist()
            if max(szs) <= cap:
                break
            while cap < max(szs):
                cap *= 2
            # raised from this rank's own copy and stored once: ranks that share the module (threads of one process) all
            # read the same start value before the gather, so each computes, and stores, the same capacity
            _ROUTED_CAP[0] = cap
        recv = np.ascontiguousarray(hb[:, 1:hdr]).view(np.int64)[:, rank].copy()   # records rank r stored into this rank's inbox
        if on_dev:   # the peers' rows are imported straight out of the all_gather buffer in HBM
            for r in range(world):
                if r != rank and szs[r]:
                    shard.callsets_import_device(allblk[r, hdr:], int(szs[r]))
        else:
            parts = [hb[r, hdr:hdr + int(szs[r]) * cw].reshape(-1, cw) for r in range(world) if r != rank and szs[r]]
            others = (np.concatenate(parts) if parts else np.zeros((0, cw), dtype=np.int32)).view(np.uint32)
            shard.callsets_import(np.ascontiguousarray(others))
        mark("callsets_exchange_import")
    else:
        # (1) sizes
        meta = torch.from_numpy(np.concatenate([[k], np.asarray(cnt, dtype=np.int64)]).astype(np.int64)).to(device)
        allmeta = torch.empty((world, 1 + world), dtype=torch.int64, device=device)
        dist.all_gather_into_tensor(allmeta.view(-1), meta)
        am = allmeta.cpu().numpy()
        szs, recv_l, send_l = am[:, 0].tolist(), am[:, 1 + rank].tolist(), [int(x) for x in cnt]
        mark("sizes_all_gather")
        # (2) callset dictionaries
        kmax = max(max(szs), 1)
        mine = torch.zeros((kmax, cw), dtype=torch.int32, device=device)
        if k:
            mine[:k] = torch.from_numpy(np.ascontiguousarray(rows).view(np.int32)).to(device)
        allrows = torch.empty((world, kmax, cw), dtype=torch.int32, device=device)
        dist.all_gather_into_tensor(allrows.view(-1), mine.view(-1))
        others = torch.cat([allrows[r, : int(szs[r])] for r in range(world) if r != rank and szs[r]] or [allrows[0, :0]]).cpu().numpy().view(np.uint32)
        shard.callsets_import(np.ascontiguousarray(others))
        mark("callsets_exchange_import")
    if routed:
        shard.route_import(recv)
        mark("route_import")
    else:
        # (3) key records by owner; re-import this rank's partition and fold it (same stream as the collective: ordered after it)
        tot_recv, tot_send = int(sum(recv_l)), int(sum(send_l))
        out = shard.recv_buffer(tot_recv)
        dist.all_to_all_single(out[:tot_recv], rec[:tot_send], output_split_sizes=recv_l, input_split_sizes=send_l)
        mark("keys_all_to_all")
        shard.keys_import(out[:tot_recv])
        mark("keys_import")
    raw = shard.finalize()
    mark("finalize")
    # (4) dense all-reduce: after (2) every rank lists the same callsets in the same order; the last element carries the unique-key count
    ncs = len(raw["callset_off"]) - 1
    dense = torch.zeros(ncs + 1, dtype=torch.int64, device=device)
    dev = shard.device_rows() if device != "cpu" and hasattr(shard, "device_rows") else None
    if dev is not None:   # the rows of nb_counts_finalize are still on the device: no host round trip
        if dev[2].numel():
            dense.index_add_(0, dev[1].to(torch.int64), dev[2])
    elif len(raw["row_callset"]):
        dense.index_add_(0, torch.from_numpy(np.asarray(raw["row_callset"]).astype(np.int64)).to(device), torch.from_numpy(np.asarray(raw["row_count"], dtype=np.int64)).to(device))
    dense[ncs] = int(raw["n_unique_keys"])
    dist.all_reduce(dense)
    hd = dense.cpu().numpy()
    mark("dense_all_reduce")
    if stats:
        print("merge: " + ", ".join("%s %.2f ms" % (marks[i][0], (marks[i][1] - marks[i - 1][1]) * 1e3) for i in range(1, len(marks))), file=sys.stderr)
    raw = dict(raw)
    raw["dense_counts"] = hd[:ncs]
    return raw, int(hd[ncs])


def merge_scoped_across_ranks(shard, torch, dist, rank, world, device, n_cells):
    """BAM mode (SURVEY.md §8e): (UMI, CB) scopes are independent, so whole scopes shard over ranks with no data-path
    exchange; only the per-cell count table is combined.  (1) all_gather of the callset dictionary rows so every rank
    numbers callsets alike, (2) dense [n_cells x n_callsets] all_reduce when that is small, else all_gather of the sparse
    (cell, callset, count) rows which every rank sums.  Returns (cells, callsets, counts) int64 arrays, sorted by (cell, callset)."""
    stats = os.environ.get("NB_MERGE_STATS") and rank == 0
    marks = []

    def mark(name):
        if stats:
            if device != "cpu":
                torch.cuda.synchronize()
            marks.append((name, time.time()))
    mark("start")
    rows = shard.callsets_export()
    k, cw = rows.shape
    mark("callsets_export")
    sizes = torch.zeros(world, dtype=torch.int64, device=device)
    sizes[rank] = k
    dist.all_reduce(sizes)
    szs = sizes.cpu().tolist()
    kmax = max(max(szs), 1)
    mine = torch.zeros((kmax, cw), dtype=torch.int32, device=device)
    if k:
        mine[:k] = torch.from_numpy(np.ascontiguousarray(rows).view(np.int32)).to(device)
    allrows = torch.empty((world, kmax, cw), dtype=torch.int32, device=device)
    dist.all_gather_into_tensor(allrows.view(-1), mine.view(-1))
    others = torch.cat([allrows[r, : int(szs[r])] for r in range(world) if r != rank and szs[r]] or [allrows[0, :0]]).cpu().numpy().view(np.uint32)
    shard.callsets_import(np.ascontiguousarray(others))
    mark("callsets_exchange_import")
    raw = shard.finalize()
    mark("finalize")
    ncs = len(raw["callset_off"]) - 1
    if n_cells * max(ncs, 1) <= (1 << 25):
        dense = torch.zeros(n_cells * max(ncs, 1), dtype=torch.int64, device=device)
        dev = shard.device_rows() if hasattr(shard, "device_rows") else None
        if dev is not None:   # rows are still on the device: no host round trip
            dcell, dcs, dcnt = dev
            if dcnt.numel():
                dense.index_add_(0, dcell.to(torch.int64) * ncs + dcs.to(torch.int64), dcnt)
        elif len(raw["row_count"]):
            cell = np.asarray(raw["row_scope"], dtype=np.int64); cs = np.asarray(raw["row_callset"], dtype=np.int64)
            dense.index_add_(0, torch.from_numpy(cell * ncs + cs).to(device), torch.from_numpy(np.asarray(raw["row_count"], dtype=np.int64)).to(device))
        mark("dense_fill")
        dist.all_reduce(dense)
        mark("all_reduce")
        if rank != 0:
            z = np.zeros(0, dtype=np.int64)
            return raw, z, z, z          # the job's table is read back on rank 0 only
        nz = torch.nonzero(dense).view(-1)
        tri = torch.stack([nz // max(ncs, 1), nz % max(ncs, 1), dense[nz]])
        if device == "cpu":
            out = tri.numpy()
        else:   # the merged table lands in pinned memory: one DMA instead of a pageable copy of ~200 MB
            k = tri.shape[1]
            if getattr(shard, "pin", None) is None or shard.pin.numel() < 3 * k:
                shard.pin = torch.empty(3 * (k + k // 4 + 1), dtype=torch.int64, pin_memory=True)
            shard.pin[: 3 * k].copy_(tri.reshape(-1), non_blocking=True)   # contiguous on both sides: one DMA
            torch.cuda.current_stream().synchronize()
            out = shard.pin[: 3 * k].view(3, k).numpy()
        mark("readback")
        if stats:
            print("scoped merge: " + ", ".join("%s %.2f ms" % (marks[i][0], (marks[i][1] - marks[i - 1][1]) * 1e3) for i in range(1, len(marks))), file=sys.stderr)
        return raw, out[0], out[1], out[2]
    dev = shard.device_rows() if device != "cpu" and hasattr(shard, "device_rows") else None
    if dev is not None:   # a device shard's finalize returns no host rows: they are still on the device
        mine = torch.stack([dev[0].to(torch.int64), dev[1].to(torch.int64), dev[2]], dim=1)
    else:
        cell = np.asarray(raw["row_scope"], dtype=np.int64); cs = np.asarray(raw["row_callset"], dtype=np.int64); cnt = np.asarray(raw["row_count"], dtype=np.int64)
        mine = torch.from_numpy(np.stack([cell, cs, cnt], axis=1)).to(device)
    n = torch.zeros(world, dtype=torch.int64, device=device)
    n[rank] = mine.shape[0]
    dist.all_reduce(n)
    ns = n.cpu().tolist(); nmax = max(max(ns), 1)
    tri = torch.zeros((nmax, 3), dtype=torch.int64, device=device)
    if mine.shape[0]:
        tri[: mine.shape[0]] = mine
    alltri = torch.empty((world, nmax, 3), dtype=torch.int64, device=device)
    dist.all_gather_into_tensor(alltri.view(-1), tri.view(-1))
    t = torch.cat([alltri[r, : int(ns[r])] for r in range(world)]).cpu().numpy()
    key = t[:, 0] * max(ncs, 1) + t[:, 1]
    uk, inv = np.unique(key, return_inverse=True)
    val = np.bincount(inv, weights=t[:, 2]).astype(np.int64) if len(uk) else np.zeros(0, dtype=np.int64)
    return raw, uk // max(ncs, 1), uk % max(ncs, 1), val


class DeviceShard:
    """One GPU's tables behind the C ABI (nb_callsets_export / nb_keys_export_partitioned / nb_callsets_import /
    nb_keys_import / nb_counts_finalize).  Buffers are allocated once: unique keys <= pairs aligned on this rank."""

    def __init__(self, ctx, nb, torch, pair_base, max_pairs, routed=False):
        self.ctx, self.nb, self.torch, self.pair_base = ctx, nb, torch, pair_base
        if routed:
            max_pairs = 0   # no export / receive buffers: the records travel inside k_pair
        self.scoped = max_pairs == 0 and not routed   # scoped (BAM) merges reduce the rows on the device
        self.pin = None
        self.rows = None
        self.rec = torch.empty((max_pairs, 4), dtype=torch.int64, device="cuda") if max_pairs else None   # (scoped merges exchange no key records)
        self.out = torch.empty((max_pairs + max_pairs // 4, 4), dtype=torch.int64, device="cuda") if max_pairs else None

    def callsets_export(self):
        nout, gcap = C.c_uint64(0), C.c_uint32(0)
        if self.rows is None:   # row width is known once the tables exist (after the first batch)
            self.nb._ck(self.nb.lib().nb_callsets_export(self.ctx.h, None, 0, C.byref(nout), C.byref(gcap)))
            self.rows = np.zeros((1 << 18, 4 + gcap.value), dtype=np.uint32)          # callset_slots default: the dictionary cannot hold more
        self.nb._ck(self.nb.lib().nb_callsets_export(self.ctx.h, self.rows.ctypes.data, self.rows.shape[0], C.byref(nout), C.byref(gcap)))
        return self.rows[: nout.value]

    def keys_export_partitioned(self, world):
        cnt = np.zeros(world, dtype=np.uint64)
        self.nb._ck(self.nb.lib().nb_keys_export_partitioned(self.ctx.h, self.rec.data_ptr(), self.rec.shape[0], self.pair_base, world, cnt.ctypes.data))
        return self.rec, cnt.astype(np.int64).tolist()

    def callsets_import(self, rows):
        self.nb._ck(self.nb.lib().nb_callsets_import(self.ctx.h, rows.ctypes.data, rows.shape[0]))

    def callsets_import_device(self, rows, n):
        self.nb._ck(self.nb.lib().nb_callsets_import_device(self.ctx.h, rows.data_ptr(), n))

    def recv_buffer(self, n):
        if n > self.out.shape[0]:
            self.out = self.torch.empty((n + n // 4, 4), dtype=self.torch.int64, device="cuda")
        return self.out

    def keys_import(self, rec):
        self.nb._ck(self.nb.lib().nb_keys_import(self.ctx.h, rec.data_ptr(), rec.shape[0]))

    def route_sent(self):
        return self.ctx.route_sent()

    def route_import(self, counts):
        return self.ctx.route_import(counts)

    def finalize(self):
        return self.ctx.counts_raw(rows=not self.scoped)

    def device_rows(self):
        a, b, c, n = self.ctx.counts_device_rows()
        if not n:
            z = self.torch.zeros(0, dtype=self.torch.int64, device="cuda")
            return z, z, z
        t = self.torch
        return t.as_tensor(a, device="cuda").view(t.int32), t.as_tensor(b, device="cuda").view(t.int32), t.as_tensor(c, device="cuda")
