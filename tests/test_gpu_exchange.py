"""Host-driven exchange between ranks on the real kernels, on one GPU: the key-record export (nb_keys_export,
nb_keys_export_partitioned), the imports (nb_keys_import, nb_callsets_import, nb_callsets_import_device) and the two
merges of multigpu.py (merge_across_ranks with DeviceShard, routed and not, and merge_scoped_across_ranks).  This is what
bench.py --merge py-p2p|py-nccl runs, and the fallback when peer routes cannot be opened.  Every "rank" is a context on
device 0 driven by its own thread; a small in-process stand-in replaces torch.distributed.  Expectations come from the
CPU oracle's per-pair records, never from the device hash: the unique insertable read_keys (R1 + R2 bases,
src/align.rs:576-579), the last insertable pair of each (src/align.rs:685) and that pair's callset."""
import ctypes as C
import functools
import json
import threading

import numpy as np
import pytest
import torch

import nimble_aligner_b200 as nb
import nimble_aligner_b200.multigpu as mg
import oracle as orc
import synth

pytestmark = pytest.mark.gpu

N = 20_000                                 # pairs per job
WORLDS = (1, 2, 3, 7, 16, 33, 64)          # nb_keys_export_partitioned accepts 1..64 ranks
BASES = (0, 123_456_789, 1 << 39)          # pair_index_base: the orders of a rank whose pairs start there


# ------------------------------------------------------------------ in-process collectives
class _Shared:
    def __init__(self, world):
        self.world = world
        self.bar = threading.Barrier(world, timeout=120)
        self.slot = [None] * world


class _Dist:
    """The torch.distributed calls multigpu.py makes, for rank threads of one process on one GPU.  Each operation:
    every rank posts its input, barrier, copies on the device, torch.cuda.synchronize(), barrier.  The synchronize
    stands in for NCCL's stream ordering: the contexts run on streams of their own and must see the received buffers,
    and no rank may overwrite an input before every rank has read it."""

    class ReduceOp:
        SUM, MIN = "sum", "min"

    def __init__(self, shared, rank):
        self.s, self.rank, self.world = shared, rank, shared.world

    def _post(self, item):
        torch.cuda.synchronize()            # inputs written on any stream (a context's included) are complete
        self.s.slot[self.rank] = item
        self.s.bar.wait()
        return list(self.s.slot)

    def _done(self):
        torch.cuda.synchronize()
        self.s.bar.wait()

    def all_gather_into_tensor(self, out, inp):
        ins = self._post(inp)
        chunks = out.view(self.world, -1)
        for r, t in enumerate(ins):
            chunks[r].copy_(t.reshape(-1))
        self._done()

    def all_to_all_single(self, out, inp, output_split_sizes, input_split_sizes):
        ins = self._post((inp, [int(x) for x in input_split_sizes]))
        at = 0
        for r, (t, splits) in enumerate(ins):
            lo, n = sum(splits[:self.rank]), splits[self.rank]
            assert n == int(output_split_sizes[r]), (r, n, output_split_sizes)
            out[at:at + n].copy_(t[lo:lo + n])
            at += n
        self._done()

    def all_reduce(self, t, op=ReduceOp.SUM):
        ins = self._post(t)
        stack = torch.empty((self.world,) + tuple(t.shape), dtype=t.dtype, device=t.device)
        for r, x in enumerate(ins):
            stack[r].copy_(x)
        self._done()                        # every rank has read every input: now they may be overwritten
        t.copy_(stack.sum(0) if op == self.ReduceOp.SUM else stack.amin(0))
        torch.cuda.synchronize()


def _run_ranks(world, fn):
    """fn(rank, dist) on `world` threads; the first real error is raised (a failing rank breaks the barrier so that the
    others stop instead of waiting)."""
    shared = _Shared(world)
    out, err = [None] * world, [None] * world

    def run(r):
        try:
            out[r] = fn(r, _Dist(shared, r))
        except BaseException as e:   # noqa: BLE001 - re-raised below
            err[r] = e
            shared.bar.abort()
    th = [threading.Thread(target=run, args=(r,)) for r in range(world)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    real = [e for e in err if e is not None and not isinstance(e, threading.BrokenBarrierError)]
    if real or any(err):
        raise (real or [e for e in err if e is not None])[0]
    return out


def test_collective_stand_in_moves_and_reduces_tensors():
    world = 3

    def rank(r, dist):
        g = torch.empty(world * 2, dtype=torch.int64, device="cuda")
        dist.all_gather_into_tensor(g, torch.tensor([10 * r, 10 * r + 1], device="cuda"))
        send = [r + q for q in range(world)]                 # rank r sends r + q rows to rank q
        inp = torch.cat([torch.full((send[q], 2), 100 * r + q, dtype=torch.int64, device="cuda") for q in range(world)])
        recv = [q + r for q in range(world)]
        out = torch.full((sum(recv) + 3, 2), -1, dtype=torch.int64, device="cuda")
        dist.all_to_all_single(out[:sum(recv)], inp, output_split_sizes=recv, input_split_sizes=send)
        s = torch.tensor([r + 1, -r], dtype=torch.int64, device="cuda")
        m = s.clone()
        dist.all_reduce(s)
        dist.all_reduce(m, op=dist.ReduceOp.MIN)
        return g.cpu().tolist(), out.cpu().tolist(), s.cpu().tolist(), m.cpu().tolist()
    for r, (g, out, s, m) in enumerate(_run_ranks(world, rank)):
        assert g == [0, 1, 10, 11, 20, 21]
        want = [[100 * q + r] * 2 for q in range(world) for _ in range(q + r)]
        assert out == want + [[-1, -1]] * 3
        assert s == [6, -3] and m == [1, -2]


# ------------------------------------------------------------------ inputs and the host reference
_ACGT = np.full(256, ord("A"), dtype=np.uint8)     # nb_batch: ACGT either case, anything else -> A
for _b in b"ACGT":
    _ACGT[_b] = _ACGT[_b + 32] = _b


class _Job:
    pass


@functools.lru_cache(maxsize=None)
def _job(mm):
    J = _Job()
    # at most 2 groups per call: ~6% of the insertable pairs end in MaxHitsExceeded, so their records carry no callset (tag 0)
    J.L = synth.SynthLibrary(seed=2468, n_fam=40, n_all=5, group_on="", num_mismatches=mm, max_hits_to_report=2)
    obj = J.L.to_json_obj()
    J.lib = nb.Library.from_text(json.dumps(obj), "unstranded")
    J.ix = nb.build_index(J.lib, 8)
    J.names = J.lib.group_names()
    J.data = synth.pairs(J.L, 0, N, seed=31, dup_rate=0.3)
    ocfg, oref = orc.parse_reference_library(obj, "unstranded")
    J.ref = orc.Oracle(ocfg, oref).run(*J.data, threads=8)
    J.want = {tuple(cs): int(c) for cs, c in J.ref["scopes"][0]}
    r1, o1, r2, o2 = J.data
    a1, a2, o1, o2 = _ACGT[r1], _ACGT[r2], o1.astype(np.int64), o2.astype(np.int64)
    ref = J.ref
    ins = (ref["read_pass"][0::2] | ref["read_pass"][1::2]).astype(bool) & (ref["pair_fr1"] != orc.R["NotMatchingPair"])
    J.insertable = np.flatnonzero(ins)
    J.key = {p: a1[o1[p]:o1[p + 1]].tobytes() + a2[o2[p]:o2[p + 1]].tobytes() for p in J.insertable.tolist()}
    rows = ref["scopes"][0]
    # every pair of a key reports that key's callset (oracle.cpp per-pair projection)
    J.callset = {p: (tuple(rows[ref["pair_callset"][p]][0]) if ref["pair_counted"][p] else None) for p in J.key}
    one = nb.Context(J.ix, J.lib)
    one.align_batch(*J.data, max_read_len=150)
    d = one.counts()
    J.single = {tuple(cs): int(k) for _, cs, k in d["rows"]}
    J.single_unique = d["n_unique_keys"]
    one.close()
    assert J.single == J.want and len(J.want) > 50
    return J


def _expect(J, lo, hi):
    """Pairs [lo, hi) of the job: {index of the last insertable pair of each unique key, relative to lo: callset or None}."""
    last = {}
    for p in J.insertable[(J.insertable >= lo) & (J.insertable < hi)].tolist():
        last[J.key[p]] = p
    return {p - lo: J.callset[p] for p in last.values()}


def _part(data, lo, hi):
    r1, o1, r2, o2 = data
    out = []
    for r, o in ((r1, o1), (r2, o2)):
        out += [np.concatenate([r[int(o[lo]):int(o[hi])], np.zeros(64, dtype=np.uint8)]), (o[lo:hi + 1] - o[lo]).astype(np.uint64)]
    return out


def _ctx(J, lo=0, hi=None, **opts):
    c = nb.Context(J.ix, J.lib, **opts)
    hi = N if hi is None else hi
    pairs = None
    if hi > lo:
        _, pairs = c.align_batch(*_part(J.data, lo, hi), max_read_len=150, want_pairs=True)
    return c, pairs


# ------------------------------------------------------------------ C-ABI wrappers
def _export_count(ctx):
    n = C.c_uint64(0)
    nb._ck(nb.lib().nb_keys_export_count(ctx.h, C.byref(n)))
    return n.value


def _export_dev(ctx, base=0):
    n = _export_count(ctx)
    buf = torch.zeros((n + 1, 4), dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()                # the contexts run on streams of their own: the fill must land first
    nb._ck(nb.lib().nb_keys_export(ctx.h, buf.data_ptr(), n, base))
    return buf[:n]


def _host(rec):
    return rec.cpu().numpy().view(np.uint64)


def _export_partitioned(ctx, world, base=0):
    n = _export_count(ctx)
    # room for twice the records: a kernel that groups records wrongly scatters them out of place, not out of bounds
    buf = torch.zeros((2 * n + 1, 4), dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    cnt = np.zeros(world, dtype=np.uint64)
    nb._ck(nb.lib().nb_keys_export_partitioned(ctx.h, buf.data_ptr(), buf.shape[0], base, world, cnt.ctypes.data))
    cnt = cnt.astype(np.int64)
    return _host(buf[:int(cnt.sum())]), cnt


def _callset_rows(ctx):
    nout, gcap = C.c_uint64(0), C.c_uint32(0)
    nb._ck(nb.lib().nb_callsets_export(ctx.h, None, 0, C.byref(nout), C.byref(gcap)))
    rows = np.zeros((max(1, nout.value), 4 + gcap.value), dtype=np.uint32)
    nb._ck(nb.lib().nb_callsets_export(ctx.h, rows.ctypes.data, rows.shape[0], C.byref(nout), C.byref(gcap)))
    return rows[: nout.value]


def _dictionary(rows, names):
    """tag -> tuple of group names."""
    return {int(r[2]) | (int(r[3]) << 32): tuple(names[g] for g in r[4:4 + int(r[1])]) for r in rows}


def _callsets_import(ctx, rows):
    rows = np.ascontiguousarray(rows)
    nb._ck(nb.lib().nb_callsets_import(ctx.h, rows.ctypes.data, rows.shape[0]))


def _keys_import(ctx, rec):
    torch.cuda.synchronize()                # rec may come from a torch kernel (cat, flip) still running
    nb._ck(nb.lib().nb_keys_import(ctx.h, rec.data_ptr(), rec.shape[0]))


def _sorted(rec):
    rec = np.asarray(rec, dtype=np.uint64).reshape(-1, 4)
    return rec[np.lexsort(rec.T[::-1])]


def _owner(rec, world):
    return (((rec[:, 0] >> np.uint64(40)) & np.uint64(0xFFFF)) % np.uint64(world)).astype(np.int64)


def _table(ctx):
    d = ctx.counts()
    return {tuple(cs): int(k) for _, cs, k in d["rows"]}, d["n_unique_keys"]


# ------------------------------------------------------------------ A. export kernels against the reference
def _check_exports(ctx, exp, pairs, names):
    """The context's key records against `exp` ({pair index: callset or None}, one entry per unique key): orders, key
    values (the k_pair results of those pairs), tags through the dictionary, and the partitioned export for every world."""
    n = _export_count(ctx)
    assert n == len(exp)
    d = _dictionary(_callset_rows(ctx), names)
    klo, khi = pairs["key_lo"].tolist(), pairs["key_hi"].tolist()
    for base in BASES:
        rec = _host(_export_dev(ctx, base))
        orders = [o - base for o in rec[:, 2].tolist()]
        assert len(set(orders)) == n and set(orders) == set(exp), base
        bad = []
        for (k0, k1, _, tag), p in zip(rec.tolist(), orders):
            want = exp[p]
            got = None if tag == 0 else d.get(tag, "tag %x not in the dictionary" % tag)
            if (k0, k1) != (klo[p], khi[p]) or got != want:
                bad.append((p, got, want))
        assert not bad, bad[:5]
        want_sorted = _sorted(rec)
        for world in WORLDS:
            part, cnt = _export_partitioned(ctx, world, base)
            assert np.array_equal(cnt, np.bincount(_owner(rec, world), minlength=world)), (base, world)
            assert np.array_equal(_sorted(part), want_sorted), (base, world)
            at = np.concatenate([[0], np.cumsum(cnt)])
            own = _owner(part, world)
            assert all((own[at[o]:at[o + 1]] == o).all() for o in range(world)), (base, world)


@pytest.mark.parametrize("grown", [False, True], ids=["default", "grown_from_1024"])
def test_key_exports_match_the_oracle(grown):
    J = _job(0)
    # 1024 slots and 1024-pair chunks: the table doubles at the first chunk and again and again up to ~14k keys at load <= 0.5
    ctx, pairs = _ctx(J, **(dict(key_slots=1024, max_batch_pairs=1024) if grown else {}))
    exp = _expect(J, 0, N)
    assert len(exp) > 8 * 1024 and sum(cs is None for cs in exp.values()) > 100
    _check_exports(ctx, exp, pairs, J.names)
    table, uniq = _table(ctx)
    assert uniq == len(exp) and table == J.want
    ctx.close()


def test_key_exports_of_one_key_and_of_no_batch():
    J = _job(0)
    p = int(J.insertable[0])
    ctx, pairs = _ctx(J, p, p + 1)
    _check_exports(ctx, {0: J.callset[p]}, pairs, J.names)
    empty = nb.Context(J.ix, J.lib)
    assert _export_count(empty) == 0
    for world in WORLDS:
        part, cnt = _export_partitioned(empty, world)
        assert len(part) == 0 and cnt.tolist() == [0] * world
    nb._ck(nb.lib().nb_keys_export(empty.h, None, 0, 0))
    ctx.close(); empty.close()


def test_key_export_misuse_fails_loudly():
    J = _job(0)
    ctx, _ = _ctx(J, 0, 2000)
    n = _export_count(ctx)
    assert n > 100
    buf = torch.zeros((n, 4), dtype=torch.int64, device="cuda")
    cnt = np.zeros(64, dtype=np.uint64)
    with pytest.raises(nb.NbError, match="too small"):
        nb._ck(nb.lib().nb_keys_export(ctx.h, buf.data_ptr(), n - 1, 0))
    with pytest.raises(nb.NbError, match="too small"):
        nb._ck(nb.lib().nb_keys_export_partitioned(ctx.h, buf.data_ptr(), n - 1, 0, 4, cnt.ctypes.data))
    for world in (0, 65):
        with pytest.raises(nb.NbError):
            nb._ck(nb.lib().nb_keys_export_partitioned(ctx.h, buf.data_ptr(), n, 0, world, cnt.ctypes.data))
    nb._ck(nb.lib().nb_keys_export_partitioned(ctx.h, buf.data_ptr(), n, 0, 64, cnt.ctypes.data))   # exactly enough room
    assert int(cnt.sum()) == n
    ctx.close()


# ------------------------------------------------------------------ B. import kernels
def test_key_import_reproduces_the_exporter():
    J = _job(0)
    E, _ = _ctx(J)
    rows, rec = _callset_rows(E), _export_dev(E)
    want = _sorted(_host(rec))
    table, uniq = _table(E)
    for reverse in (False, True):
        I = nb.Context(J.ix, J.lib, key_slots=1024)          # far below 2 x records: nb_keys_import grows the table
        _callsets_import(I, rows)
        _keys_import(I, rec.flip(0).contiguous() if reverse else rec)
        assert np.array_equal(_sorted(_host(_export_dev(I))), want), reverse
        assert _table(I) == (table, uniq) and table == J.want, reverse
        I.close()
    E.close()


def test_key_import_of_overlapping_records_keeps_the_later_pair():
    J = _job(0)
    lo_b, hi_a = 8000, 12000
    A, _ = _ctx(J, 0, hi_a)
    B, _ = _ctx(J, lo_b, N)
    ra, rb = _export_dev(A, 0), _export_dev(B, lo_b)             # global pair orders
    ha, hb = _host(ra), _host(rb)
    oa = {(k0, k1): o for k0, k1, o, _ in ha.tolist()}
    both = [(k0, k1) for k0, k1, o, _ in hb.tolist() if (k0, k1) in oa and oa[(k0, k1)] != o]
    assert len(both) > 300                                         # many keys on both sides, with different last pairs
    merged = {}
    for k0, k1, o, t in np.concatenate([ha, hb]).tolist():
        if (k0, k1) not in merged or merged[(k0, k1)][0] < o:
            merged[(k0, k1)] = (o, t)
    want = _sorted([[k0, k1, o, t] for (k0, k1), (o, t) in merged.items()])
    F, _ = _ctx(J)
    assert np.array_equal(_sorted(_host(_export_dev(F))), want)   # one context over the union holds the same records
    F.close()
    rows = np.concatenate([_callset_rows(A), _callset_rows(B)])
    for first, second in ((ra, rb), (rb, ra)):
        U = nb.Context(J.ix, J.lib, key_slots=1024)
        _callsets_import(U, rows)
        _keys_import(U, torch.cat([first, second]))
        assert np.array_equal(_sorted(_host(_export_dev(U))), want)
        table, uniq = _table(U)
        assert table == J.want and uniq == len(merged)
        U.close()
    A.close(); B.close()


def test_callsets_import_device_equals_host_import():
    J = _job(0)
    E, _ = _ctx(J, 0, 6000)
    rows, rec = _callset_rows(E), _export_dev(E)
    H = nb.Context(J.ix, J.lib)
    _callsets_import(H, rows)
    D = nb.Context(J.ix, J.lib)
    dev = torch.from_numpy(rows.view(np.int32)).cuda()
    torch.cuda.synchronize()                                       # the context reads it on a stream of its own
    nb._ck(nb.lib().nb_callsets_import_device(D.h, dev.data_ptr(), rows.shape[0]))
    strip = lambda rs: sorted(map(tuple, rs[:, 1:].tolist()))    # noqa: E731 - slots may differ, {len, tag, items} may not
    assert strip(_callset_rows(D)) == strip(_callset_rows(H)) == strip(rows) and len(rows) > 20
    _keys_import(D, rec)
    assert _table(D) == _table(E)
    for c in (E, H, D):
        c.close()


def test_key_record_with_an_unknown_callset_fails_loudly():
    J = _job(0)
    E, _ = _ctx(J, 0, 6000)
    rows, rec = _callset_rows(E), _export_dev(E)
    tag = next(t for t in _host(rec)[:, 3].tolist() if t)
    keep = rows[(rows[:, 2].astype(np.uint64) | (rows[:, 3].astype(np.uint64) << np.uint64(32))) != np.uint64(tag)]
    assert len(keep) == len(rows) - 1
    X = nb.Context(J.ix, J.lib)
    _callsets_import(X, keep)
    with pytest.raises(nb.NbError, match="never given"):
        _keys_import(X, rec)
    E.close(); X.close()


# ------------------------------------------------------------------ C. merge_across_ranks with DeviceShard
def _bounds(world):
    cuts = [N * i // world for i in range(world + 1)]
    if world == 5:
        cuts = [0, N // 4, N // 2, N // 2, 3 * N // 4, N]          # rank 2 aligns nothing
    return [(cuts[r], cuts[r + 1]) for r in range(world)]


@pytest.mark.parametrize("routed", [False, True], ids=["all_to_all", "routed"])
@pytest.mark.parametrize("mm", [0, 2])
@pytest.mark.parametrize("world", [2, 3, 5])
def test_merge_across_ranks_with_device_shards(world, mm, routed):
    J = _job(mm)
    bounds = _bounds(world)
    ctxs = [nb.Context(J.ix, J.lib, max_batch_pairs=4096) for _ in range(world)]
    saved_cap = mg._ROUTED_CAP[0]
    if routed:
        mg._ROUTED_CAP[0] = 16                                     # far below the dictionaries: the block capacity must ratchet up
        for c in ctxs:
            c.route_create(world, N)
        for r, c in enumerate(ctxs):
            c.route_attach_ctx(world, r, ctxs, bounds[r][0])
    sizes = []

    def rank(r, dist):
        c = ctxs[r]
        lo, hi = bounds[r]
        if hi > lo:
            c.align_batch(*_part(J.data, lo, hi), max_read_len=150)
        # max_pairs = 0 would make a scoped shard: an empty rank still gets a (one-record) export buffer
        shard = mg.DeviceShard(c, nb, torch, lo, max(hi - lo, 1), routed=routed)
        sizes.append(len(shard.callsets_export()))
        raw, uniq = mg.merge_across_ranks(shard, torch, dist, r, world, "cuda", routed=routed)
        names = c.decode_counts(raw)["callsets"]
        return {tuple(cs): int(k) for cs, k in zip(names, raw["dense_counts"].tolist()) if k}, uniq
    try:
        outs = _run_ranks(world, rank)
        grown_cap = mg._ROUTED_CAP[0]
    finally:
        mg._ROUTED_CAP[0] = saved_cap
        for c in ctxs:
            if routed:
                c.route_detach()
            c.close()
    for r, (table, uniq) in enumerate(outs):
        assert table == J.single == J.want, r
        assert uniq == J.single_unique, r
    if routed:
        assert grown_cap >= max(sizes) > 16


# ------------------------------------------------------------------ D. merge_scoped_across_ranks with DeviceShard(max_pairs=0)
@functools.lru_cache(maxsize=None)
def _scoped_job():
    J = _Job()
    J.L = synth.SynthLibrary(seed=78, n_fam=40, n_all=5, group_on="")
    obj = J.L.to_json_obj()
    J.lib = nb.Library.from_text(json.dumps(obj), "unstranded")
    J.ix = nb.build_index(J.lib, 8)
    J.u = u = synth.umi_reads(J.L, 0, 1200, seed=9, n_cells=50)
    J.start = np.concatenate([[0], np.cumsum(u["sizes"])]).astype(np.int64)
    n = u["n_reads"]
    ocfg, oref = orc.parse_reference_library(obj, "unstranded")
    off = u["off"][: n + 1]
    ref = orc.Oracle(ocfg, oref).run(u["bases"][: 91 * n], off, u["bases"][: 91 * n], off, q1=u["qual"], q2=u["qual"],
                                     skip1=np.ones(n, dtype=np.uint8), skip2=None, scope_off=J.start.astype(np.uint64), threads=8, want_records=False)
    J.want = {}
    for s, rows in enumerate(ref["scopes"]):
        cell = int(u["cell"][J.start[s]])
        for cs, c in rows:
            J.want[(cell, tuple(cs))] = J.want.get((cell, tuple(cs)), 0) + c
    return J


def _scoped_align(c, J, a, b):
    u, L = J.u, 91
    bases = np.concatenate([u["bases"][a * L:b * L], np.zeros(64, dtype=np.uint8)])
    qual = np.concatenate([u["qual"][a * L:b * L], np.zeros(64, dtype=np.uint8)])
    off = np.arange(b - a + 1, dtype=np.uint64) * L
    f1, f2 = np.full(b - a, nb.FLAG_SKIP_ALIGN, dtype=np.uint8), np.zeros(b - a, dtype=np.uint8)
    scope = (u["scope"][a:b] - u["scope"][a]).astype(np.uint32)
    c.align_batch(bases, off, bases, off, q1=qual, q2=qual, flags1=f1, flags2=f2, scope_id=scope, cell_id=u["cell"][a:b], max_read_len=L)


@pytest.mark.parametrize("n_cells", [50, 1 << 40], ids=["dense", "sparse"])
def test_scoped_merge_with_device_shards(n_cells):
    J = _scoped_job()
    world, ns = 3, len(J.u["sizes"])
    one = nb.Context(J.ix, J.lib)
    _scoped_align(one, J, 0, J.u["n_reads"])
    single = {(int(c), tuple(cs)): int(k) for c, cs, k in one.counts()["rows"]}
    one.close()
    assert single == J.want and len(single) > 100
    scopes = [(ns * r // world, ns * (r + 1) // world) for r in range(world)]
    ctxs = [nb.Context(J.ix, J.lib) for _ in range(world)]

    def rank(r, dist):
        c = ctxs[r]
        s0, s1 = scopes[r]
        _scoped_align(c, J, int(J.start[s0]), int(J.start[s1]))
        shard = mg.DeviceShard(c, nb, torch, 0, 0)
        assert shard.scoped
        raw, cells, css, vals = mg.merge_scoped_across_ranks(shard, torch, dist, r, world, "cuda", n_cells)
        names = c.decode_counts(raw)["callsets"]
        return {(int(ce), tuple(names[int(k)])): int(v) for ce, k, v in zip(cells.tolist(), css.tolist(), vals.tolist())}
    try:
        outs = _run_ranks(world, rank)
    finally:
        for c in ctxs:
            c.close()
    assert outs[0] == single                     # the job's table is read back on rank 0 (the sparse branch returns it everywhere)
    if n_cells > 50:
        assert all(o == single for o in outs)
