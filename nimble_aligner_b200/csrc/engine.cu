// engine.cu — execution context behind the C ABI: device copies of the index / library tables, per-batch staging,
// the K0..K4 launch sequence on one CUDA stream, and result read-back.  No CPU fallback: every entry point fails
// with NB_ERR_CUDA when the device cannot be used.
#include <time.h>
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <string>
#include <thread>
#include <unordered_map>
#include <atomic>
#include <vector>

#include <dlfcn.h>
#include <nccl.h>   // types only: the functions are resolved from libnccl.so.2 at run time (nccl_api below)

#include "host.hpp"
#include "kernels.cuh"
#include "khash.h"

using namespace nb;
using nbk::BatchDev; using nbk::Counters; using nbk::DevCfg; using nbk::DevIndex; using nbk::DevLib; using nbk::Tables;

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) return fail(NB_ERR_CUDA, std::string(#x) + ": " + cudaGetErrorString(e_)); } while (0)

namespace {

struct DBuf {
  void* p = nullptr; size_t cap = 0;
  cudaError_t ensure(size_t bytes, cudaStream_t s, bool zero = false) {
    if (bytes <= cap) return cudaSuccess;
    if (p) { cudaError_t e = cudaStreamSynchronize(s); if (e != cudaSuccess) return e; cudaFree(p); p = nullptr; cap = 0; }
    size_t want = bytes + bytes / 4 + 256;
    cudaError_t e = cudaMalloc(&p, want); if (e != cudaSuccess) { p = nullptr; return e; }
    cap = want;
    if (zero) return cudaMemsetAsync(p, 0, want, s);
    return cudaSuccess;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

template <class T> cudaError_t upload(DBuf& d, const std::vector<T>& v, cudaStream_t s, size_t pad_bytes = 0) {
  size_t bytes = v.size() * sizeof(T);
  cudaError_t e = d.ensure(bytes + pad_bytes + 16, s); if (e != cudaSuccess) return e;
  if (bytes) e = cudaMemcpyAsync(d.p, v.data(), bytes, cudaMemcpyHostToDevice, s);
  return e;
}

// one team of host threads for a whole multi-phase job: spawned once, phases separated by a spin barrier
struct HostTeam {
  u32 T; std::atomic<u32> arrived{0}; std::atomic<u32> phase{0};
  explicit HostTeam(u32 t) : T(t) {}
  void barrier() {
    if (T == 1) return;
    const u32 ph = phase.load(std::memory_order_acquire);
    if (arrived.fetch_add(1, std::memory_order_acq_rel) + 1 == T) { arrived.store(0, std::memory_order_relaxed); phase.store(ph + 1, std::memory_order_release); }
    else { u32 spins = 0; while (phase.load(std::memory_order_acquire) == ph) { if (++spins > 200) std::this_thread::yield(); } }
  }
  template <class F> void run(F fn) {
    if (T == 1) { fn(0u); return; }
    std::vector<std::thread> th; for (u32 t = 1; t < T; t++) th.emplace_back([&, t] { fn(t); });
    fn(0u);
    for (auto& x : th) x.join();
  }
};

// maxinfo tables, src/align.rs:873-897 (built once per config on the host with the same libm as the CPU reference)
i64 f64_as_i64(double v) { if (std::isnan(v)) return 0; if (v >= 9223372036854775807.0) return INT64_MAX; if (v <= -9223372036854775808.0) return INT64_MIN; return (i64)v; }
void build_maxinfo_tables(u64 target, double strictness, std::vector<i64>& ls, std::vector<i64>& qp) {
  const int LONGEST = 1000, MAXQ = 60;
  std::vector<double> l(LONGEST), q(MAXQ + 1);
  for (int i = 0; i < LONGEST; i++) { double pow1 = std::exp((double)target - (double)i - 1.0); l[i] = std::log(1.0 / (1.0 + pow1)) + std::log((double)(i + 1)) * (1.0 - strictness); }
  for (int i = 0; i <= MAXQ; i++) { double pc = 1.0 - std::pow(10.0, -((0.5 + (double)i) / 10.0)); q[i] = std::log(pc) * strictness; }
  auto ratio = [](const std::vector<double>& a) { double mx = std::fabs(a[0]); for (size_t i = 1; i < a.size(); i++) { double v = std::fabs(a[i]); if (v > mx) mx = v; } return 9223372036854775807.0 / (mx * 2000.0); };
  double r = std::fmax(ratio(l), ratio(q));
  ls.resize(LONGEST); qp.resize(MAXQ + 1);
  for (int i = 0; i < LONGEST; i++) ls[i] = f64_as_i64(l[i] * r);
  for (int i = 0; i <= MAXQ; i++) qp[i] = f64_as_i64(q[i] * r);
}

}  // namespace

struct nb_ctx {
  int device = 0; cudaStream_t stream = nullptr; bool own_stream = false;
  const nb_index* hix = nullptr; const nb_library* lib = nullptr;
  nb_config hcfg; DevCfg dcfg; DevIndex dix; DevLib dlib;
  // index + library device copies
  DBuf d_ptab, d_bloom, d_unitig, d_node, d_walk, d_ledge, d_coloff, d_colids, d_colmeta, d_rowfid, d_rowrev, d_rowof, d_featgroup, d_ent, d_ls, d_qp, d_mincov;
  DBuf d_rowuoff, d_rowupos, d_rowother, d_rowgroup;   // per-row tables of the pair stage (kernels.cuh DevLib)
  // options
  u64 max_batch_pairs = 1u << 20, arena_entries = 1u << 24, cs_slots = 1u << 18, key_slots = 1u << 22, agg_slots = 1u << 20;
  int count_work = 0; u32 min_read_len = 40;  // MIN_READ_LENGTH, src/align.rs:18 (tests pass 12, src/align.rs:1066)
  // persistent tables
  DBuf d_cstag, d_cslen, d_csitems, d_key, d_kval, d_klast, d_pslot, d_pres2, d_aggkey, d_aggcnt, d_arena, d_ctr, d_scratch, d_nout;
  u32 gcap = 16;
  bool tables_ready = false;
  // staging + per-batch buffers
  // host batches: two staging sets filled on a copy stream so that the H2D of chunk i+1 overlaps the kernels of chunk i
  struct Staging { DBuf a[2], off[2], q[2], f[2], len[2], scope, cell; cudaEvent_t copied = nullptr, consumed = nullptr; bool used = false; } stg[2];
  int stg_next = 0; cudaStream_t cstream = nullptr;
  DBuf d_pk, d_lenfull, d_lentrim, d_rres, d_pres, d_rout, d_seeded;
  // state
  int mode = -1;  // -1 unset, 0 whole-run scope (keys persist), 1 scoped (keys live for one batch)
  bool folded = false;
  u64 pairs_seen = 0, last_unique = 0;
  // Whole-run scope: how full the key table is, known without a blocking pass.  The device keeps Counters::n_live; after every
  // launch that inserts keys an 8-byte copy of it is queued into a pinned ring behind an event.  Upper bound on the current
  // count = the newest value that has arrived + every key submitted since that copy was queued.
  struct LiveRing { cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr}; u64* host = nullptr; u64 at[4] = {0, 0, 0, 0}; bool pending[4] = {false, false, false, false}; int next = 0; u64 known = 0, known_at = 0, submitted = 0; } live;
  BatchDev last_b; bool have_last = false;
  // timing
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ev_pending, ev_free;
  double map_ms = 0; u64 map_launches = 0, map_reads = 0, all_launches = 0;
  // results
  std::vector<u32> cs_items, slot_dense, dense_prev, dense_ids; std::vector<u64> cs_off;   // dense_prev: the slots slot_dense held last time (only those are reset); dense_ids: slot of callset i, uploaded to fill d_dense on the device
  bool dense_dev = false;   // d_dense holds slot_dense of the last finalize
  u32* h_csr = nullptr; size_t h_csr_cap = 0;   // pinned: compacted dictionary rows of the last finalize
  u8* h_rows = nullptr; size_t h_rows_cap = 0; u64 n_rows_dev = 0;   // pinned: row_scope | row_callset | row_count of the last finalize
  DBuf d_rowwork, d_rowout, d_dense, d_denseids;
  // peer routing of the whole-run scope (nb_route_*): own inbox = inbox_world regions of inbox_cap KeyRec, one per source rank; d_routecur = this rank's fill cursors
  DBuf d_inbox, d_routecur; u64 inbox_cap = 0; u32 inbox_world = 0; bool route_on = false; nbk::Route route; std::vector<void*> ipc_opened;
  // multi-GPU merge (nb_comm_*, nb_merge_*): the NCCL communicator this context merges over and its exchange blocks
  ncclComm_t comm = nullptr; bool own_comm = false; u32 cworld = 1, crank = 0; u64 merge_cap = 4096;
  DBuf d_blk1, d_all1, d_blk2, d_all2, d_densetab, d_densework; u64* h_hdr = nullptr;
  // per-cell table (nb_cells_*): survives nb_counts_reset.  Callsets are keyed by a persistent id (pid) because every finalize
  // renumbers them: cell_pid maps a callset's group list (as bytes) to its pid, pid_off / pid_items hold the lists in pid order
  DBuf d_cellkey, d_cellumi, d_cellreads, d_cellctr, d_cellscope, d_cellpid, d_cellwork, d_cellrows;
  u64 cell_slots = 1u << 22, cell_used = 0, cell_scopes = 0; bool cell_alloc = false;
  bool cells_rows = false, cells_rolled = false;   // the last finalize left scoped rows not rolled yet / a roll happened since nb_counts_reset
  std::unordered_map<std::string, u32> cell_pid; std::vector<u64> pid_off{0}; std::vector<u32> pid_items, pid_of_dense;
  std::vector<u64> cc_off; std::vector<u32> cc_items;   // callsets of the last nb_cells_finalize, in Vec<String> Ord
  u8* h_cellrows = nullptr; size_t h_cellrows_cap = 0;
};

static Tables make_tables(nb_ctx* c) {
  Tables t;
  t.cs_tag = (u64*)c->d_cstag.p; t.cs_len = (u32*)c->d_cslen.p; t.cs_items = (u32*)c->d_csitems.p; t.cs_mask = (u32)c->cs_slots - 1; t.gcap = c->gcap;
  t.key = (ulonglong2*)c->d_key.p; t.kval = (unsigned long long*)c->d_kval.p; t.klast = (unsigned long long*)c->d_klast.p; t.key_mask = c->key_slots - 1;
  t.agg_key = (unsigned long long*)c->d_aggkey.p; t.agg_cnt = (unsigned long long*)c->d_aggcnt.p; t.agg_mask = c->agg_slots - 1;
  t.arena = (u32*)c->d_arena.p; t.arena_cap = c->arena_entries; t.ctr = (Counters*)c->d_ctr.p;
  t.ent = (const double*)c->d_ent.p; t.ls = (const i64*)c->d_ls.p; t.qp = (const i64*)c->d_qp.p; t.mincov = (const u16*)c->d_mincov.p;
  return t;
}

static int apply_config(nb_ctx* c, const nb_config& cfg) {
  if (cfg.intersect_level < 0 || cfg.intersect_level > 2 || cfg.strand_filter < 0 || cfg.strand_filter > 3) return fail(NB_ERR_INVALID, "invalid intersect_level / strand_filter");
  u64 T = std::max<u64>(cfg.discard_multi_hits, cfg.max_hits_to_report);
  if (T + 1 > (u64)nbk::GL_MAX) return fail(NB_ERR_UNSUPPORTED, "max(discard_multi_hits, max_hits_to_report) must be < 64 on the device path");
  if (cfg.score_threshold > 0xFFFFFFFFull || cfg.num_mismatches > 0xFFFFull) return fail(NB_ERR_UNSUPPORTED, "score_threshold / num_mismatches out of range");
  u32 need_gcap = (u32)std::max<u64>(1, cfg.max_hits_to_report);
  if (c->tables_ready && need_gcap > c->gcap) return fail(NB_ERR_UNSUPPORTED, "max_hits_to_report grew beyond the callset stride chosen at context creation; create a new context");
  c->hcfg = cfg;
  DevCfg& d = c->dcfg;
  d.score_percent = cfg.score_percent; d.score_threshold = (u32)cfg.score_threshold; d.num_mismatches = (u32)cfg.num_mismatches;
  d.discard_nonzero_mismatch = cfg.discard_nonzero_mismatch; d.discard_multiple_matches = cfg.discard_multiple_matches; d.require_valid_pair = cfg.require_valid_pair;
  d.intersect_level = cfg.intersect_level; d.strand_filter = cfg.strand_filter; d.no_dedup = c->lib->no_dedup;
  d.discard_multi_hits = (u32)cfg.discard_multi_hits; d.max_hits = (u32)cfg.max_hits_to_report; d.gcap = c->gcap; d.min_read_len = c->min_read_len;
  std::vector<i64> ls, qp; build_maxinfo_tables(cfg.trim_target_length, cfg.trim_strictness, ls, qp);
  CK(upload(c->d_ls, ls, c->stream)); CK(upload(c->d_qp, qp, c->stream));
  std::vector<u16> mincov(nbk::ENT_NMAX + 1, 0);
  for (int n = 1; n <= nbk::ENT_NMAX; n++) { int m = n + 1; for (int k = 0; k <= n; k++) if ((double)k / (double)n >= cfg.score_percent) { m = k; break; } mincov[n] = (u16)m; }
  CK(upload(c->d_mincov, mincov, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return NB_OK;
}

static int alloc_tables(nb_ctx* c) {
  cudaStream_t s = c->stream;
  c->gcap = std::max<u32>(16, (u32)c->hcfg.max_hits_to_report);
  c->dcfg.gcap = c->gcap;
  CK(c->d_cstag.ensure(c->cs_slots * 8, s)); CK(c->d_cslen.ensure(c->cs_slots * 4, s)); CK(c->d_csitems.ensure(c->cs_slots * (size_t)c->gcap * 4, s));
  CK(c->d_key.ensure(c->key_slots * 16, s)); CK(c->d_kval.ensure(c->key_slots * 8, s)); CK(c->d_klast.ensure(c->key_slots * 8, s));
  CK(c->d_aggkey.ensure(c->agg_slots * 8, s)); CK(c->d_aggcnt.ensure(c->agg_slots * 8, s));
  CK(c->d_arena.ensure(c->arena_entries * 4, s)); CK(c->d_ctr.ensure(sizeof(Counters), s)); CK(c->d_nout.ensure(64, s));
  CK(cudaMemsetAsync(c->d_cstag.p, 0, c->cs_slots * 8, s)); CK(cudaMemsetAsync(c->d_key.p, 0, c->key_slots * 16, s)); CK(cudaMemsetAsync(c->d_kval.p, 0, c->key_slots * 8, s));
  CK(cudaMemsetAsync(c->d_aggkey.p, 0, c->agg_slots * 8, s)); CK(cudaMemsetAsync(c->d_aggcnt.p, 0, c->agg_slots * 8, s)); CK(cudaMemsetAsync(c->d_ctr.p, 0, sizeof(Counters), s));
  c->tables_ready = true; c->mode = -1; c->folded = false; c->pairs_seen = 0; c->have_last = false;
  for (int i = 0; i < 4; i++) { if (c->live.pending[i]) cudaEventSynchronize(c->live.ev[i]); c->live.pending[i] = false; }
  c->live.known = c->live.known_at = c->live.submitted = 0;
  return NB_OK;
}

static int check_device_errors(nb_ctx* c, Counters* out = nullptr) {
  Counters h;
  CK(cudaMemcpyAsync(&h, c->d_ctr.p, sizeof h, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  if (out) *out = h;
  if (h.err & nbk::E_FEATURE) return fail(NB_ERR_FEATURE_NOT_FOUND, "Feature not found in reference columns");
  if (h.err & nbk::E_ARENA) return fail(NB_ERR_OVERFLOW, "equivalence-class arena overflow: raise option ec_arena_entries or lower max_batch_pairs");
  if (h.err & nbk::E_CS_FULL) return fail(NB_ERR_OVERFLOW, "callset dictionary full: raise option callset_slots");
  if (h.err & nbk::E_KEY_FULL) return fail(NB_ERR_OVERFLOW, "read-key table full: raise option key_slots");
  if (h.err & nbk::E_AGG_FULL) return fail(NB_ERR_OVERFLOW, "count table full: raise option agg_slots");
  if (h.err & nbk::E_INBOX_FULL) return fail(NB_ERR_OVERFLOW, "routing inbox region full: create the routes with more records_per_peer");
  if (h.err & nbk::E_CS_UNKNOWN) return fail(NB_ERR_INVALID, "key record names a callset this rank was never given: import the peers' dictionaries (nb_callsets_import) before their key records");
  return NB_OK;
}

extern "C" {

int nb_device_count(void) { int n = 0; if (cudaGetDeviceCount(&n) != cudaSuccess) return 0; return n; }
void* nb_host_alloc(size_t bytes) { void* p = nullptr; if (cudaMallocHost(&p, bytes) != cudaSuccess) { cudaGetLastError(); return nullptr; } return p; }
void nb_host_free(void* p) { if (p) cudaFreeHost(p); }

int nb_ctx_create(const nb_index* index, const nb_library* lib, int device, void* cuda_stream, nb_ctx** out) {
  if (!index || !lib || !out) return fail(NB_ERR_INVALID, "null argument");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); return fail(NB_ERR_CUDA, "no CUDA device available: nimble_b200 has no CPU path"); }
  if (device < 0 || device >= ndev) return fail(NB_ERR_INVALID, "device ordinal out of range");
  CK(cudaSetDevice(device));
  cudaDeviceProp prop; CK(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) return fail(NB_ERR_CUDA, std::string("device is sm_") + std::to_string(prop.major) + std::to_string(prop.minor) + "; this library is built for sm_100a only");
  nb_library* mlib = const_cast<nb_library*>(lib);
  if (!mlib->derived) mlib->finalize();
  if (index->n_sequences != lib->n_rows()) return fail(NB_ERR_INVALID, "index was not built from this library (row count differs)");
  nb_ctx* c = new nb_ctx();
  c->device = device; c->hix = index; c->lib = lib;
  if (cuda_stream) c->stream = (cudaStream_t)cuda_stream; else { if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) { delete c; return fail(NB_ERR_CUDA, "cudaStreamCreate failed"); } c->own_stream = true; }
  cudaStream_t s = c->stream;
  if (cudaStreamCreateWithFlags(&c->cstream, cudaStreamNonBlocking) != cudaSuccess) { nb_ctx_free(c); return fail(NB_ERR_CUDA, "cudaStreamCreate failed"); }
  for (int i = 0; i < 2; i++) if (cudaEventCreateWithFlags(&c->stg[i].copied, cudaEventDisableTiming) != cudaSuccess || cudaEventCreateWithFlags(&c->stg[i].consumed, cudaEventDisableTiming) != cudaSuccess) { nb_ctx_free(c); return fail(NB_ERR_CUDA, "cudaEventCreate failed"); }
  int rc = NB_OK;
  auto up = [&](cudaError_t e) { if (e != cudaSuccess && rc == NB_OK) rc = fail(NB_ERR_CUDA, std::string("index upload: ") + cudaGetErrorString(e)); };
  up(upload(c->d_unitig, index->unitig, s)); up(upload(c->d_ledge, index->ledge, s)); up(upload(c->d_node, index->node, s));
  u64 n_pbuckets = nb_ptab_buckets(index->n_kmers), bloom_words = 0; u32 bloom_k = 0;
  if (rc == NB_OK) {
    // Probe table {key0, key1, value0, value1} per 32-byte bucket and, when it cannot live in L2, the Bloom prefilter: both
    // built here on the device from the artefact's flat table (khash.h), which is only staged for the build.
    if (n_pbuckets >= 0xFFFFFFFFull) rc = fail(NB_ERR_UNSUPPORTED, "index has too many k-mers for the 32-bit bucket index");
    // the prefilter always exists (80 % of all probes are misses of seed searches: one word instead of a bucket walk);
    // 16 bits per k-mer, at most 64 MB so that it stays L2-resident next to an HBM-resident table
    bloom_words = std::min<u64>(std::max<u64>(index->n_kmers / 4, 1024), (64ull << 20) / 8);
    bloom_k = index->n_kmers * 6 <= bloom_words * 64 ? 3 : 2;
    const char* env = getenv("NB_L2_HINTS");   // test knob: 0 / 1 forces the kernel variant; default: tables beyond 64 MB are HBM-resident
    c->dix.hbm = env ? (atoi(env) != 0) : (n_pbuckets * 32 > (64ull << 20));
    DBuf t_key, t_val, t_err;
    up(upload(t_key, index->table_key, s)); up(upload(t_val, index->table_val, s));
    up(c->d_ptab.ensure(n_pbuckets * 32, s)); up(t_err.ensure(4, s));
    up(c->d_bloom.ensure(bloom_words * 8, s));
    if (rc == NB_OK) {
      up(cudaMemsetAsync(c->d_ptab.p, 0, n_pbuckets * 32, s)); up(cudaMemsetAsync(t_err.p, 0, 4, s));
      up(cudaMemsetAsync(c->d_bloom.p, 0, bloom_words * 8, s));
      nbk::launch_probe_build((const u64*)t_key.p, (const u64*)t_val.p, index->table_key.size(), (u64*)c->d_ptab.p, (u32)n_pbuckets, (u64*)c->d_bloom.p, (u32)bloom_words, bloom_k, (unsigned int*)t_err.p, s);
      unsigned int herr = 0;
      up(cudaMemcpyAsync(&herr, t_err.p, 4, cudaMemcpyDeviceToHost, s)); up(cudaStreamSynchronize(s));
      if (rc == NB_OK && herr) rc = fail(NB_ERR_CUDA, "probe table build overflowed");
    }
    cudaStreamSynchronize(s); t_key.release(); t_val.release(); t_err.release();
  }
  {  // walk records (kernels.cuh DevIndex::walk), derived from the flat index arrays at upload time
    size_t nn = index->node.size(); std::vector<u32> w(16 * nn);
    auto base_at = [&](u64 pos) -> u64 { return (index->unitig[pos >> 5] >> (2 * (pos & 31))) & 3; };
    for (size_t v = 0; v < nn; v++) {
      const NodeRec& nr = index->node[v]; u32* o = &w[16 * v];
      o[0] = nr.start_lo; o[1] = nr.len; o[2] = nr.colour; o[3] = nr.exts_hi;
      memcpy(o + 4, &index->redge[4 * v], 16); memcpy(o + 8, &index->col_meta[4 * (size_t)nr.colour], 16);
      u64 st = (u64)nr.start_lo | ((u64)(nr.exts_hi >> 8) << 32), q[2] = {0, 0};
      for (u32 i = 0; i < 64 && (u32)K + i < nr.len; i++) q[i >> 5] |= base_at(st + K + i) << (2 * (i & 31));   // unitig bases [K, K + 64): a forward compare never starts below base K
      memcpy(o + 12, q, 16);
    }
    up(upload(c->d_walk, w, s));
    if (rc == NB_OK && cudaStreamSynchronize(s) != cudaSuccess) rc = fail(NB_ERR_CUDA, "index upload failed");   // the staging vector dies here
  }
  up(upload(c->d_coloff, index->col_off, s)); up(upload(c->d_colids, index->col_ids, s)); up(upload(c->d_colmeta, index->col_meta, s));
  up(upload(c->d_rowfid, lib->row_fid, s)); up(upload(c->d_rowrev, lib->row_rev, s)); up(upload(c->d_rowof, lib->row_of, s)); up(upload(c->d_featgroup, lib->feat_group, s));
  {  // per row: its component list (offset in col_ids, position in it), its other orientation, its roll-up group
    const u32 nr = lib->n_rows();
    std::vector<u32> uoff(nr, NONE32), other(nr, NONE32), group(nr, NONE32); std::vector<u8> upos(nr, 0);
    for (size_t col = 0; 4 * col + 3 < index->col_meta.size(); col++) {
      const u32 uo = index->col_meta[4 * col], us = index->col_meta[4 * col + 1];
      if (!us || (size_t)uo + us > index->col_ids.size()) continue;
      const u32 first = index->col_ids[uo];
      if (first < nr && uoff[first] == uo) continue;                      // this component's list was handled through another of its colours
      for (u32 k = 0; k < us; k++) { const u32 row = index->col_ids[uo + k]; if (row < nr) { uoff[row] = uo; upos[row] = (u8)k; } }
    }
    for (u32 r = 0; r < nr && r < lib->row_fid.size(); r++) {
      const u32 f = lib->row_fid[r]; const size_t o = 2 * (size_t)f + (1 - (lib->row_rev[r] ? 1 : 0));
      if (o < lib->row_of.size()) other[r] = lib->row_of[o];
      if (f < lib->feat_group.size()) group[r] = lib->feat_group[f];
    }
    up(upload(c->d_rowuoff, uoff, s)); up(upload(c->d_rowupos, upos, s)); up(upload(c->d_rowother, other, s)); up(upload(c->d_rowgroup, group, s));
    if (rc == NB_OK && cudaStreamSynchronize(s) != cudaSuccess) rc = fail(NB_ERR_CUDA, "library table upload failed");   // the vectors die here
  }
  {  // entropy terms f*log2(f), f = c/n, for every read length n <= ENT_NMAX (src/utils.rs:96-119)
    const int N = nbk::ENT_NMAX;
    std::vector<double> ent((size_t)(N + 1) * (N + 2) / 2, 0.0);
    for (int n = 1; n <= N; n++) for (int k = 1; k <= n; k++) { double f = (double)k / (double)n; ent[(size_t)n * (n + 1) / 2 + k] = f * std::log2(f); }
    up(upload(c->d_ent, ent, s));
  }
  if (rc == NB_OK) { cudaError_t e = cudaStreamSynchronize(s); if (e != cudaSuccess) rc = fail(NB_ERR_CUDA, cudaGetErrorString(e)); }
  if (rc != NB_OK) { nb_ctx_free(c); return rc; }
  c->dix.unitig = (const u64*)c->d_unitig.p; c->dix.ledge = (const uint4*)c->d_ledge.p;
  c->dix.ptab = (const u64*)c->d_ptab.p; c->dix.n_pbuckets = (u32)n_pbuckets; c->dix.bloom = (const u64*)c->d_bloom.p; c->dix.bloom_words = (u32)bloom_words; c->dix.bloom_k = bloom_k;
  c->dix.node = (const uint4*)c->d_node.p; c->dix.walk = (const uint4*)c->d_walk.p;
  c->dix.col_off = (const u32*)c->d_coloff.p; c->dix.col_ids = (const u32*)c->d_colids.p; c->dix.col_meta = (const uint4*)c->d_colmeta.p;
  c->dlib.row_fid = (const u32*)c->d_rowfid.p; c->dlib.row_rev = (const u8*)c->d_rowrev.p; c->dlib.row_of = (const u32*)c->d_rowof.p; c->dlib.feat_group = (const u32*)c->d_featgroup.p; c->dlib.n_rows = lib->n_rows();
  c->dlib.row_uoff = (const u32*)c->d_rowuoff.p; c->dlib.row_upos = (const u8*)c->d_rowupos.p; c->dlib.row_other = (const u32*)c->d_rowother.p; c->dlib.row_group = (const u32*)c->d_rowgroup.p;
  rc = apply_config(c, lib->cfg);
  if (rc != NB_OK) { nb_ctx_free(c); return rc; }
  *out = c;
  return NB_OK;
}

void nb_ctx_free(nb_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  if (c->cstream) cudaStreamSynchronize(c->cstream);
  if (c->stream) cudaStreamSynchronize(c->stream);
  DBuf* all[] = {&c->d_ptab, &c->d_bloom, &c->d_node, &c->d_walk, &c->d_unitig, &c->d_ledge, &c->d_coloff, &c->d_colids, &c->d_colmeta, &c->d_rowfid, &c->d_rowrev, &c->d_rowof, &c->d_featgroup, &c->d_rowuoff, &c->d_rowupos, &c->d_rowother, &c->d_rowgroup,
                 &c->d_ent, &c->d_ls, &c->d_qp, &c->d_mincov, &c->d_cstag, &c->d_cslen, &c->d_csitems, &c->d_key, &c->d_kval, &c->d_klast, &c->d_pslot, &c->d_pres2, &c->d_aggkey, &c->d_aggcnt, &c->d_arena, &c->d_ctr, &c->d_scratch, &c->d_nout,
                 &c->stg[0].a[0], &c->stg[0].a[1], &c->stg[0].off[0], &c->stg[0].off[1], &c->stg[0].q[0], &c->stg[0].q[1], &c->stg[0].f[0], &c->stg[0].f[1], &c->stg[0].len[0], &c->stg[0].len[1], &c->stg[0].scope, &c->stg[0].cell,
                 &c->stg[1].a[0], &c->stg[1].a[1], &c->stg[1].off[0], &c->stg[1].off[1], &c->stg[1].q[0], &c->stg[1].q[1], &c->stg[1].f[0], &c->stg[1].f[1], &c->stg[1].len[0], &c->stg[1].len[1], &c->stg[1].scope, &c->stg[1].cell, &c->d_pk, &c->d_lenfull, &c->d_lentrim, &c->d_rres, &c->d_pres, &c->d_rout, &c->d_seeded, &c->d_rowwork, &c->d_rowout, &c->d_dense, &c->d_denseids};
  for (DBuf* b : all) b->release();
  for (void* q : c->ipc_opened) cudaIpcCloseMemHandle(q);
  c->ipc_opened.clear(); c->d_inbox.release(); c->d_routecur.release();
  nb_comm_free(c);
  c->d_blk1.release(); c->d_all1.release(); c->d_blk2.release(); c->d_all2.release(); c->d_densetab.release(); c->d_densework.release();
  for (DBuf* b : {&c->d_cellkey, &c->d_cellumi, &c->d_cellreads, &c->d_cellctr, &c->d_cellscope, &c->d_cellpid, &c->d_cellwork, &c->d_cellrows}) b->release();
  nb_host_free(c->h_cellrows); c->h_cellrows = nullptr;
  nb_host_free(c->h_hdr); c->h_hdr = nullptr;
  for (int i = 0; i < 4; i++) if (c->live.ev[i]) cudaEventDestroy(c->live.ev[i]);
  nb_host_free(c->live.host); c->live.host = nullptr;
  nb_host_free(c->h_rows); c->h_rows = nullptr;
  nb_host_free(c->h_csr); c->h_csr = nullptr;
  for (auto& e : c->ev_pending) { cudaEventDestroy(e.first); cudaEventDestroy(e.second); }
  for (auto& e : c->ev_free) { cudaEventDestroy(e.first); cudaEventDestroy(e.second); }
  for (int i = 0; i < 2; i++) { if (c->stg[i].copied) cudaEventDestroy(c->stg[i].copied); if (c->stg[i].consumed) cudaEventDestroy(c->stg[i].consumed); }
  if (c->cstream) cudaStreamDestroy(c->cstream);
  if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
  delete c;
}

int nb_ctx_set_config(nb_ctx* c, const nb_config* cfg) { if (!c || !cfg) return fail(NB_ERR_INVALID, "null argument"); CK(cudaSetDevice(c->device)); return apply_config(c, *cfg); }
int nb_ctx_sync(nb_ctx* c) { if (!c) return fail(NB_ERR_INVALID, "null argument"); CK(cudaSetDevice(c->device)); CK(cudaStreamSynchronize(c->cstream)); CK(cudaStreamSynchronize(c->stream)); return NB_OK; }

int nb_ctx_set_option(nb_ctx* c, const char* name, uint64_t value) {
  if (!c || !name) return fail(NB_ERR_INVALID, "null argument");
  auto pow2 = [](u64 v) { u64 p = 16; while (p < v) p <<= 1; return p; };
  std::string n(name);
  if (n == "count_work") { c->count_work = value != 0; return NB_OK; }
  if (n == "min_read_length") { c->min_read_len = (u32)value; c->dcfg.min_read_len = (u32)value; return NB_OK; }
  if (n == "cell_slots") { if (c->cell_alloc) return fail(NB_ERR_INVALID, "cell_slots must be set before the first nb_cells_roll (or after nb_cells_reset)"); c->cell_slots = pow2(value); return NB_OK; }
  if (c->tables_ready) return fail(NB_ERR_INVALID, "options must be set before the first nb_align_batch (or after nb_counts_reset)");
  if (n == "max_batch_pairs") c->max_batch_pairs = std::max<u64>(1, value);
  else if (n == "ec_arena_entries") c->arena_entries = std::max<u64>(1024, value);
  else if (n == "callset_slots") { c->cs_slots = pow2(value); if (c->cs_slots > (1u << 23)) return fail(NB_ERR_INVALID, "callset_slots must be <= 2^23"); }
  else if (n == "key_slots") c->key_slots = pow2(value);
  else if (n == "agg_slots") c->agg_slots = pow2(value);
  else return fail(NB_ERR_INVALID, "unknown option " + n);
  return NB_OK;
}

static int grow_keys(nb_ctx* c, u64 need_slots) {
  u64 ns = c->key_slots; while (ns < need_slots) ns <<= 1;
  DBuf nk, nv; cudaStream_t s = c->stream;
  auto ck2 = [&](cudaError_t e) { if (e == cudaSuccess) return true; nk.release(); nv.release(); fail(NB_ERR_CUDA, std::string("key table growth: ") + cudaGetErrorString(e)); return false; };
  if (!ck2(nk.ensure(ns * 16, s)) || !ck2(nv.ensure(ns * 8, s))) return NB_ERR_CUDA;
  if (!ck2(cudaMemsetAsync(nk.p, 0, ns * 16, s)) || !ck2(cudaMemsetAsync(nv.p, 0, ns * 8, s))) return NB_ERR_CUDA;
  if (c->mode != 1) {   // scoped batches clear the table after every chunk: nothing to carry over (and Counters::n_keys, which accumulates the per-chunk unique keys there, must stay)
    Tables o = make_tables(c); Tables n = o; n.key = (ulonglong2*)nk.p; n.kval = (unsigned long long*)nv.p; n.key_mask = ns - 1;
    nbk::launch_rehash_keys(o, n, s); c->all_launches++;
  }
  if (!ck2(cudaStreamSynchronize(s))) return NB_ERR_CUDA;
  c->d_key.release(); c->d_kval.release(); c->d_key = nk; c->d_kval = nv; c->key_slots = ns;
  c->d_klast.release(); CK(c->d_klast.ensure(ns * 8, s)); CK(cudaMemsetAsync(c->d_klast.p, 0, ns * 8, s));
  return NB_OK;
}

// after a launch that inserted keys (live.submitted already counts them): queue a copy of the device's unique-key count
static int live_note(nb_ctx* c) {
  nb_ctx::LiveRing& L = c->live;
  if (!L.host) {
    L.host = (u64*)nb_host_alloc(4 * sizeof(u64)); if (!L.host) return fail(NB_ERR_CUDA, "pinned host allocation failed");
    for (int i = 0; i < 4; i++) CK(cudaEventCreateWithFlags(&L.ev[i], cudaEventDisableTiming));
  }
  const int i = L.next;
  if (L.pending[i]) { if (cudaEventQuery(L.ev[i]) != cudaSuccess) return NB_OK; L.pending[i] = false; if (L.at[i] >= L.known_at) { L.known = L.host[i]; L.known_at = L.at[i]; } }   // ring full of copies still in flight: keep them
  CK(cudaMemcpyAsync(&L.host[i], &((Counters*)c->d_ctr.p)->n_live, 8, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaEventRecord(L.ev[i], c->stream));
  L.at[i] = L.submitted; L.pending[i] = true; L.next = (i + 1) & 3;
  return NB_OK;
}
// room for `incoming` more keys at load <= 0.5; blocks (and counts exactly) only when the bound says the table might not do
static int ensure_key_capacity(nb_ctx* c, u64 incoming) {
  nb_ctx::LiveRing& L = c->live;
  for (int i = 0; i < 4; i++) if (L.pending[i] && cudaEventQuery(L.ev[i]) == cudaSuccess) { L.pending[i] = false; if (L.at[i] >= L.known_at) { L.known = L.host[i]; L.known_at = L.at[i]; } }
  u64 upper = L.known + (L.submitted - L.known_at);
  if (2 * (upper + incoming) > c->key_slots) {
    Counters h; int rc = check_device_errors(c, &h); if (rc) return rc;   // drains the stream: every queued copy has arrived too
    for (int i = 0; i < 4; i++) L.pending[i] = false;
    L.known = h.n_live; L.known_at = L.submitted;
    if (2 * (h.n_live + incoming) > c->key_slots) { rc = grow_keys(c, 2 * (h.n_live + incoming)); if (rc) return rc; }
  }
  L.submitted += incoming;
  return NB_OK;
}

static int run_chunk(nb_ctx* c, const nb_batch* bt, u64 p0, u64 p1, u32 max_len, nb_read_result* reads_out, nb_pair_result* pairs_out) {
  cudaStream_t s = c->stream;
  u64 np = p1 - p0; u32 sides = bt->r2 ? 2 : 1; u64 nr = np * sides;
  bool host = bt->location == NB_MEM_HOST;
  cudaMemcpyKind kind = host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice;
  BatchDev b; memset(&b, 0, sizeof b);
  b.n_pairs = np; b.sides = sides; b.n_reads = (u32)nr; b.W = (max_len + 31) / 32 + 1; b.order_base = c->pairs_seen;
  if (nr * (u64)b.W >= 0xFFFFFFFFull) return fail(NB_ERR_INVALID, "max_batch_pairs too large for this read length: lower option max_batch_pairs");
  const u8* src_a[2] = {bt->r1, bt->r2}; const u64* src_off[2] = {bt->r1_off, bt->r2_off}; const u8* src_q[2] = {bt->q1, bt->q2}; const u8* src_f[2] = {bt->flags1, bt->flags2};
  const u32* src_len[2] = {bt->r1_len, bt->r2_len};
  const u32 bits = bt->encoding == NB_SEQ_2BIT ? 2u : bt->encoding == NB_SEQ_BAM4 ? 4u : 8u;   // per base in r1 / r2 (offsets count bases)
  b.enc = (u32)bt->encoding;
  nb_ctx::Staging* S = nullptr; cudaStream_t cs = s;
  if (host) {
    S = &c->stg[c->stg_next]; c->stg_next ^= 1; cs = c->cstream;
    if (S->used) {
      // Reusing a staging set: the H2D copies that filled it two chunks ago must have RUN before this call returns, or the
      // documented reuse rule for the caller's host buffers (nimble_b200.h: free again once the second following call has
      // returned) would not hold — the host could otherwise run many batches ahead of the copy stream.  Blocking on that
      // copy also bounds the run-ahead to two chunks.
      CK(cudaEventSynchronize(S->copied));
      CK(cudaStreamWaitEvent(cs, S->consumed, 0));   // the kernels that read this staging set two chunks ago are done
    }
  }
  // staging buffers may be in use on either stream: drain both before a buffer is re-allocated
  auto ens = [&](DBuf& d, size_t bytes) -> cudaError_t { if (bytes <= d.cap) return cudaSuccess; cudaError_t e = cudaStreamSynchronize(c->cstream); if (e != cudaSuccess) return e; return d.ensure(bytes, s); };
  for (u32 sd = 0; sd < sides; sd++) {
    if (host) {
      u64 a0 = src_off[sd][p0], a1 = src_off[sd][p1];
      if (sd == 1 && src_a[1] == src_a[0] && src_off[1] == src_off[0] && src_q[1] == src_q[0] && src_len[1] == src_len[0]) {
        // the mate slot is the same buffer as the sequence slot (10x single-end records: the SKIP_ALIGN dummy is a clone of
        // the real record, sorted_bam_reader.rs:109-125): one copy serves both sides
        b.a[1] = b.a[0]; b.off[1] = b.off[0]; b.q[1] = b.q[0]; b.len[1] = b.len[0];
        if (src_f[sd]) { CK(ens(S->f[sd], np)); CK(cudaMemcpyAsync(S->f[sd].p, src_f[sd] + p0, np, kind, cs)); b.flags[sd] = (const u8*)S->f[sd].p; }
        continue;
      }
      const u64 ab0 = a0 * bits / 8 & ~(u64)7, ab1 = (a1 * bits + 7) / 8;   // byte range of the bases (8-byte aligned start: the packed kernels load aligned words)
      CK(ens(S->a[sd], ab1 - ab0 + 64)); CK(ens(S->off[sd], (np + 1) * 8));
      if (ab1 > ab0) CK(cudaMemcpyAsync(S->a[sd].p, src_a[sd] + ab0, ab1 - ab0, kind, cs));
      CK(cudaMemcpyAsync(S->off[sd].p, src_off[sd] + p0, (np + 1) * 8, kind, cs));
      b.a[sd] = (const u8*)S->a[sd].p - ab0; b.off[sd] = (const u64*)S->off[sd].p;
      if (src_len[sd]) { CK(ens(S->len[sd], np * 4)); CK(cudaMemcpyAsync(S->len[sd].p, src_len[sd] + p0, np * 4, kind, cs)); b.len[sd] = (const u32*)S->len[sd].p; }
      if (src_q[sd]) { CK(ens(S->q[sd], a1 - a0 + 64)); if (a1 > a0) CK(cudaMemcpyAsync(S->q[sd].p, src_q[sd] + a0, a1 - a0, kind, cs)); b.q[sd] = (const u8*)S->q[sd].p - a0; }
      if (src_f[sd]) { CK(ens(S->f[sd], np)); CK(cudaMemcpyAsync(S->f[sd].p, src_f[sd] + p0, np, kind, cs)); b.flags[sd] = (const u8*)S->f[sd].p; }
    } else {
      b.a[sd] = src_a[sd]; b.off[sd] = src_off[sd] + p0; b.q[sd] = src_q[sd]; b.flags[sd] = src_f[sd] ? src_f[sd] + p0 : nullptr; b.len[sd] = src_len[sd] ? src_len[sd] + p0 : nullptr;
    }
  }
  if (bt->scope_id) {
    if (host) { CK(ens(S->scope, np * 4)); CK(cudaMemcpyAsync(S->scope.p, bt->scope_id + p0, np * 4, kind, cs)); b.scope = (const u32*)S->scope.p; }
    else b.scope = bt->scope_id + p0;
    b.cell = b.scope;
    if (bt->cell_id) {
      if (host) { CK(ens(S->cell, np * 4)); CK(cudaMemcpyAsync(S->cell.p, bt->cell_id + p0, np * 4, kind, cs)); b.cell = (const u32*)S->cell.p; }
      else b.cell = bt->cell_id + p0;
    }
  }
  if (host) { CK(cudaEventRecord(S->copied, cs)); CK(cudaStreamWaitEvent(s, S->copied, 0)); }
  CK(c->d_pk.ensure((size_t)b.W * nr * 8 + 16, s));   /* k_walk reads up to two words past a row */ CK(c->d_lenfull.ensure(nr * 4, s)); CK(c->d_lentrim.ensure(nr * 4, s));
  CK(c->d_rres.ensure(nr * sizeof(nbk::ReadRes), s)); CK(c->d_pres.ensure(np * sizeof(nbk::PairRes), s)); CK(c->d_seeded.ensure(nr * 16, s));
  if (c->mode == 1) { CK(c->d_pslot.ensure(np * 8, s)); CK(c->d_pres2.ensure(np * sizeof(nbk::PairRes), s)); b.pslot = (u64*)c->d_pslot.p; b.pres2 = (nbk::PairRes*)c->d_pres2.p; }
  b.pk = (u64*)c->d_pk.p; b.len_full = (u32*)c->d_lenfull.p; b.len_trim = (u32*)c->d_lentrim.p; b.rres = (nbk::ReadRes*)c->d_rres.p; b.pres = (nbk::PairRes*)c->d_pres.p; b.seeded = (uint4*)c->d_seeded.p;
  // key-table capacity
  if (c->mode == 0) { int rc = ensure_key_capacity(c, np); if (rc) return rc; }
  else if (2 * np > c->key_slots) { int rc = grow_keys(c, 2 * np); if (rc) return rc; }
  Tables t = make_tables(c);
  CK(cudaMemsetAsync(&((Counters*)c->d_ctr.p)->arena_top, 0, 32, s));   // arena_top, queue, seeded_n, wqueue
  nbk::launch_pack(b, s); c->all_launches++;
  if (b.q[0] || b.q[1]) { nbk::launch_trim(b, t, s); c->all_launches++; }
  std::pair<cudaEvent_t, cudaEvent_t> ev;
  if (!c->ev_free.empty()) { ev = c->ev_free.back(); c->ev_free.pop_back(); } else { CK(cudaEventCreate(&ev.first)); CK(cudaEventCreate(&ev.second)); }
  CK(cudaEventRecord(ev.first, s));
  nbk::launch_map(b, c->dix, c->dcfg, t, c->count_work, s); c->all_launches++;
  CK(cudaEventRecord(ev.second, s));
  c->ev_pending.push_back(ev); c->map_launches++; c->map_reads += nr;
  nbk::Route rt; memset(&rt, 0, sizeof rt);
  if (c->route_on && c->mode == 0) rt = c->route;
  nbk::launch_pair(b, c->dix, c->dlib, c->dcfg, t, rt, s); c->all_launches++;
  if (c->mode == 0) { int rc = live_note(c); if (rc) return rc; }
  if (c->mode == 1) {
    nbk::launch_fold(t, b.cell, b.order_base, s); c->all_launches++;
    if (pairs_out) { nbk::launch_resolve(b, t, s); c->all_launches++; }
    CK(cudaMemsetAsync(c->d_key.p, 0, c->key_slots * 16, s)); CK(cudaMemsetAsync(c->d_kval.p, 0, c->key_slots * 8, s)); CK(cudaMemsetAsync(c->d_klast.p, 0, c->key_slots * 8, s));
  }
  if (host) { CK(cudaEventRecord(S->consumed, s)); S->used = true; }
  cudaMemcpyKind okind = host ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
  if (reads_out) {
    CK(c->d_rout.ensure(nr * sizeof(nb_read_result), s));
    nbk::launch_export_reads(b, c->dix, t, c->d_rout.p, s); c->all_launches++;
    CK(cudaMemcpyAsync(reads_out + p0 * sides, c->d_rout.p, nr * sizeof(nb_read_result), okind, s));
  }
  if (pairs_out) CK(cudaMemcpyAsync(pairs_out + p0, c->mode == 1 ? c->d_pres2.p : c->d_pres.p, np * sizeof(nb_pair_result), okind, s));
  CK(cudaGetLastError());
  c->pairs_seen += np; c->last_b = b; c->have_last = true;
  return NB_OK;
}

int nb_align_batch(nb_ctx* c, const nb_batch* bt, nb_read_result* reads_out, nb_pair_result* pairs_out) {
  if (!c || !bt) return fail(NB_ERR_INVALID, "null argument");
  static_assert(sizeof(nb_read_result) == 16 && sizeof(nb_pair_result) == 24, "ABI struct size");
  static_assert(sizeof(nbk::PairRes) == sizeof(nb_pair_result), "PairRes layout");
  CK(cudaSetDevice(c->device));
  if (bt->n_pairs && (!bt->r1 || !bt->r1_off || (bt->r2 && !bt->r2_off))) return fail(NB_ERR_INVALID, "batch needs r1/r1_off (and r2_off with r2)");
  if (bt->location != NB_MEM_HOST && bt->location != NB_MEM_DEVICE) return fail(NB_ERR_INVALID, "batch location must be NB_MEM_HOST or NB_MEM_DEVICE");
  if (bt->encoding != NB_SEQ_ASCII && bt->encoding != NB_SEQ_2BIT && bt->encoding != NB_SEQ_BAM4) return fail(NB_ERR_INVALID, "batch encoding must be NB_SEQ_ASCII, NB_SEQ_2BIT or NB_SEQ_BAM4");
  if (bt->encoding == NB_SEQ_ASCII && (bt->r1_len || bt->r2_len)) return fail(NB_ERR_INVALID, "explicit read lengths (r1_len / r2_len) belong to the packed encodings");
  if (!c->lib->injective) return fail(NB_ERR_UNSUPPORTED, "reference library not representable on the device pair stage: " + c->lib->irregular_reason);
  if (!c->tables_ready) { int rc = alloc_tables(c); if (rc) return rc; }
  if (c->folded) return fail(NB_ERR_INVALID, "counts were finalized; call nb_counts_reset before aligning more batches");
  int mode = bt->scope_id ? 1 : 0;
  if (c->mode == -1) { c->mode = mode; if (mode == 1) CK(cudaMemsetAsync(c->d_klast.p, 0, c->key_slots * 8, c->stream)); }   // klast is only used by scoped batches
  else if (c->mode != mode) return fail(NB_ERR_INVALID, "cannot mix scoped and whole-run batches in one context without nb_counts_reset");
  if (bt->n_pairs == 0) return NB_OK;
  u32 max_len = bt->max_read_len;
  if (!max_len) {
    if (bt->location != NB_MEM_HOST) return fail(NB_ERR_INVALID, "device-resident batches must state max_read_len");
    for (u64 p = 0; p < bt->n_pairs; p++) {
      max_len = std::max<u32>(max_len, bt->r1_len ? bt->r1_len[p] : (u32)(bt->r1_off[p + 1] - bt->r1_off[p]));
      if (bt->r2) max_len = std::max<u32>(max_len, bt->r2_len ? bt->r2_len[p] : (u32)(bt->r2_off[p + 1] - bt->r2_off[p]));
    }
  }
  if (max_len > (u32)nbk::ENT_NMAX) return fail(NB_ERR_UNSUPPORTED, "reads longer than 1024 bases are not supported by the device path");
  if (max_len == 0) max_len = 1;
  const u64 chunk = c->max_batch_pairs;
  for (u64 p0 = 0; p0 < bt->n_pairs;) {
    u64 p1 = std::min(bt->n_pairs, p0 + chunk);
    if (c->mode == 1 && p1 < bt->n_pairs) {  // never split a scope across chunks: its key table lives for one chunk
      if (bt->location != NB_MEM_HOST) return fail(NB_ERR_INVALID, "scoped device-resident batches must fit max_batch_pairs");
      while (p1 > p0 + 1 && bt->scope_id[p1] == bt->scope_id[p1 - 1]) p1--;
      if (bt->scope_id[p1] == bt->scope_id[p1 - 1]) {
        // one scope is larger than max_batch_pairs: it must still be de-duplicated as a whole, so the chunk grows to the
        // end of that scope (the per-chunk buffers grow with it)
        p1 = std::min(bt->n_pairs, p0 + chunk);
        while (p1 < bt->n_pairs && bt->scope_id[p1] == bt->scope_id[p1 - 1]) p1++;
      }
    }
    int rc = run_chunk(c, bt, p0, p1, max_len, reads_out, pairs_out);
    if (rc) return rc;
    p0 = p1;     // (round 1 advanced by max_batch_pairs here and silently skipped the pairs a shortened chunk left behind)
  }
  return NB_OK;
}

int nb_last_batch_ecs(nb_ctx* c, uint64_t* ec_off, uint32_t* ec_ids, uint64_t ec_cap, uint64_t* ec_total) {
  if (!c || !ec_off || !ec_total) return fail(NB_ERR_INVALID, "null argument");
  if (!c->have_last) return fail(NB_ERR_INVALID, "no batch has been aligned");
  CK(cudaSetDevice(c->device));
  const BatchDev& b = c->last_b;
  std::vector<nbk::ReadRes> rr(b.n_reads);
  CK(cudaMemcpyAsync(rr.data(), b.rres, rr.size() * sizeof(nbk::ReadRes), cudaMemcpyDeviceToHost, c->stream));
  Counters h; CK(cudaMemcpyAsync(&h, c->d_ctr.p, sizeof h, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  std::vector<u32> arena(std::min<u64>(h.arena_top, c->arena_entries));
  if (!arena.empty()) { CK(cudaMemcpy(arena.data(), c->d_arena.p, arena.size() * 4, cudaMemcpyDeviceToHost)); }
  u64 tot = 0;
  for (u32 i = 0; i < b.n_reads; i++) {
    ec_off[i] = tot;
    const nbk::ReadRes& r = rr[i];
    if (!r.ec_len) continue;
    bool big = (r.hdr >> 9) & 1;
    if (big) { for (u32 k = 0; k < r.bsize; k++) { if (ec_ids && tot < ec_cap) ec_ids[tot] = arena[r.ref + k]; tot++; } }
    else { for (u32 k = 0; k < r.bsize; k++) if ((r.mask >> k) & 1) { if (ec_ids && tot < ec_cap) ec_ids[tot] = c->hix->col_ids[r.ref + k]; tot++; } }
  }
  ec_off[b.n_reads] = tot; *ec_total = tot;
  return NB_OK;
}

struct NcclApi;
static const NcclApi* nccl_api();
static int dense_allreduce(nb_ctx* c, void* dense, u64 n);
static int dense_reduce_scatter(nb_ctx* c, void* dense, u64 chunk);
// dense_cells > 0 (nb_merge_scoped): the (cell, callset) rows of all ranks are summed through a dense [cells x callsets]
// table (all-reduce over NCCL) before they are read back; 0: this context's own rows.  shard: reduce-scatter instead — every
// rank keeps (and reads back) the rows of its own range of cells only
// d_dense = the host slot -> callset table of the last finalize (c->slot_dense), filled on the device by a scatter of the
// callset id list
static int upload_slot_map(nb_ctx* c, cudaStream_t s) {
  const std::vector<u32>& dense = c->slot_dense;
  CK(c->d_dense.ensure(dense.size() * 4, s)); CK(c->d_denseids.ensure(c->dense_ids.size() * 4 + 16, s));
  CK(cudaMemsetAsync(c->d_dense.p, 0xFF, dense.size() * 4, s));
  if (!c->dense_ids.empty()) { CK(cudaMemcpyAsync(c->d_denseids.p, c->dense_ids.data(), c->dense_ids.size() * 4, cudaMemcpyHostToDevice, s)); nbk::launch_dense_scatter((const u32*)c->d_denseids.p, c->dense_ids.size(), (u32*)c->d_dense.p, s); c->all_launches++; }
  c->dense_dev = true;
  return NB_OK;
}

static int finalize_impl(nb_ctx* c, nb_counts* out, u64 dense_cells, bool shard = false) {
  if (!c || !out) return fail(NB_ERR_INVALID, "null argument");
  CK(cudaSetDevice(c->device));
  memset(out, 0, sizeof *out);
  c->cs_items.clear(); c->cs_off.assign(1, 0); c->dense_dev = false;
  if (!c->tables_ready) { out->callset_off = c->cs_off.data(); return NB_OK; }
  cudaStream_t s = c->stream;
  Tables t = make_tables(c);
  static const bool fstats = getenv("NB_FINALIZE_STATS") != nullptr; double ft[5] = {0, 0, 0, 0, 0};
  auto fnow = []() { timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec + ts.tv_nsec * 1e-9; };
  if (fstats) { cudaStreamSynchronize(s); ft[0] = fnow(); }
  if (c->mode == 0 && !c->folded) { nbk::launch_fold(t, nullptr, 0, s); c->all_launches++; c->folded = true; }
  Counters h; int rc = check_device_errors(c, &h); if (rc) return rc;
  if (fstats) ft[1] = fnow();
  c->last_unique = h.n_keys;
  // compact the occupied entries of the (cell, callset) table and of the callset dictionary on the device, then read
  // back only those: rows of {key, count} and of {slot, len, items[gcap]}
  u64 n_agg = h.n_agg, n_cs = h.n_callsets; u32 cw = 4 + c->gcap;
  CK(c->d_scratch.ensure(n_agg * 16 + n_cs * (size_t)cw * 4 + 64, s));
  u64* d_agg = (u64*)c->d_scratch.p; u32* d_cs = (u32*)((char*)c->d_scratch.p + n_agg * 16);
  CK(cudaMemsetAsync(c->d_nout.p, 0, 16, s));
  nbk::launch_compact(t, d_agg, n_agg, d_cs, n_cs, (unsigned long long*)c->d_nout.p, s); c->all_launches += 2;
  // dictionary rows into pinned memory (a pageable vector made this 6 MB copy take a millisecond at C4)
  { const size_t need = (size_t)n_cs * cw * 4 + 64; if (c->h_csr_cap < need) { nb_host_free(c->h_csr); c->h_csr_cap = need + need / 2; c->h_csr = (u32*)nb_host_alloc(c->h_csr_cap); if (!c->h_csr) { c->h_csr_cap = 0; return fail(NB_ERR_CUDA, "pinned host allocation failed"); } } }
  const u32* csr = c->h_csr;
  if (n_cs) CK(cudaMemcpyAsync(c->h_csr, d_cs, n_cs * (size_t)cw * 4, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  if (fstats) ft[2] = fnow();
  // callsets sorted by Vec<String> Ord (utils::sort_score_vector, src/utils.rs:54-59): bytewise on the group names
  const std::vector<u32>& gr = c->lib->group_byte_rank;   // compare ranks, not strings: this sort runs once per job over every callset
  // One team of host threads does the whole host side of this phase (spawned once: sixteen threads per step of it cost more
  // than the steps): rank rows (byte ranks + 1, zero padded: a shorter list sorts first, as Vec<String> Ord has it), buckets
  // by first rank, buckets sorted as 16-byte {prefix of the first ranks, row} pairs (nearly every comparison is one integer
  // compare), then the slot -> callset-id table and the item lists in callset order.  A 40k-transcript library yields 74k
  // callsets; done serially on the dictionary rows this was 11 of the job's 15 ms.
  const u32 gc = c->gcap;
  std::vector<u32> slots(n_cs);
  std::vector<u32>& dense = c->slot_dense;
  if (dense.size() != c->cs_slots) { dense.assign(c->cs_slots, NONE32); c->dense_prev.clear(); }
  for (u32 sl : c->dense_prev) dense[sl] = NONE32;   // only the entries the previous finalize set (the table has callset_slots entries — millions for a big library)
  c->dense_prev.resize(n_cs); c->dense_ids.resize(n_cs); c->cs_off.resize((size_t)n_cs + 1); c->cs_off[0] = 0;
  if (n_cs) {
    const u64 n_groups = gr.size() + 2; const bool r16 = n_groups < 65536;
    const u32 T = n_cs >= 16384 ? std::min<u32>(16, std::max(1u, std::thread::hardware_concurrency())) : 1, NB = T == 1 ? 1 : 8 * T;
    std::unique_ptr<u32[]> km(new u32[(size_t)n_cs * gc]);
    struct PK { u64 k; u32 idx; u32 pad; };
    std::unique_ptr<PK[]> pk(new PK[n_cs]);
    std::vector<u32> bucket(n_cs), bcount((size_t)NB * T, 0), rank_of(n_cs); std::vector<u64> bstart((size_t)NB * T + 1, 0), bbeg(NB + 1, 0), part(T + 1, 0);
    std::atomic<u32> next{0};
    auto less = [&](u32 a, u32 b) { const u32* ka = &km[(size_t)a * gc]; const u32* kb = &km[(size_t)b * gc]; for (u32 x = 0; x < gc; x++) if (ka[x] != kb[x]) return ka[x] < kb[x]; return csr[(size_t)a * cw] < csr[(size_t)b * cw]; };
    HostTeam team(T);
    team.run([&](u32 t) {
      const u64 q0 = n_cs * t / T, q1 = n_cs * (t + 1) / T;
      for (u64 q = q0; q < q1; q++) {
        const u32* r = &csr[(size_t)q * cw]; u32* k = &km[(size_t)q * gc];
        for (u32 x = 0; x < gc; x++) k[x] = x < r[1] ? gr[r[4 + x]] + 1 : 0u;
        const u32 b = (u32)((u64)k[0] * NB / n_groups); bucket[q] = b; bcount[(size_t)t * NB + b]++;
      }
      team.barrier();
      if (t == 0) { u64 at = 0; for (u32 b = 0; b < NB; b++) { bbeg[b] = at; for (u32 u = 0; u < T; u++) { bstart[(size_t)u * NB + b] = at; at += bcount[(size_t)u * NB + b]; } } bbeg[NB] = n_cs; }
      team.barrier();
      for (u64 q = q0; q < q1; q++) {
        const u64 at = bstart[(size_t)t * NB + bucket[q]]++; const u32* k = &km[(size_t)q * gc];
        const u64 a = k[0], b = gc > 1 ? k[1] : 0, c2 = gc > 2 ? k[2] : 0, d = gc > 3 ? k[3] : 0;
        pk[at].k = r16 ? (a << 48) | (b << 32) | (c2 << 16) | d : (a << 32) | b; pk[at].idx = (u32)q; pk[at].pad = 0;
      }
      team.barrier();
      for (u32 b; (b = next.fetch_add(1)) < NB;) std::sort(pk.get() + bbeg[b], pk.get() + bbeg[b + 1], [&](const PK& x, const PK& y) { return x.k != y.k ? x.k < y.k : less(x.idx, y.idx); });
      team.barrier();
      { u64 sum = 0; for (u64 i = q0; i < q1; i++) { const u32 row = pk[i].idx; slots[i] = row; rank_of[row] = (u32)i; sum += csr[(size_t)row * cw + 1]; } part[t + 1] = sum; }
      team.barrier();
      if (t == 0) { for (u32 u = 0; u < T; u++) part[u + 1] += part[u]; c->cs_items.resize(part[T]); }
      // the dictionary rows arrive in (roughly) slot order — k_compact_cs walks the slots — so the table is written in ROW order
      for (u64 q = q0; q < q1; q++) { const u32 sl = csr[(size_t)q * cw]; dense[sl] = rank_of[q]; c->dense_prev[q] = sl; c->dense_ids[rank_of[q]] = sl; }
      team.barrier();
      { u64 at = part[t]; for (u64 i = q0; i < q1; i++) { const u32* r = &csr[(size_t)slots[i] * cw]; for (u32 k = 0; k < r[1]; k++) c->cs_items[at + k] = r[4 + k]; at += r[1]; c->cs_off[i + 1] = at; } }
    });
  }
  auto upload_dense = [&]() -> int { return upload_slot_map(c, s); };
  if (fstats) ft[3] = fnow();
  // rows ordered by (cell, callset): remap to dense callset ids, radix sort and split on the device (kernels.cu), then one
  // copy into pinned memory — the table can hold millions of (cell, callset) rows
  if (dense_cells) {
    // ---- scoped multi-GPU merge: after the dictionary exchange every rank numbers the callsets alike (same sort over the
    // same dictionary), so the per-cell tables add up element-wise: scatter -> all-reduce -> rows by a scan (already ordered)
    const u32 Wm = (shard && c->comm) ? c->cworld : 1;
    const u64 cells_per = (dense_cells + Wm - 1) / Wm;                 // sharded: rank r owns cells [r * cells_per, (r + 1) * cells_per)
    dense_cells = cells_per * Wm;
    const u64 ncs = std::max<u64>(1, slots.size()), nd_all = dense_cells * ncs;
    if (nd_all >= (1ull << 31)) return fail(NB_ERR_UNSUPPORTED, "cells x callsets too large for the dense merge (2^31 entries)");
    u64 nd = nd_all;
    size_t tb = nbk::merge_scan_tmp_bytes(nd);
    CK(c->d_densetab.ensure(nd * 8, s)); CK(c->d_densework.ensure(nd * 16 + tb + 16, s));
    rc = upload_dense(); if (rc) return rc;
    CK(cudaMemsetAsync(c->d_densetab.p, 0, nd * 8, s));
    nbk::launch_merge_dense_fill(t, (const u32*)c->d_dense.p, (unsigned long long*)c->d_densetab.p, ncs, dense_cells, s); c->all_launches++;
    const unsigned long long* d_tab = (const unsigned long long*)c->d_densetab.p; u32 cell_base = 0;
    if (Wm > 1) {   // in place: this rank's chunk of the sums lands where its chunk of the table is
      nd = cells_per * ncs; cell_base = (u32)(c->crank * cells_per); d_tab += (size_t)c->crank * nd;
      rc = dense_reduce_scatter(c, c->d_densetab.p, nd); if (rc) return rc;
    } else { rc = dense_allreduce(c, c->d_densetab.p, nd); if (rc) return rc; }
    unsigned long long* d_flag = (unsigned long long*)c->d_densework.p; unsigned long long* d_prefix = d_flag + nd; void* d_tmp = d_prefix + nd;
    u64 last2[2];   // row count = flag[nd-1] + prefix[nd-1]
    nbk::launch_merge_dense_scan(d_tab, nd, d_flag, d_prefix, d_tmp, tb, s); c->all_launches += 2;
    CK(cudaMemcpyAsync(&last2[0], d_flag + nd - 1, 8, cudaMemcpyDeviceToHost, s)); CK(cudaMemcpyAsync(&last2[1], d_prefix + nd - 1, 8, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    n_agg = last2[0] + last2[1];
    rc = check_device_errors(c); if (rc) return rc;
    if (c->h_rows_cap < n_agg * 16) { nb_host_free(c->h_rows); c->h_rows_cap = n_agg * 16 + n_agg * 4 + 4096; c->h_rows = (u8*)nb_host_alloc(c->h_rows_cap); if (!c->h_rows) { c->h_rows_cap = 0; return fail(NB_ERR_CUDA, "pinned host allocation failed"); } }
    c->n_rows_dev = n_agg;
    if (n_agg) {
      CK(c->d_rowout.ensure(n_agg * 16, s));
      u32* d_scope = (u32*)c->d_rowout.p; u32* d_callset = d_scope + n_agg; i64* d_count = (i64*)((char*)c->d_rowout.p + 8 * n_agg);
      nbk::launch_merge_dense_rows(d_tab, nd, ncs, d_prefix, d_scope, d_callset, d_count, cell_base, s); c->all_launches++;
      CK(cudaMemcpyAsync(c->h_rows, c->d_rowout.p, n_agg * 16, cudaMemcpyDeviceToHost, s));
      CK(cudaStreamSynchronize(s));
    }
    out->n_rows = n_agg; out->row_scope = (u32*)c->h_rows; out->row_callset = (u32*)c->h_rows + n_agg; out->row_count = (i64*)(c->h_rows + 8 * n_agg);
    out->n_callsets = slots.size(); out->callset_off = c->cs_off.data(); out->callset_items = c->cs_items.data();
    out->n_pairs_seen = c->pairs_seen; out->n_unique_keys = h.n_keys; out->n_slots = c->cs_slots; out->slot_to_callset = c->slot_dense.data();
    return NB_OK;
  }
  if (n_agg >= (1ull << 31)) return fail(NB_ERR_UNSUPPORTED, "more than 2^31 (cell, callset) rows");
  if (c->h_rows_cap < n_agg * 16) { nb_host_free(c->h_rows); c->h_rows_cap = n_agg * 16 + n_agg * 4 + 4096; c->h_rows = (u8*)nb_host_alloc(c->h_rows_cap); if (!c->h_rows) { c->h_rows_cap = 0; return fail(NB_ERR_CUDA, "pinned host allocation failed"); } }
  u32* h_scope = (u32*)c->h_rows; u32* h_callset = h_scope + n_agg; i64* h_count = (i64*)(c->h_rows + 8 * n_agg);
  c->n_rows_dev = n_agg;
  if (n_agg) {
    size_t tb = nbk::rows_sort_tmp_bytes(n_agg), work = n_agg * 32;
    CK(c->d_rowwork.ensure(work + tb, s)); CK(c->d_rowout.ensure(n_agg * 16, s));
    rc = upload_dense(); if (rc) return rc;
    u64* d_keys = (u64*)c->d_rowwork.p; i64* d_vals = (i64*)((char*)c->d_rowwork.p + n_agg * 16); void* d_tmp = (char*)c->d_rowwork.p + work;
    u32* d_scope = (u32*)c->d_rowout.p; u32* d_callset = d_scope + n_agg; i64* d_count = (i64*)((char*)c->d_rowout.p + 8 * n_agg);
    nbk::launch_rows_sort(d_agg, n_agg, (const u32*)c->d_dense.p, d_keys, d_vals, d_tmp, tb, d_scope, d_callset, d_count, c->mode == 1 ? 56 : 24, s); c->all_launches += 3;
    CK(cudaMemcpyAsync(c->h_rows, c->d_rowout.p, n_agg * 16, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
  }
  if (c->mode == 1) c->cells_rows = !c->cells_rolled;
  struct { size_t n; size_t size() const { return n; } } rows{(size_t)n_agg};
  out->n_rows = rows.size(); out->row_scope = h_scope; out->row_callset = h_callset; out->row_count = h_count;
  out->n_callsets = slots.size(); out->callset_off = c->cs_off.data(); out->callset_items = c->cs_items.data();
  out->n_pairs_seen = c->pairs_seen; out->n_unique_keys = h.n_keys; out->n_slots = c->cs_slots; out->slot_to_callset = c->slot_dense.data();
  if (fstats) { ft[4] = fnow(); fprintf(stderr, "finalize: fold+counters %.3f ms, compact+D2H %.3f ms, callset sort %.3f ms, rows %.3f ms (%llu rows, %llu callsets, key slots %llu)\n", (ft[1] - ft[0]) * 1e3, (ft[2] - ft[1]) * 1e3, (ft[3] - ft[2]) * 1e3, (ft[4] - ft[3]) * 1e3, (unsigned long long)n_agg, (unsigned long long)n_cs, (unsigned long long)c->key_slots); }
  return NB_OK;
}

int nb_counts_finalize(nb_ctx* c, nb_counts* out) { return finalize_impl(c, out, 0); }

int nb_counts_device_rows(nb_ctx* c, const void** row_scope, const void** row_callset, const void** row_count, uint64_t* n_rows) {
  if (!c || !row_scope || !row_callset || !row_count || !n_rows) return fail(NB_ERR_INVALID, "null argument");
  if (!c->folded && c->mode != 1) return fail(NB_ERR_INVALID, "no finalized counts");
  u64 n = c->n_rows_dev; *n_rows = n;
  *row_scope = c->d_rowout.p; *row_callset = (const u32*)c->d_rowout.p + n; *row_count = (const char*)c->d_rowout.p + 8 * n;
  return NB_OK;
}

int nb_counts_device_slot_map(nb_ctx* c, const void** slot_to_callset, uint64_t* n_slots) {
  if (!c || !slot_to_callset || !n_slots) return fail(NB_ERR_INVALID, "null argument");
  if (!c->folded && c->mode != 1) return fail(NB_ERR_INVALID, "no finalized counts");
  CK(cudaSetDevice(c->device));
  // finalize uploads the table only when it has rows to sort: otherwise fill it here (on the context's stream)
  if (!c->dense_dev) { const int rc = upload_slot_map(c, c->stream); if (rc) return rc; }
  *slot_to_callset = c->d_dense.p; *n_slots = c->slot_dense.size();
  return NB_OK;
}

int nb_counts_reset(nb_ctx* c) {
  if (!c) return fail(NB_ERR_INVALID, "null argument");
  CK(cudaSetDevice(c->device));
  if (c->tables_ready) { CK(cudaStreamSynchronize(c->stream)); c->tables_ready = false; }
  c->mode = -1; c->folded = false; c->pairs_seen = 0; c->have_last = false; c->n_rows_dev = 0; c->cells_rows = c->cells_rolled = false;
  if (c->d_routecur.p) CK(cudaMemsetAsync(c->d_routecur.p, 0, nbk::ROUTE_MAX * 8, c->stream));   // a job abandoned before nb_route_sent must not leak its records into the next one
  return NB_OK;
}

static nbk::CellTable cell_table(nb_ctx* c) {
  return nbk::CellTable{(unsigned long long*)c->d_cellkey.p, (unsigned long long*)c->d_cellumi.p, (unsigned long long*)c->d_cellreads.p, c->cell_slots - 1, (unsigned long long*)c->d_cellctr.p};
}

int nb_cells_roll(nb_ctx* c, const uint32_t* cell_of_scope, uint64_t n_scopes) {
  if (!c || (!cell_of_scope && n_scopes)) return fail(NB_ERR_INVALID, "null argument");
  if (!c->cells_rows) return fail(NB_ERR_INVALID, c->cells_rolled ? "these scopes were already rolled: call nb_counts_reset before the next batch" : "no finalized scoped batch to roll: call nb_counts_finalize first");
  CK(cudaSetDevice(c->device));
  const u64 n = c->n_rows_dev;
  const u32* h_scope = (const u32*)c->h_rows;
  if (n && h_scope[n - 1] >= n_scopes) return fail(NB_ERR_INVALID, "cell_of_scope has fewer entries than the batch has scopes");   // rows are sorted by scope
  for (u64 i = 0; i < n_scopes; i++) if (cell_of_scope[i] == NONE32) return fail(NB_ERR_UNSUPPORTED, "cell ids must be below 2^32 - 1");
  cudaStream_t s = c->stream;
  // persistent ids of this batch's callsets (thousands: a host map is cheap next to the batch)
  const u64 n_cs = c->cs_off.size() - 1;
  c->pid_of_dense.resize(n_cs);
  for (u64 i = 0; i < n_cs; i++) {
    const u32* it = c->cs_items.data() + c->cs_off[i]; const u64 len = c->cs_off[i + 1] - c->cs_off[i];
    auto ins = c->cell_pid.emplace(std::string((const char*)it, len * 4), (u32)(c->pid_off.size() - 1));
    if (ins.second) { c->pid_items.insert(c->pid_items.end(), it, it + len); c->pid_off.push_back(c->pid_items.size()); }
    c->pid_of_dense[i] = ins.first->second;
  }
  if (c->pid_off.size() - 1 >= NONE32) return fail(NB_ERR_UNSUPPORTED, "more than 2^32 - 1 callsets in the per-cell table");
  if (!c->cell_alloc) {
    CK(c->d_cellkey.ensure(c->cell_slots * 8, s)); CK(c->d_cellumi.ensure(c->cell_slots * 8, s)); CK(c->d_cellreads.ensure(c->cell_slots * 8, s)); CK(c->d_cellctr.ensure(16, s));
    CK(cudaMemsetAsync(c->d_cellkey.p, 0, c->cell_slots * 8, s)); CK(cudaMemsetAsync(c->d_cellumi.p, 0, c->cell_slots * 8, s)); CK(cudaMemsetAsync(c->d_cellreads.p, 0, c->cell_slots * 8, s));
    CK(cudaMemsetAsync(c->d_cellctr.p, 0, 16, s));
    c->cell_alloc = true; c->cell_used = 0;
  }
  // every row may add an entry: grow first so that the table stays at most half full (the roll then never runs out of slots)
  if (2 * (c->cell_used + n) > c->cell_slots) {
    u64 ns = c->cell_slots; while (2 * (c->cell_used + n) > ns) ns <<= 1;
    DBuf nk, nu, nr; auto rel = [&]() { nk.release(); nu.release(); nr.release(); };
    auto ck2 = [&](cudaError_t e) { if (e == cudaSuccess) return true; rel(); fail(NB_ERR_CUDA, std::string("cell table growth: ") + cudaGetErrorString(e)); return false; };
    if (!ck2(nk.ensure(ns * 8, s)) || !ck2(nu.ensure(ns * 8, s)) || !ck2(nr.ensure(ns * 8, s))) return NB_ERR_CUDA;
    if (!ck2(cudaMemsetAsync(nk.p, 0, ns * 8, s)) || !ck2(cudaMemsetAsync(nu.p, 0, ns * 8, s)) || !ck2(cudaMemsetAsync(nr.p, 0, ns * 8, s))) return NB_ERR_CUDA;
    nbk::CellTable o = cell_table(c), t = o; t.key = (unsigned long long*)nk.p; t.umis = (unsigned long long*)nu.p; t.reads = (unsigned long long*)nr.p; t.mask = ns - 1;
    nbk::launch_cells_rehash(o, t, s); c->all_launches++;
    if (!ck2(cudaStreamSynchronize(s))) return NB_ERR_CUDA;
    c->d_cellkey.release(); c->d_cellumi.release(); c->d_cellreads.release(); c->d_cellkey = nk; c->d_cellumi = nu; c->d_cellreads = nr; c->cell_slots = ns;
  }
  if (n) {
    CK(c->d_cellscope.ensure(n_scopes * 4 + 16, s)); CK(c->d_cellpid.ensure(n_cs * 4 + 16, s));
    CK(cudaMemcpyAsync(c->d_cellscope.p, cell_of_scope, n_scopes * 4, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(c->d_cellpid.p, c->pid_of_dense.data(), n_cs * 4, cudaMemcpyHostToDevice, s));
    const u32* d_scope = (const u32*)c->d_rowout.p; const u32* d_callset = d_scope + n; const i64* d_count = (const i64*)((const char*)c->d_rowout.p + 8 * n);
    nbk::launch_cells_roll(cell_table(c), d_scope, d_callset, d_count, n, (const u32*)c->d_cellscope.p, (const u32*)c->d_cellpid.p, s); c->all_launches++;
    u64 ctr[2];
    CK(cudaMemcpyAsync(ctr, c->d_cellctr.p, 16, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));   // (also: cell_of_scope and pid_of_dense may be reused once this returns)
    if (ctr[1]) return fail(NB_ERR_OVERFLOW, "per-cell table full");
    c->cell_used = ctr[0];
  }
  c->cell_scopes += n_scopes; c->cells_rows = false; c->cells_rolled = true;
  return NB_OK;
}

int nb_cells_finalize(nb_ctx* c, nb_cell_counts* out) {
  if (!c || !out) return fail(NB_ERR_INVALID, "null argument");
  CK(cudaSetDevice(c->device));
  memset(out, 0, sizeof *out);
  cudaStream_t s = c->stream;
  const u64 n = c->cell_alloc ? c->cell_used : 0, n_pid = c->pid_off.size() - 1;
  // persistent ids -> rank in Vec<String> Ord (utils::sort_score_vector): lexicographic on the groups' byte ranks, as finalize_impl
  const std::vector<u32>& gr = c->lib->group_byte_rank;
  std::vector<u32> order(n_pid), rank_of_pid(n_pid);
  for (u64 p = 0; p < n_pid; p++) order[p] = (u32)p;
  std::sort(order.begin(), order.end(), [&](u32 a, u32 b) {
    const u32* ia = &c->pid_items[c->pid_off[a]]; const u32* ib = &c->pid_items[c->pid_off[b]];
    return std::lexicographical_compare(ia, ia + (c->pid_off[a + 1] - c->pid_off[a]), ib, ib + (c->pid_off[b + 1] - c->pid_off[b]), [&](u32 x, u32 y) { return gr[x] < gr[y]; });
  });
  for (u64 r = 0; r < n_pid; r++) rank_of_pid[order[r]] = (u32)r;
  if (c->h_cellrows_cap < n * 24 + 64) { nb_host_free(c->h_cellrows); c->h_cellrows_cap = n * 24 + n * 6 + 4096; c->h_cellrows = (u8*)nb_host_alloc(c->h_cellrows_cap); if (!c->h_cellrows) { c->h_cellrows_cap = 0; return fail(NB_ERR_CUDA, "pinned host allocation failed"); } }
  u32* h_cell = (u32*)c->h_cellrows; u32* h_callset = h_cell + n; i64* h_umis = (i64*)(h_callset + n); i64* h_reads = h_umis + n;
  if (n) {
    const size_t tb = nbk::cells_sort_tmp_bytes(n), work = n * 16 + n * 8 + 64;
    CK(c->d_cellwork.ensure(work + tb, s)); CK(c->d_cellrows.ensure(n * 24, s)); CK(c->d_cellpid.ensure(n_pid * 4 + 16, s)); CK(c->d_nout.ensure(64, s));
    CK(cudaMemcpyAsync(c->d_cellpid.p, rank_of_pid.data(), n_pid * 4, cudaMemcpyHostToDevice, s));
    CK(cudaMemsetAsync(c->d_nout.p, 0, 8, s));
    u64* d_keys = (u64*)c->d_cellwork.p; u32* d_slots = (u32*)((char*)c->d_cellwork.p + n * 16); void* d_tmp = (char*)c->d_cellwork.p + work;
    nbk::launch_cells_finalize(cell_table(c), n, (const u32*)c->d_cellpid.p, d_keys, d_slots, (unsigned long long*)c->d_nout.p, d_tmp, tb, c->d_cellrows.p, s); c->all_launches += 3;
    CK(cudaMemcpyAsync(c->h_cellrows, c->d_cellrows.p, n * 24, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
  }
  // callsets without a row (interned in some batch's dictionary, never counted) are left out and the ranks closed up
  std::vector<u32> used(n_pid, 0);
  for (u64 i = 0; i < n; i++) used[h_callset[i]] = 1;
  std::vector<u32> new_id(n_pid, NONE32); u32 k = 0;
  c->cc_off.assign(1, 0); c->cc_items.clear();
  for (u64 r = 0; r < n_pid; r++) if (used[r]) {
    new_id[r] = k++; const u32 p = order[r];
    c->cc_items.insert(c->cc_items.end(), c->pid_items.begin() + c->pid_off[p], c->pid_items.begin() + c->pid_off[p + 1]); c->cc_off.push_back(c->cc_items.size());
  }
  for (u64 i = 0; i < n; i++) h_callset[i] = new_id[h_callset[i]];
  out->n_rows = n; out->row_cell = h_cell; out->row_callset = h_callset; out->row_umis = h_umis; out->row_reads = h_reads;
  out->n_callsets = k; out->callset_off = c->cc_off.data(); out->callset_items = c->cc_items.data(); out->n_scopes = c->cell_scopes;
  return NB_OK;
}

int nb_cells_reset(nb_ctx* c) {
  if (!c) return fail(NB_ERR_INVALID, "null argument");
  CK(cudaSetDevice(c->device));
  CK(cudaStreamSynchronize(c->stream));
  for (DBuf* b : {&c->d_cellkey, &c->d_cellumi, &c->d_cellreads}) b->release();
  c->cell_alloc = false; c->cell_used = 0; c->cell_scopes = 0; c->cells_rows = false;
  c->cell_pid.clear(); c->pid_off.assign(1, 0); c->pid_items.clear();
  return NB_OK;
}

int nb_ctx_work_counters(nb_ctx* c, uint64_t* out4) {
  if (!c || !out4) return fail(NB_ERR_INVALID, "null argument");
  if (!c->tables_ready) { out4[0] = out4[1] = out4[2] = out4[3] = 0; return NB_OK; }
  Counters h; int rc = check_device_errors(c, &h); if (rc) return rc;
  out4[0] = h.probes; out4[1] = h.nodes; out4[2] = h.bases; out4[3] = h.colour_elems;
  if (getenv("NB_DEBUG_KMAP")) fprintf(stderr, "k_map dbg: iters=%llu walk_lanes=%llu seed_stages=%llu reseed_lanes=%llu ring_sum=%llu drained_iters=%llu\n", h.dbg[0], h.dbg[1], h.dbg[2], h.dbg[3], h.dbg[4], h.dbg[5]);
  return NB_OK;
}

int nb_ctx_kernel_stats(nb_ctx* c, double* o, int reset) {
  if (!c || !o) return fail(NB_ERR_INVALID, "null argument");
  CK(cudaSetDevice(c->device)); CK(cudaStreamSynchronize(c->stream));
  for (auto& e : c->ev_pending) { float ms = 0; CK(cudaEventElapsedTime(&ms, e.first, e.second)); c->map_ms += ms; c->ev_free.push_back(e); }
  c->ev_pending.clear();
  o[0] = (double)c->map_launches; o[1] = c->map_ms; o[2] = (double)c->map_reads; o[3] = (double)c->all_launches;
  if (reset) { c->map_launches = 0; c->map_ms = 0; c->map_reads = 0; c->all_launches = 0; }
  return NB_OK;
}

int nb_keys_export_count(nb_ctx* c, uint64_t* n) {
  if (!c || !n) return fail(NB_ERR_INVALID, "null argument");
  if (!c->tables_ready) { *n = 0; return NB_OK; }
  CK(cudaSetDevice(c->device));
  CK(cudaMemsetAsync(&((Counters*)c->d_ctr.p)->n_keys, 0, 8, c->stream));
  nbk::launch_count_keys(make_tables(c), c->stream); c->all_launches++;
  Counters h; int rc = check_device_errors(c, &h); if (rc) return rc;
  CK(cudaMemsetAsync(&((Counters*)c->d_ctr.p)->n_keys, 0, 8, c->stream));
  *n = h.n_keys; return NB_OK;
}
int nb_keys_export(nb_ctx* c, void* dev_records, uint64_t cap, uint64_t pair_index_base) {
  if (!c || (!dev_records && cap)) return fail(NB_ERR_INVALID, "null argument");
  if (!c->tables_ready) return NB_OK;
  CK(cudaSetDevice(c->device));
  CK(cudaMemsetAsync(c->d_nout.p, 0, 8, c->stream));
  nbk::launch_keys_export(make_tables(c), dev_records, (unsigned long long*)c->d_nout.p, cap, pair_index_base, c->stream); c->all_launches++;
  u64 n = 0;
  CK(cudaMemcpyAsync(&n, c->d_nout.p, 8, cudaMemcpyDeviceToHost, c->stream)); CK(cudaStreamSynchronize(c->stream));
  if (n > cap) return fail(NB_ERR_INVALID, "record buffer too small for nb_keys_export (nb_keys_export_count gives the size)");
  return NB_OK;
}
// key records grouped by owning rank: counts_out[world] entries per owner, records of owner o start at sum(counts[0..o))
int nb_keys_export_partitioned(nb_ctx* c, void* dev_records, uint64_t cap, uint64_t pair_index_base, uint32_t world, uint64_t* counts_out) {
  if (!c || !counts_out || world == 0 || world > 64 || (!dev_records && cap)) return fail(NB_ERR_INVALID, "bad argument");
  for (u32 i = 0; i < world; i++) counts_out[i] = 0;
  if (!c->tables_ready) return NB_OK;
  CK(cudaSetDevice(c->device));
  cudaStream_t s = c->stream; Tables t = make_tables(c);
  CK(c->d_scratch.ensure(1024, s));
  unsigned long long* d_cnt = (unsigned long long*)c->d_scratch.p;
  CK(cudaMemsetAsync(d_cnt, 0, 64 * 8 * 2, s));
  nbk::launch_keys_count_owner(t, world, d_cnt, s); c->all_launches++;
  std::vector<unsigned long long> cnt(world), cur(world);
  CK(cudaMemcpyAsync(cnt.data(), d_cnt, world * 8, cudaMemcpyDeviceToHost, s)); CK(cudaStreamSynchronize(s));
  u64 tot = 0; for (u32 i = 0; i < world; i++) { cur[i] = tot; tot += cnt[i]; counts_out[i] = cnt[i]; }
  if (tot > cap) return fail(NB_ERR_INVALID, "record buffer too small for nb_keys_export_partitioned");
  CK(cudaMemcpyAsync(d_cnt + 64, cur.data(), world * 8, cudaMemcpyHostToDevice, s));
  nbk::launch_keys_scatter(t, dev_records, d_cnt + 64, pair_index_base, world, s); c->all_launches++;
  CK(cudaStreamSynchronize(s));
  return NB_OK;
}
// callset dictionary as compact rows of (4 + gcap) u32: {slot, len, tag_lo, tag_hi, items[gcap]} so that ranks can merge
// dictionaries; rows == NULL returns the count only
int nb_callsets_export(nb_ctx* c, uint32_t* rows, uint64_t cap_rows, uint64_t* n_out, uint32_t* gcap_out) {
  if (!c || !n_out) return fail(NB_ERR_INVALID, "null argument");
  *n_out = 0; if (gcap_out) *gcap_out = c->gcap;
  if (!c->tables_ready) return NB_OK;
  CK(cudaSetDevice(c->device));
  Counters h; int rc = check_device_errors(c, &h); if (rc) return rc;
  *n_out = h.n_callsets;
  if (!rows) return NB_OK;
  if (cap_rows < h.n_callsets) return fail(NB_ERR_INVALID, "row buffer too small for nb_callsets_export");
  cudaStream_t s = c->stream; u32 cw = 4 + c->gcap;
  CK(c->d_scratch.ensure(h.n_callsets * (size_t)cw * 4 + 64, s));
  CK(cudaMemsetAsync(c->d_nout.p, 0, 16, s));
  nbk::launch_compact(make_tables(c), nullptr, 0, (u32*)c->d_scratch.p, h.n_callsets, (unsigned long long*)c->d_nout.p, s); c->all_launches += 2;
  if (h.n_callsets) CK(cudaMemcpyAsync(rows, c->d_scratch.p, h.n_callsets * (size_t)cw * 4, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  return NB_OK;
}
// insert callsets received from other ranks (rows as exported; device insert with the same tag function) so that
// imported key records resolve and every rank ends up with the same dictionary
int nb_callsets_import(nb_ctx* c, const uint32_t* rows, uint64_t n) {
  if (!c || (n && !rows)) return fail(NB_ERR_INVALID, "null argument");
  CK(cudaSetDevice(c->device));
  if (!c->tables_ready) { int rc = alloc_tables(c); if (rc) return rc; }
  cudaStream_t s = c->stream; u32 cw = 4 + c->gcap;
  CK(c->d_scratch.ensure(n * (size_t)cw * 4 + 64, s));
  if (n) CK(cudaMemcpyAsync(c->d_scratch.p, rows, n * (size_t)cw * 4, cudaMemcpyHostToDevice, s));
  nbk::launch_callsets_import(make_tables(c), (const u32*)c->d_scratch.p, n, s); c->all_launches++;
  return check_device_errors(c);
}
// the same from rows already on this context's device (e.g. inside an all_gather receive buffer): no host round trip and
// no synchronisation; a full dictionary surfaces at nb_counts_finalize
int nb_callsets_import_device(nb_ctx* c, const uint32_t* dev_rows, uint64_t n) {
  if (!c || (n && !dev_rows)) return fail(NB_ERR_INVALID, "null argument");
  CK(cudaSetDevice(c->device));
  if (!c->tables_ready) { int rc = alloc_tables(c); if (rc) return rc; }
  nbk::launch_callsets_import(make_tables(c), dev_rows, n, c->stream); c->all_launches++;
  return NB_OK;
}
// replace this context's whole-run key table by the received partition (records from all ranks whose keys fall in
// this rank's range) so that nb_counts_finalize counts each unique read_key of the partition once
int nb_keys_import(nb_ctx* c, const void* dev_records, uint64_t n) {
  if (!c || (n && !dev_records)) return fail(NB_ERR_INVALID, "null argument");
  CK(cudaSetDevice(c->device));
  if (!c->tables_ready) { int rc = alloc_tables(c); if (rc) return rc; }
  if (c->mode == 1) return fail(NB_ERR_INVALID, "key exchange applies to the whole-run scope only");
  c->mode = 0;
  cudaStream_t s = c->stream;
  if (2 * n > c->key_slots) { c->d_key.release(); c->d_kval.release(); u64 ns = c->key_slots; while (ns < 2 * n) ns <<= 1; c->key_slots = ns; CK(c->d_key.ensure(ns * 16, s)); CK(c->d_kval.ensure(ns * 8, s)); }
  CK(cudaMemsetAsync(c->d_key.p, 0, c->key_slots * 16, s)); CK(cudaMemsetAsync(c->d_kval.p, 0, c->key_slots * 8, s));
  CK(cudaMemsetAsync(&((Counters*)c->d_ctr.p)->n_keys, 0, 8, s)); CK(cudaMemsetAsync(&((Counters*)c->d_ctr.p)->n_live, 0, 8, s));
  nbk::launch_keys_import(make_tables(c), dev_records, n, s); c->all_launches++;
  c->folded = false;
  Counters h; int rc = check_device_errors(c, &h);   // drains the stream: the table now holds exactly the imported partition
  for (int i = 0; i < 4; i++) c->live.pending[i] = false;
  c->live.known = h.n_live; c->live.submitted = c->live.known_at = n;
  return rc;
}

// ---- peer routing of the whole-run scope over NVLink (kernels.cuh Route; DESIGN.md "Multi-GPU")
int nb_route_create(nb_ctx* c, uint32_t world, uint64_t records_per_peer, void* ipc_handle_out) {
  if (!c || records_per_peer == 0 || world < 2 || world > (u32)nbk::ROUTE_MAX) return fail(NB_ERR_INVALID, "bad argument (2 <= world <= 16)");
  static_assert(sizeof(cudaIpcMemHandle_t) == NB_ROUTE_HANDLE_BYTES, "IPC handle size");
  CK(cudaSetDevice(c->device));
  if (c->route_on) return fail(NB_ERR_INVALID, "routes are attached; call nb_route_detach first");
  CK(cudaStreamSynchronize(c->stream));
  size_t bytes = (size_t)world * records_per_peer * sizeof(nbk::KeyRec);
  if (c->d_inbox.p && c->d_inbox.cap < bytes) c->d_inbox.release();
  if (!c->d_inbox.p) CK(c->d_inbox.ensure(bytes, c->stream));
  c->inbox_cap = records_per_peer; c->inbox_world = world;
  CK(c->d_routecur.ensure(nbk::ROUTE_MAX * 8, c->stream));
  CK(cudaMemsetAsync(c->d_routecur.p, 0, nbk::ROUTE_MAX * 8, c->stream)); CK(cudaStreamSynchronize(c->stream));
  if (ipc_handle_out) { cudaIpcMemHandle_t h; CK(cudaIpcGetMemHandle(&h, c->d_inbox.p)); memcpy(ipc_handle_out, &h, sizeof h); }
  return NB_OK;
}
static int route_fill(nb_ctx* c, u32 world, u32 rank, void* const* bases, u64 pair_index_base) {
  nbk::Route& r = c->route; memset(&r, 0, sizeof r);
  r.world = world; r.rank = rank; r.pair_base = pair_index_base; r.cap = c->inbox_cap;
  for (u32 i = 0; i < world; i++) r.inbox[i] = (nbk::KeyRec*)bases[i] + (size_t)rank * c->inbox_cap;   // this rank's region in rank i's inbox
  r.cursor = (unsigned long long*)c->d_routecur.p;
  c->route_on = true;
  return NB_OK;
}
int nb_route_attach_ipc(nb_ctx* c, uint32_t world, uint32_t rank, const void* handles, uint64_t pair_index_base) {
  if (!c || !handles || rank >= world) return fail(NB_ERR_INVALID, "bad argument");
  if (!c->d_inbox.p || c->inbox_world != world) return fail(NB_ERR_INVALID, "nb_route_create with the same world first");
  if (c->route_on) return fail(NB_ERR_INVALID, "routes already attached");
  CK(cudaSetDevice(c->device));
  void* bases[nbk::ROUTE_MAX];
  for (u32 i = 0; i < world; i++) {
    if (i == rank) { bases[i] = c->d_inbox.p; continue; }
    cudaIpcMemHandle_t h; memcpy(&h, (const char*)handles + (size_t)i * sizeof h, sizeof h);
    void* q = nullptr; cudaError_t e = cudaIpcOpenMemHandle(&q, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
      cudaGetLastError();
      for (void* o : c->ipc_opened) cudaIpcCloseMemHandle(o);
      c->ipc_opened.clear();
      return fail(NB_ERR_CUDA, std::string("cudaIpcOpenMemHandle failed for rank ") + std::to_string(i) + ": " + cudaGetErrorString(e));
    }
    c->ipc_opened.push_back(q); bases[i] = q;
  }
  return route_fill(c, world, rank, bases, pair_index_base);
}
int nb_route_attach_ctx(nb_ctx* c, uint32_t world, uint32_t rank, nb_ctx* const* peers, uint64_t pair_index_base) {
  if (!c || !peers || rank >= world || world > (u32)nbk::ROUTE_MAX || peers[rank] != c) return fail(NB_ERR_INVALID, "bad argument (peers[rank] must be this context)");
  if (c->route_on) return fail(NB_ERR_INVALID, "routes already attached");
  CK(cudaSetDevice(c->device));
  void* bases[nbk::ROUTE_MAX];
  for (u32 i = 0; i < world; i++) {
    if (!peers[i] || !peers[i]->d_inbox.p || peers[i]->inbox_world != world || peers[i]->inbox_cap != c->inbox_cap)
      return fail(NB_ERR_INVALID, "every peer needs nb_route_create with the same world and records_per_peer first");
    if (peers[i]->device != c->device) {
      int can = 0; CK(cudaDeviceCanAccessPeer(&can, c->device, peers[i]->device));
      if (!can) return fail(NB_ERR_CUDA, "no peer access between the devices of two routed contexts");
      cudaError_t e = cudaDeviceEnablePeerAccess(peers[i]->device, 0);
      if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return fail(NB_ERR_CUDA, cudaGetErrorString(e));
      cudaGetLastError();
    }
    bases[i] = peers[i]->d_inbox.p;
  }
  return route_fill(c, world, rank, bases, pair_index_base);
}
int nb_route_set_pair_base(nb_ctx* c, uint64_t pair_index_base) { if (!c) return fail(NB_ERR_INVALID, "null argument"); c->route.pair_base = pair_index_base; return NB_OK; }
int nb_route_detach(nb_ctx* c) {
  if (!c) return fail(NB_ERR_INVALID, "null argument");
  CK(cudaSetDevice(c->device)); CK(cudaStreamSynchronize(c->stream));
  for (void* q : c->ipc_opened) cudaIpcCloseMemHandle(q);
  c->ipc_opened.clear(); c->route_on = false; memset(&c->route, 0, sizeof c->route);
  return NB_OK;
}
// Records this rank has stored into each peer's inbox since the last call (sent[world], sent[rank] = 0); waits for the
// batches submitted so far and restarts the cursors for the next job.  The host hands sent[o] to rank o (one all_gather).
int nb_route_sent(nb_ctx* c, uint64_t* sent) {
  if (!c || !sent) return fail(NB_ERR_INVALID, "null argument");
  if (!c->route_on) return fail(NB_ERR_INVALID, "routes are not attached");
  CK(cudaSetDevice(c->device));
  unsigned long long h[nbk::ROUTE_MAX];
  CK(cudaMemcpyAsync(h, c->d_routecur.p, sizeof h, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaMemsetAsync(c->d_routecur.p, 0, sizeof h, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  for (u32 i = 0; i < c->route.world; i++) {
    if (h[i] > c->inbox_cap) return fail(NB_ERR_OVERFLOW, "routing inbox region overflow: create the routes with more records_per_peer");
    sent[i] = h[i];
  }
  return NB_OK;
}
// Merge the records peers stored into this context's inbox (counts[r] from rank r, counts[rank] ignored) into its key
// table with the same "later duplicate wins" rule as k_pair.  Every peer must have finished its batches of this job AND
// this rank must know it (the collective that carried the counts does); the callsets the records name must already be in
// this context's dictionary (nb_callsets_import of the peers' rows first).
int nb_route_import(nb_ctx* c, const uint64_t* counts, uint64_t* n_imported) {
  if (!c || !counts) return fail(NB_ERR_INVALID, "null argument");
  if (!c->route_on) return fail(NB_ERR_INVALID, "routes are not attached");
  CK(cudaSetDevice(c->device));
  if (!c->tables_ready) { int rc = alloc_tables(c); if (rc) return rc; }
  if (c->mode == 1) return fail(NB_ERR_INVALID, "routing applies to the whole-run scope only");
  c->mode = 0;
  cudaStream_t s = c->stream;
  u64 n = 0;
  for (u32 r = 0; r < c->route.world; r++) if (r != c->route.rank) { if (counts[r] > c->inbox_cap) return fail(NB_ERR_OVERFLOW, "routing inbox region overflow: create the routes with more records_per_peer"); n += counts[r]; }
  { int rc = ensure_key_capacity(c, n); if (rc) return rc; }
  Tables t = make_tables(c);
  for (u32 r = 0; r < c->route.world; r++) if (r != c->route.rank && counts[r]) {
    nbk::launch_keys_import(t, (const nbk::KeyRec*)c->d_inbox.p + (size_t)r * c->inbox_cap, counts[r], s); c->all_launches++;
  }
  c->folded = false;
  if (n_imported) *n_imported = n;
  return NB_OK;   // device-side errors (table full, unknown callset) surface at nb_counts_finalize
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------ multi-GPU merge over NCCL
// SURVEY.md §8(b) `nb_counts_allreduce(nb_ctx*, ncclComm_t)`, §8(e).  The reference's only parallel driver is N-1 consumer
// threads behind one producer (src/process/bam.rs:183-226); its multi-GPU counterpart is one context per GPU whose tables are
// merged here, inside the library, on the context's stream: NCCL is called from C++ (libnccl.so.2 resolved at run time, so a
// single-GPU host needs no NCCL), every import kernel reads its sizes from the gathered headers on the device, and the host
// waits once per job (the header read-back that sizes the key table) before the usual finalize.
struct NcclApi {
  ncclResult_t (*GetUniqueId)(ncclUniqueId*);
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int);
  ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*);
  ncclResult_t (*CommDestroy)(ncclComm_t);
  ncclResult_t (*CommCount)(const ncclComm_t, int*);
  ncclResult_t (*CommUserRank)(const ncclComm_t, int*);
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t);
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t);
  ncclResult_t (*ReduceScatter)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t);
  ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t);
  ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t);
  ncclResult_t (*GroupStart)();
  ncclResult_t (*GroupEnd)();
  const char* (*GetErrorString)(ncclResult_t);
};
static const NcclApi* nccl_api() {
  static NcclApi api; static int state = 0;   // 0 untried, 1 ok, -1 unavailable
  if (state == 0) {
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);   // the copy already in the process (e.g. PyTorch's) when there is one
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    bool ok = h != nullptr;
    auto sym = [&](const char* n) { void* p = ok ? dlsym(h, n) : nullptr; if (!p) ok = false; return p; };
    *(void**)&api.GetUniqueId = sym("ncclGetUniqueId"); *(void**)&api.CommInitRank = sym("ncclCommInitRank"); *(void**)&api.CommInitAll = sym("ncclCommInitAll");
    *(void**)&api.CommDestroy = sym("ncclCommDestroy"); *(void**)&api.CommCount = sym("ncclCommCount"); *(void**)&api.CommUserRank = sym("ncclCommUserRank");
    *(void**)&api.AllGather = sym("ncclAllGather"); *(void**)&api.AllReduce = sym("ncclAllReduce"); *(void**)&api.ReduceScatter = sym("ncclReduceScatter"); *(void**)&api.Send = sym("ncclSend"); *(void**)&api.Recv = sym("ncclRecv");
    *(void**)&api.GroupStart = sym("ncclGroupStart"); *(void**)&api.GroupEnd = sym("ncclGroupEnd"); *(void**)&api.GetErrorString = sym("ncclGetErrorString");
    state = ok ? 1 : -1;
  }
  return state == 1 ? &api : nullptr;
}
#define NCK(x) do { ncclResult_t r_ = (x); if (r_ != ncclSuccess) return fail(NB_ERR_CUDA, std::string(#x) + ": " + N->GetErrorString(r_)); } while (0)
#define NEED_NCCL() const NcclApi* N = nccl_api(); if (!N) return fail(NB_ERR_CUDA, "libnccl.so.2 could not be loaded: the multi-GPU merge needs NCCL")

static int dense_allreduce(nb_ctx* c, void* dense, u64 n) {
  if (!c->comm || c->cworld < 2) return NB_OK;
  NEED_NCCL();
  NCK(N->AllReduce(dense, dense, n, ncclUint64, ncclSum, c->comm, c->stream));
  return NB_OK;
}
// in place: rank r's chunk of the element-wise sums replaces elements [r * chunk, (r + 1) * chunk) of its own table
static int dense_reduce_scatter(nb_ctx* c, void* dense, u64 chunk) {
  if (!c->comm || c->cworld < 2) return NB_OK;
  NEED_NCCL();
  NCK(N->ReduceScatter(dense, (unsigned long long*)dense + (size_t)c->crank * chunk, chunk, ncclUint64, ncclSum, c->comm, c->stream));
  return NB_OK;
}

extern "C" {

int nb_comm_unique_id(void* id128_out) {
  if (!id128_out) return fail(NB_ERR_INVALID, "null argument");
  NEED_NCCL();
  static_assert(sizeof(ncclUniqueId) == NB_COMM_ID_BYTES, "ncclUniqueId size");
  ncclUniqueId id; NCK(N->GetUniqueId(&id)); memcpy(id128_out, &id, sizeof id);
  return NB_OK;
}
static int comm_adopt(nb_ctx* c, ncclComm_t comm, bool own) {
  NEED_NCCL();
  int w = 0, r = 0; NCK(N->CommCount(comm, &w)); NCK(N->CommUserRank(comm, &r));
  if (w < 1 || w > nbk::ROUTE_MAX) return fail(NB_ERR_UNSUPPORTED, "communicators of 1..16 ranks are supported");
  c->comm = comm; c->own_comm = own; c->cworld = (u32)w; c->crank = (u32)r;
  if (!c->h_hdr) { c->h_hdr = (u64*)nb_host_alloc(8 * (size_t)nbk::ROUTE_MAX * (nbk::MERGE_HDR1_WORDS + 2)); if (!c->h_hdr) return fail(NB_ERR_CUDA, "pinned host allocation failed"); }
  return NB_OK;
}
int nb_comm_init_rank(nb_ctx* c, const void* id128, uint32_t world, uint32_t rank) {
  if (!c || !id128 || rank >= world) return fail(NB_ERR_INVALID, "bad argument");
  if (c->comm) return fail(NB_ERR_INVALID, "the context already has a communicator (nb_comm_free first)");
  NEED_NCCL();
  CK(cudaSetDevice(c->device));
  ncclUniqueId id; memcpy(&id, id128, sizeof id);
  ncclComm_t comm = nullptr; NCK(N->CommInitRank(&comm, (int)world, id, (int)rank));
  return comm_adopt(c, comm, true);
}
int nb_comm_attach(nb_ctx* c, void* nccl_comm) {
  if (!c || !nccl_comm) return fail(NB_ERR_INVALID, "null argument");
  if (c->comm) return fail(NB_ERR_INVALID, "the context already has a communicator (nb_comm_free first)");
  return comm_adopt(c, (ncclComm_t)nccl_comm, false);
}
int nb_comm_init_all(nb_ctx* const* ctxs, uint32_t n) {
  if (!ctxs || n < 1 || n > (uint32_t)nbk::ROUTE_MAX) return fail(NB_ERR_INVALID, "bad argument (1..16 contexts)");
  NEED_NCCL();
  int devs[nbk::ROUTE_MAX]; ncclComm_t comms[nbk::ROUTE_MAX];
  for (u32 i = 0; i < n; i++) { if (!ctxs[i] || ctxs[i]->comm) return fail(NB_ERR_INVALID, "null context, or a context that already has a communicator"); devs[i] = ctxs[i]->device; }
  for (u32 i = 0; i < n; i++) for (u32 j = 0; j < i; j++) if (devs[i] == devs[j]) return fail(NB_ERR_INVALID, "nb_comm_init_all needs one context per distinct GPU");
  NCK(N->CommInitAll(comms, (int)n, devs));
  for (u32 i = 0; i < n; i++) { int rc = comm_adopt(ctxs[i], comms[i], true); if (rc) return rc; }
  return NB_OK;
}
int nb_comm_free(nb_ctx* c) {
  if (!c) return fail(NB_ERR_INVALID, "null argument");
  if (c->comm && c->own_comm) { const NcclApi* N = nccl_api(); cudaSetDevice(c->device); cudaStreamSynchronize(c->stream); if (N) N->CommDestroy(c->comm); }
  c->comm = nullptr; c->own_comm = false; c->cworld = 1; c->crank = 0;
  return NB_OK;
}
int nb_comm_info(nb_ctx* c, uint32_t* world, uint32_t* rank) {
  if (!c) return fail(NB_ERR_INVALID, "null argument");
  if (world) *world = c->comm ? c->cworld : 1; if (rank) *rank = c->comm ? c->crank : 0;
  return NB_OK;
}

// one process per GPU: inbox + IPC handles gathered over the communicator + peers' inboxes opened, in one call
int nb_route_setup(nb_ctx* c, uint64_t records_per_peer, uint64_t pair_index_base) {
  if (!c) return fail(NB_ERR_INVALID, "null argument");
  if (!c->comm || c->cworld < 2) return fail(NB_ERR_INVALID, "nb_route_setup needs a communicator of >= 2 ranks (nb_comm_init_rank)");
  NEED_NCCL();
  u8 mine[NB_ROUTE_HANDLE_BYTES];
  int rc = nb_route_create(c, c->cworld, records_per_peer, mine); if (rc) return rc;
  cudaStream_t s = c->stream;
  CK(c->d_blk1.ensure(NB_ROUTE_HANDLE_BYTES, s)); CK(c->d_all1.ensure((size_t)NB_ROUTE_HANDLE_BYTES * c->cworld, s));
  CK(cudaMemcpyAsync(c->d_blk1.p, mine, sizeof mine, cudaMemcpyHostToDevice, s));
  NCK(N->AllGather(c->d_blk1.p, c->d_all1.p, sizeof mine, ncclChar, c->comm, s));
  std::vector<u8> all((size_t)NB_ROUTE_HANDLE_BYTES * c->cworld);
  CK(cudaMemcpyAsync(all.data(), c->d_all1.p, all.size(), cudaMemcpyDeviceToHost, s)); CK(cudaStreamSynchronize(s));
  // every rank must end up routed or none: agree on the outcome (1 = attached) with a tiny all-reduce
  int ok = nb_route_attach_ipc(c, c->cworld, c->crank, all.data(), pair_index_base) == NB_OK;
  std::string why = ok ? std::string() : std::string(nb_last_error());
  unsigned long long flag = ok ? 1ULL : 0ULL;
  CK(cudaMemcpyAsync(c->d_blk1.p, &flag, 8, cudaMemcpyHostToDevice, s));
  NCK(N->AllReduce(c->d_blk1.p, c->d_blk1.p, 1, ncclUint64, ncclMin, c->comm, s));
  CK(cudaMemcpyAsync(&flag, c->d_blk1.p, 8, cudaMemcpyDeviceToHost, s)); CK(cudaStreamSynchronize(s));
  if (!flag) { if (ok) nb_route_detach(c); return fail(NB_ERR_CUDA, ok ? "peer routing unavailable on another rank" : "peer routing unavailable: " + why); }
  return NB_OK;
}

// dictionary exchange shared by both merges: all-gather of {k, sent[], k rows} blocks (capacity: a ratchet all ranks raise
// alike), headers to the host (the one wait of the merge), peers' rows imported straight out of the gather buffer.
// recv[r] = records rank r stored into this rank's inbox; ksum = sum of the ranks' dictionary sizes.
static int merge_dictionaries(nb_ctx* c, const unsigned long long* d_sent, u64* recv, u64* ksum) {
  NEED_NCCL();
  cudaStream_t s = c->stream; const u32 W = c->cworld, cw = 4 + c->gcap; const size_t hdr_b = 8 * (size_t)nbk::MERGE_HDR1_WORDS;
  for (;;) {
    const u64 cap = c->merge_cap; const size_t blk_b = (hdr_b + cap * cw * 4 + 15) & ~(size_t)15;
    CK(c->d_blk1.ensure(blk_b, s)); CK(c->d_all1.ensure(blk_b * W, s));
    CK(cudaMemsetAsync(c->d_nout.p, 0, 16, s));
    nbk::launch_compact(make_tables(c), nullptr, 0, (u32*)((char*)c->d_blk1.p + hdr_b), cap, (unsigned long long*)c->d_nout.p, s); c->all_launches += 2;
    nbk::launch_merge_hdr1((u64*)c->d_blk1.p, (const unsigned long long*)c->d_nout.p + 1, d_sent, W, s); c->all_launches++;
    NCK(N->AllGather(c->d_blk1.p, c->d_all1.p, blk_b, ncclChar, c->comm, s));
    CK(cudaMemcpy2DAsync(c->h_hdr, hdr_b, c->d_all1.p, blk_b, hdr_b, W, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    u64 kmax = 0; *ksum = 0;
    for (u32 r = 0; r < W; r++) { u64 k = c->h_hdr[r * nbk::MERGE_HDR1_WORDS]; kmax = std::max(kmax, k); *ksum += k; recv[r] = c->h_hdr[r * nbk::MERGE_HDR1_WORDS + 1 + c->crank]; }
    if (kmax <= cap) { nbk::launch_merge_import_callsets(make_tables(c), c->d_all1.p, blk_b, cap, W, c->crank, s); c->all_launches++; return NB_OK; }
    while (c->merge_cap < kmax) c->merge_cap *= 2;   // every rank sees the same sizes: every rank repeats with the same capacity
  }
}

int nb_merge_whole_run(nb_ctx* c, nb_counts* out) {
  if (!c || !out) return fail(NB_ERR_INVALID, "null argument");
  if (!c->comm || c->cworld < 2) return nb_counts_finalize(c, out);
  NEED_NCCL();
  CK(cudaSetDevice(c->device));
  if (!c->tables_ready) { int rc = alloc_tables(c); if (rc) return rc; }
  if (c->mode == 1) return fail(NB_ERR_INVALID, "nb_merge_whole_run applies to the whole-run scope (use nb_merge_scoped for scoped batches)");
  if (c->folded) return fail(NB_ERR_INVALID, "counts were finalized; call nb_counts_reset first");
  if (!c->route_on) return fail(NB_ERR_INVALID, "nb_merge_whole_run needs peer routing (nb_route_setup / nb_route_attach_ctx): key records travel inside k_pair");
  c->mode = 0;
  cudaStream_t s = c->stream; const u32 W = c->cworld;
  static const bool mstats = getenv("NB_MERGE_STATS") != nullptr; double mt[8]; int mi = 0;   // tuning aid: phase times with a stream sync at every mark
  auto mark = [&]() { if (!mstats) return; cudaStreamSynchronize(s); timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); mt[mi++] = ts.tv_sec + ts.tv_nsec * 1e-9; };
  mark();
  u64 recv[nbk::ROUTE_MAX], ksum = 0;
  int rc = merge_dictionaries(c, (const unsigned long long*)c->d_routecur.p, recv, &ksum); if (rc) return rc;
  mark();
  // ---- this rank's inbox: the records the peers' k_pair stored while they aligned (the all-gather above is the barrier that
  // says every peer's last batch is complete), merged with the same "later duplicate wins" rule
  u64 n_in = 0, n_max = 0;
  // (every rank looks at every rank's counts: an overflow anywhere fails the merge on ALL ranks, before the next collective —
  // a rank that left alone would leave the others waiting in it)
  for (u32 r = 0; r < W; r++) for (u32 o = 0; o < W; o++) if (r != o && c->h_hdr[r * nbk::MERGE_HDR1_WORDS + 1 + o] > c->inbox_cap) return fail(NB_ERR_OVERFLOW, "routing inbox region overflow: create the routes with more records_per_peer");
  for (u32 r = 0; r < W; r++) if (r != c->crank) { n_in += recv[r]; n_max = std::max(n_max, recv[r]); }
  rc = ensure_key_capacity(c, n_in); if (rc) return rc;
  Tables t = make_tables(c);
  const size_t blk_b = (8 * (size_t)nbk::MERGE_HDR1_WORDS + c->merge_cap * (4 + c->gcap) * 4 + 15) & ~(size_t)15;
  nbk::launch_merge_import_inbox(t, c->d_inbox.p, c->inbox_cap, n_max, c->d_all1.p, blk_b, W, c->crank, s); c->all_launches++;
  CK(cudaMemsetAsync(c->d_routecur.p, 0, nbk::ROUTE_MAX * 8, s));   // the next job's records start at the head of the regions
  mark();
  // ---- fold the keys this rank owns, then exchange {callset tag, count} rows: every rank ends with the job's counts
  nbk::launch_fold(t, nullptr, 0, s); c->all_launches++; c->folded = true;
  const u64 cap2 = std::max<u64>(1, std::min<u64>(ksum, c->cs_slots)), w2 = 2 + 2 * cap2;
  CK(c->d_blk2.ensure(w2 * 8, s)); CK(c->d_all2.ensure(w2 * 8 * W, s));
  CK(cudaMemsetAsync(c->d_blk2.p, 0, 16, s));
  nbk::launch_merge_export_counts(t, (u64*)c->d_blk2.p, cap2, s); c->all_launches++;
  NCK(N->AllGather(c->d_blk2.p, c->d_all2.p, w2 * 8, ncclChar, c->comm, s));
  CK(cudaMemsetAsync(c->d_aggkey.p, 0, c->agg_slots * 8, s)); CK(cudaMemsetAsync(c->d_aggcnt.p, 0, c->agg_slots * 8, s));
  CK(cudaMemsetAsync(&((Counters*)c->d_ctr.p)->n_keys, 0, 8, s)); CK(cudaMemsetAsync(&((Counters*)c->d_ctr.p)->n_agg, 0, 8, s));
  nbk::launch_merge_import_counts(t, (const u64*)c->d_all2.p, w2, cap2, W, s); c->all_launches++;
  mark();
  rc = finalize_impl(c, out, 0);   // (folded: no second fold) counters, dictionary order, rows — as on one GPU
  mark();
  if (mstats && c->crank == 0) fprintf(stderr, "nb_merge_whole_run: wait for the stream (alignment) %.3f ms | dictionaries all-gather + header read-back %.3f | inbox import (%llu records) %.3f | fold + counts all-gather + import %.3f | finalize %.3f\n",
                                       0.0, (mt[1] - mt[0]) * 1e3, (unsigned long long)n_in, (mt[2] - mt[1]) * 1e3, (mt[3] - mt[2]) * 1e3, (mt[4] - mt[3]) * 1e3);
  return rc;
}

static int merge_scoped_impl(nb_ctx* c, uint64_t n_cells, nb_counts* out, bool shard);
int nb_merge_scoped(nb_ctx* c, uint64_t n_cells, nb_counts* out) { return merge_scoped_impl(c, n_cells, out, false); }
int nb_merge_scoped_sharded(nb_ctx* c, uint64_t n_cells, nb_counts* out) { return merge_scoped_impl(c, n_cells, out, true); }
static int merge_scoped_impl(nb_ctx* c, uint64_t n_cells, nb_counts* out, bool shard) {
  if (!c || !out || n_cells == 0) return fail(NB_ERR_INVALID, "bad argument");
  if (!c->comm || c->cworld < 2) return nb_counts_finalize(c, out);
  CK(cudaSetDevice(c->device));
  if (!c->tables_ready) { int rc = alloc_tables(c); if (rc) return rc; }
  if (c->mode == 0) return fail(NB_ERR_INVALID, "nb_merge_scoped applies to scoped batches");
  c->mode = 1;
  u64 recv[nbk::ROUTE_MAX], ksum = 0;
  int rc = merge_dictionaries(c, nullptr, recv, &ksum); if (rc) return rc;
  // unique keys of the job = sum over ranks (scopes are disjoint): rides in the dense all-reduce's last element? no — one more tiny all-reduce
  NEED_NCCL();
  NCK(N->AllReduce(&((Counters*)c->d_ctr.p)->n_keys, &((Counters*)c->d_ctr.p)->n_keys, 1, ncclUint64, ncclSum, c->comm, c->stream));
  return finalize_impl(c, out, n_cells, shard);
}

}  // extern "C"
