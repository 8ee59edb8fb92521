// kernels.cuh — device-side data layout and the hand-written sm_100a kernels of the alignment hot path.
//
//   K0 k_pack        ASCII -> 2-bit words (word-major), optional reverse-complement      (DnaString::from_acgt_bytes,
//                    /root/reference/src/parse/fastq.rs:36, src/process/bam.rs:407-415)
//   K1 k_trim        MAXINFO trim length from raw Phred bytes, exact i64                 (src/align.rs:866-925)
//   K2 k_map         length/entropy gates + seed-and-walk pseudo-alignment + colour intersection + thresholds
//                    (src/align.rs:945-989, Pseudoaligner::map_read_with_mismatch [SURVEY.md App. B], src/filter/align.rs:4-45)
//   K3 k_pair        pair validity, orientation / strand / intersect logic, group roll-up, max-hits, callset interning,
//                    128-bit read_key and de-duplication insert                          (src/align.rs:144-375, 576-685, 732-864)
//   K4 k_fold        one vote per unique read_key -> (cell, callset) histogram            (src/align.rs:440-449, 245-251)
// Tensor cores are not used: nothing here is a dense contraction (HBM/L2-latency bound integer work).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

typedef uint8_t u8;
typedef uint16_t u16;
typedef uint32_t u32;
typedef uint64_t u64;
typedef int64_t i64;

namespace nbk {

constexpr int K = 30;
constexpr u64 KMASK = (1ULL << 60) - 1;
constexpr u32 NONE32 = 0xFFFFFFFFu;
constexpr u32 CS_NONE = 0xFFFFFFu;        // 24-bit "no callset" in the key-table value
constexpr int GL_MAX = 64;                 // per-thread group list capacity (max(discard_multi_hits, max_hits_to_report)+1 <= 64)
constexpr int ENT_NMAX = 1024;             // longest read the entropy table covers

struct DevIndex {
  const u64* ptab; u32 n_pbuckets;                   // probe table (khash.h): bucket b = {key0, key1, value0, value1}, one 32-byte sector / one 256-bit load
  const u64* bloom; u32 bloom_words; u32 bloom_k;    // blocked Bloom prefilter in front of it (64-bit words, k bits per k-mer)
  u32 hbm;                                           // the table cannot live in L2: kernels use the L2 eviction hints (filter evict_last, buckets evict_first)
  const u64* unitig;
  const uint4* node;      // {start_lo, len, colour, lext | rext<<4 | start_hi<<8}
  const uint4* walk;      // 64-byte record per unitig, everything one forward step needs in one DRAM burst / two L2 sectors:
                          // [0] node {start_lo, len, colour, exts_hi}  [1] right edges by base  [2] col_meta of its colour  [3] its bases [K, K + 64) (2 x u64)
  const uint4* ledge;
  const u32* col_off; const u32* col_ids;
  const uint4* col_meta;  // {uni_off, uni_size (0: none), mask_lo, mask_hi} per colour (host.hpp nb_index::col_meta)
};
struct DevLib {
  const u32* row_fid; const u8* row_rev; const u32* row_of; const u32* feat_group; u32 n_rows;
  // per row, derived at context creation so that the pair stage answers "is row x in this class" and "which row is x's other
  // orientation" with one load each instead of a binary search / three dependent loads:
  const u32* row_uoff; const u8* row_upos;   // the component (universe) list the row belongs to: its offset in col_ids (NONE32: none) and the row's position in it
  const u32* row_other;                      // row_of[2 * fid + (1 - rev)]
  const u32* row_group;                      // feat_group[row_fid[row]]
};
struct DevCfg {
  double score_percent; u32 score_threshold; u32 num_mismatches;
  int discard_nonzero_mismatch, discard_multiple_matches, require_valid_pair, intersect_level, strand_filter, no_dedup;
  u32 discard_multi_hits, max_hits, gcap, min_read_len;
};
// device-side error bits (Counters::err)
enum { E_ARENA = 1, E_CS_FULL = 2, E_KEY_FULL = 4, E_FEATURE = 8, E_AGG_FULL = 16, E_GCAP = 32, E_INBOX_FULL = 64, E_CS_UNKNOWN = 128 };
struct Counters {
  unsigned long long arena_top, queue, seeded_n, wqueue;   // all four zeroed before every map launch (seeded_n / wqueue: k_seed -> k_walk list)
  unsigned long long n_keys; unsigned long long n_callsets; unsigned long long n_agg;
  unsigned long long probes, nodes, bases, colour_elems;   // work counters (roofline numerator cross-check)
  unsigned int err; unsigned int pad;
  unsigned long long dbg[8];   // k_map<COUNT_WORK=1> only: loop iterations, lanes walking, seed stages, lanes re-seeding, ...
  unsigned long long n_live;   // whole-run scope: unique read_keys in the table right now (every insert path counts its new keys, one atomic per warp)
};

// internal per-read record (32 B)
struct ReadRes {
  u32 hdr;        // reason | pass<<8 | big<<9 | skip<<10 | uni<<11 (the class is a bitmap over a component list)
  u16 score, mm;
  u32 ec_len;     // elements in the raw equivalence class
  u32 bsize;      // mask mode: size of the base colour list
  u64 ref;        // mask mode: offset of the base colour in col_ids; big mode: offset in the arena
  u64 mask;       // mask mode: surviving elements of the base colour
};
struct PairRes { u32 callset; u8 triage, fr1, fr2, insertable; u64 key_lo, key_hi; };  // == nb_pair_result

struct BatchDev {
  u64 n_pairs; u32 sides; u32 n_reads; u32 W;             // W words per read incl. one zero pad word
  const u8* a[2]; const u64* off[2]; const u8* q[2]; const u8* flags[2]; const u32* scope; const u32* cell;
  u32 enc; u32 pad_; const u32* len[2];                  // nb_batch.encoding (0 ASCII, 1 2-bit, 2 BAM 4-bit: off[] then counts bases) and optional explicit read lengths
  u64* pk; u32* len_full; u32* len_trim;                  // pk[ri * W + w] (read-major), ri = p*sides + side
  ReadRes* rres; PairRes* pres;
  uint4* seeded;                                         // k_seed -> k_walk: {read, seed position, node, offset} of every read that found a seed
  u64* pslot; PairRes* pres2;                            // scoped batches: key slot per pair, per-key resolved records
  u64 order_base;
};

struct Tables {
  // callset dictionary
  u64* cs_tag; u32* cs_len; u32* cs_items; u32 cs_mask; u32 gcap;
  // de-duplication key table (128-bit keys, CAS128) and value = order<<24 | callset slot
  ulonglong2* key; unsigned long long* kval; unsigned long long* klast; u64 key_mask;   // kval = (order+1)<<24 | callset slot
  // (cell, callset) histogram
  unsigned long long* agg_key; unsigned long long* agg_cnt; u64 agg_mask;
  u32* arena; u64 arena_cap;
  Counters* ctr;
  const double* ent; const i64* ls; const i64* qp;
  const u16* mincov;   // mincov[n] = smallest coverage c with (double)c / (double)n >= score_percent (exact stand-in for the f64 division)
};

// De-duplication record exchanged between ranks: {key_lo, key_hi, global pair order, callset tag (0: none)}
struct KeyRec { u64 k0, k1, order, tag; };
// Peer routing of the whole-run scope (DESIGN.md "Multi-GPU"): every read_key has an owning rank; k_pair inserts the keys
// this rank owns into its own table and stores the others straight into the owner's inbox over NVLink, so the exchange
// rides along with the alignment instead of following it.  An inbox has one region of `cap` records per source rank and
// the fill cursors live on the SOURCE (cursor[owner], local atomics): nothing but the 32-byte record stores crosses
// the link — no remote atomic, no round trip.  inbox[o] = this rank's region inside rank o's inbox (a peer pointer from
// cudaIpcOpenMemHandle, or a plain device pointer of a context in the same process); world <= 1: routing off.
constexpr int ROUTE_MAX = 16;
struct Route { u32 world, rank; u64 pair_base, cap; KeyRec* inbox[ROUTE_MAX]; unsigned long long* cursor; };

// device probe table + prefilter from the flat k-mer table of the index artefact (tkey/tval: 4-key buckets, host.hpp)
void launch_probe_build(const u64* tkey, const u64* tval, u64 slots, u64* ptab, u32 n_pbuckets, u64* bloom, u32 bloom_words, u32 bloom_k, unsigned int* err, cudaStream_t s);
void launch_pack(const BatchDev& b, cudaStream_t s);
void launch_trim(const BatchDev& b, const Tables& t, cudaStream_t s);
void launch_map(const BatchDev& b, const DevIndex& ix, const DevCfg& cfg, const Tables& t, int count_work, cudaStream_t s);
void launch_dense_scatter(const u32* ids, u64 n, u32* dense, cudaStream_t s);   // dense[ids[i]] = i (slot -> callset id table on the device)
size_t rows_sort_tmp_bytes(u64 n);
void launch_rows_sort(const u64* agg, u64 n, const u32* dense, u64* keys, i64* vals, void* tmp, size_t tmp_bytes, u32* scope, u32* callset, i64* count, int key_bits, cudaStream_t s);
void launch_pair(const BatchDev& b, const DevIndex& ix, const DevLib& lib, const DevCfg& cfg, const Tables& t, const Route& rt, cudaStream_t s);
void launch_fold(const Tables& t, const u32* cell_of_pair, u64 order_base, cudaStream_t s);
void launch_resolve(const BatchDev& b, const Tables& t, cudaStream_t s);
void launch_compact(const Tables& t, u64* agg_out, u64 agg_cap, u32* cs_out, u64 cs_cap, unsigned long long* n_out2, cudaStream_t s);
void launch_export_reads(const BatchDev& b, const DevIndex& ix, const Tables& t, void* out, cudaStream_t s);
void launch_count_keys(const Tables& t, cudaStream_t s);
void launch_rehash_keys(const Tables& old_t, const Tables& new_t, cudaStream_t s);
void launch_keys_export(const Tables& t, void* records, unsigned long long* n_out, u64 cap, u64 order_base, cudaStream_t s);
void launch_keys_count_owner(const Tables& t, u32 world, unsigned long long* counts, cudaStream_t s);
void launch_keys_scatter(const Tables& t, void* rec, unsigned long long* cursors, u64 order_base, u32 world, cudaStream_t s);
void launch_callsets_import(const Tables& t, const u32* rows, u64 n, cudaStream_t s);
void launch_keys_import(const Tables& t, const void* records, u64 n, cudaStream_t s);

// per-cell table of the BAM driver (engine.cu nb_cells_*): open addressing on key (cell << 32 | persistent callset id) + 1
// with two counters per entry; it outlives nb_counts_reset, and the host grows it (rehash) before a roll could fill it past half.
// ctr[0] = occupied entries, ctr[1] = error bit (a probe ran through the whole table: cannot happen below half full)
struct CellTable { unsigned long long* key; unsigned long long* umis; unsigned long long* reads; u64 mask; unsigned long long* ctr; };
void launch_cells_roll(const CellTable& t, const u32* row_scope, const u32* row_callset, const i64* row_count, u64 n_rows, const u32* cell_of_scope, const u32* pid_of_dense, cudaStream_t s);
void launch_cells_rehash(const CellTable& o, const CellTable& n, cudaStream_t s);
size_t cells_sort_tmp_bytes(u64 n);
// occupied entries -> rows sorted by (cell, rank_of_pid[pid]): out = row_cell u32[n] | row_callset u32[n] | umis i64[n] | reads i64[n];
// work: 2n u64 keys + 2n u32 slots + tmp
void launch_cells_finalize(const CellTable& t, u64 n, const u32* rank_of_pid, u64* keys, u32* slots, unsigned long long* n_out, void* tmp, size_t tmp_bytes, void* out, cudaStream_t s);

// multi-GPU merge (engine.cu nb_merge_*): exchange blocks whose sizes the kernels read from the gathered headers on the device
constexpr u32 MERGE_HDR1_WORDS = 1 + ROUTE_MAX;
void launch_merge_hdr1(u64* hdr, const unsigned long long* n_rows, const unsigned long long* route_cursor, u32 world, cudaStream_t s);
void launch_merge_import_callsets(const Tables& t, const void* all, u64 blk_bytes, u64 cap, u32 world, u32 self, cudaStream_t s);
void launch_merge_import_inbox(const Tables& t, const void* inbox, u64 inbox_cap, u64 max_count, const void* all, u64 blk_bytes, u32 world, u32 self, cudaStream_t s);
void launch_merge_export_counts(const Tables& t, u64* blk2, u64 cap2, cudaStream_t s);
void launch_merge_import_counts(const Tables& t, const u64* all2, u64 blk2_words, u64 cap2, u32 world, cudaStream_t s);
void launch_merge_dense_fill(const Tables& t, const u32* dense_id, unsigned long long* dense, u64 n_cs, u64 n_cells, cudaStream_t s);
size_t merge_scan_tmp_bytes(u64 n);
void launch_merge_dense_scan(const unsigned long long* dense, u64 n, unsigned long long* flag, unsigned long long* prefix, void* tmp, size_t tmp_bytes, cudaStream_t s);
void launch_merge_dense_rows(const unsigned long long* dense, u64 n, u64 n_cs, const unsigned long long* prefix, u32* scope, u32* callset, i64* count, u32 cell_base, cudaStream_t s);

}  // namespace nbk
