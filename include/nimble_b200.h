/* nimble_b200.h — C ABI of the B200-native replacement for nimble-aligner's read-alignment hot path.
 *
 * The reference (BimberLab/nimble-aligner, pure Rust) has no FFI of its own; its boundary is the Rust library API.
 * Every entry point below names the reference interface it stands in for (paths under /root/reference).  A Rust (or
 * C++) host binds these with `extern "C"`; INTEGRATION.md shows the binding.  Conventions: plain pointers and sizes,
 * POD structs, no C++/torch types, no exceptions across the boundary; every call returns 0 or a negative nb_status
 * and nb_last_error() holds the message (the reference panics with a message instead — src/bin/main.rs:37,46,90,128).
 * The caller owns all host buffers; the library owns device memory.  An nb_index is immutable after build and may be
 * shared by several nb_ctx on the same device (the reference shares Arc<Vec<PseudoAligner>>, src/process/bam.rs:152-154).
 * There is NO CPU fallback: every compute entry point fails with NB_ERR_CUDA when no sm_100 device is usable.
 */
#ifndef NIMBLE_B200_H
#define NIMBLE_B200_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef enum nb_status {
  NB_OK = 0,
  NB_ERR_INVALID = -1,      /* bad argument */
  NB_ERR_IO = -2,           /* file could not be read / written */
  NB_ERR_PARSE = -3,        /* library JSON malformed or a config value has the wrong type (reference: expect() panics) */
  NB_ERR_CONFIG = -4,       /* sanity_check_align_config failed (src/reference_library.rs:209-226) */
  NB_ERR_UNSUPPORTED = -5,  /* input outside what the device path represents; message says what */
  NB_ERR_CUDA = -6,         /* CUDA runtime error, or no usable device */
  NB_ERR_OVERFLOW = -7,     /* a device scratch arena overflowed; message says which knob to raise */
  NB_ERR_FEATURE_NOT_FOUND = -8 /* unmap() would panic "Feature not found in reference columns" (src/align.rs:861) */
} nb_status;

/* LibraryChemistry, src/align.rs:97-103; strings of src/bin/main.rs:40-47 */
enum { NB_CHEM_UNSTRANDED = 0, NB_CHEM_FIVEPRIME = 1, NB_CHEM_THREEPRIME = 2, NB_CHEM_NONE = 3 };

/* FilterReason, src/align.rs:32-51, same order (Display strings: nb_reason_str) */
enum {
  NB_R_SCORE_BELOW_THRESHOLD = 0, NB_R_DISCARDED_MULTIPLE_MATCH, NB_R_DISCARDED_NONZERO_MISMATCH, NB_R_NO_MATCH,
  NB_R_NO_MATCH_AND_SCORE_BELOW_THRESHOLD, NB_R_DIFFERENT_FILTER_REASONS, NB_R_NOT_MATCHING_PAIR,
  NB_R_FORCE_INTERSECT_FAILURE, NB_R_SHORT_READ, NB_R_MAX_HITS_EXCEEDED, NB_R_HIGH_ENTROPY, NB_R_SUCCESSFUL_MATCH,
  NB_R_STRAND_WAS_WRONG, NB_R_TRIAGE_EMPTY_EQUIVALENCE_CLASS, NB_R_ABOVE_MISMATCH_THRESHOLD,
  NB_R_SKIPPED_ALIGN_DUE_TO_UNPAIRED_DUMMY, NB_R_NONE
};

/* AlignFilterConfig, src/align.rs:80-95 (field meaning identical; bools as int32) */
typedef struct nb_config {
  uint64_t reference_genome_size;
  double score_percent;
  uint64_t score_threshold;
  uint64_t num_mismatches;
  int32_t discard_nonzero_mismatch;
  int32_t discard_multiple_matches;
  int32_t score_filter;
  int32_t intersect_level;       /* 0 NoIntersect, 1 IntersectWithFallback, 2 ForceIntersect */
  int32_t require_valid_pair;
  int32_t strand_filter;         /* NB_CHEM_* */
  uint64_t discard_multi_hits;
  uint64_t max_hits_to_report;
  double trim_strictness;
  uint64_t trim_target_length;
} nb_config;

typedef struct nb_library nb_library;  /* Reference + AlignFilterConfig, src/reference_library.rs:11-17 */
typedef struct nb_index nb_index;      /* PseudoAligner = Pseudoaligner<Kmer30>, src/align.rs:21 */
typedef struct nb_ctx nb_ctx;          /* one (GPU, stream) execution context holding the aggregation state */

const char* nb_last_error(void);                 /* thread-local message of the last failing call */
const char* nb_reason_str(int reason);           /* Display for FilterReason, src/align.rs:53-77 */
const char* nb_version(void);

/* ---- reference_library::get_reference_library(path, strand_filter) -> (AlignFilterConfig, Reference)
 *      src/reference_library.rs:20-174: parses the 2-object JSON, U->T, appends the "name§rev" row after every row. */
int nb_library_load_json(const char* path, int strand_filter, nb_library** out);
int nb_library_parse_json(const char* text, size_t len, int strand_filter, nb_library** out);
/* Build a Reference directly (what the reference's tests do by constructing the struct, src/align.rs:1029-1040):
 * column-major strings, rows already final (no §rev rows are added). */
int nb_library_from_columns(const char* const* headers, uint32_t n_headers, const char* const* const* columns,
                            uint32_t n_rows, uint32_t group_on, uint32_t sequence_name_idx, uint32_t sequence_idx,
                            const nb_config* cfg, nb_library** out);
void nb_library_free(nb_library*);
int nb_library_get_config(const nb_library*, nb_config* out);
int nb_library_set_config(nb_library*, const nb_config* cfg);      /* e.g. --trim override, src/bin/main.rs:109-114 */
uint32_t nb_library_n_rows(const nb_library*);                     /* rows incl. §rev rows */
uint32_t nb_library_n_headers(const nb_library*);
const char* nb_library_header(const nb_library*, uint32_t col);
const char* nb_library_value(const nb_library*, uint32_t col, uint32_t row);
uint32_t nb_library_group_on(const nb_library*);
uint32_t nb_library_sequence_name_idx(const nb_library*);
uint32_t nb_library_sequence_idx(const nb_library*);
/* tests/basic-cases.rs:29-36 mutate the Reference: push a column and point group_on at it */
int nb_library_push_column(nb_library*, const char* header, const char* const* values, uint32_t n_rows, int set_group_on);

/* ---- utils::get_reference_sequence_data + debruijn_mapping::build_index::build_index::<Kmer30>(seqs, names, {}, cores)
 *      src/utils.rs:7-24, src/bin/main.rs:117-128.  Host build of the coloured compacted stranded de Bruijn graph
 *      (k = 30) into the flat GPU layout (DESIGN.md "Index layout"); the device copy is made by nb_ctx_create. */
int nb_index_build(const nb_library* lib, int n_threads, nb_index** out);
int nb_index_build_from_sequences(const uint8_t* seq_ascii, const uint64_t* seq_off, uint32_t n_seqs, int n_threads,
                                  nb_index** out);
/* K5: the same build on the GPU (sort / group / join / chain walk / cuckoo insertion as CUDA kernels); the artefact
 * equals the host build's array for array, except where a k-mer sits among its four candidate table slots.  Falls
 * back to the host builder for a library with pure k-mer cycles.  NB_ERR_CUDA when `device` is not usable. */
int nb_index_build_gpu(const nb_library* lib, int device, int n_threads, nb_index** out);
int nb_index_build_gpu_from_sequences(const uint8_t* seq_ascii, const uint64_t* seq_off, uint32_t n_seqs, int device,
                                      int n_threads, nb_index** out);
/* 0 when both artefacts describe the same index: all arrays equal and every k-mer of `a` resolves to the same
 * (node, offset) in `b`; otherwise a positive code naming the first array that differs (1 scalars, 2 unitigs, 3 nodes,
 * 4 edges, 5 colours, 6 universes, 7 table) */
int nb_index_compare(const nb_index* a, const nb_index* b);
void nb_index_free(nb_index*);
/* on-disk index cache: the flat arrays exactly as they are uploaded (the reference rebuilds its index on every run) */
int nb_index_save(const nb_index*, const char* path);
int nb_index_load(const char* path, nb_index** out);
/* the cache keyed by the library (SURVEY 8f row 4): key = 32 hex digits over the sequence column as the index sees it
 * (case and non-ACGT folded like DnaString::from_acgt_bytes) and the artefact's format tag.  nb_index_build_cached loads
 * <cache_dir>/<key>.nbix when it is there and sound, else builds on GPU `device` and writes it (temporary name + rename);
 * cache_dir NULL: $NB_INDEX_CACHE, and with neither set it is nb_index_build_gpu.  The file drivers and the CLI go through it. */
int nb_index_cache_key(const nb_library* lib, char out_hex[33]);
int nb_index_build_cached(const nb_library* lib, const char* cache_dir, int device, int n_threads, nb_index** out);
/* out[0..7] = n_kmers, n_nodes, n_colours, colour_elems, unitig_bases, table_slots, device_bytes, n_sequences */
int nb_index_stats(const nb_index*, uint64_t* out8);
/* canonical text dump (one line per unitig, sorted) used by the parity tests; returns bytes needed */
uint64_t nb_index_dump(const nb_index*, char* buf, uint64_t cap);

/* ---- execution context */
int nb_device_count(void);
int nb_ctx_create(const nb_index* index, const nb_library* lib, int device, void* cuda_stream /* NULL: own stream */,
                  nb_ctx** out);
void nb_ctx_free(nb_ctx*);
int nb_ctx_set_config(nb_ctx*, const nb_config* cfg);   /* config is read by pseudoalign / filter_and_coerce per call */
int nb_ctx_sync(nb_ctx*);
/* tuning knobs: "max_batch_pairs", "ec_arena_entries", "callset_slots", "key_slots", "agg_slots", "count_work", "cell_slots" */
int nb_ctx_set_option(nb_ctx*, const char* name, uint64_t value);

/* pinned host memory for the caller's double-buffered batches (src/parse readers feed these) */
void* nb_host_alloc(size_t bytes);
void nb_host_free(void*);

enum { NB_MEM_HOST = 0, NB_MEM_DEVICE = 1 };
enum { NB_FLAG_SKIP_ALIGN = 1 /* metadata[37]=="TRUE", src/align.rs:527 */, NB_FLAG_REVCOMP = 2 /* REVERSE, src/process/bam.rs:407-415 */ };

/* One batch of read pairs = the iterators score::call receives (src/score.rs:14-31).  Sequences are ASCII bases
 * (DnaString::from_acgt_bytes semantics: ACGT either case, anything else -> A), concatenated, with n_pairs+1 offsets.
 * r2 == NULL: single-end (mate_sequences = None).  q1/q2: raw Phred bytes (BAM record.qual(), no -33) laid out with
 * the same offsets; NULL = no metadata (FASTQ mode: no trimming, src/align.rs:521-525).  flags1/flags2: NB_FLAG_*
 * per pair side or NULL.  scope_id: aggregation scope per pair (the (UMI,CB) group of src/process/bam.rs:200-221),
 * non-decreasing; NULL = one whole-run scope (src/process/fastq.rs:15-29).  Every scope must be complete within one
 * call: a scoped batch is de-duplicated and folded into the (cell, callset) count table before the call returns. */
typedef struct nb_batch {
  uint64_t n_pairs;
  int32_t location;            /* NB_MEM_HOST (pinned recommended) or NB_MEM_DEVICE */
  uint32_t max_read_len;       /* longest read in the batch; 0 = let the library scan the offsets (host batches only) */
  const uint8_t* r1; const uint64_t* r1_off;
  const uint8_t* r2; const uint64_t* r2_off;
  const uint8_t* q1; const uint8_t* q2;
  const uint8_t* flags1; const uint8_t* flags2;
  const uint32_t* scope_id;
  const uint32_t* cell_id;     /* optional with scope_id: row key of the count table (e.g. the cell barcode); NULL = scope_id */
  int32_t encoding;            /* NB_SEQ_ASCII (0, default) | NB_SEQ_2BIT | NB_SEQ_BAM4: how r1 / r2 hold the bases */
  int32_t reserved;
  const uint32_t* r1_len; const uint32_t* r2_len;   /* packed encodings, optional: explicit read lengths when the reads are not densely packed */
} nb_batch;
/* Packed encodings: what score::call really receives are 2-bit DnaStrings (src/score.rs:14-31) and BAM stores 4-bit bases
 * (src/parse/bam.rs:186-189), so a host that already holds packed reads ships a quarter / half of the bytes.  r?_off then
 * count BASES of the packed stream (n_pairs + 1 entries; a read may start at any base); lengths are r?_off[p+1] - r?_off[p]
 * unless r?_len is given.  q1 / q2 stay one byte per base at the same base offsets.
 *   NB_SEQ_2BIT  base j = bits 2(j&3)..2(j&3)+1 of byte j>>2, A=0 C=1 G=2 T=3 (a non-ACGT base must already be 0, as
 *                DnaString::from_acgt_bytes makes it)
 *   NB_SEQ_BAM4  nibble j = byte j>>1, high nibble first (BAM's seq field), code table "=ACMGRSVTWYHKDBN": everything but
 *                A, C, G, T becomes A, exactly what the reference does with those letters
 * Buffers must be readable for 16 bytes past the last base.
 * Device-resident batches (NB_MEM_DEVICE), any encoding: the kernels fetch bases and quals as aligned 16-byte vectors, so r1 / r2
 * / q1 / q2 must be readable from the 16-byte boundary at or below their first byte to 48 bytes past their last one (any
 * cudaMalloc'ed buffer is; host batches are staged by the library and need nothing). */
enum { NB_SEQ_ASCII = 0, NB_SEQ_2BIT = 1, NB_SEQ_BAM4 = 2 };

/* Per-read outcome of align::pseudoalign (src/align.rs:945-989): reason is SuccessfulMatch when the read passed;
 * score / mismatches are map_read_with_mismatch's coverage and mismatch totals (0 when it returned None). */
typedef struct nb_read_result {
  uint8_t reason; uint8_t pass; uint16_t score; uint16_t mismatches; uint16_t trimmed_len; uint32_t ec_len; uint32_t ec_hash;
} nb_read_result;
/* Per-pair outcome: filter reasons as score_sequences records them (src/align.rs:586-600), triage as
 * filter_and_coerce_sequence_call_orientations records it (233-241), callset = id into nb_counts of this ctx
 * (0xFFFFFFFF none).  `insertable`: the pair reached score_map.insert (src/align.rs:685). */
typedef struct nb_pair_result {
  uint32_t callset; uint8_t triage; uint8_t fr1; uint8_t fr2; uint8_t insertable; uint64_t key_lo; uint64_t key_hi;
} nb_pair_result;

/* score::call on one batch (src/score.rs:14-46 -> align::get_calls src/align.rs:392-467): maps every read, applies
 * thresholds, pair / strand / orientation logic and folds the pairs into the context's per-scope de-duplicated
 * callset counts.  reads_out (2*n_pairs entries when paired, else n_pairs; side-major per pair: [2p]=sequence,
 * [2p+1]=mate) and pairs_out may be NULL.  Output buffers follow batch->location.  Asynchronous on the context's
 * stream: host buffers may be reused after nb_ctx_sync() or after the second following nb_align_batch() returns (the
 * library blocks on the copies of a staging set before it refills it, so a producer rotating THREE pinned buffers never
 * overwrites one that is still being read; with two, call nb_ctx_sync() before each refill).
 * read_key (src/align.rs:576-579: the R1 string followed by the R2 string) is represented by a 128-bit hash of the
 * concatenated 2-bit base stream, the length and the scope: two DIFFERENT pairs of one scope are merged with probability
 * about n^2 / 2^129 (1e-23 at 1e8 pairs) — the one place where the device path is exact only up to a hash.  nb_pair_result
 * carries the key (key_lo, key_hi).  A scope with more pairs than max_batch_pairs is still de-duplicated as a whole: the
 * chunk grows to the end of that scope. */
int nb_align_batch(nb_ctx*, const nb_batch* batch, nb_read_result* reads_out, nb_pair_result* pairs_out);
/* Debug / parity: full equivalence class of every read of the LAST batch: ec_off (n_reads+1) and ids. Host buffers. */
int nb_last_batch_ecs(nb_ctx*, uint64_t* ec_off, uint32_t* ec_ids, uint64_t ec_cap, uint64_t* ec_total);

/* Result of get_calls for the scopes seen since the last nb_counts_reset: rows (scope, callset, count) with the
 * callset dictionary.  Callset c = group indices callset_items[callset_off[c] .. callset_off[c+1]) into the library's
 * group-name table (nb_library_group_name); rows are sorted by scope then by Vec<String> Ord of the callset
 * (utils::sort_score_vector, src/utils.rs:54-59).  Pointers stay valid until the next finalize/reset/free. */
typedef struct nb_counts {
  uint64_t n_rows; const uint32_t* row_scope; const uint32_t* row_callset; const int64_t* row_count;
  uint64_t n_callsets; const uint64_t* callset_off; const uint32_t* callset_items;
  uint64_t n_pairs_seen; uint64_t n_unique_keys;
  uint64_t n_slots; const uint32_t* slot_to_callset;   /* nb_pair_result.callset (dictionary slot) -> callset id here */
} nb_counts;
int nb_counts_finalize(nb_ctx*, nb_counts* out);
/* device copies of the row columns of the last nb_counts_finalize (row_scope u32[n], row_callset u32[n], row_count i64[n]),
 * valid until the next finalize / reset: lets a multi-GPU host reduce per-cell tables without a host round trip */
int nb_counts_device_rows(nb_ctx*, const void** row_scope, const void** row_callset, const void** row_count, uint64_t* n_rows);
/* device copy of the last nb_counts_finalize's slot_to_callset (u32[n_slots], nb_pair_result.callset -> callset id, 0xFFFFFFFF
 * for a slot without one), on the context's stream; valid until the next finalize / reset, like nb_counts_device_rows */
int nb_counts_device_slot_map(nb_ctx*, const void** slot_to_callset, uint64_t* n_slots);
int nb_counts_reset(nb_ctx*);
uint32_t nb_library_n_groups(const nb_library*);
const char* nb_library_group_name(const nb_library*, uint32_t group);

/* Per-cell count table of BAM mode: the per-scope rows of successive scoped batches rolled up by cell, in a table of the
 * context that nb_counts_reset leaves alone.  For cell c and callset S: umis = scopes of c with a row for S (a scope has at
 * most one), reads = sum of those rows' counts (nimble_score).  Callsets are numbered persistently across batches (every
 * finalize renumbers its own).
 *   nb_cells_roll      after nb_counts_finalize of a scoped batch, once per batch: cell_of_scope[scope_id] = cell id (< 2^32 - 1,
 *                      else NB_ERR_UNSUPPORTED) for the batch's n_scopes scopes.  The table grows on the device as needed;
 *                      option "cell_slots" sets its first size (before the first roll).  Synchronous: cell_of_scope may be reused
 *   nb_cells_finalize  rows sorted by (cell id, callset); callsets = those with a row, numbered in Vec<String> Ord
 *                      (utils::sort_score_vector) with their group lists as in nb_counts.  Pointers stay valid until the next
 *                      nb_cells_finalize / nb_cells_reset / nb_ctx_free; the table itself is kept (more batches may follow)
 *   nb_cells_reset     empty table and callset numbering */
typedef struct nb_cell_counts {
  uint64_t n_rows; const uint32_t* row_cell; const uint32_t* row_callset; const int64_t* row_umis; const int64_t* row_reads;
  uint64_t n_callsets; const uint64_t* callset_off; const uint32_t* callset_items;
  uint64_t n_scopes;           /* scopes rolled in */
} nb_cell_counts;
int nb_cells_roll(nb_ctx*, const uint32_t* cell_of_scope, uint64_t n_scopes);
int nb_cells_finalize(nb_ctx*, nb_cell_counts* out);
int nb_cells_reset(nb_ctx*);

/* multi-GPU merge of the whole-run scope (SURVEY.md §8e).  Reads shard over ranks with the index replicated; counts
 * are over unique read_keys of the whole run, so ranks exchange their de-duplication records by key range
 * (all-to-all over NCCL, driven by the host), re-import the partition they own and finalize; the per-callset counts
 * are then summed across ranks (all-reduce).  Records are 32 bytes {key_lo, key_hi, order = global pair index,
 * callset_tag}; dev_records are device pointers; nb_keys_export_partitioned groups them by owning rank (a 16-bit slice of
 * key_lo mod world) so no sort is needed.  Callset dictionaries travel as rows of (4 + gcap) uint32:
 * {slot, len, tag_lo, tag_hi, items[gcap]}; after importing the union every rank's nb_counts lists the same callsets in
 * the same order, so the final merge is one all-reduce(sum) over a dense count vector.  Both exports fail with
 * NB_ERR_INVALID when cap is below the record count; nb_keys_import fails with NB_ERR_INVALID when a record's callset
 * tag is not in this context's dictionary (import the peers' rows first). */
int nb_keys_export_count(nb_ctx*, uint64_t* n);
int nb_keys_export(nb_ctx*, void* dev_records, uint64_t cap, uint64_t pair_index_base);
int nb_keys_import(nb_ctx*, const void* dev_records, uint64_t n);
int nb_keys_export_partitioned(nb_ctx*, void* dev_records, uint64_t cap, uint64_t pair_index_base, uint32_t world, uint64_t* counts_out);
int nb_callsets_export(nb_ctx*, uint32_t* rows, uint64_t cap_rows, uint64_t* n_out, uint32_t* gcap_out);
int nb_callsets_import(nb_ctx*, const uint32_t* rows, uint64_t n);
int nb_callsets_import_device(nb_ctx*, const uint32_t* dev_rows, uint64_t n);   /* rows already in this context's HBM; asynchronous */

/* Peer routing of the whole-run scope: instead of exchanging the key tables when the job ends, k_pair stores every
 * record whose key another rank owns straight into that rank's inbox over NVLink while the alignment runs; keys this
 * rank owns go into its own table with global pair orders.  An inbox has one region per source rank and the fill
 * cursors stay on the source, so only the 32-byte record stores cross the link (no remote atomics).  When the job ends
 * each rank merges its inbox (nb_route_import) — no all-to-all, no export pass over the key table.
 *   nb_route_create      allocate this context's inbox (world x records_per_peer x 32 B); returns its CUDA IPC handle (64 B).
 *                        Every rank must pass the same world and records_per_peer (a region's place in an inbox is
 *                        source rank x records_per_peer); a region that fills up fails the job loudly (NB_ERR_OVERFLOW)
 *   nb_route_attach_ipc  one process per GPU: handles = world x 64 B gathered from all ranks (own entry ignored);
 *                        NB_ERR_CUDA when a handle cannot be opened (the host then keeps the NCCL exchange above)
 *   nb_route_attach_ctx  one process driving several contexts / GPUs: peers[world], peers[rank] == this context
 *   nb_route_sent        after this rank's last batch: records stored per destination rank (sent[world]); the host
 *                        delivers sent[o] to rank o (one all_gather, which is also the barrier nb_route_import needs)
 *   nb_route_import      merge counts[r] records from each rank r; call after nb_callsets_import of the peers' dictionaries
 * pair_index_base = global index of this rank's first pair (orders decide which duplicate wins, src/align.rs:685). */
enum { NB_ROUTE_HANDLE_BYTES = 64 };
int nb_route_create(nb_ctx*, uint32_t world, uint64_t records_per_peer, void* ipc_handle_out);
int nb_route_attach_ipc(nb_ctx*, uint32_t world, uint32_t rank, const void* handles, uint64_t pair_index_base);
int nb_route_attach_ctx(nb_ctx*, uint32_t world, uint32_t rank, nb_ctx* const* peers, uint64_t pair_index_base);
int nb_route_set_pair_base(nb_ctx*, uint64_t pair_index_base);
int nb_route_sent(nb_ctx*, uint64_t* sent);
int nb_route_import(nb_ctx*, const uint64_t* counts, uint64_t* n_imported);
int nb_route_detach(nb_ctx*);

/* ---- multi-GPU merge inside the library, over NCCL (SURVEY.md §8b `nb_counts_allreduce(nb_ctx*, ncclComm_t)`, §8e).  The
 * reference's parallel driver is N-1 consumer threads behind one producer (src/process/bam.rs:183-226); here it is one
 * context per GPU.  NCCL is resolved from libnccl.so.2 at run time (a single-GPU host needs none); all collectives run on
 * the context's stream and the host waits once per merge.
 *   nb_comm_unique_id   ncclGetUniqueId (128 bytes): rank 0 creates it, the host hands it to every rank
 *   nb_comm_init_rank   one process per GPU: ncclCommInitRank on the context's device; the communicator lives in the context
 *   nb_comm_attach      adopt a communicator the host created (ncclComm_t); not destroyed by the library
 *   nb_comm_init_all    one process driving n GPUs: ncclCommInitAll over the contexts' devices (rank i = ctxs[i])
 *   nb_route_setup      one process per GPU: nb_route_create + all-gather of the IPC handles + nb_route_attach_ipc; fails on
 *                       EVERY rank when any rank cannot open its peers (no NVLink / IPC)
 *   nb_merge_whole_run  whole-run scope (FASTQ mode) with peer routing attached: dictionaries all-gathered, this rank's inbox
 *                       merged, its keys folded, {callset, count} rows all-gathered and summed: every rank's `out` holds the
 *                       job's counts (n_unique_keys = unique read_keys of the whole job), as nb_counts_finalize would on one GPU
 *   nb_merge_scoped     scoped batches (BAM mode; whole scopes shard over ranks, no data-path exchange): dictionaries
 *                       all-gathered, then the per-cell tables are summed with one dense [n_cells x callsets] all-reduce;
 *                       row_scope of `out` = cell id.  n_cells = 1 + the largest cell_id of the job (nb_merge_scoped_sharded:
 *                       every rank keeps only its own range of cells)
 * Collective calls: every rank of the communicator must make them in the same order. */
enum { NB_COMM_ID_BYTES = 128 };
int nb_comm_unique_id(void* id128_out);
int nb_comm_init_rank(nb_ctx*, const void* id128, uint32_t world, uint32_t rank);
int nb_comm_attach(nb_ctx*, void* nccl_comm);
int nb_comm_init_all(nb_ctx* const* ctxs, uint32_t n);
int nb_comm_free(nb_ctx*);
int nb_comm_info(nb_ctx*, uint32_t* world, uint32_t* rank);
int nb_route_setup(nb_ctx*, uint64_t records_per_peer, uint64_t pair_index_base);
int nb_merge_whole_run(nb_ctx*, nb_counts* out);
int nb_merge_scoped(nb_ctx*, uint64_t n_cells, nb_counts* out);
/* the same with the result left SHARDED over the ranks: a reduce-scatter instead of the all-reduce; rank r's `out` holds the
 * rows of cells [r * ceil(n_cells / world), (r + 1) * ceil(n_cells / world)) only (callsets numbered alike on every rank), so a
 * job's rows cross PCIe once, not once per GPU — the shape for a host that writes each cell's rows from one place */
int nb_merge_scoped_sharded(nb_ctx*, uint64_t n_cells, nb_counts* out);

/* timing of the dominant kernel (seed_walk_map), CUDA events on the launching stream: out[0]=launches, out[1]=total ms,
 * out[2]=reads processed, out[3]=all kernels launched by this ctx since reset */
int nb_ctx_kernel_stats(nb_ctx*, double* out4, int reset);
/* work counters of k_map when option "count_work" is 1: out[0..3] = hash probes, unitigs visited, bases compared,
 * colour ids touched (the terms of the algorithmic-bytes formula, DESIGN.md "Roofline") */
int nb_ctx_work_counters(nb_ctx*, uint64_t* out4);

/* ---- roofs (diagnostics; nothing on the data path calls them).  SURVEY.md §8(d): the probe / walk traffic of the map
 * stage (align::pseudoalign -> map_read_with_mismatch, src/align.rs:945-989) is random 32-byte buckets and 64-byte walk
 * records, so its roof is the random-record gather bandwidth of the memory level the index lives in (L2 for the 1k
 * library, HBM for the 200k one); the end-to-end number's roof is the pinned host -> device link.
 *   nb_measure_gather  bytes gathered / s over a table of table_bytes (record_bytes 32 or 64), best of reps launches
 *   nb_measure_h2d     n devices copying `bytes` x reps from pinned host memory at the same time: GB/s each and aggregate */
int nb_measure_gather(int device, uint64_t table_bytes, uint32_t record_bytes, uint32_t reps, double* gbs_out);
int nb_measure_h2d(const int* devices, uint32_t n, uint64_t bytes, uint32_t reps, double* out_per_device, double* aggregate_out);

/* ---- drivers: process::fastq::process (src/process/fastq.rs:7-30) and utils::write_to_tsv (src/utils.rs:27-51) */
int nb_write_fastq_tsv(const char* path, const nb_library* lib, const nb_counts* counts);
int nb_process_fastq(const char* const* input_files, uint32_t n_inputs, const char* const* reference_json, const char* const* output_paths,
                     uint32_t n_refs, int strand_filter, int num_cores, int device);
/* the same on several GPUs of one box: one context per device behind the one feeder, key records routed between the GPUs
 * inside k_pair, counts merged by nb_merge_whole_run (the reference's parallel shape is N-1 consumers behind one producer,
 * src/process/bam.rs:183-226; its FASTQ mode is single-threaded).  The routing inboxes are sized from the input size;
 * NB_ROUTE_RECORDS=<records per peer> overrides, an inbox that fills up fails the job with NB_ERR_OVERFLOW. */
int nb_process_fastq_devices(const char* const* input_files, uint32_t n_inputs, const char* const* reference_json, const char* const* output_paths,
                             uint32_t n_refs, int strand_filter, int num_cores, const int* devices, uint32_t n_devices);
/* host-only: the records the FASTQ feeder (src/parse/fastq.rs:21-43) hands to the device, one line per record ("SEQ" or
 * "SEQ1<TAB>SEQ2") — parity tests of the parallel plain-text parser against a sequential one.  chunk_bytes: bytes of file per
 * parse task (0 = default 8 MiB); num_cores host threads are split over the input files. */
int nb_fastq_dump(const char* const* input_files, uint32_t n_inputs, int num_cores, uint64_t chunk_bytes, const char* out_path);
/* host-only: the file drivers' own inflate (flate2 / htslib's place in src/parse/fastq.rs:21-43 and
 * src/parse/sorted_bam_reader.rs:22-41) on a buffer — parity tests against zlib.  raw != 0: one raw deflate stream in one
 * piece (a BGZF block); raw == 0: concatenated gzip members through windows of `window` bytes (0 = one window), CRC-32 and
 * ISIZE checked.  NB_ERR_PARSE on a damaged stream, NB_ERR_OVERFLOW when out_cap is too small. */
int nb_inflate(const void* in, uint64_t in_len, int raw, uint64_t window, void* out, uint64_t out_cap, uint64_t* out_len);
/* host-only: a gzip file in memory through the FASTQ feeder's parallel reader (`threads` workers enter the deflate stream
 * at guessed block headers of `chunk_bytes` byte ranges; nothing is emitted that the sequential decode does not confirm) */
/* host-only: one gzip member made by the BAM driver's TSV compressor (GzEncoder's place in src/process/bam.rs:22-42) */
int nb_gzip_fast(const void* in, uint64_t in_len, void* out, uint64_t out_cap, uint64_t* out_len);
int nb_gunzip_parallel(const void* in, uint64_t in_len, int threads, uint64_t chunk_bytes, void* out, uint64_t out_cap, uint64_t* out_len);

/* process::bam::process (src/process/bam.rs:45-243) behind the same library loop: BGZF/BAM decode on host threads,
 * UMIReader / SortedBamReader grouping (src/parse/bam.rs, src/parse/sorted_bam_reader.rs) with their quirks, one scoped
 * batch per ~512k pairs, gzip TSV rows (header + row format of src/process/bam.rs:22-42, 90-121).  `trim`: the --trim
 * option string "L:S,L:S,..." or NULL. */
/* host-only: writes the (UMI, CB) groups the producer would send (one line per record) — parity tests of the feeder */
int nb_bam_dump_groups(const char* input_file, int force_bam_paired, int num_cores, const char* out_path);
int nb_process_bam(const char* input_file, const char* const* reference_json, const char* const* output_paths, uint32_t n_refs,
                   int strand_filter, const char* trim, int num_cores, int force_bam_paired, int device);
/* The same run with a cell x feature count matrix per library (nb_cells_*): matrix_dirs[i] receives library i's matrix
 * (nb_write_cell_matrix).  The cell of a scope is the full CB of its first record; the barcodes are the CBs that start a
 * scope, in order of first appearance (one list for all libraries).  output_paths NULL: no TSV rows at all (the rows stage
 * is not run); matrix_dirs NULL: exactly nb_process_bam.  One of the two must be given. */
int nb_process_bam_cells(const char* input_file, const char* const* reference_json, const char* const* output_paths,
                         const char* const* matrix_dirs, uint32_t n_refs, int strand_filter, const char* trim, int num_cores,
                         int force_bam_paired, int device);
/* The per-cell matrices of nb_process_bam_cells (no TSV rows) from a BAM in ANY record order, e.g. Cell Ranger's
 * position-sorted possorted_genome_bam.bam: scopes come from the records' tags, not from the file order.  With ordinals
 * 0..n-1 in file order:
 *   1. kept records are filtered as SortedBamReader::fill_buffer does: no CB string aux -> skipped; UMI = UB, else UR, and a
 *      CB without either fails with NB_ERR_PARSE "Error -- Could not read UMI."; UMI AAAAAAAAAA -> skipped
 *   2. kept records are ordered by (UMI, full CB, ordinal) (byte order), on the GPU
 *   3. a scope is a maximal run in that order with equal (UMI, CB[..len-2]), compared as a pair
 *   4. each scope's records go through add_dummy_paired_reads and filter_paired_reads (src/parse/sorted_bam_reader.rs:109-162;
 *      names compared exactly); TSO clip, REVERSE and quals as in nb_process_bam
 *   5. the cell of a scope is the full CB of its first record; every scope is aligned (no "last group" is dropped)
 *   6. the barcodes are the cells of the scopes that have pairs, in order of the first kept record (by ordinal) with that CB
 * So the matrix equals nb_process_bam_cells (rows NULL) on the file G = the kept records in the order of step 2 followed by
 * one scope with a UMI no record has: same features, barcode set and (feature, barcode) counts; only the barcode order differs.
 * Every kept record's nibbles, quals and name stay in device memory (the store; NB_BAM_STATS=1 prints its size) and the
 * scoped batches point into it.  Refused: a kept record with an empty UMI string, or a UMI that the exact device key cannot
 * hold (more than 21 characters, or a character outside ACGTN): NB_ERR_UNSUPPORTED naming it; a store that does not fit:
 * NB_ERR_CUDA with the bytes needed.  There is no force_bam_paired (mates of a position-sorted file are not neighbours); the
 * TSV rows of such a file come from nb_process_bam_rows_any_order. */
int nb_process_bam_cells_any_order(const char* input_file, const char* const* reference_json, const char* const* matrix_dirs, uint32_t n_refs,
                                   int strand_filter, const char* trim, int num_cores, int device);
/* test hook: the device grouping of nb_process_bam_cells_any_order, one line per pair:
 * scope index (counting the scopes with pairs, in sorted order) TAB cell barcode TAB sequence-slot ordinal TAB mate-slot ordinal
 * TAB flags (NB_FLAG_*) of both slots TAB clipped lengths of both slots */
int nb_bam_dump_scopes_any_order(const char* input_file, int num_cores, int device, const char* out_path);
/* nb_process_bam_cells_any_order under a device-memory budget of budget_bytes (0: none, exactly
 * nb_process_bam_cells_any_order).  The budget covers every device allocation of the any-order path: the record store
 * (also while an array grows and its old and new copies are both alive), the sort, scope and pair arrays and the scratch of
 * a compaction.  It does not cover the library contexts: the index, the aggregation tables and the per-cell table.
 * Records are split by UMI bucket, the top 16 bits of the splitmix64 finalizer of the exact UMI key (nb_any_order_umi_bucket),
 * so every scope falls whole into one bucket.  Each pass reads the file from the start and keeps buckets [lo, hi), hi
 * starting at 65536; when the store, the next window and the grouping arrays would not fit the budget, hi falls to the
 * largest value whose buckets fit 3/4 of it, the store is compacted in place to the records below hi, and later records at
 * or above hi are dropped.  At the end of the file the pass groups, aligns and rolls as the single pass does; the next pass
 * starts at lo = hi.  A file that fits takes one pass.  The matrix files are the bytes of the unbudgeted run.  Refused with
 * NB_ERR_CUDA, naming the budget and the bytes needed: a budget that cannot hold one bucket.  NB_BAM_STATS=1 adds budget,
 * passes, evictions (compactions), peak device bytes and the windows time of every pass to the stats line.
 * NB_BAM_COMPACT_TILE_BYTES=N caps the compaction's scratch tile at N bytes (at least 64; default up to 16 MB). */
int nb_process_bam_cells_any_order_budget(const char* input_file, const char* const* reference_json, const char* const* matrix_dirs, uint32_t n_refs,
                                          int strand_filter, const char* trim, int num_cores, int device, uint64_t budget_bytes);
/* test hook: nb_bam_dump_scopes_any_order under a budget; every line starts with the pass index TAB, scope indices count on
 * across passes, and each line ends with TAB bases TAB quals (hex) of the sequence slot and of the mate slot, clipped, read
 * back from the device store after the pass (so after any compaction) */
int nb_bam_dump_scopes_any_order_budget(const char* input_file, int num_cores, int device, uint64_t budget_bytes, const char* out_path);
/* test hook (host-only): the UMI bucket (0..65535) of nb_process_bam_cells_any_order_budget for a UMI string, so that tests
 * can check the bucket function against a restatement; NB_ERR_UNSUPPORTED when the exact key cannot hold it */
int nb_any_order_umi_bucket(const char* umi, uint32_t len, uint32_t* bucket);
/* The TSV.gz rows of nb_process_bam (one output_paths[i] per reference library) from a BAM in ANY record order.  The file
 * is G's rows: G = the kept records (steps 1-2 of nb_process_bam_cells_any_order) in (UMI, CB) order followed by one sentinel
 * scope, and gunzip(output) equals gunzip of nb_process_bam on G byte for byte: the header, the scopes in that order, in a
 * scope the count rows in finalize order and then the zero rows in pair order, the same representative pairs, zero-row
 * rule, reason and score columns and SKIP_ALIGN values.  No row at all: an empty gzip stream.  The gzip member layout is not
 * part of the output.  Every kept record's 36 reported metadata values are formatted on the host threads and kept in device
 * memory next to its bases (a fourth byte store); the rows of each batch are assembled on the GPU and only deflated and
 * written on the host.  budget_bytes (0: none) is the budget of nb_process_bam_cells_any_order_budget, which also covers the
 * metadata store, the per-pair results and the row buffer; with P passes the file is the header, then the rows of each
 * pass in pass order, a pass's rows being G's rows of its UMI buckets in G's order.  NB_BAM_ROWS_BUFFER_KB=N sets the cap of
 * the device row buffer (default 64 MB); a batch whose rows exceed it is written in chunks of whole scopes.  The passes are
 * planned with the row buffer, the row stage's scratch and 64 KB of callset texts reserved; a batch whose callset texts
 * need more, or a scope whose rows exceed the buffer (it gets a grown buffer of its own), allocates the rest within the budget
 * when it comes.  Refused as in nb_process_bam_cells_any_order (no force_bam_paired), and such an allocation that does not fit
 * the budget: NB_ERR_CUDA naming the bytes.  NB_BAM_STATS=1 adds rows, row bytes, row chunks, the metadata store and text
 * bytes, the row buffer, the device peak and the row build and deflate times to the any-order stats line. */
int nb_process_bam_rows_any_order(const char* input_file, const char* const* reference_json, const char* const* output_paths, uint32_t n_refs,
                                  int strand_filter, const char* trim, int num_cores, int device, uint64_t budget_bytes);
/* host-only: a cell x feature matrix in the 10x v3 layout that Seurat's Read10X and scanpy's read_10x_mtx load, into `dir`
 * (created when missing; its parent must exist): matrix.mtx.gz (Matrix Market coordinate integer, features x barcodes, UMI
 * counts, 1-based lines sorted by barcode then feature), reads.mtx.gz (the same coordinates with the read counts),
 * features.tsv.gz ("callset<TAB>callset<TAB>Gene Expression", callset = group names joined by ','), barcodes.tsv.gz.  Gzip
 * members with mtime 0 and no file name: the same counts give the same bytes. */
int nb_write_cell_matrix(const char* dir, const nb_library* lib, const nb_cell_counts* counts, const char* const* barcodes, uint64_t n_barcodes);

#ifdef __cplusplus
}
#endif
#endif
