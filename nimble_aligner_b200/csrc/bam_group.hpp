// bam_group.hpp — the device record store of BAM mode in any record order (bam.cpp's process_bam_any_order, the one driver
// behind nb_process_bam_cells_any_order[_budget] and nb_process_bam_rows_any_order): the host producer stages every kept
// record's nibbles, quals, name and keys window by window; the device sorts the records by (UMI, CB), cuts the
// (UMI, CB[..len-2]) scopes, pairs each scope's records and hands out scoped batches that point into the store.  Bulk mode
// (bam.cpp's process_bam_bulk) stages no quals or cell keys and pairs the mates of the whole file by name (pair_bulk).
// Host-only declarations (bam.cpp includes them; bam_group.cu implements them).
#pragma once
#include <functional>
#include <string>

#include "host.hpp"

namespace nbg {

enum { MAX_UMI_CHARS = 21 };   // 3 bits per character of ACGTN, 63 bits

// UMI -> exact sort key: characters A C G N T as 1..5 (their byte order), first character in the highest bits, 0 after the
// end, so equal keys are equal strings and the keys sort like the strings.  false: not representable (empty, longer than
// 21 characters, or a character outside ACGTN).
inline bool pack_umi(const char* s, u32 n, u64& key) {
  if (n == 0 || n > MAX_UMI_CHARS) return false;
  u64 k = 0;
  for (u32 i = 0; i < n; i++) {
    u64 c;
    switch (s[i]) { case 'A': c = 1; break; case 'C': c = 2; break; case 'G': c = 3; break; case 'N': c = 4; break; case 'T': c = 5; break; default: return false; }
    k |= c << (60 - 3 * i);
  }
  key = k; return true;
}

// Budget mode (nb_process_bam_cells_any_order_budget) splits the records into passes by UMI bucket: every record of a
// (UMI, CB[..len-2]) scope has the same UMI, so any set of whole buckets groups on its own.  bucket = the top 16 bits of
// the splitmix64 finalizer of the exact UMI key; host and device use this one definition.
enum : u32 { N_BUCKETS = 1u << 16 };
#ifdef __CUDACC__
__host__ __device__
#endif
inline u32 umi_bucket(u64 k) {
  k ^= k >> 30; k *= 0xBF58476D1CE4E5B9ull; k ^= k >> 27; k *= 0x94D049BB133111EBull; k ^= k >> 31;
  return (u32)(k >> 48);
}

// Pinned staging of one window's kept records.  Offsets are global: nib_off = byte offset of the record's first nibble byte
// in the nibble store (its quals start at base offset 2 * nib_off of the qual store), name_off = offset in the name store.
// With rows (set_rows): meta_off / meta_len = the record's metadata text M(r) in the metadata store (its 36 reported values
// without SKIP_ALIGN, tab-joined), f0_len = the length of its field 0, the prefix of M(r).
struct Stage {
  u64 rec0 = 0, nib0 = 0, name0 = 0, meta0 = 0;        // store sizes before this window (the first record / byte this window adds)
  u64 n_rec = 0, n_nib = 0, n_name = 0, n_meta = 0;    // what this window adds
  u8* nib = nullptr; u8* qual = nullptr; char* name = nullptr;
  u64* umi = nullptr; u32* cb = nullptr; u64* nib_off = nullptr; u32* lseq = nullptr; u16* flag = nullptr; u64* name_off = nullptr; u8* name_len = nullptr;
  u64* ordinal = nullptr;
  char* meta = nullptr; u64* meta_off = nullptr; u32* meta_len = nullptr; u32* f0_len = nullptr;
};

struct Device;   // the store, the grouping buffers and the stream (bam_group.cu)

int create(int device, Device** out);
void destroy(Device*);
void* stream_of(Device*);                                  // cudaStream_t: the library contexts are created on it
int sync(Device*);                                         // waits for everything queued on that stream
// Rows mode (before the first stage): every record also carries its metadata text, and group_reserve() includes the row stage.
void set_rows(Device*, bool rows);
// Waits until the staging slot's previous upload has run, sizes it for this window and fills rec0 / nib0 / name0 / meta0.
int stage(Device*, u64 n_rec, u64 n_nib, u64 n_name, u64 n_meta, Stage*& st);
// Queues the copies of the staged window (plain cudaMemcpyAsync).  reserve: with a budget, the bytes the grouping will
// need on top of the store (group_reserve); a store array grows only so far that the store plus reserve stays in budget.
int upload(Device*, u64 reserve = 0);

// Device-memory budget.  Every cudaMalloc / cudaFree of this file goes through one counter (peak_bytes); with a budget B > 0
// an allocation that would take the counter over B fails, and a store array that grows keeps old + new copies within B.
void set_budget(Device*, u64 budget_bytes);
u64 peak_bytes(Device*);
// Drops the store and the pair arrays of the previous pass (after its batches ran): the next pass starts empty.
int begin_pass(Device*);
// Bytes group() allocates at its peak for n records and ncb CB ids: the sort and scope arrays plus the pair arrays (at most
// one pair per record).
u64 group_reserve(Device*, u64 n, u64 ncb);
// Whether a store of R records, NB nibble bytes, NM name bytes and NT metadata bytes, grown from the present arrays as
// upload() grows them, and then `reserve` bytes more, stays within the budget at every moment.
bool fits(Device*, u64 R, u64 NB, u64 NM, u64 NT, u64 reserve);
// Keeps the records whose bucket is below hi, in their order, in place: nibbles, quals, names, metadata and per-record
// arrays move down through one bounded scratch tile and the offsets are rebased.  Allocates within the budget.
int compact(Device*, u32 hi);
// The most device bytes a store of R / NB / NM grown from the present arrays to exactly what it needs, plus reserve, would
// hold at any moment: what fits() must find within the budget.
u64 need_bytes(Device*, u64 R, u64 NB, u64 NM, u64 NT, u64 reserve);
// Shrinks every store array to its contents (plus the read-past padding) where the budget has room for the copy: arrays
// that grew for records a compaction dropped stop holding room another array needs.
int trim(Device*);

struct Grouped {
  u64 n_records = 0, n_scopes = 0, n_pairs = 0;
  std::vector<u64> scope_pair0;   // n_scopes + 1: first pair of every scope
  std::vector<u32> scope_cb;      // CB id (the producer's dictionary) of every scope's first record
};
// cb_rank[id] = rank of CB id in byte order, cb_prefix[id] = id of its CB[..len-2]
int group(Device*, const std::vector<u32>& cb_rank, const std::vector<u32>& cb_prefix, Grouped& g);
// Fills a device-resident NB_SEQ_BAM4 batch over pairs [p0, p1) whose scope ids are local to the batch (scope - scope0);
// bulk mode: a whole-run batch (scope0 unused).
int batch(Device*, u64 p0, u64 p1, u64 scope0, u32 max_read_len, nb_batch& b);
// Test hook: per pair the file ordinals of both slots, their flags and clipped lengths.
int pairs_to_host(Device*, std::vector<u64>& ord1, std::vector<u64>& ord2, std::vector<u8>& f1, std::vector<u8>& f2, std::vector<u32>& l1, std::vector<u32>& l2);
// Test hook: per pair the base offsets of both slots into the store, and the nibble and qual stores as they are now.
int slots_to_host(Device*, std::vector<u64>& off1, std::vector<u64>& off2, std::vector<u8>& nib, std::vector<u8>& qual);
// ---- bulk mode (nb_process_bam_bulk): FASTQ-mode counts of a BAM without cell barcodes, mates paired by name on the device
// Before the first stage: the store keeps nibbles, names, offsets, lengths, flags and ordinals only (no quals, UMI keys or
// CB ids are staged or uploaded), and batch() hands out whole-run batches (no scope ids, no quals; r2 = NULL single-end).
void set_bulk(Device*, bool bulk);
struct BulkPairs {
  u64 n_pairs = 0;
  u64 singletons = 0, unsplit = 0, multi = 0;   // dropped records: templates of one record, of two that are not READ1-only + READ2-only, of three or more
  u32 max_len = 0;                              // longest read of a pair
};
// After the last upload.  paired: every kept record has flag 0x1 (else none has): a template is the kept records with
// byte-equal QNAME, and one of exactly two records, one READ1-only (0x40 without 0x80) and one READ2-only, is a pair
// (R1 in slot 1); every other record is dropped.  The name key is a 64-bit hash of the QNAME (hash_bits < 64 keeps its
// low bits: tests force collisions); one radix sort of (key -> kept index), runs of equal key, and per run a count pass,
// a scan and a write pass resolve the templates by exact name compare (a thread per run, a warp per run of more than 32
// records).  Single-end: one slot per kept record.  A REVERSE record's slot carries NB_FLAG_REVCOMP_FASTQ.  No TSO clip.
int pair_bulk(Device*, bool paired, u32 hash_bits, BulkPairs& bp);

u64 store_records(Device*);     // records in the store
u64 store_bytes(Device*);       // device bytes of the record store (nibbles, quals, names, per-record keys)
u64 group_bytes(Device*);       // device bytes of the sort, scope and pair arrays
u64 meta_bytes(Device*);        // device bytes of the metadata store (rows mode; part of store_bytes)

// ---- the rows of nb_process_bam_rows_any_order, assembled on the device
// Row buffer cap: NB_BAM_ROWS_BUFFER_KB, default 64 MB; independent of the batch size.
u64 rows_buffer_cap();
// After group(): allocates, within the budget, the per-read / per-pair result buffers and the row stage's scratch for
// batches of up to max_batch_pairs pairs, and the row buffer.  Released by begin_pass / destroy.  group_reserve() holds
// these, 64 KB of callset texts and the reason table; texts beyond that and a row buffer grown for an oversize scope are
// allocated by rows_build within the budget but outside the reserve (NB_ERR_CUDA naming the bytes when they do not fit).
int rows_begin(Device*, u64 max_batch_pairs);
// The device result buffers nb_align_batch writes for a batch of this device (NB_MEM_DEVICE).
void rows_results(Device*, nb_read_result** rres, nb_pair_result** pres);
// What one batch of one library gives the row stage, after nb_counts_finalize: its pairs [p0, p1) of the grouping, the
// device count rows (nb_counts_device_rows), the device slot map (nb_counts_device_slot_map) and the text of every callset
// id of that finalize (group names joined by ','): feats[feat_off[c] .. feat_off[c + 1]).  reasons[r] = nb_reason_str(r).
struct RowsBatch {
  u64 p0 = 0, p1 = 0;
  const void* row_scope = nullptr; const void* row_callset = nullptr; const void* row_count = nullptr; u64 n_rows = 0;
  const void* slot_map = nullptr; u64 n_slots = 0;
  const std::string* feats = nullptr; const std::vector<u64>* feat_off = nullptr; const std::vector<std::string>* reasons = nullptr;
};
struct RowsStats { u64 rows = 0, bytes = 0, chunks = 0, batches = 0, max_chunks = 0; double t_device = 0; };
// Plans the batch's rows on the device (representatives, zero rows, byte lengths, CUB scans), then writes them in chunks of
// whole scopes into the row buffer; each chunk is copied into pinned memory (two buffers, alternating) and handed to
// sink(bytes, n) in order.  The sink may go on reading a buffer until its next call returns, not longer.
int rows_build(Device*, const RowsBatch&, const std::function<int(const char*, u64)>& sink, RowsStats& st);

}  // namespace nbg
