// host.hpp — host-side types shared by the library loader, the index builder and the CUDA context.
#pragma once
#include <cstdint>
#include <string>
#include <vector>

#include "../../include/nimble_b200.h"

typedef uint8_t u8;
typedef uint16_t u16;
typedef uint32_t u32;
typedef uint64_t u64;
typedef int64_t i64;

namespace nb {

constexpr int K = 30;  // Kmer30, src/align.rs:21
constexpr u64 KMASK = (1ULL << 60) - 1;
constexpr u32 NONE32 = 0xFFFFFFFFu;

void set_error(const std::string& msg);
int fail(int code, const std::string& msg);

// DnaString::from_acgt_bytes: ACGT either case -> 0..3, anything else -> 0 ('A')
inline u8 base_code(u8 c) {
  switch (c) {
    case 'A': case 'a': return 0;
    case 'C': case 'c': return 1;
    case 'G': case 'g': return 2;
    case 'T': case 't': return 3;
    default: return 0;
  }
}

int natural_lexical_cmp(const std::string& a, const std::string& b);

// nb_process_samples (fastq.cpp): a failing sample keeps the code and message of its single run behind "sample <name>: "
inline int sample_failed(const char* name, int rc) { return fail(rc, std::string("sample ") + name + ": " + nb_last_error()); }
// its bulk samples (bam.cpp), after the checks: inputs[2 s] = sample s's BAM, outs[s * n_refs + li] = library li's TSV of it
int bulk_samples(const char* const* names, const char* const* inputs, u32 n_samples, const char* const* reference_json, const std::vector<std::string>& outs,
                 u32 n_refs, int strand_filter, int num_cores, int device);

}  // namespace nb

// Reference + AlignFilterConfig (src/reference_library.rs:11-17, src/align.rs:80-95) plus the integer tables the
// device pair stage uses instead of the reference's per-pair string work (src/align.rs:144-375, 802-864).
struct nb_library {
  nb_config cfg;
  std::vector<std::string> headers;
  std::vector<std::vector<std::string>> columns;  // column-major, rows include the §rev rows
  u32 group_on = 0, name_idx = 0, seq_idx = 0;
  // ---- derived by finalize()
  bool derived = false;
  bool injective = false;            // row -> (feature, orientation) is one-to-one and parse_calls == strip_suffix
  std::string irregular_reason;
  bool no_dedup = false;             // headers[group_on] == "nt_sequence" (src/align.rs:810)
  u32 n_features = 0;
  std::vector<u32> row_fid;          // row -> feature id
  std::vector<u8> row_rev;           // row -> 1 if parse_calls says reverse
  std::vector<u32> row_of;           // [2*fid + rev] -> row or NONE32
  std::vector<u32> feat_group;       // fid -> group rank of unmap(feature) row, NONE32 when unmap would panic
  std::vector<std::string> group_names;  // rank -> string; ranks follow natural_lexical_cmp
  std::vector<u32> group_byte_rank;      // rank -> position of that string in plain byte order (distinct strings: no ties)
  void finalize();
  u32 n_rows() const { return columns.empty() ? 0 : (u32)columns[0].size(); }
};

// Flat index artefact (DESIGN.md "Index layout"); the same bytes are uploaded to HBM.
struct NodeRec { u32 start_lo; u32 len; u32 colour; u32 exts_hi; };  // exts_hi: lext | rext<<4 | start_hi<<8
struct nb_index {
  // k-mer table (khash.h): bucket b = slots 4b .. 4b+3 (one 32-byte sector of keys); home bucket or the next with room
  std::vector<u64> table_key;  // device k-mer form (first base in the low bits) | bit63 set when occupied
  std::vector<u64> table_val;  // node | off<<32
  u64 table_buckets = 0;       // n_buckets (any size, khash.h); table_key.size() == 4 * n_buckets
  std::vector<u64> unitig;     // 2-bit packed, base i at bits 2*(i&31) of word i>>5, 2 zero pad words
  std::vector<NodeRec> node;
  std::vector<u32> redge, ledge;  // 4 per node, NONE32 when absent
  std::vector<u32> col_off, col_ids;   // colour c = col_ids[col_off[c] .. col_off[c+1]); universe lists are appended after the colours
  // Per colour {uni_off, uni_size, mask_lo, mask_hi}: sequences that ever share a colour form components ("universes");
  // for a component of <= 64 sequences every colour is a 64-bit mask over its sorted member list
  // col_ids[uni_off .. uni_off+uni_size), so intersecting two colours is one AND.  uni_size == 0: list path only.
  std::vector<u32> col_meta;
  u64 n_kmers = 0, unitig_bases = 0, n_sequences = 0;
  u64 device_bytes() const {
    return table_key.size() * 16 + unitig.size() * 8 + node.size() * 16 + (redge.size() + ledge.size()) * 4 + (col_off.size() + col_ids.size() + col_meta.size()) * 4;
  }
};

int nb_build_index_impl(const std::vector<std::vector<u8>>& seqs, int n_threads, nb_index** out);
int nb_build_universes(nb_index* ix, u32 n_seq);
int nb_build_index_gpu(const std::vector<std::vector<u8>>& seqs, int device, int n_threads, nb_index** out);
