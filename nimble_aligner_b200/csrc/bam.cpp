// bam.cpp — BAM-mode host pipeline: BGZF inflate on host threads, BAM record decode, UMI / cell-barcode grouping with the
// reference's quirks, scoped batches into the device path, gzip TSV rows.
//
// Mirrors (paths under /root/reference):
//   src/parse/sorted_bam_reader.rs:31-185  fill_buffer / add_dummy_paired_reads / filter_paired_reads / next
//   src/parse/bam.rs:70-287                UMIReader: group key = UMI + CB[..len-2], 13-base TSO clip iff len == 124,
//                                          38 metadata fields per record (BAM_FIELDS_TO_REPORT 9-49)
//   src/process/bam.rs:45-243              producer loop (the last group is never sent when there are >= 2, 163-179),
//                                          header + row format (22-42, 90-121), zero rows (329-353), reasons (356-396)
// The reference runs cores-1 consumer threads over an mpsc channel; here one GPU context per library takes whole
// batches of groups (scope_id = group number) and the row order is group order (the reference's order is arbitrary).
// The device needs a tenth of the time of the host stages around it, so those are written for throughput: the file is
// mapped and its BGZF blocks inflated in parallel by inflate.hpp (CRC-32 checked), the window's record chain and UMI runs
// are found on all threads, a row's 2 x 36 values are formatted in one pass over each record's aux block, and the rows are
// compressed in parallel gzip members by deflate_fast.hpp.
#include <unistd.h>
#include <zlib.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <future>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include <errno.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include "host.hpp"
#include "inflate.hpp"
#include "deflate_fast.hpp"
#include "bam_group.hpp"

using namespace nb;
typedef int32_t i32;

namespace {

const char* FIELDS[38] = {"QNAME", "QUAL", "REVERSE", "MATE_REVERSE", "PAIRED", "PROPER_PAIRED", "PAIR_ORIENTATION", "UNMAPPED", "MATE_UNMAPPED",
  "FIRST_IN_TEMPLATE", "LAST_IN_TEMPLATE", "STRAND", "MAPQ", "POS", "MATE_POS", "SEQ", "SEQ_LEN", "INSERT_SIZE", "QUALITY_FAILED", "SECONDARY",
  "DUPLICATE", "SUPPLEMENTARY", "NH", "HI", "AS", "GN", "TX", "AN", "nM", "fx", "RE", "CR", "CY", "CB", "UR", "UY", "UB", "SKIP_ALIGN"};
const size_t CLIP_LENGTH = 13;   // src/parse/bam.rs:7

// ------------------------------------------------------------------ BGZF: all blocks located up front, inflated by a thread pool
// byte buffer without value-initialisation: the inflate threads are the first to touch the pages (a zero-filling
// std::vector costs a single-threaded pass over gigabytes before the first block is inflated)
struct RawBuf {
  u8* p = nullptr; size_t n = 0;
  ~RawBuf() { free(p); }
  bool alloc(size_t bytes) { free(p); p = (u8*)malloc(bytes ? bytes : 1); n = p ? bytes : 0; return p != nullptr; }
  void release() { free(p); p = nullptr; n = 0; }
  size_t size() const { return n; } const u8* data() const { return p; } u8* data() { return p; }
  const u8& operator[](size_t i) const { return p[i]; } u8& operator[](size_t i) { return p[i]; }
};

// Streaming BGZF reader: the file is consumed window by window (about `target` inflated bytes at a time), each window's
// blocks inflated in parallel on the host threads; nothing but the current windows is ever resident (the reference's reader
// holds one UMI at a time, src/parse/sorted_bam_reader.rs:31-107, and its channel 50 groups, src/process/bam.rs:149).
struct Bgzf {
  FILE* f = nullptr; std::string path; std::vector<u8> cbuf; size_t cpos = 0, cend = 0; bool file_done = false;
  const u8* map = nullptr; size_t map_size = 0;   // a regular file is mapped: the blocks are inflated straight out of the page cache (fread copied every compressed byte once more, on one thread)
  RawBuf data;   // whole-stream mode (window = everything): kept for callers that want one buffer
  ~Bgzf() { if (map) munmap((void*)map, map_size); if (f) fclose(f); }
  const u8* cdata() const { return map ? map : cbuf.data(); }
  int open(const std::string& p) {
    path = p; f = fopen(p.c_str(), "rb");
    if (!f) return fail(NB_ERR_IO, "could not open " + p);
    cpos = cend = 0; file_done = false;
    struct stat st;
    if (!getenv("NB_BAM_NO_MMAP") && fstat(fileno(f), &st) == 0 && S_ISREG(st.st_mode) && st.st_size > 0) {
      void* q = mmap(nullptr, (size_t)st.st_size, PROT_READ, MAP_PRIVATE, fileno(f), 0);
      if (q != MAP_FAILED) { map = (const u8*)q; map_size = (size_t)st.st_size; madvise(q, map_size, MADV_SEQUENTIAL); cend = map_size; file_done = true; }
    }
    return NB_OK;
  }
  // Appends the inflated bytes of the next blocks (at least one block, about `target` bytes, everything left when target is
  // SIZE_MAX) behind the first `keep` bytes of `out` (the carry-over of the previous window, already in place).  eof: the
  // file is exhausted after this window.
  int next(RawBuf& out, size_t keep, size_t target, int threads, size_t& n_out, bool& eof) {
    struct Blk { size_t off, clen, uoff, ulen; };
    std::vector<Blk> blks; size_t utot = 0;
    for (;;) {
      const size_t avail = cend - cpos;
      if (avail < 18) { if (!refill(18)) { if (avail == 0) break; return fail(NB_ERR_PARSE, "truncated BGZF block at the end of " + path); } continue; }
      const u8* const cb = cdata(); const u8* h = cb + cpos;
      if (h[0] != 31 || h[1] != 139 || h[2] != 8 || !(h[3] & 4)) return fail(NB_ERR_PARSE, "not a BGZF file: " + path);
      // every size field comes from the file: nothing is read or handed to inflate() before it is checked against the
      // block and the bytes that are really there (a damaged BAM must fail with NB_ERR_PARSE, never read out of bounds)
      const size_t xlen = h[10] | (h[11] << 8);
      if (avail < 12 + xlen) { if (!refill(12 + xlen)) return fail(NB_ERR_PARSE, "corrupt BGZF block (extra field runs past the end of the file) in " + path); continue; }
      size_t q = cpos + 12, xend = q + xlen, bsize = 0;
      while (q + 4 <= xend) { size_t slen = cb[q + 2] | (cb[q + 3] << 8); if (q + 4 + slen > xend) break; if (cb[q] == 'B' && cb[q + 1] == 'C' && slen == 2) bsize = (cb[q + 4] | (cb[q + 5] << 8)) + 1; q += 4 + slen; }
      if (!bsize || 12 + xlen + 8 > bsize) return fail(NB_ERR_PARSE, "corrupt BGZF block in " + path);
      if (avail < bsize) { if (!refill(bsize)) return fail(NB_ERR_PARSE, "corrupt BGZF block (runs past the end of the file) in " + path); continue; }
      const size_t isize = cb[cpos + bsize - 4] | (cb[cpos + bsize - 3] << 8) | (cb[cpos + bsize - 2] << 16) | ((size_t)cb[cpos + bsize - 1] << 24);
      if (isize > 65536) return fail(NB_ERR_PARSE, "corrupt BGZF block (ISIZE beyond 64 KiB) in " + path);
      blks.push_back({xend, bsize - (xend - cpos) - 8, utot, isize});
      utot += isize; cpos += bsize;
      if (utot >= target) break;
    }
    // peek: is anything left after this window?
    if (cend == cpos && !file_done) refill(65536);
    eof = file_done && cend == cpos;
    // grow `out` keeping its first `keep` bytes
    if (out.size() < keep + utot) { RawBuf nb2; if (!nb2.alloc(keep + utot + (utot >> 3) + 64)) return fail(NB_ERR_IO, "out of memory inflating " + path); if (keep) memcpy(nb2.data(), out.data(), keep); std::swap(out.p, nb2.p); std::swap(out.n, nb2.n); }
    std::atomic<size_t> next_blk(0); std::atomic<int> bad(0);
    u8* dst = out.data() + keep; const u8* src = cdata();
    const bool check_crc = !getenv("NB_BAM_NO_CRC");
    auto work = [&]() {
      // inflate.hpp's decoder, one block in one piece into its place in the window (it never writes past the block's
      // ISIZE bytes: the neighbouring blocks are being written by other threads); the block's CRC-32 is checked like htslib does
      std::unique_ptr<nbz::Inflater> inf(new nbz::Inflater());
      for (;;) { size_t i = next_blk.fetch_add(1); if (i >= blks.size()) break; const Blk& b = blks[i]; if (!b.ulen) continue;
        inf->start(src + b.off, src + b.off + b.clen);
        u8* const o = dst + b.uoff; u8* q = o;
        const int rc = inf->run(o, q, o + b.ulen);
        u32 want; memcpy(&want, src + b.off + b.clen, 4);
        if (rc != nbz::INF_END || (size_t)(q - o) != b.ulen || (check_crc && (u32)crc32_z(0L, o, b.ulen) != want)) bad = 1; }
    };
    std::vector<std::thread> th; for (int t = 1; t < std::max(1, threads) && (size_t)t < blks.size(); t++) th.emplace_back(work);
    work(); for (auto& t : th) t.join();
    if (bad) return fail(NB_ERR_PARSE, "BGZF inflate failed in " + path);
    n_out = utot;
    return NB_OK;
  }
  // whole file into `data` (tests and the whole-file fallback)
  int load(const std::string& p, int threads) { int rc = open(p); if (rc) return rc; size_t n = 0; bool eof = false; rc = next(data, 0, SIZE_MAX, threads, n, eof); if (rc) return rc; data.n = n; return NB_OK; }
 private:
  // makes at least `want` unread bytes available when the file has them; false when nothing more could be read
  bool refill(size_t want) {
    if (file_done) return false;
    // blocks already handed out in this window are still referenced by offset: compaction only happens between windows,
    // so within a window the buffer only grows
    size_t need = cend + std::max<size_t>(want, (size_t)8 << 20);
    if (cbuf.size() < need) cbuf.resize(need + (need >> 2));
    size_t got = fread(&cbuf[cend], 1, cbuf.size() - cend, f);
    if (got == 0) { file_done = true; return false; }
    cend += got;
    return true;
  }
 public:
  // between windows: drop the consumed compressed bytes
  void compact() { if (map) return; if (cpos) { memmove(cbuf.data(), cbuf.data() + cpos, cend - cpos); cend -= cpos; cpos = 0; } }
};

struct Rec {   // one decoded BAM record (views into Bgzf::data stay valid for the run)
  const u8* p = nullptr;        // start of the fixed fields (after block_size)
  u32 block = 0;
  int skip_align = -1;          // the "SK" string aux the reference appends (sorted_bam_reader.rs:114-121): -1 absent (-p mode), 0 "FALSE", 1 "TRUE"
  const char* cb = nullptr; const char* umi = nullptr; u32 cb_len = 0, umi_len = 0;   // CB:Z and UB:Z (else UR:Z) values, found once by scan_keys(); nullptr = absent / not a string
  // one pass over the aux block for the grouping keys (same first-match-by-two-bytes rule as aux_z)
  void scan_keys() {
    const u8* a = aux(); const u8* e = end(); const char* ub = nullptr; const char* ur = nullptr; u32 ub_len = 0, ur_len = 0; bool seen_cb = false, seen_ub = false, seen_ur = false;
    cb = umi = nullptr; cb_len = umi_len = 0;
    while (a + 3 <= e) {
      char t0 = (char)a[0], t1 = (char)a[1], ty = (char)a[2]; a += 3; const u8* v = a; u32 zlen = 0; bool zok = false;
      if (!aux_skip(ty, a, e, zlen, zok)) break;
      if (t0 == 'C' && t1 == 'B' && !seen_cb) { seen_cb = true; if (ty == 'Z' && zok) { cb = (const char*)v; cb_len = zlen; } }
      else if (t0 == 'U' && t1 == 'B' && !seen_ub) { seen_ub = true; if (ty == 'Z' && zok) { ub = (const char*)v; ub_len = zlen; } }
      else if (t0 == 'U' && t1 == 'R' && !seen_ur) { seen_ur = true; if (ty == 'Z' && zok) { ur = (const char*)v; ur_len = zlen; } }
    }
    umi = ub ? ub : ur; umi_len = ub ? ub_len : ur_len;
  }
  // Steps `a` over one aux value of type `ty` without ever passing `e` (the end of the record): false when the value is
  // cut off or the type is unknown (the scan stops there).  Z / H: zlen = bytes before the NUL, zok = a NUL was found
  // inside the record (an unterminated string is not a value: strlen() on it would run off the record).
  static bool aux_skip(char ty, const u8*& a, const u8* e, u32& zlen, bool& zok) {
    size_t left = (size_t)(e - a), w = 0;
    switch (ty) {
      case 'A': case 'c': case 'C': w = 1; break; case 's': case 'S': w = 2; break; case 'i': case 'I': case 'f': w = 4; break;
      case 'Z': case 'H': { const u8* z = (const u8*)memchr(a, 0, left); if (!z) { a = e; return false; } zlen = (u32)(z - a); zok = true; a = z + 1; return true; }
      case 'B': { if (left < 5) { a = e; return false; } char st = (char)a[0]; u32 n; memcpy(&n, a + 1, 4); size_t ew = (st == 'c' || st == 'C') ? 1 : (st == 's' || st == 'S') ? 2 : 4;
                  if ((size_t)n > (left - 5) / ew) { a = e; return false; } a += 5 + ew * n; return true; }
      default: a = e; return false;
    }
    if (w > left) { a = e; return false; }
    a += w; return true;
  }
  const char* qname_ptr() const { return (const char*)p + 32; } u32 qname_len() const { u32 l = l_read_name(); return l ? l - 1 : 0; }
  i32 refid() const { return rd32(0); } i32 pos() const { return rd32(4); }
  u32 l_read_name() const { return p[8]; } u32 mapq() const { return p[9]; }
  u32 n_cigar() const { return p[12] | (p[13] << 8); } u32 flag() const { return p[14] | (p[15] << 8); }
  u32 l_seq() const { return (u32)rd32(16); } i32 mrefid() const { return rd32(20); } i32 mpos() const { return rd32(24); } i32 tlen() const { return rd32(28); }
  i32 rd32(size_t o) const { i32 v; memcpy(&v, p + o, 4); return v; }
  std::string qname() const { u32 l = l_read_name(); return std::string((const char*)p + 32, l ? l - 1 : 0); }
  const u8* seq4() const { return p + 32 + l_read_name() + 4 * n_cigar(); }
  const u8* qual() const { return seq4() + (l_seq() + 1) / 2; }
  const u8* aux() const { return qual() + l_seq(); }
  const u8* end() const { return p + block; }
  bool is_paired() const { return flag() & 1; } bool is_reverse() const { return flag() & 16; } bool is_first() const { return flag() & 64; }
  // Aux::String lookup by the first two bytes of `tag` (htslib bam_aux_get semantics)
  bool aux_z(const char* tag, std::string& out) const {
    const u8* a = aux(); const u8* e = end();
    while (a + 3 <= e) {
      char t0 = (char)a[0], t1 = (char)a[1], ty = (char)a[2]; a += 3; const u8* v = a; u32 zlen = 0; bool zok = false;
      bool ok = aux_skip(ty, a, e, zlen, zok);
      if (t0 == tag[0] && t1 == tag[1]) { if (ty != 'Z' || !zok) return false; out.assign((const char*)v, zlen); return true; }
      if (!ok) return false;
    }
    return false;
  }
  std::string seq_ascii() const { static const char* T = "=ACMGRSVTWYHKDBN"; u32 n = l_seq(); std::string s(n, 'N'); const u8* q = seq4(); for (u32 i = 0; i < n; i++) s[i] = T[(q[i >> 1] >> ((~i & 1) << 2)) & 15]; return s; }
};

struct ParsedRec {   // what UMIReader keeps per record: clipped sequence, the 38 string fields, flags for the device
  std::string seq;   // DnaString::from_acgt_bytes(clipped).to_string() (uppercase ACGT)
  std::string qual;  // clipped raw Phred bytes, NOT reversed (the device reverses with NB_FLAG_REVCOMP); field 1 holds the reversed string
  std::vector<std::string> f; bool reverse = false, skip = false;
};

std::string bstr(bool b) { return b ? "true" : "false"; }

void parse_fields(const Rec& r, ParsedRec& o) {   // src/parse/bam.rs:186-236
  bool rev = r.is_reverse(); o.reverse = rev; o.skip = r.skip_align == 1;
  std::string raw = r.seq_ascii(); const u8* q = r.qual(); size_t n = raw.size();
  size_t a = 0, b = n;
  if (n == 124) { if (rev) b = n - CLIP_LENGTH; else a = CLIP_LENGTH; }                 // strip_nonbio_regions 258-268
  o.seq.assign(b - a, 'A');
  for (size_t i = a; i < b; i++) { char c = raw[i]; o.seq[i - a] = (c == 'C' || c == 'c') ? 'C' : (c == 'G' || c == 'g') ? 'G' : (c == 'T' || c == 't') ? 'T' : 'A'; }
  o.qual.assign((const char*)q + a, b - a);
  std::string qfield = o.qual; if (rev) std::reverse(qfield.begin(), qfield.end());     // strip_nonbio_regions_qual 271-286
  u32 fl = r.flag(); bool paired = fl & 1, unm = fl & 4, munm = fl & 8, mrev = fl & 32, first = fl & 64;
  std::string orient = "None";   // rust-htslib read_pair_orientation
  if (paired && !unm && !munm && r.refid() == r.mrefid() && r.pos() != r.mpos()) {
    i64 p1, p2; bool f1, f2;
    if (first) { p1 = r.pos(); p2 = r.mpos(); f1 = !rev; f2 = !mrev; } else { p1 = r.mpos(); p2 = r.pos(); f1 = !mrev; f2 = !rev; }
    if (p1 < p2) orient = std::string(f1 ? "F1" : "R1") + (f2 ? "F2" : "R2"); else orient = std::string(f2 ? "F2" : "R2") + (f1 ? "F1" : "R1");
  }
  o.f.resize(38);
  for (int i = 0; i < 38; i++) {
    std::string z;
    if (i == 37 && r.skip_align >= 0) { o.f[i] = r.skip_align ? "TRUE" : "FALSE"; continue; }   // the appended "SK" string aux
    if (r.aux_z(FIELDS[i], z)) { o.f[i] = z; continue; }
    switch (i) {
      case 0: o.f[i] = r.qname(); break; case 1: o.f[i] = qfield; break; case 2: o.f[i] = bstr(rev); break; case 3: o.f[i] = bstr(mrev); break;
      case 4: o.f[i] = bstr(paired); break; case 5: o.f[i] = bstr(fl & 2); break; case 6: o.f[i] = orient; break; case 7: o.f[i] = bstr(unm); break;
      case 8: o.f[i] = bstr(munm); break; case 9: o.f[i] = bstr(first); break; case 10: o.f[i] = bstr(fl & 128); break; case 11: o.f[i] = rev ? "-" : "+"; break;
      case 12: o.f[i] = std::to_string(r.mapq()); break; case 13: o.f[i] = std::to_string(r.pos()); break; case 14: o.f[i] = std::to_string(r.mpos()); break;
      case 15: o.f[i] = o.seq; break; case 16: o.f[i] = std::to_string(r.l_seq()); break; case 17: o.f[i] = std::to_string(r.tlen()); break;
      case 18: o.f[i] = bstr(fl & 512); break; case 19: o.f[i] = bstr(fl & 256); break; case 20: o.f[i] = bstr(fl & 1024); break; case 21: o.f[i] = bstr(fl & 2048); break;
      default: o.f[i].clear(); break;   // non-string aux (NH, HI, AS, nM, RE ...) -> String::new()
    }
  }
}

void parallel_ranges(int threads, size_t n, const std::function<void(size_t, size_t, int)>& fn) {
  if (threads <= 1 || n < 2) { fn(0, n, 0); return; }
  std::vector<std::thread> th;
  for (int t = 0; t < threads; t++) th.emplace_back(fn, n * (size_t)t / threads, n * (size_t)(t + 1) / threads, t);
  for (auto& x : th) x.join();
}

// ------------------------------------------------------------------ SortedBamReader (src/parse/sorted_bam_reader.rs)
inline bool same(const char* a, u32 al, const char* b, u32 bl) { return al == bl && (al == 0 || !memcmp(a, b, al)); }
inline int cmp_bytes(const char* a, u32 al, const char* b, u32 bl) { int c = memcmp(a, b, std::min(al, bl)); return c ? c : (al < bl ? -1 : al > bl ? 1 : 0); }

struct SortedReader {
  const Bgzf& z; size_t cur = 0; bool force_paired; bool header_done = false;
  std::vector<Rec> all; size_t next_rec = 0;   // every record of the file, keys already scanned (prepare())
  std::string current_umi, next_umi; std::vector<Rec> buffer, next_records;   // buffer is popped from the back
  SortedReader(const Bgzf& zz, bool fp) : z(zz), force_paired(fp) {}
  int skip_header() {
    const RawBuf& d = z.data;
    if (d.size() < 12 || memcmp(d.data(), "BAM\1", 4)) return fail(NB_ERR_PARSE, "not a BAM file");
    u32 l_text; memcpy(&l_text, &d[4], 4); size_t p = 8 + (size_t)l_text; u32 n_ref; if (p + 4 > d.size()) return fail(NB_ERR_PARSE, "truncated BAM header"); memcpy(&n_ref, &d[p], 4); p += 4;
    for (u32 i = 0; i < n_ref; i++) { if (p + 4 > d.size()) return fail(NB_ERR_PARSE, "truncated BAM header"); u32 l; memcpy(&l, &d[p], 4); p += 4 + (size_t)l + 4; }
    cur = p; header_done = true; return NB_OK;
  }
  // locate the records (serial walk over block sizes), then scan their grouping keys on `threads` threads
  int prepare(int threads) {
    const RawBuf& d = z.data;
    while (cur + 4 <= d.size()) {
      u32 bs; memcpy(&bs, &d[cur], 4);
      if (bs < 32 || cur + 4 + bs > d.size()) break;
      Rec r; r.p = &d[cur + 4]; r.block = bs;
      // l_read_name, n_cigar and l_seq come from the file: qname / cigar / 4-bit bases / quals must lie inside the record
      if (32ull + r.l_read_name() + 4ull * r.n_cigar() + ((u64)r.l_seq() + 1) / 2 + (u64)r.l_seq() > bs) return fail(NB_ERR_PARSE, "corrupt BAM record (field lengths exceed its block size)");
      all.push_back(r); cur += 4 + bs;
      if (all.size() == 4096) all.reserve((size_t)((double)d.size() / (double)cur * 4096 * 1.1) + 4096);   // one allocation for the whole file
    }
    parallel_ranges(threads, all.size(), [&](size_t a, size_t b, int) { for (size_t i = a; i < b; i++) all[i].scan_keys(); });
    return NB_OK;
  }
  bool read_record(Rec& r) { if (next_rec >= all.size()) return false; r = all[next_rec++]; return true; }
  int fill_buffer() {   // 31-107
    buffer.clear(); buffer.swap(next_records); next_records.clear();
    current_umi = next_umi;
    Rec r;
    while (read_record(r)) {
      if (!r.is_paired() && force_paired) continue;
      if (!r.cb) continue;
      if (!r.umi) return fail(NB_ERR_PARSE, "Error -- Could not read UMI.");
      if (r.umi_len == 10 && !memcmp(r.umi, "AAAAAAAAAA", 10)) continue;
      if (current_umi.empty()) current_umi.assign(r.umi, r.umi_len);
      if (!same(current_umi.data(), (u32)current_umi.size(), r.umi, r.umi_len)) {
        std::stable_sort(buffer.begin(), buffer.end(), [](const Rec& a, const Rec& b) { return cmp_bytes(a.cb, a.cb_len, b.cb, b.cb_len) < 0; });
        next_records.push_back(r); next_umi.assign(r.umi, r.umi_len);
        return NB_OK;
      }
      buffer.push_back(r);
    }
    return NB_OK;   // end of file: this last buffer is NOT sorted by CB (quirk kept)
  }
  std::vector<Rec> tmp;   // scratch reused across buffers (one UMI buffer is a handful of records: allocation would dominate)
  void add_dummy_paired_reads() {   // 109-125
    std::vector<Rec>& nb2 = tmp; nb2.clear();
    for (const Rec& r : buffer) { Rec m = r; m.skip_align = 0; nb2.push_back(m); if (!r.is_paired()) { Rec d = r; d.skip_align = 1; nb2.push_back(d); } }
    buffer.swap(nb2);
  }
  void filter_paired_reads() {      // 127-162
    std::vector<Rec>& out = tmp; out.clear(); size_t i = 0;
    while (i < buffer.size()) {
      if (i + 1 >= buffer.size()) break;
      if (same(buffer[i].qname_ptr(), buffer[i].qname_len(), buffer[i + 1].qname_ptr(), buffer[i + 1].qname_len())) {
        if (buffer[i].is_first()) { out.push_back(buffer[i]); out.push_back(buffer[i + 1]); } else { out.push_back(buffer[i + 1]); out.push_back(buffer[i]); }
        i += 2;
      } else i += 1;
    }
    buffer.swap(out);
  }
  // 164-185; returns 1 record, 0 end of input, <0 error
  int next(Rec& r) {
    if (!buffer.empty()) { r = buffer.back(); buffer.pop_back(); return 1; }
    int rc = fill_buffer(); if (rc) return rc;
    if (!force_paired) add_dummy_paired_reads();
    filter_paired_reads();
    std::reverse(buffer.begin(), buffer.end());
    if (buffer.empty()) return 0;
    r = buffer.back(); buffer.pop_back(); return 1;
  }
};

// ------------------------------------------------------------------ UMIReader (src/parse/bam.rs:100-253), on undecoded records:
// the 38 strings per record are only materialised for the rows that get written (and by the writer threads)
struct UmiReader {
  SortedReader rd; std::vector<Rec> current, nextg; std::string current_key, next_key, current_umi, next_umi;
  UmiReader(const Bgzf& z, bool fp) : rd(z, fp) {}
  // returns 1: a following group exists (Some(true)); 0: end of input (None); <0 error
  int get_umi() {
    current.swap(nextg); nextg.clear(); current_key = next_key; next_key.clear(); current_umi = next_umi; next_umi.clear();
    std::string key;
    for (;;) {
      Rec r; int g = rd.next(r);
      if (g < 0) return g;
      if (g == 0) return 0;
      if (!r.umi) return fail(NB_ERR_PARSE, "Error -- Could not read UMI.");
      if (!r.cb) return fail(NB_ERR_PARSE, "Error Read without cell barcode, cannot excise read-mate.");
      key.assign(r.umi, r.umi_len); if (r.cb_len >= 2) key.append(r.cb, r.cb_len - 2);
      if (current_umi.empty()) current_umi.assign(r.umi, r.umi_len);
      if (current_key.empty()) current_key = key;
      if (current_key == key) current.push_back(r);
      else { nextg.push_back(r); next_umi.assign(r.umi, r.umi_len); next_key = key; return 1; }
    }
  }
};

// The groups the producer loop sends, in order (src/process/bam.rs:157-180): records of group g are
// stream[gstart[g] .. gstart[g+1]); the last group is never sent when a group was sent before.
int collect_groups_serial(const Bgzf& z, bool force_paired, int threads, std::vector<Rec>& stream, std::vector<u64>& gstart) {
  UmiReader reader(z, force_paired);
  int rc = reader.rd.skip_header(); if (rc) return rc;
  rc = reader.rd.prepare(threads); if (rc) return rc;
  stream.clear(); gstart.assign(1, 0);
  bool has_aligned = false;
  for (;;) {
    int g = reader.get_umi();
    if (g < 0) return g;
    bool final_umi = g == 0;
    if (final_umi && has_aligned) break;
    stream.insert(stream.end(), reader.current.begin(), reader.current.end()); gstart.push_back(stream.size());
    has_aligned = true;
    if (final_umi) break;
  }
  return NB_OK;
}

// group key of UMIReader: UMI + CB without its last two characters, compared without building the strings
inline bool key_equal(const Rec& a, const Rec& b) {
  u32 ca = a.cb_len >= 2 ? a.cb_len - 2 : 0, cb = b.cb_len >= 2 ? b.cb_len - 2 : 0;
  if (a.umi_len + ca != b.umi_len + cb) return false;
  if (a.umi_len == b.umi_len) return !memcmp(a.umi, b.umi, a.umi_len) && !memcmp(a.cb, b.cb, ca);
  std::string x(a.umi, a.umi_len), y(b.umi, b.umi_len); x.append(a.cb, ca); y.append(b.cb, cb); return x == y;   // different split of the same concatenation
}

// The complete records of d[cur, len) in file order (tail = first byte that is not part of one; a record cut by the end of the
// window is left for the next window).  eof: d holds the end of the file.
int walk_records(const RawBuf& d, size_t len, size_t cur, bool eof, int threads, std::vector<Rec>& all, size_t& tail) {
  all.clear();
  const size_t walk_from = cur;
  // complete records of the window.  The records form a chain (each block_size leads to the next record), and walking it
  // serially was a quarter of the producer's critical path, every step a cache miss on data another core just inflated.
  // So the window is cut into segments walked at the same time: a segment starts at a GUESSED record start (the first
  // offset behind its boundary from which four consecutive records look sound) and the guess is never trusted — the
  // segments are only accepted if each one begins exactly where the previous one's walk ended, else the serial walk runs.
  auto sound = [&](size_t o, size_t& next) -> bool {   // does a complete, self-consistent record start at o?
    if (o + 36 > len) return false;
    u32 bs; memcpy(&bs, &d[o], 4);
    if (bs < 32 || bs > (1u << 24) || o + 4 + bs > len) return false;
    const u8* q = &d[o + 4]; const u32 lrn = q[8], ncig = q[12] | (q[13] << 8); u32 lseq; memcpy(&lseq, q + 16, 4);
    i32 refid; memcpy(&refid, q, 4);
    if (lrn == 0 || refid < -1 || 32ull + lrn + 4ull * ncig + ((u64)lseq + 1) / 2 + (u64)lseq > bs || q[32 + lrn - 1] != 0) return false;
    next = o + 4 + bs; return true;
  };
  bool walked = false;
  const size_t par_min_bytes = getenv("NB_BAM_PAR_MIN_BYTES") ? (size_t)strtoull(getenv("NB_BAM_PAR_MIN_BYTES"), nullptr, 10) : ((size_t)8 << 20);   // (tests force the parallel passes on small files)
  const int WT = (len - cur > par_min_bytes) ? threads : 1;
  if (WT > 1) {
    std::vector<std::vector<Rec>> part(WT); std::vector<size_t> seg_start(WT, 0), seg_end(WT, 0); std::vector<char> ok(WT, 1);
    const size_t span = len - walk_from;
    parallel_ranges(WT, (size_t)WT, [&](size_t ta, size_t tb, int) {
      for (size_t t = ta; t < tb; t++) {
        const size_t lo = walk_from + span * t / WT, hi = walk_from + span * (t + 1) / WT;   // records STARTING in [lo, hi) belong to segment t
        size_t o = lo;
        if (t > 0) {   // guess: first offset >= lo that begins a chain of four sound records (or runs into the window's end)
          bool found = false;
          for (; o < hi && o < lo + ((size_t)1 << 20); o++) { size_t n1 = o, n2; int k = 0; while (k < 4 && sound(n1, n2)) { n1 = n2; k++; } if (k == 4 || (k > 0 && n1 + 4 > len)) { found = true; break; } }
          if (!found) { ok[t] = 0; continue; }
        }
        seg_start[t] = o;
        std::vector<Rec>& out = part[t]; out.reserve((hi - lo) / 160 + 16);
        while (o < hi) { size_t nx; if (!sound(o, nx)) break; Rec r; r.p = &d[o + 4]; r.block = (u32)(nx - o - 4); out.push_back(r); o = nx; }
        seg_end[t] = o;     // first offset this segment did not consume: a record start >= hi, the cut record, or something unsound
      }
    });
    bool good = true;
    for (int t = 0; t < WT && good; t++) good = ok[t] && (t == 0 || seg_start[t] == seg_end[t - 1]);
    if (good) {
      // the last segment's end must be where the serial walk would stop: at a record the window cuts (or at the window's end)
      const size_t e = seg_end[WT - 1]; u32 bs = 0; if (e + 4 <= len) memcpy(&bs, &d[e], 4);
      good = e + 4 > len || (bs >= 32 && e + 4 + bs > len);
      if (good) {
        size_t total = 0; std::vector<size_t> at(WT + 1, 0); for (int t = 0; t < WT; t++) { at[t] = total; total += part[t].size(); }
        all.resize(total);
        parallel_ranges(WT, (size_t)WT, [&](size_t ta, size_t tb, int) { for (size_t t = ta; t < tb; t++) if (!part[t].empty()) memcpy(&all[at[t]], part[t].data(), part[t].size() * sizeof(Rec)); });
        cur = e; walked = true;
      }
    }
  }
  while (!walked && cur + 4 <= len) {
    u32 bs; memcpy(&bs, &d[cur], 4);
    if (bs < 32) { if (!eof) return fail(NB_ERR_PARSE, "corrupt BAM record (block size below the fixed fields)"); break; }   // (trailing garbage at the very end is ignored, as before)
    if (cur + 4 + bs > len) break;                                                        // cut by the window: carried over
    Rec r; r.p = &d[cur + 4]; r.block = bs;
    // l_read_name, n_cigar and l_seq come from the file: qname / cigar / 4-bit bases / quals must lie inside the record
    if (32ull + r.l_read_name() + 4ull * r.n_cigar() + ((u64)r.l_seq() + 1) / 2 + (u64)r.l_seq() > bs) return fail(NB_ERR_PARSE, "corrupt BAM record (field lengths exceed its block size)");
    all.push_back(r); cur += 4 + bs;
  }
  tail = cur;
  return NB_OK;
}

// ------------------------------------------------------------------ windowed producer
// The same stream and groups as collect_groups_serial, computed window by window on `threads` threads with bounded memory.
// The serial readers above define the semantics; this restates them over whole runs: a SortedBamReader buffer is a maximal
// run of kept records with one UMI (the last run of the FILE is the one that is not CB-sorted), buffers are independent,
// the stream ends at the first buffer that is empty after pairing (next() returns None there), UMIReader's groups are runs
// of equal keys, and the last group is never sent when a group was sent before.  A window that is not the file's last one
// holds back its last complete non-empty run and everything behind it (a handful of records), so every group it emits is
// complete and known not to be the last; the held-back bytes open the next window.
// NEED_WHOLE: a kept record has an empty UMI string, or two different UMIs give the same UMI+CB concatenation across a
// window boundary (both quirks of the serial readers that need the whole file): the caller restarts with one window.
const int NEED_WHOLE = 1000;
struct Window {
  RawBuf data; size_t len = 0;                         // inflated bytes: carry-over of the previous window + this window's blocks
  std::vector<Rec> all;                                // complete records, file order, keys scanned
  std::vector<Rec> stream; std::vector<u64> gstart;    // what the producer sends: records and group boundaries
  size_t carry_from = 0;                               // offset in data of the first held-back byte (== len: nothing held back)
};
struct GroupStreamer {
  Bgzf z; bool force_paired = false; int threads = 1; size_t window_bytes = (size_t)256 << 20;
  bool header_done = false, eof = false, ended = false; u64 groups_sent = 0, records_seen = 0; size_t peak_window = 0;
  std::string last_umi, last_cb; bool have_last = false;     // key of the last record sent (cross-window coincidence check)
  double t_inflate = 0, t_scan = 0, t_keys = 0, t_runs = 0, t_emit = 0, t_groups = 0;   // phase times (NB_BAM_STATS)
  static double clk() { timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec + ts.tv_nsec * 1e-9; }
  int open(const std::string& path, bool fp, int th, size_t wb) { force_paired = fp; threads = std::max(1, th); window_bytes = std::max<size_t>(wb, 1 << 16); return z.open(path); }
  // fills w from the file position and the carry-over of `prev` (nullptr for the first window).  done: nothing was produced
  // and nothing more will come.
  int next(Window& w, const Window* prev, bool& done) {
    done = false; w.all.clear(); w.stream.clear(); w.gstart.assign(1, 0); w.len = 0; w.carry_from = 0;
    const bool has_carry = prev && prev->carry_from < prev->len;
    if (ended || (eof && !has_carry)) { done = true; return NB_OK; }
    if (has_carry) {
      const size_t keep = prev->len - prev->carry_from;
      if (w.data.size() < keep + 64) { if (!w.data.alloc(keep + window_bytes + (window_bytes >> 3) + 64)) return fail(NB_ERR_IO, "out of memory"); }
      memcpy(w.data.data(), prev->data.data() + prev->carry_from, keep);
      w.len = keep;
    }
    size_t grow = window_bytes;
    for (;;) {   // (repeats only when the window could not emit anything: one giant UMI run, or a header larger than the window)
      double tc = clk();
      if (!eof) { size_t n_out = 0; int rc = z.next(w.data, w.len, grow, threads, n_out, eof); if (rc) return rc; z.compact(); w.len += n_out; }
      t_inflate += clk() - tc; tc = clk();
      peak_window = std::max(peak_window, w.len);
      size_t cur = 0;
      if (!header_done) {
        const RawBuf& d = w.data; bool ok = w.len >= 12;
        if (ok && memcmp(d.data(), "BAM\1", 4)) return fail(NB_ERR_PARSE, "not a BAM file");
        size_t p = 0;
        if (ok) { u32 l_text; memcpy(&l_text, &d[4], 4); p = 8 + (size_t)l_text; ok = p + 4 <= w.len; }
        if (ok) { u32 n_ref; memcpy(&n_ref, &d[p], 4); p += 4; for (u32 i = 0; i < n_ref && ok; i++) { if (p + 4 > w.len) { ok = false; break; } u32 l; memcpy(&l, &d[p], 4); p += 4 + (size_t)l + 4; } ok = ok && p <= w.len; }
        if (!ok) { if (eof) return fail(NB_ERR_PARSE, w.len < 12 ? "not a BAM file" : "truncated BAM header"); grow *= 2; continue; }
        cur = p;
      }
      size_t cur_end = cur;
      { int rw = walk_records(w.data, w.len, cur, eof, threads, w.all, cur_end); if (rw) return rw; }
      cur = cur_end;
      const RawBuf& d = w.data;
      const size_t par_min_recs = getenv("NB_BAM_PAR_MIN_RECS") ? (size_t)strtoull(getenv("NB_BAM_PAR_MIN_RECS"), nullptr, 10) : 65536;
      const size_t tail = cur;    // first byte that is not part of a complete record
      std::vector<Rec>& all = w.all;
      t_scan += clk() - tc; tc = clk();
      parallel_ranges(threads, all.size(), [&](size_t a, size_t b, int) { for (size_t i = a; i < b; i++) all[i].scan_keys(); });
      t_keys += clk() - tc; tc = clk();
      if (all.size() >= 0xFFFFFFFFull) return fail(NB_ERR_UNSUPPORTED, "more than 2^32 records in one window");
      // which records the sorted reader keeps, and where its UMI runs start: flags in parallel, compaction by thread-local
      // counts; the first offending record IN FILE ORDER decides between the two failures, as the serial loop did
      std::vector<u32> kept; std::vector<size_t> run;
      {
        const int T = all.size() > par_min_recs ? threads : 1;
        std::vector<u8> flag(all.size(), 0); std::vector<size_t> cnt(T + 1, 0), bad_at(T, (size_t)-1); std::vector<int> bad_kind(T, 0);
        parallel_ranges(T, all.size(), [&](size_t a, size_t b, int t) {
          size_t c = 0;
          for (size_t i = a; i < b; i++) {
            const Rec& r = all[i];
            if (!r.is_paired() && force_paired) continue;
            if (!r.cb) continue;
            if (!r.umi) { bad_at[t] = i; bad_kind[t] = 1; break; }
            if (r.umi_len == 10 && !memcmp(r.umi, "AAAAAAAAAA", 10)) continue;
            if (r.umi_len == 0) { bad_at[t] = i; bad_kind[t] = 2; break; }
            flag[i] = 1; c++;
          }
          cnt[t + 1] = c;
        });
        { size_t first = (size_t)-1; int kind = 0; for (int t = 0; t < T; t++) if (bad_at[t] < first) { first = bad_at[t]; kind = bad_kind[t]; }
          if (kind == 1) return fail(NB_ERR_PARSE, "Error -- Could not read UMI.");
          if (kind == 2) return NEED_WHOLE; }
        for (int t = 0; t < T; t++) cnt[t + 1] += cnt[t];
        kept.resize(cnt[T]);
        parallel_ranges(T, all.size(), [&](size_t a, size_t b, int t) { size_t at = cnt[t]; for (size_t i = a; i < b; i++) if (flag[i]) kept[at++] = (u32)i; });
        // run heads
        const size_t nk = kept.size(); std::vector<u8> head(nk, 0); std::vector<size_t> hc(T + 1, 0);
        parallel_ranges(T, nk, [&](size_t a, size_t b, int t) { size_t c = 0; for (size_t j = a; j < b; j++) if (j == 0 || !same(all[kept[j]].umi, all[kept[j]].umi_len, all[kept[j - 1]].umi, all[kept[j - 1]].umi_len)) { head[j] = 1; c++; } hc[t + 1] = c; });
        for (int t = 0; t < T; t++) hc[t + 1] += hc[t];
        run.resize(hc[T]);
        parallel_ranges(T, nk, [&](size_t a, size_t b, int t) { size_t at = hc[t]; for (size_t j = a; j < b; j++) if (head[j]) run[at++] = j; });
      }
      const size_t nr = run.size(); run.push_back(kept.size());
      t_runs += clk() - tc; tc = clk();
      // one run -> the records the sorted reader hands on (CB sort unless it is the file's last run, dummy mates, pairing)
      auto emit_run = [&](size_t r, std::vector<Rec>& out, std::vector<Rec>& buf, std::vector<Rec>& tmp) {
        buf.clear(); for (size_t j = run[r]; j < run[r + 1]; j++) buf.push_back(all[kept[j]]);
        if (!(eof && r + 1 == nr)) std::stable_sort(buf.begin(), buf.end(), [](const Rec& a, const Rec& b) { return cmp_bytes(a.cb, a.cb_len, b.cb, b.cb_len) < 0; });   // the file's last buffer is not sorted (quirk kept)
        if (!force_paired) { tmp.clear(); for (const Rec& x : buf) { Rec m = x; m.skip_align = 0; tmp.push_back(m); if (!x.is_paired()) { Rec d2 = x; d2.skip_align = 1; tmp.push_back(d2); } } buf.swap(tmp); }
        size_t before = out.size(), i = 0;
        while (i + 1 < buf.size()) {   // filter_paired_reads
          if (same(buf[i].qname_ptr(), buf[i].qname_len(), buf[i + 1].qname_ptr(), buf[i + 1].qname_len())) {
            if (buf[i].is_first()) { out.push_back(buf[i]); out.push_back(buf[i + 1]); } else { out.push_back(buf[i + 1]); out.push_back(buf[i]); }
            i += 2;
          } else i += 1;
        }
        return out.size() - before;
      };
      size_t R = nr;   // runs [0, R) are emitted by this window
      if (!eof) {
        // hold back from the last COMPLETE run (index <= nr - 2) that is non-empty after pairing: what precedes it is then
        // known to be followed by another group
        std::vector<Rec> o, b1, b2; size_t rstar = (size_t)-1;
        for (size_t r = nr >= 2 ? nr - 2 : (size_t)-1; r != (size_t)-1; r--) { o.clear(); if (emit_run(r, o, b1, b2)) { rstar = r; break; } if (r == 0) break; }
        if (rstar == (size_t)-1 || rstar == 0) {
          // nothing can be emitted yet: one run spans the window (or nothing complete and non-empty precedes the last run) -> read more into the same window
          grow = std::max(grow, w.len); continue;
        }
        R = rstar;
        w.carry_from = (size_t)((all[kept[run[rstar]]].p - 4) - d.data());
      } else w.carry_from = w.len;
      (void)tail;
      if (kept.empty() || R == 0) {
        if (eof && groups_sent == 0) w.gstart.push_back(0);   // the producer sends one (empty) group when there is nothing at all
        records_seen += all.size(); header_done = true;
        done = w.gstart.size() < 2;
        return NB_OK;
      }
      const int T = std::max(1, std::min<int>(threads, (int)((R + 63) / 64)));
      std::vector<std::vector<Rec>> outs(T); std::vector<size_t> first_empty(T, (size_t)-1);
      parallel_ranges(T, R, [&](size_t ra, size_t rb, int) {
        size_t t = 0; for (int k = 0; k < T; k++) if (R * (size_t)k / T == ra) t = k;   // the slice parallel_ranges gave this thread
        std::vector<Rec>& out = outs[t]; std::vector<Rec> buf, tmp;
        out.reserve((force_paired ? 1 : 2) * (run[rb] - run[ra]));   // (a dummy mate per unpaired record at most)
        for (size_t r = ra; r < rb; r++) if (!emit_run(r, out, buf, tmp)) { first_empty[t] = r; return; }   // next() returns None on an empty buffer: the stream ends here
      });
      std::vector<Rec>& stream = w.stream; bool cut = false;
      // the slices' records in order, up to the slice where the stream ends (copied by all threads: tens of millions of records per window)
      int t_used = 0; std::vector<size_t> at(T + 1, 0);
      for (int t = 0; t < T; t++) { at[t + 1] = at[t] + outs[t].size(); t_used = t + 1; if (first_empty[t] != (size_t)-1) { cut = true; break; } }
      stream.resize(at[t_used]);
      parallel_ranges(std::min(T, t_used), (size_t)t_used, [&](size_t ta, size_t tb, int) { for (size_t t = ta; t < tb; t++) { if (!outs[t].empty()) memcpy((void*)&stream[at[t]], (const void*)outs[t].data(), outs[t].size() * sizeof(Rec)); std::vector<Rec>().swap(outs[t]); } });
      if (cut) { ended = true; w.carry_from = w.len; }   // the reference's reader stops for good at an empty buffer
      const bool final = eof || ended;
      header_done = true; records_seen += all.size();
      t_emit += clk() - tc; tc = clk();
      std::vector<u64>& gstart = w.gstart; gstart.clear();
      if (stream.empty()) { gstart.assign(1, 0); if (final && groups_sent == 0) gstart.push_back(0); done = gstart.size() < 2; return NB_OK; }
      // groups: runs of equal (UMI + CB[..len-2]) over the stream
      if (have_last) { Rec lr; lr.umi = last_umi.data(); lr.umi_len = (u32)last_umi.size(); lr.cb = last_cb.data(); lr.cb_len = (u32)last_cb.size(); if (key_equal(lr, stream[0])) return NEED_WHOLE; }
      std::vector<char> head(stream.size(), 0);
      parallel_ranges(threads, stream.size(), [&](size_t a, size_t b, int) { for (size_t j = a; j < b; j++) head[j] = (j == 0 || !key_equal(stream[j - 1], stream[j])) ? 1 : 0; });
      for (size_t j = 0; j < stream.size(); j++) if (head[j]) gstart.push_back(j);
      gstart.push_back(stream.size());
      if (final && groups_sent + (gstart.size() - 1) >= 2) { stream.resize(gstart[gstart.size() - 2]); gstart.pop_back(); }   // the last group is never sent when a group was sent before
      groups_sent += gstart.size() - 1;
      if (!stream.empty()) { const Rec& l = stream.back(); last_umi.assign(l.umi, l.umi_len); last_cb.assign(l.cb ? l.cb : "", l.cb_len); have_last = true; }
      t_groups += clk() - tc;
      return NB_OK;
    }
  }
};

// clipped length / start of a record's sequence (strip_nonbio_regions, src/parse/bam.rs:258-268)
inline void clip_of(const Rec& r, size_t& a, size_t& b) { size_t n = r.l_seq(); a = 0; b = n; if (n == 124) { if (r.is_reverse()) b = n - CLIP_LENGTH; else a = CLIP_LENGTH; } }

// ---- the rows stage's formatter.  A 10x run writes two records' worth of metadata per output row (hundreds of millions of
// records), so this is written for throughput: one pass over the aux block, no per-field search, no snprintf, one resize.
// The reference looks a field up by the first two bytes of its NAME (rust-htslib aux(b"QNAME") -> bam_aux_get reads two
// bytes), so several fields share a tag ("MA": MATE_REVERSE, MATE_UNMAPPED, MAPQ, MATE_POS): fields are put into CLASSES
// by those two bytes, and the aux pass records the first occurrence of each class.
struct FieldClasses {
  u8 of_key[65536]; u8 of_field[38]; int n = 0;
  FieldClasses() { memset(of_key, 0, sizeof of_key); for (int i = 0; i < 38; i++) { u32 key = (u8)FIELDS[i][0] | ((u32)(u8)FIELDS[i][1] << 8); if (!of_key[key]) of_key[key] = (u8)++n; of_field[i] = of_key[key]; } }
};
const FieldClasses FCLS;
inline char* put_u32(char* p, u32 v) { char t[10]; int n = 0; do { t[n++] = (char)('0' + v % 10); v /= 10; } while (v); while (n) *p++ = t[--n]; return p; }
inline char* put_i32(char* p, i32 v) { if (v < 0) { *p++ = '-'; return put_u32(p, (u32)(-(i64)v)); } return put_u32(p, (u32)v); }
inline char* put_bool(char* p, bool b) { if (b) { memcpy(p, "true", 4); return p + 4; } memcpy(p, "false", 5); return p + 5; }

// the 36 reported metadata values of one record, tab-joined, straight into the output line (same values as parse_fields);
// skip_align = false leaves out the last one (SKIP_ALIGN and its tab): the any-order rows store that text once per record
// and add the value of the slot it fills
void append_data_values(const Rec& r, std::string& s, bool skip_align = true) {
  const char* zv[40]; u32 zl[40]; u64 seen = 0, isz = 0;
  { const u8* a = r.aux(); const u8* e = r.end();
    while (a + 3 <= e) {   // same rule as Rec::aux_z: the FIRST aux with the tag decides, a string only when NUL-terminated inside the record
      const u32 key = a[0] | ((u32)a[1] << 8); const char ty = (char)a[2]; a += 3; const u8* v = a; u32 zlen = 0; bool zok = false;
      const bool ok = Rec::aux_skip(ty, a, e, zlen, zok);
      const u32 c = FCLS.of_key[key];
      if (c && !((seen >> c) & 1)) { seen |= 1ull << c; if (ty == 'Z' && zok) { isz |= 1ull << c; zv[c] = (const char*)v; zl[c] = zlen; } }
      if (!ok) break;
    } }
  size_t bound = 36 * 13 + r.qname_len();
  if (isz) for (int i = 0; i < 38; i++) { const u32 c = FCLS.of_field[i]; if ((isz >> c) & 1) bound += zl[c]; }
  const size_t old = s.size(); s.resize(old + bound);
  char* p = &s[old];
  const u32 fl = r.flag(); const bool rev = fl & 16, paired = fl & 1, unm = fl & 4, munm = fl & 8, mrev = fl & 32, first = fl & 64;
  for (int i = 0; i < (skip_align ? 38 : 37); i++) {
    if (i == 1 || i == 15) continue;
    if (i) *p++ = '\t';
    if (i == 37 && r.skip_align >= 0) { if (r.skip_align) { memcpy(p, "TRUE", 4); p += 4; } else { memcpy(p, "FALSE", 5); p += 5; } continue; }
    const u32 c = FCLS.of_field[i];
    if ((isz >> c) & 1) { memcpy(p, zv[c], zl[c]); p += zl[c]; continue; }
    switch (i) {
      case 0: memcpy(p, r.qname_ptr(), r.qname_len()); p += r.qname_len(); break;
      case 2: p = put_bool(p, rev); break; case 3: p = put_bool(p, mrev); break; case 4: p = put_bool(p, paired); break; case 5: p = put_bool(p, fl & 2); break;
      case 6: {
        if (paired && !unm && !munm && r.refid() == r.mrefid() && r.pos() != r.mpos()) {   // rust-htslib read_pair_orientation
          i64 p1, p2; bool f1, f2;
          if (first) { p1 = r.pos(); p2 = r.mpos(); f1 = !rev; f2 = !mrev; } else { p1 = r.mpos(); p2 = r.pos(); f1 = !mrev; f2 = !rev; }
          const char* x = f1 ? "F1" : "R1"; const char* y = f2 ? "F2" : "R2";
          if (p1 < p2) { memcpy(p, x, 2); memcpy(p + 2, y, 2); } else { memcpy(p, y, 2); memcpy(p + 2, x, 2); }
        } else memcpy(p, "None", 4);
        p += 4; break; }
      case 7: p = put_bool(p, unm); break; case 8: p = put_bool(p, munm); break; case 9: p = put_bool(p, first); break; case 10: p = put_bool(p, fl & 128); break;
      case 11: *p++ = rev ? '-' : '+'; break;
      case 12: p = put_u32(p, r.mapq()); break; case 13: p = put_i32(p, r.pos()); break; case 14: p = put_i32(p, r.mpos()); break;
      case 16: p = put_u32(p, r.l_seq()); break; case 17: p = put_i32(p, r.tlen()); break;
      case 18: p = put_bool(p, fl & 512); break; case 19: p = put_bool(p, fl & 256); break; case 20: p = put_bool(p, fl & 1024); break; case 21: p = put_bool(p, fl & 2048); break;
      default: break;   // non-string aux (NH, HI, AS, nM, RE ...) -> String::new()
    }
  }
  s.resize((size_t)(p - s.data()));
}
// field 0 of a record as the row logic sees it (QNAME, or a "QN" string aux when one exists — aux lookup by two bytes), as a view
inline void field0(const Rec& r, const char*& ptr, u32& len) {
  const u8* a = r.aux(); const u8* e = r.end();
  while (a + 3 <= e) {
    const char t0 = (char)a[0], t1 = (char)a[1], ty = (char)a[2]; a += 3; const u8* v = a; u32 zlen = 0; bool zok = false;
    const bool ok = Rec::aux_skip(ty, a, e, zlen, zok);
    if (t0 == 'Q' && t1 == 'N') { if (ty == 'Z' && zok) { ptr = (const char*)v; len = zlen; return; } break; }
    if (!ok) break;
  }
  ptr = r.qname_ptr(); len = r.qname_len();
}

std::string data_header(const char* prefix) { std::string s; for (int i = 0; i < 38; i++) { if (i == 1 || i == 15) continue; if (!s.empty()) s += "\t"; s += prefix; s += "_"; s += FIELDS[i]; } return s; }

// one gzip member (concatenated members are one valid .gz stream): lets the writer threads deflate independently
bool gzip_member(const char* text, size_t len, int level, std::string& out) {
  z_stream zs; memset(&zs, 0, sizeof zs);
  if (deflateInit2(&zs, level, Z_DEFLATED, 15 + 16, 8, Z_DEFAULT_STRATEGY) != Z_OK) return false;
  out.resize(deflateBound(&zs, (uLong)len) + 32);
  zs.next_in = (Bytef*)text; zs.avail_in = (uInt)len; zs.next_out = (Bytef*)&out[0]; zs.avail_out = (uInt)out.size();
  int rc = deflate(&zs, Z_FINISH); size_t n = zs.total_out; deflateEnd(&zs);
  if (rc != Z_STREAM_END) return false;
  out.resize(n); return true;
}
bool gzip_member(const std::string& text, int level, std::string& out) { return gzip_member(text.data(), text.size(), level, out); }

// The rows' gzip members (nb_process_bam and nb_process_bam_rows_any_order): a part of the rows with the rows' own
// compressor, or zlib at NB_BAM_GZ_LEVEL=1..9; the header member before the first rows; an empty stream when there is no row.
int rows_gz_level() { int v = 0; if (const char* e = getenv("NB_BAM_GZ_LEVEL")) v = atoi(e); return v >= 1 && v <= 9 ? v : 0; }
bool rows_member(const char* text, size_t n, int level, std::string& out) {
  if (level) return gzip_member(text, n, level, out);
  std::unique_ptr<nbz::FastDeflate> fd(new nbz::FastDeflate()); out.reserve(n / 16 + 4096); fd->gzip_member((const u8*)text, n, out); return true;
}
int write_rows_header(FILE* f, int level) {
  const std::string header = "nimble_features\tnimble_score\t" + data_header("r1") + "\t" + data_header("r2") + "\tr1_filter_forward\tr1_forward_score\tr1_filter_reverse\tr1_reverse_score\tr2_filter_forward\tr2_forward_score\tr2_filter_reverse\tr2_reverse_score\ttriage_reason\taligndirection\n";
  std::string hm; if (!gzip_member(header, level ? level : 2, hm) || fwrite(hm.data(), 1, hm.size(), f) != hm.size()) return fail(NB_ERR_IO, "short write on the TSV");
  return NB_OK;
}
int write_rows_empty(FILE* f, int level) {   // no row at all: an empty gzip stream, like the reference's untouched GzEncoder
  std::string em; if (!gzip_member(std::string(), level ? level : 2, em) || fwrite(em.data(), 1, em.size(), f) != em.size()) return fail(NB_ERR_IO, "short write on the TSV");
  return NB_OK;
}

// Run-wide cell barcodes (nb_process_bam_cells): id = order of first appearance.  The fill stage hashes the CB of every
// group and looks it up (find: read-only, full-string check) on all threads; one serial pass in group order then adds the
// barcodes not found (tens of millions of groups: a std::unordered_map<std::string, ...> lookup per group, or any serial
// pass touching every group's record, would cost seconds).
struct CellDict {
  std::string names; std::vector<u64> off{0}, hash; std::vector<u32> slot;   // names: NUL-terminated, back to back
  CellDict() { clear(); }
  void clear() { names.clear(); off.assign(1, 0); hash.clear(); slot.assign((size_t)1 << 16, NONE32); }
  size_t size() const { return hash.size(); }
  static u64 hash_of(const char* p, u32 n) {
    u64 h = 0x9E3779B97F4A7C15ull ^ n; u32 i = 0;
    for (; i + 8 <= n; i += 8) { u64 w; memcpy(&w, p + i, 8); h = (h ^ w) * 0xFF51AFD7ED558CCDull; h ^= h >> 32; }
    u64 w = 0; memcpy(&w, p + i, n - i); h = (h ^ w) * 0xC4CEB9FE1A85EC53ull; return h ^ (h >> 29);
  }
  u32 find(const char* p, u32 n, u64 h) const {
    const u64 m = slot.size() - 1;
    for (u64 i = h & m;; i = (i + 1) & m) {
      const u32 id = slot[i]; if (id == NONE32) return NONE32;
      if (hash[id] == h && off[id + 1] - off[id] - 1 == n && !memcmp(&names[off[id]], p, n)) return id;
    }
  }
  u32 intern(const char* p, u32 n, u64 h) {
    if (2 * (hash.size() + 1) > slot.size()) {   // grow: the stored hashes place every id again
      slot.assign(slot.size() * 2, NONE32); const u64 m = slot.size() - 1;
      for (u32 id = 0; id < hash.size(); id++) { u64 i = hash[id] & m; while (slot[i] != NONE32) i = (i + 1) & m; slot[i] = id; }
    }
    const u32 found = find(p, n, h); if (found != NONE32) return found;
    const u64 m = slot.size() - 1; u64 i = h & m;
    while (slot[i] != NONE32) i = (i + 1) & m;
    const u32 id = (u32)hash.size(); slot[i] = id; hash.push_back(h); names.append(p, n); names.push_back('\0'); off.push_back(names.size());
    return id;
  }
};

// text -> gzip members of the rows' compressor, written to `path`; the text is cut into pieces of a fixed size (compressed on
// several threads) so that the bytes do not depend on the thread count
int write_gz_pieces(const std::string& path, const std::vector<std::string>& pieces) {
  std::vector<std::string> member(pieces.size());
  const int T = (int)std::max<size_t>(1, std::min<size_t>(pieces.size(), std::max(1u, std::min(16u, std::thread::hardware_concurrency()))));
  std::atomic<size_t> next(0);
  parallel_ranges(T, (size_t)T, [&](size_t, size_t, int) {
    std::unique_ptr<nbz::FastDeflate> fd(new nbz::FastDeflate());
    for (size_t i; (i = next.fetch_add(1)) < pieces.size();) fd->gzip_member((const u8*)pieces[i].data(), pieces[i].size(), member[i]);
  });
  FILE* f = fopen(path.c_str(), "wb"); if (!f) return fail(NB_ERR_IO, "could not open " + path);
  bool ok = true;
  for (const std::string& m : member) ok = ok && fwrite(m.data(), 1, m.size(), f) == m.size();
  ok = fclose(f) == 0 && ok;
  return ok ? NB_OK : fail(NB_ERR_IO, "short write on " + path);
}
inline char* put_u64(char* p, u64 v) { char t[20]; int n = 0; do { t[n++] = (char)('0' + v % 10); v /= 10; } while (v); while (n) *p++ = t[--n]; return p; }

}  // namespace

extern "C" int nb_write_cell_matrix(const char* dir, const nb_library* lib, const nb_cell_counts* cc, const char* const* barcodes, uint64_t n_barcodes) {
  if (!dir || !*dir || !lib || !cc || (!barcodes && n_barcodes)) return fail(NB_ERR_INVALID, "null argument");
  const u64 n = cc->n_rows, ncs = cc->n_callsets;
  if ((n && (!cc->row_cell || !cc->row_callset || !cc->row_umis || !cc->row_reads)) || (ncs && (!cc->callset_off || !cc->callset_items))) return fail(NB_ERR_INVALID, "null array in the cell counts");
  for (u64 b = 0; b < n_barcodes; b++) if (!barcodes[b]) return fail(NB_ERR_INVALID, "null barcode");
  const u32 n_groups = nb_library_n_groups(lib);
  for (u64 c = 0; c < ncs; c++) for (u64 k = cc->callset_off[c]; k < cc->callset_off[c + 1]; k++) if (cc->callset_items[k] >= n_groups) return fail(NB_ERR_INVALID, "callset item is not a group of the library");
  for (u64 i = 0; i < n; i++) {
    if (cc->row_cell[i] >= n_barcodes || cc->row_callset[i] >= ncs) return fail(NB_ERR_INVALID, "row outside the barcodes / callsets");
    if (cc->row_umis[i] < 0 || cc->row_reads[i] < 0) return fail(NB_ERR_INVALID, "negative count");
    if (i && (cc->row_cell[i] < cc->row_cell[i - 1] || (cc->row_cell[i] == cc->row_cell[i - 1] && cc->row_callset[i] <= cc->row_callset[i - 1]))) return fail(NB_ERR_INVALID, "rows are not sorted by (cell, callset)");
  }
  if (mkdir(dir, 0777) != 0 && errno != EEXIST) return fail(NB_ERR_IO, std::string("could not create ") + dir);
  struct stat st; if (stat(dir, &st) != 0 || !S_ISDIR(st.st_mode)) return fail(NB_ERR_IO, std::string(dir) + " is not a directory");
  const std::string d(dir);
  std::vector<std::string> pieces(1);
  for (u64 c = 0; c < ncs; c++) {
    std::string name;
    for (u64 k = cc->callset_off[c]; k < cc->callset_off[c + 1]; k++) { if (k > cc->callset_off[c]) name += ','; name += nb_library_group_name(lib, cc->callset_items[k]); }
    pieces[0] += name; pieces[0] += '\t'; pieces[0] += name; pieces[0] += "\tGene Expression\n";
  }
  int rc = write_gz_pieces(d + "/features.tsv.gz", pieces); if (rc) return rc;
  pieces.assign(1, std::string());
  for (u64 b = 0; b < n_barcodes; b++) { pieces[0] += barcodes[b]; pieces[0] += '\n'; }
  rc = write_gz_pieces(d + "/barcodes.tsv.gz", pieces); if (rc) return rc;
  // Matrix Market: features are the rows, barcodes the columns; lines in (barcode, feature) order as the counts come
  const u64 PIECE = (u64)1 << 20;   // lines per gzip member
  for (int which = 0; which < 2; which++) {
    const i64* val = which ? cc->row_reads : cc->row_umis;
    pieces.assign(1 + (n + PIECE - 1) / PIECE, std::string());
    pieces[0] = "%%MatrixMarket matrix coordinate integer general\n" + std::to_string(ncs) + " " + std::to_string(n_barcodes) + " " + std::to_string(n) + "\n";
    parallel_ranges((int)std::min<u64>(16, pieces.size() - 1), pieces.size() - 1, [&](size_t a, size_t b, int) {
      for (size_t q = a; q < b; q++) {
        const u64 r0 = q * PIECE, r1 = std::min(n, r0 + PIECE);
        std::string& t = pieces[q + 1]; t.resize((r1 - r0) * 64); char* p = &t[0];
        for (u64 i = r0; i < r1; i++) { p = put_u64(p, (u64)cc->row_callset[i] + 1); *p++ = ' '; p = put_u64(p, (u64)cc->row_cell[i] + 1); *p++ = ' '; p = put_u64(p, (u64)val[i]); *p++ = '\n'; }
        t.resize((size_t)(p - t.data()));
      } });
    rc = write_gz_pieces(d + (which ? "/reads.mtx.gz" : "/matrix.mtx.gz"), pieces); if (rc) return rc;
  }
  return NB_OK;
}

// host-only: one gzip member made by the rows stage's compressor (deflate_fast.hpp) — tests inflate it with zlib
extern "C" int nb_gzip_fast(const void* in, uint64_t in_len, void* out, uint64_t out_cap, uint64_t* out_len) {
  if ((!in && in_len) || (!out && out_cap) || !out_len) return fail(NB_ERR_INVALID, "null argument");
  std::unique_ptr<nbz::FastDeflate> fd(new nbz::FastDeflate()); std::string o;
  fd->gzip_member((const u8*)in, in_len, o);
  *out_len = o.size();
  if (o.size() > out_cap) return fail(NB_ERR_OVERFLOW, "output buffer too small");
  memcpy(out, o.data(), o.size());
  return NB_OK;
}

extern "C" int nb_process_bam(const char* input_file, const char* const* reference_json, const char* const* output_paths, uint32_t n_refs, int strand_filter,
                              const char* trim, int num_cores, int force_bam_paired, int device) {
  if (!output_paths) return fail(NB_ERR_INVALID, "need an input BAM and >=1 reference/output pair");
  return nb_process_bam_cells(input_file, reference_json, output_paths, nullptr, n_refs, strand_filter, trim, num_cores, force_bam_paired, device);
}

// process::bam::process behind main.rs's library loop (src/bin/main.rs:95-156); matrix_dirs: per-cell matrices as well,
// output_paths NULL: no TSV rows
extern "C" int nb_process_bam_cells(const char* input_file, const char* const* reference_json, const char* const* output_paths, const char* const* matrix_dirs,
                                    uint32_t n_refs, int strand_filter, const char* trim /* "L:S,L:S" or NULL */, int num_cores, int force_bam_paired, int device) {
  if (!input_file || !reference_json || (!output_paths && !matrix_dirs) || n_refs < 1) return fail(NB_ERR_INVALID, "need an input BAM and >=1 reference/output pair");
  const bool want_rows = output_paths != nullptr, want_cells = matrix_dirs != nullptr;
  int threads = std::max(1, num_cores);
  std::vector<nb_library*> libs(n_refs, nullptr); std::vector<nb_index*> idx(n_refs, nullptr); std::vector<nb_ctx*> ctx(n_refs, nullptr); std::vector<FILE*> outs(n_refs, nullptr);
  std::vector<bool> first_write(n_refs, true);
  int rc = NB_OK;
  auto cleanup = [&]() { for (u32 i = 0; i < n_refs; i++) { if (outs[i]) fclose(outs[i]); nb_ctx_free(ctx[i]); nb_index_free(idx[i]); nb_library_free(libs[i]); } };
  std::vector<std::pair<u64, double>> trims;
  if (trim && *trim) {   // src/bin/main.rs:74-93
    std::string t(trim); size_t p = 0;
    while (p <= t.size()) { size_t e = t.find(',', p); if (e == std::string::npos) e = t.size(); std::string one = t.substr(p, e - p); size_t c = one.find(':'); if (c == std::string::npos) return fail(NB_ERR_INVALID, "Invalid strictness"); trims.push_back({strtoull(one.substr(0, c).c_str(), nullptr, 10), strtod(one.substr(c + 1).c_str(), nullptr)}); p = e + 1; }
    if (trims.size() != n_refs) return fail(NB_ERR_INVALID, "The number of trim options does not match the number of reference libraries");
  }
  for (u32 i = 0; i < n_refs && rc == NB_OK; i++) {
    rc = nb_library_load_json(reference_json[i], strand_filter, &libs[i]);
    if (rc == NB_OK && !trims.empty()) { nb_config c; nb_library_get_config(libs[i], &c); c.trim_target_length = trims[i].first; c.trim_strictness = trims[i].second; rc = nb_library_set_config(libs[i], &c); }
    if (rc == NB_OK) rc = nb_index_build_cached(libs[i], nullptr, device, threads, &idx[i]);   // K5: the CUDA builder (same artefact as the host builder), or $NB_INDEX_CACHE
    if (rc == NB_OK) rc = nb_ctx_create(idx[i], libs[i], device, nullptr, &ctx[i]);
    if (rc == NB_OK) rc = nb_ctx_set_option(ctx[i], "agg_slots", 1u << 23);   // a batch of 2^20 pairs can hold that many one-pair scopes, each with its own (scope, callset) row: stay under half full
    if (rc == NB_OK && want_rows) { outs[i] = fopen(output_paths[i], "wb"); if (!outs[i]) rc = fail(NB_ERR_IO, std::string("could not open output ") + output_paths[i]); }
  }
  auto now = []() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  double t_load = 0, t_group = 0, t_fill = 0, t_gpu = 0, t_rows = 0, t_align = 0, t_final = 0, t_roll = 0, t_cells = 0, t0 = now(); const double t_start = t0;   // NB_BAM_STATS=1 prints the phase times
  // window size of the streaming producer: NB_BAM_WINDOW_MB (inflated bytes per window; tests use small ones), default 256 MB
  size_t window_bytes = (size_t)256 << 20;
  if (const char* e = getenv("NB_BAM_WINDOW_KB")) window_bytes = (size_t)strtoull(e, nullptr, 10) << 10;
  else if (const char* e2 = getenv("NB_BAM_WINDOW_MB")) window_bytes = (size_t)strtoull(e2, nullptr, 10) << 20;
  if (rc != NB_OK) { cleanup(); return rc; }
  const size_t BATCH_PAIRS = 1u << 20;
  const int GZ_LEVEL = rows_gz_level();   // 0: the rows' own compressor (deflate_fast.hpp); NB_BAM_GZ_LEVEL=1..9: zlib at that level (the rows are the same, the members smaller or slower to make)
  // Three stages run concurrently on consecutive batches: (F) the host threads fill batch k+1 into pinned buffers,
  // (D) the device aligns batch k and its counts are finalized, (R) the host threads format + gzip the rows of batch k-1.
  struct Pinned { u8* p = nullptr; size_t cap = 0; int ensure(size_t n) { if (n <= cap) return NB_OK; nb_host_free(p); cap = n + n / 4 + 4096; p = (u8*)nb_host_alloc(cap); if (!p) { cap = 0; return fail(NB_ERR_CUDA, "pinned host allocation failed"); } return NB_OK; } ~Pinned() { nb_host_free(p); } };
  struct BatchIn { const std::vector<Rec>* stream = nullptr; const std::vector<u64>* gstart = nullptr; size_t g0 = 0, g1 = 0, np = 0; u32 maxlen = 1; std::vector<u64> pair0, o1, o2; std::vector<u32> l1, l2; std::vector<u8> f1, f2; std::vector<u32> scope, cell; std::vector<u64> cb_hash; Pinned r1, r2, q1, q2; };
  struct BatchOut { std::vector<nb_read_result> rres; std::vector<nb_pair_result> pres; std::vector<u64> row_begin, callset_off; std::vector<u32> row_callset, callset_items, slot_to_callset; std::vector<i64> row_count; };
  BatchIn bin[3]; BatchOut bout[2];
  // the window being processed (its records and groups): set by the window loop below, read by the three stages
  const std::vector<Rec>* cur_stream = nullptr; const std::vector<u64>* cur_gstart = nullptr;
  std::atomic<u64> ns_fill(0), ns_rows(0);
  CellDict cells;   // (matrix_dirs) cell of a scope = the full CB of its first record; fills run in stream order, so ids are first-appearance order
  // ---- (F) batch arrays: even record = sequence slot, odd = mate slot (src/process/bam.rs:257-292)
  auto fill = [&](BatchIn& B, size_t g0, size_t g1) -> int {
    double tb = now();
    B.stream = cur_stream; B.gstart = cur_gstart; const std::vector<Rec>& stream = *B.stream; const std::vector<u64>& gstart = *B.gstart;
    B.g0 = g0; B.g1 = g1; const size_t ng = g1 - g0;
    B.pair0.assign(ng + 1, 0);
    for (size_t g = 0; g < ng; g++) B.pair0[g + 1] = B.pair0[g] + (gstart[g0 + g + 1] - gstart[g0 + g]) / 2;
    const size_t np = B.np = B.pair0[ng];
    // The bases travel as BAM stores them — 4-bit nibbles (NB_SEQ_BAM4: the device turns =ACMGRSVTWYHKDBN into A/C/G/T with
    // everything else A, exactly DnaString::from_acgt_bytes on the letters) — so a read is a byte copy out of its record, not a
    // per-base expansion, and half the PCIe bytes.  Every read starts on a byte of the batch stream; offsets count BASES
    // (2 x byte + the odd nibble a TSO clip may start on), lengths are explicit, quals sit one byte per base at the same offsets.
    B.o1.assign(np + 1, 0); B.o2.assign(np + 1, 0); B.l1.resize(np); B.l2.resize(np); B.f1.resize(np); B.f2.resize(np); B.scope.resize(np);
    std::vector<u64>& by1 = B.o1; std::vector<u64>& by2 = B.o2;   // first: nibble bytes per read, then their running sum, then base offsets
    parallel_ranges(threads, ng, [&](size_t a, size_t b, int) {
      for (size_t g = a; g < b; g++) { const Rec* v = &stream[gstart[g0 + g]];
        for (size_t j = 0; j < B.pair0[g + 1] - B.pair0[g]; j++) { size_t x, y; const size_t p = B.pair0[g] + j;
          clip_of(v[2 * j], x, y); by1[p + 1] = ((y + 1) >> 1) - (x >> 1); B.l1[p] = (u32)(y - x);
          clip_of(v[2 * j + 1], x, y); by2[p + 1] = ((y + 1) >> 1) - (x >> 1); B.l2[p] = (u32)(y - x); } } });
    B.maxlen = 1;
    for (size_t p = 0; p < np; p++) { B.maxlen = std::max<u32>(B.maxlen, std::max(B.l1[p], B.l2[p])); by1[p + 1] += by1[p]; by2[p + 1] += by2[p]; }
    const u64 tot1 = by1[np], tot2 = by2[np];
    int e = B.r1.ensure(tot1 + 64); if (!e) e = B.q1.ensure(2 * tot1 + 64); if (!e) e = B.r2.ensure(tot2 + 64); if (!e) e = B.q2.ensure(2 * tot2 + 64); if (e) return e;
    parallel_ranges(threads, ng, [&](size_t a, size_t b, int) {
      for (size_t g = a; g < b; g++) { const Rec* v = &stream[gstart[g0 + g]];
        for (size_t j = 0; j < B.pair0[g + 1] - B.pair0[g]; j++) {
          size_t p = B.pair0[g] + j;
          for (int side = 0; side < 2; side++) {
            const Rec& r = v[2 * j + side]; size_t x, y; clip_of(r, x, y);
            const u64 byte0 = side ? by2[p] : by1[p], base0 = 2 * byte0 + (x & 1);
            memcpy((side ? B.r2.p : B.r1.p) + byte0, r.seq4() + (x >> 1), ((y + 1) >> 1) - (x >> 1));
            memcpy((side ? B.q2.p : B.q1.p) + base0, r.qual() + x, y - x);
            u8 fl = (u8)((r.skip_align == 1 ? NB_FLAG_SKIP_ALIGN : 0) | (r.is_reverse() ? NB_FLAG_REVCOMP : 0));
            if (side) B.f2[p] = fl; else B.f1[p] = fl;
          }
          B.scope[p] = (u32)g;
        } } });
    // byte positions -> base offsets (in place, after every copy has used the byte positions): the odd start nibble of read p
    parallel_ranges(threads, ng, [&](size_t a, size_t b, int) {
      for (size_t g = a; g < b; g++) { const Rec* v = &stream[gstart[g0 + g]];
        for (size_t j = 0; j < B.pair0[g + 1] - B.pair0[g]; j++) { size_t x, y; const size_t p = B.pair0[g] + j;
          clip_of(v[2 * j], x, y); by1[p] = 2 * by1[p] + (x & 1); clip_of(v[2 * j + 1], x, y); by2[p] = 2 * by2[p] + (x & 1); } } });
    by1[np] = 2 * tot1; by2[np] = 2 * tot2;
    if (want_cells) {
      B.cell.assign(ng, 0); B.cb_hash.resize(ng);
      std::vector<std::vector<u32>> miss(threads);   // groups whose CB the dictionary did not know yet, per thread in group order
      parallel_ranges(threads, ng, [&](size_t a, size_t b, int t) {
        for (size_t g = a; g < b; g++) if (gstart[g0 + g + 1] > gstart[g0 + g]) {   // (a group without records has no pairs: its cell is never read)
          const Rec& r = stream[gstart[g0 + g]]; const u64 h = B.cb_hash[g] = CellDict::hash_of(r.cb, r.cb_len);
          if ((B.cell[g] = cells.find(r.cb, r.cb_len, h)) == NONE32) miss[t].push_back((u32)g);
        } });
      for (const std::vector<u32>& mt : miss) for (u32 g : mt) { const Rec& r = stream[gstart[g0 + g]]; B.cell[g] = cells.intern(r.cb, r.cb_len, B.cb_hash[g]); }
    }
    ns_fill += (u64)((now() - tb) * 1e9);
    return NB_OK;
  };
  // ---- (D) device: align + finalize; the count rows are copied out (the context reuses that memory on the next finalize)
  auto on_device = [&](const BatchIn& B, u32 li, BatchOut& O) -> int {
    if (!B.np) { O.row_begin.assign(B.g1 - B.g0 + 1, 0); return NB_OK; }
    double tb = now();
    nb_batch b; memset(&b, 0, sizeof b);
    b.n_pairs = B.np; b.location = NB_MEM_HOST; b.max_read_len = B.maxlen; b.r1 = B.r1.p; b.r1_off = B.o1.data(); b.r2 = B.r2.p; b.r2_off = B.o2.data();
    b.q1 = B.q1.p; b.q2 = B.q2.p; b.flags1 = B.f1.data(); b.flags2 = B.f2.data(); b.scope_id = B.scope.data();
    b.encoding = NB_SEQ_BAM4; b.r1_len = B.l1.data(); b.r2_len = B.l2.data();
    if (want_rows) { O.rres.resize(2 * B.np); O.pres.resize(B.np); }
    double ta = now();
    int e = nb_counts_reset(ctx[li]); if (e) return e;
    e = nb_ctx_set_option(ctx[li], "max_batch_pairs", std::max<size_t>(B.np, 1)); if (e) return e;
    double tb1 = now();
    e = nb_align_batch(ctx[li], &b, want_rows ? O.rres.data() : nullptr, want_rows ? O.pres.data() : nullptr); if (e) return e;
    double tb2 = now(); nb_ctx_sync(ctx[li]); double tb3 = now();
    if (getenv("NB_BAM_STATS")) fprintf(stderr, "  batch: np=%zu resize %.1f ms, reset+opt %.1f ms, align call %.1f ms, sync %.1f ms\n", B.np, (ta - tb) * 1e3, (tb1 - ta) * 1e3, (tb2 - tb1) * 1e3, (tb3 - tb2) * 1e3);
    t_align += now() - tb; double tf = now();
    nb_counts cts; e = nb_counts_finalize(ctx[li], &cts); if (e) return e;
    t_final += now() - tf;
    const size_t ng = B.g1 - B.g0;
    if (want_cells) { const double tr = now(); e = nb_cells_roll(ctx[li], B.cell.data(), ng); t_roll += now() - tr; if (e) return e; }
    if (!want_rows) { t_gpu += now() - tb; return NB_OK; }
    O.row_begin.assign(ng + 1, 0);
    for (u64 r = 0; r < cts.n_rows; r++) O.row_begin[cts.row_scope[r] + 1]++;
    for (size_t g = 0; g < ng; g++) O.row_begin[g + 1] += O.row_begin[g];
    O.row_callset.assign(cts.row_callset, cts.row_callset + cts.n_rows); O.row_count.assign(cts.row_count, cts.row_count + cts.n_rows);
    O.callset_off.assign(cts.callset_off, cts.callset_off + cts.n_callsets + 1); O.callset_items.assign(cts.callset_items, cts.callset_items + cts.callset_off[cts.n_callsets]);
    O.slot_to_callset.assign(cts.slot_to_callset, cts.slot_to_callset + cts.n_slots);
    t_gpu += now() - tb;
    return NB_OK;
  };
  // ---- (R) rows: every writer thread formats a contiguous range of groups and deflates it into its own gzip member
  auto rows = [&](const BatchIn& B, u32 li, const BatchOut& O) -> int {
    if (!B.np) return NB_OK;
    double tb = now();
    const std::vector<Rec>& stream = *B.stream; const std::vector<u64>& gstart = *B.gstart;
    const size_t ng = B.g1 - B.g0, np = B.np, g0 = B.g0;
    const std::vector<u64>& pair0 = B.pair0; const std::vector<u64>& row_begin = O.row_begin;
    const int parts = std::max(1, std::min<int>(threads, (int)((np + 4095) / 4096)));
    std::vector<std::string> member(parts); std::vector<int> bad(parts, 0); std::vector<char> wrote(parts, 0);
    std::vector<size_t> cut(parts + 1, ng);   // group ranges balanced by pair count
    cut[0] = 0; for (int t = 1; t < parts; t++) cut[t] = (size_t)(std::lower_bound(pair0.begin(), pair0.end(), np * (u64)t / parts) - pair0.begin());
    for (int t = 1; t <= parts; t++) cut[t] = std::min(std::max(cut[t], cut[t - 1]), ng);
    cut[parts] = ng;
    parallel_ranges(parts, (size_t)parts, [&](size_t ta, size_t tb2, int) {
      for (size_t t = ta; t < tb2; t++) {
        std::string text; text.reserve((size_t)(pair0[cut[t + 1]] - pair0[cut[t]]) * 448 + 4096); char num[32];   // (about 400 bytes per row)
        std::vector<std::string> feats_of(O.callset_off.size()); std::vector<char> feats_made(O.callset_off.size(), 0);    // callset -> "name,name,..." (made on first use)
        const std::string no_feats;
        auto put_num = [&](long long x) { char* e = num; if (x < 0) { *e++ = '-'; x = -x; } if ((unsigned long long)x <= 0xFFFFFFFFull) e = put_u32(e, (u32)x); else e += snprintf(e, 24, "%lld", x); text.append(num, (size_t)(e - num)); };
        std::vector<std::pair<const char*, u32>> scored;   // field 0 of the records that got a count row in this scope (a handful at most)
        auto is_scored = [&](const Rec& x) { const char* q; u32 l; field0(x, q, l); for (const auto& sc : scored) if (same(sc.first, sc.second, q, l)) return true; return false; };
        for (size_t g = cut[t]; g < cut[t + 1]; g++) {
          if (row_begin[g + 1] == row_begin[g]) continue;   // scopes without a callset emit nothing at all (src/process/bam.rs:329-331)
          const Rec* v = &stream[gstart[g0 + g]]; const size_t gp = pair0[g + 1] - pair0[g], pbase = pair0[g];
          scored.clear();
          auto emit = [&](const std::string& feats, long long score, size_t pj) {
            const Rec& sq = v[2 * pj]; const Rec& mt = v[2 * pj + 1]; const nb_pair_result& pr = O.pres[pbase + pj];
            const nb_read_result& ra = O.rres[2 * (pbase + pj)]; const nb_read_result& rb = O.rres[2 * (pbase + pj) + 1];
            text += feats; text += '\t'; put_num(score); text += '\t';
            append_data_values(mt, text); text += '\t'; append_data_values(sq, text); text += '\t';      // "r1" = mate slot, "r2" = sequence slot (108-117)
            text += nb_reason_str(pr.fr2); text += '\t'; put_num(rb.pass ? rb.score : 0); text += "\tNone\t0\t";
            text += nb_reason_str(pr.fr1); text += '\t'; put_num(ra.pass ? ra.score : 0); text += "\tNone\t0\t";
            text += nb_reason_str(pr.triage); text += "\tNone\n";
          };
          for (u64 r = row_begin[g]; r < row_begin[g + 1]; r++) {
            const u32 cs = O.row_callset[r]; std::string& feats = feats_of[cs];
            if (!feats_made[cs]) { feats_made[cs] = 1; for (u64 k = O.callset_off[cs]; k < O.callset_off[cs + 1]; k++) { if (!feats.empty()) feats += ","; feats += nb_library_group_name(libs[li], O.callset_items[k]); } }
            // representative: the last pair of the scope whose read_key resolved to this callset (the reference keeps an arbitrary one)
            size_t rep = gp;
            for (size_t pj = gp; pj-- > 0;) { u32 slot = O.pres[pbase + pj].callset; if (slot != NONE32 && O.slot_to_callset[slot] == cs) { rep = pj; break; } }
            if (rep == gp) continue;
            { const char* q; u32 l; field0(v[2 * rep], q, l); scored.push_back({q, l}); }
            emit(feats, (long long)O.row_count[r], rep);
          }
          for (size_t pj = 0; pj < gp; pj++) { if (!scored.empty() && is_scored(v[2 * pj + 1])) continue; emit(no_feats, 0, pj); }   // zero rows (332-353)
        }
        if (!text.empty()) {
          wrote[t] = 1;
          if (!rows_member(text.data(), text.size(), GZ_LEVEL, member[t])) bad[t] = 1;
        }
      } });
    bool any = false; for (int t = 0; t < parts; t++) { if (bad[t]) return fail(NB_ERR_IO, "gzip of the TSV rows failed"); any = any || wrote[t]; }
    if (any && first_write[li]) { const int e = write_rows_header(outs[li], GZ_LEVEL); if (e) return e; first_write[li] = false; }
    for (int t = 0; t < parts; t++) if (wrote[t] && fwrite(member[t].data(), 1, member[t].size(), outs[li]) != member[t].size()) return fail(NB_ERR_IO, "short write on the TSV");
    ns_rows += (u64)((now() - tb) * 1e9);
    return NB_OK;
  };
  // Errors of the async stages are raised on their own threads (nb_last_error is thread-local): the stage returns the
  // message with its code and the joining thread re-raises it.
  typedef std::pair<int, std::string> Res;
  auto wrap = [](int e) { return Res(e, e ? std::string(nb_last_error()) : std::string()); };
  auto join = [](std::future<Res>& f) { if (!f.valid()) return 0; Res r = f.get(); if (r.first) set_error(r.second); return r.first; };
  std::future<Res> fut_fill, fut_rows, fut_win;
  size_t it_global = 0, bin_next = 0, n_groups_total = 0, n_records_total = 0;
  // one window = a run of whole groups: its batches go through the three stages; the next window is read, inflated and
  // grouped on the host threads meanwhile
  auto process_window = [&](const std::vector<Rec>& stream, const std::vector<u64>& gstart) -> int {
    const size_t n_groups = gstart.size() - 1;
    n_groups_total += n_groups; n_records_total += stream.size();
    std::vector<std::pair<size_t, size_t>> batches;
    for (size_t g0 = 0; g0 < n_groups;) { size_t g1 = g0, pairs = 0; while (g1 < n_groups && pairs < BATCH_PAIRS) { pairs += (gstart[g1 + 1] - gstart[g1]) / 2; g1++; } batches.push_back({g0, g1}); g0 = g1; }
    cur_stream = &stream; cur_gstart = &gstart;
    const size_t nb_ = batches.size();
    int e = 0;
    size_t slot = bin_next;
    if (nb_) e = fill(bin[slot % 3], batches[0].first, batches[0].second);
    for (size_t k = 0; k < nb_ && !e; k++) {
      for (u32 li = 0; li < n_refs && !e; li++, it_global++) {
        if (li == 0 && k + 1 < nb_) fut_fill = std::async(std::launch::async, [&, k, slot]() { return wrap(fill(bin[(slot + k + 1) % 3], batches[k + 1].first, batches[k + 1].second)); });
        e = on_device(bin[(slot + k) % 3], li, bout[it_global % 2]);
        { int er = join(fut_rows); if (er && !e) e = er; }
        if (!e && want_rows) { const BatchIn* bi = &bin[(slot + k) % 3]; const BatchOut* bo = &bout[it_global % 2]; fut_rows = std::async(std::launch::async, [&, bi, bo, li]() { return wrap(rows(*bi, li, *bo)); }); }
        if (li + 1 == n_refs) { int ef = join(fut_fill); if (ef && !e) e = ef; }
      }
    }
    { int ef = join(fut_fill); if (ef && !e) e = ef; }
    { int er = join(fut_rows); if (er && !e) e = er; }   // the rows stage reads this window's records: finish before the window is recycled
    bin_next = (slot + nb_) % 3;
    return e;
  };
  double t_prod = 0; size_t peak_window = 0; bool whole_file = false;
  {
    GroupStreamer gs; Window win[2];
    rc = gs.open(input_file, force_bam_paired != 0, threads, window_bytes);
    bool done = false; int cur = 0;
    if (rc == NB_OK) { double tp = now(); rc = gs.next(win[0], nullptr, done); t_prod += now() - tp; }
    while (rc == NB_OK && !done) {
      // produce the next window while this one is processed (it only reads this window's carry-over bytes)
      bool ndone = false;
      fut_win = std::async(std::launch::async, [&, cur]() { double tp = now(); int e = gs.next(win[cur ^ 1], &win[cur], ndone); t_prod += now() - tp; return wrap(e); });
      int e = process_window(win[cur].stream, win[cur].gstart);
      Res rw = fut_win.get();
      if (rw.first && rw.first != NEED_WHOLE) set_error(rw.second);
      rc = e ? e : rw.first;
      done = ndone; cur ^= 1;
    }
    peak_window = gs.peak_window;
    if (rc == NEED_WHOLE) whole_file = true;
  }
  if (whole_file) {
    // the serial readers' empty-UMI / key-concatenation quirks need the whole file: start over with everything resident
    rc = NB_OK;
    for (u32 li = 0; li < n_refs && rc == NB_OK && want_rows; li++) { if (ftruncate(fileno(outs[li]), 0) != 0 || fseek(outs[li], 0, SEEK_SET) != 0) rc = fail(NB_ERR_IO, "could not rewind the output"); first_write[li] = true; }
    if (want_cells) { cells.clear(); for (u32 li = 0; li < n_refs && rc == NB_OK; li++) rc = nb_cells_reset(ctx[li]); }
    Bgzf z; std::vector<Rec> stream; std::vector<u64> gstart;
    if (rc == NB_OK) rc = z.load(input_file, threads);
    if (rc == NB_OK) rc = collect_groups_serial(z, force_bam_paired != 0, threads, stream, gstart);
    n_groups_total = n_records_total = 0;
    if (rc == NB_OK) rc = process_window(stream, gstart);
  }
  t_load = t_prod; t_group = 0;
  t_fill = ns_fill.load() * 1e-9; t_rows = ns_rows.load() * 1e-9;
  if (rc == NB_OK && want_rows) for (u32 li = 0; li < n_refs && rc == NB_OK; li++) if (first_write[li]) rc = write_rows_empty(outs[li], GZ_LEVEL);
  if (rc == NB_OK && want_cells) {
    const double tc = now();
    std::vector<const char*> bc(cells.size()); for (size_t i = 0; i < bc.size(); i++) bc[i] = cells.names.data() + cells.off[i];
    for (u32 li = 0; li < n_refs && rc == NB_OK; li++) { nb_cell_counts cc; rc = nb_cells_finalize(ctx[li], &cc); if (rc == NB_OK) rc = nb_write_cell_matrix(matrix_dirs[li], libs[li], &cc, bc.data(), bc.size()); }
    t_cells = now() - tc;
  }
  if (getenv("NB_BAM_STATS")) {
    // peak resident set of THIS process image (VmHWM belongs to the mm, so unlike ru_maxrss it does not start at the forking parent's size)
    double hwm_mb = 0; if (FILE* st = fopen("/proc/self/status", "r")) { char line[256]; while (fgets(line, sizeof line, st)) if (!strncmp(line, "VmHWM:", 6)) hwm_mb = strtod(line + 6, nullptr) / 1024.0; fclose(st); }
    fprintf(stderr, "nb_process_bam: %zu records in %zu groups%s; windows (read+inflate+group, overlapped) %.2fs, largest window %.0f MB, batch fill %.2fs, device align+finalize %.2fs (align %.2fs, finalize %.2fs), rows+gzip+write %.2fs (fill and rows overlap the device stage), cell roll %.3fs, cell finalize+matrix write %.3fs, total %.2fs, peak RSS %.0f MB\n", n_records_total, n_groups_total, whole_file ? " (whole-file fallback)" : "", t_load, peak_window / 1048576.0, t_fill, t_gpu, t_align, t_final, t_rows, t_roll, t_cells, now() - t_start, hwm_mb);
  }
  cleanup();
  return rc;
}

// Host-only view of the feeder for parity tests: the groups the producer loop would send, one line per record:
// group index, clipped sequence, hex of the clipped (unreversed) quals, then the 38 metadata fields (QUAL as hex).
extern "C" int nb_bam_dump_groups(const char* input_file, int force_bam_paired, int num_cores, const char* out_path) {
  if (!input_file || !out_path) return fail(NB_ERR_INVALID, "null argument");
  size_t window_bytes = (size_t)256 << 20;
  if (const char* e = getenv("NB_BAM_WINDOW_KB")) window_bytes = (size_t)strtoull(e, nullptr, 10) << 10;
  else if (const char* e2 = getenv("NB_BAM_WINDOW_MB")) window_bytes = (size_t)strtoull(e2, nullptr, 10) << 20;
  FILE* f = fopen(out_path, "wb"); if (!f) return fail(NB_ERR_IO, std::string("could not open ") + out_path);
  auto hex = [](const std::string& s) { static const char* H = "0123456789abcdef"; std::string o; for (unsigned char c : s) { o += H[c >> 4]; o += H[c & 15]; } return o; };
  size_t gi0 = 0;
  auto dump = [&](const std::vector<Rec>& stream, const std::vector<u64>& gstart) {
    for (size_t gi = 0; gi + 1 < gstart.size(); gi++) {
      for (u64 k = gstart[gi]; k < gstart[gi + 1]; k++) {
        ParsedRec r; parse_fields(stream[k], r);
        fprintf(f, "%zu\t%s\t%s", gi0 + gi, r.seq.c_str(), hex(r.qual).c_str());
        for (int i = 0; i < 38; i++) fprintf(f, "\t%s", i == 1 ? hex(r.f[i]).c_str() : r.f[i].c_str());
        fputc('\n', f);
      }
    }
    gi0 += gstart.size() - 1;
  };
  // NB_BAM_DUMP_ROWFMT: instead, one line per record made by the rows stage's own formatter (append_data_values: the 36
  // reported fields, tab-joined) — tests hold it against the fields above, and it times the formatter without a device
  const bool rowfmt = getenv("NB_BAM_DUMP_ROWFMT") != nullptr;
  auto dump_rowfmt = [&](const std::vector<Rec>& stream, bool write) { std::string line; for (const Rec& r : stream) { line.clear(); append_data_values(r, line); line += '\n'; if (write) fwrite(line.data(), 1, line.size(), f); } };
  int rc = NB_OK;
  {
    GroupStreamer gs; Window win[2]; bool done = false; int cur = 0;
    rc = getenv("NB_BAM_SERIAL_GROUPING") ? NEED_WHOLE : gs.open(input_file, force_bam_paired != 0, std::max(1, num_cores), window_bytes);
    if (rc == NB_OK) rc = gs.next(win[0], nullptr, done);
    const bool none = out_path[0] && !strcmp(out_path, "/dev/null") && getenv("NB_BAM_DUMP_NONE");   // producer only (timing the reader)
    double t_fmt = 0; size_t n_fmt = 0;
    while (rc == NB_OK && !done) {
      if (rowfmt) { double tf = GroupStreamer::clk(); dump_rowfmt(win[cur].stream, !none); n_fmt += win[cur].stream.size(); t_fmt += GroupStreamer::clk() - tf; }
      else if (!none) dump(win[cur].stream, win[cur].gstart);
      rc = gs.next(win[cur ^ 1], &win[cur], done); cur ^= 1;
    }
    if (rowfmt && getenv("NB_BAM_STATS")) fprintf(stderr, "row formatter: %zu records in %.2f s = %.0f ns per record (one thread)\n", n_fmt, t_fmt, n_fmt ? t_fmt / n_fmt * 1e9 : 0.0);
    if (getenv("NB_BAM_STATS")) fprintf(stderr, "bam producer: inflate %.2fs, record scan %.2fs, key scan %.2fs, runs %.2fs, emit %.2fs, groups %.2fs\n", gs.t_inflate, gs.t_scan, gs.t_keys, gs.t_runs, gs.t_emit, gs.t_groups);
  }
  if (rc == NEED_WHOLE) {
    if (ftruncate(fileno(f), 0) != 0 || fseek(f, 0, SEEK_SET) != 0) { fclose(f); return fail(NB_ERR_IO, "could not rewind the output"); }
    gi0 = 0;
    Bgzf z; rc = z.load(input_file, std::max(1, num_cores));
    std::vector<Rec> stream; std::vector<u64> gstart;
    if (rc == NB_OK) rc = collect_groups_serial(z, force_bam_paired != 0, std::max(1, num_cores), stream, gstart);
    if (rc == NB_OK) { if (rowfmt) dump_rowfmt(stream, true); else dump(stream, gstart); }
  }
  if (rc) { fclose(f); return rc; }
  fclose(f);
  return NB_OK;
}

// ------------------------------------------------------------------ BAM mode in any record order (bam_group.hpp)
namespace {

struct AnyOrderLoad {   // what the producer saw (NB_BAM_STATS)
  u64 n_records = 0, n_kept = 0, meta_text = 0; u32 max_len = 1; size_t peak_window = 0; double t_wait = 0, t_meta = 0;   // meta_text: M(r) bytes staged
};

// Budget mode: a pass stages the records of UMI buckets [lo, hi) (nbg::umi_bucket); hi starts at N_BUCKETS and only falls.
struct Passes {
  u64 budget = 0; int pass = 0; u32 lo = 0, hi = nbg::N_BUCKETS; u64 evictions = 0; bool rows = false;
  std::vector<u64> b_rec, b_nib, b_name, b_meta;   // what this pass has staged (or is about to) of every bucket
  void begin(u32 lo_) { lo = lo_; hi = nbg::N_BUCKETS; b_rec.assign(nbg::N_BUCKETS, 0); b_nib.assign(nbg::N_BUCKETS, 0); b_name.assign(nbg::N_BUCKETS, 0); b_meta.assign(nbg::N_BUCKETS, 0); }
};

// Before a window is staged in budget mode (the per-bucket counts already hold it): when the store plus the window plus the
// grouping arrays would not fit, hi falls to the largest value whose buckets fit the fill target (3/4 of the budget, grouping
// arrays included) and the device keeps only the records below it.  The caller drops the window's records at or above hi.
int plan_window(nbg::Device* dev, Passes& P, u64 ncb, bool& lowered) {
  lowered = false;
  const u32 lo = P.lo, hi = P.hi;
  std::vector<u64> R(hi - lo + 1, 0), NB(hi - lo + 1, 0), NM(hi - lo + 1, 0), NT(hi - lo + 1, 0);   // sums over buckets [lo, lo + k)
  for (u32 k = 0; k < hi - lo; k++) { R[k + 1] = R[k] + P.b_rec[lo + k]; NB[k + 1] = NB[k] + P.b_nib[lo + k]; NM[k + 1] = NM[k] + P.b_name[lo + k]; NT[k + 1] = NT[k] + P.b_meta[lo + k]; }
  auto fits = [&](u32 k) { return nbg::fits(dev, R[k], NB[k], NM[k], NT[k], nbg::group_reserve(dev, R[k], ncb)); };
  if (fits(hi - lo)) return NB_OK;
  const u64 per_rec = P.rows ? 43 + 16 : 43;   // store bytes per record (rows: metadata offset, length and field-0 length)
  auto under_target = [&](u32 k) { return 3 * NB[k] + NM[k] + NT[k] + per_rec * R[k] + nbg::group_reserve(dev, R[k], ncb) <= P.budget / 4 * 3 && fits(k); };
  u32 a = 0, b = hi - lo;   // the largest k in (0, hi - lo) under the target: ok(a) (or a = 0), !ok(b)
  while (b - a > 1) { const u32 m = a + (b - a) / 2; if (under_target(m)) a = m; else b = m; }
  bool compacted = false;
  if (a == 0) {
    if (!fits(1)) {
      // the store may hold arrays sized for records of other buckets: keep bucket lo alone, shrink the arrays, look again
      if (nbg::store_records(dev)) { const int rc = nbg::compact(dev, lo + 1); if (rc) return rc; P.evictions++; compacted = true; }
      { const int rc = nbg::trim(dev); if (rc) return rc; }
      if (!fits(1)) {
        const u64 need = nbg::need_bytes(dev, R[1], NB[1], NM[1], NT[1], nbg::group_reserve(dev, R[1], ncb));
        return fail(NB_ERR_CUDA, "the device budget of " + std::to_string(P.budget) + " bytes is too small: UMI bucket " + std::to_string(lo) + " needs " + std::to_string(need) +
                                 " bytes (" + std::to_string(R[1]) + " records with their grouping arrays)");
      }
    }
    a = 1;
  }
  const u32 nh = lo + a;
  if (!compacted && nbg::store_records(dev)) { const int rc = nbg::compact(dev, nh); if (rc) return rc; P.evictions++; }   // an eviction: records already on the device leave
  for (u32 x = nh; x < hi; x++) P.b_rec[x] = P.b_nib[x] = P.b_name[x] = P.b_meta[x] = 0;
  P.hi = nh; lowered = true;
  return NB_OK;
}

// Streams the file window by window: the kept records of every window (SortedBamReader::fill_buffer's filters, in its
// order) are staged into pinned memory on all threads and uploaded into the device store while the next window inflates.
// cells: every kept record's full CB, ids in order of first appearance.  With P (budget mode) only the records of buckets
// [P->lo, P->hi) are staged, and passes after the first only look the CBs up.  rows: every staged record also gets its
// metadata text M(r) (append_data_values without SKIP_ALIGN) and the length of its field 0, formatted on the host threads.
int any_order_load(const char* input_file, int threads, size_t window_bytes, nbg::Device* dev, CellDict& cells, AnyOrderLoad& st, bool rows, Passes* P = nullptr) {
  auto now = []() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  Bgzf z; int rc = z.open(input_file); if (rc) return rc;
  RawBuf data; size_t len = 0; bool eof = false, header_done = false;
  std::vector<Rec> all;
  const bool lookup_only = P && P->pass > 0;
  for (;;) {
    if (!eof) { size_t n_out = 0; rc = z.next(data, len, window_bytes, threads, n_out, eof); if (rc) return rc; z.compact(); len += n_out; }
    st.peak_window = std::max(st.peak_window, len);
    if (!header_done) {
      bool ok = len >= 12; size_t p = 0;
      if (ok && memcmp(data.data(), "BAM\1", 4)) return fail(NB_ERR_PARSE, "not a BAM file");
      if (ok) { u32 l_text; memcpy(&l_text, &data[4], 4); p = 8 + (size_t)l_text; ok = p + 4 <= len; }
      if (ok) { u32 n_ref; memcpy(&n_ref, &data[p], 4); p += 4; for (u32 i = 0; i < n_ref && ok; i++) { if (p + 4 > len) { ok = false; break; } u32 l; memcpy(&l, &data[p], 4); p += 4 + (size_t)l + 4; } ok = ok && p <= len; }
      if (!ok) { if (eof) return fail(NB_ERR_PARSE, len < 12 ? "not a BAM file" : "truncated BAM header"); continue; }
      memmove(data.data(), data.data() + p, len - p); len -= p; header_done = true;
    }
    size_t tail = 0;
    rc = walk_records(data, len, 0, eof, threads, all, tail); if (rc) return rc;
    if (all.empty()) { if (eof) break; continue; }   // one record larger than the window: read on
    const size_t n = all.size();
    const int T = n > 65536 ? threads : 1;
    parallel_ranges(T, n, [&](size_t a, size_t b, int) { for (size_t i = a; i < b; i++) all[i].scan_keys(); });
    // keep / skip / fail per record; the first failing record in file order decides the error
    std::vector<u8> keep(n, 0); std::vector<u64> umi(n); std::vector<u32> cb(n, NONE32); std::vector<u64> cb_hash(n);
    std::vector<size_t> bad_at(T, (size_t)-1); std::vector<int> bad_kind(T, 0); std::vector<u64> cnt(T + 1, 0), nib(T + 1, 0), nam(T + 1, 0); std::vector<u32> mx(T, 1);
    std::vector<std::vector<u32>> miss(T);
    std::vector<u32> bucket(P ? n : 0);
    parallel_ranges(T, n, [&](size_t a, size_t b, int t) {
      u64 c = 0, nb_ = 0, nm = 0; u32 m = 1;
      for (size_t i = a; i < b; i++) {
        const Rec& r = all[i];
        if (!r.cb) continue;
        if (!r.umi) { bad_at[t] = i; bad_kind[t] = 1; break; }
        if (r.umi_len == 10 && !memcmp(r.umi, "AAAAAAAAAA", 10)) continue;
        if (r.umi_len == 0) { bad_at[t] = i; bad_kind[t] = 2; break; }
        if (!nbg::pack_umi(r.umi, r.umi_len, umi[i])) { bad_at[t] = i; bad_kind[t] = 3; break; }
        size_t x, y; clip_of(r, x, y); m = std::max<u32>(m, (u32)(y - x));
        const u64 h = cb_hash[i] = CellDict::hash_of(r.cb, r.cb_len);
        if ((cb[i] = cells.find(r.cb, r.cb_len, h)) == NONE32) { if (lookup_only) { bad_at[t] = i; bad_kind[t] = 4; break; } miss[t].push_back((u32)i); }
        if (P) { const u32 bk = bucket[i] = nbg::umi_bucket(umi[i]); if (bk < P->lo || bk >= P->hi) continue; }
        keep[i] = 1; c++; nb_ += (r.l_seq() + 1) / 2; nm += r.qname_len();
      }
      cnt[t + 1] = c; nib[t + 1] = nb_; nam[t + 1] = nm; mx[t] = m;
    });
    { size_t first = (size_t)-1; int kind = 0; for (int t = 0; t < T; t++) if (bad_at[t] < first) { first = bad_at[t]; kind = bad_kind[t]; }
      if (kind == 1) return fail(NB_ERR_PARSE, "Error -- Could not read UMI.");
      if (kind == 2) return fail(NB_ERR_UNSUPPORTED, "a kept record has an empty UMI string (where the reference groups it depends on the file order): record " + std::to_string(st.n_records + first) + " of " + input_file);
      if (kind == 3) return fail(NB_ERR_UNSUPPORTED, "UMI \"" + std::string(all[first].umi, all[first].umi_len) + "\" of record " + std::to_string(st.n_records + first) + " cannot be packed into the exact device key (at most " + std::to_string((int)nbg::MAX_UMI_CHARS) + " characters of ACGTN)");
      if (kind == 4) return fail(NB_ERR_IO, std::string("the input changed between passes: record ") + std::to_string(st.n_records + first) + " of " + input_file + " has a cell barcode the first pass did not see"); }
    for (int t = 0; t < T; t++) for (u32 i : miss[t]) cb[i] = cells.intern(all[i].cb, all[i].cb_len, cb_hash[i]);   // file order: ids follow first appearance
    // rows: M(r) of the kept records, back to back per thread slice (the slices of every parallel_ranges(T, n) below)
    std::vector<std::string> mt(rows ? T : 0); std::vector<u32> mlen(rows ? n : 0), f0l(rows ? n : 0); std::vector<u64> met(T + 1, 0);
    if (rows) {
      const double tf = now();
      parallel_ranges(T, n, [&](size_t a, size_t b, int t) {
        std::string& o = mt[t]; u64 m = 0;
        for (size_t i = a; i < b; i++) if (keep[i]) {
          const size_t at = o.size(); append_data_values(all[i], o, false); mlen[i] = (u32)(o.size() - at); m += mlen[i];
          const char* q; u32 l; field0(all[i], q, l); f0l[i] = l;
        }
        met[t + 1] = m;
      });
      st.t_meta += now() - tf;
    }
    if (P) {
      for (size_t i = 0; i < n; i++) if (keep[i]) { const u32 bk = bucket[i]; P->b_rec[bk]++; P->b_nib[bk] += (all[i].l_seq() + 1) / 2; P->b_name[bk] += all[i].qname_len(); if (rows) P->b_meta[bk] += mlen[i]; }
      bool lowered = false;
      rc = plan_window(dev, *P, cells.size(), lowered); if (rc) return rc;
      if (lowered) parallel_ranges(T, n, [&](size_t a, size_t b, int t) {   // drop this window's records at or above the new hi
        u64 c = 0, nb_ = 0, nm = 0, mm = 0;
        for (size_t i = a; i < b; i++) {
          if (keep[i] && bucket[i] >= P->hi) keep[i] = 0;
          if (keep[i]) { c++; nb_ += (all[i].l_seq() + 1) / 2; nm += all[i].qname_len(); if (rows) mm += mlen[i]; }
        }
        cnt[t + 1] = c; nib[t + 1] = nb_; nam[t + 1] = nm; met[t + 1] = mm;
      });
    }
    for (int t = 0; t < T; t++) { cnt[t + 1] += cnt[t]; nib[t + 1] += nib[t]; nam[t + 1] += nam[t]; met[t + 1] += met[t]; st.max_len = std::max(st.max_len, mx[t]); }
    const double tw = now();
    nbg::Stage* sg = nullptr;
    rc = nbg::stage(dev, cnt[T], nib[T], nam[T], met[T], sg); if (rc) return rc;
    st.meta_text += met[T];
    st.t_wait += now() - tw;
    const u64 ord0 = st.n_records;
    parallel_ranges(T, n, [&](size_t a, size_t b, int t) {
      u64 k = cnt[t], bo = nib[t], no = nam[t], mo = met[t]; size_t src = 0;   // src: this slice's read position in mt[t]
      for (size_t i = a; i < b; i++) {
        if (keep[i]) {
          const Rec& r = all[i]; const u32 l = r.l_seq(), nbytes = (l + 1) / 2, ql = r.qname_len();
          memcpy(sg->nib + bo, r.seq4(), nbytes);
          memcpy(sg->qual + 2 * bo, r.qual(), l);   // one qual byte per base, at the base's offset
          memcpy(sg->name + no, r.qname_ptr(), ql);
          sg->umi[k] = umi[i]; sg->cb[k] = cb[i]; sg->nib_off[k] = sg->nib0 + bo; sg->lseq[k] = l; sg->flag[k] = (u16)r.flag();
          sg->name_off[k] = sg->name0 + no; sg->name_len[k] = (u8)ql; sg->ordinal[k] = ord0 + i;
          if (rows) { memcpy(sg->meta + mo, mt[t].data() + src, mlen[i]); sg->meta_off[k] = sg->meta0 + mo; sg->meta_len[k] = mlen[i]; sg->f0_len[k] = f0l[i]; mo += mlen[i]; }
          k++; bo += nbytes; no += ql;
        }
        if (rows) src += mlen[i];   // (a record dropped by a lowered hi was formatted too)
      } });
    rc = nbg::upload(dev, P ? nbg::group_reserve(dev, nbg::store_records(dev) + cnt[T], cells.size()) : 0); if (rc) return rc;
    st.n_records += n; st.n_kept += cnt[T];
    memmove(data.data(), data.data() + tail, len - tail); len -= tail;
    if (eof) break;
  }
  return NB_OK;
}

// At the end of the file: the byte-order rank of every CB and an id for every CB[..len-2], then the device grouping.
int any_order_group(nbg::Device* dev, const CellDict& cells, nbg::Grouped& g) {
  const size_t nc = cells.size();
  auto name = [&](u32 id) { return std::make_pair(cells.names.data() + cells.off[id], (u32)(cells.off[id + 1] - cells.off[id] - 1)); };
  std::vector<u32> order(nc), rank(nc), prefix(nc);
  for (u32 i = 0; i < nc; i++) order[i] = i;
  std::sort(order.begin(), order.end(), [&](u32 a, u32 b) { auto x = name(a), y = name(b); return cmp_bytes(x.first, x.second, y.first, y.second) < 0; });
  for (u32 i = 0; i < nc; i++) rank[order[i]] = i;
  std::unordered_map<std::string, u32> pre;
  for (u32 i = 0; i < nc; i++) { auto x = name(i); prefix[i] = pre.emplace(std::string(x.first, x.second >= 2 ? x.second - 2 : 0), (u32)pre.size()).first->second; }
  return nbg::group(dev, rank, prefix, g);
}

// What a run in any record order did over all its passes (NB_BAM_STATS).
struct AnyOrderRun {
  AnyOrderLoad ld;                       // the first pass's producer (every pass reads the same records)
  int passes = 0; u64 evictions = 0, n_kept = 0, n_scopes = 0, n_pairs = 0, meta_text = 0;   // meta_text: the M(r) text of the records staged in all passes (dropped ones included)
  std::vector<double> t_windows; double t_group = 0;
};

// The passes over the file: one without a budget; with one, each pass takes the UMI buckets from where the previous one
// stopped up to the hi its windows left.  After each pass's grouping: on_pass(pass, grouped, max_read_len) aligns it.
template <class F>
int any_order_passes(const char* input_file, int threads, size_t window_bytes, nbg::Device* dev, u64 budget, bool rows, CellDict& cells, AnyOrderRun& run, F on_pass) {
  auto now = []() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  Passes P; P.budget = budget; P.rows = rows;
  nbg::set_budget(dev, budget); nbg::set_rows(dev, rows);
  for (u32 lo = 0;;) {
    int rc = NB_OK;
    if (budget) { P.begin(lo); if (P.pass) rc = nbg::begin_pass(dev); }
    const double t0 = now();
    AnyOrderLoad ld;
    if (rc == NB_OK) rc = any_order_load(input_file, threads, window_bytes, dev, cells, ld, rows, budget ? &P : nullptr);
    if (rc == NB_OK) { const double tw = now(); rc = nbg::sync(dev); ld.t_wait += now() - tw; }
    const double t1 = now(); run.t_windows.push_back(t1 - t0);
    nbg::Grouped g;
    if (rc == NB_OK) rc = any_order_group(dev, cells, g);
    run.t_group += now() - t1;
    if (rc) return rc;
    if (P.pass == 0) run.ld = ld;
    else if (ld.n_records != run.ld.n_records) return fail(NB_ERR_IO, std::string("the input changed between passes: ") + input_file);
    else { run.ld.t_wait += ld.t_wait; run.ld.t_meta += ld.t_meta; run.ld.peak_window = std::max(run.ld.peak_window, ld.peak_window); }
    run.passes++; run.meta_text += ld.meta_text; run.n_kept += g.n_records; run.n_scopes += g.n_scopes; run.n_pairs += g.n_pairs;
    rc = on_pass(P.pass, (const nbg::Grouped&)g, run.ld.max_len); if (rc) return rc;
    if (!budget || P.hi == nbg::N_BUCKETS) break;
    lo = P.hi; P.pass++;
  }
  run.evictions = P.evictions;
  return NB_OK;
}

size_t any_order_window_bytes() {
  size_t window_bytes = (size_t)256 << 20;
  if (const char* e = getenv("NB_BAM_WINDOW_KB")) window_bytes = std::max<size_t>((size_t)strtoull(e, nullptr, 10) << 10, 1 << 16);
  else if (const char* e2 = getenv("NB_BAM_WINDOW_MB")) window_bytes = std::max<size_t>((size_t)strtoull(e2, nullptr, 10) << 20, 1 << 16);
  return window_bytes;
}

// The device store and one library context per reference of an any-order run, all on the store's stream (the batches'
// scope ids are written on it).
struct AnyOrderSetup {
  nbg::Device* dev = nullptr; u32 n = 0;
  std::vector<nb_library*> libs; std::vector<nb_index*> idx; std::vector<nb_ctx*> ctx;
  ~AnyOrderSetup() { for (u32 i = 0; i < n; i++) { nb_ctx_free(ctx[i]); nb_index_free(idx[i]); nb_library_free(libs[i]); } nbg::destroy(dev); }
  int open(const char* const* reference_json, uint32_t n_refs, int strand_filter, const char* trim, int threads, int device) {
    std::vector<std::pair<u64, double>> trims;
    if (trim && *trim) {   // src/bin/main.rs:74-93
      std::string t(trim); size_t p = 0;
      while (p <= t.size()) { size_t e = t.find(',', p); if (e == std::string::npos) e = t.size(); std::string one = t.substr(p, e - p); size_t c = one.find(':'); if (c == std::string::npos) return fail(NB_ERR_INVALID, "Invalid strictness"); trims.push_back({strtoull(one.substr(0, c).c_str(), nullptr, 10), strtod(one.substr(c + 1).c_str(), nullptr)}); p = e + 1; }
      if (trims.size() != n_refs) return fail(NB_ERR_INVALID, "The number of trim options does not match the number of reference libraries");
    }
    n = n_refs; libs.assign(n, nullptr); idx.assign(n, nullptr); ctx.assign(n, nullptr);
    int rc = nbg::create(device, &dev);
    for (u32 i = 0; i < n && rc == NB_OK; i++) {
      rc = nb_library_load_json(reference_json[i], strand_filter, &libs[i]);
      if (rc == NB_OK && !trims.empty()) { nb_config c; nb_library_get_config(libs[i], &c); c.trim_target_length = trims[i].first; c.trim_strictness = trims[i].second; rc = nb_library_set_config(libs[i], &c); }
      if (rc == NB_OK) rc = nb_index_build_cached(libs[i], nullptr, device, threads, &idx[i]);
      if (rc == NB_OK) rc = nb_ctx_create(idx[i], libs[i], device, nbg::stream_of(dev), &ctx[i]);
      if (rc == NB_OK) rc = nb_ctx_set_option(ctx[i], "agg_slots", 1u << 23);
    }
    return rc;
  }
};

// The NB_BAM_STATS line of an any-order run; rows: the rows mode's fields, which go before the budget's
void any_order_stats(const AnyOrderRun& run, nbg::Device* dev, u64 budget, u64 n_batches, size_t n_barcodes, double t_setup, double t_align, double t_roll, double t_out, double t_total, const std::string& rows) {
  double hwm_mb = 0; if (FILE* stf = fopen("/proc/self/status", "r")) { char line[256]; while (fgets(line, sizeof line, stf)) if (!strncmp(line, "VmHWM:", 6)) hwm_mb = strtod(line + 6, nullptr) / 1024.0; fclose(stf); }
  const AnyOrderLoad& ld = run.ld;
  double t_win = 0; std::string per_pass;
  for (double t : run.t_windows) { t_win += t; char b[32]; snprintf(b, sizeof b, "%s%.2fs", per_pass.empty() ? "" : "/", t); per_pass += b; }
  std::string extra = rows;
  if (budget) { char b[256]; snprintf(b, sizeof b, ", budget %llu bytes, passes %d, evictions %llu, peak device bytes %llu, windows per pass ", (unsigned long long)budget, run.passes, (unsigned long long)run.evictions, (unsigned long long)(dev ? nbg::peak_bytes(dev) : 0)); extra += b + per_pass; }
  fprintf(stderr, "nb_process_bam_any_order: %llu records, %llu kept, %llu scopes, %llu pairs, %llu batches, %zu barcodes; setup %.2fs, windows (read+inflate+stage+upload) %.2fs, upload wait %.3fs, largest window %.0f MB, key+sort+scope build %.3fs, device align+finalize %.3fs, cell roll %.3fs, cell finalize+matrix write %.3fs, total %.2fs, store %llu bytes, grouping %llu bytes, peak RSS %.0f MB%s\n",
          (unsigned long long)ld.n_records, (unsigned long long)run.n_kept, (unsigned long long)run.n_scopes, (unsigned long long)run.n_pairs, (unsigned long long)n_batches, n_barcodes,
          t_setup, t_win, ld.t_wait, ld.peak_window / 1048576.0, run.t_group, t_align, t_roll, t_out, t_total,
          (unsigned long long)(dev ? nbg::store_bytes(dev) : 0), (unsigned long long)(dev ? nbg::group_bytes(dev) : 0), hwm_mb, extra.c_str());
}

int process_bam_cells_any_order(const char* input_file, const char* const* reference_json, const char* const* matrix_dirs, uint32_t n_refs,
                                int strand_filter, const char* trim, int num_cores, int device, u64 budget) {
  if (!input_file || !reference_json || !matrix_dirs || n_refs < 1) return fail(NB_ERR_INVALID, "need an input BAM and >=1 reference library / matrix directory pair");
  auto now = []() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  const double t_start = now();
  const int threads = std::max(1, num_cores);
  const size_t window_bytes = any_order_window_bytes();
  AnyOrderSetup S;
  int rc = S.open(reference_json, n_refs, strand_filter, trim, threads, device);
  if (rc != NB_OK) return rc;
  nbg::Device* dev = S.dev; std::vector<nb_library*>& libs = S.libs; std::vector<nb_ctx*>& ctx = S.ctx;
  const double t_setup = now();
  CellDict cells; AnyOrderRun run;
  // barcodes: the cells of the scopes that have pairs, in order of first appearance.  Without a budget the one pass knows
  // them before it rolls; with one, the passes roll dictionary ids and the rows are renumbered after the last pass (an
  // order-preserving map, so the (cell, rank) order of the rows holds).
  std::vector<u32> remap; std::vector<u8> used; std::vector<const char*> bc;
  const u64 BATCH_PAIRS = 1u << 20;   // batches: whole scopes, at most 2^20 pairs (a larger scope is a batch of its own)
  double t_align = 0, t_roll = 0; u64 n_batches = 0;
  rc = any_order_passes(input_file, threads, window_bytes, dev, budget, false, cells, run, [&](int, const nbg::Grouped& g, u32 max_len) -> int {
    std::vector<u32> cell_of_scope(g.n_scopes, 0);   // scopes without pairs get cell 0 (no rows)
    if (!budget) {
      remap.assign(cells.size(), NONE32);
      for (u64 s = 0; s < g.n_scopes; s++) if (g.scope_pair0[s + 1] > g.scope_pair0[s]) remap[g.scope_cb[s]] = 0;
      for (u32 id = 0; id < cells.size(); id++) if (remap[id] != NONE32) { remap[id] = (u32)bc.size(); bc.push_back(cells.names.data() + cells.off[id]); }
      for (u64 s = 0; s < g.n_scopes; s++) if (g.scope_pair0[s + 1] > g.scope_pair0[s]) cell_of_scope[s] = remap[g.scope_cb[s]];
    } else {
      used.resize(cells.size(), 0);
      for (u64 s = 0; s < g.n_scopes; s++) if (g.scope_pair0[s + 1] > g.scope_pair0[s]) { cell_of_scope[s] = g.scope_cb[s]; used[g.scope_cb[s]] = 1; }
    }
    int e = NB_OK;
    for (u64 s0 = 0; e == NB_OK && s0 < g.n_scopes;) {
      u64 s1 = s0 + 1;
      while (s1 < g.n_scopes && g.scope_pair0[s1 + 1] - g.scope_pair0[s0] <= BATCH_PAIRS) s1++;
      const u64 p0 = g.scope_pair0[s0], p1 = g.scope_pair0[s1];
      if (p1 > p0) {
        n_batches++;
        nb_batch b; e = nbg::batch(dev, p0, p1, s0, max_len, b);
        for (u32 li = 0; li < n_refs && e == NB_OK; li++) {
          const double tb = now();
          e = nb_counts_reset(ctx[li]);
          if (e == NB_OK) e = nb_ctx_set_option(ctx[li], "max_batch_pairs", p1 - p0);   // scoped device batches must fit one chunk
          if (e == NB_OK) e = nb_align_batch(ctx[li], &b, nullptr, nullptr);
          nb_counts cts;
          if (e == NB_OK) e = nb_counts_finalize(ctx[li], &cts);
          const double tr = now(); t_align += tr - tb;
          if (e == NB_OK) e = nb_cells_roll(ctx[li], cell_of_scope.data() + s0, s1 - s0);
          t_roll += now() - tr;
        }
      }
      s0 = s1;
    }
    return e;
  });
  const double t_aligned = now();
  if (rc == NB_OK && budget) {
    remap.assign(cells.size(), NONE32);
    for (u32 id = 0; id < used.size(); id++) if (used[id]) { remap[id] = (u32)bc.size(); bc.push_back(cells.names.data() + cells.off[id]); }
  }
  std::vector<u32> row_cell;
  for (u32 li = 0; li < n_refs && rc == NB_OK; li++) {
    nb_cell_counts cc; rc = nb_cells_finalize(ctx[li], &cc);
    if (rc == NB_OK && budget) { row_cell.resize(cc.n_rows); for (u64 k = 0; k < cc.n_rows; k++) row_cell[k] = remap[cc.row_cell[k]]; cc.row_cell = row_cell.data(); }
    if (rc == NB_OK) rc = nb_write_cell_matrix(matrix_dirs[li], libs[li], &cc, bc.data(), bc.size());
  }
  const double t_end = now();
  if (getenv("NB_BAM_STATS")) any_order_stats(run, dev, budget, n_batches, bc.size(), t_setup - t_start, t_align, t_roll, t_end - t_aligned, t_end - t_start, std::string());
  return rc;
}

// The TSV.gz rows of the grouped driver on G (nb_process_bam_rows_any_order): every batch of every library is aligned
// into device result buffers and its rows are assembled on the device (nbg::rows_build); the host only deflates each
// chunk, cut at row boundaries into parts compressed on its threads, and writes the members in order.  The deflate of a
// chunk runs while the device builds the next one.
int process_bam_rows_any_order(const char* input_file, const char* const* reference_json, const char* const* output_paths, uint32_t n_refs,
                               int strand_filter, const char* trim, int num_cores, int device, u64 budget) {
  if (!input_file || !reference_json || !output_paths || n_refs < 1) return fail(NB_ERR_INVALID, "need an input BAM and >=1 reference library / output pair");
  auto now = []() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  const double t_start = now();
  const int threads = std::max(1, num_cores);
  const int GZ_LEVEL = rows_gz_level();
  AnyOrderSetup S;
  int rc = S.open(reference_json, n_refs, strand_filter, trim, threads, device);
  if (rc != NB_OK) return rc;
  nbg::Device* dev = S.dev;
  std::vector<FILE*> outs(n_refs, nullptr); std::vector<bool> first_write(n_refs, true);
  struct Closer { std::vector<FILE*>& f; ~Closer() { for (FILE* x : f) if (x) fclose(x); } } closer{outs};
  for (u32 i = 0; i < n_refs && rc == NB_OK; i++) { outs[i] = fopen(output_paths[i], "wb"); if (!outs[i]) rc = fail(NB_ERR_IO, std::string("could not open output ") + output_paths[i]); }
  if (rc != NB_OK) return rc;
  const double t_setup = now();
  std::vector<std::string> reasons(256); for (int r = 0; r < 256; r++) reasons[r] = nb_reason_str(r);
  // the deflate + write of one chunk, on its own thread while the device goes on; errors come back through the future
  typedef std::pair<int, std::string> Res;
  std::future<Res> fut; double t_deflate = 0;
  auto join = [&]() -> int { if (!fut.valid()) return NB_OK; Res r = fut.get(); if (r.first) set_error(r.second); return r.first; };
  auto write_chunk = [&, threads, GZ_LEVEL](FILE* f, const char* p, u64 n) -> Res {
    const double t0 = now();
    const u64 PART = (u64)1 << 20;
    std::vector<u64> cut(1, 0);   // parts of about PART bytes, each ending at the end of a row
    while (cut.back() < n) { u64 e = cut.back() + PART; if (e >= n) e = n; else { const char* nl = (const char*)memchr(p + e - 1, '\n', n - (e - 1)); e = nl ? (u64)(nl - p) + 1 : n; } cut.push_back(e); }
    const size_t parts = cut.size() - 1;
    std::vector<std::string> member(parts); std::vector<char> bad(parts, 0); std::atomic<size_t> next(0);
    parallel_ranges((int)std::min<size_t>(threads, parts), (size_t)std::min<size_t>(threads, parts), [&](size_t, size_t, int) {
      for (size_t i; (i = next.fetch_add(1)) < parts;) if (!rows_member(p + cut[i], cut[i + 1] - cut[i], GZ_LEVEL, member[i])) bad[i] = 1; });
    for (size_t i = 0; i < parts; i++) {
      if (bad[i]) return Res(NB_ERR_IO, "gzip of the TSV rows failed");
      if (fwrite(member[i].data(), 1, member[i].size(), f) != member[i].size()) return Res(NB_ERR_IO, "short write on the TSV");
    }
    t_deflate += now() - t0;
    return Res(NB_OK, std::string());
  };
  CellDict cells; AnyOrderRun run; nbg::RowsStats rst;
  const u64 BATCH_PAIRS = 1u << 20;   // batches: whole scopes, at most 2^20 pairs (a larger scope is a batch of its own)
  double t_align = 0; u64 n_batches = 0;
  std::string feats; std::vector<u64> feat_off;
  rc = any_order_passes(input_file, threads, any_order_window_bytes(), dev, budget, true, cells, run, [&](int, const nbg::Grouped& g, u32 max_len) -> int {
    std::vector<std::pair<u64, u64>> batches; u64 maxp = 0;
    for (u64 s0 = 0; s0 < g.n_scopes;) {
      u64 s1 = s0 + 1;
      while (s1 < g.n_scopes && g.scope_pair0[s1 + 1] - g.scope_pair0[s0] <= BATCH_PAIRS) s1++;
      if (g.scope_pair0[s1] > g.scope_pair0[s0]) { batches.push_back({s0, s1}); maxp = std::max(maxp, g.scope_pair0[s1] - g.scope_pair0[s0]); }
      s0 = s1;
    }
    if (batches.empty()) return NB_OK;
    int e = nbg::rows_begin(dev, maxp); if (e) return e;
    nb_read_result* rres = nullptr; nb_pair_result* pres = nullptr; nbg::rows_results(dev, &rres, &pres);
    for (const auto& bt : batches) {
      const u64 s0 = bt.first, p0 = g.scope_pair0[s0], p1 = g.scope_pair0[bt.second];
      n_batches++;
      nb_batch b; e = nbg::batch(dev, p0, p1, s0, max_len, b); if (e) return e;
      for (u32 li = 0; li < n_refs; li++) {
        const double tb = now();
        e = nb_counts_reset(S.ctx[li]);
        if (e == NB_OK) e = nb_ctx_set_option(S.ctx[li], "max_batch_pairs", p1 - p0);
        if (e == NB_OK) e = nb_align_batch(S.ctx[li], &b, rres, pres);
        nb_counts cts;
        if (e == NB_OK) e = nb_counts_finalize(S.ctx[li], &cts);
        nbg::RowsBatch RB; RB.p0 = p0; RB.p1 = p1; RB.reasons = &reasons;
        if (e == NB_OK) e = nb_counts_device_rows(S.ctx[li], &RB.row_scope, &RB.row_callset, &RB.row_count, &RB.n_rows);
        if (e == NB_OK) e = nb_counts_device_slot_map(S.ctx[li], &RB.slot_map, &RB.n_slots);
        t_align += now() - tb;
        if (e) return e;
        if (!RB.n_rows) continue;
        // the text of every callset of this finalize: its group names joined by ','
        feats.clear(); feat_off.assign(1, 0);
        for (u64 c = 0; c < cts.n_callsets; c++) {
          for (u64 k = cts.callset_off[c]; k < cts.callset_off[c + 1]; k++) { if (k > cts.callset_off[c]) feats += ','; feats += nb_library_group_name(S.libs[li], cts.callset_items[k]); }
          feat_off.push_back(feats.size());
        }
        RB.feats = &feats; RB.feat_off = &feat_off;
        FILE* f = outs[li];
        e = nbg::rows_build(dev, RB, [&, f, li](const char* p, u64 n) -> int {
          int er = join(); if (er) return er;
          if (first_write[li]) { er = write_rows_header(f, GZ_LEVEL); if (er) return er; first_write[li] = false; }
          fut = std::async(std::launch::async, [&write_chunk, f, p, n]() { return write_chunk(f, p, n); });
          return NB_OK;
        }, rst);
        if (e) return e;
      }
    }
    return NB_OK;
  });
  { const int er = join(); if (er && rc == NB_OK) rc = er; }
  for (u32 li = 0; li < n_refs && rc == NB_OK; li++) if (first_write[li]) rc = write_rows_empty(outs[li], GZ_LEVEL);
  for (u32 li = 0; li < n_refs; li++) { if (outs[li] && fclose(outs[li]) != 0 && rc == NB_OK) rc = fail(NB_ERR_IO, std::string("short write on ") + output_paths[li]); outs[li] = nullptr; }
  const double t_end = now();
  if (getenv("NB_BAM_STATS")) {
    char b[1024];
    snprintf(b, sizeof b, ", rows %llu, row bytes %llu, row chunks %llu (at most %llu per batch), metadata %llu bytes, metadata text %llu bytes, metadata formatting %.2fs, row buffer %llu bytes, device peak %llu bytes, device row build %.3fs, deflate+write %.3fs",
             (unsigned long long)rst.rows, (unsigned long long)rst.bytes, (unsigned long long)rst.chunks, (unsigned long long)rst.max_chunks, (unsigned long long)(dev ? nbg::meta_bytes(dev) : 0),
             (unsigned long long)run.meta_text, run.ld.t_meta, (unsigned long long)nbg::rows_buffer_cap(), (unsigned long long)(dev ? nbg::peak_bytes(dev) : 0), rst.t_device, t_deflate);
    any_order_stats(run, dev, budget, n_batches, 0, t_setup - t_start, t_align, 0, 0, t_end - t_start, b);
  }
  return rc;
}

// The device grouping, one line per pair in batch order: scope index (counting the scopes with pairs), the scope's cell
// barcode, the file ordinals of the sequence-slot and mate-slot records, both NB_FLAG_* and both clipped lengths.  With
// slots: the pass index first, and each slot's clipped bases and quals (hex) as the store holds them after the pass.
int dump_scopes_any_order(const char* input_file, int num_cores, int device, u64 budget, const char* out_path, bool slots) {
  if (!input_file || !out_path) return fail(NB_ERR_INVALID, "null argument");
  nbg::Device* dev = nullptr;
  int rc = nbg::create(device, &dev);
  CellDict cells; AnyOrderRun run;
  std::string out; u64 shown = 0;
  static const char* SEQ = "=ACMGRSVTWYHKDBN"; static const char* H = "0123456789abcdef";
  if (rc == NB_OK) rc = any_order_passes(input_file, std::max(1, num_cores), any_order_window_bytes(), dev, budget, false, cells, run, [&](int pass, const nbg::Grouped& g, u32) -> int {
    std::vector<u64> o1, o2, b1, b2; std::vector<u8> f1, f2, nib, qual; std::vector<u32> l1, l2;
    int e = nbg::pairs_to_host(dev, o1, o2, f1, f2, l1, l2);
    if (e == NB_OK && slots) e = nbg::slots_to_host(dev, b1, b2, nib, qual);
    if (e) return e;
    auto slot = [&](u64 at, u32 n) {
      out += '\t'; for (u64 k = at; k < at + n; k++) out += SEQ[(nib[k >> 1] >> ((k & 1) ? 0 : 4)) & 15];
      out += '\t'; for (u64 k = at; k < at + n; k++) { out += H[qual[k] >> 4]; out += H[qual[k] & 15]; }
    };
    char line[256];
    for (u64 s = 0; s < g.n_scopes; s++) {
      if (g.scope_pair0[s + 1] == g.scope_pair0[s]) continue;
      const char* cb = cells.names.data() + cells.off[g.scope_cb[s]];
      for (u64 p = g.scope_pair0[s]; p < g.scope_pair0[s + 1]; p++) {
        if (slots) { snprintf(line, sizeof line, "%d\t", pass); out += line; }
        snprintf(line, sizeof line, "%llu\t", (unsigned long long)shown); out += line; out += cb;
        snprintf(line, sizeof line, "\t%llu\t%llu\t%u\t%u\t%u\t%u", (unsigned long long)o1[p], (unsigned long long)o2[p], f1[p], f2[p], l1[p], l2[p]); out += line;
        if (slots) { slot(b1[p], l1[p]); slot(b2[p], l2[p]); }
        out += '\n';
      }
      shown++;
    }
    return NB_OK;
  });
  nbg::destroy(dev);
  if (rc) return rc;
  FILE* f = fopen(out_path, "wb"); if (!f) return fail(NB_ERR_IO, std::string("could not open ") + out_path);
  const bool ok = fwrite(out.data(), 1, out.size(), f) == out.size();
  if (fclose(f) != 0 || !ok) return fail(NB_ERR_IO, std::string("short write on ") + out_path);
  return NB_OK;
}

}  // namespace

extern "C" int nb_process_bam_cells_any_order(const char* input_file, const char* const* reference_json, const char* const* matrix_dirs, uint32_t n_refs,
                                              int strand_filter, const char* trim, int num_cores, int device) {
  return process_bam_cells_any_order(input_file, reference_json, matrix_dirs, n_refs, strand_filter, trim, num_cores, device, 0);
}

extern "C" int nb_process_bam_cells_any_order_budget(const char* input_file, const char* const* reference_json, const char* const* matrix_dirs, uint32_t n_refs,
                                                     int strand_filter, const char* trim, int num_cores, int device, uint64_t budget_bytes) {
  return process_bam_cells_any_order(input_file, reference_json, matrix_dirs, n_refs, strand_filter, trim, num_cores, device, budget_bytes);
}

extern "C" int nb_process_bam_rows_any_order(const char* input_file, const char* const* reference_json, const char* const* output_paths, uint32_t n_refs,
                                             int strand_filter, const char* trim, int num_cores, int device, uint64_t budget_bytes) {
  return process_bam_rows_any_order(input_file, reference_json, output_paths, n_refs, strand_filter, trim, num_cores, device, budget_bytes);
}

extern "C" int nb_bam_dump_scopes_any_order(const char* input_file, int num_cores, int device, const char* out_path) {
  return dump_scopes_any_order(input_file, num_cores, device, 0, out_path, false);
}

extern "C" int nb_bam_dump_scopes_any_order_budget(const char* input_file, int num_cores, int device, uint64_t budget_bytes, const char* out_path) {
  return dump_scopes_any_order(input_file, num_cores, device, budget_bytes, out_path, true);
}

extern "C" int nb_any_order_umi_bucket(const char* umi, uint32_t len, uint32_t* bucket) {
  if (!umi || !bucket) return fail(NB_ERR_INVALID, "null argument");
  u64 key;
  if (!nbg::pack_umi(umi, len, key)) return fail(NB_ERR_UNSUPPORTED, "UMI \"" + std::string(umi, len) + "\" cannot be packed into the exact device key");
  *bucket = nbg::umi_bucket(key);
  return NB_OK;
}
