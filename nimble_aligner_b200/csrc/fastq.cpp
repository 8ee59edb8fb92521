// fastq.cpp — FASTQ(.gz) feeder, FASTQ-mode TSV writer and the process::fastq::process driver.
// Mirrors /root/reference/src/parse/fastq.rs:8-43 (niffler gz autodetect + bio fastq records -> DnaString::from_acgt_bytes),
// src/utils.rs:27-51 (write_to_tsv: append, header iff empty, features TAB-joined) and src/process/fastq.rs:7-30.
//
// Three feeders behind one interface (a stream of parsed segments: bases concatenated in pinned memory + offsets):
//   MapStream  plain FASTQ: the file is mapped and cut into byte chunks that T host threads parse at the same time.  A chunk
//              starts at the first record start at or after its byte boundary, found by a local pattern test ('@' line whose
//              next-but-one line starts with '+' and whose sequence and quality lines are equally long).  That guess is never
//              trusted: the consumer accepts chunk c only if it began exactly where the parse of chunk c-1 ended, and parses
//              it again from that position otherwise (multi-line records can defeat the pattern; the result is then still
//              that of the sequential parse, only slower).
//   GzParStream  gzip input (sniffed by its magic bytes, like niffler) with two or more threads for the file: pgunzip.hpp
//              inflates it on all of them (entry points at guessed block headers, confirmed by a chain through the chunks),
//              each worker parses the text of its chunk, the consumer parses the few lines at the chunk junctions.
//   GzStream   gzip input with one thread: one thread inflates (inflate.hpp over the mapped file), a second one parses.
// The consumer hands min(records left in R1's segment, records left in R2's) pairs to nb_align_batch at a time, so the two
// files never have to be cut at the same record numbers.
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>
#include <time.h>
#include <zlib.h>

#include <algorithm>
#include <atomic>
#include <cerrno>
#include <condition_variable>
#include <cstdio>
#include <cstring>
#include <deque>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "host.hpp"
#include "inflate.hpp"
#include "pgunzip.hpp"

using namespace nb;

namespace {

std::atomic<bool> g_pageable{false};   // nb_fastq_dump (host-only parity tests of the feeder) runs without a CUDA device
struct Pinned {
  u8* p = nullptr; size_t cap = 0; bool pageable = false;
  void drop() { if (pageable) free(p); else nb_host_free(p); p = nullptr; cap = 0; }
  ~Pinned() { drop(); }
  bool ensure(size_t n, size_t keep) {
    if (n <= cap) return true;
    const size_t nc = std::max(n, cap * 2 + (1 << 20)); const bool pg = g_pageable.load();
    u8* q = (u8*)(pg ? malloc(nc) : nb_host_alloc(nc)); if (!q) return false;
    if (keep) memcpy(q, p, keep);
    drop(); p = q; cap = nc; pageable = pg; return true;
  }
};

// records of one stretch of one input stream: bases concatenated in pinned memory, n + 1 offsets (pinned too: they are copied
// to the device asynchronously)
struct Segment {
  Pinned seq, offb; u64 n = 0; u32 maxlen = 0; size_t used = 0;
  int status = 1;               // 1 more may follow, 0 end of file, -1 malformed, -2 out of pinned memory, -3 damaged gzip stream
  size_t start = 0, end = 0;    // MapStream: byte positions of the first record and behind the last one
  u64* off() const { return (u64*)offb.p; }
  void clear() { n = 0; maxlen = 0; used = 0; status = 1; }
  bool push_off() { if (!offb.ensure((n + 2) * 8, (n + 1) * 8)) return false; off()[n + 1] = used; return true; }
  bool begin() { clear(); if (!offb.ensure(1 << 16, 0)) return false; off()[0] = 0; return true; }
};

struct SegStream {
  virtual ~SegStream() {}
  virtual Segment* next() = 0;            // blocks; the caller gives every segment back with recycle()
  virtual void recycle(Segment*) = 0;
  virtual void finish() = 0;              // stops the threads (also mid-stream, after an error elsewhere)
};

// ------------------------------------------------------------------------------------------------ gzip: inflate thread -> parse thread
// A gzip stream cannot be entered in the middle, so one .gz file is inflated by ONE thread — with the decoder of inflate.hpp
// over the mapped file (zlib's gzread ran at 0.4 GB/s per stream and was the whole cost of the .gz path) — into text chunks
// that a second thread parses while the next chunk is inflated.  A chunk buffer starts with the 32 KiB of text before it
// (the deflate window), then up to GZ_CHUNK bytes of new text.
struct GzText {
  static const size_t HIST = 32768; size_t GZ_CHUNK = (size_t)4 << 20;   // NB_GZ_CHUNK_KB overrides (tests: lines that straddle many chunk borders)
  struct Chunk { std::vector<u8> buf; size_t len = 0; int status = 1; const char* data() const { return (const char*)buf.data() + HIST; } };   // status: 1 more follows, 0 last, -3 damaged gzip stream
  int fd = -1; const u8* map = nullptr; size_t size = 0; nbz::GzipStream gz;
  std::vector<std::unique_ptr<Chunk>> chunks; std::vector<Chunk*> free_q; std::deque<Chunk*> filled_q; std::mutex m; std::condition_variable cv; bool stop = false; std::thread th;
  bool open(const std::string& p) {
    fd = ::open(p.c_str(), O_RDONLY); if (fd < 0) return false;
    struct stat st; if (fstat(fd, &st) != 0) return false;
    size = (size_t)st.st_size;
    if (size) { void* q = mmap(nullptr, size, PROT_READ, MAP_PRIVATE, fd, 0); if (q == MAP_FAILED) return false; map = (const u8*)q; madvise(q, size, MADV_SEQUENTIAL); }
    gz.open(map, size);
    if (const char* e = getenv("NB_GZ_CHUNK_KB")) { const size_t kb = (size_t)strtoull(e, nullptr, 10); if (kb >= 1) GZ_CHUNK = kb << 10; }
    for (int i = 0; i < 4; i++) { chunks.emplace_back(new Chunk()); chunks.back()->buf.resize(HIST + GZ_CHUNK); free_q.push_back(chunks.back().get()); }
    th = std::thread([this] { run(); });
    return true;
  }
  void run() {
    Chunk* prev = nullptr;
    for (;;) {
      Chunk* c;
      { std::unique_lock<std::mutex> lk(m); cv.wait(lk, [&] { return stop || !free_q.empty(); }); if (stop) return; c = free_q.back(); free_q.pop_back(); }
      u8* b = c->buf.data();
      if (prev) memcpy(b, prev->buf.data() + prev->len, HIST);      // the last HIST bytes of [history | text] of the chunk before (still intact: only this thread writes chunks)
      const ptrdiff_t n = gz.read(prev ? b : b + HIST, b + HIST, b + HIST + GZ_CHUNK);
      c->len = n < 0 ? 0 : (size_t)n; c->status = n < 0 ? -3 : gz.done() ? 0 : 1;
      const int st = c->status; prev = c;
      { std::lock_guard<std::mutex> lk(m); filled_q.push_back(c); }
      cv.notify_all();
      if (st != 1) return;
    }
  }
  Chunk* next() { std::unique_lock<std::mutex> lk(m); cv.wait(lk, [&] { return !filled_q.empty(); }); Chunk* c = filled_q.front(); filled_q.pop_front(); return c; }
  void recycle(Chunk* c) { { std::lock_guard<std::mutex> lk(m); free_q.insert(free_q.begin(), c); } cv.notify_all(); }   // (reused last: the inflate thread copies its history from the newest chunk)
  void finish() { { std::lock_guard<std::mutex> lk(m); stop = true; } cv.notify_all(); if (th.joinable()) th.join(); }
  ~GzText() { finish(); if (map) munmap((void*)map, size); if (fd >= 0) ::close(fd); }
};
// One FASTQ.gz stream parsed in place: lines are views into the text chunks (a line that straddles two chunks is put
// together in `carry`), no per-line strings.
struct FastqReader {
  GzText src; GzText::Chunk* cur = nullptr; size_t pos = 0; bool eof = false, damaged = false, carry_out = false; std::string carry;
  bool open(const std::string& p) { return src.open(p); }
  // one line without its terminator; false at end of input (or at a damaged gzip stream: `damaged`)
  bool line(const char*& out, size_t& n) {
    if (carry_out) { carry.clear(); carry_out = false; }
    for (;;) {
      if (cur) {
        const char* s = cur->data() + pos; const size_t left = cur->len - pos;
        const char* nl = left ? (const char*)memchr(s, '\n', left) : nullptr;
        if (nl) {
          const size_t k = (size_t)(nl - s); pos += k + 1;
          if (carry.empty()) { out = s; n = k; } else { carry.append(s, k); out = carry.data(); n = carry.size(); carry_out = true; }
          if (n && out[n - 1] == '\r') n--;
          return true;
        }
        carry.append(s, left);
        const int st = cur->status; src.recycle(cur); cur = nullptr;
        if (st != 1) { eof = true; damaged = st < 0; }
      }
      if (eof) {
        if (damaged || carry.empty()) return false;
        out = carry.data(); n = carry.size(); carry_out = true; if (n && out[n - 1] == '\r') n--; return true;   // last line without a newline
      }
      cur = src.next(); pos = 0;
    }
  }
};

// fills g from r; multi-line records are accepted like bio::io::fastq does
void parse_block(FastqReader& r, Segment& g, u64 want) {
  if (!g.begin()) { g.status = -2; return; }
  const char* s; size_t n;
  while (g.n < want) {
    do { if (!r.line(s, n)) { g.status = r.damaged ? -3 : 0; return; } } while (n == 0);
    if (s[0] != '@') { g.status = -1; return; }
    size_t start = g.used;
    for (;;) {
      if (!r.line(s, n)) { g.status = r.damaged ? -3 : -1; return; }
      if (n && s[0] == '+') break;
      if (!g.seq.ensure(g.used + n + 64, g.used)) { g.status = -2; return; }
      memcpy(g.seq.p + g.used, s, n); g.used += n;
    }
    size_t slen = g.used - start, qlen = 0;
    while (qlen < slen) { if (!r.line(s, n)) { g.status = r.damaged ? -3 : -1; return; } qlen += n; }
    if (qlen != slen) { g.status = -1; return; }
    if (!g.push_off()) { g.status = -2; return; }
    g.maxlen = std::max<u32>(g.maxlen, (u32)slen); g.n++;
  }
}

struct GzStream : SegStream {
  FastqReader rd; std::vector<std::unique_ptr<Segment>> blocks; std::vector<Segment*> free_q; std::deque<Segment*> filled_q; std::mutex m; std::condition_variable cv; bool stop = false; std::thread th; u64 want;
  GzStream(u64 w, int extra) : want(w) { for (int i = 0; i < 4 + extra; i++) blocks.emplace_back(new Segment()); }   // the consumer holds up to 3 + extra segments
  bool open(const std::string& p) { if (!rd.open(p)) return false; for (auto& b : blocks) free_q.push_back(b.get()); th = std::thread([this] { run(); }); return true; }
  void run() {
    for (;;) {
      Segment* b;
      { std::unique_lock<std::mutex> lk(m); cv.wait(lk, [&] { return stop || !free_q.empty(); }); if (stop) return; b = free_q.back(); free_q.pop_back(); }
      parse_block(rd, *b, want);
      { std::lock_guard<std::mutex> lk(m); filled_q.push_back(b); }
      cv.notify_all();
      if (b->status != 1) return;
    }
  }
  Segment* next() override { std::unique_lock<std::mutex> lk(m); cv.wait(lk, [&] { return !filled_q.empty(); }); Segment* b = filled_q.front(); filled_q.pop_front(); return b; }
  void recycle(Segment* b) override { { std::lock_guard<std::mutex> lk(m); free_q.push_back(b); } cv.notify_all(); }
  void finish() override { { std::lock_guard<std::mutex> lk(m); stop = true; } cv.notify_all(); if (th.joinable()) th.join(); }
  ~GzStream() override { finish(); }
};

// ------------------------------------------------------------------------------------------------ plain text: mapped file, parallel chunks
inline size_t next_line(const char* d, size_t size, size_t pos) {   // start of the line after the one holding pos (size when there is none)
  if (pos >= size) return size;
  const char* nl = (const char*)memchr(d + pos, '\n', size - pos);
  return nl ? (size_t)(nl - d) + 1 : size;
}
inline size_t line_len(const char* d, size_t size, size_t pos) {    // without terminator / '\r'
  size_t e = next_line(d, size, pos); size_t n = e - pos;
  if (n && d[pos + n - 1] == '\n') n--;
  if (n && d[pos + n - 1] == '\r') n--;
  return n;
}
inline size_t skip_blank(const char* d, size_t size, size_t pos) {  // parse_block's `while (n == 0)`: empty lines between records
  while (pos < size) { if (d[pos] == '\n') pos++; else if (d[pos] == '\r' && pos + 1 < size && d[pos + 1] == '\n') pos += 2; else if (d[pos] == '\r' && pos + 1 == size) pos++; else break; }
  return pos;
}
// records whose first byte lies in [pos, bound): same grammar and the same failures as parse_block.  Appends to g; returns
// the position of the next record (blank lines skipped).
size_t parse_range(const char* d, size_t size, size_t pos, size_t bound, Segment& g, bool* ran_out = nullptr) {   // ran_out: the data ended inside a record (status -1, nothing of that record kept)
  pos = skip_blank(d, size, pos);
  while (pos < bound && pos < size) {
    if (d[pos] != '@') { g.status = -1; return pos; }
    size_t p = next_line(d, size, pos);
    const size_t start = g.used;
    for (;;) {                                      // sequence lines up to the '+' line
      if (p >= size) { g.status = -1; g.used = start; if (ran_out) *ran_out = true; return pos; }
      size_t e = next_line(d, size, p), n = e - p;
      if (n && d[p + n - 1] == '\n') n--;
      if (n && d[p + n - 1] == '\r') n--;
      if (n && d[p] == '+') { p = e; break; }
      if (!g.seq.ensure(g.used + n + 64, g.used)) { g.status = -2; return pos; }
      memcpy(g.seq.p + g.used, d + p, n); g.used += n; p = e;
    }
    const size_t slen = g.used - start; size_t qlen = 0;
    while (qlen < slen) {
      if (p >= size) { g.status = -1; g.used = start; if (ran_out) *ran_out = true; return pos; }
      size_t e = next_line(d, size, p), n = e - p;
      if (n && d[p + n - 1] == '\n') n--;
      if (n && d[p + n - 1] == '\r') n--;
      qlen += n; p = e;
    }
    if (qlen != slen) { g.status = -1; g.used = start; return pos; }
    if (!g.push_off()) { g.status = -2; return pos; }
    g.maxlen = std::max<u32>(g.maxlen, (u32)slen); g.n++;
    pos = skip_blank(d, size, p);
  }
  return pos;
}
// first position >= from that LOOKS like a record start (see the file comment); size when there is none
size_t guess_start(const char* d, size_t size, size_t from) {
  if (from == 0) return skip_blank(d, size, 0);
  size_t pos = next_line(d, size, from - 1);
  for (int tries = 0; tries < 4096; tries++) {
    pos = skip_blank(d, size, pos);
    if (pos >= size) return size;
    if (d[pos] == '@') {
      size_t l1 = next_line(d, size, pos), l2 = next_line(d, size, l1);
      if (l2 < size && d[l2] == '+') { size_t l3 = next_line(d, size, l2); if (line_len(d, size, l1) == line_len(d, size, l3)) return pos; }
    }
    pos = next_line(d, size, pos);
  }
  return pos;
}

struct MapStream : SegStream {
  const char* d = nullptr; size_t size = 0; int fd = -1; size_t chunk = 8u << 20; u64 n_chunks = 0;
  struct Slot { Segment seg; bool filled = false; };
  std::vector<std::unique_ptr<Slot>> ring; std::vector<std::thread> th;
  std::mutex m; std::condition_variable cv; bool stop = false;
  std::atomic<u64> next_chunk{0}; u64 take = 0, released = 0;   // chunks handed to the consumer / given back by it
  size_t expected = 0; Segment tail;                               // tail: the empty end-of-file segment of an empty input

  bool open(const std::string& p, int threads, size_t chunk_bytes, int extra) {
    fd = ::open(p.c_str(), O_RDONLY); if (fd < 0) return false;
    struct stat st; if (fstat(fd, &st) != 0 || !S_ISREG(st.st_mode)) { ::close(fd); fd = -1; return false; }
    size = (size_t)st.st_size; chunk = std::max<size_t>(chunk_bytes, 4096);
    if (size) {
      void* q = mmap(nullptr, size, PROT_READ, MAP_PRIVATE, fd, 0);
      if (q == MAP_FAILED) { ::close(fd); fd = -1; return false; }
      d = (const char*)q; madvise(q, size, MADV_SEQUENTIAL);
    }
    n_chunks = (size + chunk - 1) / chunk;
    threads = (int)std::max<u64>(1, std::min<u64>((u64)std::max(threads, 1), n_chunks));
    for (int i = 0; i < 2 * threads + 4 + extra; i++) ring.emplace_back(new Slot());   // the consumer holds up to 3 + extra segments
    expected = skip_blank(d, size, 0);
    for (int i = 0; i < threads && n_chunks; i++) th.emplace_back([this] { work(); });
    return true;
  }
  void parse_chunk(u64 c, size_t from, Segment& g) {
    const size_t bound = std::min(size, (size_t)(c + 1) * chunk);
    if (!g.begin()) { g.status = -2; g.start = g.end = from; return; }
    g.start = from;
    if (from >= bound) { g.end = from; return; }
    if (!g.seq.ensure((bound - from) / 2 + (1 << 16), 0)) { g.status = -2; g.end = from; return; }
    g.end = parse_range(d, size, from, bound, g);
  }
  void work() {
    const u64 R = ring.size();
    for (;;) {
      const u64 c = next_chunk.fetch_add(1);
      if (c >= n_chunks) return;
      Slot& s = *ring[c % R];
      { std::unique_lock<std::mutex> lk(m); cv.wait(lk, [&] { return stop || c < released + R; }); if (stop) return; }   // slot c % R is free once chunk c - R came back
      parse_chunk(c, guess_start(d, size, (size_t)c * chunk), s.seg);
      { std::lock_guard<std::mutex> lk(m); s.filled = true; }
      cv.notify_all();
    }
  }
  Segment* next() override {
    if (take >= n_chunks) { tail.status = tail.begin() ? 0 : -2; tail.n = 0; return &tail; }   // empty input (or a caller that asks again after the end)
    const u64 c = take++; Slot& s = *ring[c % ring.size()];
    { std::unique_lock<std::mutex> lk(m); cv.wait(lk, [&] { return s.filled; }); s.filled = false; }
    Segment& g = s.seg;
    const size_t bound = std::min(size, (size_t)(c + 1) * chunk);
    if (expected >= bound) { g.begin(); g.start = g.end = expected; }             // a record of the previous chunk runs past this whole chunk
    else if (g.start != expected) parse_chunk(c, expected, g);                      // the guess was wrong: this chunk again, from where the sequential parse stands
    expected = g.end;
    if (g.status == 1 && c + 1 == n_chunks) g.status = 0;
    return &g;
  }
  void recycle(Segment* g) override {
    if (g == &tail) return;
    // slots are reused in chunk order, so segments must come back in the order next() handed them out (consume() and the
    // driver's `held` queue do)
    { std::lock_guard<std::mutex> lk(m); released++; }
    cv.notify_all();
  }
  void finish() override {
    { std::lock_guard<std::mutex> lk(m); stop = true; }
    cv.notify_all();
    for (auto& t : th) if (t.joinable()) t.join();
    th.clear();
  }
  ~MapStream() override { finish(); if (d) munmap((void*)d, size); if (fd >= 0) ::close(fd); }
};

// ------------------------------------------------------------------------------------------------ gzip on several threads
// pgunzip.hpp inflates one .gz file on T threads, chunk by chunk; each worker also PARSES the text of its chunk, from the
// first position that looks like a record start (guess_start) to the last record that is complete in the chunk.  What lies in
// front of the guess and behind the last complete record are a few lines per chunk; the consumer parses those — the bytes
// carried over from the chunk before plus this chunk's head — in file order, and takes the worker's records only if that
// parse ends exactly at the guess (then the guess was a record boundary of the sequential parse, and the worker's records
// are what the sequential parse yields from there).  Otherwise it parses the chunk's text again from the carried bytes.
struct GzParStream : SegStream {
  int fd = -1; const u8* map = nullptr; size_t size = 0; nbz::ParallelGunzip pg;
  struct Parsed { Segment* seg = nullptr; size_t head_end = 0, tail_start = 0; };   // a worker's result, carried by the chunk (user_ptr, user_a, user_b)
  std::vector<std::unique_ptr<Segment>> segs; std::vector<Segment*> free_segs; std::mutex m; std::condition_variable cv; bool stop = false;
  std::deque<Segment*> ready; std::string carry, piece; bool ended = false;
  Segment* take_seg() { std::unique_lock<std::mutex> lk(m); cv.wait(lk, [&] { return stop || !free_segs.empty(); }); if (stop) return nullptr; Segment* g = free_segs.back(); free_segs.pop_back(); return g; }
  void give_seg(Segment* g) { { std::lock_guard<std::mutex> lk(m); free_segs.push_back(g); } cv.notify_all(); }
  bool open(const std::string& p, int threads, int extra) {
    fd = ::open(p.c_str(), O_RDONLY); if (fd < 0) return false;
    struct stat st; if (fstat(fd, &st) != 0) return false;
    size = (size_t)st.st_size;
    if (size) { void* q = mmap(nullptr, size, PROT_READ, MAP_PRIVATE, fd, 0); if (q == MAP_FAILED) return false; map = (const u8*)q; madvise(q, size, MADV_SEQUENTIAL); }
    // compressed bytes per chunk: 2 MiB is about 8 MB of text = 25 k records, the plain-text parser's granularity (one
    // nb_align_batch call per segment: smaller chunks made the calls, not the inflate, the bound on the box); 4 MiB for a file
    // that still gives every worker eight of them
    size_t cbytes = std::min((size_t)4 << 20, std::max((size_t)2 << 20, size / ((size_t)std::max(1, threads) * 8)));
    if (const char* e = getenv("NB_GZ_CHUNK_KB")) { const size_t kb = (size_t)strtoull(e, nullptr, 10); if (kb >= 1) cbytes = kb << 10; }
    const int n_segs = 2 * (2 * threads + 2) + 3 + extra + 4;                         // two per chunk in flight (its records, the junction's) + what the consumer holds
    for (int i = 0; i < n_segs; i++) { segs.emplace_back(new Segment()); free_segs.push_back(segs.back().get()); }
    pg.open(map, size, threads, cbytes, [this](size_t k, nbz::PgChunk& c) { parse_chunk(k, c); });
    return true;
  }
  // worker: the records that lie completely inside this chunk's text
  void parse_chunk(size_t k, nbz::PgChunk& c) {
    Parsed p;
    struct Put { Parsed& p; nbz::PgChunk& c; ~Put() { c.user_ptr = p.seg; c.user_a = p.head_end; c.user_b = p.tail_start; } } put{p, c};
    const char* d = (const char*)c.text.data(); const size_t n = c.text.size();
    p.head_end = p.tail_start = n;
    if (c.status < 0 || !n) return;
    const size_t g = k == 0 ? skip_blank(d, n, 0) : guess_start(d, n, 1);
    if (g >= n) return;
    Segment* sg = take_seg(); if (!sg) return;
    if (!sg->begin() || !sg->seq.ensure(n / 2 + 65536, 0) || !sg->offb.ensure((n / 64 + 1024) * 8, 8)) { sg->status = -2; p.seg = sg; p.head_end = g; return; }   // sized once: growing a pinned buffer step by step costs a cudaMallocHost and a copy each time
    bool ran_out = false;
    const size_t e = parse_range(d, n, g, n, *sg, &ran_out);
    if (sg->status == -1 && ran_out) sg->status = 1;                                  // the last record continues in the next chunk
    p.seg = sg; p.head_end = g; p.tail_start = e;                                     // (status -1 left: not a record where the guess said — the consumer parses again)
  }
  Segment* next() override {
    while (ready.empty()) {
      if (ended) return nullptr;
      nbz::PgChunk* c = pg.next();
      Segment* out = take_seg(); if (!out) return nullptr;
      if (!c || c->status < 0 || !out->begin()) { out->clear(); out->status = !c || c->status < 0 ? -3 : -2; ready.push_back(out); ended = true; if (c) pg.recycle(c); break; }
      Parsed p; p.seg = (Segment*)c->user_ptr; p.head_end = c->user_a; p.tail_start = c->user_b; c->user_ptr = nullptr;
      const char* d = (const char*)c->text.data(); const size_t n = c->text.size(); const bool last = c->status == 0;
      bool taken = false;
      if (p.seg && p.seg->status == 1 && p.head_end < n) {
        piece.assign(carry); piece.append(d, p.head_end);
        bool ro = false; const size_t e = parse_range(piece.data(), piece.size(), 0, piece.size(), *out, &ro);
        if (out->status == 1 && e >= piece.size()) {                                   // the junction parses up to the guess: the worker's records follow
          ready.push_back(out); ready.push_back(p.seg); p.seg = nullptr;
          carry.assign(d + p.tail_start, n - p.tail_start); taken = true;
        } else if (out->status == -2) { ready.push_back(out); ended = true; pg.recycle(c); break; }
        else out->begin();
      }
      if (!taken) {                                                                    // no usable guess in this chunk: its text behind the carried bytes, sequentially
        if (p.seg) { if (p.seg->status == -2) { out->clear(); out->status = -2; } give_seg(p.seg); p.seg = nullptr; }
        if (out->status == 1) {
          piece.assign(carry); piece.append(d, n);
          bool ro = false; const size_t e = parse_range(piece.data(), piece.size(), 0, piece.size(), *out, &ro);
          if (out->status == -1 && ro) out->status = 1;
          carry.assign(piece.data() + e, piece.size() - e);
        }
        ready.push_back(out);
        if (out->status != 1) { ended = true; pg.recycle(c); break; }
      }
      pg.recycle(c);
      if (last) {
        ended = true;
        Segment* fin = ready.back();
        if (!carry.empty()) { fin->status = -1; }                                      // the file ends inside a record
        else fin->status = 0;
      }
    }
    Segment* g = ready.front(); ready.pop_front(); return g;
  }
  void recycle(Segment* g) override { give_seg(g); }
  void finish() override { { std::lock_guard<std::mutex> lk(m); stop = true; } cv.notify_all(); pg.finish(); }
  ~GzParStream() override { finish(); if (map) munmap((void*)map, size); if (fd >= 0) ::close(fd); }
};

bool is_gzip(const std::string& p) { FILE* f = fopen(p.c_str(), "rb"); if (!f) return false; unsigned char h[2] = {0, 0}; size_t n = fread(h, 1, 2, f); fclose(f); return n == 2 && h[0] == 0x1f && h[1] == 0x8b; }

// extra: segments the consumer may hold beyond the usual three (a driver feeding W contexts in turn holds 2 W + 1)
std::unique_ptr<SegStream> open_stream(const std::string& path, int threads, u64 gz_block_records, size_t chunk_bytes, int extra = 0) {
  if (is_gzip(path)) {
    int gt = threads; if (const char* e = getenv("NB_GZ_THREADS")) gt = atoi(e);      // (1: the serial reader)
    if (gt >= 2) { std::unique_ptr<GzParStream> g(new GzParStream()); if (!g->open(path, gt, extra)) return nullptr; return g; }
    std::unique_ptr<GzStream> g(new GzStream(gz_block_records, extra)); if (!g->open(path)) return nullptr; return g;
  }
  std::unique_ptr<MapStream> s(new MapStream());
  if (!s->open(path, threads, chunk_bytes, extra)) return nullptr;
  return s;
}
u64 file_bytes(const char* p) { struct stat st; return stat(p, &st) == 0 ? (u64)st.st_size : 0; }
// Bytes of plain FASTQ per parse task = records per segment = pairs per nb_align_batch call.  A call costs about a
// millisecond whatever it carries (both drivers measured at one call per ms: 780 calls / 0.80 s on 10 M plain pairs,
// 453 calls / 0.46 s on 2 M .gz pairs), so a big file is cut into bigger chunks — as long as every parser thread still gets
// eight of them — and a small one keeps 8 MiB (25 k records).  NB_FASTQ_CHUNK overrides.
size_t chunk_bytes_default(u64 file_bytes = 0, int threads = 1) {
  const char* e = getenv("NB_FASTQ_CHUNK"); size_t v = e ? (size_t)strtoull(e, nullptr, 10) : 0; if (v) return v;
  const size_t lo = (size_t)8 << 20, hi = (size_t)32 << 20; const size_t want = (size_t)(file_bytes / ((u64)std::max(1, threads) * 8));
  return std::min(hi, std::max(lo, want));
}

int write_tsv(const std::string& path, const nb_library* lib, const nb_counts& cts) {  // utils::write_to_tsv
  FILE* f = fopen(path.c_str(), "ab");
  if (!f) return fail(NB_ERR_IO, "Unable to open file " + path);
  fseek(f, 0, SEEK_END);
  if (ftell(f) == 0) fputs("feature\tscore\n", f);
  for (u64 r = 0; r < cts.n_rows; r++) {
    u32 cs = cts.row_callset[r];
    for (u64 i = cts.callset_off[cs]; i < cts.callset_off[cs + 1]; i++) { fputs(nb_library_group_name(lib, cts.callset_items[i]), f); fputc('\t', f); }
    fprintf(f, "%lld\n", (long long)cts.row_count[r]);
  }
  fclose(f);
  return NB_OK;
}

// The consumer loop shared by the driver and the host-only dump: walks the one or two segment streams in lockstep and calls
// emit(seg1, first1, seg2, first2, m) for every stretch of m records both current segments still hold.  Error precedence
// follows the reference's zip over the two readers (src/process/fastq.rs:20-24): the first bad record wins, R1 before R2.
template <class Emit, class Retire>
int consume(SegStream* s1, SegStream* s2, Emit emit, Retire retire) {
  Segment* c1 = nullptr; Segment* c2 = nullptr; u64 k1 = 0, k2 = 0; bool end1 = false, end2 = !s2;
  int rc = NB_OK;
  for (;;) {
    while (!end1 && (!c1 || k1 == c1->n)) {
      if (c1) { int st = c1->status; retire(s1, c1); c1 = nullptr; if (st == 0) { end1 = true; break; } if (st == -2) return fail(NB_ERR_CUDA, "pinned allocation failed"); if (st == -3) return fail(NB_ERR_PARSE, "Error -- could not read R1: damaged or truncated gzip stream."); if (st == -1) return fail(NB_ERR_PARSE, "Error -- could not parse read. Input R1 data malformed."); }
      c1 = s1->next(); k1 = 0;
    }
    while (s2 && !end2 && (!c2 || k2 == c2->n)) {
      if (c2) { int st = c2->status; retire(s2, c2); c2 = nullptr; if (st == 0) { end2 = true; break; } if (st == -2) return fail(NB_ERR_CUDA, "pinned allocation failed"); if (st == -3) return fail(NB_ERR_PARSE, "Error -- could not read R2: damaged or truncated gzip stream."); if (st == -1) return fail(NB_ERR_PARSE, "Error -- could not parse reverse read. Input R2 data malformed."); }
      c2 = s2->next(); k2 = 0;
    }
    if (s2 && end1 != end2) return fail(NB_ERR_PARSE, "Error -- read and reverse read files do not have matching lengths: ");
    if (end1) break;
    u64 m = c1->n - k1; if (s2) m = std::min<u64>(m, c2->n - k2);
    if (m) { rc = emit(c1, k1, c2, k2, m); if (rc != NB_OK) return rc; }
    k1 += m; k2 += m;
  }
  return NB_OK;
}

}  // namespace

extern "C" int nb_write_fastq_tsv(const char* path, const nb_library* lib, const nb_counts* counts) {
  if (!path || !lib || !counts) return fail(NB_ERR_INVALID, "null argument");
  return write_tsv(path, lib, *counts);
}

// host-only: the file drivers' inflate (inflate.hpp) on a buffer, for parity tests against zlib.  raw != 0: one raw deflate
// stream decoded in one piece (how bam.cpp inflates a BGZF block; the output must fit out_cap exactly or loosely);
// raw == 0: concatenated gzip members decoded through windows of `window` bytes behind a 32 KiB history (how fastq.cpp
// reads a .gz file; window 0 = one window).  NB_ERR_PARSE on a damaged stream, NB_ERR_OVERFLOW when out_cap is too small.
extern "C" int nb_inflate(const void* in, uint64_t in_len, int raw, uint64_t window, void* out, uint64_t out_cap, uint64_t* out_len) {
  if ((!in && in_len) || (!out && out_cap) || !out_len) return fail(NB_ERR_INVALID, "null argument");
  const u8* src = (const u8*)in; u8* dst = (u8*)out; *out_len = 0;
  if (raw) {
    std::unique_ptr<nbz::Inflater> inf(new nbz::Inflater()); inf->start(src, src + in_len);
    u8* q = dst; const int r = inf->run(dst, q, dst + out_cap);
    *out_len = (uint64_t)(q - dst);
    if (r == nbz::INF_MORE) return fail(NB_ERR_OVERFLOW, "output buffer too small");
    if (r != nbz::INF_END) return fail(NB_ERR_PARSE, "damaged deflate stream");
    return NB_OK;
  }
  std::unique_ptr<nbz::GzipStream> gz(new nbz::GzipStream()); gz->open(src, in_len);
  if (!window) {
    while (!gz->done()) {
      const ptrdiff_t n = gz->read(dst, dst + *out_len, dst + out_cap);
      if (n < 0) return fail(NB_ERR_PARSE, "damaged gzip stream");
      *out_len += (uint64_t)n;
      if (!gz->done() && n == 0) return fail(NB_ERR_OVERFLOW, "output buffer too small");
    }
    return NB_OK;
  }
  if (window < 300) return fail(NB_ERR_INVALID, "window must hold the longest match");
  const size_t HIST = 32768; std::vector<u8> a(HIST + window), b(HIST + window); u8* cur = a.data(); u8* prev = nullptr; size_t prev_len = 0;
  while (!gz->done()) {
    if (prev) memcpy(cur, prev + prev_len, HIST);
    const ptrdiff_t n = gz->read(prev ? cur : cur + HIST, cur + HIST, cur + HIST + window);
    if (n < 0) return fail(NB_ERR_PARSE, "damaged gzip stream");
    if (*out_len + (uint64_t)n > out_cap) return fail(NB_ERR_OVERFLOW, "output buffer too small");
    memcpy(dst + *out_len, cur + HIST, (size_t)n); *out_len += (uint64_t)n;
    prev = cur; prev_len = (size_t)n; cur = cur == a.data() ? b.data() : a.data();
  }
  return NB_OK;
}

// host-only: a gzip file in memory through the parallel reader (pgunzip.hpp) with `threads` workers and `chunk_bytes` of
// compressed data per chunk — parity tests against zlib
extern "C" int nb_gunzip_parallel(const void* in, uint64_t in_len, int threads, uint64_t chunk_bytes, void* out, uint64_t out_cap, uint64_t* out_len) {
  if ((!in && in_len) || (!out && out_cap) || !out_len) return fail(NB_ERR_INVALID, "null argument");
  *out_len = 0;
  nbz::ParallelGunzip pg; pg.open((const u8*)in, in_len, threads, chunk_bytes);
  while (nbz::PgChunk* c = pg.next()) {
    if (c->status < 0) return fail(NB_ERR_PARSE, "damaged gzip stream");
    if (*out_len + c->text.size() > out_cap) return fail(NB_ERR_OVERFLOW, "output buffer too small");
    memcpy((u8*)out + *out_len, c->text.data(), c->text.size()); *out_len += c->text.size();
    pg.recycle(c);
  }
  return NB_OK;
}

// host-only: the records the feeder hands to the device, one line per record ("SEQ" or "SEQ1\tSEQ2") — parity tests of the
// parallel parser against a sequential one need no GPU.  chunk_bytes 0 = default.
extern "C" int nb_fastq_dump(const char* const* input_files, uint32_t n_inputs, int num_cores, uint64_t chunk_bytes, const char* out_path) {
  if (!input_files || n_inputs < 1 || n_inputs > 2 || !out_path) return fail(NB_ERR_INVALID, "need 1-2 inputs and an output path");
  g_pageable = true;
  struct Unset { ~Unset() { g_pageable = false; } } unset;
  const int T = std::max(1, num_cores / (int)n_inputs);
  std::unique_ptr<SegStream> s1 = open_stream(input_files[0], T, 1u << 16, chunk_bytes ? chunk_bytes : chunk_bytes_default()), s2;
  if (!s1) return fail(NB_ERR_IO, std::string("could not open ") + input_files[0]);
  if (n_inputs > 1) { s2 = open_stream(input_files[1], T, 1u << 16, chunk_bytes ? chunk_bytes : chunk_bytes_default()); if (!s2) return fail(NB_ERR_IO, std::string("could not open ") + input_files[1]); }
  FILE* f = out_path[0] ? fopen(out_path, "wb") : nullptr;   // "" = parse only (timing the feeder)
  if (!f && out_path[0]) return fail(NB_ERR_IO, std::string("Unable to open file ") + out_path);
  int rc = consume(s1.get(), s2.get(),
    [&](Segment* a, u64 ka, Segment* b, u64 kb, u64 m) {
      for (u64 i = 0; f && i < m; i++) {
        fwrite(a->seq.p + a->off()[ka + i], 1, a->off()[ka + i + 1] - a->off()[ka + i], f);
        if (b) { fputc('\t', f); fwrite(b->seq.p + b->off()[kb + i], 1, b->off()[kb + i + 1] - b->off()[kb + i], f); }
        fputc('\n', f);
      }
      return (int)NB_OK;
    },
    [&](SegStream* s, Segment* g) { s->recycle(g); });
  if (f) fclose(f);
  s1->finish(); if (s2) s2->finish();
  return rc;
}

namespace {

double now() { timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec + ts.tv_nsec * 1e-9; }

// One reference library of a FASTQ run: the library, its index (the CUDA builder, or $NB_INDEX_CACHE) and one context per
// device.  nb_process_fastq_devices sets one up per library in turn; nb_process_samples sets up all of them once and runs
// every sample through them.
struct FastqLib {
  nb_library* lib = nullptr; nb_index* ix = nullptr; std::vector<nb_ctx*> ctx;
  double t_lib = 0, t_index = 0, t_ctx = 0;
  ~FastqLib() { for (nb_ctx* c : ctx) nb_ctx_free(c); nb_index_free(ix); nb_library_free(lib); }
  int open(const char* reference_json, int strand_filter, int num_cores, const int* devices, u32 W) {
    const u64 BATCH = 1u << 20;
    ctx.assign(W, nullptr);
    const double t0 = now();
    int rc = nb_library_load_json(reference_json, strand_filter, &lib);
    const double t1 = now();
    if (rc == NB_OK) rc = nb_index_build_cached(lib, nullptr, devices[0], std::max(1, num_cores), &ix);   // K5: the CUDA builder (same artefact as nb_index_build), or $NB_INDEX_CACHE
    const double t2 = now();
    for (u32 d = 0; d < W && rc == NB_OK; d++) { rc = nb_ctx_create(ix, lib, devices[d], nullptr, &ctx[d]); if (rc == NB_OK) rc = nb_ctx_set_option(ctx[d], "max_batch_pairs", BATCH); }
    t_lib = t1 - t0; t_index = t2 - t1; t_ctx = now() - t2;
    return rc;
  }
};

struct FastqJob { u64 pairs = 0, calls = 0; double t_align = 0, t_final = 0; };

// One job of a library: the FASTQs streamed into nb_align_batch (batches dealt to the contexts in turn), the counts
// finalized (merged across the contexts when there are several) and appended to output_path by write_tsv.  The contexts
// are fresh or reset (nb_counts_reset).
int fastq_job(FastqLib& L, const char* const* input_files, u32 n_inputs, int num_cores, const char* output_path, FastqJob& st) {
  const int T = std::max(1, num_cores / (int)n_inputs);
  const u32 W = (u32)L.ctx.size();
  std::vector<nb_ctx*>& ctx = L.ctx;
  const double t3 = now(); u64 n_pairs_fed = 0, n_calls = 0;
  int rc = NB_OK;
  std::unique_ptr<SegStream> s1, s2;
  s1 = open_stream(input_files[0], T, 1u << 19, chunk_bytes_default(file_bytes(input_files[0]), T), 2 * (int)W); if (!s1) rc = fail(NB_ERR_IO, std::string("could not open ") + input_files[0]);
  if (rc == NB_OK && n_inputs > 1) { s2 = open_stream(input_files[1], T, 1u << 19, chunk_bytes_default(file_bytes(input_files[1]), T), 2 * (int)W); if (!s2) rc = fail(NB_ERR_IO, std::string("could not open ") + input_files[1]); }
  if (rc == NB_OK) {
    // A segment goes back to its stream once the copies out of it have run: nb_align_batch blocks on the copies of a staging
    // set before refilling it, so everything a context was given before its last two calls is free again (nimble_b200.h);
    // with W contexts fed in turn that is everything older than 2 W calls.
    struct Held { SegStream* s; Segment* g; u64 call; };
    std::deque<Held> held; u64 calls = 0;
    std::vector<u64> fed(W, 0);
    auto release = [&](bool all) { while (!held.empty() && (all || held.front().call + 2 * W <= calls)) { held.front().s->recycle(held.front().g); held.pop_front(); } };
    rc = consume(s1.get(), s2.get(),
      [&](Segment* a, u64 ka, Segment* b2, u64 kb, u64 m) {
        const u32 d = (u32)(calls % W);
        nb_batch b; memset(&b, 0, sizeof b);
        b.n_pairs = m; b.location = NB_MEM_HOST; b.max_read_len = std::max<u32>(a->maxlen, b2 ? b2->maxlen : 0);
        b.r1 = a->seq.p; b.r1_off = a->off() + ka;
        if (b2) { b.r2 = b2->seq.p; b.r2_off = b2->off() + kb; }
        int r = NB_OK;
        if (W > 1) r = nb_route_set_pair_base(ctx[d], n_pairs_fed - fed[d]);   // this batch's pairs are numbered n_pairs_fed.. in the job; the context adds its own count
        if (r == NB_OK) r = nb_align_batch(ctx[d], &b, nullptr, nullptr);
        calls++; release(false); n_pairs_fed += m; fed[d] += m; n_calls++;
        return r;
      },
      [&](SegStream* s, Segment* g) { held.push_back({s, g, calls}); release(false); });
    for (u32 d = 0; d < W; d++) if (nb_ctx_sync(ctx[d]) != NB_OK && rc == NB_OK) rc = NB_ERR_CUDA;
    release(true);
  }
  if (s1) s1->finish();
  if (s2) s2->finish();
  const double t4 = now();
  std::vector<nb_counts> cts(W);
  if (rc == NB_OK && W == 1) rc = nb_counts_finalize(ctx[0], &cts[0]);
  if (rc == NB_OK && W > 1) {   // collective: every context's call must be in flight at the same time
    std::vector<int> rcs(W, NB_OK); std::vector<std::string> msgs(W); std::vector<std::thread> th;
    for (u32 d = 0; d < W; d++) th.emplace_back([&, d] { rcs[d] = nb_merge_whole_run(ctx[d], &cts[d]); if (rcs[d] != NB_OK) msgs[d] = nb_last_error(); });
    for (auto& x : th) x.join();
    for (u32 d = 0; d < W && rc == NB_OK; d++) if (rcs[d] != NB_OK) rc = fail(rcs[d], msgs[d]);
  }
  if (rc == NB_OK) rc = write_tsv(output_path, L.lib, cts[0]);
  s1.reset(); s2.reset();
  st.pairs = n_pairs_fed; st.calls = n_calls; st.t_align = t4 - t3; st.t_final = now() - t4;
  return rc;
}

}  // namespace

// process::fastq::process with the library loop of src/bin/main.rs:95-133 in front of it, on one or several GPUs.
// Several devices: one context per GPU behind the one feeder (the reference's shape is N-1 consumers behind one producer,
// src/process/bam.rs:183-226); batches go to the contexts in turn with their global pair numbers, k_pair routes every
// read_key record to the GPU that owns the key (peer stores), and nb_merge_whole_run — NCCL inside the library, one host
// thread per context for the collective calls — leaves the whole job's counts on every context.
extern "C" int nb_process_fastq_devices(const char* const* input_files, uint32_t n_inputs, const char* const* reference_json, const char* const* output_paths,
                                        uint32_t n_refs, int strand_filter, int num_cores, const int* devices, uint32_t n_devices) {
  if (!input_files || !reference_json || !output_paths || n_inputs < 1 || n_inputs > 2 || n_refs < 1) return fail(NB_ERR_INVALID, "need 1-2 inputs and >=1 reference/output pair");
  if (!devices || n_devices < 1 || n_devices > 16) return fail(NB_ERR_INVALID, "need 1-16 devices");
  const u32 W = n_devices;
  const bool stats = getenv("NB_FASTQ_STATS") != nullptr;   // phase times on stderr
  for (u32 li = 0; li < n_refs; li++) {
    FastqLib L; FastqJob st;
    int rc = L.open(reference_json[li], strand_filter, num_cores, devices, W);
    std::vector<nb_ctx*>& ctx = L.ctx;
    if (rc == NB_OK && W > 1) {
      // inbox regions hold every record a peer sends during the job: sized from the input (a record of a 100-base read is
      // about 230 bytes of text, gzip packs it about five-fold); NB_ROUTE_RECORDS overrides; a region that fills up fails loudly
      const double t0 = now();
      const char* e = getenv("NB_ROUTE_RECORDS");
      u64 est = file_bytes(input_files[0]) / 100; if (is_gzip(input_files[0])) est *= 6;
      const u64 rpp = e ? strtoull(e, nullptr, 10) : est * 2 / ((u64)W * W) + 65536;
      rc = nb_comm_init_all(ctx.data(), W);
      for (u32 d = 0; d < W && rc == NB_OK; d++) rc = nb_route_create(ctx[d], W, rpp, nullptr);
      for (u32 d = 0; d < W && rc == NB_OK; d++) rc = nb_route_attach_ctx(ctx[d], W, d, ctx.data(), 0);
      L.t_ctx += now() - t0;
    }
    if (rc == NB_OK) rc = fastq_job(L, input_files, n_inputs, num_cores, output_paths[li], st);
    if (stats) fprintf(stderr, "nb_process_fastq: library %.3f s, index (GPU) %.3f s, %u context(s) %.3f s, parse+align %.3f s (%llu pairs in %llu calls, %d parser threads per file: %.1f M reads/s), finalize+tsv %.3f s\n",
                       L.t_lib, L.t_index, W, L.t_ctx, st.t_align, (unsigned long long)st.pairs, (unsigned long long)st.calls, std::max(1, num_cores / (int)n_inputs),
                       (double)st.pairs * n_inputs / std::max(st.t_align, 1e-9) / 1e6, st.t_final);
    if (rc != NB_OK) return rc;
  }
  return NB_OK;
}

extern "C" int nb_process_fastq(const char* const* input_files, uint32_t n_inputs, const char* const* reference_json, const char* const* output_paths,
                                uint32_t n_refs, int strand_filter, int num_cores, int device) {
  return nb_process_fastq_devices(input_files, n_inputs, reference_json, output_paths, n_refs, strand_filter, num_cores, &device, 1);
}

namespace {

bool ends_with(const std::string& s, const char* suf) { const size_t n = strlen(suf); return s.size() >= n && s.compare(s.size() - n, n, suf) == 0; }

// What nb_process_samples checks before any device work, in this order: names, every sample's inputs (count and kind, as
// the CLI dispatches -i on the extension), that every input opens, and that every output directory exists or can be made.
int check_samples(const char* const* names, const char* const* inputs, u32 n_samples, const char* const* output_dirs, u32 n_refs, bool bulk) {
  std::vector<std::string> seen;
  for (u32 s = 0; s < n_samples; s++) {
    const std::string name = names[s] ? names[s] : "";
    auto bad = [&](int code, const std::string& m) { return fail(code, "sample " + name + ": " + m); };
    bool legal = !name.empty() && name != "." && name != "..";
    for (char c : name) legal = legal && ((c >= 'A' && c <= 'Z') || (c >= 'a' && c <= 'z') || (c >= '0' && c <= '9') || c == '.' || c == '_' || c == '-');
    if (!legal) return bad(NB_ERR_INVALID, "a sample name matches [A-Za-z0-9._-]+ and is not '.' or '..'");
    if (std::find(seen.begin(), seen.end(), name) != seen.end()) return bad(NB_ERR_INVALID, "the name is used by an earlier sample");
    seen.push_back(name);
    const char* in[2] = {inputs[2 * s], inputs[2 * s + 1]};
    if (!in[0]) return bad(NB_ERR_INVALID, "no input");
    if (bulk && in[1]) return bad(NB_ERR_INVALID, "a bulk sample has exactly one .bam input");
    for (int k = 0; k < 2 && in[k]; k++) {
      std::string lower = in[k]; std::transform(lower.begin(), lower.end(), lower.begin(), ::tolower);
      const bool fastq = ends_with(in[k], ".fastq.gz") || ends_with(lower, ".fastq"), bam = ends_with(lower, ".bam");
      if (bulk && !bam) return bad(NB_ERR_INVALID, std::string("a bulk sample has exactly one .bam input, not ") + in[k]);
      if (!bulk && bam) return bad(NB_ERR_INVALID, std::string(in[k]) + " is a BAM: BAM samples run in bulk mode (--bulk)");
      if (!bulk && !fastq) return bad(NB_ERR_INVALID, std::string("unsupported file format of ") + in[k] + ": FASTQ samples have .fastq or .fastq.gz inputs");
    }
  }
  for (u32 s = 0; s < n_samples; s++)
    for (int k = 0; k < 2 && inputs[2 * s + k]; k++) {
      const int fd = ::open(inputs[2 * s + k], O_RDONLY);
      if (fd < 0) return fail(NB_ERR_IO, std::string("sample ") + names[s] + ": could not open " + inputs[2 * s + k] + ": " + strerror(errno));
      ::close(fd);
    }
  for (u32 li = 0; li < n_refs; li++) {   // created when missing, its parent must exist (as nb_write_cell_matrix does)
    const char* dir = output_dirs[li];
    if (!dir || !*dir) return fail(NB_ERR_INVALID, "empty output directory");
    if (mkdir(dir, 0777) != 0 && errno != EEXIST) return fail(NB_ERR_IO, std::string("could not create output directory ") + dir + ": " + strerror(errno));
    struct stat st; if (stat(dir, &st) != 0 || !S_ISDIR(st.st_mode)) return fail(NB_ERR_IO, std::string("output directory ") + dir + " is not a directory");
  }
  return NB_OK;
}

// FASTQ samples on one device: every library set up once (FastqLib), then sample by sample, library by library, a job on
// the reset context.
int fastq_samples(const char* const* names, const char* const* inputs, u32 n_samples, const char* const* reference_json, const std::vector<std::string>& outs,
                  u32 n_refs, int strand_filter, int num_cores, int device) {
  const bool stats = getenv("NB_FASTQ_STATS") != nullptr;
  const double t0 = now();
  std::vector<std::unique_ptr<FastqLib>> L(n_refs);
  double t_lib = 0, t_index = 0, t_ctx = 0;
  for (u32 li = 0; li < n_refs; li++) {
    L[li].reset(new FastqLib());
    const int rc = L[li]->open(reference_json[li], strand_filter, num_cores, &device, 1);
    t_lib += L[li]->t_lib; t_index += L[li]->t_index; t_ctx += L[li]->t_ctx;
    if (rc != NB_OK) return rc;
  }
  if (stats) fprintf(stderr, "nb_process_samples: setup %.3f s (CUDA start-up included): %u libraries, library %.3f s, index (GPU) %.3f s, contexts %.3f s\n", now() - t0, n_refs, t_lib, t_index, t_ctx);
  for (u32 s = 0; s < n_samples; s++) {
    const u32 n_inputs = inputs[2 * s + 1] ? 2 : 1;
    FastqJob sum;
    int rc = NB_OK;
    for (u32 li = 0; li < n_refs && rc == NB_OK; li++) {
      FastqJob st;
      rc = nb_counts_reset(L[li]->ctx[0]);
      if (rc == NB_OK) rc = fastq_job(*L[li], inputs + 2 * s, n_inputs, num_cores, outs[(size_t)s * n_refs + li].c_str(), st);
      sum.pairs = st.pairs; sum.t_align += st.t_align; sum.t_final += st.t_final;
    }
    if (stats) fprintf(stderr, "nb_process_samples: sample %s: %llu pairs, parse+align %.3f s, finalize+tsv %.3f s\n", names[s], (unsigned long long)sum.pairs, sum.t_align, sum.t_final);
    if (rc != NB_OK) return sample_failed(names[s], rc);
  }
  return NB_OK;
}

}  // namespace

extern "C" int nb_process_samples(const char* const* names, const char* const* inputs, uint32_t n_samples, const char* const* reference_json,
                                  const char* const* output_dirs, uint32_t n_refs, int strand_filter, int num_cores, int device, int bulk) {
  if (!names || !inputs || !reference_json || !output_dirs || n_samples < 1 || n_refs < 1) return fail(NB_ERR_INVALID, "need >=1 sample and >=1 reference library / output directory pair");
  for (u32 li = 0; li < n_refs; li++) if (!reference_json[li]) return fail(NB_ERR_INVALID, "null reference library");
  int rc = check_samples(names, inputs, n_samples, output_dirs, n_refs, bulk != 0);
  if (rc != NB_OK) return rc;
  std::vector<std::string> outs;   // library li's TSV of sample s: outs[s * n_refs + li] = <output_dirs[li]>/<name>.tsv
  for (u32 s = 0; s < n_samples; s++) for (u32 li = 0; li < n_refs; li++) outs.push_back(std::string(output_dirs[li]) + "/" + names[s] + ".tsv");
  if (bulk) return bulk_samples(names, inputs, n_samples, reference_json, outs, n_refs, strand_filter, num_cores, device);
  return fastq_samples(names, inputs, n_samples, reference_json, outs, n_refs, strand_filter, num_cores, device);
}
