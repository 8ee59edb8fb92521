// synth.cpp — deterministic synthetic workloads of the shapes BASELINE.json names (SURVEY.md §8d): MHC/KIR-like family
// libraries and 2x150 read pairs / 10x-style single-end records.  Test + bench infrastructure only (not product, not
// oracle).  Counter-based RNG: pair i depends only on (seed, i), so any shard can be produced by any rank or thread.
#include <cmath>
#include <cstdint>
#include <cstring>
#include <functional>
#include <thread>
#include <vector>
#include <cstdio>
#include <string>
#include <zlib.h>
typedef uint8_t u8; typedef uint16_t u16; typedef uint32_t u32; typedef uint64_t u64;
namespace {
struct Rng { u64 s; explicit Rng(u64 a, u64 b) { s = a * 0x9E3779B97F4A7C15ULL ^ (b + 0xD1B54A32D192ED03ULL) * 0xBF58476D1CE4E5B9ULL; next(); }
  u64 next() { u64 z = (s += 0x9E3779B97F4A7C15ULL); z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL; z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL; return z ^ (z >> 31); }
  double uni() { return (double)(next() >> 11) * (1.0 / 9007199254740992.0); }
  u64 below(u64 n) { return next() % n; }
  double normal() { double u1 = uni(), u2 = uni(); if (u1 < 1e-300) u1 = 1e-300; return std::sqrt(-2.0 * std::log(u1)) * std::cos(6.283185307179586 * u2); } };
const char B[5] = "ACGT";
inline char comp(char c) { switch (c) { case 'A': return 'T'; case 'C': return 'G'; case 'G': return 'C'; default: return 'A'; } }
void par(int threads, u64 n, const std::function<void(u64, u64)>& f) { if (threads <= 1 || n < 1024) { f(0, n); return; } std::vector<std::thread> th; for (int t = 0; t < threads; t++) th.emplace_back(f, n * (u64)t / threads, n * (u64)(t + 1) / threads); for (auto& x : th) x.join(); }
}

extern "C" {
// Library: n_fam families x n_all alleles; family base length U[900,1300]; allele = base with SNPs at rate U[0.5%,3%].
// Pass seqs=NULL to get the total size; off has n_fam*n_all+1 entries.
u64 synth_library(u64 seed, u32 n_fam, u32 n_all, char* seqs, u64* off) {
  u64 tot = 0; u64 idx = 0;
  for (u32 f = 0; f < n_fam; f++) {
    Rng r(seed, f); u32 len = 900 + (u32)r.below(401);
    std::vector<char> base(len); for (u32 i = 0; i < len; i++) base[i] = B[r.below(4)];
    for (u32 a = 0; a < n_all; a++) {
      Rng ra(seed ^ 0xA11E1EULL, (u64)f * 64 + a); double rate = 0.005 + 0.025 * ra.uni();
      if (off) off[idx] = tot;
      if (seqs) for (u32 i = 0; i < len; i++) { char c = base[i]; if (a > 0 && ra.uni() < rate) { char d; do d = B[ra.below(4)]; while (d == c); c = d; } seqs[tot + i] = c; }
      tot += len; idx++;
    }
  }
  if (off) off[idx] = tot;
  return tot;
}

struct PairPlan { u32 kind; u32 l1, l2; };  // kind: 0 on-target, 1 off-target, 2 low complexity, 3 short
static u64 source_index(u64 seed, u64 i, double dup_rate) {  // PCR duplicates: pair i repeats an earlier pair exactly
  if (i == 0 || dup_rate <= 0) return i;
  Rng r(seed ^ 0xD0BULL, i); if (r.uni() >= dup_rate) return i; return r.below(i);
}
static PairPlan plan(u64 seed, u64 src, u32 read_len) {
  Rng r(seed, src); double u = r.uni(); PairPlan p; p.l1 = p.l2 = read_len;
  if (u < 0.15) p.kind = 1; else if (u < 0.155) p.kind = 2; else if (u < 0.16) { p.kind = 3; p.l1 = 20 + (u32)r.below(20); p.l2 = 20 + (u32)r.below(20); } else p.kind = 0;
  return p;
}
static void fill_pair(u64 seed, u64 src, u32 read_len, const char* lib, const u64* lib_off, u32 n_seqs, char* o1, char* o2, bool paired, double err) {
  Rng r(seed, src); double u = r.uni(); u32 l1 = read_len, l2 = read_len;
  if (u < 0.15) { for (u32 i = 0; i < l1; i++) o1[i] = B[r.below(4)]; if (paired) for (u32 i = 0; i < l2; i++) o2[i] = B[r.below(4)]; return; }
  if (u < 0.155) { u32 per = 1 + (u32)r.below(2); char m[2] = {B[r.below(4)], B[r.below(4)]}; for (u32 i = 0; i < l1; i++) o1[i] = m[i % per]; if (paired) for (u32 i = 0; i < l2; i++) o2[i] = m[(i + 1) % per]; return; }
  if (u < 0.16) { l1 = 20 + (u32)r.below(20); l2 = 20 + (u32)r.below(20); }
  u32 t = (u32)r.below(n_seqs); u64 t0 = lib_off[t]; u32 tlen = (u32)(lib_off[t + 1] - t0);
  int fl = (int)std::lround(350.0 + 50.0 * r.normal()); u32 need = l1 > l2 ? l1 : l2;
  if (fl < (int)need) fl = (int)need; if ((u32)fl > tlen) fl = (int)tlen;
  u32 st = (u32)r.below((u64)tlen - (u32)fl + 1); bool flip = r.uni() < 0.5;
  // fragment base j (0-based, in fragment orientation)
  auto frag = [&](u32 j) -> char { return flip ? comp(lib[t0 + st + (u32)fl - 1 - j]) : lib[t0 + st + j]; };
  for (u32 i = 0; i < l1; i++) o1[i] = frag(i);
  if (paired) for (u32 i = 0; i < l2; i++) o2[i] = comp(frag((u32)fl - 1 - i));
  auto mutate = [&](char* o, u32 l) { for (u32 i = 0; i < l; i++) if (r.uni() < err) { char d; do d = B[r.below(4)]; while (d == o[i]); o[i] = d; } };
  mutate(o1, l1); if (paired) mutate(o2, l2);
}
// offsets for pairs [first, first+n): r1_off / r2_off have n+1 entries each (relative to this shard)
void synth_pair_offsets(u64 seed, u64 first, u64 n, u32 read_len, double dup_rate, u64* r1_off, u64* r2_off, int threads) {
  std::vector<u32> a(n), b(n);
  par(threads, n, [&](u64 x, u64 y) { for (u64 i = x; i < y; i++) { PairPlan p = plan(seed, source_index(seed, first + i, dup_rate), read_len); a[i] = p.l1; b[i] = p.l2; } });
  r1_off[0] = 0; if (r2_off) r2_off[0] = 0;
  for (u64 i = 0; i < n; i++) { r1_off[i + 1] = r1_off[i] + a[i]; if (r2_off) r2_off[i + 1] = r2_off[i] + b[i]; }
}
void synth_pairs(u64 seed, u64 first, u64 n, u32 read_len, double dup_rate, double err, const char* lib, const u64* lib_off, u32 n_seqs,
                 char* r1, const u64* r1_off, char* r2, const u64* r2_off, int threads) {
  par(threads, n, [&](u64 x, u64 y) { char dummy[2048]; for (u64 i = x; i < y; i++) fill_pair(seed, source_index(seed, first + i, dup_rate), read_len, lib, lib_off, n_seqs, r1 + r1_off[i], r2 ? r2 + r2_off[i] : dummy, r2 != nullptr, err); });
}
// 10x-style single-end records (C3): n UMI groups starting at group `first`; reads/UMI ~ 1 + Geometric(mean 4 total);
// each read L bases from one transcript of the group's gene (forward strand = cDNA sense), 10% of reads get a Q2 tail.
// Outputs: group sizes (n), then per read: bases, raw phred, cell id, scope id (group index).
u64 synth_umi_sizes(u64 seed, u64 first, u64 n, u32* sizes) { u64 tot = 0; for (u64 g = 0; g < n; g++) { Rng r(seed ^ 0x5C0FEULL, first + g); u32 k = 1; while (r.uni() < 0.75 && k < 64) k++; sizes[g] = k; tot += k; } return tot; }
void synth_umi_reads(u64 seed, u64 first, u64 n, const u32* sizes, const u64* read_start, u32 L, u32 n_cells, double err, const char* lib, const u64* lib_off, u32 n_seqs,
                     char* bases, u8* qual, u32* cell, u32* scope, int threads) {
  par(threads, n, [&](u64 x, u64 y) {
    for (u64 g = x; g < y; g++) {
      Rng r(seed ^ 0xBA3ULL, first + g); u32 c = (u32)r.below(n_cells); u32 t = (u32)r.below(n_seqs); bool offt = r.uni() < 0.15;
      u64 t0 = lib_off[t]; u32 tlen = (u32)(lib_off[t + 1] - t0);
      for (u32 k = 0; k < sizes[g]; k++) {
        u64 ri = read_start[g] + k; char* o = bases + ri * L; u8* q = qual + ri * L; cell[ri] = c; scope[ri] = (u32)g;
        bool dup = k > 0 && r.uni() < 0.3;   // PCR duplicate of the previous read of this UMI
        if (dup) { memcpy(o, o - L, L); }
        else if (offt) { for (u32 i = 0; i < L; i++) o[i] = B[r.below(4)]; }
        else { u32 st = (u32)r.below((u64)tlen - L + 1); bool flip = r.uni() < 0.1; for (u32 i = 0; i < L; i++) o[i] = flip ? comp(lib[t0 + st + L - 1 - i]) : lib[t0 + st + i];
               for (u32 i = 0; i < L; i++) if (r.uni() < err) { char d; do d = B[r.below(4)]; while (d == o[i]); o[i] = d; } }
        bool tail = r.uni() < 0.1; u32 tail_at = tail ? 30 + (u32)r.below(L - 30) : L;
        // Phred ~ N(36, 3) approximated by a sum of uniforms (Irwin-Hall, 8 x U[0,255]: sd = 209): no transcendental per base
        for (u32 i = 0; i < L; i++) { int v = 2; if (i < tail_at) { u64 z = r.next(); int sum = 0; for (int k = 0; k < 8; k++) sum += (int)((z >> (8 * k)) & 255); v = 36 + (sum - 1020) * 3 / 209; if (v < 2) v = 2; if (v > 41) v = 41; } q[i] = (u8)v; }
      }
    }
  });
}

// 10x-style unaligned BAM of the reads synth_umi_reads made (C3): one record per read, tags CB:Z:<16 nt>-1, UB:Z / UR:Z
// <12 nt> derived from the cell / group ids, CR, NH:i, RE:A; records of one group are contiguous (what UMIReader needs,
// src/parse/sorted_bam_reader.rs:84).  BGZF blocks are deflated on `threads` threads.  Record i is named r<name_id[i]>, or
// r<i> when name_id is null (so a reordering of another file's records can keep their names).  Returns bytes written, 0 on error.
static void nt_of(u64 v, int n, char* o) { for (int i = 0; i < n; i++) { o[i] = B[v & 3]; v >>= 2; } }
u64 synth_write_bam(const char* path, u64 n_reads, u32 L, const char* bases, const u8* qual, const u32* cell, const u32* scope, u32 first_scope, int level, int threads, const u64* name_id) {
  static const u8 code[256] = {0};
  u8 c4[256]; memset(c4, 15, 256); c4[(u8)'A'] = 1; c4[(u8)'C'] = 2; c4[(u8)'G'] = 4; c4[(u8)'T'] = 8; (void)code;
  const char* text = "@HD\tVN:1.6\tSO:unsorted\n@SQ\tSN:chr1\tLN:100000000\n";
  std::string raw; raw.append("BAM\1", 4);
  auto put32 = [&](std::string& d, u32 v) { d.append((const char*)&v, 4); };
  put32(raw, (u32)strlen(text)); raw.append(text); put32(raw, 1); put32(raw, 5); raw.append("chr1\0", 5); put32(raw, 100000000);
  const u64 rec_guess = 36 + 16 + (L + 1) / 2 + L + 80;
  std::vector<std::string> parts(threads > 0 ? threads : 1);
  par((int)parts.size(), n_reads, [&](u64 x, u64 y) {
    size_t pi = 0; for (size_t t = 0; t < parts.size(); t++) if (n_reads * (u64)t / parts.size() == x) pi = t;   // the slice `par` gave this thread
    std::string& d = parts[pi];
    d.reserve((y - x) * rec_guess);
    char name[32], cb[20], ub[13];
    for (u64 i = x; i < y; i++) {
      int ln = snprintf(name, sizeof name, "r%llu", (unsigned long long)(name_id ? name_id[i] : i)) + 1;
      u64 g = (u64)scope[i] + first_scope; nt_of(g * 0x9E3779B97F4A7C15ULL >> 8, 12, ub); ub[12] = 0; nt_of((u64)cell[i] * 0xD1B54A32D192ED03ULL >> 8, 16, cb); cb[16] = '-'; cb[17] = '1'; cb[18] = 0;
      std::string aux; aux.append("CBZ"); aux.append(cb, 19); aux.append("CRZ"); aux.append(cb, 16); aux.push_back(0); aux.append("UBZ"); aux.append(ub, 13); aux.append("URZ"); aux.append(ub, 13);
      aux.append("NHC"); aux.push_back(1); aux.append("REA"); aux.push_back('E');
      u32 body = 32 + ln + (L + 1) / 2 + L + (u32)aux.size();
      put32(d, body); put32(d, (u32)-1); put32(d, (u32)-1);
      u8 hdr8[4] = {(u8)ln, 255, (u8)(4680 & 255), (u8)(4680 >> 8)}; d.append((const char*)hdr8, 4);
      u16 ncig = 0, flag = 4; d.append((const char*)&ncig, 2); d.append((const char*)&flag, 2);
      put32(d, L); put32(d, (u32)-1); put32(d, (u32)-1); put32(d, 0);
      d.append(name, ln);
      const char* sq = bases + i * (u64)L;
      for (u32 k = 0; k < L; k += 2) d.push_back((char)((c4[(u8)sq[k]] << 4) | (k + 1 < L ? c4[(u8)sq[k + 1]] : 0)));
      d.append((const char*)(qual + i * (u64)L), L);
      d.append(aux);
    }
  });
  for (auto& d : parts) { raw.append(d); std::string().swap(d); }
  const u64 BS = 60000; u64 nblk = (raw.size() + BS - 1) / BS;
  std::vector<std::string> comp(nblk + 1);
  auto deflate_block = [&](const char* src, u32 n, std::string& out) {
    z_stream z; memset(&z, 0, sizeof z); deflateInit2(&z, level, Z_DEFLATED, -15, 8, Z_DEFAULT_STRATEGY);
    std::string buf(deflateBound(&z, n) + 64, '\0'); z.next_in = (Bytef*)src; z.avail_in = n; z.next_out = (Bytef*)&buf[0]; z.avail_out = (uInt)buf.size();
    deflate(&z, Z_FINISH); u32 clen = (u32)z.total_out; deflateEnd(&z);
    u8 h[18] = {31, 139, 8, 4, 0, 0, 0, 0, 0, 255, 6, 0, 66, 67, 2, 0, 0, 0}; u16 bsize = (u16)(clen + 25); h[16] = (u8)(bsize & 255); h[17] = (u8)(bsize >> 8);
    out.assign((const char*)h, 18); out.append(buf.data(), clen); u32 crc = (u32)crc32(crc32(0, nullptr, 0), (const Bytef*)src, n); out.append((const char*)&crc, 4); out.append((const char*)&n, 4);
  };
  par(threads, nblk, [&](u64 x, u64 y) { for (u64 b = x; b < y; b++) deflate_block(raw.data() + b * BS, (u32)std::min<u64>(BS, raw.size() - b * BS), comp[b]); });
  deflate_block("", 0, comp[nblk]);
  FILE* f = fopen(path, "wb"); if (!f) return 0;
  u64 tot = 0; for (auto& c : comp) { if (fwrite(c.data(), 1, c.size(), f) != c.size()) { fclose(f); return 0; } tot += c.size(); }
  fclose(f); return tot;
}

// FASTQ (plain, or gzip when the path ends in .gz) of reads r[off[i]..off[i+1]); names @r<i>/<mate>, quality 'I'.
u64 synth_write_fastq(const char* path, u64 n, const char* r, const u64* off, int mate, int level) {
  size_t pl = strlen(path); bool gz = pl > 3 && !strcmp(path + pl - 3, ".gz");
  std::string buf; buf.reserve(1 << 24); u64 tot = 0;
  FILE* f = nullptr; gzFile g = nullptr;
  if (gz) { char mode[8]; snprintf(mode, sizeof mode, "wb%d", level); g = gzopen(path, mode); if (!g) return 0; } else { f = fopen(path, "wb"); if (!f) return 0; }
  auto flush = [&]() { if (gz) gzwrite(g, buf.data(), (unsigned)buf.size()); else fwrite(buf.data(), 1, buf.size(), f); tot += buf.size(); buf.clear(); };
  char name[48];
  for (u64 i = 0; i < n; i++) {
    int ln = snprintf(name, sizeof name, "@r%llu/%d\n", (unsigned long long)i, mate); buf.append(name, ln);
    u64 a = off[i], b = off[i + 1]; buf.append(r + a, b - a); buf.append("\n+\n"); buf.append(b - a, 'I'); buf.push_back('\n');
    if (buf.size() > (1u << 23)) flush();
  }
  flush();
  if (gz) gzclose(g); else fclose(f);
  return tot;
}
// ASCII bases -> NB_SEQ_2BIT stream (base j = bits 2(j&3) of byte j>>2; non-ACGT -> A), threaded: what a producer that holds
// packed reads would hand over; here only so that the bench can ship the same reads packed.  dst needs (n + 3) / 4 bytes.
void synth_encode_2bit(const u8* src, u64 n_bases, u8* dst, int threads) {
  u8 lut[256]; memset(lut, 0, sizeof lut); lut['C'] = lut['c'] = 1; lut['G'] = lut['g'] = 2; lut['T'] = lut['t'] = 3;
  u64 nb4 = (n_bases + 3) / 4;
  par(threads, nb4, [&](u64 a, u64 b) {
    for (u64 i = a; i < b; i++) { u8 v = 0; for (int k = 0; k < 4; k++) { u64 j = 4 * i + k; if (j < n_bases) v |= (u8)(lut[src[j]] << (2 * k)); } dst[i] = v; }
  });
}
}
