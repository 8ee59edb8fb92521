// kernels.cu — hand-written sm_100a kernels (see kernels.cuh for the map to the reference functions).
#include <float.h>
#include <stdlib.h>
#include <string.h>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <algorithm>

#include "kernels.cuh"
#include "khash.h"

namespace nbk {

// FilterReason values used on the device (src/align.rs:32-51 order)
enum { R_SCORE_BELOW = 0, R_MULTI = 1, R_NONZERO_MM = 2, R_NO_MATCH = 3, R_NOT_MATCHING_PAIR = 6, R_SHORT = 8, R_MAX_HITS = 9,
       R_ENTROPY = 10, R_SUCCESS = 11, R_TRIAGE_EMPTY = 13, R_ABOVE_MM = 14, R_SKIPPED = 15, R_NONE = 16 };

__host__ __device__ __forceinline__ u64 mix64(u64 x) {
  x ^= x >> 33; x *= 0xff51afd7ed558ccdULL; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ULL; x ^= x >> 33; return x;
}

// ------------------------------------------------------------------------------------------------ K0 pack
// One thread per (read, 32-base word).  The 32 source bytes are fetched as two or three aligned 16-byte loads and
// realigned in registers (word select + funnel shift); 4 bases are classified per SIMD-in-register compare (non-ACGT
// -> A like DnaString::from_acgt_bytes).  (Nine 4-byte loads per thread ran at 2.4 TB/s; staging the block's span in
// shared memory was slower still — 8-way bank conflicts on the 32-byte-stride reads.)
__device__ __forceinline__ u32 codes4(u32 v) {   // exact for any byte values: the fall-back of codes4_fast
  u32 u = v & 0xDFDFDFDFu;
  u32 c4 = (__vcmpeq4(u, 0x43434343u) & 0x01010101u) | (__vcmpeq4(u, 0x47474747u) & 0x02020202u) | (__vcmpeq4(u, 0x54545454u) & 0x03030303u);
  c4 = (c4 | (c4 >> 6)) & 0x000F000Fu;
  return (c4 | (c4 >> 12)) & 0xFFu;
}
// Four bases in about a dozen instructions.  For the eight valid letters the code is bits (1^2, 2^3) of the byte
// (A 0x41 -> 0, C 0x43 -> 1, G 0x47 -> 2, T 0x54 -> 3, bit 5 = case is never looked at); one multiply gathers the four
// 2-bit codes into the product's top byte (shifts 24/18/12/6: no two partial products overlap, so nothing carries).
// Validity is checked bitwise: bits 7,6,3 must read 0,1,0 and (bit4,bit2,bit1,bit0) must be 0001/0011/0111 (A/C/G) or
// 1100 (T) <=> T(b0,b1,b2) & (b0 ^ b4) with T = b0 ? (!b2 | b1) : (b2 & !b1).  Offending bits accumulate in `bad`; the
// caller redoes the whole word with codes4 when any are set (non-ACGT -> A, rare).
__device__ __forceinline__ u32 codes4_fast(u32 v, u32& bad) {
  u32 s1 = v >> 1, s2 = v >> 2, s4 = v >> 4;
  u32 code = (s1 ^ s2) & 0x03030303u;
  u32 t = (v & (~s2 | s1)) | (~v & s2 & ~s1);
  u32 ok = t & (v ^ s4);
  bad |= (~ok & 0x01010101u) | ((v & 0xC8C8C8C8u) ^ 0x40404040u);
  return code * 0x01041040u;   // top byte = the four codes, first base in the low bits
}
__device__ __forceinline__ u64 rev2(u64 x) {  // reverse the order of the 32 2-bit groups
  x = __brevll(x);
  return ((x >> 1) & 0x5555555555555555ULL) | ((x & 0x5555555555555555ULL) << 1);
}

// one (read, data word) straight from global memory: 2-3 aligned 16-byte loads realigned in registers (round 1's k_pack; kept
// for blocks whose span does not fit the staging buffer — reads longer than the batch declared)
__device__ __forceinline__ void pack_word_direct(const BatchDev& b, u32 idx) {
  // one thread per DATA word; the last data word's thread also writes the read's zero pad word (a thread per pad word
  // idled one lane in W: measured 2.00 -> 2.03 G reads/s on the C2 step)
  const u32 Wd = b.W - 1;
  if (idx >= b.n_reads * Wd) return;
  u32 ri = idx / Wd, w = idx - ri * Wd;                    // 32-bit divide by a small runtime constant
  if (w == Wd - 1) b.pk[(u64)ri * b.W + Wd] = 0;
  u32 side = b.sides == 2 ? (ri & 1) : 0; u64 p = b.sides == 2 ? (ri >> 1) : ri;
  u64 o0 = b.off[side][p]; u32 len = (u32)(b.off[side][p + 1] - o0);
  bool rc = b.flags[side] != nullptr && (b.flags[side][p] & 2);
  if (w == 0) { b.len_full[ri] = len; b.len_trim[ri] = len; }
  u64 word = 0; u32 s = w * 32;
  if (s < len) {
    u32 cnt = min(32u, len - s);
    u64 src = rc ? (o0 + len - s - cnt) : (o0 + s);
    const u8* addr = b.a[side] + src;
    const uint4* al = (const uint4*)((uintptr_t)addr & ~(uintptr_t)15);
    u32 sh = (u32)((uintptr_t)addr & 15), need = sh + cnt;   // bytes wanted from al on: <= 47
    uint4 c0 = __ldg(al), c1 = make_uint4(0x41414141u, 0x41414141u, 0x41414141u, 0x41414141u), c2 = c1;
    if (need > 16) c1 = __ldg(al + 1);
    if (need > 32) c2 = __ldg(al + 2);
    u32 wv[12] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w, c2.x, c2.y, c2.z, c2.w};
    if (sh & 8) {
#pragma unroll
      for (int j = 0; j < 10; j++) wv[j] = wv[j + 2];
      wv[10] = wv[11] = 0;
    }
    if (sh & 4) {
#pragma unroll
      for (int j = 0; j < 11; j++) wv[j] = wv[j + 1];
      wv[11] = 0;
    }
    // bytes behind the read's end (the next read's bases, or the 'A' fill of a chunk that was not needed) are classified
    // too and masked off below; only a non-ACGT byte anywhere in the 32 sends the word through the exact path
    u32 al4[8], pr[8], bad = 0;
#pragma unroll
    for (int j = 0; j < 8; j++) { al4[j] = __funnelshift_r(wv[j], wv[j + 1], (sh & 3) * 8); pr[j] = codes4_fast(al4[j], bad); }
    if (bad == 0) {
      u32 lo = __byte_perm(__byte_perm(pr[0], pr[1], 0x0073), __byte_perm(pr[2], pr[3], 0x0073), 0x5410);
      u32 hi = __byte_perm(__byte_perm(pr[4], pr[5], 0x0073), __byte_perm(pr[6], pr[7], 0x0073), 0x5410);
      word = (u64)lo | ((u64)hi << 32);
    } else {
#pragma unroll
      for (int j = 0; j < 8; j++) word |= (u64)codes4(al4[j]) << (8 * j);
    }
    if (cnt < 32) word &= (1ULL << (2 * cnt)) - 1;
    if (rc) { word = rev2(word) >> (64 - 2 * cnt); word ^= cnt < 32 ? ((1ULL << (2 * cnt)) - 1) : ~0ULL; }
  }
  b.pk[(u64)ri * b.W + w] = word;
}


// K0, staged variant (NB_PACK_BULK=1): ASCII -> 2-bit through shared memory, staged by bulk asynchronous copies.
// A block owns RB consecutive reads (RB * Wd <= 256 word-threads; RB even when paired) = one contiguous ASCII span per side.
//   A  one elected thread arms an mbarrier with the byte count and issues one cp.async.bulk (TMA engine, global -> shared)
//      per side for the 16-byte-aligned cover of the span; the block waits on the barrier's phase
//   B  every thread classifies aligned 16-byte chunks (conflict-free 128-bit shared loads, no realignment: the reads'
//      arbitrary start offsets do not matter yet) into 32 bits of 2-bit codes -> a contiguous 2-bit image of the span
//   C  thread (read, word) cuts its 64-bit window out of that image at the read's base offset (three 32-bit shared loads
//      + two funnel shifts), masks the tail, reverse-complements if asked, writes the word (+ the zero pad word, lengths)
// Round 1's kernel did the realignment on the ASCII bytes in registers (per thread: 2-3 misaligned-by-construction 16-byte
// global loads, a 12-word select network, 8 funnel shifts) and ran at 0.48 of the HBM stream peak, issue-bound at 256
// instructions per 32 bases; classifying aligned data first and realigning the 4x smaller 2-bit image halves that.
constexpr int PACK_T = 256;
constexpr int PACK_RAW = 8192 + 64;     // RB reads x at most 32 * Wd bytes <= 256 * 32, + the alignment slack of two spans
__device__ __forceinline__ u32 smem_u32(const void* p) { return (u32)__cvta_generic_to_shared(p); }
__global__ void __launch_bounds__(PACK_T) k_pack_bulk(BatchDev b, u32 RB, u32 inv_wd) {
  __shared__ __align__(16) u8 s_raw[PACK_RAW];
  __shared__ u32 s_bits[PACK_RAW / 16 + 2];
  __shared__ __align__(8) unsigned long long s_bar;
  __shared__ u64 s_g0[2]; __shared__ u32 s_lead[2], s_bytes[2];
  const u32 tid = threadIdx.x, Wd = b.W - 1, sides = b.sides;
  const u32 r0 = blockIdx.x * RB, rn = min(RB, b.n_reads - r0);          // this block's reads [r0, r0 + rn)
  const u64 p0 = r0 / sides; const u32 pn = (rn + sides - 1) / sides;      // ... = pairs [p0, p0 + pn) on every side
  if (tid < sides) {
    const u64 g0 = b.off[tid][p0], g1 = b.off[tid][p0 + pn];
    const uintptr_t a = (uintptr_t)(b.a[tid] + g0);
    s_g0[tid] = g0; s_lead[tid] = (u32)(a & 15); s_bytes[tid] = (u32)min(((a & 15) + (g1 - g0) + 15) & ~(u64)15, (u64)0x40000000);
  }
  if (tid == 0) {
    if (sides == 1) { s_bytes[1] = 0; s_lead[1] = 0; s_g0[1] = 0; }
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(smem_u32(&s_bar)));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  const u32 bytes0 = s_bytes[0], bytes1 = s_bytes[1], total = bytes0 + bytes1;
  if (total > (u32)PACK_RAW) {   // a read longer than the batch declared: no staging for this block
    if (tid < rn * Wd) pack_word_direct(b, r0 * Wd + tid);
    return;
  }
  // ---- A: bulk copies (global -> shared) signalled through the mbarrier's transaction count
  if (total) {
    if (tid == 0) {
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(&s_bar)), "r"(total) : "memory");
      if (bytes0) asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                               :: "r"(smem_u32(s_raw)), "l"((const u8*)(((uintptr_t)(b.a[0] + s_g0[0])) & ~(uintptr_t)15)), "r"(bytes0), "r"(smem_u32(&s_bar)) : "memory");
      if (bytes1) asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                               :: "r"(smem_u32(s_raw + bytes0)), "l"((const u8*)(((uintptr_t)(b.a[1] + s_g0[1])) & ~(uintptr_t)15)), "r"(bytes1), "r"(smem_u32(&s_bar)) : "memory");
    }
    asm volatile("{\n\t.reg .pred p;\n\tNB_PACK_WAIT:\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%0], 0;\n\t@p bra NB_PACK_DONE;\n\tbra NB_PACK_WAIT;\n\tNB_PACK_DONE:\n\t}" :: "r"(smem_u32(&s_bar)) : "memory");
  }
  // ---- B: 16 aligned bytes -> 16 two-bit codes
  for (u32 ch = tid; ch < total / 16; ch += PACK_T) {
    const uint4 v = ((const uint4*)s_raw)[ch];
    u32 bad = 0;
    const u32 q0 = codes4_fast(v.x, bad), q1 = codes4_fast(v.y, bad), q2 = codes4_fast(v.z, bad), q3 = codes4_fast(v.w, bad);
    u32 w;
    if (bad == 0) w = __byte_perm(__byte_perm(q0, q1, 0x0073), __byte_perm(q2, q3, 0x0073), 0x5410);
    else w = codes4(v.x) | (codes4(v.y) << 8) | (codes4(v.z) << 16) | (codes4(v.w) << 24);   // a non-ACGT byte (-> A): the exact compares
    s_bits[ch] = w;
  }
  if (tid < 2) s_bits[total / 16 + tid] = 0;
  __syncthreads();
  // ---- C: one thread per (read, data word); the last data word's thread also writes the read's zero pad word
  if (tid >= rn * Wd) return;
  const u32 rl = (tid * inv_wd) >> 16, w = tid - rl * Wd, ri = r0 + rl;   // tid / Wd by a 16-bit reciprocal (exact for tid < 256, Wd <= 32)
  const u32 side = sides == 2 ? (ri & 1) : 0; const u64 p = sides == 2 ? (ri >> 1) : ri;
  const u64 o0 = b.off[side][p]; const u32 len = (u32)(b.off[side][p + 1] - o0);
  const bool rc = b.flags[side] != nullptr && (b.flags[side][p] & 2);
  if (w == Wd - 1) b.pk[(u64)ri * b.W + Wd] = 0;
  if (w == 0) { b.len_full[ri] = len; b.len_trim[ri] = len; }
  u64 word = 0; const u32 s = w * 32;
  if (s < len) {
    const u32 cnt = min(32u, len - s);
    // base index of the stretch's first base in the 2-bit image (one base per staged byte)
    const u32 bi = (side ? bytes0 : 0u) + s_lead[side] + (u32)(o0 - s_g0[side]) + (rc ? len - s - cnt : s);
    const u32* q = s_bits + (bi >> 4); const u32 sh = (bi & 15) * 2;
    const u32 x0 = q[0], x1 = q[1], x2 = q[2];
    word = (u64)__funnelshift_r(x0, x1, sh) | ((u64)__funnelshift_r(x1, x2, sh) << 32);
    if (cnt < 32) word &= (1ULL << (2 * cnt)) - 1;
    if (rc) { word = rev2(word) >> (64 - 2 * cnt); word ^= cnt < 32 ? ((1ULL << (2 * cnt)) - 1) : ~0ULL; }
  }
  b.pk[(u64)ri * b.W + w] = word;
}

__global__ void __launch_bounds__(256) k_pack(BatchDev b) { pack_word_direct(b, blockIdx.x * blockDim.x + threadIdx.x); }

// ---- packed input encodings (nb_batch.encoding): the host ships 2 or 4 bits per base instead of 8 — the boundary the
// reference's hot path really has (score::call takes 2-bit DnaStrings, src/score.rs:14-31; BAM stores 4-bit nibbles,
// src/parse/bam.rs:186-189) and a quarter / half of the PCIe bytes.  off[] counts BASES of the packed stream; a read may
// start at any base position.  One thread per (read, data word) as above.
//   NB_SEQ_2BIT  base j of the stream = bits 2(j&3) of byte j>>2 (A0 C1 G2 T3): the device word is a 64-bit window at an
//                arbitrary bit offset (two aligned 8-byte loads + funnel shift)
//   NB_SEQ_BAM4  nibble j = byte j>>1, HIGH nibble first (the BAM layout), codes "=ACMGRSVTWYHKDBN": 1,2,4,8 are A,C,G,T,
//                everything else becomes A exactly as DnaString::from_acgt_bytes treats the letters M, R, ..., N
__device__ __forceinline__ u64 ld_al64(const u8* al, u32 i) { return __ldg((const unsigned long long*)al + i); }
__device__ __forceinline__ u64 swap_nibbles(u64 x) { return ((x & 0x0F0F0F0F0F0F0F0FULL) << 4) | ((x >> 4) & 0x0F0F0F0F0F0F0F0FULL); }
// 16 nibbles (one-hot 1,2,4,8 = A,C,G,T; else A) -> 16 two-bit codes in the low 32 bits
__device__ __forceinline__ u64 nib16_to_codes(u64 x) {
  const u64 M = 0x1111111111111111ULL;
  u64 m1 = x & M, m2 = (x >> 1) & M, m4 = (x >> 2) & M, m8 = (x >> 3) & M;
  u64 sum = m1 + m2 + m4 + m8;                                   // per nibble 0..4, no carry between nibbles
  u64 v = sum & ~(sum >> 1) & ~(sum >> 2) & M;                   // exactly one bit set
  u64 c = ((m2 | m8) & v) | ((((m4 | m8) & v)) << 1);            // code bits at [0,1] of every nibble
  c = (c | (c >> 2)) & 0x0F0F0F0F0F0F0F0FULL; c = (c | (c >> 4)) & 0x00FF00FF00FF00FFULL;
  c = (c | (c >> 8)) & 0x0000FFFF0000FFFFULL; c = (c | (c >> 16)) & 0xFFFFFFFFULL;
  return c;
}
template <int ENC>
__global__ void __launch_bounds__(256) k_pack_enc(BatchDev b) {
  u32 idx = blockIdx.x * blockDim.x + threadIdx.x;
  const u32 Wd = b.W - 1;
  if (idx >= b.n_reads * Wd) return;
  u32 ri = idx / Wd, w = idx - ri * Wd;
  if (w == Wd - 1) b.pk[(u64)ri * b.W + Wd] = 0;
  u32 side = b.sides == 2 ? (ri & 1) : 0; u64 p = b.sides == 2 ? (ri >> 1) : ri;
  u64 o0 = b.off[side][p]; u32 len = b.len[side] ? b.len[side][p] : (u32)(b.off[side][p + 1] - o0);
  bool rc = b.flags[side] != nullptr && (b.flags[side][p] & 2);
  if (w == 0) { b.len_full[ri] = len; b.len_trim[ri] = len; }
  u64 word = 0; u32 s = w * 32;
  if (s < len) {
    u32 cnt = min(32u, len - s);
    u64 src = rc ? (o0 + len - s - cnt) : (o0 + s);        // first base of the 32-base source stretch
    if (ENC == 1) {
      const u8* addr = b.a[side] + (src >> 2);
      const u8* al = (const u8*)((uintptr_t)addr & ~(uintptr_t)7);
      u32 sh = (u32)((uintptr_t)addr & 7) * 8 + (u32)(src & 3) * 2;          // <= 62
      u64 lo = ld_al64(al, 0), hi = (sh + 2 * cnt > 64) ? ld_al64(al, 1) : 0ULL;
      word = sh ? (lo >> sh) | (hi << (64 - sh)) : lo;
    } else {
      const u8* addr = b.a[side] + (src >> 1);
      const u8* al = (const u8*)((uintptr_t)addr & ~(uintptr_t)7);
      u32 sh = (u32)((uintptr_t)addr & 7) * 8 + (u32)(src & 1) * 4;          // <= 60
      u32 need = sh + 4 * cnt;                                                 // bits wanted from al on: <= 188
      u64 w0 = swap_nibbles(ld_al64(al, 0)), w1 = need > 64 ? swap_nibbles(ld_al64(al, 1)) : 0ULL, w2 = need > 128 ? swap_nibbles(ld_al64(al, 2)) : 0ULL;
      u64 lo = sh ? (w0 >> sh) | (w1 << (64 - sh)) : w0, hi = sh ? (w1 >> sh) | (w2 << (64 - sh)) : w1;
      word = nib16_to_codes(lo) | (nib16_to_codes(hi) << 32);
    }
    if (cnt < 32) word &= (1ULL << (2 * cnt)) - 1;
    if (rc) { word = rev2(word) >> (64 - 2 * cnt); word ^= cnt < 32 ? ((1ULL << (2 * cnt)) - 1) : ~0ULL; }
  }
  b.pk[(u64)ri * b.W + w] = word;
}

// ------------------------------------------------------------------------------------------------ K1 trim (maxinfo)
// maxinfo, src/align.rs:873-925: position of the LAST maximum of (double)(ls[i] + sum_{j<=i} qp[q_j]) over the read.
// Thread per read; the quality row is read as aligned 16-byte vectors (it starts at an arbitrary byte), the two tables live in
// shared memory.  The reference compares f64 conversions of the i64 scores (`score as f64 >= max_score`): conversion is
// monotonic, so s >= best (integers) already decides "true", and s < best can only still compare equal after rounding when the
// two are within one ulp of 2^63 — only then are the doubles compared.  `best` is the score of the latest update, so
// (double)best is always the running max_score.
__global__ void __launch_bounds__(256) k_trim(BatchDev b, Tables t) {
  __shared__ i64 s_ls[1024], s_qp[256];
  for (u32 i = threadIdx.x; i < 1024; i += blockDim.x) s_ls[i] = i < 1000 ? t.ls[i] : 0;
  s_qp[threadIdx.x] = t.qp[min(threadIdx.x, 60u)];          // indexed by the raw byte (blockDim.x == 256): qualities above 60 count as 60
  __syncthreads();
  // thread -> read: all sequence-side reads first, then all mates, so that a warp works on one side (its quality rows are
  // neighbours in one buffer) and the warps of a side whose reads are all SKIP_ALIGN dummies retire at once
  const u32 tix = blockIdx.x * blockDim.x + threadIdx.x;
  if (tix >= b.n_reads) return;
  const u32 half = b.n_reads / b.sides, side = b.sides == 2 ? tix / half : 0u; const u64 p = b.sides == 2 ? tix - side * half : tix;
  const u32 ri = (u32)(p * b.sides + side);
  if (b.q[side] == nullptr) return;
  if (b.flags[side] != nullptr && (b.flags[side][p] & 1)) return;       // SKIP_ALIGN: the reference never trims (nor aligns) these, src/align.rs:527-528
  const u64 o0 = b.off[side][p]; const u32 len = b.len_full[ri];        // written by k_pack (packed encodings may carry explicit lengths)
  const bool rc = b.flags[side] != nullptr && (b.flags[side][p] & 2);
  const uintptr_t a0 = (uintptr_t)(b.q[side] + o0), a1 = a0 + len;
  i64 acc = 0, best = INT64_MIN; u32 pos = 0, i = 0;
  auto step = [&](u32 qq) {
    acc += s_qp[qq];
    const i64 sc = s_ls[i] + acc;
    i++;
    bool upd = sc >= best;
    if (!upd && best - sc <= 4096) upd = (double)sc >= (double)best;     // (never taken for scores below 2^53)
    best = upd ? sc : best; pos = upd ? i : pos;
  };
  if (len) {
    const uintptr_t c0 = a0 & ~(uintptr_t)15, c1 = (a1 - 1) & ~(uintptr_t)15;      // first and last aligned chunk
    if (!rc) {
      for (uintptr_t c = c0; c <= c1; c += 16) {
        const uint4 v = __ldg((const uint4*)c); const u32 w[4] = {v.x, v.y, v.z, v.w};
        if (c >= a0 && c + 16 <= a1) {
#pragma unroll
          for (int k = 0; k < 16; k++) step((w[k >> 2] >> (8 * (k & 3))) & 0xFFu);
        } else {
#pragma unroll
          for (int k = 0; k < 16; k++) if (c + k >= a0 && c + k < a1) step((w[k >> 2] >> (8 * (k & 3))) & 0xFFu);
        }
      }
    } else {
      for (uintptr_t c = c1;; c -= 16) {
        const uint4 v = __ldg((const uint4*)c); const u32 w[4] = {v.x, v.y, v.z, v.w};
        if (c >= a0 && c + 16 <= a1) {
#pragma unroll
          for (int k = 15; k >= 0; k--) step((w[k >> 2] >> (8 * (k & 3))) & 0xFFu);
        } else {
#pragma unroll
          for (int k = 15; k >= 0; k--) if (c + k >= a0 && c + k < a1) step((w[k >> 2] >> (8 * (k & 3))) & 0xFFu);
        }
        if (c == c0) break;
      }
    }
  }
  const u32 r = (pos < 1 || best == 0) ? 0u : min(pos, len);      // max_score == 0.0 <=> best == 0
  b.len_trim[ri] = r;
}

// ------------------------------------------------------------------------------------------------ K2 map
struct ReadView {   // one packed read: W words, zero padded; either global (read-major, stride 1) or a shared-memory column (stride 32)
  const u64* p; u32 stride;
  __device__ __forceinline__ u64 word(u32 w) const { return p[(size_t)w * stride]; }
  // 32 bases from base `pos` on.  (Three 32-bit loads + two funnel shifts instead of two 64-bit loads + 64-bit shifts
  // were measured: fewer ALU instructions, one more load per window, +4 % map time — the load/store unit is the scarcer resource.)
  __device__ __forceinline__ u64 win(u32 pos) const {
    u32 w = pos >> 5, sh = (pos & 31) * 2; u64 lo = word(w);
    if (!sh) return lo;
    return (lo >> sh) | (word(w + 1) << (64 - sh));
  }
  __device__ __forceinline__ u32 base(u32 pos) const { return (((const u32*)p)[pos >> 4] >> ((pos & 15) * 2)) & 3u; }
};
__device__ __forceinline__ u64 uwin(const u64* U, u64 pos) {
  u64 w = pos >> 5; u32 sh = (u32)(pos & 31) * 2; u64 lo = __ldg(U + w);
  if (!sh) return lo;
  return (lo >> sh) | (__ldg(U + w + 1) << (64 - sh));
}
// the same from three 32-bit loads and two funnel shifts (fewer ALU instructions, one more load: for the rarer paths)
__device__ __forceinline__ u64 uwin3(const u64* U, u64 pos) {
  const u32* p = (const u32*)U + (pos >> 4); const u32 sh = (u32)(pos & 15) * 2;
  const u32 a = __ldg(p), b = __ldg(p + 1), c = __ldg(p + 2);
  return (u64)__funnelshift_r(a, b, sh) | ((u64)__funnelshift_r(b, c, sh) << 32);
}
__device__ __forceinline__ bool bsearch32(const u32* a, u32 n, u32 x, u32& idx) {
  u32 lo = 0, hi = n;
  while (lo < hi) { u32 mid = (lo + hi) >> 1; if (__ldg(a + mid) < x) lo = mid + 1; else hi = mid; }
  idx = lo; return lo < n && __ldg(a + lo) == x;
}

struct WorkCnt { u32 probes, nodes, bases, colour_elems; };

// Running intersection of the colours of the visited unitigs.  "mask mode": survivors are a 64-bit mask over the
// smallest-so-far colour list (<= 64 ids); "big mode": a private copy in the arena that shrinks in place.
// "universe mode" (the fast path): the colour has a precomputed 64-bit mask over its component of <= 64 sequences
// (col_meta), so the running intersection is one AND; colours of different components are disjoint.
struct EcAcc {
  const u32* col_off; const u32* col_ids; const uint4* col_meta; u32* arena; Counters* ctr; u64 arena_cap;
  bool any, big, uni; u32 last, prev2, base, bsize, alen; u64 boff, aoff, mask;
  __device__ void init(const DevIndex& ix, const Tables& t) { col_off = ix.col_off; col_ids = ix.col_ids; col_meta = ix.col_meta; arena = t.arena; ctr = t.ctr; arena_cap = t.arena_cap; any = big = uni = false; last = prev2 = NONE32; base = NONE32; bsize = alen = 0; boff = aoff = 0; mask = 0; }
  __device__ void reset() { any = big = uni = false; last = prev2 = NONE32; base = NONE32; bsize = alen = 0; boff = aoff = 0; mask = 0; }
  __device__ void add(u32 cid, WorkCnt& wc) { if (cid == last) return; add(cid, __ldg(col_meta + cid), wc); }
  // same, with col_meta[cid] already in hand (it rides in the unitig's walk record)
  __device__ void add(u32 cid, uint4 cm, WorkCnt& wc) {
    if (cid == last) { return; }
    last = cid;
    if (cm.y) {   // bitmap colour
      u64 cmask = (u64)cm.z | ((u64)cm.w << 32);
      wc.colour_elems += (u32)__popcll(cmask);
      if (!any) { any = true; uni = true; boff = cm.x; bsize = cm.y; mask = cmask; }
      else if (uni) mask = (cm.x == (u32)boff) ? (mask & cmask) : 0ULL;
      else if (big) alen = 0;          // list state vs. a colour of another (small) component: disjoint
      else mask = 0;
      return;
    }
    if (uni) { mask = 0; return; }     // small-component state vs. a colour of a big component: disjoint
    u32 o = __ldg(col_off + cid), s = __ldg(col_off + cid + 1) - o;
    wc.colour_elems += s;
    if (!any) {
      any = true; base = cid; boff = o; bsize = s;
      if (s <= 64) mask = s == 64 ? ~0ULL : ((1ULL << s) - 1);
      else {
        big = true; alen = s;
        aoff = atomicAdd(&ctr->arena_top, (unsigned long long)s);
        if (aoff + s > arena_cap) { atomicOr(&ctr->err, (unsigned)E_ARENA); alen = 0; aoff = 0; return; }
        for (u32 i = 0; i < s; i++) arena[aoff + i] = __ldg(col_ids + o + i);
      }
      return;
    }
    if (!big) {
      if (cid == base || cid == prev2) return;     // intersecting with an already-applied colour changes nothing
      prev2 = cid;
      u64 m = mask;
      if (s <= 16) {  // small colours (the common case): one linear merge pass over both sorted lists
        u32 j = 0, cj = s ? __ldg(col_ids + o) : NONE32;
        while (m) {
          int i = __ffsll((long long)m) - 1; m &= m - 1;
          u32 e = __ldg(col_ids + boff + i);
          while (j < s && cj < e) { j++; cj = j < s ? __ldg(col_ids + o + j) : NONE32; }
          if (j >= s || cj != e) mask &= ~(1ULL << i);
        }
      } else {
        while (m) { int i = __ffsll((long long)m) - 1; m &= m - 1; u32 idx; if (!bsearch32(col_ids + o, s, __ldg(col_ids + boff + i), idx)) mask &= ~(1ULL << i); }
      }
    } else if (s <= 64) {
      u64 nm = 0;
      for (u32 i = 0; i < s; i++) { u32 e = __ldg(col_ids + o + i); u32 lo = 0, hi = alen; while (lo < hi) { u32 mid = (lo + hi) >> 1; if (arena[aoff + mid] < e) lo = mid + 1; else hi = mid; } if (lo < alen && arena[aoff + lo] == e) nm |= 1ULL << i; }
      big = false; base = cid; boff = o; bsize = s; mask = nm;
    } else {
      u32 j = 0;
      for (u32 i = 0; i < alen; i++) { u32 e = arena[aoff + i], idx; if (bsearch32(col_ids + o, s, e, idx)) arena[aoff + j++] = e; }
      alen = j;
    }
  }
  __device__ u32 ec_len() const { return !any ? 0u : (big ? alen : (u32)__popcll(mask)); }
};

// backward compare: unitig positions uhi-i vs read positions rhi-i, i in [0, m)
__device__ __forceinline__ void cmp_bwd(const u64* U, u64 uhi, const ReadView& rd, u32 rhi, u32 m, u32 allowed, u32& mb, u32& snp, bool& brk) {
  mb = 0; snp = 0; brk = false;
  while (mb < m) {
    u32 c = min(32u, m - mb);
    u64 x = uwin(U, uhi - mb - (c - 1)) ^ rd.win(rhi - mb - (c - 1));
    u64 d = (x | (x >> 1)) & 0x5555555555555555ULL;
    if (c < 32) d &= (1ULL << (2 * c)) - 1;
    u32 cnt = (u32)__popcll(d);
    if (snp + cnt <= allowed) { snp += cnt; mb += c; continue; }
    u32 need = allowed - snp;
    for (u32 i = 0; i < need; i++) d &= ~(1ULL << (63 - __clzll((long long)d)));
    u32 j = (u32)(63 - __clzll((long long)d)) >> 1;
    mb += c - 1 - j;
    snp = allowed + 1; brk = true; break;
  }
}

#include "kmap.cuh"

// ------------------------------------------------------------------------------------------------ K3 pair
struct EcView { const u32* list; u64 mask; u32 lsize; u32 n; bool big; bool uni; u32 ref32; };
__device__ __forceinline__ EcView make_view(const ReadRes& r, const DevIndex& ix, const Tables& t) {
  EcView e; e.n = 0; e.list = nullptr; e.mask = 0; e.lsize = 0; e.big = false; e.uni = false; e.ref32 = 0;
  if (!((r.hdr >> 8) & 1)) return e;   // only passing alignments contribute an equivalence class (src/align.rs:561-572)
  e.big = (r.hdr >> 9) & 1; e.uni = (r.hdr >> 11) & 1; e.n = r.ec_len; e.lsize = r.bsize; e.mask = r.mask; e.ref32 = (u32)r.ref;
  e.list = e.big ? (t.arena + r.ref) : (ix.col_ids + r.ref);
  return e;
}
__device__ __forceinline__ bool ec_has(const EcView& e, const DevLib& L, u32 x) {
  if (e.n == 0 || x == NONE32) return false;
  if (e.uni) return L.row_uoff[x] == e.ref32 && ((e.mask >> L.row_upos[x]) & 1);   // bitmap over a component list: two loads, no search
  u32 lo = 0, hi = e.lsize;
  while (lo < hi) { u32 mid = (lo + hi) >> 1; if (e.list[mid] < x) lo = mid + 1; else hi = mid; }
  if (lo >= e.lsize || e.list[lo] != x) return false;
  return e.big ? true : ((e.mask >> lo) & 1);
}
template <class F> __device__ __forceinline__ void ec_each(const EcView& e, F f) {
  if (e.n == 0) return;
  if (e.big) { for (u32 i = 0; i < e.lsize; i++) if (!f(e.list[i])) return; }
  else { u64 m = e.mask; while (m) { int i = __ffsll((long long)m) - 1; m &= m - 1; if (!f(e.list[i])) return; } }
}
// membership after filter_read_calls_with_orientation (src/align.rs:144-171): a feature called in both orientations
// by one mate is dropped from that mate's list
__device__ __forceinline__ bool in_side(const EcView& e, const DevLib& L, u32 row) {
  if (row == NONE32 || !ec_has(e, L, row)) return false;
  return !ec_has(e, L, L.row_other[row]);
}

struct GroupList {
  u32 g[GL_MAX]; u32 n; u32 limit; bool dedup; bool sat;
  __device__ void add(u32 x) {
    if (sat) return;
    u32 i = 0;
    while (i < n && g[i] < x) i++;
    if (dedup && i < n && g[i] == x) return;
    if (n >= limit) { sat = true; return; }
    for (u32 j = n; j > i; j--) g[j] = g[j - 1];
    g[i] = x; n++;
  }
};

__device__ __forceinline__ void cas128(ulonglong2* addr, u64 n0, u64 n1, u64& o0, u64& o1) {
  asm volatile("{\n\t.reg .b128 c, n, o;\n\tmov.b128 c, {%2, %3};\n\tmov.b128 n, {%4, %5};\n\tatom.global.cas.b128 o, [%6], c, n;\n\tmov.b128 {%0, %1}, o;\n\t}\n"
               : "=l"(o0), "=l"(o1) : "l"(0ULL), "l"(0ULL), "l"(n0), "l"(n1), "l"(addr) : "memory");
}
// insert-or-find a 128-bit key; returns slot or ~0 when the table is full; fresh = this call created the entry
__device__ __forceinline__ u64 key_insert(const Tables& t, u64 k0, u64 k1, bool& fresh) {
  u64 h = (k0 ^ (k1 >> 17)) & t.key_mask;
  fresh = false;
  for (u64 probes = 0; probes <= t.key_mask; probes++) {
    // the 128-bit CAS is also the (atomic) read: a plain 16-byte load could be torn against a concurrent insert
    u64 o0, o1; cas128(t.key + h, k0, k1, o0, o1);
    if (o0 == 0 && o1 == 0) { fresh = true; return h; }
    if (o0 == k0 && o1 == k1) return h;
    h = (h + 1) & t.key_mask;
  }
  return ~0ULL;
}
__device__ __forceinline__ u32 callset_intern(const Tables& t, const u32* g, u32 n) {
  u64 tag = 0x9E3779B97F4A7C15ULL ^ n;
  for (u32 i = 0; i < n; i++) tag = mix64(tag ^ g[i]) + 0x632BE59BD9B4E019ULL;
  tag = mix64(tag) | 1ULL;
  u32 h = (u32)(tag >> 24) & t.cs_mask;
  for (u32 probes = 0; probes <= t.cs_mask; probes++) {
    unsigned long long old = atomicCAS((unsigned long long*)(t.cs_tag + h), 0ULL, (unsigned long long)tag);
    if (old == 0ULL) {
      t.cs_len[h] = n;
      for (u32 i = 0; i < n; i++) t.cs_items[(u64)h * t.gcap + i] = g[i];
      atomicAdd(&t.ctr->n_callsets, 1ULL);
      return h;
    }
    if (old == tag) return h;
    h = (h + 1) & t.cs_mask;
  }
  return NONE32;
}

// owning rank of a read_key in a multi-GPU whole-run scope: a 16-bit slice of key_lo mod world
__device__ __forceinline__ u32 key_owner(u64 k0, u32 world) { return (u32)((k0 >> 40) & 0xFFFFu) % world; }

// one pair; returns true when the pair created a new entry of the whole-run key table (k_pair counts those per block)
__device__ __forceinline__ bool pair_one(const BatchDev& b, const DevIndex& ix, const DevLib& L, const DevCfg& cfg, const Tables& t, const Route& rt, u64 p) {
  bool paired = b.sides == 2;
  u32 ri1 = (u32)(p * b.sides);
  ReadRes r1 = b.rres[ri1], r2;
  if (paired) r2 = b.rres[ri1 + 1]; else { r2.hdr = R_SUCCESS; r2.ec_len = 0; r2.bsize = 0; r2.ref = 0; r2.mask = 0; r2.score = r2.mm = 0; }
  EcView e1 = make_view(r1, ix, t), e2 = make_view(r2, ix, t);
  PairRes out; out.callset = NONE32; out.triage = R_NONE; out.insertable = 0; out.fr1 = (u8)(r1.hdr & 0xFF); out.fr2 = (u8)(r2.hdr & 0xFF);
  // ---- read_key = R1 string + R2 string (untrimmed, after revcomp), src/align.rs:576-579 — hashed to 128 bits over
  // the concatenated 2-bit stream so that, like the reference's string concatenation, only the joined bases matter.
  u32 n1 = b.len_full[ri1], n2 = paired ? b.len_full[ri1 + 1] : 0, tot = n1 + n2;
  ReadView rd1{b.pk + (u64)ri1 * b.W, 1}, rd2{b.pk + (u64)(ri1 + 1) * b.W, 1};
  u64 h0 = 0x243F6A8885A308D3ULL, h1 = 0x13198A2E03707344ULL;
  for (u32 s = 0; s < tot; s += 32) {
    u64 w;
    if (s + 32 <= n1) w = rd1.win(s);
    else if (s >= n1) w = rd2.win(s - n1);
    else { u32 c1 = n1 - s; w = rd1.win(s) & ((1ULL << (2 * c1)) - 1); if (n2) w |= rd2.win(0) << (2 * c1); }
    h0 = (h0 ^ w) * 0x9E3779B97F4A7C15ULL; h0 ^= h0 >> 29;          // two multiply-xorshift lanes, avalanche at the end
    h1 = (h1 + w) * 0xC2B2AE3D27D4EB4FULL; h1 ^= h1 >> 31;
  }
  u32 scope = b.scope ? b.scope[p] : 0u;
  h0 = mix64(h0 ^ tot ^ ((u64)scope << 32)); h1 = mix64(h1 + (u64)tot * 0xD6E8FEB86659FD93ULL + scope);
  if ((h0 | h1) == 0) h0 = 1;
  out.key_lo = h0; out.key_hi = h1;
  // ---- require_valid_pair, src/align.rs:582-588 + filter_pair 732-760
  if (paired && cfg.require_valid_pair) {
    bool bad = e1.n == 0 || e2.n == 0 || e1.n != e2.n;
    if (!bad) ec_each(e1, [&](u32 x) { if (!ec_has(e2, L, x)) { bad = true; return false; } return true; });
    if (bad) { out.fr1 = out.fr2 = R_NOT_MATCHING_PAIR; e1.n = e2.n = 0; }
  }
  u32 cs = CS_NONE;
  const bool scoped = b.scope != nullptr;
  if (e1.n != 0 || e2.n != 0) {   // else failed alignment: bookkeeping only (src/align.rs:686-725)
  out.insertable = 1;
  // ---- filter_and_coerce_sequence_call_orientations, src/align.rs:178-252, on integer ids
  int chem = cfg.strand_filter;
  auto in_ua = [&](u32 row) { return in_side(e1, L, row) && !in_side(e2, L, row); };
  auto qual_a = [&](u32 row) -> bool {   // row comes from e1
    if (!in_side(e1, L, row)) return false;
    if (chem == 3) return true;
    if (in_side(e2, L, row)) return false;
    if (chem == 0) return true;
    bool rev = L.row_rev[row];
    return chem == 1 ? !rev : rev;
  };
  auto qual_b = [&](u32 row) -> bool {   // row comes from e2
    if (!in_side(e2, L, row)) return false;
    if (chem == 3) return true;
    if (in_side(e1, L, row)) return false;
    if (chem == 0) return true;
    u32 f = L.row_fid[row]; bool rev = L.row_rev[row];
    u32 rf = L.row_of[2 * (u64)f], rr_ = L.row_of[2 * (u64)f + 1];
    if (chem == 1) { if (in_ua(rr_)) return false; return rev || in_ua(rf); }        // filter_five_prime 311-342
    if (in_ua(rf)) return false; return !rev || in_ua(rr_);                           // filter_three_prime 344-375
  };
  auto feat_in_b = [&](u32 f) -> bool {
    u32 rf = L.row_of[2 * (u64)f], rr_ = L.row_of[2 * (u64)f + 1];
    return (ec_has(e2, L, rf) && qual_b(rf)) || (ec_has(e2, L, rr_) && qual_b(rr_));
  };
  u32 T = max(cfg.discard_multi_hits, cfg.max_hits);
  GroupList gl; gl.n = 0; gl.limit = T + 1; gl.dedup = !cfg.no_dedup; gl.sat = false;
  bool feat_missing = false;
  auto add_feat = [&](u32 f) { u32 g = L.feat_group[f]; if (g == NONE32) { feat_missing = true; return; } gl.add(g); };
  auto add_row = [&](u32 row) { u32 g = L.row_group[row]; if (g == NONE32) { feat_missing = true; return; } gl.add(g); };   // = add_feat(row_fid[row])
  bool use_intersection = false;
  if (cfg.intersect_level != 0) {   // get_intersecting_reads 763-785 (array_tool Intersect: unique(A) kept when in B)
    ec_each(e1, [&](u32 row) { if (qual_a(row) && feat_in_b(L.row_fid[row])) { use_intersection = true; return false; } return true; });
  }
  if (use_intersection) {
    ec_each(e1, [&](u32 row) { if (qual_a(row) && feat_in_b(L.row_fid[row])) add_feat(L.row_fid[row]); return !gl.sat; });
  } else if (cfg.intersect_level != 2) {   // get_all_calls 788-796 (concat; duplicates collapse in the roll-up unless nt_sequence)
    ec_each(e1, [&](u32 row) { if (qual_a(row)) add_row(row); return !gl.sat; });
    ec_each(e2, [&](u32 row) { if (qual_b(row)) add_row(row); return !gl.sat; });
  }
  if (feat_missing) atomicOr(&t.ctr->err, (unsigned)E_FEATURE);
  // roll-up + discard_multi_hits + max hits, src/align.rs:229-242, 842-848
  u32 cnt = gl.sat ? T + 1 : gl.n;
  if (cfg.discard_multi_hits > 0 && cnt > cfg.discard_multi_hits) cnt = 0;
  u32 triage = R_NONE;
  if (cnt > cfg.max_hits) triage = R_MAX_HITS;
  else if (cnt == 0) triage = R_TRIAGE_EMPTY;
  if (triage == R_NONE) {
    u32 slot = callset_intern(t, gl.g, gl.n);
    if (slot == NONE32 || slot >= CS_NONE) atomicOr(&t.ctr->err, (unsigned)E_CS_FULL); else { cs = slot; out.callset = slot; }
  }
  out.triage = (u8)triage;
  }
  // ---- score_map.insert(read_key, ...): later duplicates overwrite (src/align.rs:685) => keep the highest order.
  // Scoped (BAM) batches also register non-insertable pairs: filter_reasons is keyed by read_key for every pair
  // (src/align.rs:586-600) and k_resolve reports per-key outcomes.
  // Whole-run scope sharded over ranks (rt.world > 1): orders are global pair indices and a key this rank does not own
  // goes to its owner's inbox over NVLink — one local atomicAdd per (warp, owner) reserves slots in this rank's region
  // of that inbox, then each lane stores its 32-byte record (peer stores: the only traffic on the link); the owner
  // merges its inbox when the job ends (nb_route_import).
  const bool routed = rt.world > 1 && !scoped;
  u32 owner = routed ? key_owner(h0, rt.world) : 0u;
  bool send = routed && out.insertable && owner != rt.rank;
  bool fresh = false;
  if ((out.insertable || scoped) && !send) {
    u64 slot = key_insert(t, h0, h1, fresh);
    if (slot == ~0ULL) atomicOr(&t.ctr->err, (unsigned)E_KEY_FULL);
    else {
      unsigned long long ord1 = (routed ? rt.pair_base : 0ULL) + b.order_base + p + 1;
      if (out.insertable) atomicMax(t.kval + slot, (ord1 << 24) | cs);
      if (scoped) { atomicMax(t.klast + slot, ord1); b.pslot[p] = slot; }
    }
  }
  if (routed) {
    unsigned sm = __ballot_sync(__activemask(), send);
    if (send) {
      unsigned peers = __match_any_sync(sm, owner); u32 lane = threadIdx.x & 31; int leader = __ffs(peers) - 1;
      unsigned long long base = 0;
      if ((int)lane == leader) base = atomicAdd(rt.cursor + owner, (unsigned long long)__popc(peers));
      base = __shfl_sync(peers, base, leader);
      u64 at = base + __popc(peers & ((1u << lane) - 1));
      if (at >= rt.cap) atomicOr(&t.ctr->err, (unsigned)E_INBOX_FULL);
      else {
        KeyRec r; r.k0 = h0; r.k1 = h1; r.order = rt.pair_base + b.order_base + p; r.tag = cs == CS_NONE ? 0ULL : t.cs_tag[cs];
        uint4* dst = (uint4*)(rt.inbox[owner] + at);
        dst[0] = make_uint4((u32)r.k0, (u32)(r.k0 >> 32), (u32)r.k1, (u32)(r.k1 >> 32));
        dst[1] = make_uint4((u32)r.order, (u32)(r.order >> 32), (u32)r.tag, (u32)(r.tag >> 32));
      }
    }
  }
  b.pres[p] = out;
  return fresh && !scoped;
}
// Counters::n_live += the block's new keys: one shared-memory atomic per warp, one global atomic per block.  (A per-warp
// global atomic issued from inside the divergent pair logic — several convergence groups per warp — cost 1.5 ms per 10 M pairs
// on that one address.)
#ifndef NB_PAIR_MINB
#define NB_PAIR_MINB 1
#endif
__global__ void __launch_bounds__(128, NB_PAIR_MINB) k_pair(BatchDev b, DevIndex ix, DevLib L, DevCfg cfg, Tables t, Route rt) {
  __shared__ u32 s_new;
  if (threadIdx.x == 0) s_new = 0;
  __syncthreads();
  const u64 p = blockIdx.x * (u64)blockDim.x + threadIdx.x;
  bool fresh = false;
  if (p < b.n_pairs) fresh = pair_one(b, ix, L, cfg, t, rt, p);
  __syncwarp();
  const unsigned fm = __ballot_sync(0xFFFFFFFFu, fresh);
  if ((threadIdx.x & 31) == 0 && fm) atomicAdd(&s_new, (u32)__popc(fm));
  __syncthreads();
  if (threadIdx.x == 0 && s_new) atomicAdd(&t.ctr->n_live, (unsigned long long)s_new);
}

// Per-pair records as the reference reports them (per read_key): filter reasons of the LAST pair carrying the key
// (filter_reasons.insert overwrites, src/align.rs:586-600), triage / callset of the last pair that reached score_map
// (src/align.rs:685, 440-449).  Scoped batches only; all pairs of a key live in the same batch.
__global__ void __launch_bounds__(256) k_resolve(BatchDev b, Tables t) {
  u64 p = blockIdx.x * (u64)blockDim.x + threadIdx.x;
  if (p >= b.n_pairs) return;
  PairRes out = b.pres[p];
  u64 slot = b.pslot[p];
  u64 last = t.klast[slot], v = t.kval[slot];
  if (last) { const PairRes& l = b.pres[last - 1 - b.order_base]; out.fr1 = l.fr1; out.fr2 = l.fr2; }
  if (v >> 24) { const PairRes& r = b.pres[(v >> 24) - 1 - b.order_base]; out.triage = r.triage; out.callset = r.callset; }
  else { out.triage = R_NONE; out.callset = NONE32; }
  b.pres2[p] = out;
}

// ------------------------------------------------------------------------------------------------ K4 fold
// One vote per unique read_key (src/align.rs:440-449): results[callset] += 1 (245-251), keyed here by (cell, callset).
// Each block walks a contiguous range of key slots.  In the whole-run scope the votes land on a few thousand callsets,
// so a block first counts them in a shared-memory table and adds each (callset, count) to the global table once
// (7 M same-address global atomics per 10 M-pair job otherwise: the kernel was atomics-bound at 0.8 TB/s).  Scoped
// batches have about as many (cell, callset) rows as votes and go to the global table directly.
// returns 1 when the call created the (cell, callset) row: the caller adds those up and bumps Counters::n_agg once per
// block (a scoped batch creates about one row per two votes — that many atomics on ONE address were most of k_fold's time)
__device__ __forceinline__ u32 agg_add(const Tables& t, unsigned long long ak, unsigned long long n) {
  u64 h = mix64(ak) & t.agg_mask;
  for (u64 probes = 0; probes <= t.agg_mask; probes++) {
    unsigned long long old = atomicCAS(t.agg_key + h, 0ULL, ak);
    if (old == 0ULL || old == ak) { atomicAdd(t.agg_cnt + h, n); return old == 0ULL ? 1u : 0u; }
    h = (h + 1) & t.agg_mask;
  }
  atomicOr(&t.ctr->err, (unsigned)E_AGG_FULL);
  return 0u;
}
constexpr int FOLD_S = 2048;   // shared-memory vote table entries per block (24 KB)
__global__ void __launch_bounds__(256) k_fold(Tables t, const u32* cell_of_pair, u64 order_base, u64 slots_per_block) {
  __shared__ unsigned long long s_key[FOLD_S];
  __shared__ u32 s_cnt[FOLD_S];
  __shared__ u32 s_occ, s_new;
  const bool local = cell_of_pair == nullptr;
  if (local) for (u32 i = threadIdx.x; i < FOLD_S; i += blockDim.x) { s_key[i] = 0ULL; s_cnt[i] = 0; }
  if (threadIdx.x == 0) { s_occ = 0; s_new = 0; }
  __syncthreads();
  u64 lo = blockIdx.x * slots_per_block, hi = min(lo + slots_per_block, t.key_mask + 1);
  u32 nocc = 0, nnew = 0;
  for (u64 idx = lo + threadIdx.x; idx < hi; idx += blockDim.x) {
    ulonglong2 k = t.key[idx];
    if (k.x == 0 && k.y == 0) continue;
    nocc++;                                          // unique read_keys
    u64 v = t.kval[idx]; u32 cs = (u32)(v & 0xFFFFFFu);
    if ((v >> 24) == 0 || cs == CS_NONE) continue;   // key never reached score_map (scoped batches register every key) / triaged
    u32 cell = cell_of_pair ? cell_of_pair[(v >> 24) - 1 - order_base] : 0u;
    unsigned long long ak = (((unsigned long long)cell << 24) | cs) + 1ULL;
    bool done = false;
    if (local) {
      u32 h = (u32)mix64(ak) & (FOLD_S - 1);
      for (int probes = 0; probes < 8 && !done; probes++) {
        unsigned long long old = atomicCAS(s_key + h, 0ULL, ak);
        if (old == 0ULL || old == ak) { atomicAdd(s_cnt + h, 1u); done = true; }
        h = (h + 1) & (FOLD_S - 1);
      }
    }
    if (!done) nnew += agg_add(t, ak, 1ULL);
  }
  for (int o = 16; o; o >>= 1) nocc += __shfl_xor_sync(0xFFFFFFFFu, nocc, o);
  if ((threadIdx.x & 31) == 0 && nocc) atomicAdd(&s_occ, nocc);
  __syncthreads();
  if (threadIdx.x == 0 && s_occ) atomicAdd(&t.ctr->n_keys, (unsigned long long)s_occ);
  if (local) for (u32 i = threadIdx.x; i < FOLD_S; i += blockDim.x) if (s_key[i]) nnew += agg_add(t, s_key[i], (unsigned long long)s_cnt[i]);
  for (int o = 16; o; o >>= 1) nnew += __shfl_xor_sync(0xFFFFFFFFu, nnew, o);
  if ((threadIdx.x & 31) == 0 && nnew) atomicAdd(&s_new, nnew);
  __syncthreads();
  if (threadIdx.x == 0 && s_new) atomicAdd(&t.ctr->n_agg, (unsigned long long)s_new);
}

// ------------------------------------------------------------------------------------------------ exports
struct ReadOut { u8 reason, pass; u16 score, mm, trimmed_len; u32 ec_len, ec_hash; };  // == nb_read_result
__global__ void __launch_bounds__(256) k_export_reads(BatchDev b, DevIndex ix, Tables t, ReadOut* out) {
  u32 ri = blockIdx.x * blockDim.x + threadIdx.x;
  if (ri >= b.n_reads) return;
  ReadRes r = b.rres[ri];
  ReadOut o; o.reason = (u8)(r.hdr & 0xFF); o.pass = (u8)((r.hdr >> 8) & 1); o.score = r.score; o.mm = r.mm; o.trimmed_len = (u16)b.len_trim[ri]; o.ec_len = r.ec_len;
  u32 h = 2166136261u;
  if (r.ec_len) {
    EcView e; e.big = (r.hdr >> 9) & 1; e.n = r.ec_len; e.lsize = r.bsize; e.mask = r.mask; e.list = e.big ? (t.arena + r.ref) : (ix.col_ids + r.ref);
    ec_each(e, [&](u32 x) { h = (h ^ x) * 16777619u; return true; });
  }
  o.ec_hash = h;
  out[ri] = o;
}

__global__ void __launch_bounds__(256) k_rehash_keys(Tables o, Tables n) {
  u64 idx = blockIdx.x * (u64)blockDim.x + threadIdx.x;
  if (idx > o.key_mask) return;
  ulonglong2 k = o.key[idx];
  if (k.x == 0 && k.y == 0) return;
  bool fresh;
  u64 slot = key_insert(n, k.x, k.y, fresh);
  if (slot == ~0ULL) { atomicOr(&n.ctr->err, (unsigned)E_KEY_FULL); return; }
  n.kval[slot] = o.kval[idx];
}

__global__ void __launch_bounds__(256) k_keys_export(Tables t, KeyRec* rec, unsigned long long* n_out, u64 cap, u64 order_base) {
  u64 idx = blockIdx.x * (u64)blockDim.x + threadIdx.x;
  if (idx > t.key_mask) return;
  ulonglong2 k = t.key[idx];
  if (k.x == 0 && k.y == 0) return;
  u64 v = t.kval[idx]; u32 cs = (u32)(v & 0xFFFFFFu);
  unsigned long long at = atomicAdd(n_out, 1ULL);
  if (at >= cap) return;
  KeyRec r; r.k0 = k.x; r.k1 = k.y; r.order = (v >> 24) - 1 + order_base; r.tag = ((v >> 24) == 0 || cs == CS_NONE) ? 0ULL : t.cs_tag[cs];   // as k_keys_scatter
  rec[at] = r;
}
// import records from other ranks: the tag must already be present in this rank's dictionary (the host merges
// dictionaries first); records whose tag is 0 carry "no callset" and only shadow older duplicates.
__global__ void __launch_bounds__(256) k_keys_import(Tables t, const KeyRec* rec, u64 n);

// ---- multi-GPU exchange helpers: key records grouped by owning rank (owner = a 16-bit slice of key_lo mod world), so the
// host can hand them to an all-to-all without sorting; warp-aggregated cursors (a handful of hot counters otherwise)
__global__ void __launch_bounds__(256) k_keys_count_owner(Tables t, u32 world, unsigned long long* counts) {
  u64 idx = blockIdx.x * (u64)blockDim.x + threadIdx.x;
  bool occ = false; u32 owner = 0;
  if (idx <= t.key_mask) { ulonglong2 k = t.key[idx]; occ = !(k.x == 0 && k.y == 0); owner = key_owner(k.x, world); }
  unsigned act = __ballot_sync(0xFFFFFFFFu, occ);
  if (!occ) return;
  unsigned peers = __match_any_sync(act, owner);
  if ((threadIdx.x & 31) == (unsigned)(__ffs(peers) - 1)) atomicAdd(counts + owner, (unsigned long long)__popc(peers));
}
__global__ void __launch_bounds__(256) k_keys_scatter(Tables t, KeyRec* rec, unsigned long long* cursors, u64 order_base, u32 world) {
  u64 idx = blockIdx.x * (u64)blockDim.x + threadIdx.x;
  bool occ = false; u32 owner = 0; ulonglong2 k = make_ulonglong2(0, 0);
  if (idx <= t.key_mask) { k = t.key[idx]; occ = !(k.x == 0 && k.y == 0); owner = key_owner(k.x, world); }
  unsigned act = __ballot_sync(0xFFFFFFFFu, occ);
  if (!occ) return;
  unsigned peers = __match_any_sync(act, owner); u32 lane = threadIdx.x & 31; int leader = __ffs(peers) - 1;
  unsigned long long base = 0;
  if ((int)lane == leader) base = atomicAdd(cursors + owner, (unsigned long long)__popc(peers));
  base = __shfl_sync(peers, base, leader);
  u64 at = base + __popc(peers & ((1u << lane) - 1));
  u64 v = t.kval[idx]; u32 cs = (u32)(v & 0xFFFFFFu);
  KeyRec r; r.k0 = k.x; r.k1 = k.y; r.order = (v >> 24) - 1 + order_base; r.tag = ((v >> 24) == 0 || cs == CS_NONE) ? 0ULL : t.cs_tag[cs];
  rec[at] = r;
}
// callsets received from other ranks (same tag function as callset_intern)
__global__ void __launch_bounds__(256) k_callsets_import(Tables t, const u32* rows, u64 n) {
  u64 idx = blockIdx.x * (u64)blockDim.x + threadIdx.x;
  if (idx >= n) return;
  const u32* r = rows + idx * (4 + t.gcap);
  u64 tag = (u64)r[2] | ((u64)r[3] << 32); u32 len = r[1];
  u32 h = (u32)(tag >> 24) & t.cs_mask;
  for (u32 probes = 0; probes <= t.cs_mask; probes++) {
    unsigned long long old = atomicCAS((unsigned long long*)(t.cs_tag + h), 0ULL, (unsigned long long)tag);
    if (old == 0ULL) { t.cs_len[h] = len; for (u32 i = 0; i < len; i++) t.cs_items[(u64)h * t.gcap + i] = r[4 + i]; atomicAdd(&t.ctr->n_callsets, 1ULL); return; }
    if (old == tag) return;
    h = (h + 1) & t.cs_mask;
  }
  atomicOr(&t.ctr->err, (unsigned)E_CS_FULL);
}
// ---- count rows in output order, on the device: compacted (cell, callset slot) entries -> (cell, dense callset id) keys,
// radix sort, split into the three output columns (the host used to do this with a 4-pass LSD sort: 240 ms for the 5 M
// rows of a C3-sized batch)
__global__ void __launch_bounds__(256) k_rows_remap(const u64* agg, u64 n, const u32* dense, u64* keys, i64* vals) {
  u64 i = blockIdx.x * (u64)blockDim.x + threadIdx.x;
  if (i >= n) return;
  u64 k = agg[2 * i] - 1;
  keys[i] = ((k >> 24) << 24) | (u64)dense[(u32)(k & 0xFFFFFF)]; vals[i] = (i64)agg[2 * i + 1];
}
__global__ void __launch_bounds__(256) k_rows_split(const u64* keys, const i64* vals, u64 n, u32* scope, u32* callset, i64* count) {
  u64 i = blockIdx.x * (u64)blockDim.x + threadIdx.x;
  if (i >= n) return;
  u64 k = keys[i]; scope[i] = (u32)(k >> 24); callset[i] = (u32)(k & 0xFFFFFF); count[i] = vals[i];
}
// ------------------------------------------------------------------------------------------------ launchers
static inline unsigned blocks_for(u64 n, unsigned bs) { return (unsigned)((n + bs - 1) / bs); }
// ------------------------------------------------------------------------------------------------ multi-GPU merge (nb_merge_*)
// The exchange blocks of engine.cu's merge: block 1 = {k, sent[ROUTE_MAX]} + k dictionary rows, block 2 = {n, n_keys} + n
// rows {callset tag, count} (whole-run) — every kernel reads its sizes from the gathered headers ON THE DEVICE, so the host
// never has to wait between the collective and the import.
constexpr u32 MERGE_HDR1 = 1 + ROUTE_MAX;   // u64 words
__global__ void k_merge_hdr1(u64* hdr, const unsigned long long* n_rows, const unsigned long long* route_cursor, u32 world) {
  u32 i = threadIdx.x;
  if (i == 0) hdr[0] = *n_rows;
  if (i < (u32)ROUTE_MAX) hdr[1 + i] = (route_cursor && i < world) ? route_cursor[i] : 0ULL;
}
__device__ __forceinline__ void callset_import_row(const Tables& t, const u32* r) {
  u64 tag = (u64)r[2] | ((u64)r[3] << 32); u32 len = r[1];
  u32 h = (u32)(tag >> 24) & t.cs_mask;
  for (u32 probes = 0; probes <= t.cs_mask; probes++) {
    unsigned long long old = atomicCAS((unsigned long long*)(t.cs_tag + h), 0ULL, (unsigned long long)tag);
    if (old == 0ULL) { t.cs_len[h] = len; for (u32 i = 0; i < len; i++) t.cs_items[(u64)h * t.gcap + i] = r[4 + i]; atomicAdd(&t.ctr->n_callsets, 1ULL); return; }
    if (old == tag) return;
    h = (h + 1) & t.cs_mask;
  }
  atomicOr(&t.ctr->err, (unsigned)E_CS_FULL);
}
// peers' dictionary rows straight out of the all-gather buffer: grid (rows, world), rank `self` skipped
__global__ void __launch_bounds__(256) k_merge_import_callsets(Tables t, const u8* all, u64 blk_bytes, u64 cap, u32 self) {
  const u32 r = blockIdx.y; if (r == self) return;
  const u8* blk = all + (u64)r * blk_bytes; const u64 k = min(*(const u64*)blk, cap);
  const u64 idx = blockIdx.x * (u64)blockDim.x + threadIdx.x; if (idx >= k) return;
  callset_import_row(t, (const u32*)(blk + 8 * MERGE_HDR1) + idx * (4 + t.gcap));
}
// returns 1 when the record created a key-table entry (the caller adds those up: Counters::n_live takes one atomic per warp)
__device__ __forceinline__ u32 key_import_rec(const Tables& t, const KeyRec& r) {
  u32 cs = CS_NONE;
  if (r.tag) {
    u32 h = (u32)(r.tag >> 24) & t.cs_mask; bool ok = false;
    for (u32 probes = 0; probes <= t.cs_mask; probes++) { u64 tg = t.cs_tag[h]; if (tg == r.tag) { ok = true; break; } if (tg == 0) break; h = (h + 1) & t.cs_mask; }
    if (!ok) { atomicOr(&t.ctr->err, (unsigned)E_CS_UNKNOWN); return 0u; }
    cs = h;
  }
  bool fresh;
  u64 slot = key_insert(t, r.k0, r.k1, fresh);
  if (slot == ~0ULL) { atomicOr(&t.ctr->err, (unsigned)E_KEY_FULL); return 0u; }
  atomicMax(t.kval + slot, (unsigned long long)(((r.order + 1) << 24) | cs));
  return fresh ? 1u : 0u;
}
__device__ __forceinline__ void add_live(const Tables& t, u32 n_new) {   // every lane of the warp calls it, converged
  for (int o = 16; o; o >>= 1) n_new += __shfl_xor_sync(0xFFFFFFFFu, n_new, o);
  if ((threadIdx.x & 31) == 0 && n_new) atomicAdd(&t.ctr->n_live, (unsigned long long)n_new);
}
__global__ void __launch_bounds__(256) k_keys_import(Tables t, const KeyRec* rec, u64 n) {
  const u64 idx = blockIdx.x * (u64)blockDim.x + threadIdx.x;
  u32 n_new = 0;
  if (idx < n) n_new = key_import_rec(t, rec[idx]);
  __syncwarp();
  add_live(t, n_new);
}
// the records peers stored into this rank's inbox, region by region; counts come from the gathered headers (sent[self] of rank r)
__global__ void __launch_bounds__(256) k_merge_import_inbox(Tables t, const KeyRec* inbox, u64 inbox_cap, const u8* all, u64 blk_bytes, u32 self) {
  const u32 r = blockIdx.y; if (r == self) return;
  const u64 n = min(((const u64*)(all + (u64)r * blk_bytes))[1 + self], inbox_cap);
  u32 n_new = 0;
  for (u64 idx = blockIdx.x * (u64)blockDim.x + threadIdx.x; idx < n; idx += (u64)gridDim.x * blockDim.x) {
    const uint4* p = (const uint4*)(inbox + (u64)r * inbox_cap + idx);
    uint4 a = __ldcg(p), b = __ldcg(p + 1);      // written by a peer GPU: read through L2, never a stale L1 line
    KeyRec rec; rec.k0 = (u64)a.x | ((u64)a.y << 32); rec.k1 = (u64)a.z | ((u64)a.w << 32); rec.order = (u64)b.x | ((u64)b.y << 32); rec.tag = (u64)b.z | ((u64)b.w << 32);
    n_new += key_import_rec(t, rec);
  }
  __syncwarp();
  add_live(t, n_new);
}
// this rank's folded counts as {callset tag, count} rows + header {n, unique keys}
__global__ void __launch_bounds__(256) k_merge_export_counts(Tables t, u64* blk2, u64 cap2) {
  u64 idx = blockIdx.x * (u64)blockDim.x + threadIdx.x;
  if (idx == 0) blk2[1] = t.ctr->n_keys;
  if (idx > t.agg_mask) return;
  unsigned long long k = t.agg_key[idx];
  if (!k) return;
  unsigned long long at = atomicAdd((unsigned long long*)blk2, 1ULL);
  if (at < cap2) { u32 slot = (u32)((k - 1) & 0xFFFFFF); blk2[2 + 2 * at] = t.cs_tag[slot]; blk2[3 + 2 * at] = t.agg_cnt[idx]; }
}
// every rank's rows (own included) summed into the (cleared) count table by callset slot: after this each rank holds the job's counts
__global__ void __launch_bounds__(256) k_merge_import_counts(Tables t, const u64* all2, u64 blk2_words, u64 cap2) {
  const u32 r = blockIdx.y; const u64* blk = all2 + (u64)r * blk2_words; const u64 n = min(blk[0], cap2);
  const u64 idx = blockIdx.x * (u64)blockDim.x + threadIdx.x;
  if (idx == 0) atomicAdd(&t.ctr->n_keys, (unsigned long long)blk[1]);
  if (idx >= n) return;
  const u64 tag = blk[2 + 2 * idx];
  u32 h = (u32)(tag >> 24) & t.cs_mask;
  for (u32 probes = 0; probes <= t.cs_mask; probes++) { u64 tg = t.cs_tag[h]; if (tg == tag) { if (agg_add(t, (unsigned long long)h + 1ULL, blk[3 + 2 * idx])) atomicAdd(&t.ctr->n_agg, 1ULL); return; } if (tg == 0) break; h = (h + 1) & t.cs_mask; }
  atomicOr(&t.ctr->err, (unsigned)E_CS_FULL);
}
// scoped merge: (cell, callset slot) counts -> dense [cells x callsets] table by the job-wide callset numbering, and back
__global__ void __launch_bounds__(256) k_merge_dense_fill(Tables t, const u32* dense_id, unsigned long long* dense, u64 n_cs, u64 n_cells) {
  u64 idx = blockIdx.x * (u64)blockDim.x + threadIdx.x;
  if (idx > t.agg_mask) return;
  unsigned long long k = t.agg_key[idx];
  if (!k) return;
  k -= 1; u64 cell = k >> 24; u32 id = dense_id[(u32)(k & 0xFFFFFF)];
  if (cell >= n_cells || id == NONE32) { atomicOr(&t.ctr->err, (unsigned)E_AGG_FULL); return; }
  atomicAdd(dense + cell * n_cs + id, t.agg_cnt[idx]);
}
__global__ void __launch_bounds__(256) k_merge_dense_rows(const unsigned long long* dense, u64 n, u64 n_cs, const unsigned long long* prefix, u32* scope, u32* callset, i64* count, u32 cell_base) {
  // `prefix` = exclusive scan of (dense != 0): rows come out ordered by (cell, callset) without a sort
  u64 i = blockIdx.x * (u64)blockDim.x + threadIdx.x;
  if (i >= n) return;
  unsigned long long v = dense[i];
  if (!v) return;
  u64 at = prefix[i]; scope[at] = cell_base + (u32)(i / n_cs); callset[at] = (u32)(i % n_cs); count[at] = (i64)v;
}
__global__ void __launch_bounds__(256) k_merge_nonzero(const unsigned long long* dense, u64 n, unsigned long long* flag) {
  u64 i = blockIdx.x * (u64)blockDim.x + threadIdx.x;
  if (i < n) flag[i] = dense[i] ? 1ULL : 0ULL;
}
void launch_merge_hdr1(u64* hdr, const unsigned long long* n_rows, const unsigned long long* route_cursor, u32 world, cudaStream_t s) { k_merge_hdr1<<<1, 32, 0, s>>>(hdr, n_rows, route_cursor, world); }
void launch_merge_import_callsets(const Tables& t, const void* all, u64 blk_bytes, u64 cap, u32 world, u32 self, cudaStream_t s) {
  if (cap && world > 1) k_merge_import_callsets<<<dim3(blocks_for(cap, 256), world), 256, 0, s>>>(t, (const u8*)all, blk_bytes, cap, self);
}
void launch_merge_import_inbox(const Tables& t, const void* inbox, u64 inbox_cap, u64 max_count, const void* all, u64 blk_bytes, u32 world, u32 self, cudaStream_t s) {
  if (max_count && world > 1) k_merge_import_inbox<<<dim3(std::min<unsigned>(blocks_for(max_count, 256), 148 * 16), world), 256, 0, s>>>(t, (const KeyRec*)inbox, inbox_cap, (const u8*)all, blk_bytes, self);
}
void launch_merge_export_counts(const Tables& t, u64* blk2, u64 cap2, cudaStream_t s) { k_merge_export_counts<<<blocks_for(t.agg_mask + 1, 256), 256, 0, s>>>(t, blk2, cap2); }
void launch_merge_import_counts(const Tables& t, const u64* all2, u64 blk2_words, u64 cap2, u32 world, cudaStream_t s) {
  k_merge_import_counts<<<dim3(blocks_for(std::max<u64>(cap2, 1), 256), world), 256, 0, s>>>(t, all2, blk2_words, cap2);
}
void launch_merge_dense_fill(const Tables& t, const u32* dense_id, unsigned long long* dense, u64 n_cs, u64 n_cells, cudaStream_t s) { k_merge_dense_fill<<<blocks_for(t.agg_mask + 1, 256), 256, 0, s>>>(t, dense_id, dense, n_cs, n_cells); }
size_t merge_scan_tmp_bytes(u64 n) { size_t tb = 0; cub::DeviceScan::ExclusiveSum(nullptr, tb, (const unsigned long long*)nullptr, (unsigned long long*)nullptr, (int)n); return tb + 256; }
// dense table -> rows (scope, callset, count) ordered by (cell, callset), in two steps so that the host can size the row
// buffers: (1) non-zero flags + exclusive scan (row count = flag[n-1] + prefix[n-1]), (2) the rows
void launch_merge_dense_scan(const unsigned long long* dense, u64 n, unsigned long long* flag, unsigned long long* prefix, void* tmp, size_t tmp_bytes, cudaStream_t s) {
  if (!n) return;
  k_merge_nonzero<<<blocks_for(n, 256), 256, 0, s>>>(dense, n, flag);
  cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, (const unsigned long long*)flag, prefix, (int)n, s);
}
void launch_merge_dense_rows(const unsigned long long* dense, u64 n, u64 n_cs, const unsigned long long* prefix, u32* scope, u32* callset, i64* count, u32 cell_base, cudaStream_t s) {
  if (n) k_merge_dense_rows<<<blocks_for(n, 256), 256, 0, s>>>(dense, n, n_cs, prefix, scope, callset, count, cell_base);
}
void launch_keys_count_owner(const Tables& t, u32 world, unsigned long long* counts, cudaStream_t s) { k_keys_count_owner<<<blocks_for(t.key_mask + 1, 256), 256, 0, s>>>(t, world, counts); }
void launch_keys_scatter(const Tables& t, void* rec, unsigned long long* cursors, u64 order_base, u32 world, cudaStream_t s) { k_keys_scatter<<<blocks_for(t.key_mask + 1, 256), 256, 0, s>>>(t, (KeyRec*)rec, cursors, order_base, world); }
void launch_callsets_import(const Tables& t, const u32* rows, u64 n, cudaStream_t s) { if (n) k_callsets_import<<<blocks_for(n, 256), 256, 0, s>>>(t, rows, n); }

void launch_pack(const BatchDev& b, cudaStream_t s) {
  u64 n = (u64)b.n_reads * (b.W - 1); if (!n) return;
  if (b.enc == 1) k_pack_enc<1><<<blocks_for(n, 256), 256, 0, s>>>(b);
  else if (b.enc == 2) k_pack_enc<2><<<blocks_for(n, 256), 256, 0, s>>>(b);
  else {
    // Measured on B200 (C2, 2 M reads per launch): the direct kernel 110 us, the bulk-copy kernel 145 us — one tile per block
    // leaves each block's chain offsets -> TMA -> wait -> classify -> cut exposed (8 resident blocks do not cover it) and the
    // classification, not the realignment, is most of the instructions.  The direct kernel stays the default;
    // NB_PACK_BULK=1 selects the staged one (same results: the parity suite runs green on both).
    const char* env = getenv("NB_PACK_BULK"); const bool bulk = env && atoi(env) != 0;   // read per launch: the tests switch it
    const u32 Wd = b.W - 1;
    if (!bulk || Wd > 32) { k_pack<<<blocks_for(n, 256), 256, 0, s>>>(b); return; }
    u32 RB = PACK_T / Wd; if (b.sides == 2) RB &= ~1u;
    k_pack_bulk<<<blocks_for(b.n_reads, RB), PACK_T, 0, s>>>(b, RB, (65536u + Wd - 1) / Wd);
  }
}
void launch_trim(const BatchDev& b, const Tables& t, cudaStream_t s) { if (b.n_reads) k_trim<<<blocks_for(b.n_reads, 256), 256, 0, s>>>(b, t); }
void launch_map(const BatchDev& b, const DevIndex& ix, const DevCfg& cfg, const Tables& t, int count_work, cudaStream_t s) {
  if (!b.n_reads) return;
  // k_walk: persistent warps popping seeded reads from the global list (counters zeroed by the host before the launch):
  // enough blocks to fill every SM at the kernel's occupancy, never more than the work needs
  static int sms = 0, per_sm[4] = {0, 0, 0, 0};
  if (!sms) {
    int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev); if (sms <= 0) sms = 148;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm[0], k_walk<0, 0>, 128, 0) != cudaSuccess || per_sm[0] < 1) per_sm[0] = 8;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm[1], k_walk<1, 0>, 128, 0) != cudaSuccess || per_sm[1] < 1) per_sm[1] = 8;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm[2], k_walk<0, 1>, 128, 0) != cudaSuccess || per_sm[2] < 1) per_sm[2] = 8;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm[3], k_walk<1, 1>, 128, 0) != cudaSuccess || per_sm[3] < 1) per_sm[3] = 8;
  }
  const int v = (count_work ? 1 : 0) | (ix.hbm ? 2 : 0);
  unsigned sb = blocks_for(b.n_reads, SEED_BLOCK), wb = min(blocks_for(b.n_reads, 128), (unsigned)(sms * per_sm[v]));
  switch (v) {
    case 0: k_seed<0, 0><<<sb, SEED_BLOCK, 0, s>>>(b, ix, cfg, t); k_walk<0, 0><<<wb, 128, 0, s>>>(b, ix, cfg, t); break;
    case 1: k_seed<1, 0><<<sb, SEED_BLOCK, 0, s>>>(b, ix, cfg, t); k_walk<1, 0><<<wb, 128, 0, s>>>(b, ix, cfg, t); break;
    case 2: k_seed<0, 1><<<sb, SEED_BLOCK, 0, s>>>(b, ix, cfg, t); k_walk<0, 1><<<wb, 128, 0, s>>>(b, ix, cfg, t); break;
    default: k_seed<1, 1><<<sb, SEED_BLOCK, 0, s>>>(b, ix, cfg, t); k_walk<1, 1><<<wb, 128, 0, s>>>(b, ix, cfg, t); break;
  }
}
// ---- probe table + Bloom prefilter, built on the device from the artefact's flat table when a context is created
__global__ void __launch_bounds__(256) k_probe_build(const u64* tkey, const u64* tval, u64 slots, u64* ptab, u32 n_pbuckets, u64* bloom, u32 bloom_words, u32 bloom_k, unsigned int* err) {
  u64 i = blockIdx.x * (u64)blockDim.x + threadIdx.x;
  if (i >= slots) return;
  const u64 key = tkey[i];
  if (!(key >> 63)) return;
  const u64 val = tval[i], hh = nb_khash(key & KMASK); const u32 h = (u32)hh;
  if (bloom_words) atomicOr((unsigned long long*)(bloom + __umulhi((u32)(hh >> 32), bloom_words)), (unsigned long long)nb_bloom_bits(h, bloom_k));
  u32 b = __umulhi(h, n_pbuckets);
  for (u32 tries = 0; tries < n_pbuckets; tries++) {
    unsigned long long* q = (unsigned long long*)(ptab + 4 * (u64)b);
    if (atomicCAS(q, 0ULL, (unsigned long long)key) == 0ULL) { ptab[4 * (u64)b + 2] = val; return; }   // slot 0 first: occupied slots stay a prefix
    if (atomicCAS(q + 1, 0ULL, (unsigned long long)key) == 0ULL) { ptab[4 * (u64)b + 3] = val; return; }
    if (++b == n_pbuckets) b = 0;
  }
  atomicOr(err, 1u);
}
void launch_probe_build(const u64* tkey, const u64* tval, u64 slots, u64* ptab, u32 n_pbuckets, u64* bloom, u32 bloom_words, u32 bloom_k, unsigned int* err, cudaStream_t s) {
  if (slots) k_probe_build<<<blocks_for(slots, 256), 256, 0, s>>>(tkey, tval, slots, ptab, n_pbuckets, bloom, bloom_words, bloom_k, err);
}
__global__ void __launch_bounds__(256) k_dense_scatter(const u32* ids, u64 n, u32* dense) { u64 i = blockIdx.x * (u64)blockDim.x + threadIdx.x; if (i < n) dense[ids[i]] = (u32)i; }
void launch_dense_scatter(const u32* ids, u64 n, u32* dense, cudaStream_t s) { if (n) k_dense_scatter<<<blocks_for(n, 256), 256, 0, s>>>(ids, n, dense); }
size_t rows_sort_tmp_bytes(u64 n) { size_t tb = 0; cub::DeviceRadixSort::SortPairs(nullptr, tb, (const u64*)nullptr, (u64*)nullptr, (const i64*)nullptr, (i64*)nullptr, (int)n, 0, 56); return tb + 256; }
// work: 2n u64 keys + 2n i64 values + temp; out: n u32 + n u32 + n i64 (all device)
void launch_rows_sort(const u64* agg, u64 n, const u32* dense, u64* keys, i64* vals, void* tmp, size_t tmp_bytes, u32* scope, u32* callset, i64* count, int key_bits, cudaStream_t s) {
  if (!n) return;
  k_rows_remap<<<blocks_for(n, 256), 256, 0, s>>>(agg, n, dense, keys, vals);
  cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, (const u64*)keys, keys + n, (const i64*)vals, vals + n, (int)n, 0, key_bits, s);   // whole-run scope: 24 key bits = 3 passes instead of 7
  k_rows_split<<<blocks_for(n, 256), 256, 0, s>>>(keys + n, vals + n, n, scope, callset, count);
}
void launch_pair(const BatchDev& b, const DevIndex& ix, const DevLib& lib, const DevCfg& cfg, const Tables& t, const Route& rt, cudaStream_t s) {
  if (b.n_pairs) k_pair<<<blocks_for(b.n_pairs, 128), 128, 0, s>>>(b, ix, lib, cfg, t, rt);
}
void launch_fold(const Tables& t, const u32* cell_of_pair, u64 order_base, cudaStream_t s) {
  // contiguous slot ranges, a few blocks per SM (148 SMs x 8): enough votes per block for the shared-memory table to pay
  u64 slots = t.key_mask + 1, blocks = std::min<u64>((slots + 255) / 256, 148 * 8), per = ((slots + blocks - 1) / blocks + 255) / 256 * 256;
  k_fold<<<(unsigned)((slots + per - 1) / per), 256, 0, s>>>(t, cell_of_pair, order_base, per);
}
void launch_resolve(const BatchDev& b, const Tables& t, cudaStream_t s) { if (b.n_pairs) k_resolve<<<blocks_for(b.n_pairs, 256), 256, 0, s>>>(b, t); }
void launch_export_reads(const BatchDev& b, const DevIndex& ix, const Tables& t, void* out, cudaStream_t s) {
  if (b.n_reads) k_export_reads<<<blocks_for(b.n_reads, 256), 256, 0, s>>>(b, ix, t, (ReadOut*)out);
}
// occupied entries of the count table -> {key, count} rows; of the callset dictionary -> {slot, len, tag_lo, tag_hi, items[gcap]} rows
__global__ void __launch_bounds__(256) k_compact_agg(Tables t, u64* out, u64 cap, unsigned long long* n_out) {
  u64 idx = blockIdx.x * (u64)blockDim.x + threadIdx.x;
  if (idx > t.agg_mask) return;
  unsigned long long k = t.agg_key[idx];
  if (!k) return;
  unsigned long long at = atomicAdd(n_out, 1ULL);
  if (at < cap) { out[2 * at] = k; out[2 * at + 1] = t.agg_cnt[idx]; }
}
__global__ void __launch_bounds__(256) k_compact_cs(Tables t, u32* out, u64 cap, unsigned long long* n_out) {
  u32 idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx > t.cs_mask) return;
  if (!t.cs_tag[idx]) return;
  unsigned long long at = atomicAdd(n_out, 1ULL);
  if (at >= cap) return;
  u32* r = out + at * (4 + t.gcap); u32 n = t.cs_len[idx]; u64 tag = t.cs_tag[idx];
  r[0] = idx; r[1] = n; r[2] = (u32)tag; r[3] = (u32)(tag >> 32);
  for (u32 i = 0; i < t.gcap; i++) r[4 + i] = i < n ? t.cs_items[(u64)idx * t.gcap + i] : 0u;
}
void launch_compact(const Tables& t, u64* agg_out, u64 agg_cap, u32* cs_out, u64 cs_cap, unsigned long long* n_out2, cudaStream_t s) {
  k_compact_agg<<<blocks_for(t.agg_mask + 1, 256), 256, 0, s>>>(t, agg_out, agg_cap, n_out2);
  k_compact_cs<<<blocks_for((u64)t.cs_mask + 1, 256), 256, 0, s>>>(t, cs_out, cs_cap, n_out2 + 1);
}
__global__ void __launch_bounds__(256) k_count_keys(Tables t) {
  u64 idx = blockIdx.x * (u64)blockDim.x + threadIdx.x;
  bool occ = false;
  if (idx <= t.key_mask) { ulonglong2 k = t.key[idx]; occ = !(k.x == 0 && k.y == 0); }
  unsigned ob = __ballot_sync(0xFFFFFFFFu, occ);
  if ((threadIdx.x & 31) == 0 && ob) atomicAdd(&t.ctr->n_keys, (unsigned long long)__popc(ob));
}
void launch_count_keys(const Tables& t, cudaStream_t s) { k_count_keys<<<blocks_for(t.key_mask + 1, 256), 256, 0, s>>>(t); }
void launch_rehash_keys(const Tables& o, const Tables& n, cudaStream_t s) { k_rehash_keys<<<blocks_for(o.key_mask + 1, 256), 256, 0, s>>>(o, n); }
void launch_keys_export(const Tables& t, void* records, unsigned long long* n_out, u64 cap, u64 order_base, cudaStream_t s) {
  k_keys_export<<<blocks_for(t.key_mask + 1, 256), 256, 0, s>>>(t, (KeyRec*)records, n_out, cap, order_base);
}
void launch_keys_import(const Tables& t, const void* records, u64 n, cudaStream_t s) { if (n) k_keys_import<<<blocks_for(n, 256), 256, 0, s>>>(t, (const KeyRec*)records, n); }

// ------------------------------------------------------------------------------------------------ per-cell table (nb_cells_*)
// returns the slot of `key`, claiming it when absent (fresh = 1); ~0 when every slot was probed
__device__ __forceinline__ u64 cell_slot(const CellTable& t, unsigned long long key, u32& fresh) {
  u64 h = mix64(key) & t.mask;
  for (u64 probes = 0; probes <= t.mask; probes++) {
    unsigned long long old = atomicCAS(t.key + h, 0ULL, key);
    if (old == 0ULL || old == key) { fresh = old == 0ULL; return h; }
    h = (h + 1) & t.mask;
  }
  atomicOr(t.ctr + 1, 1ULL);
  return ~0ULL;
}
// one thread per per-scope row of a finalized scoped batch: umis += 1 (a scope has at most one row per callset), reads += count
__global__ void __launch_bounds__(256) k_cells_roll(CellTable t, const u32* row_scope, const u32* row_callset, const i64* row_count, u64 n, const u32* cell_of_scope, const u32* pid_of_dense) {
  u64 i = blockIdx.x * (u64)blockDim.x + threadIdx.x;
  u32 fresh = 0;
  if (i < n) {
    const unsigned long long key = (((unsigned long long)cell_of_scope[row_scope[i]] << 32) | pid_of_dense[row_callset[i]]) + 1ULL;
    const u64 h = cell_slot(t, key, fresh);
    if (h != ~0ULL) { atomicAdd(t.umis + h, 1ULL); atomicAdd(t.reads + h, (unsigned long long)row_count[i]); }
  }
  const u32 nw = __popc(__ballot_sync(0xFFFFFFFFu, fresh));   // new entries: one atomic per warp
  if ((threadIdx.x & 31) == 0 && nw) atomicAdd(t.ctr, (unsigned long long)nw);
}
__global__ void __launch_bounds__(256) k_cells_rehash(CellTable o, CellTable n) {
  u64 idx = blockIdx.x * (u64)blockDim.x + threadIdx.x;
  if (idx > o.mask) return;
  const unsigned long long k = o.key[idx];
  if (!k) return;
  u32 fresh = 0;
  const u64 h = cell_slot(n, k, fresh);
  if (h != ~0ULL) { n.umis[h] = o.umis[idx]; n.reads[h] = o.reads[idx]; }
}
__global__ void __launch_bounds__(256) k_cells_compact(CellTable t, const u32* rank_of_pid, u64* keys, u32* slots, u64 cap, unsigned long long* n_out) {
  u64 idx = blockIdx.x * (u64)blockDim.x + threadIdx.x;
  if (idx > t.mask) return;
  const unsigned long long k = t.key[idx];
  if (!k) return;
  const unsigned long long at = atomicAdd(n_out, 1ULL);
  if (at >= cap) return;
  const u64 ck = k - 1;
  keys[at] = (ck & 0xFFFFFFFF00000000ULL) | rank_of_pid[(u32)ck]; slots[at] = (u32)idx;
}
__global__ void __launch_bounds__(256) k_cells_split(CellTable t, const u64* keys, const u32* slots, u64 n, u32* cell, u32* callset, i64* umis, i64* reads) {
  u64 i = blockIdx.x * (u64)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const u64 k = keys[i]; const u32 sl = slots[i];
  cell[i] = (u32)(k >> 32); callset[i] = (u32)k; umis[i] = (i64)t.umis[sl]; reads[i] = (i64)t.reads[sl];
}
void launch_cells_roll(const CellTable& t, const u32* row_scope, const u32* row_callset, const i64* row_count, u64 n_rows, const u32* cell_of_scope, const u32* pid_of_dense, cudaStream_t s) {
  if (n_rows) k_cells_roll<<<blocks_for(n_rows, 256), 256, 0, s>>>(t, row_scope, row_callset, row_count, n_rows, cell_of_scope, pid_of_dense);
}
void launch_cells_rehash(const CellTable& o, const CellTable& n, cudaStream_t s) { k_cells_rehash<<<blocks_for(o.mask + 1, 256), 256, 0, s>>>(o, n); }
size_t cells_sort_tmp_bytes(u64 n) { size_t tb = 0; cub::DeviceRadixSort::SortPairs(nullptr, tb, (const u64*)nullptr, (u64*)nullptr, (const u32*)nullptr, (u32*)nullptr, (int)n, 0, 64); return tb + 256; }
void launch_cells_finalize(const CellTable& t, u64 n, const u32* rank_of_pid, u64* keys, u32* slots, unsigned long long* n_out, void* tmp, size_t tmp_bytes, void* out, cudaStream_t s) {
  if (!n) return;
  k_cells_compact<<<blocks_for(t.mask + 1, 256), 256, 0, s>>>(t, rank_of_pid, keys, slots, n, n_out);
  cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, (const u64*)keys, keys + n, (const u32*)slots, slots + n, (int)n, 0, 64, s);
  u32* cell = (u32*)out; u32* callset = cell + n; i64* umis = (i64*)(callset + n); i64* reads = umis + n;
  k_cells_split<<<blocks_for(n, 256), 256, 0, s>>>(t, keys + n, slots + n, n, cell, callset, umis, reads);
}

}  // namespace nbk
