// bam_group.cu — BAM mode in any record order: the device record store and the (UMI, CB) grouping (bam_group.hpp).
//
// The host producer (bam.cpp) stages every kept record of a window and this file uploads it into HBM.  At the end of the
// file the records are put in (UMI, full CB, ordinal) order by two stable CUB radix sorts (CB rank, then UMI key, ordinals
// as values), a scope starts wherever (UMI, CB[..len-2]) changes, and one thread per scope restates
// SortedBamReader::add_dummy_paired_reads + filter_paired_reads (src/parse/sorted_bam_reader.rs:109-162) over the scope's
// records in that order: a count pass, a scan, a write pass.  Pairs are (base offset, clipped length, flags) into the store,
// so no bases move: the scoped batches handed to nb_align_batch are NB_MEM_DEVICE views of the store.  Under a device
// budget every allocation here is counted against it, and compact() drops the records of the UMI buckets a pass gives up.
// Rows mode (nb_process_bam_rows_any_order) keeps every record's metadata text in a fourth byte store, and the row kernels
// below turn each aligned batch into the grouped driver's TSV rows next to it.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <algorithm>
#include <chrono>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <string>
#include <type_traits>

#include "bam_group.hpp"

using namespace nb;

namespace nbg {

#define GK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) return fail(NB_ERR_CUDA, std::string(#x) + ": " + cudaGetErrorString(e_)); } while (0)

namespace {

const u64 PAD = 64;   // the kernels read bases and quals as aligned 16-byte vectors past a read's end (nimble_b200.h)

// every device allocation of this file: one counter, its peak, and the budget (0: none) it may not pass
struct Mem {
  u64 live = 0, peak = 0, budget = 0;
  cudaError_t alloc(void** p, u64 n) {
    if (budget && live + n > budget) return cudaErrorMemoryAllocation;
    const cudaError_t e = cudaMalloc(p, n);
    if (e == cudaSuccess) { live += n; peak = std::max(peak, live); }
    return e;
  }
  void release(void*& p, u64 n) { if (p) { cudaFree(p); live -= n; } p = nullptr; }
};

// The capacity a store array of capacity cap grows to for need bytes, 0 when the budget cannot hold it.  With a budget
// the old and new copies are both alive while the contents move (live + want <= B), and afterwards the store leaves room
// for the grouping arrays (live - cap + want + reserve <= B).  exact: no growth slack.
u64 grow_to(u64 cap, u64 need, const Mem& m, u64 reserve, bool exact = false) {
  const u64 want = exact ? need + PAD : std::max<u64>(need + PAD, cap + cap / 2);
  if (!m.budget) return want;
  const u64 after = m.live - cap + reserve;
  if (m.live >= m.budget || after >= m.budget) return 0;
  const u64 w = std::min({want, m.budget - m.live, m.budget - after});
  return w >= need + PAD ? w : 0;
}

// a device array that keeps its contents when it grows (the store is appended to window by window)
struct Grow {
  void* p = nullptr; u64 cap = 0;
  int ensure(u64 need, u64 keep, cudaStream_t s, const char* what, u64 store_total, Mem& m, u64 reserve, bool exact) {
    if (need + PAD <= cap) return NB_OK;
    u64 want = grow_to(cap, need, m, reserve, exact);
    if (!want) return fail(NB_ERR_CUDA, "the device budget of " + std::to_string(m.budget) + " bytes cannot hold the record store: " + what + " needs " + std::to_string(need + PAD) + " bytes (the store needs " + std::to_string(store_total) + " bytes so far)");
    void* q = nullptr;
    if (m.alloc(&q, want) != cudaSuccess) {
      cudaGetLastError();
      want = need + PAD;
      if (m.alloc(&q, want) != cudaSuccess) { cudaGetLastError(); return fail(NB_ERR_CUDA, std::string("not enough device memory for the record store: ") + what + " needs " + std::to_string(need + PAD) + " bytes (the store needs " + std::to_string(store_total) + " bytes so far)"); }
    }
    if (p) { if (keep) GK(cudaMemcpyAsync(q, p, keep, cudaMemcpyDeviceToDevice, s)); GK(cudaStreamSynchronize(s)); m.release(p, cap); }
    p = q; cap = want;
    return NB_OK;
  }
  void release(Mem& m) { m.release(p, cap); cap = 0; }
};

struct Pinned {
  void* p = nullptr; u64 cap = 0;
  int ensure(u64 n) {
    if (n <= cap) return NB_OK;
    if (p) cudaFreeHost(p);
    p = nullptr; cap = 0;
    const u64 want = n + n / 4 + 4096;
    if (cudaHostAlloc(&p, want, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); p = nullptr; return fail(NB_ERR_CUDA, "pinned host allocation failed"); }
    cap = want; return NB_OK;
  }
  ~Pinned() { if (p) cudaFreeHost(p); }
};

// ------------------------------------------------------------------------------------------------ kernels
__global__ void k_cb_keys(const u32* __restrict__ cb, const u32* __restrict__ rank, u32* __restrict__ key, u32* __restrict__ val, u32 n) {
  const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) { key[i] = rank[cb[i]]; val[i] = i; }
}
__global__ void k_umi_gather(const u64* __restrict__ umi, const u32* __restrict__ perm, u64* __restrict__ key, u32 n) {
  const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) key[i] = umi[perm[i]];
}
// head of a scope: (UMI, CB[..len-2]) differs from the previous record in sorted order
__global__ void k_heads(const u64* __restrict__ umi_sorted, const u32* __restrict__ perm, const u32* __restrict__ cb, const u32* __restrict__ prefix, u32* __restrict__ head, u32 n) {
  const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  head[i] = (i == 0 || umi_sorted[i] != umi_sorted[i - 1] || prefix[cb[perm[i]]] != prefix[cb[perm[i - 1]]]) ? 1u : 0u;
}
// sid = inclusive sum of the heads: scope s = sid - 1 starts at i
__global__ void k_starts(const u32* __restrict__ head, const u32* __restrict__ sid, u32* __restrict__ start, u32 n) {
  const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (head[i]) start[sid[i] - 1] = i;
  if (i == n - 1) start[sid[i]] = n;
}

struct Recs {   // the store's per-record arrays, indexed by kept index (file order of the kept records)
  const u32* perm; const u64* nib_off; const u32* lseq; const u16* flag; const u64* name_off; const u8* name_len; const char* names; const u32* cb;
};
struct PairsOut { u64* o1; u64* o2; u32* l1; u32* l2; u8* f1; u8* f2; u32* scope; u32* idx1; u32* idx2; };

__device__ __forceinline__ bool same_name(const Recs& d, u32 a, u32 b) {
  if (a == b) return true;   // a record and its dummy mate
  const u32 la = d.name_len[a];
  if (la != d.name_len[b]) return false;
  const char* x = d.names + d.name_off[a]; const char* y = d.names + d.name_off[b];
  for (u32 i = 0; i < la; i++) if (x[i] != y[i]) return false;
  return true;
}

// One scope's records at sorted positions [s0, s1): add_dummy_paired_reads (every unpaired record is followed by a
// SKIP_ALIGN copy of itself) and filter_paired_reads (neighbours with equal names form a pair, the first-in-template one
// in the sequence slot; otherwise the left one is dropped), walked over (position, copy) without materialising the list.
template <bool WRITE>
__device__ u64 walk_scope(const Recs& d, u32 s0, u32 s1, const PairsOut& out, u64 at, u32 scope) {
  if (s0 >= s1) return 0;
  auto next = [&](u32& j, u32& k) { if (k == 0 && !(d.flag[d.perm[j]] & 1)) k = 1; else { j++; k = 0; } };
  u32 ja = s0, ka = 0, jb = s0, kb = 0; next(jb, kb);
  u64 np = 0;
  while (jb < s1) {
    const u32 ra = d.perm[ja], rb = d.perm[jb];
    if (same_name(d, ra, rb)) {
      if (WRITE) {
        const bool a_first = d.flag[ra] & 64;
        const u32 rs = a_first ? ra : rb, rm = a_first ? rb : ra, ks = a_first ? ka : kb, km = a_first ? kb : ka;
        const u64 p = at + np;
        #pragma unroll
        for (int side = 0; side < 2; side++) {
          const u32 r = side ? rm : rs, k = side ? km : ks;
          const u32 n = d.lseq[r]; const bool rev = d.flag[r] & 16;
          u32 x = 0, y = n;
          if (n == 124) { if (rev) y = n - 13; else x = 13; }   // strip_nonbio_regions (src/parse/bam.rs:258-268)
          const u64 o = 2 * d.nib_off[r] + x; const u8 f = (u8)((k ? NB_FLAG_SKIP_ALIGN : 0) | (rev ? NB_FLAG_REVCOMP : 0));
          if (side) { out.o2[p] = o; out.l2[p] = y - x; out.f2[p] = f; out.idx2[p] = r; }
          else { out.o1[p] = o; out.l1[p] = y - x; out.f1[p] = f; out.idx1[p] = r; }
        }
        out.scope[p] = scope;
      }
      np++;
      ja = jb; ka = kb; next(ja, ka);
      if (ja >= s1) break;
      jb = ja; kb = ka; next(jb, kb);
    } else {
      ja = jb; ka = kb; next(jb, kb);
    }
  }
  return np;
}

__global__ void k_pair_count(Recs d, const u32* __restrict__ start, u64* __restrict__ cnt, u32* __restrict__ scope_cb, u32 n_scopes) {
  const u32 s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s > n_scopes) return;
  if (s == n_scopes) { cnt[s] = 0; return; }
  const PairsOut none{};
  cnt[s] = walk_scope<false>(d, start[s], start[s + 1], none, 0, s);
  scope_cb[s] = d.cb[d.perm[start[s]]];
}
__global__ void k_pair_write(Recs d, const u32* __restrict__ start, const u64* __restrict__ pair0, PairsOut out, u32 n_scopes) {
  const u32 s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s < n_scopes) walk_scope<true>(d, start[s], start[s + 1], out, pair0[s], s);
}
__global__ void k_local_scope(const u32* __restrict__ scope, u32* __restrict__ local, u64 n, u32 base) {
  const u64 i = blockIdx.x * (u64)blockDim.x + threadIdx.x;
  if (i < n) local[i] = scope[i] - base;
}

inline u32 blocks(u64 n, u32 t = 256) { return (u32)((n + t - 1) / t); }

// ---------------------------------------------------------------------------------------- compaction (budget mode)
// keep flag of every record (its UMI bucket is below hi) and its kept nibble / name bytes; entry n is 0, so exclusive
// scans of the n + 1 entries give destinations and totals
// (rows mode: td = the kept metadata bytes, else meta_len is null)
__global__ void k_keep(const u64* __restrict__ umi, const u32* __restrict__ lseq, const u8* __restrict__ name_len, const u32* __restrict__ meta_len, u32 hi,
                       u32* __restrict__ pos, u64* __restrict__ nd, u64* __restrict__ md, u64* __restrict__ td, u32 n) {
  const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i > n) return;
  const bool k = i < n && umi_bucket(umi[i]) < hi;
  pos[i] = k; nd[i] = k ? (lseq[i] + 1) / 2 : 0; md[i] = k ? name_len[i] : 0;
  if (meta_len) td[i] = k ? meta_len[i] : 0;
}

// per-record arrays, one tile of records [t0, t1): the kept values go to the tile in order, then to their destination
template <class T>
__global__ void k_rec_gather(const T* __restrict__ src, const u32* __restrict__ pos, T* __restrict__ tile, u32 t0, u32 t1) {
  const u32 i = t0 + blockIdx.x * blockDim.x + threadIdx.x;
  if (i < t1 && pos[i + 1] > pos[i]) tile[pos[i] - pos[t0]] = src[i];
}
template <class T>
__global__ void k_rec_scatter(const T* __restrict__ tile, const u32* __restrict__ pos, T* __restrict__ dst, u32 t0, u32 t1) {
  const u32 j = blockIdx.x * blockDim.x + threadIdx.x, base = pos[t0];
  if (j < pos[t1] - base) dst[base + j] = tile[j];
}

// Byte runs: record i owns [mul * so[i], mul * so[i + 1]) of the array (so = its old nibble or name offset; the runs are
// back to back in record order) and, when kept, moves to mul * dn[i] (dn = exclusive scan of the kept run lengths).
__device__ __forceinline__ u64 umin(u64 a, u64 b) { return a < b ? a : b; }
__device__ __forceinline__ u64 umax(u64 a, u64 b) { return a > b ? a : b; }
// last record whose run starts at or before byte b
__device__ u32 run_at(const u64* so, u32 n, u64 mul, u64 b) {
  u32 lo = 0, hi = n;   // so[0] = 0 <= b
  while (hi - lo > 1) { const u32 m = (lo + hi) / 2; if (mul * so[m] <= b) lo = m; else hi = m; }
  return lo;
}
// kept bytes before byte b = where byte b's tile starts at the destination
__device__ u64 kept_before(const u64* so, const u64* dn, u32 n, u64 mul, u64 b) {
  const u32 r = run_at(so, n, mul, b);
  const u64 len = mul * (dn[r + 1] - dn[r]);
  return mul * dn[r] + (len ? umin(b - mul * so[r], len) : 0);
}
// one warp copies n bytes, 16 at a time where source and destination share their alignment
__device__ __forceinline__ void warp_copy(u8* __restrict__ dst, const u8* __restrict__ src, u64 n, u32 lane) {
  if ((((uintptr_t)dst ^ (uintptr_t)src) & 15) == 0) {
    const u64 head = umin((16 - ((uintptr_t)src & 15)) & 15, n), nv = (n - head) / 16;
    for (u64 k = lane; k < head; k += 32) dst[k] = src[k];
    const uint4* s4 = (const uint4*)(src + head); uint4* d4 = (uint4*)(dst + head);
    for (u64 k = lane; k < nv; k += 32) d4[k] = s4[k];
    for (u64 k = head + 16 * nv + lane; k < n; k += 32) dst[k] = src[k];
  } else {
    for (u64 k = lane; k < n; k += 32) dst[k] = src[k];
  }
}
// source bytes [b0, b1): each kept run's part in it goes to tile[dest - d0 + (d0 & 15)] with d0 = kept_before(b0), one warp
// per run; the tile holds its bytes at d0's alignment, so the scatter below copies 16 bytes at a time
__global__ void k_run_gather(const u8* __restrict__ src, u8* __restrict__ tile, const u64* __restrict__ so, const u64* __restrict__ dn, u32 n, u32 mul, u64 b0, u64 b1) {
  __shared__ u32 r0; __shared__ u64 d0;
  if (threadIdx.x == 0) { r0 = run_at(so, n, mul, b0); d0 = kept_before(so, dn, n, mul, b0); }
  __syncthreads();
  const u32 lane = threadIdx.x & 31, warps = gridDim.x * (blockDim.x / 32);
  for (u64 i = r0 + blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32; i < n; i += warps) {
    const u64 s = mul * so[i];
    if (s >= b1) break;
    const u64 len = mul * (dn[i + 1] - dn[i]);
    const u64 c0 = umax(s, b0), c1 = umin(s + len, b1);
    if (c0 < c1) warp_copy(tile + (mul * dn[i] + (c0 - s) - d0 + (d0 & 15)), src + c0, c1 - c0, lane);
  }
}
// the tile back to the destination [kept_before(b0), kept_before(b1)), which lies at or below b1: later tiles' sources are untouched
__global__ void k_run_scatter(const u8* __restrict__ tile, u8* __restrict__ dst, const u64* __restrict__ so, const u64* __restrict__ dn, u32 n, u32 mul, u64 b0, u64 b1) {
  __shared__ u64 d0, d1;
  if (threadIdx.x == 0) { d0 = kept_before(so, dn, n, mul, b0); d1 = kept_before(so, dn, n, mul, b1); }
  __syncthreads();
  const u64 CH = 4096, m = d1 - d0;
  const u32 lane = threadIdx.x & 31, warps = gridDim.x * (blockDim.x / 32);
  for (u64 c = blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32; c * CH < m; c += warps) warp_copy(dst + d0 + c * CH, tile + (d0 & 15) + c * CH, umin(CH, m - c * CH), lane);
}

// ---------------------------------------------------------------------------------------------- rows (rows mode)
// The grouped driver's rows (bam.cpp, nb_process_bam_cells' rows stage), restated on the device for one scoped batch.  A
// scope emits rows only when it has count rows: each count row (finalize order) whose representative exists — the last
// pair of the scope whose slot resolves to the row's callset — then a zero row for every pair whose mate slot's field 0 is
// not the sequence slot's field 0 of a representative.
struct RowDesc { u32 pair; u32 cs; i64 score; };   // cs = NONE32: a zero row
const u32 NONE = 0xFFFFFFFFu;
const u32 REASON_W = 48;                           // the reason table: 256 slots of REASON_W bytes + a length byte each

struct RowsView {
  const u32* local; const u32* idx1; const u32* idx2; const u8* f1; const u8* f2;   // the batch's pairs (from p0)
  const nb_read_result* rres; const nb_pair_result* pres;
  const char* meta; const u64* meta_off; const u32* meta_len; const u32* f0_len;
  const u32* row_scope; const u32* row_callset; const i64* row_count;
  const u32* slot_map; u64 n_slots;
  const char* feats; const u64* feat_off;
  const char* reasons; const u8* reason_len;
  u32 np;
};

// first pair in [0, n) whose batch-local scope is >= s (the pairs are in scope order)
__device__ __forceinline__ u32 lower_pair(const u32* local, u32 n, u32 s) {
  u32 lo = 0, hi = n;
  while (lo < hi) { const u32 m = (lo + hi) / 2; if (local[m] < s) lo = m + 1; else hi = m; }
  return lo;
}
__device__ __forceinline__ bool same_f0(const RowsView& v, u32 a, u32 b) {
  const u32 la = v.f0_len[a];
  if (la != v.f0_len[b]) return false;
  const char* x = v.meta + v.meta_off[a]; const char* y = v.meta + v.meta_off[b];
  for (u32 i = 0; i < la; i++) if (x[i] != y[i]) return false;
  return true;
}

// head of a scope's count rows
__global__ void k_row_heads(const u32* __restrict__ row_scope, u32* __restrict__ head, u32 n) {
  const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) head[i] = (i == 0 || row_scope[i] != row_scope[i - 1]) ? 1u : 0u;
}

// One warp per scope with count rows (u < nu, its rows [ustart[u], ustart[u + 1])): the representative of every count row
// (rep, NONE when there is none), the zero-row flag of every pair of the scope, and the number of rows it emits.
__global__ void k_rows_plan(RowsView v, const u32* __restrict__ ustart, u32 nu, u32* __restrict__ rep, u8* __restrict__ zero, u32* __restrict__ ucount) {
  const u32 u = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (u > nu) return;
  if (u == nu) { if (lane == 0) ucount[nu] = 0; return; }
  const u32 r0 = ustart[u], r1 = ustart[u + 1], s = v.row_scope[r0];
  const u32 pa = lower_pair(v.local, v.np, s), pb = lower_pair(v.local, v.np, s + 1);
  u32 n_rep = 0;
  for (u32 r = r0; r < r1; r++) {
    const u32 cs = v.row_callset[r]; u32 found = NONE;
    for (u32 top = pb; top > pa && found == NONE;) {   // 32 pairs at a time from the scope's end
      const u32 base = top - pa > 32 ? top - 32 : pa;
      bool m = false;
      if (top - 1 - lane >= base && lane < top - base) { const u32 sl = v.pres[top - 1 - lane].callset; m = sl != NONE && sl < v.n_slots && v.slot_map[sl] == cs; }
      const unsigned b = __ballot_sync(0xFFFFFFFFu, m);
      if (b) found = top - 1 - (__ffs(b) - 1);
      top = base;
    }
    if (lane == 0) rep[r] = found;
    n_rep += found != NONE;
  }
  __syncwarp();
  u32 nz = 0;
  for (u32 c0 = pa; c0 < pb; c0 += 32) {
    const u32 pj = c0 + lane; bool z = false;
    if (pj < pb) {
      z = true;
      const u32 mate = v.idx2[pj];
      for (u32 r = r0; r < r1 && z; r++) { const u32 rp = rep[r]; if (rp != NONE && same_f0(v, v.idx1[rp], mate)) z = false; }
      zero[pj] = z;
    }
    nz += __popc(__ballot_sync(0xFFFFFFFFu, z));
  }
  if (lane == 0) ucount[u] = n_rep + nz;
}

// One warp per scope with count rows: its row descriptors from out0[u] on, count rows first, then zero rows in pair order.
__global__ void k_rows_desc(RowsView v, const u32* __restrict__ ustart, const u32* __restrict__ out0, u32 nu, const u32* __restrict__ rep, const u8* __restrict__ zero, RowDesc* __restrict__ desc) {
  const u32 u = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (u >= nu) return;
  const u32 r0 = ustart[u], r1 = ustart[u + 1], s = v.row_scope[r0];
  const u32 pa = lower_pair(v.local, v.np, s), pb = lower_pair(v.local, v.np, s + 1);
  u32 j = out0[u];
  for (u32 r = r0; r < r1; r++) { const u32 rp = rep[r]; if (rp == NONE) continue; if (lane == 0) desc[j] = RowDesc{rp, v.row_callset[r], v.row_count[r]}; j++; }
  for (u32 c0 = pa; c0 < pb; c0 += 32) {
    const u32 pj = c0 + lane; const bool z = pj < pb && zero[pj];
    const unsigned b = __ballot_sync(0xFFFFFFFFu, z);
    if (z) desc[j + __popc(b & ((1u << lane) - 1))] = RowDesc{pj, NONE, 0};
    j += __popc(b);
  }
}

__device__ __forceinline__ u32 dec_len(i64 x) { u64 a = x < 0 ? (u64)(-(x + 1)) + 1 : (u64)x; u32 n = x < 0 ? 2 : 1; while (a >= 10) { a /= 10; n++; } return n; }
__device__ __forceinline__ void put_dec(char* p, i64 x, u32 n) { u64 a = x < 0 ? (u64)(-(x + 1)) + 1 : (u64)x; if (x < 0) *p = '-'; char* e = p + n; do { *--e = (char)('0' + a % 10); a /= 10; } while (a); }

// One row, as the grouped driver's emit() writes it: feats TAB score TAB M(mate) TAB skip TAB M(seq) TAB skip TAB then the
// reason / score / None / 0 columns of both reads and the triage.  WRITE = false: the length only (one thread); WRITE = true:
// the bytes at dst (one warp: long runs by warp_copy, the short fields by lane 0).
template <bool WRITE>
__device__ u64 emit_row(const RowsView& v, const RowDesc& d, char* dst, u32 lane) {
  u64 c = 0;
  auto small = [&](const char* t, u32 n) { if (WRITE && lane == 0) for (u32 k = 0; k < n; k++) dst[c + k] = t[k]; c += n; };
  auto big = [&](const char* t, u64 n) { if (WRITE) warp_copy((u8*)dst + c, (const u8*)t, n, lane); c += n; };
  auto num = [&](i64 x) { const u32 n = dec_len(x); if (WRITE && lane == 0) put_dec(dst + c, x, n); c += n; };
  auto reason = [&](u8 r) { small(v.reasons + (u64)r * REASON_W, v.reason_len[r]); };
  const u32 p = d.pair, sq = v.idx1[p], mt = v.idx2[p];
  const nb_pair_result& pr = v.pres[p]; const nb_read_result& ra = v.rres[2 * (u64)p]; const nb_read_result& rb = v.rres[2 * (u64)p + 1];
  if (d.cs != NONE) big(v.feats + v.feat_off[d.cs], v.feat_off[d.cs + 1] - v.feat_off[d.cs]);
  small("\t", 1); num(d.score); small("\t", 1);
  big(v.meta + v.meta_off[mt], v.meta_len[mt]); if (v.f2[p] & NB_FLAG_SKIP_ALIGN) small("\tTRUE\t", 6); else small("\tFALSE\t", 7);
  big(v.meta + v.meta_off[sq], v.meta_len[sq]); if (v.f1[p] & NB_FLAG_SKIP_ALIGN) small("\tTRUE\t", 6); else small("\tFALSE\t", 7);
  reason(pr.fr2); small("\t", 1); num(rb.pass ? rb.score : 0); small("\tNone\t0\t", 8);
  reason(pr.fr1); small("\t", 1); num(ra.pass ? ra.score : 0); small("\tNone\t0\t", 8);
  reason(pr.triage); small("\tNone\n", 6);
  return c;
}
// len has n + 1 entries (the last 0): an exclusive scan of it gives every row's byte offset and the total
__global__ void k_rows_len(RowsView v, const RowDesc* __restrict__ desc, u64* __restrict__ len, u32 n) {
  const u32 j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < n) len[j] = emit_row<false>(v, desc[j], nullptr, 0);
  else if (j == n) len[n] = 0;
}
// byte offset of every scope's first row (u <= nu; out0[nu] = the number of rows)
__global__ void k_rows_scope_bytes(const u32* __restrict__ out0, const u64* __restrict__ off, u64* __restrict__ ubyte, u32 nu) {
  const u32 u = blockIdx.x * blockDim.x + threadIdx.x;
  if (u <= nu) ubyte[u] = off[out0[u]];
}
// one warp per row of [j0, j1), written at off[j] - base
__global__ void k_rows_write(RowsView v, const RowDesc* __restrict__ desc, const u64* __restrict__ off, u32 j0, u32 j1, u64 base, char* __restrict__ buf) {
  const u32 j = j0 + ((blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (j < j1) emit_row<true>(v, desc[j], buf + (off[j] - base), lane);
}


}  // namespace

struct Device {
  int device = 0; cudaStream_t s = nullptr;
  Mem mem;
  // the record store (kept index = position in file order of the kept records); rows mode adds the metadata store
  Grow nib, qual, name, umi, cb, nib_off, lseq, flag, name_off, name_len, ordinal, meta, meta_off, meta_len, f0_len;
  u64 n_rec = 0, n_nib = 0, n_name = 0, n_meta = 0;
  bool rows = false;
  // staging: two slots, the producer fills one while the other's copies run
  struct Slot { Stage st; Pinned nib, qual, name, umi, cb, nib_off, lseq, flag, name_off, name_len, ordinal, meta, meta_off, meta_len, f0_len; cudaEvent_t done = nullptr; bool used = false; } slot[2];
  int cur = 0;
  // grouping
  void* g_buf = nullptr; u64 g_bytes = 0;
  u64 *o1 = nullptr, *o2 = nullptr; u32 *l1 = nullptr, *l2 = nullptr, *scope = nullptr, *idx1 = nullptr, *idx2 = nullptr, *local = nullptr; u8 *f1 = nullptr, *f2 = nullptr;
  void* p_buf = nullptr; u64 p_bytes = 0, n_pairs = 0;
  // rows (rows_begin): result buffers and plan scratch in one allocation, the row buffer, the batch's callset texts, the
  // reason strings, and two pinned buffers the chunks go to
  void* r_buf = nullptr; u64 r_bytes = 0, r_maxp = 0;
  void* rowbuf = nullptr; u64 rowbuf_cap = 0;
  void* feat = nullptr; u64 feat_cap = 0;
  void* reasons = nullptr; u64 reasons_bytes = 0;
  Pinned host[2]; int host_cur = 0;
  u64 total() const { u64 t = 0; for (const Grow* g : arrays) t += g->cap; return t; }
  // the store arrays in the order upload() grows them (the last four only in rows mode), and their bytes for R records,
  // NB nibble bytes, NM name bytes, NT metadata bytes
  enum { N_ARR = 15, N_ARR_MATRIX = 11 };
  Grow* arrays[N_ARR] = {&nib, &qual, &name, &umi, &cb, &nib_off, &lseq, &flag, &name_off, &name_len, &ordinal, &meta, &meta_off, &meta_len, &f0_len};
  int n_arr() const { return rows ? N_ARR : N_ARR_MATRIX; }
  static void needs(u64 R, u64 NB, u64 NM, u64 NT, u64 out[N_ARR]) {
    const u64 v[N_ARR] = {NB, 2 * NB, NM, 8 * R, 4 * R, 8 * R, 4 * R, 2 * R, 8 * R, R, 8 * R, NT, 8 * R, 4 * R, 4 * R};
    for (int k = 0; k < N_ARR; k++) out[k] = v[k];
  }
};

namespace {
const char* const WHAT[Device::N_ARR] = {"the nibble store", "the qual store", "the name store", "the UMI keys", "the CB ids", "the record offsets", "the record lengths", "the record flags", "the name offsets",
                                         "the name lengths", "the ordinals", "the metadata store", "the metadata offsets", "the metadata lengths", "the field-0 lengths"};

// one allocation for the sort and scope arrays: rank (ncb) | prefix (ncb) | key32 x2 (n) | val x3 (n) | umi keys x2 (n) | head, sid (n) | start (n+1) | cnt, pair0 (n+1) | scope_cb (n) | cub temp
struct GroupLayout {
  int rank_bits = 1; size_t tmp_bytes = 0, bytes = 0;
  size_t o_rank, o_pre, o_k1, o_k2, o_v0, o_v1, o_v2, o_u1, o_u2, o_head, o_sid, o_start, o_cnt, o_p0, o_scb, o_tmp;
};
inline size_t al256(size_t x) { return (x + 255) & ~(size_t)255; }
int group_layout(u32 n, u32 ncb, cudaStream_t s, GroupLayout& L) {
  while (L.rank_bits < 32 && (1ull << L.rank_bits) < ncb) L.rank_bits++;
  size_t tb_sort1 = 0, tb_sort2 = 0, tb_scan1 = 0, tb_scan2 = 0;
  GK(cub::DeviceRadixSort::SortPairs(nullptr, tb_sort1, (const u32*)nullptr, (u32*)nullptr, (const u32*)nullptr, (u32*)nullptr, (int)n, 0, L.rank_bits, s));
  GK(cub::DeviceRadixSort::SortPairs(nullptr, tb_sort2, (const u64*)nullptr, (u64*)nullptr, (const u32*)nullptr, (u32*)nullptr, (int)n, 0, 64, s));
  GK(cub::DeviceScan::InclusiveSum(nullptr, tb_scan1, (const u32*)nullptr, (u32*)nullptr, (int)n, s));
  GK(cub::DeviceScan::ExclusiveSum(nullptr, tb_scan2, (const u64*)nullptr, (u64*)nullptr, (int)n + 1, s));
  L.tmp_bytes = std::max(std::max(tb_sort1, tb_sort2), std::max(tb_scan1, tb_scan2)) + 256;
  size_t off = 0; auto take = [&](size_t bytes) { size_t o = off; off += al256(bytes); return o; };
  L.o_rank = take(4ull * ncb); L.o_pre = take(4ull * ncb); L.o_k1 = take(4ull * n); L.o_k2 = take(4ull * n); L.o_v0 = take(4ull * n); L.o_v1 = take(4ull * n); L.o_v2 = take(4ull * n);
  L.o_u1 = take(8ull * n); L.o_u2 = take(8ull * n); L.o_head = take(4ull * n); L.o_sid = take(4ull * n); L.o_start = take(4ull * (n + 1)); L.o_cnt = take(8ull * (n + 1));
  L.o_p0 = take(8ull * (n + 1)); L.o_scb = take(4ull * n); L.o_tmp = take(L.tmp_bytes);
  L.bytes = off;
  return NB_OK;
}
// the pair arrays: o1 o2 l1 l2 f1 f2 scope idx1 idx2 local, each for np pairs
struct PairLayout { size_t o[10]; size_t bytes; };
PairLayout pair_layout(u64 np) {
  PairLayout P; size_t off = 0; const u64 w[10] = {8, 8, 4, 4, 1, 1, 4, 4, 4, 4};
  for (int k = 0; k < 10; k++) { P.o[k] = off; off += al256(w[k] * np + w[k]); }
  P.bytes = off; return P;
}

// the row stage's scratch for batches of up to P pairs (at most P count rows, 2P output rows):
// rres | pres | head | uid | ustart | rep | zero | out0 | desc | len (offsets) | ubyte | cub temp
struct RowsLayout { size_t o_rres, o_pres, o_head, o_uid, o_ust, o_rep, o_zero, o_out0, o_desc, o_len, o_ub, o_tmp, tmp_bytes, bytes; };
int rows_layout(u64 P, cudaStream_t s, RowsLayout& L) {
  size_t t1 = 0, t2 = 0, t3 = 0;
  GK(cub::DeviceScan::InclusiveSum(nullptr, t1, (const u32*)nullptr, (u32*)nullptr, (int)P + 1, s));
  GK(cub::DeviceScan::ExclusiveSum(nullptr, t2, (const u32*)nullptr, (u32*)nullptr, (int)P + 2, s));
  GK(cub::DeviceScan::ExclusiveSum(nullptr, t3, (const u64*)nullptr, (u64*)nullptr, (int)(2 * P + 1), s));
  L.tmp_bytes = std::max({t1, t2, t3}) + 256;
  size_t off = 0; auto take = [&](size_t b) { const size_t o = off; off += al256(b); return o; };
  L.o_rres = take(sizeof(nb_read_result) * 2 * P); L.o_pres = take(sizeof(nb_pair_result) * P);
  L.o_head = take(4 * (P + 1)); L.o_uid = take(4 * (P + 1)); L.o_ust = take(4 * (P + 2)); L.o_rep = take(4 * P); L.o_zero = take(P);
  L.o_out0 = take(4 * (P + 2)); L.o_desc = take(sizeof(RowDesc) * 2 * P); L.o_len = take(8 * (2 * P + 1)); L.o_ub = take(8 * (P + 2)); L.o_tmp = take(L.tmp_bytes);
  L.bytes = off;
  return NB_OK;
}
// What the reserve allows for a batch's callset texts.  The texts have no bound the planning can know before the batch is
// finalized (a callset is any list of group names), so a batch whose texts pass this, like a row buffer grown for a scope
// larger than the cap, allocates beyond the reserve: still through the budget counter, and when the budget has no room
// left rows_build fails with NB_ERR_CUDA naming the bytes rather than passing it.
const u64 FEAT_ALLOWANCE = 64ull << 10;
u64 rows_reserve(Device* d, u64 P) {
  RowsLayout L;
  if (rows_layout(std::max<u64>(P, 1), d->s, L)) return ~0ull;
  return L.bytes + rows_buffer_cap() + 256 * (REASON_W + 1) + FEAT_ALLOWANCE;
}
void rows_release(Device* d) {
  d->mem.release(d->r_buf, d->r_bytes); d->r_bytes = 0; d->r_maxp = 0;
  d->mem.release(d->rowbuf, d->rowbuf_cap); d->rowbuf_cap = 0;
  d->mem.release(d->feat, d->feat_cap); d->feat_cap = 0;
}
}  // namespace

int create(int device, Device** out) {
  *out = nullptr;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || device < 0 || device >= n) { cudaGetLastError(); return fail(NB_ERR_CUDA, "no usable CUDA device " + std::to_string(device)); }
  GK(cudaSetDevice(device));
  Device* d = new Device(); d->device = device;
  if (cudaStreamCreateWithFlags(&d->s, cudaStreamNonBlocking) != cudaSuccess) { delete d; return fail(NB_ERR_CUDA, "cudaStreamCreate failed"); }
  for (auto& sl : d->slot) if (cudaEventCreateWithFlags(&sl.done, cudaEventDisableTiming) != cudaSuccess) { destroy(d); return fail(NB_ERR_CUDA, "cudaEventCreate failed"); }
  *out = d; return NB_OK;
}

void destroy(Device* d) {
  if (!d) return;
  cudaSetDevice(d->device);
  if (d->s) cudaStreamSynchronize(d->s);
  for (Grow* g : d->arrays) g->release(d->mem);
  d->mem.release(d->g_buf, d->g_bytes);
  d->mem.release(d->p_buf, d->p_bytes);
  rows_release(d); d->mem.release(d->reasons, d->reasons_bytes);
  for (auto& sl : d->slot) if (sl.done) cudaEventDestroy(sl.done);
  if (d->s) cudaStreamDestroy(d->s);
  delete d;
}

void* stream_of(Device* d) { return (void*)d->s; }
int sync(Device* d) { GK(cudaSetDevice(d->device)); GK(cudaStreamSynchronize(d->s)); return NB_OK; }
u64 store_records(Device* d) { return d->n_rec; }
u64 store_bytes(Device* d) { return d->total(); }
u64 group_bytes(Device* d) { return d->g_bytes + d->p_bytes; }
void set_budget(Device* d, u64 budget_bytes) { d->mem.budget = budget_bytes; }
void set_rows(Device* d, bool rows) { d->rows = rows; }
u64 meta_bytes(Device* d) { return d->meta.cap + d->meta_off.cap + d->meta_len.cap + d->f0_len.cap; }
u64 peak_bytes(Device* d) { return d->mem.peak; }

int begin_pass(Device* d) {
  GK(cudaSetDevice(d->device));
  GK(cudaStreamSynchronize(d->s));
  for (Grow* g : d->arrays) g->release(d->mem);
  d->mem.release(d->p_buf, d->p_bytes); d->p_bytes = 0; d->g_bytes = 0; d->n_pairs = 0;
  rows_release(d);
  d->n_rec = d->n_nib = d->n_name = d->n_meta = 0;
  return NB_OK;
}

u64 group_reserve(Device* d, u64 n, u64 ncb) {
  if (n == 0) return 0;
  GroupLayout L;
  if (group_layout((u32)n, (u32)ncb, d->s, L)) return ~0ull;
  return L.bytes + pair_layout(n).bytes + (d->rows ? rows_reserve(d, std::min<u64>(n, 1u << 20)) : 0);
}

namespace {
// upload()'s growth, array by array, on a copy of the counter
bool grows_within(Device* d, u64 R, u64 NB, u64 NM, u64 NT, u64 reserve, bool exact) {
  Mem m = d->mem;
  u64 need[Device::N_ARR]; Device::needs(R, NB, NM, NT, need);
  for (int k = 0; k < d->n_arr(); k++) {
    const u64 cap = d->arrays[k]->cap;
    if (need[k] + PAD <= cap) continue;
    const u64 w = grow_to(cap, need[k], m, reserve, exact);
    if (!w) return false;
    m.live += w - cap;
  }
  return !m.budget || m.live + reserve <= m.budget;
}
}  // namespace

// with growth slack where the budget leaves room for it, else exactly: false only when need_bytes() passes the budget
bool fits(Device* d, u64 R, u64 NB, u64 NM, u64 NT, u64 reserve) { return grows_within(d, R, NB, NM, NT, reserve, false) || grows_within(d, R, NB, NM, NT, reserve, true); }

u64 need_bytes(Device* d, u64 R, u64 NB, u64 NM, u64 NT, u64 reserve) {
  u64 need[Device::N_ARR]; Device::needs(R, NB, NM, NT, need);
  u64 live = d->mem.live, peak = live;
  for (int k = 0; k < d->n_arr(); k++) {   // each array grown to exactly what it needs, old and new copies alive at once
    const u64 cap = d->arrays[k]->cap;
    if (need[k] + PAD <= cap) continue;
    peak = std::max(peak, live + need[k] + PAD);
    live += need[k] + PAD - cap;
  }
  return std::max(peak, live + reserve);
}

int trim(Device* d) {
  GK(cudaSetDevice(d->device));
  u64 need[Device::N_ARR]; Device::needs(d->n_rec, d->n_nib, d->n_name, d->n_meta, need);
  for (int k = 0; k < d->n_arr(); k++) {
    Grow& g = *d->arrays[k];
    if (d->n_rec == 0) { g.release(d->mem); continue; }
    if (g.cap <= need[k] + PAD) continue;
    void* q = nullptr;
    if (d->mem.alloc(&q, need[k] + PAD) != cudaSuccess) { cudaGetLastError(); continue; }   // no room for the copy: keep it as it is
    if (need[k]) GK(cudaMemcpyAsync(q, g.p, need[k], cudaMemcpyDeviceToDevice, d->s));
    GK(cudaStreamSynchronize(d->s));
    d->mem.release(g.p, g.cap);
    g.p = q; g.cap = need[k] + PAD;
  }
  return NB_OK;
}

int stage(Device* d, u64 n_rec, u64 n_nib, u64 n_name, u64 n_meta, Stage*& st) {
  GK(cudaSetDevice(d->device));
  Device::Slot& sl = d->slot[d->cur];
  if (sl.used) GK(cudaEventSynchronize(sl.done));
  int e = NB_OK;
  const u64 r = std::max<u64>(n_rec, 1);
  if (!e) e = sl.nib.ensure(n_nib + 1); if (!e) e = sl.qual.ensure(2 * n_nib + 1); if (!e) e = sl.name.ensure(n_name + 1);
  if (!e) e = sl.umi.ensure(8 * r); if (!e) e = sl.cb.ensure(4 * r); if (!e) e = sl.nib_off.ensure(8 * r); if (!e) e = sl.lseq.ensure(4 * r);
  if (!e) e = sl.flag.ensure(2 * r); if (!e) e = sl.name_off.ensure(8 * r); if (!e) e = sl.name_len.ensure(r); if (!e) e = sl.ordinal.ensure(8 * r);
  if (d->rows) { if (!e) e = sl.meta.ensure(n_meta + 1); if (!e) e = sl.meta_off.ensure(8 * r); if (!e) e = sl.meta_len.ensure(4 * r); if (!e) e = sl.f0_len.ensure(4 * r); }
  if (e) return e;
  Stage& t = sl.st;
  t.rec0 = d->n_rec; t.nib0 = d->n_nib; t.name0 = d->n_name; t.meta0 = d->n_meta; t.n_rec = n_rec; t.n_nib = n_nib; t.n_name = n_name; t.n_meta = d->rows ? n_meta : 0;
  t.meta = (char*)sl.meta.p; t.meta_off = (u64*)sl.meta_off.p; t.meta_len = (u32*)sl.meta_len.p; t.f0_len = (u32*)sl.f0_len.p;
  t.nib = (u8*)sl.nib.p; t.qual = (u8*)sl.qual.p; t.name = (char*)sl.name.p; t.umi = (u64*)sl.umi.p; t.cb = (u32*)sl.cb.p; t.nib_off = (u64*)sl.nib_off.p;
  t.lseq = (u32*)sl.lseq.p; t.flag = (u16*)sl.flag.p; t.name_off = (u64*)sl.name_off.p; t.name_len = (u8*)sl.name_len.p; t.ordinal = (u64*)sl.ordinal.p;
  st = &t;
  return NB_OK;
}

int upload(Device* d, u64 reserve) {
  Device::Slot& sl = d->slot[d->cur];
  const Stage& t = sl.st;
  const u64 R = d->n_rec + t.n_rec, NB = d->n_nib + t.n_nib, NM = d->n_name + t.n_name, NT = d->n_meta + t.n_meta;
  if (R >= 0x7FFFFFFFull) return fail(NB_ERR_UNSUPPORTED, "more than 2^31 - 1 kept records");
  cudaStream_t s = d->s;
  u64 need[Device::N_ARR], keep[Device::N_ARR]; Device::needs(R, NB, NM, NT, need); Device::needs(d->n_rec, d->n_nib, d->n_name, d->n_meta, keep);
  u64 tot = 0; for (int k = 0; k < d->n_arr(); k++) tot += need[k];
  const bool exact = d->mem.budget && !grows_within(d, R, NB, NM, NT, reserve, false);   // the slack would not fit: grow exactly
  for (int k = 0; k < d->n_arr(); k++) { const int e = d->arrays[k]->ensure(need[k], keep[k], s, WHAT[k], tot, d->mem, reserve, exact); if (e) return e; }
  auto cp = [&](Grow& g, u64 at, const void* src, u64 n) -> cudaError_t { return n ? cudaMemcpyAsync((char*)g.p + at, src, n, cudaMemcpyHostToDevice, s) : cudaSuccess; };
  const u64 r0 = d->n_rec, n = t.n_rec;
  GK(cp(d->nib, d->n_nib, t.nib, t.n_nib)); GK(cp(d->qual, 2 * d->n_nib, t.qual, 2 * t.n_nib)); GK(cp(d->name, d->n_name, t.name, t.n_name));
  GK(cp(d->umi, 8 * r0, t.umi, 8 * n)); GK(cp(d->cb, 4 * r0, t.cb, 4 * n)); GK(cp(d->nib_off, 8 * r0, t.nib_off, 8 * n)); GK(cp(d->lseq, 4 * r0, t.lseq, 4 * n));
  GK(cp(d->flag, 2 * r0, t.flag, 2 * n)); GK(cp(d->name_off, 8 * r0, t.name_off, 8 * n)); GK(cp(d->name_len, r0, t.name_len, n)); GK(cp(d->ordinal, 8 * r0, t.ordinal, 8 * n));
  if (d->rows) { GK(cp(d->meta, d->n_meta, t.meta, t.n_meta)); GK(cp(d->meta_off, 8 * r0, t.meta_off, 8 * n)); GK(cp(d->meta_len, 4 * r0, t.meta_len, 4 * n)); GK(cp(d->f0_len, 4 * r0, t.f0_len, 4 * n)); }
  GK(cudaEventRecord(sl.done, s));
  sl.used = true;
  d->n_rec = R; d->n_nib = NB; d->n_name = NM; d->n_meta = NT;
  d->cur ^= 1;
  return NB_OK;
}

int compact(Device* d, u32 hi) {
  GK(cudaSetDevice(d->device));
  cudaStream_t s = d->s;
  const u32 n = (u32)d->n_rec;
  if (n == 0) return NB_OK;
  // scratch: pos (n+1) | nd (n+1) | md (n+1) | td (n+1, rows mode) | cub temp | tile; the tile takes what the budget leaves, up to 16 MB
  size_t tb32 = 0, tb64 = 0;
  GK(cub::DeviceScan::ExclusiveSum(nullptr, tb32, (u32*)nullptr, (u32*)nullptr, (int)n + 1, s));
  GK(cub::DeviceScan::ExclusiveSum(nullptr, tb64, (u64*)nullptr, (u64*)nullptr, (int)n + 1, s));
  const size_t o_pos = 0, o_nd = o_pos + al256(4ull * (n + 1)), o_md = o_nd + al256(8ull * (n + 1)), o_td = o_md + al256(8ull * (n + 1)),
               o_tmp = o_td + (d->rows ? al256(8ull * (n + 1)) : 0), o_tile = o_tmp + al256(std::max(tb32, tb64) + 256);
  const u64 room = d->mem.budget ? (d->mem.budget > d->mem.live ? d->mem.budget - d->mem.live : 0) : ~0ull;
  if (room < o_tile + 4096) return fail(NB_ERR_CUDA, "the device budget of " + std::to_string(d->mem.budget) + " bytes leaves no room to compact the record store: " + std::to_string(o_tile + 4096) + " bytes needed");
  u64 tile_bytes = std::min<u64>(16ull << 20, (room - o_tile) & ~(u64)255);
  // NB_BAM_COMPACT_TILE_BYTES caps the tile (at least 64 bytes), so that small inputs cross many tile boundaries too
  if (const char* e = getenv("NB_BAM_COMPACT_TILE_BYTES")) tile_bytes = std::min<u64>(tile_bytes, std::max<u64>(64, strtoull(e, nullptr, 10)));
  void* buf = nullptr; const u64 buf_bytes = o_tile + tile_bytes;
  if (d->mem.alloc(&buf, buf_bytes) != cudaSuccess) { cudaGetLastError(); return fail(NB_ERR_CUDA, "not enough device memory to compact the record store: " + std::to_string(buf_bytes) + " bytes needed"); }
  char* B = (char*)buf;
  u32* pos = (u32*)(B + o_pos); u64* nd = (u64*)(B + o_nd); u64* md = (u64*)(B + o_md); u64* td = d->rows ? (u64*)(B + o_td) : nullptr; void* tmp = B + o_tmp; void* tile = B + o_tile;
  int rc = NB_OK;
  auto run = [&]() -> int {
    k_keep<<<blocks((u64)n + 1), 256, 0, s>>>((const u64*)d->umi.p, (const u32*)d->lseq.p, (const u8*)d->name_len.p, d->rows ? (const u32*)d->meta_len.p : nullptr, hi, pos, nd, md, td, n);
    size_t tb = tb32; GK(cub::DeviceScan::ExclusiveSum(tmp, tb, pos, pos, (int)n + 1, s));
    tb = tb64; GK(cub::DeviceScan::ExclusiveSum(tmp, tb, nd, nd, (int)n + 1, s));
    tb = tb64; GK(cub::DeviceScan::ExclusiveSum(tmp, tb, md, md, (int)n + 1, s));
    if (td) { tb = tb64; GK(cub::DeviceScan::ExclusiveSum(tmp, tb, td, td, (int)n + 1, s)); }
    u32 keep_rec = 0; u64 keep_nib = 0, keep_name = 0, keep_meta = 0;
    GK(cudaMemcpyAsync(&keep_rec, pos + n, 4, cudaMemcpyDeviceToHost, s)); GK(cudaMemcpyAsync(&keep_nib, nd + n, 8, cudaMemcpyDeviceToHost, s)); GK(cudaMemcpyAsync(&keep_name, md + n, 8, cudaMemcpyDeviceToHost, s));
    if (td) GK(cudaMemcpyAsync(&keep_meta, td + n, 8, cudaMemcpyDeviceToHost, s));
    GK(cudaStreamSynchronize(s));
    // the byte runs first (they read the old offsets): nibbles, quals at twice the nibble offsets, names
    auto runs = [&](Grow& g, const Grow& off, const u64* dn, u32 mul, u64 total) {
      const u64 span = tile_bytes - 16;   // the tile's first (d0 & 15) bytes stay unused
      for (u64 b0 = 0; b0 < total; b0 += span) {
        const u64 b1 = std::min(total, b0 + span);
        k_run_gather<<<1024, 256, 0, s>>>((const u8*)g.p, (u8*)tile, (const u64*)off.p, dn, n, mul, b0, b1);
        k_run_scatter<<<256, 256, 0, s>>>((const u8*)tile, (u8*)g.p, (const u64*)off.p, dn, n, mul, b0, b1);
      }
    };
    runs(d->nib, d->nib_off, nd, 1, d->n_nib); runs(d->qual, d->nib_off, nd, 2, 2 * d->n_nib); runs(d->name, d->name_off, md, 1, d->n_name);
    if (td) runs(d->meta, d->meta_off, td, 1, d->n_meta);
    // then the per-record arrays, the offsets rebased to the scans
    auto recs = [&](auto* tag, const void* src, Grow& dst) {
      using T = std::remove_pointer_t<decltype(tag)>;
      const u32 per = (u32)std::min<u64>(tile_bytes / sizeof(T), 1u << 30);
      for (u64 t0 = 0; t0 < n; t0 += per) {
        const u32 t1 = (u32)std::min<u64>(t0 + per, n);
        k_rec_gather<T><<<blocks(t1 - t0), 256, 0, s>>>((const T*)src, pos, (T*)tile, (u32)t0, t1);
        k_rec_scatter<T><<<blocks(t1 - t0), 256, 0, s>>>((const T*)tile, pos, (T*)dst.p, (u32)t0, t1);
      }
    };
    recs((u64*)nullptr, d->umi.p, d->umi); recs((u32*)nullptr, d->cb.p, d->cb); recs((u64*)nullptr, nd, d->nib_off); recs((u32*)nullptr, d->lseq.p, d->lseq);
    recs((u16*)nullptr, d->flag.p, d->flag); recs((u64*)nullptr, md, d->name_off); recs((u8*)nullptr, d->name_len.p, d->name_len); recs((u64*)nullptr, d->ordinal.p, d->ordinal);
    if (td) { recs((u64*)nullptr, td, d->meta_off); recs((u32*)nullptr, d->meta_len.p, d->meta_len); recs((u32*)nullptr, d->f0_len.p, d->f0_len); }
    GK(cudaGetLastError());
    GK(cudaStreamSynchronize(s));
    d->n_rec = keep_rec; d->n_nib = keep_nib; d->n_name = keep_name; d->n_meta = keep_meta;
    return NB_OK;
  };
  rc = run();
  d->mem.release(buf, buf_bytes);
  return rc;
}

int group(Device* d, const std::vector<u32>& cb_rank, const std::vector<u32>& cb_prefix, Grouped& g) {
  GK(cudaSetDevice(d->device));
  cudaStream_t s = d->s;
  const u32 n = (u32)d->n_rec;
  g.n_records = n; g.n_scopes = 0; g.n_pairs = 0; g.scope_pair0.assign(1, 0); g.scope_cb.clear();
  if (n == 0) return NB_OK;
  const u32 ncb = (u32)cb_rank.size();
  GroupLayout L;
  if (int e = group_layout(n, ncb, s, L)) return e;
  const size_t tmp_bytes = L.tmp_bytes;
  d->mem.release(d->g_buf, d->g_bytes); d->g_bytes = 0;
  if (d->mem.alloc(&d->g_buf, L.bytes) != cudaSuccess) { cudaGetLastError(); d->g_buf = nullptr; return fail(NB_ERR_CUDA, "not enough device memory to group the records: " + std::to_string(L.bytes) + " bytes needed"); }
  d->g_bytes = L.bytes;
  char* B = (char*)d->g_buf;
  u32* rank = (u32*)(B + L.o_rank); u32* pre = (u32*)(B + L.o_pre); u32* k1 = (u32*)(B + L.o_k1); u32* k2 = (u32*)(B + L.o_k2);
  u32* v0 = (u32*)(B + L.o_v0); u32* v1 = (u32*)(B + L.o_v1); u32* perm = (u32*)(B + L.o_v2); u64* u1 = (u64*)(B + L.o_u1); u64* u2 = (u64*)(B + L.o_u2);
  u32* head = (u32*)(B + L.o_head); u32* sid = (u32*)(B + L.o_sid); u32* start = (u32*)(B + L.o_start); u64* cnt = (u64*)(B + L.o_cnt); u64* pair0 = (u64*)(B + L.o_p0);
  u32* scb = (u32*)(B + L.o_scb); void* tmp = B + L.o_tmp;
  if (ncb) { GK(cudaMemcpyAsync(rank, cb_rank.data(), 4ull * ncb, cudaMemcpyHostToDevice, s)); GK(cudaMemcpyAsync(pre, cb_prefix.data(), 4ull * ncb, cudaMemcpyHostToDevice, s)); }
  // (UMI, CB rank, ordinal): stable sort by CB rank, then stable sort by UMI key
  k_cb_keys<<<blocks(n), 256, 0, s>>>((const u32*)d->cb.p, rank, k1, v0, n);
  size_t tb = tmp_bytes;
  GK(cub::DeviceRadixSort::SortPairs(tmp, tb, k1, k2, v0, v1, (int)n, 0, L.rank_bits, s));
  k_umi_gather<<<blocks(n), 256, 0, s>>>((const u64*)d->umi.p, v1, u1, n);
  tb = tmp_bytes;
  GK(cub::DeviceRadixSort::SortPairs(tmp, tb, u1, u2, v1, perm, (int)n, 0, 63, s));
  // scopes
  k_heads<<<blocks(n), 256, 0, s>>>(u2, perm, (const u32*)d->cb.p, pre, head, n);
  tb = tmp_bytes;
  GK(cub::DeviceScan::InclusiveSum(tmp, tb, head, sid, (int)n, s));
  k_starts<<<blocks(n), 256, 0, s>>>(head, sid, start, n);
  u32 n_scopes = 0;
  GK(cudaMemcpyAsync(&n_scopes, sid + n - 1, 4, cudaMemcpyDeviceToHost, s));
  GK(cudaStreamSynchronize(s));
  // pairs: count, scan, write
  Recs R{perm, (const u64*)d->nib_off.p, (const u32*)d->lseq.p, (const u16*)d->flag.p, (const u64*)d->name_off.p, (const u8*)d->name_len.p, (const char*)d->name.p, (const u32*)d->cb.p};
  k_pair_count<<<blocks((u64)n_scopes + 1, 128), 128, 0, s>>>(R, start, cnt, scb, n_scopes);
  tb = tmp_bytes;
  GK(cub::DeviceScan::ExclusiveSum(tmp, tb, cnt, pair0, (int)n_scopes + 1, s));
  g.n_scopes = n_scopes;
  g.scope_pair0.resize((size_t)n_scopes + 1); g.scope_cb.resize(n_scopes);
  GK(cudaMemcpyAsync(g.scope_pair0.data(), pair0, 8ull * (n_scopes + 1), cudaMemcpyDeviceToHost, s));
  GK(cudaMemcpyAsync(g.scope_cb.data(), scb, 4ull * n_scopes, cudaMemcpyDeviceToHost, s));
  GK(cudaStreamSynchronize(s));
  const u64 np = g.n_pairs = g.scope_pair0[n_scopes];
  d->n_pairs = np;
  d->mem.release(d->p_buf, d->p_bytes); d->p_bytes = 0;
  const PairLayout P = pair_layout(np);
  if (d->mem.alloc(&d->p_buf, P.bytes) != cudaSuccess) { cudaGetLastError(); d->p_buf = nullptr; return fail(NB_ERR_CUDA, "not enough device memory for the pairs: " + std::to_string(P.bytes) + " bytes needed"); }
  d->p_bytes = P.bytes;
  char* Q = (char*)d->p_buf;
  d->o1 = (u64*)(Q + P.o[0]); d->o2 = (u64*)(Q + P.o[1]); d->l1 = (u32*)(Q + P.o[2]); d->l2 = (u32*)(Q + P.o[3]); d->f1 = (u8*)(Q + P.o[4]); d->f2 = (u8*)(Q + P.o[5]);
  d->scope = (u32*)(Q + P.o[6]); d->idx1 = (u32*)(Q + P.o[7]); d->idx2 = (u32*)(Q + P.o[8]); d->local = (u32*)(Q + P.o[9]);
  PairsOut out{d->o1, d->o2, d->l1, d->l2, d->f1, d->f2, d->scope, d->idx1, d->idx2};
  if (np) k_pair_write<<<blocks(n_scopes, 128), 128, 0, s>>>(R, start, pair0, out, n_scopes);
  GK(cudaGetLastError());
  GK(cudaStreamSynchronize(s));
  // the sort and scope arrays are not needed any more: the batches only read the store and the pair arrays
  { const u64 gb = d->g_bytes; d->mem.release(d->g_buf, gb); }
  return NB_OK;
}

int batch(Device* d, u64 p0, u64 p1, u64 scope0, u32 max_read_len, nb_batch& b) {
  memset(&b, 0, sizeof b);
  const u64 np = p1 - p0;
  if (np) k_local_scope<<<(u32)((np + 255) / 256), 256, 0, d->s>>>(d->scope + p0, d->local + p0, np, (u32)scope0);
  GK(cudaGetLastError());
  b.n_pairs = np; b.location = NB_MEM_DEVICE; b.max_read_len = max_read_len; b.encoding = NB_SEQ_BAM4;
  b.r1 = b.r2 = (const u8*)d->nib.p; b.q1 = b.q2 = (const u8*)d->qual.p;
  b.r1_off = d->o1 + p0; b.r2_off = d->o2 + p0; b.r1_len = d->l1 + p0; b.r2_len = d->l2 + p0;
  b.flags1 = d->f1 + p0; b.flags2 = d->f2 + p0; b.scope_id = d->local + p0;
  return NB_OK;
}

int pairs_to_host(Device* d, std::vector<u64>& ord1, std::vector<u64>& ord2, std::vector<u8>& f1, std::vector<u8>& f2, std::vector<u32>& l1, std::vector<u32>& l2) {
  GK(cudaSetDevice(d->device));
  const u64 np = d->n_pairs; cudaStream_t s = d->s;
  std::vector<u32> i1(np), i2(np); std::vector<u64> ord(d->n_rec);
  f1.resize(np); f2.resize(np); l1.resize(np); l2.resize(np); ord1.resize(np); ord2.resize(np);
  if (np) {
    GK(cudaMemcpyAsync(i1.data(), d->idx1, 4 * np, cudaMemcpyDeviceToHost, s)); GK(cudaMemcpyAsync(i2.data(), d->idx2, 4 * np, cudaMemcpyDeviceToHost, s));
    GK(cudaMemcpyAsync(f1.data(), d->f1, np, cudaMemcpyDeviceToHost, s)); GK(cudaMemcpyAsync(f2.data(), d->f2, np, cudaMemcpyDeviceToHost, s));
    GK(cudaMemcpyAsync(l1.data(), d->l1, 4 * np, cudaMemcpyDeviceToHost, s)); GK(cudaMemcpyAsync(l2.data(), d->l2, 4 * np, cudaMemcpyDeviceToHost, s));
  }
  if (d->n_rec) GK(cudaMemcpyAsync(ord.data(), d->ordinal.p, 8 * d->n_rec, cudaMemcpyDeviceToHost, s));
  GK(cudaStreamSynchronize(s));
  for (u64 p = 0; p < np; p++) { ord1[p] = ord[i1[p]]; ord2[p] = ord[i2[p]]; }
  return NB_OK;
}

int slots_to_host(Device* d, std::vector<u64>& off1, std::vector<u64>& off2, std::vector<u8>& nib, std::vector<u8>& qual) {
  GK(cudaSetDevice(d->device));
  const u64 np = d->n_pairs; cudaStream_t s = d->s;
  off1.resize(np); off2.resize(np); nib.resize(d->n_nib); qual.resize(2 * d->n_nib);
  if (np) { GK(cudaMemcpyAsync(off1.data(), d->o1, 8 * np, cudaMemcpyDeviceToHost, s)); GK(cudaMemcpyAsync(off2.data(), d->o2, 8 * np, cudaMemcpyDeviceToHost, s)); }
  if (d->n_nib) { GK(cudaMemcpyAsync(nib.data(), d->nib.p, d->n_nib, cudaMemcpyDeviceToHost, s)); GK(cudaMemcpyAsync(qual.data(), d->qual.p, 2 * d->n_nib, cudaMemcpyDeviceToHost, s)); }
  GK(cudaStreamSynchronize(s));
  return NB_OK;
}

u64 rows_buffer_cap() {
  if (const char* e = getenv("NB_BAM_ROWS_BUFFER_KB")) return std::max<u64>(strtoull(e, nullptr, 10), 1) << 10;
  return 64ull << 20;
}

int rows_begin(Device* d, u64 max_batch_pairs) {
  GK(cudaSetDevice(d->device));
  const u64 P = std::max<u64>(max_batch_pairs, 1);
  if (P > 0x7FFFFFFFull) return fail(NB_ERR_UNSUPPORTED, "a batch of more than 2^31 - 1 pairs");
  RowsLayout L; if (int e = rows_layout(P, d->s, L)) return e;
  if (d->r_maxp < P) {
    d->mem.release(d->r_buf, d->r_bytes); d->r_bytes = 0; d->r_maxp = 0;
    if (d->mem.alloc(&d->r_buf, L.bytes) != cudaSuccess) { cudaGetLastError(); d->r_buf = nullptr; return fail(NB_ERR_CUDA, "not enough device memory for the row stage of batches of " + std::to_string(P) + " pairs: " + std::to_string(L.bytes) + " bytes needed"); }
    d->r_bytes = L.bytes; d->r_maxp = P;
  }
  if (!d->rowbuf) {
    const u64 cap = rows_buffer_cap();
    if (d->mem.alloc(&d->rowbuf, cap) != cudaSuccess) { cudaGetLastError(); d->rowbuf = nullptr; return fail(NB_ERR_CUDA, "not enough device memory for the row buffer: " + std::to_string(cap) + " bytes needed"); }
    d->rowbuf_cap = cap;
  }
  return NB_OK;
}

void rows_results(Device* d, nb_read_result** rres, nb_pair_result** pres) {
  RowsLayout L; rows_layout(std::max<u64>(d->r_maxp, 1), d->s, L);
  *rres = (nb_read_result*)((char*)d->r_buf + L.o_rres); *pres = (nb_pair_result*)((char*)d->r_buf + L.o_pres);
}

int rows_build(Device* d, const RowsBatch& B, const std::function<int(const char*, u64)>& sink, RowsStats& st) {
  auto now = []() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  GK(cudaSetDevice(d->device));
  const u64 np = B.p1 - B.p0, n_rows = B.n_rows;
  if (!np || !n_rows) return NB_OK;   // no count row: the batch emits nothing
  if (np > d->r_maxp) return fail(NB_ERR_INVALID, "rows_build: a batch larger than rows_begin's");
  double t0 = now(), t_sink = 0;
  cudaStream_t s = d->s;
  RowsLayout L; if (int e = rows_layout(d->r_maxp, s, L)) return e;
  char* W = (char*)d->r_buf;
  // the reason strings once, the batch's callset texts every batch
  if (!d->reasons) {
    std::vector<char> t(256 * (REASON_W + 1), 0);
    for (int r = 0; r < 256; r++) { const std::string& x = (*B.reasons)[r]; const u32 n = (u32)std::min<size_t>(x.size(), REASON_W); memcpy(&t[r * REASON_W], x.data(), n); t[256 * REASON_W + r] = (char)n; }
    if (d->mem.alloc(&d->reasons, t.size()) != cudaSuccess) { cudaGetLastError(); d->reasons = nullptr; return fail(NB_ERR_CUDA, "not enough device memory for the reason strings"); }
    d->reasons_bytes = t.size();
    GK(cudaMemcpyAsync(d->reasons, t.data(), t.size(), cudaMemcpyHostToDevice, s));
    GK(cudaStreamSynchronize(s));
  }
  const std::vector<u64>& fo = *B.feat_off;
  const u64 fo_at = al256(B.feats->size() + 1), feat_need = fo_at + 8 * fo.size();
  if (d->feat_cap < feat_need) {
    d->mem.release(d->feat, d->feat_cap); d->feat_cap = 0;
    if (d->mem.alloc(&d->feat, feat_need) != cudaSuccess) { cudaGetLastError(); d->feat = nullptr; return fail(NB_ERR_CUDA, "the callset texts of a batch (" + std::to_string(feat_need) + " bytes) do not fit the device" + (d->mem.budget ? " budget of " + std::to_string(d->mem.budget) + " bytes" : std::string(" memory"))); }
    d->feat_cap = feat_need;
  }
  if (!B.feats->empty()) GK(cudaMemcpyAsync(d->feat, B.feats->data(), B.feats->size(), cudaMemcpyHostToDevice, s));
  GK(cudaMemcpyAsync((char*)d->feat + fo_at, fo.data(), 8 * fo.size(), cudaMemcpyHostToDevice, s));
  RowsView v;
  v.local = d->local + B.p0; v.idx1 = d->idx1 + B.p0; v.idx2 = d->idx2 + B.p0; v.f1 = d->f1 + B.p0; v.f2 = d->f2 + B.p0;
  v.rres = (const nb_read_result*)(W + L.o_rres); v.pres = (const nb_pair_result*)(W + L.o_pres);
  v.meta = (const char*)d->meta.p; v.meta_off = (const u64*)d->meta_off.p; v.meta_len = (const u32*)d->meta_len.p; v.f0_len = (const u32*)d->f0_len.p;
  v.row_scope = (const u32*)B.row_scope; v.row_callset = (const u32*)B.row_callset; v.row_count = (const i64*)B.row_count;
  v.slot_map = (const u32*)B.slot_map; v.n_slots = B.n_slots;
  v.feats = (const char*)d->feat; v.feat_off = (const u64*)((char*)d->feat + fo_at);
  v.reasons = (const char*)d->reasons; v.reason_len = (const u8*)d->reasons + 256 * REASON_W;
  v.np = (u32)np;
  u32* head = (u32*)(W + L.o_head); u32* uid = (u32*)(W + L.o_uid); u32* ustart = (u32*)(W + L.o_ust); u32* rep = (u32*)(W + L.o_rep); u8* zero = (u8*)(W + L.o_zero);
  u32* out0 = (u32*)(W + L.o_out0); RowDesc* desc = (RowDesc*)(W + L.o_desc); u64* len = (u64*)(W + L.o_len); u64* ubyte = (u64*)(W + L.o_ub); void* tmp = W + L.o_tmp;
  const u32 nr = (u32)n_rows;
  // the scopes with count rows
  k_row_heads<<<blocks(nr), 256, 0, s>>>(v.row_scope, head, nr);
  size_t tb = L.tmp_bytes; GK(cub::DeviceScan::InclusiveSum(tmp, tb, head, uid, (int)nr, s));
  k_starts<<<blocks(nr), 256, 0, s>>>(head, uid, ustart, nr);
  u32 nu = 0;
  GK(cudaMemcpyAsync(&nu, uid + nr - 1, 4, cudaMemcpyDeviceToHost, s));
  GK(cudaStreamSynchronize(s));
  // representatives and zero rows, then every row's descriptor, byte length and offset
  k_rows_plan<<<blocks(32ull * (nu + 1), 128), 128, 0, s>>>(v, ustart, nu, rep, zero, out0);
  tb = L.tmp_bytes; GK(cub::DeviceScan::ExclusiveSum(tmp, tb, out0, out0, (int)nu + 1, s));
  k_rows_desc<<<blocks(32ull * nu, 128), 128, 0, s>>>(v, ustart, out0, nu, rep, zero, desc);
  u32 nout = 0;
  GK(cudaMemcpyAsync(&nout, out0 + nu, 4, cudaMemcpyDeviceToHost, s));
  GK(cudaStreamSynchronize(s));
  k_rows_len<<<blocks((u64)nout + 1), 256, 0, s>>>(v, desc, len, nout);
  tb = L.tmp_bytes; GK(cub::DeviceScan::ExclusiveSum(tmp, tb, len, len, (int)nout + 1, s));
  k_rows_scope_bytes<<<blocks((u64)nu + 1), 256, 0, s>>>(out0, len, ubyte, nu);
  std::vector<u64> hb(nu + 1); std::vector<u32> hr(nu + 1);
  GK(cudaMemcpyAsync(hb.data(), ubyte, 8ull * (nu + 1), cudaMemcpyDeviceToHost, s)); GK(cudaMemcpyAsync(hr.data(), out0, 4ull * (nu + 1), cudaMemcpyDeviceToHost, s));
  GK(cudaGetLastError());
  GK(cudaStreamSynchronize(s));
  // chunks of whole scopes within the row buffer; a scope larger than the buffer gets a chunk of its own in a grown buffer
  const u64 cap = rows_buffer_cap(); u64 chunks = 0;
  for (u32 a = 0; a < nu;) {
    u32 b = a + 1;
    while (b < nu && hb[b + 1] - hb[a] <= cap) b++;
    const u64 bytes = hb[b] - hb[a];
    if (bytes > d->rowbuf_cap) {
      d->mem.release(d->rowbuf, d->rowbuf_cap); d->rowbuf_cap = 0;
      if (d->mem.alloc(&d->rowbuf, bytes) != cudaSuccess) { cudaGetLastError(); d->rowbuf = nullptr; return fail(NB_ERR_CUDA, "the rows of one scope (" + std::to_string(bytes) + " bytes) do not fit the device" + (d->mem.budget ? " budget of " + std::to_string(d->mem.budget) + " bytes" : std::string(" memory"))); }
      d->rowbuf_cap = bytes;
    }
    if (bytes) {
      const u32 j0 = hr[a], j1 = hr[b];
      k_rows_write<<<blocks(32ull * (j1 - j0), 128), 128, 0, s>>>(v, desc, len, j0, j1, hb[a], (char*)d->rowbuf);
      Pinned& h = d->host[d->host_cur];
      if (int e = h.ensure(bytes)) return e;
      GK(cudaMemcpyAsync(h.p, d->rowbuf, bytes, cudaMemcpyDeviceToHost, s));
      GK(cudaGetLastError());
      GK(cudaStreamSynchronize(s));
      const double ts = now();
      if (int e = sink((const char*)h.p, bytes)) return e;
      t_sink += now() - ts;
      d->host_cur ^= 1; chunks++;
    }
    a = b;
  }
  st.rows += nout; st.bytes += hb[nu]; st.chunks += chunks; st.batches++; st.max_chunks = std::max(st.max_chunks, chunks);
  st.t_device += now() - t0 - t_sink;
  return NB_OK;
}

}  // namespace nbg
