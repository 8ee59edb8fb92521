// bam_group.cu — BAM mode in any record order: the device record store and the (UMI, CB) grouping (bam_group.hpp).
//
// The host producer (bam.cpp) stages every kept record of a window and this file uploads it into HBM.  At the end of the
// file the records are put in (UMI, full CB, ordinal) order by two stable CUB radix sorts (CB rank, then UMI key, ordinals
// as values), a scope starts wherever (UMI, CB[..len-2]) changes, and one thread per scope restates
// SortedBamReader::add_dummy_paired_reads + filter_paired_reads (src/parse/sorted_bam_reader.rs:109-162) over the scope's
// records in that order: a count pass, a scan, a write pass.  Pairs are (base offset, clipped length, flags) into the store,
// so no bases move: the scoped batches handed to nb_align_batch are NB_MEM_DEVICE views of the store.  Under a device
// budget every allocation here is counted against it, and compact() drops the records of the UMI buckets a pass gives up.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <algorithm>
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
__global__ void k_keep(const u64* __restrict__ umi, const u32* __restrict__ lseq, const u8* __restrict__ name_len, u32 hi, u32* __restrict__ pos, u64* __restrict__ nd, u64* __restrict__ md, u32 n) {
  const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i > n) return;
  const bool k = i < n && umi_bucket(umi[i]) < hi;
  pos[i] = k; nd[i] = k ? (lseq[i] + 1) / 2 : 0; md[i] = k ? name_len[i] : 0;
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


}  // namespace

struct Device {
  int device = 0; cudaStream_t s = nullptr;
  Mem mem;
  // the record store (kept index = position in file order of the kept records)
  Grow nib, qual, name, umi, cb, nib_off, lseq, flag, name_off, name_len, ordinal;
  u64 n_rec = 0, n_nib = 0, n_name = 0;
  // staging: two slots, the producer fills one while the other's copies run
  struct Slot { Stage st; Pinned nib, qual, name, umi, cb, nib_off, lseq, flag, name_off, name_len, ordinal; cudaEvent_t done = nullptr; bool used = false; } slot[2];
  int cur = 0;
  // grouping
  void* g_buf = nullptr; u64 g_bytes = 0;
  u64 *o1 = nullptr, *o2 = nullptr; u32 *l1 = nullptr, *l2 = nullptr, *scope = nullptr, *idx1 = nullptr, *idx2 = nullptr, *local = nullptr; u8 *f1 = nullptr, *f2 = nullptr;
  void* p_buf = nullptr; u64 p_bytes = 0, n_pairs = 0;
  u64 total() const { return nib.cap + qual.cap + name.cap + umi.cap + cb.cap + nib_off.cap + lseq.cap + flag.cap + name_off.cap + name_len.cap + ordinal.cap; }
  // the store arrays in the order upload() grows them, and their bytes for R records, NB nibble bytes, NM name bytes
  Grow* arrays[11] = {&nib, &qual, &name, &umi, &cb, &nib_off, &lseq, &flag, &name_off, &name_len, &ordinal};
  static void needs(u64 R, u64 NB, u64 NM, u64 out[11]) {
    const u64 v[11] = {NB, 2 * NB, NM, 8 * R, 4 * R, 8 * R, 4 * R, 2 * R, 8 * R, R, 8 * R};
    for (int k = 0; k < 11; k++) out[k] = v[k];
  }
};

namespace {
const char* const WHAT[11] = {"the nibble store", "the qual store", "the name store", "the UMI keys", "the CB ids", "the record offsets", "the record lengths", "the record flags", "the name offsets", "the name lengths", "the ordinals"};

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
u64 peak_bytes(Device* d) { return d->mem.peak; }

int begin_pass(Device* d) {
  GK(cudaSetDevice(d->device));
  GK(cudaStreamSynchronize(d->s));
  for (Grow* g : d->arrays) g->release(d->mem);
  d->mem.release(d->p_buf, d->p_bytes); d->p_bytes = 0; d->g_bytes = 0; d->n_pairs = 0;
  d->n_rec = d->n_nib = d->n_name = 0;
  return NB_OK;
}

u64 group_reserve(Device* d, u64 n, u64 ncb) {
  if (n == 0) return 0;
  GroupLayout L;
  if (group_layout((u32)n, (u32)ncb, d->s, L)) return ~0ull;
  return L.bytes + pair_layout(n).bytes;
}

namespace {
// upload()'s growth, array by array, on a copy of the counter
bool grows_within(Device* d, u64 R, u64 NB, u64 NM, u64 reserve, bool exact) {
  Mem m = d->mem;
  u64 need[11]; Device::needs(R, NB, NM, need);
  for (int k = 0; k < 11; k++) {
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
bool fits(Device* d, u64 R, u64 NB, u64 NM, u64 reserve) { return grows_within(d, R, NB, NM, reserve, false) || grows_within(d, R, NB, NM, reserve, true); }

u64 need_bytes(Device* d, u64 R, u64 NB, u64 NM, u64 reserve) {
  u64 need[11]; Device::needs(R, NB, NM, need);
  u64 live = d->mem.live, peak = live;
  for (int k = 0; k < 11; k++) {   // each array grown to exactly what it needs, old and new copies alive at once
    const u64 cap = d->arrays[k]->cap;
    if (need[k] + PAD <= cap) continue;
    peak = std::max(peak, live + need[k] + PAD);
    live += need[k] + PAD - cap;
  }
  return std::max(peak, live + reserve);
}

int trim(Device* d) {
  GK(cudaSetDevice(d->device));
  u64 need[11]; Device::needs(d->n_rec, d->n_nib, d->n_name, need);
  for (int k = 0; k < 11; k++) {
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

int stage(Device* d, u64 n_rec, u64 n_nib, u64 n_name, Stage*& st) {
  GK(cudaSetDevice(d->device));
  Device::Slot& sl = d->slot[d->cur];
  if (sl.used) GK(cudaEventSynchronize(sl.done));
  int e = NB_OK;
  const u64 r = std::max<u64>(n_rec, 1);
  if (!e) e = sl.nib.ensure(n_nib + 1); if (!e) e = sl.qual.ensure(2 * n_nib + 1); if (!e) e = sl.name.ensure(n_name + 1);
  if (!e) e = sl.umi.ensure(8 * r); if (!e) e = sl.cb.ensure(4 * r); if (!e) e = sl.nib_off.ensure(8 * r); if (!e) e = sl.lseq.ensure(4 * r);
  if (!e) e = sl.flag.ensure(2 * r); if (!e) e = sl.name_off.ensure(8 * r); if (!e) e = sl.name_len.ensure(r); if (!e) e = sl.ordinal.ensure(8 * r);
  if (e) return e;
  Stage& t = sl.st;
  t.rec0 = d->n_rec; t.nib0 = d->n_nib; t.name0 = d->n_name; t.n_rec = n_rec; t.n_nib = n_nib; t.n_name = n_name;
  t.nib = (u8*)sl.nib.p; t.qual = (u8*)sl.qual.p; t.name = (char*)sl.name.p; t.umi = (u64*)sl.umi.p; t.cb = (u32*)sl.cb.p; t.nib_off = (u64*)sl.nib_off.p;
  t.lseq = (u32*)sl.lseq.p; t.flag = (u16*)sl.flag.p; t.name_off = (u64*)sl.name_off.p; t.name_len = (u8*)sl.name_len.p; t.ordinal = (u64*)sl.ordinal.p;
  st = &t;
  return NB_OK;
}

int upload(Device* d, u64 reserve) {
  Device::Slot& sl = d->slot[d->cur];
  const Stage& t = sl.st;
  const u64 R = d->n_rec + t.n_rec, NB = d->n_nib + t.n_nib, NM = d->n_name + t.n_name;
  if (R >= 0x7FFFFFFFull) return fail(NB_ERR_UNSUPPORTED, "more than 2^31 - 1 kept records");
  cudaStream_t s = d->s;
  const u64 tot = NB + 2 * NB + NM + R * (8 + 4 + 8 + 4 + 2 + 8 + 1 + 8);
  u64 need[11], keep[11]; Device::needs(R, NB, NM, need); Device::needs(d->n_rec, d->n_nib, d->n_name, keep);
  const bool exact = d->mem.budget && !grows_within(d, R, NB, NM, reserve, false);   // the slack would not fit: grow exactly
  for (int k = 0; k < 11; k++) { const int e = d->arrays[k]->ensure(need[k], keep[k], s, WHAT[k], tot, d->mem, reserve, exact); if (e) return e; }
  auto cp = [&](Grow& g, u64 at, const void* src, u64 n) -> cudaError_t { return n ? cudaMemcpyAsync((char*)g.p + at, src, n, cudaMemcpyHostToDevice, s) : cudaSuccess; };
  const u64 r0 = d->n_rec, n = t.n_rec;
  GK(cp(d->nib, d->n_nib, t.nib, t.n_nib)); GK(cp(d->qual, 2 * d->n_nib, t.qual, 2 * t.n_nib)); GK(cp(d->name, d->n_name, t.name, t.n_name));
  GK(cp(d->umi, 8 * r0, t.umi, 8 * n)); GK(cp(d->cb, 4 * r0, t.cb, 4 * n)); GK(cp(d->nib_off, 8 * r0, t.nib_off, 8 * n)); GK(cp(d->lseq, 4 * r0, t.lseq, 4 * n));
  GK(cp(d->flag, 2 * r0, t.flag, 2 * n)); GK(cp(d->name_off, 8 * r0, t.name_off, 8 * n)); GK(cp(d->name_len, r0, t.name_len, n)); GK(cp(d->ordinal, 8 * r0, t.ordinal, 8 * n));
  GK(cudaEventRecord(sl.done, s));
  sl.used = true;
  d->n_rec = R; d->n_nib = NB; d->n_name = NM;
  d->cur ^= 1;
  return NB_OK;
}

int compact(Device* d, u32 hi) {
  GK(cudaSetDevice(d->device));
  cudaStream_t s = d->s;
  const u32 n = (u32)d->n_rec;
  if (n == 0) return NB_OK;
  // scratch: pos (n+1) | nd (n+1) | md (n+1) | cub temp | tile; the tile takes what the budget leaves, up to 16 MB
  size_t tb32 = 0, tb64 = 0;
  GK(cub::DeviceScan::ExclusiveSum(nullptr, tb32, (u32*)nullptr, (u32*)nullptr, (int)n + 1, s));
  GK(cub::DeviceScan::ExclusiveSum(nullptr, tb64, (u64*)nullptr, (u64*)nullptr, (int)n + 1, s));
  const size_t o_pos = 0, o_nd = o_pos + al256(4ull * (n + 1)), o_md = o_nd + al256(8ull * (n + 1)), o_tmp = o_md + al256(8ull * (n + 1)), o_tile = o_tmp + al256(std::max(tb32, tb64) + 256);
  const u64 room = d->mem.budget ? (d->mem.budget > d->mem.live ? d->mem.budget - d->mem.live : 0) : ~0ull;
  if (room < o_tile + 4096) return fail(NB_ERR_CUDA, "the device budget of " + std::to_string(d->mem.budget) + " bytes leaves no room to compact the record store: " + std::to_string(o_tile + 4096) + " bytes needed");
  u64 tile_bytes = std::min<u64>(16ull << 20, (room - o_tile) & ~(u64)255);
  // NB_BAM_COMPACT_TILE_BYTES caps the tile (at least 64 bytes), so that small inputs cross many tile boundaries too
  if (const char* e = getenv("NB_BAM_COMPACT_TILE_BYTES")) tile_bytes = std::min<u64>(tile_bytes, std::max<u64>(64, strtoull(e, nullptr, 10)));
  void* buf = nullptr; const u64 buf_bytes = o_tile + tile_bytes;
  if (d->mem.alloc(&buf, buf_bytes) != cudaSuccess) { cudaGetLastError(); return fail(NB_ERR_CUDA, "not enough device memory to compact the record store: " + std::to_string(buf_bytes) + " bytes needed"); }
  char* B = (char*)buf;
  u32* pos = (u32*)(B + o_pos); u64* nd = (u64*)(B + o_nd); u64* md = (u64*)(B + o_md); void* tmp = B + o_tmp; void* tile = B + o_tile;
  int rc = NB_OK;
  auto run = [&]() -> int {
    k_keep<<<blocks((u64)n + 1), 256, 0, s>>>((const u64*)d->umi.p, (const u32*)d->lseq.p, (const u8*)d->name_len.p, hi, pos, nd, md, n);
    size_t tb = tb32; GK(cub::DeviceScan::ExclusiveSum(tmp, tb, pos, pos, (int)n + 1, s));
    tb = tb64; GK(cub::DeviceScan::ExclusiveSum(tmp, tb, nd, nd, (int)n + 1, s));
    tb = tb64; GK(cub::DeviceScan::ExclusiveSum(tmp, tb, md, md, (int)n + 1, s));
    u32 keep_rec = 0; u64 keep_nib = 0, keep_name = 0;
    GK(cudaMemcpyAsync(&keep_rec, pos + n, 4, cudaMemcpyDeviceToHost, s)); GK(cudaMemcpyAsync(&keep_nib, nd + n, 8, cudaMemcpyDeviceToHost, s)); GK(cudaMemcpyAsync(&keep_name, md + n, 8, cudaMemcpyDeviceToHost, s));
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
    GK(cudaGetLastError());
    GK(cudaStreamSynchronize(s));
    d->n_rec = keep_rec; d->n_nib = keep_nib; d->n_name = keep_name;
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

}  // namespace nbg
