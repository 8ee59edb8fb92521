// bam_group.cu — BAM mode in any record order: the device record store and the (UMI, CB) grouping (bam_group.hpp).
//
// The host producer (bam.cpp) stages every kept record of a window and this file uploads it into HBM.  At the end of the
// file the records are put in (UMI, full CB, ordinal) order by two stable CUB radix sorts (CB rank, then UMI key, ordinals
// as values), a scope starts wherever (UMI, CB[..len-2]) changes, and one thread per scope restates
// SortedBamReader::add_dummy_paired_reads + filter_paired_reads (src/parse/sorted_bam_reader.rs:109-162) over the scope's
// records in that order: a count pass, a scan, a write pass.  Pairs are (base offset, clipped length, flags) into the store,
// so no bases move: the scoped batches handed to nb_align_batch are NB_MEM_DEVICE views of the store.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <algorithm>
#include <cstring>
#include <string>

#include "bam_group.hpp"

using namespace nb;

namespace nbg {

#define GK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) return fail(NB_ERR_CUDA, std::string(#x) + ": " + cudaGetErrorString(e_)); } while (0)

namespace {

const u64 PAD = 64;   // the kernels read bases and quals as aligned 16-byte vectors past a read's end (nimble_b200.h)

// a device array that keeps its contents when it grows (the store is appended to window by window)
struct Grow {
  void* p = nullptr; u64 cap = 0;
  int ensure(u64 need, u64 keep, cudaStream_t s, const char* what, u64 store_total) {
    if (need + PAD <= cap) return NB_OK;
    u64 want = std::max<u64>(need + PAD, cap + cap / 2);
    void* q = nullptr;
    if (cudaMalloc(&q, want) != cudaSuccess) {
      cudaGetLastError();
      want = need + PAD;
      if (cudaMalloc(&q, want) != cudaSuccess) { cudaGetLastError(); return fail(NB_ERR_CUDA, std::string("not enough device memory for the record store: ") + what + " needs " + std::to_string(need + PAD) + " bytes (the store needs " + std::to_string(store_total) + " bytes so far)"); }
    }
    if (p) { if (keep) GK(cudaMemcpyAsync(q, p, keep, cudaMemcpyDeviceToDevice, s)); GK(cudaStreamSynchronize(s)); cudaFree(p); }
    p = q; cap = want;
    return NB_OK;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
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

}  // namespace

struct Device {
  int device = 0; cudaStream_t s = nullptr;
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
};

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
  for (Grow* g : {&d->nib, &d->qual, &d->name, &d->umi, &d->cb, &d->nib_off, &d->lseq, &d->flag, &d->name_off, &d->name_len, &d->ordinal}) g->release();
  if (d->g_buf) cudaFree(d->g_buf);
  if (d->p_buf) cudaFree(d->p_buf);
  for (auto& sl : d->slot) if (sl.done) cudaEventDestroy(sl.done);
  if (d->s) cudaStreamDestroy(d->s);
  delete d;
}

void* stream_of(Device* d) { return (void*)d->s; }
int sync(Device* d) { GK(cudaSetDevice(d->device)); GK(cudaStreamSynchronize(d->s)); return NB_OK; }
u64 store_bytes(Device* d) { return d->total(); }
u64 group_bytes(Device* d) { return d->g_bytes + d->p_bytes; }

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

int upload(Device* d) {
  Device::Slot& sl = d->slot[d->cur];
  const Stage& t = sl.st;
  const u64 R = d->n_rec + t.n_rec, NB = d->n_nib + t.n_nib, NM = d->n_name + t.n_name;
  if (R >= 0x7FFFFFFFull) return fail(NB_ERR_UNSUPPORTED, "more than 2^31 - 1 kept records");
  cudaStream_t s = d->s;
  const u64 tot = NB + 2 * NB + NM + R * (8 + 4 + 8 + 4 + 2 + 8 + 1 + 8);
  int e = NB_OK;
  if (!e) e = d->nib.ensure(NB, d->n_nib, s, "the nibble store", tot);
  if (!e) e = d->qual.ensure(2 * NB, 2 * d->n_nib, s, "the qual store", tot);
  if (!e) e = d->name.ensure(NM, d->n_name, s, "the name store", tot);
  if (!e) e = d->umi.ensure(8 * R, 8 * d->n_rec, s, "the UMI keys", tot);
  if (!e) e = d->cb.ensure(4 * R, 4 * d->n_rec, s, "the CB ids", tot);
  if (!e) e = d->nib_off.ensure(8 * R, 8 * d->n_rec, s, "the record offsets", tot);
  if (!e) e = d->lseq.ensure(4 * R, 4 * d->n_rec, s, "the record lengths", tot);
  if (!e) e = d->flag.ensure(2 * R, 2 * d->n_rec, s, "the record flags", tot);
  if (!e) e = d->name_off.ensure(8 * R, 8 * d->n_rec, s, "the name offsets", tot);
  if (!e) e = d->name_len.ensure(R, d->n_rec, s, "the name lengths", tot);
  if (!e) e = d->ordinal.ensure(8 * R, 8 * d->n_rec, s, "the ordinals", tot);
  if (e) return e;
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

int group(Device* d, const std::vector<u32>& cb_rank, const std::vector<u32>& cb_prefix, Grouped& g) {
  GK(cudaSetDevice(d->device));
  cudaStream_t s = d->s;
  const u32 n = (u32)d->n_rec;
  g.n_records = n; g.n_scopes = 0; g.n_pairs = 0; g.scope_pair0.assign(1, 0); g.scope_cb.clear();
  if (n == 0) return NB_OK;
  const u32 ncb = (u32)cb_rank.size();
  int rank_bits = 1; while (rank_bits < 32 && (1ull << rank_bits) < ncb) rank_bits++;
  // one allocation for the sort and scope arrays: rank (ncb) | prefix (ncb) | key32 x2 (n) | val x3 (n) | umi keys x2 (n) | head, sid (n) | start (n+1) | cnt, pair0 (n+1) | scope_cb (n) | cub temp
  size_t tb_sort1 = 0, tb_sort2 = 0, tb_scan1 = 0, tb_scan2 = 0;
  GK(cub::DeviceRadixSort::SortPairs(nullptr, tb_sort1, (const u32*)nullptr, (u32*)nullptr, (const u32*)nullptr, (u32*)nullptr, (int)n, 0, rank_bits, s));
  GK(cub::DeviceRadixSort::SortPairs(nullptr, tb_sort2, (const u64*)nullptr, (u64*)nullptr, (const u32*)nullptr, (u32*)nullptr, (int)n, 0, 64, s));
  GK(cub::DeviceScan::InclusiveSum(nullptr, tb_scan1, (const u32*)nullptr, (u32*)nullptr, (int)n, s));
  GK(cub::DeviceScan::ExclusiveSum(nullptr, tb_scan2, (const u64*)nullptr, (u64*)nullptr, (int)n + 1, s));
  const size_t tmp_bytes = std::max(std::max(tb_sort1, tb_sort2), std::max(tb_scan1, tb_scan2)) + 256;
  auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
  size_t off = 0; auto take = [&](size_t bytes) { size_t o = off; off += al(bytes); return o; };
  const size_t o_rank = take(4ull * ncb), o_pre = take(4ull * ncb), o_k1 = take(4ull * n), o_k2 = take(4ull * n), o_v0 = take(4ull * n), o_v1 = take(4ull * n), o_v2 = take(4ull * n),
               o_u1 = take(8ull * n), o_u2 = take(8ull * n), o_head = take(4ull * n), o_sid = take(4ull * n), o_start = take(4ull * (n + 1)), o_cnt = take(8ull * (n + 1)),
               o_p0 = take(8ull * (n + 1)), o_scb = take(4ull * n), o_tmp = take(tmp_bytes);
  if (d->g_buf) { cudaFree(d->g_buf); d->g_buf = nullptr; d->g_bytes = 0; }
  if (cudaMalloc(&d->g_buf, off) != cudaSuccess) { cudaGetLastError(); d->g_buf = nullptr; return fail(NB_ERR_CUDA, "not enough device memory to group the records: " + std::to_string(off) + " bytes needed"); }
  d->g_bytes = off;
  char* B = (char*)d->g_buf;
  u32* rank = (u32*)(B + o_rank); u32* pre = (u32*)(B + o_pre); u32* k1 = (u32*)(B + o_k1); u32* k2 = (u32*)(B + o_k2);
  u32* v0 = (u32*)(B + o_v0); u32* v1 = (u32*)(B + o_v1); u32* perm = (u32*)(B + o_v2); u64* u1 = (u64*)(B + o_u1); u64* u2 = (u64*)(B + o_u2);
  u32* head = (u32*)(B + o_head); u32* sid = (u32*)(B + o_sid); u32* start = (u32*)(B + o_start); u64* cnt = (u64*)(B + o_cnt); u64* pair0 = (u64*)(B + o_p0);
  u32* scb = (u32*)(B + o_scb); void* tmp = B + o_tmp;
  if (ncb) { GK(cudaMemcpyAsync(rank, cb_rank.data(), 4ull * ncb, cudaMemcpyHostToDevice, s)); GK(cudaMemcpyAsync(pre, cb_prefix.data(), 4ull * ncb, cudaMemcpyHostToDevice, s)); }
  // (UMI, CB rank, ordinal): stable sort by CB rank, then stable sort by UMI key
  k_cb_keys<<<blocks(n), 256, 0, s>>>((const u32*)d->cb.p, rank, k1, v0, n);
  size_t tb = tmp_bytes;
  GK(cub::DeviceRadixSort::SortPairs(tmp, tb, k1, k2, v0, v1, (int)n, 0, rank_bits, s));
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
  if (d->p_buf) { cudaFree(d->p_buf); d->p_buf = nullptr; d->p_bytes = 0; }
  off = 0;
  const size_t q_o1 = take(8 * np + 8), q_o2 = take(8 * np + 8), q_l1 = take(4 * np + 4), q_l2 = take(4 * np + 4), q_f1 = take(np + 1), q_f2 = take(np + 1),
               q_sc = take(4 * np + 4), q_i1 = take(4 * np + 4), q_i2 = take(4 * np + 4), q_loc = take(4 * np + 4);
  if (cudaMalloc(&d->p_buf, off) != cudaSuccess) { cudaGetLastError(); d->p_buf = nullptr; return fail(NB_ERR_CUDA, "not enough device memory for the pairs: " + std::to_string(off) + " bytes needed"); }
  d->p_bytes = off;
  char* P = (char*)d->p_buf;
  d->o1 = (u64*)(P + q_o1); d->o2 = (u64*)(P + q_o2); d->l1 = (u32*)(P + q_l1); d->l2 = (u32*)(P + q_l2); d->f1 = (u8*)(P + q_f1); d->f2 = (u8*)(P + q_f2);
  d->scope = (u32*)(P + q_sc); d->idx1 = (u32*)(P + q_i1); d->idx2 = (u32*)(P + q_i2); d->local = (u32*)(P + q_loc);
  PairsOut out{d->o1, d->o2, d->l1, d->l2, d->f1, d->f2, d->scope, d->idx1, d->idx2};
  if (np) k_pair_write<<<blocks(n_scopes, 128), 128, 0, s>>>(R, start, pair0, out, n_scopes);
  GK(cudaGetLastError());
  GK(cudaStreamSynchronize(s));
  // the sort and scope arrays are not needed any more: the batches only read the store and the pair arrays
  cudaFree(d->g_buf); d->g_buf = nullptr;
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

}  // namespace nbg
