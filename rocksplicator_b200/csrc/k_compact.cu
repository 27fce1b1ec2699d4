// k_compact.cu — flush and compaction: memtable / sorted runs -> one new sorted run.
//
// Replaces RocksDB's background flush + compaction behind ApplicationDB::CompactRange
// (rocksdb_admin/application_db.cpp:138-144) and the write-buffer / L0 triggers of
// examples/counter_service/rocksdb_options.cpp:78-93.  Per shard ("job"):
//
//   k_compact_fill  : one SortItem {8-byte big-endian key prefix, entry ref, source|rank} per entry, one segment per
//                     source; a run's segment is sorted as stored
//   k_compact_sort  : bitonic sort of the MEMTABLE segment by (user key asc, newest first) — prefix compare, full key
//                     on ties (the unsorted source; tiles of 4096 items in shared memory)
//   k_merge_partition / k_merge_tiles : merge of the sorted segments without re-sorting them (merge path): a thread
//                     per tile boundary finds how many items of each segment precede it (multi-sequence selection
//                     under the strict order key / source / rank), then one CTA per 2048-item tile gathers its
//                     sub-ranges into shared memory, orders them there and writes the tile — many CTAs per shard
//   k_compact_size  : per user key: keep what a read can still observe (newest Put; tombstone unless
//                     bottom-most; Merge operands folded with the device operators, otherwise the
//                     operand stack down to its base), then an exclusive scan -> output offsets
//   k_compact_write : copy / synthesise the kept entries into the new heap, write the restart array
//                     (ent_off), the block index (first-key prefix per 32 entries) and the bucketised
//                     hash index
#include <algorithm>
#include <atomic>

#include "kernels.h"

namespace rsp {

constexpr u32 KEEP_UNITS_MASK = 0x00ffffffu;
constexpr u32 KEEP_HEAD = 1u << 24;
constexpr u32 KEEP_MODE_SHIFT = 28;
enum : u32 { MODE_COPY = 0, MODE_PUT_IMM = 1, MODE_PUT_BYTES = 2, MODE_MERGE_IMM = 3 };
constexpr u32 PAD_REF = 0xffffffffu;

struct EntView {
  const u8* e;
  u32 type, klen, vlen;
  u64 seqtype;
  const u64* key;
  const u8* val;
};
__device__ __forceinline__ EntView view_item(const CompactJob& j, const SortItem& it) {
  const u32 src = it.srcrank >> 28;
  EntView v;
  v.e = j.src_heap[src] + (u64)it.ref * 16u;
  const uint4 hd = *reinterpret_cast<const uint4*>(v.e);
  v.seqtype = ((u64)hd.y << 32) | hd.x;
  v.type = hd.x & 0xffu;
  v.klen = hd.z;
  v.vlen = hd.w;
  const u32 koff = j.src_is_mem[src] ? 32u : 16u;
  v.key = reinterpret_cast<const u64*>(v.e + koff);
  v.val = v.e + koff + 16u * units_of(v.klen);
  return v;
}

__device__ __forceinline__ bool item_less(const CompactJob& j, const SortItem& a, const SortItem& b) {
  if (a.ref == PAD_REF) return false;
  if (b.ref == PAD_REF) return true;
  if (a.prefix != b.prefix) return a.prefix < b.prefix;
  const EntView x = view_item(j, a), y = view_item(j, b);
  const int c = cmp_padded(x.key, x.klen, y.key, y.klen);
  if (c) return c < 0;
  return a.srcrank < b.srcrank;
}
__device__ __forceinline__ bool same_key(const CompactJob& j, const SortItem& a, const SortItem& b) {
  if (a.prefix != b.prefix) return false;
  const EntView x = view_item(j, a), y = view_item(j, b);
  return cmp_padded(x.key, x.klen, y.key, y.klen) == 0;
}

__global__ void __launch_bounds__(256) k_compact_fill(const CompactJob* jobs) {
  const CompactJob& j = jobs[blockIdx.y];
  const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= j.items_len) return;
  SortItem it;
  u32 src = 0;
  while (src + 1 < j.n_src && i >= j.seg_start[src + 1]) src++;
  const u32 k = i - j.seg_start[src];
  if (k >= j.src_n[src]) {  // padding of the memtable segment up to its power-of-two sort size
    it.prefix = ~0ull; it.ref = PAD_REF; it.srcrank = ~0u;
  } else {
    it.ref = j.src_ent_off[src][k];
    // ascending rank == newest first: the memtable's ordinals grow with sequence, a run is already
    // stored newest-first within a key
    it.srcrank = (src << 28) | (j.src_is_mem[src] ? (j.src_n[src] - 1u - k) : k);
    const u8* e = j.src_heap[src] + (u64)it.ref * 16u;
    const u32 klen = reinterpret_cast<const u32*>(e)[2];
    const u64 w0 = klen ? *reinterpret_cast<const u64*>(e + (j.src_is_mem[src] ? 32u : 16u)) : 0ull;
    it.prefix = bswap64(w0);
  }
  j.items[i] = it;
}

// Bitonic sort, one CTA per job.  Every compare-exchange step whose stride fits a 4096-item tile (64 KB of
// shared memory) runs on the tile in shared memory; only the strides >= the tile size go through global memory.
// For a 16 K-item shard that is 6 tile passes over global memory instead of 105 step passes.
constexpr u32 SORT_TILE = 4096;

__device__ __forceinline__ void sort_tile_steps(const CompactJob& j, SortItem* tile, u32 tile_n, u32 base, u32 k,
                                                u32 first_stride) {
  for (u32 s = first_stride; s > 0; s >>= 1) {
    for (u32 li = threadIdx.x; li < tile_n; li += blockDim.x) {
      const u32 lp = li ^ s;
      if (lp > li) {
        const SortItem a = tile[li], b = tile[lp];
        const bool asc = ((base + li) & k) == 0;
        if (item_less(j, b, a) == asc) { tile[li] = b; tile[lp] = a; }
      }
    }
    __syncthreads();
  }
}

__global__ void __launch_bounds__(1024) k_compact_sort(const CompactJob* jobs) {
#ifdef RSP_EMUL
  unsigned char* sort_smem = emul_dyn_smem;  // tests/emul: dynamic shared memory of the running block
#else
  extern __shared__ __align__(16) unsigned char sort_smem[];
#endif
  SortItem* tile = reinterpret_cast<SortItem*>(sort_smem);
  const CompactJob& j = jobs[blockIdx.x];
  const u32 n = j.n_pow2;  // the memtable segment at items[0 .. n_pow2); nothing to sort without a memtable
  if (n < 2 || j.totals[7] == 0) return;  // (totals[7] == 0: k_flush_sort has sorted it)
  SortItem* it = j.items;
  const u32 tile_n = n < SORT_TILE ? n : SORT_TILE;
  // phase 1: every tile fully sorted (all steps with k <= tile_n), directions by GLOBAL index
  for (u32 base = 0; base < n; base += tile_n) {
    for (u32 li = threadIdx.x; li < tile_n; li += blockDim.x) tile[li] = it[base + li];
    __syncthreads();
    for (u32 k = 2; k <= tile_n; k <<= 1) sort_tile_steps(j, tile, tile_n, base, k, k >> 1);
    for (u32 li = threadIdx.x; li < tile_n; li += blockDim.x) it[base + li] = tile[li];
    __syncthreads();
  }
  // phase 2: merge stages above the tile size
  for (u32 k = tile_n << 1; k <= n && k != 0; k <<= 1) {
    for (u32 s = k >> 1; s >= tile_n; s >>= 1) {  // strides that leave the tile: global memory
      for (u32 i = threadIdx.x; i < n; i += blockDim.x) {
        const u32 p = i ^ s;
        if (p > i) {
          const SortItem a = it[i], b = it[p];
          const bool asc = (i & k) == 0;
          if (item_less(j, b, a) == asc) { it[i] = b; it[p] = a; }
        }
      }
      __syncthreads();
    }
    for (u32 base = 0; base < n; base += tile_n) {  // the remaining strides: one shared-memory pass per tile
      for (u32 li = threadIdx.x; li < tile_n; li += blockDim.x) tile[li] = it[base + li];
      __syncthreads();
      sort_tile_steps(j, tile, tile_n, base, k, tile_n >> 1);
      for (u32 li = threadIdx.x; li < tile_n; li += blockDim.x) it[base + li] = tile[li];
      __syncthreads();
    }
  }
}


// ------------------------------------------------------------------------------------------------------------
// k_flush_sort — the memtable segment by LSD radix sort in shared memory (one CTA per shard).
//
// The sort key of an entry is its 8-byte big-endian key prefix; within a shard the prefixes differ in their low V bits
// only (V from min ^ max), so an item packs into ONE 64-bit word: (varying prefix bits << 16) | rank, the rank (newest
// first) in the low 16 bits.  ceil(V / 8) stable counting passes order the words by prefix and, being stable, leave
// equal prefixes in rank order — what the compaction wants for the versions of one key.  A pass: every warp owns a
// contiguous range, rows of 32 are ranked with __match_any_sync (no atomics: one histogram row per warp), the digit
// totals are scanned, the words are scattered.  The two buffers are shared memory and the (dead) front half of the
// job's own items[] in global memory, alternating so that the last pass lands in shared memory, from where the sorted
// SortItems are written out coalesced.  Afterwards neighbours with equal prefixes are compared in full: distinct keys
// that share their first 8 bytes (or V > 48, or a memtable beyond the shared-memory budget) leave the job to the
// generic comparison sort (k_compact_sort), flagged in totals[7].  The bitonic network this replaces moved every
// 16-byte item through shared memory ~180 times per 8 K-entry memtable; here it is 2 x ceil(V / 8) + 2 times.
// ------------------------------------------------------------------------------------------------------------
constexpr u32 FS_THREADS = 512;
constexpr u32 FS_WARPS = FS_THREADS / 32;
constexpr u32 FS_MAX_ITEMS = 24576;  // 192 KB of packed words + 8 KB of histograms: one CTA per SM at that size

__global__ void __launch_bounds__(FS_THREADS) k_flush_sort(const CompactJob* jobs, u32 cap) {
#ifdef RSP_EMUL
  unsigned char* fs_smem = emul_dyn_smem;
#else
  extern __shared__ __align__(16) unsigned char fs_smem[];
#endif
  __shared__ unsigned long long s_min, s_max;
  __shared__ u32 s_bad, s_dig_tot[256], s_dig_base[256];
  const CompactJob& j = jobs[blockIdx.x];
  const u32 tid = threadIdx.x, lane = tid & 31u, wid = tid >> 5;
  const u32 n = (j.n_src >= 1 && j.src_is_mem[0]) ? j.src_n[0] : 0u;
  if (tid == 0) { j.totals[7] = n >= 2 ? 1u : 0u; s_min = ~0ull; s_max = 0ull; s_bad = 0; }  // 1: the generic sort is still needed
  if (n < 2 || n > cap) return;
  u64* keys = reinterpret_cast<u64*>(fs_smem);                          // [cap]
  u16* hist = reinterpret_cast<u16*>(fs_smem + (size_t)cap * 8);        // [FS_WARPS][256]
  SortItem* items = j.items;
  u64* gbuf = reinterpret_cast<u64*>(items);  // n words over items[0 .. n/2): dead once the prefixes sit in shared memory
  __syncthreads();
  // ---- range of the prefixes
  {
    u64 mn = ~0ull, mx = 0ull;
    for (u32 i = tid; i < n; i += FS_THREADS) {
      const u64 p = items[i].prefix;
      mn = min(mn, p); mx = max(mx, p);
    }
#pragma unroll
    for (u32 d = 16; d > 0; d >>= 1) {
      mn = min(mn, __shfl_xor_sync(0xffffffffu, mn, d));
      mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, d));
    }
    if (lane == 0) { atomicMin(&s_min, (unsigned long long)mn); atomicMax(&s_max, (unsigned long long)mx); }
  }
  __syncthreads();
  const u64 pmin = s_min, diff = s_min ^ s_max;
  const u32 V = diff ? 64u - (u32)__clzll((long long)diff) : 0u;
  if (V > 48u) return;  // (uniform) the varying bits do not fit beside the rank
  const u64 vmask = V ? (~0ull >> (64u - V)) : 0ull;
  const u32 P = (V + 7u) / 8u;
  // ---- packed words in rank order: rank r = item n-1-r (k_compact_fill stores the memtable in ordinal order)
  for (u32 r = tid; r < n; r += FS_THREADS) keys[r] = ((items[n - 1u - r].prefix & vmask) << 16) | (u64)r;
  __syncthreads();
  if (P & 1u) {  // an odd number of passes starts from the global buffer, so that the last one ends in shared memory
    for (u32 r = tid; r < n; r += FS_THREADS) __stcg(reinterpret_cast<unsigned long long*>(gbuf) + r, (unsigned long long)keys[r]);
    __syncthreads();
  }
  const u32 per = ((n + FS_WARPS - 1u) / FS_WARPS + 31u) & ~31u;  // a warp's contiguous range, whole rows
  const u32 w_lo = min(n, wid * per), w_hi = min(n, w_lo + per);
  u16* my_hist = hist + wid * 256u;
  const u32 lt_mask = (1u << lane) - 1u;
  for (u32 pass = 0; pass < P; pass++) {
    const u32 shift = 16u + 8u * pass;
    const bool src_smem = ((P - pass) & 1u) == 0u;
    for (u32 i = tid; i < FS_WARPS * 256u; i += FS_THREADS) hist[i] = 0;
    __syncthreads();
    // count
    for (u32 row = w_lo; row < w_hi; row += 32u) {
      const u32 i = row + lane;
      const bool valid = i < w_hi;
      const u64 key = valid ? (src_smem ? keys[i] : (u64)__ldcg(reinterpret_cast<const unsigned long long*>(gbuf) + i)) : 0ull;
      const u32 d = valid ? (u32)(key >> shift) & 255u : (256u + lane);
      const u32 m = __match_any_sync(0xffffffffu, d);
      if (valid && (m & lt_mask) == 0u) my_hist[d] = (u16)(my_hist[d] + __popc(m));
      __syncwarp();
    }
    __syncthreads();
    // digit-major, warp-minor exclusive offsets
    if (tid < 256u) {
      u32 run = 0;
      for (u32 w = 0; w < FS_WARPS; w++) {
        const u32 c = hist[w * 256u + tid];
        hist[w * 256u + tid] = (u16)run;
        run += c;
      }
      s_dig_tot[tid] = run;
    }
    __syncthreads();
    if (wid == 0) {
      u32 v[8], sum = 0;
#pragma unroll
      for (u32 q = 0; q < 8; q++) { v[q] = s_dig_tot[lane * 8u + q]; sum += v[q]; }
      u32 incl = sum;
#pragma unroll
      for (u32 d = 1; d < 32; d <<= 1) {
        const u32 o = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += o;
      }
      u32 base = incl - sum;
#pragma unroll
      for (u32 q = 0; q < 8; q++) { s_dig_base[lane * 8u + q] = base; base += v[q]; }
    }
    __syncthreads();
    // scatter (the source rows are re-read: a word is 8 bytes, a register array of a whole range is not)
    for (u32 row = w_lo; row < w_hi; row += 32u) {
      const u32 i = row + lane;
      const bool valid = i < w_hi;
      const u64 key = valid ? (src_smem ? keys[i] : (u64)__ldcg(reinterpret_cast<const unsigned long long*>(gbuf) + i)) : 0ull;
      const u32 d = valid ? (u32)(key >> shift) & 255u : (256u + lane);
      const u32 m = __match_any_sync(0xffffffffu, d);
      u32 dst = 0;
      if (valid) dst = s_dig_base[d] + my_hist[d] + (u32)__popc(m & lt_mask);
      __syncwarp();
      if (valid && (m & lt_mask) == 0u) my_hist[d] = (u16)(my_hist[d] + __popc(m));
      __syncwarp();
      if (valid) {
        if (src_smem) __stcg(reinterpret_cast<unsigned long long*>(gbuf) + dst, (unsigned long long)key);
        else keys[dst] = key;
      }
    }
    __syncthreads();
  }
  // (a shared-memory source is scattered into global memory and the other way round: no pass overwrites what another
  // warp still reads)
  // ---- the sorted SortItems, coalesced; neighbours with equal prefixes must be versions of ONE key
  const u8* heap = j.src_heap[0];
  const u32* ent_off = j.src_ent_off[0];
  const u64 phigh = pmin & ~vmask;
  for (u32 p = tid; p < n; p += FS_THREADS) {
    const u64 key = keys[p];
    const u32 r = (u32)key & 0xffffu;
    SortItem it;
    it.prefix = phigh | (key >> 16);
    it.ref = ent_off[n - 1u - r];
    it.srcrank = r;  // source 0 (the memtable) | rank
    if (p > 0) {
      const u64 prev = keys[p - 1];
      if ((prev >> 16) == (key >> 16)) {
        const u8* a = heap + (u64)ent_off[n - 1u - ((u32)prev & 0xffffu)] * 16u;
        const u8* b = heap + (u64)it.ref * 16u;
        const u32 ka = reinterpret_cast<const u32*>(a)[2], kb = reinterpret_cast<const u32*>(b)[2];
        if (cmp_padded(reinterpret_cast<const u64*>(a + 32), ka, reinterpret_cast<const u64*>(b + 32), kb) != 0) s_bad = 1;
      }
    }
    items[p] = it;
  }
  __syncthreads();
  if (tid == 0) j.totals[7] = s_bad ? 1u : 0u;
}

// ---- merge of the sorted segments (merge path) -------------------------------------------------------
// number of items of segment [lo, hi) of `seg` that order before x
__device__ __forceinline__ u32 seg_lower_bound(const CompactJob& j, const SortItem* seg, u32 lo, u32 hi, const SortItem& x) {
  while (lo < hi) {
    const u32 m = (lo + hi) >> 1;
    if (item_less(j, seg[m], x)) lo = m + 1; else hi = m;
  }
  return lo;
}

// One thread per tile boundary b: coranks[b * n_src + s] = how many items of segment s are among the first
// b * MERGE_TILE items of the merged order.  Multi-sequence selection: the order (key, source, rank) is strict, so the
// split is unique; every round halves the widest remaining range.
__global__ void __launch_bounds__(64) k_merge_partition(const CompactJob* jobs) {
  const CompactJob& j = jobs[blockIdx.y];
  const u32 b = blockIdx.x * blockDim.x + threadIdx.x;
  if (j.n_src < 2 || b > j.n_tiles) return;
  const u32 ns = j.n_src;
  u32* out = j.coranks + (u64)b * ns;
  const u32 p = min(b * MERGE_TILE, j.n_items);
  u32 lo[RSP_MAX_RUNS + 1], hi[RSP_MAX_RUNS + 1];
  for (u32 s = 0; s < ns; s++) { lo[s] = 0; hi[s] = j.src_n[s]; }
  if (p == 0) { for (u32 s = 0; s < ns; s++) out[s] = 0; return; }
  if (p == j.n_items) { for (u32 s = 0; s < ns; s++) out[s] = j.src_n[s]; return; }
  for (;;) {
    u32 widest = 0, width = 0;
    for (u32 s = 0; s < ns; s++) if (hi[s] - lo[s] > width) { width = hi[s] - lo[s]; widest = s; }
    if (width == 0) break;
    const u32 mid = lo[widest] + (width >> 1);
    const SortItem pivot = j.items[j.seg_start[widest] + mid];
    u32 pos[RSP_MAX_RUNS + 1];
    u32 total = 0;
    for (u32 s = 0; s < ns; s++) {
      pos[s] = s == widest ? mid : seg_lower_bound(j, j.items + j.seg_start[s], lo[s], hi[s], pivot);
      total += pos[s];
    }
    if (total == p) { for (u32 s = 0; s < ns; s++) lo[s] = hi[s] = pos[s]; break; }
    if (total < p) {  // the pivot is among the first p items: everything before it is too
      for (u32 s = 0; s < ns; s++) lo[s] = pos[s];
      lo[widest] = mid + 1;
    } else {          // the pivot is beyond the boundary: so is everything after it
      for (u32 s = 0; s < ns; s++) hi[s] = pos[s];
    }
  }
  for (u32 s = 0; s < ns; s++) out[s] = lo[s];
}

// One CTA per tile: gather the tile's sub-range of every segment into shared memory (together MERGE_TILE items, the
// last tile fewer), order them there (bitonic network over 2048 items: 66 compare-exchange steps, no global traffic),
// write the tile of the merged order.
__global__ void __launch_bounds__(512) k_merge_tiles(const CompactJob* jobs) {
  __shared__ SortItem tile[MERGE_TILE];
  const CompactJob& j = jobs[blockIdx.y];
  const u32 b = blockIdx.x;
  if (j.n_src < 2 || b >= j.n_tiles) return;
  const u32 ns = j.n_src;
  const u32* c0 = j.coranks + (u64)b * ns;
  const u32* c1 = c0 + ns;
  u32 at = 0;
  for (u32 s = 0; s < ns; s++) {
    const u32 from = c0[s], cnt = c1[s] - from;
    const SortItem* seg = j.items + j.seg_start[s] + from;
    for (u32 i = threadIdx.x; i < cnt; i += blockDim.x) tile[at + i] = seg[i];
    at += cnt;
  }
  SortItem pad;
  pad.prefix = ~0ull; pad.ref = PAD_REF; pad.srcrank = ~0u;
  for (u32 i = at + threadIdx.x; i < MERGE_TILE; i += blockDim.x) tile[i] = pad;
  __syncthreads();
  for (u32 k = 2; k <= MERGE_TILE; k <<= 1) sort_tile_steps(j, tile, MERGE_TILE, 0, k, k >> 1);
  SortItem* out = j.items2 + (u64)b * MERGE_TILE;
  for (u32 i = threadIdx.x; i < at; i += blockDim.x) out[i] = tile[i];
}

__device__ __forceinline__ u32 imm_units(u32 klen) { return 1u + units_of(klen) + 1u; }

__global__ void __launch_bounds__(1024) k_compact_size(const CompactJob* jobs) {
  const CompactJob& j = jobs[blockIdx.x];
  const u32 n = j.n_items;
  const SortItem* it = j.sorted;
  const bool foldable = j.merge_op == 1 || j.merge_op == 2;
  for (u32 i = threadIdx.x; i < n; i += blockDim.x) {
    if (i > 0 && same_key(j, it[i - 1], it[i])) continue;  // not the newest version of its key
    // i heads a group of versions of one user key, newest first
    const EntView e0 = view_item(j, it[i]);
    u32 g_end = i + 1;  // exclusive end of the group
    while (g_end < n && same_key(j, it[i], it[g_end])) g_end++;
    for (u32 k = i; k < g_end; k++) { j.keep_units[k] = 0; j.out_ord[k] = 0; }
    // the head's shape for the pass below (which would otherwise read the entry header from the heap again: a second
    // random sector per item); out_pos / out_ord get their real contents after that pass
    if (e0.klen <= 0xffffu && e0.vlen <= 0xffffu) { j.out_pos[i] = e0.klen | (e0.vlen << 16); j.out_ord[i] = 0x100u | e0.type; }
    if (e0.type == kTypeValue) {
      j.keep_units[i] = entry_units(e0.type, e0.klen, e0.vlen, false) | KEEP_HEAD;
    } else if (e0.type != kTypeMerge) {  // Delete / SingleDelete
      if (!j.bottom) j.keep_units[i] = entry_units(e0.type, e0.klen, e0.vlen, false) | KEEP_HEAD;
    } else {
      // operands i .. m-1, optional base at m
      u32 m = i, n_bad = 0;
      u64 sum = 0;
      while (m < g_end) {
        const EntView x = view_item(j, it[m]);
        if (x.type != kTypeMerge) break;
        if (x.vlen == 8) sum += *reinterpret_cast<const u64*>(x.val); else n_bad++;
        m++;
      }
      const u32 n_ops = m - i;
      const bool has_base_ent = m < g_end;
      EntView base;
      bool base_put = false;
      if (has_base_ent) { base = view_item(j, it[m]); base_put = base.type == kTypeValue; }
      u32 mode = MODE_COPY;
      bool folded = false;
      u64 val = 0;
      if (foldable) {
        if (base_put) {
          if (j.merge_op == 1) { if (n_bad == 0 && base.vlen == 8) { folded = true; val = sum + *reinterpret_cast<const u64*>(base.val); } }
          else { folded = true; val = sum + (base.vlen == 8 ? *reinterpret_cast<const u64*>(base.val) : 0ull); }
          mode = MODE_PUT_IMM;
        } else if (has_base_ent || j.bottom) {  // existing value == nullptr
          if (j.merge_op == 1) {
            if (n_ops == 1) { folded = true; mode = MODE_PUT_BYTES; }
            else if (n_bad == 0) { folded = true; val = sum; mode = MODE_PUT_IMM; }
          } else { folded = true; val = sum; mode = MODE_PUT_IMM; }
        } else if (n_ops >= 2 && (j.merge_op == 2 || n_bad == 0)) {  // partial merge of the operands
          folded = true; val = sum; mode = MODE_MERGE_IMM;
        }
      }
      if (folded) {
        const u32 units = mode == MODE_PUT_BYTES ? entry_units(kTypeValue, e0.klen, e0.vlen, false) : imm_units(e0.klen);
        j.keep_units[i] = units | KEEP_HEAD | (mode << KEEP_MODE_SHIFT);
        j.fold_val[i] = val;
      } else {
        // keep the operand stack and its base as they are (reads fold them); a Delete base at the
        // bottom is equivalent to "no existing value" and is dropped
        for (u32 k = i; k < m; k++) {
          const EntView x = view_item(j, it[k]);
          j.keep_units[k] = entry_units(x.type, x.klen, x.vlen, false) | (k == i ? KEEP_HEAD : 0u);
        }
        if (has_base_ent && (base_put || !j.bottom))
          j.keep_units[m] = entry_units(base.type, base.klen, base.vlen, false);
      }
    }
  }
  __syncthreads();
  // ---- exclusive scans of units and entry counts (one CTA, chunk per thread)
  __shared__ u32 s_units[1024], s_cnt[1024], s_keys[1024], s_min[1024], s_max[1024], s_np[1024], s_kvmin[1024], s_kvmax[1024];
  const u32 chunk = (n + blockDim.x - 1) / blockDim.x;
  const u32 lo = min(n, threadIdx.x * chunk), hi = min(n, lo + chunk);
  u32 su = 0, sc = 0, sk = 0, mn = ~0u, mx = 0, np = 0, kvmin = ~0u, kvmax = 0;
  for (u32 i = lo; i < hi; i++) {
    const u32 ku = j.keep_units[i];
    const u32 u = ku & KEEP_UNITS_MASK;
    if (u) {
      su += u; sc++; mn = min(mn, u); mx = max(mx, u); if (ku & KEEP_HEAD) sk++;
      // entry shape as it will be written (folded merges become 8-byte Puts / Merges)
      const u32 mode = ku >> KEEP_MODE_SHIFT;
      u32 x_type, x_klen, x_vlen;
      const u32 cached = j.out_ord[i];
      if (cached & 0x100u) {
        const u32 kvc = j.out_pos[i];
        x_type = cached & 0xffu; x_klen = kvc & 0xffffu; x_vlen = kvc >> 16;
      } else {
        const EntView x = view_item(j, it[i]);
        x_type = x.type; x_klen = x.klen; x_vlen = x.vlen;
      }
      const u32 type = (mode == MODE_PUT_IMM || mode == MODE_PUT_BYTES) ? (u32)kTypeValue : (mode == MODE_MERGE_IMM ? (u32)kTypeMerge : x_type);
      const u32 vlen = (mode == MODE_PUT_IMM || mode == MODE_MERGE_IMM) ? 8u : x_vlen;
      if (type != kTypeValue || x_klen > 0xffffu || vlen > 0xffffu) np++;
      const u32 kv = (x_klen & 0xffffu) | (vlen << 16);
      kvmin = min(kvmin, kv); kvmax = max(kvmax, kv);
    }
  }
  s_units[threadIdx.x] = su; s_cnt[threadIdx.x] = sc; s_keys[threadIdx.x] = sk;
  s_min[threadIdx.x] = mn; s_max[threadIdx.x] = mx;
  s_np[threadIdx.x] = np; s_kvmin[threadIdx.x] = kvmin; s_kvmax[threadIdx.x] = kvmax;
  __syncthreads();
  if (threadIdx.x == 0) {
    u32 au = 0, ac = 0, ak = 0, amn = ~0u, amx = 0, anp = 0, akmin = ~0u, akmax = 0;
    for (u32 t = 0; t < blockDim.x; t++) {
      const u32 u = s_units[t], c = s_cnt[t];
      s_units[t] = au; s_cnt[t] = ac;
      au += u; ac += c; ak += s_keys[t];
      amn = min(amn, s_min[t]); amx = max(amx, s_max[t]);
      anp += s_np[t]; akmin = min(akmin, s_kvmin[t]); akmax = max(akmax, s_kvmax[t]);
    }
    j.totals[0] = au; j.totals[1] = ac; j.totals[2] = (ac && amn == amx) ? amn : 0u; j.totals[3] = ak;
    j.totals[4] = anp; j.totals[5] = akmin; j.totals[6] = akmax;  // ([7]: k_flush_sort's flag, read by the host)
  }
  __syncthreads();
  u32 pu = s_units[threadIdx.x], pc = s_cnt[threadIdx.x];
  for (u32 i = lo; i < hi; i++) {
    const u32 u = j.keep_units[i] & KEEP_UNITS_MASK;
    j.out_pos[i] = pu; j.out_ord[i] = pc;
    if (u) { pu += u; pc++; }
  }
}

// several loads in flight before the first store (the kernel is latency-bound: one entry per thread)
__device__ __forceinline__ void copy_units(u8* dst, const u8* src, u32 units) {
  const uint4* s = reinterpret_cast<const uint4*>(src);
  uint4* d = reinterpret_cast<uint4*>(dst);
  u32 u = 0;
  for (; u + 4 <= units; u += 4) {
    const uint4 a = s[u], b = s[u + 1], c = s[u + 2], e = s[u + 3];
    d[u] = a; d[u + 1] = b; d[u + 2] = c; d[u + 3] = e;
  }
  if (u + 2 <= units) {
    const uint4 a = s[u], b = s[u + 1];
    d[u] = a; d[u + 1] = b;
    u += 2;
  }
  if (u < units) d[u] = s[u];
}

__global__ void __launch_bounds__(256) k_compact_write(const CompactJob* jobs) {
  const CompactJob& j = jobs[blockIdx.y];
  const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= j.n_items) return;
  const u32 ku = j.keep_units[i];
  const u32 units = ku & KEEP_UNITS_MASK;
  if (!units) return;
  const u32 mode = ku >> KEEP_MODE_SHIFT;
  const EntView x = view_item(j, j.sorted[i]);
  const u32 pos = j.out_pos[i], ord = j.out_ord[i];
  u8* d = j.out_heap + (u64)pos * 16u;
  const u32 ku_key = units_of(x.klen);
  u32 type = x.type, vlen = x.vlen;
  if (mode == MODE_PUT_IMM || mode == MODE_PUT_BYTES) type = kTypeValue;
  if (mode == MODE_PUT_IMM || mode == MODE_MERGE_IMM) vlen = 8;
  const u64 st = (x.seqtype & ~0xffull) | type;
  *reinterpret_cast<uint4*>(d) = make_uint4((u32)st, (u32)(st >> 32), x.klen, vlen);
  if (mode == MODE_PUT_IMM || mode == MODE_MERGE_IMM) {
    copy_units(d + 16, reinterpret_cast<const u8*>(x.key), ku_key);
    const u64 v = j.fold_val[i];
    *reinterpret_cast<uint4*>(d + 16u + 16u * ku_key) = make_uint4((u32)v, (u32)(v >> 32), 0u, 0u);
  } else {
    // key and value units follow each other in a memtable entry as in a run entry: one copy
    copy_units(d + 16, reinterpret_cast<const u8*>(x.key), ku_key + units_of(x.vlen));
  }
  j.out_ent_off[ord] = pos;
  if (ord % RSP_BLOCK_ENTRIES == 0) j.out_blk_pfx[ord / RSP_BLOCK_ENTRIES] = j.sorted[i].prefix;
  if (ku & KEEP_HEAD) {
    const u64 h = hash_key_padded(x.key, x.klen);
    const u32 val = (((u32)(h >> 32) >> j.out_ord_bits) << j.out_ord_bits) | (ord + 1u);
    u32 bucket = (u32)(((u64)(u32)h * j.out_n_buckets) >> 32);
    for (u32 tries = 0; tries <= j.out_n_buckets; tries++) {  // (load <= 0.5: a free slot exists; bounded anyway)
      u32* b = j.out_hslots + (u64)bucket * RUN_BUCKET_SLOTS;
      bool placed = false;
      for (u32 s = 0; s < RUN_BUCKET_SLOTS && !placed; s++) {
        if (b[s] == 0 && atomicCAS(b + s, 0u, val) == 0u) placed = true;
      }
      if (placed) break;
      bucket = bucket + 1 == j.out_n_buckets ? 0 : bucket + 1;
    }
  }
}

// ---- maintenance helpers: one launch per batch of shards ---------------------------------------------------
__global__ void __launch_bounds__(256) k_zero_out_hslots(const CompactJob* jobs) {
  const CompactJob& j = jobs[blockIdx.y];
  uint4* p = reinterpret_cast<uint4*>(j.out_hslots);
  const u32 n = j.out_n_buckets * (RUN_BUCKET_SLOTS * 4u / 16u);
  for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) p[i] = make_uint4(0u, 0u, 0u, 0u);
}
void launch_zero_out_hslots(const CompactJob* d_jobs, u32 n_jobs, u32 max_buckets, cudaStream_t s) {
  if (!n_jobs || !max_buckets) return;
  const u32 units = max_buckets * (RUN_BUCKET_SLOTS * 4u / 16u);
  const u32 gx = std::min<u32>(64u, (units + 1023u) / 1024u);
  k_zero_out_hslots<<<dim3(std::max<u32>(gx, 1u), n_jobs), 256, 0, s>>>(d_jobs);
}

__global__ void __launch_bounds__(128) k_upload_shards(const ShardUpload* up, ShardDev* shards, ShardFast* fast, ShardFast* fast_runs,
                                                        u32* mt_filter) {
  const ShardUpload& u = up[blockIdx.x];
  const u32 ix = u.index;
  {
    constexpr u32 words = sizeof(ShardDev) / 4, keep = offsetof(ShardDev, n_runs) / 4;
    const u32* src = reinterpret_cast<const u32*>(&u.sd);
    u32* dst = reinterpret_cast<u32*>(shards + ix);
    for (u32 w = (u.runs_only ? keep : 0u) + threadIdx.x; w < words; w += blockDim.x) dst[w] = src[w];
  }
  {
    // (runs_only: run 0 + meta; mt_count is written by the sequencing kernels)
    const u32 words = u.runs_only ? offsetof(ShardFast, mt_count) / 4 : sizeof(ShardFast) / 4;
    if (threadIdx.x < words) reinterpret_cast<u32*>(fast + ix)[threadIdx.x] = reinterpret_cast<const u32*>(&u.fast)[threadIdx.x];
  }
  {
    constexpr u32 words = sizeof(ShardFast) * RSP_MAX_RUNS / 4;
    const u32* src = reinterpret_cast<const u32*>(u.fast_runs);
    u32* dst = reinterpret_cast<u32*>(fast_runs + (size_t)ix * RSP_MAX_RUNS);
    for (u32 w = threadIdx.x; w < words; w += blockDim.x) dst[w] = src[w];
  }
  if (u.zero_mt && u.sd.mt_slots) {
    uint4* p = reinterpret_cast<uint4*>(u.sd.mt_slots);
    const u32 n = (u.sd.mt_slot_mask + 1u) / 2u;  // 8-byte slots, 16-byte stores (the table holds >= 16 slots)
    for (u32 i = threadIdx.x; i < n; i += blockDim.x) p[i] = make_uint4(0u, 0u, 0u, 0u);
    uint4* f = reinterpret_cast<uint4*>(mt_filter + (size_t)ix * MT_FILTER_WORDS);  // and its filter
    for (u32 i = threadIdx.x; i < MT_FILTER_WORDS / 4u; i += blockDim.x) f[i] = make_uint4(0u, 0u, 0u, 0u);
  }
}
void launch_upload_shards(const ShardUpload* d_up, u32 n, ShardDev* shards, ShardFast* fast, ShardFast* fast_runs, u32* mt_filter,
                          cudaStream_t s) {
  if (!n) return;
  k_upload_shards<<<n, 128, 0, s>>>(d_up, shards, fast, fast_runs, mt_filter);
}

// An ingested run takes the sequence number of the ingest, all its entries alike: the scratch shard it was built on
// numbered them 1..n, which may be below the versions of the same keys in older runs.
__global__ void __launch_bounds__(256) k_set_run_seq(u8* heap, const u32* ent_off, u32 n, u64 seq) {
  const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  u64* st = reinterpret_cast<u64*>(heap + (u64)ent_off[i] * 16u);
  *st = (seq << 8) | (*st & 0xffull);
}
void launch_set_run_seq(u8* heap, const u32* ent_off, u32 n, u64 seq, cudaStream_t s) {
  if (!n) return;
  k_set_run_seq<<<(n + 255) / 256, 256, 0, s>>>(heap, ent_off, n, seq);
}

void launch_compact_sort(const CompactJob* d_jobs, const CompactJob* h_jobs, u32 n_jobs, cudaStream_t s) {
  if (!n_jobs) return;
  u32 max_len = 0, max_sort = 0, max_tiles = 0;
  for (u32 i = 0; i < n_jobs; i++) {
    max_len = std::max(max_len, h_jobs[i].items_len);
    max_sort = std::max(max_sort, h_jobs[i].n_pow2);
    if (h_jobs[i].n_src > 1) max_tiles = std::max(max_tiles, h_jobs[i].n_tiles);
  }
  if (!max_len) return;
  k_compact_fill<<<dim3((max_len + 255) / 256, n_jobs), 256, 0, s>>>(d_jobs);
  if (max_sort >= 2) {
    // the opt-ins are per-DEVICE function attributes: one engine per GPU may live in the same process
    static std::atomic<unsigned long long> opted_in{0};
    int dev = 0;
    cudaGetDevice(&dev);
    const unsigned long long bit = 1ull << (dev & 63);
    if (!(opted_in.load(std::memory_order_acquire) & bit)) {
      cudaFuncSetAttribute(k_compact_sort, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(SORT_TILE * sizeof(SortItem)));
      cudaFuncSetAttribute(k_flush_sort, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(FS_MAX_ITEMS * 8 + FS_WARPS * 256 * 2));
      opted_in.fetch_or(bit, std::memory_order_release);
    }
    // radix sort in shared memory for the memtables that fit; the comparison sort takes what is left (flag in totals[7])
    u32 cap = 32;
    for (u32 i = 0; i < n_jobs; i++)
      if (h_jobs[i].n_src && h_jobs[i].src_is_mem[0]) cap = std::max(cap, std::min(h_jobs[i].src_n[0], FS_MAX_ITEMS));
    cap = (cap + 31u) & ~31u;
    k_flush_sort<<<n_jobs, FS_THREADS, (size_t)cap * 8 + FS_WARPS * 256 * 2, s>>>(d_jobs, cap);
    k_compact_sort<<<n_jobs, 1024, SORT_TILE * sizeof(SortItem), s>>>(d_jobs);
  }
  if (max_tiles) {
    k_merge_partition<<<dim3((max_tiles + 1 + 63) / 64, n_jobs), 64, 0, s>>>(d_jobs);
    k_merge_tiles<<<dim3(max_tiles, n_jobs), 512, 0, s>>>(d_jobs);
  }
}
void launch_compact_size(const CompactJob* d_jobs, u32 n_jobs, cudaStream_t s) {
  if (!n_jobs) return;
  k_compact_size<<<n_jobs, 1024, 0, s>>>(d_jobs);
}
void launch_compact_write(const CompactJob* d_jobs, u32 n_jobs, u32 max_items, cudaStream_t s) {
  if (!n_jobs || !max_items) return;
  dim3 grid((max_items + 255) / 256, n_jobs);
  k_compact_write<<<grid, 256, 0, s>>>(d_jobs);
}

}  // namespace rsp
