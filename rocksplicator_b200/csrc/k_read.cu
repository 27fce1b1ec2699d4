// k_read.cu — Get / MultiGet / range-scan kernels.
//
// Replaces what ApplicationDB::Get / MultiGet / NewIterator hand to rocksdb::DB
// (rocksdb_admin/application_db.cpp:78-120): for each key, walk the versions newest -> oldest
// (memtable chain, then each sorted run newest first); Put answers, Delete/SingleDelete hides,
// Merge operands accumulate and are folded oldest -> newest with the AssociativeMergeOperator rules
// of examples/counter_service/merge_operator.cpp:23-45 / RocksDB's uint64add on the device, or are
// handed to the host for any other operator.
//
// A query is served by a group of G lanes (8 for MultiGet): one 32-byte sector of hash slots is one
// coalesced group load, an entry is read as consecutive 16-byte units, the value leaves as
// consecutive 16-byte stores.  All lanes of a group run the same control flow.
#include <algorithm>
#include <cstddef>

#include "kernels.h"

namespace rsp {

__device__ __forceinline__ u64 ldcg64(const void* p) { return __ldcg(reinterpret_cast<const unsigned long long*>(p)); }
__device__ __forceinline__ u32 ldcg32(const void* p) { return __ldcg(reinterpret_cast<const u32*>(p)); }

// ---- merge accumulator (device-resident operators) ------------------------------------------------
struct Acc {
  u32 n_ops, n_bad;
  u64 sum;             // wrapping sum of the 8-byte operands seen so far
  const u8* last_ptr;  // oldest operand seen so far
  u32 last_len;
  u32 merge_op;
  // result
  bool done, imm;
  i32 status;
  u32 msg;
  const u8* res_ptr;
  u32 res_len;
  u64 res_imm;
  __device__ void init(u32 op) {
    n_ops = n_bad = 0; sum = 0; last_ptr = nullptr; last_len = 0; merge_op = op;
    done = false; imm = false; status = 1; msg = 0; res_ptr = nullptr; res_len = 0; res_imm = 0;
  }
  __device__ void fail(i32 st, u32 m) { status = st; msg = m; done = true; }
  // fold the collected operands onto `base` (nullptr = no existing value)
  __device__ void finish(const u8* base, u32 base_len) {
    done = true;
    if (merge_op == 1) {  // RSP_MERGE_COUNTER
      if (base) {
        if (base_len != 8 || n_bad) return fail(2, MSG_MERGE_FAILED);
        res_imm = sum + ldcg64(base);
      } else if (n_ops == 1) {  // existing == nullptr -> the operand itself, any size
        status = 0; res_ptr = last_ptr; res_len = last_len;
        return;
      } else {
        if (n_bad) return fail(2, MSG_MERGE_FAILED);
        res_imm = sum;
      }
    } else {  // RSP_MERGE_UINT64ADD: malformed operands count as 0
      res_imm = sum + ((base && base_len == 8) ? ldcg64(base) : 0ull);
    }
    status = 0; imm = true; res_len = 8;
  }
  // one version, newest first.  returns done.
  __device__ bool visit(u32 type, const u8* vptr, u32 vlen) {
    if (type == kTypeValue) {
      if (n_ops == 0) { status = 0; res_ptr = vptr; res_len = vlen; done = true; }
      else finish(vptr, vlen);
    } else if (type == kTypeMerge) {
      if (merge_op == 0) fail(4, MSG_MERGE_NOT_INIT);
      else if (merge_op > 2) fail(ST_NEED_HOST_MERGE, 0);
      else {
        n_ops++;
        if (vlen == 8) sum += ldcg64(vptr); else n_bad++;
        last_ptr = vptr; last_len = vlen;
      }
    } else {  // Delete / SingleDelete
      if (n_ops == 0) { status = 1; done = true; }
      else finish(nullptr, 0);
    }
    return done;
  }
  __device__ void end_of_versions() {
    if (done) return;
    if (n_ops) finish(nullptr, 0);
    else { status = 1; done = true; }
  }
};

// ---- version walk over one shard ---------------------------------------------------------------------
// V: visitor with bool visit(u32 type, const u8* vptr, u32 vlen) (true = stop).
template <u32 G, class V>
__device__ __forceinline__ void walk_memtable(const ShardDev* sd, const u8* kp, u32 klen, u64 h, u64 snap,
                                              u32 lane, u32 gmask, u32 gbase, V& v) {
  const u64* slots = sd->mt_slots;
  const u8* heap = sd->mt_heap;
  const u32 mask = sd->mt_slot_mask;
  const u32 tag = hash_tag32(h);
  u32 idx = (u32)h & mask;
  for (u32 probes = 0; probes <= mask; probes += G) {
    const u64 sv = ldcg64(slots + ((idx + lane) & mask));
    const u32 empty_m = (__ballot_sync(gmask, sv == 0) >> gbase) & ((1u << G) - 1u);
    u32 match_m = (__ballot_sync(gmask, (u32)(sv >> 32) == tag && sv != 0) >> gbase) & ((1u << G) - 1u);
    const u32 first_empty = empty_m ? (u32)(__ffs(empty_m) - 1) : G;
    match_m &= (first_empty >= 32u) ? 0xffffffffu : ((1u << first_empty) - 1u);
    while (match_m) {
      const u32 m = (u32)(__ffs(match_m) - 1);
      match_m &= match_m - 1;
      u32 c = (u32)__shfl_sync(gmask, (u32)sv, gbase + m);
      const u8* he = heap + (u64)(c - 1u) * 16u;
      const u32 hklen = ldcg32(he + 8);
      if (!eq_key_vs_padded_cg(kp, klen, reinterpret_cast<const u64*>(he + 32), hklen)) continue;
      // my key: walk the chain newest -> oldest, skipping versions newer than the published snapshot
      while (c) {
        const u8* e = heap + (u64)(c - 1u) * 16u;
        const uint4 hd = __ldcg(reinterpret_cast<const uint4*>(e));
        const u64 st = ((u64)hd.y << 32) | hd.x;
        if ((st >> 8) <= snap) {
          if (v.visit((u32)(st & 0xffu), e + 32u + 16u * units_of(hd.z), hd.w)) return;
        }
        c = ldcg32(e + 16);
      }
      return;  // chain exhausted, older versions live in the runs
    }
    if (empty_m) return;
    idx = (idx + G) & mask;
  }
}

__device__ __forceinline__ const u8* run_entry(const RunDev& r, u32 ord) {
  const u32 unit = r.uniform_units ? ord * r.uniform_units : __ldg(r.ent_off + ord);
  return r.heap + (u64)unit * 16u;
}

template <u32 G, class V>
__device__ __forceinline__ bool walk_run(const RunDev& r, const u8* kp, u32 klen, u64 h, u32 lane, u32 gmask,
                                         u32 gbase, V& v) {
  if (r.n_ent == 0) return false;
  const u32 tag = (u32)(h >> 32) >> r.ord_bits;
  const u32 ord_mask = (1u << r.ord_bits) - 1u;
  u32 bucket = (u32)(((u64)(u32)h * r.n_buckets) >> 32);
  for (u32 nb = 0; nb < r.n_buckets; nb++) {
    // one 32-byte sector of slots per bucket; with G < 8 lanes each lane covers several slots
    u32 sv[RUN_BUCKET_SLOTS / G > 0 ? RUN_BUCKET_SLOTS / G : 1];
    bool any_empty = false;
#pragma unroll
    for (u32 i = 0; i < RUN_BUCKET_SLOTS / G; i++) {
      sv[i] = __ldg(r.hslots + (u64)bucket * RUN_BUCKET_SLOTS + i * G + lane);
      any_empty |= sv[i] == 0;
    }
    const bool grp_empty = __ballot_sync(gmask, any_empty) != 0;
#pragma unroll
    for (u32 i = 0; i < RUN_BUCKET_SLOTS / G; i++) {
      u32 match_m = (__ballot_sync(gmask, sv[i] != 0 && (sv[i] >> r.ord_bits) == tag) >> gbase) & ((1u << G) - 1u);
      while (match_m) {
        const u32 m = (u32)(__ffs(match_m) - 1);
        match_m &= match_m - 1;
        u32 ord = (__shfl_sync(gmask, sv[i], gbase + m) & ord_mask) - 1u;
        const u8* e = run_entry(r, ord);
        uint4 hd = __ldg(reinterpret_cast<const uint4*>(e));
        if (!eq_key_vs_padded(kp, klen, reinterpret_cast<const u64*>(e + 16), hd.z)) continue;
        // first (newest) version of my key in this run; older versions follow in sort order
        for (;;) {
          if (v.visit(hd.x & 0xffu, e + 16u + 16u * units_of(hd.z), hd.w)) return true;
          if (++ord >= r.n_ent) return true;
          e = run_entry(r, ord);
          hd = __ldg(reinterpret_cast<const uint4*>(e));
          if (!eq_key_vs_padded(kp, klen, reinterpret_cast<const u64*>(e + 16), hd.z)) return true;
        }
      }
    }
    if (grp_empty) return false;
    bucket = bucket + 1 == r.n_buckets ? 0 : bucket + 1;
  }
  return false;
}

template <u32 G, class V>
__device__ __forceinline__ void walk_shard(const ShardDev* sd, const u8* kp, u32 klen, u32 lane, u32 gmask,
                                           u32 gbase, V& v, bool& stopped) {
  const u64 h = hash_key(kp, klen);
  const u64 snap = ldcg64(&sd->pub_seq);
  stopped = false;
  if (ldcg32(&sd->mt_count) != 0) {
    walk_memtable<G>(sd, kp, klen, h, snap, lane, gmask, gbase, v);
    if (v.done) { stopped = true; return; }
  }
  const u32 n_runs = sd->n_runs;
  for (u32 ri = 0; ri < n_runs; ri++) {
    walk_run<G>(sd->runs[ri], kp, klen, h, lane, gmask, gbase, v);
    if (v.done) { stopped = true; return; }
  }
}

// ------------------------------------------------------------------------------------------------
// k_multi_get
// ------------------------------------------------------------------------------------------------
constexpr u32 MG_LANES = 8;

__device__ __forceinline__ void group_copy_out(u8* dst, const u8* src, u32 n, u32 lane, u32 lanes) {
  if ((reinterpret_cast<uintptr_t>(dst) & 15u) == 0) {
    const u32 full = n >> 4;
    for (u32 u = lane; u < full; u += lanes)
      reinterpret_cast<uint4*>(dst)[u] = __ldcg(reinterpret_cast<const uint4*>(src) + u);
    for (u32 b = (full << 4) + lane; b < n; b += lanes) dst[b] = src[b];
  } else {
    for (u32 b = lane; b < n; b += lanes) dst[b] = src[b];
  }
}

// generic path: any key length, any entry shape, memtable chains, merges, multiple runs
__device__ __noinline__ void lookup_generic(const GetArgs& a, u32 q, u32 lane, u32 gmask, u32 gbase) {
  const u32 six = __ldg(a.shard_ix + q);
  if (six >= a.max_shards || !a.shards[six].live) {  // unknown / closed shard
    if (lane == 0) {
      a.st[q] = 4;
      a.vlen[q] = 0;
      if (a.n_special) atomicAdd(a.n_special, 1u);
    }
    return;
  }
  const ShardDev* sd = a.shards + six;
  const u8* kp;
  u32 klen;
  if (a.klen_fixed) {
    klen = a.klen_fixed;
    kp = a.keys + (u64)q * klen;
  } else {
    const u64 o = __ldg(a.koff + q);
    klen = (u32)(__ldg(a.koff + q + 1) - o);
    kp = a.keys + o;
  }
  Acc acc;
  acc.init(sd->merge_op);
  bool stopped;
  walk_shard<MG_LANES>(sd, kp, klen, lane, gmask, gbase, acc, stopped);
  acc.end_of_versions();
  i32 st = acc.status;
  u32 vlen = 0;
  if (st == 0) {
    vlen = acc.res_len;
    if ((u64)vlen > a.val_stride) {
      st = 7;  // RSP_INCOMPLETE: vlen reports the size needed
    } else {
      u8* dst = a.vals + (u64)q * a.val_stride;
      if (acc.imm) {
        if (lane == 0) {
#pragma unroll
          for (u32 b = 0; b < 8; b++) dst[b] = (u8)(acc.res_imm >> (8u * b));
        }
      } else {
        group_copy_out(dst, acc.res_ptr, vlen, lane, MG_LANES);
      }
    }
  } else if (st != 1 && st != ST_NEED_HOST_MERGE) {
    vlen = acc.msg;  // message id rides in vlen for error statuses
  }
  if (lane == 0) {
    a.st[q] = st;
    a.vlen[q] = vlen;
    if (st != 0 && st != 1 && st != 7 && a.n_special) atomicAdd(a.n_special, 1u);
  }
}

__global__ void __launch_bounds__(256) k_multi_get(GetArgs a) {
  const u32 q = (blockIdx.x * blockDim.x + threadIdx.x) / MG_LANES;
  const u32 lane = threadIdx.x & (MG_LANES - 1);
  const u32 gbase = (threadIdx.x & 31u) & ~(MG_LANES - 1u);
  const u32 gmask = ((1u << MG_LANES) - 1u) << gbase;
  if (q >= a.n) return;
  lookup_generic(a, q, lane, gmask, gbase);
}

// Measured and dropped in r02 (profiles/r02_experiments/): hash-addressed entry slots instead of the index
// (0.38 / 0.32 / 0.18 of the roofline at load 0.25 / 0.5 / 0.75 against 0.41) and software prefetch of later lookups'
// sectors (0.18).
// ---- the hot kernel: 16-byte keys, TWO lanes per lookup, three dependent memory round trips ----------
//   1. shard id + query key (coalesced across the warp) and the 32-byte ShardFast descriptor
//      (32 B x #shards: L1/L2-resident); both lanes load the same words (one broadcast transaction)
//   2. the hash bucket: one 32-byte sector of run 0's index, four u32 slots (one 16-byte load) per lane
//      (when the memtable is not empty: eight u64 memtable slots first, four per lane)
//   3. the entry: both lanes read the header and key units (same sector, broadcast) and decide alike with
//      no shuffles; lane L then moves value units L, L+2, .. straight from its registers to the output
//      (2 lanes x 2 x 16 B = the 64-byte value)
// The kernel is issue-bound before it is HBM-bound, so the lane count per lookup is what the instruction
// budget allows: 8 lanes cost ~70 warp instructions per lookup, 2 lanes ~1/4 of that.
// Anything else — tag false positive, probe longer than 4 buckets, Delete / Merge, version chains, several
// runs, odd sizes — is appended to the pending list and served by the generic path (k_multi_get_pending).
static_assert(offsetof(ShardDev, mt_slot_mask) == 24 && offsetof(ShardDev, pub_seq) == 56, "ShardDev units 0-3");
static_assert(sizeof(ShardFast) == 32, "ShardFast");

constexpr u32 FL = 2;  // lanes per lookup

// L2 residency control (createpolicy + ld/st .L2::cache_hint): the hash-index sectors are the only
// data with reuse across lookups (80 MB at 10 M keys vs a 126 MB L2); entries, query keys and results
// stream through once.  RSP_MG_HINTS: 0 = none, 1 = index evict_last (+1 %), 2 = also streams evict_first
// (measured 20 % SLOWER on B200: kept only as an experiment switch).  RSP_MG_NOALLOC: entry units bypass L1.
#ifndef RSP_MG_HINTS
#define RSP_MG_HINTS 1
#endif
__device__ __forceinline__ u64 pol_evict_last() {
  u64 p;
#ifdef RSP_EMUL  // tests/emul: cache policies have no meaning on the CPU
  p = 0;
#else
  asm("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
#endif
  return p;
}
__device__ __forceinline__ u64 pol_evict_first() {
  u64 p;
#ifdef RSP_EMUL
  p = 0;
#else
  asm("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
#endif
  return p;
}
__device__ __forceinline__ uint4 ldg_pol(const uint4* p, u64 pol) {
  uint4 v;
#ifdef RSP_EMUL
  (void)pol;
  v = *p;
#else
  asm("ld.global.nc.L2::cache_hint.v4.u32 {%0,%1,%2,%3}, [%4], %5;"
      : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p), "l"(pol));
#endif
  return v;
}
__device__ __forceinline__ void stg_pol(uint4* p, const uint4& v, u64 pol) {
#ifdef RSP_EMUL
  (void)pol;
  *p = v;
#else
  asm volatile("st.global.L2::cache_hint.v4.u32 [%0], {%1,%2,%3,%4}, %5;"
               :: "l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w), "l"(pol) : "memory");
#endif
}
#ifndef RSP_MG_TPB
#define RSP_MG_TPB 64
#endif
#ifndef RSP_MG_MINB
#define RSP_MG_MINB 24
#endif

// Candidate entry at `ent`: header unit 0, key unit KU, value units KU+1.. (U units in all).
// Returns 0 = served, 1 = not my key (tag false positive), 2 = needs the generic path.
#ifndef RSP_MG_NOALLOC
#define RSP_MG_NOALLOC 0  // measured 5 % slower with L1::no_allocate on the entry units
#endif
#ifndef RSP_MG_MEMSET
#define RSP_MG_MEMSET 1
#endif
__device__ __forceinline__ uint4 ldg_noalloc(const uint4* p) {
  uint4 v;
#ifdef RSP_EMUL
  v = *p;
#else
  asm("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
#endif
  return v;
}
template <bool CG>
__device__ __forceinline__ uint4 ld_entry_unit(const uint4* p, u64 pol) {
  if (CG) return __ldcg(p);
#if RSP_MG_HINTS >= 2
  return ldg_pol(p, pol);
#elif RSP_MG_NOALLOC
  return ldg_noalloc(p);
#else
  return __ldg(p);
#endif
}
template <bool CG, bool BIG>
__device__ __forceinline__ u32 fast_entry(const u8* ent, u32 U, u32 KU, const uint4& kq, u64 snap, u8* dst,
                                          u64 val_stride, u32 lane, u32& vlen_out, u64 pol) {
  const uint4* ep = reinterpret_cast<const uint4*>(ent);
  const uint4 hd = ld_entry_unit<CG>(ep, pol);
  const uint4 ek = ld_entry_unit<CG>(ep + KU, pol);
  const u32 fv = KU + 1;  // first value unit; lane L owns value units L, L+2, L+4, ...
  uint4 v0 = make_uint4(0, 0, 0, 0), v1 = v0, v2 = v0;
  if (!CG) {
    // a run: the entry size U is known before the header arrives, so the first six value units are
    // requested together with header and key (one round trip for values up to 96 bytes)
    if (fv + lane < U) v0 = ld_entry_unit<CG>(ep + fv + lane, pol);
    if (fv + lane + 2 < U) v1 = ld_entry_unit<CG>(ep + fv + lane + 2, pol);
    if (fv + lane + 4 < U) v2 = ld_entry_unit<CG>(ep + fv + lane + 4, pol);
  }
  if (ek.x != kq.x || ek.y != kq.y || ek.z != kq.z || ek.w != kq.w || hd.z != 16) return 1;
  const u64 seq = (((u64)hd.y << 32) | hd.x) >> 8;
  const u32 vu = (hd.w + 15u) >> 4;
  if ((hd.x & 0xffu) != kTypeValue || seq > snap || (!CG && fv + vu > U) || (u64)vu * 16u > val_stride || (!BIG && vu > 6)) return 2;
  uint4* out = reinterpret_cast<uint4*>(dst);
  if (CG) {
    // the memtable: the entry's size is only known from its header, so the value follows in a second trip
    for (u32 u = lane; u < vu; u += FL) out[u] = ld_entry_unit<CG>(ep + fv + u, pol);
  } else {
#if RSP_MG_HINTS >= 2
    if (lane < vu) stg_pol(out + lane, v0, pol);
    if (lane + 2 < vu) stg_pol(out + lane + 2, v1, pol);
    if (lane + 4 < vu) stg_pol(out + lane + 4, v2, pol);
#else
    if (lane < vu) out[lane] = v0;
    if (lane + 2 < vu) out[lane + 2] = v1;
    if (lane + 4 < vu) out[lane + 4] = v2;
#endif
    if (BIG)
      for (u32 u = lane + 6; u < vu; u += FL) out[u] = ld_entry_unit<CG>(ep + fv + u, pol);  // values > 96 bytes
  }
  vlen_out = hd.w;
  return 0;
}

// BIG = false: values up to 96 bytes (larger ones take the pending list); BIG = true adds the tail loop for
// larger values at the price of a few registers — the host picks by the caller's value stride.
template <bool BIG>
__global__ void __launch_bounds__(RSP_MG_TPB, RSP_MG_MINB) k_multi_get16(GetArgs a) {
  const u32 q = (blockIdx.x * blockDim.x + threadIdx.x) / FL;
  const u32 lane = threadIdx.x & (FL - 1);
  const u32 pbase = (threadIdx.x & 31u) & ~1u;
  const u32 pmask = 3u << pbase;  // the two lanes of this lookup always branch together
  if (q >= a.n) return;
  // (1)
  const u64 pol_stream = pol_evict_first();
  u32 six = __ldg(a.shard_ix + q);
  const bool bad_shard = six >= a.max_shards;
  if (bad_shard) six = 0;
#if RSP_MG_HINTS >= 2
  const uint4 kq = ldg_pol(reinterpret_cast<const uint4*>(a.keys) + q, pol_stream);
#else
  const uint4 kq = __ldg(reinterpret_cast<const uint4*>(a.keys) + q);
#endif
  const uint4 f0 = __ldg(reinterpret_cast<const uint4*>(a.fast + six));
  const uint4 f1 = __ldg(reinterpret_cast<const uint4*>(a.fast + six) + 1);
  const u32 n_buckets = f1.x, ord_bits = f1.y & 0xffu, U = (f1.y >> 8) & 0xffu, n_runs = (f1.y >> 16) & 0xffu;
  const u64 k0 = ((u64)kq.y << 32) | kq.x, k1 = ((u64)kq.w << 32) | kq.z;
  const u64 h = hash_final(hash_step(hash_step(hash_init(16), k0), k1));
  u8* dst = a.vals + (u64)q * a.val_stride;
  u32 state = 3;  // 0 served, 2 generic path, 3 undecided, 4 not found
  u32 vlen = 0;
  if (n_runs > 1 || ((a.val_stride | reinterpret_cast<uintptr_t>(a.vals)) & 15u) || bad_shard || !(f1.y >> 24)) state = 2;
  bool in_mem = false;
  if (state == 3 && f1.z /* mt_count */) {
    // the shard's memtable filter (L2-resident, behind the descriptors): a clear bit = the key is not in the memtable
    const u32 fb = mt_filter_bit(h);
    const u32 fw = __ldcg(reinterpret_cast<const u32*>(a.fast + (size_t)a.max_shards * (1u + RSP_MAX_RUNS)) + (size_t)six * MT_FILTER_WORDS + (fb >> 5));
    in_mem = (fw >> (fb & 31u)) & 1u;
  }
  if (in_mem) {
    // ---- memtable: eight u64 slots from the home position, four per lane; descriptor through L2
    const uint4* dp = reinterpret_cast<const uint4*>(a.shards + six);
    const uint4 d0 = __ldcg(dp), d1 = __ldcg(dp + 1), d3 = __ldcg(dp + 3);
    const u8* heap = reinterpret_cast<const u8*>(((u64)d0.y << 32) | d0.x);
    const u64* sp = reinterpret_cast<const u64*>(((u64)d0.w << 32) | d0.z);
    const u32 mask = d1.z;
    const u64 snap = ((u64)d3.w << 32) | d3.z;
    const u32 tag = hash_tag32(h);
    u32 cand = 0, info = 0;  // info: matches | (position of my first empty + 1) << 8
#pragma unroll
    for (u32 i = 0; i < 4; i++) {
      const u64 sv = ldcg64(sp + (((u32)h + 4u * lane + i) & mask));
      if (sv == 0) { if (!(info >> 8)) info |= (4u * lane + i + 1u) << 8; }
      else if ((u32)(sv >> 32) == tag && !(info >> 8)) { if (!cand) cand = (u32)sv; info++; }
    }
    const u32 o_cand = __shfl_xor_sync(pmask, cand, 1), o_info = __shfl_xor_sync(pmask, info, 1);
    // lane 1's slots come after lane 0's in probe order: they count only if lane 0 saw no empty slot
    const u32 lo_info = lane ? o_info : info, hi_info = lane ? info : o_info;
    const u32 lo_cand = lane ? o_cand : cand, hi_cand = lane ? cand : o_cand;
    const bool lo_empty = (lo_info >> 8) != 0;
    const u32 n_match = (lo_info & 0xffu) + (lo_empty ? 0u : (hi_info & 0xffu));
    const bool any_empty = lo_empty || (hi_info >> 8) != 0;
    if (n_match == 1) {
      const u32 c = (lo_info & 0xffu) ? lo_cand : hi_cand;
      // memtable entry: unit0 header, unit1 link, unit2 key, units 3.. value
      const u32 r = fast_entry<true, BIG>(heap + (u64)(c - 1u) * 16u, 7, 2, kq, snap, dst, a.val_stride, lane, vlen, pol_stream);
      state = r == 0 ? 0 : 2;
    } else if (n_match > 1 || !any_empty) {
      state = 2;
    }
  }
  if (state == 3) {
    if (n_runs == 0) state = 4;
    else if (U == 0 || U >= 255) state = 2;
    else {
      // ---- run 0 through its hash index: one bucket = one 32-byte sector, four slots per lane
      const u8* heap = reinterpret_cast<const u8*>(((u64)f0.y << 32) | f0.x);
      const uint4* hs = reinterpret_cast<const uint4*>(((u64)f0.w << 32) | f0.z);
      u32 bucket = (u32)(((u64)(u32)h * n_buckets) >> 32);
      const u32 tag = (u32)(h >> 32) >> ord_bits;
      // Walk the tag matches in probe order; a false positive (18-bit tags at 16 K entries: ~1 per 60 K
      // lookups) just moves on to the next candidate, a full bucket to the next bucket.
      u32 m8 = 0, e8 = 1, probe = 0;  // e8 != 0 before the first load only so that the loop loads first
      uint4 sv = make_uint4(0, 0, 0, 0);
      state = 2;
#pragma unroll 1
      for (;;) {
        if (!m8) {
          if (probe && e8) { state = 4; break; }  // an empty slot ends the probe: NOT_FOUND
          if (probe == n_buckets) { state = 4; break; }  // (a table without an empty slot)
          if (probe) bucket = bucket + 1 == n_buckets ? 0 : bucket + 1;
          probe++;
#if RSP_MG_HINTS >= 1
          sv = ldg_pol(hs + (u64)bucket * 2u + lane, pol_evict_last());
#else
          sv = __ldg(hs + (u64)bucket * 2u + lane);
#endif
          const u32 m = ((sv.x && (sv.x >> ord_bits) == tag) ? 1u : 0u) | ((sv.y && (sv.y >> ord_bits) == tag) ? 2u : 0u) |
                        ((sv.z && (sv.z >> ord_bits) == tag) ? 4u : 0u) | ((sv.w && (sv.w >> ord_bits) == tag) ? 8u : 0u);
          const u32 e = (sv.x == 0 || sv.y == 0 || sv.z == 0 || sv.w == 0) ? 1u : 0u;
          const u32 mine = m | (e << 4);
          const u32 other = __shfl_xor_sync(pmask, mine, 1);
          m8 = lane ? ((other & 15u) | ((mine & 15u) << 4)) : ((mine & 15u) | ((other & 15u) << 4));
          e8 = (mine | other) >> 4;
          if (!m8) continue;
        }
        const u32 p = __ffs(m8) - 1;
        m8 &= m8 - 1;
        const u32 pick = (p & 2u) ? ((p & 1u) ? sv.w : sv.z) : ((p & 1u) ? sv.y : sv.x);
        const u32 val = __shfl_sync(pmask, pick, pbase + (p >> 2));
        // run entry: unit0 header, unit1 key, units 2.. value
        const u32 r = fast_entry<false, BIG>(heap + (u64)((val & ((1u << ord_bits) - 1u)) - 1u) * U * 16u, U, 1, kq, ~0ull, dst,
                                        a.val_stride, lane, vlen, pol_stream);
        if (r == 0) { state = 0; break; }
        if (r == 2) break;
      }
    }
  }
  if (lane == 0) {
    if (state == 2) {
      a.pending[atomicAdd(a.n_pending + a.parity, 1u)] = q;
    } else {
      a.st[q] = state == 0 ? 0 : 1;
      a.vlen[q] = vlen;
    }
  }
  // this launch counts in n_pending[parity].  Clearing the other counter here instead of a memset node
  // before the launch measured 20 % SLOWER end to end on B200 (14.98 -> 12.08 G lookups/s), so the
  // memset node stays (RSP_MG_MEMSET=1).
#if !RSP_MG_MEMSET
  if (blockIdx.x == 0 && threadIdx.x == 0) a.n_pending[a.parity ^ 1u] = 0;
#endif
}

// Candidate entry at `ent`: header unit 0, key unit KU, value units KU+1.. (U units in all).
// Returns 0 = served, 1 = not my key (tag false positive), 2 = needs the generic path.
template <bool CG>
__device__ __forceinline__ uint4 ld_entry_unit_m(const uint4* p) {
  if (CG) return __ldcg(p);
  return __ldg(p);
}
template <bool CG, bool BIG>
__device__ __forceinline__ u32 fast_entry_m(const u8* ent, u32 U, u32 KU, const uint4& kq, u64 snap, u8* dst,
                                          u64 val_stride, u32 lane, u32& vlen_out) {
  const uint4* ep = reinterpret_cast<const uint4*>(ent);
  const uint4 hd = ld_entry_unit_m<CG>(ep);
  const uint4 ek = ld_entry_unit_m<CG>(ep + KU);
  const u32 fv = KU + 1;  // first value unit; lane L owns value units L, L+2, L+4, ...
  uint4 v0 = make_uint4(0, 0, 0, 0), v1 = v0, v2 = v0;
  if (!CG) {
    // a run: the entry size U is known before the header arrives, so the first six value units are
    // requested together with header and key (one round trip for values up to 96 bytes)
    if (fv + lane < U) v0 = ld_entry_unit_m<CG>(ep + fv + lane);
    if (fv + lane + 2 < U) v1 = ld_entry_unit_m<CG>(ep + fv + lane + 2);
    if (fv + lane + 4 < U) v2 = ld_entry_unit_m<CG>(ep + fv + lane + 4);
  }
  if (ek.x != kq.x || ek.y != kq.y || ek.z != kq.z || ek.w != kq.w || hd.z != 16) return 1;
  const u64 seq = (((u64)hd.y << 32) | hd.x) >> 8;
  const u32 vu = (hd.w + 15u) >> 4;
  if ((hd.x & 0xffu) != kTypeValue || seq > snap || (!CG && fv + vu > U) || (u64)vu * 16u > val_stride || (!BIG && vu > 6)) return 2;
  uint4* out = reinterpret_cast<uint4*>(dst);
  if (CG) {
    // the memtable: the entry's size is only known from its header, so the value follows in a second trip
    for (u32 u = lane; u < vu; u += FL) out[u] = ld_entry_unit_m<CG>(ep + fv + u);
  } else {
    if (lane < vu) out[lane] = v0;
    if (lane + 2 < vu) out[lane + 2] = v1;
    if (lane + 4 < vu) out[lane + 4] = v2;
    if (BIG)
      for (u32 u = lane + 6; u < vu; u += FL) out[u] = ld_entry_unit_m<CG>(ep + fv + u);  // values > 96 bytes
  }
  vlen_out = hd.w;
  return 0;
}

// One sorted run through its hash index: g0/g1 are the run's 32-byte descriptor in ShardFast's layout (heap pointer,
// index pointer, bucket count, meta).  One bucket = one 32-byte sector, four slots per lane.  Walks the tag matches in
// probe order; a false positive (18-bit tags at 16 K entries: ~1 per 60 K lookups) just moves on to the next
// candidate, a full bucket to the next bucket.  Returns 0 = served, 2 = generic path, 4 = not in this run.
template <bool BIG>
__device__ __forceinline__ u32 probe_one_run(const uint4& g0, const uint4& g1, const uint4& kq, u64 h, u8* dst, u64 val_stride,
                                             u32 lane, u32 pmask, u32 pbase, u32& vlen) {
  const u8* heap = reinterpret_cast<const u8*>(((u64)g0.y << 32) | g0.x);
  const u32 n_buckets = g1.x, ord_bits = g1.y & 0xffu, U = (g1.y >> 8) & 0xffu;
  if (U == 0 || U >= 255) return 2;
  const uint4* hs = reinterpret_cast<const uint4*>(((u64)g0.w << 32) | g0.z);
  u32 bucket = (u32)(((u64)(u32)h * n_buckets) >> 32);
  const u32 tag = (u32)(h >> 32) >> ord_bits;
  u32 m8 = 0, e8 = 1, probe = 0;  // e8 != 0 before the first load only so that the loop loads first
  uint4 sv = make_uint4(0, 0, 0, 0);
#pragma unroll 1
  for (;;) {
    if (!m8) {
      if (probe && e8) return 4;           // an empty slot ends the probe: not here
      if (probe == n_buckets) return 4;    // (a table without an empty slot)
      if (probe) bucket = bucket + 1 == n_buckets ? 0 : bucket + 1;
      probe++;
      sv = ldg_pol(hs + (u64)bucket * 2u + lane, pol_evict_last());
      const u32 m = ((sv.x && (sv.x >> ord_bits) == tag) ? 1u : 0u) | ((sv.y && (sv.y >> ord_bits) == tag) ? 2u : 0u) |
                    ((sv.z && (sv.z >> ord_bits) == tag) ? 4u : 0u) | ((sv.w && (sv.w >> ord_bits) == tag) ? 8u : 0u);
      const u32 e = (sv.x == 0 || sv.y == 0 || sv.z == 0 || sv.w == 0) ? 1u : 0u;
      const u32 mine = m | (e << 4);
      const u32 other = __shfl_xor_sync(pmask, mine, 1);
      m8 = lane ? ((other & 15u) | ((mine & 15u) << 4)) : ((mine & 15u) | ((other & 15u) << 4));
      e8 = (mine | other) >> 4;
      if (!m8) continue;
    }
    const u32 p = __ffs(m8) - 1;
    m8 &= m8 - 1;
    const u32 pick = (p & 2u) ? ((p & 1u) ? sv.w : sv.z) : ((p & 1u) ? sv.y : sv.x);
    const u32 val = __shfl_sync(pmask, pick, pbase + (p >> 2));
    // run entry: unit0 header, unit1 key, units 2.. value
    const u32 r = fast_entry_m<false, BIG>(heap + (u64)((val & ((1u << ord_bits) - 1u)) - 1u) * U * 16u, U, 1, kq, ~0ull, dst,
                                         val_stride, lane, vlen);
    if (r == 0) return 0;
    if (r == 2) return 2;
  }
}

// k_multi_get16m: the same lookup for engines where some shard has SEVERAL sorted runs (between a flush and the next
// merge): the runs are walked newest first, a run that does not hold the key hands over to the next older one
// (per-run descriptors behind the ShardFast array).  The single-run kernel above is kept exactly as measured in r01:
// folding both into one template cost it 20 % (13.3 instead of 16.2 G lookups/s on the same B200, same instruction
// mix — profiles/r02_regression_bisect.md), so the host picks the kernel per launch instead.
template <bool BIG>
__global__ void __launch_bounds__(RSP_MG_TPB, RSP_MG_MINB) k_multi_get16m(GetArgs a) {
  constexpr bool MULTI = true;
  const u32 q = (blockIdx.x * blockDim.x + threadIdx.x) / FL;
  const u32 lane = threadIdx.x & (FL - 1);
  const u32 pbase = (threadIdx.x & 31u) & ~1u;
  const u32 pmask = 3u << pbase;  // the two lanes of this lookup always branch together
  if (q >= a.n) return;
  // (1)
  u32 six = __ldg(a.shard_ix + q);
  const bool bad_shard = six >= a.max_shards;
  if (bad_shard) six = 0;
  const uint4 kq = __ldg(reinterpret_cast<const uint4*>(a.keys) + q);
  const uint4 f0 = __ldg(reinterpret_cast<const uint4*>(a.fast + six));
  const uint4 f1 = __ldg(reinterpret_cast<const uint4*>(a.fast + six) + 1);
  const u32 n_runs = (f1.y >> 16) & 0xffu;
  const u64 k0 = ((u64)kq.y << 32) | kq.x, k1 = ((u64)kq.w << 32) | kq.z;
  const u64 h = hash_final(hash_step(hash_step(hash_init(16), k0), k1));
  u8* dst = a.vals + (u64)q * a.val_stride;
  u32 state = 3;  // 0 served, 2 generic path, 3 undecided, 4 not found
  u32 vlen = 0;
  if ((!MULTI && n_runs > 1) || ((a.val_stride | reinterpret_cast<uintptr_t>(a.vals)) & 15u) || bad_shard || !(f1.y & FAST_META_LIVE)) state = 2;
  bool in_mem = false;
  if (state == 3 && f1.z /* mt_count */) {
    // the shard's memtable filter (L2-resident, behind the descriptors): a clear bit = the key is not in the memtable
    const u32 fb = mt_filter_bit(h);
    const u32 fw = __ldcg(reinterpret_cast<const u32*>(a.fast + (size_t)a.max_shards * (1u + RSP_MAX_RUNS)) + (size_t)six * MT_FILTER_WORDS + (fb >> 5));
    in_mem = (fw >> (fb & 31u)) & 1u;
  }
  if (in_mem) {
    // ---- memtable: eight u64 slots from the home position, four per lane; descriptor through L2
    const uint4* dp = reinterpret_cast<const uint4*>(a.shards + six);
    const uint4 d0 = __ldcg(dp), d1 = __ldcg(dp + 1), d3 = __ldcg(dp + 3);
    const u8* heap = reinterpret_cast<const u8*>(((u64)d0.y << 32) | d0.x);
    const u64* sp = reinterpret_cast<const u64*>(((u64)d0.w << 32) | d0.z);
    const u32 mask = d1.z;
    const u64 snap = ((u64)d3.w << 32) | d3.z;
    const u32 tag = hash_tag32(h);
    u32 cand = 0, info = 0;  // info: matches | (position of my first empty + 1) << 8
#pragma unroll
    for (u32 i = 0; i < 4; i++) {
      const u64 sv = ldcg64(sp + (((u32)h + 4u * lane + i) & mask));
      if (sv == 0) { if (!(info >> 8)) info |= (4u * lane + i + 1u) << 8; }
      else if ((u32)(sv >> 32) == tag && !(info >> 8)) { if (!cand) cand = (u32)sv; info++; }
    }
    const u32 o_cand = __shfl_xor_sync(pmask, cand, 1), o_info = __shfl_xor_sync(pmask, info, 1);
    // lane 1's slots come after lane 0's in probe order: they count only if lane 0 saw no empty slot
    const u32 lo_info = lane ? o_info : info, hi_info = lane ? info : o_info;
    const u32 lo_cand = lane ? o_cand : cand, hi_cand = lane ? cand : o_cand;
    const bool lo_empty = (lo_info >> 8) != 0;
    const u32 n_match = (lo_info & 0xffu) + (lo_empty ? 0u : (hi_info & 0xffu));
    const bool any_empty = lo_empty || (hi_info >> 8) != 0;
    if (n_match == 1) {
      const u32 c = (lo_info & 0xffu) ? lo_cand : hi_cand;
      // memtable entry: unit0 header, unit1 link, unit2 key, units 3.. value
      const u32 r = fast_entry_m<true, BIG>(heap + (u64)(c - 1u) * 16u, 7, 2, kq, snap, dst, a.val_stride, lane, vlen);
      state = r == 0 ? 0 : 2;
    } else if (n_match > 1 || !any_empty) {
      state = 2;
    }
  }
  if (state == 3) {
    // ---- the sorted runs, newest first
    state = 4;
    const u32 nr = MULTI ? n_runs : min(n_runs, 1u);
    for (u32 r = 0; r < nr; r++) {
      uint4 g0 = f0, g1 = f1;
      if (MULTI && r) {
        const uint4* fr = reinterpret_cast<const uint4*>(a.fast + a.max_shards) + ((u64)six * RSP_MAX_RUNS + r) * 2u;
        g0 = __ldg(fr);
        g1 = __ldg(fr + 1);
      }
      const u32 rs = probe_one_run<BIG>(g0, g1, kq, h, dst, a.val_stride, lane, pmask, pbase, vlen);
      if (rs != 4) { state = rs; break; }
    }
  }
  if (lane == 0) {
    if (state == 2) {
      a.pending[atomicAdd(a.n_pending + a.parity, 1u)] = q;
    } else {
      a.st[q] = state == 0 ? 0 : 1;
      a.vlen[q] = vlen;
    }
  }
}

// generic path over the queries the fast kernel deferred; a small fixed grid strides over the list
__global__ void __launch_bounds__(256) k_multi_get_pending(GetArgs a) {
  const u32 lane = threadIdx.x & (MG_LANES - 1);
  const u32 gbase = (threadIdx.x & 31u) & ~(MG_LANES - 1u);
  const u32 gmask = ((1u << MG_LANES) - 1u) << gbase;
  const u32 n = __ldcg(a.n_pending + a.parity);
  const u32 groups = gridDim.x * (blockDim.x / MG_LANES);
  for (u32 i = (blockIdx.x * blockDim.x + threadIdx.x) / MG_LANES; i < n; i += groups)
    lookup_generic(a, __ldcg(a.pending + i), lane, gmask, gbase);
}

void launch_multi_get(const GetArgs& a, cudaStream_t s) {
  if (!a.n) return;
  const u32 per_block = 256 / MG_LANES;
  const u32 grid = (a.n + per_block - 1) / per_block;
  if (a.klen_fixed == 16 && (reinterpret_cast<uintptr_t>(a.keys) & 15u) == 0 && a.pending && a.fast) {
    // this launch counts in n_pending[parity]; a memset node clears it
#if RSP_MG_MEMSET
    cudaMemsetAsync(a.n_pending + a.parity, 0, 4, s);
#endif
    const u32 g16 = (a.n + RSP_MG_TPB / FL - 1) / (RSP_MG_TPB / FL);
    const bool multi = a.multirun != 0;
    if (a.val_stride > 96) {
      if (multi) k_multi_get16m<true><<<g16, RSP_MG_TPB, 0, s>>>(a); else k_multi_get16<true><<<g16, RSP_MG_TPB, 0, s>>>(a);
    } else {
      if (multi) k_multi_get16m<false><<<g16, RSP_MG_TPB, 0, s>>>(a); else k_multi_get16<false><<<g16, RSP_MG_TPB, 0, s>>>(a);
    }
    k_multi_get_pending<<<std::min<u32>(grid, 148u), 256, 0, s>>>(a);
  } else {
    k_multi_get<<<grid, 256, 0, s>>>(a);
  }
}

// ------------------------------------------------------------------------------------------------
// k_get_versions — slow path for host-folded merge operators: dump the version stack
// ------------------------------------------------------------------------------------------------
struct DumpVisitor {
  u8* out;
  u64 cap;
  u32 used, n_rec;
  bool done;
  __device__ bool visit(u32 type, const u8* vptr, u32 vlen) {
    const u32 rec = 8u + ((vlen + 3u) & ~3u);
    if ((u64)used + rec <= cap) {
      *reinterpret_cast<u32*>(out + used) = type;
      *reinterpret_cast<u32*>(out + used + 4) = vlen;
      for (u32 b = 0; b < vlen; b++) out[used + 8 + b] = __ldcg(vptr + b);
      n_rec++;
    }
    used += rec;
    if (type != kTypeMerge) done = true;
    return done;
  }
};

__global__ void k_get_versions(VersionsArgs a) {
  const u32 q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= a.n) return;
  const u32 lane_in_warp = threadIdx.x & 31u;
  const ShardDev* sd = a.views ? nullptr : a.shards + a.shard_ix[q];
  const u64 o = a.koff[q];
  const u32 klen = (u32)(a.koff[q + 1] - o);
  DumpVisitor v{a.out + (u64)q * a.out_stride, a.out_stride, 0, 0, false};
  bool stopped;
  if (a.views) {  // a pinned iterator snapshot: sorted runs only
    const ScanView& vw = a.views[q];
    const u64 h = hash_key(a.keys + o, klen);
    for (u32 ri = 0; ri < vw.n_runs && !v.done; ri++)
      walk_run<1>(vw.runs[ri], a.keys + o, klen, h, 0, 1u << lane_in_warp, lane_in_warp, v);
  } else {
    walk_shard<1>(sd, a.keys + o, klen, 0, 1u << lane_in_warp, lane_in_warp, v, stopped);
  }
  a.n_rec[q] = v.n_rec;
  a.need[q] = v.used;
}

void launch_get_versions(const VersionsArgs& a, cudaStream_t s) {
  if (!a.n) return;
  k_get_versions<<<(a.n + 63) / 64, 64, 0, s>>>(a);
}

// ------------------------------------------------------------------------------------------------
// k_multi_scan — Seek + N x Next/Prev over the sorted runs (one warp per scan)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int cmp_run_key(const RunDev& r, u32 ord, const u8* kp, u32 klen) {
  const u8* e = run_entry(r, ord);
  const u32 eklen = __ldg(reinterpret_cast<const u32*>(e) + 2);
  return -cmp_key_vs_padded(kp, klen, reinterpret_cast<const u64*>(e + 16), eklen);  // sign of (entry - key)
}
// first ordinal whose key is >= key (strict: > key)
__device__ u32 run_lower_bound(const RunDev& r, const u8* kp, u32 klen, bool strict) {
  u32 lo = 0, hi = r.n_ent;
  // block index first: 8-byte big-endian prefixes of every RSP_BLOCK_ENTRIES-th entry
  if (r.n_blocks > 1 && klen) {
    const u64 pfx = key_prefix_be(kp, klen);
    u32 bl = 0, bh = r.n_blocks;  // last block whose first prefix < pfx bounds the answer from below
    while (bl < bh) {
      const u32 m = (bl + bh) >> 1;
      if (__ldg(r.blk_pfx + m) < pfx) bl = m + 1; else bh = m;
    }
    lo = bl ? (bl - 1) * RSP_BLOCK_ENTRIES : 0;
    // first block whose prefix > pfx bounds it from above
    u32 cl = bl, ch = r.n_blocks;
    while (cl < ch) {
      const u32 m = (cl + ch) >> 1;
      if (__ldg(r.blk_pfx + m) <= pfx) cl = m + 1; else ch = m;
    }
    hi = min(r.n_ent, cl * RSP_BLOCK_ENTRIES);
  }
  while (lo < hi) {
    const u32 m = (lo + hi) >> 1;
    const int c = cmp_run_key(r, m, kp, klen);
    if (c < 0 || (strict && c == 0)) lo = m + 1; else hi = m;
  }
  return lo;
}

struct EntRef {
  const u8* e;
  u32 klen, vlen, type;
  __device__ const u64* key() const { return reinterpret_cast<const u64*>(e + 16); }
  __device__ const u8* val() const { return e + 16u + 16u * units_of(klen); }
};
__device__ __forceinline__ EntRef load_ent(const RunDev& r, u32 ord) {
  EntRef x;
  x.e = run_entry(r, ord);
  const uint4 hd = __ldg(reinterpret_cast<const uint4*>(x.e));
  x.type = hd.x & 0xffu; x.klen = hd.z; x.vlen = hd.w;
  return x;
}

__device__ __forceinline__ void warp_copy_bytes(u8* dst, const u8* src, u32 n, u32 lane) {
  for (u32 b = lane; b < n; b += 32) dst[b] = src[b];
}

// ---- TMA-staged block index + warp-ballot search (Seek on a sorted run) --------------------------------
// The run's block index (8-byte big-endian first-key prefix per RSP_BLOCK_ENTRIES entries) is pulled into
// shared memory with ONE bulk asynchronous copy (cp.async.bulk global -> shared, completion on an mbarrier:
// the TMA engine, SASS UBLKCP) instead of a dependent chain of ~log2(n_blocks) global loads; the warp then
// counts prefixes below / not above the target 32 at a time with ballots, and resolves the final position
// inside the 1-2 candidate blocks by comparing 32 entry keys at once.
// independent loads per lane in the streaming loop: 4 gives 181 M scans/s, the plain loop (one load in flight per
// warp: LDG, STG, LDG, ...) 115 M (profiles/r02_experiments/)
#define RSP_SCAN_UNROLL 4
constexpr u32 SCAN_WARPS = 4;
constexpr u32 SCAN_STAGE_PFX = 512;  // prefixes staged per warp (4 KB): runs up to 16 K entries

#ifdef RSP_EMUL
// tests/emul: the bulk copy completes at issue; the mbarrier word counts completed phases
__device__ __forceinline__ void tma_load_1d(void* smem_dst, const void* gmem_src, u32 bytes, u64* mbar) {
  memcpy(smem_dst, gmem_src, bytes);
  *mbar += 1;
}
__device__ __forceinline__ void mbar_init(u64* mbar, u32) { *mbar = 0; }
__device__ __forceinline__ bool mbar_wait(u64* mbar, u32 parity) {
  while ((*mbar & 1u) == parity) emul_yield();
  return true;
}
#else
__device__ __forceinline__ void tma_load_1d(void* smem_dst, const void* gmem_src, u32 bytes, u64* mbar) {
  const u32 dst = (u32)__cvta_generic_to_shared(smem_dst);
  const u32 bar = (u32)__cvta_generic_to_shared(mbar);
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(gmem_src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_init(u64* mbar, u32 count) {
  const u32 bar = (u32)__cvta_generic_to_shared(mbar);
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
// Bounded wait: try_wait itself blocks for a hardware time slice per attempt, so 2^20 attempts are seconds, not a
// hang.  false = the bulk copy never completed (never seen; the caller then searches the index in global memory).
__device__ __forceinline__ bool mbar_wait(u64* mbar, u32 parity) {
  const u32 bar = (u32)__cvta_generic_to_shared(mbar);
  for (u32 tries = 0; tries < (1u << 20); tries++) {
    u32 ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n" : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    if (ok) return true;
  }
  return false;
}
#endif

// warp-cooperative lower bound: first ordinal of R whose key is >= key (strict: > key)
__device__ u32 run_lower_bound_warp(const RunDev& R, const u8* kp, u32 klen, bool strict, u64* s_pfx, u64* mbar,
                                    u32 lane) {
  u32 lo = 0, hi = R.n_ent;
  if (R.n_blocks > 1 && klen) {
    if (lane == 0) tma_load_1d(s_pfx, R.blk_pfx, (R.n_blocks * 8u + 15u) & ~15u, mbar);
    const u64 pfx = key_prefix_be(kp, klen);
    if (!__all_sync(0xffffffffu, mbar_wait(mbar, 0))) return run_lower_bound(R, kp, klen, strict);
    u32 n_lt = 0, n_le = 0;
    for (u32 b = 0; b < R.n_blocks; b += 32) {
      const u64 p = b + lane < R.n_blocks ? s_pfx[b + lane] : ~0ull;
      const u32 in = b + lane < R.n_blocks;
      n_lt += __popc(__ballot_sync(0xffffffffu, in && p < pfx));
      n_le += __popc(__ballot_sync(0xffffffffu, in && p <= pfx));
    }
    lo = n_lt ? (n_lt - 1) * RSP_BLOCK_ENTRIES : 0;
    hi = min(R.n_ent, n_le * RSP_BLOCK_ENTRIES);
  }
  // entries [lo, hi) are sorted: the answer is lo + #(entries below the target)
  u32 below = 0;
  for (u32 b = lo; b < hi; b += 32) {
    bool is_below = false;
    if (b + lane < hi) {
      const int c = cmp_run_key(R, b + lane, kp, klen);
      is_below = c < 0 || (strict && c == 0);
    }
    const u32 m = __ballot_sync(0xffffffffu, is_below);
    below += __popc(m);
    if (m != 0xffffffffu) break;  // sorted: once an entry is not below, none after it is
  }
  return lo + below;
}

__device__ __forceinline__ void multi_scan_body(const ScanArgs& a) {
  __shared__ __align__(16) u64 s_pfx_all[SCAN_WARPS][SCAN_STAGE_PFX];
  __shared__ __align__(8) u64 s_mbar[SCAN_WARPS];
  {
    const u32 wi = threadIdx.x >> 5;
    if ((threadIdx.x & 31u) == 0) mbar_init(&s_mbar[wi], 1);
    __syncwarp();
  }
  const u32 q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const u32 lane = threadIdx.x & 31u;
  if (q >= a.n) return;
  const RunDev* runs;
  u32 n_runs, merge_op;
  if (a.views) {
    runs = a.views[q].runs; n_runs = a.views[q].n_runs; merge_op = a.views[q].merge_op;
  } else {
    // unknown / closed shard: InvalidArgument, no output bytes.  An unknown id reads slot 0 (never past the table), so
    // that `live` is loaded together with the fields below rather than ahead of them: an extra dependent load at the
    // head of every scan costs the short-lived scan warps a third of their rate
    const u32 six = a.shard_ix[q];
    const bool known = six < a.max_shards;
    const ShardDev* sd = a.shards + (known ? six : 0u);
    runs = sd->runs; n_runs = sd->n_runs; merge_op = sd->merge_op;
    if (!known || !sd->live) {
      if (lane == 0) {
        a.n_out[q] = 0;
        a.st[q] = 4;
      }
      return;
    }
  }
  const u8* kp;
  u32 klen;
  if (a.klen_fixed) { klen = a.klen_fixed; kp = a.keys + (u64)q * klen; }
  else { const u64 o = a.koff[q]; klen = (u32)(a.koff[q + 1] - o); kp = a.keys + o; }
  const u32 fl = a.flags ? a.flags[q] : 0u;
  const bool exclusive = fl & 1u, reverse = fl & 2u, extreme = fl & 4u;
  u8* out = a.out + (u64)q * a.out_stride;
  u64 used = 0;
  u32 n_out = 0;
  i32 st = 0;

  // ---- fast path: one fully compacted run of fixed-size Puts, forward scan.  Seek (block index + binary
  // search), then the warp streams the consecutive entries out as 8-byte words: record i =
  // [u32 klen][u32 vlen][key][value] at out + i * (8 + klen + vlen).
  if (n_runs == 1 && !reverse && (runs[0].flags & RUN_ALL_PUT_FIXED)) {
    const RunDev& R = runs[0];
    const u32 kl = R.kv_len & 0xffffu, vl = R.kv_len >> 16;
    const u32 rec = 8u + kl + vl;
    if ((kl & 15u) == 0 && (vl & 7u) == 0 && ((reinterpret_cast<uintptr_t>(out) | a.out_stride) & 7u) == 0) {
      u32 start = 0;
      if (!extreme) {
        const u32 wi = threadIdx.x >> 5;
        start = R.n_blocks <= SCAN_STAGE_PFX ? run_lower_bound_warp(R, kp, klen, exclusive, s_pfx_all[wi], &s_mbar[wi], lane)
                                             : run_lower_bound(R, kp, klen, exclusive);
      }
      u32 cnt = min(a.max_entries, R.n_ent - start);
      i32 fst = 0;
      if ((u64)cnt * rec > a.out_stride) { cnt = (u32)(a.out_stride / rec); fst = 7; }
      const u32 wpr = rec >> 3;  // 8-byte words per record
      const u64* src = reinterpret_cast<const u64*>(R.heap) + (u64)start * R.uniform_units * 2u;
      u64* dst = reinterpret_cast<u64*>(out);
      const u32 total = cnt * wpr;
      // RSP_SCAN_UNROLL loads are issued before the first of their stores: with one load in flight per warp (what
      // the plain loop compiles to: LDG, STG, LDG, ...) the kernel is bound by latency x occupancy, not by HBM
      for (u32 w0 = lane; w0 < total; w0 += 32u * RSP_SCAN_UNROLL) {
        u64 v[RSP_SCAN_UNROLL];
#pragma unroll
        for (u32 u = 0; u < RSP_SCAN_UNROLL; u++) {
          const u32 w = w0 + 32u * u;
          if (w < total) {
            const u32 r = w / wpr, jw = w - r * wpr;
            // source words of entry r: word 1 = (klen, vlen); key from word 2; value follows (klen % 16 == 0)
            v[u] = __ldg(src + (u64)r * R.uniform_units * 2u + 1 + jw);
          }
        }
#pragma unroll
        for (u32 u = 0; u < RSP_SCAN_UNROLL; u++) {
          const u32 w = w0 + 32u * u;
          if (w < total) dst[w] = v[u];
        }
      }
      if (lane == 0) {
        a.n_out[q] = cnt;
        a.st[q] = fst;
      }
      return;
    }
  }

  // ---- general path: k-way newest-wins merge over the pinned runs.
  // FORWARD scans are lane-parallel: lane r owns run r's cursor and keeps its head entry cached (pointer, lengths,
  // type, 8-byte big-endian key prefix).  Every lane seeks its own run at the same time; per output key the warp takes
  // the minimum prefix by shuffles, settles prefix ties by full-key compares done in parallel by the tied lanes, and
  // the runs that hold the key are visited newest first while their lanes already load their next heads.
  // REVERSE scans (Iterator::Prev, rare) keep the scalar walk: every lane executes the same code.
  u32 cur[RSP_MAX_RUNS];
  // forward state of lane r (r < n_runs)
  u32 my_cur = 0, h_klen = 0, h_vlen = 0, h_type = 0;
  const u8* h_e = nullptr;
  u64 h_pfx = 0;
  bool h_valid = false;
  auto load_head = [&]() {
    h_valid = lane < n_runs && my_cur < runs[lane].n_ent;
    if (h_valid) {
      h_e = run_entry(runs[lane], my_cur);
      const uint4 hd = __ldg(reinterpret_cast<const uint4*>(h_e));
      h_type = hd.x & 0xffu; h_klen = hd.z; h_vlen = hd.w;
      h_pfx = h_klen ? bswap64(__ldg(reinterpret_cast<const u64*>(h_e + 16))) : 0ull;
    }
  };
  if (!reverse) {
    if (lane < n_runs) my_cur = extreme ? 0u : run_lower_bound(runs[lane], kp, klen, exclusive);
    load_head();
  } else {
    for (u32 r = 0; r < n_runs; r++) {
      if (extreme) cur[r] = runs[r].n_ent;
      else cur[r] = run_lower_bound(runs[r], kp, klen, !exclusive);  // entries < key (or <= key)
    }
  }

  while (n_out < a.max_entries) {
    EntRef bk;
    Acc acc;
    acc.init(merge_op);
    if (!reverse) {
      const u32 vmask = __ballot_sync(0xffffffffu, h_valid);
      if (!vmask) break;
      // minimum prefix over the valid heads (lanes 0 .. 7 hold the runs: three butterfly steps)
      u64 mp = h_valid ? h_pfx : ~0ull;
#pragma unroll
      for (u32 d = 1; d < RSP_MAX_RUNS; d <<= 1) {
        const u64 o = __shfl_xor_sync(0xffffffffu, mp, d);
        mp = o < mp ? o : mp;
      }
      mp = __shfl_sync(0xffffffffu, mp, 0);
      u32 cand = __ballot_sync(0xffffffffu, h_valid && h_pfx == mp);
      u32 group, w;
      for (;;) {  // the smallest full key among the tied prefixes, and every run whose head is that key
        w = (u32)__ffs(cand) - 1u;
        const u64 wk = __shfl_sync(0xffffffffu, (u64)reinterpret_cast<uintptr_t>(h_e), w);
        const u32 wkl = __shfl_sync(0xffffffffu, h_klen, w);
        int c = 0;
        const bool mine = ((cand >> lane) & 1u) && lane != w;
        if (mine) c = cmp_padded(reinterpret_cast<const u64*>(h_e + 16), h_klen, reinterpret_cast<const u64*>(reinterpret_cast<const u8*>(wk) + 16), wkl);
        const u32 less = __ballot_sync(0xffffffffu, mine && c < 0);
        if (less) { cand = less; continue; }
        group = __ballot_sync(0xffffffffu, mine && c == 0) | (1u << w);
        break;
      }
      bk.e = reinterpret_cast<const u8*>(__shfl_sync(0xffffffffu, (u64)reinterpret_cast<uintptr_t>(h_e), w));
      bk.klen = __shfl_sync(0xffffffffu, h_klen, w);
      bk.vlen = 0; bk.type = 0;
      // newest run first; inside a run the versions of a key follow each other, newest first
      for (u32 g = group; g;) {
        const u32 r = (u32)__ffs(g) - 1u;
        g &= g - 1u;
        for (;;) {
          const u32 t = __shfl_sync(0xffffffffu, h_type, r), vl = __shfl_sync(0xffffffffu, h_vlen, r);
          const u64 ep = __shfl_sync(0xffffffffu, (u64)reinterpret_cast<uintptr_t>(h_e), r);
          const u32 kl = __shfl_sync(0xffffffffu, h_klen, r);
          if (!acc.done) acc.visit(t, reinterpret_cast<const u8*>(ep) + 16u + 16u * units_of(kl), vl);
          bool same = false;
          if (lane == r) {
            my_cur++;
            load_head();
            same = h_valid && cmp_padded(reinterpret_cast<const u64*>(h_e + 16), h_klen, bk.key(), bk.klen) == 0;
          }
          if (!__shfl_sync(0xffffffffu, (u32)same, r)) break;
        }
      }
    } else {
    // pick the next user key: the maximum over the reverse cursors (newest run wins ties)
    int best = -1;
    for (u32 r = 0; r < n_runs; r++) {
      if (cur[r] == 0) continue;
      const EntRef x = load_ent(runs[r], cur[r] - 1);
      if (best < 0) { best = (int)r; bk = x; continue; }
      const int c = cmp_padded(x.key(), x.klen, bk.key(), bk.klen);
      if (c > 0) { best = (int)r; bk = x; }
    }
    if (best < 0) break;
    // resolve this key across the runs that hold it, newest run first
    for (u32 r = 0; r < n_runs; r++) {
      const RunDev& R = runs[r];
      // group = [g, cur[r]) with the same key; versions are newest-first from g upward
      u32 g = cur[r];
      while (g > 0) {
        const EntRef x = load_ent(R, g - 1);
        if (cmp_padded(x.key(), x.klen, bk.key(), bk.klen) != 0) break;
        g--;
      }
      for (u32 o = g; o < cur[r] && !acc.done; o++) {
        const EntRef x = load_ent(R, o);
        acc.visit(x.type, x.val(), x.vlen);
      }
      cur[r] = g;
    }
    }
    acc.end_of_versions();
    if (acc.status == 1) continue;  // deleted
    u32 vlen = 0;
    bool host_fold = false, merge_failed = false;
    if (acc.status == ST_NEED_HOST_MERGE) {
      // the operator lives on the host: hand back the key alone (vlen marker 0xffffffff)
      if (st == 0) st = ST_NEED_HOST_MERGE;
      host_fold = true;
    } else if (acc.status != 0) {
      // DBIter keeps the key with an empty value and records the (sticky) status; the record carries the marker
      // SCAN_VLEN_MERGE_FAILED so that an iterator can raise the status when it REACHES this key, as DBIter does
      st = (i32)mk_status((u32)acc.status, acc.msg);
      merge_failed = true;
    } else {
      vlen = acc.res_len;
    }
    const u64 rec = 8ull + bk.klen + vlen;
    // out of room: INCOMPLETE, or its flag on top of a status that is already there (host-fold request, failed merge)
    if (used + rec > a.out_stride) { st = st == 0 ? 7 : (st | SCAN_ST_TRUNCATED); break; }
    if (lane == 0) {
      u8 hdr[8];
      const u32 vl_out = host_fold ? SCAN_VLEN_HOST_FOLD : (merge_failed ? SCAN_VLEN_MERGE_FAILED : vlen);
      for (u32 b = 0; b < 4; b++) { hdr[b] = (u8)(bk.klen >> (8 * b)); hdr[4 + b] = (u8)(vl_out >> (8 * b)); }
      for (u32 b = 0; b < 8; b++) out[used + b] = hdr[b];
    }
    warp_copy_bytes(out + used + 8, reinterpret_cast<const u8*>(bk.key()), bk.klen, lane);
    if (vlen) {
      if (acc.imm) {
        if (lane < 8) out[used + 8 + bk.klen + lane] = (u8)(acc.res_imm >> (8u * lane));
      } else {
        warp_copy_bytes(out + used + 8 + bk.klen, acc.res_ptr, vlen, lane);
      }
    }
    used += rec;
    n_out++;
  }
  if (lane == 0) {
    a.n_out[q] = n_out;
    a.st[q] = st;
  }
}

__global__ void __launch_bounds__(128) k_multi_scan(ScanArgs a) { multi_scan_body(a); }

void launch_multi_scan(const ScanArgs& a, cudaStream_t s) {
  if (!a.n) return;
  k_multi_scan<<<(a.n + 3) / 4, 128, 0, s>>>(a);
}
}  // namespace rsp
