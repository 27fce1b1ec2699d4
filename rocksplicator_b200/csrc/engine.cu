// engine.cu — host side of librsp_b200.so: device memory, shard bookkeeping, the batching front-end of
// the apply path, flush/compaction scheduling, iterators, and the extern "C" ABI of include/rsp_b200.h.
//
// What it stands in for: the rocksdb::DB object the reference keeps behind
// rocksdb_replicator/rocksdb_wrapper.cpp (Write / GetLatestSequenceNumber) and
// rocksdb_admin/application_db.cpp:78-144 (Get / MultiGet / NewIterator / CompactRange).
// No oracle, no CPU fallback: every data-path call ends in the kernels of k_*.cu or fails.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <stdexcept>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include "../../include/rsp_b200.h"
#include "arena.h"
#include "stager.h"
#include "kernels.h"

using namespace rsp;

// A failed CUDA call inside the library must not take the host process down (the header promises status codes): it
// is thrown, unwinds through the RAII locks, and is turned into RSP_IO_ERROR at the C ABI (abi_guard below); the text
// is kept for rsp_engine_last_error.  Device-side faults are sticky in the CUDA context: later calls fail the same way.
struct CudaFailure : public std::runtime_error {
  explicit CudaFailure(const std::string& m) : std::runtime_error(m) {}
};
static std::mutex g_fail_mu;
static std::string g_fail_text;
[[noreturn]] static void throw_cuda(cudaError_t e, const char* file, int line) {
  char buf[384];
  snprintf(buf, sizeof(buf), "CUDA error %s at %s:%d: %s", cudaGetErrorName(e), file, line, cudaGetErrorString(e));
  fprintf(stderr, "[rsp_b200] %s\n", buf);
  {
    std::lock_guard<std::mutex> g(g_fail_mu);
    g_fail_text = buf;
  }
  throw CudaFailure(buf);
}
#define CUDA_OK(x)                                            \
  do {                                                        \
    cudaError_t e_ = (x);                                     \
    if (e_ != cudaSuccess) throw_cuda(e_, __FILE__, __LINE__); \
  } while (0)
// what an extern "C" entry point answers when its body threw
static int abi_caught() noexcept {
  try {
    throw;
  } catch (const CudaFailure&) {
    return RSP_IO_ERROR;
  } catch (const std::bad_alloc&) {
    std::lock_guard<std::mutex> g(g_fail_mu);
    g_fail_text = "out of host memory";
    return RSP_IO_ERROR;
  } catch (const std::exception& ex) {
    std::lock_guard<std::mutex> g(g_fail_mu);
    g_fail_text = ex.what();
    return RSP_IO_ERROR;
  } catch (...) {
    return RSP_IO_ERROR;
  }
}

static const char* kMsgText[MSG_COUNT] = {
    "",
    "Corruption: malformed WriteBatch (too small)",
    "Corruption: bad WriteBatch Put",
    "Corruption: bad WriteBatch Delete",
    "Corruption: bad WriteBatch Merge",
    "Corruption: bad WriteBatch Blob",
    "Corruption: unknown WriteBatch tag",
    "Corruption: WriteBatch has wrong count",
    "Invalid argument: Invalid column family specified in write batch",
    "Not implemented: WriteBatch tag outside the replicated hot path",
    "Invalid argument: merge_operator is not properly initialized.",
    "Corruption: Error: Could not perform merge.",
    "Busy: update larger than the reserved memtable",
    "Corruption: bad EndPrepare XID",
    "Corruption: bad Commit XID",
    "Corruption: bad Rollback XID",
    "Corruption: bad WriteBatch DeleteRange",
};

// ------------------------------------------------------------------------------------------------
// device arena (arena.h): best-fit blocks with splitting and coalescing over cudaMalloc'ed slabs
// ------------------------------------------------------------------------------------------------
static void* arena_slab_alloc(size_t n) {
  void* p = nullptr;
  CUDA_OK(cudaMalloc(&p, n));
  return p;
}
static void arena_slab_free(void* p) { cudaFree(p); }

// growable device / pinned scratch
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  void* get(size_t n) {
    if (n > cap) {
      if (p) CUDA_OK(cudaFree(p));
      cap = std::max(n, cap * 2);
      CUDA_OK(cudaMalloc(&p, cap));
    }
    return p;
  }
  void destroy() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};
struct PinBuf {
  void* p = nullptr;
  size_t cap = 0;
  void* get(size_t n) {
    if (n > cap) {
      if (p) CUDA_OK(cudaFreeHost(p));
      cap = std::max(n, cap * 2);
      CUDA_OK(cudaHostAlloc(&p, cap, cudaHostAllocDefault));
    }
    return p;
  }
  void destroy() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
};

// ------------------------------------------------------------------------------------------------
// the block index is staged by one TMA bulk copy, whose size is a multiple of 16 bytes (k_read.cu run_lower_bound_warp)
static inline size_t blk_pfx_bytes(u32 n_blocks) { return ((size_t)n_blocks * 8 + 15) & ~(size_t)15; }

struct Run {
  Arena* arena;
  u8* heap = nullptr;
  u32* ent_off = nullptr;
  u32* hslots = nullptr;
  u64* blk_pfx = nullptr;
  u32 n_ent = 0, heap_units = 0, n_buckets = 0, ord_bits = 0, uniform_units = 0, n_blocks = 0, flags = 0, kv_len = 0;
  RunDev dev() const {
    RunDev r;
    r.heap = heap; r.ent_off = ent_off; r.hslots = hslots; r.blk_pfx = blk_pfx;
    r.n_ent = n_ent; r.n_buckets = n_buckets; r.ord_bits = ord_bits; r.uniform_units = uniform_units;
    r.n_blocks = n_blocks; r.heap_units = heap_units; r.flags = flags; r.kv_len = kv_len;
    return r;
  }
  size_t bytes() const { return (size_t)heap_units * 16; }
  ~Run() {
    arena->release(heap, (size_t)heap_units * 16);
    arena->release(ent_off, (size_t)n_ent * 4);
    arena->release(hslots, (size_t)n_buckets * RUN_BUCKET_SLOTS * 4);
    arena->release(blk_pfx, blk_pfx_bytes(n_blocks));
  }
};

struct rsp_engine;

struct rsp_shard {
  rsp_engine* eng;
  std::string name;
  u32 index;
  rsp_shard_opts opts;
  ShardDev h;  // host mirror of the device descriptor
  // upper bounds of ticks that were reserved (and possibly launched) but whose results are not folded into `h` yet:
  // a later tick is reserved against mirror + in-flight, so several ticks can be on the device back to back
  u64 inflight_units = 0, inflight_ents = 0;
  std::atomic<u64> last_seq{0};
  u32 latch = 0;
  std::vector<std::shared_ptr<Run>> runs;  // [0] newest
  std::string last_error;
  std::mutex err_mu;
  rsp_stats stats{};
  size_t mt_heap_bytes = 0, mt_slot_bytes = 0, mt_ent_bytes = 0;
  bool counted_multirun = false;  // this shard is counted in the engine's n_multirun
  bool merging = false;           // a background merge of runs [bg_first_pinned ..] is in flight
  u64 uid = 0;                    // never reused: a background merge recognises the shard it planned for
  const Run* bg_first_pinned = nullptr;
};

struct rsp_staged {
  rsp_engine* eng;
  size_t n = 0;
  std::vector<u32> order;       // staged position -> caller's batch index
  std::vector<rsp_shard*> group_shard;
  std::vector<u32> need_units, need_ents;
  void* dev = nullptr;          // device image
  size_t dev_bytes = 0;
  TickDev tick{};
  cudaStream_t last_stream = nullptr;
  size_t res_bytes = 0;         // gres + per-batch status words, contiguous
  std::vector<u32> group_first;  // staged position of each group's first batch (+ total at the end)
  bool identity_order = false;   // packed ticks: staged position == caller's batch index
  bool fused = false;            // small batches: the whole tick is one launch of k_tick_fused
  FusedTick ftick{};
  mutable bool reserved = false; // its upper bounds are counted in the shards' in-flight totals until the results are folded
};

struct ReadCombiner;
struct ApplyCombiner;
struct Compactor;

struct rsp_engine {
  int device = 0;
  // staging combiners (created on first use): concurrent readers / writers share device batches (stager.h)
  std::mutex comb_mu;
  ReadCombiner* read_comb = nullptr;
  ApplyCombiner* apply_comb = nullptr;
  std::atomic<ReadCombiner*> read_comb_ready{nullptr};
  std::atomic<ApplyCombiner*> apply_comb_ready{nullptr};
  rsp_engine_cfg cfg{};
  std::mutex mu;  // serialises GPU work issued through the ABI
  cudaStream_t st = nullptr;
  cudaStream_t cs[3] = {nullptr, nullptr, nullptr};  // chunk streams of the pipelined host MultiGet
  cudaEvent_t cs_done[3] = {nullptr, nullptr, nullptr};
  Arena arena;
  ShardDev* d_shards = nullptr;
  ShardFast* d_fast = nullptr;
  std::vector<rsp_shard*> slots;
  std::unordered_map<std::string, rsp_shard*> by_name;
  PinBuf pin_in, pin_out, pin_up, pin_totals;
  DevBuf dev_tick, dev_q, dev_pending, dev_ops, dev_up;
  cudaEvent_t pending_ev = nullptr;  // the last device-form MultiGet launch (the pending list is per engine)
  bool pending_ev_recorded = false;
  cudaStream_t pending_last_stream = nullptr;
  cudaEvent_t up_ev = nullptr;  // the last batched descriptor upload (its staging buffers are reused)
  bool up_ev_recorded = false;
  std::vector<u32> gid_scratch;
  std::vector<u8> seen_scratch;
  // ordering between reads launched on caller streams and memtable flushes / re-allocations on the engine stream
  cudaEvent_t reader_ev[8] = {};
  u32 reader_head = 0, reader_pending = 0;
  cudaEvent_t mut_ev = nullptr;
  bool mut_recorded = false;
  size_t stage_threads = 1;
  // per-run descriptors of every shard ([max_shards][RSP_MAX_RUNS], behind d_fast in the same allocation): the fast
  // MultiGet kernel walks a shard's runs newest first when some shard has more than one (n_multirun counts them)
  ShardFast* d_fast_runs = nullptr;
  u32* d_mt_filter = nullptr;  // behind d_fast_runs in the same allocation (format.cuh: memtable filter)
  std::atomic<u32> n_multirun{0};
  bool fused_ticks = true;  // RSP_FUSED_TICK=0: always the four general kernels (k_decode .. k_publish)
  bool bg_compaction = true;  // RSP_BG_COMPACT=0: merges run on the apply path (r01 behaviour)
  struct Compactor* compactor = nullptr;
  u32 mg_parity = 0;
  size_t pending_cap = 0;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  std::map<std::string, float> last_ms;
  std::atomic<u64> launches{0};
};

static void set_err(rsp_shard* s, const std::string& m) {
  std::lock_guard<std::mutex> g(s->err_mu);
  s->last_error = m;
}

// Reads launched on a caller's stream (rsp_multi_get_device / rsp_multi_scan_device) are lock-free against apply
// ticks, but a flush or a memtable re-allocation recycles memory they may be reading: the engine stream waits for
// the outstanding reader events first, and later reads wait for the mutation event.
static void wait_readers(rsp_engine* e) {
  const u32 n = std::min<u32>(e->reader_pending, 8);
  for (u32 k = 0; k < n; k++) CUDA_OK(cudaStreamWaitEvent(e->st, e->reader_ev[(e->reader_head + 8 - 1 - k) % 8], 0));
  e->reader_pending = 0;
}
static void note_mutation(rsp_engine* e) {
  CUDA_OK(cudaEventRecord(e->mut_ev, e->st));
  e->mut_recorded = true;
}
static void reader_begin(rsp_engine* e, cudaStream_t s) {
  if (s != e->st && e->mut_recorded) CUDA_OK(cudaStreamWaitEvent(s, e->mut_ev, 0));
}
static void reader_end(rsp_engine* e, cudaStream_t s) {
  if (s == e->st) return;
  CUDA_OK(cudaEventRecord(e->reader_ev[e->reader_head], s));
  e->reader_head = (e->reader_head + 1) % 8;
  e->reader_pending++;
}

// runs_only: only the run set changed (a background merge was installed).  The sequencing state of the descriptor
// (last_seq, pub_seq, mt_tail, mt_count, latch) belongs to the DEVICE while ticks are in flight — the host mirror may
// lag behind pre-staged ticks — so it is not written then.
// host bookkeeping + the compact descriptors of a shard (ShardFast, one per run) from its run list
static void describe_shard(rsp_engine* e, rsp_shard* s, ShardFast* f_out, ShardFast* fr) {
  s->h.n_runs = (u32)s->runs.size();
  for (u32 i = 0; i < RSP_MAX_RUNS; i++) {
    if (i < s->runs.size()) s->h.runs[i] = s->runs[i]->dev();
    else memset(&s->h.runs[i], 0, sizeof(RunDev));
  }
  auto describe = [](const Run& r, ShardFast* f) {
    f->run0_heap = (u64)r.heap; f->run0_hslots = (u64)r.hslots; f->n_buckets = r.n_buckets;
    f->meta = r.ord_bits | (std::min<u32>(r.uniform_units, 255u) << 8);
  };
  ShardFast f;
  memset(&f, 0, sizeof(f));
  if (!s->runs.empty()) describe(*s->runs[0], &f);
  memset(fr, 0, sizeof(ShardFast) * RSP_MAX_RUNS);
  for (size_t i = 0; i < s->runs.size() && i < RSP_MAX_RUNS; i++) describe(*s->runs[i], &fr[i]);
  const bool multi_now = s->runs.size() > 1;
  if (multi_now != s->counted_multirun) {
    if (multi_now) e->n_multirun++; else e->n_multirun--;
    s->counted_multirun = multi_now;
  }
  f.meta |= (u32)std::min<size_t>(s->runs.size(), 255) << 16;
  f.meta |= 1u << 24;  // live
  f.mt_count = s->h.mt_count;
  f.merge_op = s->h.merge_op;
  *f_out = f;
}
static void upload_shard(rsp_engine* e, rsp_shard* s, bool runs_only = false) {
  ShardFast f, fr[RSP_MAX_RUNS];
  describe_shard(e, s, &f, fr);
  if (runs_only) {
    const size_t from = offsetof(ShardDev, n_runs);
    CUDA_OK(cudaMemcpyAsync((u8*)(e->d_shards + s->index) + from, (const u8*)&s->h + from, sizeof(ShardDev) - from,
                            cudaMemcpyHostToDevice, e->st));
  } else {
    CUDA_OK(cudaMemcpyAsync(e->d_shards + s->index, &s->h, sizeof(ShardDev), cudaMemcpyHostToDevice, e->st));
  }
  CUDA_OK(cudaMemcpyAsync(e->d_fast_runs + (size_t)s->index * RSP_MAX_RUNS, fr, sizeof(fr), cudaMemcpyHostToDevice, e->st));
  // (runs_only: the first 24 bytes = run 0 + meta; mt_count is written by the sequencing kernels)
  CUDA_OK(cudaMemcpyAsync(e->d_fast + s->index, &f, runs_only ? offsetof(ShardFast, mt_count) : sizeof(f), cudaMemcpyHostToDevice, e->st));
  // the host mirror is pageable: the copy above is staged before the call returns
}
// The same for a batch of shards (a flush / merge batch installs up to thousands of descriptors): records staged in
// pinned memory, one copy, one launch (k_upload_shards) — three pageable copies and a memset per shard cost the
// install of a 1024-shard flush tens of milliseconds of driver calls.
struct UploadBatch {
  std::vector<ShardUpload> recs;
};
static void stage_upload(rsp_engine* e, rsp_shard* s, bool runs_only, bool zero_mt, UploadBatch* b) {
  b->recs.emplace_back();
  ShardUpload& u = b->recs.back();
  describe_shard(e, s, &u.fast, u.fast_runs);
  u.index = s->index; u.runs_only = runs_only ? 1u : 0u; u.zero_mt = zero_mt ? 1u : 0u; u.pad = 0;
  u.sd = s->h;
}
static void commit_uploads(rsp_engine* e, UploadBatch* b) {
  const size_t n = b->recs.size();
  if (!n) return;
  const size_t bytes = n * sizeof(ShardUpload);
  if (e->up_ev_recorded) CUDA_OK(cudaEventSynchronize(e->up_ev));  // the staging buffers of the previous batch
  void* pin = e->pin_up.get(bytes);
  memcpy(pin, b->recs.data(), bytes);
  ShardUpload* d_up = (ShardUpload*)e->dev_up.get(bytes);
  CUDA_OK(cudaMemcpyAsync(d_up, pin, bytes, cudaMemcpyHostToDevice, e->st));
  launch_upload_shards(d_up, (u32)n, e->d_shards, e->d_fast, e->d_fast_runs, e->d_mt_filter, e->st);
  CUDA_OK(cudaGetLastError());
  CUDA_OK(cudaEventRecord(e->up_ev, e->st));
  e->up_ev_recorded = true;
  e->launches += 1;
  b->recs.clear();
}

static u32 next_pow2(u32 x) {
  u32 p = 1;
  while (p < x) p <<= 1;
  return p;
}

// (re)allocate an empty memtable able to hold at least `units` heap units and `ents` entries
static void alloc_memtable(rsp_engine* e, rsp_shard* s, u64 units, u64 ents) {
  Arena& a = e->arena;
  if (s->h.mt_heap) {
    wait_readers(e);
    CUDA_OK(cudaStreamSynchronize(e->st));  // nothing may still read the buffers being recycled
    a.release(s->h.mt_heap, s->mt_heap_bytes);
    a.release(s->h.mt_slots, s->mt_slot_bytes);
    a.release(s->h.mt_ent_off, s->mt_ent_bytes);
  }
  u64 want_units = std::max<u64>(units, (s->opts.write_buffer_bytes ? s->opts.write_buffer_bytes : (1u << 20)) / 16);
  u64 want_ents = std::max<u64>(ents, want_units / 7);  // a 16 B/64 B Put is 7 units
  u32 slot_cap = next_pow2((u32)std::max<u64>(16, want_ents * 2));
  s->mt_heap_bytes = want_units * 16;
  s->mt_slot_bytes = (size_t)slot_cap * 8;
  s->mt_ent_bytes = want_ents * 4;
  s->h.mt_heap = (u8*)a.alloc(s->mt_heap_bytes);
  s->h.mt_slots = (u64*)a.alloc(s->mt_slot_bytes);
  s->h.mt_ent_off = (u32*)a.alloc(s->mt_ent_bytes);
  s->h.mt_slot_mask = slot_cap - 1;
  s->h.mt_heap_cap = (u32)want_units;
  s->h.mt_ent_cap = (u32)want_ents;
  s->h.mt_tail = 0;
  s->h.mt_count = 0;
  CUDA_OK(cudaMemsetAsync(s->h.mt_slots, 0, s->mt_slot_bytes, e->st));
  CUDA_OK(cudaMemsetAsync(e->d_mt_filter + (size_t)s->index * MT_FILTER_WORDS, 0, MT_FILTER_WORDS * 4, e->st));
}

// ------------------------------------------------------------------------------------------------
// flush / compaction of a set of shards in one batched pass
// ------------------------------------------------------------------------------------------------
struct JobHost {
  rsp_shard* s;
  u32 index;        // s->index / s->uid at planning time: a background install checks that the shard is still the same
  u64 uid;
  bool full;        // every run of the shard takes part: the output is the shard's only run
  bool has_mem;     // the memtable is a source (flush)
  size_t n_merged;  // srcs.size(): the runs replaced by the output
  std::vector<std::shared_ptr<Run>> srcs;
  size_t items_b, items2_b, coranks_b, keep_b, fold_b;
  bool generic_sort = false;  // the memtable took the comparison sort (k_flush_sort left it: totals[7])
};
// one batch of flush / merge jobs: planned under the engine mutex, run on a stream, installed under the mutex again
struct CompactPlan {
  std::vector<JobHost> jh;
  std::vector<CompactJob> jobs;
  std::vector<std::shared_ptr<Run>> outs;
  CompactJob* d_jobs = nullptr;
  u32* d_totals = nullptr;  // [8 x jobs], contiguous: one copy brings every job's sizes back
  float ms = 0;
};
enum CompactMode {
  COMPACT_FLUSH,     // memtable -> new run; the newest runs join only when the run table is nearly full
  COMPACT_FULL,      // everything into one run (CompactRange(nullptr, nullptr))
  COMPACT_SNAPSHOT,  // memtable -> a private sorted run for an iterator; the shard is left untouched
  COMPACT_MERGE      // background: the size-tiered merge set of the runs, no memtable
};

// Which runs are merged?  Size-tiered (the role of RocksDB's level0_file_num_compaction_trigger + level sizing,
// examples/counter_service/rocksdb_options.cpp:82-93): at the trigger the newest runs are merged, stopping before a
// run more than twice as large as everything gathered so far — the big bottom run is rewritten only when the small
// ones have grown to its order of magnitude, so write amplification stays logarithmic in the shard size instead of
// shard_bytes / write_buffer.  `acc` starts with what is merged anyway (the memtable of a foreground flush).  Runs
// pinned by a background merge in flight (from s->bg_first_pinned on) are not touched.
static size_t tiered_set(const rsp_shard* s, u64 acc, size_t limit, bool must_shrink) {
  size_t j = 0;
  const size_t min_take = acc ? 1 : 2;  // a merge needs two inputs
  while (j < limit) {
    const u64 sz = s->runs[j]->bytes();
    if (j >= min_take && !(must_shrink && j < 2) && sz > 2 * acc) break;
    acc += sz;
    j++;
  }
  return j;
}
static size_t unpinned_runs(const rsp_shard* s) {
  if (!s->merging) return s->runs.size();
  for (size_t i = 0; i < s->runs.size(); i++) if (s->runs[i].get() == s->bg_first_pinned) return i;
  return s->runs.size();
}

static void bg_request(rsp_engine* e, rsp_shard* s);

// ---- plan (engine mutex held) ------------------------------------------------------------------------
static void plan_jobs(rsp_engine* e, const std::vector<rsp_shard*>& shards, CompactMode mode, CompactPlan* plan) {
  Arena& a = e->arena;
  for (rsp_shard* s : shards) {
    const bool has_mem = mode != COMPACT_MERGE && s->h.mt_count > 0;
    size_t n_merged = 0;
    const size_t avail = unpinned_runs(s);
    if (mode == COMPACT_FULL) n_merged = s->runs.size();  // (the caller waited for the shard's background merge)
    else if (mode == COMPACT_MERGE) {
      if (s->merging || s->runs.size() < e->cfg.l0_compaction_trigger) continue;
      n_merged = tiered_set(s, 0, s->runs.size(), false);
      if (n_merged < 2) continue;
    } else if (mode == COMPACT_FLUSH) {
      const bool table_full = s->runs.size() + 1 > RSP_MAX_RUNS - 1;
      if (!e->bg_compaction) {
        if (s->runs.size() + (has_mem ? 1 : 0) >= e->cfg.l0_compaction_trigger || table_full)
          n_merged = tiered_set(s, has_mem ? (u64)s->h.mt_tail * 16 : 0, avail, table_full);
      } else if (table_full) {
        // merges belong to the background thread; the foreground only merges when the run table itself fills up
        n_merged = tiered_set(s, has_mem ? (u64)s->h.mt_tail * 16 : 0, avail, true);
      }
    }
    // the run table must never overflow: if the flush would, everything is merged right here (a background merge of
    // some of these runs then finds its sources gone at install time and drops its output)
    if (mode == COMPACT_FLUSH && has_mem && s->runs.size() - n_merged + 1 > RSP_MAX_RUNS) n_merged = s->runs.size();
    const bool full = n_merged == s->runs.size();
    if (!has_mem && n_merged <= 1) {
      // nothing to flush; a single run is already fully compacted unless it holds tombstones
      if (!(mode == COMPACT_FULL && s->runs.size() == 1)) continue;
    }
    CompactJob j;
    memset(&j, 0, sizeof(j));
    JobHost h{s, s->index, s->uid, full, has_mem, n_merged, {}, 0, 0, 0, 0, 0};
    u32 ns = 0;
    if (has_mem) {
      j.src_heap[ns] = s->h.mt_heap; j.src_ent_off[ns] = s->h.mt_ent_off; j.src_n[ns] = s->h.mt_count;
      j.src_is_mem[ns] = 1; ns++;
      j.n_pow2 = next_pow2(std::max<u32>(2, s->h.mt_count));
    }
    for (size_t r = 0; r < n_merged; r++) {
      auto& run = s->runs[r];
      j.src_heap[ns] = run->heap; j.src_ent_off[ns] = run->ent_off; j.src_n[ns] = run->n_ent; j.src_is_mem[ns] = 0;
      ns++;
      h.srcs.push_back(run);
    }
    j.n_src = ns;
    u64 n = 0, at = 0;
    for (u32 i = 0; i < ns; i++) {
      j.seg_start[i] = (u32)at;
      at += (i == 0 && has_mem) ? j.n_pow2 : j.src_n[i];
      n += j.src_n[i];
    }
    j.n_items = (u32)n;
    j.items_len = (u32)at;
    j.n_tiles = ns > 1 ? (u32)((n + MERGE_TILE - 1) / MERGE_TILE) : 0;
    j.bottom = (full && mode != COMPACT_SNAPSHOT) ? 1 : 0;
    j.merge_op = s->opts.merge_op;
    h.items_b = (size_t)std::max<u32>(1, j.items_len) * sizeof(SortItem);
    h.items2_b = ns > 1 ? (size_t)std::max<u32>(1, j.n_items) * sizeof(SortItem) : 0;
    h.coranks_b = ns > 1 ? (size_t)(j.n_tiles + 1) * ns * 4 : 0;
    h.keep_b = (size_t)std::max<u32>(1, j.n_items) * 4;
    h.fold_b = (size_t)std::max<u32>(1, j.n_items) * 8;
    j.items = (SortItem*)a.alloc(h.items_b);
    j.items2 = ns > 1 ? (SortItem*)a.alloc(h.items2_b) : nullptr;
    j.coranks = ns > 1 ? (u32*)a.alloc(h.coranks_b) : nullptr;
    j.sorted = ns > 1 ? j.items2 : j.items;
    j.keep_units = (u32*)a.alloc(h.keep_b);
    j.out_pos = (u32*)a.alloc(h.keep_b);
    j.out_ord = (u32*)a.alloc(h.keep_b);
    j.fold_val = (u64*)a.alloc(h.fold_b);
    if (mode == COMPACT_MERGE) {
      s->merging = true;
      s->bg_first_pinned = h.srcs.front().get();
    }
    plan->jh.push_back(h);
    plan->jobs.push_back(j);
  }
}

// ---- run (no engine mutex needed: sources are pinned, outputs are private until installed) -----------------
static void run_jobs(rsp_engine* e, CompactPlan* plan, cudaStream_t st, cudaEvent_t ev0, cudaEvent_t ev1, PinBuf* pin_totals) {
  Arena& a = e->arena;
  std::vector<CompactJob>& jobs = plan->jobs;
  const u32 nj = (u32)jobs.size();
  plan->d_jobs = (CompactJob*)a.alloc(sizeof(CompactJob) * nj);
  plan->d_totals = (u32*)a.alloc((size_t)32 * nj);
  for (u32 i = 0; i < nj; i++) jobs[i].totals = plan->d_totals + 8 * (size_t)i;
  CUDA_OK(cudaMemsetAsync(plan->d_totals, 0, (size_t)32 * nj, st));
  CompactJob* d_jobs = plan->d_jobs;
  CUDA_OK(cudaMemcpyAsync(d_jobs, jobs.data(), sizeof(CompactJob) * nj, cudaMemcpyHostToDevice, st));
  CUDA_OK(cudaEventRecord(ev0, st));
  launch_compact_sort(d_jobs, jobs.data(), nj, st);
  launch_compact_size(d_jobs, nj, st);
  CUDA_OK(cudaGetLastError());  // a refused launch (e.g. shared-memory opt-in) must not pass as an unsorted run
  e->launches += 5;
  // the sizing round trip: ONE copy into pinned memory (r02 issued a 32-byte pageable copy per job)
  const u32* totals = (const u32*)pin_totals->get((size_t)32 * nj);
  CUDA_OK(cudaMemcpyAsync((void*)totals, plan->d_totals, (size_t)32 * nj, cudaMemcpyDeviceToHost, st));
  CUDA_OK(cudaStreamSynchronize(st));
  u32 max_items = 0, max_buckets = 0;
  plan->outs.resize(nj);
  for (u32 i = 0; i < nj; i++) {
    CompactJob& j = jobs[i];
    const u32 units = totals[8 * i], ents = totals[8 * i + 1], uni = totals[8 * i + 2], keys = totals[8 * i + 3];
    const u32 non_put = totals[8 * i + 4], kvmin = totals[8 * i + 5], kvmax = totals[8 * i + 6];
    plan->jh[i].generic_sort = totals[8 * i + 7] != 0;
    auto r = std::make_shared<Run>();
    r->arena = &a;
    r->n_ent = ents; r->heap_units = units; r->uniform_units = uni;
    if (ents && uni && non_put == 0 && kvmin == kvmax) { r->flags = RUN_ALL_PUT_FIXED; r->kv_len = kvmin; }
    r->n_blocks = (ents + RSP_BLOCK_ENTRIES - 1) / RSP_BLOCK_ENTRIES;
    // 8-slot buckets at load <= 0.5: a key overflows its home bucket with p ~ 2 % (Poisson(4) > 8), and
    // an overflow costs the 16-lookup warp of k_multi_get16 one more dependent sector read
    r->n_buckets = std::max<u32>(1, (u32)(((u64)keys + 3) / 4));
    r->ord_bits = 1;
    while ((1ull << r->ord_bits) <= ents) r->ord_bits++;
    r->heap = (u8*)a.alloc((size_t)units * 16);
    r->ent_off = (u32*)a.alloc((size_t)ents * 4);
    r->hslots = (u32*)a.alloc((size_t)r->n_buckets * RUN_BUCKET_SLOTS * 4);
    r->blk_pfx = (u64*)a.alloc(blk_pfx_bytes(r->n_blocks));
    max_buckets = std::max(max_buckets, r->n_buckets);
    j.out_heap = r->heap; j.out_ent_off = r->ent_off; j.out_hslots = r->hslots; j.out_blk_pfx = r->blk_pfx;
    j.out_n_buckets = r->n_buckets; j.out_ord_bits = r->ord_bits;
    plan->outs[i] = r;
    max_items = std::max(max_items, j.n_items);
  }
  CUDA_OK(cudaMemcpyAsync(d_jobs, jobs.data(), sizeof(CompactJob) * nj, cudaMemcpyHostToDevice, st));
  launch_zero_out_hslots(d_jobs, nj, max_buckets, st);  // every output's hash index in one launch
  launch_compact_write(d_jobs, nj, max_items, st);
  CUDA_OK(cudaGetLastError());
  e->launches += 2;
  CUDA_OK(cudaEventRecord(ev1, st));
  CUDA_OK(cudaStreamSynchronize(st));
  cudaEventElapsedTime(&plan->ms, ev0, ev1);
}

static void release_work(rsp_engine* e, CompactPlan* plan) {
  Arena& a = e->arena;
  for (size_t i = 0; i < plan->jobs.size(); i++) {
    const CompactJob& j = plan->jobs[i];
    const JobHost& h = plan->jh[i];
    a.release(j.items, h.items_b);
    if (j.items2) a.release(j.items2, h.items2_b);
    if (j.coranks) a.release(j.coranks, h.coranks_b);
    a.release(j.keep_units, h.keep_b);
    a.release(j.out_pos, h.keep_b);
    a.release(j.out_ord, h.keep_b);
    a.release(j.fold_val, h.fold_b);
  }
  if (plan->d_jobs) a.release(plan->d_jobs, sizeof(CompactJob) * plan->jobs.size());
  if (plan->d_totals) a.release(plan->d_totals, (size_t)32 * plan->jobs.size());
  plan->d_jobs = nullptr;
  plan->d_totals = nullptr;
}

// ---- install (engine mutex held): the new run takes the place of its sources in the shard's run list; readers keep
// the old descriptors until this point and the old runs live until every reader launched before it has finished
static void install_jobs(rsp_engine* e, CompactPlan* plan, CompactMode mode) {
  const u32 nj = (u32)plan->jobs.size();
  if (mode == COMPACT_MERGE) wait_readers(e);  // (the foreground path did this before it touched a memtable)
  UploadBatch up;
  up.recs.reserve(nj);
  for (u32 i = 0; i < nj; i++) {
    JobHost& h = plan->jh[i];
    rsp_shard* s = h.s;
    if (mode == COMPACT_MERGE) {
      // the shard may have been closed, or its runs merged by a foreground CompactRange, while the kernels ran: the
      // output is only installed over exactly the sources it was built from
      const bool alive = h.index < e->slots.size() && e->slots[h.index] == s && s->uid == h.uid;
      if (!alive) { h.s = nullptr; continue; }
      size_t at = 0;
      while (at < s->runs.size() && s->runs[at].get() != h.srcs.front().get()) at++;
      bool intact = at + h.n_merged <= s->runs.size();
      for (size_t k = 0; intact && k < h.n_merged; k++) intact = s->runs[at + k].get() == h.srcs[k].get();
      s->merging = false;
      s->bg_first_pinned = nullptr;
      if (!intact) { h.s = nullptr; continue; }
    }
    u64 read_b = 0;
    if (h.has_mem) read_b += (u64)s->h.mt_tail * 16;
    for (auto& r : h.srcs) read_b += r->bytes();
    s->stats.compaction_bytes_read += read_b;
    s->stats.compaction_bytes_written += plan->outs[i]->bytes();
    if (h.has_mem) s->stats.flushes++;
    if (h.has_mem && h.generic_sort) s->stats.flush_comparison_sorts++;
    // the sources sit where they were planned, possibly behind runs that were flushed meanwhile (background merges)
    size_t at = 0;
    if (h.n_merged) {
      while (at < s->runs.size() && s->runs[at].get() != h.srcs.front().get()) at++;
      s->stats.compactions++;
      s->runs.erase(s->runs.begin() + at, s->runs.begin() + at + h.n_merged);
    }
    if (plan->outs[i]->n_ent) s->runs.insert(s->runs.begin() + at, plan->outs[i]);
    if (h.has_mem) {
      s->h.mt_tail = 0;
      s->h.mt_count = 0;
    }
    stage_upload(e, s, mode == COMPACT_MERGE, h.has_mem, &up);  // (+ the flushed memtable's slot table cleared)
  }
  commit_uploads(e, &up);
  note_mutation(e);
  CUDA_OK(cudaStreamSynchronize(e->st));  // sources may be released once nothing reads them
  e->last_ms["compact"] = plan->ms;
  e->last_ms["compact_total"] += plan->ms;  // kernels of every flush / merge so far (sizing round trip included)
  for (u32 i = 0; i < nj; i++) {
    rsp_shard* s = plan->jh[i].s;
    if (s && e->bg_compaction && s->runs.size() >= e->cfg.l0_compaction_trigger && !s->merging) bg_request(e, s);
  }
}

// foreground flush / full compaction of a set of shards in one batched pass (engine mutex held throughout)
static void compact_shards(rsp_engine* e, const std::vector<rsp_shard*>& shards, bool force_full) {
  CompactPlan plan;
  const CompactMode mode = force_full ? COMPACT_FULL : COMPACT_FLUSH;
  plan_jobs(e, shards, mode, &plan);
  if (plan.jobs.empty()) return;
  wait_readers(e);
  try {
    run_jobs(e, &plan, e->st, e->ev0, e->ev1, &e->pin_totals);
  } catch (...) {  // (out of device memory, typically): nothing was installed; the work buffers and partial outputs go back
    cudaStreamSynchronize(e->st);
    release_work(e, &plan);
    throw;
  }
  install_jobs(e, &plan, mode);
  release_work(e, &plan);
}

// the memtable's contents as a private sorted run (an iterator's snapshot): nothing about the shard changes
static std::shared_ptr<Run> snapshot_memtable(rsp_engine* e, rsp_shard* s) {
  CompactPlan plan;
  plan_jobs(e, {s}, COMPACT_SNAPSHOT, &plan);
  if (plan.jobs.empty()) return nullptr;
  try {
    run_jobs(e, &plan, e->st, e->ev0, e->ev1, &e->pin_totals);
  } catch (...) {
    cudaStreamSynchronize(e->st);
    release_work(e, &plan);
    throw;
  }
  release_work(e, &plan);
  s->stats.compaction_bytes_read += (u64)s->h.mt_tail * 16;
  return plan.outs[0]->n_ent ? plan.outs[0] : nullptr;
}

// ---- background merges ------------------------------------------------------------------------------------
// Flushes stay on the apply path (they are what makes room in a memtable); merging sorted runs is deferred to this
// thread: planned and installed under the engine mutex, but its kernels run on their own stream with the mutex
// released, so applies and reads go on while runs are merged (readers keep the old run set until the install).
struct Compactor {
  rsp_engine* e = nullptr;
  std::mutex mu;
  std::condition_variable cv;
  std::vector<rsp_shard*> pending;
  bool stop = false, busy = false;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  PinBuf pin_totals;  // this thread's sizing round trips
  std::thread th;
  void loop();
};
static void bg_request(rsp_engine* e, rsp_shard* s) {
  Compactor* c = e->compactor;
  if (!c) return;
  {
    std::lock_guard<std::mutex> g(c->mu);
    if (std::find(c->pending.begin(), c->pending.end(), s) == c->pending.end()) c->pending.push_back(s);
  }
  c->cv.notify_one();
}
void Compactor::loop() {
  cudaSetDevice(e->device);
  for (;;) {
    std::vector<rsp_shard*> take;
    {
      std::unique_lock<std::mutex> l(mu);
      busy = false;
      cv.notify_all();
      cv.wait(l, [this] { return stop || !pending.empty(); });
      if (stop) return;
      take.swap(pending);
      busy = true;
    }
    // in parts bounded by source bytes (<= 8 GB, <= 256 shards): a uniform load brings every shard to its merge trigger at
    // the same time, and one plan over all of them needs their outputs and work buffers at once (the config-2 stretch
    // point ran out of HBM that way)
    size_t pos = 0;
    while (pos < take.size()) {
      CompactPlan plan;
      try {
        {
          std::lock_guard<std::mutex> g(e->mu);
          std::vector<rsp_shard*> part;
          u64 part_bytes = 0;
          while (pos < take.size() && part.size() < 256) {
            rsp_shard* s = take[pos];
            if (std::find(e->slots.begin(), e->slots.end(), s) != e->slots.end()) {
              u64 b = 0;
              for (auto& r : s->runs) b += r->bytes();
              if (!part.empty() && part_bytes + b > (8ull << 30)) break;
              part.push_back(s);
              part_bytes += b;
            }
            pos++;
          }
          plan_jobs(e, part, COMPACT_MERGE, &plan);
        }
        if (plan.jobs.empty()) continue;
        run_jobs(e, &plan, stream, ev0, ev1, &pin_totals);
        {
          std::lock_guard<std::mutex> g(e->mu);
          cudaSetDevice(e->device);
          install_jobs(e, &plan, COMPACT_MERGE);
        }
        release_work(e, &plan);
      } catch (...) {
        abi_caught();  // a CUDA failure: recorded; the shards keep their runs, the work buffers go back
        cudaStreamSynchronize(stream);
        std::lock_guard<std::mutex> g(e->mu);
        for (JobHost& h : plan.jh)
          if (h.s && h.index < e->slots.size() && e->slots[h.index] == h.s && h.s->uid == h.uid) { h.s->merging = false; h.s->bg_first_pinned = nullptr; }
        release_work(e, &plan);
        plan.outs.clear();
      }
    }
  }
}
// ------------------------------------------------------------------------------------------------
// apply path
// ------------------------------------------------------------------------------------------------
static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
static inline double now_us() {
  return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now().time_since_epoch()).count();
}
static const bool g_trace = getenv("RSP_TRACE") != nullptr;

// Build the tick image (pinned) for n batches and copy it to the device.  Layout of the image:
//   [BatchDesc x n][GroupDesc x g][blob ...] ; results [BatchRes x n][GroupRes x g] ; [OpRec x ops]
// Cut every group into chunks of <= FUSED_CHUNK_BATCHES batches and <= FUSED_STAGE_BYTES of blob (k_tick_chunks: a CTA
// per chunk); start(i) / end(i) = byte offsets of staged batch i in the blob.  GroupDesc.pad receives the chunk count.
template <class Start, class End>
static void cut_chunks(GroupDesc* groups, size_t ng, Start start, End end, std::vector<ChunkDesc>* out) {
  out->clear();
  for (size_t g = 0; g < ng; g++) {
    const size_t first = groups[g].first_batch, last = first + groups[g].n_batches;
    u32 ci = 0;
    for (size_t b = first; b < last;) {
      const u64 base = start(b);
      size_t e = b + 1;  // (a batch beyond the stage cannot reach here: such ticks take the general kernels)
      while (e < last && e - b < FUSED_CHUNK_BATCHES && end(e) - base <= FUSED_STAGE_BYTES) e++;
      out->push_back(ChunkDesc{(u32)g, (u32)b, (u32)(e - b), ci++, groups[g].shard_ix, 0u, 0u, 0u});
      b = e;
    }
    groups[g].pad = ci;
    for (size_t k = out->size() - ci; k < out->size(); k++) (*out)[k].group_chunks = ci;
  }
}

// Pitch of a batch in a staged image: whole 4-byte words, an ODD number of them — k_tick_fused walks a batch per thread
// in shared memory, and equal-sized batches at an even word pitch (r02 padded to 16 bytes: 128 for the 115-byte
// replication unit) put all 32 lanes of a warp on the same bank (ncu: 29.7-way conflicts, 97 % of the wavefronts).
static inline size_t stage_pitch(size_t len_eff) {
  const size_t w = (len_eff + 3) / 4;
  return 4 * (w | 1);
}

static int stage_build(rsp_engine* e, size_t n, const uint32_t* shard_ix, const uint8_t* blob, const uint64_t* off,
                       const uint64_t* ts_ms, rsp_staged* sg, bool own_dev) {
  sg->eng = e;
  sg->n = n;
  const double t_a = now_us();
  // group by shard, preserving submission order within a shard (counting sort over shard ids)
  std::vector<u32>& gid_of = e->gid_scratch;
  if (gid_of.size() < e->slots.size()) gid_of.assign(e->slots.size(), 0xffffffffu);
  std::vector<u32> g_count, g_of_batch(n);
  for (size_t i = 0; i < n; i++) {
    const u32 six = shard_ix[i];
    if (six >= e->slots.size() || !e->slots[six]) {
      for (rsp_shard* s : sg->group_shard) gid_of[s->index] = 0xffffffffu;
      return RSP_INVALID_ARGUMENT;
    }
    u32 g = gid_of[six];
    if (g == 0xffffffffu) {
      g = gid_of[six] = (u32)sg->group_shard.size();
      sg->group_shard.push_back(e->slots[six]);
      g_count.push_back(0);
    }
    g_of_batch[i] = g;
    g_count[g]++;
  }
  for (rsp_shard* s : sg->group_shard) gid_of[s->index] = 0xffffffffu;
  std::vector<u32> g_start(g_count.size() + 1, 0);
  for (size_t g = 0; g < g_count.size(); g++) g_start[g + 1] = g_start[g] + g_count[g];
  std::vector<u32> by_group(n);
  {
    std::vector<u32> fill(g_start.begin(), g_start.end() - 1);
    for (size_t i = 0; i < n; i++) by_group[fill[g_of_batch[i]]++] = (u32)i;
  }
  const size_t ng = sg->group_shard.size();
  const size_t trailer = ts_ms ? 10 : 0;
  const double t_b = now_us();
  // ---- plan (serial, no byte copies): staged order, blob offsets, reserved op slots, capacity bounds
  sg->order.resize(n);
  sg->need_units.assign(ng, 0);
  sg->need_ents.assign(ng, 0);
  std::vector<u32> p_boff(n), p_cap(n), p_opbase(n);
  size_t boff = 0;
  u64 ops_cap = 0;
  {
    size_t pos = 0;
    for (size_t g = 0; g < ng; g++) {
      for (u32 bi = g_start[g]; bi < g_start[g + 1]; bi++, pos++) {
        const u32 i = by_group[bi];
        const size_t len = (size_t)(off[i + 1] - off[i]);
        const size_t len_eff = len + trailer;
        u32 claimed = 0;
        if (len >= 12) memcpy(&claimed, blob + off[i] + 8, 4);
        else if (len_eff >= 12) {  // the header straddles the appended LogData record
          u8 hdr[12];
          memcpy(hdr, blob + off[i], len);
          const u8 tr[10] = {0x03, 8, (u8)ts_ms[i], (u8)(ts_ms[i] >> 8), (u8)(ts_ms[i] >> 16), (u8)(ts_ms[i] >> 24),
                             (u8)(ts_ms[i] >> 32), (u8)(ts_ms[i] >> 40), (u8)(ts_ms[i] >> 48), (u8)(ts_ms[i] >> 56)};
          memcpy(hdr + len, tr, 12 - len);
          memcpy(&claimed, hdr + 8, 4);
        }
        const u32 max_ops = len_eff > 12 ? (u32)((len_eff - 12) / 2) : 0;
        const u32 cap = std::min(claimed, max_ops);
        sg->order[pos] = i;
        p_boff[pos] = (u32)boff;
        p_cap[pos] = cap;
        p_opbase[pos] = (u32)ops_cap;
        ops_cap += cap;
        // upper bound on heap units: 2 header units + padding per op, payload bytes / 16
        sg->need_units[g] += cap * 4u + (u32)(len_eff / 16) + 1u;
        sg->need_ents[g] += cap;
        boff += stage_pitch(len_eff);
        if (boff > 0xf0000000ull) return RSP_INVALID_ARGUMENT;
      }
    }
  }
  if (ops_cap > 0xfff00000ull) return RSP_INVALID_ARGUMENT;
  const size_t blob_bytes = align_up(boff + 64, 256);  // slack for the insert kernel's aligned word reads; what follows stays aligned
  // [BatchDesc x n][GroupDesc x g][u64 off x n][u32 len x n] | blob : the last two feed the fused tick kernel
  const size_t o_foff = align_up(n * sizeof(BatchDesc) + ng * sizeof(GroupDesc), 16);
  const size_t o_flen = o_foff + n * 8;
  const size_t desc_b = align_up(o_flen + n * 4, 256);
  const size_t in_b = desc_b + blob_bytes;
  u8* pin = (u8*)e->pin_in.get(in_b);
  BatchDesc* bd = (BatchDesc*)pin;
  GroupDesc* gd = (GroupDesc*)(pin + n * sizeof(BatchDesc));
  u8* pblob = pin + desc_b;
  for (size_t g = 0; g < ng; g++) {
    gd[g].shard_ix = sg->group_shard[g]->index;
    gd[g].first_batch = g_start[g];
    gd[g].n_batches = g_count[g];
    gd[g].pad = 0;
  }
  const double t_c = now_us();
  // ---- copy (parallel over staged positions): batch bytes + the follower's LogData record + descriptors
  const u32* order = sg->order.data();
  const u32* g_of = g_of_batch.data();
  auto copy_range = [&](size_t lo, size_t hi) {
    for (size_t pos = lo; pos < hi; pos++) {
      const u32 i = order[pos];
      const size_t len = (size_t)(off[i + 1] - off[i]);
      const size_t len_eff = len + trailer;
      u8* dst = pblob + p_boff[pos];
      memcpy(dst, blob + off[i], len);
      if (ts_ms) {  // rocksdb_wrapper.cpp:19-20: PutLogData(&timestamp, 8) appended to the rep
        dst[len] = 0x03;
        dst[len + 1] = 8;
        memcpy(dst + len + 2, &ts_ms[i], 8);
      }
      const size_t padded = stage_pitch(len_eff);
      if (padded > len_eff) memset(dst + len_eff, 0, padded - len_eff);
      BatchDesc& b = bd[pos];
      const u32 g = g_of[i];
      b.shard_ix = gd[g].shard_ix; b.boff = p_boff[pos]; b.len = (u32)len_eff;
      b.op_base = p_opbase[pos]; b.op_cap = p_cap[pos]; b.group = g; b.raw_len = (u32)len_eff; b.pad1 = 0;
      reinterpret_cast<u64*>(pin + o_foff)[pos] = p_boff[pos];
      reinterpret_cast<u32*>(pin + o_flen)[pos] = (u32)len_eff;
    }
  };
  const size_t n_workers = n >= 16384 ? std::min<size_t>(e->stage_threads, 8) : 1;
  if (n_workers <= 1) {
    copy_range(0, n);
  } else {
    std::vector<std::thread> th;
    const size_t per = (n + n_workers - 1) / n_workers;
    for (size_t w = 1; w < n_workers; w++) th.emplace_back(copy_range, std::min(n, w * per), std::min(n, (w + 1) * per));
    copy_range(0, std::min(n, per));
    for (auto& t : th) t.join();
  }
  memset(pblob + boff, 0, 64);
  const double t_d = now_us();
  if (g_trace) fprintf(stderr, "[rsp trace] stage n=%zu group %.0f us plan %.0f us copy %.0f us\n", n, t_b - t_a, t_c - t_b, t_d - t_c);
  // device image: [descs | blob] [BatchRes x n] [GroupRes x g | u32 status x n] [OpRec x ops]
  const size_t bres_b = align_up(n * sizeof(BatchRes), 256);
  const size_t out_b = align_up(ng * sizeof(GroupRes) + n * 4, 256);
  const size_t ops_b = (size_t)ops_cap * sizeof(OpRec);
  // k_tick_chunks (groups longer than one chunk): chunk table, chain records, per-group counters behind everything else
  std::vector<ChunkDesc> chunks;
  {
    size_t mg = 0, ml = 0;
    for (size_t g = 0; g < ng; g++) mg = std::max<size_t>(mg, g_count[g]);
    for (size_t pos = 0; pos < n; pos++) ml = std::max<size_t>(ml, reinterpret_cast<const u32*>(pin + o_flen)[pos]);
    if (!fused_small_shape((u32)mg, (u32)(ml + 16)) && ml <= FUSED_MAX_BATCH_BYTES) {
      const u32* lens = reinterpret_cast<const u32*>(pin + o_flen);
      cut_chunks(gd, ng, [&](size_t i) { return (u64)p_boff[i]; }, [&](size_t i) { return (u64)p_boff[i] + lens[i]; }, &chunks);
    }
  }
  const size_t dev_b_base = align_up(in_b + bres_b + out_b + ops_b, 256);
  const size_t dev_b = dev_b_base + align_up(chunks.size() * sizeof(ChunkDesc), 256) + chunks.size() * 32 + ng * 4 + 256;
  u8* dev;
  if (own_dev) {
    CUDA_OK(cudaMalloc(&sg->dev, dev_b));
    sg->dev_bytes = dev_b;
    dev = (u8*)sg->dev;
  } else {
    dev = (u8*)e->dev_tick.get(dev_b);
  }
  CUDA_OK(cudaMemcpyAsync(dev, pin, in_b, cudaMemcpyHostToDevice, e->st));
  TickDev& t = sg->tick;
  t.ts = nullptr;  // the LogData record is physically in the staged blob
  t.batches = (const BatchDesc*)dev;
  t.groups = (const GroupDesc*)(dev + n * sizeof(BatchDesc));
  t.blob = dev + desc_b;
  t.bres = (BatchRes*)(dev + in_b);
  t.gres = (GroupRes*)(dev + in_b + bres_b);
  t.bstat = (u32*)(dev + in_b + bres_b + ng * sizeof(GroupRes));
  t.ops = (OpRec*)(dev + in_b + bres_b + out_b);
  t.n_batches = (u32)n; t.n_groups = (u32)ng; t.n_ops_cap = (u32)ops_cap;
  sg->res_bytes = ng * sizeof(GroupRes) + n * 4;  // what comes back: per-shard results + one status word per batch
  sg->group_first.assign(g_start.begin(), g_start.end());
  {
    // one launch for the whole tick when every batch is small (a thread walks a batch there) and no group is so long
    // that its CTA would serialise the tick
    size_t max_len = 0, max_group = 0;
    for (size_t i = 0; i < n; i++) max_len = std::max<size_t>(max_len, (size_t)(off[i + 1] - off[i]) + trailer);
    for (size_t g = 0; g < ng; g++) max_group = std::max<size_t>(max_group, g_count[g]);
    sg->fused = e->fused_ticks && max_len <= FUSED_MAX_BATCH_BYTES;
    FusedTick& f = sg->ftick;
    f.blob = t.blob; f.off = (const u64*)(dev + o_foff); f.len = (const u32*)(dev + o_flen); f.ts = nullptr;
    f.groups = t.groups; f.bstat = t.bstat; f.gres = t.gres; f.n_groups = (u32)ng; f.n_batches = (u32)n;
    f.max_group = (u32)max_group; f.max_len = (u32)(max_len + 16);
    f.chunks = (const ChunkDesc*)(dev + dev_b_base); f.n_chunks = (u32)chunks.size(); f.pad = 0;
    f.chain = (u64*)(dev + dev_b_base + align_up(chunks.size() * sizeof(ChunkDesc), 256));
    f.group_done = (u32*)((u8*)f.chain + chunks.size() * 32);
    if (!chunks.empty())
      CUDA_OK(cudaMemcpyAsync(dev + dev_b_base, chunks.data(), chunks.size() * sizeof(ChunkDesc), cudaMemcpyHostToDevice, e->st));
  }
  if (own_dev) CUDA_OK(cudaStreamSynchronize(e->st));  // the pinned staging buffer is reused
  return RSP_OK;
}

// make sure every shard of the tick has room; flush (batched) or grow memtables as needed
static void unreserve(const rsp_staged* sg) {
  if (!sg->reserved) return;
  for (size_t g = 0; g < sg->group_shard.size(); g++) {
    rsp_shard* s = sg->group_shard[g];
    s->inflight_units -= std::min<u64>(s->inflight_units, sg->need_units[g]);
    s->inflight_ents -= std::min<u64>(s->inflight_ents, sg->need_ents[g]);
  }
  sg->reserved = false;
}

// pre-staged ticks launched on the device whose results are not folded into the host mirror yet: maintenance that
// rewrites the memtable from the mirror must not run now (the caller folds them first: rsp_apply_staged_finish)
static inline bool ticks_in_flight(const rsp_shard* s) { return s->inflight_units != 0 || s->inflight_ents != 0; }

// Make room for the tick's upper bounds.  Returns 1 when memtables were flushed or re-sized (work on the engine
// stream), 0 when nothing had to be done, -1 when a shard is full while earlier ticks are still in flight (their
// results must be folded first: rsp_apply_staged_finish).
static int reserve_for(rsp_engine* e, const rsp_staged* sg) {
  bool did_work = false;
  unreserve(sg);  // reserving twice counts once
  auto fits = [](const rsp_shard* s, u64 nu, u64 ne) {
    const u64 tail = (u64)s->h.mt_tail + s->inflight_units, cnt = (u64)s->h.mt_count + s->inflight_ents;
    return tail + nu <= s->h.mt_heap_cap && cnt + ne <= s->h.mt_ent_cap && (cnt + ne) * 2 <= (u64)s->h.mt_slot_mask + 1;
  };
  std::vector<rsp_shard*> to_flush;
  for (size_t g = 0; g < sg->group_shard.size(); g++) {
    rsp_shard* s = sg->group_shard[g];
    if (fits(s, sg->need_units[g], sg->need_ents[g])) continue;
    if (s->inflight_units || s->inflight_ents) return -1;  // the mirror lags the device: neither flush nor re-size now
    if (s->h.mt_count) to_flush.push_back(s);
  }
  if (!to_flush.empty()) { compact_shards(e, to_flush, false); did_work = true; }
  for (size_t g = 0; g < sg->group_shard.size(); g++) {
    rsp_shard* s = sg->group_shard[g];
    const u64 nu = sg->need_units[g], ne = sg->need_ents[g];
    if (!fits(s, nu, ne)) {  // empty but too small for this tick
      alloc_memtable(e, s, nu + nu / 2, ne + ne / 2);
      upload_shard(e, s);
      did_work = true;
    }
  }
  for (size_t g = 0; g < sg->group_shard.size(); g++) {
    sg->group_shard[g]->inflight_units += sg->need_units[g];
    sg->group_shard[g]->inflight_ents += sg->need_ents[g];
  }
  sg->reserved = true;
  return did_work ? 1 : 0;
}

static void tick_launch(rsp_engine* e, rsp_staged* sg, cudaStream_t st) {
  if (sg->fused) {
    launch_tick_fused(sg->ftick, e->d_shards, e->d_fast, e->d_mt_filter, st);
    CUDA_OK(cudaGetLastError());
    e->launches += 1;
    return;
  }
  launch_decode(sg->tick, st);
  launch_sequence(sg->tick, e->d_shards, e->d_fast, st);
  launch_insert(sg->tick, e->d_shards, e->d_mt_filter, st);
  launch_publish(sg->tick, e->d_shards, st);
  CUDA_OK(cudaGetLastError());
  e->launches += 4;
}

// fold a tick's results (per-shard state + one status word per batch) into the host mirrors
static int tick_results(rsp_staged* sg, const u8* pout, int32_t* st_out) {
  unreserve(sg);  // the mirrors below now include this tick
  const size_t ng = sg->group_shard.size();
  const GroupRes* gr = (const GroupRes*)pout;
  const u32* bs = (const u32*)(pout + ng * sizeof(GroupRes));
  int worst = RSP_OK;
  for (size_t g = 0; g < ng; g++) {
    rsp_shard* s = sg->group_shard[g];
    s->h.last_seq = gr[g].last_seq;
    s->h.pub_seq = gr[g].last_seq;
    s->h.mt_tail = gr[g].tail;
    s->h.mt_count = gr[g].count;
    s->h.latch = gr[g].latch;
    s->latch = gr[g].latch;
    s->last_seq.store(gr[g].last_seq, std::memory_order_release);
  }
  bool any_bad = false;
  for (size_t p = 0; p < sg->n; p++) {
    const u32 code = bs[p] >> 8;
    if (st_out) st_out[sg->identity_order ? p : sg->order[p]] = (int32_t)code;
    any_bad |= code != 0;
  }
  if (any_bad) {
    for (size_t g = 0; g < ng; g++) {
      for (u32 p = sg->group_first[g]; p < sg->group_first[g + 1]; p++) {
        if (bs[p]) {  // text of the first failing batch of the shard
          const u32 msg = bs[p] & 0xff;
          set_err(sg->group_shard[g], msg < MSG_COUNT ? kMsgText[msg] : "error");
          worst = (int)(bs[p] >> 8);
          break;
        }
      }
    }
  }
  return worst;
}

// Packed tick: when the caller's batches are already grouped by shard (each shard's batches contiguous, in
// order — what a per-shard aggregator produces), nothing is re-laid out on the host: the caller's blob, offsets and
// timestamps go to the device as they are (four copies), k_prepare derives the descriptors there, and the
// follower's LogData(timestamp) record is a VIRTUAL suffix the decode kernel synthesises.  Host work per batch: one
// comparison.  Returns -1 when the input does not qualify (the general, host-staged path takes over).
static int apply_many_locked(rsp_engine* e, size_t n, const uint32_t* shard_ix, const uint8_t* blob, const uint64_t* off,
                             const uint64_t* ts_ms, int32_t* st_out, bool allow_packed = true);

static int apply_many_packed(rsp_engine* e, size_t n, const uint32_t* shard_ix, const uint8_t* blob, const uint64_t* off,
                             const uint64_t* ts_ms, int32_t* st_out) {
  if (n < 1024 || off[0] != 0 || off[n] > 0xe0000000ull) return -1;
  const double t0 = now_us();
  rsp_staged sg;
  sg.eng = e;
  sg.n = n;
  sg.identity_order = true;
  std::vector<GroupDesc> groups;
  std::vector<u8>& seen = e->seen_scratch;
  if (seen.size() < e->slots.size()) seen.assign(e->slots.size(), 0);
  bool ok = true;
  size_t max_len = 0, max_group = 0;
  for (size_t i = 0; i < n; i++) {
    const u32 six = shard_ix[i];
    if (groups.empty() || six != groups.back().shard_ix) {
      if (six >= e->slots.size() || !e->slots[six] || seen[six]) { ok = false; break; }  // unknown, or not grouped
      seen[six] = 1;
      groups.push_back(GroupDesc{six, (u32)i, 0, 0});
      sg.group_shard.push_back(e->slots[six]);
    }
    groups.back().n_batches++;
    max_len = std::max<size_t>(max_len, (size_t)(off[i + 1] - off[i]));
  }
  for (const GroupDesc& g : groups) { seen[g.shard_ix] = 0; max_group = std::max<size_t>(max_group, g.n_batches); }
  if (!ok) return -1;
  const size_t ng = groups.size();
  const size_t trailer = ts_ms ? 10 : 0;
  sg.group_first.resize(ng + 1);
  for (size_t g = 0; g < ng; g++) sg.group_first[g] = groups[g].first_batch;
  sg.group_first[ng] = (u32)n;
  const size_t blob_b = (size_t)off[n];
  const bool fused = e->fused_ticks && max_len + trailer <= FUSED_MAX_BATCH_BYTES;
  // device image: [groups][off][ts][need | total][BatchDesc][blob + slack][BatchRes][GroupRes | status]
  // (the fused tick needs neither the descriptors nor the per-batch results: those regions are empty then)
  const size_t o_groups = 0, o_off = align_up(ng * sizeof(GroupDesc), 256), o_ts = o_off + align_up((n + 1) * 8, 256);
  const size_t o_need = o_ts + align_up(n * 8, 256), o_desc = o_need + align_up((2 * ng + 1) * 4, 256);
  const size_t o_blob = o_desc + (fused ? 0 : align_up(n * sizeof(BatchDesc), 256)), o_bres = o_blob + align_up(blob_b + 64, 256);
  const size_t o_out = o_bres + (fused ? 0 : align_up(n * sizeof(BatchRes), 256));
  // groups longer than one chunk: k_tick_chunks' chunk table, chain records and per-group counters
  std::vector<ChunkDesc> chunks;
  if (fused && !fused_small_shape((u32)max_group, (u32)(max_len + trailer + 16)))
    cut_chunks(groups.data(), ng, [&](size_t i) { return (u64)off[i]; }, [&](size_t i) { return (u64)off[i + 1]; }, &chunks);
  const size_t o_chunks = o_out + align_up(ng * sizeof(GroupRes) + n * 4, 256);
  const size_t o_chain = o_chunks + align_up(chunks.size() * sizeof(ChunkDesc), 256);
  const size_t total = o_chain + align_up(chunks.size() * 32 + ng * 4, 256);
  sg.res_bytes = ng * sizeof(GroupRes) + n * 4;
  sg.need_units.resize(ng);
  sg.need_ents.resize(ng);
  if (fused) {
    // No sizing round trip: the memtable room is reserved from an ESTIMATE (bytes / 16 units of payload plus two
    // header units per expected entry); the kernel's own capacity guard refuses what does not fit after all (status
    // Busy, unlatched) and those batches are retried below through the general path, which reserves exact bounds.
    for (size_t g = 0; g < ng; g++) {
      const size_t first = groups[g].first_batch, nb = groups[g].n_batches;
      const u64 bytes = off[first + nb] - off[first] + nb * trailer;
      const u64 ents = nb + bytes / 256;
      sg.need_ents[g] = (u32)ents;
      sg.need_units[g] = (u32)(bytes / 16 + 2 * ents + 1);
    }
    if (reserve_for(e, &sg) < 0) {
      if (st_out) for (size_t i = 0; i < n; i++) st_out[i] = RSP_BUSY;
      return RSP_BUSY;
    }
  }
  u8* dev = (u8*)e->dev_tick.get(total);
  CUDA_OK(cudaMemcpyAsync(dev + o_groups, groups.data(), ng * sizeof(GroupDesc), cudaMemcpyHostToDevice, e->st));
  CUDA_OK(cudaMemcpyAsync(dev + o_off, off, (n + 1) * 8, cudaMemcpyHostToDevice, e->st));
  if (ts_ms) CUDA_OK(cudaMemcpyAsync(dev + o_ts, ts_ms, n * 8, cudaMemcpyHostToDevice, e->st));
  CUDA_OK(cudaMemcpyAsync(dev + o_blob, blob, blob_b, cudaMemcpyHostToDevice, e->st));
  CUDA_OK(cudaMemsetAsync(dev + o_blob + blob_b, 0, 64, e->st));
  u32* pneed = (u32*)e->pin_out.get((2 * ng + 1) * 4 + ng * sizeof(GroupRes) + n * 4 + 256);
  u8* pout = (u8*)pneed + align_up((2 * ng + 1) * 4, 16);
  double t1 = now_us();
  if (fused) {
    sg.fused = true;
    FusedTick& f = sg.ftick;
    f.blob = dev + o_blob; f.off = (const u64*)(dev + o_off); f.len = nullptr; f.ts = ts_ms ? (const u64*)(dev + o_ts) : nullptr;
    f.groups = (const GroupDesc*)(dev + o_groups); f.gres = (GroupRes*)(dev + o_out);
    f.bstat = (u32*)(dev + o_out + ng * sizeof(GroupRes)); f.n_groups = (u32)ng; f.n_batches = (u32)n;
    f.max_group = (u32)max_group; f.max_len = (u32)(max_len + trailer + 16);
    f.chunks = (const ChunkDesc*)(dev + o_chunks); f.n_chunks = (u32)chunks.size(); f.pad = 0;
    f.chain = (u64*)(dev + o_chain); f.group_done = (u32*)(dev + o_chain + chunks.size() * 32);
    if (!chunks.empty())
      CUDA_OK(cudaMemcpyAsync(dev + o_chunks, chunks.data(), chunks.size() * sizeof(ChunkDesc), cudaMemcpyHostToDevice, e->st));
    sg.tick.gres = f.gres;
  } else {
    CUDA_OK(cudaMemsetAsync(dev + o_need, 0, (2 * ng + 1) * 4, e->st));
    PrepareArgs pa;
    pa.blob = dev + o_blob; pa.off = (const u64*)(dev + o_off); pa.ts = ts_ms ? (const u64*)(dev + o_ts) : nullptr;
    pa.groups = (const GroupDesc*)(dev + o_groups); pa.n_groups = (u32)ng; pa.n_batches = (u32)n;
    pa.batches = (BatchDesc*)(dev + o_desc); pa.need = (u32*)(dev + o_need); pa.total_ops = (u32*)(dev + o_need) + 2 * ng;
    launch_prepare(pa, e->st);
    e->launches++;
    CUDA_OK(cudaMemcpyAsync(pneed, dev + o_need, (2 * ng + 1) * 4, cudaMemcpyDeviceToHost, e->st));
    CUDA_OK(cudaStreamSynchronize(e->st));
    t1 = now_us();
    for (size_t g = 0; g < ng; g++) { sg.need_units[g] = pneed[2 * g]; sg.need_ents[g] = pneed[2 * g + 1]; }
    const u32 total_ops = pneed[2 * ng];
    if (reserve_for(e, &sg) < 0) {
      // pre-staged ticks are still in flight on these shards and the memtable is full: the caller folds them first
      if (st_out) for (size_t i = 0; i < n; i++) st_out[i] = RSP_BUSY;
      return RSP_BUSY;
    }
    TickDev& t = sg.tick;
    t.blob = dev + o_blob; t.ts = pa.ts; t.batches = pa.batches; t.groups = pa.groups;
    t.bres = (BatchRes*)(dev + o_bres); t.gres = (GroupRes*)(dev + o_out);
    t.bstat = (u32*)(dev + o_out + ng * sizeof(GroupRes));
    t.ops = (OpRec*)e->dev_ops.get((size_t)std::max<u32>(total_ops, 1) * sizeof(OpRec));
    t.n_batches = (u32)n; t.n_groups = (u32)ng; t.n_ops_cap = total_ops;
  }
  CUDA_OK(cudaEventRecord(e->ev0, e->st));
  tick_launch(e, &sg, e->st);
  CUDA_OK(cudaEventRecord(e->ev1, e->st));
  CUDA_OK(cudaMemcpyAsync(pout, sg.tick.gres, sg.res_bytes, cudaMemcpyDeviceToHost, e->st));
  CUDA_OK(cudaStreamSynchronize(e->st));
  float ms = 0;
  cudaEventElapsedTime(&ms, e->ev0, e->ev1);
  e->last_ms["apply"] = ms;
  const double t2 = now_us();
  std::vector<int32_t> st_local;
  if (fused && !st_out) { st_local.assign(n, 0); st_out = st_local.data(); }
  int worst = tick_results(&sg, pout, st_out);
  if (g_trace) fprintf(stderr, "[rsp trace] apply_many(packed%s) n=%zu copy%s %.0f us tick+sync %.0f us (kernels %.0f us) results %.0f us\n",
                       fused ? ", fused" : "", n, fused ? "" : "+prepare", t1 - t0, t2 - t1, ms * 1e3, now_us() - t2);
  if (fused) {
    // batches the capacity guard refused (the estimate was too small for their shard): again, in order, with exact bounds
    std::vector<uint32_t> again;
    for (size_t i = 0; i < n; i++)
      if (st_out[i] == RSP_BUSY && !e->slots[shard_ix[i]]->latch) again.push_back((uint32_t)i);
    if (!again.empty()) {
      const size_t m = again.size();
      std::vector<uint32_t> six(m);
      std::vector<uint64_t> off2(m + 1, 0), ts2(m);
      std::vector<uint8_t> blob2;
      for (size_t k = 0; k < m; k++) {
        const size_t i = again[k];
        six[k] = shard_ix[i];
        blob2.insert(blob2.end(), blob + off[i], blob + off[i + 1]);
        off2[k + 1] = blob2.size();
        if (ts_ms) ts2[k] = ts_ms[i];
      }
      blob2.push_back(0);
      std::vector<int32_t> st2(m, 0);
      const int rc2 = apply_many_locked(e, m, six.data(), blob2.data(), off2.data(), ts_ms ? ts2.data() : nullptr, st2.data(), false);
      for (size_t k = 0; k < m; k++) st_out[again[k]] = st2[k];
      worst = RSP_OK;
      for (size_t i = 0; i < n; i++) if (st_out[i]) { worst = st_out[i]; break; }
      if (rc2 == RSP_BUSY) worst = RSP_BUSY;
    }
  }
  return worst;
}

static int apply_many_locked(rsp_engine* e, size_t n, const uint32_t* shard_ix, const uint8_t* blob,
                             const uint64_t* off, const uint64_t* ts_ms, int32_t* st_out, bool allow_packed) {
  if (n == 0) return RSP_OK;
  if (allow_packed && !getenv("RSP_NO_PACKED")) {
    const int prc = apply_many_packed(e, n, shard_ix, blob, off, ts_ms, st_out);
    if (prc >= 0) return prc;
  }
  rsp_staged sg;
  // reserve first (may flush), then stage: staging uses the engine's tick buffers
  // sizes are only known after grouping, so build the grouping twice is avoided by staging first into
  // pinned memory and reserving before the H2D copy is consumed (same stream => ordered)
  const double t0 = now_us();
  int rc = stage_build(e, n, shard_ix, blob, off, ts_ms, &sg, false);
  if (rc != RSP_OK) return rc;
  const double t1 = now_us();
  if (reserve_for(e, &sg) < 0) {
    // pre-staged ticks are still in flight on these shards and the memtable is full: the caller folds them first
    if (st_out) for (size_t i = 0; i < n; i++) st_out[i] = RSP_BUSY;
    return RSP_BUSY;
  }
  CUDA_OK(cudaEventRecord(e->ev0, e->st));
  tick_launch(e, &sg, e->st);
  CUDA_OK(cudaEventRecord(e->ev1, e->st));
  u8* pout = (u8*)e->pin_out.get(sg.res_bytes);
  CUDA_OK(cudaMemcpyAsync(pout, sg.tick.gres, sg.res_bytes, cudaMemcpyDeviceToHost, e->st));
  CUDA_OK(cudaStreamSynchronize(e->st));
  float ms = 0;
  cudaEventElapsedTime(&ms, e->ev0, e->ev1);
  e->last_ms["apply"] = ms;
  const double t2 = now_us();
  const int worst = tick_results(&sg, pout, st_out);
  if (g_trace) fprintf(stderr, "[rsp trace] apply_many n=%zu stage %.0f us device+sync %.0f us (kernels %.0f us) results %.0f us\n", n, t1 - t0, t2 - t1, ms * 1e3, now_us() - t2);
  return worst;
}

// ------------------------------------------------------------------------------------------------
// host-side merge folding (operators that do not live on the device)
// ------------------------------------------------------------------------------------------------
struct OutCtx { std::string* s; };
static void out_set_cb(void* ctx, const uint8_t* b, size_t n) { ((OutCtx*)ctx)->s->assign((const char*)b, n); }

static bool host_merge_one(rsp_shard* s, const std::string& key, bool has, const std::string& ex,
                           const std::string& operand, std::string* out) {
  switch (s->opts.merge_op) {
    case RSP_MERGE_APPEND:
      *out = has ? ex + operand : operand;
      return true;
    case RSP_MERGE_CALLBACK: {
      if (!s->opts.merge_fn) return false;
      OutCtx c{out};
      return s->opts.merge_fn(s->opts.merge_state, (const uint8_t*)key.data(), key.size(),
                              has ? (const uint8_t*)ex.data() : nullptr, has ? ex.size() : 0,
                              (const uint8_t*)operand.data(), operand.size(), out_set_cb, &c) != 0;
    }
    default:
      return false;
  }
}

// resolve one key through the version-dump kernel and the host operator
static int host_fold_get(rsp_engine* e, rsp_shard* s, const uint8_t* key, size_t klen, std::string* value,
                         const ScanView* d_view = nullptr) {
  size_t stride = 4096;
  for (;;) {
    u8* d = (u8*)e->dev_q.get(klen + 64 + stride + 64);
    u64 koff[2] = {0, klen};
    u32 six = s->index;
    // layout: [koff 16][six 4 pad 12][n_rec 4][need 4][pad 8][key ...][out ...]
    u8* d_koff = d; u8* d_six = d + 16; u8* d_nrec = d + 32; u8* d_need = d + 36;
    u8* d_key = d + 48; u8* d_out = d + 48 + align_up(klen, 16) + 16;
    CUDA_OK(cudaMemcpyAsync(d_koff, koff, 16, cudaMemcpyHostToDevice, e->st));
    CUDA_OK(cudaMemcpyAsync(d_six, &six, 4, cudaMemcpyHostToDevice, e->st));
    if (klen) CUDA_OK(cudaMemcpyAsync(d_key, key, klen, cudaMemcpyHostToDevice, e->st));
    VersionsArgs a{e->d_shards, d_view, (const u32*)d_six, d_key, (const u64*)d_koff, d_out, stride - 64, (u32*)d_nrec, (u32*)d_need, 1};
    launch_get_versions(a, e->st);
    e->launches++;
    u32 res[2];
    CUDA_OK(cudaMemcpyAsync(res, d_nrec, 8, cudaMemcpyDeviceToHost, e->st));
    CUDA_OK(cudaStreamSynchronize(e->st));
    if (res[1] > stride - 64) { stride = (size_t)res[1] * 2 + 128; continue; }
    std::vector<u8> buf(res[1] ? res[1] : 1);
    if (res[1]) CUDA_OK(cudaMemcpy(buf.data(), d_out, res[1], cudaMemcpyDeviceToHost));
    // records newest -> oldest; fold oldest -> newest
    struct Rec { u32 type; std::string v; };
    std::vector<Rec> recs;
    size_t at = 0;
    for (u32 i = 0; i < res[0]; i++) {
      u32 type, vlen;
      memcpy(&type, &buf[at], 4);
      memcpy(&vlen, &buf[at + 4], 4);
      recs.push_back({type, std::string((const char*)&buf[at + 8], vlen)});
      at += 8 + ((vlen + 3) & ~3u);
    }
    if (recs.empty()) return RSP_NOT_FOUND;
    bool has = false;
    std::string cur;
    size_t n_ops = recs.size();
    if (recs.back().type != kTypeMerge) {
      n_ops--;
      if (recs.back().type == kTypeValue) { has = true; cur = recs.back().v; }
    }
    if (n_ops == 0) {
      if (!has) return RSP_NOT_FOUND;
      *value = cur;
      return RSP_OK;
    }
    const std::string k((const char*)key, klen);
    for (size_t i = n_ops; i-- > 0;) {
      std::string nv;
      if (!host_merge_one(s, k, has, cur, recs[i].v, &nv)) {
        set_err(s, kMsgText[MSG_MERGE_FAILED]);
        return RSP_CORRUPTION;
      }
      cur.swap(nv);
      has = true;
    }
    *value = cur;
    return RSP_OK;
  }
}

// ------------------------------------------------------------------------------------------------
// reads
// ------------------------------------------------------------------------------------------------
// pending-list scratch of the 16-byte-key kernel: [2 counters][n indices]; the counters alternate per launch
// ONE list per engine: a launch that would share it with a launch still running on ANOTHER stream waits for that one
// (launches on one stream are ordered anyway; ADVICE r01: two device-form launches on different streams wrote the
// same list).
static void pending_order(rsp_engine* e, cudaStream_t stream) {
  if (e->pending_ev_recorded && e->pending_last_stream != stream) CUDA_OK(cudaStreamWaitEvent(stream, e->pending_ev, 0));
}
static void pending_mark(rsp_engine* e, cudaStream_t stream) {
  CUDA_OK(cudaEventRecord(e->pending_ev, stream));
  e->pending_ev_recorded = true;
  e->pending_last_stream = stream;
}
static void set_pending(rsp_engine* e, GetArgs& a, size_t n, cudaStream_t stream) {
  pending_order(e, stream);
  if ((n + 8) * 4 > e->pending_cap) {
    if (e->pending_ev_recorded) CUDA_OK(cudaEventSynchronize(e->pending_ev));  // the old list may still be read
    e->pending_cap = std::max<size_t>((n + 8) * 4, e->pending_cap * 2);
    u32* p = (u32*)e->dev_pending.get(e->pending_cap);
    CUDA_OK(cudaMemsetAsync(p, 0, 16, stream));
    e->mg_parity = 0;
  }
  a.n_special = (u32*)e->dev_pending.p;
  a.n_pending = (u32*)e->dev_pending.p + 2;
  a.pending = a.n_pending + 2;
  a.parity = e->mg_parity;
  e->mg_parity ^= 1u;
}

// One MultiGet over host buffers.  Large fixed-key batches are cut into chunks that ride three streams
// (H2D -> kernel -> D2H per chunk), so the copy engines and the SMs overlap: the end-to-end rate is set by
// the slower PCIe direction, not by the sum of both plus the kernel.
static int multi_get_locked(rsp_engine* e, size_t n, const uint32_t* shard_ix, const uint8_t* keys, const uint64_t* koff,
                            uint32_t klen_fixed, uint8_t* vals, size_t val_stride, uint32_t* vlen, int32_t* st) {
  if (n == 0) return RSP_OK;
  const size_t key_bytes = klen_fixed ? n * klen_fixed : (size_t)koff[n];
  const size_t o_six = 0, o_koff = align_up(n * 4, 256), o_keys = o_koff + (klen_fixed ? 0 : align_up((n + 1) * 8, 256));
  const size_t o_vlen = o_keys + align_up(key_bytes + 16, 256), o_st = o_vlen + align_up(n * 4, 256);
  const size_t o_vals = o_st + align_up(n * 4, 256);
  const size_t total = o_vals + n * val_stride + 256;
  u8* d = (u8*)e->dev_q.get(total);
  const size_t CH = 1u << 18;
  const bool piped = klen_fixed && n >= 2 * CH;
  const size_t n_chunks = piped ? (n + CH - 1) / CH : 1;
  // scratch: [n_special][pad][2 counters per chunk][pending indices]
  const size_t scratch_u32 = 4 + 2 * n_chunks + n + 16;
  if (e->pending_ev_recorded) {  // a device-form launch on a caller's stream may still use the list: this call is
    CUDA_OK(cudaEventSynchronize(e->pending_ev));  // synchronous anyway
    e->pending_ev_recorded = false;
  }
  if (scratch_u32 * 4 > e->pending_cap) {
    e->pending_cap = std::max(scratch_u32 * 4, e->pending_cap * 2);
    e->dev_pending.get(e->pending_cap);
  }
  u32* scratch = (u32*)e->dev_pending.p;
  CUDA_OK(cudaMemsetAsync(scratch, 0, (4 + 2 * n_chunks) * 4, e->st));
  e->mg_parity = 0;
  CUDA_OK(cudaEventRecord(e->ev0, e->st));
  for (size_t c = 0; c < n_chunks; c++) {
    const size_t c0 = c * CH, cn = piped ? std::min(CH, n - c0) : n;
    cudaStream_t cs = piped ? e->cs[c % 3] : e->st;
    if (piped && c < 3) CUDA_OK(cudaStreamWaitEvent(cs, e->ev0, 0));
    CUDA_OK(cudaMemcpyAsync(d + o_six + c0 * 4, shard_ix + c0, cn * 4, cudaMemcpyHostToDevice, cs));
    if (!klen_fixed) CUDA_OK(cudaMemcpyAsync(d + o_koff, koff, (n + 1) * 8, cudaMemcpyHostToDevice, cs));
    const size_t kb0 = klen_fixed ? c0 * klen_fixed : 0, kbn = klen_fixed ? cn * klen_fixed : key_bytes;
    if (kbn) CUDA_OK(cudaMemcpyAsync(d + o_keys + kb0, keys + kb0, kbn, cudaMemcpyHostToDevice, cs));
    GetArgs a;
    a.shards = e->d_shards; a.fast = e->d_fast; a.max_shards = e->cfg.max_shards;
    a.shard_ix = (const u32*)(d + o_six) + c0; a.keys = d + o_keys + kb0;
    a.koff = klen_fixed ? nullptr : (const u64*)(d + o_koff); a.klen_fixed = klen_fixed;
    a.vals = d + o_vals + c0 * val_stride; a.val_stride = val_stride;
    a.vlen = (u32*)(d + o_vlen) + c0; a.st = (i32*)(d + o_st) + c0; a.n = (u32)cn;
    a.n_special = scratch; a.n_pending = scratch + 4 + 2 * c; a.pending = scratch + 4 + 2 * n_chunks + c0; a.parity = 0;
    a.multirun = e->n_multirun.load() ? 1u : 0u;
    launch_multi_get(a, cs);
    e->launches += 2;
    CUDA_OK(cudaMemcpyAsync(vlen + c0, d + o_vlen + c0 * 4, cn * 4, cudaMemcpyDeviceToHost, cs));
    CUDA_OK(cudaMemcpyAsync(st + c0, d + o_st + c0 * 4, cn * 4, cudaMemcpyDeviceToHost, cs));
    if (val_stride) CUDA_OK(cudaMemcpyAsync(vals + c0 * val_stride, d + o_vals + c0 * val_stride, cn * val_stride, cudaMemcpyDeviceToHost, cs));
  }
  if (piped) {
    for (int k = 0; k < 3; k++) {
      CUDA_OK(cudaEventRecord(e->cs_done[k], e->cs[k]));
      CUDA_OK(cudaStreamWaitEvent(e->st, e->cs_done[k], 0));
    }
  }
  CUDA_OK(cudaEventRecord(e->ev1, e->st));
  u32 n_special = 0;
  CUDA_OK(cudaMemcpyAsync(&n_special, scratch, 4, cudaMemcpyDeviceToHost, e->st));
  CUDA_OK(cudaStreamSynchronize(e->st));
  float ms = 0;
  cudaEventElapsedTime(&ms, e->ev0, e->ev1);
  e->last_ms["multi_get"] = ms;
  if (!n_special) return RSP_OK;
  // post-process the rare statuses: error texts, host-folded merges, unknown shards
  for (size_t i = 0; i < n; i++) {
    if (st[i] == ST_NEED_HOST_MERGE) {
      rsp_shard* s = e->slots[shard_ix[i]];
      const uint8_t* k = klen_fixed ? keys + i * klen_fixed : keys + koff[i];
      const size_t kl = klen_fixed ? klen_fixed : (size_t)(koff[i + 1] - koff[i]);
      std::string v;
      int rc = host_fold_get(e, s, k, kl, &v);
      st[i] = rc;
      vlen[i] = 0;
      if (rc == RSP_OK) {
        vlen[i] = (u32)v.size();
        if (v.size() > val_stride) st[i] = RSP_INCOMPLETE;
        else memcpy(vals + i * val_stride, v.data(), v.size());
      }
    } else if (st[i] != RSP_OK && st[i] != RSP_NOT_FOUND && st[i] != RSP_INCOMPLETE) {
      const u32 msg = vlen[i];
      if (shard_ix[i] < e->slots.size() && e->slots[shard_ix[i]])
        set_err(e->slots[shard_ix[i]], msg < MSG_COUNT ? kMsgText[msg] : "error");
      vlen[i] = 0;
    }
  }
  return RSP_OK;
}

// ------------------------------------------------------------------------------------------------
// iterator
// ------------------------------------------------------------------------------------------------
struct rsp_iter {
  rsp_shard* s;
  std::vector<std::shared_ptr<Run>> pinned;
  ScanView* d_view = nullptr;
  struct Ent { std::string first, second; int status; };  // status != 0: the merge of this key failed (empty value)
  std::vector<Ent> buf;
  size_t pos = 0;
  bool valid = false;
  bool reverse = false;      // direction the buffer was fetched in
  bool exhausted = true;     // no more entries beyond the buffer in that direction
  int status = 0;
  size_t want = 16;
  size_t stride = 16384;
};

// DBIter's status_ is sticky and is raised when the iterator REACHES a key whose merge fails (it keeps that key, with
// an empty value); entries are fetched ahead in chunks, so the status travels with the entry
static inline void iter_landed(rsp_iter* it) {
  if (it->valid && it->buf[it->pos].status) it->status = it->buf[it->pos].status;
}

// fetch up to it->want entries starting at `key` (or the extreme) in the given direction
static void iter_fetch(rsp_iter* it, const std::string* key, bool exclusive, bool reverse) {
  rsp_engine* e = it->s->eng;
  std::lock_guard<std::mutex> g(e->mu);
  CUDA_OK(cudaSetDevice(e->device));
  it->buf.clear();
  it->pos = 0;
  it->reverse = reverse;
  std::string fetch_key;
  for (;;) {
    const size_t klen = key ? key->size() : 0;
    const size_t o_key = 64, o_out = 64 + align_up(klen + 16, 256);
    u8* d = (u8*)e->dev_q.get(o_out + it->stride + 256);
    // header: [koff 2x8][flags 1][pad][n_out 4 @32][st 4 @36]
    u64 koff[2] = {0, klen};
    u8 flags = (exclusive ? 1 : 0) | (reverse ? 2 : 0) | (key ? 0 : 4);
    CUDA_OK(cudaMemcpyAsync(d, koff, 16, cudaMemcpyHostToDevice, e->st));
    CUDA_OK(cudaMemcpyAsync(d + 16, &flags, 1, cudaMemcpyHostToDevice, e->st));
    if (klen) CUDA_OK(cudaMemcpyAsync(d + o_key, key->data(), klen, cudaMemcpyHostToDevice, e->st));
    ScanArgs a;
    a.shards = nullptr; a.views = it->d_view; a.shard_ix = nullptr; a.keys = d + o_key; a.koff = (const u64*)d;
    a.klen_fixed = 0; a.flags = d + 16; a.max_entries = (u32)it->want; a.out = d + o_out; a.out_stride = it->stride;
    a.n_out = (u32*)(d + 32); a.st = (i32*)(d + 36); a.n = 1; a.max_shards = 0;
    launch_multi_scan(a, e->st);
    e->launches++;
    u32 res[2];
    CUDA_OK(cudaMemcpyAsync(res, d + 32, 8, cudaMemcpyDeviceToHost, e->st));
    CUDA_OK(cudaStreamSynchronize(e->st));
    const u32 n_out = res[0];
    const bool truncated = (i32)res[1] == RSP_INCOMPLETE || ((i32)res[1] & SCAN_ST_TRUNCATED) != 0;
    const i32 st = (i32)res[1] & ~SCAN_ST_TRUNCATED;
    if (n_out == 0 && truncated) { it->stride *= 4; continue; }
    std::vector<u8> h(it->stride);
    if (n_out) CUDA_OK(cudaMemcpy(h.data(), d + o_out, it->stride, cudaMemcpyDeviceToHost));
    size_t at = 0;
    std::string last_key;
    for (u32 i = 0; i < n_out; i++) {
      u32 kl, vl;
      memcpy(&kl, &h[at], 4);
      memcpy(&vl, &h[at + 4], 4);
      std::string k((const char*)&h[at + 8], kl);
      last_key = k;
      if (vl == SCAN_VLEN_HOST_FOLD) {  // operator lives on the host: fold this key against the pinned view
        std::string v;
        const int rc = host_fold_get(e, it->s, (const uint8_t*)k.data(), k.size(), &v, it->d_view);
        if (rc == RSP_OK) it->buf.push_back({std::move(k), std::move(v), 0});
        else if (rc != RSP_NOT_FOUND) it->buf.push_back({std::move(k), std::string(), rc});
        at += 8 + kl;
        // (the scan kernel's scratch was reused by the fold: the copy in `h` is what we keep reading)
      } else if (vl == SCAN_VLEN_MERGE_FAILED) {
        it->buf.push_back({std::move(k), std::string(), st > 255 ? (int)(st >> 8) : RSP_CORRUPTION});
        at += 8 + kl;
      } else {
        it->buf.push_back({std::move(k), std::string((const char*)&h[at + 8 + kl], vl), 0});
        at += 8 + kl + vl;
      }
    }
    it->exhausted = !(truncated || n_out == it->want);
    if (g_trace) fprintf(stderr, "[rsp trace] iter_fetch want=%zu stride=%zu reverse=%d exclusive=%d klen=%zu -> n_out=%u st=%d kept=%zu exhausted=%d\n",
                         it->want, it->stride, (int)reverse, (int)exclusive, key ? key->size() : 0, n_out, st, it->buf.size(), (int)it->exhausted);
    if (it->buf.empty() && !it->exhausted) {
      // every fetched key folded to "deleted": keep going from the last key the kernel returned
      fetch_key = last_key; key = &fetch_key; exclusive = true;
      continue;
    }
    break;
  }
  it->valid = !it->buf.empty();
  if (it->want < 1024) it->want *= 4;
  iter_landed(it);
}

// ------------------------------------------------------------------------------------------------
// staging combiners: concurrent callers of the reference's seams share device batches (stager.h)
// ------------------------------------------------------------------------------------------------
// Asynchronous completions run here, not on a dispatcher thread (a dispatcher that runs user code cannot launch).
// One task = ALL the completions of one device batch, run back to back by one thread: a wake-up per batch, not per
// response (the box's CPU time is capped: a thread hand-off per response was most of the follower's cost,
// profiles/r02_seams_trace.md); a large batch is split over a few threads, eight completions or more each.
struct CompletionPool {
  std::mutex mu;
  std::condition_variable cv;
  std::deque<std::vector<std::function<void()>>> q;
  bool stop = false;
  size_t idle = 0;
  std::vector<std::thread> th;
  void start(size_t n) {
    for (size_t i = 0; i < n; i++) th.emplace_back([this] {
      for (;;) {
        std::vector<std::function<void()>> fs;
        {
          std::unique_lock<std::mutex> l(mu);
          idle++;
          cv.wait(l, [this] { return stop || !q.empty(); });
          idle--;
          if (q.empty()) return;  // stop requested and drained
          fs = std::move(q.front());
          q.pop_front();
        }
        for (auto& f : fs) {
          try { f(); } catch (...) { abi_caught(); }  // (a caller's completion must not take the pool thread down)
        }
      }
    });
  }
  void add_many(std::vector<std::function<void()>>& fs) {
    if (fs.empty()) return;
    // tasks of >= kMinPerTask completions: a batch of a thousand shards' responses is shared by a few threads
    constexpr size_t kMinPerTask = 8;
    const size_t n_tasks = std::max<size_t>(1, std::min(th.size(), fs.size() / kMinPerTask));
    size_t wake;
    {
      std::lock_guard<std::mutex> g(mu);
      if (n_tasks == 1) {
        q.emplace_back(std::move(fs));
      } else {
        const size_t per = (fs.size() + n_tasks - 1) / n_tasks;
        for (size_t lo = 0; lo < fs.size(); lo += per) {
          q.emplace_back();
          auto& v = q.back();
          for (size_t i = lo; i < std::min(fs.size(), lo + per); i++) v.push_back(std::move(fs[i]));
        }
      }
      wake = std::min(idle, n_tasks);
    }
    fs.clear();
    for (size_t i = 0; i < wake; i++) cv.notify_one();
  }
  void shutdown() {
    {
      std::lock_guard<std::mutex> g(mu);
      stop = true;
    }
    cv.notify_all();
    for (auto& t : th) t.join();
    th.clear();
  }
};

static size_t env_size(const char* name, size_t dflt) {
  const char* v = getenv(name);
  return v && atoll(v) > 0 ? (size_t)atoll(v) : dflt;
}
static u32 stride_class(size_t want) {  // value strides are batched by power-of-two class (>= 64 bytes)
  u32 c = 64;
  while (c < want && c < (1u << 30)) c <<= 1;
  return c;
}

// pinned + mapped staging: the device reads small batches straight from it (no copy calls at all)
static u8* pinned_mapped(size_t bytes, u8** dev_alias) {
  void* p = nullptr;
  CUDA_OK(cudaHostAlloc(&p, bytes, cudaHostAllocMapped | cudaHostAllocPortable));
  void* d = nullptr;
  CUDA_OK(cudaHostGetDevicePointer(&d, p, 0));
  *dev_alias = (u8*)d;
  return (u8*)p;
}

struct ReadStage {
  u8* pin = nullptr;
  u8* pin_dev = nullptr;  // the same memory through its device address
  u8* dev = nullptr;      // HBM mirror for large batches
  u32* d_pending = nullptr;
  std::atomic<u32> not16{0};  // a key of this batch is not 16 bytes long
};
struct ReadCombiner {
  rsp_engine* e = nullptr;
  size_t cap_items = 0, cap_key_bytes = 0, cap_val_bytes = 0, zero_copy_max = 0;
  size_t o_six = 0, o_koff = 0, o_keys = 0, o_st = 0, o_vlen = 0, o_vals = 0, total = 0;
  ReadStage st[Stager::kBuffers];
  cudaStream_t stream = nullptr;
  std::unique_ptr<Stager> stager;

  void run(const Stager::BatchInfo& info) {
    try {
      run_batch(info);
    } catch (...) {  // (the dispatcher thread must survive: the callers of this batch get an IO error)
      const int rc = abi_caught();
      i32* stp = reinterpret_cast<i32*>(st[info.buf].pin + o_st);
      for (size_t i = 0; i < info.n_items; i++) stp[i] = rc;
    }
  }
  void run_batch(const Stager::BatchInfo& info) {
    ReadStage& S = st[info.buf];
    const size_t n = info.n_items;
    const u32 stride = info.klass;
    CUDA_OK(cudaSetDevice(e->device));
    reinterpret_cast<u64*>(S.pin + o_koff)[n] = info.n_bytes;
    const bool fixed16 = S.not16.exchange(0) == 0 && info.n_bytes == n * 16;
    const bool zc = n <= zero_copy_max;
    u8* base = zc ? S.pin_dev : S.dev;
    if (!zc) {
      CUDA_OK(cudaMemcpyAsync(S.dev + o_six, S.pin + o_six, n * 4, cudaMemcpyHostToDevice, stream));
      if (!fixed16) CUDA_OK(cudaMemcpyAsync(S.dev + o_koff, S.pin + o_koff, (n + 1) * 8, cudaMemcpyHostToDevice, stream));
      if (info.n_bytes) CUDA_OK(cudaMemcpyAsync(S.dev + o_keys, S.pin + o_keys, info.n_bytes, cudaMemcpyHostToDevice, stream));
    }
    GetArgs a;
    a.shards = e->d_shards; a.fast = e->d_fast; a.max_shards = e->cfg.max_shards;
    a.shard_ix = (const u32*)(base + o_six); a.keys = base + o_keys;
    a.koff = fixed16 ? nullptr : (const u64*)(base + o_koff); a.klen_fixed = fixed16 ? 16u : 0u;
    a.vals = base + o_vals; a.val_stride = stride; a.vlen = (u32*)(base + o_vlen); a.st = (i32*)(base + o_st); a.n = (u32)n;
    a.n_special = nullptr; a.n_pending = S.d_pending; a.pending = S.d_pending + 4; a.parity = 0;
    a.multirun = e->n_multirun.load() ? 1u : 0u;
    {
      // ordering against flushes / memtable re-allocations on the engine stream (reader_begin / reader_end)
      std::lock_guard<std::mutex> g(e->mu);
      reader_begin(e, stream);
      launch_multi_get(a, stream);
      CUDA_OK(cudaGetLastError());
      reader_end(e, stream);
    }
    e->launches += 2;
    if (!zc) {
      CUDA_OK(cudaMemcpyAsync(S.pin + o_st, S.dev + o_st, n * 4, cudaMemcpyDeviceToHost, stream));
      CUDA_OK(cudaMemcpyAsync(S.pin + o_vlen, S.dev + o_vlen, n * 4, cudaMemcpyDeviceToHost, stream));
      CUDA_OK(cudaMemcpyAsync(S.pin + o_vals, S.dev + o_vals, n * (size_t)stride, cudaMemcpyDeviceToHost, stream));
    }
    CUDA_OK(cudaStreamSynchronize(stream));
  }
  void destroy() {
    stager.reset();  // joins the dispatcher
    cudaSetDevice(e->device);
    for (auto& S : st) {
      if (S.pin) cudaFreeHost(S.pin);
      if (S.dev) cudaFree(S.dev);
      if (S.d_pending) cudaFree(S.d_pending);
    }
    if (stream) cudaStreamDestroy(stream);
  }
};

static ReadCombiner* read_combiner(rsp_engine* e) {
  if (ReadCombiner* c = e->read_comb_ready.load(std::memory_order_acquire)) return c;
  std::lock_guard<std::mutex> g(e->comb_mu);
  if (e->read_comb) return e->read_comb;
  CUDA_OK(cudaSetDevice(e->device));
  ReadCombiner* c = new ReadCombiner();
  c->e = e;
  c->cap_items = env_size("RSP_READ_COMBINE_ITEMS", 1u << 18);
  c->cap_key_bytes = env_size("RSP_READ_COMBINE_KEY_BYTES", c->cap_items * 24);
  c->cap_val_bytes = env_size("RSP_READ_COMBINE_VAL_BYTES", c->cap_items * 128);
  c->zero_copy_max = getenv("RSP_READ_ZERO_COPY") ? (size_t)atoll(getenv("RSP_READ_ZERO_COPY")) : 2048;
  c->o_six = 0;
  c->o_koff = align_up(c->cap_items * 4, 256);
  c->o_keys = c->o_koff + align_up((c->cap_items + 1) * 8, 256);
  c->o_st = c->o_keys + align_up(c->cap_key_bytes + 64, 256);
  c->o_vlen = c->o_st + align_up(c->cap_items * 4, 256);
  c->o_vals = c->o_vlen + align_up(c->cap_items * 4, 256);
  c->total = c->o_vals + c->cap_val_bytes + 256;
  for (auto& S : c->st) {
    S.pin = pinned_mapped(c->total, &S.pin_dev);
    CUDA_OK(cudaMalloc(&S.dev, c->total));
    CUDA_OK(cudaMalloc(&S.d_pending, (c->cap_items + 16) * 4));
    CUDA_OK(cudaMemset(S.d_pending, 0, 16));
  }
  CUDA_OK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  c->stager.reset(new Stager(c->cap_items, c->cap_key_bytes, [c](const Stager::BatchInfo& b) { c->run(b); }));
  e->read_comb = c;
  e->read_comb_ready.store(c, std::memory_order_release);
  return c;
}

// One read request through the combiner.  six_at(i) -> shard index, key_at(i, &len) -> key pointer, on_res(i, st,
// value, vlen) with the device's status (7 = the value needs more than `stride` bytes, vlen = needed; statuses
// other than 0 / 1 / 7 are the generic kernel's special cases: the caller re-runs the request on the direct path).
// Returns false when the request does not fit the staging buffers (direct path).
template <class SixAt, class KeyAt, class OnRes>
static bool read_combined(rsp_engine* e, size_t n, size_t key_bytes, u32 stride, SixAt six_at, KeyAt key_at, OnRes on_res) {
  ReadCombiner* c = read_combiner(e);
  const size_t max_items = std::min(c->cap_items, c->cap_val_bytes / stride);
  if (n > max_items / 2 || key_bytes > c->cap_key_bytes / 2) return false;
  Stager::Ticket t;
  if (!c->stager->begin(n, key_bytes, stride, max_items, &t)) return false;
  ReadStage& S = c->st[t.buf];
  u32* six = reinterpret_cast<u32*>(S.pin + c->o_six) + t.item0;
  u64* koff = reinterpret_cast<u64*>(S.pin + c->o_koff) + t.item0;
  u8* keys = S.pin + c->o_keys;
  size_t at = t.byte0;
  bool all16 = true;
  for (size_t i = 0; i < n; i++) {
    size_t len = 0;
    const uint8_t* p = key_at(i, &len);
    six[i] = six_at(i);
    koff[i] = at;
    if (len) memcpy(keys + at, p, len);
    at += len;
    all16 &= len == 16;
  }
  if (!all16) S.not16.store(1, std::memory_order_relaxed);
  c->stager->commit(t);
  c->stager->wait(t);
  struct Release {  // (the caller's result handler may throw: a slice that is never released would park its buffer for good)
    Stager* s; const Stager::Ticket& t;
    ~Release() { s->release(t); }
  } release{c->stager.get(), t};
  const i32* st = reinterpret_cast<const i32*>(S.pin + c->o_st) + t.item0;
  const u32* vlen = reinterpret_cast<const u32*>(S.pin + c->o_vlen) + t.item0;
  const u8* vals = S.pin + c->o_vals + t.item0 * (size_t)stride;
  for (size_t i = 0; i < n; i++) on_res(i, st[i], vals + i * (size_t)stride, vlen[i]);
  return true;
}

// ---- applies --------------------------------------------------------------------------------------
struct ApplyStage {
  u8* pin = nullptr;
  u8* pin_dev = nullptr;
};
struct ApplyCombiner {
  rsp_engine* e = nullptr;
  size_t cap_items = 0, cap_bytes = 0;
  size_t o_six = 0, o_off = 0, o_ts = 0, o_blob = 0, o_st = 0, total = 0;
  ApplyStage st[Stager::kBuffers];
  std::unique_ptr<Stager> stager;
  CompletionPool pool;
  std::vector<std::function<void()>> done_now;  // dispatcher thread only: completions of the batch that just ran
  // diagnostics of the asynchronous form: ns from commit to the batch having run, from there to a completion thread
  // picking the callback up, inside the callback; and the number of callbacks
  std::atomic<u64> dbg_ns[3] = {}, dbg_n{0};

  void run(const Stager::BatchInfo& info) {
    ApplyStage& S = st[info.buf];
    const size_t n = info.n_items;
    u64* off = reinterpret_cast<u64*>(S.pin + o_off);
    off[n] = info.n_bytes;
    int32_t* stv = reinterpret_cast<int32_t*>(S.pin + o_st);
    memset(stv, 0, n * 4);
    int rc;
    try {
      std::lock_guard<std::mutex> g(e->mu);
      CUDA_OK(cudaSetDevice(e->device));
      rc = apply_many_locked(e, n, reinterpret_cast<const u32*>(S.pin + o_six), S.pin + o_blob, off,
                             info.klass == 0 ? reinterpret_cast<const u64*>(S.pin + o_ts) : nullptr, stv);
    } catch (...) {
      // this is the dispatcher thread: an exception that leaves it ends the process.  A failed CUDA call (out of device
      // memory while making room, typically) fails the batch instead, every caller of it with an IO error.
      rc = abi_caught();
      for (size_t i = 0; i < n; i++) stv[i] = rc;
    }
    if (rc == RSP_INVALID_ARGUMENT || rc == RSP_BUSY)
      for (size_t i = 0; i < n; i++) if (stv[i] == 0) stv[i] = rc;
  }
  void destroy() {
    stager.reset();
    pool.shutdown();
    cudaSetDevice(e->device);
    for (auto& S : st) if (S.pin) cudaFreeHost(S.pin);
  }
};

static ApplyCombiner* apply_combiner(rsp_engine* e) {
  if (ApplyCombiner* c = e->apply_comb_ready.load(std::memory_order_acquire)) return c;
  std::lock_guard<std::mutex> g(e->comb_mu);
  if (e->apply_comb) return e->apply_comb;
  CUDA_OK(cudaSetDevice(e->device));
  ApplyCombiner* c = new ApplyCombiner();
  c->e = e;
  c->cap_items = env_size("RSP_APPLY_COMBINE_ITEMS", 1u << 17);
  c->cap_bytes = env_size("RSP_APPLY_COMBINE_BYTES", c->cap_items * 160);
  c->o_six = 0;
  c->o_off = align_up(c->cap_items * 4, 256);
  c->o_ts = c->o_off + align_up((c->cap_items + 1) * 8, 256);
  c->o_blob = c->o_ts + align_up(c->cap_items * 8, 256);
  c->o_st = c->o_blob + align_up(c->cap_bytes + 64, 256);
  c->total = c->o_st + align_up(c->cap_items * 4, 256);
  for (auto& S : c->st) S.pin = pinned_mapped(c->total, &S.pin_dev);
  c->pool.start(env_size("RSP_COMPLETION_THREADS", 8));
  c->stager.reset(new Stager(c->cap_items, c->cap_bytes, [c](const Stager::BatchInfo& b) { c->run(b); },
                             [c] { c->pool.add_many(c->done_now); }));
  e->apply_comb = c;
  e->apply_comb_ready.store(c, std::memory_order_release);
  return c;
}

// n updates of ONE shard, in order, through the apply combiner.  done == nullptr: returns after the tick with the
// first failing status (0 when all were applied) and *n_applied.  Otherwise returns RSP_OK at once and done runs on
// a completion thread.  The updates are copied before the call returns.
static int apply_combined(rsp_shard* s, size_t n, const rsp_slice* batches, const uint64_t* ts_ms, bool has_ts,
                          rsp_done_fn done, void* ctx, size_t* n_applied) {
  rsp_engine* e = s->eng;
  if (n_applied) *n_applied = 0;
  if (n == 0) {
    if (done) done(ctx, RSP_OK, 0, rsp_latest_seq(s));
    return RSP_OK;
  }
  size_t bytes = 0;
  for (size_t i = 0; i < n; i++) bytes += batches[i].size;
  ApplyCombiner* c = apply_combiner(e);
  Stager::Ticket t;
  if (n > c->cap_items / 2 || bytes > c->cap_bytes / 2 || !c->stager->begin(n, bytes, has_ts ? 0u : 1u, c->cap_items, &t)) {
    // too large for the staging buffers: one tick of its own
    std::vector<uint32_t> six(n, s->index);
    std::vector<uint64_t> off(n + 1, 0);
    std::vector<uint8_t> blob(bytes + 1);
    for (size_t i = 0; i < n; i++) {
      off[i + 1] = off[i] + batches[i].size;
      if (batches[i].size) memcpy(&blob[off[i]], batches[i].data, batches[i].size);
    }
    std::vector<int32_t> stv(n, 0);
    int rc;
    {
      std::lock_guard<std::mutex> g(e->mu);
      CUDA_OK(cudaSetDevice(e->device));
      rc = apply_many_locked(e, n, six.data(), blob.data(), off.data(), has_ts ? ts_ms : nullptr, stv.data());
    }
    size_t ok = 0;
    while (ok < n && stv[ok] == 0) ok++;
    const int first = ok < n ? (stv[ok] ? stv[ok] : rc) : RSP_OK;
    if (n_applied) *n_applied = ok;
    if (done) { done(ctx, first, ok, rsp_latest_seq(s)); return RSP_OK; }
    return first;
  }
  ApplyStage& S = c->st[t.buf];
  u32* six = reinterpret_cast<u32*>(S.pin + c->o_six) + t.item0;
  u64* off = reinterpret_cast<u64*>(S.pin + c->o_off) + t.item0;
  u64* ts = reinterpret_cast<u64*>(S.pin + c->o_ts) + t.item0;
  u8* blob = S.pin + c->o_blob;
  size_t at = t.byte0;
  for (size_t i = 0; i < n; i++) {
    six[i] = s->index;
    off[i] = at;
    ts[i] = has_ts ? ts_ms[i] : 0;
    if (batches[i].size) memcpy(blob + at, batches[i].data, batches[i].size);
    at += batches[i].size;
  }
  const int32_t* stv = reinterpret_cast<const int32_t*>(S.pin + c->o_st) + t.item0;
  auto result = [stv, n](size_t* ok_out) {
    size_t ok = 0;
    while (ok < n && stv[ok] == 0) ok++;
    *ok_out = ok;
    return ok < n ? (int)stv[ok] : (int)RSP_OK;
  };
  if (done) {
    const double t_commit = now_us();
    c->stager->commit_async(t, [c, s, done, ctx, result, t_commit] {
      size_t ok = 0;
      const int first = result(&ok);
      const uint64_t seq = rsp_latest_seq(s);
      const double t_ran = now_us();
      c->dbg_ns[0].fetch_add((u64)(1e3 * (t_ran - t_commit)), std::memory_order_relaxed);
      c->done_now.push_back([c, done, ctx, first, ok, seq, t_ran] {
        const double t_start = now_us();
        done(ctx, first, ok, seq);
        c->dbg_ns[1].fetch_add((u64)(1e3 * (t_start - t_ran)), std::memory_order_relaxed);
        c->dbg_ns[2].fetch_add((u64)(1e3 * (now_us() - t_start)), std::memory_order_relaxed);
        c->dbg_n.fetch_add(1, std::memory_order_relaxed);
      });
    });
    return RSP_OK;
  }
  c->stager->commit(t);
  c->stager->wait(t);
  size_t ok = 0;
  const int first = result(&ok);
  c->stager->release(t);
  if (n_applied) *n_applied = ok;
  return first;
}

// ------------------------------------------------------------------------------------------------
// extern "C"
// ------------------------------------------------------------------------------------------------
extern "C" {

const char* rsp_version(void) { return "rocksplicator_b200 0.1 (sm_100a)"; }

int rsp_engine_create(int device, const rsp_engine_cfg* cfg, rsp_engine** out) {
  try {
  if (!out) return RSP_INVALID_ARGUMENT;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) {
    fprintf(stderr, "[rsp_b200] no CUDA device %d (the engine has no CPU fallback)\n", device);
    return RSP_IO_ERROR;
  }
  CUDA_OK(cudaSetDevice(device));
  {
    // random 96-byte entry reads: ask L2 for sector-sized DRAM fetches (default is wider)
    const char* g = getenv("RSP_L2_FETCH_BYTES");
    const size_t gran = g ? (size_t)atoi(g) : 32;
    if (gran) cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, gran);
  }
  rsp_engine* e = new rsp_engine();
  e->device = device;
  if (cfg) e->cfg = *cfg;
  if (!e->cfg.max_shards) e->cfg.max_shards = 16384;
  if (!e->cfg.arena_bytes) e->cfg.arena_bytes = 1ull << 30;
  if (!e->cfg.l0_compaction_trigger) e->cfg.l0_compaction_trigger = 4;
  if (e->cfg.l0_compaction_trigger > RSP_MAX_RUNS) e->cfg.l0_compaction_trigger = RSP_MAX_RUNS;
  e->arena.slab_bytes = e->cfg.arena_bytes;
  e->arena.slab_alloc = arena_slab_alloc;
  e->arena.slab_free = arena_slab_free;
  // measured on the B200 host (128 cores): 2 staging threads 29 M applies/s, 1: 27, 8: 19 (spawn cost wins)
  e->stage_threads = 2;
  if (const char* t = getenv("RSP_STAGE_THREADS")) e->stage_threads = (size_t)std::max(1, atoi(t));
  if (const char* t = getenv("RSP_FUSED_TICK")) e->fused_ticks = atoi(t) != 0;
  if (const char* t = getenv("RSP_BG_COMPACT")) e->bg_compaction = atoi(t) != 0;
  CUDA_OK(cudaStreamCreateWithFlags(&e->st, cudaStreamNonBlocking));
  for (int k = 0; k < 3; k++) {
    CUDA_OK(cudaStreamCreateWithFlags(&e->cs[k], cudaStreamNonBlocking));
    CUDA_OK(cudaEventCreateWithFlags(&e->cs_done[k], cudaEventDisableTiming));
  }
  for (int k = 0; k < 8; k++) CUDA_OK(cudaEventCreateWithFlags(&e->reader_ev[k], cudaEventDisableTiming));
  CUDA_OK(cudaEventCreateWithFlags(&e->mut_ev, cudaEventDisableTiming));
  CUDA_OK(cudaEventCreate(&e->ev0));
  CUDA_OK(cudaEventCreate(&e->ev1));
  CUDA_OK(cudaEventCreateWithFlags(&e->up_ev, cudaEventDisableTiming));
  CUDA_OK(cudaEventCreateWithFlags(&e->pending_ev, cudaEventDisableTiming));
  CUDA_OK(cudaMalloc(&e->d_shards, sizeof(ShardDev) * e->cfg.max_shards));
  CUDA_OK(cudaMemset(e->d_shards, 0, sizeof(ShardDev) * e->cfg.max_shards));
  {
    // [ShardFast x max_shards][ShardFast x max_shards x RSP_MAX_RUNS][memtable filter: MT_FILTER_WORDS x max_shards]
    const size_t n_fast = (size_t)e->cfg.max_shards * (1 + RSP_MAX_RUNS);
    const size_t fast_b = sizeof(ShardFast) * n_fast + (size_t)e->cfg.max_shards * MT_FILTER_WORDS * 4;
    CUDA_OK(cudaMalloc(&e->d_fast, fast_b));
    CUDA_OK(cudaMemset(e->d_fast, 0, fast_b));
    e->d_fast_runs = e->d_fast + e->cfg.max_shards;
    e->d_mt_filter = reinterpret_cast<u32*>(e->d_fast + n_fast);
  }
  if (e->bg_compaction) {
    Compactor* c = new Compactor();
    c->e = e;
    CUDA_OK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    CUDA_OK(cudaEventCreate(&c->ev0));
    CUDA_OK(cudaEventCreate(&c->ev1));
    e->compactor = c;
    c->th = std::thread([c] { c->loop(); });
  }
  *out = e;
  return RSP_OK;
  } catch (...) { return abi_caught(); }
}

void rsp_engine_destroy(rsp_engine* e) {
  if (!e) return;
  if (Compactor* c = e->compactor) {  // let a merge in flight finish, then stop the thread
    {
      std::lock_guard<std::mutex> g(c->mu);
      c->stop = true;
      c->pending.clear();
    }
    c->cv.notify_all();
    if (c->th.joinable()) c->th.join();
    cudaSetDevice(e->device);
    cudaStreamDestroy(c->stream);
    cudaEventDestroy(c->ev0);
    cudaEventDestroy(c->ev1);
    c->pin_totals.destroy();
    delete c;
    e->compactor = nullptr;
  }
  if (e->read_comb) { e->read_comb->destroy(); delete e->read_comb; }
  if (e->apply_comb) { e->apply_comb->destroy(); delete e->apply_comb; }
  cudaSetDevice(e->device);
  cudaStreamSynchronize(e->st);
  for (rsp_shard* s : e->slots)
    if (s) { s->runs.clear(); delete s; }
  e->arena.destroy();
  e->pin_in.destroy(); e->pin_out.destroy(); e->pin_up.destroy(); e->pin_totals.destroy(); e->dev_up.destroy(); e->dev_tick.destroy(); e->dev_q.destroy(); e->dev_pending.destroy(); e->dev_ops.destroy();
  cudaFree(e->d_shards);
  cudaFree(e->d_fast);
  cudaEventDestroy(e->ev0); cudaEventDestroy(e->ev1); cudaEventDestroy(e->up_ev); cudaEventDestroy(e->pending_ev);
  for (int k = 0; k < 8; k++) cudaEventDestroy(e->reader_ev[k]);
  cudaEventDestroy(e->mut_ev);
  for (int k = 0; k < 3; k++) { cudaStreamDestroy(e->cs[k]); cudaEventDestroy(e->cs_done[k]); }
  cudaStreamDestroy(e->st);
  delete e;
}

int rsp_engine_device(const rsp_engine* e) { return e->device; }
void* rsp_engine_stream(const rsp_engine* e) { return (void*)e->st; }

static int shard_open_locked(rsp_engine* e, const char* name, const rsp_shard_opts* opts, rsp_shard** out) {
  if (e->by_name.count(name)) return RSP_INVALID_ARGUMENT;
  u32 ix = 0;
  while (ix < e->slots.size() && e->slots[ix]) ix++;
  if (ix >= e->cfg.max_shards) return RSP_BUSY;
  if (ix == e->slots.size()) e->slots.push_back(nullptr);
  rsp_shard* s = new rsp_shard();
  static std::atomic<u64> next_uid{1};
  s->uid = next_uid++;
  s->eng = e; s->name = name; s->index = ix;
  memset(&s->opts, 0, sizeof(s->opts));
  if (opts) s->opts = *opts;
  memset(&s->h, 0, sizeof(s->h));
  s->h.merge_op = s->opts.merge_op;
  s->h.live = 1;
  alloc_memtable(e, s, 0, 0);
  upload_shard(e, s);
  CUDA_OK(cudaStreamSynchronize(e->st));
  e->slots[ix] = s;
  e->by_name[name] = s;
  *out = s;
  return RSP_OK;
}

static void shard_close_locked(rsp_shard* s) {
  rsp_engine* e = s->eng;
  wait_readers(e);
  CUDA_OK(cudaStreamSynchronize(e->st));
  e->slots[s->index] = nullptr;
  e->by_name.erase(s->name);
  if (s->counted_multirun) { e->n_multirun--; s->counted_multirun = false; }
  ShardDev z;
  memset(&z, 0, sizeof(z));
  CUDA_OK(cudaMemcpy(e->d_shards + s->index, &z, sizeof(z), cudaMemcpyHostToDevice));
  CUDA_OK(cudaMemset(e->d_fast + s->index, 0, sizeof(ShardFast)));
  CUDA_OK(cudaMemset(e->d_fast_runs + (size_t)s->index * RSP_MAX_RUNS, 0, sizeof(ShardFast) * RSP_MAX_RUNS));
  CUDA_OK(cudaMemset(e->d_mt_filter + (size_t)s->index * MT_FILTER_WORDS, 0, MT_FILTER_WORDS * 4));
  e->arena.release(s->h.mt_heap, s->mt_heap_bytes);
  e->arena.release(s->h.mt_slots, s->mt_slot_bytes);
  e->arena.release(s->h.mt_ent_off, s->mt_ent_bytes);
  s->runs.clear();
  delete s;
}

int rsp_shard_open(rsp_engine* e, const char* name, const rsp_shard_opts* opts, rsp_shard** out) {
  try {
  if (!e || !name || !out) return RSP_INVALID_ARGUMENT;
  std::lock_guard<std::mutex> g(e->mu);
  CUDA_OK(cudaSetDevice(e->device));
  return shard_open_locked(e, name, opts, out);
  } catch (...) { return abi_caught(); }
}

int rsp_shard_close(rsp_shard* s) {
  try {
  if (!s) return RSP_INVALID_ARGUMENT;
  rsp_engine* e = s->eng;
  std::lock_guard<std::mutex> g(e->mu);
  if (ticks_in_flight(s)) return RSP_BUSY;
  CUDA_OK(cudaSetDevice(e->device));
  shard_close_locked(s);
  return RSP_OK;
  } catch (...) { return abi_caught(); }
}

// first / last user key of a run (two small copies: the run is immutable)
static void run_key_range(rsp_engine* e, const Run& r, std::string* first, std::string* last) {
  auto key_at = [&](u32 unit, std::string* out) {
    u32 hd[4];
    CUDA_OK(cudaMemcpy(hd, r.heap + (size_t)unit * 16, 16, cudaMemcpyDeviceToHost));
    out->resize(hd[2]);
    if (hd[2]) CUDA_OK(cudaMemcpy(&(*out)[0], r.heap + (size_t)unit * 16 + 16, hd[2], cudaMemcpyDeviceToHost));
  };
  u32 first_unit = 0, last_unit = 0;
  CUDA_OK(cudaMemcpy(&first_unit, r.ent_off, 4, cudaMemcpyDeviceToHost));
  CUDA_OK(cudaMemcpy(&last_unit, r.ent_off + (r.n_ent - 1), 4, cudaMemcpyDeviceToHost));
  key_at(first_unit, first);
  key_at(last_unit, last);
  (void)e;
}

// DB::IngestExternalFile for a sorted set of Puts (rocksdb_admin/admin_handler.cpp:1820-1845, sequence rules of
// rocksdb_replicator/tests/rocksdb_assumption_test.cpp:248-283): the keys become ONE new sorted run.  When its key
// range intersects existing data the run is newer than everything and the shard's sequence number advances by one
// (refused unless allow_global_seqno); otherwise the sequence number does not move.  The run is produced by the
// ordinary apply + flush kernels on a scratch shard and then handed to the target (sequence numbers inside runs are
// not consulted by reads: recency is the run order).
int rsp_ingest_sorted(rsp_shard* s, size_t n, const uint8_t* keys, const uint64_t* koff, const uint8_t* vals,
                      const uint64_t* voff, int allow_global_seqno, uint64_t* seq_out) {
  try {
  if (!s || !n || !keys || !koff || !voff) return RSP_INVALID_ARGUMENT;
  rsp_engine* e = s->eng;
  std::lock_guard<std::mutex> g(e->mu);
  CUDA_OK(cudaSetDevice(e->device));
  auto key = [&](size_t i) { return std::string((const char*)keys + koff[i], (size_t)(koff[i + 1] - koff[i])); };
  for (size_t i = 1; i < n; i++) {
    const size_t al = (size_t)(koff[i] - koff[i - 1]), bl = (size_t)(koff[i + 1] - koff[i]);
    const int c = memcmp(keys + koff[i - 1], keys + koff[i], std::min(al, bl));
    if (c > 0 || (c == 0 && al >= bl)) { set_err(s, "Invalid argument: Keys must be added in order"); return RSP_INVALID_ARGUMENT; }
  }
  if (s->latch) return (int)(s->latch >> 8);
  if (ticks_in_flight(s)) return RSP_BUSY;
  // everything the shard holds must be in runs before ranges are compared
  if (s->h.mt_count) compact_shards(e, {s}, false);
  if (s->runs.size() + 1 > RSP_MAX_RUNS) compact_shards(e, {s}, true);
  const std::string lo = key(0), hi = key(n - 1);
  bool overlap = false;
  for (auto& r : s->runs) {
    if (!r->n_ent) continue;
    std::string rf, rl;
    run_key_range(e, *r, &rf, &rl);
    if (!(hi < rf) && !(rl < lo)) { overlap = true; break; }
  }
  if (overlap && !allow_global_seqno) {
    set_err(s, "Invalid argument: Global seqno is required, but disabled");
    return RSP_INVALID_ARGUMENT;
  }
  // build the run on a scratch shard with the ordinary apply + flush path
  rsp_shard* tmp = nullptr;
  rsp_shard_opts so;
  memset(&so, 0, sizeof(so));
  size_t payload = (size_t)koff[n] + (size_t)voff[n];
  so.write_buffer_bytes = payload + n * 64 + (1u << 20);
  static std::atomic<u64> ctr{0};
  const std::string tname = "__ingest_" + std::to_string(ctr++);
  int rc = shard_open_locked(e, tname.c_str(), &so, &tmp);
  if (rc != RSP_OK) return rc;
  const size_t CH = 1u << 16;
  for (size_t c0 = 0; c0 < n && rc == RSP_OK; c0 += CH) {
    const size_t cn = std::min(CH, n - c0);
    std::string blob;
    std::vector<uint64_t> off(cn + 1, 0);
    std::vector<uint32_t> six(cn, tmp->index);
    for (size_t i = 0; i < cn; i++) {
      const std::string k = key(c0 + i);
      const size_t vl = (size_t)(voff[c0 + i + 1] - voff[c0 + i]);
      off[i] = blob.size();
      blob.append(8, '\0');
      const uint32_t one = 1;
      blob.append((const char*)&one, 4);
      blob.push_back(0x1);
      for (uint32_t v = (uint32_t)k.size(); ; v >>= 7) { if (v >= 128) blob.push_back((char)((v & 127) | 128)); else { blob.push_back((char)v); break; } }
      blob.append(k);
      for (uint32_t v = (uint32_t)vl; ; v >>= 7) { if (v >= 128) blob.push_back((char)((v & 127) | 128)); else { blob.push_back((char)v); break; } }
      blob.append((const char*)vals + voff[c0 + i], vl);
    }
    off[cn] = blob.size();
    blob.push_back('\0');
    std::vector<int32_t> st(cn, 0);
    rc = apply_many_locked(e, cn, six.data(), (const uint8_t*)blob.data(), off.data(), nullptr, st.data());
  }
  if (rc == RSP_OK) {
    compact_shards(e, {tmp}, false);
    if (tmp->runs.size() > 1) compact_shards(e, {tmp}, true);
    std::shared_ptr<Run> in;
    if (!tmp->runs.empty()) {
      in = tmp->runs[0];
      s->runs.insert(s->runs.begin(), in);
      tmp->runs.clear();
    }
    if (overlap) {
      const u64 seq = s->last_seq.load() + 1;
      s->h.last_seq = seq;
      s->h.pub_seq = seq;
      s->last_seq.store(seq, std::memory_order_release);
    }
    if (in) {  // (before the descriptor upload below: no reader sees the run yet)
      launch_set_run_seq(in->heap, in->ent_off, in->n_ent, s->last_seq.load(), e->st);
      CUDA_OK(cudaGetLastError());
      e->launches += 1;
    }
    upload_shard(e, s);
    note_mutation(e);
    CUDA_OK(cudaStreamSynchronize(e->st));
  }
  shard_close_locked(tmp);
  if (seq_out) *seq_out = s->last_seq.load();
  return rc;
  } catch (...) { return abi_caught(); }
}

uint32_t rsp_shard_index(const rsp_shard* s) { return s->index; }
const char* rsp_shard_name(const rsp_shard* s) { return s->name.c_str(); }
uint64_t rsp_latest_seq(const rsp_shard* s) { return s->last_seq.load(std::memory_order_acquire); }

int rsp_set_latest_seq(rsp_shard* s, uint64_t seq) {
  try {
  if (!s) return RSP_INVALID_ARGUMENT;
  rsp_engine* e = s->eng;
  std::lock_guard<std::mutex> g(e->mu);
  if (ticks_in_flight(s)) return RSP_BUSY;
  if (seq < s->last_seq.load()) return RSP_INVALID_ARGUMENT;
  CUDA_OK(cudaSetDevice(e->device));
  s->h.last_seq = seq;
  s->h.pub_seq = seq;
  s->last_seq.store(seq, std::memory_order_release);
  upload_shard(e, s);
  note_mutation(e);
  CUDA_OK(cudaStreamSynchronize(e->st));
  return RSP_OK;
  } catch (...) { return abi_caught(); }
}

size_t rsp_last_error(const rsp_shard* s, char* buf, size_t cap) {
  try {
  rsp_shard* m = const_cast<rsp_shard*>(s);
  std::lock_guard<std::mutex> g(m->err_mu);
  if (buf && cap) snprintf(buf, cap, "%s", m->last_error.c_str());
  return m->last_error.size();
  } catch (...) { abi_caught(); return 0; }
}

int rsp_apply_many(rsp_engine* e, size_t n, const uint32_t* shard_ix, const uint8_t* blob, const uint64_t* off,
                   const uint64_t* ts_ms, int32_t* st_out) {
  try {
  if (!e || (n && (!shard_ix || !off))) return RSP_INVALID_ARGUMENT;
  std::lock_guard<std::mutex> g(e->mu);
  CUDA_OK(cudaSetDevice(e->device));
  return apply_many_locked(e, n, shard_ix, blob, off, ts_ms, st_out);
  } catch (...) {
    // (a failed CUDA call — out of device memory while making room, typically: before the tick ran, nothing of it applied)
    const int rc = abi_caught();
    if (st_out) for (size_t i = 0; i < n; i++) st_out[i] = rc;
    return rc;
  }
}

int rsp_apply(rsp_shard* s, const uint8_t* batch, size_t len, uint64_t ts_ms, uint64_t* seq_out) {
  try {
  if (!s) return RSP_INVALID_ARGUMENT;
  static const uint8_t empty = 0;
  const rsp_slice b{batch ? batch : &empty, len};
  const int rc = apply_combined(s, 1, &b, &ts_ms, true, nullptr, nullptr, nullptr);  // concurrent callers share one device tick
  if (seq_out) *seq_out = rsp_latest_seq(s);
  return rc;
  } catch (...) { return abi_caught(); }
}

int rsp_write(rsp_shard* s, const uint8_t* batch, size_t len, uint64_t* seq_out) {
  try {
  if (!s) return RSP_INVALID_ARGUMENT;
  static const uint8_t empty = 0;
  const rsp_slice b{batch ? batch : &empty, len};
  const int rc = apply_combined(s, 1, &b, nullptr, false, nullptr, nullptr, nullptr);
  if (seq_out) *seq_out = rsp_latest_seq(s);
  return rc;
  } catch (...) { return abi_caught(); }
}

int rsp_apply_updates(rsp_shard* s, size_t n, const rsp_slice* batches, const uint64_t* ts_ms, rsp_done_fn done,
                      void* ctx, size_t* n_applied) {
  try {
  if (!s || (n && !batches)) return RSP_INVALID_ARGUMENT;
  return apply_combined(s, n, batches, ts_ms, ts_ms != nullptr, done, ctx, n_applied);
  } catch (...) { return abi_caught(); }
}

// statuses the fast / generic kernels settle themselves; anything else (host-folded merges, error texts, unknown
// shards) is post-processed by the direct path
static inline bool plain_status(int32_t st) { return st == RSP_OK || st == RSP_NOT_FOUND || st == RSP_INCOMPLETE; }

static int multi_get_direct(rsp_engine* e, size_t n, const uint32_t* shard_ix, const uint8_t* keys, const uint64_t* koff,
                            uint32_t klen_fixed, uint8_t* vals, size_t val_stride, uint32_t* vlen, int32_t* st) {
  std::lock_guard<std::mutex> g(e->mu);
  CUDA_OK(cudaSetDevice(e->device));
  return multi_get_locked(e, n, shard_ix, keys, koff, klen_fixed, vals, val_stride, vlen, st);
}

// rsp_multi_get / rsp_multi_get_fixed: through the read combiner when the request fits its staging buffers
static int multi_get_any(rsp_engine* e, size_t n, const uint32_t* shard_ix, const uint8_t* keys, const uint64_t* koff,
                         uint32_t klen_fixed, uint8_t* vals, size_t val_stride, uint32_t* vlen, int32_t* st) {
  if (n == 0) return RSP_OK;
  const size_t key_bytes = klen_fixed ? n * (size_t)klen_fixed : (size_t)(koff[n] - koff[0]);
  const u32 stride = stride_class(val_stride);
  bool special = false;
  const bool combined = val_stride <= (1u << 20) && read_combined(
      e, n, key_bytes, stride, [&](size_t i) { return shard_ix[i]; },
      [&](size_t i, size_t* len) {
        if (klen_fixed) { *len = klen_fixed; return keys + i * (size_t)klen_fixed; }
        *len = (size_t)(koff[i + 1] - koff[i]);
        return keys + koff[i];
      },
      [&](size_t i, int32_t s_i, const u8* v, u32 vl) {
        st[i] = s_i;
        vlen[i] = vl;
        if (s_i == RSP_OK) {
          if (vl > val_stride) st[i] = RSP_INCOMPLETE;
          else if (vl) memcpy(vals + i * val_stride, v, vl);
        } else if (!plain_status(s_i)) special = true;
      });
  if (combined && !special) return RSP_OK;
  return multi_get_direct(e, n, shard_ix, keys, koff, klen_fixed, vals, val_stride, vlen, st);
}

int rsp_multi_get(rsp_engine* e, size_t n, const uint32_t* shard_ix, const uint8_t* keys, const uint64_t* koff,
                  uint8_t* vals, size_t val_stride, uint32_t* vlen, int32_t* st) {
  try {
  if (!e || (n && (!shard_ix || !koff || !vlen || !st))) return RSP_INVALID_ARGUMENT;
  return multi_get_any(e, n, shard_ix, keys, koff, 0, vals, val_stride, vlen, st);
  } catch (...) { return abi_caught(); }
}

int rsp_multi_get_fixed(rsp_engine* e, size_t n, const uint32_t* shard_ix, const uint8_t* keys, uint32_t klen,
                        uint8_t* vals, size_t val_stride, uint32_t* vlen, int32_t* st) {
  try {
  if (!e || !klen || (n && (!shard_ix || !keys || !vlen || !st))) return RSP_INVALID_ARGUMENT;
  return multi_get_any(e, n, shard_ix, keys, nullptr, klen, vals, val_stride, vlen, st);
  } catch (...) { return abi_caught(); }
}

int rsp_multi_get_slices(rsp_shard* s, size_t n, const rsp_slice* keys, size_t value_hint, rsp_value_fn fn, void* ctx) {
  try {
  if (!s || !fn || (n && !keys)) return RSP_INVALID_ARGUMENT;
  if (n == 0) return RSP_OK;
  rsp_engine* e = s->eng;
  size_t key_bytes = 0;
  for (size_t i = 0; i < n; i++) key_bytes += keys[i].size;
  static const uint8_t empty = 0;
  std::vector<uint32_t> again;  // values larger than the stride of the first pass
  size_t need = 0;
  bool special = false;
  const u32 stride = stride_class(value_hint ? value_hint : 256);
  const bool combined = read_combined(
      e, n, key_bytes, stride, [&](size_t) { return s->index; },
      [&](size_t i, size_t* len) { *len = keys[i].size; return keys[i].data ? keys[i].data : &empty; },
      [&](size_t i, int32_t st, const u8* v, u32 vl) {
        if (st == RSP_INCOMPLETE) { again.push_back((uint32_t)i); need = std::max<size_t>(need, vl); }
        else if (!plain_status(st)) special = true;
        else if (!special) fn(ctx, i, st, st == RSP_OK ? v : nullptr, st == RSP_OK ? vl : 0);
      });
  if (combined && !special && again.empty()) return RSP_OK;
  // the rest (oversized values; or everything when the request did not fit / met a special status) on the direct path
  std::vector<uint32_t> idx;
  if (combined && !special) idx.swap(again);
  else { idx.resize(n); for (size_t i = 0; i < n; i++) idx[i] = (uint32_t)i; }
  const size_t m = idx.size();
  std::vector<uint32_t> six(m, s->index), vlen(m);
  std::vector<uint64_t> koff(m + 1, 0);
  std::vector<int32_t> st(m);
  std::string blob;
  for (size_t j = 0; j < m; j++) { blob.append((const char*)keys[idx[j]].data, keys[idx[j]].size); koff[j + 1] = blob.size(); }
  blob.push_back('\0');
  size_t vs = std::max<size_t>(stride_class(std::max<size_t>(need, value_hint ? value_hint : 256)), 64);
  for (;;) {
    std::vector<uint8_t> vals(m * vs);
    const int rc = multi_get_direct(e, m, six.data(), (const uint8_t*)blob.data(), koff.data(), 0, vals.data(), vs, vlen.data(), st.data());
    if (rc != RSP_OK) return rc;
    size_t more = 0;
    for (size_t j = 0; j < m; j++) if (st[j] == RSP_INCOMPLETE) more = std::max<size_t>(more, vlen[j]);
    if (more) { vs = stride_class(more); continue; }
    for (size_t j = 0; j < m; j++) fn(ctx, idx[j], st[j], st[j] == RSP_OK ? &vals[j * vs] : nullptr, st[j] == RSP_OK ? vlen[j] : 0);
    return RSP_OK;
  }
  } catch (...) { return abi_caught(); }
}

int rsp_get(rsp_shard* s, const uint8_t* key, size_t klen, uint8_t* val, size_t cap, size_t* vlen) {
  try {
  if (!s) return RSP_INVALID_ARGUMENT;
  const uint64_t koff[2] = {0, klen};
  const uint32_t six = s->index;
  uint32_t vl = 0;
  int32_t st = 0;
  static const uint8_t empty = 0;
  // n = 1 through the read combiner: concurrent Get callers (up to 256 thrift workers in the reference) share launches
  int rc = multi_get_any(s->eng, 1, &six, key ? key : &empty, koff, 0, val, cap, &vl, &st);
  if (rc != RSP_OK) return rc;
  if (vlen) *vlen = vl;
  return st;
  } catch (...) { return abi_caught(); }
}


// ---- router: one process, several engines (include/rsp_b200.h) ------------------------------------------------
struct rsp_router {
  std::vector<rsp_engine*> engines;
  std::mutex mu;  // the shard table
  std::unordered_map<uint32_t, std::pair<uint32_t, uint32_t>> where;  // router id -> (engine ordinal, shard index there)
};

int rsp_router_create(size_t n_engines, rsp_engine* const* engines, rsp_router** out) {
  try {
  if (!n_engines || !engines || !out) return RSP_INVALID_ARGUMENT;
  rsp_router* r = new rsp_router();
  r->engines.assign(engines, engines + n_engines);
  *out = r;
  return RSP_OK;
  } catch (...) { return abi_caught(); }
}
void rsp_router_destroy(rsp_router* r) { delete r; }
int rsp_router_add_shard(rsp_router* r, uint32_t shard_id, rsp_shard* s) {
  try {
  if (!r || !s) return RSP_INVALID_ARGUMENT;
  for (size_t k = 0; k < r->engines.size(); k++) {
    if (r->engines[k] != s->eng) continue;
    std::lock_guard<std::mutex> g(r->mu);
    if (r->where.count(shard_id)) return RSP_INVALID_ARGUMENT;
    r->where[shard_id] = {(uint32_t)k, s->index};
    return RSP_OK;
  }
  return RSP_INVALID_ARGUMENT;  // the shard lives on an engine the router does not know
  } catch (...) { return abi_caught(); }
}
int rsp_router_remove_shard(rsp_router* r, uint32_t shard_id) {
  try {
  if (!r) return RSP_INVALID_ARGUMENT;
  std::lock_guard<std::mutex> g(r->mu);
  return r->where.erase(shard_id) ? RSP_OK : RSP_NOT_FOUND;
  } catch (...) { return abi_caught(); }
}

extern "C++" {
namespace {
// requests bucketed by engine, caller order kept inside a bucket
struct Buckets {
  std::vector<std::vector<uint32_t>> idx;    // [engine] -> caller indices
  std::vector<std::vector<uint32_t>> local;  // [engine] -> shard index on that engine
  std::vector<uint32_t> unknown;             // caller indices with an unregistered shard id
};
Buckets bucket_by_engine(rsp_router* r, size_t n, const uint32_t* shard_id) {
  Buckets b;
  b.idx.resize(r->engines.size());
  b.local.resize(r->engines.size());
  std::lock_guard<std::mutex> g(r->mu);
  uint32_t last_id = 0;
  const std::pair<uint32_t, uint32_t>* last = nullptr;
  for (size_t i = 0; i < n; i++) {
    if (!last || shard_id[i] != last_id) {  // batches come grouped by shard more often than not
      auto it = r->where.find(shard_id[i]);
      last = it == r->where.end() ? nullptr : &it->second;
      last_id = shard_id[i];
    }
    if (!last) { b.unknown.push_back((uint32_t)i); continue; }
    b.idx[last->first].push_back((uint32_t)i);
    b.local[last->first].push_back(last->second);
  }
  return b;
}
// run fn(k) for every engine with work, concurrently (each call drives its own device and synchronises it)
template <class F> void for_each_engine(const Buckets& b, F fn) {
  std::vector<std::thread> th;
  int first = -1;
  for (size_t k = 0; k < b.idx.size(); k++) {
    if (b.idx[k].empty()) continue;
    if (first < 0) { first = (int)k; continue; }
    th.emplace_back(fn, k);
  }
  if (first >= 0) fn((size_t)first);  // one engine's part on the calling thread
  for (auto& t : th) t.join();
}
}  // namespace

static int router_multi_get(rsp_router* r, size_t n, const uint32_t* shard_id, const uint8_t* keys, const uint64_t* koff,
                            uint32_t klen_fixed, uint8_t* vals, size_t val_stride, uint32_t* vlen, int32_t* st) {
  if (n == 0) return RSP_OK;
  const Buckets b = bucket_by_engine(r, n, shard_id);
  for (uint32_t i : b.unknown) { st[i] = RSP_INVALID_ARGUMENT; vlen[i] = 0; }
  std::atomic<int> worst{RSP_OK};
  for_each_engine(b, [&](size_t k) {
    const std::vector<uint32_t>& ix = b.idx[k];
    const size_t m = ix.size();
    // gather this engine's keys, run, scatter
    std::vector<uint64_t> off;
    std::vector<uint8_t> kb;
    if (klen_fixed) {
      kb.resize(m * (size_t)klen_fixed + 16);
      for (size_t j = 0; j < m; j++) memcpy(&kb[j * (size_t)klen_fixed], keys + (size_t)ix[j] * klen_fixed, klen_fixed);
    } else {
      off.assign(m + 1, 0);
      for (size_t j = 0; j < m; j++) off[j + 1] = off[j] + (koff[ix[j] + 1] - koff[ix[j]]);
      kb.resize((size_t)off[m] + 16);
      for (size_t j = 0; j < m; j++) memcpy(&kb[off[j]], keys + koff[ix[j]], (size_t)(off[j + 1] - off[j]));
    }
    std::vector<uint8_t> v(m * val_stride + 1);
    std::vector<uint32_t> vl(m);
    std::vector<int32_t> s(m);
    const int rc = multi_get_any(r->engines[k], m, b.local[k].data(), kb.data(), klen_fixed ? nullptr : off.data(), klen_fixed,
                                 v.data(), val_stride, vl.data(), s.data());
    if (rc != RSP_OK) worst = rc;
    for (size_t j = 0; j < m; j++) {
      st[ix[j]] = rc == RSP_OK ? s[j] : rc;
      vlen[ix[j]] = vl[j];
      if (rc == RSP_OK && s[j] == RSP_OK && vl[j]) memcpy(vals + (size_t)ix[j] * val_stride, &v[j * val_stride], std::min<size_t>(vl[j], val_stride));
    }
  });
  return worst.load();
}
}  // extern "C++"

int rsp_router_multi_get(rsp_router* r, size_t n, const uint32_t* shard_id, const uint8_t* keys, const uint64_t* koff,
                         uint8_t* vals, size_t val_stride, uint32_t* vlen, int32_t* st) {
  try {
  if (!r || (n && (!shard_id || !koff || !vlen || !st))) return RSP_INVALID_ARGUMENT;
  return router_multi_get(r, n, shard_id, keys, koff, 0, vals, val_stride, vlen, st);
  } catch (...) { return abi_caught(); }
}
int rsp_router_multi_get_fixed(rsp_router* r, size_t n, const uint32_t* shard_id, const uint8_t* keys, uint32_t klen,
                               uint8_t* vals, size_t val_stride, uint32_t* vlen, int32_t* st) {
  try {
  if (!r || !klen || (n && (!shard_id || !keys || !vlen || !st))) return RSP_INVALID_ARGUMENT;
  return router_multi_get(r, n, shard_id, keys, nullptr, klen, vals, val_stride, vlen, st);
  } catch (...) { return abi_caught(); }
}

int rsp_router_apply_many(rsp_router* r, size_t n, const uint32_t* shard_id, const uint8_t* blob, const uint64_t* off,
                          const uint64_t* ts_ms, int32_t* st_out) {
  try {
  if (!r || (n && (!shard_id || !off))) return RSP_INVALID_ARGUMENT;
  if (n == 0) return RSP_OK;
  const Buckets b = bucket_by_engine(r, n, shard_id);
  if (st_out) for (uint32_t i : b.unknown) st_out[i] = RSP_INVALID_ARGUMENT;
  std::atomic<int> worst{b.unknown.empty() ? RSP_OK : RSP_INVALID_ARGUMENT};
  for_each_engine(b, [&](size_t k) {
    const std::vector<uint32_t>& ix = b.idx[k];
    const size_t m = ix.size();
    std::vector<uint64_t> off2(m + 1, 0), ts2(ts_ms ? m : 0);
    for (size_t j = 0; j < m; j++) off2[j + 1] = off2[j] + (off[ix[j] + 1] - off[ix[j]]);
    std::vector<uint8_t> bb((size_t)off2[m] + 16);
    for (size_t j = 0; j < m; j++) {
      memcpy(&bb[off2[j]], blob + off[ix[j]], (size_t)(off2[j + 1] - off2[j]));
      if (ts_ms) ts2[j] = ts_ms[ix[j]];
    }
    std::vector<int32_t> s(m, 0);
    const int rc = rsp_apply_many(r->engines[k], m, b.local[k].data(), bb.data(), off2.data(), ts_ms ? ts2.data() : nullptr, s.data());
    if (rc != RSP_OK) worst = rc;
    if (st_out) for (size_t j = 0; j < m; j++) st_out[ix[j]] = s[j] ? s[j] : (rc == RSP_INVALID_ARGUMENT ? rc : 0);
  });
  return worst.load();
  } catch (...) { return abi_caught(); }
}

int rsp_flush(rsp_shard* s) {
  try {
  if (!s) return RSP_INVALID_ARGUMENT;
  rsp_engine* e = s->eng;
  std::lock_guard<std::mutex> g(e->mu);
  if (ticks_in_flight(s)) return RSP_BUSY;
  CUDA_OK(cudaSetDevice(e->device));
  compact_shards(e, {s}, false);
  return RSP_OK;
  } catch (...) { return abi_caught(); }
}
int rsp_compact(rsp_shard* s) {
  try {
  if (!s) return RSP_INVALID_ARGUMENT;
  rsp_engine* e = s->eng;
  std::lock_guard<std::mutex> g(e->mu);
  if (ticks_in_flight(s)) return RSP_BUSY;
  CUDA_OK(cudaSetDevice(e->device));
  compact_shards(e, {s}, true);
  return RSP_OK;
  } catch (...) { return abi_caught(); }
}
static int all_shards(rsp_engine* e, bool full) {
  std::lock_guard<std::mutex> g(e->mu);
  CUDA_OK(cudaSetDevice(e->device));
  std::vector<rsp_shard*> v;
  for (rsp_shard* s : e->slots) if (s) v.push_back(s);
  for (rsp_shard* s : v) if (ticks_in_flight(s)) return RSP_BUSY;
  // bounded batches keep the work buffers modest: <= 256 shards and <= 8 GB of sources (a batch needs about half its
  // sources again for sort items / scratch, plus its outputs, before the sources are released)
  std::vector<rsp_shard*> part;
  u64 part_bytes = 0;
  auto run_part = [&] {
    if (!part.empty()) compact_shards(e, part, full);
    part.clear();
    part_bytes = 0;
  };
  for (rsp_shard* s : v) {
    u64 b = (u64)s->h.mt_tail * 16;
    for (auto& r : s->runs) b += r->bytes();
    if (!part.empty() && (part.size() >= 256 || part_bytes + b > (8ull << 30))) run_part();
    part.push_back(s);
    part_bytes += b;
  }
  run_part();
  return RSP_OK;
}
int rsp_flush_all(rsp_engine* e) {
  try {
    return e ? all_shards(e, false) : RSP_INVALID_ARGUMENT;
  } catch (...) { return abi_caught(); }
}
int rsp_compact_all(rsp_engine* e) {
  try {
    return e ? all_shards(e, true) : RSP_INVALID_ARGUMENT;
  } catch (...) { return abi_caught(); }
}

int rsp_get_stats(const rsp_shard* s, rsp_stats* out) {
  try {
  if (!s || !out) return RSP_INVALID_ARGUMENT;
  rsp_engine* e = s->eng;
  std::lock_guard<std::mutex> g(e->mu);
  *out = s->stats;
  out->latest_seq = s->last_seq.load();
  out->memtable_entries = s->h.mt_count;
  out->memtable_bytes = (u64)s->h.mt_tail * 16;
  out->n_runs = s->runs.size();
  out->run_entries = 0; out->run_bytes = 0;
  for (auto& r : s->runs) { out->run_entries += r->n_ent; out->run_bytes += r->bytes(); }
  return RSP_OK;
  } catch (...) { return abi_caught(); }
}

// ---- iterator ----
rsp_iter* rsp_iter_create(rsp_shard* s) {
  try {
  if (!s) return nullptr;
  rsp_engine* e = s->eng;
  std::lock_guard<std::mutex> g(e->mu);
  if (ticks_in_flight(s)) return nullptr;  // fold the pre-staged ticks first (rsp_apply_staged_finish)
  rsp_iter* it = new rsp_iter();
  it->s = s;
  CUDA_OK(cudaSetDevice(e->device));
  // The memtable is unordered: its contents are sorted into a PRIVATE run (the same kernels as a flush), which the
  // iterator pins in front of the shard's runs.  The shard itself is not touched: no new run, no compaction trigger,
  // writers go on filling the same memtable (RocksDB: an iterator pins the memtable and the current version).
  if (s->h.mt_count) {
    wait_readers(e);
    if (auto snap = snapshot_memtable(e, s)) it->pinned.push_back(snap);
  }
  it->pinned.insert(it->pinned.end(), s->runs.begin(), s->runs.end());
  if (it->pinned.size() > RSP_MAX_RUNS) {  // the view has room for RSP_MAX_RUNS runs: fold the memtable in after all
    it->pinned.clear();
    compact_shards(e, {s}, false);
    it->pinned = s->runs;
  }
  ScanView v;
  memset(&v, 0, sizeof(v));
  v.n_runs = (u32)it->pinned.size();
  v.merge_op = s->opts.merge_op;
  for (u32 i = 0; i < v.n_runs; i++) v.runs[i] = it->pinned[i]->dev();
  it->d_view = (ScanView*)e->arena.alloc(sizeof(ScanView));
  CUDA_OK(cudaMemcpyAsync(it->d_view, &v, sizeof(v), cudaMemcpyHostToDevice, e->st));
  CUDA_OK(cudaStreamSynchronize(e->st));
  return it;
  } catch (...) { abi_caught(); return nullptr; }
}
void rsp_iter_destroy(rsp_iter* it) {
  try {
  if (!it) return;
  rsp_engine* e = it->s->eng;
  {
    std::lock_guard<std::mutex> g(e->mu);
    CUDA_OK(cudaSetDevice(e->device));
    CUDA_OK(cudaStreamSynchronize(e->st));
    e->arena.release(it->d_view, sizeof(ScanView));
    it->pinned.clear();
  }
  delete it;
  } catch (...) { abi_caught(); }
}
void rsp_iter_seek_to_first(rsp_iter* it) {
  try {
    it->want = 16; iter_fetch(it, nullptr, false, false);
  } catch (...) { abi_caught(); it->valid = false; it->status = RSP_IO_ERROR; }
}
void rsp_iter_seek_to_last(rsp_iter* it) {
  try {
    it->want = 16; iter_fetch(it, nullptr, false, true);
  } catch (...) { abi_caught(); it->valid = false; it->status = RSP_IO_ERROR; }
}
void rsp_iter_seek(rsp_iter* it, const uint8_t* key, size_t klen) {
  try {
  std::string k((const char*)key, klen);
  it->want = 16;
  iter_fetch(it, &k, false, false);
  } catch (...) { abi_caught(); }
}
void rsp_iter_next(rsp_iter* it) {
  try {
  if (!it->valid) return;
  if (it->reverse) {  // direction change: refetch forward from the current key, exclusive
    std::string k = it->buf[it->pos].first;
    it->want = 16;
    iter_fetch(it, &k, true, false);
    return;
  }
  if (it->pos + 1 < it->buf.size()) { it->pos++; iter_landed(it); return; }
  if (it->exhausted) { it->valid = false; return; }
  std::string k = it->buf[it->pos].first;
  iter_fetch(it, &k, true, false);
  } catch (...) { abi_caught(); }
}
void rsp_iter_prev(rsp_iter* it) {
  try {
  if (!it->valid) return;
  if (!it->reverse) {
    std::string k = it->buf[it->pos].first;
    it->want = 16;
    iter_fetch(it, &k, true, true);
    return;
  }
  if (it->pos + 1 < it->buf.size()) { it->pos++; iter_landed(it); return; }
  if (it->exhausted) { it->valid = false; return; }
  std::string k = it->buf[it->pos].first;
  iter_fetch(it, &k, true, true);
  } catch (...) { abi_caught(); }
}
int rsp_iter_valid(const rsp_iter* it) { return it->valid ? 1 : 0; }
const uint8_t* rsp_iter_key(const rsp_iter* it, size_t* klen) {
  if (!it->valid) { if (klen) *klen = 0; return nullptr; }
  if (klen) *klen = it->buf[it->pos].first.size();
  return (const uint8_t*)it->buf[it->pos].first.data();
}
const uint8_t* rsp_iter_value(const rsp_iter* it, size_t* vlen) {
  if (!it->valid) { if (vlen) *vlen = 0; return nullptr; }
  if (vlen) *vlen = it->buf[it->pos].second.size();
  return (const uint8_t*)it->buf[it->pos].second.data();
}
int rsp_iter_status(const rsp_iter* it) { return it->status; }

// ---- batched scans (host buffers) ----
int rsp_multi_scan(rsp_engine* e, size_t n, const uint32_t* shard_ix, const uint8_t* keys, const uint64_t* koff,
                   uint32_t max_entries, uint8_t* out, size_t out_stride, uint32_t* n_out, int32_t* st) {
  try {
  if (!e || (n && (!shard_ix || !koff || !out || !n_out || !st))) return RSP_INVALID_ARGUMENT;
  std::lock_guard<std::mutex> g(e->mu);
  CUDA_OK(cudaSetDevice(e->device));
  if (n == 0) return RSP_OK;
  std::vector<rsp_shard*> fl;
  for (size_t i = 0; i < n; i++) {
    if (shard_ix[i] >= e->slots.size() || !e->slots[shard_ix[i]]) return RSP_INVALID_ARGUMENT;
    rsp_shard* s = e->slots[shard_ix[i]];
    if (ticks_in_flight(s)) return RSP_BUSY;
    if (s->h.mt_count && std::find(fl.begin(), fl.end(), s) == fl.end()) fl.push_back(s);
  }
  if (!fl.empty()) compact_shards(e, fl, false);
  const size_t key_bytes = (size_t)koff[n];
  const size_t o_koff = align_up(n * 4, 256), o_keys = o_koff + align_up((n + 1) * 8, 256);
  const size_t o_nout = o_keys + align_up(key_bytes + 16, 256), o_st = o_nout + align_up(n * 4, 256);
  const size_t o_out = o_st + align_up(n * 4, 256);
  u8* d = (u8*)e->dev_q.get(o_out + n * out_stride + 256);
  CUDA_OK(cudaMemcpyAsync(d, shard_ix, n * 4, cudaMemcpyHostToDevice, e->st));
  CUDA_OK(cudaMemcpyAsync(d + o_koff, koff, (n + 1) * 8, cudaMemcpyHostToDevice, e->st));
  if (key_bytes) CUDA_OK(cudaMemcpyAsync(d + o_keys, keys, key_bytes, cudaMemcpyHostToDevice, e->st));
  ScanArgs a;
  a.shards = e->d_shards; a.views = nullptr; a.shard_ix = (const u32*)d; a.keys = d + o_keys;
  a.koff = (const u64*)(d + o_koff); a.klen_fixed = 0; a.flags = nullptr; a.max_entries = max_entries;
  a.out = d + o_out; a.out_stride = out_stride; a.n_out = (u32*)(d + o_nout); a.st = (i32*)(d + o_st); a.n = (u32)n;
  a.max_shards = e->cfg.max_shards;
  CUDA_OK(cudaEventRecord(e->ev0, e->st));
  launch_multi_scan(a, e->st);
  e->launches++;
  CUDA_OK(cudaEventRecord(e->ev1, e->st));
  CUDA_OK(cudaMemcpyAsync(n_out, d + o_nout, n * 4, cudaMemcpyDeviceToHost, e->st));
  CUDA_OK(cudaMemcpyAsync(st, d + o_st, n * 4, cudaMemcpyDeviceToHost, e->st));
  CUDA_OK(cudaMemcpyAsync(out, d + o_out, n * out_stride, cudaMemcpyDeviceToHost, e->st));
  CUDA_OK(cudaStreamSynchronize(e->st));
  float ms = 0;
  cudaEventElapsedTime(&ms, e->ev0, e->ev1);
  e->last_ms["scan"] = ms;
  for (size_t i = 0; i < n; i++) {
    st[i] &= ~SCAN_ST_TRUNCATED;  // (n_out[i] < max_entries tells the caller that the scan stopped early)
    if (st[i] == ST_NEED_HOST_MERGE) st[i] = RSP_NOT_SUPPORTED;  // host-folded operators: use the iterator
    else if (st[i] > 255) {
      // a merge failed somewhere in this scan: its record reads as an empty value, the status is the scan's
      st[i] = st[i] >> 8;
      u8* r = out + i * out_stride;
      for (u32 k = 0; k < n_out[i]; k++) {
        u32 kl, vl;
        memcpy(&kl, r, 4);
        memcpy(&vl, r + 4, 4);
        if (vl == SCAN_VLEN_MERGE_FAILED) { vl = 0; memcpy(r + 4, &vl, 4); }
        r += 8 + kl + vl;
      }
    }
  }
  return RSP_OK;
  } catch (...) { return abi_caught(); }
}

// ---- device-pointer forms ----
int rsp_multi_get_device(rsp_engine* e, size_t n, const uint32_t* d_shard_ix, const uint8_t* d_keys, uint32_t klen,
                         uint8_t* d_vals, uint32_t val_stride, uint32_t* d_vlen, int32_t* d_st, void* stream) {
  try {
  if (!e || !klen) return RSP_INVALID_ARGUMENT;
  GetArgs a;
  a.shards = e->d_shards; a.fast = e->d_fast; a.shard_ix = d_shard_ix; a.keys = d_keys; a.koff = nullptr; a.klen_fixed = klen;
  a.vals = d_vals; a.val_stride = val_stride; a.vlen = d_vlen; a.st = d_st; a.n = (u32)n;
  {
    std::lock_guard<std::mutex> g(e->mu);  // the pending-list scratch is per engine
    cudaStream_t rs = stream ? (cudaStream_t)stream : e->st;
    set_pending(e, a, n, rs);
    a.max_shards = e->cfg.max_shards;
    reader_begin(e, rs);
    a.multirun = e->n_multirun.load() ? 1u : 0u;
    launch_multi_get(a, rs);
    reader_end(e, rs);
    pending_mark(e, rs);
  }
  e->launches += 2;
  return cudaPeekAtLastError() == cudaSuccess ? RSP_OK : RSP_IO_ERROR;
  } catch (...) { return abi_caught(); }
}

int rsp_multi_scan_device(rsp_engine* e, size_t n, const uint32_t* d_shard_ix, const uint8_t* d_keys, uint32_t klen,
                          uint32_t max_entries, uint8_t* d_out, uint64_t out_stride, uint32_t* d_n_out, int32_t* d_st,
                          void* stream) {
  try {
  if (!e || !klen) return RSP_INVALID_ARGUMENT;
  ScanArgs a;
  a.shards = e->d_shards; a.views = nullptr; a.shard_ix = d_shard_ix; a.keys = d_keys; a.koff = nullptr;
  a.klen_fixed = klen; a.flags = nullptr; a.max_entries = max_entries; a.out = d_out; a.out_stride = out_stride;
  a.n_out = d_n_out; a.st = d_st; a.n = (u32)n; a.max_shards = e->cfg.max_shards;
  {
    std::lock_guard<std::mutex> g(e->mu);
    cudaStream_t rs = stream ? (cudaStream_t)stream : e->st;
    reader_begin(e, rs);
    launch_multi_scan(a, rs);
    reader_end(e, rs);
  }
  e->launches++;
  return cudaPeekAtLastError() == cudaSuccess ? RSP_OK : RSP_IO_ERROR;
  } catch (...) { return abi_caught(); }
}

int rsp_stage_build(rsp_engine* e, size_t n, const uint32_t* shard_ix, const uint8_t* blob, const uint64_t* off,
                    const uint64_t* ts_ms, rsp_staged** out) {
  try {
  if (!e || !out || !n) return RSP_INVALID_ARGUMENT;
  std::lock_guard<std::mutex> g(e->mu);
  CUDA_OK(cudaSetDevice(e->device));
  rsp_staged* sg = new rsp_staged();
  int rc = stage_build(e, n, shard_ix, blob, off, ts_ms, sg, true);
  if (rc != RSP_OK) { delete sg; return rc; }
  *out = sg;
  return RSP_OK;
  } catch (...) { return abi_caught(); }
}
void rsp_stage_free(rsp_staged* sg) {
  if (!sg) return;
  if (sg->reserved) { std::lock_guard<std::mutex> g(sg->eng->mu); unreserve(sg); }
  if (sg->dev) { cudaSetDevice(sg->eng->device); cudaFree(sg->dev); }
  delete sg;
}
int rsp_reserve(rsp_engine* e, const rsp_staged* sg) {
  try {
  if (!e || !sg) return RSP_INVALID_ARGUMENT;
  std::lock_guard<std::mutex> g(e->mu);
  CUDA_OK(cudaSetDevice(e->device));
  // flushes / re-allocations run on the engine stream: wait only when there were any, so that a tick
  // launched on another stream is ordered after them
  const int r = reserve_for(e, sg);
  if (r < 0) return RSP_BUSY;  // fold the results of the ticks in flight (rsp_apply_staged_finish), then retry
  if (r > 0) CUDA_OK(cudaStreamSynchronize(e->st));
  return RSP_OK;
  } catch (...) { return abi_caught(); }
}
int rsp_apply_staged_device(rsp_engine* e, rsp_staged* sg, void* stream) {
  try {
  if (!e || !sg) return RSP_INVALID_ARGUMENT;
  sg->last_stream = stream ? (cudaStream_t)stream : e->st;
  cudaEventRecord(e->ev0, sg->last_stream);
  tick_launch(e, sg, sg->last_stream);
  cudaEventRecord(e->ev1, sg->last_stream);
  return cudaPeekAtLastError() == cudaSuccess ? RSP_OK : RSP_IO_ERROR;
  } catch (...) { return abi_caught(); }
}
int rsp_apply_staged_finish(rsp_engine* e, rsp_staged* sg, int32_t* st_out) {
  try {
  if (!e || !sg) return RSP_INVALID_ARGUMENT;
  std::lock_guard<std::mutex> g(e->mu);
  CUDA_OK(cudaSetDevice(e->device));
  u8* pout = (u8*)e->pin_out.get(sg->res_bytes);
  cudaStream_t st = sg->last_stream ? sg->last_stream : e->st;
  CUDA_OK(cudaMemcpyAsync(pout, sg->tick.gres, sg->res_bytes, cudaMemcpyDeviceToHost, st));
  CUDA_OK(cudaStreamSynchronize(st));
  float ms = 0;
  if (cudaEventElapsedTime(&ms, e->ev0, e->ev1) == cudaSuccess) e->last_ms["apply"] = ms;
  return tick_results(sg, pout, st_out);
  } catch (...) { return abi_caught(); }
}

float rsp_last_kernel_ms(const rsp_engine* e, const char* what) {
  try {
  rsp_engine* m = const_cast<rsp_engine*>(e);
  std::lock_guard<std::mutex> g(m->mu);
  auto it = m->last_ms.find(what);
  return it == m->last_ms.end() ? -1.f : it->second;
  } catch (...) { abi_caught(); return -1.f; }
}
uint64_t rsp_kernel_launches(const rsp_engine* e) { return e->launches.load(); }

void rsp_debug_arena(rsp_engine* e, uint64_t out[4]) {
  for (int i = 0; i < 4; i++) out[i] = 0;
  if (!e) return;
  std::lock_guard<std::mutex> g(e->arena.mu);
  out[0] = e->arena.in_use;       // bytes handed out (rounded to 256)
  out[1] = e->arena.reserved;     // bytes reserved from the device (slabs)
  out[2] = e->arena.blocks.size();  // blocks, free and used
  out[3] = e->arena.free_bytes;   // free inside the slabs
}

int rsp_debug_run(rsp_shard* s, uint32_t r, rsp_debug_run_info* info, uint8_t* heap, uint32_t* ent_off,
                  uint64_t* blk_pfx, uint32_t* hslots) {
  try {
  if (!s || !info) return RSP_INVALID_ARGUMENT;
  rsp_engine* e = s->eng;
  std::lock_guard<std::mutex> g(e->mu);
  if (r >= s->runs.size()) return RSP_NOT_FOUND;
  CUDA_OK(cudaSetDevice(e->device));
  static_assert(sizeof(rsp_debug_run_desc) == sizeof(RunDev) && sizeof(rsp_debug_fast_desc) == sizeof(ShardFast), "layout");
  const Run& run = *s->runs[r];
  // the buffers were sized from an earlier call: copy only into buffers sized for THIS run
  if ((heap || ent_off || blk_pfx || hslots) && info->host.heap != (uint64_t)run.heap) return RSP_BUSY;
  memset(info, 0, sizeof(*info));
  const RunDev hd = run.dev();
  memcpy(&info->host, &hd, sizeof(RunDev));
  info->n_runs = (u32)s->runs.size();
  const ShardDev* d = e->d_shards + s->index;
  CUDA_OK(cudaMemcpyAsync(&info->dev_n_runs, &d->n_runs, 4, cudaMemcpyDeviceToHost, e->st));
  CUDA_OK(cudaMemcpyAsync(&info->dev, &d->runs[r], sizeof(RunDev), cudaMemcpyDeviceToHost, e->st));
  CUDA_OK(cudaMemcpyAsync(&info->fast_run, e->d_fast_runs + (size_t)s->index * RSP_MAX_RUNS + r, sizeof(ShardFast),
                          cudaMemcpyDeviceToHost, e->st));
  if (r == 0) CUDA_OK(cudaMemcpyAsync(&info->fast, e->d_fast + s->index, sizeof(ShardFast), cudaMemcpyDeviceToHost, e->st));
  if (heap && run.heap_units) CUDA_OK(cudaMemcpyAsync(heap, run.heap, (size_t)run.heap_units * 16, cudaMemcpyDeviceToHost, e->st));
  if (ent_off && run.n_ent) CUDA_OK(cudaMemcpyAsync(ent_off, run.ent_off, (size_t)run.n_ent * 4, cudaMemcpyDeviceToHost, e->st));
  if (blk_pfx && run.n_blocks) CUDA_OK(cudaMemcpyAsync(blk_pfx, run.blk_pfx, (size_t)run.n_blocks * 8, cudaMemcpyDeviceToHost, e->st));
  if (hslots && run.n_buckets)
    CUDA_OK(cudaMemcpyAsync(hslots, run.hslots, (size_t)run.n_buckets * RUN_BUCKET_SLOTS * 4, cudaMemcpyDeviceToHost, e->st));
  CUDA_OK(cudaStreamSynchronize(e->st));
  return RSP_OK;
  } catch (...) { return abi_caught(); }
}

void rsp_debug_combiner_stats(rsp_engine* e, int which, uint64_t out[9]) {
  for (int i = 0; i < 9; i++) out[i] = 0;
  if (!e) return;
  if (which == 0) { if (ReadCombiner* c = e->read_comb_ready.load(std::memory_order_acquire)) c->stager->stats(out); }
  else if (ApplyCombiner* c = e->apply_comb_ready.load(std::memory_order_acquire)) {
    c->stager->stats(out);
    for (int k = 0; k < 3; k++) out[5 + k] = c->dbg_ns[k].load(std::memory_order_relaxed);
    out[8] = c->dbg_n.load(std::memory_order_relaxed);
  }
}

// diagnostics: how many lookups of the last MultiGet launch took the generic path (synchronises)
uint32_t rsp_debug_last_pending(rsp_engine* e, uint32_t* first, uint32_t cap) {
  try {
  std::lock_guard<std::mutex> g(e->mu);
  cudaSetDevice(e->device);
  cudaDeviceSynchronize();
  if (!e->dev_pending.p) return 0;
  u32 n = 0;
  cudaMemcpy(&n, (u32*)e->dev_pending.p + 2 + (e->mg_parity ^ 1u), 4, cudaMemcpyDeviceToHost);
  if (first && cap) cudaMemcpy(first, (u32*)e->dev_pending.p + 4, 4 * std::min(n, cap), cudaMemcpyDeviceToHost);
  return n;
  } catch (...) { abi_caught(); return 0; }
}

}  // extern "C"
