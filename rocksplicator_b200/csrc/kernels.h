// kernels.h — launch wrappers of the engine's CUDA kernels (implemented in k_*.cu).
#pragma once
#include "format.cuh"

namespace rsp {

// ---- apply tick image (device) -------------------------------------------------------------------
struct BatchDesc {
  u32 shard_ix;
  u32 boff;    // byte offset of the batch in the tick blob
  u32 len;     // bytes, including the appended LogData(timestamp) record when present
  u32 op_base; // first reserved slot in the op table
  u32 op_cap;  // reserved slots (min(header count, (len-12)/2))
  u32 group;
  u32 raw_len; // bytes physically present in the blob; [raw_len, len) is the VIRTUAL LogData record
               // {0x03, 0x08, timestamp LE} (packed ticks: nobody copies the batch to append it)
  u32 pad1;
};
struct GroupDesc {
  u32 shard_ix;
  u32 first_batch;
  u32 n_batches;
  u32 pad;
};
struct BatchRes {
  u32 status;    // k_decode: mk_status(code,msg) or 0; k_sequence: final status
  u32 n_ops;
  u32 units;
  u32 unit_base; // k_sequence
  u64 seq_base;  // k_sequence: sequence of the first op
  u32 ord_base;  // k_sequence: insertion ordinal of the first op
  u32 accepted;  // k_sequence
};
struct GroupRes {
  u64 last_seq;
  u32 tail;
  u32 count;
  u32 latch;
  u32 pad;
};
struct __align__(16) OpRec {
  u32 koff, klen;  // key bytes in the blob
  u32 voff, vlen;  // value bytes in the blob
  u32 rel_units;   // entry offset (units) relative to the batch's unit_base
  u32 type;        // kTypeValue / kTypeDeletion / kTypeSingleDeletion / kTypeMerge / kTypeInvalid
  u32 batch_ix;
  u32 op_ix;       // index within the batch (sequence = seq_base + op_ix)
};

struct TickDev {
  const u8* blob;
  const u64* ts;   // packed ticks: timestamp of batch i (virtual trailer); nullptr when the trailer is in the blob
  const BatchDesc* batches;
  const GroupDesc* groups;
  BatchRes* bres;
  GroupRes* gres;
  u32* bstat;     // final status word of each batch (k_sequence): what the host reads back
  OpRec* ops;
  u32 n_batches;
  u32 n_groups;
  u32 n_ops_cap;
};

// packed tick: descriptors are derived on the device from the caller's own arrays (no host re-layout)
struct PrepareArgs {
  const u8* blob;       // the caller's blob as given
  const u64* off;       // [n+1]
  const u64* ts;        // [n] or nullptr
  const GroupDesc* groups;
  u32 n_groups;
  u32 n_batches;
  BatchDesc* batches;   // out
  u32* need;            // out [2 * n_groups]: upper bounds (heap units, entries) per group
  u32* total_ops;       // out [1]
};
void launch_prepare(const PrepareArgs& a, cudaStream_t s);

// the whole tick in one launch (ticks of small batches): batch i of group g is blob[off[i] .. off[i] + len[i]) (len ==
// nullptr: the batches are contiguous, length off[i+1] - off[i]); ts != nullptr: the follower's LogData(timestamp)
// record is a virtual suffix of every batch
// one chunk of a group (cut by the host): <= FUSED_CHUNK_BATCHES consecutive batches, <= FUSED_STAGE_BYTES of blob
struct ChunkDesc {
  u32 group;
  u32 first_batch;     // staged position of the chunk's first batch
  u32 n_batches;
  u32 index_in_group;  // the chunks of a group are consecutive
  u32 shard_ix;        // (the group's, so that a chunk's CTA reaches its shard with one dependent load less)
  u32 group_chunks;    // chunks of its group
  u32 pad0, pad1;
};
constexpr u32 FUSED_CHUNK_BATCHES = 128;
constexpr u32 FUSED_STAGE_BYTES = 16384;
struct FusedTick {
  const u8* blob;
  const u64* off;
  const u32* len;
  const u64* ts;
  const GroupDesc* groups;
  u32* bstat;     // [n_batches] final status word
  GroupRes* gres; // [n_groups]
  u32 n_groups;
  u32 n_batches;
  u32 max_group;  // batches of the longest group and bytes of the longest batch: pick the kernel (64 threads /
  u32 max_len;    // 8 KB stage, a CTA per group, when no group holds more than 64 batches and no batch more than 4 KB)
  // otherwise k_tick_chunks, a CTA per chunk:
  const ChunkDesc* chunks;
  u64* chain;        // [n_chunks][4]: the group's sequencing state after each chunk (zeroed before the launch)
  u32* group_done;   // [n_groups]: chunks of the group that have finished (zeroed before the launch)
  u32 n_chunks;
  u32 pad;
};
inline bool fused_small_shape(u32 max_group, u32 max_len) { return max_group <= 64 && max_len <= 4096; }
constexpr u32 FUSED_MAX_BATCH_BYTES = 16384;  // larger batches take the general kernels (one thread walks a batch here)
void launch_tick_fused(const FusedTick& t, ShardDev* shards, ShardFast* fast, u32* mt_filter, cudaStream_t s);
void launch_decode(const TickDev& t, cudaStream_t s);
void launch_sequence(const TickDev& t, ShardDev* shards, ShardFast* fast, cudaStream_t s);
void launch_insert(const TickDev& t, ShardDev* shards, u32* mt_filter, cudaStream_t s);
void launch_publish(const TickDev& t, ShardDev* shards, cudaStream_t s);

// ---- reads ---------------------------------------------------------------------------------------
struct GetArgs {
  const ShardDev* shards;
  const ShardFast* fast;   // compact per-shard descriptors for the 16-byte-key kernel (may be nullptr)
  const u32* shard_ix;   // [n]
  const u8* keys;        // key bytes
  const u64* koff;       // [n+1] or nullptr when klen_fixed > 0
  u32 klen_fixed;
  u8* vals;              // value i at vals + i * val_stride
  u64 val_stride;
  u32* vlen;             // [n]
  i32* st;               // [n]
  u32 n;
  u32* pending;          // [n] scratch: queries deferred by the fast kernel (may be nullptr)
  u32* n_pending;        // [2] counters (launch parity)
  u32 parity;
  u32* n_special;        // [1] counts lookups whose status is none of OK / NotFound / Incomplete (may be nullptr)
  u32 max_shards;        // shard ids >= this answer InvalidArgument
  u32 multirun;          // some live shard has more than one run: k_multi_get16m walks the runs newest first; the per-run
                         // descriptors ([max_shards][RSP_MAX_RUNS]) follow the ShardFast array in the same allocation.
                         // (The struct keeps its r01 size and field offsets: growing it by eight bytes changes the
                         // register allocation of k_multi_get16 and costs it 20 % — profiles/r02_regression_bisect.md)
};
static_assert(sizeof(GetArgs) == 128, "GetArgs layout is part of k_multi_get16's measured code generation");
void launch_multi_get(const GetArgs& a, cudaStream_t s);

// dump the version stack of each key (newest first, up to and including the first Put/Delete) for
// host-side merge folding: records [u32 type][u32 vlen][value, padded to 4] at out + i*stride
struct ScanView;
struct VersionsArgs {
  const ShardDev* shards;
  const ScanView* views;   // when set: one pinned view per query (runs only), shards/shard_ix unused
  const u32* shard_ix;
  const u8* keys;
  const u64* koff;
  u8* out;
  u64 out_stride;
  u32* n_rec;   // [n] records written
  u32* need;    // [n] bytes needed
  u32 n;
};
void launch_get_versions(const VersionsArgs& a, cudaStream_t s);

// range scan over a pinned set of runs (the memtable is flushed first by the host)
struct ScanView {
  RunDev runs[RSP_MAX_RUNS];
  u32 n_runs;
  u32 merge_op;
  u32 pad0, pad1;
};
// vlen markers in scan records (the value is absent: the record is [u32 klen][u32 marker][key])
constexpr u32 SCAN_VLEN_HOST_FOLD = 0xffffffffu;     // the merge operator lives on the host: fold this key there
constexpr u32 SCAN_VLEN_MERGE_FAILED = 0xfffffffeu;  // the merge failed: empty value, the scan's st holds the status
// scan status word: 0, 7 (Incomplete: the output stride was too small for max_entries), ST_NEED_HOST_MERGE, or
// mk_status(code, msg) of a failed merge; the last two carry SCAN_ST_TRUNCATED when the scan ALSO ran out of room
constexpr i32 SCAN_ST_TRUNCATED = 1 << 30;
struct ScanArgs {
  const ShardDev* shards;   // used when views == nullptr (shard_ix indexes it)
  const ScanView* views;    // or explicit pinned views (one per request)
  const u32* shard_ix;
  const u8* keys;
  const u64* koff;
  u32 klen_fixed;
  const u8* flags;          // per request: bit0 = exclusive start, bit1 = reverse, bit2 = from extreme
  u32 max_entries;
  u8* out;
  u64 out_stride;
  u32* n_out;
  i32* st;
  u32 n;
  u32 max_shards;           // with `shards`: ids >= this (and closed shards) answer InvalidArgument
};
void launch_multi_scan(const ScanArgs& a, cudaStream_t s);

// ---- flush / compaction ---------------------------------------------------------------------------
struct SortItem {
  u64 prefix;   // big-endian first 8 key bytes
  u32 ref;      // unit offset of the entry in its source heap
  u32 srcrank;  // src << 28 | rank : ascending == newest first among equal keys
};
struct CompactJob {
  // sources: src 0 = memtable (optional), 1.. = runs newest first
  const u8* src_heap[RSP_MAX_RUNS + 1];
  const u32* src_ent_off[RSP_MAX_RUNS + 1];
  u32 src_n[RSP_MAX_RUNS + 1];
  u32 src_is_mem[RSP_MAX_RUNS + 1];
  u32 n_src;
  u32 n_items;      // sum of src_n
  u32 n_pow2;       // sort size of the memtable segment (0 when there is none): only the memtable needs sorting
  u32 bottom;       // 1 = no older data below the output: tombstones can be dropped
  u32 merge_op;
  u32 items_len;    // length of items[]: n_pow2 (memtable segment, padded) + the runs' entries
  u32 seg_start[RSP_MAX_RUNS + 1];  // first item of each source's segment in items[]
  u32 n_tiles;      // merge tiles of MERGE_TILE items (n_src > 1)
  u32 pad;
  // work buffers
  SortItem* items;  // [items_len]: one sorted segment per source (the runs are sorted as stored)
  SortItem* items2; // [n_items]: the segments merged (n_src > 1)
  u32* coranks;     // [(n_tiles + 1) * n_src]: how many items of each segment precede each tile boundary
  const SortItem* sorted;  // what the sizing / writing passes read: items (one source) or items2
  u32* keep_units;  // [n_items] output size in units of each sorted item (0 = dropped)
  u32* out_pos;     // [n_items] exclusive scan of keep_units
  u32* out_ord;     // [n_items] exclusive scan of (keep_units != 0)
  u64* fold_val;    // [n_items] folded 8-byte merge results
  u32* totals;      // [8]: units, entries, uniform_units (or 0), distinct keys, non-Put entries, min/max klen<<16|vlen..
  // outputs (allocated by the host after the sizing pass)
  u8* out_heap;
  u32* out_ent_off;
  u32* out_hslots;
  u64* out_blk_pfx;
  u32 out_n_buckets;
  u32 out_ord_bits;
};
constexpr u32 MERGE_TILE = 2048;
// fill the per-source item segments, sort the memtable segment, merge the segments (merge path: co-ranks per tile
// boundary, then one CTA per tile)
void launch_compact_sort(const CompactJob* d_jobs, const CompactJob* h_jobs, u32 n_jobs, cudaStream_t s);
void launch_compact_size(const CompactJob* d_jobs, u32 n_jobs, cudaStream_t s);
void launch_compact_write(const CompactJob* d_jobs, u32 n_jobs, u32 max_items, cudaStream_t s);
// zero the hash index of every job's output run (out_hslots, out_n_buckets buckets): one launch for the whole batch
void launch_set_run_seq(u8* heap, const u32* ent_off, u32 n, u64 seq, cudaStream_t s);
void launch_zero_out_hslots(const CompactJob* d_jobs, u32 n_jobs, u32 max_buckets, cudaStream_t s);

// ---- batched descriptor upload ------------------------------------------------------------------------
// One record per shard whose descriptors changed (a flush / merge batch installs up to thousands at once): staged in
// pinned memory, ONE copy, ONE launch that scatters them — instead of three small pageable copies and a memset per shard.
struct ShardUpload {
  u32 index;
  u32 runs_only;  // 1: only the run set changed — the sequencing state (last_seq .. latch) stays the device's
  u32 zero_mt;    // 1: clear the memtable's slot table (the memtable was flushed)
  u32 pad;
  ShardDev sd;
  ShardFast fast;
  ShardFast fast_runs[RSP_MAX_RUNS];
};
static_assert(sizeof(ShardUpload) % 32 == 0, "records are copied as words from an array");
void launch_upload_shards(const ShardUpload* d_up, u32 n, ShardDev* shards, ShardFast* fast, ShardFast* fast_runs, u32* mt_filter,
                          cudaStream_t s);

}  // namespace rsp
