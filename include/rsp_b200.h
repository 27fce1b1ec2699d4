/*
 * rsp_b200.h — the C ABI of librsp_b200.so: the drop-in boundary of the B200 engine.
 *
 * Everything the reference's hot path asks of RocksDB goes through these entry points; the C++
 * mirror of the reference interfaces (rocksplicator_b200/host/: rocksdb:: shim, replicator::DbWrapper
 * implementation, RocksDBReplicator, admin::ApplicationDB) and the Python binding are thin layers
 * above it.  Plain pointers and sizes only; no CUDA, torch or C++ types cross this line; nothing
 * throws across it.
 *
 * Return values are rocksdb::Status::Code numbers (the codes the reference surfaces through
 * rocksdb::Status at rocksdb_admin/application_db.cpp:85-136 and maps to bool at
 * rocksdb_replicator/rocksdb_wrapper.cpp:22-27).
 *
 * Threading: every function is thread-safe (rocksdb_replicator/rocksdb_replicator.h:80-82).  Applies
 * to ONE shard are ordered by call order (the pull loop is serial per shard,
 * rocksdb_replicator/replicated_db.cpp:369-383, 430); reads issued after an apply returned observe it.
 */
#ifndef RSP_B200_H_
#define RSP_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RSP_ABI_VERSION 1

/* rocksdb::Status::Code */
enum rsp_status {
  RSP_OK = 0,
  RSP_NOT_FOUND = 1,
  RSP_CORRUPTION = 2,
  RSP_NOT_SUPPORTED = 3,
  RSP_INVALID_ARGUMENT = 4,
  RSP_IO_ERROR = 5,
  RSP_MERGE_IN_PROGRESS = 6,
  RSP_INCOMPLETE = 7, /* output buffer too small: *vlen holds the size needed */
  RSP_SHUTDOWN = 8,
  RSP_TIMED_OUT = 9,
  RSP_ABORTED = 10,
  RSP_BUSY = 11
};

/* merge operators that run on the device; anything else is folded on the host through a callback */
enum rsp_merge_op {
  RSP_MERGE_NONE = 0,      /* Merge records are stored; reads answer InvalidArgument as RocksDB does */
  RSP_MERGE_COUNTER = 1,   /* examples/counter_service/merge_operator.cpp:23-45 (int64 LE add) */
  RSP_MERGE_UINT64ADD = 2, /* RocksDB built-in "uint64add" (malformed operand == 0) */
  RSP_MERGE_APPEND = 3,    /* rocksdb_replicator/tests/rocksdb_assumption_test.cpp:58-77 (host fold) */
  RSP_MERGE_CALLBACK = 4   /* rsp_shard_opts.merge_fn (host fold) */
};

typedef struct rsp_engine rsp_engine; /* one per GPU */
typedef struct rsp_shard rsp_shard;   /* one per DB ("segment%05d", common/segment_utils.cpp:26-29) */
typedef struct rsp_iter rsp_iter;

/* AssociativeMergeOperator::Merge (examples/counter_service/merge_operator.h): existing may be NULL.
 * Write the result with out_set(out_ctx, bytes, len) and return 1; return 0 for failure. */
typedef int (*rsp_merge_fn)(void* state, const uint8_t* key, size_t klen, const uint8_t* existing,
                            size_t elen, const uint8_t* operand, size_t olen,
                            void (*out_set)(void* out_ctx, const uint8_t* bytes, size_t len),
                            void* out_ctx);

typedef struct rsp_engine_cfg {
  uint32_t abi_version;      /* RSP_ABI_VERSION */
  uint32_t max_shards;       /* shard-table capacity on the device (default 16384) */
  uint64_t arena_bytes;      /* device arena slab size (default 1 GiB; grows by slabs) */
  uint64_t staging_bytes;    /* reserved (pinned staging grows on demand) */
  uint32_t l0_compaction_trigger; /* runs per shard before a merge (rocksdb_options.cpp:82; default 4) */
  uint32_t reserved;
} rsp_engine_cfg;

typedef struct rsp_shard_opts {
  uint32_t merge_op;          /* enum rsp_merge_op */
  uint32_t reserved;
  uint64_t write_buffer_bytes; /* memtable entry-heap capacity (options.write_buffer_size); 0 = 1 MiB */
  rsp_merge_fn merge_fn;       /* RSP_MERGE_CALLBACK */
  void* merge_state;
} rsp_shard_opts;

typedef struct rsp_stats {
  uint64_t latest_seq;
  uint64_t memtable_entries, memtable_bytes;
  uint64_t n_runs, run_entries, run_bytes;
  uint64_t flushes, compactions;
  uint64_t compaction_bytes_read, compaction_bytes_written;
  uint64_t flush_comparison_sorts; /* flushes whose memtable took the comparison sort (distinct keys sharing their first
                                    * 8 bytes, or a memtable beyond the radix sort's shared-memory budget) */
} rsp_stats;

/* ---- engine / shard lifecycle -----------------------------------------------------------------
 * replaces rocksdb::DB::Open + RocksDBReplicator::addDB's wrapping of the DB
 * (rocksdb_admin/admin_handler.cpp:640, rocksdb_replicator/rocksdb_replicator.cpp:96-133). */
int rsp_engine_create(int device, const rsp_engine_cfg* cfg, rsp_engine** out);
void rsp_engine_destroy(rsp_engine* e);
int rsp_engine_device(const rsp_engine* e);
/* the engine's CUDA stream (cudaStream_t as void*): lets a caller order its own work / events with it */
void* rsp_engine_stream(const rsp_engine* e);
int rsp_shard_open(rsp_engine* e, const char* name, const rsp_shard_opts* opts, rsp_shard** out);
int rsp_shard_close(rsp_shard* s); /* frees the shard's HBM (removeDB + DB close); the caller drains its own calls on
                                     * the shard first, as RocksDBReplicator::removeDB does (rocksdb_replicator.cpp:143-151) */
uint32_t rsp_shard_index(const rsp_shard* s); /* index used by the batched calls below */
const char* rsp_shard_name(const rsp_shard* s);

/* ---- apply path --------------------------------------------------------------------------------
 * rsp_apply  == RocksDbWrapper::HandleReplicateResponse (rocksdb_replicator/rocksdb_wrapper.cpp:13-28):
 *               WriteBatch(bytes) -> PutLogData(&ts_ms, 8) -> DB::Write(default WriteOptions).
 * rsp_write  == RocksDbWrapper::WriteToLeader (rocksdb_wrapper.cpp:5-8): DB::Write of the batch as is.
 * On success *seq_out (optional) is DB::GetLatestSequenceNumber() after the write.  A failed write
 * leaves the shard unchanged and LATCHES the error for later writes, as RocksDB 5.x does.
 * Concurrent callers share device ticks (the apply combiner, see rsp_apply_updates). */
int rsp_apply(rsp_shard* s, const uint8_t* batch, size_t len, uint64_t ts_ms, uint64_t* seq_out);
int rsp_write(rsp_shard* s, const uint8_t* batch, size_t len, uint64_t* seq_out);

/* The batching front-end: n updates for any mix of shards in one device tick (what the >=16
 * replicator executor threads of rocksdb_replicator.cpp:58-67 call concurrently, one call here).
 * Batch i is blob[off[i] .. off[i+1]); batches of the same shard apply in index order.
 * ts_ms == NULL means rsp_write semantics (no LogData append).  st_out[i] gets each batch's status. */
int rsp_apply_many(rsp_engine* e, size_t n, const uint32_t* shard_ix, const uint8_t* blob,
                   const uint64_t* off, const uint64_t* ts_ms, int32_t* st_out);

/* The pull loop's unit of work: the <= replicator_max_updates_per_response updates of ONE ReplicateResponse, applied in
 * order (rocksdb_replicator/replicated_db.cpp:369-383 calls HandleReplicateResponse once per update; here the whole
 * response is one call).  batches[i] has the layout of rocksdb::Slice / folly::IOBuf's contiguous bytes; ts_ms[i] is
 * update i's timestamp (NULL = rsp_write semantics: nothing appended).  The bytes are copied before the call returns.
 * Calls from many threads (one per shard's response) share device ticks: each caller copies its updates into the open
 * tick's pinned staging buffer in parallel, a dispatcher thread runs one tick after the other (stager.h).
 *   done == NULL : blocks until the tick has run; returns the first failing update's status (RSP_OK when all were
 *                  applied) and, through *n_applied, how many leading updates were applied.
 *   done != NULL : returns RSP_OK at once; done(ctx, status, n_applied, latest_seq) runs on an engine-owned completion
 *                  thread after the tick (the follower then issues its next pull, replicated_db.cpp:430). */
typedef struct rsp_slice { const uint8_t* data; size_t size; } rsp_slice;
typedef void (*rsp_done_fn)(void* ctx, int status, size_t n_applied, uint64_t latest_seq);
int rsp_apply_updates(rsp_shard* s, size_t n, const rsp_slice* batches, const uint64_t* ts_ms, rsp_done_fn done,
                      void* ctx, size_t* n_applied);

/* RocksDbWrapper::LatestSequenceNumber (rocksdb_wrapper.cpp:4) */
uint64_t rsp_latest_seq(const rsp_shard* s);
/* Restore from a backup (rocksdb_admin/admin_handler.cpp:768-860 restoreDBHelper): after the saved contents have been
 * ingested, the shard continues at the sequence number the backup was taken at, so that it resumes pulling from its
 * upstream where the backed-up replica stood.  Only forwards; InvalidArgument otherwise. */
int rsp_set_latest_seq(rsp_shard* s, uint64_t seq);
/* text of the last non-OK status on this shard ("Corruption: bad WriteBatch Put" ...) */
size_t rsp_last_error(const rsp_shard* s, char* buf, size_t cap);

/* ---- read path ---------------------------------------------------------------------------------
 * rsp_get == ApplicationDB::Get (rocksdb_admin/application_db.cpp:85-111).
 * RSP_INCOMPLETE when cap is too small (*vlen = needed). */
int rsp_get(rsp_shard* s, const uint8_t* key, size_t klen, uint8_t* val, size_t cap, size_t* vlen);

/* rsp_multi_get == ApplicationDB::MultiGet (application_db.cpp:113-120), across shards.
 * Key i is keys[koff[i] .. koff[i+1]); value i is written at vals + i*val_stride (at most val_stride
 * bytes; st[i] = RSP_INCOMPLETE and vlen[i] = needed size when it does not fit). */
int rsp_multi_get(rsp_engine* e, size_t n, const uint32_t* shard_ix, const uint8_t* keys,
                  const uint64_t* koff, uint8_t* vals, size_t val_stride, uint32_t* vlen,
                  int32_t* st);

/* ApplicationDB::MultiGet as the reference calls it: one shard, an array of rocksdb::Slice keys, results delivered one
 * by one (fn(ctx, i, status, value, vlen) on the calling thread, straight from the pinned result buffer: the caller
 * assigns its std::string from there, no intermediate copy).  value_hint = expected largest value (0 = unknown); larger
 * values are fetched in a second pass.  Concurrent callers (and rsp_get / rsp_multi_get callers) share launches. */
typedef void (*rsp_value_fn)(void* ctx, size_t i, int status, const uint8_t* value, size_t vlen);
int rsp_multi_get_slices(rsp_shard* s, size_t n, const rsp_slice* keys, size_t value_hint, rsp_value_fn fn, void* ctx);

/* Fixed-key-length form with host buffers (pinned or pageable): keys[i*klen .. +klen). */
int rsp_multi_get_fixed(rsp_engine* e, size_t n, const uint32_t* shard_ix, const uint8_t* keys,
                        uint32_t klen, uint8_t* vals, size_t val_stride, uint32_t* vlen, int32_t* st);

/* ---- one process, several GPUs: the router --------------------------------------------------------------------
 * Shards partition shard_id -> GPU (one engine per device, no collective: nothing is exchanged between shards).  The
 * reference's router hashes a key to its shard and fans a request out to the hosts that own the shards
 * (examples/counter_service/counter_router.cpp:36-66); inside one box the same fan-out goes to the engines: a
 * cross-shard batch is bucketed by engine on the host (order within a shard preserved), every engine runs its part
 * concurrently on its own device, and the results are scattered back to the caller's order.
 * Shards are addressed by the id they were registered under (rsp_router_add_shard; e.g. the segment number). */
typedef struct rsp_router rsp_router;
int rsp_router_create(size_t n_engines, rsp_engine* const* engines, rsp_router** out);
void rsp_router_destroy(rsp_router* r); /* the engines and shards stay open */
int rsp_router_add_shard(rsp_router* r, uint32_t shard_id, rsp_shard* s);
int rsp_router_remove_shard(rsp_router* r, uint32_t shard_id);
/* rsp_multi_get / rsp_multi_get_fixed / rsp_apply_many with router shard ids; an unknown id answers InvalidArgument */
int rsp_router_multi_get(rsp_router* r, size_t n, const uint32_t* shard_id, const uint8_t* keys, const uint64_t* koff,
                         uint8_t* vals, size_t val_stride, uint32_t* vlen, int32_t* st);
int rsp_router_multi_get_fixed(rsp_router* r, size_t n, const uint32_t* shard_id, const uint8_t* keys, uint32_t klen,
                               uint8_t* vals, size_t val_stride, uint32_t* vlen, int32_t* st);
int rsp_router_apply_many(rsp_router* r, size_t n, const uint32_t* shard_id, const uint8_t* blob, const uint64_t* off,
                          const uint64_t* ts_ms, int32_t* st_out);

/* ---- iterator: ApplicationDB::NewIterator (application_db.cpp:78-83) + rocksdb::Iterator ------- */
rsp_iter* rsp_iter_create(rsp_shard* s);
void rsp_iter_destroy(rsp_iter* it);
void rsp_iter_seek_to_first(rsp_iter* it);
void rsp_iter_seek_to_last(rsp_iter* it);
void rsp_iter_seek(rsp_iter* it, const uint8_t* key, size_t klen);
void rsp_iter_next(rsp_iter* it);
void rsp_iter_prev(rsp_iter* it);
int rsp_iter_valid(const rsp_iter* it);
const uint8_t* rsp_iter_key(const rsp_iter* it, size_t* klen);
const uint8_t* rsp_iter_value(const rsp_iter* it, size_t* vlen);
int rsp_iter_status(const rsp_iter* it);

/* Batched range scans (BASELINE config 4: Seek + 128 x Next).  Memtables of the shards involved are flushed first
 * (the device form below scans the sorted runs only: call rsp_flush_all before it if memtables are not empty).  Scan i starts at the first key >=
 * start key i and returns up to max_entries live entries in key order.  Output i is a sequence of
 * [u32 klen][u32 vlen][key][value] records at out + i*out_stride; n_out[i] = entries written;
 * st[i] = RSP_INCOMPLETE when out_stride was too small for max_entries (n_out[i] entries are valid); a key whose
 * merge fails is returned with an empty value and st[i] = the failure (what DBIter does).  In the device form such a
 * record carries vlen = 0xfffffffe (and no value bytes), a key that needs a host-side merge operator 0xffffffff, and a
 * status other than 0 / RSP_INCOMPLETE has bit 30 set when the scan also ran out of room. */
int rsp_multi_scan(rsp_engine* e, size_t n, const uint32_t* shard_ix, const uint8_t* keys,
                   const uint64_t* koff, uint32_t max_entries, uint8_t* out, size_t out_stride,
                   uint32_t* n_out, int32_t* st);

/* ---- maintenance: DB::Flush / ApplicationDB::CompactRange(nullptr, nullptr)
 * (application_db.cpp:138-144; triggers admin_handler.cpp:1846,2174) -------------------------------- */
int rsp_flush(rsp_shard* s);
int rsp_compact(rsp_shard* s);
int rsp_flush_all(rsp_engine* e);
int rsp_compact_all(rsp_engine* e);
int rsp_get_stats(const rsp_shard* s, rsp_stats* out);

/* ---- bulk load: DB::IngestExternalFile for n sorted Puts (rocksdb_admin/admin_handler.cpp:1820-1845) -----------
 * Key i is keys[koff[i] .. koff[i+1]) (strictly increasing), value i vals[voff[i] .. voff[i+1]).  The keys become one
 * new sorted run.  Sequence numbers follow rocksdb_replicator/tests/rocksdb_assumption_test.cpp:248-283: unchanged when
 * the key range does not intersect existing data, +1 (the file's global sequence number) when it does — refused with
 * InvalidArgument unless allow_global_seqno.  host/sst/sst_format.h turns an SST file into these arrays. */
int rsp_ingest_sorted(rsp_shard* s, size_t n, const uint8_t* keys, const uint64_t* koff, const uint8_t* vals,
                      const uint64_t* voff, int allow_global_seqno, uint64_t* seq_out);

/* ---- device-pointer forms (kernel-level measurement; inputs/outputs already in HBM) -------------
 * `stream` is a cudaStream_t passed as void* (0 = the engine's own read stream).  No host
 * synchronisation is performed; the caller owns ordering and timing.  A lookup that needs a host-side merge operator
 * (RSP_MERGE_CALLBACK shards with merge operands on the key) cannot be finished on the device: its d_st is 100 and the
 * caller resolves it with rsp_get / rsp_multi_get. */
int rsp_multi_get_device(rsp_engine* e, size_t n, const uint32_t* d_shard_ix, const uint8_t* d_keys,
                         uint32_t klen, uint8_t* d_vals, uint32_t val_stride, uint32_t* d_vlen,
                         int32_t* d_st, void* stream);
/* The raw form of rsp_multi_scan: d_st / the vlen markers as described there, untranslated.  A scan whose shard id is
 * >= max_shards or names a shard that is not open answers d_st = RSP_INVALID_ARGUMENT, d_n_out = 0 and writes no output
 * bytes (as rsp_multi_get_device answers such lookups); the other scans of the launch are unaffected. */
int rsp_multi_scan_device(rsp_engine* e, size_t n, const uint32_t* d_shard_ix, const uint8_t* d_keys,
                          uint32_t klen, uint32_t max_entries, uint8_t* d_out, uint64_t out_stride,
                          uint32_t* d_n_out, int32_t* d_st, void* stream);
/* One apply tick from a pre-staged device image (see rsp_stage_*): decode + sequence + insert.
 * Memtable capacity must have been reserved with rsp_reserve. */
typedef struct rsp_staged rsp_staged;
int rsp_stage_build(rsp_engine* e, size_t n, const uint32_t* shard_ix, const uint8_t* blob,
                    const uint64_t* off, const uint64_t* ts_ms, rsp_staged** out); /* H2D once */
void rsp_stage_free(rsp_staged* st);
/* Reserve memtable room for the tick (flushing / re-sizing as needed).  Several ticks may be reserved and launched back to
 * back before their results are folded (rsp_apply_staged_finish, in launch order): each reservation counts the earlier
 * ones.  RSP_BUSY: a shard is full while earlier ticks are in flight — finish those, then reserve again. */
int rsp_reserve(rsp_engine* e, const rsp_staged* st);
int rsp_apply_staged_device(rsp_engine* e, rsp_staged* st, void* stream); /* kernels only */
int rsp_apply_staged_finish(rsp_engine* e, rsp_staged* st, int32_t* st_out); /* D2H + host seq update */

/* device timing helper: elapsed ms of the engine's last kernel group named `what`
 * ("multi_get", "apply", "scan", "flush", "compact"), measured with CUDA events on its own stream */
float rsp_last_kernel_ms(const rsp_engine* e, const char* what);
/* number of engine kernels launched so far (bench.py's gpu_launches) */
uint64_t rsp_kernel_launches(const rsp_engine* e);

/* diagnostics: lookups of the last MultiGet launch that left the fast kernel for the generic path */
uint32_t rsp_debug_last_pending(rsp_engine* e, uint32_t* first, uint32_t cap);

/* diagnostics: the staging combiners' counters — which = 0 reads, 1 applies; out = {batches run, items carried,
 * ns inside the device batches, ns waiting for callers still copying, ns idle, and for the asynchronous applies
 * (rsp_apply_updates): ns from the call to its batch having run, ns until a completion thread picked the callback
 * up, ns inside the callbacks, number of callbacks}; zeros before first use */
void rsp_debug_combiner_stats(rsp_engine* e, int which, uint64_t out[9]);

/* diagnostics: the device arena — out = {bytes handed out, bytes reserved from the device (slabs), number of blocks,
 * bytes free inside the slabs} */
void rsp_debug_arena(rsp_engine* e, uint64_t out[4]);

/* diagnostics, not part of the product path: read back run r of a shard (0 = newest) as flush and compaction built it,
 * for tests that check a run's structure entry by entry.  Synchronises the engine stream; changes no state.
 * info gets the engine's descriptor of the run (host), the descriptor the readers use (ShardDev.runs[r] and
 * ShardDev.n_runs, copied back from the device), the run's row of the per-run fast descriptors and, for r == 0, the
 * shard's fast descriptor (zero otherwise).  A run is identified by host.heap, its heap's device address.  With all of
 * heap, ent_off, blk_pfx and hslots NULL only info is filled (the sizes).  Otherwise *info must hold what an earlier
 * call returned for this run, and the non-NULL buffers receive a copy of heap (host.heap_units x 16 bytes), ent_off
 * (host.n_ent x 4), blk_pfx (host.n_blocks x 8) and hslots (host.n_buckets x 32); RSP_BUSY and nothing copied when run
 * r has been replaced since (a background merge).  RSP_NOT_FOUND when the shard has no run r. */
typedef struct rsp_debug_run_desc { /* RunDev (format.cuh) */
  uint64_t heap, ent_off, hslots, blk_pfx; /* device addresses */
  uint32_t n_ent, n_buckets, ord_bits, uniform_units, n_blocks, heap_units, flags, kv_len;
} rsp_debug_run_desc;
typedef struct rsp_debug_fast_desc { /* ShardFast (format.cuh) */
  uint64_t run0_heap, run0_hslots;
  uint32_t n_buckets, meta, mt_count, merge_op;
} rsp_debug_fast_desc;
typedef struct rsp_debug_run_info {
  uint32_t n_runs;     /* runs of the shard (host) */
  uint32_t dev_n_runs; /* ShardDev.n_runs on the device */
  rsp_debug_run_desc host, dev;
  rsp_debug_fast_desc fast_run; /* the per-run fast descriptor of run r on the device */
  rsp_debug_fast_desc fast;     /* r == 0: the shard's ShardFast on the device */
} rsp_debug_run_info;
int rsp_debug_run(rsp_shard* s, uint32_t r, rsp_debug_run_info* info, uint8_t* heap, uint32_t* ent_off,
                  uint64_t* blk_pfx, uint32_t* hslots);

const char* rsp_version(void);

#ifdef __cplusplus
}
#endif
#endif /* RSP_B200_H_ */
