/*
 * evstore_b200 -- C-ABI of the B200-native EVStore embedding-lookup hot path.
 *
 * This header is the drop-in boundary.  It has two parts:
 *
 *  (1) the LEGACY entry points of the reference's libcachemanager.so
 *      (/root/reference/mixed_precs_caching/cache_manager.cpp), same names, same
 *      signatures, same "process-global cache + library-owned float buffer"
 *      contract, so cache_algo/cpp_socket_client.py:63-83 binds them unchanged;
 *
 *  (2) a runtime-configured, batched API that replaces the reference's
 *      compile-time #defines (cache_manager.cpp:13-20) and its one-sample-per-call
 *      limit.  Plain pointers and sizes only; no torch / C++ types.  Groups:
 *        evs_create / evs_destroy / evs_stats / evs_check ...          handle life cycle and bookkeeping
 *        evs_lookup_batch / _batches / _bags / _batch_host / evs_submit_host   the hot path (device or host buffers,
 *                                                                      one batch, a queue of batches, bags with pooling)
 *        evs_probe_batch / evs_probe_bags / evs_lookup_bags_agg        exact agg_hit over a collective transport
 *        evs_prefetch, evs_note_replays                                look-ahead; the lookup inside a caller's CUDA graph
 *        evs_update_rows                                               new row values, ordered between batches
 *        evs_state_bytes / evs_save_state / evs_load_state             snapshot of a warm cache's policy state, and restore
 *        evs_shard_*                                                   table-wise sharding over NVLink peer memory
 *        evs_embedding_bag, evs_interact, evs_knn                      the ops either side of the cache; alt-key generation
 *        evs_host_alloc / evs_host_free                                host memory for backing rows (large device pages)
 *
 * Conventions
 *  - table ids are 0-based here; the reference's keys are "<table+1>-<row>"
 *    (evlfu_32.cpp:477).  A key is (table << 40) | row in every key stream.
 *  - every call returns EVS_OK (0) or a negative evs_status; nothing calls exit()
 *    (the reference's error path is printf + exit(-1), cache_manager.cpp:213-217).
 *  - one handle == one stream-ordered, single-writer cache (the reference is
 *    not thread safe either: globals, no locks).
 *  - "dev" pointers are CUDA device pointers on cfg.device; "host" pointers are
 *    ordinary host memory (pinned memory makes the copies asynchronous).
 */
#ifndef EVSTORE_B200_H
#define EVSTORE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EVS_MAX_TABLES 32      /* keys of one sample are handled by one warp */
#define EVS_MAX_TIERS 2        /* C1 and C2 (C3 holds alternative keys, not rows) */

typedef enum {
    EVS_OK = 0,
    EVS_ERR_INVALID = -1,      /* bad argument / unsupported configuration */
    EVS_ERR_CUDA = -2,         /* a CUDA runtime call failed (see evs_last_error) */
    EVS_ERR_INDEX = -3,        /* an index was outside [0, rows[table]) */
    EVS_ERR_CAPACITY = -4,     /* internal structure overflow (should not happen) */
    EVS_ERR_NOT_CONFIGURED = -5,
    EVS_ERR_PEER = -6          /* table-wise sharding: a peer rank did not answer within 4 s */
} evs_status;

typedef struct evs_handle_s *evs_handle;
typedef struct evs_shard_s *evs_shard;

/* Replaces cache_manager.cpp:13-20 (N_CACHING_LAYER, MAIN_PRECISION,
 * SECONDARY_PRECISION, TOTAL_SIZE, SIZE_PROPORTION) plus the hard-coded
 * EV_DIMENSION / N_EV_TABLE (cache_manager.hpp:30-31) and file roots
 * (evlfu_32.hpp:61, evlfu_8.hpp:58, evlfu_4.hpp:61, aprx_embedding.hpp:39). */
typedef struct {
    int32_t device;              /* CUDA device ordinal */
    int32_t n_tables;            /* tables served by this cache (<= EVS_MAX_TABLES) */
    int32_t n_tables_total;      /* agg_hit range: buckets 0..n_tables_total (26 in the reference) */
    int32_t table_base;          /* global id of local table 0 (table-wise sharding), else 0 */
    int32_t dim;                 /* embedding dimension (reference: 36) */
    int32_t n_layers;            /* 1, 2 or 3  (N_CACHING_LAYER) */
    int32_t main_precision;      /* 32, 16, 8 or 4  (MAIN_PRECISION) */
    int32_t secondary_precision; /* 16, 8 or 4, lower than main (SECONDARY_PRECISION); 0 if n_layers == 1 */
    int64_t total_size;          /* TOTAL_SIZE, in fp32-row units */
    int32_t prop_c1, prop_c2, prop_c3; /* SIZE_PROPORTION "c1-c2-c3" in percent; all 0 = even split */
    int32_t max_batch;           /* largest B passed to evs_lookup_batch */
    int32_t approx_emb_thres;    /* EvLFU_C1.request_to_ev_lfu approx_emb_thres; <= 0 disables */
    int32_t high_agghit_threshold; /* evlfu_32.hpp:74; 0 = default 23 */
    float flush_rate;            /* 0 = default 0.3  (evlfu_32.hpp:53) */
    float perfect_item_cap;      /* 0 = default 0.95 (evlfu_32.hpp:54) */
    const int64_t *rows;         /* [n_tables] table cardinalities */
    /* Backing store (stands in for emb_storage/* and EVLFU_*::get_from_file): per table a
     * host pointer to rows*dim*precision/8 bytes, row-major, the layout of
     * binary/ev-table-N.bin (script/convert_ev_to_binary.py).  The library page-locks and
     * maps the memory (zero-copy); it must stay valid until evs_destroy. */
    const void *const *store_main;       /* [n_tables] rows at main_precision */
    const void *const *store_secondary;  /* [n_tables] rows at secondary_precision, or NULL */
    /* Alternative keys for C3 (aprx_embedding.cpp): per table a host pointer to rows uint32
     * alt_key = alt_row*100 + (alt_table+1), host byte order (the file is big-endian,
     * convert_altkeys_to_binary.py:35); NULL unless n_layers == 3. */
    const uint32_t *const *alt_keys;
    int32_t store_in_hbm;        /* testing aid: copy the backing store into HBM instead of mapping it */
    int32_t record_events;       /* keep per-batch eviction / flush key streams for evs_last_events */
    /* Replacement policy of the (single) tier: EVS_POLICY_EVLFU = the EvLFU of cache_algo/EvLFU_C1.py and
     * mixed_precs_caching/ (default, every layer count); EVS_POLICY_LRU = the comparison policy of
     * cache_algo/LRU.py:15-37 (n_layers == 1 only), selected in the reference by --cache-algo
     * (dlrm_s_pytorch_C1_C2_C3.py:249-254). */
    int32_t policy;
    /* Table placement (table-wise sharding): global id of each local table, [n_tables], strictly increasing, each
     * in [0, n_tables_total).  NULL = the contiguous slice table_base .. table_base + n_tables - 1 that
     * ext_dist.get_my_slice gives a rank (extend_distributed.py:47-51).  A non-contiguous placement (e.g. tables
     * balanced by rows) departs from the reference's split; keys, tier routing and the output column of a table
     * always follow its global id. */
    const int32_t *table_ids;
} evs_config;

#define EVS_POLICY_EVLFU 0
#define EVS_POLICY_LRU 1
#define EVS_POLICY_LFU 2   /* cache_algo/LFU.py: one FIFO list per frequency, saturating at n_tables_total + 1 (n_layers == 1 only) */

typedef struct {
    uint64_t lookups;            /* keys looked up */
    uint64_t samples;
    uint64_t hits[EVS_MAX_TIERS];       /* served from C1 / C2 */
    uint64_t c3_hits;            /* "C3 Indiv-Hit" (evlfu_8.cpp:539) */
    uint64_t approx_subst;       /* EvLFU_C1 approximate substitutions (EvLFU_C1.py:150) */
    uint64_t misses;             /* fetched from the backing store */
    uint64_t perfect_hits;       /* samples whose every key hit ("Perfect hit", cache_manager.cpp:288) */
    uint64_t inserts[EVS_MAX_TIERS];
    uint64_t evictions[EVS_MAX_TIERS];
    uint64_t flushed[EVS_MAX_TIERS];
    uint64_t size[EVS_MAX_TIERS];       /* resident entries now */
    uint64_t capacity[EVS_MAX_TIERS];
    uint64_t c3_size, c3_capacity;
    uint64_t batches;
} evs_stats_t;

/* ---- lifecycle ------------------------------------------------------------------ */
int evs_create(const evs_config *cfg, evs_handle *out);
int evs_destroy(evs_handle h);
const char *evs_last_error(void);       /* text of the last failure on this thread */
int evs_version(void);

/* ---- the hot path ---------------------------------------------------------------- *
 * One batch: probe -> EvLFU promote -> fetch misses -> insert/evict -> dequantise ->
 * fp32 rows.  Replaces B calls of ev_lookup (cache_manager.cpp:231) /
 * EvLFU_C1.request_to_ev_lfu (EvLFU_C1.py:97).
 *   idx_dev   int64 [n_tables][B]          (the reference's lS_i, table-major)
 *   out_dev   fp32  B rows of n_tables*dim, consecutive samples out_stride floats apart
 *             (out_stride 0 == n_tables*dim)
 *   hit_dev   uint8 [B][n_tables] or NULL  (aggHitMissRecord; 1 = answered from a cache tier)
 *   agg_in    uint8 [B] or NULL: externally supplied agg_hit per sample (exact
 *             groupability under table-wise sharding); NULL = count locally
 *   stream    cudaStream_t (NULL = the handle's own stream)
 * Asynchronous with respect to the host. */
int evs_lookup_batch(evs_handle h, const int64_t *idx_dev, int32_t B, float *out_dev, int64_t out_stride,
                     uint8_t *hit_dev, const uint8_t *agg_in, void *stream);

/* Bags on the cached path (pooling factor > 1): the (lS_o, lS_i) pairs of apply_emb (dlrm_s_pytorch_C1_C2_C3.py:191-223;
 * --data-generation=random draws up to 10 indices per bag, dlrm_data_pytorch.py:961-1007).
 *   idx_dev  int64 [nnz]          all bags' indices, table 0's bags first
 *   off_dev  int64 [n_tables*B+1] bag (t, s) = idx_dev[off[t*B+s] .. off[t*B+s+1]);  off[n_tables*B] = nnz
 *   max_per_bag  P <= 32, B*P <= max_batch; a larger bag, a negative index or malformed offsets raise EVS_ERR_INDEX
 *   out_dev  fp32 [B][n_tables][dim]: out[s][t] = sum over the bag's rows, j ascending, single fp32 adds (an empty bag
 *            gives zeros) -- nn.EmbeddingBag(mode="sum") over the rows the cache serves (dequantised at the serving tier)
 *   hit_dev  uint8 [nnz] hit code per index (as evs_lookup_batch), or NULL
 * Policy: the batch is looked up as B*P slices -- slice s*P+j = the j-th index of every table's bag of sample s -- each one
 * a request group in the reference's sense (its agg_hit counts the hits among its own keys). */
int evs_lookup_bags(evs_handle h, const int64_t *idx_dev, const int64_t *off_dev, int32_t B, int64_t nnz, int32_t max_per_bag,
                    float *out_dev, int64_t out_stride, uint8_t *hit_dev, void *stream);
/* Bags for a table-wise sharded cache over a collective transport (probe -> all-reduce of the slice counts -> lookup ->
 * all-to-all of the POOLED rows), the bags form of evs_probe_batch / evs_lookup_batch(agg_in):
 *   evs_probe_bags      agg_out_dev uint8 [B*P]: each slice's local hit count (absent positions count nothing); no state change
 *   evs_lookup_bags_agg agg_in uint8 [B*P]: each slice's agg_hit summed over the ranks; otherwise evs_lookup_bags
 * Same arguments, limits and refusals as evs_lookup_bags (P = max_per_bag). */
int evs_probe_bags(evs_handle h, const int64_t *idx_dev, const int64_t *off_dev, int32_t B, int64_t nnz, int32_t max_per_bag,
                   uint8_t *agg_out_dev, void *stream);
int evs_lookup_bags_agg(evs_handle h, const int64_t *idx_dev, const int64_t *off_dev, int32_t B, int64_t nnz, int32_t max_per_bag,
                        float *out_dev, int64_t out_stride, uint8_t *hit_dev, const uint8_t *agg_in, void *stream);

/* n consecutive batches of B samples in one call: exactly the results of n evs_lookup_batch calls in that order (the
 * batches stay strictly ordered on the device), but groups of 4 batches go to the device as ONE captured graph, so only
 * every fourth batch pays the graph-to-graph launch boundary, and the misses of batches 1..n-1 are staged by the
 * look-ahead (evs_prefetch) without further calls.  A serving loop whose requests are queued uses this; announce the
 * first batch of the next call with evs_prefetch.  idx_dev / out_dev / hit_dev: n pointers each (hit_dev or its entries
 * may be NULL); the output buffers may alias each other if the caller consumes only the last one. */
int evs_lookup_batches(evs_handle h, int32_t n, const int64_t *const *idx_dev, int32_t B, float *const *out_dev,
                       int64_t out_stride, uint8_t *const *hit_dev, void *stream);

/* Capturing evs_lookup_batch into the CALLER's CUDA graph (e.g. a whole sequential_forward, dlrm_s_pytorch_C1_C2_C3.py:742-768):
 * when `stream` is being captured the batch is recorded as plain kernels with its arguments frozen (same index / output
 * buffers on every replay: refill them before each launch); the device numbers the replays itself.  After launching the
 * captured graph n times call evs_note_replays(h, n, stream) -- it keeps the host's batch count and the ring bookkeeping
 * in step (and returns a pending index / peer error).  Replays and direct calls may be mixed. */
int evs_note_replays(evs_handle h, int64_t n, void *stream);

/* Look-ahead: idx_dev is the index batch the NEXT evs_lookup_batch / evs_shard_lookup call on this handle will pass
 * (same pointer, same B).  The library probes it and stages the rows of its probable misses from the host-pinned
 * backing store into HBM on its own stream, under the kernels of the batch in flight; the next call then finds
 * its missing rows staged instead of waiting for the PCIe reads (the longest part of a step).  Pure data movement:
 * every hit / eviction decision is still taken by the next call itself, results are identical with and without.
 *   ready_event  cudaEvent_t recorded after idx_dev was written, or NULL if the indices are already complete
 * Optional; a call that was not announced (or whose announcement does not match) runs as before. */
int evs_prefetch(evs_handle h, const int64_t *idx_dev, int32_t B, void *ready_event);

/* Refreshing a model in service: new fp32 values for the rows of n keys, written into the backing store at every
 * precision the handle has (store_main / store_secondary: the caller's host arrays through the device mapping, or the HBM
 * copy with store_in_hbm) and into every cached copy (the C1 / C2 slab row of a resident key).
 *   keys_dev    int64 [n] in the library's key format, (global table << 40) | row (as evs_dump_state returns them)
 *   values_dev  fp32 rows of dim floats, value_stride floats apart (0 = dim)
 *   where_dev   uint8 [n] or NULL: bit 0 = the C1 copy was refreshed, bit 1 = the C2 copy, bit 2 = the backing store was
 *               written; 0x80 = rejected, nothing written.  A key is rejected when its row is outside [0, rows[table]) or
 *               its table is not served by this handle (this also raises the sticky EVS_ERR_INDEX of evs_check), or when a
 *               quantised precision of the handle cannot hold one of its values: non-finite at 16 / 8 / 4 bits, outside
 *               [-1, 1] at 8 bits, a 16-bit code outside [0, 65535] (|v| above about 6).  At 32 bits every bit pattern is
 *               stored as given.  A key given several times takes the row of its LAST occurrence, whole; the earlier
 *               occurrences write nothing and report 0 (the last one is still rejected on its own values).
 * Stream-ordered: lookups enqueued on `stream` before the call see the old rows, lookups after it the new ones, whichever
 * way a row is served (C1 / C2 / C3 / approximate substitution / miss / look-ahead, bags, evs_store_ptr readers).  The
 * call changes no policy state (hit codes, buckets, eviction order, C3, statistics are what they would be without it);
 * it cancels a pending evs_prefetch announcement, so the next batch fetches its misses itself.  Asynchronous; not
 * allowed while `stream` is being captured (EVS_ERR_INVALID).  n == 0 is a no-op. */
int evs_update_rows(evs_handle h, const int64_t *keys_dev, int64_t n, const float *values_dev, int64_t value_stride,
                    uint8_t *where_dev, void *stream);

/* ---- snapshots of the policy state: keep a warm cache across a restart ------------------------------- *
 * A snapshot holds a handle's policy state with KEYS ONLY: per tier (C1, C2) its resident keys bucket by bucket in
 * eviction (FIFO) order and n_perfect; for C3 the raw FIFO window, stale and duplicate records included, and the map
 * entries (key, alt key, recency flag).  Rows are re-read from the loading handle's backing store at its own
 * precisions, so a snapshot survives evs_update_rows and loads into a handle whose tiers use other precisions.
 * Guarantee: handle A saves after some batches, handle B loads the snapshot; given the same batches from then on, A and
 * B return bit-identical rows, hit codes and agg_hit, the same evs_last_events streams, evs_dump_state / evs_dump_c3
 * and statistics deltas, for every policy and lookup path.  Slot assignments may differ; nothing observable depends
 * on them.  Loading replaces the whole state (B may have served traffic).
 * The loading handle must match policy, n_layers, n_tables_total, the served global table ids and rows[]; each tier's
 * key count and C3's size must fit its capacities, and C3's window must leave room in its ring for one batch's
 * appends (2 * max_batch * n_tables records).  dim, precisions, max_batch, larger
 * capacities, store_in_hbm and the device may differ.
 *
 * Blob, little-endian: a 464-byte header
 *     char magic[8] "EVSSTATE"; u32 version (1); u32 header bytes (464); u64 total bytes;
 *     i32 policy, n_layers, n_tables_total, n_tables; i32 dim, main_precision, secondary_precision, n_buckets;
 *     u64 cap[2], c3_cap; i32 table_ids[32] (-1 past n_tables); i64 rows[32] (0 past n_tables)
 *     (dim, precisions and capacities are informational), then u64 words:
 *     per tier (1 or 2):  n_perfect; count[n_buckets]; the keys, (global table << 40) | row, bucket 0 first, each
 *                         bucket oldest first
 *     C3 (three layers):  size; W; the W window records, oldest first; size map entries (key, alt | flag << 32)
 *
 * evs_state_bytes: an upper bound of a snapshot's size, from the capacities (no synchronisation).
 * evs_save_state: writes the snapshot into buf (host memory of any kind, cap bytes) and its size into *bytes
 *   (EVS_ERR_INVALID with *bytes set when cap is too small).  Reflects every batch enqueued on `stream` before it.
 * evs_load_state: replaces the handle's state with the snapshot; every batch enqueued on `stream` after it sees it.
 *   It cancels a pending evs_prefetch announcement and leaves the cumulative statistics alone.  The header and
 *   every count are checked on the host first: a mismatch returns EVS_ERR_INVALID with the reason in evs_last_error and
 *   the handle untouched.  The device then checks each key (table served, row in range, at most once per tier, C3 map
 *   keys unique); a key that fails returns EVS_ERR_INVALID and leaves the handle EMPTY, as after evs_create.
 * Both are stream-ordered, synchronise before returning, and are refused while `stream` is being captured. */
int evs_state_bytes(evs_handle h, uint64_t *bound);
int evs_save_state(evs_handle h, void *buf, uint64_t cap, uint64_t *bytes, void *stream);
int evs_load_state(evs_handle h, const void *buf, uint64_t bytes, void *stream);

/* Probe only: per-sample local hit counts (for the sharded exact mode the ranks
 * all-reduce these and pass the sum back as agg_in).  Does not change state. */
int evs_probe_batch(evs_handle h, const int64_t *idx_dev, int32_t B, uint8_t *agg_out_dev, void *stream);

/* Same batch through host buffers: H2D of idx, the hot path, D2H of out (and hit),
 * then a stream synchronise.  This is what a reference-side caller (ctypes / cgo) uses. */
int evs_lookup_batch_host(evs_handle h, const int64_t *idx_host, int32_t B, float *out_host, uint8_t *hit_host);

/* Pipelined variant of the same: returns at once with a ticket, at most 4 batches in flight (the
 * call blocks on the oldest when all staging slots are taken).  H2D of the next batch and D2H of
 * the previous one overlap the kernels of the current one; batches stay strictly ordered.  The
 * host buffers must stay valid (and should be page-locked) until evs_wait_host(ticket) returns. */
int evs_submit_host(evs_handle h, const int64_t *idx_host, int32_t B, float *out_host, uint8_t *hit_host, int64_t *ticket);
int evs_wait_host(evs_handle h, int64_t ticket);

int evs_sync(evs_handle h);
int evs_stats(evs_handle h, evs_stats_t *out, int reset);
/* Cheap error poll (no synchronisation, no device round trip): the kernels mirror their error word into pinned
 * host memory.  Returns EVS_OK, or the sticky EVS_ERR_INDEX / EVS_ERR_PEER of a batch that has already run;
 * evs_wait_host and evs_lookup_batch_host call it after their synchronisation.  clear != 0 resets it. */
int evs_check(evs_handle h, int clear);
/* Device memory the handle holds (index, slabs, rings, staging), in bytes: the slab is slot-indexed at a load
 * factor <= 1/3, so this is a multiple of TOTAL_SIZE * row bytes (the reference's budget, cache_manager.cpp:16). */
int evs_memory_footprint(evs_handle h, uint64_t *hbm_bytes);

/* ---- measurement ------------------------------------------------------------------- *
 * Every kernel launch of a handle is counted.  With profiling on, each launch is also bracketed
 * by CUDA events on its launching stream; evs_kernel_times synchronises and returns, per kernel
 * name, the summed device time, the number of timed launches and the number of launches.
 * *n in: capacity of the arrays, out: number of kernel kinds. */
int evs_set_profiling(evs_handle h, int enable);
int evs_kernel_times(evs_handle h, int32_t *n, const char **names, double *total_ms, uint64_t *timed,
                     uint64_t *launches, int reset);
uint64_t evs_launch_count(evs_handle h);
/* %globaltimer stamps (ns) of the LAST batch: [0] k_serve start, [7] k_serve end (last CTA),
 * [2] k_update start, [3] all CTAs done (claims, appends, miss fetch), [4] ring tails advanced,
 * [5] evictions done, [6] C3 done.  Synchronises. */
int evs_phase_times(evs_handle h, uint64_t *ns8);   /* ns8: 32 entries */

/* ---- parity / introspection (used by tests; cheap, off the hot path) -------------- */
/* Keys evicted / flushed by the LAST batch of tier (0 = C1, 1 = C2), in eviction order.
 * Needs cfg.record_events.  *n_* in: capacity of the arrays, out: count. */
int evs_last_events(evs_handle h, int tier, int64_t *evicted, int64_t *n_evicted, int64_t *flushed,
                    int64_t *n_flushed);
/* Resident keys of a tier in eviction order: bucket_off[b]..bucket_off[b+1] index keys of
 * agg_hit bucket b (FIFO).  keys capacity in *n_keys (in) -> count (out); bucket_off has
 * n_tables_total+2 entries. */
int evs_dump_state(evs_handle h, int tier, int64_t *keys, int64_t *n_keys, int64_t *bucket_off,
                   int64_t *n_perfect);
/* Resident keys of C3 in FIFO order with their alt keys and recency flags. */
int evs_dump_c3(evs_handle h, int64_t *keys, uint32_t *alt, uint8_t *recency, int64_t *n);

/* ---- feature interaction (dlrm_s_pytorch_C1_C2_C3.py:625-658, "dot") ---------------- *
 *   x_dev  fp32 [B][dim]        bottom-MLP output
 *   ly_dev fp32 [B][n_f][dim]   pooled embeddings (evs_lookup_batch output)
 *   r_dev  fp32 [B][dim + (n_f+1)*n_f/2]   (arch_interaction_itself = 0)
 * Pairs are fp32-accurate (DESIGN.md section 4); a NaN or +-Inf input makes every pair of its row NaN or non-finite.
 * EVS_ERR_INVALID when one sample's (n_f+1) x (dim+1) floats exceed the device's shared memory per block (only for
 * n_f + 1 > 32 or dim > 128).
 */
int evs_interact(const float *x_dev, const float *ly_dev, float *r_dev, int32_t B, int32_t n_f, int32_t dim,
                 void *stream);

/* ---- table-wise sharding over NVLink peer memory ------------------------------------------- *
 * The embedding part of DLRM_Net.distributed_forward (dlrm_s_pytorch.py:544-570): rank r owns the tables
 * get_my_slice(n_tables_total) (extend_distributed.py:47-62; build its handle with table_base / n_tables_total),
 * looks the WHOLE global batch up in them, and the pooled rows [B, T_local*d] must end up batch-sharded,
 * [B/world, n_tables_total*d] (ext_dist.alltoall, extend_distributed.py:541-576; all_to_all_single :414).
 * Here the exchange is part of the kernels: every rank exports one block of device memory over CUDA IPC
 * (evs_shard_export, 64 bytes, exchanged by the caller), maps its peers' blocks (evs_shard_connect), and
 *   - the probe kernel stores each sample's local hit count into every peer's count table, so that agg_hit is the
 *     exact sum over all tables (the reference never ran its cache sharded; agg_hit is its only cross-table coupling);
 *   - the gather and miss-fetch kernels store every fp32 row straight into the receive buffer of the rank that owns the
 *     sample, already in the [B/world][n_tables_total][dim] layout;
 *   - epoch words in peer memory order the two phases (no host synchronisation, no NCCL call).
 * evs_shard_lookup: idx_dev int64 [n_tables][B] for the whole global batch B (a multiple of world); *out_dev receives
 * this rank's [B/world][n_tables_total][dim] fp32 buffer, valid until four batches later (four alternate).  hit_dev as in
 * evs_lookup_batch.  Every rank must make the same sequence of calls. */
int evs_shard_create(evs_handle h, int32_t rank, int32_t world, int32_t batch_max, evs_shard *out);
int evs_shard_export(evs_shard s, void *handle64);
int evs_shard_connect(evs_shard s, const void *handles /* world x 64 bytes, rank order */);
int evs_shard_lookup(evs_shard s, const int64_t *idx_dev, int32_t B, uint8_t *hit_dev, float **out_dev, void *stream);
/* n consecutive global batches in one call: what n evs_shard_lookup calls deliver, but groups of 4 batches reach the device
 * as one captured graph on every rank (every rank must make the same calls).  out_dev[i] receives this rank's buffer of
 * batch i; the buffers rotate through 4, so each stays valid until four batches later. */
int evs_shard_lookup_many(evs_shard s, int32_t n, const int64_t *const *idx_dev, int32_t B, uint8_t *const *hit_dev,
                          float **out_dev, void *stream);
/* Bags on a rank of a sharded cache: a sharded bag batch gives exactly what evs_lookup_bags gives on one GPU with every
 * table, agg_hit summed over the ranks.  idx_dev / off_dev: the evs_lookup_bags layout for THIS rank's tables over the
 * whole global batch B (a multiple of world).  Every rank expands its bags into B*P slices (slice s*P+j = the j-th index
 * of each bag of sample s; P = max_per_bag <= 32, B*P <= batch_max); a slice's agg_hit is the sum over the ranks of the hits
 * among its present keys, and each rank runs the policy on its slices.  The rank pools its tables locally (j ascending,
 * single fp32 adds from +0.0; an empty bag gives zeros) and stores only the pooled rows into the owner ranks' receive
 * buffers: *out_dev receives this rank's [B/world][n_tables_total][dim] buffer, each table at the column of its global
 * id, valid until four batches later.  hit_dev uint8 [nnz] per index as evs_lookup_bags, or NULL.  Malformed offsets or a
 * bag larger than P raise the sticky EVS_ERR_INDEX.  One batch per call (no grouping, no look-ahead); plain and bag
 * batches share the epoch sequence and the receive buffers and may be mixed freely.  Every rank makes the same calls. */
int evs_shard_lookup_bags(evs_shard s, const int64_t *idx_dev, const int64_t *off_dev, int32_t B, int64_t nnz, int32_t max_per_bag,
                          uint8_t *hit_dev, float **out_dev, void *stream);
int evs_shard_destroy(evs_shard s);

/* ---- sum pooling: nn.EmbeddingBag(mode="sum") of apply_emb_ori_dlrm ------------------- *
 * (dlrm_s_pytorch_C1_C2_C3.py:191-223)   out[b] = sum_{j = off[b] .. off[b+1]-1} w[j] * W[idx[j]], j ascending.
 *   table_dev  device-visible rows of ONE table, rows*dim*precision/8 bytes, the binary/ev-table-N.bin
 *              layout at 32 / 16 / 8 / 4 bits (HBM, or mapped pinned host memory: evs_store_ptr)
 *   idx_dev    int64 [nnz], off_dev int64 [B] (bag b ends where bag b+1 starts, the last at nnz)
 *   per_sample_weights fp32 [nnz] or NULL; out_dev fp32 [B] rows of dim, out_stride floats apart (0 = dim)
 * Out-of-range indices read row 0 and make evs_embedding_bag_status() (synchronising) return EVS_ERR_INDEX. */
int evs_embedding_bag(const void *table_dev, int64_t rows, int32_t dim, int32_t precision, const int64_t *idx_dev,
                      const int64_t *off_dev, int64_t nnz, int32_t B, const float *per_sample_weights, float *out_dev,
                      int64_t out_stride, void *stream);
int evs_embedding_bag_status(void);
/* Device-visible alias of the handle's backing rows of (tier, table): the storage_manager no-cache
 * path (request_to_emb_storage, emb_storage/storage_manager.py:125) reads it with evs_embedding_bag. */
int evs_store_ptr(evs_handle h, int tier, int table, const void **dev_ptr, int32_t *precision);

/* ---- alt-key generation for C3 (script/approximate_embedding/phase2_similarity_analysis/) ---------- *
 * get_neighbors_GPU.ipynb: every embedding row of every table in one matrix, brute-force Euclidean k-NN (n_neighbors = 11,
 * entry [0] -- the row itself -- dropped); most_popular_neighbor.ipynb: of those k = 10 the one with the highest workload
 * frequency (first maximum, absent = 0) becomes the row's alternative key, alt_row * 100 + alt_table (tables 1-based,
 * convert_altkeys_to_binary.py:50).  One fused tensor-core kernel (distances by 3xTF32 mma.sync: fp32-accurate) + a merge.
 *   x_dev  fp32 [n][dim] the database (n < 2^31, dim <= 64);  q_dev fp32 [nq][dim] the query rows (may point into x_dev)
 *   nbr_dev int64 [nq][k] global row ids, nearest first (ties by index), -1 where the database has fewer rows; or NULL
 *   dist_dev fp32 [nq][k] squared distances (non-finite where nbr is -1), or NULL
 *   A database row with a NaN or +-Inf element, or whose squared norm overflows fp32, is never a neighbour or an alt key;
 *   a query row with a NaN or +-Inf element gets -1 everywhere, non-finite distances and alt key 0.
 *   alt_dev uint32 [nq] alt keys, or NULL; then table_off_dev int64 [n_tables + 1] = first global row of each table and
 *           freq_dev uint32 [n] request counts per global row (or NULL: every neighbour counts 0, the nearest wins) */
int evs_knn(const float *x_dev, int64_t n, const float *q_dev, int64_t nq, int32_t dim, int32_t k, int64_t *nbr_dev,
            float *dist_dev, const uint32_t *freq_dev, const int64_t *table_off_dev, int32_t n_tables, uint32_t *alt_dev,
            void *stream);

/* ---- host memory for the backing rows (get_from_file's ev-table-N.bin contents, evlfu_32.cpp:283-316) --- *
 * Any host array works as a backing store (pinned allocations are used as they are, pageable ones are
 * page-locked by evs_create).  Memory from evs_host_alloc is additionally mapped into `device` with large
 * pages: the zero-copy miss fetch over a multi-GB table runs at about twice the row rate (managed memory
 * that lives in host memory and is never migrated; the host reads / writes / fread()s into it as usual).
 * Free with evs_host_free after every handle created over it has been destroyed. */
int evs_host_alloc(void **ptr, uint64_t bytes, int32_t device);
int evs_host_free(void *ptr);

/* ---- legacy libcachemanager.so surface (cache_manager.cpp) ------------------------ *
 * A process-global cache answers one sample per call.  Where the reference fixes its
 * configuration at compile time, call evs_legacy_configure once first (or set
 * EVSTORE_B200_LEGACY=... and let the Python shim do it); ev_lookup before that
 * prints an error and returns NULL instead of exiting. */
int evs_legacy_configure(const evs_config *cfg);
evs_handle evs_legacy_handle(void);
float *ev_lookup(int *arr);                    /* cache_manager.cpp:231 */
float *get_ev_values(int *arr);                /* cache_manager.cpp:257 */
void print_perfect_hit(void);                  /* cache_manager.cpp:262 (prints, then resets) */
void test_arr(int *arr);                       /* cache_manager.cpp:154 */
int ev_lookup_based_on_list_keys(int *arr);    /* cache_manager.cpp:239 (deprecated there; returns -1 here) */

#ifdef __cplusplus
}
#endif
#endif /* EVSTORE_B200_H */
