// Device-side data layout of the EvLFU cache tiers (C1, C2) and the alternative-key map (C3).
//
// What the reference keeps in std::unordered_map<string, Cache_data> vals_C1 plus
// vector<unordered_set<string>> lists_C1 (evlfu_32.hpp:47-49) is, per tier, in HBM:
//
//   slots[]   open-addressing index (linear probing), 16 B per slot {kw, meta}
//             kw   = pass << 48 | key   (key 48 bits, all ones = empty).  pass counts the resident
//                    keys whose probe path crosses the slot, so a probe stops at the first slot
//                    nobody crosses and deletions need no tombstones; one 128-bit load answers
//                    "is it my key / may I stop / which bucket".
//             meta = (bucket+1) << 56 | position of the entry's live record in its bucket ring;
//                    0 on an occupied slot = claimed by the batch in flight, not in a bucket yet
//   slab[]    the rows themselves, indexed BY SLOT (row_stride bytes each, precision dependent):
//             no row indirection and no free list -- claiming a slot is one CAS
//   ring[b][] per agg_hit bucket b a FIFO log of slot ids (lists_C1[b]); a record is live iff
//             slots[slot].meta still points at it, so promotion / eviction never edit a log
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace evs {

constexpr int kMaxTables = 32;
constexpr int kMaxBuckets = 32;              // agg_hit 0..n_tables_total (<= 31)
constexpr int kMaxTiers = 2;
// append sequences: group 0 = C1 (promotions and inserts interleaved in position order, as the
// reference's C1 loop does, evlfu_8.cpp:629-652), group 1 = C2 promotions, group 2 = C2 inserts
// (phase_2 updates every hit before it inserts any miss, evlfu_8.cpp:416-442)
constexpr int kSeqGroups = 3;
constexpr int kSeqs = kSeqGroups * kMaxBuckets;
constexpr int kTierCtas = 192;               // CTAs of k_evict per tier
constexpr int kEvictWindow = 256;            // ring records per eviction chunk (one per thread)
constexpr int kSamplesPerCta = 8;            // warps per serve / update CTA (one sample per warp when T > 16)
constexpr int kLookupThreads = kSamplesPerCta * 32;
constexpr int kKeyShift = 40;
constexpr unsigned long long kKeyMask = 0x0000FFFFFFFFFFFFull;
constexpr unsigned long long kEmptyKey = kKeyMask;           // 48 one bits
constexpr unsigned long long kPassOne = 1ull << 48;
constexpr unsigned kNoSlot = 0xFFFFFFFFu;
constexpr unsigned kClaimedBit = 0x80000000u;     // pos_slot: this position claimed the slot (it fills the slab row)

// flags[p]: 0 = nothing to do; bits 0-5 = bucket+1 of the append this position asks for;
// bit 6 = tier of the append; bit 7 = the position missed: claim a slot and fetch the row
constexpr uint8_t kFlagMiss = 0x80;
constexpr uint8_t kFlagTier = 0x40;

// hit[p] codes (nonzero == answered without touching the backing store)
constexpr uint8_t kHitMiss = 0, kHitC1 = 1, kHitC2 = 2, kHitC3 = 3, kHitApprox = 4;
constexpr uint8_t kHitAbsent = 255;               // bags: no key at this position of the slice (evs_bags.cuh)

struct __align__(16) Slot {
    unsigned long long kw;
    unsigned long long meta;
};

// What a tier's k_evict CTA 0 derives from the counters (its plan), left for whichever CTA closes the batch.
struct EvictOut {
    unsigned long long head[kMaxBuckets];      // ring heads before the victims
    unsigned long long tail[kMaxBuckets];      // ring tails after this batch's appends
    unsigned long long total_v;                // records of the buckets that give up victims
    unsigned int count[kMaxBuckets];           // entries per bucket once the victims are out
    unsigned int take_mask;                    // buckets that give up victims
    unsigned int size, need, top_left, any_perfect, flush, appended, pad;
};

struct TierCtl {
    unsigned long long head[kMaxBuckets];
    unsigned long long tail[kMaxBuckets];
    unsigned long long kept[kMaxBuckets];        // k_evict: first live record left in place (~0: none)
    unsigned long long scan_end[kMaxBuckets];    // k_evict: end of the scanned part of the ring
    unsigned int count[kMaxBuckets];       // live entries per bucket
    unsigned int ticket;                   // k_evict: next eviction chunk
    unsigned int done_ctas;                // k_evict, flush path: CTAs of this tier that have their plan
    unsigned int stop;                     // k_evict: the victims are complete, take no more chunks
    unsigned int n_taken;                  // k_evict: victims evicted by this batch
    unsigned int n_perfect;                // n_perfect_item_C1 (evlfu_32.hpp:51)
    unsigned int full_at_start;            // size >= cap when the batch began (two-tier routing, evlfu_32.cpp:373)
    // per batch (reset by the evict kernel)
    unsigned int n_new;
    unsigned int any_perfect;
    unsigned long long prot;               // max over new keys of pack_prot(bucket+1, position, slot)
    unsigned int n_evicted_last;
    unsigned int n_flushed_last;
    unsigned int error;
    unsigned int pad;
    // cumulative
    unsigned long long stat_inserts, stat_evictions, stat_flushed;
    EvictOut out;                          // k_evict: the plan of the batch in flight
};

struct TierDev {
    Slot *slots;
    unsigned int hash_mask;
    unsigned int row_stride;               // bytes, multiple of 16
    unsigned char *slab;                   // [hash_cap][row_stride]
    unsigned int row_bytes;                // dim*prec/8 (bytes of one backing-store row)
    int prec;                              // 32/16/8/4
    unsigned int *ring;                    // [n_buckets][ring_cap] slot ids
    unsigned int ring_cap;                 // power of two
    unsigned int cap;                      // policy capacity (entries)
    unsigned int max_perfect;              // int(cap * 0.95)
    unsigned int flush_n;                  // int(0.3 * cap) + 1
    int n_buckets;                         // n_tables_total + 1
    TierCtl *ctl;
    const unsigned char *const *store;     // [n_tables] device-visible backing rows at this precision
    unsigned long long *evicted;           // [N] keys evicted by the last batch (rank order)
    unsigned long long *flushed;           // [flush_n] keys flushed by the last batch (or null)
    unsigned long long *lookback;          // [lb_cap] k_evict chunk states: status << 32 | count
    unsigned int lb_cap;
};

// C3 (aprx_embedding.cpp): key -> alternative key, FIFO with second-chance eviction.
struct C3Ctl {
    unsigned long long head, tail;         // FIFO ring window (lists_C3)
    unsigned int size;                     // vals_C3.size()
    unsigned int error;
    unsigned long long stat_inserts, stat_evictions;
};
struct __align__(16) C3Slot {
    unsigned long long kw;                 // pass << 48 | key, as in Slot
    unsigned int alt;                      // alt_row*100 + alt_table(1-based)   (convert_altkeys_to_binary.py:50)
    unsigned int flag;                     // recency flag (aprx_embedding.cpp:402)
};
struct C3Dev {
    C3Slot *slots;
    unsigned int hash_mask;
    unsigned int ring_cap;
    unsigned long long *ring;              // FIFO of keys; may hold stale duplicates like the reference's queue
    unsigned int cap;
    int active;
    C3Ctl *ctl;
    const unsigned int *const *alt;        // [n_tables] device-visible alt-key tables
    unsigned int *scratch;                 // [window] duplicate detection
};

struct GlobalCtl {
    unsigned long long lookups, samples, hits[2], c3_hits, approx_subst, misses, perfect_hits, batches;
    unsigned int error;                    // 1 = index out of range, 7 = a peer did not answer in time
    unsigned int fetch_done_seq;           // number of the last batch whose miss-fetch role has finished (it no longer reads its staging rows)
    unsigned int auto_seq;                 // number of the last batch started; a batch launched with BatchArgs::seq == 0 (a replay of a
                                           // graph the CALLER captured: its arguments are frozen) takes the next number from here
    unsigned int pool_arrived;             // k_bags_pool on a sharded handle: CTAs done with their pooled rows (the last resets it)
};
constexpr unsigned long long kPeerTimeoutNs = 4000000000ull;   // spin-waits on peer flags give up after 4 s

// Arguments that change from batch to batch.  k_serve receives them as a kernel parameter (the
// only graph node whose parameters are updated per batch) and stores them in device memory for
// the kernels that follow it.
constexpr int kMaxPeers = 8;                 // GPUs of one NVSwitch box

// Table-wise sharding over peer memory (evs_shard_*): every rank maps one exchange block of each
// peer (CUDA IPC).  Pooled rows are stored straight into the batch-sharded buffer of the rank
// that owns the sample, per-sample hit counts straight into every peer's count table.  A count is one 32-bit word
// that carries its batch's epoch, so it is valid the moment it arrives (no flag, no fence: a sample waits only for
// ITS counts, not for the peers' whole probe phase); an epoch word per peer says when a batch's rows are complete.  All pointers below are
// addresses in THIS process (peer r's memory for index r, our own for index rank).
struct ShardArgs {
    int world;                             // 0 = not sharded
    int rank;
    int Bl;                                // samples per rank (B / world)
    int T_total;                           // tables of the whole model
    unsigned epoch;                        // batch number, >= 1
    float *recv[kMaxPeers];                // peer r's receive buffer of this epoch's parity: [Bl][T_total][D]
    unsigned *parts[kMaxPeers];            // peer r's count table of this parity, OUR row: [B] words epoch << 5 | hit count
    unsigned *out_flag[kMaxPeers];         // peer r's "rank `rank` has written its rows of epoch e" word
    const unsigned *my_parts;              // our count table of this parity: [world][B]; an entry is valid once it carries this epoch
    const unsigned *my_out_flags;          // [world]
    int fused;                             // 1: k_serve sends its counts, gathers, THEN waits for the peers' counts (one pass);
                                           // 0: a probe_only pass sends the counts first (grids too large to be co-resident)
};

struct BatchArgs {
    const long long *idx;                  // [T][B]
    float *out;
    long long out_stride;                  // floats between samples
    uint8_t *hit;                          // [B][T] or null
    const uint8_t *agg_in;                 // [B] or null
    uint8_t *agg_out;                      // [B]
    int B;
    int probe_only;
    unsigned seq;                          // number of this batch on the handle (>= 1)
    unsigned pf_gen;                       // != 0: evs_prefetch staged rows for this batch (Params::pf_*), tagged with this generation
    int bags;                              // 1: the batch holds slices of ragged bags; a negative index = no key at that position.
                                           // Sharded: the counts still go through the exchange, but the slice rows stay local (out)
                                           // and k_bags_pool sends the pooled rows and raises the completion words
    ShardArgs sh;
};

// Arguments of the look-ahead kernel (k_prefetch, evs_prefetch.cuh)
struct PrefetchArgs {
    const long long *idx;                  // [T][B] of the NEXT batch
    int B;
    unsigned seq;                          // the number that batch will get (its parity selects the staging buffer)
    unsigned gen;                          // generation of this announcement (>= 1): the tag of the rows it stages
    int mode;                              // 0 = probe + stage; 1 = probe and L2 warm-up only (experiments)
};

// Everything a kernel of the batch pipeline needs; constant for the life of a handle.
struct Params {
    TierDev tier[kMaxTiers];
    C3Dev c3;
    int n_tiers;
    int T, D;
    int L, L_shift;                        // lanes per sample: next_pow2(T) and its log2
    int spc;                               // samples per serve / update CTA: 8 warps * 32 / L
    int table_base;
    int tid[kMaxTables];                   // global id of local table t (keys, tier routing parity); table_base + t unless table_ids given
    int col[kMaxTables];                   // output column of local table t: t, or tid[t] in the batch-sharded receive buffers
    int loc[kMaxTables];                   // local index of global table g (-1: not served here)
    int n_perfect_agg;                     // agg value that counts as a perfect hit (n_tables_total)
    int approx_thres;
    int high_thres;                        // high_agghit_threshold (evlfu_32.hpp:74)
    int n_chunks_max;
    int quad_max;                          // batches of more serve CTAs than this get their append offsets from k_scan
    int policy;                            // 0 = EvLFU, 1 = LRU (single tier: one recency ring, every hit re-appends), 2 = LFU (single tier: bucket = frequency - 1)
    const long long *rows;                 // [T] cardinalities
    BatchArgs *args;
    GlobalCtl *g;
    // per-batch scratch
    uint8_t *flags;                        // [N]
    unsigned int *pos_slot;                // [N] slot (in the flag's tier) of a promoted / inserted key
    unsigned int *hist;                    // [kSeqs][n_chunks_max]: per-CTA append counts (prefixes after k_scan)
    unsigned int *tot;                     // [kSeqs] batch totals of the same (k_serve adds, k_evict clears)
    unsigned int stage_stride;             // max row_stride of the tiers (shared-memory staging of unaligned rows)
    unsigned int *done;                    // k_evict: CTAs arrived (every eviction CTA, the last fetch CTA); the last closes the batch
    unsigned int *miss_list;               // [N] position | tier << 31 of every miss of the batch in flight
    unsigned int *miss_ctl;                // [0] entries in miss_list, [1] fetch CTAs finished
    int evict_ctas;                        // CTAs per tier of the eviction roles of k_evict
    int fetch_ctas;                        // CTAs of its miss-fetch role
    int pdl;                               // kernels of a batch are chained by programmatic dependent launch
    unsigned int *err_host;                // mapped pinned copy of g->error: the host sees it without a device round trip
    unsigned long long *ring_host;         // mapped pinned, per tier: batch number << 32 | max over the buckets of tail - head
    // look-ahead staging (evs_prefetch): rows of the next batch's probable misses, by position, two parities
    unsigned int *pf_tag;                  // [2][n_max]: generation << 1 | tier once the row is complete
    unsigned char *pf_rows;                // [2][n_max][stage_stride]
    unsigned int n_max;                    // max_batch * T
    int store_aligned;                     // bit t: every backing row of tier t starts 16-byte aligned
    unsigned long long *dbg;               // [16] %globaltimer stamps of the last batch's phases (ns)
};

__host__ __device__ inline unsigned long long pack_meta(int bucket, unsigned long long q) {
    return (static_cast<unsigned long long>(bucket + 1) << 56) | (q & 0x00FFFFFFFFFFFFFFull);
}
__host__ __device__ inline int meta_bucket(unsigned long long m) { return static_cast<int>(m >> 56) - 1; }
__host__ __device__ inline unsigned long long meta_pos(unsigned long long m) { return m & 0x00FFFFFFFFFFFFFFull; }

// TierCtl::prot: the batch's newest key (highest (bucket, position) among its claims) together with the slot it claimed, so
// that the eviction plan has the protected slot without a dependent load.  6 + 27 + 31 bits: positions < 2^27 (evs_create).
constexpr unsigned long long kMaxProtPositions = 1ull << 27;
__host__ __device__ inline unsigned long long pack_prot(unsigned bucket1, unsigned pos, unsigned slot) {
    return (static_cast<unsigned long long>(bucket1) << 58) | (static_cast<unsigned long long>(pos) << 31) | (slot & 0x7FFFFFFFu);
}
__host__ __device__ inline int prot_bucket(unsigned long long prot) { return static_cast<int>(prot >> 58) - 1; }
__host__ __device__ inline unsigned prot_slot(unsigned long long prot) { return static_cast<unsigned>(prot) & 0x7FFFFFFFu; }

__host__ __device__ inline unsigned long long make_key(int table, long long row) {
    return (static_cast<unsigned long long>(table) << kKeyShift) | static_cast<unsigned long long>(row);
}

// 64-bit finaliser (splitmix64); the slot is the low bits
__host__ __device__ inline unsigned int hash_key(unsigned long long k, unsigned int mask) {
    k ^= k >> 30; k *= 0xbf58476d1ce4e5b9ull;
    k ^= k >> 27; k *= 0x94d049bb133111ebull;
    k ^= k >> 31;
    return static_cast<unsigned int>(k) & mask;
}

}  // namespace evs
