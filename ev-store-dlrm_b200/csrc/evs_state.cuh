// evs_save_state / evs_load_state: the policy state of a handle (keys only, no row bytes) as a snapshot, and back.
//
//   k_state_save      one CTA per (tier, bucket): walks the bucket's ring window [head, tail), keeps the live records
//                     (state_live below) and compacts their keys in FIFO order with a block scan; one more CTA copies
//                     C3's raw FIFO window (stale and duplicate records included) and compacts its map entries.  The
//                     output is the snapshot's body, packed, in a device staging area (offsets from the TierCtl counts).
//                     evs_dump_state / evs_dump_c3 read the same output.
//   k_state_load      after k_init_tier: a group of lanes per key claims a slot (claim_slot: the probing and pass
//                     accounting of a batch's insert), writes meta = pack_meta(bucket, i) and ring[bucket][i] = slot,
//                     and copies the key's backing row into the slab (16-byte loads where the store allows, as the miss
//                     fetch).  Keys of unserved tables, rows out of range and a key twice in one tier set the error word.
//   k_state_load_c3   after k_init_c3: claims the map entries (c3_claim), writes the raw window at [0, W)
//   k_state_load_ctl  one CTA: every TierCtl / C3Ctl field of the loaded (or, after an error, the empty) state
// The rings come out compacted (head = 0, tail = count), which changes no later decision (k_compact does the same).
#pragma once
#include "evs_c3.cuh"

namespace evs {

constexpr int kStateThreads = 1024;
constexpr int kStateMetaWords = 128;         // staging words ahead of the body: [0] body words, [1] status, [2 + 32 t + b] live
                                             // records of bucket b of tier t
constexpr unsigned kStateBadBucket = 1, kStateBadC3 = 2, kStateOverCap = 4;   // save status bits
constexpr unsigned kStateBadKey = 1, kStateDupKey = 2;                         // load error bits

// The live-record rule: record q of bucket b's ring is live iff the slot it names still points back at it.
__device__ __forceinline__ bool state_live(const TierDev &tier, int b, unsigned long long q, unsigned slot, unsigned long long meta) {
    return slot <= tier.hash_mask && meta == pack_meta(b, q);
}

// Words of tier t's section in the body: n_perfect, count[n_buckets], keys.
__device__ __forceinline__ unsigned long long state_tier_words(const TierDev &tier, unsigned long long &n_keys) {
    n_keys = 0;
    for (int b = 0; b < tier.n_buckets; ++b) n_keys += tier.ctl->count[b];
    return 1ull + tier.n_buckets + n_keys;
}

__global__ void __launch_bounds__(kStateThreads) k_state_save(const __grid_constant__ Params p, unsigned long long *meta) {
    __shared__ unsigned s_w[33];
    unsigned long long *out = meta + kStateMetaWords;
    unsigned long long n_keys[kMaxTiers] = {0, 0}, base[kMaxTiers + 1] = {0, 0, 0};
    for (int t = 0; t < p.n_tiers; ++t) base[t + 1] = base[t] + state_tier_words(p.tier[t], n_keys[t]);
    const int nb = p.tier[0].n_buckets;
    const int role = blockIdx.x;
    if (role == 0 && threadIdx.x == 0) {
        unsigned long long words = base[p.n_tiers];
        if (p.c3.active) words += 2ull + (p.c3.ctl->tail - p.c3.ctl->head) + 2ull * p.c3.ctl->size;
        meta[0] = words;
    }
    if (role < p.n_tiers * nb) {
        const int t = role / nb, b = role - t * nb;
        const TierDev &tier = p.tier[t];
        const TierCtl *c = tier.ctl;
        const unsigned cnt = c->count[b];
        unsigned long long kb = base[t] + 1 + nb;
        for (int bb = 0; bb < b; ++bb) kb += c->count[bb];
        if (threadIdx.x == 0) {
            if (b == 0) out[base[t]] = c->n_perfect;
            out[base[t] + 1 + b] = cnt;
        }
        // a tier over capacity cannot occur between batches; its keys would not fit the bound evs_state_bytes gives
        const bool over = n_keys[t] > tier.cap;
        if (over && threadIdx.x == 0) atomicOr(reinterpret_cast<unsigned *>(meta + 1), kStateOverCap);
        const unsigned long long head = c->head[b], tail = c->tail[b];
        const unsigned *ring = tier.ring + static_cast<size_t>(b) * tier.ring_cap;
        unsigned long long live = 0;
        constexpr int R = 4;
        for (unsigned long long q0 = head; q0 < tail; q0 += static_cast<unsigned long long>(kStateThreads) * R) {
            unsigned slot[R];
            uint4 sv[R];
            bool on[R];
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const unsigned long long q = q0 + static_cast<unsigned long long>(threadIdx.x) * R + r;
                slot[r] = (q < tail) ? __ldcg(ring + (q & (tier.ring_cap - 1))) : kNoSlot;
            }
#pragma unroll
            for (int r = 0; r < R; ++r)
                if (slot[r] <= tier.hash_mask) sv[r] = __ldcg(reinterpret_cast<const uint4 *>(tier.slots + slot[r]));
            unsigned mine = 0;
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const unsigned long long q = q0 + static_cast<unsigned long long>(threadIdx.x) * R + r;
                on[r] = slot[r] <= tier.hash_mask && state_live(tier, b, q, slot[r], u64_of(sv[r].z, sv[r].w));
                mine += on[r] ? 1u : 0u;
            }
            unsigned total;
            unsigned idx = block_excl_scan(mine, s_w, &total);
#pragma unroll
            for (int r = 0; r < R; ++r)
                if (on[r]) {
                    const unsigned long long i = live + idx++;
                    if (i < cnt && !over) out[kb + i] = u64_of(sv[r].x, sv[r].y) & kKeyMask;
                }
            live += total;
        }
        if (threadIdx.x == 0) {
            meta[2 + kMaxBuckets * t + b] = live;
            if (live != cnt) atomicOr(reinterpret_cast<unsigned *>(meta + 1), kStateBadBucket);
        }
        return;
    }
    // C3: size, the raw window, the map entries (key, alt | flag << 32) in slot order
    const C3Dev &c3 = p.c3;
    const unsigned long long head = c3.ctl->head, W = c3.ctl->tail - head;
    const unsigned size = c3.ctl->size;
    unsigned long long *o = out + base[p.n_tiers];
    if (threadIdx.x == 0) {
        o[0] = size;
        o[1] = W;
    }
    for (unsigned long long i = threadIdx.x; i < W; i += kStateThreads) o[2 + i] = __ldcg(c3.ring + ((head + i) & (c3.ring_cap - 1)));
    unsigned long long *m = o + 2 + W;
    unsigned n = 0;
    for (unsigned s0 = 0; s0 <= c3.hash_mask; s0 += kStateThreads) {
        const unsigned s = s0 + threadIdx.x;
        const bool in = s <= c3.hash_mask;
        unsigned long long kw = kEmptyKey;
        if (in) kw = __ldcg(&c3.slots[s].kw);
        const bool occ = in && (kw & kKeyMask) != kEmptyKey;
        unsigned total;
        const unsigned j = n + block_excl_scan(occ ? 1u : 0u, s_w, &total);
        if (occ && j < size) {
            m[2 * static_cast<size_t>(j)] = kw & kKeyMask;
            m[2 * static_cast<size_t>(j) + 1] = u64_of(__ldcg(&c3.slots[s].alt), __ldcg(&c3.slots[s].flag));
        }
        n += total;
    }
    if (threadIdx.x == 0 && n != size) atomicOr(reinterpret_cast<unsigned *>(meta + 1), kStateBadC3);
}

struct StateLoadArgs {
    const unsigned long long *keys[kMaxTiers];     // per tier: keys bucket by bucket
    unsigned off[kMaxTiers][kMaxBuckets + 1];     // per tier: first key of each bucket, off[t][n_buckets] = keys of the tier
    unsigned n_perfect[kMaxTiers];
    const unsigned long long *window;              // C3: the FIFO records, oldest first
    unsigned long long W;
    const unsigned long long *map;                 // C3: n_map entries (key, alt | flag << 32)
    unsigned n_map;
    unsigned *err;                                 // kStateBadKey / kStateDupKey
};

// Local table of key, or -1 when its table is not served here or its row is outside [0, rows[table]).
__device__ __forceinline__ int state_table(const Params &p, unsigned long long key, long long &row) {
    row = static_cast<long long>(key & ((1ull << kKeyShift) - 1ull));
    if ((key >> kKeyShift) >= static_cast<unsigned long long>(kMaxTables)) return -1;
    const int t = p.loc[key >> kKeyShift];
    if (t < 0 || row >= __ldg(p.rows + t)) return -1;
    return t;
}

__global__ void __launch_bounds__(256) k_state_load(const __grid_constant__ Params p, const __grid_constant__ StateLoadArgs a) {
    const int G = fetch_gsize(p, p.n_tiers);
    const int lane = threadIdx.x & 31, grp = lane / G, gl = lane - grp * G;
    const unsigned n0 = a.off[0][p.tier[0].n_buckets];
    const unsigned n = n0 + (p.n_tiers == 2 ? a.off[1][p.tier[1].n_buckets] : 0u);
    const unsigned kpw = 32 / G;
    const unsigned gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = (gridDim.x * blockDim.x) >> 5;
    for (unsigned j0 = gw * kpw; j0 < n; j0 += nw * kpw) {                  // uniform per warp: the shuffles see every lane
        const unsigned j = j0 + grp;
        const bool on = j < n;
        const int t = (on && j >= n0) ? 1 : 0;
        const TierDev &tier = p.tier[t];
        const unsigned i = on ? j - (t ? n0 : 0u) : 0u;
        unsigned long long key = 0;
        long long row = 0;
        int lt = -1;
        unsigned slot = 0;
        if (on) {
            key = a.keys[t][i];
            lt = state_table(p, key, row);
        }
        if (on && gl == 0) {
            if (lt < 0) {
                atomicOr(a.err, kStateBadKey);
            } else {
                int b = 0;
                while (a.off[t][b + 1] <= i) ++b;
                bool claimed;
                slot = claim_slot(tier, key, claimed);
                if (!claimed) atomicOr(a.err, kStateDupKey);
                tier.slots[slot].meta = pack_meta(b, i - a.off[t][b]);
                tier.ring[static_cast<size_t>(b) * tier.ring_cap + (i - a.off[t][b])] = slot;
            }
        }
        slot = __shfl_sync(kFull, slot, grp * G);
        if (lt < 0) continue;                                               // uniform per group
        const unsigned char *src = tier.store[lt] + static_cast<size_t>(row) * tier.row_bytes;
        unsigned char *dst = tier.slab + static_cast<size_t>(slot) * tier.row_stride;
        if (p.store_aligned & (1 << t)) {
            for (unsigned c = gl; c < (tier.row_stride >> 4); c += G)
                reinterpret_cast<uint4 *>(dst)[c] = ldg16(src + (c << 4));
        } else {
            fetch_row(src, tier.row_bytes, dst, tier.row_stride, lane);     // G == 32 here (fetch_gsize)
        }
    }
}

__global__ void __launch_bounds__(256) k_state_load_c3(const __grid_constant__ Params p, const __grid_constant__ StateLoadArgs a) {
    const C3Dev &c = p.c3;
    const unsigned long long stride = static_cast<unsigned long long>(gridDim.x) * blockDim.x;
    for (unsigned long long i = static_cast<unsigned long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < a.n_map + a.W; i += stride) {
        long long row;
        if (i < a.n_map) {
            const unsigned long long key = a.map[2 * i], v = a.map[2 * i + 1];
            if (state_table(p, key, row) < 0) {
                atomicOr(a.err, kStateBadKey);
                continue;
            }
            bool claimed;
            const unsigned s = c3_claim(c, key, claimed);
            if (!claimed) atomicOr(a.err, kStateDupKey);
            c.slots[s].alt = static_cast<unsigned>(v);
            c.slots[s].flag = static_cast<unsigned>(v >> 32);
        } else {
            const unsigned long long q = i - a.n_map, key = a.window[q];
            if (state_table(p, key, row) < 0) atomicOr(a.err, kStateBadKey);
            c.ring[q] = key;
        }
    }
}

__global__ void k_state_load_ctl(const __grid_constant__ Params p, const __grid_constant__ StateLoadArgs a) {
    const int b = threadIdx.x;
    for (int t = 0; t < p.n_tiers; ++t) {
        const TierDev &tier = p.tier[t];
        TierCtl *c = tier.ctl;
        if (b < kMaxBuckets) {
            const unsigned cnt = b < tier.n_buckets ? a.off[t][b + 1] - a.off[t][b] : 0u;
            c->head[b] = 0ull;
            c->tail[b] = cnt;
            c->count[b] = cnt;
            c->kept[b] = ~0ull;
            c->scan_end[b] = 0ull;
        }
        if (b == 0) {
            const unsigned size = a.off[t][tier.n_buckets];
            c->n_perfect = a.n_perfect[t];
            c->full_at_start = (size >= tier.cap) ? 1u : 0u;       // the next batch's two-tier routing (k_evict sets it per batch)
            c->ticket = 0;
            c->done_ctas = 0;
            c->stop = 0;
            c->n_taken = 0;
            c->n_new = 0;
            c->any_perfect = 0;
            c->prot = 0ull;
            c->n_evicted_last = 0;
            c->n_flushed_last = 0;
        }
    }
    if (b == 0 && p.c3.active) {
        p.c3.ctl->head = 0ull;
        p.c3.ctl->tail = a.W;
        p.c3.ctl->size = a.n_map;
    }
}

}  // namespace evs
