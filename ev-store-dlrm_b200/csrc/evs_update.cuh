// k_update and k_evict: everything of a batch that changes the cache.
//
//   k_update   same warp <-> sample, lane <-> table mapping as k_serve.  A flagged position
//              (a) claims an index slot if it missed (CAS; same-batch duplicates converge on one slot),
//              (b) appends a record to the FIFO ring of its bucket at the position its rank among the flagged positions of
//                  the batch dictates (sample-major, table-minor: the order EvLFU_C1.py processes them; in C2 all
//                  promotions come before all inserts, as phase_2 does, evlfu_8.cpp:416-442), computed from k_serve's
//                  per-CTA counts,
//              (c) atomicMax on the slot's meta picks the winning occurrence of a key (highest (bucket, position)), bucket
//                  counters follow.
//   k_evict    one grid, blockIdx.y = role.  Eviction roles (one per tier, p.evict_ctas CTAs): advance the ring tails, then
//              evict down to capacity in (bucket, FIFO) order -- the candidate records form one virtual sequence cut into
//              chunks of kEvictWindow records, a CTA's first chunk is its block index, further ones go by ticket, and a chunk
//              learns how many victims precede it by a decoupled look-back over its predecessors' counts.  A batch that
//              triggers the flush rule (rare) takes the single-CTA path of evs_kernels.cuh.  Miss-fetch role
//              (p.fetch_ctas CTAs): fetch_list_body (evs_kernels.cuh).  Every eviction CTA and the last fetch CTA arrive on
//              one counter; the last to arrive (close_batch) writes every tier's counters back, inserts the victims into
//              C3, mirrors the ring occupancy to the host and -- sharded -- exchanges the "rows delivered" words.
#pragma once
#include "evs_c3.cuh"
#include "evs_kernels.cuh"

namespace evs {

// NG = sequence groups in use: 1 for a single tier (only C1's interleaved sequence exists), kSeqGroups with a C2.
// XU = rounds of 32 per-CTA counts a lane holds in registers across the claim.
//
// Ring positions need, per append sequence (group, bucket), the number of records the EARLIER serve CTAs appended.  Unless
// k_scan has turned the per-CTA counts into prefixes (batches of more than quad_max serve CTAs), they are summed here, by
// loads that are issued BEFORE the claim's chain of dependent accesses and consumed after it (a warp issues in order: loads
// placed after the CAS loop would only start when it ends), so they cost no round trip of their own:
//   COOP = false (a sample is a whole warp, the 26 tables of an unsharded model): the warp of a flagged sample sums the
//          counts of its one bucket, lane = earlier CTA;
//   COOP = true  (packed warps: a rank of a sharded cache owns 3-13 tables and a warp carries 2-8 samples): the CTA sums
//          once for all its samples -- the sequences that occur in the CTA are dealt out to the warps, lane = earlier CTA.
//          (Per-sample sums by groups of 4-16 lanes were a serial chain of up to 8 round trips, and handles of fewer than
//          8 tables needed a k_scan launch.)
constexpr int kSeqPerWarp = 4;               // COOP: sequences a warp sums per round
__device__ __forceinline__ bool kth_present(const unsigned *present, int ng, int k, int &g, int &b) {
    for (g = 0; g < ng; ++g) {
        const int c = __popc(present[g]);
        if (k < c) {
            b = static_cast<int>(__fns(present[g], 0, k + 1));
            return true;
        }
        k -= c;
    }
    return false;
}

// LFU (needs COOP, NG = 1): the appends of one sample go to different buckets (bucket = the key's own frequency), so a
// position's rank inside the CTA is counted per bucket -- lanes of a warp that share a bucket find each other with
// match.any, the warps of the CTA add up in sample order -- instead of per sample.
template <int NG, int XU, bool COOP, bool LFU = false>
__global__ void __launch_bounds__(kLookupThreads, COOP ? 3 : (NG == 1 ? 5 : 4)) k_update(const __grid_constant__ Params p) {
    static_assert(!LFU || (COOP && NG == 1), "the LFU path is single-tier and sums per CTA");
    __shared__ unsigned s_wcnt[LFU ? kSamplesPerCta : 1][kMaxBuckets];      // LFU: appends per warp and bucket
    __shared__ unsigned s_cnt[kLookupThreads][kSeqGroups];      // per sample of the CTA (at most 256 when L = 1)
    __shared__ int s_b[kLookupThreads];
    __shared__ int s_delta[kMaxTiers * kMaxBuckets];
    __shared__ unsigned s_new[kMaxTiers], s_ins[kMaxTiers];
    __shared__ unsigned long long s_prot[kMaxTiers];
    __shared__ unsigned s_base[kSeqGroups * kMaxBuckets];       // COOP: records the earlier CTAs append, per sequence
    __shared__ unsigned s_present[kSeqGroups];                  // COOP: buckets that occur in this CTA, per group

    griddep_launch(p);
    if (threadIdx.x < kMaxTiers * kMaxBuckets) s_delta[threadIdx.x] = 0;
    if (threadIdx.x < kMaxTiers) {
        s_new[threadIdx.x] = 0;
        s_ins[threadIdx.x] = 0;
        s_prot[threadIdx.x] = 0ull;
    }
    if (threadIdx.x < kSeqGroups) s_present[threadIdx.x] = 0u;
    if (LFU) s_wcnt[threadIdx.x >> 5][threadIdx.x & 31] = 0u;
    griddep_wait(p);
    if (blockIdx.x == 0 && threadIdx.x == 0) p.dbg[2] = gtime();
    const BatchArgs a = *p.args;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int T = p.T, B = a.B;
    const Grp q = make_grp(p, lane);
    const int spc = p.spc;
    const int n_chunks = (B + spc - 1) / spc;
    if (static_cast<int>(blockIdx.x) >= n_chunks) return;
    const int j = warp * (32 >> p.L_shift) + q.g;      // sample within the CTA
    const int s = blockIdx.x * spc + j;
    const int tbl = q.gl;
    const bool act = (s < B) && (tbl < T);
    const int pos = s * T + tbl;
    const unsigned f = act ? p.flags[pos] : 0u;
    long long r = 0;
    if (f & kFlagMiss) {
        r = __ldg(a.idx + static_cast<size_t>(tbl) * B + s);
        if (r < 0 || r >= __ldg(p.rows + tbl)) r = 0;
    }

    const int tr = (f & kFlagTier) ? 1 : 0;
    const int b = static_cast<int>(f & 0x3Fu) - 1;
    // sequence group of this position: 0 = C1, 1 = C2 promotion, 2 = C2 insert
    const int grp = (f == 0u) ? -1 : (tr == 0 ? 0 : ((f & kFlagMiss) ? 2 : 1));
    const unsigned m0 = __ballot_sync(kFull, grp == 0) & q.mask;
    const unsigned m1 = __ballot_sync(kFull, grp == 1) & q.mask;
    const unsigned m2 = __ballot_sync(kFull, grp == 2) & q.mask;
    const unsigned any = m0 | m1 | m2;
    const int wb = __shfl_sync(kFull, b, any ? (__ffs(any) - 1) : q.base);    // all flagged lanes of a sample share it
    unsigned lfu_rank = 0;
    if (LFU) {
        const unsigned fm = __ballot_sync(kFull, f != 0u);
        if (f) {
            const unsigned peers = __match_any_sync(fm, b);
            lfu_rank = __popc(peers & ((1u << lane) - 1u));
            if (lfu_rank == 0) {
                s_wcnt[warp][b] = __popc(peers);
                atomicOr(&s_present[0], 1u << b);
            }
        }
    }
    if (q.gl == 0) {
        s_cnt[j][0] = __popc(m0);
        s_cnt[j][1] = __popc(m1);
        s_cnt[j][2] = __popc(m2);
        s_b[j] = any ? wb : -1;
        if (COOP && !LFU && any) {
            if (m0) atomicOr(&s_present[0], 1u << wb);
            if (NG > 1 && m1) atomicOr(&s_present[1], 1u << wb);
            if (NG > 1 && m2) atomicOr(&s_present[2], 1u << wb);
        }
    }
    __syncthreads();

    const bool direct = n_chunks <= p.quad_max;
    const int nc = static_cast<int>(blockIdx.x);
    const unsigned msk3[kSeqGroups] = {m0, m1, m2};
    unsigned base[kSeqGroups] = {0, 0, 0};
    // ---- loads that do not depend on the claim ----------------------------------------------------------------------
    constexpr int NX = COOP ? kSeqPerWarp : NG;
    unsigned x[NX][XU];
#pragma unroll
    for (int i = 0; i < NX; ++i)
#pragma unroll
        for (int u = 0; u < XU; ++u) x[i][u] = 0u;
    if (direct) {
        if (COOP) {
            unsigned pres[kSeqGroups] = {s_present[0], NG > 1 ? s_present[1] : 0u, NG > 1 ? s_present[2] : 0u};
#pragma unroll
            for (int i = 0; i < kSeqPerWarp; ++i) {
                int g, bb;
                if (!kth_present(pres, NG, warp + 8 * i, g, bb)) break;
                const unsigned *h = p.hist + static_cast<size_t>(g * kMaxBuckets + bb) * p.n_chunks_max;
#pragma unroll
                for (int u = 0; u < XU; ++u) {
                    const int c = u * 32 + lane;
                    if (c < nc) x[i][u] = __ldcg(h + c);
                }
            }
        } else if (any) {
#pragma unroll
            for (int g = 0; g < NG; ++g) {
                if (!msk3[g]) continue;
                const unsigned *h = p.hist + static_cast<size_t>(g * kMaxBuckets + wb) * p.n_chunks_max;
#pragma unroll
                for (int u = 0; u < XU; ++u) {
                    const int c = u * 32 + lane;
                    if (c < nc) x[g][u] = __ldcg(h + c);
                }
            }
        }
    } else if (any) {
        // k_scan made the counts prefixes
        if (LFU) {
            if (f) base[0] = __ldcg(p.hist + static_cast<size_t>(b) * p.n_chunks_max + blockIdx.x);
        } else {
#pragma unroll
            for (int g = 0; g < NG; ++g)
                if (msk3[g]) base[g] = __ldcg(p.hist + static_cast<size_t>(g * kMaxBuckets + wb) * p.n_chunks_max + blockIdx.x);
        }
    }
    const unsigned tot_p1 = (any && m2) ? __ldcg(p.tot + kMaxBuckets + wb) : 0u;
    unsigned long long tail_b = 0ull;
    if (f) tail_b = static_cast<const volatile TierCtl *>(p.tier[tr].ctl)->tail[b];

    unsigned slot = 0;
    if (f & kFlagMiss) {
        bool claimed = false;
        slot = claim_slot(p.tier[tr], make_key(p.tid[tbl], r), claimed);
        p.pos_slot[pos] = slot | (claimed ? kClaimedBit : 0u);
        if (claimed) atomicAdd(&s_new[tr], 1u);
        atomicMax(&s_prot[tr], pack_prot(f & 0x3Fu, static_cast<unsigned>(pos), slot));
    } else if (f) {
        slot = p.pos_slot[pos];
    }

    // ---- sum the earlier CTAs' counts ----------------------------------------------------------------------------------
    if (direct && COOP) {
        unsigned pres[kSeqGroups] = {s_present[0], NG > 1 ? s_present[1] : 0u, NG > 1 ? s_present[2] : 0u};
        const int n_present = __popc(pres[0]) + __popc(pres[1]) + __popc(pres[2]);
        for (int i0 = 0; warp + 8 * i0 < n_present; i0 += kSeqPerWarp) {
#pragma unroll
            for (int i = 0; i < kSeqPerWarp; ++i) {
                int g, bb;
                if (!kth_present(pres, NG, warp + 8 * (i0 + i), g, bb)) break;
                const unsigned *h = p.hist + static_cast<size_t>(g * kMaxBuckets + bb) * p.n_chunks_max;
                unsigned acc = 0u;
                if (i0 == 0) {
#pragma unroll
                    for (int u = 0; u < XU; ++u) acc += x[i][u];
                }
                for (int c0 = (i0 == 0 ? XU * 32 : 0); c0 < nc; c0 += 128) {       // the rest: 4 loads per lane and round
                    unsigned y[4] = {0, 0, 0, 0};
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const int c = c0 + u * 32 + lane;
                        if (c < nc) y[u] = __ldcg(h + c);
                    }
                    acc += y[0] + y[1] + y[2] + y[3];
                }
#pragma unroll
                for (int d = 16; d > 0; d >>= 1) acc += __shfl_xor_sync(kFull, acc, d);
                if (lane == 0) s_base[g * kMaxBuckets + bb] = acc;
            }
        }
    }
    if (COOP) __syncthreads();

    if (LFU) {
        if (f) {
            unsigned bs = direct ? s_base[b] : base[0];
            for (int w = 0; w < warp; ++w) bs += s_wcnt[w][b];
            const TierDev &tier = p.tier[0];
            const unsigned long long qq = tail_b + bs + lfu_rank;
            tier.ring[static_cast<size_t>(b) * tier.ring_cap + (qq & (tier.ring_cap - 1))] = slot;
            const unsigned long long mine = pack_meta(b, qq);
            const unsigned long long old = atomicMax(&tier.slots[slot].meta, mine);
            if (mine > old) {
                const int ob = meta_bucket(old);
                if (ob != b) {
                    atomicAdd(&s_delta[b], 1);
                    if (ob >= 0) atomicSub(&s_delta[ob], 1);
                    else atomicAdd(&s_ins[0], 1u);
                }
            }
        }
    } else if (any) {
        if (direct && COOP) {
#pragma unroll
            for (int g = 0; g < NG; ++g)
                if (msk3[g]) base[g] = s_base[g * kMaxBuckets + wb];
        } else if (direct) {
            unsigned acc[NG];
#pragma unroll
            for (int g = 0; g < NG; ++g) {
                acc[g] = 0u;
#pragma unroll
                for (int u = 0; u < XU; ++u) acc[g] += x[g][u];
            }
            for (int c0 = XU * 32; c0 < nc; c0 += 128) {       // the rest: 4 loads per lane, group and round
#pragma unroll
                for (int g = 0; g < NG; ++g) {
                    if (!msk3[g]) continue;
                    const unsigned *h = p.hist + static_cast<size_t>(g * kMaxBuckets + wb) * p.n_chunks_max;
                    unsigned y[4] = {0, 0, 0, 0};
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const int c = c0 + u * 32 + lane;
                        if (c < nc) y[u] = __ldcg(h + c);
                    }
                    acc[g] += y[0] + y[1] + y[2] + y[3];
                }
            }
#pragma unroll
            for (int g = 0; g < NG; ++g) {
#pragma unroll
                for (int d = 16; d > 0; d >>= 1) acc[g] += __shfl_xor_sync(kFull, acc[g], d);
                base[g] = acc[g];
            }
        }
        // records of earlier samples of this chunk
        for (int w = 0; w < j; ++w)
            if (s_b[w] == wb) {
#pragma unroll
                for (int g = 0; g < NG; ++g) base[g] += s_cnt[w][g];
            }
        // C2 inserts start after ALL of the batch's C2 promotions in this bucket
        if (m2) base[2] += tot_p1;

        if (f) {
            const TierDev &tier = p.tier[tr];
            const unsigned mine_mask = grp == 0 ? m0 : (grp == 1 ? m1 : m2);
            const unsigned rank = __popc(mine_mask & ((1u << lane) - 1u));
            const unsigned long long qq = tail_b + (grp == 0 ? base[0] : (grp == 1 ? base[1] : base[2])) + rank;
            tier.ring[static_cast<size_t>(b) * tier.ring_cap + (qq & (tier.ring_cap - 1))] = slot;
            const unsigned long long mine = pack_meta(b, qq);
            const unsigned long long old = atomicMax(&tier.slots[slot].meta, mine);
            if (mine > old) {
                const int ob = meta_bucket(old);
                if (ob != b) {
                    atomicAdd(&s_delta[tr * kMaxBuckets + b], 1);
                    if (ob >= 0) atomicSub(&s_delta[tr * kMaxBuckets + ob], 1);
                    else atomicAdd(&s_ins[tr], 1u);
                }
            }
        }
    }

    // ---- publish this CTA's counter deltas ----------------------------------------------------
    __syncthreads();
    if (threadIdx.x < kMaxTiers * kMaxBuckets) {
        const int d = s_delta[threadIdx.x];
        if (d != 0) {
            const int t = threadIdx.x / kMaxBuckets, bb = threadIdx.x - t * kMaxBuckets;
            atomicAdd(&p.tier[t].ctl->count[bb], static_cast<unsigned>(d));
        }
    } else if (threadIdx.x < kMaxTiers * kMaxBuckets + kMaxTiers) {
        const int t = threadIdx.x - kMaxTiers * kMaxBuckets;
        if (t < p.n_tiers) {
            if (s_new[t]) atomicAdd(&p.tier[t].ctl->n_new, s_new[t]);
            if (s_ins[t]) atomicAdd(&p.tier[t].ctl->stat_inserts, static_cast<unsigned long long>(s_ins[t]));
            if (s_prot[t]) atomicMax(&p.tier[t].ctl->prot, s_prot[t]);
        }
    }
    if (threadIdx.x == 0) atomicMax(&p.dbg[3], gtime());
}

// ---- k_evict -------------------------------------------------------------------------------
// What every CTA of a tier derives from the tier's counters (identically): the new ring tails,
// how many victims each bucket gives up, and the virtual record sequence V the chunks index.
struct EvictPlan {
    unsigned long long head[kMaxBuckets];
    unsigned long long tail[kMaxBuckets];      // after this batch's appends
    unsigned count[kMaxBuckets];
    unsigned take[kMaxBuckets];                // victims this bucket gives up
    int seg_b[kMaxBuckets];                    // buckets that give up victims, ascending
    unsigned long long seg_off[kMaxBuckets + 1];   // their offsets in V
    int n_seg;
    unsigned size, need, n_new, n_perfect, any_perfect, flush, prot_slot, appended;
    int prot_b;
};

__device__ __forceinline__ unsigned long long ld_volatile_u64(const unsigned long long *p) {
    return *reinterpret_cast<const volatile unsigned long long *>(p);
}

// Look-back entries of the eviction chunks: status << 62 | own count << 31 | inclusive prefix.
// status 1: the chunk knows its own count; status 2: it also knows how many candidates precede it.
__device__ __forceinline__ unsigned long long lb_pack(unsigned status, unsigned own, unsigned incl) {
    return (static_cast<unsigned long long>(status) << 62) | (static_cast<unsigned long long>(own) << 31) | incl;
}
__device__ __forceinline__ unsigned lb_status(unsigned long long e) { return static_cast<unsigned>(e >> 62); }
__device__ __forceinline__ unsigned lb_own(unsigned long long e) { return static_cast<unsigned>(e >> 31) & 0x7FFFFFFFu; }
__device__ __forceinline__ unsigned lb_incl(unsigned long long e) { return static_cast<unsigned>(e) & 0x7FFFFFFFu; }

// Warp 0 of a chunk: publish this chunk's victim-candidate count, sum the counts of all earlier
// chunks (decoupled look-back: walk back 32 entries at a time until one carries a full prefix),
// publish the inclusive prefix.
__device__ __forceinline__ unsigned lookback_excl(unsigned long long *lb, unsigned ch, unsigned total, int lane) {
    if (ch == 0) {
        if (lane == 0) atomicExch(&lb[0], lb_pack(2u, total, total));
        return 0u;
    }
    if (lane == 0) atomicExch(&lb[ch], lb_pack(1u, total, 0u));
    unsigned excl = 0;
    long long j = static_cast<long long>(ch) - 1;
    while (true) {
        const long long k = j - lane;
        unsigned long long e = lb_pack(2u, 0u, 0u);          // before chunk 0: inclusive prefix 0
        if (k >= 0) {
            do {
                e = ld_volatile_u64(lb + k);
            } while (lb_status(e) == 0u);
        }
        const unsigned incl = __ballot_sync(kFull, lb_status(e) == 2u);
        unsigned v = lb_status(e) == 2u ? lb_incl(e) : lb_own(e);
        if (incl) {
            const int first = __ffs(incl) - 1;               // nearest predecessor with a full prefix
            if (lane > first) v = 0;
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(kFull, v, d);
        excl += v;
        if (incl) break;
        j -= 32;
    }
    if (lane == 0) atomicExch(&lb[ch], lb_pack(2u, total, excl + total));
    return excl;
}

// The same for one of the first blockDim.x chunks, by the whole CTA in one round trip: thread i reads
// the own count of chunk i < ch (every chunk publishes it before it waits for anything), the CTA sums.
__device__ __forceinline__ unsigned lookback_excl_wide(unsigned long long *lb, unsigned ch, unsigned total, unsigned *s_w) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    if (threadIdx.x == 0) atomicExch(&lb[ch], lb_pack(1u, total, 0u));
    unsigned v = 0;
    if (threadIdx.x < ch) {
        unsigned long long e;
        do {
            e = ld_volatile_u64(lb + threadIdx.x);
        } while (lb_status(e) == 0u);
        v = lb_own(e);
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(kFull, v, d);
    __syncthreads();                            // s_w may still be read from the block scan
    if (lane == 0) s_w[warp] = v;
    __syncthreads();
    unsigned excl = 0;
    for (int w = 0; w < nwarp; ++w) excl += s_w[w];
    if (threadIdx.x == 0) atomicExch(&lb[ch], lb_pack(2u, total, excl + total));
    return excl;
}

// The CTA that arrives last closes the batch.  Its chain is one round of independent loads (every tier's published plan,
// the chunks' results, the phase stamps), then stores only:
//   warp t < n_tiers   lane = bucket: write tier t's counters back, reset its per-batch scratch, and keep the longest ring
//                      window in a register for the host's mirror;
//   warp kPhaseWarp    lane = phase-accounting word (p.dbg).
// Then C3, the sharded completion words, the ring mirror (a store into mapped host memory that no fence waits for) and
// the running phase sums.
constexpr int kPhaseWarp = kMaxTiers;
static_assert(kEvictThreads >= (kPhaseWarp + 1) * 32, "close_batch needs a warp per tier plus one");
__device__ __forceinline__ void close_batch(const Params &p) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned nev = static_cast<unsigned>(p.evict_ctas);
    unsigned long long used = 0ull;          // warp t < n_tiers: max over tier t's buckets of tail - head
    unsigned long long d = 0ull, t5 = 0ull;  // warp kPhaseWarp: p.dbg[lane], the closing CTA's start
    const unsigned seq = p.args->seq;
    // a bags batch has delivered no rows yet: k_bags_pool raises and waits for the completion words after pooling
    const int world = p.args->bags ? 0 : p.args->sh.world;
    if (warp < p.n_tiers) {
        const int t = warp, b = lane;
        const TierDev &tier = p.tier[t];
        TierCtl *ctl = tier.ctl;
        volatile TierCtl *c = ctl;
        const volatile EvictOut &o = c->out;
        const bool in = b < tier.n_buckets;
        const unsigned long long oh = o.head[b], ot = o.tail[b], kept = c->kept[b], se = c->scan_end[b];
        const unsigned ocnt = o.count[b];
        const unsigned mask = o.take_mask, size = o.size, need = o.need, top_left = o.top_left, any_perfect = o.any_perfect,
                       flush = o.flush, appended = o.appended;
        const unsigned long long total_v = o.total_v;
        const unsigned taken = c->n_taken, ticket = c->ticket;
        if (!flush) {
            unsigned long long head = oh;
            if ((mask >> b) & 1u) head = (kept != ~0ull) ? kept : (se > oh ? se : oh);
            if (ocnt == 0) head = ot;
            if (in) {
                if (ot - head > tier.ring_cap) c->error = 4u;
                c->head[b] = head;
                c->tail[b] = ot;
                c->count[b] = ocnt;
                used = ot - head;
            }
            if (lane == 0) {
                if (any_perfect) c->n_perfect = top_left;       // EvLFU_C1.py:163-165
                atomicAdd(&ctl->stat_evictions, static_cast<unsigned long long>(taken));
                c->n_evicted_last = taken;
                c->n_flushed_last = 0;
                c->full_at_start = (size - taken >= tier.cap) ? 1u : 0u;
                c->n_new = 0;
                c->prot = 0ull;
                c->any_perfect = 0;
                if (taken != need) c->error = 4u;
                atomicAdd(&p_dbg_appends, static_cast<unsigned long long>(appended));
            }
        } else if (in) {
            used = c->tail[b] - c->head[b];          // evict_tier wrote the counters (rare: a second round trip)
        }
        // per-batch scratch of the tier
        const unsigned n_tk = min(ticket + nev, tier.lb_cap);
        for (unsigned i = lane; i < n_tk; i += 32) tier.lookback[i] = 0ull;
        c->kept[b] = ~0ull;
        c->scan_end[b] = 0ull;
        if (t == 0) {
            p.tot[b] = 0u;
        } else {
            p.tot[kMaxBuckets + b] = 0u;
            p.tot[2 * kMaxBuckets + b] = 0u;
        }
        if (lane == 0) {
            c->ticket = 0;
            c->done_ctas = 0;
            c->stop = 0;
            c->n_taken = 0;
            if (t == 0) {
                atomicAdd(&p.dbg[20], static_cast<unsigned long long>(ticket + nev));
                atomicAdd(&p.dbg[21], total_v);
            }
        }
#pragma unroll
        for (int k = 16; k > 0; k >>= 1) {
            const unsigned long long x = __shfl_xor_sync(kFull, used, k);
            used = x > used ? x : used;
        }
    } else if (warp == kPhaseWarp) {
        t5 = gtime();
        d = __ldcg(&p.dbg[lane]);
    }
    // C3 reads both tiers' n_evicted_last
    __syncthreads();
    if (p.c3.active) c3_update(p);
    if (warp == 0 && world > 1) {
        // every row this rank owes its peers has been stored (k_serve's gather, the fetch role): tell them, then
        // hold the stream until every peer has said the same to us
        const ShardArgs *sh = &p.args->sh;
        const unsigned epoch = sh->epoch;
        __threadfence_system();
        if (lane < world) *reinterpret_cast<volatile unsigned *>(sh->out_flag[lane]) = epoch;
        const unsigned long long tw0 = gtime();
        wait_flags(sh->my_out_flags, world, epoch, lane, p);
        if (lane == 0) p.dbg[29] += gtime() - tw0;
    }
    // the host's view of the ring occupancy (maintain_rings): one 8-byte store into mapped pinned memory per tier, tagged
    // with the batch number; nothing waits for it to land
    if (warp < p.n_tiers && lane == 0)
        *reinterpret_cast<volatile unsigned long long *>(p.ring_host + warp) =
            (static_cast<unsigned long long>(seq) << 32) | (used & 0xFFFFFFFFull);
    if (warp == kPhaseWarp) {
        // phase accounting, one accumulator per lane, from the words loaded with the plans above:
        // running sums over batches (ns): [8] serve, [9] gap, [10] update, [11] gap, [12] evict(+c3), [13] count;
        // k_evict in detail: [22] plan, [23] chunk loops (slowest CTA), [24] wait for the last arrival, [25] close + C3
        t5 = __shfl_sync(kFull, t5, 0);
        unsigned long long t6 = (lane == 0) ? gtime() : 0ull;
        t6 = __shfl_sync(kFull, t6, 0);
        const unsigned long long v0 = __shfl_sync(kFull, d, 0), v1 = __shfl_sync(kFull, d, 1), v2 = __shfl_sync(kFull, d, 2),
                                 v3 = __shfl_sync(kFull, d, 3), v4 = __shfl_sync(kFull, d, 4), v16 = __shfl_sync(kFull, d, 16),
                                 v17 = __shfl_sync(kFull, d, 17);
        const unsigned long long nv = lane == 5 ? t5 : lane == 6 ? t6 : lane == 7 ? v1 : lane == 8 ? d + (v1 - v0)
                                    : lane == 9 ? d + (v2 - v1) : lane == 10 ? d + (v3 - v2) : lane == 11 ? d + (v4 - v3)
                                    : lane == 12 ? d + (t6 - v4) : lane == 13 ? d + 1ull : lane == 18 ? t5
                                    : lane == 22 ? d + (v16 - v4) : lane == 23 ? d + (v17 - v16) : lane == 24 ? d + (t5 - v17)
                                    : d + (t6 - t5);
        const bool wr = (lane >= 5 && lane <= 13) || lane == 18 || (lane >= 22 && lane <= 25);
        if (wr) p.dbg[lane] = nv;
        if (lane == 0) atomicAdd(&p.g->batches, 1ull);
    }
}

// One launch, three kinds of CTA (blockIdx.y = role): roles 0 .. n_tiers-1 evict from that tier (p.evict_ctas CTAs each),
// role n_tiers fetches the batch's missing rows (p.fetch_ctas CTAs: fetch_list_body, evs_kernels.cuh).  The two do not
// depend on each other -- both follow k_update -- so they used to be two kernels on two streams joined by events;
// as roles of one grid the batch is a linear chain of three launches (no fork / join inside the graph).
// The last CTA to arrive, of any role, closes the batch (close_batch): the tiers' counters, C3 insertions, and for a
// sharded handle the "my rows are delivered" words to the peers and the wait for theirs.
template <int P0, int P1>
__global__ void __launch_bounds__(kEvictThreads) k_evict(const __grid_constant__ Params p) {
    extern __shared__ __align__(16) unsigned char s_stage[];    // fetch role: warps * max(row_stride); unaligned rows only
    __shared__ CodecLut s_lut;
    __shared__ EvictPlan P;
    __shared__ unsigned s_w[33];
    __shared__ unsigned s_chunk, s_excl, s_last, s_taken, s_more;
    const int role = blockIdx.y;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    griddep_launch(p);                  // the next batch's k_serve may be made resident: it waits for this grid to finish
    if (role == p.n_tiers) {
        if (static_cast<int>(blockIdx.x) >= p.fetch_ctas) return;
        codec_lut_init<P0, P1>(&s_lut);
        griddep_wait(p);
        __syncthreads();
        if (!fetch_list_body<P0, P1>(p, blockIdx.x, static_cast<unsigned>(p.fetch_ctas), s_stage, &s_lut, &s_last)) return;
    } else {
    if (static_cast<int>(blockIdx.x) >= p.evict_ctas) return;
    const unsigned nev = static_cast<unsigned>(p.evict_ctas);
    const int t = role;
    const TierDev &tier = p.tier[t];
    TierCtl *ctl = tier.ctl;
    volatile TierCtl *c = ctl;
    const int top = tier.n_buckets - 1;
    constexpr unsigned W = kEvictWindow;
    static_assert(kEvictWindow == kEvictThreads, "one ring record per thread");
    griddep_wait(p);
    if (t == 0 && blockIdx.x == 0 && threadIdx.x == 0) {
        p.dbg[4] = gtime();
        if (p.dbg[0] > p.dbg[2]) p.dbg[14] += 1000ull;      // the next batch's k_serve already started (must not happen)
    }

    // ---- plan: lane = bucket; every input in one round of independent loads ----------------
    if (warp == 0) {
        const int b = lane;
        const bool in = b < tier.n_buckets;
        unsigned app = 0;
        if (in) app = (t == 0) ? __ldcg(p.tot + b) : __ldcg(p.tot + kMaxBuckets + b) + __ldcg(p.tot + 2 * kMaxBuckets + b);
        const unsigned long long head = in ? c->head[b] : 0ull;
        const unsigned long long tail = in ? c->tail[b] + app : 0ull;
        const unsigned cnt = in ? c->count[b] : 0u;
        const unsigned n_new = c->n_new;
        const unsigned long long prot = c->prot;
        const unsigned n_perfect = c->n_perfect;
        const unsigned any_perfect = c->any_perfect;
        unsigned size = cnt, appended = app;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            size += __shfl_xor_sync(kFull, size, d);
            appended += __shfl_xor_sync(kFull, appended, d);
        }
        const int prot_b = n_new ? prot_bucket(prot) : -1;
        const unsigned need = size > tier.cap ? size - tier.cap : 0u;
        const unsigned avail = cnt - ((b == prot_b && cnt > 0) ? 1u : 0u);
        unsigned incl = avail;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned n = __shfl_up_sync(kFull, incl, d);
            if (lane >= d) incl += n;
        }
        const unsigned excl = incl - avail;
        const unsigned take = need > excl ? min(avail, need - excl) : 0u;
        const unsigned long long len = take > 0 ? tail - head : 0ull;
        unsigned long long lincl = len;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned long long n = __shfl_up_sync(kFull, lincl, d);
            if (lane >= d) lincl += n;
        }
        const unsigned has = __ballot_sync(kFull, take > 0);
        const int si = __popc(has & ((1u << lane) - 1u));
        P.head[b] = head;
        P.tail[b] = tail;
        P.count[b] = cnt;
        P.take[b] = take;
        if (take > 0) {
            P.seg_b[si] = b;
            P.seg_off[si] = lincl - len;
        }
        const unsigned long long total_v = __shfl_sync(kFull, lincl, 31);
        const unsigned top_left = __shfl_sync(kFull, cnt - take, top);
        const bool overflow = total_v > static_cast<unsigned long long>(tier.lb_cap) * W;     // cannot happen unless a ring overflowed
        const unsigned flush = (n_new > 0 && n_perfect >= tier.max_perfect) ? 1u : 0u;
        if (lane == 0) {
            const int n = __popc(has);
            P.n_seg = n;
            P.seg_off[n] = total_v;
            P.size = size;
            P.need = overflow ? 0u : need;
            if (overflow) c->error = 5u;
            P.n_new = n_new;
            P.n_perfect = n_perfect;
            P.any_perfect = any_perfect;
            P.flush = flush;
            P.prot_b = prot_b;
            P.prot_slot = n_new ? prot_slot(prot) : kNoSlot;
            P.appended = appended;
            s_taken = 0;
        }
        if (blockIdx.x == 0) {
            // the plan, for whichever CTA closes the batch (close_batch)
            EvictOut &o = ctl->out;
            o.head[b] = head;
            o.tail[b] = tail;
            o.count[b] = cnt - take;
            if (lane == 0) {
                o.total_v = total_v;
                o.take_mask = has;
                o.size = size;
                o.need = overflow ? 0u : need;
                o.top_left = top_left;
                o.any_perfect = any_perfect;
                o.flush = flush;
                o.appended = appended;
            }
        }
    }
    __syncthreads();
    if (t == 0 && blockIdx.x == 0 && threadIdx.x == 0) p.dbg[16] = gtime();

    if (P.flush) {
        // flush rule (EvLFU_C1.py:36-44): rare; CTA 0 does flush + eviction alone
        if (blockIdx.x == 0) {
            // the tier's counters may change only after every other CTA has derived its plan from them
            // (they do nothing else in this case and are not waiting for anything)
            if (threadIdx.x == 0)
                while (c->done_ctas < nev - 1) {}
            __syncthreads();
            if (threadIdx.x < tier.n_buckets) c->tail[threadIdx.x] = P.tail[threadIdx.x];
            __syncthreads();
            evict_tier(tier, p);
        } else if (threadIdx.x == 0) {
            atomicAdd(&ctl->done_ctas, 1u);
        }
    } else if (P.need > 0) {
        const unsigned need = P.need;
        const int n_seg = P.n_seg;
        const unsigned long long total_v = P.seg_off[n_seg];
        bool first = true;
        while (true) {
            // the first chunk of a CTA is its block index (no round trip); further ones are handed out
            // by ticket, so a chunk's predecessors always belong to CTAs that are already running
            __syncthreads();
            if (threadIdx.x == 0) s_chunk = first ? blockIdx.x : (c->stop ? kNoSlot : nev + atomicAdd(&ctl->ticket, 1u));
            first = false;
            __syncthreads();
            const unsigned ch = s_chunk;
            if (ch == kNoSlot || static_cast<unsigned long long>(ch) * W >= total_v) break;
            if (ch >= tier.lb_cap) {
                if (threadIdx.x == 0) c->error = 5u;
                break;
            }
            // my record of the chunk
            const unsigned long long v = static_cast<unsigned long long>(ch) * W + threadIdx.x;
            const bool inr = v < total_v;
            int sg = 0, b = 0;
            unsigned long long q = 0;
            unsigned slot = kNoSlot;
            if (inr) {
                while (sg + 1 < n_seg && P.seg_off[sg + 1] <= v) ++sg;
                b = P.seg_b[sg];
                q = P.head[b] + (v - P.seg_off[sg]);
                slot = __ldcg(tier.ring + static_cast<size_t>(b) * tier.ring_cap + (q & (tier.ring_cap - 1)));
            }
            uint4 sv = make_uint4(0, 0, 0, 0);
            const bool okslot = inr && slot <= tier.hash_mask;
            if (okslot) sv = __ldcg(reinterpret_cast<const uint4 *>(tier.slots + slot));
            const bool live = okslot && (u64_of(sv.z, sv.w) == pack_meta(b, q));
            const bool cand = live && slot != P.prot_slot;
            unsigned total;
            const unsigned idx = block_excl_scan(cand ? 1u : 0u, s_w, &total);
            unsigned before;
            if (ch < blockDim.x) {
                before = lookback_excl_wide(tier.lookback, ch, total, s_w);
            } else {
                if (warp == 0) {
                    const unsigned e = lookback_excl(tier.lookback, ch, total, lane);
                    if (lane == 0) s_excl = e;
                }
                __syncthreads();
                before = s_excl;
            }
            if (threadIdx.x == 0) {
                // Does this CTA go on to another chunk?  Not when the victims are complete at or before
                // this chunk, nor when -- at the density seen so far -- the chunks already handed out
                // reach the last victim with a margin.  The CTA holding the LAST chunk handed out is the
                // one that must not leave while victims are missing (it then takes a ticket; so does
                // every CTA whose estimate says the static chunks fall short, and they work in parallel).
                const unsigned incl = before + total;
                unsigned more = 0u;
                if (incl >= need) {
                    if (before < need) {
                        c->stop = 1u;
                        atomicAdd(&p.dbg[26], static_cast<unsigned long long>(ch));
                        atomicMax(&p.dbg[27], static_cast<unsigned long long>(ch));
                    }
                } else {
                    const unsigned long long pred = (static_cast<unsigned long long>(ch) + 1ull) * need / max(incl, 1u) + 1ull;
                    const bool covered = pred + (pred >> 2) + 2ull <= nev;
                    if (!covered) more = 1u;
                    else if (ch + 1u >= nev) more = (ch + 1u == nev + c->ticket) ? 1u : 0u;
                }
                s_more = more;
            }
            const bool takeit = cand && (before + idx < need);
            if (takeit) {
                const unsigned long long key = u64_of(sv.x, sv.y) & kKeyMask;
                evict_slot(tier, slot, key);
                tier.evicted[before + idx] = key;
            }
            // first live record left in place, per bucket: within a warp q grows with the lane.  The plain pre-check keeps
            // the same-address atomics few (a bare atomicMin from every warp measured no faster)
            const bool stays = live && !takeit;
            unsigned pending = __ballot_sync(kFull, stays);
            while (pending) {
                const int leader = __ffs(pending) - 1;
                const int lb_ = __shfl_sync(kFull, b, leader);
                const unsigned same = __ballot_sync(kFull, stays && b == lb_);
                if (lane == leader && q < ld_volatile_u64(&ctl->kept[b])) atomicMin(&ctl->kept[b], q);
                pending &= ~same;
            }
            if (before < need) {
                // everything of these buckets up to here has been examined
                const bool seg_end = inr && (threadIdx.x == W - 1 || v + 1 == total_v || v + 1 == P.seg_off[sg + 1]);
                if (seg_end) atomicMax(&ctl->scan_end[b], q + 1);
                const unsigned nt = __popc(__ballot_sync(kFull, takeit));
                if (lane == 0 && nt) atomicAdd(&s_taken, nt);
            }
            __syncthreads();
            if (!s_more) break;
        }
    }

    // ---- arrival ----------------------------------------------------------------------------
    __syncthreads();
    if (t == 0 && threadIdx.x == 0) atomicMax(&p.dbg[17], gtime());
    if (threadIdx.x == 0 && s_taken) atomicAdd(&ctl->n_taken, s_taken);

    }   // eviction role

    // ---- one arrival level: every eviction CTA of every tier and the last fetch CTA; the last to arrive closes the batch
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        const unsigned n_arrivals = static_cast<unsigned>(p.n_tiers * p.evict_ctas) + 1u;
        const unsigned prev = atomicAdd(p.done, 1u);
        s_last = (prev == n_arrivals - 1u) ? 1u : 0u;
        if (s_last) *p.done = 0u;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    close_batch(p);
}

}  // namespace evs
