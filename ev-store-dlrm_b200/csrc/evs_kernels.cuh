// Kernels of one batch of the embedding-lookup hot path, for one or two cache tiers (+ C3).
//
//   k_serve    probe both tiers -> per-sample agg_hit -> route (EvLFU promote / insert per tier; LRU / LFU variants) ->
//              gather + dequantise every resident row into the fp32 output; writes the batch's flags, per-CTA append
//              counts and compact miss list.  Read-only on the cache (C3 recency flags excepted).  As a rank of a
//              table-wise sharded cache it also sends the per-sample hit counts to the peers, stores its rows into the
//              owner ranks' receive buffers and waits for the peers' counts.
//   k_scan     only for batches of more than kQuadMaxChunks serve CTAs: per (group, bucket) exclusive scan of the per-CTA
//              append counts (smaller batches sum their predecessors in k_update)
//   k_update   (evs_update.cuh) claim index slots for missing keys (dedup by CAS), append promoted / inserted entries to
//              their bucket's FIFO ring in position order
//   k_evict    (evs_update.cuh) roles of one grid: eviction of each tier down to capacity in (bucket, FIFO) order (flush
//              rule first), and the miss fetch (fetch_list_body below) from the look-ahead's staging rows or zero-copy from
//              the host backing store; the last role closes the batch (C3, peers)
//   k_prefetch (evs_prefetch.cuh) look-ahead for the next batch on its own stream
//   k_compact  squeeze dead records out of one bucket ring (rare, host-triggered)
// The kernels of a batch (and the batches inside one graph) are joined by programmatic dependent launch: a kernel
// boundary costs ~0.8 us that way, a dependent L2 / HBM access 0.3 - 0.8 us.
#pragma once
#include "evs_codec.cuh"
#include "evs_types.cuh"

namespace evs {

constexpr unsigned kFull = 0xFFFFFFFFu;
constexpr int kEvictThreads = 256;         // small CTAs: they must fit on SMs that k_fetch occupies
constexpr int kEvictPerThread = 4;           // ring records one thread examines per window
constexpr int kQuadMaxChunks = 512;          // above this a k_scan launch replaces the direct prefix sums (B = 16384: 150 -> 141 us)

__device__ __forceinline__ uint4 ldg16(const void *p) { return __ldg(reinterpret_cast<const uint4 *>(p)); }
__device__ __forceinline__ unsigned long long gtime() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ unsigned long long u64_of(unsigned lo, unsigned hi) {
    return (static_cast<unsigned long long>(hi) << 32) | lo;
}

// Programmatic dependent launch (Params::pdl): a kernel of the batch is launched while its predecessor drains; it may
// run its preamble, and blocks here until the predecessor's grid has completed and its writes are visible.
__device__ __forceinline__ void griddep_wait(const Params &p) {
    if (p.pdl) asm volatile("griddepcontrol.wait;" ::: "memory");
}
__device__ __forceinline__ void griddep_launch(const Params &p) {
    if (p.pdl) asm volatile("griddepcontrol.launch_dependents;");
}

// Where the fp32 rows of sample s go: the caller's buffer, or -- table-wise sharded -- the receive
// buffer of the rank that owns the sample (peer memory over NVLink).  Local table t lands at column p.col[t].
// A bags batch keeps its slice rows local on a sharded handle too (a.out: the handle's slice staging); k_bags_pool sends
// the pooled rows.
__device__ __forceinline__ float *out_row(const BatchArgs &a, const Params &p, int s) {
    if (a.sh.world <= 1 || a.bags) return a.out + static_cast<size_t>(s) * a.out_stride;
    const int dst = s / a.sh.Bl, ls = s - dst * a.sh.Bl;
    return a.sh.recv[dst] + static_cast<size_t>(ls) * a.sh.T_total * p.D;
}
__device__ __forceinline__ bool out_vec_ok(const BatchArgs &a, int D) {
    if (a.sh.world > 1 && !a.bags) return (D & 3) == 0;   // receive buffers are cudaMalloc'ed blocks
    return ((reinterpret_cast<uintptr_t>(a.out) & 15u) == 0) && ((a.out_stride & 3) == 0) && ((D & 3) == 0);
}
__device__ __forceinline__ void set_error(const Params &p, unsigned code) {
    p.g->error = code;
    *reinterpret_cast<volatile unsigned *>(p.err_host) = code;
}

// Lanes 0..world-1 wait until every rank's flag word has reached `epoch` (the words live in OUR
// memory, peers store into them).  Gives up after kPeerTimeoutNs and reports error 7.
__device__ __forceinline__ void wait_flags(const unsigned *flags, int world, unsigned epoch, int lane, const Params &p) {
    if (lane < world) {
        const volatile unsigned *f = flags + lane;
        if (static_cast<int>(*f - epoch) < 0) {
            const unsigned long long t0 = gtime();
            while (static_cast<int>(*f - epoch) < 0) {
                if (gtime() - t0 > kPeerTimeoutNs) {
                    set_error(p, 7u);
                    break;
                }
                __nanosleep(64);
            }
        }
        __threadfence();
    }
    __syncwarp();
}

// ---- index probe ---------------------------------------------------------------------
// Linear probing.  The walk ends at the key or at the first slot no resident key's path crosses
// (pass == 0).  A dependent HBM access costs ~0.4 us here, so a probe never walks slot by slot:
// it loads 4 consecutive slots at once (two 32-byte sectors), then 8 per round; at the <= 1/3
// load factor of the index > 98 % of the probes end in the first round.
template <int N>
__device__ __forceinline__ void probe_load(const Slot *__restrict__ slots, unsigned mask, unsigned i, uint4 (&v)[N]) {
#pragma unroll
    for (int k = 0; k < N; ++k) v[k] = ldg16(slots + ((i + k) & mask));
}
// 1 = found, 0 = absent, -1 = undecided after these N slots
template <int N>
__device__ __forceinline__ int probe_check(const uint4 (&v)[N], unsigned mask, unsigned long long key, unsigned i,
                                           unsigned &slot_out, unsigned long long &meta_out) {
    // branch-free, last slot first, so that the FIRST decisive slot wins and the loaded words stay in
    // registers (an early return inside the loop made ptxas spill the array to local memory)
    int res = -1;
#pragma unroll
    for (int k = N - 1; k >= 0; --k) {
        const unsigned long long kw = u64_of(v[k].x, v[k].y);
        const bool match = (kw & kKeyMask) == key;
        const bool stop = (kw >> 48) == 0ull;
        if (match) {
            slot_out = (i + k) & mask;
            meta_out = u64_of(v[k].z, v[k].w);
        }
        res = match ? 1 : (stop ? 0 : res);
    }
    return res;
}
__device__ __forceinline__ bool probe_rest(const Slot *__restrict__ slots, unsigned mask, unsigned long long key, unsigned i,
                                           unsigned &slot_out, unsigned long long &meta_out) {
    while (true) {
        uint4 v[8];
        probe_load<8>(slots, mask, i, v);
        const int r = probe_check<8>(v, mask, key, i, slot_out, meta_out);
        if (r >= 0) return r == 1;
        i += 8;
    }
}
__device__ __forceinline__ bool probe(const TierDev &t, unsigned long long key, unsigned &slot, unsigned long long &meta) {
    const unsigned i = hash_key(key, t.hash_mask);
    uint4 v[4];
    probe_load<4>(t.slots, t.hash_mask, i, v);
    const int r = probe_check<4>(v, t.hash_mask, key, i, slot, meta);
    if (r >= 0) return r == 1;
    return probe_rest(t.slots, t.hash_mask, key, i + 4, slot, meta);
}

// C3: key -> alt key (aprx_embedding.cpp:344 get_altkey_str).  Plain loads: the recency flag of
// these slots is written by this same kernel.
__device__ __forceinline__ bool c3_find(const C3Dev &c, unsigned long long key, unsigned &slot_out, unsigned &alt_out) {
    unsigned i = hash_key(key, c.hash_mask);
    while (true) {
        const unsigned long long kw = __ldcg(&c.slots[i].kw);
        if ((kw & kKeyMask) == key) {
            slot_out = i;
            alt_out = __ldcg(&c.slots[i].alt);
            return true;
        }
        if ((kw >> 48) == 0ull) return false;
        i = (i + 1) & c.hash_mask;
    }
}

// ---- miss fetch ---------------------------------------------------------------------------
// Copy one backing-store row (row_bytes, arbitrary alignment) into a 16-byte aligned staging
// row of `stride` bytes, zero padded.  Zero-copy reads when the store lives in pinned host memory.
__device__ __forceinline__ void fetch_row(const unsigned char *__restrict__ src, unsigned row_bytes,
                                          unsigned char *stage, unsigned stride, int lane) {
    const uintptr_t a = reinterpret_cast<uintptr_t>(src);
    if (((a | row_bytes) & 3u) == 0) {
        for (unsigned o = lane * 4u; o < row_bytes; o += 128u)
            *reinterpret_cast<unsigned *>(stage + o) = __ldg(reinterpret_cast<const unsigned *>(src + o));
    } else if (((a | row_bytes) & 1u) == 0) {
        for (unsigned o = lane * 2u; o < row_bytes; o += 64u)
            *reinterpret_cast<unsigned short *>(stage + o) = __ldg(reinterpret_cast<const unsigned short *>(src + o));
    } else {
        for (unsigned o = lane; o < row_bytes; o += 32u) stage[o] = __ldg(src + o);
    }
    for (unsigned o = row_bytes + lane; o < stride; o += 32u) stage[o] = 0;
}

// Fetch one missing row from `src` (its backing-store row, or the copy evs_prefetch staged in HBM): dequantised
// into the output and, raw, into the slab row of the slot the position claimed (dst; null for a same-batch
// duplicate of a key another position claimed).  Executed by a group of `gsize` consecutive lanes
// (glane = lane within the group) straight through registers when rows are 16-byte aligned
// (stage == nullptr), else by the whole warp via a shared-memory staging row.
template <int PREC>
__device__ __forceinline__ void fetch_one(const TierDev &tier, const unsigned char *src, bool coherent, float *orow, int D,
                                          unsigned char *dst, int lane, int glane, int gsize, unsigned char *stage,
                                          bool vec, const CodecLut *lut) {
    const int cpr = static_cast<int>(tier.row_stride >> 4);
    if (stage == nullptr) {
        for (int c = glane; c < cpr; c += gsize) {
            const uint4 v = coherent ? __ldcg(reinterpret_cast<const uint4 *>(src + (c << 4))) : ldg16(src + (c << 4));
            if (dst != nullptr) *reinterpret_cast<uint4 *>(dst + (c << 4)) = v;
            decode_store<PREC>(v, orow, c, D, vec, lut);
        }
    } else {
        fetch_row(src, tier.row_bytes, stage, tier.row_stride, lane);
        __syncwarp();
        for (int c = lane; c < cpr; c += 32) {
            const uint4 v = *reinterpret_cast<const uint4 *>(stage + (c << 4));
            if (dst != nullptr) *reinterpret_cast<uint4 *>(dst + (c << 4)) = v;
            decode_store<PREC>(v, orow, c, D, vec, lut);
        }
        __syncwarp();
    }
}

// Lanes per row when every stored row is 16-byte aligned (a power of two covering the widest row's chunks), else 32.
__device__ __forceinline__ int fetch_gsize(const Params &p, int n_tiers) {
    const bool al0 = (p.store_aligned & 1) != 0, al1 = (n_tiers < 2) || (p.store_aligned & 2) != 0;
    if (!(al0 && al1)) return 32;
    unsigned cpr = p.tier[0].row_stride >> 4;
    if (n_tiers == 2 && (p.tier[1].row_stride >> 4) > cpr) cpr = p.tier[1].row_stride >> 4;
    int gsize = 1;
    while (gsize < static_cast<int>(cpr) && gsize < 32) gsize <<= 1;
    return gsize;
}

// ---- the miss-fetch role of k_evict ---------------------------------------------------------
// Driven by the compact miss list k_serve wrote (entry = position | tier << 31): every group of lanes takes one
// missing row per round, so a SMALL number of CTAs keeps a bounded number of PCIe reads in flight all the time.
// Why: the link serves 55-110 row reads / us whatever is asked of it (the GPU's address translation for system
// memory is the limit once the table exceeds ~512 MB: profiles/r2_zc_page_probe.txt); letting every miss of the
// batch issue at once only delays the HBM accesses of the eviction CTAs running next to it (profiles/r1_fetch_list_ab.md).
// A row that evs_prefetch already staged in HBM for this batch (tag == generation << 1 | tier) is copied from there
// instead -- the common case when the caller announces its next batch.
// Returns true in the CTA that finished last (all rows of the batch are in place).
template <int P0, int P1>
__device__ __forceinline__ bool fetch_list_body(const Params &p, unsigned cta, unsigned n_ctas, unsigned char *s_stage,
                                                const CodecLut *s_lut, unsigned *s_flag) {
    // the few per-batch arguments this role needs, in registers (a by-value copy of BatchArgs would live in
    // local memory: ShardArgs' pointer arrays are indexed dynamically); peers' buffers are looked up on demand
    const BatchArgs *ga = p.args;
    const long long *idx = ga->idx;
    const int B = ga->B;
    float *out = ga->out;
    const long long out_stride = ga->out_stride;
    const int world = ga->bags ? 0 : ga->sh.world, Bl = ga->sh.Bl, T_total = ga->sh.T_total;   // bags: as out_row()
    const unsigned want_tag = ga->pf_gen << 1;
    const bool use_pf = ga->pf_gen != 0u;
    const unsigned par = ga->seq & 1u;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int wpc = blockDim.x >> 5;
    const int T = p.T, D = p.D;
    const unsigned n = __ldcg(p.miss_ctl);
    const TierDev &t0 = p.tier[0];
    const TierDev &t1 = p.tier[1];
    const bool vec = (world > 1) ? ((D & 3) == 0)
                                 : (((reinterpret_cast<uintptr_t>(out) & 15u) == 0) && ((out_stride & 3) == 0) && ((D & 3) == 0));
    const bool al0 = (p.store_aligned & 1) != 0, al1 = (P1 == 0) || (p.store_aligned & 2) != 0;
    const int gsize = fetch_gsize(p, P1 == 0 ? 1 : 2);
    const int rpw = 32 / gsize, grp = lane / gsize, gl = lane - grp * gsize;
    unsigned char *stage = s_stage + static_cast<size_t>(warp) * p.stage_stride;
    const unsigned gw = cta * wpc + warp, nw = n_ctas * wpc;
    for (unsigned i0 = gw * rpw; i0 < n; i0 += nw * rpw) {
        const unsigned i = i0 + grp;
        if (i < n) {
            const unsigned e = __ldcg(p.miss_list + i);
            const int pos = static_cast<int>(e & 0x7FFFFFFFu);
            const unsigned tr = (P1 == 0) ? 0u : (e >> 31);
            const int s = pos / T, t = pos - s * T;
            const unsigned sw = __ldcg(p.pos_slot + pos);       // the slot this position claimed in k_update, if it is the claimer
            bool staged = false;
            if (use_pf) staged = __ldcg(p.pf_tag + static_cast<size_t>(par) * p.n_max + pos) == (want_tag | tr);
            float *orow;
            if (world <= 1) {
                orow = out + static_cast<size_t>(s) * out_stride + p.col[t] * D;
            } else {                                            // as out_row(): the owner rank's receive buffer
                const int dst = s / Bl, ls = s - dst * Bl;
                orow = ga->sh.recv[dst] + (static_cast<size_t>(ls) * T_total + p.col[t]) * D;
            }
            const TierDev &tier = tr ? t1 : t0;
            const unsigned char *src;
            if (staged) {
                __threadfence();                                // the row was written before its tag
                src = p.pf_rows + (static_cast<size_t>(par) * p.n_max + pos) * p.stage_stride;
            } else {
                long long r = __ldg(idx + static_cast<size_t>(t) * B + s);
                if (r < 0 || r >= __ldg(p.rows + t)) r = 0;
                src = tier.store[t] + static_cast<size_t>(r) * tier.row_bytes;
            }
            unsigned char *dst = (sw & kClaimedBit) ? tier.slab + static_cast<size_t>(sw & ~kClaimedBit) * tier.row_stride : nullptr;
            if (P1 == 0 || !tr)
                fetch_one<P0>(t0, src, staged, orow, D, dst, lane, gl, gsize, (al0 || staged) ? nullptr : stage, vec, s_lut);
            else
                fetch_one<(P1 != 0 ? P1 : 32)>(t1, src, staged, orow, D, dst, lane, gl, gsize, (al1 || staged) ? nullptr : stage, vec, s_lut);
        }
    }
    // the last CTA empties the list for the next batch (every CTA has read the count by then)
    __syncthreads();
    if (threadIdx.x == 0) {
        if (world > 1) __threadfence_system();      // rows stored into peers' receive buffers
        else __threadfence();
        const bool last = atomicAdd(p.miss_ctl + 1, 1u) == n_ctas - 1;
        if (last) {
            p.miss_ctl[0] = 0u;
            p.miss_ctl[1] = 0u;
            p.dbg[28] += gtime() - p.dbg[4];      // fetch span, counted from the start of the k_evict it is part of
            // the staging rows of this batch's parity are free: the look-ahead for batch seq + 2 may overwrite them
            *reinterpret_cast<volatile unsigned *>(&p.g->fetch_done_seq) = ga->seq;
        }
        *s_flag = last ? 1u : 0u;
    }
    __syncthreads();
    return *s_flag != 0u;
}

// ---- k_serve ---------------------------------------------------------------------------
// A sample is handled by a GROUP of L = next_pow2(T) consecutive lanes (lane gl of the group holds
// the key of table gl); a warp carries 32 / L samples.  With the 26 tables of the whole model
// L = 32 and a warp is one sample; a rank of a table-wise sharded run owns 3-13 tables and packs
// 8-2 samples into each warp instead of idling most lanes.
struct Grp {
    int L, g, gl;            // lanes per sample, group of this lane, lane within the group
    unsigned mask;           // the group's lanes
    int base;                // first lane of the group
};
__device__ __forceinline__ Grp make_grp(const Params &p, int lane) {
    Grp q;
    q.L = p.L;
    q.g = lane >> p.L_shift;
    q.gl = lane & (q.L - 1);
    q.base = q.g << p.L_shift;
    q.mask = (q.L == 32) ? kFull : (((1u << q.L) - 1u) << q.base);
    return q;
}
// sum over the lanes of a group (L a power of two, groups aligned)
__device__ __forceinline__ int grp_sum(int v, int L) {
    for (int d = L >> 1; d > 0; d >>= 1) v += __shfl_xor_sync(kFull, v, d);
    return v;
}

// Gather the rows tier `k` serves for this group's sample: the group's lanes walk the sample's
// T*CPR 16-byte chunks so consecutive lanes read consecutive 16 B of a row and write consecutive
// floats of the output; all loads of an unrolled round are issued before the first decode/store.
template <int PREC>
__device__ __forceinline__ void gather_tier(const Params &p, const TierDev &t, int k, int src_t, unsigned src_s, float *orow, bool sact,
                                            int T, int D, bool vec, const Grp &q, const CodecLut *lut) {
    if (__ballot_sync(kFull, src_t == k) == 0u) return;
    constexpr int U = 4;
    const int cpr = static_cast<int>(t.row_stride >> 4);
    const int total = T * cpr;
    for (int c0 = 0; c0 < total; c0 += q.L * U) {
        uint4 v[U];
        int tt[U], part[U];
        bool ok[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int c = c0 + u * q.L + q.gl;
            const bool inb = c < total;
            tt[u] = inb ? c / cpr : 0;
            part[u] = c - tt[u] * cpr;
            const int st = __shfl_sync(kFull, src_t, q.base + tt[u]);
            const unsigned sl = __shfl_sync(kFull, src_s, q.base + tt[u]);
            ok[u] = inb && sact && (st == k);
            if (ok[u]) v[u] = ldg16(t.slab + static_cast<size_t>(sl) * t.row_stride + (part[u] << 4));
        }
#pragma unroll
        for (int u = 0; u < U; ++u)
            if (ok[u]) decode_store<PREC>(v[u], orow + p.col[tt[u]] * D, part[u], D, vec, lut);
    }
}

// A CTA covers p.spc = 8 * (32 / L) consecutive samples, so the int64 index tile is read as T runs
// of 8*spc contiguous bytes.  P1 == 0: single tier.  The cache state is only read here (C3 recency
// flags excepted).
// SH: the handle is one rank of a table-wise sharded cache.  With a.sh.fused the kernel is the whole exchange: it
// stores each sample's local hit count into every rank's count table, gathers the rows it can already serve
// straight into the owner ranks' receive buffers (which row serves a key does not depend on agg_hit), and only then
// waits for the peers' counts -- their NVLink round trip runs under the gather -- to derive agg_hit, the EvLFU
// flags and the miss list.  Every CTA spins on words that the peers' LAST CTAs raise, so the grid must be
// co-resident (evs_shard_connect checks the occupancy and falls back to a separate probe_only pass otherwise).
template <int P0, int P1, bool SH>
__global__ void __launch_bounds__(kLookupThreads, (P1 == 0) ? 5 : 1) k_serve(const __grid_constant__ Params p, const __grid_constant__ BatchArgs a) {
    __shared__ long long s_idx[kLookupThreads];          // [sample in CTA][L]
    __shared__ unsigned s_hist[kSeqs];
    __shared__ unsigned s_stat[8];           // hits C1, hits C2, C3, approx, misses, perfect, positions without a key (bags)
    __shared__ CodecLut s_lut;

    // Launched without a graph, k_serve is programmatically dependent on the previous batch's k_evict (which lets its
    // dependents go at once): the launch latency of this kernel runs under that kernel's tail.  Nothing -- not even
    // the caller's index batch, whose producer may be the kernel before us -- is touched before the wait.
    griddep_wait(p);
    const unsigned long long t_start = gtime();
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        p.dbg[0] = t_start;
        if (p.dbg[4] > p.dbg[6]) p.dbg[14] += 1ull;       // previous batch's k_evict has not finished (must stay 0)
        *p.args = a;                                       // the later kernels of this batch read the arguments here
        if (a.seq != 0u) p.g->auto_seq = a.seq;
        else p.args->seq = (p.g->auto_seq += 1u);          // replayed from a caller's graph: the device numbers the batch
    }
    griddep_launch(p);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int T = p.T, B = a.B, D = p.D;
    const Grp q = make_grp(p, lane);
    const int spc = p.spc;
    const int s0 = blockIdx.x * spc;
    if (s0 >= B) return;

    for (int i = threadIdx.x; i < spc * T; i += kLookupThreads) {
        const int t = i / spc, j = i - t * spc;
        const int s = s0 + j;
        s_idx[(j << p.L_shift) + t] = (s < B) ? __ldg(a.idx + static_cast<size_t>(t) * B + s) : 0;
    }
    if (threadIdx.x < kSeqs) s_hist[threadIdx.x] = 0;
    if (threadIdx.x < 8) s_stat[threadIdx.x] = 0;
    codec_lut_init<P0, P1>(&s_lut);
    const TierDev &t0 = p.tier[0];
    const TierDev &t1 = p.tier[1];
    const int full = (P1 != 0) ? static_cast<int>(t0.ctl->full_at_start) : 0;
    __syncthreads();

    const int j = warp * (32 >> p.L_shift) + q.g;     // sample within the CTA
    const int s = s0 + j;
    const bool sact = s < B;                   // a group past the batch end only joins the warp-wide operations
    bool act = sact && q.gl < T;
    const int tbl = q.gl;
    const int gtbl = act ? p.tid[tbl] : 0;     // global table id
    unsigned long long key = 0, m0 = 0, m1 = 0;
    unsigned slot0 = 0, slot1 = 0;
    bool h0 = false, h1 = false;
    // bags: a negative index = this slice has no key for the table (the bag is shorter): nothing to probe, count or serve
    const bool absent = act && a.bags != 0 && s_idx[(j << p.L_shift) + tbl] < 0;
    if (absent) act = false;
    if (act) {
        long long r = s_idx[(j << p.L_shift) + tbl];
        if (r < 0 || r >= __ldg(p.rows + tbl)) {
            set_error(p, 1u);                  // EVS_ERR_INDEX; answer from row 0
            r = 0;
        }
        key = make_key(gtbl, r);
        // both tiers' first rounds are in flight together
        const unsigned i0 = hash_key(key, t0.hash_mask);
        uint4 v0[4];
        probe_load<4>(t0.slots, t0.hash_mask, i0, v0);
        if (P1 != 0) {
            const unsigned i1 = hash_key(key, t1.hash_mask);
            uint4 v1[4];
            probe_load<4>(t1.slots, t1.hash_mask, i1, v1);
            const int r1 = probe_check<4>(v1, t1.hash_mask, key, i1, slot1, m1);
            h1 = (r1 >= 0) ? (r1 == 1) : probe_rest(t1.slots, t1.hash_mask, key, i1 + 4, slot1, m1);
        }
        const int r0 = probe_check<4>(v0, t0.hash_mask, key, i0, slot0, m0);
        h0 = (r0 >= 0) ? (r0 == 1) : probe_rest(t0.slots, t0.hash_mask, key, i0 + 4, slot0, m0);
    }

    // C3 (evlfu_8.cpp:474-489, 528-558): a double miss whose alternative key is resident in C1,
    // else C2, is answered with that row; the C3 entry gets its recency flag.
    bool c3hit = false;
    int c3_tier = 0;
    unsigned c3_slot = 0;
    if (P1 != 0 && p.c3.active) {
        if (act && !h0 && !h1) {
            unsigned cs, alt;
            if (c3_find(p.c3, key, cs, alt)) {
                const unsigned long long akey = make_key(static_cast<int>(alt % 100u) - 1, static_cast<long long>(alt / 100u));
                unsigned long long am;
                if (probe(t0, akey, c3_slot, am)) {
                    c3hit = true;
                    c3_tier = 0;
                } else if (probe(t1, akey, c3_slot, am)) {
                    c3hit = true;
                    c3_tier = 1;
                }
                if (c3hit) p.c3.slots[cs].flag = 1u;       // set_recency_flag_c3 (aprx_embedding.cpp:402)
            }
        }
    }

    const unsigned m_h0 = __ballot_sync(kFull, h0) & q.mask;
    const unsigned m_h1 = __ballot_sync(kFull, h1) & q.mask;
    const unsigned m_c3 = __ballot_sync(kFull, c3hit) & q.mask;
    int agg;
    if (P1 == 0) agg = __popc(m_h0);                                   // evlfu_32.cpp:477-492
    else if (full) agg = __popc(m_h0 | m_h1) + __popc(m_c3);           // evlfu_8.cpp:512-541
    else agg = __popc(m_h0);                                           // evlfu_8.cpp:601 (C1 not full)
    const int local_agg = agg;
    const bool fused = SH && a.sh.world > 1 && a.sh.fused != 0 && a.agg_in == nullptr;
    if (SH && a.sh.world > 1 && (a.probe_only || fused)) {
        // our count of every sample goes into every rank's count table (ours included), tagged with the batch's epoch
        if (sact)
            for (int r = q.gl; r < a.sh.world; r += q.L) a.sh.parts[r][s] = (a.sh.epoch << 5) | static_cast<unsigned>(local_agg);
    }
    if (a.probe_only) {
        if (!(SH && a.sh.world > 1) && q.gl == 0 && sact) a.agg_out[s] = static_cast<uint8_t>(local_agg);
        return;
    }

    // which resident row answers a key does not depend on agg_hit (the approximate substitution excepted)
    uint8_t hc = kHitMiss;
    int src_t = -1;
    unsigned src_s = 0;
    if (act) {
        if (h0) {                                                      // C1 serves (and overrides C2)
            hc = kHitC1;
            src_t = 0;
            src_s = slot0;
        } else if (c3hit) {
            hc = kHitC3;
            src_t = c3_tier;
            src_s = c3_slot;
        } else if (P1 != 0 && full && h1) {                            // C2 serves
            hc = kHitC2;
            src_t = 1;
            src_s = slot1;
        }
    }
    float *orow = sact ? out_row(a, p, s) : nullptr;
    const bool vec = out_vec_ok(a, D);
    const bool early = fused && !(P1 == 0 && p.approx_thres > 0);
    if (SH && early) {
        gather_tier<P0>(p, t0, 0, src_t, src_s, orow, sact, T, D, vec, q, &s_lut);
        if (P1 != 0) gather_tier<(P1 != 0 ? P1 : 32)>(p, t1, 1, src_t, src_s, orow, sact, T, D, vec, q, &s_lut);
    }

    if (a.agg_in != nullptr) {
        if (sact) agg = a.agg_in[s];
    } else if (SH && a.sh.world > 1) {
        // exact groupability: agg_hit = sum over the ranks of their local hit counts
        // every sample waits for ITS counts only: the peers' warps that serve the same sample run at about the same
        // time, so the words are usually there once the early gather above is done
        const unsigned long long tw0 = gtime();
        int v = 0;
        if (sact)
            for (int r = q.gl; r < a.sh.world; r += q.L) {
                const volatile unsigned *e = a.sh.my_parts + static_cast<size_t>(r) * a.B + s;
                unsigned x = *e;
                while ((x >> 5) != a.sh.epoch) {
                    if (gtime() - tw0 > kPeerTimeoutNs) {
                        set_error(p, 7u);
                        x = a.sh.epoch << 5;
                        break;
                    }
                    x = *e;
                }
                v += static_cast<int>(x & 31u);
            }
        __syncwarp();
        if (blockIdx.x == 0 && threadIdx.x == 0) p.dbg[30] += gtime() - tw0;      // CTA 0, warp 0: its wait for the peers' counts
        agg = grp_sum(v, q.L);
    }
    const bool approx = (P1 == 0) && (p.approx_thres > 0) && (agg >= p.approx_thres) && (m_h0 != 0u);
    // LRU (cache_algo/LRU.py): one recency ring (bucket 0); every hit moves its key to the MRU end (:30)
    const bool lru = (P1 == 0) && (p.policy == 1);
    // LFU (cache_algo/LFU.py): bucket = frequency - 1; a hit moves its key to the next frequency list (saturating at the last
    // one), a miss enters list 1 -- the bucket is a property of the key, not of the sample (oracle.lru.BatchLFU)
    const bool lfu = (P1 == 0) && (p.policy == 2);
    const int bkt = (lru || lfu) ? 0 : agg;

    uint8_t f = 0;
    const int pos = s * T + tbl;
    if (act) {
        if (hc == kHitC1) {
            if (lfu) {
                f = static_cast<uint8_t>(min(meta_bucket(m0) + 1, t0.n_buckets - 1) + 1);
                p.pos_slot[pos] = slot0;
            } else if (lru || meta_bucket(m0) < agg) {
                f = static_cast<uint8_t>(bkt + 1);
                p.pos_slot[pos] = slot0;
            }
        } else if (hc == kHitC3) {
        } else if (hc == kHitC2) {
            if (meta_bucket(m1) < agg) {
                f = static_cast<uint8_t>(kFlagTier | (agg + 1));
                p.pos_slot[pos] = slot1;
            }
        } else if (approx) {                                           // EvLFU_C1.py:140-152
            hc = kHitApprox;
            src_t = 0;
        } else {
            // fetch and insert.  C1 not full: everything goes to C1 (evlfu_8.cpp:590-602).  C1 full:
            // odd tables to C1, even to C2 while agg < high_agghit_threshold, else all to C2 (:573-588).
            int tier_ins = 0;
            if (P1 != 0 && full) tier_ins = (agg < p.high_thres && (gtbl & 1)) ? 0 : 1;
            f = static_cast<uint8_t>(kFlagMiss | (tier_ins ? kFlagTier : 0) | (bkt + 1));
        }
        p.flags[pos] = f;
        if (a.hit != nullptr) a.hit[pos] = hc;
    } else if (absent) {
        p.flags[pos] = 0;
        if (a.hit != nullptr) a.hit[pos] = kHitAbsent;
    }
    if (P1 == 0 && p.approx_thres > 0) {
        // value of the latest earlier hit in table order, else of the first hit
        const unsigned gm = m_h0 >> q.base;
        const unsigned lower = gm & ((1u << q.gl) - 1u);
        const int jj = lower ? (31 - __clz(lower)) : (gm ? __ffs(gm) - 1 : 0);
        const unsigned subst = __shfl_sync(kFull, slot0, q.base + jj);
        if (hc == kHitApprox) src_s = subst;
    }

    const unsigned m_f0 = __ballot_sync(kFull, f != 0 && !(f & kFlagTier)) & q.mask;
    const unsigned m_p1 = __ballot_sync(kFull, (f & kFlagTier) != 0 && !(f & kFlagMiss)) & q.mask;
    const unsigned m_i1 = __ballot_sync(kFull, (f & kFlagTier) != 0 && (f & kFlagMiss) != 0) & q.mask;
    const unsigned m_miss = __ballot_sync(kFull, (f & kFlagMiss) != 0) & q.mask;
    const unsigned m_c2 = __ballot_sync(kFull, hc == kHitC2) & q.mask;
    const unsigned m_ap = __ballot_sync(kFull, hc == kHitApprox) & q.mask;
    const unsigned m_abs = __ballot_sync(kFull, absent) & q.mask;
    // compact miss list for the fetch role of k_evict: one atomic per sample that missed anything, issued here so that
    // its round trip hides behind the gather below
    unsigned mbase = 0;
    if (q.gl == 0 && sact && m_miss) mbase = atomicAdd(p.miss_ctl, static_cast<unsigned>(__popc(m_miss)));
    if (q.gl == 0 && sact) {
        a.agg_out[s] = static_cast<uint8_t>(agg);
        if (m_f0 && !lfu) atomicAdd(&s_hist[bkt], static_cast<unsigned>(__popc(m_f0)));
        if (m_p1) atomicAdd(&s_hist[kMaxBuckets + agg], static_cast<unsigned>(__popc(m_p1)));
        if (m_i1) atomicAdd(&s_hist[2 * kMaxBuckets + agg], static_cast<unsigned>(__popc(m_i1)));
        if (m_h0) atomicAdd(&s_stat[0], static_cast<unsigned>(__popc(m_h0)));
        if (m_c2) atomicAdd(&s_stat[1], static_cast<unsigned>(__popc(m_c2)));
        if (m_c3) atomicAdd(&s_stat[2], static_cast<unsigned>(__popc(m_c3)));
        if (m_ap) atomicAdd(&s_stat[3], static_cast<unsigned>(__popc(m_ap)));
        if (m_miss) atomicAdd(&s_stat[4], static_cast<unsigned>(__popc(m_miss)));
        if (agg == p.n_perfect_agg) atomicAdd(&s_stat[5], 1u);
        if (m_abs) atomicAdd(&s_stat[6], static_cast<unsigned>(__popc(m_abs)));
    }

    if (lfu && f != 0) atomicAdd(&s_hist[(f & 0x3Fu) - 1u], 1u);       // LFU: the appends of a sample go to different buckets

    if (!(SH && early)) {
        gather_tier<P0>(p, t0, 0, src_t, src_s, orow, sact, T, D, vec, q, &s_lut);
        if (P1 != 0) gather_tier<(P1 != 0 ? P1 : 32)>(p, t1, 1, src_t, src_s, orow, sact, T, D, vec, q, &s_lut);
    }

    {
        mbase = __shfl_sync(kFull, mbase, q.base);
        if (f & kFlagMiss)
            p.miss_list[mbase + __popc(m_miss & ((1u << lane) - 1u))] = static_cast<unsigned>(pos) | ((f & kFlagTier) ? 0x80000000u : 0u);
    }

    __syncthreads();
    const int n_seq = (p.n_tiers == 1) ? kMaxBuckets : kSeqs;
    if (threadIdx.x < n_seq) {
        const unsigned v = s_hist[threadIdx.x];
        p.hist[static_cast<size_t>(threadIdx.x) * p.n_chunks_max + blockIdx.x] = v;
        if (v) atomicAdd(&p.tot[threadIdx.x], v);
    }
    if (threadIdx.x == 0) {
        const unsigned long long t_end = gtime();
        atomicMax(&p.dbg[1], t_end);
        GlobalCtl *g = p.g;
        const int ns = min(spc, B - s0);
        atomicAdd(&g->lookups, static_cast<unsigned long long>(ns) * T - s_stat[6]);
        atomicAdd(&g->samples, static_cast<unsigned long long>(ns));
        if (s_stat[0]) atomicAdd(&g->hits[0], static_cast<unsigned long long>(s_stat[0]));
        if (s_stat[1]) atomicAdd(&g->hits[1], static_cast<unsigned long long>(s_stat[1]));
        if (s_stat[2]) atomicAdd(&g->c3_hits, static_cast<unsigned long long>(s_stat[2]));
        if (s_stat[3]) atomicAdd(&g->approx_subst, static_cast<unsigned long long>(s_stat[3]));
        if (s_stat[4]) atomicAdd(&g->misses, static_cast<unsigned long long>(s_stat[4]));
        if (s_stat[5]) {
            atomicAdd(&g->perfect_hits, static_cast<unsigned long long>(s_stat[5]));
            if (p.policy != 2) t0.ctl->any_perfect = 1u;           // EvLFU_C1.py:163-165 (LFU has no perfect-item bookkeeping)
            if (P1 != 0 && full) t1.ctl->any_perfect = 1u;         // evlfu_8.cpp:439-441 (only when C2 is updated)
        }
    }
}

// ---- k_scan ------------------------------------------------------------------------------
// hist[seq][chunk] (append requests of serve-CTA `chunk` for sequence seq) -> offset of that
// chunk's first record inside the sequence.  One CTA per (group, bucket).
__global__ void __launch_bounds__(256) k_scan(const __grid_constant__ Params p) {
    __shared__ unsigned s_w[8];
    griddep_launch(p);
    griddep_wait(p);
    const int B = p.args->B;
    const int n_chunks = (B + p.spc - 1) / p.spc;
    if (n_chunks <= p.quad_max) return;                          // k_update sums its predecessors' counts itself
    const int nb = p.tier[0].n_buckets;
    const int grp = blockIdx.x / nb, b = blockIdx.x - grp * nb;
    unsigned *h = p.hist + static_cast<size_t>(grp * kMaxBuckets + b) * p.n_chunks_max;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned running = 0;
    for (int base = 0; base < n_chunks; base += 256) {
        const int i = base + threadIdx.x;
        const unsigned v = (i < n_chunks) ? h[i] : 0u;
        unsigned incl = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned n = __shfl_up_sync(kFull, incl, d);
            if (lane >= d) incl += n;
        }
        if (lane == 31) s_w[warp] = incl;
        __syncthreads();
        unsigned woff = 0, tot = 0;
#pragma unroll
        for (int w = 0; w < 8; ++w) {
            const unsigned x = s_w[w];
            if (w < warp) woff += x;
            tot += x;
        }
        if (i < n_chunks) h[i] = running + woff + incl - v;
        running += tot;
        __syncthreads();
    }
}

// ---- k_update ----------------------------------------------------------------------------
// Claim a slot for `key` (or find the slot a same-batch duplicate already claimed).  Only inserts
// run concurrently here, so the key field goes EMPTY -> occupied monotonically and every thread
// inserting the same key converges on one slot.  pass bits of the word may change under us
// (other claimers crossing), hence the CAS retry on the same slot.
__device__ __forceinline__ unsigned claim_slot(const TierDev &tier, unsigned long long key, bool &claimed) {
    const unsigned mask = tier.hash_mask;
    const unsigned home = hash_key(key, mask);
    unsigned i = home;
    claimed = false;
    while (true) {
        // look at 4 slots per round trip (L2-coherent loads: other claimers write these words)
        unsigned long long kw[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) kw[k] = __ldcg(&tier.slots[(i + k) & mask].kw);
        int k = 0;
        for (; k < 4; ++k) {
            unsigned long long cur = kw[k];
            const unsigned j = (i + k) & mask;
            bool done = false;
            while (true) {
                const unsigned long long kk = cur & kKeyMask;
                if (kk == key) {
                    done = true;
                    break;
                }
                if (kk != kEmptyKey) break;                       // someone else's key: next slot
                const unsigned long long old = atomicCAS(&tier.slots[j].kw, cur, (cur & ~kKeyMask) | key);
                if (old == cur) {
                    claimed = true;
                    done = true;
                    break;
                }
                cur = old;                                          // pass bits moved or the slot got taken: re-examine
            }
            if (done) {
                i = j;
                break;
            }
        }
        if (k < 4) break;
        i = (i + 4) & mask;
    }
    if (claimed) {
        // 16 bits of pass: a 65 535-key probe cluster cannot form at the <= 1/3 load factor used here
        for (unsigned j = home; j != i; j = (j + 1) & mask) atomicAdd(&tier.slots[j].kw, kPassOne);
    }
    return i;
}

// ---- k_evict ---------------------------------------------------------------------------
__device__ __forceinline__ void evict_slot(const TierDev &tier, unsigned slot, unsigned long long key) {
    const unsigned mask = tier.hash_mask;
    for (unsigned j = hash_key(key, mask); j != slot; j = (j + 1) & mask) atomicAdd(&tier.slots[j].kw, ~kPassOne + 1ull);
    tier.slots[slot].meta = 0ull;
    atomicOr(&tier.slots[slot].kw, kEmptyKey);        // keep the pass bits: other keys may cross this slot
}

// Per-tier eviction state of the evicting CTA (a copy of the bucket heads / tails / counts that
// is written back once at the end).
__device__ unsigned long long p_dbg_appends;      // ring records appended (cumulative, debug)
__device__ unsigned long long p_dbg_scanned;      // ring records examined by evictions (cumulative, debug)
struct EvictShared {
    unsigned long long head[kMaxBuckets];      // first record that may still be live
    unsigned long long cur[kMaxBuckets];       // scan cursor (>= head)
    unsigned long long tail[kMaxBuckets];
    unsigned long long kept[kMaxBuckets];      // first live record left in place by this call (~0: none)
    unsigned count[kMaxBuckets];
    // one window
    int seg_b[kMaxBuckets];
    unsigned long long seg_q0[kMaxBuckets];
    unsigned seg_off[kMaxBuckets + 1];
    unsigned seg_taken[kMaxBuckets];
    int n_seg;
    unsigned wsum[33];
};

// Pop up to `want` live records in (bucket, FIFO) order from buckets b_lo..b_hi (whole CTA).  One
// window of blockDim.x * R ring records can span several sparsely filled buckets, so the cost is
// a function of the records scanned, not of the buckets visited.  The protected slot is skipped
// but keeps its place.  Returns the number popped (uniform across the CTA).
__device__ unsigned pop_range(const TierDev &tier, EvictShared &S, int b_lo, int b_hi, unsigned want, unsigned prot_slot,
                              unsigned long long *out_keys, unsigned out_base) {
    constexpr int R = kEvictPerThread;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    const unsigned W = blockDim.x * R;
    unsigned got = 0;
    while (got < want) {
        __syncthreads();
        if (warp == 0) {
            // lane = bucket: unscanned ring length of every bucket in range, clipped so that the
            // window holds at most W records; buckets without live entries are skipped for good
            const int b = lane;
            const bool in = b >= b_lo && b <= b_hi;
            unsigned long long len = 0;
            if (in) {
                if (S.count[b] == 0) S.cur[b] = S.tail[b];
                len = S.tail[b] - S.cur[b];
            }
            const unsigned l32 = len > W ? W : static_cast<unsigned>(len);
            unsigned incl = l32;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const unsigned n = __shfl_up_sync(kFull, incl, d);
                if (lane >= d) incl += n;
            }
            const unsigned excl = incl - l32;
            const unsigned take = excl >= W ? 0u : (l32 < W - excl ? l32 : W - excl);
            const unsigned has = __ballot_sync(kFull, take > 0);
            const int si = __popc(has & ((1u << lane) - 1u));
            if (take > 0) {
                S.seg_b[si] = b;
                S.seg_q0[si] = S.cur[b];
                S.seg_off[si] = excl;
                S.seg_taken[si] = 0;
            }
            const unsigned total_take = __shfl_sync(kFull, incl < W ? incl : W, 31);
            if (lane == 0) {
                const int n = __popc(has);
                S.seg_off[n] = total_take;
                S.n_seg = n;
            }
        }
        __syncthreads();
        const int n_seg = S.n_seg;
        if (n_seg == 0) break;
        const unsigned n_rec = S.seg_off[n_seg];
        unsigned slot[R];
        unsigned long long q[R];
        int seg[R];
        uint4 sv[R];
        bool live[R], cand[R];
        const unsigned v0 = threadIdx.x * R;
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const unsigned v = v0 + r;
            slot[r] = kNoSlot;
            seg[r] = 0;
            q[r] = 0;
            if (v < n_rec) {
                int sg = 0;
                while (sg + 1 < n_seg && S.seg_off[sg + 1] <= v) ++sg;
                seg[r] = sg;
                q[r] = S.seg_q0[sg] + (v - S.seg_off[sg]);
                const unsigned *ring = tier.ring + static_cast<size_t>(S.seg_b[sg]) * tier.ring_cap;
                slot[r] = __ldcg(ring + (q[r] & (tier.ring_cap - 1)));
            }
        }
#pragma unroll
        for (int r = 0; r < R; ++r)
            if (slot[r] <= tier.hash_mask) sv[r] = __ldcg(reinterpret_cast<const uint4 *>(tier.slots + slot[r]));
        unsigned mycnt = 0;
#pragma unroll
        for (int r = 0; r < R; ++r) {
            live[r] = (slot[r] <= tier.hash_mask) && (u64_of(sv[r].z, sv[r].w) == pack_meta(S.seg_b[seg[r]], q[r]));
            cand[r] = live[r] && (slot[r] != prot_slot);
            mycnt += cand[r] ? 1u : 0u;
        }
        unsigned incl = mycnt;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned n = __shfl_up_sync(kFull, incl, d);
            if (lane >= d) incl += n;
        }
        if (lane == 31) S.wsum[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            const unsigned x = (lane < nwarp) ? S.wsum[lane] : 0u;
            unsigned wi = x;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const unsigned n = __shfl_up_sync(kFull, wi, d);
                if (lane >= d) wi += n;
            }
            S.wsum[lane] = wi - x;
            if (lane == 31) S.wsum[32] = wi;
        }
        __syncthreads();
        unsigned idx = S.wsum[warp] + incl - mycnt;
        const unsigned total = S.wsum[32];
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const bool take = cand[r] && (got + idx < want);
            if (take) {
                const unsigned long long key = u64_of(sv[r].x, sv[r].y) & kKeyMask;
                evict_slot(tier, slot[r], key);
                if (out_keys != nullptr) out_keys[out_base + got + idx] = key;
            }
            // victims per segment, one shared-memory atomic per warp and segment
            unsigned pending = __ballot_sync(kFull, take);
            while (pending) {
                const int leader = __ffs(pending) - 1;
                const int sg = __shfl_sync(kFull, seg[r], leader);
                const unsigned same = __ballot_sync(kFull, take && seg[r] == sg);
                if (lane == leader) atomicAdd(&S.seg_taken[sg], static_cast<unsigned>(__popc(same)));
                pending &= ~same;
            }
            // first live record left in place, per bucket; the plain pre-check keeps the same-address
            // shared-memory atomics to a handful per bucket (benign race: atomicMin decides)
            if (live[r] && !take && q[r] < *reinterpret_cast<volatile unsigned long long *>(&S.kept[S.seg_b[seg[r]]]))
                atomicMin(&S.kept[S.seg_b[seg[r]]], q[r]);
            idx += cand[r] ? 1u : 0u;
        }
        __syncthreads();
        if (threadIdx.x == 0) atomicAdd(&p_dbg_scanned, static_cast<unsigned long long>(n_rec));
        if (threadIdx.x < n_seg) {
            const int b = S.seg_b[threadIdx.x];
            S.cur[b] = S.seg_q0[threadIdx.x] + (S.seg_off[threadIdx.x + 1] - S.seg_off[threadIdx.x]);
            S.count[b] -= S.seg_taken[threadIdx.x];
        }
        got += min(total, want - got);
    }
    __syncthreads();
    return got;
}

// Flush rule, then evict down to capacity (whole CTA).
__device__ void evict_tier(const TierDev &tier, const Params &p) {
    __shared__ EvictShared S;
    __shared__ unsigned s_size;
    volatile TierCtl *c = tier.ctl;
    const int top = tier.n_buckets - 1;
    __syncthreads();
    if (threadIdx.x < kMaxBuckets) {
        const int b = threadIdx.x;
        const bool in = b < tier.n_buckets;
        S.head[b] = in ? c->head[b] : 0ull;
        S.cur[b] = S.head[b];
        S.tail[b] = in ? c->tail[b] : 0ull;
        S.kept[b] = ~0ull;
        const unsigned cnt = in ? c->count[b] : 0u;
        S.count[b] = cnt;
        unsigned sum = cnt;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) sum += __shfl_xor_sync(kFull, sum, d);
        if (b == 0) s_size = sum;
    }
    const unsigned n_new = c->n_new;
    const unsigned long long prot = c->prot;
    const unsigned n_perfect = c->n_perfect;
    const unsigned any_perfect = c->any_perfect;
    __syncthreads();
    unsigned size = s_size;

    // flush rule (EvLFU_C1.py:36-44, evlfu_32.cpp:209-218): bucket `top` is trimmed FIFO
    unsigned flushed = 0;
    unsigned new_n_perfect = n_perfect;
    if (n_new > 0 && n_perfect >= tier.max_perfect) {
        const unsigned want = min(tier.flush_n, S.count[top]);
        flushed = pop_range(tier, S, top, top, want, kNoSlot, tier.flushed, 0);
        size -= flushed;
        new_n_perfect = S.count[top];
        // records the flush scanned but kept stay ahead of later scans
        if (threadIdx.x == 0) {
            if (S.kept[top] != ~0ull) S.cur[top] = S.kept[top];
            S.head[top] = S.cur[top];
            S.kept[top] = ~0ull;
        }
        __syncthreads();
    }

    // evict down to capacity, lowest bucket first, FIFO inside a bucket; the highest ranked
    // new key is never the victim (the reference evicts before it inserts)
    unsigned prot_slot = kNoSlot;
    if (n_new > 0) prot_slot = evs::prot_slot(prot);
    const unsigned need = size > tier.cap ? size - tier.cap : 0u;
    unsigned ev = 0;
    if (need > 0) ev = pop_range(tier, S, 0, top, need, prot_slot, tier.evicted, 0);
    size -= ev;

    if (threadIdx.x < tier.n_buckets) {
        const int b = threadIdx.x;
        c->head[b] = (S.kept[b] != ~0ull) ? S.kept[b] : S.cur[b];
        c->count[b] = S.count[b];
    }
    if (threadIdx.x == 0) {
        c->n_perfect = any_perfect ? S.count[top] : new_n_perfect;      // EvLFU_C1.py:163-165
        c->stat_evictions += ev;
        c->stat_flushed += flushed;
        c->n_evicted_last = ev;
        c->n_flushed_last = flushed;
        c->full_at_start = (size >= tier.cap) ? 1u : 0u;
        c->n_new = 0;
        c->prot = 0ull;
        c->any_perfect = 0;
        if (ev < need) c->error = 4u;
    }
    __syncthreads();
}

// ---- k_compact ---------------------------------------------------------------------------
// Rewrites bucket b's ring so that [head, tail) holds only live records, order preserved.
__global__ void __launch_bounds__(1024) k_compact(TierDev tier, int b) {
    __shared__ unsigned s_wsum[32];
    __shared__ unsigned s_total;
    TierCtl *c = tier.ctl;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    const unsigned long long h = c->head[b], tl = c->tail[b];
    unsigned long long dst = h;
    unsigned *ring = tier.ring + static_cast<size_t>(b) * tier.ring_cap;
    for (unsigned long long base = h; base < tl; base += blockDim.x) {
        const unsigned long long q = base + threadIdx.x;
        bool valid = false;
        unsigned slot = kNoSlot;
        if (q < tl) {
            slot = ring[q & (tier.ring_cap - 1)];
            if (slot <= tier.hash_mask) valid = (tier.slots[slot].meta == pack_meta(b, q));
        }
        const unsigned bal = __ballot_sync(kFull, valid);
        if (lane == 0) s_wsum[warp] = __popc(bal);
        __syncthreads();                    // also: every record of this window has been read
        if (warp == 0) {
            const unsigned v = (lane < nwarp) ? s_wsum[lane] : 0u;
            unsigned incl = v;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const unsigned n = __shfl_up_sync(kFull, incl, d);
                if (lane >= d) incl += n;
            }
            s_wsum[lane] = incl - v;
            if (lane == 31) s_total = incl;
        }
        __syncthreads();
        if (valid) {
            const unsigned long long nq = dst + s_wsum[warp] + __popc(bal & ((1u << lane) - 1u));
            ring[nq & (tier.ring_cap - 1)] = slot;
            tier.slots[slot].meta = pack_meta(b, nq);
        }
        dst += s_total;
        __syncthreads();
    }
    if (threadIdx.x == 0) c->tail[b] = dst;
}

// ---- one-time initialisation --------------------------------------------------------------
__global__ void k_init_tier(TierDev tier) {
    const size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
    const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
    for (size_t j = i; j <= tier.hash_mask; j += stride) {
        tier.slots[j].kw = kEmptyKey;
        tier.slots[j].meta = 0ull;
    }
    if (i < kMaxBuckets) tier.ctl->kept[i] = ~0ull;
}

}  // namespace evs
