// Alternative-key generation for C3 (SURVEY.md 8(f) rank 3): the offline step that produces the alt-key tables
// aprx_embedding.cpp serves from.  The reference does it in two notebooks
// (script/approximate_embedding/phase2_similarity_analysis/):
//   get_neighbors_GPU.ipynb      all embedding rows of all tables in ONE matrix, brute-force Euclidean k-NN with
//                                n_neighbors = 11 (cuML NearestNeighbors, algorithm='brute'); neighbour [0] -- the row
//                                itself -- is dropped, the other 10 are written as "table-row" (tables 1-based);
//   most_popular_neighbor.ipynb  of the 10, the one requested most often in the workload (first maximum; rows that never
//                                occur count 0) becomes the row's alternative key.
//
// k_knn -- fused distance + selection.  A CTA owns 128 query rows and walks a range of the database in tiles of 64 rows:
//   * dist(q, x) is ranked by |x|^2 - 2 q.x; the dot products of a 128 x 64 tile run on the tensor cores
//     (mma.sync.m16n8k8 TF32, warp w = query rows 16w .. 16w+15).  Operands are split hi + lo (hi = the value rounded to
//     TF32's mantissa with an integer add, lo = the exact remainder, which the tensor core truncates to TF32) and a product
//     is hi*hi + hi*lo + lo*hi, within 5 * 2^-22 of the exact product: a neighbour list is only as good as its near-ties,
//     and plain TF32 (10 mantissa bits) reorders them.  lo is not rounded: the rounding add carries a NaN's mantissa into
//     the sign bit (0x7FFFFFFF -> -0.0), so a NaN row would rank as a zero row.  Unrounded, lo is NaN for a NaN or +-Inf
//     element, every ranking value of its row (or query) is NaN and never passes a threshold: such a row is never a
//     neighbour, such a query gets none.  The split of a database tile is done ONCE, by the
//     thread that stages it (global -> registers -> hi / lo planes in shared memory, the next tile's loads in flight under
//     the current tile's math); the queries' split fragments live in registers for d <= 16;
//   * every thread keeps, for each of its two query rows, a sorted list (in shared memory) of the 11 best (distance, index)
//     pairs among the columns it sees; a candidate is first compared with the row's threshold -- the smallest of the worst
//     entries of the four lists of the row's quad -- so after the first tiles an element costs one FFMA and one compare.  At
//     the end the four lists of a query row (the accumulator layout spreads a row over a quad) are merged.
// With d = 16 there are only 2 x 16 multiply-adds per pair against ~4 selection instructions: the kernel is bound by the
// ALU work of the selection, not by the tensor pipe (which is why the 3x split is free) and not by HBM (a tile is read once
// per 128 queries).
// k_knn_merge -- merges the per-split lists of a query, drops entry [0], writes the k neighbours and, if asked, the
// most popular one as an alt key (alt_row * 100 + alt_table, tables 1-based: convert_altkeys_to_binary.py:50).
#pragma once
#include "evs_host.h"
#include "evs_interact.cuh"

namespace evs {

constexpr int kKnnQ = 128;                   // query rows per CTA
constexpr int kKnnT = 64;                    // database rows per tile
constexpr int kKnnSel = 11;                  // list length: the row itself + 10 neighbours (get_neighbors_GPU.ipynb)
constexpr int kKnnThreads = 256;
constexpr int kKnnMaxD = 64;

__device__ __forceinline__ unsigned tf32_rn(float v) { return (__float_as_uint(v) + 0x1000u) & 0xFFFFE000u; }

__device__ __forceinline__ bool knn_better(float a, int ia, float b, int ib) { return a < b || (a == b && ia < ib); }
// A thread's list of a query row: kKnnSel (distance, index) pairs in SHARED memory, sorted ascending.  Insertions are rare
// once the lists have warmed up (a candidate must beat the row's threshold first), so the insertion is one out-of-line
// routine: inlined at the 32 candidate sites of a tile, its unrolled register version was ~5000 instructions -- the kernel
// spent its time fetching them -- and 44 registers per thread.  Returns the list's new worst distance.
__device__ __noinline__ float knn_insert(float2 *list, float v, int i) {
    float2 last = list[kKnnSel - 1];
    if (!knn_better(v, i, last.x, __float_as_int(last.y))) return last.x;
    int p = kKnnSel - 1;
    while (p > 0) {
        const float2 e = list[p - 1];
        if (!knn_better(v, i, e.x, __float_as_int(e.y))) break;
        list[p] = e;
        --p;
    }
    list[p] = make_float2(v, __int_as_float(i));
    return list[kKnnSel - 1].x;
}

// x: database [n][D] fp32, q: queries [nq][D] fp32 (may alias x), part: [nq][splits][kKnnSel] (distance, index) pairs.
// KSR: k-steps of the queries' split fragments held in registers (2: d <= 16); 0: re-read from shared memory per tile.
template <int KSR>
__global__ void __launch_bounds__(kKnnThreads, 2) k_knn(const float *__restrict__ x, long long n, const float *__restrict__ q, long long nq,
                                                        int D, int Dp, int ld, long long rows_per_split, float2 *__restrict__ part) {
    extern __shared__ __align__(16) unsigned char s_raw[];
    // layout: lists[128 rows][4 threads of the row's quad][11] (distance, index) | Qhi[128][ld] Qlo[128][ld] | Xhi[64][ld] Xlo[64][ld] | norm[64]
    float2 *s_cand = reinterpret_cast<float2 *>(s_raw);
    unsigned *s_qhi = reinterpret_cast<unsigned *>(s_raw + static_cast<size_t>(kKnnQ) * 4 * kKnnSel * sizeof(float2));
    unsigned *s_qlo = s_qhi + kKnnQ * ld;
    unsigned *s_xhi = s_qlo + kKnnQ * ld;
    unsigned *s_xlo = s_xhi + kKnnT * ld;
    float *s_norm = reinterpret_cast<float *>(s_xlo + kKnnT * ld);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = lane >> 2, tq = lane & 3;
    const long long q0 = static_cast<long long>(blockIdx.x) * kKnnQ;
    const long long n0 = static_cast<long long>(blockIdx.y) * rows_per_split;
    const long long n1 = min(n, n0 + rows_per_split);
    const int d4 = Dp >> 2;                                  // float4 pieces per (padded) row

    // ---- queries: split once, into shared memory (zero rows past nq, zero columns past D) ------------------------------------
    for (int e = threadIdx.x; e < kKnnQ * Dp; e += kKnnThreads) {
        const int r = e / Dp, c = e - r * Dp;
        float v = 0.0f;
        if (q0 + r < nq && c < D) v = __ldg(q + (q0 + r) * D + c);
        const unsigned h = tf32_rn(v);
        s_qhi[r * ld + c] = h;
        s_qlo[r * ld + c] = __float_as_uint(v - __uint_as_float(h));      // exact; NaN for NaN / Inf (see the header)
    }
    __syncthreads();
    // A fragments of this warp's 16 query rows; logical k slots tq / tq + 4 of a k-step take columns k0 + 2 tq, k0 + 2 tq + 1
    constexpr bool AREG = KSR > 0;
    constexpr int KS = AREG ? KSR : 1;                       // k-steps held in registers
    unsigned ahi[KS][4], alo[KS][4];
    const unsigned *qh = s_qhi + (16 * warp + g) * ld + 2 * tq, *ql = s_qlo + (16 * warp + g) * ld + 2 * tq;
    if (AREG) {
#pragma unroll
        for (int ks = 0; ks < KS; ++ks) {
            if (ks * 8 < Dp) {
                const uint2 h0 = *reinterpret_cast<const uint2 *>(qh + ks * 8), h1 = *reinterpret_cast<const uint2 *>(qh + 8 * ld + ks * 8);
                const uint2 l0 = *reinterpret_cast<const uint2 *>(ql + ks * 8), l1 = *reinterpret_cast<const uint2 *>(ql + 8 * ld + ks * 8);
                ahi[ks][0] = h0.x, ahi[ks][1] = h1.x, ahi[ks][2] = h0.y, ahi[ks][3] = h1.y;
                alo[ks][0] = l0.x, alo[ks][1] = l1.x, alo[ks][2] = l0.y, alo[ks][3] = l1.y;
            } else {
#pragma unroll
                for (int i = 0; i < 4; ++i) ahi[ks][i] = alo[ks][i] = 0u;
            }
        }
    }

    // this thread's lists: rows 16 warp + g and 16 warp + g + 8; their worst distances are mirrored in registers
    float2 *list[2] = {s_cand + ((16 * warp + g) * 4 + tq) * kKnnSel, s_cand + ((16 * warp + g + 8) * 4 + tq) * kKnnSel};
    float worst[2];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        for (int i = 0; i < kKnnSel; ++i) list[r][i] = make_float2(__int_as_float(0x7f800000), __int_as_float(0x7fffffff));
        worst[r] = __int_as_float(0x7f800000);
    }

    // ---- staging: thread t owns float4 pieces t, t + 256, ... of a tile (64 rows x d4 pieces) ----------------------------------
    constexpr int PMAX = (KSR > 0 ? kKnnT * (KSR * 8 / 4) : kKnnT * (kKnnMaxD / 4)) / kKnnThreads;      // pieces per thread: 1 (d <= 16) or 4
    const int n_pieces = kKnnT * d4;
    const bool vec = ((D & 3) == 0) && ((reinterpret_cast<uintptr_t>(x) & 15u) == 0);
    float4 stage[PMAX];
    auto load_tile = [&](long long base) {
#pragma unroll
        for (int i = 0; i < PMAX; ++i) {
            const int e = threadIdx.x + i * kKnnThreads;
            stage[i] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (e < n_pieces) {
                const int r = e / d4, c4 = e - r * d4;
                const long long row = base + r;
                if (row < n1) {
                    if (vec) {
                        if ((c4 << 2) < D) stage[i] = __ldg(reinterpret_cast<const float4 *>(x + row * D) + c4);
                    } else {
                        float t[4];
#pragma unroll
                        for (int k = 0; k < 4; ++k) t[k] = ((c4 << 2) + k < D) ? __ldg(x + row * D + (c4 << 2) + k) : 0.0f;
                        stage[i] = make_float4(t[0], t[1], t[2], t[3]);
                    }
                }
            }
        }
    };
    // |x|^2 of a tile's rows: when a row's pieces sit in d4 neighbouring lanes (d4 = 2, 4, 8, 16) the lanes add up their pieces
    // in a fixed butterfly (the same x gets the same norm in every CTA: the ranking must not depend on who computed it), else
    // one thread per row walks the row in shared memory (hi + lo there is the value itself, or NaN for a NaN or Inf: the
    // norm is never finite for a non-finite row on either path).  Rows past the end of the range get +inf: never selected.
    const bool shfl_norm = (32 % d4) == 0;
    auto store_tile = [&](long long base) {
        __syncthreads();                                     // the previous tile's reads are over
#pragma unroll
        for (int i = 0; i < PMAX; ++i) {
            const int e = threadIdx.x + i * kKnnThreads;
            const bool on = e < n_pieces;
            const int r = on ? e / d4 : 0, c4 = on ? e - r * d4 : 0;
            const float v[4] = {stage[i].x, stage[i].y, stage[i].z, stage[i].w};
            uint4 h, l;
            unsigned *hp = &h.x, *lp = &l.x;
            float nn = 0.0f;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                hp[k] = tf32_rn(v[k]);
                lp[k] = __float_as_uint(v[k] - __uint_as_float(hp[k]));
                nn = fmaf(v[k], v[k], nn);
            }
            if (on) {
                *reinterpret_cast<uint4 *>(s_xhi + r * ld + (c4 << 2)) = h;
                *reinterpret_cast<uint4 *>(s_xlo + r * ld + (c4 << 2)) = l;
            }
            if (shfl_norm) {
                for (int o = 1; o < d4; o <<= 1) nn += __shfl_xor_sync(0xFFFFFFFFu, nn, o);
                if (on && c4 == 0) s_norm[r] = (base + r < n1) ? nn : __int_as_float(0x7f800000);
            }
        }
        __syncthreads();
        if (!shfl_norm) {
            if (threadIdx.x < kKnnT) {
                float nn = 0.0f;
                for (int c = 0; c < Dp; ++c) {
                    const float v = __uint_as_float(s_xhi[threadIdx.x * ld + c]) + __uint_as_float(s_xlo[threadIdx.x * ld + c]);
                    nn = fmaf(v, v, nn);
                }
                s_norm[threadIdx.x] = (base + threadIdx.x < n1) ? nn : __int_as_float(0x7f800000);
            }
            __syncthreads();
        }
    };

    long long base = n0;
    if (base < n1) load_tile(base);
    for (; base < n1; base += kKnnT) {
        store_tile(base);
        if (base + kKnnT < n1) load_tile(base + kKnnT);      // the next tile's loads fly under this tile's math
        float acc[kKnnT / 8][4];
#pragma unroll
        for (int j = 0; j < kKnnT / 8; ++j)
#pragma unroll
            for (int k = 0; k < 4; ++k) acc[j][k] = 0.0f;
        const unsigned *xh = s_xhi + g * ld + 2 * tq, *xl = s_xlo + g * ld + 2 * tq;
        if (AREG) {
#pragma unroll
            for (int ks = 0; ks < KS; ++ks) {
                if (ks * 8 < Dp) {
#pragma unroll
                    for (int j = 0; j < kKnnT / 8; ++j) {
                        const uint2 bh = *reinterpret_cast<const uint2 *>(xh + 8 * j * ld + ks * 8);
                        const uint2 bl = *reinterpret_cast<const uint2 *>(xl + 8 * j * ld + ks * 8);
                        mma_tf32(acc[j], ahi[ks][0], ahi[ks][1], ahi[ks][2], ahi[ks][3], bh.x, bh.y);
                        mma_tf32(acc[j], ahi[ks][0], ahi[ks][1], ahi[ks][2], ahi[ks][3], bl.x, bl.y);
                        mma_tf32(acc[j], alo[ks][0], alo[ks][1], alo[ks][2], alo[ks][3], bh.x, bh.y);
                    }
                }
            }
        } else {
            for (int k0 = 0; k0 < Dp; k0 += 8) {
                const uint2 h0 = *reinterpret_cast<const uint2 *>(qh + k0), h1 = *reinterpret_cast<const uint2 *>(qh + 8 * ld + k0);
                const uint2 l0 = *reinterpret_cast<const uint2 *>(ql + k0), l1 = *reinterpret_cast<const uint2 *>(ql + 8 * ld + k0);
#pragma unroll
                for (int j = 0; j < kKnnT / 8; ++j) {
                    const uint2 bh = *reinterpret_cast<const uint2 *>(xh + 8 * j * ld + k0);
                    const uint2 bl = *reinterpret_cast<const uint2 *>(xl + 8 * j * ld + k0);
                    mma_tf32(acc[j], h0.x, h1.x, h0.y, h1.y, bh.x, bh.y);
                    mma_tf32(acc[j], h0.x, h1.x, h0.y, h1.y, bl.x, bl.y);
                    mma_tf32(acc[j], l0.x, l1.x, l0.y, l1.y, bh.x, bh.y);
                }
            }
        }
        // ---- selection: |x|^2 - 2 q.x against the row's threshold -------------------------------------------------------------
        // A query row is spread over the four threads of a quad, each with its own list.  Whatever a thread's list holds, 11
        // candidates at or below its worst entry exist, so nothing above the SMALLEST of the quad's four worst entries can be
        // among the row's 11 best: one threshold per row and tile (two shuffles) cuts the insertions -- the divergent, expensive
        // part (ncu: 2/3 of the kernel's stall samples) -- by about four.
        float thr[2];
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            float w = worst[r];
            w = fminf(w, __shfl_xor_sync(0xFFFFFFFFu, w, 1));
            w = fminf(w, __shfl_xor_sync(0xFFFFFFFFu, w, 2));
            thr[r] = w;
        }
#pragma unroll
        for (int j = 0; j < kKnnT / 8; ++j) {
            const int c = 8 * j + 2 * tq;
            const float2 nn = *reinterpret_cast<const float2 *>(s_norm + c);
            const int id = static_cast<int>(base) + c;
            const float v0 = fmaf(-2.0f, acc[j][0], nn.x), v1 = fmaf(-2.0f, acc[j][1], nn.y);
            const float v2 = fmaf(-2.0f, acc[j][2], nn.x), v3 = fmaf(-2.0f, acc[j][3], nn.y);
            if (v0 <= thr[0]) worst[0] = knn_insert(list[0], v0, id);
            if (v1 <= thr[0]) worst[0] = knn_insert(list[0], v1, id + 1);
            if (v2 <= thr[1]) worst[1] = knn_insert(list[1], v2, id);
            if (v3 <= thr[1]) worst[1] = knn_insert(list[1], v3, id + 1);
        }
    }

    // ---- merge the four sorted lists of a query row (the quad's threads) ---------------------------------------------------------
    __syncthreads();
    if (threadIdx.x < kKnnQ && q0 + threadIdx.x < nq) {
        const float2 *c = s_cand + threadIdx.x * 4 * kKnnSel;
        int head[4] = {0, 0, 0, 0};
        float2 *out = part + ((q0 + threadIdx.x) * gridDim.y + blockIdx.y) * kKnnSel;
        for (int i = 0; i < kKnnSel; ++i) {
            int w = -1;
            float bd = 0.f;
            int bi = 0;
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                if (head[t] >= kKnnSel) continue;
                const float2 e = c[t * kKnnSel + head[t]];
                if (w < 0 || knn_better(e.x, __float_as_int(e.y), bd, bi)) {
                    w = t;
                    bd = e.x;
                    bi = __float_as_int(e.y);
                }
            }
            out[i] = make_float2(bd, __int_as_float(bi));
#pragma unroll
            for (int t = 0; t < 4; ++t)
                if (t == w) ++head[t];
        }
    }
}

// part [nq][splits][11] -> nbr [nq][k] (nearest first, entry [0] of the merged list dropped), dist [nq][k] or null (squared
// distances, |q|^2 added back), alt [nq] or null: the neighbour with the highest freq (first maximum) as an alt key.
__global__ void __launch_bounds__(256) k_knn_merge(const float2 *__restrict__ part, int splits, long long nq, int k, const float *__restrict__ q,
                                                   int D, long long *__restrict__ nbr, float *__restrict__ dist,
                                                   const unsigned *__restrict__ freq, const long long *__restrict__ table_off, int n_tables,
                                                   unsigned *__restrict__ alt) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= nq) return;
    const float2 *c = part + i * splits * kKnnSel;
    float qn = 0.0f;
    if (dist != nullptr)
        for (int e = 0; e < D; ++e) qn = fmaf(q[i * D + e], q[i * D + e], qn);
    // the lists are sorted: a (splits)-way merge, one head per split
    int best_alt = -1;
    unsigned best_f = 0;
    float last_d = -__int_as_float(0x7f800000);
    int last_i = -1;
    for (int o = 0; o <= k; ++o) {
        // smallest (distance, index) strictly after the last one taken
        float bd = __int_as_float(0x7f800000);
        int bi = 0x7fffffff;
        for (int e = 0; e < splits * kKnnSel; ++e) {
            const float2 v = c[e];
            const int vi = __float_as_int(v.y);
            if (!knn_better(last_d, last_i, v.x, vi)) continue;
            if (knn_better(v.x, vi, bd, bi)) bd = v.x, bi = vi;
        }
        last_d = bd;
        last_i = bi;
        if (o == 0) continue;                                 // the row itself (get_neighbors_GPU.ipynb drops indices[j][0])
        const bool none = bi == 0x7fffffff || !(bd < __int_as_float(0x7f800000));      // fewer than k + 1 rows in the database
        if (nbr != nullptr) nbr[i * k + (o - 1)] = none ? -1 : bi;
        if (dist != nullptr) dist[i * k + (o - 1)] = bd + qn;
        if (alt != nullptr && !none) {
            const unsigned f = freq != nullptr ? freq[bi] : 0u;
            if (best_alt < 0 || f > best_f) best_alt = bi, best_f = f;      // first maximum (most_popular_neighbor.ipynb: index(max))
        }
    }
    if (alt != nullptr) {
        unsigned key = 0u;
        if (best_alt >= 0) {
            int t = 0;
            while (t + 1 < n_tables && table_off[t + 1] <= best_alt) ++t;
            key = static_cast<unsigned>(best_alt - table_off[t]) * 100u + static_cast<unsigned>(t + 1);
        }
        alt[i] = key;
    }
}

inline int launch_knn(const float *x, long long n, const float *q, long long nq, int D, int k, long long *nbr, float *dist,
                      const unsigned *freq, const long long *table_off, int n_tables, unsigned *alt, float2 *part, int splits,
                      cudaStream_t st) {
    if (x == nullptr || q == nullptr || n < 1 || nq < 0 || D < 1 || D > kKnnMaxD || k < 1 || k > kKnnSel - 1 || n >= (1ll << 31) ||
        part == nullptr || splits < 1 || (alt != nullptr && (table_off == nullptr || n_tables < 1)))
        return EVS_ERR_INVALID;
    if (nq == 0) return EVS_OK;
    const int Dp = (D + 7) & ~7;
    const int ld = (Dp & 15) == 8 ? Dp : Dp + 8;             // = 8 mod 16: conflict-free 64-bit fragment reads
    const size_t smem = static_cast<size_t>(kKnnQ) * 4 * kKnnSel * 8 + static_cast<size_t>(2 * kKnnQ + 2 * kKnnT) * ld * 4 + kKnnT * 4;
    const long long tiles = (n + kKnnT - 1) / kKnnT;
    const long long rows_per_split = ((tiles + splits - 1) / splits) * kKnnT;
    const dim3 grid(static_cast<unsigned>((nq + kKnnQ - 1) / kKnnQ), static_cast<unsigned>(splits));
    auto fn = Dp <= 16 ? k_knn<2> : k_knn<0>;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
        if (e != cudaSuccess) {
            set_error(std::string("k_knn smem: ") + cudaGetErrorString(e));
            return EVS_ERR_CUDA;
        }
    }
    fn<<<grid, kKnnThreads, smem, st>>>(x, n, q, nq, D, Dp, ld, rows_per_split, part);
    EVS_CUDA(cudaGetLastError());
    k_knn_merge<<<static_cast<unsigned>((nq + 255) / 256), 256, 0, st>>>(part, splits, nq, k, q, D, nbr, dist, freq, table_off, n_tables, alt);
    EVS_CUDA(cudaGetLastError());
    return EVS_OK;
}

}  // namespace evs
