// evs_update_rows: new fp32 values for the rows of n keys, written into the backing store at every precision the handle
// has and into every resident slab copy, between two batches.
//
//   k_update_rows_claim  a thread per key: validates the key and records, in a scratch hash of the call's keys, the last
//                        position at which it occurs (atomicMax), so that duplicates resolve to their last occurrence
//   k_update_rows        a group of lanes per key (8 elements per lane and round, as the fetch role shares a row): the
//                        winning occurrence validates its values at every quantised precision, then encodes them and
//                        writes the store row(s) and the slab row of every tier the key is resident in
// Only bytes move: no TierCtl, slot meta, ring or C3 word is touched, so every policy decision stays what it would have
// been without the call.  Rows are written with exactly row_bytes bytes (packed rows need not be 16-byte aligned, and a
// wider read-modify-write would race with the writer of the neighbouring row).
#pragma once
#include "evs_kernels.cuh"

namespace evs {

constexpr int kRefreshThreads = 256;
constexpr uint8_t kWhereC1 = 1, kWhereC2 = 2, kWhereStore = 4, kWhereRejected = 0x80;
constexpr unsigned long long kRefreshEmpty = ~0ull;    // no key of the library's format has all bits set

struct RefreshArgs {
    const long long *keys;                 // [n] (global table << 40) | row
    long long n;
    const float *values;                   // [n] rows of D floats, vstride floats apart
    long long vstride;
    uint8_t *where;                        // [n] outcome bits, or null
    unsigned long long *hkey;              // [hmask + 1] scratch hash: keys of this call (kRefreshEmpty = free)
    long long *hpos;                       // [hmask + 1] last position of that key (-1 before the claim)
    unsigned hmask;
    int gsize;                             // lanes per key: next_pow2(ceil(D / 8)), at most 32
};

// Local table of a key, or -1 when its table is not served here or its row is outside [0, rows[table]).
__device__ __forceinline__ int refresh_table(const Params &p, long long key, long long &row) {
    row = key & ((1ll << kKeyShift) - 1);
    if (key < 0 || (key >> kKeyShift) >= kMaxTables) return -1;
    const int t = p.loc[key >> kKeyShift];
    if (t < 0 || row >= __ldg(p.rows + t)) return -1;
    return t;
}

__device__ __forceinline__ unsigned refresh_find(const RefreshArgs &a, long long key) {
    unsigned j = hash_key(static_cast<unsigned long long>(key), a.hmask);
    while (a.hkey[j] != static_cast<unsigned long long>(key)) j = (j + 1) & a.hmask;
    return j;
}

__global__ void __launch_bounds__(kRefreshThreads) k_update_rows_claim(const __grid_constant__ Params p, const __grid_constant__ RefreshArgs a) {
    const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < a.n; i += stride) {
        const long long key = a.keys[i];
        long long row;
        if (refresh_table(p, key, row) < 0) {
            set_error(p, 1u);                  // EVS_ERR_INDEX, as a lookup with a bad index
            continue;
        }
        unsigned j = hash_key(static_cast<unsigned long long>(key), a.hmask);
        while (true) {
            const unsigned long long prev = atomicCAS(a.hkey + j, kRefreshEmpty, static_cast<unsigned long long>(key));
            if (prev == kRefreshEmpty || prev == static_cast<unsigned long long>(key)) {
                atomicMax(a.hpos + j, i);
                break;
            }
            j = (j + 1) & a.hmask;
        }
    }
}

// Encode up to 8 elements (raw fp32 bits x[0 .. ne-1]) at PREC bits into the first PREC bytes of w.  False if one of
// them cannot be stored at this precision.
template <int PREC>
__device__ __forceinline__ bool encode_unit(const unsigned (&x)[8], int ne, unsigned (&w)[8]) {
    bool ok = true;
#pragma unroll
    for (int k = 0; k < 8; ++k) w[k] = (PREC == 32) ? x[k] : 0u;     // 32 bits: every pattern as given, NaN included
    if constexpr (PREC != 32) {
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            if (e >= ne) break;
            const float v = __uint_as_float(x[e]);
            unsigned q = 0;
            if (PREC == 16) {
                ok = enc16(v, q) && ok;
                w[e >> 1] |= q << (16 * (e & 1));
            } else if (PREC == 8) {
                ok = enc8(v, q) && ok;
                w[e >> 2] |= q << (8 * (e & 3));
            } else {
                ok = enc4(v, q) && ok;
                w[0] |= q << (8 * (e >> 1) + ((e & 1) ? 0 : 4));      // element 2k in the high nibble of byte k
            }
        }
    }
    return ok;
}

// Store the first nb bytes of w at dst, with the widest stores dst's alignment allows and never a byte past nb.
__device__ __forceinline__ void put_bytes(unsigned char *dst, const unsigned (&w)[8], int nb) {
    const uintptr_t ad = reinterpret_cast<uintptr_t>(dst);
    if ((ad & 15u) == 0 && (nb == 16 || nb == 32)) {
        reinterpret_cast<uint4 *>(dst)[0] = make_uint4(w[0], w[1], w[2], w[3]);
        if (nb == 32) reinterpret_cast<uint4 *>(dst)[1] = make_uint4(w[4], w[5], w[6], w[7]);
    } else if ((ad & 3u) == 0 && (nb & 3) == 0) {
#pragma unroll
        for (int k = 0; k < 8; ++k)
            if (4 * k < nb) reinterpret_cast<unsigned *>(dst)[k] = w[k];
    } else {
#pragma unroll
        for (int b = 0; b < 32; ++b)
            if (b < nb) dst[b] = static_cast<unsigned char>(w[b >> 2] >> (8 * (b & 3)));
    }
}

template <int PREC>
__device__ __forceinline__ void write_unit(const unsigned (&x)[8], int ne, int u, unsigned char *store_row, unsigned char *slab_row) {
    unsigned w[8];
    encode_unit<PREC>(x, ne, w);
    const int nb = ne * PREC / 8;
    put_bytes(store_row + u * PREC, w, nb);                     // unit u starts at element 8u = byte u * PREC
    if (slab_row != nullptr) put_bytes(slab_row + u * PREC, w, nb);
}

__device__ __forceinline__ void load_unit(const float *src, int ne, unsigned (&x)[8]) {
#pragma unroll
    for (int e = 0; e < 8; ++e) x[e] = (e < ne) ? __float_as_uint(__ldg(src + e)) : 0u;
}

template <int P0, int P1>
__global__ void __launch_bounds__(kRefreshThreads) k_update_rows(const __grid_constant__ Params p, const __grid_constant__ RefreshArgs a) {
    const int D = p.D, G = a.gsize, nu = (D + 7) >> 3;
    const int lane = threadIdx.x & 31, grp = lane / G, gl = lane - grp * G;
    const unsigned gmask = (G == 32) ? kFull : (((1u << G) - 1u) << (grp * G));
    const long long kpw = 32 / G;
    const long long gw = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const long long nw = (static_cast<long long>(gridDim.x) * blockDim.x) >> 5;
    const TierDev &t0 = p.tier[0];
    const TierDev &t1 = p.tier[1];
    for (long long i0 = gw * kpw; i0 < a.n; i0 += nw * kpw) {           // uniform per warp: the ballot below sees every lane
        const long long i = i0 + grp;
        const bool on = i < a.n;
        const long long key = on ? a.keys[i] : -1;
        long long row = 0;
        const int t = on ? refresh_table(p, key, row) : -1;
        const bool win = t >= 0 && a.hpos[refresh_find(a, key)] == i;
        const float *src = a.values + i * a.vstride;
        bool ok = true;
        if (win && (P0 != 32 || P1 != 0)) {
            for (int u = gl; u < nu; u += G) {
                unsigned x[8], w[8];
                const int ne = min(8, D - 8 * u);
                load_unit(src + 8 * u, ne, x);
                ok = encode_unit<P0>(x, ne, w) && ok;
                if (P1 != 0) ok = encode_unit<(P1 != 0 ? P1 : 32)>(x, ne, w) && ok;
            }
        }
        ok = (__ballot_sync(kFull, !ok) & gmask) == 0u;
        uint8_t res = (t < 0 || (win && !ok)) ? kWhereRejected : 0;
        if (win && ok) {
            unsigned s0 = 0, s1 = 0;
            unsigned long long m;
            const bool h0 = probe(t0, static_cast<unsigned long long>(key), s0, m);
            const bool h1 = P1 != 0 && probe(t1, static_cast<unsigned long long>(key), s1, m);
            unsigned char *st0 = const_cast<unsigned char *>(t0.store[t]) + static_cast<size_t>(row) * t0.row_bytes;
            unsigned char *sl0 = h0 ? t0.slab + static_cast<size_t>(s0) * t0.row_stride : nullptr;
            unsigned char *st1 = nullptr, *sl1 = nullptr;
            if (P1 != 0) {
                st1 = const_cast<unsigned char *>(t1.store[t]) + static_cast<size_t>(row) * t1.row_bytes;
                sl1 = h1 ? t1.slab + static_cast<size_t>(s1) * t1.row_stride : nullptr;
            }
            for (int u = gl; u < nu; u += G) {
                unsigned x[8];
                const int ne = min(8, D - 8 * u);
                load_unit(src + 8 * u, ne, x);
                write_unit<P0>(x, ne, u, st0, sl0);
                if (P1 != 0) write_unit<(P1 != 0 ? P1 : 32)>(x, ne, u, st1, sl1);
            }
            res = kWhereStore | (h0 ? kWhereC1 : 0) | (h1 ? kWhereC2 : 0);
        }
        if (on && gl == 0 && a.where != nullptr) a.where[i] = res;
    }
}

}  // namespace evs
