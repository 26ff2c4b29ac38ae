// Bags on the cached path (evs_lookup_bags): pooling factor > 1, the lS_o / lS_i pairs of apply_emb
// (dlrm_s_pytorch_C1_C2_C3.py:191-223; the random data generator draws up to --num-indices-per-lookup = 10 indices per
// bag, dlrm_data_pytorch.py:961-1007).
//
// A batch of B samples whose bags hold at most P indices is looked up as B*P SLICES: slice s*P + j holds the j-th index
// of every table's bag of sample s (no key where the bag is shorter).  Each slice is a request group in the reference's
// sense -- its agg_hit counts the hits among its keys, its keys are promoted / inserted into bucket agg_hit -- so the
// policy kernels run unchanged on a batch of B*P groups (oracle: oracle.evlfu.expand_bags + BatchEvLFU).  The rows of
// the slices land in a staging buffer (hits by k_serve's gather, misses by the fetch role of k_evict, which finishes
// last), and k_bags_pool sums them per (sample, table) in ascending j with single fp32 adds -- the order of
// nn.EmbeddingBag(mode="sum").
//
// On a rank of a table-wise sharded cache (evs_shard_lookup_bags) the rank expands its own tables' bags of the whole
// global batch into the same B*P slices; a slice's agg_hit is the sum over the ranks of their counts (the count exchange
// of a plain batch, indexed by slice).  The slice rows stay in the local staging, and k_bags_pool pools where the rows are
// and sends the POOLED rows to the owner ranks' receive buffers: P times fewer NVLink bytes than sending slice rows.
#pragma once
#include "evs_kernels.cuh"

namespace evs {

constexpr int kMaxPerBag = 32;

// idx: int64 [nnz], off: int64 [T*B + 1] (bag (t, s) = idx[off[t*B+s] .. off[t*B+s+1])) -> idxv int64 [T][B*P], -1 = no key
__global__ void __launch_bounds__(256) k_bags_expand(const __grid_constant__ Params p, const long long *__restrict__ idx,
                                                     const long long *__restrict__ off, int B, int P, long long nnz,
                                                     long long *__restrict__ idxv) {
    const int T = p.T;
    const long long Bv = static_cast<long long>(B) * P;
    const long long total = Bv * T;
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int t = static_cast<int>(i / Bv);
        const long long v = i - t * Bv;
        const int s = static_cast<int>(v / P), j = static_cast<int>(v - static_cast<long long>(s) * P);
        const long long o0 = __ldg(off + static_cast<size_t>(t) * B + s), o1 = __ldg(off + static_cast<size_t>(t) * B + s + 1);
        long long n = o1 - o0;
        if (o0 < 0 || o1 > nnz || n < 0 || n > P) {         // malformed offsets or a bag larger than max_per_bag
            set_error(p, 1u);
            n = 0;
        }
        long long r = -1;
        if (j < n) {
            r = __ldg(idx + o0 + j);
            if (r < 0) {                                     // a negative index is an error here, not "no key"
                set_error(p, 1u);
                r = 0;
            }
        }
        idxv[i] = r;
    }
}

// rows_v fp32 [B*P][W][D], local table t at column p.col[t] (W = T on one GPU, n_tables_total on a sharded handle) ->
// out[s][col(t)][:] = sum_j rows_v[s*P + j][col(t)][:] over the bag's indices, j ascending;
// hit_v uint8 [B*P][T] -> hit_out[off[t*B+s] + j] (one code per index, aligned with idx).
// Sharded (sh.world > 1): B is the global batch and sample s goes to row s % Bl of rank s / Bl's receive buffer
// ([Bl][T_total][D], out is unused).  Then every CTA fences at system scope and arrives; the last one raises
// "rank `rank` has written its rows of epoch e" at every peer and holds the stream until every peer has said the same
// to us, as close_batch does for a plain batch.  After this kernel our receive buffer holds the pooled batch.
template <bool VEC>
__global__ void __launch_bounds__(256) k_bags_pool(const __grid_constant__ Params p, const __grid_constant__ ShardArgs sh,
                                                   const float *__restrict__ rows_v, const uint8_t *__restrict__ hit_v,
                                                   const long long *__restrict__ off, int B, int P, long long nnz, int W,
                                                   float *__restrict__ out, long long out_stride, uint8_t *__restrict__ hit_out) {
    __shared__ unsigned s_last;
    const int T = p.T, D = p.D;
    const int cpr = VEC ? (D >> 2) : D;                     // work items per row
    const long long total = static_cast<long long>(B) * T * cpr;
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int c = static_cast<int>(i % cpr);
        const long long st = i / cpr;
        const int t = static_cast<int>(st % T), s = static_cast<int>(st / T);
        const int col = p.col[t];
        const long long o0 = __ldg(off + static_cast<size_t>(t) * B + s);
        long long n = __ldg(off + static_cast<size_t>(t) * B + s + 1) - o0;
        if (o0 < 0 || n < 0 || n > P || o0 + n > nnz) n = 0;   // malformed: k_bags_expand raised EVS_ERR_INDEX
        const float *src = rows_v + (static_cast<size_t>(s) * P * W + col) * D;
        float *dst;
        if (sh.world > 1) {
            const int r = s / sh.Bl, ls = s - r * sh.Bl;
            dst = sh.recv[r] + (static_cast<size_t>(ls) * sh.T_total + col) * D;
        } else {
            dst = out + static_cast<size_t>(s) * out_stride + static_cast<size_t>(col) * D;
        }
        if (VEC) {
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
            for (int j = 0; j < n; ++j) {
                const float4 x = *reinterpret_cast<const float4 *>(src + static_cast<size_t>(j) * W * D + (c << 2));
                acc.x = __fadd_rn(acc.x, x.x);
                acc.y = __fadd_rn(acc.y, x.y);
                acc.z = __fadd_rn(acc.z, x.z);
                acc.w = __fadd_rn(acc.w, x.w);
            }
            *reinterpret_cast<float4 *>(dst + (c << 2)) = acc;
        } else {
            float acc = 0.f;
            for (int j = 0; j < n; ++j) acc = __fadd_rn(acc, src[static_cast<size_t>(j) * W * D + c]);
            dst[c] = acc;
        }
        if (c == 0 && hit_out != nullptr)
            for (int j = 0; j < n; ++j) hit_out[o0 + j] = hit_v[(static_cast<size_t>(s) * P + j) * T + t];
    }
    if (sh.world <= 1) return;
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence_system();                              // our pooled rows, stored into the peers' receive buffers
        const bool last = atomicAdd(&p.g->pool_arrived, 1u) == gridDim.x - 1;
        if (last) p.g->pool_arrived = 0u;                     // every CTA has arrived: reset for the next bags batch
        s_last = last ? 1u : 0u;
    }
    __syncthreads();
    if (s_last != 0u && threadIdx.x < 32) {
        const int lane = threadIdx.x;
        __threadfence_system();
        if (lane < sh.world) *reinterpret_cast<volatile unsigned *>(sh.out_flag[lane]) = sh.epoch;
        wait_flags(sh.my_out_flags, sh.world, sh.epoch, lane, p);
    }
}

}  // namespace evs
