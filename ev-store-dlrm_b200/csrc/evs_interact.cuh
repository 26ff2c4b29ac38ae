// Pairwise-dot feature interaction (dlrm_s_pytorch_C1_C2_C3.py:625-658, op "dot",
// arch_interaction_itself = 0):  T = [x ; ly] in [B, n_f+1, d],  Z = T T^t  (torch.bmm at :632),
// R = [x, Z[i][j] for i > j in row-major order]  ->  [B, d + (n_f+1) n_f / 2].
//
// k_interact_mma -- the tensor-core path (n_f + 1 <= 32, d <= 128): one warp per sample.
//   * T is staged in shared memory with 128-bit loads (rows padded to 32, d padded to a multiple of 8, row stride
//     = 4 mod 8 floats so that the fragment reads below are bank-conflict free);
//   * Z = T T^t as 32x32xd on the tensor cores with mma.sync.m16n8k8 TF32: T serves as the row-major A operand and,
//     unchanged, as the "column-major" B operand (B[k][n] = T[n][k]), so a lane loads 8 values per k-step and uses
//     them for both.  Only the 6 of 8 accumulator tiles that touch the strict lower triangle are computed;
//   * fp32 accuracy from TF32 hardware: every operand is split hi + lo (hi = the value rounded to TF32's mantissa, lo = the
//     exact remainder, which the tensor core truncates to TF32) and a tile is the sum of hi*hi + hi*lo + lo*hi (the
//     "3xTF32" scheme: the dropped lo*lo term and lo's truncation are 5 * 2^-22 relative together).  NaN and Inf inputs
//     give NaN pairs (lo = v - hi is NaN for both); a finite value within 2^-11 of FLT_MAX rounds to hi = Inf and gives
//     NaN as well.  The kernel is bound by issue slots (7-11 FLOP/B), so the 3x tensor work is free;
//   * the accumulators go back through shared memory so that the 351 packed outputs are written as consecutive floats.
// k_interact (fp32 FMA) remains for shapes outside those limits.
#pragma once
#include "evs_host.h"

namespace evs {

constexpr int kInteractWarps = 4;            // at most; fewer when (n_f + 1) (d + 1) floats per warp do not fit 4 times

__global__ void __launch_bounds__(kInteractWarps * 32) k_interact(const float *__restrict__ x, const float *__restrict__ ly,
                                                                  float *__restrict__ r, int B, int n_f, int D) {
    extern __shared__ float s_t[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpc = blockDim.x >> 5;
    const int nt = n_f + 1, ld = D + 1;
    float *t = s_t + static_cast<size_t>(warp) * nt * ld;
    const int n_pairs = nt * (nt - 1) / 2;
    const int out_w = D + n_pairs;
    for (int s = blockIdx.x * wpc + warp; s < B; s += gridDim.x * wpc) {
        const float *xs = x + static_cast<size_t>(s) * D;
        const float *ls = ly + static_cast<size_t>(s) * n_f * D;
        float *rs = r + static_cast<size_t>(s) * out_w;
        for (int e = lane; e < D; e += 32) {
            const float v = __ldg(xs + e);
            t[e] = v;
            rs[e] = v;
        }
        for (int e = lane; e < n_f * D; e += 32) {
            const int f = e / D, k = e - f * D;
            t[(f + 1) * ld + k] = __ldg(ls + e);
        }
        __syncwarp();
        for (int pr = lane; pr < n_pairs; pr += 32) {
            // invert pr = i(i-1)/2 + j, 0 <= j < i
            int i = static_cast<int>((1.0f + sqrtf(1.0f + 8.0f * static_cast<float>(pr))) * 0.5f);
            while (i * (i - 1) / 2 > pr) --i;
            while ((i + 1) * i / 2 <= pr) ++i;
            const int j = pr - i * (i - 1) / 2;
            const float *a = t + i * ld, *b = t + j * ld;
            float acc = 0.0f;
            for (int k = 0; k < D; ++k) acc = fmaf(a[k], b[k], acc);
            rs[D + pr] = acc;
        }
        __syncwarp();
    }
}

// ---- tensor-core path -------------------------------------------------------------------------------------------
constexpr int kMmaWarps = 8;

__device__ __forceinline__ unsigned to_tf32(float v) {
    unsigned r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
    return r;
}
// D += A(16x8, row) * B(8x8, col), TF32 inputs, fp32 accumulate
__device__ __forceinline__ void mma_tf32(float (&c)[4], unsigned a0, unsigned a1, unsigned a2, unsigned a3, unsigned b0, unsigned b1) {
    asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

__device__ __forceinline__ void cp_async16(void *smem, const void *gmem) {
    const unsigned sa = static_cast<unsigned>(__cvta_generic_to_shared(smem));
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sa), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

// ld: floats between rows of the staged T (>= Dp, = 8 mod 16: the 64-bit fragment reads below are bank-conflict free).
// A warp owns two buffers of `region` floats (region >= 32 * ld and >= (n_f + 1) * kZld): while it computes sample s out
// of one, cp.async fills the other with the T of its next sample, so a warp always has a sample's worth of HBM reads in
// flight; the grid is sized to what is resident at once and every warp walks the batch with the grid's stride.
// The kernel was issue-bound (ncu, profiles/r2_interact_*: 932 warp instructions per sample at d = 16, issue slots 64 % busy,
// DRAM 12 %), so everything that does not depend on the sample is hoisted out of the sample loop: the (row, column) walk
// of the staging copy is incremental (no division), the shared-memory offsets of a lane's packed pairs live in registers
// (no pair table), and the fragments / accumulators move as 64-bit words.
constexpr int kZld = 40;                     // row stride of the staged Z: the accumulators' 64-bit stores are conflict free
constexpr int kPairSlots = 16;               // packed pairs per lane: 32 * 16 >= 31 * 32 / 2

__global__ void __launch_bounds__(kMmaWarps * 32, 3) k_interact_mma(const float *__restrict__ x, const float *__restrict__ ly,
                                                                 float *__restrict__ r, int B, int n_f, int D, int Dp, int ld, int region) {
    extern __shared__ __align__(16) float s_t[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpc = blockDim.x >> 5;
    const int nt = n_f + 1;
    const int n_pairs = nt * (nt - 1) / 2;
    const int out_w = D + n_pairs;
    // offset in the staged Z of packed pair pr = i(i-1)/2 + j (0 <= j < i): a table built once by the CTA, from which a lane
    // takes the pairs lane + 32 k it writes, two 16-bit offsets per register (a warp lives for only a handful of samples:
    // per-lane square roots for all 16 slots cost as much as a whole sample)
    __shared__ unsigned short s_off[32 * kPairSlots];
    for (int pr = threadIdx.x; pr < 32 * kPairSlots; pr += blockDim.x) {
        unsigned o = 0;
        if (pr < n_pairs) {
            int i = static_cast<int>((1.0f + sqrtf(1.0f + 8.0f * static_cast<float>(pr))) * 0.5f);
            while (i * (i - 1) / 2 > pr) --i;
            while ((i + 1) * i / 2 <= pr) ++i;
            o = static_cast<unsigned>(i * kZld + (pr - i * (i - 1) / 2));
        }
        s_off[pr] = static_cast<unsigned short>(o);
    }
    __syncthreads();
    unsigned poff[kPairSlots / 2];
#pragma unroll
    for (int k = 0; k < kPairSlots; k += 2)
        poff[k >> 1] = static_cast<unsigned>(s_off[lane + 32 * k]) | (static_cast<unsigned>(s_off[lane + 32 * (k + 1)]) << 16);
    float *buf0 = s_t + static_cast<size_t>(warp) * 2 * region;
    const int g = lane >> 2, tq = lane & 3;
    const bool vec = ((D & 3) == 0) && ((reinterpret_cast<uintptr_t>(x) & 15u) == 0) && ((reinterpret_cast<uintptr_t>(ly) & 15u) == 0);
    const int d4 = D >> 2, n4 = nt * d4;
    const int stride = gridDim.x * wpc;
    // the staging walk of this lane: 16-byte piece e = lane + 32 i of [x ; ly] sits in row e / d4 of T.  x and the rows of
    // ly are contiguous in global memory, so the source is a base pointer + 16 e; the destination is 16 e plus the row's
    // padding, row * (ld - D) floats -- only the row is tracked (incrementally: no division in the loop), and shared-memory
    // addresses are 32-bit
    const int row0 = vec ? lane / d4 : 0, c40 = vec ? lane - row0 * d4 : 0;
    const int dr = vec ? 32 / d4 : 0, dc = vec ? 32 - dr * d4 : 0;
    const int pad = ld - D;

    // stage T = [x ; ly] of sample s into t (asynchronously when rows are 16-byte aligned)
    auto stage = [&](int s, float *t) {
        const float *xs = x + static_cast<size_t>(s) * D;
        const float *ls = ly + static_cast<size_t>(s) * n_f * D;
        if (vec) {
            const float *lsm = ls - D;                        // piece e >= d4 is at ls + 4 (e - d4)
            const unsigned sa = static_cast<unsigned>(__cvta_generic_to_shared(t));
            int row = row0, c4 = c40;
            for (int e = lane; e < n4; e += 32) {
                const float *src = (e < d4 ? xs : lsm) + (e << 2);
                const unsigned dst = sa + (static_cast<unsigned>((e << 2) + row * pad) << 2);
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
                c4 += dc;
                row += dr;
                if (c4 >= d4) {
                    c4 -= d4;
                    ++row;
                }
            }
        } else {
            for (int e = lane; e < nt * D; e += 32) {
                const int row = e / D, c = e - row * D;
                t[row * ld + c] = __ldg(row == 0 ? xs + c : ls + static_cast<size_t>(row - 1) * D + c);
            }
        }
        cp_async_commit();
    };

    int s = blockIdx.x * wpc + warp;
    int cur = 0;
    if (s < B) stage(s, buf0);
    for (; s < B; s += stride) {
        float *t = buf0 + cur * region;
        const int s_next = s + stride;
        if (s_next < B) {
            stage(s_next, buf0 + (cur ^ 1) * region);
            cp_async_wait<1>();
        } else {
            cp_async_wait<0>();
        }
        __syncwarp();
        float *rs = r + static_cast<size_t>(s) * out_w;
        if (Dp > D) {
            for (int e = lane; e < nt * (Dp - D); e += 32) {
                const int row = e / (Dp - D), c = D + (e - row * (Dp - D));
                t[row * ld + c] = 0.0f;
            }
            __syncwarp();
        }
        // x goes to the head of the output row
        if (lane < D) rs[lane] = t[lane];
        for (int e = lane + 32; e < D; e += 32) rs[e] = t[e];
        // ---- Z = T T^t on the tensor cores (rows >= nt hold stale data: they only reach outputs nobody reads) ----
        // The contraction index may be permuted as long as A and B agree: the fragment slots "k = tq" and "k = tq + 4"
        // of a lane take the adjacent columns k0 + 2 tq and k0 + 2 tq + 1, so a lane reads one 64-bit word per row group.
        float acc[6][4];
#pragma unroll
        for (int i = 0; i < 6; ++i)
#pragma unroll
            for (int k = 0; k < 4; ++k) acc[i][k] = 0.0f;
        const float *tl = t + g * ld + 2 * tq;
        for (int k0 = 0; k0 < Dp; k0 += 8) {
            unsigned hi[4][2], lo[4][2];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                // hi = the value rounded to TF32's 10 mantissa bits with two integer instructions (add half an ulp, mask):
                // cvt.rna.tf32 runs at a quarter of the ALU rate, and at d = 64 its 256 conversions per sample were the
                // longest pipe.  lo = v - hi is exact and goes in unrounded: the tensor core ignores its low 13 bits, so
                // |v - hi - lo_tf32| < 2^-21 |v|.  Rounding lo as well would halve that, but the add can carry a NaN's
                // mantissa into the sign bit (0x7FFFFFFF -> -0.0): hi of a NaN may be +-0 or Inf, and lo must stay NaN
                const float2 v = *reinterpret_cast<const float2 *>(tl + 8 * j * ld + k0);
                hi[j][0] = (__float_as_uint(v.x) + 0x1000u) & 0xFFFFE000u;
                lo[j][0] = __float_as_uint(v.x - __uint_as_float(hi[j][0]));
                hi[j][1] = (__float_as_uint(v.y) + 0x1000u) & 0xFFFFE000u;
                lo[j][1] = __float_as_uint(v.y - __uint_as_float(hi[j][1]));
            }
            // tile (m, n): rows 16m .. 16m+15 (A from row groups 2m, 2m+1), cols 8n .. 8n+7 (B from row group n)
#define EVS_TILE(ti, m, n)                                                                                           \
    mma_tf32(acc[ti], hi[2 * m][0], hi[2 * m + 1][0], hi[2 * m][1], hi[2 * m + 1][1], hi[n][0], hi[n][1]);              \
    mma_tf32(acc[ti], hi[2 * m][0], hi[2 * m + 1][0], hi[2 * m][1], hi[2 * m + 1][1], lo[n][0], lo[n][1]);              \
    mma_tf32(acc[ti], lo[2 * m][0], lo[2 * m + 1][0], lo[2 * m][1], lo[2 * m + 1][1], hi[n][0], hi[n][1]);
            EVS_TILE(0, 0, 0)
            EVS_TILE(1, 0, 1)
            EVS_TILE(2, 1, 0)
            EVS_TILE(3, 1, 1)
            EVS_TILE(4, 1, 2)
            EVS_TILE(5, 1, 3)
#undef EVS_TILE
        }
        __syncwarp();                                   // every lane has read its last fragment: T may be overwritten
        // ---- accumulators -> Z[nt][kZld] in the same buffer (rows >= nt are never read) ------------------------------
        {
            const int tm[6] = {0, 0, 1, 1, 1, 1}, tn[6] = {0, 1, 0, 1, 2, 3};
#pragma unroll
            for (int ti = 0; ti < 6; ++ti) {
                const int row = 16 * tm[ti] + g, col = 8 * tn[ti] + 2 * tq;
                if (row < nt) *reinterpret_cast<float2 *>(t + row * kZld + col) = make_float2(acc[ti][0], acc[ti][1]);
                if (row + 8 < nt) *reinterpret_cast<float2 *>(t + (row + 8) * kZld + col) = make_float2(acc[ti][2], acc[ti][3]);
            }
        }
        __syncwarp();
        // ---- strict lower triangle row-major behind x, consecutive lanes write consecutive floats ------------------
        float *rp = rs + D + lane;
#pragma unroll
        for (int k = 0; k < kPairSlots; ++k)
            if (lane + 32 * k < n_pairs) rp[32 * k] = t[(poff[k >> 1] >> (16 * (k & 1))) & 0xFFFFu];
        __syncwarp();
        cur ^= 1;
    }
}

inline int launch_interact(const float *x, const float *ly, float *r, int B, int n_f, int D, cudaStream_t st) {
    if (B < 0 || n_f < 1 || D < 1 || x == nullptr || ly == nullptr || r == nullptr) return EVS_ERR_INVALID;
    if (B == 0) return EVS_OK;
    static const bool force_fma = [] {
        const char *e = getenv("EVSTORE_B200_INTERACT_FMA");     // A/B aid: 1 = the fp32 FMA kernel for every shape
        return e && e[0] == '1';
    }();
    if (n_f + 1 <= 32 && D <= 128 && !force_fma) {
        const int Dp = (D + 7) & ~7;
        const int ld = (Dp & 15) == 8 ? Dp : Dp + 8;            // = 8 mod 16: conflict-free 64-bit fragment reads
        const int region = std::max(32 * ld, (n_f + 1) * kZld);
        // two buffers per warp; fewer warps per CTA when the rows are wide, so that several CTAs stay resident
        const int warps = (static_cast<size_t>(kMmaWarps) * 2 * region * sizeof(float) > 72 * 1024) ? 4 : kMmaWarps;
        const size_t smem = static_cast<size_t>(warps) * 2 * region * sizeof(float);
        static int sms = 0;
        if (sms == 0) {
            int dev = 0;
            cudaGetDevice(&dev);
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        }
        if (smem > 48 * 1024) {
            cudaError_t e = cudaFuncSetAttribute(k_interact_mma, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
            if (e != cudaSuccess) {
                cudaGetLastError();                         // not left behind for the caller's next launch check
                set_error(std::string("k_interact_mma smem: ") + cudaGetErrorString(e));
                return EVS_ERR_CUDA;
            }
        }
        int per_sm = 1;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_interact_mma, warps * 32, smem) != cudaSuccess || per_sm < 1) per_sm = 1;
        const int ctas = std::min((B + warps - 1) / warps, per_sm * sms);
        k_interact_mma<<<ctas, warps * 32, smem, st>>>(x, ly, r, B, n_f, D, Dp, ld, region);
        EVS_CUDA(cudaGetLastError());
        return EVS_OK;
    }
    // the fp32 FMA kernel: a warp stages its sample's T in (n_f + 1) (d + 1) floats; as many warps per CTA (4 down to 1)
    // as the device's opt-in shared memory holds
    int dev = 0, optin = 0;
    EVS_CUDA(cudaGetDevice(&dev));
    EVS_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    const size_t per_warp = static_cast<size_t>(n_f + 1) * (D + 1) * sizeof(float);
    if (per_warp > static_cast<size_t>(optin)) {
        set_error("evs_interact: n_f = " + std::to_string(n_f) + ", dim = " + std::to_string(D) + " stages " +
                  std::to_string(per_warp) + " B of shared memory per sample, more than the device's limit of " +
                  std::to_string(optin) + " B per block");
        return EVS_ERR_INVALID;
    }
    const int warps = static_cast<int>(std::min<size_t>(kInteractWarps, optin / per_warp));
    const size_t smem = warps * per_warp;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(k_interact, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
        if (e != cudaSuccess) {
            cudaGetLastError();
            set_error(std::string("k_interact smem: ") + cudaGetErrorString(e));
            return EVS_ERR_CUDA;
        }
    }
    const int ctas = static_cast<int>(std::min<long long>((static_cast<long long>(B) + warps - 1) / warps, 148 * 8));
    k_interact<<<ctas, warps * 32, smem, st>>>(x, ly, r, B, n_f, D);
    EVS_CUDA(cudaGetLastError());
    return EVS_OK;
}

}  // namespace evs
