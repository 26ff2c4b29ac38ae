// Dequantisers of the reference's storage formats, 16 bytes (one 128-bit load) at a time.
//
//   32-bit: raw IEEE fp32 rows                        (evlfu_32.cpp:530 memcpy)
//   16-bit: ushort codebook, v <= 65000 -> v*0.00002-0.65 evaluated in double then narrowed,
//           v > 65000 -> +-(0.65 + (v-65000)/100), odd = negative   (evlfu_16.cpp:332-356)
//   8-bit : (v/254)*2-1 in float                       (evlfu_8.cpp:370-378)
//   4-bit : two nibbles per byte, high nibble first, 15-entry table (evlfu_4.hpp:46,
//           evlfu_4.cpp:319-341); code 15 is out of range in the reference (the quantiser
//           never emits it, reduce_precision.py:163) and is defined as -1.0 here.
// All four are bit-exact with the C++ expressions (no FMA contraction, same rounding).
#pragma once
#include "evs_types.cuh"

namespace evs {

__device__ __forceinline__ float dec16(unsigned v) {
    if (v > 65000u) {
        float diff = __fdiv_rn(static_cast<float>(v - 65000u), 100.0f);
        double r = __dadd_rn(0.65, static_cast<double>(diff));
        return static_cast<float>((v & 1u) ? -r : r);
    }
    return static_cast<float>(__dsub_rn(__dmul_rn(static_cast<double>(static_cast<float>(v)), 0.00002), 0.65));
}

__device__ __forceinline__ float dec8(unsigned v) {
    return __fsub_rn(__fmul_rn(__fdiv_rn(static_cast<float>(v), 254.0f), 2.0f), 1.0f);
}

__device__ __forceinline__ float dec4(unsigned v) {
    // value_mapping, evlfu_4.hpp:46
    switch (v & 15u) {
        case 0: return 1.0f;          case 1: return 0.8f;        case 2: return 0.6f;
        case 3: return 0.4f;          case 4: return 0.0625f;     case 5: return 0.00390625f;
        case 6: return 0.0000153f;    case 7: return 0.0f;        case 8: return -0.0000153f;
        case 9: return -0.00390625f;  case 10: return -0.0625f;   case 11: return -0.4f;
        case 12: return -0.6f;        case 13: return -0.8f;      default: return -1.0f;
    }
}

// Quantisers (evs_update_rows): bit-exact with codecs.encode_table / oracle/codecs.quantize_table, which evaluate
// reduce_precision.py's expressions in float64 on float32 inputs.  Explicit _rn intrinsics keep nvcc from contracting
// them into FMAs.  Each returns false for a value the format cannot hold, where numpy's astype would wrap silently.
//   16-bit: trunc((v+0.65)/1.3*65000) inside +-0.65; outside, 65000 + trunc(+-100*(..)) made odd (negative) or even
//           (positive); the code must land in [0, 65535] (|v| up to about 6)
//   8-bit : rint((v+1)/2*254), round half to even; v must lie in [-1, 1]
//   4-bit : searchsorted(side="right") over the edges: v == 0 (either sign) -> 7, -0.00025 <= v < 0 -> 8
__device__ __forceinline__ bool enc16(float x, unsigned &q) {
    if (!isfinite(x)) return false;
    const double v = static_cast<double>(x);
    double c;
    if (v < -0.65) {
        double b = trunc(__dmul_rn(-100.0, __dadd_rn(0.65, v)));
        if (fmod(b, 2.0) == 0.0) b = __dadd_rn(b, 1.0);
        c = __dadd_rn(65000.0, b);
    } else if (v > 0.65) {
        double t = trunc(__dmul_rn(100.0, __dsub_rn(v, 0.65)));
        if (fmod(t, 2.0) == 1.0) t = __dsub_rn(t, 1.0);
        c = __dadd_rn(65000.0, t);
    } else {
        c = trunc(__dmul_rn(__ddiv_rn(__dadd_rn(v, 0.65), 1.3), 65000.0));
    }
    if (!(c >= 0.0 && c <= 65535.0)) return false;
    q = static_cast<unsigned>(c);
    return true;
}

__device__ __forceinline__ bool enc8(float x, unsigned &q) {
    if (!(x >= -1.0f && x <= 1.0f)) return false;          // NaN fails too
    q = static_cast<unsigned>(rint(__dmul_rn(__ddiv_rn(__dadd_rn(static_cast<double>(x), 1.0), 2.0), 254.0)));
    return true;
}

__device__ __forceinline__ bool enc4(float x, unsigned &q) {
    if (!isfinite(x)) return false;
    const double v = static_cast<double>(x);
    if (v == 0.0) {
        q = 7u;
    } else if (v > 0.0) {
        q = 6u - (v >= 0.00025) - (v >= 0.015) - (v >= 0.25) - (v >= 0.4) - (v >= 0.6) - (v >= 0.8);
    } else if (v >= -0.00025) {
        q = 8u;
    } else {
        q = 15u - (v >= -1.0) - (v >= -0.8) - (v >= -0.6) - (v >= -0.4) - (v >= -0.25) - (v >= -0.015);
    }
    return true;
}

// Shared-memory lookup tables for the byte codecs (filled once per CTA).
struct CodecLut {
    float lut8[256];
    float lut4[16];
};

// Fills the tables the two precisions of a tier pair need (P1 == 0: single tier).
template <int P0, int P1>
__device__ __forceinline__ void codec_lut_init(CodecLut *l) {
    if (P0 == 8 || P1 == 8) {
        for (int i = threadIdx.x; i < 256; i += blockDim.x) l->lut8[i] = dec8(i);
    }
    if (P0 == 4 || P1 == 4) {
        if (threadIdx.x < 16) l->lut4[threadIdx.x] = dec4(threadIdx.x);
    }
}

template <int PREC>
struct ElemsPerChunk {
    static constexpr int value = 128 / PREC;     // 4, 8, 16, 32 floats per 16-byte chunk
};

__device__ __forceinline__ void store4(float *dst, bool vec, int e, int D, float a, float b, float c, float d) {
    if (vec && e + 4 <= D) {
        *reinterpret_cast<float4 *>(dst + e) = make_float4(a, b, c, d);
    } else {
        if (e < D) dst[e] = a;
        if (e + 1 < D) dst[e + 1] = b;
        if (e + 2 < D) dst[e + 2] = c;
        if (e + 3 < D) dst[e + 3] = d;
    }
}

// Decode chunk `part` (16 bytes) of a stored row into dst[part*EPC ...], elements >= D dropped.
// `vec` = dst is 16-byte aligned for every 4-element group (uniform per launch).
template <int PREC>
__device__ __forceinline__ void decode_store(uint4 v, float *dst, int part, int D, bool vec, const CodecLut *l) {
    const int e0 = part * ElemsPerChunk<PREC>::value;
    const unsigned w[4] = {v.x, v.y, v.z, v.w};
    if (PREC == 32) {
        store4(dst, vec, e0, D, __uint_as_float(v.x), __uint_as_float(v.y), __uint_as_float(v.z),
               __uint_as_float(v.w));
    } else if (PREC == 16) {
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            unsigned a = w[2 * i], b = w[2 * i + 1];
            store4(dst, vec, e0 + 4 * i, D, dec16(a & 0xFFFFu), dec16(a >> 16), dec16(b & 0xFFFFu), dec16(b >> 16));
        }
    } else if (PREC == 8) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            unsigned a = w[i];
            store4(dst, vec, e0 + 4 * i, D, l->lut8[a & 0xFFu], l->lut8[(a >> 8) & 0xFFu], l->lut8[(a >> 16) & 0xFFu],
                   l->lut8[a >> 24]);
        }
    } else {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            unsigned a = w[i];
            // byte k of the word holds elements 2k (high nibble) and 2k+1 (low nibble)
            store4(dst, vec, e0 + 8 * i, D, l->lut4[(a >> 4) & 15u], l->lut4[a & 15u], l->lut4[(a >> 12) & 15u],
                   l->lut4[(a >> 8) & 15u]);
            store4(dst, vec, e0 + 8 * i + 4, D, l->lut4[(a >> 20) & 15u], l->lut4[(a >> 16) & 15u],
                   l->lut4[(a >> 28) & 15u], l->lut4[(a >> 24) & 15u]);
        }
    }
}

}  // namespace evs
