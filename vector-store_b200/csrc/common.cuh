// common.cuh — shared device helpers of libvsb200 (sm_100a).
//
// Canonical distance arithmetic (mirrored bit-for-bit by oracle/exact.c):
//   a stored row is a sequence of 16-byte chunks; chunk c belongs to lane (c % 32);
//   a lane walks its chunks in increasing c and the elements of a chunk in
//   increasing index with ONE fp32 accumulator and explicit fmaf; the 32 lane
//   sums are combined by the xor butterfly 16,8,4,2,1 (every lane ends with the
//   same bits).  i8 accumulates in int32 and b1 in popcounts, which are order-free.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>

#define VSB_METRIC_L2SQ 0
#define VSB_METRIC_COS 1
#define VSB_METRIC_IP 2
#define VSB_METRIC_HAMMING 3

#define VSB_ST_F32 0
#define VSB_ST_F16 1
#define VSB_ST_BF16 2
#define VSB_ST_I8 3
#define VSB_ST_B1 4

namespace vsb {

constexpr uint32_t kInvalidSlot = 0xFFFFFFFFu;
constexpr uint64_t kInvalidPacked = 0xFFFFFFFFFFFFFFFFull;
constexpr uint32_t kFullMask = 0xFFFFFFFFu;
constexpr uint32_t kExpandedBit = 0x80000000u;  // graph search: "already expanded" flag in the slot word
constexpr uint64_t kRowMask48 = 0x0000FFFFFFFFFFFFull;

// ---- order-preserving float <-> uint -----------------------------------------------------------
__host__ __device__ __forceinline__ uint32_t f32_to_ord(float f) {
#ifdef __CUDA_ARCH__
    uint32_t u = __float_as_uint(f);
#else
    uint32_t u;
    memcpy(&u, &f, 4);
#endif
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__host__ __device__ __forceinline__ float ord_to_f32(uint32_t o) {
    uint32_t u = (o & 0x80000000u) ? (o & 0x7FFFFFFFu) : ~o;
#ifdef __CUDA_ARCH__
    return __uint_as_float(u);
#else
    float f;
    memcpy(&f, &u, 4);
    return f;
#endif
}
__host__ __device__ __forceinline__ uint64_t pack_ds(float d, uint32_t slot) {
    return ((uint64_t)f32_to_ord(d) << 32) | slot;
}
__host__ __device__ __forceinline__ uint32_t packed_hi(uint64_t p) { return (uint32_t)(p >> 32); }
__host__ __device__ __forceinline__ uint32_t packed_lo(uint64_t p) { return (uint32_t)p; }

__device__ __forceinline__ bool bit_test(const uint32_t* bm, uint32_t i) {
    return (bm[i >> 5] >> (i & 31)) & 1u;
}

// Filtered search: the bitmaps of a call lie back to back, ceil(bits / 32) words each; query q tests bitmap
// allow_of_q[q] (a null index array means bitmap 0 for every query)
__device__ __forceinline__ const uint32_t* query_allow(const uint32_t* allow, uint64_t bits, const uint32_t* allow_of_q,
                                                       uint32_t q) {
    return allow_of_q == nullptr ? allow : allow + (size_t)allow_of_q[q] * (size_t)((bits + 31) / 32);
}

// ---- warp helpers ------------------------------------------------------------------------------
__device__ __forceinline__ float butterfly_sum(float v) {
    v = __fadd_rn(v, __shfl_xor_sync(kFullMask, v, 16));
    v = __fadd_rn(v, __shfl_xor_sync(kFullMask, v, 8));
    v = __fadd_rn(v, __shfl_xor_sync(kFullMask, v, 4));
    v = __fadd_rn(v, __shfl_xor_sync(kFullMask, v, 2));
    v = __fadd_rn(v, __shfl_xor_sync(kFullMask, v, 1));
    return v;
}
__device__ __forceinline__ int butterfly_sum_i(int v) {
    v += __shfl_xor_sync(kFullMask, v, 16);
    v += __shfl_xor_sync(kFullMask, v, 8);
    v += __shfl_xor_sync(kFullMask, v, 4);
    v += __shfl_xor_sync(kFullMask, v, 2);
    v += __shfl_xor_sync(kFullMask, v, 1);
    return v;
}

__device__ __forceinline__ uint4 ldg_nc_v4(const void* p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}

// ---- storage traits ----------------------------------------------------------------------------
// ELEMS = elements per 16-byte chunk.  unpack() turns a chunk into ELEMS floats (exact).
template <int ST>
struct Storage;

template <>
struct Storage<VSB_ST_F32> {
    static constexpr int ELEMS = 4;
    static constexpr bool kFloat = true;
    __device__ static __forceinline__ void unpack(const uint4& c, float* f) {
        f[0] = __uint_as_float(c.x);
        f[1] = __uint_as_float(c.y);
        f[2] = __uint_as_float(c.z);
        f[3] = __uint_as_float(c.w);
    }
};
template <>
struct Storage<VSB_ST_BF16> {
    static constexpr int ELEMS = 8;
    static constexpr bool kFloat = true;
    __device__ static __forceinline__ void unpack(const uint4& c, float* f) {
        f[0] = __uint_as_float(c.x << 16);
        f[1] = __uint_as_float(c.x & 0xFFFF0000u);
        f[2] = __uint_as_float(c.y << 16);
        f[3] = __uint_as_float(c.y & 0xFFFF0000u);
        f[4] = __uint_as_float(c.z << 16);
        f[5] = __uint_as_float(c.z & 0xFFFF0000u);
        f[6] = __uint_as_float(c.w << 16);
        f[7] = __uint_as_float(c.w & 0xFFFF0000u);
    }
};
template <>
struct Storage<VSB_ST_F16> {
    static constexpr int ELEMS = 8;
    static constexpr bool kFloat = true;
    __device__ static __forceinline__ void unpack(const uint4& c, float* f) {
        const uint32_t w[4] = {c.x, c.y, c.z, c.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            __half2 h = *reinterpret_cast<const __half2*>(&w[i]);
            float2 v = __half22float2(h);
            f[2 * i] = v.x;
            f[2 * i + 1] = v.y;
        }
    }
};
template <>
struct Storage<VSB_ST_I8> {
    static constexpr int ELEMS = 16;
    static constexpr bool kFloat = false;
    __device__ static __forceinline__ void unpack(const uint4& c, float* f) {
        const uint32_t w[4] = {c.x, c.y, c.z, c.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
#pragma unroll
            for (int b = 0; b < 4; ++b) f[4 * i + b] = (float)(int)(int8_t)((w[i] >> (8 * b)) & 0xFF);
        }
    }
};
template <>
struct Storage<VSB_ST_B1> {
    static constexpr int ELEMS = 128;
    static constexpr bool kFloat = false;
};

// Per-(query,row) partial state produced by a lane for its chunks, then reduced.
// FLOAT storages: acc = canonical fp32 partial.  I8: int dot / int l2.  B1: popcount.
template <int ST, int METRIC>
struct ChunkAcc {
    float f = 0.0f;
    int i = 0;
    __device__ __forceinline__ void add(const uint4& q, const uint4& x) {
        if constexpr (ST == VSB_ST_B1) {
            i += __popc(q.x ^ x.x) + __popc(q.y ^ x.y) + __popc(q.z ^ x.z) + __popc(q.w ^ x.w);
        } else if constexpr (ST == VSB_ST_I8) {
            if constexpr (METRIC == VSB_METRIC_L2SQ) {
                const uint32_t qa[4] = {q.x, q.y, q.z, q.w};
                const uint32_t xa[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
                for (int w = 0; w < 4; ++w) {
#pragma unroll
                    for (int b = 0; b < 4; ++b) {
                        int d = (int)(int8_t)((qa[w] >> (8 * b)) & 0xFF) - (int)(int8_t)((xa[w] >> (8 * b)) & 0xFF);
                        i += d * d;
                    }
                }
            } else {
                i = __dp4a((int)q.x, (int)x.x, i);
                i = __dp4a((int)q.y, (int)x.y, i);
                i = __dp4a((int)q.z, (int)x.z, i);
                i = __dp4a((int)q.w, (int)x.w, i);
            }
        } else {
            float qf[Storage<ST>::ELEMS], xf[Storage<ST>::ELEMS];
            Storage<ST>::unpack(q, qf);
            Storage<ST>::unpack(x, xf);
            add_f(qf, xf);
        }
    }
    // float path with the query chunk already unpacked (graph search keeps it in registers)
    __device__ __forceinline__ void add_f(const float* qf, const float* xf) {
        constexpr int E = (ST == VSB_ST_F32) ? 4 : 8;
#pragma unroll
        for (int e = 0; e < E; ++e) {
            if constexpr (METRIC == VSB_METRIC_L2SQ) {
                float d = __fsub_rn(qf[e], xf[e]);
                f = __fmaf_rn(d, d, f);
            } else {
                f = __fmaf_rn(qf[e], xf[e], f);
            }
        }
    }
};

// Final scalar distance from the warp-reduced accumulator.  qn / xn are sqrt(sum of squares)
// (COS only).  Must match oracle/exact.c :: finish_distance.
template <int ST, int METRIC>
__device__ __forceinline__ float finish_distance(float facc, int iacc, float qn, float xn) {
    if constexpr (ST == VSB_ST_B1) {
        return (float)iacc;
    } else {
        float dot = Storage<ST>::kFloat ? facc : (float)iacc;
        if constexpr (METRIC == VSB_METRIC_L2SQ) {
            return dot;
        } else if constexpr (METRIC == VSB_METRIC_IP) {
            if constexpr (ST == VSB_ST_I8) dot = __fdiv_rn(dot, 16129.0f);
            return __fsub_rn(1.0f, dot);
        } else {
            if (qn == 0.0f && xn == 0.0f) return 0.0f;
            if (qn == 0.0f || xn == 0.0f) return 1.0f;
            float d = __fsub_rn(1.0f, __fdiv_rn(dot, __fmul_rn(qn, xn)));
            d = d < 0.0f ? 0.0f : d;
            d = d > 2.0f ? 2.0f : d;
            return d;
        }
    }
}

// Full canonical distance between two stored rows, executed by one warp. All lanes return it.
template <int ST, int METRIC>
__device__ __forceinline__ float warp_distance(const uint4* __restrict__ q, const uint4* __restrict__ x,
                                               int n_chunks, float qn, float xn, int lane) {
    ChunkAcc<ST, METRIC> acc;
    for (int c = lane; c < n_chunks; c += 32) acc.add(q[c], ldg_nc_v4(x + c));
    float f = 0.0f;
    int i = 0;
    if constexpr (Storage<ST>::kFloat)
        f = butterfly_sum(acc.f);
    else
        i = butterfly_sum_i(acc.i);
    return finish_distance<ST, METRIC>(f, i, qn, xn);
}

// ---- dispatch helpers --------------------------------------------------------------------------
#define VSB_DISPATCH_ST(st, ...)                                              \
    switch (st) {                                                             \
        case VSB_ST_F32: { constexpr int ST = VSB_ST_F32; __VA_ARGS__; } break;   \
        case VSB_ST_F16: { constexpr int ST = VSB_ST_F16; __VA_ARGS__; } break;   \
        case VSB_ST_BF16: { constexpr int ST = VSB_ST_BF16; __VA_ARGS__; } break; \
        case VSB_ST_I8: { constexpr int ST = VSB_ST_I8; __VA_ARGS__; } break;     \
        default: { constexpr int ST = VSB_ST_B1; __VA_ARGS__; } break;            \
    }
#define VSB_DISPATCH_METRIC(m, ...)                                                   \
    switch (m) {                                                                      \
        case VSB_METRIC_L2SQ: { constexpr int METRIC = VSB_METRIC_L2SQ; __VA_ARGS__; } break; \
        case VSB_METRIC_COS: { constexpr int METRIC = VSB_METRIC_COS; __VA_ARGS__; } break;   \
        case VSB_METRIC_IP: { constexpr int METRIC = VSB_METRIC_IP; __VA_ARGS__; } break;     \
        default: { constexpr int METRIC = VSB_METRIC_HAMMING; __VA_ARGS__; } break;           \
    }

}  // namespace vsb
