// convert.cu — K0: cast f32 rows to the storage scalar (on add AND on the query, like
// usearch's cast on `add`/`search`, reference call sites vs_index/usearch.rs:191-222) and
// compute the per-row canonical sum of squares / its square root.
//   f16/bf16: round-to-nearest-even.  i8: round-half-away(clamp(x,-1,1)*127)
//   (pinned by tests/integration/quantization.rs:35-39: 0.9 -> 114, 0.1 -> 13).
//   b1: bit i (LSB first) of byte j = v[8j+i] > 0 (usearch.rs:1179-1205).
// One warp per row; lane l owns chunks l, l+32, ... (the canonical order of common.cuh).
#include "kernels.h"

namespace vsb {

template <int ST>
__global__ void __launch_bounds__(256) convert_rows_kernel(const float* __restrict__ in, uint32_t n_rows,
                                                           uint32_t dim, uint8_t* __restrict__ out,
                                                           uint32_t row_bytes, float* __restrict__ sq,
                                                           float* __restrict__ nrm) {
    constexpr int E = Storage<ST>::ELEMS;
    const int lane = threadIdx.x & 31;
    const uint32_t row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= n_rows) return;
    const float* src = in + (size_t)row * dim;
    uint4* dst = reinterpret_cast<uint4*>(out + (size_t)row * row_bytes);
    const int n_chunks = row_bytes / 16;
    float facc = 0.0f;
    int iacc = 0;
    for (int c = lane; c < n_chunks; c += 32) {
        uint32_t w[4] = {0, 0, 0, 0};
        const uint32_t base = (uint32_t)c * E;
        if constexpr (ST == VSB_ST_F32) {
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                float v = (base + e < dim) ? src[base + e] : 0.0f;
                w[e] = __float_as_uint(v);
                facc = __fmaf_rn(v, v, facc);
            }
        } else if constexpr (ST == VSB_ST_BF16) {
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                float v = (base + e < dim) ? src[base + e] : 0.0f;
                __nv_bfloat16 b = __float2bfloat16_rn(v);
                uint32_t bits = (uint32_t)__bfloat16_as_ushort(b);
                w[e >> 1] |= bits << (16 * (e & 1));
                float r = __uint_as_float(bits << 16);
                facc = __fmaf_rn(r, r, facc);
            }
        } else if constexpr (ST == VSB_ST_F16) {
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                float v = (base + e < dim) ? src[base + e] : 0.0f;
                __half h = __float2half_rn(v);
                uint32_t bits = (uint32_t)__half_as_ushort(h);
                w[e >> 1] |= bits << (16 * (e & 1));
                float r = __half2float(h);
                facc = __fmaf_rn(r, r, facc);
            }
        } else if constexpr (ST == VSB_ST_I8) {
#pragma unroll
            for (int e = 0; e < 16; ++e) {
                float v = (base + e < dim) ? src[base + e] : 0.0f;
                v = fminf(fmaxf(v, -1.0f), 1.0f);
                int q = (int)roundf(__fmul_rn(v, 127.0f));
                w[e >> 2] |= ((uint32_t)(q & 0xFF)) << (8 * (e & 3));
                iacc += q * q;
            }
        } else {
#pragma unroll 4
            for (int e = 0; e < 128; ++e) {
                float v = (base + e < dim) ? src[base + e] : 0.0f;
                if (v > 0.0f) {
                    w[e >> 5] |= 1u << (e & 31);
                    iacc += 1;
                }
            }
        }
        dst[c] = make_uint4(w[0], w[1], w[2], w[3]);
    }
    float s;
    if constexpr (Storage<ST>::kFloat)
        s = butterfly_sum(facc);
    else
        s = (float)butterfly_sum_i(iacc);
    if (lane == 0) {
        sq[row] = s;
        nrm[row] = __fsqrt_rn(s);
    }
}

// Scaled int8 rows for the cosine traversal copy (VSB_FLAG_I8_TRAVERSAL): x_j ~ s * q_j with the per-row scale
// s = max|x_j| / 127 and q_j = rint(x_j / s) in [-127, 127].  The row's "norm" is stored in units of s
// (|x| / s), so that K4's int8 cosine  1 - dot_i8 / (|q|/s_q * |x|/s_x)  equals  1 - <q,x> / (|q||x|)  up to
// the quantisation error (relative 1/254 of the largest component per element) — no kernel change needed.
__global__ void __launch_bounds__(256) convert_rows_i8s_kernel(const float* __restrict__ in, uint32_t n_rows, uint32_t dim,
                                                               uint32_t in_stride, uint8_t* __restrict__ out,
                                                               uint32_t row_bytes, float* __restrict__ sq,
                                                               float* __restrict__ nrm) {
    const int lane = threadIdx.x & 31;
    const uint32_t row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= n_rows) return;
    const float* src = in + (size_t)row * in_stride;
    float mx = 0.0f, ss = 0.0f;
    for (uint32_t j = lane; j < dim; j += 32) {
        const float v = src[j];
        mx = fmaxf(mx, fabsf(v));
        ss = __fmaf_rn(v, v, ss);
    }
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(kFullMask, mx, o));
    ss = butterfly_sum(ss);
    const float scale = mx > 0.0f ? mx / 127.0f : 1.0f;
    const float inv = 1.0f / scale;
    uint4* dst = reinterpret_cast<uint4*>(out + (size_t)row * row_bytes);
    const int n_chunks = row_bytes / 16;
    for (int c = lane; c < n_chunks; c += 32) {
        uint32_t w[4] = {0, 0, 0, 0};
        const uint32_t base = (uint32_t)c * 16;
#pragma unroll
        for (int e = 0; e < 16; ++e) {
            const float v = (base + e < dim) ? src[base + e] : 0.0f;
            int q = __float2int_rn(v * inv);
            q = max(-127, min(127, q));
            w[e >> 2] |= ((uint32_t)(q & 0xFF)) << (8 * (e & 3));
        }
        dst[c] = make_uint4(w[0], w[1], w[2], w[3]);
    }
    if (lane == 0) {
        sq[row] = ss;
        nrm[row] = __fsqrt_rn(ss) * inv;
    }
}

// gathers rows (and their norms) by slot into a contiguous block — used for the seed layer
__global__ void gather_rows_kernel(const uint8_t* __restrict__ rows, uint32_t row_bytes,
                                   const float* __restrict__ sq, const float* __restrict__ nrm,
                                   const uint32_t* __restrict__ slots, uint32_t n, uint8_t* __restrict__ out_rows,
                                   float* __restrict__ out_sq, float* __restrict__ out_nrm) {
    const int lane = threadIdx.x & 31;
    const uint32_t i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (i >= n) return;
    const uint32_t s = slots[i];
    const uint4* src = reinterpret_cast<const uint4*>(rows + (size_t)s * row_bytes);
    uint4* dst = reinterpret_cast<uint4*>(out_rows + (size_t)i * row_bytes);
    for (int c = lane; c < (int)(row_bytes / 16); c += 32) dst[c] = src[c];
    if (lane == 0) {
        out_sq[i] = sq[s];
        out_nrm[i] = nrm[s];
    }
}

__global__ void gather_u64_kernel(const uint64_t* __restrict__ in, const uint32_t* __restrict__ slots, uint32_t n,
                                  uint64_t* __restrict__ out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = in[slots[i]];
}

void launch_gather_u64(const uint64_t* in, const uint32_t* slots, uint32_t n, uint64_t* out, cudaStream_t stream) {
    if (n == 0) return;
    gather_u64_kernel<<<(n + 255) / 256, 256, 0, stream>>>(in, slots, n, out);
    g_kernel_launches += 1;
}

__global__ void gather_u32_kernel(const uint32_t* __restrict__ in, const uint32_t* __restrict__ slots, uint32_t n,
                                  uint32_t* __restrict__ out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = in[slots[i]];
}

void launch_gather_u32(const uint32_t* in, const uint32_t* slots, uint32_t n, uint32_t* out, cudaStream_t stream) {
    if (n == 0) return;
    gather_u32_kernel<<<(n + 255) / 256, 256, 0, stream>>>(in, slots, n, out);
    g_kernel_launches += 1;
}

// one thread per result entry; thread 0 of a row also moves its count
__global__ void scatter_topk_kernel(const uint64_t* __restrict__ keys, const float* __restrict__ dists,
                                    const uint32_t* __restrict__ counts, const uint32_t* __restrict__ map, uint32_t n,
                                    uint32_t k, uint64_t* __restrict__ out_keys, float* __restrict__ out_dists,
                                    uint32_t* __restrict__ out_counts) {
    const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (uint64_t)n * k) return;
    const uint32_t i = (uint32_t)(e / k), j = (uint32_t)(e % k);
    const uint64_t dst = (uint64_t)map[i] * k + j;
    out_keys[dst] = keys[e];
    out_dists[dst] = dists[e];
    if (j == 0 && counts != nullptr && out_counts != nullptr) out_counts[map[i]] = counts[i];
}

void launch_scatter_topk(const uint64_t* keys, const float* dists, const uint32_t* counts, const uint32_t* map, uint32_t n,
                         uint32_t k, uint64_t* out_keys, float* out_dists, uint32_t* out_counts, cudaStream_t stream) {
    if (n == 0) return;
    const uint64_t total = (uint64_t)n * k;
    scatter_topk_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(keys, dists, counts, map, n, k, out_keys,
                                                                            out_dists, out_counts);
    g_kernel_launches += 1;
}

void launch_convert_rows(int storage, const float* in, uint32_t n_rows, uint32_t dim, uint8_t* out,
                         uint32_t row_bytes, float* sq, float* nrm, cudaStream_t stream) {
    if (n_rows == 0) return;
    const int warps = 8;
    dim3 grid((n_rows + warps - 1) / warps), block(warps * 32);
    VSB_DISPATCH_ST(storage, (convert_rows_kernel<ST><<<grid, block, 0, stream>>>(in, n_rows, dim, out, row_bytes, sq, nrm)));
    g_kernel_launches += 1;
}

void launch_convert_rows_i8s(const float* in, uint32_t n_rows, uint32_t dim, uint32_t in_stride, uint8_t* out,
                             uint32_t row_bytes, float* sq, float* nrm, cudaStream_t stream) {
    if (n_rows == 0) return;
    const int warps = 8;
    convert_rows_i8s_kernel<<<(n_rows + warps - 1) / warps, warps * 32, 0, stream>>>(in, n_rows, dim, in_stride, out,
                                                                                  row_bytes, sq, nrm);
    g_kernel_launches += 1;
}

void launch_gather_rows(const uint8_t* rows, uint32_t row_bytes, const float* sq, const float* nrm,
                        const uint32_t* slots, uint32_t n, uint8_t* out_rows, float* out_sq, float* out_nrm,
                        cudaStream_t stream) {
    if (n == 0) return;
    const int warps = 8;
    gather_rows_kernel<<<(n + warps - 1) / warps, warps * 32, 0, stream>>>(rows, row_bytes, sq, nrm, slots, n,
                                                                          out_rows, out_sq, out_nrm);
    g_kernel_launches += 1;
}

}  // namespace vsb
