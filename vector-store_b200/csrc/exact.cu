// exact.cu — exact brute-force k-NN (SURVEY §8a A7 "K1/K2/K3").
//
//   K1  exact_candidates_kernel : register-tiled distance tiles (generic over all five storage
//       scalars) with the top-k' selection fused into the tile epilogue — the Q×N distance matrix
//       is never written.  Distances here are "candidate grade" (norm trick, any summation
//       order); the list is over-fetched to k' > k.
//   K3  exact_rerank_kernel     : merges the per-split lists, re-evaluates every surviving
//       candidate with the canonical fp32 order of common.cuh (bit-identical to oracle/exact.c),
//       sorts by (distance, key) and emits the top k.
//
// Replaces: usearch::Index::search as called at vs_index/usearch.rs:203-222 when the caller
// wants exact results (ground truth, the un-graphed tail, filtered search, kNN-graph build).
#include <algorithm>

#include <cub/device/device_segmented_sort.cuh>

#include "kernels.h"
#include "select.cuh"

namespace vsb {

namespace {

constexpr int TQ = 64;    // queries per CTA tile
constexpr int TN = 128;   // corpus rows per CTA tile
constexpr int BK = 32;    // elements per k-slab
constexpr int BUFCAP = 32;
constexpr int K1_THREADS = 256;

// bits per element of a storage scalar
template <int ST>
__device__ __host__ constexpr int elem_bits() {
    return ST == VSB_ST_F32 ? 32 : (ST == VSB_ST_F16 || ST == VSB_ST_BF16) ? 16 : ST == VSB_ST_I8 ? 8 : 1;
}

// Loads NE consecutive elements starting at element `e0` (multiple of NE) of a stored row and
// widens them to float.  Bytes past the padded row read as zero.
template <int ST, int NE>
__device__ __forceinline__ void load_elems(const uint8_t* __restrict__ row, uint32_t row_bytes, uint32_t e0,
                                           float* out) {
    constexpr int BYTES = NE * elem_bits<ST>() / 8;
    const uint32_t off = e0 * elem_bits<ST>() / 8;
    uint32_t w[(BYTES + 3) / 4];
#pragma unroll
    for (int i = 0; i < (BYTES + 3) / 4; ++i) w[i] = 0;
    if (off < row_bytes) {
        if constexpr (BYTES >= 16) {
#pragma unroll
            for (int i = 0; i < BYTES / 16; ++i) {
                if (off + 16 * i < row_bytes) {
                    uint4 v = *reinterpret_cast<const uint4*>(row + off + 16 * i);
                    w[4 * i] = v.x;
                    w[4 * i + 1] = v.y;
                    w[4 * i + 2] = v.z;
                    w[4 * i + 3] = v.w;
                }
            }
        } else if constexpr (BYTES == 8) {
            uint2 v = *reinterpret_cast<const uint2*>(row + off);
            w[0] = v.x;
            w[1] = v.y;
        } else if constexpr (BYTES == 4) {
            w[0] = *reinterpret_cast<const uint32_t*>(row + off);
        } else if constexpr (BYTES == 2) {
            w[0] = *reinterpret_cast<const uint16_t*>(row + off);
        } else {
            w[0] = *(row + off);
        }
    }
#pragma unroll
    for (int e = 0; e < NE; ++e) {
        if constexpr (ST == VSB_ST_F32) {
            out[e] = __uint_as_float(w[e]);
        } else if constexpr (ST == VSB_ST_BF16) {
            out[e] = __uint_as_float(((w[e >> 1] >> (16 * (e & 1))) & 0xFFFFu) << 16);
        } else if constexpr (ST == VSB_ST_F16) {
            out[e] = __half2float(__ushort_as_half((unsigned short)((w[e >> 1] >> (16 * (e & 1))) & 0xFFFFu)));
        } else if constexpr (ST == VSB_ST_I8) {
            out[e] = (float)(int)(int8_t)((w[e >> 2] >> (8 * (e & 3))) & 0xFFu);
        } else {
            out[e] = (float)((w[e >> 5] >> (e & 31)) & 1u);
        }
    }
}

template <int ST, int METRIC>
__device__ __forceinline__ float candidate_distance(float dot, float qsq, float xsq, float qn, float xn) {
    if constexpr (METRIC == VSB_METRIC_L2SQ || METRIC == VSB_METRIC_HAMMING) {
        float d = qsq + xsq - 2.0f * dot;
        return d < 0.0f ? 0.0f : d;
    } else if constexpr (METRIC == VSB_METRIC_IP) {
        if constexpr (ST == VSB_ST_I8) dot = dot / 16129.0f;
        return 1.0f - dot;
    } else {
        if (qn == 0.0f && xn == 0.0f) return 0.0f;
        if (qn == 0.0f || xn == 0.0f) return 1.0f;
        float d = 1.0f - dot / (qn * xn);
        return fminf(fmaxf(d, 0.0f), 2.0f);
    }
}

struct K1Args {
    const uint8_t* q_rows;
    const float* q_sq;
    const float* q_nrm;
    uint32_t nq, q_row_bytes;
    const uint8_t* x_rows;
    const float* x_sq;
    const float* x_nrm;
    uint32_t x_row_bytes, x_lo, x_hi;
    const uint32_t* deny;
    const uint64_t* keys;
    const uint32_t* allow;
    uint64_t allow_bits;
    const uint32_t* allow_of_q;  // [nq] bitmap index per query (nullable: bitmap 0)
    uint32_t kp, n_splits, rows_per_split, n_slabs;
    uint64_t* part;
    RangeParams range;  // RANGE instantiations only
};

// RANGE = false: the split's top-kp list per query.  RANGE = true: every admissible row within the query's bound
// (count or fill pass, see RangeParams); kp = 0, no lists.
template <int ST, int METRIC, bool RANGE>
__global__ void __launch_bounds__(K1_THREADS, 2) exact_candidates_kernel(K1Args a) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    float* As = reinterpret_cast<float*>(smem_raw);                  // [BK][TQ]
    float* Bs = As + BK * TQ;                                        // [BK][TN]
    uint64_t* top = reinterpret_cast<uint64_t*>(Bs + BK * TN);       // [TQ][kp]
    uint64_t* buf = top + (size_t)TQ * a.kp;                         // [TQ][BUFCAP]
    uint32_t* thr = reinterpret_cast<uint32_t*>(buf + TQ * BUFCAP);  // [TQ] ordered-distance threshold
    int* cnt = reinterpret_cast<int*>(thr + TQ);                     // [TQ]

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int ty = tid >> 4, tx = tid & 15;
    const uint32_t q0 = blockIdx.x * TQ;
    const uint32_t split = blockIdx.y;
    const uint32_t r_lo = a.x_lo + split * a.rows_per_split;
    const uint32_t r_hi = min(a.x_hi, r_lo + a.rows_per_split);
    const LessByKey less{a.keys};

    for (uint32_t i = tid; i < TQ * a.kp; i += K1_THREADS) top[i] = kInvalidPacked;
    if (tid < TQ) {
        thr[tid] = 0xFFFFFFFFu;
        cnt[tid] = 0;
    }

    // per-thread query metadata for the 4 rows of its micro tile
    float qsq[4], qn[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        uint32_t q = q0 + ty * 4 + i;
        qsq[i] = q < a.nq ? a.q_sq[q] : 0.0f;
        qn[i] = q < a.nq ? a.q_nrm[q] : 0.0f;
    }
    // range mode: each row's bound (-inf for padding rows), its count from the count pass, rows counted so far
    float rthr[4];
    uint32_t rcap[4], rcnt[4];
    if constexpr (RANGE) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const uint32_t q = q0 + ty * 4 + i;
            rthr[i] = q < a.nq ? a.range.thr[q] : __int_as_float(0xFF800000);
            rcap[i] = q < a.nq && a.range.off != nullptr ? a.range.count[q] : 0u;
            rcnt[i] = 0;
        }
    }
    __syncthreads();

    for (uint32_t n0 = r_lo; n0 < r_hi; n0 += TN) {
        float acc[4][8];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[i][j] = 0.0f;

        for (uint32_t slab = 0; slab < a.n_slabs; ++slab) {
            // A: thread -> (row tid&63, 8 elements)
            {
                const int r = tid & 63, part8 = tid >> 6;
                float v[8];
                uint32_t q = q0 + r;
                if (q < a.nq)
                    load_elems<ST, 8>(a.q_rows + (size_t)q * a.q_row_bytes, a.q_row_bytes, slab * BK + part8 * 8, v);
                else {
#pragma unroll
                    for (int e = 0; e < 8; ++e) v[e] = 0.0f;
                }
#pragma unroll
                for (int e = 0; e < 8; ++e) As[(part8 * 8 + e) * TQ + r] = v[e];
            }
            // B: thread -> (row tid&127, 16 elements)
            {
                const int r = tid & 127, half = tid >> 7;
                float v[16];
                uint32_t n = n0 + r;
                if (n < r_hi)
                    load_elems<ST, 16>(a.x_rows + (size_t)n * a.x_row_bytes, a.x_row_bytes, slab * BK + half * 16, v);
                else {
#pragma unroll
                    for (int e = 0; e < 16; ++e) v[e] = 0.0f;
                }
#pragma unroll
                for (int e = 0; e < 16; ++e) Bs[(half * 16 + e) * TN + r] = v[e];
            }
            __syncthreads();
#pragma unroll
            for (int k = 0; k < BK; ++k) {
                const float4 av = *reinterpret_cast<const float4*>(&As[k * TQ + ty * 4]);
                const float4 b0 = *reinterpret_cast<const float4*>(&Bs[k * TN + tx * 4]);
                const float4 b1 = *reinterpret_cast<const float4*>(&Bs[k * TN + 64 + tx * 4]);
                const float ar[4] = {av.x, av.y, av.z, av.w};
                const float br[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(ar[i], br[j], acc[i][j]);
            }
            __syncthreads();
        }

        if constexpr (RANGE) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const uint32_t q = q0 + ty * 4 + i;
                float d[8];
                uint32_t hit = 0;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const uint32_t n = n0 + (j < 4 ? tx * 4 + j : 64 + tx * 4 + (j - 4));
                    const bool nvalid = n < r_hi;
                    d[j] = candidate_distance<ST, METRIC>(acc[i][j], qsq[i], nvalid ? a.x_sq[n] : 0.0f, qn[i],
                                                          nvalid ? a.x_nrm[n] : 0.0f);
                    if (!nvalid || !(d[j] <= rthr[i])) continue;
                    bool ok = !(a.deny != nullptr && bit_test(a.deny, n));
                    if (ok && a.allow != nullptr) {
                        const uint64_t rid = a.keys[n] & kRowMask48;
                        ok = rid < a.allow_bits && bit_test(query_allow(a.allow, a.allow_bits, a.allow_of_q, q), (uint32_t)rid);
                    }
                    if (ok) hit |= 1u << j;
                }
                if (hit == 0) continue;
                if (a.range.off == nullptr) {
                    rcnt[i] += __popc(hit);
                    continue;
                }
                uint32_t pos = atomicAdd(&a.range.cursor[q], (uint32_t)__popc(hit));
                uint64_t* seg = a.range.out + a.range.off[q];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    if (!((hit >> j) & 1u)) continue;
                    const uint32_t n = n0 + (j < 4 ? tx * 4 + j : 64 + tx * 4 + (j - 4));
                    if (pos < rcap[i]) seg[pos] = pack_ds(d[j], n);
                    ++pos;
                }
            }
            continue;
        }

        // ---- fused selection epilogue ----
        uint32_t pending = 0;
        uint32_t dord[4][8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const uint32_t n = n0 + (j < 4 ? tx * 4 + j : 64 + tx * 4 + (j - 4));
            const bool nvalid = n < r_hi;
            const float xsq = nvalid ? a.x_sq[n] : 0.0f;
            const float xn = nvalid ? a.x_nrm[n] : 0.0f;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                float d = candidate_distance<ST, METRIC>(acc[i][j], qsq[i], xsq, qn[i], xn);
                dord[i][j] = f32_to_ord(d);
                if (nvalid && (q0 + ty * 4 + i) < a.nq) pending |= 1u << (i * 8 + j);
            }
        }
        while (true) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int row = ty * 4 + i;
                const uint32_t t = thr[row];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const uint32_t bit = 1u << (i * 8 + j);
                    if (!(pending & bit)) continue;
                    if (dord[i][j] > t) {
                        pending &= ~bit;
                        continue;
                    }
                    const uint32_t n = n0 + (j < 4 ? tx * 4 + j : 64 + tx * 4 + (j - 4));
                    bool ok = true;
                    if (a.deny != nullptr && bit_test(a.deny, n)) ok = false;
                    if (ok && a.allow != nullptr) {
                        const uint64_t rid = a.keys[n] & kRowMask48;
                        ok = rid < a.allow_bits && bit_test(query_allow(a.allow, a.allow_bits, a.allow_of_q, q0 + row),
                                                            (uint32_t)rid);
                    }
                    if (!ok) {
                        pending &= ~bit;
                        continue;
                    }
                    const int pos = atomicAdd(&cnt[row], 1);
                    if (pos < BUFCAP) {
                        buf[row * BUFCAP + pos] = ((uint64_t)dord[i][j] << 32) | n;
                        pending &= ~bit;
                    }
                }
            }
            __syncthreads();
            int overflow = 0;
            for (int rr = 0; rr < TQ / (K1_THREADS / 32); ++rr) {
                const int row = warp * (TQ / (K1_THREADS / 32)) + rr;
                const int c = cnt[row];
                if (c == 0) continue;
                if (c > BUFCAP) overflow = 1;
                uint64_t v = lane < min(c, BUFCAP) ? buf[row * BUFCAP + lane] : kInvalidPacked;
                v = warp_sort32(v, lane, less);
                warp_list_merge(top + (size_t)row * a.kp, (int)a.kp, v, lane, less);
                if (lane == 0) {
                    thr[row] = packed_hi(top[(size_t)row * a.kp + a.kp - 1]);
                    cnt[row] = 0;
                }
            }
            if (!__syncthreads_or(overflow)) break;
        }
    }

    if constexpr (RANGE) {
        if (a.range.off == nullptr) {
#pragma unroll
            for (int i = 0; i < 4; ++i)
                if (rcnt[i] != 0) atomicAdd(&a.range.count[q0 + ty * 4 + i], rcnt[i]);
        }
        return;
    }
    // write the split's lists
    for (uint32_t i = tid; i < TQ * a.kp; i += K1_THREADS) {
        const uint32_t row = i / a.kp, c = i % a.kp;
        const uint32_t q = q0 + row;
        if (q < a.nq) a.part[((size_t)q * a.n_splits + split) * a.kp + c] = top[i];
    }
}

struct K3Args {
    const uint8_t* q_rows;
    const float* q_nrm;
    uint32_t nq, q_row_bytes;
    const uint8_t* x_rows;
    const float* x_nrm;
    uint32_t x_row_bytes;
    const uint64_t* keys;
    const uint64_t* part;
    uint32_t kp, n_splits, k, kf;
    uint64_t* out_keys;
    float* out_dists;
    uint32_t* out_counts;
    uint64_t* out_packed;
    int64_t self_base;
    // certification of a reduced-precision candidate stage (see ExactCert in kernels.h); all nullable
    const float* x_nrm_max;
    float cert_rel, cert_sum;
    uint32_t* uncert_flags;
    uint32_t* uncert_count;
    const uint32_t* q_map;  // query q of this launch is query q_map[q] of the caller (outputs, self slot)
};

constexpr int K3_WARPS = 4;   // warp-per-query variant: queries per CTA
constexpr int K3C_WARPS = 8;  // CTA-per-query variant (small batches): warps sharing one query's candidates

// canonical distances of up to four candidate rows, evaluated by one warp (four rows in flight: 4x the
// memory-level parallelism of a one-by-one loop, each accumulator still follows the canonical order)
template <int ST, int METRIC>
__device__ __forceinline__ void k3_eval4(const K3Args& a, const uint4* qrow, int n_chunks, float qn, const uint32_t (&slot)[4],
                                         const bool (&on)[4], float (&d)[4], int lane) {
    ChunkAcc<ST, METRIC> acc[4];
    const uint4* xr[4];
#pragma unroll
    for (int u = 0; u < 4; ++u)
        xr[u] = reinterpret_cast<const uint4*>(a.x_rows + (size_t)(on[u] ? slot[u] : 0u) * a.x_row_bytes);
    for (int ch = lane; ch < n_chunks; ch += 32) {
        const uint4 qv = qrow[ch];
        uint4 xv[4];
#pragma unroll
        for (int u = 0; u < 4; ++u)
            if (on[u]) xv[u] = ldg_nc_v4(xr[u] + ch);
#pragma unroll
        for (int u = 0; u < 4; ++u)
            if (on[u]) acc[u].add(qv, xv[u]);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        d[u] = 0.0f;
        if (!on[u]) continue;
        float f = 0.0f;
        int i = 0;
        if constexpr (Storage<ST>::kFloat)
            f = butterfly_sum(acc[u].f);
        else
            i = butterfly_sum_i(acc[u].i);
        d[u] = finish_distance<ST, METRIC>(f, i, qn, a.x_nrm[slot[u]]);
    }
}

// CTA == false: one warp per query, K3_WARPS queries per CTA (large batches).
// CTA == true : one CTA of K3C_WARPS warps per query; the candidates are re-evaluated four per warp in parallel
//               (a single-query call would otherwise walk its 2k candidates with one warp).
template <int ST, int METRIC, bool CTA>
__global__ void __launch_bounds__((CTA ? K3C_WARPS : K3_WARPS) * 32) exact_rerank_kernel(K3Args a) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t q = CTA ? blockIdx.x : blockIdx.x * K3_WARPS + warp;
    if (q >= a.nq) return;
    uint64_t* cand = reinterpret_cast<uint64_t*>(smem_raw) + (CTA ? 0 : (size_t)warp * (a.kp + a.kf));  // [kp]
    uint64_t* fin = cand + a.kp;                                                                         // [kf]
    uint64_t* res_s = fin + a.kf;                                                                        // [kp] (CTA only)
    const LessByKey less{a.keys};
    const bool lead = !CTA || warp == 0;

    // 1. merge the split lists by candidate-grade distance
    if (lead) {
        for (uint32_t i = lane; i < a.kp; i += 32) cand[i] = a.part[((size_t)q * a.n_splits) * a.kp + i];
        for (uint32_t i = lane; i < a.kf; i += 32) fin[i] = kInvalidPacked;
        __syncwarp();
        for (uint32_t s = 1; s < a.n_splits; ++s) {
            const uint64_t* src = a.part + ((size_t)q * a.n_splits + s) * a.kp;
            for (uint32_t b = 0; b < a.kp; b += 32) {
                uint64_t v = src[b + lane];  // already ascending inside the list
                if (shfl_u64(v, 0) == kInvalidPacked) break;
                warp_list_merge(cand, (int)a.kp, v, lane, less);
            }
        }
        __syncwarp();
    }
    if constexpr (CTA) {
        for (uint32_t i = threadIdx.x; i < a.kp; i += K3C_WARPS * 32) res_s[i] = kInvalidPacked;
        __syncthreads();
    }
    // every row that is NOT a candidate has a candidate-stage distance >= the worst kept one
    const uint64_t cand_floor = cand[a.kp - 1];
    const uint32_t oq = a.q_map != nullptr ? a.q_map[q] : q;

    // 2. canonical re-evaluation
    const uint4* qrow = reinterpret_cast<const uint4*>(a.q_rows + (size_t)q * a.q_row_bytes);
    const int n_chunks = a.x_row_bytes / 16;
    const float qn = a.q_nrm[q];
    const uint32_t self_slot = a.self_base >= 0 ? (uint32_t)(a.self_base + oq) : kInvalidSlot;
    if constexpr (CTA) {
        for (uint32_t g = warp; g * 4 < a.kp; g += K3C_WARPS) {
            uint32_t slot[4];
            bool on[4];
            bool any = false;
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const uint64_t pc = cand[g * 4 + u];
                slot[u] = packed_lo(pc);
                on[u] = pc != kInvalidPacked && slot[u] != self_slot;
                any = any || on[u];
            }
            if (!any) continue;
            float d[4];
            k3_eval4<ST, METRIC>(a, qrow, n_chunks, qn, slot, on, d, lane);
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (lane == u && on[u]) res_s[g * 4 + u] = pack_ds(d[u], slot[u]);
        }
        __syncthreads();
        if (warp != 0) return;
        for (uint32_t b = 0; b < a.kp; b += 32) {
            uint64_t res = res_s[b + lane];
            if (__ballot_sync(kFullMask, res != kInvalidPacked) == 0) continue;
            res = warp_sort32(res, lane, less);
            warp_list_merge(fin, (int)a.kf, res, lane, less);
        }
    } else {
        for (uint32_t b = 0; b < a.kp; b += 32) {
            const uint64_t mine = cand[b + lane];
            uint64_t res = kInvalidPacked;
            bool end_of_list = false;
            for (int c0 = 0; c0 < 32 && !end_of_list; c0 += 4) {
                uint32_t slot[4];
                bool on[4];
                bool any = false;
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const uint64_t pc = shfl_u64(mine, c0 + u);
                    if (pc == kInvalidPacked) end_of_list = true;  // ascending: the rest of the block is padding
                    slot[u] = packed_lo(pc);
                    on[u] = pc != kInvalidPacked && slot[u] != self_slot;
                    any = any || on[u];
                }
                if (!any) continue;
                float d[4];
                k3_eval4<ST, METRIC>(a, qrow, n_chunks, qn, slot, on, d, lane);
#pragma unroll
                for (int u = 0; u < 4; ++u)
                    if (on[u] && lane == c0 + u) res = pack_ds(d[u], slot[u]);
            }
            if (__ballot_sync(kFullMask, res != kInvalidPacked) == 0) continue;
            res = warp_sort32(res, lane, less);
            warp_list_merge(fin, (int)a.kf, res, lane, less);
        }
    }

    // 3. emit
    uint32_t count = 0;
    for (uint32_t i = lane; i < a.kf; i += 32) {
        const uint64_t p = fin[i];
        const bool valid = p != kInvalidPacked && i < a.k;
        if (i < a.k) {
            if (a.out_packed != nullptr) a.out_packed[(size_t)oq * a.k + i] = valid ? p : kInvalidPacked;
            if (a.out_keys != nullptr) {
                a.out_keys[(size_t)oq * a.k + i] = valid ? a.keys[packed_lo(p)] : 0xFFFFFFFFFFFFFFFFull;
                a.out_dists[(size_t)oq * a.k + i] = valid ? ord_to_f32(packed_hi(p)) : __int_as_float(0x7F800000);
            }
        }
        count += __popc(__ballot_sync(kFullMask, valid));
    }
    if (lane == 0 && a.out_counts != nullptr) a.out_counts[oq] = count;

    // 4. certificate: the candidate stage summed in its own order / at reduced precision (TF32).  A non-candidate
    //    row x has candidate-stage distance >= cand_floor, hence canonical distance >= cand_floor - eps(q).  If
    //    the k-th canonical distance found is strictly below that bound, no such row can enter (or tie into) the
    //    top-k and the result equals the canonical brute force.  Otherwise the query is flagged for the next stage.
    if (a.uncert_flags != nullptr && lane == 0) {
        bool ok = true;
        if (cand_floor != kInvalidPacked) {  // list full: rows were dropped
            const uint64_t pk = fin[a.k - 1];
            if (pk == kInvalidPacked) {
                ok = false;
            } else {
                const float floor_d = ord_to_f32(packed_hi(cand_floor)), dk = ord_to_f32(packed_hi(pk));
                // |candidate-stage distance - canonical distance| <= eps for every row of the block
                const float eps = cert_margin<METRIC>(a.cert_rel, a.cert_sum, qn, *a.x_nrm_max);
                ok = dk + eps < floor_d;  // false for NaN
            }
        }
        a.uncert_flags[q] = ok ? 0u : 1u;
        if (!ok) atomicAdd(a.uncert_count, 1u);
    }
}

// K1c — canonical scan: every admissible row of [x_lo, x_hi) is evaluated in the canonical order against a
// block of SCAN_QB queries; each warp keeps one (distance, key)-ordered list of kf entries per query.  No
// candidate stage, hence nothing to certify: this is the last resort for queries whose certificate failed
// (near-ties below the resolution of the tiled stages), bandwidth-amortised over SCAN_QB queries per row read.
constexpr int SCAN_WARPS = 4, SCAN_QB = 8;
struct ScanArgs {
    const uint8_t* q_rows;
    const float* q_nrm;
    uint32_t nq, q_row_bytes;
    const uint8_t* x_rows;
    const float* x_nrm;
    uint32_t x_row_bytes, x_lo, x_hi;
    const uint32_t* deny;
    const uint64_t* keys;
    const uint32_t* allow;
    uint64_t allow_bits;
    const uint32_t* allow_of_q;  // [nq] bitmap index per query (nullable: bitmap 0)
    uint32_t kf, n_splits, rows_per_split;
    uint64_t* part;  // [nq][n_splits * SCAN_WARPS][kf]
};

template <int ST, int METRIC>
__global__ void __launch_bounds__(SCAN_WARPS * 32) exact_scan_kernel(ScanArgs a) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t q0 = blockIdx.x * SCAN_QB, split = blockIdx.y;
    const int nv = (int)min((uint32_t)SCAN_QB, a.nq - q0);
    uint64_t* lists = reinterpret_cast<uint64_t*>(smem_raw) + (size_t)warp * SCAN_QB * a.kf;  // [SCAN_QB][kf]
    for (uint32_t i = lane; i < SCAN_QB * a.kf; i += 32) lists[i] = kInvalidPacked;
    __syncwarp();
    const LessByKey less{a.keys};
    const int n_chunks = a.x_row_bytes / 16;
    const uint32_t lo = a.x_lo + split * a.rows_per_split;
    const uint32_t hi = min(lo + a.rows_per_split, a.x_hi);
    float qn[SCAN_QB];
#pragma unroll
    for (int j = 0; j < SCAN_QB; ++j) qn[j] = j < nv ? a.q_nrm[q0 + j] : 0.0f;
    // word offset of each query's own bitmap (in shared memory: registers are what this kernel is short of)
    __shared__ size_t q_allow_off[SCAN_QB];
    if (threadIdx.x < SCAN_QB)
        q_allow_off[threadIdx.x] = a.allow_of_q != nullptr && (int)threadIdx.x < nv
                                       ? (size_t)a.allow_of_q[q0 + threadIdx.x] * (size_t)((a.allow_bits + 31) / 32) : 0;
    __syncthreads();

    for (uint32_t r0 = lo + warp * 32; r0 < hi; r0 += 32 * SCAN_WARPS) {
        const uint32_t row = r0 + lane;
        // bit j: the row is admissible for query j of the block; a row is evaluated if any query admits it
        uint32_t adm = 0;
        if (row < hi && !(a.deny != nullptr && bit_test(a.deny, row))) {
            if (a.allow == nullptr) {
                adm = (1u << nv) - 1;
            } else {
                const uint64_t rid = a.keys[row] & kRowMask48;
                if (rid < a.allow_bits) {
#pragma unroll
                    for (int j = 0; j < SCAN_QB; ++j)
                        if (j < nv && bit_test(a.allow + q_allow_off[j], (uint32_t)rid)) adm |= 1u << j;
                }
            }
        }
        uint32_t mask = __ballot_sync(kFullMask, adm != 0);
        uint64_t res[SCAN_QB];
#pragma unroll
        for (int j = 0; j < SCAN_QB; ++j) res[j] = kInvalidPacked;
        while (mask) {  // two rows in flight
            const int c0 = __ffs(mask) - 1;
            mask &= mask - 1;
            const int c1 = mask ? __ffs(mask) - 1 : -1;
            if (c1 >= 0) mask &= mask - 1;
            const uint32_t s0 = r0 + c0, s1 = c1 >= 0 ? r0 + c1 : s0;
            const uint4* x0 = reinterpret_cast<const uint4*>(a.x_rows + (size_t)s0 * a.x_row_bytes);
            const uint4* x1 = reinterpret_cast<const uint4*>(a.x_rows + (size_t)s1 * a.x_row_bytes);
            ChunkAcc<ST, METRIC> acc0[SCAN_QB], acc1[SCAN_QB];
            for (int ch = lane; ch < n_chunks; ch += 32) {
                const uint4 xv0 = ldg_nc_v4(x0 + ch), xv1 = ldg_nc_v4(x1 + ch);
#pragma unroll
                for (int j = 0; j < SCAN_QB; ++j) {
                    if (j < nv) {
                        const uint4 qv = __ldg(reinterpret_cast<const uint4*>(a.q_rows + (size_t)(q0 + j) * a.q_row_bytes) + ch);
                        acc0[j].add(qv, xv0);
                        acc1[j].add(qv, xv1);
                    }
                }
            }
            const float xn0 = a.x_nrm[s0], xn1 = a.x_nrm[s1];
#pragma unroll
            for (int j = 0; j < SCAN_QB; ++j) {
                if (j < nv) {
                    float f0 = 0.0f, f1 = 0.0f;
                    int i0 = 0, i1 = 0;
                    if constexpr (Storage<ST>::kFloat) {
                        f0 = butterfly_sum(acc0[j].f);
                        f1 = butterfly_sum(acc1[j].f);
                    } else {
                        i0 = butterfly_sum_i(acc0[j].i);
                        i1 = butterfly_sum_i(acc1[j].i);
                    }
                    const float d0 = finish_distance<ST, METRIC>(f0, i0, qn[j], xn0);
                    const float d1 = finish_distance<ST, METRIC>(f1, i1, qn[j], xn1);
                    if (lane == c0 && (adm >> j & 1u)) res[j] = pack_ds(d0, s0);
                    if (lane == c1 && (adm >> j & 1u)) res[j] = pack_ds(d1, s1);
                }
            }
        }
#pragma unroll
        for (int j = 0; j < SCAN_QB; ++j) {
            if (j < nv) {
                uint64_t* list = lists + (size_t)j * a.kf;
                const uint64_t tail = list[a.kf - 1];
                if (__ballot_sync(kFullMask, res[j] != kInvalidPacked && less(res[j], tail)) == 0) continue;
                const uint64_t sorted = warp_sort32(res[j], lane, less);
                warp_list_merge(list, (int)a.kf, sorted, lane, less);
            }
        }
    }
    __syncwarp();
    for (int j = 0; j < nv; ++j)
        for (uint32_t i = lane; i < a.kf; i += 32)
            a.part[(((size_t)(q0 + j) * a.n_splits + split) * SCAN_WARPS + warp) * a.kf + i] = lists[(size_t)j * a.kf + i];
}

template <int ST, int METRIC>
void launch_scan(const ScanArgs& a, dim3 grid, size_t smem, cudaStream_t stream) {
    cudaFuncSetAttribute(exact_scan_kernel<ST, METRIC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    exact_scan_kernel<ST, METRIC><<<grid, SCAN_WARPS * 32, smem, stream>>>(a);
}

// max over a block of row norms (non-negative floats order like their bit patterns); *out must be zeroed
__global__ void max_norm_kernel(const float* nrm, uint32_t lo, uint32_t hi, float* out) {
    float m = 0.0f;
    for (uint32_t i = lo + blockIdx.x * blockDim.x + threadIdx.x; i < hi; i += gridDim.x * blockDim.x) m = fmaxf(m, nrm[i]);
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(kFullMask, m, o));
    if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<unsigned int*>(out), __float_as_uint(m));
}

template <int ST, int METRIC, bool RANGE = false>
void launch_k1(const K1Args& a, dim3 grid, size_t smem, cudaStream_t stream) {
    cudaFuncSetAttribute(exact_candidates_kernel<ST, METRIC, RANGE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    exact_candidates_kernel<ST, METRIC, RANGE><<<grid, K1_THREADS, smem, stream>>>(a);
}

// ---- range search: bound, canonical re-evaluation, emit ----
template <int ST, int METRIC>
__global__ void range_bound_kernel(const float* q_nrm, const float* max_distance, uint32_t n, const float* x_nrm_max,
                                   float rel, float sum, float* thr) {
    const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n) return;
    const float qn = q_nrm[q], r = max_distance[q];
    float eps = 0.0f;
    if constexpr (Storage<ST>::kFloat)
        eps = cert_margin<METRIC>(rel, sum, qn, *x_nrm_max);
    else if constexpr (ST == VSB_ST_I8 && METRIC == VSB_METRIC_L2SQ)
        eps = cert_margin<METRIC>(0.0f, sum, qn, *x_nrm_max);
    float t = __fadd_ru(r, eps);
    if constexpr (METRIC == VSB_METRIC_COS)
        if (qn == 0.0f) t = __int_as_float(0x7F800000);
    thr[q] = t;
}

constexpr int RE_WARPS = 8;

template <int ST, int METRIC>
__global__ void __launch_bounds__(RE_WARPS * 32) range_eval_kernel(K3Args a, const float* max_distance, const uint32_t* count,
                                                                   const uint32_t* cursor, const uint32_t* seg_off,
                                                                   const uint32_t* grp_off, uint32_t n_groups,
                                                                   const uint64_t* cand, uint64_t* key_out,
                                                                   uint32_t* dord_out, uint32_t* kept, uint32_t* mismatch) {
    const int lane = threadIdx.x & 31;
    const uint32_t w = blockIdx.x * RE_WARPS + (threadIdx.x >> 5);
    if (w >= n_groups) return;
    // the query of this group: the last q with grp_off[q] <= w (queries without entries own no group)
    uint32_t lo = 0, hi = a.nq;
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) / 2;
        if (grp_off[mid] <= w) lo = mid;
        else hi = mid;
    }
    const uint32_t q = lo, g = w - grp_off[q];
    const uint32_t cnt = count[q];
    const uint32_t have = min(cnt, cursor[q]);
    const uint32_t base = seg_off[q] + 4 * g;
    uint32_t slot[4];
    bool on[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        on[u] = 4 * g + u < have;
        slot[u] = on[u] ? packed_lo(cand[base + u]) : 0u;
    }
    float d[4];
    k3_eval4<ST, METRIC>(a, reinterpret_cast<const uint4*>(a.q_rows + (size_t)q * a.q_row_bytes), a.x_row_bytes / 16,
                         a.q_nrm[q], slot, on, d, lane);
    const float r = max_distance[q];
    uint32_t n_kept = 0;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        const bool keep = on[u] && d[u] <= r;
        n_kept += keep ? 1u : 0u;
        if (lane == u && 4 * g + u < cnt) {
            key_out[base + u] = on[u] ? a.keys[slot[u]] : 0xFFFFFFFFFFFFFFFFull;
            dord_out[base + u] = keep ? f32_to_ord(d[u]) : 0xFFFFFFFFu;
        }
    }
    if (lane == 0 && n_kept != 0) atomicAdd(&kept[q], n_kept);
}

// queries whose fill-pass cursor differs from their count-pass count (queries without candidates included)
__global__ void range_check_kernel(const uint32_t* count, const uint32_t* cursor, uint32_t n, uint32_t* mismatch) {
    const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q < n && count[q] != cursor[q]) atomicAdd(mismatch, 1u);
}

__global__ void range_emit_kernel(const uint32_t* dord, const uint64_t* key, const uint32_t* seg_off, const uint32_t* out_off,
                                  uint32_t n, uint32_t total, uint64_t* keys_out, float* dists_out) {
    const uint32_t e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= total) return;
    uint32_t lo = 0, hi = n;
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) / 2;
        if (out_off[mid] <= e) lo = mid;
        else hi = mid;
    }
    const uint32_t src = seg_off[lo] + (e - out_off[lo]);
    keys_out[e] = key[src];
    dists_out[e] = ord_to_f32(dord[src]);
}

template <int ST, int METRIC>
void launch_k3(const K3Args& a, bool cta, cudaStream_t stream) {
    if (cta) {
        const size_t smem = (size_t)(2 * a.kp + a.kf) * 8;
        exact_rerank_kernel<ST, METRIC, true><<<a.nq, K3C_WARPS * 32, smem, stream>>>(a);
    } else {
        const size_t smem = (size_t)K3_WARPS * (a.kp + a.kf) * 8;
        exact_rerank_kernel<ST, METRIC, false><<<(a.nq + K3_WARPS - 1) / K3_WARPS, K3_WARPS * 32, smem, stream>>>(a);
    }
}

}  // namespace

size_t exact_part_elems(uint32_t nq, uint32_t n_splits, uint32_t kp) { return (size_t)nq * n_splits * kp; }

uint32_t exact_pick_splits(uint32_t nq, uint32_t n_rows, int sm_count) {
    const uint32_t q_tiles = (nq + TQ - 1) / TQ;
    const uint32_t want = (2u * (uint32_t)sm_count + q_tiles - 1) / q_tiles;  // >= 2 CTAs per SM
    const uint32_t max_by_rows = (n_rows + 4 * TN - 1) / (4 * TN);            // >= 4 tiles per split
    uint32_t s = want < max_by_rows ? want : max_by_rows;
    if (s < 1) s = 1;
    if (s > 1024) s = 1024;
    return s;
}

#define VSB_DISPATCH_PAIR(st, metric, CALL)                                        \
    do {                                                                           \
        if ((st) == VSB_ST_B1) {                                                   \
            constexpr int ST = VSB_ST_B1, METRIC = VSB_METRIC_HAMMING;             \
            CALL;                                                                  \
        } else {                                                                   \
            switch ((st) * 4 + (metric)) {                                         \
                case VSB_ST_F32 * 4 + VSB_METRIC_L2SQ: { constexpr int ST = VSB_ST_F32, METRIC = VSB_METRIC_L2SQ; CALL; } break; \
                case VSB_ST_F32 * 4 + VSB_METRIC_COS: { constexpr int ST = VSB_ST_F32, METRIC = VSB_METRIC_COS; CALL; } break;   \
                case VSB_ST_F32 * 4 + VSB_METRIC_IP: { constexpr int ST = VSB_ST_F32, METRIC = VSB_METRIC_IP; CALL; } break;     \
                case VSB_ST_F16 * 4 + VSB_METRIC_L2SQ: { constexpr int ST = VSB_ST_F16, METRIC = VSB_METRIC_L2SQ; CALL; } break; \
                case VSB_ST_F16 * 4 + VSB_METRIC_COS: { constexpr int ST = VSB_ST_F16, METRIC = VSB_METRIC_COS; CALL; } break;   \
                case VSB_ST_F16 * 4 + VSB_METRIC_IP: { constexpr int ST = VSB_ST_F16, METRIC = VSB_METRIC_IP; CALL; } break;     \
                case VSB_ST_BF16 * 4 + VSB_METRIC_L2SQ: { constexpr int ST = VSB_ST_BF16, METRIC = VSB_METRIC_L2SQ; CALL; } break; \
                case VSB_ST_BF16 * 4 + VSB_METRIC_COS: { constexpr int ST = VSB_ST_BF16, METRIC = VSB_METRIC_COS; CALL; } break;   \
                case VSB_ST_BF16 * 4 + VSB_METRIC_IP: { constexpr int ST = VSB_ST_BF16, METRIC = VSB_METRIC_IP; CALL; } break;     \
                case VSB_ST_I8 * 4 + VSB_METRIC_L2SQ: { constexpr int ST = VSB_ST_I8, METRIC = VSB_METRIC_L2SQ; CALL; } break;   \
                case VSB_ST_I8 * 4 + VSB_METRIC_COS: { constexpr int ST = VSB_ST_I8, METRIC = VSB_METRIC_COS; CALL; } break;     \
                default: { constexpr int ST = VSB_ST_I8, METRIC = VSB_METRIC_IP; CALL; } break;                                  \
            }                                                                      \
        }                                                                          \
    } while (0)

void launch_exact_candidates(const ExactParams& p, cudaStream_t stream) {
    if (p.q.n == 0 || p.x_hi <= p.x_lo) return;
    K1Args a;
    a.q_rows = p.q.rows; a.q_sq = p.q.sq; a.q_nrm = p.q.nrm; a.nq = p.q.n; a.q_row_bytes = p.q.row_bytes;
    a.x_rows = p.x.rows; a.x_sq = p.x.sq; a.x_nrm = p.x.nrm; a.x_row_bytes = p.x.row_bytes;
    a.x_lo = p.x_lo; a.x_hi = p.x_hi;
    a.deny = p.deny; a.keys = p.keys; a.allow = p.allow.bm; a.allow_bits = p.allow.bits; a.allow_of_q = p.allow.of_q;
    a.kp = p.kp; a.n_splits = p.n_splits;
    const uint32_t rows = p.x_hi - p.x_lo;
    uint32_t rps = (rows + p.n_splits - 1) / p.n_splits;
    a.rows_per_split = ((rps + TN - 1) / TN) * TN;
    const uint32_t bits = p.x.row_bytes * 8;
    const int eb = p.storage == VSB_ST_F32 ? 32 : (p.storage == VSB_ST_F16 || p.storage == VSB_ST_BF16) ? 16
                   : p.storage == VSB_ST_I8 ? 8 : 1;
    const uint32_t elems = bits / eb;
    a.n_slabs = (elems + BK - 1) / BK;
    a.part = p.part;
    dim3 grid((p.q.n + TQ - 1) / TQ, p.n_splits);
    const size_t smem = (size_t)(BK * TQ + BK * TN) * 4 + (size_t)TQ * p.kp * 8 + (size_t)TQ * BUFCAP * 8 + TQ * 8;
    VSB_DISPATCH_PAIR(p.storage, p.metric, (launch_k1<ST, METRIC>(a, grid, smem, stream)));
    g_kernel_launches += 1;
}

uint32_t exact_scan_pick_splits(uint32_t nq, uint32_t n_rows, int sm_count) {
    const uint32_t q_blocks = (nq + SCAN_QB - 1) / SCAN_QB;
    const uint32_t want = (4u * (uint32_t)sm_count + q_blocks - 1) / q_blocks;
    const uint32_t max_by_rows = (n_rows + 1023) / 1024;
    uint32_t s = want < max_by_rows ? want : max_by_rows;
    return s < 1 ? 1 : s;
}

uint32_t exact_scan_lists_per_query(uint32_t n_splits) { return n_splits * SCAN_WARPS; }

void launch_exact_scan(const ExactParams& p, uint32_t k, cudaStream_t stream) {
    if (p.q.n == 0 || p.x_hi <= p.x_lo) return;
    ScanArgs a;
    a.q_rows = p.q.rows; a.q_nrm = p.q.nrm; a.nq = p.q.n; a.q_row_bytes = p.q.row_bytes;
    a.x_rows = p.x.rows; a.x_nrm = p.x.nrm; a.x_row_bytes = p.x.row_bytes; a.x_lo = p.x_lo; a.x_hi = p.x_hi;
    a.deny = p.deny; a.keys = p.keys; a.allow = p.allow.bm; a.allow_bits = p.allow.bits; a.allow_of_q = p.allow.of_q;
    a.kf = p.kp;  // the caller sets kp = round_up(k (+1 for self), 32): lists hold exactly what K3 needs
    (void)k;
    a.n_splits = p.n_splits;
    const uint32_t rows = p.x_hi - p.x_lo;
    a.rows_per_split = ((rows + p.n_splits - 1) / p.n_splits + 31) / 32 * 32;
    a.part = p.part;
    dim3 grid((p.q.n + SCAN_QB - 1) / SCAN_QB, p.n_splits);
    const size_t smem = (size_t)SCAN_WARPS * SCAN_QB * a.kf * 8;
    VSB_DISPATCH_PAIR(p.storage, p.metric, (launch_scan<ST, METRIC>(a, grid, smem, stream)));
    g_kernel_launches += 1;
}

void launch_max_norm(const float* nrm, uint32_t lo, uint32_t hi, float* out, cudaStream_t stream) {
    cudaMemsetAsync(out, 0, sizeof(float), stream);
    if (hi <= lo) return;
    const uint32_t blocks = std::min<uint32_t>((hi - lo + 1023) / 1024, 296);
    max_norm_kernel<<<blocks, 256, 0, stream>>>(nrm, lo, hi, out);
    g_kernel_launches += 1;
}

void launch_exact_rerank(const ExactParams& p, uint32_t k, uint64_t* out_keys, float* out_dists,
                         uint32_t* out_counts, uint64_t* out_packed, int64_t self_base, cudaStream_t stream,
                         const ExactCert* cert, const uint32_t* q_map) {
    if (p.q.n == 0) return;
    K3Args a;
    a.q_rows = p.q.rows; a.q_nrm = p.q.nrm; a.nq = p.q.n; a.q_row_bytes = p.q.row_bytes;
    a.x_rows = p.x.rows; a.x_nrm = p.x.nrm; a.x_row_bytes = p.x.row_bytes;
    a.keys = p.keys; a.part = p.part; a.kp = p.kp; a.n_splits = p.n_splits;
    a.k = k; a.kf = ((k + 31) / 32) * 32;
    a.out_keys = out_keys; a.out_dists = out_dists; a.out_counts = out_counts; a.out_packed = out_packed;
    a.self_base = self_base;
    a.x_nrm_max = cert ? cert->x_nrm_max : nullptr;
    a.cert_rel = cert ? cert->rel : 0.0f;
    a.cert_sum = cert ? cert->sum : 0.0f;
    a.uncert_flags = cert ? cert->flags : nullptr;
    a.uncert_count = cert ? cert->count : nullptr;
    a.q_map = q_map;
    // small batches: a CTA per query (candidates spread over 8 warps) instead of a warp per query
    const bool cta = p.q.n <= 1024 && a.kp >= 8;
    VSB_DISPATCH_PAIR(p.storage, p.metric, (launch_k3<ST, METRIC>(a, cta, stream)));
    g_kernel_launches += 1;
}

void launch_range_candidates(const ExactParams& p, const RangeParams& r, cudaStream_t stream) {
    if (p.q.n == 0 || p.x_hi <= p.x_lo) return;
    ExactParams pr = p;
    pr.kp = 0;
    K1Args a;
    a.q_rows = pr.q.rows; a.q_sq = pr.q.sq; a.q_nrm = pr.q.nrm; a.nq = pr.q.n; a.q_row_bytes = pr.q.row_bytes;
    a.x_rows = pr.x.rows; a.x_sq = pr.x.sq; a.x_nrm = pr.x.nrm; a.x_row_bytes = pr.x.row_bytes;
    a.x_lo = pr.x_lo; a.x_hi = pr.x_hi;
    a.deny = pr.deny; a.keys = pr.keys; a.allow = pr.allow.bm; a.allow_bits = pr.allow.bits; a.allow_of_q = pr.allow.of_q;
    a.kp = 0; a.n_splits = pr.n_splits;
    const uint32_t rows = pr.x_hi - pr.x_lo;
    const uint32_t rps = (rows + pr.n_splits - 1) / pr.n_splits;
    a.rows_per_split = ((rps + TN - 1) / TN) * TN;
    const int eb = pr.storage == VSB_ST_F32 ? 32 : (pr.storage == VSB_ST_F16 || pr.storage == VSB_ST_BF16) ? 16
                   : pr.storage == VSB_ST_I8 ? 8 : 1;
    a.n_slabs = (pr.x.row_bytes * 8 / eb + BK - 1) / BK;
    a.part = nullptr;
    a.range = r;
    dim3 grid((pr.q.n + TQ - 1) / TQ, pr.n_splits);
    const size_t smem = (size_t)(BK * TQ + BK * TN) * 4 + (size_t)TQ * BUFCAP * 8 + TQ * 8;
    VSB_DISPATCH_PAIR(pr.storage, pr.metric, (launch_k1<ST, METRIC, true>(a, grid, smem, stream)));
    g_kernel_launches += 1;
}

void launch_range_bound(int storage, int metric, const float* q_nrm, const float* max_distance, uint32_t n,
                        const float* x_nrm_max, float rel, float sum, float* thr, cudaStream_t stream) {
    if (n == 0) return;
    VSB_DISPATCH_PAIR(storage, metric,
                      (range_bound_kernel<ST, METRIC><<<(n + 255) / 256, 256, 0, stream>>>(q_nrm, max_distance, n, x_nrm_max,
                                                                                             rel, sum, thr)));
    g_kernel_launches += 1;
}

void launch_range_eval(const ExactParams& p, const float* max_distance, const uint32_t* count, const uint32_t* cursor,
                       const uint32_t* seg_off, const uint32_t* grp_off, uint32_t n_groups, const uint64_t* cand,
                       uint64_t* key_out, uint32_t* dord_out, uint32_t* kept, uint32_t* mismatch, cudaStream_t stream) {
    if (p.q.n == 0) return;
    range_check_kernel<<<(p.q.n + 255) / 256, 256, 0, stream>>>(count, cursor, p.q.n, mismatch);
    g_kernel_launches += 1;
    if (n_groups == 0) return;
    K3Args a{};
    a.q_rows = p.q.rows; a.q_nrm = p.q.nrm; a.nq = p.q.n; a.q_row_bytes = p.q.row_bytes;
    a.x_rows = p.x.rows; a.x_nrm = p.x.nrm; a.x_row_bytes = p.x.row_bytes;
    a.keys = p.keys;
    const uint32_t blocks = (n_groups + RE_WARPS - 1) / RE_WARPS;
    VSB_DISPATCH_PAIR(p.storage, p.metric,
                      (range_eval_kernel<ST, METRIC><<<blocks, RE_WARPS * 32, 0, stream>>>(
                          a, max_distance, count, cursor, seg_off, grp_off, n_groups, cand, key_out, dord_out, kept, mismatch)));
    g_kernel_launches += 1;
}

// Two segmented passes: by key (unique among live rows), then a STABLE pass by distance, which leaves equal
// distances in key order.
size_t range_sort_temp_bytes(uint32_t n_entries, uint32_t n_segments) {
    size_t a = 0, b = 0;
    cub::DeviceSegmentedSort::SortPairs(nullptr, a, (const uint64_t*)nullptr, (uint64_t*)nullptr, (const uint32_t*)nullptr,
                                        (uint32_t*)nullptr, (int)n_entries, (int)n_segments, (const uint32_t*)nullptr,
                                        (const uint32_t*)nullptr);
    cub::DeviceSegmentedSort::StableSortPairs(nullptr, b, (const uint32_t*)nullptr, (uint32_t*)nullptr,
                                              (const uint64_t*)nullptr, (uint64_t*)nullptr, (int)n_entries, (int)n_segments,
                                              (const uint32_t*)nullptr, (const uint32_t*)nullptr);
    return std::max(a, b);
}

cudaError_t launch_range_sort(uint32_t* dord, uint64_t* key, uint32_t* alt_dord, uint64_t* alt_key, uint32_t n_entries,
                              const uint32_t* seg_off, uint32_t n_segments, void* temp, size_t temp_bytes,
                              cudaStream_t stream) {
    if (n_entries == 0) return cudaSuccess;
    size_t tb = temp_bytes;
    cudaError_t e = cub::DeviceSegmentedSort::SortPairs(temp, tb, key, alt_key, dord, alt_dord, (int)n_entries, (int)n_segments,
                                                        seg_off, seg_off + 1, stream);
    if (e != cudaSuccess) return e;
    tb = temp_bytes;
    e = cub::DeviceSegmentedSort::StableSortPairs(temp, tb, alt_dord, dord, alt_key, key, (int)n_entries, (int)n_segments,
                                                  seg_off, seg_off + 1, stream);
    g_kernel_launches += 2;
    return e;
}

void launch_range_emit(const uint32_t* dord, const uint64_t* key, const uint32_t* seg_off, const uint32_t* out_off,
                       uint32_t n, uint32_t total, uint64_t* keys_out, float* dists_out, cudaStream_t stream) {
    if (total == 0) return;
    range_emit_kernel<<<(total + 255) / 256, 256, 0, stream>>>(dord, key, seg_off, out_off, n, total, keys_out, dists_out);
    g_kernel_launches += 1;
}

}  // namespace vsb
