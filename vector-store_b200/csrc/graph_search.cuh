// graph_search.cuh — K4: warp-per-query beam search over the fixed-degree graph.
//
// Replaces the HNSW base-layer traversal inside usearch::Index::search (reference call site
// vs_index/usearch.rs:203-222, SURVEY §8a A7).  One warp owns one query:
//   * the query lives in registers (each lane keeps the 16-byte chunks it will ever touch);
//   * the candidate list (itopk = ef entries, packed ord(dist)<<32|slot, ascending) and the
//     visited hash live in shared memory;
//   * every iteration expands the best un-expanded candidate: one coalesced 128-byte read of its
//     graph row, a visited-hash filter, then the surviving neighbours' vectors are streamed with
//     128-bit ld.global.nc loads (a 1536-byte bf16 row = 3 fully coalesced warp loads),
//     reduced with the canonical butterfly, sorted with a shuffle bitonic network and folded
//     into the list.
// HBM-bound by design: bytes/query = E * row_bytes + P * R * 4 (E, P counted in-kernel).
#pragma once
#ifdef VSB_K4B_PROFILE
#include <cstdio>
#endif
#include "kernels.h"
#include "select.cuh"

namespace vsb {

constexpr int K4_WARPS = 4;
constexpr uint32_t kHashEmpty = 0xFFFFFFFFu;

struct K4Args {
    const uint8_t* q_rows;
    const float* q_nrm;
    uint32_t nq, q_row_bytes;
    const uint8_t* x_rows;
    const float* x_nrm;
    uint32_t x_row_bytes;
    const uint32_t* graph;
    uint32_t graph_stride, degree;
    const uint64_t* seed_lists;  // [nq][seed_splits][32]
    uint32_t seed_splits, n_seeds;
    const uint32_t* seed_slots;
    const uint32_t* deny;
    const uint64_t* keys;
    uint32_t itopk, max_iters, k, hash_bits, search_width, queue_cap;
    int metric;
    uint64_t* out_keys;
    float* out_dists;
    uint32_t* out_counts;
    uint64_t* out_packed;  // if set: emit the first k live entries as packed (ord(dist)<<32 | slot) for K3 instead of keys
    long long self_base;   // >= 0: query i is row self_base + i of x and is left out of its own result
    uint32_t out_stride;   // entries per query in out_packed (>= k; the rest is padded with kInvalidPacked)
    unsigned long long* counters;
    const uint32_t* allow;  // filtered ANN: admissibility bitmap over (key & 2^48-1); only the FILTER instantiation reads it
    uint64_t allow_bits;
    const uint32_t* allow_of_q;  // [nq] bitmap index per query (nullable: bitmap 0)
    uint32_t rk;            // length of the result list of the FILTER instantiation (k rounded up to 32)
    uint32_t mma;           // 1: 16-bit rows are evaluated on the tensor cores (mma.sync), distances are candidate-grade
    uint32_t compact;       // 1: survivors of an iteration are compacted before the sort + merge
    uint32_t l2pf;          // rows of prefetch distance into L2 (0 = off), warp-per-query kernel
};

__device__ __forceinline__ bool hash_insert(uint32_t* tab, uint32_t mask, uint32_t bits, uint32_t slot) {
    uint32_t h = (slot * 0x9E3779B1u) >> (32 - bits);
#pragma unroll 1
    for (int probe = 0; probe < 64; ++probe) {
        const uint32_t old = atomicCAS(&tab[h], kHashEmpty, slot);
        if (old == kHashEmpty) return true;
        if (old == slot) return false;
        h = (h + 1) & mask;
    }
    return false;  // saturated neighbourhood: treat as visited
}

// Visited filter of the warp-per-query kernel: the same open-addressing table with 16-bit TAGS instead of the
// 32-bit slot ids.  Half the shared memory per query (8 KB for 4096 entries) is what lets a fourth / fifth CTA
// fit on the SM — the kernel is bound by rows in flight per SM.  Two different slots that share a probe position
// AND a tag read as "visited": ~2 probes x 2^-16 per insert, i.e. one skipped candidate in ~12 queries of 2600
// evaluations each, far below the recall resolution (checked by the ANN recall tests).
constexpr uint16_t kTagEmpty = 0xFFFFu;
__device__ __forceinline__ bool hash_insert16(uint16_t* tab, uint32_t mask, uint32_t bits, uint32_t slot) {
    uint32_t h = (slot * 0x9E3779B1u) >> (32 - bits);
    uint32_t t = (slot * 0x85EBCA6Bu) >> 16;
    const unsigned short tag = (unsigned short)(t == kTagEmpty ? 0xFFFEu : t);
#pragma unroll 1
    for (int probe = 0; probe < 64; ++probe) {
        const unsigned short old = atomicCAS(reinterpret_cast<unsigned short*>(&tab[h]), (unsigned short)kTagEmpty, tag);
        if (old == kTagEmpty) return true;
        if (old == tag) return false;
        h = (h + 1) & mask;
    }
    return false;  // saturated neighbourhood: treat as visited
}

// ---- shared evaluation helpers (K4 and K4b) -----------------------------------------------------
// A "group" is U stored rows in flight in registers.  Loads are unpredicated when every lane owns a
// full set of chunks (`full`), and indices past the end of the queue are clamped to its last entry
// (the duplicate result is simply not written back), so the hot loop carries no per-chunk predicates.
template <int CPL, int U>
struct VecGroup {
    uint4 x[U][CPL];
};

template <int CPL, int U>
__device__ __forceinline__ void group_load(VecGroup<CPL, U>& g, const uint8_t* __restrict__ x_rows, uint32_t row_bytes,
                                           const uint32_t* newq, uint32_t base, uint32_t stride, uint32_t last,
                                           int lane, int n_chunks, bool full) {
#pragma unroll
    for (int u = 0; u < U; ++u) {
        uint32_t idx = base + u * stride;
        idx = idx < last ? idx : last;
        const uint4* xrow = reinterpret_cast<const uint4*>(x_rows + (size_t)newq[idx] * row_bytes) + lane;
        if (full) {
#pragma unroll
            for (int j = 0; j < CPL; ++j) g.x[u][j] = ldg_nc_v4(xrow + j * 32);
        } else {
#pragma unroll
            for (int j = 0; j < CPL; ++j) {
                g.x[u][j] = make_uint4(0, 0, 0, 0);
                if (j * 32 + lane < n_chunks) g.x[u][j] = ldg_nc_v4(xrow + j * 32);
            }
        }
    }
}

// raw = canonical butterfly sum (dot or squared-L2) as float; integer storages convert once at the end
template <int ST, int CPL, int U>
__device__ __forceinline__ void group_reduce(const VecGroup<CPL, U>& g, const float* qf, const uint4* qc, bool is_l2,
                                             float* newd, uint32_t base, uint32_t stride, uint32_t n_new, int lane) {
    constexpr int E = Storage<ST>::ELEMS;
    constexpr bool kFloat = Storage<ST>::kFloat;
#pragma unroll
    for (int u = 0; u < U; ++u) {
        const uint32_t idx = base + u * stride;
        float raw;
        if constexpr (kFloat) {
            float f;
            if (is_l2) {
                ChunkAcc<ST, VSB_METRIC_L2SQ> acc;
#pragma unroll
                for (int j = 0; j < CPL; ++j) {
                    float xf[E];
                    Storage<ST>::unpack(g.x[u][j], xf);
                    acc.add_f(&qf[j * E], xf);
                }
                f = acc.f;
            } else {
                ChunkAcc<ST, VSB_METRIC_IP> acc;
#pragma unroll
                for (int j = 0; j < CPL; ++j) {
                    float xf[E];
                    Storage<ST>::unpack(g.x[u][j], xf);
                    acc.add_f(&qf[j * E], xf);
                }
                f = acc.f;
            }
            raw = butterfly_sum(f);
        } else {
            int i;
            if (is_l2) {
                ChunkAcc<ST, VSB_METRIC_L2SQ> acc;
#pragma unroll
                for (int j = 0; j < CPL; ++j) acc.add(qc[j], g.x[u][j]);
                i = acc.i;
            } else {
                ChunkAcc<ST, VSB_METRIC_IP> acc;
#pragma unroll
                for (int j = 0; j < CPL; ++j) acc.add(qc[j], g.x[u][j]);
                i = acc.i;
            }
            raw = (float)butterfly_sum_i(i);
        }
        if (lane == 0 && idx < n_new) newd[idx] = raw;
    }
}

// raw sum -> distance; the same arithmetic as finish_distance (common.cuh), executed once per candidate
// by the lane that owns it instead of once per candidate by the whole warp
template <int ST>
__device__ __forceinline__ float finish_raw(float raw, int metric, float qn, float xn) {
    if constexpr (ST == VSB_ST_B1) {
        return raw;
    } else {
        if (metric == VSB_METRIC_L2SQ) return raw;
        if (metric == VSB_METRIC_IP) {
            if constexpr (ST == VSB_ST_I8) raw = __fdiv_rn(raw, 16129.0f);
            return __fsub_rn(1.0f, raw);
        }
        if (qn == 0.0f && xn == 0.0f) return 0.0f;
        if (qn == 0.0f || xn == 0.0f) return 1.0f;
        float d = __fsub_rn(1.0f, __fdiv_rn(raw, __fmul_rn(qn, xn)));
        d = d < 0.0f ? 0.0f : d;
        d = d > 2.0f ? 2.0f : d;
        return d;
    }
}

// ---- tensor-core evaluation of 16-bit rows (warp-per-query kernel) -------------------------------------------------
// mma.sync.m16n8k16 (bf16 / f16 in, fp32 accumulate).  The unpack of bf16 rows to fp32 was the hottest line of the SIMT
// evaluation (one shift or mask per element before every FFMA); the tensor core consumes the packed rows as they come
// out of the 128-bit loads.  A first layout that gave each thread quad 64 contiguous bytes of 16 different rows
// (natural for the fragments) was measured SLOWER than SIMT once the per-row pieces dropped to 192 bytes per pipeline
// stage (10.1 vs 9.2 ms): HBM wants long contiguous bursts per row.  group_reduce_mma therefore keeps the SIMT
// kernel's loads (one warp load = 512 contiguous bytes of one row) and adapts the fragments to them.  The accumulation
// order is the tensor core's, not the canonical one: results are candidate-grade and the caller re-ranks what it
// returns (K3).
template <int ST>
__device__ __forceinline__ void mma_16816(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                                          uint32_t b1) {
    if constexpr (ST == VSB_ST_BF16) {
        asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                     : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                     : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
    } else {
        asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                     : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                     : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
    }
}

// tensor-core form of group_reduce for one group of U rows held in registers (same loads, same double buffering as the
// SIMT form): rows are taken two at a time, lane l's 16-byte piece of row u fills the fragment slots of MMA row
// g = l / 4 (piece of row u + 1: MMA row g + 8), lane l's piece of the query fills column g.  D[g][g] is then the
// partial dot product of the pieces held by quad g (D[g + 8][g] for the second row); the off-diagonal entries pair
// pieces of different offsets and are ignored.  The diagonal entry of quad g sits in thread t = g / 2, register g % 2.
template <int ST, int CPL, int U>
__device__ __forceinline__ void group_reduce_mma(const VecGroup<CPL, U>& grp, const uint4* qc, float* newd, uint32_t base,
                                                 uint32_t stride, uint32_t n_new, int lane) {
    const int g = lane >> 2, t = lane & 3;
    const bool diag = t == (g >> 1);
    const bool odd = (g & 1) != 0;
#pragma unroll
    for (int u = 0; u < U; u += 2) {
        constexpr bool kPair = U > 1;
        float c[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int j = 0; j < CPL; ++j) {
            const uint4 xa = grp.x[u][j];
            const uint4 xb = kPair ? grp.x[kPair ? u + 1 : u][j] : xa;
            mma_16816<ST>(c, xa.x, xb.x, xa.y, xb.y, qc[j].x, qc[j].y);
            mma_16816<ST>(c, xa.z, xb.z, xa.w, xb.w, qc[j].z, qc[j].w);
        }
        float v0 = diag ? (odd ? c[1] : c[0]) : 0.0f;
        float v1 = diag ? (odd ? c[3] : c[2]) : 0.0f;
        v0 = butterfly_sum(v0);
        if (kPair) v1 = butterfly_sum(v1);
        if (lane == 0) {
            const uint32_t i0 = base + u * stride, i1 = base + (u + 1) * stride;
            if (i0 < n_new) newd[i0] = v0;
            if (kPair && i1 < n_new) newd[i1] = v1;
        }
    }
}

// all queue entries of this warp: index(m) = first + m * stride, m < mine.  Double buffered: the loads of
// group m+1 are in flight while group m is reduced.
// whole-row prefetch into L2 by the bulk-copy engine: one instruction per row, nothing comes back to the SM
__device__ __forceinline__ void prefetch_row_l2(const void* p, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}

// l2pf > 0: rows `l2pf` positions ahead of the group being loaded are prefetched into L2 (all rows of an iteration are
// known when it starts).  The register double buffer holds at most 2 U rows in flight per warp; at HBM latency that is
// what bounds the kernel, at L2 latency it is plenty — the bulk prefetches carry the HBM latency instead and cost
// neither registers nor issue slots.
template <int ST, int CPL, int U, bool MMA = false>
__device__ __forceinline__ void evaluate_entries(const uint8_t* __restrict__ x_rows, uint32_t row_bytes,
                                                 const uint32_t* newq, float* newd, uint32_t first, uint32_t stride,
                                                 uint32_t mine, uint32_t n_new, const float* qf, const uint4* qc,
                                                 bool is_l2, int lane, int n_chunks, bool full, uint32_t l2pf = 0) {
    if (mine == 0) return;
    const uint32_t last = first + (mine - 1) * stride;
    if (l2pf != 0) {
        for (uint32_t m = 2 * U + lane; m < l2pf + 2 * U && m < mine; m += 32)
            prefetch_row_l2(x_rows + (size_t)newq[first + m * stride] * row_bytes, row_bytes);
    }
    auto reduce = [&](const VecGroup<CPL, U>& grp, uint32_t base) {
        if constexpr (MMA) group_reduce_mma<ST, CPL, U>(grp, qc, newd, base, stride, n_new, lane);
        else group_reduce<ST, CPL, U>(grp, qf, qc, is_l2, newd, base, stride, n_new, lane);
    };
    VecGroup<CPL, U> ga, gb;
    group_load<CPL, U>(ga, x_rows, row_bytes, newq, first, stride, last, lane, n_chunks, full);
    for (uint32_t m0 = 0; m0 < mine; m0 += 2 * U) {
        const bool has_b = m0 + U < mine;
        if (l2pf != 0) {
            const uint32_t m = m0 + 2 * U + l2pf + lane;
            if (lane < 2 * U && m < mine) prefetch_row_l2(x_rows + (size_t)newq[first + m * stride] * row_bytes, row_bytes);
        }
        if (has_b) group_load<CPL, U>(gb, x_rows, row_bytes, newq, first + (m0 + U) * stride, stride, last, lane, n_chunks, full);
        reduce(ga, first + m0 * stride);
        if (has_b) {
            if (m0 + 2 * U < mine)
                group_load<CPL, U>(ga, x_rows, row_bytes, newq, first + (m0 + 2 * U) * stride, stride, last, lane, n_chunks, full);
            reduce(gb, first + (m0 + U) * stride);
        }
    }
}

// Compile-time cap of search_width.  8 was measured: the wider unrolled parent / neighbour loops slow EVERY width down
// (1.25 M x 768 bf16, ef 64, 2 parents: 3.65 ms with a cap of 4, 4.39 ms with a cap of 8), which costs more than
// 8 parents per iteration gain on long searches.
#ifndef VSB_K4_MAX_WIDTH
#define VSB_K4_MAX_WIDTH 4
#endif
constexpr int K4_MAX_WIDTH = VSB_K4_MAX_WIDTH;  // parents expanded per iteration (search_width)

// resident CTAs per SM the register budget is sized for: short int8 rows (the scaled-int8 traversal copy) need
// few load registers, and the kernel is bound by the number of rows in flight per SM, not by bytes
// tools/rowgather_probe.py (profiles/r2_random_row_gather_probe.jsonl): a kernel that does nothing but gather random
// 1.5 KB rows reaches 6.6 TB/s with >= 32 resident warps x 2 rows in flight, 4.4 TB/s with 16 warps x 4 rows, 2.6 TB/s
// with 8 warps x 8 rows: the ceiling for this access pattern is the copy peak, but only with ~100 rows in flight per
// SM.  K4 holds 12 warps x <= 8 rows with a ~50 % duty cycle, which is where its 0.75 comes from.  Measured and NOT
// kept: 2 rows per group + four CTAs per SM for the tensor-core form (117 registers, 16 warps: 8.8 ms vs 8.3-8.6 ms).
template <int ST, int CPL, bool MMA = false>
constexpr int k4_min_blocks() { return (ST == VSB_ST_I8 && CPL <= 2) ? 4 : 3; }
template <int CPL, bool MMA>
constexpr int k4_rows_per_group() { return CPL <= 3 ? 4 : (CPL <= 6 ? 2 : 1); }

// FILTER = true (vsb_search_filtered): the traversal is unchanged, but every evaluated row whose key is admissible is
// ALSO folded into a second list of rk entries, and that list is what the kernel emits.  The beam still walks through
// inadmissible rows, exactly like usearch's predicate search (usearch.rs:224-248).
// MMA = true (16-bit float storages): the rows of a group are multiplied on the tensor cores (group_reduce_mma) instead
// of being unpacked and FMA'd lane by lane; the query stays packed in registers; the distances are candidate-grade.
template <int ST, int CPL, bool FILTER, bool MMA = false>
__global__ void __launch_bounds__(K4_WARPS * 32, k4_min_blocks<ST, CPL, MMA>()) graph_search_kernel(K4Args a) {
    constexpr int E = Storage<ST>::ELEMS;
    constexpr bool kFloat = Storage<ST>::kFloat;
    constexpr int U = k4_rows_per_group<CPL, MMA>();  // vectors per load group
    constexpr int QF = (kFloat && !MMA) ? CPL * E : 1;

    extern __shared__ __align__(16) uint8_t smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t q = blockIdx.x * K4_WARPS + warp;
    if (q >= a.nq) return;

    const uint32_t hsize = 1u << a.hash_bits, hmask = hsize - 1;
    const uint32_t qcap = a.queue_cap;
    const size_t per_warp = (size_t)a.itopk * 8 + (size_t)hsize * 2 + (size_t)qcap * 8 + (FILTER ? (size_t)a.rk * 8 : 0) + 64 * 8;
    uint64_t* list = reinterpret_cast<uint64_t*>(smem_raw + (size_t)warp * per_warp);
    uint16_t* hash = reinterpret_cast<uint16_t*>(list + a.itopk);  // [hsize] 16-bit tags
    uint32_t* newq = reinterpret_cast<uint32_t*>(hash + hsize);   // [qcap] un-visited neighbour slots of this iteration
    float* newd = reinterpret_cast<float*>(newq + qcap);     // [qcap] their raw sums
    uint64_t* rlist = reinterpret_cast<uint64_t*>(newd + qcap);  // [rk] FILTER: best admissible rows seen so far
    uint64_t* stage = rlist + (FILTER ? a.rk : 0);               // [64] candidates of this iteration that can enter the list
    const uint32_t* allow = nullptr;  // FILTER: this query's own bitmap
    if constexpr (FILTER) {
        for (uint32_t i = lane; i < a.rk; i += 32) rlist[i] = kInvalidPacked;
        allow = query_allow(a.allow, a.allow_bits, a.allow_of_q, q);
    }
    const LessBySlot less;
    const bool is_l2 = a.metric == VSB_METRIC_L2SQ;
    const bool is_cos = a.metric == VSB_METRIC_COS;
    const int n_chunks = a.x_row_bytes / 16;
    const bool full = n_chunks == CPL * 32;

    for (uint32_t i = lane; i < a.itopk; i += 32) list[i] = kInvalidPacked;
    for (uint32_t i = lane; i < hsize; i += 32) hash[i] = kTagEmpty;

    // ---- query into registers ----
    const uint4* qrow = reinterpret_cast<const uint4*>(a.q_rows + (size_t)q * a.q_row_bytes);
    float qf[QF];
    uint4 qc[(kFloat && !MMA) ? 1 : CPL];  // integer storages and the tensor-core form keep the query packed
#pragma unroll
    for (int j = 0; j < CPL; ++j) {
        const int c = j * 32 + lane;
        uint4 v = make_uint4(0, 0, 0, 0);
        if (c < n_chunks) v = qrow[c];
        if constexpr (kFloat && !MMA)
            Storage<ST>::unpack(v, &qf[j * E]);
        else
            qc[j] = v;
    }
    if constexpr (MMA) qf[0] = 0.0f;
    const float qn = a.q_nrm[q];
    __syncwarp();

    uint32_t n_hashed = 0, n_new = 0;
    unsigned long long n_evals = 0, n_parents = 0;

    // visited filter + compaction of one candidate per lane into the iteration queue
    auto enqueue = [&](uint32_t nb) {
        bool is_new = false;
        if (nb != kInvalidSlot) is_new = hash_insert16(hash, hmask, a.hash_bits, nb);
        const uint32_t m = __ballot_sync(kFullMask, is_new);
        if (is_new) newq[n_new + __popc(m & ((1u << lane) - 1))] = nb;
        n_new += __popc(m);
        n_hashed += __popc(m);
    };

    // distances of everything queued, then fold the candidates that can still enter the list
    auto evaluate_queue = [&]() {
        __syncwarp();
        if (n_new == 0) return;
        n_evals += n_new;
        // MMA: the candidates' norms are a dependent gather that would otherwise start only after the rows have been
        // multiplied, with nothing else of this warp in flight — fetch the first 64 before the rows
        float xn_pre[2] = {0.0f, 0.0f};
        if constexpr (MMA) {
            if (is_cos || is_l2) {
                if (lane < n_new) xn_pre[0] = __ldg(a.x_nrm + newq[lane]);
                if (32 + lane < n_new) xn_pre[1] = __ldg(a.x_nrm + newq[32 + lane]);
            }
        }
        evaluate_entries<ST, CPL, U, MMA>(a.x_rows, a.x_row_bytes, newq, newd, 0, 1, n_new, n_new, qf, qc, is_l2, lane,
                                          n_chunks, full, a.l2pf);
        __syncwarp();
        // Candidates that cannot enter the list (most of them once the beam has converged) are dropped first and the
        // survivors of ALL batches of this iteration are compacted into `stage`, so the shuffle sort + list merge — the
        // longest dependent chain of an iteration — runs once per 32 survivors, not once per 32 candidates.
        uint64_t worst = list[a.itopk - 1];
        uint32_t n_stage = 0;
        auto fold_stage = [&](uint32_t n) {  // sort + merge stage[0, n), n <= 32
            __syncwarp();
            uint64_t v = lane < n ? stage[lane] : kInvalidPacked;
            v = warp_sort32(v, lane, less);
            warp_list_merge(list, (int)a.itopk, v, lane, less);
            worst = list[a.itopk - 1];
        };
        for (uint32_t base = 0; base < n_new; base += 32) {
            uint64_t res = kInvalidPacked;
            if (base + lane < n_new) {
                const uint32_t slot = newq[base + lane];
                float xn = 0.0f;
                if (MMA && base < 64) xn = base == 0 ? xn_pre[0] : xn_pre[1];
                else if (is_cos || (MMA && is_l2)) xn = __ldg(a.x_nrm + slot);
                float raw = newd[base + lane];
                if constexpr (MMA) {
                    // the tensor-core sum is the dot product; squared L2 from the norms (candidate-grade like the rest)
                    if (is_l2) raw = fmaxf(fmaf(-2.0f, raw, fmaf(qn, qn, xn * xn)), 0.0f);
                }
                res = pack_ds(finish_raw<ST>(raw, a.metric, qn, xn), slot);
            }
            if constexpr (FILTER) {
                uint64_t adm = kInvalidPacked;
                if (res != kInvalidPacked) {
                    const uint64_t row_id = a.keys[packed_lo(res)] & kRowMask48;
                    if (row_id < a.allow_bits && (allow[row_id >> 5] >> (row_id & 31) & 1u)) adm = res;
                }
                if (__ballot_sync(kFullMask, adm < rlist[a.rk - 1]) != 0) {
                    adm = warp_sort32(adm, lane, less);
                    warp_list_merge(rlist, (int)a.rk, adm, lane, less);
                }
            }
            const bool keep = res < worst;
            const uint32_t km = __ballot_sync(kFullMask, keep);
            if (km == 0) continue;  // nothing here can enter the list
            if (!a.compact || n_new <= 32) {  // a single batch (or VSB_K4_COMPACT=0): sort + merge it directly
                res = warp_sort32(res, lane, less);
                warp_list_merge(list, (int)a.itopk, res, lane, less);
                continue;
            }
            if (keep) stage[n_stage + __popc(km & ((1u << lane) - 1))] = res;  // < 64 entries
            n_stage += __popc(km);
            if (n_stage >= 32) {
                fold_stage(32);
                __syncwarp();
                const uint64_t mv = lane + 32 < n_stage ? stage[32 + lane] : kInvalidPacked;
                __syncwarp();
                if (lane + 32 < n_stage) stage[lane] = mv;
                n_stage -= 32;
            }
        }
        if (n_stage != 0) fold_stage(n_stage);
        n_new = 0;
    };

    // ---- seeds: the seed layer hands over `seed_splits` blocks of 32 packed (distance, seed index)
    // entries (sorted lists from K1, or unsorted per-tile winners from the tensor-core kernel) ----
    {
        uint64_t sv = kInvalidPacked;
        for (uint32_t s = 0; s < a.seed_splits; ++s) {
            uint64_t v = a.seed_lists[((size_t)q * a.seed_splits + s) * 32 + lane];
            v = warp_sort32(v, lane, less);
            const uint64_t rc = shfl_u64(v, 31 - lane);
            sv = warp_bitonic_merge32(rc < sv ? rc : sv, lane, less);
        }
        uint32_t nb = kInvalidSlot;
        if (lane < (int)a.n_seeds && sv != kInvalidPacked) nb = a.seed_slots[packed_lo(sv)];
        enqueue(nb);
        evaluate_queue();
    }

    // ---- main loop ----
    const uint32_t width = a.search_width;
    for (uint32_t it = 0; it < a.max_iters; ++it) {
        // visited hash getting crowded: forget everything except what is still in the list
        if (n_hashed > (hsize >> 2) * 3) {
            for (uint32_t i = lane; i < hsize; i += 32) hash[i] = kTagEmpty;
            __syncwarp();
            n_hashed = 0;
            for (uint32_t b = 0; b < a.itopk; b += 32) {
                const uint64_t e = list[b + lane];
                if (e != kInvalidPacked) hash_insert16(hash, hmask, a.hash_bits, packed_lo(e) & ~kExpandedBit);
                n_hashed += __popc(__ballot_sync(kFullMask, e != kInvalidPacked));
            }
            __syncwarp();
        }
        // best un-expanded candidates (up to `width`)
        uint32_t par[K4_MAX_WIDTH];
        uint32_t np = 0;
#pragma unroll
        for (int i = 0; i < K4_MAX_WIDTH; ++i) par[i] = kInvalidSlot;
        for (uint32_t b = 0; b < a.itopk && np < width; b += 32) {
            const uint64_t e = list[b + lane];
            const bool unexp = e != kInvalidPacked && !(packed_lo(e) & kExpandedBit);
            uint32_t m = __ballot_sync(kFullMask, unexp);
            bool mine = false;
            while (m && np < width) {
                const int src = __ffs(m) - 1;
                m &= m - 1;
                const uint32_t pslot = __shfl_sync(kFullMask, packed_lo(e), src);
#pragma unroll
                for (int i = 0; i < K4_MAX_WIDTH; ++i)
                    if (i == (int)np) par[i] = pslot;
                if (lane == src) mine = true;
                ++np;
            }
            if (mine) list[b + lane] = e | kExpandedBit;
        }
        __syncwarp();
        if (np == 0) break;
        n_parents += np;
        // all graph rows of this iteration in flight together, then filter + queue
        uint32_t nbs[K4_MAX_WIDTH][2];
#pragma unroll
        for (int i = 0; i < K4_MAX_WIDTH; ++i) {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                nbs[i][h] = kInvalidSlot;
                const uint32_t r = h * 32 + lane;
                if (i < (int)np && r < a.degree) nbs[i][h] = __ldg(a.graph + (size_t)par[i] * a.graph_stride + r);
            }
        }
#pragma unroll
        for (int i = 0; i < K4_MAX_WIDTH; ++i) {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                if (i < (int)np && h * 32 < (int)a.degree) enqueue(nbs[i][h]);
            }
        }
        evaluate_queue();
    }

    // ---- emit the first k live entries (of the admissible list when filtering) ----
    __syncwarp();
    const uint64_t* src_list = FILTER ? rlist : list;
    const uint32_t src_len = FILTER ? a.rk : a.itopk;
    uint32_t count = 0;
    for (uint32_t b = 0; b < src_len; b += 32) {
        const uint64_t e = src_list[b + lane];
        const uint32_t slot = packed_lo(e) & ~kExpandedBit;
        bool valid = e != kInvalidPacked;
        if (valid && a.deny != nullptr && bit_test(a.deny, slot)) valid = false;
        if (valid && a.self_base >= 0 && slot == (uint32_t)(a.self_base + q)) valid = false;
        const uint32_t m = __ballot_sync(kFullMask, valid);
        const uint32_t pos = count + __popc(m & ((1u << lane) - 1));
        if (valid && pos < a.k) {
            if (a.out_packed != nullptr) {
                a.out_packed[(size_t)q * a.out_stride + pos] = ((uint64_t)packed_hi(e) << 32) | slot;
            } else {
                a.out_keys[(size_t)q * a.k + pos] = a.keys[slot];
                a.out_dists[(size_t)q * a.k + pos] = ord_to_f32(packed_hi(e));
            }
        }
        count += __popc(m);
    }
    if (count > a.k) count = a.k;
    if (a.out_packed != nullptr) {
        for (uint32_t i = count + lane; i < a.out_stride; i += 32) a.out_packed[(size_t)q * a.out_stride + i] = kInvalidPacked;
    }
    for (uint32_t i = count + lane; i < a.k; i += 32) {
        if (a.out_packed != nullptr) {
        } else {
            a.out_keys[(size_t)q * a.k + i] = 0xFFFFFFFFFFFFFFFFull;
            a.out_dists[(size_t)q * a.k + i] = __int_as_float(0x7F800000);
        }
    }
    if (lane == 0) {
        if (a.out_counts != nullptr) a.out_counts[q] = count;
        if (a.counters != nullptr) {
            atomicAdd(&a.counters[0], n_evals);
            atomicAdd(&a.counters[1], n_parents);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// K4b: CTA-per-query variant for small batches (batch-1 latency, SURVEY §8d "p99 batch-1").
// Same algorithm and the same canonical distances as the warp kernel, but 8 warps share one candidate
// list / visited hash and split every iteration's neighbour evaluations, and up to 8 parents are
// expanded per iteration, so a query needs ~ef/8 dependent memory round trips instead of ~ef.
constexpr int K4B_WARPS = 8;
constexpr int K4B_MAX_WIDTH = 8;
constexpr int K4B_PICK_ROUNDS = 4;  // list entries per thread in the parallel parent pick (itopk <= 1024)

// -DVSB_K4B_PROFILE: thread 0 of CTA 0 accumulates clock64() per phase of the iteration and prints the split
#ifdef VSB_K4B_PROFILE
#define K4B_T(i)                                       \
    do {                                               \
        const long long now_ = clock64();              \
        prof_[i] += now_ - prof_t_;                    \
        prof_t_ = now_;                                \
    } while (0)
#else
#define K4B_T(i) do { } while (0)
#endif

template <int ST, int CPL>
__global__ void __launch_bounds__(K4B_WARPS * 32, 1) graph_search_cta_kernel(K4Args a) {
    constexpr int E = Storage<ST>::ELEMS;
    constexpr bool kFloat = Storage<ST>::kFloat;
    constexpr int U = CPL <= 3 ? 4 : (CPL <= 6 ? 2 : 1);
    constexpr int QF = kFloat ? CPL * E : 1;

    extern __shared__ __align__(16) uint8_t smem_raw[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t q = blockIdx.x;
    const uint32_t hsize = 1u << a.hash_bits, hmask = hsize - 1;
    const uint32_t qcap = a.queue_cap;
    uint64_t* list = reinterpret_cast<uint64_t*>(smem_raw);       // [itopk] current list
    uint64_t* list_alt = list + a.itopk;                          // [itopk] target of the next parallel merge
    uint64_t* newp = list_alt + a.itopk;                          // [qcap] sorted groups of 32
    uint32_t* hash = reinterpret_cast<uint32_t*>(newp + qcap);    // [hsize]
    uint32_t* newq = hash + hsize;                                // [qcap]
    float* newd = reinterpret_cast<float*>(newq + qcap);          // [qcap]
    uint32_t* par = reinterpret_cast<uint32_t*>(newd + qcap);     // [K4B_MAX_WIDTH]
    uint32_t* ctrl = par + K4B_MAX_WIDTH;                         // [0]=n_new [1]=np [2]=n_hashed [3]=n_keep
    uint32_t* wcnt = ctrl + 4;                                    // [K4B_PICK_ROUNDS * K4B_WARPS] unexpanded per warp
    const LessBySlot less;
    const bool is_l2 = a.metric == VSB_METRIC_L2SQ;
    const bool is_cos = a.metric == VSB_METRIC_COS;
    const int n_chunks = a.x_row_bytes / 16;
    const bool full = n_chunks == CPL * 32;

    for (uint32_t i = tid; i < a.itopk; i += K4B_WARPS * 32) list[i] = kInvalidPacked;
    for (uint32_t i = tid; i < hsize; i += K4B_WARPS * 32) hash[i] = kHashEmpty;
    if (tid < 4) ctrl[tid] = 0;

    const uint4* qrow = reinterpret_cast<const uint4*>(a.q_rows + (size_t)q * a.q_row_bytes);
    float qf[QF];
    uint4 qc[kFloat ? 1 : CPL];
#pragma unroll
    for (int j = 0; j < CPL; ++j) {
        const int c = j * 32 + lane;
        uint4 v = make_uint4(0, 0, 0, 0);
        if (c < n_chunks) v = qrow[c];
        if constexpr (kFloat)
            Storage<ST>::unpack(v, &qf[j * E]);
        else
            qc[j] = v;
    }
    const float qn = a.q_nrm[q];
    unsigned long long n_evals = 0, n_parents = 0;
    __syncthreads();
#ifdef VSB_K4B_PROFILE
    long long prof_[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    long long prof_t_ = clock64();
    const long long prof_start_ = prof_t_;
#endif

    const uint32_t width = a.search_width;
    const uint32_t deg_pad = ((a.degree + 31) / 32) * 32;
    // all threads: the `width` best unexpanded list entries become the next parents (rank among the unexpanded
    // entries by ballot + per-warp counts); the graph rows of the `width` after them are prefetched into L2
    // (they are the likely parents of the following iteration).  Ends with a barrier.
    auto pick_parents = [&]() {
        uint64_t e[K4B_PICK_ROUNDS];
        uint32_t m[K4B_PICK_ROUNDS];
#pragma unroll
        for (int r = 0; r < K4B_PICK_ROUNDS; ++r) {
            const uint32_t t = r * K4B_WARPS * 32 + tid;
            e[r] = t < a.itopk ? list[t] : kInvalidPacked;
            const bool unexp = e[r] != kInvalidPacked && !(packed_lo(e[r]) & kExpandedBit);
            m[r] = __ballot_sync(kFullMask, unexp);
            if (lane == 0) wcnt[r * K4B_WARPS + warp] = __popc(m[r]);
        }
        __syncthreads();
        uint32_t before = 0, total = 0;
#pragma unroll
        for (int r = 0; r < K4B_PICK_ROUNDS; ++r) {
#pragma unroll
            for (int w = 0; w < K4B_WARPS; ++w) {
                const uint32_t c = wcnt[r * K4B_WARPS + w];
                total += c;
            }
        }
#pragma unroll
        for (int r = 0; r < K4B_PICK_ROUNDS; ++r) {
            uint32_t base = before;
#pragma unroll
            for (int w = 0; w < K4B_WARPS; ++w) {
                const uint32_t c = wcnt[r * K4B_WARPS + w];
                if (w < warp) base += c;
                before += c;
            }
            if (m[r] >> lane & 1u) {
                const uint32_t rank = base + __popc(m[r] & ((1u << lane) - 1));
                if (rank < width) {
                    par[rank] = packed_lo(e[r]);
                    list[r * K4B_WARPS * 32 + tid] = e[r] | kExpandedBit;
                } else if (rank < 2 * width) {
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(a.graph + (size_t)packed_lo(e[r]) * a.graph_stride));
                }
            }
        }
        const uint32_t np = total < width ? total : width;
        if (tid == 0) {
            ctrl[1] = np;
            n_parents += np;
        }
        __syncthreads();
    };

    // first index of the ascending run [seq, seq + len) whose value is not below x
    auto lower_bound = [&](const uint64_t* seq, uint32_t len, uint64_t x) -> uint32_t {
        uint32_t lo = 0, n = len;
        while (n > 0) {
            const uint32_t half = n >> 1;
            const bool go = seq[lo + half] < x;
            lo = go ? lo + half + 1 : lo;
            n = go ? n - half - 1 : half;
        }
        return lo;
    };

    // all warps: evaluate the queue (warp w takes entries w, w+8, ...), keep what can enter the list, sort it in
    // groups of 32, then merge list and groups IN PARALLEL: every element finds its final position as its own index
    // plus its rank in each other sorted run (packed values are unique), and is scattered into the other list buffer
    auto evaluate_queue = [&]() {
        K4B_T(0);  // own share of the neighbour fetch + visited filter
        __syncthreads();
        K4B_T(1);  // waiting for the rest of the CTA
        const uint32_t n_new = ctrl[0];
        if (n_new != 0) {
            const uint32_t mine = n_new > (uint32_t)warp ? (n_new - warp + K4B_WARPS - 1) / K4B_WARPS : 0;
            // the norm of the entry this thread will finish below: issued now so that its latency hides behind
            // the row loads instead of adding a dependent global round trip to every iteration
            float xn_first = 0.0f;
            if (is_cos && (uint32_t)tid < n_new) xn_first = __ldg(a.x_nrm + newq[tid]);
            evaluate_entries<ST, CPL, U>(a.x_rows, a.x_row_bytes, newq, newd, (uint32_t)warp, K4B_WARPS, mine, n_new, qf, qc,
                                         is_l2, lane, n_chunks, full);
            K4B_T(2);  // row loads + partial sums of warp 0's entries
            __syncthreads();
            K4B_T(3);  // waiting for the slowest warp
            const uint64_t worst = list[a.itopk - 1];
            for (uint32_t i = tid; i < n_new; i += K4B_WARPS * 32) {
                const uint32_t slot = newq[i];
                const float xn = !is_cos ? 0.0f : (i == (uint32_t)tid ? xn_first : __ldg(a.x_nrm + slot));
                const uint64_t res = pack_ds(finish_raw<ST>(newd[i], a.metric, qn, xn), slot);
                if (res < worst) newp[atomicAdd(&ctrl[3], 1u)] = res;
            }
            for (uint32_t i = tid; i < a.itopk; i += K4B_WARPS * 32) list_alt[i] = kInvalidPacked;
            __syncthreads();
            K4B_T(4);  // finish + filter
            const uint32_t n_keep = ctrl[3];
            for (uint32_t g = warp; g * 32 < n_keep; g += K4B_WARPS) {
                const uint64_t res = g * 32 + lane < n_keep ? newp[g * 32 + lane] : kInvalidPacked;
                newp[g * 32 + lane] = warp_sort32(res, lane, less);
            }
            __syncthreads();
            K4B_T(5);  // group sort
            if (n_keep != 0) {
                const uint32_t n_groups = (n_keep + 31) / 32;
                for (uint32_t i = tid; i < a.itopk + n_groups * 32; i += K4B_WARPS * 32) {
                    const bool from_list = i < a.itopk;
                    const uint32_t own_g = from_list ? 0xFFFFFFFFu : (i - a.itopk) >> 5;
                    const uint64_t x = from_list ? list[i] : newp[i - a.itopk];
                    if (x == kInvalidPacked) continue;
                    uint32_t pos = from_list ? i : ((i - a.itopk) & 31u) + lower_bound(list, a.itopk, x);
                    for (uint32_t g = 0; g < n_groups; ++g)
                        if (g != own_g) pos += lower_bound(newp + g * 32, 32, x);
                    if (pos < a.itopk) list_alt[pos] = x;
                }
                uint64_t* t = list;
                list = list_alt;
                list_alt = t;
            }
            if (tid == 0) {
                ctrl[2] += n_new;
                ctrl[0] = 0;
                ctrl[3] = 0;
                n_evals += n_new;
            }
            __syncthreads();
        }
        K4B_T(6);  // parallel merge into the list
        pick_parents();
        K4B_T(7);  // parent pick
    };

    // ---- seeds (warp 0) ----
    if (warp == 0) {
        uint64_t sv = kInvalidPacked;
        for (uint32_t s = 0; s < a.seed_splits; ++s) {
            uint64_t v = a.seed_lists[((size_t)q * a.seed_splits + s) * 32 + lane];
            v = warp_sort32(v, lane, less);
            const uint64_t rc = shfl_u64(v, 31 - lane);
            sv = warp_bitonic_merge32(rc < sv ? rc : sv, lane, less);
        }
        uint32_t nb = kInvalidSlot;
        if (lane < (int)a.n_seeds && sv != kInvalidPacked) nb = a.seed_slots[packed_lo(sv)];
        bool is_new = false;
        if (nb != kInvalidSlot) is_new = hash_insert(hash, hmask, a.hash_bits, nb);
        const uint32_t m = __ballot_sync(kFullMask, is_new);
        if (is_new) newq[__popc(m & ((1u << lane) - 1))] = nb;
        if (lane == 0) ctrl[0] = __popc(m);
    }
    evaluate_queue();

    for (uint32_t it = 0; it < a.max_iters; ++it) {
        if (ctrl[2] > (hsize >> 2) * 3) {  // uniform: written before the last barrier
            __syncthreads();
            for (uint32_t i = tid; i < hsize; i += K4B_WARPS * 32) hash[i] = kHashEmpty;
            __syncthreads();
            uint32_t cnt = 0;
            for (uint32_t i = tid; i < a.itopk; i += K4B_WARPS * 32) {
                const uint64_t e = list[i];
                if (e != kInvalidPacked) {
                    hash_insert(hash, hmask, a.hash_bits, packed_lo(e) & ~kExpandedBit);
                    ++cnt;
                }
            }
            if (tid == 0) ctrl[2] = 0;
            __syncthreads();
            if (cnt) atomicAdd(&ctrl[2], cnt);
            __syncthreads();
        }
        const uint32_t np = ctrl[1];  // picked by warp 0 at the end of the previous evaluate_queue
        if (np == 0) break;
        for (uint32_t t = tid; t < np * deg_pad; t += K4B_WARPS * 32) {
            const uint32_t i = t / deg_pad, r = t % deg_pad;
            if (r < a.degree) {
                const uint32_t nb = __ldg(a.graph + (size_t)par[i] * a.graph_stride + r);
                if (nb != kInvalidSlot && hash_insert(hash, hmask, a.hash_bits, nb)) newq[atomicAdd(&ctrl[0], 1u)] = nb;
            }
        }
        evaluate_queue();
    }

#ifdef VSB_K4B_PROFILE
    if (tid == 0 && q == 0)
        printf("k4b cycles: total %lld | fetch %lld wait %lld | rows %lld wait %lld | finish %lld sort %lld fold %lld pick %lld | "
               "evals %llu parents %llu\n",
               clock64() - prof_start_, prof_[0], prof_[1], prof_[2], prof_[3], prof_[4], prof_[5], prof_[6], prof_[7], n_evals,
               n_parents);
#endif
    // ---- emit (warp 0) ----
    if (warp == 0) {
        uint32_t count = 0;
        for (uint32_t b = 0; b < a.itopk; b += 32) {
            const uint64_t e = list[b + lane];
            const uint32_t slot = packed_lo(e) & ~kExpandedBit;
            bool valid = e != kInvalidPacked;
            if (valid && a.deny != nullptr && bit_test(a.deny, slot)) valid = false;
            if (valid && a.self_base >= 0 && slot == (uint32_t)(a.self_base + q)) valid = false;
            const uint32_t m = __ballot_sync(kFullMask, valid);
            const uint32_t pos = count + __popc(m & ((1u << lane) - 1));
            if (valid && pos < a.k) {
                if (a.out_packed != nullptr) {
                    a.out_packed[(size_t)q * a.out_stride + pos] = ((uint64_t)packed_hi(e) << 32) | slot;
                } else {
                    a.out_keys[(size_t)q * a.k + pos] = a.keys[slot];
                    a.out_dists[(size_t)q * a.k + pos] = ord_to_f32(packed_hi(e));
                }
            }
            count += __popc(m);
        }
        if (count > a.k) count = a.k;
        if (a.out_packed != nullptr) {
            for (uint32_t i = count + lane; i < a.out_stride; i += 32) a.out_packed[(size_t)q * a.out_stride + i] = kInvalidPacked;
        }
        for (uint32_t i = count + lane; i < a.k; i += 32) {
            if (a.out_packed != nullptr) {
            } else {
                a.out_keys[(size_t)q * a.k + i] = 0xFFFFFFFFFFFFFFFFull;
                a.out_dists[(size_t)q * a.k + i] = __int_as_float(0x7F800000);
            }
        }
        if (lane == 0) {
            if (a.out_counts != nullptr) a.out_counts[q] = count;
            if (a.counters != nullptr) {
                atomicAdd(&a.counters[0], n_evals);
                atomicAdd(&a.counters[1], n_parents);
            }
        }
    }
}

// Seed layer for tiny batches: every warp scans 4 seed rows with the canonical distance, every CTA
// emits its best row -> [q][blocks][32] packed winners (the format K4 consumes).
constexpr int SEED_SCAN_WARPS = 8;
constexpr int SEED_SCAN_ROWS_PER_WARP = 4;

template <int ST>
__global__ void __launch_bounds__(SEED_SCAN_WARPS * 32) seed_scan_kernel(const uint8_t* __restrict__ q_rows,
                                                                          const float* __restrict__ q_nrm,
                                                                          uint32_t q_row_bytes,
                                                                          const uint8_t* __restrict__ s_rows,
                                                                          const float* __restrict__ s_nrm,
                                                                          uint32_t n_seed_rows, uint32_t row_bytes,
                                                                          int metric, uint32_t n_blocks,
                                                                          uint64_t* __restrict__ out) {
    __shared__ uint64_t best[SEED_SCAN_WARPS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t q = blockIdx.y;
    const uint4* qrow = reinterpret_cast<const uint4*>(q_rows + (size_t)q * q_row_bytes);
    const float qn = q_nrm[q];
    const int n_chunks = row_bytes / 16;
    const uint32_t r0 = (blockIdx.x * SEED_SCAN_WARPS + warp) * SEED_SCAN_ROWS_PER_WARP;
    uint64_t mine = kInvalidPacked;
#pragma unroll
    for (int i = 0; i < SEED_SCAN_ROWS_PER_WARP; ++i) {
        const uint32_t r = r0 + i;
        if (r >= n_seed_rows) break;
        const uint4* xrow = reinterpret_cast<const uint4*>(s_rows + (size_t)r * row_bytes);
        float d;
        if constexpr (ST == VSB_ST_B1) {
            d = warp_distance<ST, VSB_METRIC_HAMMING>(qrow, xrow, n_chunks, qn, 0.0f, lane);
        } else {
            if (metric == VSB_METRIC_L2SQ) d = warp_distance<ST, VSB_METRIC_L2SQ>(qrow, xrow, n_chunks, qn, 0.0f, lane);
            else if (metric == VSB_METRIC_IP) d = warp_distance<ST, VSB_METRIC_IP>(qrow, xrow, n_chunks, qn, 0.0f, lane);
            else d = warp_distance<ST, VSB_METRIC_COS>(qrow, xrow, n_chunks, qn, s_nrm[r], lane);
        }
        const uint64_t p = pack_ds(d, r);
        mine = p < mine ? p : mine;
    }
    if (lane == 0) best[warp] = mine;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint64_t b = best[0];
        for (int w = 1; w < SEED_SCAN_WARPS; ++w) b = best[w] < b ? best[w] : b;
        out[(size_t)q * n_blocks * 32 + blockIdx.x] = b;
    }
}

template <int ST, int CPL>
void launch_k4_inst(const K4Args& a, dim3 grid, size_t smem, cudaStream_t stream) {
    if (a.allow != nullptr) {
        cudaFuncSetAttribute(graph_search_kernel<ST, CPL, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        graph_search_kernel<ST, CPL, true><<<grid, K4_WARPS * 32, smem, stream>>>(a);
        return;
    }
    if constexpr (ST == VSB_ST_BF16 || ST == VSB_ST_F16) {
        if (a.mma) {
            cudaFuncSetAttribute(graph_search_kernel<ST, CPL, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            graph_search_kernel<ST, CPL, false, true><<<grid, K4_WARPS * 32, smem, stream>>>(a);
            return;
        }
    }
    cudaFuncSetAttribute(graph_search_kernel<ST, CPL, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    graph_search_kernel<ST, CPL, false><<<grid, K4_WARPS * 32, smem, stream>>>(a);
}

template <int ST, int CPL>
void launch_k4b_inst(const K4Args& a, dim3 grid, size_t smem, cudaStream_t stream) {
    cudaFuncSetAttribute(graph_search_cta_kernel<ST, CPL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    graph_search_cta_kernel<ST, CPL><<<grid, K4B_WARPS * 32, smem, stream>>>(a);
}

template <int ST>
void launch_k4b_storage(const K4Args& a, int cpl, dim3 grid, size_t smem, cudaStream_t stream) {
    switch (cpl) {
        case 1: launch_k4b_inst<ST, 1>(a, grid, smem, stream); break;
        case 2: launch_k4b_inst<ST, 2>(a, grid, smem, stream); break;
        case 3: launch_k4b_inst<ST, 3>(a, grid, smem, stream); break;
        case 4: launch_k4b_inst<ST, 4>(a, grid, smem, stream); break;
        case 6: launch_k4b_inst<ST, 6>(a, grid, smem, stream); break;
        case 8: launch_k4b_inst<ST, 8>(a, grid, smem, stream); break;
        default: launch_k4b_inst<ST, 12>(a, grid, smem, stream); break;
    }
}

struct SeedScanArgs {
    const uint8_t* q_rows; const float* q_nrm; uint32_t nq, q_row_bytes;
    const uint8_t* s_rows; const float* s_nrm; uint32_t n_seed_rows, row_bytes;
    int metric; uint32_t n_blocks; uint64_t* out;
};
template <int ST>
void launch_seed_scan_storage(const SeedScanArgs& s, cudaStream_t stream) {
    const uint32_t ctas = (s.n_seed_rows + SEED_SCAN_WARPS * SEED_SCAN_ROWS_PER_WARP - 1) /
                          (SEED_SCAN_WARPS * SEED_SCAN_ROWS_PER_WARP);
    seed_scan_kernel<ST><<<dim3(ctas, s.nq), SEED_SCAN_WARPS * 32, 0, stream>>>(
        s.q_rows, s.q_nrm, s.q_row_bytes, s.s_rows, s.s_nrm, s.n_seed_rows, s.row_bytes, s.metric, s.n_blocks, s.out);
}

// one translation unit per storage scalar instantiates this
template <int ST>
void launch_k4_storage(const K4Args& a, int cpl, dim3 grid, size_t smem, cudaStream_t stream) {
    switch (cpl) {
        case 1: launch_k4_inst<ST, 1>(a, grid, smem, stream); break;
        case 2: launch_k4_inst<ST, 2>(a, grid, smem, stream); break;
        case 3: launch_k4_inst<ST, 3>(a, grid, smem, stream); break;
        case 4: launch_k4_inst<ST, 4>(a, grid, smem, stream); break;
        case 6: launch_k4_inst<ST, 6>(a, grid, smem, stream); break;
        case 8: launch_k4_inst<ST, 8>(a, grid, smem, stream); break;
        default: launch_k4_inst<ST, 12>(a, grid, smem, stream); break;
    }
}

#define VSB_K4_DECL(name)                                                                              \
    void launch_k4b_##name(const K4Args& a, int cpl, dim3 grid, size_t smem, cudaStream_t stream);     \
    void launch_seed_scan_##name(const SeedScanArgs& s, cudaStream_t stream);
VSB_K4_DECL(f32)
VSB_K4_DECL(f16)
VSB_K4_DECL(bf16)
VSB_K4_DECL(i8)
VSB_K4_DECL(b1)
void launch_k4_f32(const K4Args& a, int cpl, dim3 grid, size_t smem, cudaStream_t stream);
void launch_k4_f16(const K4Args& a, int cpl, dim3 grid, size_t smem, cudaStream_t stream);
void launch_k4_bf16(const K4Args& a, int cpl, dim3 grid, size_t smem, cudaStream_t stream);
void launch_k4_i8(const K4Args& a, int cpl, dim3 grid, size_t smem, cudaStream_t stream);
void launch_k4_b1(const K4Args& a, int cpl, dim3 grid, size_t smem, cudaStream_t stream);

}  // namespace vsb
