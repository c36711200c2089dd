// graph_build.cu — K6: turn exact k_init-NN lists into the fixed-degree search graph.
//
// Replaces the link-selection half of usearch::Index::add (reference call site
// vs_index/usearch.rs:191-197, SURVEY §8a A5): instead of HNSW's per-insert neighbour heuristic
// the bulk build prunes a kNN graph by rank-based detour counting (CAGRA), then adds reverse
// edges.  Everything here is integer work on slot ids and is fully deterministic, so the graph is
// compared bit-for-bit with oracle/graph_oracle.py.
//
//   1. prune_detour_kernel : for node u with list L (ascending by distance), edge u->L[j] gets
//      detour[j] = #{ i<j : L[j] appears in knn(L[i]) at a position t < j }.  Keep the R edges with
//      the smallest (detour, j).
//   2. reverse edges       : every kept edge u->v at rank r proposes u to v.  Proposals are radix
//      sorted by (v, r, u) so each node's reverse list is its R best-ranked proposers, ties by slot.
//   3. merge_graph_kernel  : row = fwd[0:R/2] ++ reverse (new ones only) ++ fwd[R/2:R], cut at R.
#include <cub/device/device_radix_sort.cuh>

#include "kernels.h"
#include "select.cuh"

namespace vsb {

namespace {

constexpr int K6_WARPS = 4;
constexpr int K6_MAXK = 128;   // k_init upper bound
constexpr int K6_HASH = 256;   // >= 2 * K6_MAXK

__global__ void __launch_bounds__(K6_WARPS * 32) prune_detour_kernel(const uint64_t* __restrict__ knn, uint32_t n,
                                                                     uint32_t k_init, uint32_t R,
                                                                     const uint32_t* __restrict__ deny,
                                                                     uint32_t* __restrict__ fwd) {
    __shared__ uint32_t sL[K6_WARPS][K6_MAXK];
    __shared__ uint32_t sDet[K6_WARPS][K6_MAXK];
    __shared__ uint32_t sHid[K6_WARPS][K6_HASH];
    __shared__ uint32_t sHrank[K6_WARPS][K6_HASH];
    __shared__ uint64_t sOrd[K6_WARPS][K6_MAXK];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t u = blockIdx.x * K6_WARPS + warp;
    if (u >= n) return;
    if (deny != nullptr && bit_test(deny, u)) {  // tombstoned rows keep no edges and propose none
        for (uint32_t r = lane; r < R; r += 32) fwd[(size_t)u * R + r] = kInvalidSlot;
        return;
    }
    uint32_t* L = sL[warp];
    uint32_t* det = sDet[warp];
    uint32_t* hid = sHid[warp];
    uint32_t* hrank = sHrank[warp];
    uint64_t* ord = sOrd[warp];

    for (int i = lane; i < K6_HASH; i += 32) hid[i] = kInvalidSlot;
    uint32_t k0 = 0;
    for (uint32_t j = lane; j < K6_MAXK; j += 32) {
        uint32_t v = kInvalidSlot;
        if (j < k_init) {
            const uint64_t p = knn[(size_t)u * k_init + j];
            if (p != kInvalidPacked) v = packed_lo(p);
        }
        L[j] = v;
        det[j] = 0;
        ord[j] = kInvalidPacked;
        k0 += __popc(__ballot_sync(kFullMask, v != kInvalidSlot));
    }
    __syncwarp();
    for (uint32_t j = lane; j < k0; j += 32) {
        const uint32_t v = L[j];
        uint32_t h = (v * 0x9E3779B1u) >> 24;
        while (true) {
            const uint32_t old = atomicCAS(&hid[h], kInvalidSlot, v);
            if (old == kInvalidSlot) {
                hrank[h] = j;
                break;
            }
            h = (h + 1) & (K6_HASH - 1);
        }
    }
    __syncwarp();
    for (uint32_t i = 0; i < k0; ++i) {
        const uint64_t* row = knn + (size_t)L[i] * k_init;
        for (uint32_t t = lane; t < k_init; t += 32) {
            const uint64_t p = row[t];
            if (p == kInvalidPacked) continue;
            const uint32_t y = packed_lo(p);
            uint32_t h = (y * 0x9E3779B1u) >> 24;
            while (true) {
                const uint32_t id = hid[h];
                if (id == kInvalidSlot) break;
                if (id == y) {
                    const uint32_t j = hrank[h];
                    if (j > i && t < j) atomicAdd(&det[j], 1u);
                    break;
                }
                h = (h + 1) & (K6_HASH - 1);
            }
        }
    }
    __syncwarp();
    // order by (detour, rank)
    const LessBySlot less;
    for (uint32_t b = 0; b < K6_MAXK; b += 32) {
        const uint32_t j = b + lane;
        uint64_t v = j < k0 ? (((uint64_t)det[j] << 32) | j) : kInvalidPacked;
        if (__ballot_sync(kFullMask, v != kInvalidPacked) == 0) break;
        v = warp_sort32(v, lane, less);
        warp_list_merge(ord, K6_MAXK, v, lane, less);
    }
    for (uint32_t r = lane; r < R; r += 32) {
        const uint64_t o = r < K6_MAXK ? ord[r] : kInvalidPacked;
        fwd[(size_t)u * R + r] = (o == kInvalidPacked) ? kInvalidSlot : L[packed_lo(o)];
    }
}

// proposals: key = v << 36 | r << 28 | u   (n < 2^28, r < 256)
__global__ void make_proposals_kernel(const uint32_t* __restrict__ fwd, uint32_t n, uint32_t R,
                                      uint64_t* __restrict__ out) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)n * R) return;
    const uint32_t u = (uint32_t)(i / R), r = (uint32_t)(i % R);
    const uint32_t v = fwd[i];
    out[i] = (v == kInvalidSlot) ? kInvalidPacked : (((uint64_t)v << 36) | ((uint64_t)r << 28) | u);
}

__global__ void mark_segments_kernel(const uint64_t* __restrict__ sorted, size_t m, uint32_t* __restrict__ seg_start) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const uint64_t p = sorted[i];
    if (p == kInvalidPacked) return;
    const uint32_t v = (uint32_t)(p >> 36);
    if (i == 0 || (uint32_t)(sorted[i - 1] >> 36) != v) seg_start[v] = (uint32_t)i;
}

__global__ void scatter_reverse_kernel(const uint64_t* __restrict__ sorted, size_t m,
                                       const uint32_t* __restrict__ seg_start, uint32_t R,
                                       uint32_t* __restrict__ rev, uint32_t* __restrict__ rev_cnt) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const uint64_t p = sorted[i];
    if (p == kInvalidPacked) return;
    const uint32_t v = (uint32_t)(p >> 36);
    const uint32_t u = (uint32_t)(p & 0x0FFFFFFFu);
    const uint32_t pos = (uint32_t)i - seg_start[v];
    if (pos < R) {
        rev[(size_t)v * R + pos] = u;
        atomicMax(&rev_cnt[v], pos + 1);
    }
}

constexpr int K6_MAXR = 128;

__global__ void merge_graph_kernel(const uint32_t* __restrict__ fwd, const uint32_t* __restrict__ rev,
                                   const uint32_t* __restrict__ rev_cnt, uint32_t n, uint32_t R,
                                   uint32_t* __restrict__ graph, uint32_t graph_stride) {
    const uint32_t u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= n) return;
    uint32_t out[K6_MAXR];
    uint32_t c = 0;
    auto push_unique = [&](uint32_t v) {
        if (v == kInvalidSlot || v == u || c >= R) return;
        for (uint32_t i = 0; i < c; ++i)
            if (out[i] == v) return;
        out[c++] = v;
    };
    const uint32_t half = R / 2;
    for (uint32_t r = 0; r < half; ++r) push_unique(fwd[(size_t)u * R + r]);
    const uint32_t rc = rev_cnt[u];
    for (uint32_t r = 0; r < rc; ++r) push_unique(rev[(size_t)u * R + r]);
    for (uint32_t r = half; r < R; ++r) push_unique(fwd[(size_t)u * R + r]);
    for (uint32_t r = 0; r < graph_stride; ++r) graph[(size_t)u * graph_stride + r] = r < c ? out[r] : kInvalidSlot;
}

}  // namespace

void launch_prune_detour(const uint64_t* knn, uint32_t n, uint32_t k_init, uint32_t R, const uint32_t* deny,
                         uint32_t* fwd, cudaStream_t stream) {
    if (n == 0) return;
    prune_detour_kernel<<<(n + K6_WARPS - 1) / K6_WARPS, K6_WARPS * 32, 0, stream>>>(knn, n, k_init, R, deny, fwd);
    g_kernel_launches += 1;
}

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

size_t reverse_edges_scratch_bytes(uint32_t n, uint32_t R) {
    const size_t m = (size_t)n * R;
    size_t temp = 0;
    cub::DeviceRadixSort::SortKeys(nullptr, temp, (const uint64_t*)nullptr, (uint64_t*)nullptr, m, 0, 64);
    return align_up(m * 8, 256) * 2 + align_up((size_t)n * 4, 256) + align_up(temp, 256);
}

void launch_reverse_edges(const uint32_t* fwd, uint32_t n, uint32_t R, uint32_t* rev, uint32_t* rev_cnt,
                          void* scratch, size_t scratch_bytes, cudaStream_t stream) {
    if (n == 0) return;
    const size_t m = (size_t)n * R;
    uint8_t* base = static_cast<uint8_t*>(scratch);
    uint64_t* prop = reinterpret_cast<uint64_t*>(base);
    uint64_t* sorted = reinterpret_cast<uint64_t*>(base + align_up(m * 8, 256));
    uint32_t* seg_start = reinterpret_cast<uint32_t*>(base + 2 * align_up(m * 8, 256));
    void* temp = base + 2 * align_up(m * 8, 256) + align_up((size_t)n * 4, 256);
    size_t temp_bytes = scratch_bytes - (2 * align_up(m * 8, 256) + align_up((size_t)n * 4, 256));
    const int T = 256;
    make_proposals_kernel<<<(unsigned)((m + T - 1) / T), T, 0, stream>>>(fwd, n, R, prop);
    cub::DeviceRadixSort::SortKeys(temp, temp_bytes, prop, sorted, m, 0, 64, stream);
    cudaMemsetAsync(rev_cnt, 0, (size_t)n * 4, stream);
    cudaMemsetAsync(rev, 0xFF, (size_t)n * R * 4, stream);
    mark_segments_kernel<<<(unsigned)((m + T - 1) / T), T, 0, stream>>>(sorted, m, seg_start);
    scatter_reverse_kernel<<<(unsigned)((m + T - 1) / T), T, 0, stream>>>(sorted, m, seg_start, R, rev, rev_cnt);
    g_kernel_launches += 3;  // + the CUB radix-sort passes, which are library kernels and not counted
}

void launch_merge_graph(const uint32_t* fwd, const uint32_t* rev, const uint32_t* rev_cnt, uint32_t n,
                        uint32_t R, uint32_t* graph, uint32_t graph_stride, cudaStream_t stream) {
    if (n == 0) return;
    const int T = 128;
    merge_graph_kernel<<<(n + T - 1) / T, T, 0, stream>>>(fwd, rev, rev_cnt, n, R, graph, graph_stride);
    g_kernel_launches += 1;
}

}  // namespace vsb

// ------------------------------------------------------------------------------------------------
// K7: streaming insert (SURVEY §8a A5 "HNSW insert", config C5).  The batch of new rows has been searched with
// K4 (beam = expansion_add) and `cand` holds each new row's C best candidates (packed, ascending,
// kInvalidPacked padded; C <= 128, normally 2R).  Two kernels, so that the row of a new node is complete before
// any edge points at it (searches may be walking the same buffer, index_impl.h):
//   stream_link_fwd : one warp per new row u.  Neighbour selection is the bulk build's rank-based detour count
//                     with the GRAPH rows of the candidates standing in for their kNN lists:
//                     detour[j] = #{ i < j : cand[j] is a neighbour of cand[i] }  (u -> cand[i] -> cand[j] exists),
//                     keep the R candidates with the smallest (detour, j) — a diverse neighbourhood instead of
//                     the R closest, which is what keeps recall from decaying between refinement passes.
//   stream_link_rev : each of the R/2 first neighbours v of u gets u written into the reverse half of row(v):
//                     an empty slot if there is one, otherwise a pseudo-randomly chosen one is replaced.  The
//                     batch's proposals are radix sorted by (v, rank, u) and one warp applies all proposals to
//                     row(v) in that order: the closest links first, as when the batch's warps step through
//                     their ranks together, but independent of the order warps run in.  A reverse edge is one
//                     32-bit store: searches walking the same buffer never see a torn row.
// Rows of one batch do not link to each other; refinement passes re-optimise the graph.
namespace vsb {
namespace {
constexpr int K7_WARPS = 4;

__global__ void __launch_bounds__(K7_WARPS * 32) stream_link_fwd_kernel(const uint64_t* __restrict__ cand, uint32_t n_new,
                                                                        uint32_t C, uint32_t first_slot, uint32_t R,
                                                                        uint32_t* __restrict__ graph, uint32_t graph_stride) {
    __shared__ uint32_t sL[K7_WARPS][K6_MAXK];
    __shared__ uint32_t sDet[K7_WARPS][K6_MAXK];
    __shared__ uint32_t sHid[K7_WARPS][K6_HASH];
    __shared__ uint32_t sHrank[K7_WARPS][K6_HASH];
    __shared__ uint64_t sOrd[K7_WARPS][K6_MAXK];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t i = blockIdx.x * K7_WARPS + warp;
    if (i >= n_new) return;
    const uint32_t u = first_slot + i;
    uint32_t* L = sL[warp];
    uint32_t* det = sDet[warp];
    uint32_t* hid = sHid[warp];
    uint32_t* hrank = sHrank[warp];
    uint64_t* ord = sOrd[warp];
    for (int t = lane; t < K6_HASH; t += 32) hid[t] = kInvalidSlot;
    const uint32_t k0 = C < (uint32_t)K6_MAXK ? C : (uint32_t)K6_MAXK;
    for (uint32_t j = lane; j < K6_MAXK; j += 32) {
        uint32_t v = kInvalidSlot;
        if (j < k0) {
            const uint64_t p = cand[(size_t)i * C + j];
            if (p != kInvalidPacked && packed_lo(p) != u) v = packed_lo(p);
        }
        L[j] = v;  // holes (padding, u itself) are skipped everywhere below
        det[j] = 0;
        ord[j] = kInvalidPacked;
    }
    __syncwarp();
    for (uint32_t j = lane; j < k0; j += 32) {
        const uint32_t v = L[j];
        if (v == kInvalidSlot) continue;
        uint32_t h = (v * 0x9E3779B1u) >> 24;
        while (true) {
            const uint32_t old = atomicCAS(&hid[h], kInvalidSlot, v);
            if (old == kInvalidSlot) {
                hrank[h] = j;
                break;
            }
            if (old == v) break;  // duplicate candidate: the first rank stands
            h = (h + 1) & (K6_HASH - 1);
        }
    }
    __syncwarp();
    for (uint32_t a = 0; a < k0; ++a) {
        if (L[a] == kInvalidSlot) continue;
        const uint32_t* row = graph + (size_t)L[a] * graph_stride;
        for (uint32_t t = lane; t < R; t += 32) {
            const uint32_t y = row[t];
            if (y == kInvalidSlot) continue;
            uint32_t h = (y * 0x9E3779B1u) >> 24;
            while (true) {
                const uint32_t id = hid[h];
                if (id == kInvalidSlot) break;
                if (id == y) {
                    const uint32_t j = hrank[h];
                    if (j > a) atomicAdd(&det[j], 1u);
                    break;
                }
                h = (h + 1) & (K6_HASH - 1);
            }
        }
    }
    __syncwarp();
    const LessBySlot less;
    for (uint32_t b = 0; b < K6_MAXK; b += 32) {
        const uint32_t j = b + lane;
        uint64_t v = (j < k0 && L[j] != kInvalidSlot) ? (((uint64_t)det[j] << 32) | j) : kInvalidPacked;
        if (__ballot_sync(kFullMask, v != kInvalidPacked) == 0) continue;
        v = warp_sort32(v, lane, less);
        warp_list_merge(ord, K6_MAXK, v, lane, less);
    }
    __syncwarp();
    // the kept edges go back into distance order (rank order), so the R/2 first ones are the closest kept ones
    for (int t = lane; t < K6_HASH; t += 32) hid[t] = 0;  // the hash is done: reuse it as "kept" flags by rank
    __syncwarp();
    for (uint32_t r = lane; r < R && r < (uint32_t)K6_MAXK; r += 32) {
        const uint64_t o = ord[r];
        if (o != kInvalidPacked) hid[packed_lo(o)] = 1;
    }
    __syncwarp();
    uint32_t* out = graph + (size_t)u * graph_stride;
    uint32_t count = 0;
    for (uint32_t b = 0; b < k0; b += 32) {
        const uint32_t j = b + lane;
        const bool kept = j < k0 && hid[j] == 1;
        const uint32_t m = __ballot_sync(kFullMask, kept);
        if (kept) out[count + __popc(m & ((1u << lane) - 1))] = L[j];
        count += __popc(m);
    }
    for (uint32_t r = count + lane; r < graph_stride; r += 32) out[r] = kInvalidSlot;
}

// reverse-edge proposals of one batch: key = v << 32 | r * n_new + (u - first_slot)  (n_new * half < 2^32)
__global__ void stream_proposals_kernel(const uint32_t* __restrict__ graph, uint32_t graph_stride, uint32_t n_new,
                                        uint32_t first_slot, uint32_t half, uint64_t* __restrict__ out) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)n_new * half) return;
    const uint32_t u = first_slot + (uint32_t)(i / half), r = (uint32_t)(i % half);
    const uint32_t v = graph[(size_t)u * graph_stride + r];
    out[i] = (v == kInvalidSlot || v >= first_slot) ? kInvalidPacked
                                                    : (((uint64_t)v << 32) | ((uint64_t)r * n_new + (u - first_slot)));
}

// one warp per target row v (the warp of its segment's first entry) applies the segment's proposals in sorted order;
// the lanes scan the reverse half of row(v) 32 slots at a time
__global__ void __launch_bounds__(256) stream_link_rev_kernel(const uint64_t* __restrict__ sorted, size_t m, uint32_t n_new,
                                                              uint32_t first_slot, uint32_t R, uint32_t* __restrict__ graph,
                                                              uint32_t graph_stride) {
    const int lane = threadIdx.x & 31;
    const size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (i >= m || sorted[i] == kInvalidPacked) return;  // uniform across the warp
    const uint32_t v = (uint32_t)(sorted[i] >> 32);
    if (i > 0 && (uint32_t)(sorted[i - 1] >> 32) == v) return;
    const uint32_t half = R / 2;
    uint32_t* vrow = graph + (size_t)v * graph_stride;
    for (size_t e = i; e < m && (uint32_t)(sorted[e] >> 32) == v; ++e) {  // kInvalidPacked >> 32 is no slot
        const uint32_t idx = (uint32_t)sorted[e];
        const uint32_t u = first_slot + idx % n_new, r = idx / n_new;
        bool linked = false;
        uint32_t empty = kInvalidSlot;
        for (uint32_t base = half; base < R; base += 32) {
            const uint32_t pos = base + lane;
            const uint32_t cur = pos < R ? vrow[pos] : 0u;
            linked |= __ballot_sync(kFullMask, pos < R && cur == u) != 0;
            const uint32_t empties = __ballot_sync(kFullMask, pos < R && cur == kInvalidSlot);
            if (empty == kInvalidSlot && empties != 0) empty = base + __ffs(empties) - 1;
        }
        if (!linked && lane == 0)
            vrow[empty != kInvalidSlot ? empty : half + ((u * 0x9E3779B1u + r * 0x85EBCA6Bu) >> 16) % (R - half)] = u;
        __syncwarp();  // the next proposal's scan sees this store
    }
}

// compaction: new_graph[old2new[u]][r] = old2new[graph[u][r]] (edges to removed rows dropped)
__global__ void remap_graph_kernel(const uint32_t* __restrict__ graph, uint32_t n_old, uint32_t stride,
                                   const uint32_t* __restrict__ old2new, uint32_t* __restrict__ out) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (size_t)n_old * stride) return;
    const uint32_t u = (uint32_t)(t / stride), r = (uint32_t)(t % stride);
    const uint32_t nu = old2new[u];
    if (nu == kInvalidSlot) return;
    const uint32_t v = graph[t];
    out[(size_t)nu * stride + r] = (v == kInvalidSlot || v >= n_old) ? kInvalidSlot : old2new[v];
}
}  // namespace

size_t stream_link_scratch_bytes(uint32_t n_new, uint32_t R) {
    const size_t m = (size_t)n_new * (R / 2);
    size_t temp = 0;
    cub::DeviceRadixSort::SortKeys(nullptr, temp, (const uint64_t*)nullptr, (uint64_t*)nullptr, m, 0, 64);
    return align_up(m * 8, 256) * 2 + align_up(temp, 256);
}

cudaError_t launch_stream_link(const uint64_t* cand, uint32_t n_new, uint32_t cand_stride, uint32_t first_slot, uint32_t R,
                               uint32_t* graph, uint32_t graph_stride, void* scratch, size_t scratch_bytes,
                               cudaStream_t stream) {
    if (n_new == 0) return cudaSuccess;
    stream_link_fwd_kernel<<<(n_new + K7_WARPS - 1) / K7_WARPS, K7_WARPS * 32, 0, stream>>>(cand, n_new, cand_stride, first_slot,
                                                                                            R, graph, graph_stride);
    const size_t m = (size_t)n_new * (R / 2);
    uint8_t* base = static_cast<uint8_t*>(scratch);
    uint64_t* prop = reinterpret_cast<uint64_t*>(base);
    uint64_t* sorted = reinterpret_cast<uint64_t*>(base + align_up(m * 8, 256));
    size_t temp_bytes = scratch_bytes - 2 * align_up(m * 8, 256);
    const int T = 256;
    stream_proposals_kernel<<<(unsigned)((m + T - 1) / T), T, 0, stream>>>(graph, graph_stride, n_new, first_slot, R / 2, prop);
    g_kernel_launches += 2;
    // targets are below first_slot: the key's high word needs bit_width(first_slot - 1) bits (kInvalidPacked still sorts last)
    const int end_bit = 32 + (first_slot > 1 ? 32 - __builtin_clz(first_slot - 1) : 1);
    cudaError_t e = cub::DeviceRadixSort::SortKeys(base + 2 * align_up(m * 8, 256), temp_bytes, prop, sorted, m, 0, end_bit,
                                                   stream);
    if (e != cudaSuccess) return e;
    stream_link_rev_kernel<<<(unsigned)((m * 32 + T - 1) / T), T, 0, stream>>>(sorted, m, n_new, first_slot, R, graph, graph_stride);
    g_kernel_launches += 1;  // + the CUB radix-sort passes, which are library kernels and not counted
    return cudaGetLastError();
}

void launch_remap_graph(const uint32_t* graph, uint32_t n_old, uint32_t stride, const uint32_t* old2new, uint32_t* out,
                        cudaStream_t stream) {
    if (n_old == 0) return;
    const size_t m = (size_t)n_old * stride;
    remap_graph_kernel<<<(unsigned)((m + 255) / 256), 256, 0, stream>>>(graph, n_old, stride, old2new, out);
    g_kernel_launches += 1;
}
// ---- reachability of the graph from the entry-point sample -----------------------------------------------------
// A kNN-derived graph over well separated clusters can fall apart into components; the beam search only ever sees
// the components that hold a seed.  After every (re)sampling of the seeds the host runs this frontier expansion to
// a fixed point and promotes one node of each unreached component to an extra seed (index.cu::sample_seeds).
// state: 0 = unreached, 1 = reached / to expand, 2 = expanded.
__global__ void reach_mark_kernel(uint8_t* state, const uint32_t* seeds, uint32_t n_seeds) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_seeds) state[seeds[i]] = 1;
}

__global__ void __launch_bounds__(256) reach_step_kernel(const uint32_t* __restrict__ graph, uint32_t n, uint32_t stride,
                                                         uint32_t degree, uint8_t* state, uint32_t* changed) {
    const int lane = threadIdx.x & 31;
    const uint32_t u = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (u >= n || state[u] != 1) return;
    bool any = false;
    for (uint32_t r = lane; r < degree; r += 32) {
        const uint32_t v = graph[(size_t)u * stride + r];
        if (v < n && state[v] == 0) {
            state[v] = 1;  // benign race: every writer stores the same value
            any = true;
        }
    }
    __syncwarp();
    if (lane == 0) state[u] = 2;
    if (__ballot_sync(kFullMask, any) != 0 && lane == 0) *changed = 1;
}

__global__ void first_unreached_kernel(const uint8_t* __restrict__ state, const uint32_t* __restrict__ deny, uint32_t n,
                                       uint32_t* out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || state[i] != 0) return;
    if (deny != nullptr && bit_test(deny, i)) return;
    atomicMin(out, i);
}

// The first `cap` unreached live nodes in slot order (deterministic): ONE CTA, thread t owns a contiguous 16-byte
// aligned range of the state array; count, block-scan, then write.  out[0] = how many were found (<= cap),
// out[1..] = their slots.
__global__ void __launch_bounds__(1024) collect_unreached_kernel(const uint8_t* __restrict__ state,
                                                                 const uint32_t* __restrict__ deny, uint32_t n, uint32_t cap,
                                                                 uint32_t* __restrict__ out) {
    __shared__ uint32_t s_cnt[1024];
    const uint32_t t = threadIdx.x;
    const uint32_t chunk = (((n + 1023) / 1024) + 15) / 16 * 16;
    const uint32_t lo = min(n, t * chunk), hi = min(n, lo + chunk);
    auto unreached = [&](uint32_t i) { return state[i] == 0 && !(deny != nullptr && bit_test(deny, i)); };
    uint32_t c = 0;
    for (uint32_t i = lo; i < hi; i += 16) {
        const uint4 v = *reinterpret_cast<const uint4*>(state + i);  // the buffer is padded to 16 bytes past n
        auto all_nonzero = [](uint32_t w) { return ((w | (w >> 1)) & 0x01010101u) == 0x01010101u; };  // states are 0, 1, 2
        if (all_nonzero(v.x) && all_nonzero(v.y) && all_nonzero(v.z) && all_nonzero(v.w)) continue;  // the common case
        for (uint32_t j = i; j < min(hi, i + 16); ++j) c += unreached(j) ? 1u : 0u;
    }
    s_cnt[t] = c;
    __syncthreads();
    // exclusive scan (Hillis-Steele over 1024 entries)
    for (uint32_t off = 1; off < 1024; off <<= 1) {
        const uint32_t v = t >= off ? s_cnt[t - off] : 0u;
        __syncthreads();
        s_cnt[t] += v;
        __syncthreads();
    }
    const uint32_t total = s_cnt[1023];
    uint32_t pos = s_cnt[t] - c;
    if (t == 0) out[0] = total < cap ? total : cap;
    if (c == 0 || pos >= cap) return;
    for (uint32_t i = lo; i < hi && pos < cap; ++i)
        if (unreached(i)) out[1 + pos++] = i;
}

void launch_collect_unreached(const uint8_t* state, const uint32_t* deny, uint32_t n, uint32_t cap, uint32_t* out,
                              cudaStream_t stream) {
    collect_unreached_kernel<<<1, 1024, 0, stream>>>(state, deny, n, cap, out);
    g_kernel_launches += 1;
}

void launch_reach_mark(uint8_t* state, const uint32_t* seeds, uint32_t n_seeds, cudaStream_t stream) {
    if (n_seeds == 0) return;
    reach_mark_kernel<<<(n_seeds + 255) / 256, 256, 0, stream>>>(state, seeds, n_seeds);
    g_kernel_launches += 1;
}

void launch_reach_step(const uint32_t* graph, uint32_t n, uint32_t stride, uint32_t degree, uint8_t* state,
                       uint32_t* changed, cudaStream_t stream) {
    if (n == 0) return;
    reach_step_kernel<<<(n + 7) / 8, 256, 0, stream>>>(graph, n, stride, degree, state, changed);
    g_kernel_launches += 1;
}

void launch_first_unreached(const uint8_t* state, const uint32_t* deny, uint32_t n, uint32_t* out, cudaStream_t stream) {
    if (n == 0) return;
    first_unreached_kernel<<<(n + 255) / 256, 256, 0, stream>>>(state, deny, n, out);
    g_kernel_launches += 1;
}

}  // namespace vsb
