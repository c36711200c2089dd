// kernels.h — host-callable launchers of every CUDA kernel in libvsb200 (internal).
#pragma once
#include <atomic>

#include "common.cuh"

namespace vsb {

// every launcher adds the number of kernels it enqueued (reported as gpu_launches by bench.py)
extern std::atomic<uint64_t> g_kernel_launches;
extern std::atomic<uint64_t> g_tc_launches;

// A block of stored rows: storage-typed bytes + canonical norms.
struct RowsView {
    const uint8_t* rows = nullptr;  // [n][row_bytes]
    const float* sq = nullptr;      // canonical sum of squares (popcount for b1)
    const float* nrm = nullptr;     // sqrt(sq)
    uint32_t row_bytes = 0;
    uint32_t n = 0;
    // rows [first, first + count) of this block
    RowsView slice(uint32_t first, uint32_t count) const {
        return RowsView{rows + (size_t)first * row_bytes, sq + first, nrm + first, row_bytes, count};
    }
};

// A filter: bitmaps over (key & 2^48-1), ceil(bits / 32) words each, back to back; query i tests bitmap of_q[i]
// (of_q null: every query tests the first bitmap).  bm null: no filter.
struct Allow {
    const uint32_t* bm = nullptr;
    uint64_t bits = 0;
    const uint32_t* of_q = nullptr;
    // the same filter for the queries from q0 on
    Allow from(uint64_t q0) const { return Allow{bm, bits, of_q ? of_q + q0 : nullptr}; }
};

// K0 ------------------------------------------------------------------------------------------
void launch_convert_rows(int storage, const float* in, uint32_t n_rows, uint32_t dim, uint8_t* out,
                         uint32_t row_bytes, float* sq, float* nrm, cudaStream_t stream);
// scaled int8 copy for the cosine traversal (per-row scale max|x|/127; nrm = |x| in units of the scale)
void launch_convert_rows_i8s(const float* in, uint32_t n_rows, uint32_t dim, uint32_t in_stride, uint8_t* out,
                             uint32_t row_bytes, float* sq, float* nrm, cudaStream_t stream);
// row i of the output = row slots[i] of src
void launch_gather_rows(const RowsView& src, const uint32_t* slots, uint32_t n, uint8_t* out_rows, float* out_sq,
                        float* out_nrm, cudaStream_t stream);

void launch_gather_u64(const uint64_t* in, const uint32_t* slots, uint32_t n, uint64_t* out, cudaStream_t stream);
void launch_gather_u32(const uint32_t* in, const uint32_t* slots, uint32_t n, uint32_t* out, cudaStream_t stream);
// result row i of [n][k] (keys, dists, counts) goes to row map[i] of the output (counts / out_counts nullable)
void launch_scatter_topk(const uint64_t* keys, const float* dists, const uint32_t* counts, const uint32_t* map, uint32_t n,
                         uint32_t k, uint64_t* out_keys, float* out_dists, uint32_t* out_counts, cudaStream_t stream);

// K1 + K3 (exact.cu) ----------------------------------------------------------------------------
struct ExactParams {
    int storage = 0, metric = 0;
    RowsView q;                       // converted queries
    RowsView x;                       // corpus block; candidate slots are x_base + row index
    uint32_t x_lo = 0, x_hi = 0;      // row range inside x
    const uint32_t* deny = nullptr;   // tombstone bitmap over rows of x (nullable)
    const uint64_t* keys = nullptr;   // u64 key per row of x (tie-break + output)
    Allow allow;                      // N1: filter over (key & 2^48-1), of_q indexed by query of q
    uint32_t kp = 32;                 // candidate list length, multiple of 32, <= 256
    uint32_t n_splits = 1;
    uint64_t* part = nullptr;         // scratch [q.n][n_splits][kp]
    // tensor-core launches only (exact_tc.cu): a tile-strided sample of the rows, and sampled initial list bounds
    uint32_t tile_step = 0;           // rows between tile starts (0 = contiguous tiles)
    uint32_t max_tiles = 0;           // at most this many tiles per row split (0 = all)
    const float* thr_init = nullptr;  // [q.n] rows farther than this never enter the query's lists
};
size_t exact_part_elems(uint32_t nq, uint32_t n_splits, uint32_t kp);
uint32_t exact_pick_splits(uint32_t nq, uint32_t n_rows, int sm_count);
// candidates by approximate distance (any summation order), over-fetched to kp
void launch_exact_candidates(const ExactParams& p, cudaStream_t stream);
// merge the split lists, re-evaluate the canonical distance, sort by (distance,key), emit top-k.
//   out_keys/out_dists/out_counts: user-facing result (nullable)
//   out_packed: [q.n][k] packed (ord(dist)<<32 | slot), kInvalidPacked padded (nullable; used by the build)
//   self_base: if >= 0 the query i is row (self_base + i) of x and is dropped from its own list
//   cert: the candidate stage ran at reduced precision; flag every query whose top-k is not PROVABLY the
//         full-precision one (see exact_rerank_kernel step 4) so the caller can re-run those on the SIMT path
//   q_map: query i of this launch is query q_map[i] of the caller (outputs are written to row q_map[i])
struct ExactCert {
    const float* x_nrm_max = nullptr;  // device scalar: max row norm of the searched block
    float rel = 0.0f;                  // bound on |dot_candidate - dot_canonical| / (|q| |x|)
    float sum = 0.0f;                  // relative rounding bound of an fp32 sum of `dim` terms
    uint32_t* flags = nullptr;         // [q.n] 1 = not certified
    uint32_t* count = nullptr;         // device scalar, incremented per flagged query (zeroed by the caller)
};
void launch_exact_rerank(const ExactParams& p, uint32_t k, uint64_t* out_keys, float* out_dists,
                         uint32_t* out_counts, uint64_t* out_packed, int64_t self_base, cudaStream_t stream,
                         const ExactCert* cert = nullptr, const uint32_t* q_map = nullptr);
// K1c canonical scan (no candidate stage): writes exact_scan_lists_per_query(n_splits) lists of p.kp entries
// per query into p.part; follow with launch_exact_rerank on ExactParams{kp, n_splits = lists per query}.
uint32_t exact_scan_pick_splits(uint32_t nq, uint32_t n_rows, int sm_count);
uint32_t exact_scan_lists_per_query(uint32_t n_splits);
void launch_exact_scan(const ExactParams& p, uint32_t k, cudaStream_t stream);
void launch_max_norm(const float* nrm, uint32_t lo, uint32_t hi, float* out, cudaStream_t stream);

// Bound on |candidate-stage distance - canonical distance| for every row of a block whose largest row norm is xm:
// rel bounds the dot-product error relative to |q||x|, sum the rounding of an fp32 sum of `dim` terms (the norms of
// the L2 expansion, the canonical sum itself).  The K3 certificate and the range-search margin both use it.
template <int METRIC>
__host__ __device__ __forceinline__ float cert_margin(float rel, float sum, float qn, float xm) {
    if constexpr (METRIC == VSB_METRIC_COS)
        return rel + 1e-6f;
    else if constexpr (METRIC == VSB_METRIC_L2SQ)
        return (rel + sum) * (qn * qn + xm * xm);
    else
        return rel * qn * xm + 0x1p-22f * (1.0f + qn * xm);
}

// Range search: the K1 tiles with a fixed per-query bound instead of a k'-list (exact.cu, exact_tc.cu).
//   count pass (off == nullptr): count[q] += admissible rows whose candidate-stage distance is <= thr[q]
//   fill pass: the same rows, as packed (candidate distance, slot) entries, go to out[off[q] + i] for
//              i = cursor[q]++ (space reserved once per flush), and only while i < count[q]; the caller checks that
//              every cursor ends equal to its count
struct RangeParams {
    const float* thr = nullptr;     // [q.n]
    uint32_t* count = nullptr;      // [q.n]
    const uint32_t* off = nullptr;  // [q.n] segment starts in out (fill pass)
    uint32_t* cursor = nullptr;     // [q.n] zeroed by the caller (fill pass)
    uint64_t* out = nullptr;
};
void launch_range_candidates(const ExactParams& p, const RangeParams& r, cudaStream_t stream);
// false if the TMA descriptors could not be encoded (nothing launched)
bool launch_range_candidates_tc(const ExactParams& p, const RangeParams& r, cudaStream_t stream);
// thr[q] = max_distance[q] + cert_margin(rel, sum, |q|, *x_nrm_max), rounded up; integer storages are exact in the
// candidate stage (margin 0) except int8 L2sq, whose norm expansion can round above 2^24; cosine queries of norm 0
// get +inf (their candidate distance is 1, the canonical one 0 or 1)
void launch_range_bound(int storage, int metric, const float* q_nrm, const float* max_distance, uint32_t n,
                        const float* x_nrm_max, float rel, float sum, float* thr, cudaStream_t stream);
// Canonical re-evaluation of the fill pass's entries, four rows per warp (K3's evaluation).  Query q's segment is
// cand[seg_off[q] .. seg_off[q + 1]), its warps are groups grp_off[q] .. grp_off[q + 1] (ceil(count / 4) each).  Per
// entry: key_out = its key, dord_out = ord(canonical distance) if that is <= max_distance[q], else 0xFFFFFFFF;
// kept[q] += rows kept.  *mismatch += queries of p.q whose cursor differs from their count, every query checked
// (entries past the smaller of the two are never read).
void launch_range_eval(const ExactParams& p, const float* max_distance, const uint32_t* count, const uint32_t* cursor,
                       const uint32_t* seg_off, const uint32_t* grp_off, uint32_t n_groups, const uint64_t* cand,
                       uint64_t* key_out, uint32_t* dord_out, uint32_t* kept, uint32_t* mismatch, cudaStream_t stream);
// Sorts every segment of (dord, key) by (dord, key) in place; alt_* are buffers of the same size, temp from
// range_sort_temp_bytes.  Deterministic.
size_t range_sort_temp_bytes(uint32_t n_entries, uint32_t n_segments);
cudaError_t launch_range_sort(uint32_t* dord, uint64_t* key, uint32_t* alt_dord, uint64_t* alt_key, uint32_t n_entries,
                              const uint32_t* seg_off, uint32_t n_segments, void* temp, size_t temp_bytes,
                              cudaStream_t stream);
// Output entry e of query q (out_off[q] <= e < out_off[q + 1]) = entry seg_off[q] + (e - out_off[q]) of the sorted
// segments, as (key, float distance).
void launch_range_emit(const uint32_t* dord, const uint64_t* key, const uint32_t* seg_off, const uint32_t* out_off,
                       uint32_t n, uint32_t total, uint64_t* keys_out, float* dists_out, cudaStream_t stream);

// K1 on tcgen05 tensor cores (exact_tc.cu): same contract as launch_exact_candidates.
bool exact_tc_supported(int storage, int metric);
uint32_t exact_tc_pick_splits(uint32_t nq, uint32_t n_rows, int sm_count, uint32_t kp);
bool launch_exact_candidates_tc(const ExactParams& p, cudaStream_t stream, bool tile_min = false);
// tile-min launches write a DENSE array of exact_tc_tile_min_entries(rows) packed winners per query into p.part (one
// per 256-row tile half, in row order; padding and empty tiles = kInvalidPacked, the caller pre-fills the padding with
// 0xFF) whatever p.n_splits is; p.x_lo must be 0.
uint32_t exact_tc_tile_min_entries(uint32_t n_rows);
// sampled list bounds (see tc_sample_threshold_kernel): sample_part = [nq][exact_tc_halves()][32] lists of a sample pass
uint32_t exact_tc_halves();
void launch_tc_sample_threshold(const uint64_t* sample_part, uint32_t nq, uint32_t m, float* thr, cudaStream_t stream);
void launch_tc_count_short(const uint64_t* part, uint32_t nq, uint32_t lists, uint32_t kp, uint32_t need, uint32_t* counter,
                           cudaStream_t stream);

// K6 (graph_build.cu) ---------------------------------------------------------------------------
// knn: [n][k_init] packed lists (ascending); produces fwd [n][R] pruned by detour count.
void launch_prune_detour(const uint64_t* knn, uint32_t n, uint32_t k_init, uint32_t R, const uint32_t* deny,
                         uint32_t* fwd, cudaStream_t stream);
// deterministic reverse-edge lists: rev [n][R] (sorted by (rank in source list, source slot)), rev_cnt[n]
size_t reverse_edges_scratch_bytes(uint32_t n, uint32_t R);
void launch_reverse_edges(const uint32_t* fwd, uint32_t n, uint32_t R, uint32_t* rev, uint32_t* rev_cnt,
                          void* scratch, size_t scratch_bytes, cudaStream_t stream);
// final rows: fwd[0:R/2] ++ reverse edges (unique) ++ remaining fwd, padded with kInvalidSlot
void launch_merge_graph(const uint32_t* fwd, const uint32_t* rev, const uint32_t* rev_cnt, uint32_t n,
                        uint32_t R, uint32_t* graph, uint32_t graph_stride, cudaStream_t stream);

// reachability from the seed sample (graph_build.cu): state bytes 0 = unreached, 1 = frontier, 2 = expanded
void launch_reach_mark(uint8_t* state, const uint32_t* seeds, uint32_t n_seeds, cudaStream_t stream);
void launch_reach_step(const uint32_t* graph, uint32_t n, uint32_t stride, uint32_t degree, uint8_t* state,
                       uint32_t* changed, cudaStream_t stream);
// out[0] = number found (<= cap), out[1..] = the first `cap` unreached live slots in slot order; state must be
// readable 16 bytes past n
void launch_collect_unreached(const uint8_t* state, const uint32_t* deny, uint32_t n, uint32_t cap, uint32_t* out,
                              cudaStream_t stream);
void launch_first_unreached(const uint8_t* state, const uint32_t* deny, uint32_t n, uint32_t* out, cudaStream_t stream);

// compaction: renumber the rows and the edges of a graph through old2new (kInvalidSlot = removed)
void launch_remap_graph(const uint32_t* graph, uint32_t n_old, uint32_t stride, const uint32_t* old2new, uint32_t* out,
                        cudaStream_t stream);

// K7 (graph_build.cu): link a batch of already-searched new rows into the graph (detour-pruned forward rows,
// then reverse edges in a deterministic order); cand = [n_new][cand_stride] packed ascending candidates
size_t stream_link_scratch_bytes(uint32_t n_new, uint32_t R);
cudaError_t launch_stream_link(const uint64_t* cand, uint32_t n_new, uint32_t cand_stride, uint32_t first_slot, uint32_t R,
                               uint32_t* graph, uint32_t graph_stride, void* scratch, size_t scratch_bytes,
                               cudaStream_t stream);

// K4 (graph_search.cu) ---------------------------------------------------------------------------
struct SearchParams {
    int storage = 0, metric = 0;
    RowsView q;
    RowsView x;
    const uint32_t* graph = nullptr;  // [n_graphed][graph_stride]
    uint32_t graph_stride = 32, degree = 32;
    uint32_t n_graphed = 0;
    const uint64_t* seed_lists = nullptr;  // [q.n][seed_stride] packed (approx dist, seed index)
    uint32_t seed_stride = 32, n_seeds = 32;
    const uint32_t* seed_slots = nullptr;  // seed index -> slot
    const uint32_t* deny = nullptr;
    const uint64_t* keys = nullptr;
    uint32_t itopk = 64, max_iters = 0, k = 10, search_width = 1;
    uint64_t* out_keys = nullptr;
    float* out_dists = nullptr;
    uint32_t* out_counts = nullptr;
    uint64_t* out_packed = nullptr;          // packed (dist, slot) output for a following K3 re-rank
    long long self_base = -1;                // >= 0: query i is row self_base + i (excluded from its own list)
    uint32_t out_stride = 0;                 // packed entries per query (0 = k)
    unsigned long long* counters = nullptr;  // [2]: distance evals, parent expansions (instrumented only)
    // filtered ANN (usearch.rs:224-248): every row is traversed, only rows whose bit (key & 2^48-1) is set enter the
    // result list (a second list next to the traversal list)
    Allow allow;
    // 16-bit float rows, warp-per-query kernel only: evaluate the rows on the tensor cores (mma.sync, candidate-grade
    // distances — the caller re-ranks the rows it returns).  graph_search_uses_mma() tells which launches honour it.
    bool mma = false;
};
bool graph_search_uses_mma(int storage, uint32_t n_queries, bool filtered, uint32_t itopk);
void launch_graph_search(const SearchParams& p, cudaStream_t stream);
bool graph_search_supported(uint32_t row_bytes);  // rows up to 6144 bytes
uint32_t graph_search_small_batch();
uint32_t seed_scan_blocks(uint32_t n_seed_rows);
void launch_seed_scan(int storage, int metric, const RowsView& q, const RowsView& seeds, uint64_t* out,
                      cudaStream_t stream);

// K8 (merge.cu) ----------------------------------------------------------------------------------
// key_part_stride / dist_part_stride: elements between consecutive parts (0 = q*k, parts back to back)
void launch_merge_topk(const uint64_t* keys, const float* dists, uint32_t parts, uint64_t q, uint32_t k,
                       uint64_t* out_keys, float* out_dists, uint32_t* out_counts, cudaStream_t stream,
                       uint64_t key_part_stride = 0, uint64_t dist_part_stride = 0);
// fills [n] key/dist arrays with the padding values
void launch_fill_empty(uint64_t* keys, float* dists, uint32_t* counts, uint64_t q, uint32_t k, cudaStream_t stream);

}  // namespace vsb
