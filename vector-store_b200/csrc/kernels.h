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
};

// K0 ------------------------------------------------------------------------------------------
void launch_convert_rows(int storage, const float* in, uint32_t n_rows, uint32_t dim, uint8_t* out,
                         uint32_t row_bytes, float* sq, float* nrm, cudaStream_t stream);
// scaled int8 copy for the cosine traversal (per-row scale max|x|/127; nrm = |x| in units of the scale)
void launch_convert_rows_i8s(const float* in, uint32_t n_rows, uint32_t dim, uint32_t in_stride, uint8_t* out,
                             uint32_t row_bytes, float* sq, float* nrm, cudaStream_t stream);
void launch_gather_rows(const uint8_t* rows, uint32_t row_bytes, const float* sq, const float* nrm,
                        const uint32_t* slots, uint32_t n, uint8_t* out_rows, float* out_sq, float* out_nrm,
                        cudaStream_t stream);

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
    const uint32_t* allow = nullptr;  // N1: bitmap over (key & 2^48-1) (nullable)
    uint64_t allow_bits = 0;
    // [q.n] index of each query's bitmap: query i tests allow + allow_of_q[i] * ceil(allow_bits / 32)
    // (nullable: every query uses the first bitmap)
    const uint32_t* allow_of_q = nullptr;
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
    const uint32_t* allow = nullptr;
    uint64_t allow_bits = 0;
    const uint32_t* allow_of_q = nullptr;  // per-query bitmap index, as in ExactParams (nullable)
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
