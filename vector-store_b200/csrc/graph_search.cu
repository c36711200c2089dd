// graph_search.cu — host launcher of K4 (kernel in graph_search.cuh, instantiated per storage scalar).
#include "graph_search.cuh"

namespace vsb {

static int pick_cpl(int n_chunks) {
    const int need = (n_chunks + 31) / 32;
    const int set[7] = {1, 2, 3, 4, 6, 8, 12};
    for (int i = 0; i < 7; ++i)
        if (set[i] >= need) return set[i];
    return -1;
}

bool graph_search_supported(uint32_t row_bytes) { return pick_cpl((int)(row_bytes / 16)) > 0; }

// batches up to this size use the CTA-per-query kernel (one CTA per SM-slot still fills the GPU)
uint32_t graph_search_small_batch() { return 256; }

uint32_t seed_scan_blocks(uint32_t n_seed_rows) {
    const uint32_t ctas = (n_seed_rows + SEED_SCAN_WARPS * SEED_SCAN_ROWS_PER_WARP - 1) /
                          (SEED_SCAN_WARPS * SEED_SCAN_ROWS_PER_WARP);
    return (ctas + 31) / 32;
}

// [q][blocks][32] packed per-CTA winners, kInvalidPacked padded (caller pre-fills the buffer with 0xFF)
void launch_seed_scan(int storage, int metric, const RowsView& q, const RowsView& seeds, uint64_t* out,
                      cudaStream_t stream) {
    if (q.n == 0 || seeds.n == 0) return;
    SeedScanArgs s;
    s.q_rows = q.rows; s.q_nrm = q.nrm; s.nq = q.n; s.q_row_bytes = q.row_bytes;
    s.s_rows = seeds.rows; s.s_nrm = seeds.nrm; s.n_seed_rows = seeds.n; s.row_bytes = seeds.row_bytes;
    s.metric = metric; s.n_blocks = seed_scan_blocks(seeds.n); s.out = out;
    switch (storage) {
        case VSB_ST_F32: launch_seed_scan_f32(s, stream); break;
        case VSB_ST_F16: launch_seed_scan_f16(s, stream); break;
        case VSB_ST_BF16: launch_seed_scan_bf16(s, stream); break;
        case VSB_ST_I8: launch_seed_scan_i8(s, stream); break;
        default: launch_seed_scan_b1(s, stream); break;
    }
    g_kernel_launches += 1;
}

// Tensor-core evaluation of 16-bit rows pays for its re-rank (a fixed ~0.09 ms per 10 000 queries) and its
// candidate-grade bookkeeping only on long searches: 10 M rows at ef = 224 gain 6 % (9.19 -> 8.66 ms), 1.25 M-row
// shards at ef = 32 lose 10 % (1.29 -> 1.42 ms + the re-rank).  Automatic: beams of at least 96 entries.
bool graph_search_uses_mma(int storage, uint32_t n_queries, bool filtered, uint32_t itopk) {
    if (filtered || n_queries <= graph_search_small_batch()) return false;
    if (storage != VSB_ST_BF16 && storage != VSB_ST_F16) return false;
    return itopk >= 96;
}

// Visited hash: 16 KB per warp (4096 slots) = 3 CTAs x 4 query warps per SM, the same residency the register budget
// allows; it is reset to "what is still in the list" when 3/4 full (forgotten nodes cost a re-evaluation, never a
// duplicate).
constexpr uint32_t K4_HASH_BITS = 12;

void launch_graph_search(const SearchParams& p, cudaStream_t stream) {
    if (p.q.n == 0) return;
    K4Args a;
    a.q_rows = p.q.rows; a.q_nrm = p.q.nrm; a.nq = p.q.n; a.q_row_bytes = p.q.row_bytes;
    a.x_rows = p.x.rows; a.x_nrm = p.x.nrm; a.x_row_bytes = p.x.row_bytes;
    a.graph = p.graph; a.graph_stride = p.graph_stride; a.degree = p.degree;
    a.seed_lists = p.seed_lists; a.seed_splits = p.seed_stride / 32; a.n_seeds = p.n_seeds;
    a.seed_slots = p.seed_slots; a.deny = p.deny; a.keys = p.keys;
    a.itopk = ((p.itopk + 31) / 32) * 32;
    if (a.itopk < ((p.k + 31) / 32) * 32) a.itopk = ((p.k + 31) / 32) * 32;
    a.search_width = p.search_width < 1 ? 1 : (p.search_width > (uint32_t)K4_MAX_WIDTH ? (uint32_t)K4_MAX_WIDTH : p.search_width);
    a.max_iters = p.max_iters ? p.max_iters : (2 * a.itopk) / a.search_width + 8;
    a.k = p.k;
    a.hash_bits = K4_HASH_BITS;
    const uint32_t deg_pad = ((p.degree + 31) / 32) * 32;
    a.queue_cap = a.search_width * deg_pad < 32 ? 32 : a.search_width * deg_pad;
    a.metric = p.metric;
    a.out_keys = p.out_keys; a.out_dists = p.out_dists; a.out_counts = p.out_counts; a.out_packed = p.out_packed; a.self_base = p.self_base; a.counters = p.counters;
    a.out_stride = p.out_stride ? p.out_stride : p.k;
    a.allow = p.allow.bm;
    a.allow_bits = p.allow.bits;
    a.allow_of_q = p.allow.of_q;
    a.rk = p.allow.bm != nullptr ? ((p.k + 31) / 32) * 32 : 0;
    a.mma = 0;
    const int cpl = pick_cpl((int)(p.x.row_bytes / 16));
    // filtered ANN always runs the warp-per-query kernel (the second list lives there)
    if (p.q.n <= graph_search_small_batch() && p.allow.bm == nullptr) {
        // CTA-per-query kernel: 8 warps and up to 8 parents per iteration for one query
        a.search_width = a.search_width < 4 ? 8 : (a.search_width > 8 ? 8 : a.search_width);
        a.max_iters = p.max_iters ? p.max_iters : (2 * a.itopk) / a.search_width + 8;
        a.queue_cap = a.search_width * deg_pad;
        dim3 gridb(p.q.n);
        const size_t smemb = (size_t)a.itopk * 16 + (size_t)a.queue_cap * 16 + ((size_t)4 << K4_HASH_BITS) + 64 + 128;
        switch (p.storage) {
            case VSB_ST_F32: launch_k4b_f32(a, cpl, gridb, smemb, stream); break;
            case VSB_ST_F16: launch_k4b_f16(a, cpl, gridb, smemb, stream); break;
            case VSB_ST_BF16: launch_k4b_bf16(a, cpl, gridb, smemb, stream); break;
            case VSB_ST_I8: launch_k4b_i8(a, cpl, gridb, smemb, stream); break;
            default: launch_k4b_b1(a, cpl, gridb, smemb, stream); break;
        }
        g_kernel_launches += 1;
        return;
    }
    dim3 grid((p.q.n + K4_WARPS - 1) / K4_WARPS);
    a.mma = (p.mma && p.allow.bm == nullptr && (p.storage == VSB_ST_BF16 || p.storage == VSB_ST_F16)) ? 1u : 0u;
    const size_t smem = (size_t)K4_WARPS * ((size_t)a.itopk * 8 + ((size_t)2 << K4_HASH_BITS) + (size_t)a.queue_cap * 8 + (size_t)a.rk * 8 + 64 * 8);
    switch (p.storage) {
        case VSB_ST_F32: launch_k4_f32(a, cpl, grid, smem, stream); break;
        case VSB_ST_F16: launch_k4_f16(a, cpl, grid, smem, stream); break;
        case VSB_ST_BF16: launch_k4_bf16(a, cpl, grid, smem, stream); break;
        case VSB_ST_I8: launch_k4_i8(a, cpl, grid, smem, stream); break;
        default: launch_k4_b1(a, cpl, grid, smem, stream); break;
    }
    g_kernel_launches += 1;
}

}  // namespace vsb
