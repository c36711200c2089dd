// exact_tc.cu — K1 on the 5th-generation tensor cores: Q x N distance tiles with tcgen05.mma,
// operands staged by TMA into 128B-swizzled shared memory, accumulators in TMEM, and the top-k'
// selection (K2) fused into the TMEM epilogue so the Q x N matrix never exists.
//
// Used for the dense parts of the path (SURVEY §8a K1/K5): the seed layer of every ANN search,
// exact search on 16-bit storage, and the all-pairs kNN lists of the bulk graph build — the work
// `usearch::Index::add` / `search` spend in SimSIMD distance loops in the reference
// (vs_index/usearch.rs:191-222).  Output format is identical to exact.cu's K1 (per-split sorted
// candidate lists), so K3 (exact_rerank_kernel) finishes both the same way.
//
// CTA = 320 threads, one CTA per SM (TMEM 512 columns, ~217 KB smem):
//   warp 0      TMA producer: A = 128 queries x 128 B of K, B = 256 corpus rows x 128 B of K,
//               3-stage mbarrier ring (full/empty)
//   warp 1      tcgen05.mma issuer (one elected lane): D[128 x 256] fp32 in TMEM, double buffered
//               (2 x 256 columns) so the epilogue of tile t overlaps the MMAs of tile t+1
//   warps 2-9   epilogue, two warps per TMEM lane quarter, each owning 128 of the tile's 256 columns
//               (a "column half" = its own candidate list per query, merged by K3 like a split):
//               tcgen05.ld 32 lanes x 32 columns at a time; thread = one query row; distance from
//               the dot product and per-column norms; a 32-bit hit mask against the row's current
//               k'-th best (register); the columns in which ANY row of the warp hit are revisited
//               in a warp-uniform loop (one tcgen05.ld.x1 each) and the survivors go to a 32-entry
//               per-row smem buffer that is sorted with the shuffle bitonic network and folded into
//               the row's list when full (tc_flush_rows, kept out of line: the tile loop stays
//               small enough for the instruction cache).
// kind::f16 (bf16 / f16 storage, exact products) or kind::tf32 (f32 storage, candidate grade).
#include <cuda.h>

#include <algorithm>
#include <cmath>
#include <cstdlib>

#include "kernels.h"
#include "select.cuh"

namespace vsb {

namespace {

constexpr int TC_M = 128;
constexpr int TC_N = 256;
constexpr int TC_KBYTES = 128;
constexpr int TC_STAGES = 3;       // 1-CTA variant: 3 x 48 KB
constexpr int TC2_STAGES = 4;      // 2-CTA variant: 4 x 32 KB (each CTA stages its own A and half of B)
constexpr int TC_BUFCAP = 32;        // candidates buffered per (query row, column half) before a flush
constexpr int TC_HALVES = 2;         // epilogue warps per TMEM lane quarter = candidate lists per (query, row split)
constexpr int TC_HALF_N = TC_N / TC_HALVES;
constexpr int TC_EPI_WARPS = 4 * TC_HALVES;
constexpr int TC_THREADS = 64 + 32 * TC_EPI_WARPS;
constexpr uint32_t TC_A_BYTES = TC_M * TC_KBYTES;   // 16 KB
constexpr uint32_t TC_B_BYTES = TC_N * TC_KBYTES;   // 32 KB
constexpr uint32_t TC_STAGE_BYTES = TC_A_BYTES + TC_B_BYTES;
constexpr uint32_t TC_OFF_BUF = TC_STAGES * TC_STAGE_BYTES;
constexpr uint32_t TC_OFF_COLP = TC_OFF_BUF + TC_HALVES * TC_M * TC_BUFCAP * 8;
constexpr uint32_t TC_OFF_BAR = TC_OFF_COLP + TC_EPI_WARPS * 2 * TC_HALF_N * 4;  // per epilogue warp, per accumulator stage
constexpr uint32_t TC_SMEM_BYTES = TC_OFF_BAR + 128 + 1024;  // + alignment slack
// both variants use the same offsets for buf / colp / barriers: 4 x 32 KB < 3 x 48 KB
static_assert(TC2_STAGES * (TC_A_BYTES + TC_B_BYTES / 2) <= TC_OFF_BUF, "2-CTA stages must fit the stage area");
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;  // shared::cluster address of the same offset in the even (leader) CTA

enum { KIND_BF16 = 0, KIND_F16 = 1, KIND_TF32 = 2 };

struct TcArgs {
    const float* q_sq;
    const float* q_nrm;
    uint32_t nq;
    const float* x_sq;
    const float* x_nrm;
    uint32_t x_lo, x_hi, row_bytes;
    const uint32_t* deny;
    const uint64_t* keys;
    const uint32_t* allow;
    uint64_t allow_bits;
    const uint32_t* allow_of_q;  // [nq] bitmap index per query (nullable: bitmap 0)
    uint32_t kp, n_splits, rows_per_split;  // n_splits = lists per query = TC_HALVES * gridDim.y
    uint64_t* part;
    int tile_min;  // 1: emit only each tile's best row per query (seed layer), no list maintenance
    uint32_t tile_min_stride;  // tile-min mode: entries per query in `part`, entry = (global tile) * TC_HALVES + half
    uint32_t tile_step;        // rows between the starts of consecutive tiles (TC_N; larger = a tile-strided SAMPLE of the rows)
    uint32_t max_tiles;        // 0 = every tile of the split; else at most this many (sample passes)
    const float* thr_init;     // [nq] initial k'-th-best bound per query (nullable): rows farther than this are never listed
};

// ---- PTX wrappers ------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra WAIT_DONE;\n"
        "bra WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
            smem_u32(smem_dst)),
        "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d_2sm(void* smem_dst, const CUtensorMap* map, uint64_t* leader_bar, int c0,
                                                int c1) {
    // issued by both CTAs of the pair; the transaction bytes are credited to the leader CTA's barrier
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], "
        "[%2];" ::"r"(smem_u32(smem_dst)),
        "l"(map), "r"(smem_u32(leader_bar) & kPeerBitMask), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void mbar_arrive_remote(uint64_t* bar, uint32_t cta_rank) {
    asm volatile(
        "{\n.reg .b32 ra;\nmapa.shared::cluster.u32 ra, %0, %1;\nmbarrier.arrive.shared::cluster.b64 _, [ra];\n}\n" ::"r"(
            smem_u32(bar)),
        "r"(cta_rank)
        : "memory");
}
__device__ __forceinline__ void tc_commit_2sm(uint64_t* bar) {
    // arrives on the barrier at this offset in BOTH CTAs of the pair once the MMAs issued so far retire
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                     smem_u32(bar)),
                 "h"((uint16_t)3)
                 : "memory");
}
template <int KIND>
__device__ __forceinline__ void tc_mma_2sm(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    if constexpr (KIND == KIND_TF32) {
        asm volatile(
            "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
            "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, {%5, %5, %5, %5, %5, %5, %5, %5}, p;\n}\n" ::"r"(tmem_d),
            "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc), "r"(0u)
            : "memory");
    } else {
        asm volatile(
            "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
            "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, {%5, %5, %5, %5, %5, %5, %5, %5}, p;\n}\n" ::"r"(tmem_d),
            "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc), "r"(0u)
            : "memory");
    }
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t cluster_cta_rank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
template <int KIND>
__device__ __forceinline__ void tc_mma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    if constexpr (KIND == KIND_TF32) {
        asm volatile(
            "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
            "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n}\n" ::"r"(tmem_d),
            "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc), "r"(0u)
            : "memory");
    } else {
        asm volatile(
            "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
            "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n}\n" ::"r"(tmem_d),
            "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc), "r"(0u)
            : "memory");
    }
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* v) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

__device__ __forceinline__ uint32_t tmem_ld1(uint32_t taddr) {
    uint32_t v;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];\n" : "=r"(v) : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    return v;
}

__device__ __forceinline__ uint32_t tmem_ld1_nowait(uint32_t taddr) {
    uint32_t v;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];\n" : "=r"(v) : "r"(taddr));
    return v;
}
// the loaded registers are operands of the wait, so no use of them can be scheduled above it
__device__ __forceinline__ void tmem_wait_ld4(uint32_t& a, uint32_t& b, uint32_t& c, uint32_t& d) {
    asm volatile("tcgen05.wait::ld.sync.aligned;" : "+r"(a), "+r"(b), "+r"(c), "+r"(d)::"memory");
}

// Candidate-stage distance of one (query, corpus row) pair from the tile's dot product.  col = per-column parameter
// (|x|^2, 1/|x|, 1), qpar = per-query parameter (|q|^2, -1/|q|, unused).  One definition for the hit test and for the
// value that is stored, so both see the same bits.
template <int METRIC>
__device__ __forceinline__ float tc_dist(float dot, float col, float qpar) {
    if constexpr (METRIC == VSB_METRIC_L2SQ) return __fadd_rn(__fmaf_rn(dot, -2.0f, col), qpar);
    else if constexpr (METRIC == VSB_METRIC_COS) return __fmaf_rn(__fmul_rn(dot, col), qpar, 1.0f);
    else return __fmaf_rn(dot, -1.0f, col);
}

// Folds the buffered candidates of the rows in `need_mask` (bit r = row r of this warp) into their lists: the whole
// warp sorts one row's buffer (shuffle bitonic network) and carry-merges it into the row's sorted list in global
// memory.  Returns the calling lane's threshold: the new k'-th best of its row if that row was flushed and its list
// is full, `thr` otherwise.  Out of line on purpose (called from the tile loop's rare path).
__device__ __noinline__ float tc_flush_rows(uint32_t need_mask, uint64_t* warp_lists, size_t list_stride, uint32_t kp,
                                            const uint64_t* keys, const uint64_t* warp_buf, int cnt, float thr, int lane) {
    const LessByKey less{keys};
    constexpr int MAXB = 8;  // kp <= 256
    const int nb = (int)(kp >> 5);
    __syncwarp();  // make every lane's buffered candidates visible to the warp
    // The lists live in global memory (L2): all blocks of a row's list are fetched with independent loads BEFORE the
    // buffer is sorted, and the next row's list is fetched while this row's is merged, so a flush pays the L2
    // latency once instead of once per 32-entry block (the build's all-pairs lists are 128 long and flush ~60 times
    // per row and launch).
    uint64_t blk[MAXB], nxt[MAXB];
    int r = __ffs(need_mask) - 1;
    need_mask &= need_mask - 1;
    {
        const uint64_t* list = warp_lists + (size_t)r * list_stride;
#pragma unroll
        for (int b = 0; b < MAXB; ++b) blk[b] = b < nb ? list[b * 32 + lane] : kInvalidPacked;
    }
    while (true) {
        const int r_next = need_mask ? __ffs(need_mask) - 1 : -1;
        need_mask &= need_mask - 1;
        if (r_next >= 0) {
            const uint64_t* list = warp_lists + (size_t)r_next * list_stride;
#pragma unroll
            for (int b = 0; b < MAXB; ++b) nxt[b] = b < nb ? list[b * 32 + lane] : kInvalidPacked;
        }
        const int c = __shfl_sync(kFullMask, cnt, r);
        uint64_t* list = warp_lists + (size_t)r * list_stride;
        uint64_t carry = lane < c ? warp_buf[(size_t)r * TC_BUFCAP + lane] : kInvalidPacked;
        carry = warp_sort32(carry, lane, less);
        uint64_t worst = kInvalidPacked;
        // one ROLLED loop over the blocks (the body — two bitonic merges — is the bulk of this function's code and
        // must stay small for the instruction cache); the prefetched blocks rotate through blk[0]
#pragma unroll 1
        for (int b = 0; b < nb; ++b) {
            uint64_t cur = blk[0];
#pragma unroll
            for (int i = 0; i + 1 < MAXB; ++i) blk[i] = blk[i + 1];
            // nothing in the carry beats this block's maximum -> block unchanged, carry unchanged
            const uint64_t blk_max = shfl_u64(cur, 31);
            const uint64_t carry_min = shfl_u64(carry, 0);
            if (less(carry_min, blk_max)) {
                const uint64_t rc = shfl_u64(carry, 31 - lane);
                const bool rc_less = less(rc, cur);
                uint64_t lo = rc_less ? rc : cur;
                uint64_t hi = rc_less ? cur : rc;
                lo = warp_bitonic_merge32(lo, lane, less);
                hi = warp_bitonic_merge32(hi, lane, less);
                list[b * 32 + lane] = lo;
                cur = lo;
                carry = hi;
            }
            worst = shfl_u64(cur, 31);  // after the last block: the list's k'-th best
        }
        if (lane == r && worst != kInvalidPacked) thr = ord_to_f32(packed_hi(worst));
        if (r_next < 0) break;
        r = r_next;
#pragma unroll
        for (int b = 0; b < MAXB; ++b) blk[b] = nxt[b];
    }
    __syncwarp();
    return thr;
}

// K-major, 128B-swizzled operand tile: rows of 128 bytes, 8-row atoms 1024 bytes apart.
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);   // start address
    d |= (uint64_t)1 << 16;                        // leading byte offset (unused for swizzled K-major)
    d |= (uint64_t)(1024 >> 4) << 32;              // stride byte offset: 8 rows * 128 B
    d |= (uint64_t)1 << 46;                        // descriptor version (Blackwell)
    d |= (uint64_t)2 << 61;                        // SWIZZLE_128B
    return d;
}

// CTA2 = true: the kernel runs as clusters of two CTAs (cta_group::2).  Each CTA owns its own 128 query rows
// (its half of the M = 256 accumulator) and stages only 128 of the tile's 256 corpus rows; the leader CTA issues
// the MMAs for the pair, so a CTA moves 32 KB instead of 48 KB per K slab and a fourth stage fits.
template <int KIND, int METRIC, bool TILE_MIN, bool CTA2>
__global__ void __launch_bounds__(TC_THREADS, 1)
    exact_candidates_tc_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_x,
                               TcArgs a) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint64_t* buf = reinterpret_cast<uint64_t*>(smem + TC_OFF_BUF);
    float* colp = reinterpret_cast<float*>(smem + TC_OFF_COLP);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + TC_OFF_BAR);
    uint64_t* full = bars;                    // [<= TC2_STAGES]
    uint64_t* empty = bars + TC2_STAGES;      // [<= TC2_STAGES]
    uint64_t* tmem_full = bars + 2 * TC2_STAGES;  // [2]
    uint64_t* tmem_empty = tmem_full + 2;         // [2]
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_empty + 2);

    const int warp = __shfl_sync(kFullMask, (int)(threadIdx.x >> 5), 0);
    const int lane = threadIdx.x & 31;
    const uint32_t q0 = blockIdx.x * TC_M;
    const uint32_t split = blockIdx.y;
    const uint32_t r_lo = a.x_lo + split * a.rows_per_split;
    const uint32_t r_hi = min(a.x_hi, r_lo + a.rows_per_split);
    uint32_t n_tiles = r_hi > r_lo ? (r_hi - r_lo + a.tile_step - 1) / a.tile_step : 0;
    if (a.max_tiles != 0 && n_tiles > a.max_tiles) n_tiles = a.max_tiles;
    const uint32_t n_slabs = (a.row_bytes + TC_KBYTES - 1) / TC_KBYTES;
    constexpr int ELEMS_PER_SLAB = KIND == KIND_TF32 ? 32 : 64;
    constexpr int STAGES = CTA2 ? TC2_STAGES : TC_STAGES;
    constexpr uint32_t B_BYTES = CTA2 ? TC_B_BYTES / 2 : TC_B_BYTES;
    constexpr uint32_t STAGE_BYTES = TC_A_BYTES + B_BYTES;
    const uint32_t cta_rank = CTA2 ? cluster_cta_rank() : 0u;
    const bool leader = cta_rank == 0;

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_q) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_x) : "memory");
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], 1);
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&tmem_full[i], 1);
            mbar_init(&tmem_empty[i], CTA2 ? 2 * TC_EPI_WARPS : TC_EPI_WARPS);  // the leader also waits for the peer CTA's epilogue warps
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        if constexpr (CTA2) {
            asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr)),
                         "r"(512u));
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::);
        } else {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr)),
                         "r"(512u));
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
        }
    }
    tc_fence_before();
    if constexpr (CTA2) cluster_sync_all(); else __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;

    if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0) {
            uint32_t stage = 0, phase = 0;
            for (uint32_t t = 0; t < n_tiles; ++t) {
                const int n0 = (int)(r_lo + t * a.tile_step);
                for (uint32_t slab = 0; slab < n_slabs; ++slab) {
                    mbar_wait(&empty[stage], phase ^ 1);
                    uint8_t* sa = smem + stage * STAGE_BYTES;
                    if constexpr (CTA2) {
                        // both CTAs load their own halves; all bytes are credited to the leader's barrier
                        if (leader) mbar_arrive_expect_tx(&full[stage], 2 * STAGE_BYTES);
                        tma_load_2d_2sm(sa, &tmap_q, &full[stage], (int)(slab * ELEMS_PER_SLAB), (int)q0);
                        tma_load_2d_2sm(sa + TC_A_BYTES, &tmap_x, &full[stage], (int)(slab * ELEMS_PER_SLAB),
                                        n0 + (int)cta_rank * (TC_N / 2));
                    } else {
                        mbar_arrive_expect_tx(&full[stage], STAGE_BYTES);
                        tma_load_2d(sa, &tmap_q, &full[stage], (int)(slab * ELEMS_PER_SLAB), (int)q0);
                        tma_load_2d(sa + TC_A_BYTES, &tmap_x, &full[stage], (int)(slab * ELEMS_PER_SLAB), n0);
                    }
                    if (++stage == STAGES) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer =====
        if (lane == 0 && leader) {
            constexpr uint32_t fmt = KIND == KIND_BF16 ? 1u : (KIND == KIND_F16 ? 0u : 2u);
            constexpr uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(TC_N >> 3) << 17) |
                                       ((uint32_t)((CTA2 ? 2 * TC_M : TC_M) >> 4) << 24);
            uint32_t stage = 0, phase = 0;
            for (uint32_t t = 0; t < n_tiles; ++t) {
                const uint32_t acc = t & 1, acc_phase = (t >> 1) & 1;
                mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
                tc_fence_after();
                const uint32_t tmem_d = tmem_base + acc * TC_N;
                for (uint32_t slab = 0; slab < n_slabs; ++slab) {
                    mbar_wait(&full[stage], phase);
                    tc_fence_after();
                    const uint32_t sa = smem_u32(smem + stage * STAGE_BYTES);
                    const uint64_t adesc = make_smem_desc(sa);
                    const uint64_t bdesc = make_smem_desc(sa + TC_A_BYTES);
#pragma unroll
                    for (uint32_t k = 0; k < TC_KBYTES / 32; ++k) {
                        // +32 bytes of K inside the swizzle atom = +2 in the (addr >> 4) field
                        if constexpr (CTA2)
                            tc_mma_2sm<KIND>(tmem_d, adesc + 2 * k, bdesc + 2 * k, idesc, (slab | k) != 0 ? 1u : 0u);
                        else
                            tc_mma<KIND>(tmem_d, adesc + 2 * k, bdesc + 2 * k, idesc, (slab | k) != 0 ? 1u : 0u);
                    }
                    if constexpr (CTA2) tc_commit_2sm(&empty[stage]); else tc_commit(&empty[stage]);
                    if (++stage == STAGES) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
                if constexpr (CTA2) tc_commit_2sm(&tmem_full[acc]); else tc_commit(&tmem_full[acc]);
            }
        }
    } else {
        // ===== epilogue: one thread per (query row, column half) =====
        const int quarter = warp & 3;                // TMEM lane quarter this warp may read (hardware: warp id % 4)
        const int half = (warp - 2) >> 2;            // which 128 columns of every tile this warp owns
        const int row = quarter * 32 + lane;         // row inside the CTA tile
        const uint32_t q = q0 + row;
        const bool q_valid = q < a.nq;
        const uint32_t list_id = split * TC_HALVES + half;   // a.n_splits = TC_HALVES * (row splits)
        uint64_t* my_buf = buf + ((size_t)half * TC_M + row) * TC_BUFCAP;
        float qpar = 0.f;   // L2sq: |q|^2; cosine: -1/|q|
        if (q_valid) {
            if constexpr (METRIC == VSB_METRIC_L2SQ) qpar = a.q_sq[q];
            if constexpr (METRIC == VSB_METRIC_COS) {
                const float qn = a.q_nrm[q];
                qpar = qn > 0.f ? -(1.0f / qn) : 0.f;
            }
        }
        // this warp's 32 lists live in global memory (L2 resident); row r's list is r * list_stride further on
        const size_t list_stride = (size_t)a.n_splits * a.kp;
        uint64_t* warp_lists = a.part + ((size_t)(q0 + quarter * 32) * a.n_splits + list_id) * a.kp;
        const uint64_t* warp_buf = buf + ((size_t)half * TC_M + quarter * 32) * TC_BUFCAP;
        if constexpr (!TILE_MIN) {  // (tile-min mode writes one dense entry per tile half; the caller pre-fills the padding)
            for (int r = 0; r < 32; ++r) {
                if (q0 + quarter * 32 + r >= a.nq) break;
                uint64_t* list = warp_lists + (size_t)r * list_stride;
                for (uint32_t i = lane; i < a.kp; i += 32) list[i] = kInvalidPacked;
            }
            __syncwarp();
        }
        float thr = q_valid ? (a.thr_init != nullptr ? a.thr_init[q] : __int_as_float(0x7F800000)) : __int_as_float(0xFF800000);
        int cnt = 0;
        const uint32_t* deny = a.deny;
        // this thread's query row is tested against its own bitmap
        const uint32_t* allow = a.allow != nullptr && q_valid ? query_allow(a.allow, a.allow_bits, a.allow_of_q, q) : a.allow;
        const uint64_t* keys = a.keys;
        const uint64_t allow_bits = a.allow_bits;

        for (uint32_t t = 0; t < n_tiles; ++t) {
            const uint32_t acc = t & 1, acc_phase = (t >> 1) & 1;
            const uint32_t n0 = r_lo + t * a.tile_step + half * TC_HALF_N;   // first corpus row of this warp's columns
            float best_d = __int_as_float(0x7F800000);
            uint32_t best_c = kInvalidSlot;
            // per-column parameter of this tile (NaN marks columns outside the split); every epilogue warp keeps
            // its own copy so the warps never wait for each other
            float* cp = colp + ((warp - 2) * 2 + acc) * TC_HALF_N;
            for (int c = lane; c < TC_HALF_N; c += 32) {
                const uint32_t n = n0 + c;
                float pv = __int_as_float(0x7FC00000);
                if (n < r_hi) {
                    if constexpr (METRIC == VSB_METRIC_L2SQ) pv = a.x_sq[n];
                    else if constexpr (METRIC == VSB_METRIC_COS) {
                        const float xn = a.x_nrm[n];
                        pv = xn > 0.f ? 1.0f / xn : 0.f;
                    } else pv = 1.0f;
                }
                cp[c] = pv;
            }
            __syncwarp();
            mbar_wait(&tmem_full[acc], acc_phase);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + acc * TC_N + half * TC_HALF_N;
#pragma unroll 1
            for (int ch = 0; ch < TC_HALF_N / 32; ++ch) {
                uint32_t v[32];
                tmem_ld32(taddr + ch * 32, v);
                const float4* cp4 = reinterpret_cast<const float4*>(cp + ch * 32);
                if constexpr (TILE_MIN) {
                    float d[32];
                    float dmin = __int_as_float(0x7F800000);
#pragma unroll
                    for (int j4 = 0; j4 < 8; ++j4) {
                        const float4 p4 = cp4[j4];
                        const float pj[4] = {p4.x, p4.y, p4.z, p4.w};
#pragma unroll
                        for (int jj = 0; jj < 4; ++jj) {
                            const int j = j4 * 4 + jj;
                            d[j] = tc_dist<METRIC>(__uint_as_float(v[j]), pj[jj], qpar);
                            dmin = fminf(dmin, d[j]);  // NaN (masked column) never wins
                        }
                    }
                    if (dmin < best_d) {
#pragma unroll
                        for (int j = 31; j >= 0; --j)
                            if (d[j] == dmin) best_c = (uint32_t)(ch * 32 + j);
                        best_d = dmin;
                    }
                } else {
                    // bit j = column j of this chunk beats (or ties) the row's k'-th best; NaN never does
                    uint32_t hit = 0;
#pragma unroll
                    for (int j4 = 0; j4 < 8; ++j4) {
                        const float4 p4 = cp4[j4];
                        const float pj[4] = {p4.x, p4.y, p4.z, p4.w};
#pragma unroll
                        for (int jj = 0; jj < 4; ++jj) {
                            const int j = j4 * 4 + jj;
                            if (tc_dist<METRIC>(__uint_as_float(v[j]), pj[jj], qpar) <= thr) hit |= 1u << j;
                        }
                    }
                    // The columns in which ANY row of the warp hit, one at a time (warp-uniform loop): the dot product
                    // comes back from TMEM with a one-column load (registers cannot be indexed by a run-time j), the
                    // same tc_dist gives the same bits, and only the rows that hit append.  With warmed-up lists
                    // the loop body runs for well under one column per chunk (exact search) to a few (the build's
                    // all-pairs lists, k' = 96 over 131 072 rows).
                    uint32_t any_hit = __reduce_or_sync(kFullMask, hit);
                    while (any_hit != 0) {
                        // up to four hit columns per round trip to TMEM: four one-column loads, ONE wait
                        int jj[4];
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            jj[u] = any_hit != 0 ? __ffs(any_hit) - 1 : -1;
                            any_hit &= any_hit - 1;  // 0 stays 0
                        }
                        uint32_t dv[4];
#pragma unroll
                        for (int u = 0; u < 4; ++u) dv[u] = tmem_ld1_nowait(taddr + ch * 32 + (jj[u] >= 0 ? jj[u] : jj[0]));
                        tmem_wait_ld4(dv[0], dv[1], dv[2], dv[3]);
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            if (jj[u] < 0) break;  // warp-uniform
                            const int j = jj[u];
                            if ((hit >> j) & 1u) {
                                const uint32_t n = n0 + ch * 32 + j;
                                bool ok = true;
                                if (deny != nullptr && bit_test(deny, n)) ok = false;
                                if (ok && allow != nullptr) {
                                    const uint64_t rid = keys[n] & kRowMask48;
                                    ok = rid < allow_bits && bit_test(allow, (uint32_t)rid);
                                }
                                if (ok) {
                                    float dd = tc_dist<METRIC>(__uint_as_float(dv[u]), cp[ch * 32 + j], qpar);
                                    if constexpr (METRIC == VSB_METRIC_L2SQ) dd = fmaxf(dd, 0.0f);
                                    if constexpr (METRIC == VSB_METRIC_COS) dd = fminf(fmaxf(dd, 0.0f), 2.0f);
                                    my_buf[cnt++] = pack_ds(dd, n);
                                }
                            }
                            const uint32_t full_rows = __ballot_sync(kFullMask, cnt == TC_BUFCAP);
                            if (full_rows != 0) {
                                thr = tc_flush_rows(full_rows, warp_lists, list_stride, a.kp, keys, warp_buf, cnt, thr, lane);
                                if ((full_rows >> lane) & 1u) cnt = 0;
                            }
                        }
                    }
                }
            }
            if constexpr (TILE_MIN) {
                if (q_valid) {
                    // dense layout: K4 sorts ceil(2 * tiles / 32) blocks of 32 entries per query, however the rows
                    // were split over CTAs
                    if constexpr (METRIC == VSB_METRIC_L2SQ) best_d = fmaxf(best_d, 0.0f);
                    if constexpr (METRIC == VSB_METRIC_COS) best_d = fminf(fmaxf(best_d, 0.0f), 2.0f);
                    const uint32_t gt = split * (a.rows_per_split / TC_N) + t;
                    a.part[(size_t)q * a.tile_min_stride + gt * TC_HALVES + half] =
                        best_c != kInvalidSlot ? pack_ds(best_d, n0 + best_c) : kInvalidPacked;
                }
            }
            // accumulator drained: hand the TMEM buffer back to the MMA warp
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                if (CTA2 && !leader) mbar_arrive_remote(&tmem_empty[acc], 0);
                else mbar_arrive(&tmem_empty[acc]);
            }
        }
        if constexpr (!TILE_MIN) {
            const uint32_t rest = __ballot_sync(kFullMask, cnt > 0);
            if (rest) tc_flush_rows(rest, warp_lists, list_stride, a.kp, keys, warp_buf, cnt, thr, lane);
        }
    }

    tc_fence_before();
    if constexpr (CTA2) cluster_sync_all(); else __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        if constexpr (CTA2)
            asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u));
        else
            asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u));
    }
}

// Sampled thresholds for long lists over few rows (the build's all-pairs kNN lists: k' = 96 over 131 072 rows cost
// ~1 450 list insertions per row if every list starts empty).  A first pass lists the 32 best rows of a tile-strided
// SAMPLE per query; the m-th best of the sample, m ~ 3 * k' * sample / rows, bounds the k'-th best of all rows with
// room to spare, and the main pass starts every list at that bound: ~3 k' candidates per row instead of ~15 k'.
// One warp per query: merge the two column-half lists of the sample pass, take rank m - 1.
__global__ void __launch_bounds__(256) tc_sample_threshold_kernel(const uint64_t* __restrict__ part, uint32_t nq, uint32_t m,
                                                                  float* __restrict__ thr) {
    const int lane = threadIdx.x & 31;
    const uint32_t q = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (q >= nq) return;
    const LessBySlot less;
    const uint64_t a0 = part[((size_t)q * TC_HALVES + 0) * 32 + lane];        // ascending
    const uint64_t b0 = part[((size_t)q * TC_HALVES + 1) * 32 + (31 - lane)];  // descending
    uint64_t v = b0 < a0 ? b0 : a0;  // bitonic: the 32 smallest of the 64
    v = warp_bitonic_merge32(v, lane, less);
    const uint64_t pick = shfl_u64(v, (int)m - 1);
    if (lane == 0) thr[q] = pick == kInvalidPacked ? __int_as_float(0x7F800000) : ord_to_f32(packed_hi(pick));
}

// queries whose lists of the thresholded pass hold fewer than `need` rows in total (the bound was too tight for them)
__global__ void __launch_bounds__(256) tc_count_short_kernel(const uint64_t* __restrict__ part, uint32_t nq, uint32_t lists,
                                                             uint32_t kp, uint32_t need, uint32_t* __restrict__ counter) {
    const int lane = threadIdx.x & 31;
    const uint32_t q = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (q >= nq) return;
    uint32_t have = 0;
    for (uint32_t i = lane; i < lists * kp; i += 32) have += part[(size_t)q * lists * kp + i] != kInvalidPacked ? 1u : 0u;
    have = (uint32_t)butterfly_sum_i((int)have);
    if (lane == 0 && have < need) atomicAdd(counter, 1u);
}

// ---- host side ---------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (fn == nullptr) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

bool make_map(CUtensorMap* map, int kind, const void* base, uint32_t rows, uint32_t row_bytes, uint32_t box_rows) {
    EncodeTiledFn fn = get_encode_fn();
    if (fn == nullptr || rows == 0) return false;
    const uint32_t esz = kind == KIND_TF32 ? 4 : 2;
    const CUtensorMapDataType dt = kind == KIND_TF32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                                   : kind == KIND_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16
                                                       : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
    cuuint64_t dims[2] = {row_bytes / esz, rows};
    cuuint64_t strides[1] = {row_bytes};
    cuuint32_t box[2] = {TC_KBYTES / esz, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, dt, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS;
}

template <int KIND, int METRIC, bool TILE_MIN, bool CTA2>
void launch_tc_one(const CUtensorMap& mq, const CUtensorMap& mx, const TcArgs& a, dim3 grid, cudaStream_t stream) {
    auto kern = exact_candidates_tc_kernel<KIND, METRIC, TILE_MIN, CTA2>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TC_SMEM_BYTES);
    if constexpr (CTA2) {
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = grid;
        cfg.blockDim = dim3(TC_THREADS);
        cfg.dynamicSmemBytes = TC_SMEM_BYTES;
        cfg.stream = stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = 2;
        attr[0].val.clusterDim.y = 1;
        attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        cudaLaunchKernelEx(&cfg, kern, mq, mx, a);
    } else {
        kern<<<grid, TC_THREADS, TC_SMEM_BYTES, stream>>>(mq, mx, a);
    }
}

template <int KIND, int METRIC>
void launch_tc_inst(const CUtensorMap& mq, const CUtensorMap& mx, const TcArgs& a, dim3 grid, cudaStream_t stream,
                    bool cta2) {
    if (a.tile_min) {
        launch_tc_one<KIND, METRIC, true, false>(mq, mx, a, grid, stream);  // the seed layer is tiny: 1-CTA form
    } else if (cta2) {
        launch_tc_one<KIND, METRIC, false, true>(mq, mx, a, grid, stream);
    } else {
        launch_tc_one<KIND, METRIC, false, false>(mq, mx, a, grid, stream);
    }
}

template <int KIND>
void launch_tc_kind(int metric, const CUtensorMap& mq, const CUtensorMap& mx, const TcArgs& a, dim3 grid,
                    cudaStream_t stream, bool cta2) {
    switch (metric) {
        case VSB_METRIC_L2SQ: launch_tc_inst<KIND, VSB_METRIC_L2SQ>(mq, mx, a, grid, stream, cta2); break;
        case VSB_METRIC_COS: launch_tc_inst<KIND, VSB_METRIC_COS>(mq, mx, a, grid, stream, cta2); break;
        default: launch_tc_inst<KIND, VSB_METRIC_IP>(mq, mx, a, grid, stream, cta2); break;
    }
}

}  // namespace

// cta_group::2 form of the list-maintaining kernel (VSB_TC_2CTA=0/1); the seed layer's tile-min kernel is always 1-CTA
static bool tc_use_cta_pairs() {
    static const bool on = [] {
        const char* e = getenv("VSB_TC_2CTA");
        return e != nullptr ? e[0] == '1' : true;  // default on: 1 046 vs 964 TFLOP/s on 10 000 x 1 M x 768 bf16
    }();
    return on;
}

bool exact_tc_supported(int storage, int metric) {
    if (metric == VSB_METRIC_HAMMING) return false;
    return storage == VSB_ST_F32 || storage == VSB_ST_BF16 || storage == VSB_ST_F16;
}

// tile-min mode: entries per query of the dense winner array (one per tile half, padded to whole blocks of 32)
uint32_t exact_tc_tile_min_entries(uint32_t n_rows) {
    const uint32_t tiles = (n_rows + TC_N - 1) / TC_N;
    return (tiles * TC_HALVES + 31) / 32 * 32;
}

// Returns the number of candidate LISTS per query (what ExactParams::n_splits means to K3 and to the part buffer):
// TC_HALVES lists — one per epilogue column half — for each row split of the corpus.
uint32_t exact_tc_pick_splits(uint32_t nq, uint32_t n_rows, int sm_count, uint32_t kp) {
    // One CTA per SM: the sweep takes ceil(q_tiles * s / SMs) waves of 1/s of the corpus each.  Pick the row-split
    // count s that minimises waves / s, i.e. fills the last wave (79 query tiles x 1 split would leave 69 of 148 SMs
    // idle; x 13 splits = 1027 CTAs = 6.94 waves) — weighed against the list work it adds: every list warms up on
    // its own (~ kp * (1 + ln(rows_per_list / kp)) insertions, each worth ~200 scanned elements of epilogue time —
    // calibrated on 10 000 x 1 M x 768: 19.7 ms at weight 10, 15.6 ms at 100..300, 19.4 ms at 1000) and K3
    // merges them all.  Short lists over many rows (exact search) split freely; the build's all-pairs lists
    // (k' = 96 over 131 072 rows) stay at one split.  kp = 0: tile-min mode, no lists.  CTAs of one wave walk the
    // same row split in step, so the corpus stream stays L2-resident however many splits there are.
    uint32_t q_tiles = (nq + TC_M - 1) / TC_M;
    if (kp != 0 && tc_use_cta_pairs()) q_tiles = (q_tiles + 1) & ~1u;  // CTA pairs: an odd tail tile gets a partner
    const uint32_t min_tiles = kp == 0 ? 2 : 8;
    uint32_t max_by_rows = n_rows / (min_tiles * TC_N);
    if (max_by_rows < 1) max_by_rows = 1;
    const uint32_t s_max = max_by_rows < 64 ? max_by_rows : 64;
    static const double insert_cost = [] {
        const char* e = getenv("VSB_TC_SPLIT_PENALTY");
        return e ? atof(e) : 200.0;
    }();
    uint32_t best = 1;
    double best_cost = 1e30;
    for (uint32_t s = 1; s <= s_max; ++s) {
        const uint32_t ctas = q_tiles * s;
        const uint32_t waves = (ctas + (uint32_t)sm_count - 1) / (uint32_t)sm_count;
        const double lists = (double)TC_HALVES * s;
        const double per_list = (double)n_rows / lists;
        const double inserts = kp == 0 ? 1.0 : (double)kp * (1.0 + std::log(std::max(1.0, per_list / kp)));
        const double cost = (double)waves / s * (1.0 + insert_cost * lists * inserts / (double)n_rows);
        if (cost < best_cost - 1e-12) {
            best_cost = cost;
            best = s;
        }
    }
    return TC_HALVES * best;
}

// Same contract as launch_exact_candidates (exact.cu); returns false if the TMA descriptors could
// not be encoded (caller falls back to the SIMT K1, which is still the CUDA path).
bool launch_exact_candidates_tc(const ExactParams& p, cudaStream_t stream, bool tile_min) {
    if (p.q.n == 0 || p.x_hi <= p.x_lo) return true;
    const int kind = p.storage == VSB_ST_F32 ? KIND_TF32 : (p.storage == VSB_ST_BF16 ? KIND_BF16 : KIND_F16);
    const bool cta2 = tc_use_cta_pairs() && !tile_min;
    CUtensorMap mq, mx;
    if (!make_map(&mq, kind, p.q.rows, p.q.n, p.q.row_bytes, TC_M)) return false;
    if (!make_map(&mx, kind, p.x.rows, p.x_hi, p.x.row_bytes, cta2 ? TC_N / 2 : TC_N)) return false;
    TcArgs a;
    a.q_sq = p.q.sq; a.q_nrm = p.q.nrm; a.nq = p.q.n;
    a.x_sq = p.x.sq; a.x_nrm = p.x.nrm; a.x_lo = p.x_lo; a.x_hi = p.x_hi; a.row_bytes = p.x.row_bytes;
    a.deny = p.deny; a.keys = p.keys; a.allow = p.allow; a.allow_bits = p.allow_bits; a.allow_of_q = p.allow_of_q;
    a.kp = p.kp; a.n_splits = p.n_splits;
    if (p.n_splits % TC_HALVES != 0) return false;  // callers size the lists with exact_tc_pick_splits
    const uint32_t row_splits = p.n_splits / TC_HALVES;
    const uint32_t rows = p.x_hi - p.x_lo;
    const uint32_t rps = (rows + row_splits - 1) / row_splits;
    a.rows_per_split = ((rps + TC_N - 1) / TC_N) * TC_N;
    a.part = p.part;
    a.tile_min = tile_min ? 1 : 0;
    a.tile_min_stride = exact_tc_tile_min_entries(p.x_hi - p.x_lo);
    a.tile_step = (!tile_min && p.tile_step >= (uint32_t)TC_N) ? p.tile_step / TC_N * TC_N : (uint32_t)TC_N;
    a.max_tiles = tile_min ? 0u : p.max_tiles;
    a.thr_init = tile_min ? nullptr : p.thr_init;
    uint32_t q_tiles = (p.q.n + TC_M - 1) / TC_M;
    if (cta2) q_tiles = (q_tiles + 1) & ~1u;  // CTA pairs: an odd tail tile gets an all-padding partner
    dim3 grid(q_tiles, row_splits);
    switch (kind) {
        case KIND_BF16: launch_tc_kind<KIND_BF16>(p.metric, mq, mx, a, grid, stream, cta2); break;
        case KIND_F16: launch_tc_kind<KIND_F16>(p.metric, mq, mx, a, grid, stream, cta2); break;
        default: launch_tc_kind<KIND_TF32>(p.metric, mq, mx, a, grid, stream, cta2); break;
    }
    g_kernel_launches += 1;
    g_tc_launches += 1;
    return true;
}

void launch_tc_sample_threshold(const uint64_t* sample_part, uint32_t nq, uint32_t m, float* thr, cudaStream_t stream) {
    if (nq == 0) return;
    tc_sample_threshold_kernel<<<(nq + 7) / 8, 256, 0, stream>>>(sample_part, nq, m < 1 ? 1 : (m > 32 ? 32 : m), thr);
    g_kernel_launches += 1;
}

void launch_tc_count_short(const uint64_t* part, uint32_t nq, uint32_t lists, uint32_t kp, uint32_t need, uint32_t* counter,
                           cudaStream_t stream) {
    if (nq == 0) return;
    tc_count_short_kernel<<<(nq + 7) / 8, 256, 0, stream>>>(part, nq, lists, kp, need, counter);
    g_kernel_launches += 1;
}

uint32_t exact_tc_halves() { return TC_HALVES; }

}  // namespace vsb
