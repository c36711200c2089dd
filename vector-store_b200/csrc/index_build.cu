// index_build.cu — graph construction: bulk build (K5 + K6), streaming insert (K7), refinement, entry points.
// Replaces the HNSW insert inside usearch::Index::add (vs_index/usearch.rs:191-197).  Everything here runs under
// mut_mu on the mutator stream with the mutator scratch, reads and extends the working view `w`, and leaves the
// publication of the result to the entry point that called it (index.cu).
#include <algorithm>
#include <cmath>
#include <cstdlib>

#include <nvtx3/nvToolsExt.h>

#include "index_impl.h"

using vsbi::DevBuf;
using vsbi::fail;
using vsbi::round_up;

namespace {
// CUDA-event stopwatch on one stream; stop() synchronises on the end event only
struct EvTimer {
    cudaEvent_t a = nullptr, b = nullptr;
    cudaStream_t s;
    explicit EvTimer(cudaStream_t st) : s(st) {
        cudaEventCreate(&a);
        cudaEventCreate(&b);
        cudaEventRecord(a, s);
    }
    uint64_t stop() {
        cudaEventRecord(b, s);
        cudaEventSynchronize(b);
        float ms = 0.f;
        cudaEventElapsedTime(&ms, a, b);
        return (uint64_t)((double)ms * 1e6);
    }
    ~EvTimer() {
        cudaEventDestroy(a);
        cudaEventDestroy(b);
    }
};
}  // namespace

vsb_status vsb_index::build() {
    CU(cudaSetDevice(device));
    bstats = vsb_build_stats{};
    if (w.any_tombstone) ST(compact(false));
    struct Flag {
        bool& f;
        explicit Flag(bool& r) : f(r) { f = true; }
        ~Flag() { f = false; }
    } building(in_build);
    churn_since_refine = 0;
    bstats.rows = w.n_slots;
    bstats.traversal_row_bytes = trav16 ? row_bytes16 : row_bytes;
    if (live < min_graph_size || !vsb::graph_search_supported(row_bytes)) {
        w.n_graphed = 0;
        w.gr.reset();
        w.sd.reset();
        return VSB_OK;
    }
    // The graph is built beside the published one: searches keep using the old graph until vsb_build publishes.
    w.n_graphed = 0;
    w.gr.reset();
    w.sd.reset();
    const uint32_t n_slots = w.n_slots;
    // All-pairs kNN lists cost 2*n^2*D flop: above `allpairs_max` rows only the first `allpairs_prefix` rows are
    // built that way and the remaining rows are linked in with the streaming insert (K7, O(n log n)).
    const uint32_t n = n_slots <= allpairs_max ? n_slots : std::min<uint32_t>(n_slots, allpairs_prefix);
    const uint32_t kin = std::min<uint32_t>(k_init, 128);
    DevBuf knn;
    CU(knn.alloc((size_t)n * kin * 8));
    const vsb::RowsView x = rows_view(w);
    const vsbi::Store& st = *w.st;
    // f32 storage: the all-pairs candidate stage runs on a bf16 copy (kNN lists only need candidate-grade
    // distances; K3 re-evaluates the survivors on the f32 rows in the canonical order)
    DevBuf sh_rows, sh_sq, sh_nrm;
    vsb::RowsView shx;
    const bool use_shadow = storage == VSB_F32 && tc_enabled && n >= tc_min_rows;
    if (use_shadow) {
        if (trav16) {  // the traversal copy IS that shadow
            shx.rows = st.rows16.as<uint8_t>();
            shx.sq = st.sq16.as<float>();
            shx.nrm = st.nrm16.as<float>();
            shx.row_bytes = row_bytes16;
            shx.n = n;
        } else {
            const uint32_t dim_pad = row_bytes / 4;
            shx.row_bytes = ((dim_pad * 2 + 15) / 16) * 16;
            shx.n = n;
            CU(sh_rows.alloc((size_t)n * shx.row_bytes));
            CU(sh_sq.alloc((size_t)n * 4));
            CU(sh_nrm.alloc((size_t)n * 4));
            vsb::launch_convert_rows(VSB_BF16, reinterpret_cast<const float*>(x.rows), n, dim_pad, sh_rows.as<uint8_t>(),
                                     shx.row_bytes, sh_sq.as<float>(), sh_nrm.as<float>(), mstream);
            CU(cudaGetLastError());
            shx.rows = sh_rows.as<uint8_t>();
            shx.sq = sh_sq.as<float>();
            shx.nrm = sh_nrm.as<float>();
        }
    }
    {
        nvtxRangePushA("build.allpairs");
        EvTimer t(mstream);
        // query blocks of one 128-row tensor-core tile per SM: a block is exactly one wave of K1-TC CTAs
        const uint32_t QB = std::max<uint32_t>(16384, (uint32_t)sm_count * 128);
        for (uint32_t b0 = 0; b0 < n; b0 += QB) {
            vsb::RowsView q;
            q.n = std::min(QB, n - b0);
            q.rows = x.rows + (size_t)b0 * row_bytes;
            q.sq = x.sq + b0;
            q.nrm = x.nrm + b0;
            q.row_bytes = row_bytes;
            vsb::RowsView shq = shx;
            if (use_shadow) {
                shq.n = q.n;
                shq.rows = shx.rows + (size_t)b0 * shx.row_bytes;
                shq.sq = shx.sq + b0;
                shq.nrm = shx.nrm + b0;
            }
            ST(exact_block(w, ms, q, x, 0, n, nullptr, st.keys.as<uint64_t>(), nullptr, 0, nullptr, kin, nullptr, nullptr, nullptr,
                           knn.as<uint64_t>() + (size_t)b0 * kin, (int64_t)b0, mstream, true, use_shadow ? &shq : nullptr,
                           use_shadow ? &shx : nullptr));
        }
        bstats.allpairs_ns = t.stop();
        bstats.allpairs_rows = n;
        bstats.allpairs_flops = 2ull * n * n * dim;
        nvtxRangePop();
    }
    sh_rows.release();
    sh_sq.release();
    sh_nrm.release();
    ST(graph_from_knn(knn.as<uint64_t>(), n, kin, nullptr));
    knn.release();
    // the reachability pass (extra seeds for lost components) runs on the FINAL graph only
    ST(sample_seeds(n, n >= n_slots));
    if (n < n_slots) {
        // large index: link the remaining rows with the streaming insert (K7), then rebuild every row's
        // list from an ANN search over that navigable graph and prune it exactly like the all-pairs lists
        ST(stream_insert());
        ST(sample_seeds(n_slots, refine_passes == 0));  // entry points drawn from every row, not only the all-pairs prefix
        for (uint32_t pass = 0; pass < refine_passes; ++pass) {
            ST(refine_graph());
            ST(sample_seeds(n_slots, pass + 1 == refine_passes));
        }
    }
    return VSB_OK;
}

// K6 pipeline: packed kNN lists [n][kin] -> fixed-degree graph rows (a NEW graph buffer, n_graphed = n)
vsb_status vsb_index::graph_from_knn(const uint64_t* knn, uint32_t n, uint32_t kin, const uint32_t* deny_bm) {
    nvtxRangePushA("build.prune");
    EvTimer t(mstream);
    const uint32_t R = degree;
    DevBuf fwd, rev, rev_cnt, scratch;
    CU(fwd.alloc((size_t)n * R * 4));
    CU(rev.alloc((size_t)n * R * 4));
    CU(rev_cnt.alloc((size_t)n * 4));
    vsb::launch_prune_detour(knn, n, kin, R, deny_bm, fwd.as<uint32_t>(), mstream);
    CU(cudaGetLastError());
    const size_t sb = vsb::reverse_edges_scratch_bytes(n, R);
    CU(scratch.alloc(sb));
    vsb::launch_reverse_edges(fwd.as<uint32_t>(), n, R, rev.as<uint32_t>(), rev_cnt.as<uint32_t>(), scratch.p,
                              scratch.bytes, mstream);
    CU(cudaGetLastError());
    auto ng = std::make_shared<vsbi::Graph>();
    ng->cap_rows = std::max<uint64_t>(w.st->capacity, n);  // room for streamed rows
    CU(ng->g.alloc((size_t)ng->cap_rows * graph_stride * 4));
    vsb::launch_merge_graph(fwd.as<uint32_t>(), rev.as<uint32_t>(), rev_cnt.as<uint32_t>(), n, R, ng->g.as<uint32_t>(),
                            graph_stride, mstream);
    CU(cudaGetLastError());
    bstats.prune_ns += t.stop();
    w.gr = ng;
    w.n_graphed = n;
    nvtxRangePop();
    return VSB_OK;
}

// One refinement pass over a complete (streamed) graph: every row searches the graph for its own
// k_init nearest rows (K4, beam = expansion_add) and the lists go through the K6 pipeline again.
vsb_status vsb_index::refine_graph() {
    if (w.n_graphed == 0) return VSB_OK;
    // rows are cheap to move on this machine: drop the tombstoned ones first, so the new lists never hold them
    if (n_tombstones * 20 >= w.n_slots && n_tombstones > 0) ST(compact(true));
    const uint32_t n = w.n_graphed;
    if (n == 0) return VSB_OK;
    nvtxRangePushA("build.refine");
    const uint32_t kin = std::min<uint32_t>(k_init, 128);
    const uint32_t ef_add = ef_add_rt ? ef_add_rt : (opt.expansion_add ? opt.expansion_add : 128);
    const uint32_t ef = std::min<uint32_t>(round_up(std::max(ef_add, kin + 1), 32), 512);
    const vsbi::Store& st = *w.st;
    const uint32_t* deny_bm = w.any_tombstone ? st.deny.as<uint32_t>() : nullptr;
    DevBuf knn;
    CU(knn.alloc((size_t)n * kin * 8));
    GraphRun run;
    run.itopk = ef;
    run.max_iters = 0;
    run.n_seeds = 32;
    run.search_width = build_search_width;  // 2 parents per iteration: ~10 % more evaluations, but twice the rows in flight per warp
    {
        EvTimer t(mstream);
        const uint32_t QB = 16384;
        for (uint32_t b0 = 0; b0 < n; b0 += QB) {
            const uint32_t nb = std::min(QB, n - b0);
            vsb::RowsView qv;
            qv.rows = st.rows.as<uint8_t>() + (size_t)b0 * row_bytes;
            qv.sq = st.sq.as<float>() + b0;
            qv.nrm = st.nrm.as<float>() + b0;
            qv.row_bytes = row_bytes;
            qv.n = nb;
            vsb::RowsView q16;
            if (trav16) {
                q16.rows = st.rows16.as<uint8_t>() + (size_t)b0 * row_bytes16;
                q16.sq = st.sq16.as<float>() + b0;
                q16.nrm = st.nrm16.as<float>() + b0;
                q16.row_bytes = row_bytes16;
                q16.n = nb;
            }
            ST(graph_block(w, ms, run, qv, nb, kin, nullptr, nullptr, nullptr, knn.as<uint64_t>() + (size_t)b0 * kin,
                           trav16 ? &q16 : nullptr, mstream, (long long)b0, false, &bstats.refine_evals,
                           &bstats.refine_parents));
        }
        bstats.refine_ns += t.stop();
        bstats.refine_rows += n;
    }
    ST(graph_from_knn(knn.as<uint64_t>(), n, kin, deny_bm));
    nvtxRangePop();
    return VSB_OK;
}

// Entry-point sample ("upper layer"): a stride permutation of the live slots below n_rows
// (deterministic, seed-shifted), gathered into a contiguous block (+ bf16 shadow for f32 storage).
vsb_status vsb_index::sample_seeds(uint32_t n, bool ensure_reach) {
    nvtxRangePushA("build.seeds");
    EvTimer t(mstream);
    const vsb::RowsView x = rows_view(w);
    const vsbi::Store& st = *w.st;
    uint64_t live_below = 0;
    for (uint32_t wd = 0; wd < (n + 31) / 32; ++wd) live_below += __builtin_popcount(~h_deny[wd]);
    if (n % 32) live_below -= 32 - (n % 32);
    // S = 4 * sqrt(live rows), in whole 256-row tensor-core tiles, at most 8192: the seed GEMM costs Q * S * D flop per
    // batch whatever the shard size, so a shard of n/G rows gets a sample (and a seed-layer time) ~1/sqrt(G) as large
    // The cap keeps the seed GEMM at the cost of 8192 rows of 768 dimensions: short rows get proportionally more
    // entry points (C4's 125 M x 128 shards: 4 * sqrt(n) = 44 800 seeds — with 8192 most of its 64 000 clusters had no
    // entry point and recall@10 stalled at 0.946 for ef = 512).
    const double target = 4.0 * std::sqrt((double)live_below);
    const uint32_t seed_cap = std::min<uint32_t>(65536, 8192u * std::max<uint32_t>(1, 768u / std::max<uint32_t>(dim, 1)));
    uint32_t S = std::min<uint32_t>(seed_cap, std::max<uint32_t>(256, round_up((uint32_t)std::ceil(target), 256)));
    if (S > live_below / 4) S = (uint32_t)std::max<uint64_t>(32, live_below / 4);
    std::vector<uint32_t> h_seeds;
    h_seeds.reserve(S);
    {
        uint64_t step = (uint64_t)((double)n * 0.6180339887498949) | 1ull;
        auto gcd = [](uint64_t a, uint64_t b) { while (b) { uint64_t r = a % b; a = b; b = r; } return a; };
        while (gcd(step, n) != 1) step += 2;
        uint64_t pos = opt.seed % n;
        for (uint32_t i = 0; i < n && h_seeds.size() < S; ++i) {
            const uint32_t slot = (uint32_t)pos;
            pos = (pos + step) % n;
            if (h_deny[slot >> 5] >> (slot & 31) & 1u) continue;
            h_seeds.push_back(slot);
        }
    }
    S = (uint32_t)h_seeds.size();
    auto sd = std::make_shared<vsbi::Seeds>();
    // every live graph node must be reachable from the seed set: expand the frontier from the sample to a fixed
    // point, then promote the first unreached live node to an extra seed and continue, once per lost component
    uint32_t extra_seeds = 0;
    if (w.n_graphed >= n && n > 0 && S > 0 && reach_fix && ensure_reach) {
        DevBuf reach_state;
        const size_t flag_off = ((size_t)n + 16 + 15) / 16 * 16;  // the state array is readable 16 bytes past n
        constexpr uint32_t kPromote = 64;                          // unreached nodes promoted per round
        CU(reach_state.alloc(flag_off + 16 + (size_t)(1 + kPromote) * 4));
        uint8_t* state = reach_state.as<uint8_t>();
        uint32_t* flag = reinterpret_cast<uint32_t*>(state + flag_off);  // [0] changed
        uint32_t* found = flag + 4;                                      // [0] count, [1..] slots
        CU(sd->slots.alloc((size_t)(S + reach_budget) * 4));
        CU(cudaMemsetAsync(state, 0, flag_off, mstream));
        CU(cudaMemcpyAsync(sd->slots.p, h_seeds.data(), (size_t)S * 4, cudaMemcpyHostToDevice, mstream));
        vsb::launch_reach_mark(state, sd->slots.as<uint32_t>(), S, mstream);
        const uint32_t* deny_bm = w.any_tombstone ? st.deny.as<uint32_t>() : nullptr;
        auto expand = [&]() -> vsb_status {
            for (int round = 0; round < 4096; ++round) {
                CU(cudaMemsetAsync(flag, 0, 4, mstream));
                for (int i = 0; i < 4; ++i)
                    vsb::launch_reach_step(w.gr->g.as<uint32_t>(), n, graph_stride, degree, state, flag, mstream);
                uint32_t changed = 0;
                vsbi::HostReadback rb(ms.pin, mstream);
                CU(rb.reserve(4));
                CU(rb.copy(&changed, flag, 4));
                CU(rb.finish());
                if (!changed) break;
            }
            return VSB_OK;
        };
        ST(expand());
        // unreached live nodes become extra seeds, up to kPromote of them (in slot order) per round: a lost component
        // usually is a single node nobody links to, so promoting a batch and expanding once beats one round per node
        std::vector<uint32_t> h_found(1 + kPromote);
        while (extra_seeds < reach_budget) {
            const uint32_t room = std::min<uint32_t>(kPromote, reach_budget - extra_seeds);
            vsb::launch_collect_unreached(state, deny_bm, n, room, found, mstream);
            {
                vsbi::HostReadback rb(ms.pin, mstream);
                CU(rb.reserve((size_t)(1 + room) * 4));
                CU(rb.copy(h_found.data(), found, (size_t)(1 + room) * 4));
                CU(rb.finish());
            }
            const uint32_t cnt = std::min(h_found[0], room);
            if (cnt == 0) break;
            for (uint32_t i = 0; i < cnt; ++i) h_seeds.push_back(h_found[1 + i]);
            vsb::launch_reach_mark(state, found + 1, cnt, mstream);
            extra_seeds += cnt;
            ST(expand());
        }
        CU(cudaGetLastError());
        S = (uint32_t)h_seeds.size();
    } else {
        CU(sd->slots.alloc((size_t)std::max<uint32_t>(S, 1) * 4));
    }
    sd->extra = extra_seeds;
    CU(sd->rows.alloc((size_t)S * row_bytes));
    CU(sd->sq.alloc((size_t)S * 4));
    CU(sd->nrm.alloc((size_t)S * 4));
    CU(cudaMemcpyAsync(sd->slots.p, h_seeds.data(), (size_t)S * 4, cudaMemcpyHostToDevice, mstream));
    vsb::launch_gather_rows(x.rows, row_bytes, x.sq, x.nrm, sd->slots.as<uint32_t>(), S, sd->rows.as<uint8_t>(),
                            sd->sq.as<float>(), sd->nrm.as<float>(), mstream);
    CU(cudaGetLastError());
    if (storage == VSB_F32) {
        const uint32_t dim_pad = row_bytes / 4;
        const uint32_t rb16 = ((dim_pad * 2 + 15) / 16) * 16;
        CU(sd->rows16.alloc((size_t)S * rb16));
        CU(sd->sq16.alloc((size_t)S * 4));
        CU(sd->nrm16.alloc((size_t)S * 4));
        vsb::launch_convert_rows(VSB_BF16, sd->rows.as<float>(), S, dim_pad, sd->rows16.as<uint8_t>(), rb16,
                                 sd->sq16.as<float>(), sd->nrm16.as<float>(), mstream);
        CU(cudaGetLastError());
    }
    CU(cudaStreamSynchronize(mstream));
    sd->n = S;
    sd->sampled_rows = n;
    w.sd = sd;
    bstats.seeds_ns += t.stop();
    nvtxRangePop();
    return VSB_OK;
}

// K7: link every un-graphed tail row into the existing graph (batched HNSW-style insert: search with
// beam = expansion_add, choose R of the 2R closest by detour count over the graph rows of the candidates,
// then add reverse edges).  The graph buffer is extended IN PLACE: rows of the new nodes are complete before
// any reverse edge points at them (two kernels), and a reverse edge replaces one 32-bit word, so a search
// running on the published view of the same buffer always reads valid rows.
vsb_status vsb_index::stream_insert() {
    if (w.n_graphed == 0 || w.n_graphed >= w.n_slots) return VSB_OK;
    CU(cudaSetDevice(device));
    nvtxRangePushA("build.stream_insert");
    const vsbi::Store& st = *w.st;
    if (w.gr->cap_rows < st.capacity) {
        auto ng = std::make_shared<vsbi::Graph>();
        ng->cap_rows = st.capacity;
        CU(ng->g.alloc((size_t)st.capacity * graph_stride * 4));
        CU(cudaMemcpyAsync(ng->g.p, w.gr->g.p, (size_t)w.n_graphed * graph_stride * 4, cudaMemcpyDeviceToDevice, mstream));
        CU(cudaStreamSynchronize(mstream));
        w.gr = ng;
    }
    const uint32_t R = degree;
    const uint32_t ef_add = ef_add_rt ? ef_add_rt : (opt.expansion_add ? opt.expansion_add : 128);
    const uint32_t ef = std::min<uint32_t>(round_up(std::max(ef_add, R), 32), 512);
    const uint32_t C = std::min<uint32_t>(std::min<uint32_t>(ef, 2 * R), 128);  // candidates handed to the link stage
    GraphRun run;
    run.itopk = ef;
    run.max_iters = 0;
    run.n_seeds = 32;
    run.search_width = build_search_width;
    DevBuf cand, link_scratch;
    const uint32_t QB = 8192;
    CU(cand.alloc((size_t)QB * C * 8));
    const size_t link_bytes = vsb::stream_link_scratch_bytes(QB, R);
    CU(link_scratch.alloc(link_bytes));
    EvTimer t(mstream);
    while (w.n_graphed < w.n_slots) {
        // the entry points follow the graph: a sample drawn when the graph was half its size (at the start of a bulk
        // build: from the all-pairs prefix only) leaves the newer regions without a nearby seed
        if (w.sd && w.n_graphed >= 2 * std::max<uint32_t>(w.sd->sampled_rows, 1024)) ST(sample_seeds(w.n_graphed, false));
        const uint32_t t0 = w.n_graphed;
        const uint32_t nb = std::min(QB, w.n_slots - t0);
        vsb::RowsView qv;
        qv.rows = st.rows.as<uint8_t>() + (size_t)t0 * row_bytes;
        qv.sq = st.sq.as<float>() + t0;
        qv.nrm = st.nrm.as<float>() + t0;
        qv.row_bytes = row_bytes;
        qv.n = nb;
        vsb::RowsView q16;
        if (trav16) {
            q16.rows = st.rows16.as<uint8_t>() + (size_t)t0 * row_bytes16;
            q16.sq = st.sq16.as<float>() + t0;
            q16.nrm = st.nrm16.as<float>() + t0;
            q16.row_bytes = row_bytes16;
            q16.n = nb;
        }
        ST(graph_block(w, ms, run, qv, nb, C, nullptr, nullptr, nullptr, cand.as<uint64_t>(), trav16 ? &q16 : nullptr, mstream,
                       -1, false, &bstats.stream_evals, &bstats.stream_parents));
        CU(vsb::launch_stream_link(cand.as<uint64_t>(), nb, C, t0, R, w.gr->g.as<uint32_t>(), graph_stride, link_scratch.p,
                                   link_bytes, mstream));
        w.n_graphed = t0 + nb;  // later batches may link to these rows (stream order)
        churn_since_refine += nb;
        bstats.stream_rows += nb;
    }
    bstats.stream_ns += t.stop();
    nvtxRangePop();
    // Streamed links are a little worse than built ones and tombstoned rows keep occupying beam slots: once
    // 10 % of the graph has churned, one refinement pass (K4 kNN lists of every row -> K6) restores the
    // quality of a fresh build and drops the tombstoned rows from every list.  Searches are not held up:
    // the pass builds a new graph beside the published one.
    if (!in_build && churn_refine && churn_since_refine * 10 >= w.n_graphed && w.n_graphed >= min_graph_size) {
        publish();  // the streamed rows are navigable from here on
        ST(refine_graph());
        ST(sample_seeds(w.n_graphed));
        churn_since_refine = 0;
    }
    return VSB_OK;
}
