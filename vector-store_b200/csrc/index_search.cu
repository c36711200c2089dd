// index_search.cu — the search side of the index: exact blocks (K1 + K3 with the exactness certificate), graph
// blocks (seed layer + K4 [+ K3 re-rank]), and the two entry points (device pointers / host pointers).
// Replaces usearch::Index::search / filtered_search behind vs_index/usearch.rs:203-248.
#include <algorithm>
#include <chrono>
#include <cstring>

#include <nvtx3/nvToolsExt.h>

#include "index_impl.h"

using vsbi::DevBuf;
using vsbi::fail;
using vsbi::round_up;
using vsbi::Scratch;
using vsbi::TopK;
using vsbi::View;

// the filter of queries map[0..n) of a block: their bitmap indices gathered into `fidx`
static vsb_status gather_allow(const vsb::Allow& a, const uint32_t* map, uint32_t n, DevBuf& fidx, cudaStream_t s,
                               vsb::Allow& out) {
    out = a;
    if (a.of_q == nullptr) return VSB_OK;
    CU(fidx.ensure((size_t)n * 4));
    vsb::launch_gather_u32(a.of_q, map, n, fidx.as<uint32_t>(), s);
    out.of_q = fidx.as<uint32_t>();
    return VSB_OK;
}

vsb::ExactParams vsb_index::exact_in(const View& v, const vsb::RowsView& q, uint32_t x_lo, uint32_t x_hi,
                                     const vsb::Allow& allow) const {
    vsb::ExactParams p;
    p.storage = storage;
    p.metric = metric;
    p.q = q;
    p.x = v.st->rows.view(v.n_slots);
    p.x_lo = x_lo;
    p.x_hi = x_hi;
    p.deny = v.any_tombstone ? v.st->deny.as<uint32_t>() : nullptr;
    p.keys = v.st->keys.as<uint64_t>();
    p.allow = allow;
    return p;
}

// exact top-k of the queries in.q against rows [in.x_lo, in.x_hi) of in.x (K1 + K3)
vsb_status vsb_index::exact_block(Scratch& sc, const vsb::ExactParams& in, uint32_t k, const TopK& out, cudaStream_t s,
                                  bool approx_ok, const vsb::RowsView* shadow_q, const vsb::RowsView* shadow_x) {
    vsb::ExactParams p = in;
    const vsb::RowsView& q = in.q;
    const uint32_t x_lo = in.x_lo, x_hi = in.x_hi;
    const int64_t self_base = out.self_base;
    const uint32_t extra = std::max<uint32_t>(16, k / 4) + (self_base >= 0 ? 1 : 0);
    p.kp = round_up(k + extra, 32);
    if (p.kp > 256) return fail(VSB_EINVAL, "k=%u too large for the exact path (max 200)", k);
    // Tensor-core tiles: 16-bit storages multiply exactly, f32 rows run as TF32.  Any tiled stage (tensor core
    // or SIMT) sums in its own order, so its lists are candidate-grade; for exact results on float storages K3
    // CERTIFIES each query (no dropped row can reach or tie into the canonical top-k) and the queries it
    // cannot certify fall through: TF32 tiles -> fp32 SIMT tiles -> canonical scan (K1c, needs no certificate).
    // Integer storages (i8, b1) are exact in every stage and ordered by (distance, key) throughout.
    const bool tc_shape = tc_enabled && vsb::exact_tc_supported(storage, metric) && (x_hi - x_lo) >= tc_min_rows;
    const bool is_float = storage == VSB_F32 || storage == VSB_F16 || storage == VSB_BF16;
    const bool certify = is_float && !approx_ok && cert_enabled;
    bool tc = tc_shape && (approx_ok || storage != VSB_F32 || certify);
    const uint32_t kp_simt = p.kp;
    constexpr uint32_t kCertKp16 = 32;  // certified tensor-core list length of 16-bit rows (f32 rows: cert_kp)
    if (certify && tc) p.kp = std::min<uint32_t>(256, std::max<uint32_t>(p.kp, round_up(storage == VSB_F32 ? cert_kp : kCertKp16, 32)));
    p.n_splits = tc ? vsb::exact_tc_pick_splits(q.n, x_hi - x_lo, sm_count, p.kp)
                    : vsb::exact_pick_splits(q.n, x_hi - x_lo, sm_count);
    CU(sc.part.ensure(vsb::exact_part_elems(q.n, p.n_splits, p.kp) * 8));
    p.part = sc.part.as<uint64_t>();
    if (tc) {
        vsb::ExactParams pc = p;
        if (shadow_q != nullptr && shadow_x != nullptr && !certify) {
            // candidate stage on the bf16 shadow (half the bytes, kind::f16 rate); K3 re-ranks on the real rows
            pc.storage = VSB_BF16;
            pc.q = *shadow_q;
            pc.x = *shadow_x;
        }
        // Long lists over few rows (the all-pairs kNN lists of a build): bound every list by the m-th best row of a
        // tile-strided 8192-row sample first, so the main pass lists ~3 k' rows per query instead of ~15 k'.  The
        // bound is statistical: if more than 2 % of the queries end up with fewer than k rows the block is redone
        // without it (rows stored in the order of their clusters would do that).
        const uint32_t rows = x_hi - x_lo;
        const bool sampled = approx_ok && !certify && self_base >= 0 && rows >= 65536 && p.kp >= 64 &&
                             p.n_splits == vsb::exact_tc_halves() && p.allow.bm == nullptr;
        if (sampled) {
            const uint32_t sample_tiles = 32, halves = vsb::exact_tc_halves();
            vsb::ExactParams ps = pc;
            ps.kp = 32;
            ps.n_splits = halves;
            ps.tile_step = rows / 256 / sample_tiles * 256;
            ps.max_tiles = sample_tiles;
            CU(sc.thr_part.ensure((size_t)q.n * halves * 32 * 8));
            CU(sc.thr.ensure((size_t)q.n * 4));
            CU(sc.thr_cnt.ensure(16));
            ps.part = sc.thr_part.as<uint64_t>();
            tc = vsb::launch_exact_candidates_tc(ps, s);
            if (tc) {
                const double frac = (double)sample_tiles * 256.0 / (double)rows;
                const uint32_t m = (uint32_t)std::min(32.0, std::max(4.0, std::ceil(3.0 * (double)p.kp * frac)));
                vsb::launch_tc_sample_threshold(sc.thr_part.as<uint64_t>(), q.n, m, sc.thr.as<float>(), s);
                pc.thr_init = sc.thr.as<float>();
                CU(cudaMemsetAsync(sc.thr_cnt.p, 0, 4, s));
                tc = vsb::launch_exact_candidates_tc(pc, s);
                vsb::launch_tc_count_short(p.part, q.n, p.n_splits, p.kp, k + (self_base >= 0 ? 1u : 0u),
                                           sc.thr_cnt.as<uint32_t>(), s);
                uint32_t n_short = 0;
                CU(vsbi::HostReadback::read(sc.pin, s, &n_short, sc.thr_cnt.p, 4));
                if ((uint64_t)n_short * 50 > q.n) {
                    pc.thr_init = nullptr;
                    tc = vsb::launch_exact_candidates_tc(pc, s);
                }
            }
        } else {
            tc = vsb::launch_exact_candidates_tc(pc, s);
        }
    }
    if (!tc) {
        if (p.kp != kp_simt) {  // the tensor-core launch was refused: plain SIMT with its own list length
            p.kp = kp_simt;
            p.n_splits = vsb::exact_pick_splits(q.n, x_hi - x_lo, sm_count);
            CU(sc.part.ensure(vsb::exact_part_elems(q.n, p.n_splits, p.kp) * 8));
            p.part = sc.part.as<uint64_t>();
        }
        vsb::launch_exact_candidates(p, s);
    }
    CU(cudaGetLastError());
    if (!certify) {
        vsb::launch_exact_rerank(p, k, out.keys, out.dists, out.counts, out.packed, self_base, s);
        CU(cudaGetLastError());
        return VSB_OK;
    }

    // cert_state: [0] = max row norm of the block, [1] = number of flagged queries, [2..] flags
    CU(sc.cert_state.ensure((size_t)(q.n + 2) * 4));
    float* d_xmax = sc.cert_state.as<float>();
    uint32_t* d_count = sc.cert_state.as<uint32_t>() + 1;
    uint32_t* d_flags = sc.cert_state.as<uint32_t>() + 2;
    vsb::launch_max_norm(in.x.nrm, x_lo, x_hi, d_xmax, s);
    vsb::ExactCert cert;
    cert.x_nrm_max = d_xmax;
    cert.flags = d_flags;
    cert.count = d_count;
    cert.sum = cert_sum();
    cert.rel = cert_rel(tc && storage == VSB_F32);

    // flagged queries of one stage -> compact map (indices into the caller's query block) + gathered rows, and the
    // gathered bitmap index of each query (a filtered call whose queries carry their own bitmaps)
    vsb::ExactParams pf = p;
    std::vector<uint32_t> map, flags;
    auto collect = [&](uint32_t n_stage, const std::vector<uint32_t>* prev) -> vsb_status {
        flags.resize(n_stage);
        CU(vsbi::HostReadback::read(sc.pin, s, flags.data(), d_flags, (size_t)n_stage * 4));
        std::vector<uint32_t> next;
        for (uint32_t i = 0; i < n_stage; ++i)
            if (flags[i]) next.push_back(prev ? (*prev)[i] : i);
        map.swap(next);
        const uint32_t nf = (uint32_t)map.size();
        CU(sc.fb_map.ensure((size_t)nf * 4));
        CU(sc.fb.ensure(nf, q.row_bytes));
        CU(cudaMemcpyAsync(sc.fb_map.p, map.data(), (size_t)nf * 4, cudaMemcpyHostToDevice, s));
        vsbi::gather_rows(q, sc.fb_map.as<uint32_t>(), nf, sc.fb, s);
        ST(gather_allow(p.allow, sc.fb_map.as<uint32_t>(), nf, sc.fb_fidx, s, pf.allow));
        pf.q = sc.fb.view(nf);
        CU(cudaStreamSynchronize(s));  // `map` is pageable and is rebuilt by the next stage
        return VSB_OK;
    };

    CU(cudaMemsetAsync(d_count, 0, 4, s));
    vsb::launch_exact_rerank(p, k, out.keys, out.dists, out.counts, out.packed, self_base, s, &cert);
    CU(cudaGetLastError());
    uint32_t n_flagged = 0;
    CU(vsbi::HostReadback::read(sc.pin, s, &n_flagged, d_count, 4));
    cert_ok += q.n - n_flagged;
    cert_fallback += n_flagged;
    if (n_flagged == 0) return VSB_OK;
    ST(collect(q.n, nullptr));

    if (tc && storage == VSB_F32) {
        // second stage: full fp32 products on the SIMT tiles, same certificate with the fp32 bound
        pf.kp = kp_simt;
        pf.n_splits = vsb::exact_pick_splits(pf.q.n, x_hi - x_lo, sm_count);
        CU(sc.part.ensure(vsb::exact_part_elems(pf.q.n, pf.n_splits, pf.kp) * 8));
        pf.part = sc.part.as<uint64_t>();
        vsb::launch_exact_candidates(pf, s);
        CU(cudaGetLastError());
        cert.rel = cert_rel(false);
        CU(cudaMemsetAsync(d_count, 0, 4, s));
        vsb::launch_exact_rerank(pf, k, out.keys, out.dists, out.counts, out.packed, self_base, s, &cert,
                                 sc.fb_map.as<uint32_t>());
        CU(cudaGetLastError());
        CU(vsbi::HostReadback::read(sc.pin, s, &n_flagged, d_count, 4));
        if (n_flagged == 0) return VSB_OK;
        const std::vector<uint32_t> prev = map;
        ST(collect(pf.q.n, &prev));
    }

    // last stage: canonical scan of the whole block for what is left
    cert_scanned += pf.q.n;
    pf.kp = round_up(k + (self_base >= 0 ? 1 : 0), 32);
    const uint32_t scan_splits = vsb::exact_scan_pick_splits(pf.q.n, x_hi - x_lo, sm_count);
    pf.n_splits = scan_splits;
    const uint32_t lists = vsb::exact_scan_lists_per_query(scan_splits);
    CU(sc.part.ensure(vsb::exact_part_elems(pf.q.n, lists, pf.kp) * 8));
    pf.part = sc.part.as<uint64_t>();
    vsb::launch_exact_scan(pf, k, s);
    CU(cudaGetLastError());
    pf.n_splits = lists;
    vsb::launch_exact_rerank(pf, k, out.keys, out.dists, out.counts, out.packed, self_base, s, nullptr,
                             sc.fb_map.as<uint32_t>());
    CU(cudaGetLastError());
    return VSB_OK;
}

// Seeds + K4 (+ K3 re-rank on the bf16-traversal path) for the converted queries `qv`.  out.packed: the raw K4 list
// ([n][k], used by the streaming insert and the refinement) instead of the user-facing top-k.
vsb_status vsb_index::graph_block(const View& v, Scratch& sc, const GraphRun& run, const vsb::RowsView& qv, uint32_t k,
                                  const TopK& out, const vsb::RowsView* q16_in, cudaStream_t s) {
    const vsbi::Store& st = *v.st;
    const vsbi::Seeds& sd = *v.sd;
    const vsb::RowsView x = st.rows.view(v.n_slots);
    const uint32_t nb = qv.n;
    const bool tp = run.timed;
    uint64_t* packed_out = out.packed;
    const uint32_t* deny_bm = v.any_tombstone ? st.deny.as<uint32_t>() : nullptr;
    // the traversal copies serve searches; `native` (a runtime override, searches only) walks the stored rows instead
    const bool t16 = trav16 && !(run.native && packed_out == nullptr);
    // 16-bit float rows (stored, or the bf16 traversal copy) in a large batch are evaluated on the tensor cores: the
    // distances K4 ranks by are then candidate-grade and the rows a SEARCH returns are re-ranked by K3 in the canonical
    // order, exactly like the results of the bf16 / int8 traversal copies (the build only needs the ranking)
    const int trav_storage = t16 ? (int)VSB_BF16 : storage;
    const bool use8_early = trav8 && t16 && packed_out == nullptr;
    const bool mma = !use8_early && vsb::graph_search_uses_mma(trav_storage, nb, run.allow.bm != nullptr, std::max(run.itopk, k));
    const bool rerank = (t16 || mma) && packed_out == nullptr;
    // ---- bf16 shadow of the queries (f32 storage: tensor-core seed layer and/or bf16 traversal) ----
    bool seed_tc = tc_enabled && vsb::exact_tc_supported(storage, metric) && nb >= 16;
    vsb::RowsView q16v;
    if (q16_in != nullptr) {
        q16v = *q16_in;
    } else if (storage == VSB_F32 && (seed_tc || t16)) {
        CU(sc.q16.ensure(nb, row_bytes16));
        vsb::launch_convert_rows(VSB_BF16, reinterpret_cast<const float*>(qv.rows), nb, row_bytes / 4, sc.q16.rows.as<uint8_t>(),
                                 row_bytes16, sc.q16.sq.as<float>(), sc.q16.nrm.as<float>(), s);
        CU(cudaGetLastError());
        q16v = sc.q16.view(nb);
    }
    // ---- seed layer: distances to the contiguous entry-point sample ----
    vsb::ExactParams sp;
    sp.storage = storage;
    sp.metric = metric;
    sp.q = qv;
    sp.x = sd.rows.view(sd.n);
    sp.x_lo = 0;
    sp.x_hi = sd.n;
    sp.keys = nullptr;  // ties fall back to the seed index (LessByKey with null keys)
    sp.kp = 32;
    const vsb::ExactParams sp_native = sp;
    if (seed_tc) {
        // tensor cores: one winner per 256-row tile per query (no list maintenance);
        // f32 storage multiplies the bf16 shadows of the queries and of the seed block
        sp.n_splits = vsb::exact_tc_pick_splits(nb, sd.n, sm_count, 0);
        if (storage == VSB_F32) {
            sp.storage = VSB_BF16;
            sp.q = q16v;
            sp.x = sd.bf16.view(sd.n);
        }
    } else {
        sp.n_splits = vsb::exact_pick_splits(nb, sd.n, sm_count);
    }
    const bool seed_scan = !seed_tc && nb <= vsb::graph_search_small_batch();
    if (seed_scan) sp.n_splits = vsb::seed_scan_blocks(sd.n);
    const uint32_t seed_dense = vsb::exact_tc_tile_min_entries(sd.n);  // tensor-core seed layer: dense winners per query
    CU(sc.seed_part.ensure(std::max<size_t>(vsb::exact_part_elems(nb, sp.n_splits, 32), (size_t)nb * seed_dense) * 8));
    sp.part = sc.seed_part.as<uint64_t>();
    if (tp) t_begin(PH_SEED, s);
    if (seed_tc) {
        CU(cudaMemsetAsync(sc.seed_part.p, 0xFF, (size_t)nb * seed_dense * 8, s));
        seed_tc = vsb::launch_exact_candidates_tc(sp, s, true);
    }
    if (!seed_tc) {
        const uint32_t splits = sp.n_splits;
        sp = sp_native;
        sp.n_splits = splits;
        sp.part = sc.seed_part.as<uint64_t>();
        if (seed_scan) {
            // tiny batch: one warp per 4 seed rows, one winner per CTA
            CU(cudaMemsetAsync(sc.seed_part.p, 0xFF, vsb::exact_part_elems(nb, sp.n_splits, 32) * 8, s));
            vsb::launch_seed_scan(storage, metric, qv, sp.x, sc.seed_part.as<uint64_t>(), s);
        } else {
            vsb::launch_exact_candidates(sp, s);
        }
    }
    if (tp) t_end(s);
    CU(cudaGetLastError());
    // ---- K4 beam search (on the bf16 traversal copy when VSB_FLAG_BF16_TRAVERSAL is set) ----
    vsb::SearchParams gp;
    gp.storage = t16 ? VSB_BF16 : storage;
    gp.metric = metric;
    gp.q = t16 ? q16v : qv;
    gp.x = t16 ? st.bf16.view(v.n_slots) : x;
    const bool use8 = trav8 && rerank;  // searches only: the build keeps the bf16 traversal
    if (use8) {
        CU(sc.q8.ensure(nb, row_bytes8));
        vsb::launch_convert_rows_i8s(reinterpret_cast<const float*>(qv.rows), nb, dim, row_bytes / 4, sc.q8.rows.as<uint8_t>(),
                                     row_bytes8, sc.q8.sq.as<float>(), sc.q8.nrm.as<float>(), s);
        CU(cudaGetLastError());
        gp.storage = VSB_I8;
        gp.q = sc.q8.view(nb);
        gp.x = st.i8.view(v.n_slots);
    }
    gp.graph = v.gr->g.as<uint32_t>();
    gp.graph_stride = graph_stride;
    gp.degree = degree;
    gp.n_graphed = v.n_graphed;
    gp.seed_lists = sc.seed_part.as<uint64_t>();
    gp.seed_stride = seed_tc ? seed_dense : sp.n_splits * 32;
    gp.n_seeds = run.n_seeds;
    gp.seed_slots = sd.slots.as<uint32_t>();
    gp.deny = deny_bm;
    gp.keys = st.keys.as<uint64_t>();
    gp.itopk = std::max(run.itopk, k);
    gp.max_iters = run.max_iters;
    gp.search_width = run.search_width;
    gp.k = k;
    gp.out_keys = out.keys;
    gp.out_dists = out.dists;
    gp.out_counts = out.counts;
    gp.self_base = out.self_base;
    gp.allow = run.allow;
    gp.mma = mma;
    uint32_t kr = 0;
    if (packed_out != nullptr) {
        gp.out_packed = packed_out;
        gp.out_counts = nullptr;
    }
    if (rerank) {
        // hand the best kr bf16-ranked candidates to K3 for the canonical fp32 re-rank
        // (2k for small k, k + 32 + k/4 for large k, at least k + 6; bf16 ranking errors only reorder
        // candidates near the k-th distance and are far smaller than that margin)
        // int8 traversal ranks more coarsely: 4k candidates go to the re-rank
        constexpr uint32_t kRerankMult8 = 4;
        const uint32_t kv = use8 ? std::min<uint32_t>(std::max(kRerankMult8 * k, k + 16), 256)
                                 : std::max(std::min(2 * k, k + 32 + k / 4), k + 6);
        kr = std::min<uint32_t>(round_up(kv, 32), 256);
        if (kr < k) return fail(VSB_EINVAL, "k=%u too large for the bf16-traversal re-rank (max 256)", k);
        CU(sc.rr_packed.ensure((size_t)nb * kr * 8));
        gp.k = std::min(kv, kr);
        gp.out_stride = kr;
        gp.out_packed = sc.rr_packed.as<uint64_t>();
        gp.out_counts = nullptr;
    }
    const bool count = run.count || run.evals != nullptr;
    if (count) {
        CU(sc.counters.ensure(16));
        CU(cudaMemsetAsync(sc.counters.p, 0, 16, s));
        gp.counters = sc.counters.as<unsigned long long>();
    }
    if (tp) t_begin(PH_GRAPH, s);
    vsb::launch_graph_search(gp, s);
    if (tp) t_end(s);
    CU(cudaGetLastError());
    if (rerank) {
        vsb::ExactParams rp;
        rp.storage = storage;
        rp.metric = metric;
        rp.q = qv;
        rp.x = x;
        rp.keys = st.keys.as<uint64_t>();
        rp.part = sc.rr_packed.as<uint64_t>();
        rp.kp = kr;
        rp.n_splits = 1;
        if (tp) t_begin(PH_EXACT, s);
        vsb::launch_exact_rerank(rp, k, out.keys, out.dists, out.counts, nullptr, -1, s);
        if (tp) t_end(s);
        CU(cudaGetLastError());
    }
    if (count) {
        unsigned long long h[2];
        CU(vsbi::HostReadback::read(sc.pin, s, h, sc.counters.p, 16));
        if (run.evals) *run.evals += h[0];
        if (run.parents) *run.parents += h[1];
        if (run.count) {
            last_evals = h[0];
            last_parents = h[1];
            last_queries = nb;
        }
    }
    return VSB_OK;
}

vsb_status vsb_index::search_block(const View& v, Scratch& sc, const vsb::RowsView& qv, uint32_t k, const TopK& out,
                                    cudaStream_t s, bool graph, const vsb::Allow& allow) {
    const uint32_t nb = qv.n;
    uint64_t* o_keys = out.keys;
    float* o_dists = out.dists;
    uint32_t* o_counts = out.counts;
    const bool use_graph = graph && v.n_graphed > 0 && k <= 1024;
    const uint32_t tail_lo = use_graph ? v.n_graphed : 0, tail_hi = v.n_slots;
    const bool have_tail = tail_hi > tail_lo;
    // the brute-force tail contributes at most its 200 best rows to an ANN answer (list length of K1)
    const uint32_t k_tail = use_graph ? std::min<uint32_t>(k, 200) : k;
    uint64_t* g_keys = o_keys;
    float* g_dists = o_dists;
    uint64_t* t_keys = o_keys;
    float* t_dists = o_dists;
    if (use_graph && have_tail) {
        CU(sc.tmp_keys.ensure((size_t)2 * nb * k * 8));
        CU(sc.tmp_dists.ensure((size_t)2 * nb * k * 4));
        g_keys = sc.tmp_keys.as<uint64_t>();
        g_dists = sc.tmp_dists.as<float>();
        t_keys = g_keys + (size_t)nb * k;
        t_dists = g_dists + (size_t)nb * k;
    }
    if (use_graph) {
        GraphRun run;
        run.itopk = itopk;
        run.max_iters = max_iters;
        run.n_seeds = n_seeds;
        run.search_width = search_width;
        run.count = instrumented;
        run.native = native_traversal;
        run.timed = true;
        run.allow = allow;
        TopK g;
        g.keys = g_keys;
        g.dists = g_dists;
        g.counts = have_tail ? nullptr : o_counts;
        ST(graph_block(v, sc, run, qv, k, g, nullptr, s));
    }
    if (have_tail) {
        t_begin(PH_EXACT, s);
        const vsb::ExactParams tail = exact_in(v, qv, tail_lo, tail_hi, allow);
        vsb_status est;
        if (k_tail == k) {
            TopK t;
            t.keys = t_keys;
            t.dists = t_dists;
            t.counts = use_graph ? nullptr : o_counts;
            est = exact_block(sc, tail, k, t, s, /*approx_ok=*/use_graph);  // the ANN tail needs no certificate (no host sync)
        } else {
            // k > 200 with a tail: the tail's best 200 rows, laid out with stride k so that K8 can merge them
            vsb::launch_fill_empty(t_keys, t_dists, nullptr, nb, k, s);
            DevBuf& tk = sc.fb.rows;  // scratch that the ANN path does not otherwise touch
            CU(tk.ensure((size_t)nb * k_tail * 12));
            TopK c;
            c.keys = tk.as<uint64_t>();
            c.dists = reinterpret_cast<float*>(c.keys + (size_t)nb * k_tail);
            est = exact_block(sc, tail, k_tail, c, s, true);
            if (est == VSB_OK) {
                CU(cudaMemcpy2DAsync(t_keys, (size_t)k * 8, c.keys, (size_t)k_tail * 8, (size_t)k_tail * 8, nb, cudaMemcpyDeviceToDevice, s));
                CU(cudaMemcpy2DAsync(t_dists, (size_t)k * 4, c.dists, (size_t)k_tail * 4, (size_t)k_tail * 4, nb, cudaMemcpyDeviceToDevice, s));
            }
        }
        t_end(s);
        ST(est);
    }
    if (use_graph && have_tail) {
        t_begin(PH_MERGE, s);
        vsb::launch_merge_topk(g_keys, g_dists, 2, nb, k, o_keys, o_dists, o_counts, s);
        t_end(s);
        CU(cudaGetLastError());
    }
    return VSB_OK;
}

// search_mu held by the caller
vsb_status vsb_index::search_dev(const float* d_q, uint64_t nq, uint32_t k, uint64_t* d_keys, float* d_dists,
                                 uint32_t* d_counts, cudaStream_t s, bool exact, const vsbi::Filters& f) {
    if (nq == 0) return VSB_OK;
    if (k == 0) return fail(VSB_EINVAL, "k must be > 0");
    if (d_q == nullptr || d_keys == nullptr || d_dists == nullptr) return fail(VSB_EINVAL, "null buffer");
    CU(cudaSetDevice(device));
    last_search_ns.store(std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now().time_since_epoch()).count(),
                         std::memory_order_relaxed);
    const View v = snapshot();
    ST(begin_search(s));
    Scratch& sc = ss;
    const bool filtered = f.allow.bm != nullptr;
    // filtered search, per bitmap: graph traversal with the bitmap unless too few rows are admissible (then the exact
    // scan wins).  Queries whose bitmaps take different routes are split by route below.
    std::vector<uint8_t> graph_of_filter(filtered ? f.n : 0, 0);
    if (filtered && !exact && v.n_graphed > 0 && k <= 256) {
        const uint64_t live_rows = live_atomic.load();
        for (uint32_t i = 0; i < f.n; ++i)
            graph_of_filter[i] = f.pop[i] * 100 >= (uint64_t)filter_min_pct * std::max<uint64_t>(live_rows, 1) && filter_min_pct <= 100;
    }
    const uint64_t QCHUNK = 65536;
    for (uint64_t q0 = 0; q0 < nq; q0 += QCHUNK) {
        const uint32_t nb = (uint32_t)std::min<uint64_t>(QCHUNK, nq - q0);
        TopK o;
        o.keys = d_keys + q0 * k;
        o.dists = d_dists + q0 * k;
        o.counts = d_counts ? d_counts + q0 : nullptr;
        if (v.n_slots == 0) {
            vsb::launch_fill_empty(o.keys, o.dists, o.counts, nb, k, s);
            CU(cudaGetLastError());
            continue;
        }
        CU(sc.q.ensure(nb, row_bytes));
        t_begin(PH_CONVERT, s);
        vsb::launch_convert_rows(storage, d_q + q0 * dim, nb, dim, sc.q.rows.as<uint8_t>(), row_bytes, sc.q.sq.as<float>(),
                                 sc.q.nrm.as<float>(), s);
        t_end(s);
        CU(cudaGetLastError());
        const vsb::RowsView qv = sc.q.view(nb);
        if (!filtered) {
            ST(search_block(v, sc, qv, k, o, s, !exact, vsb::Allow{}));
            continue;
        }
        const vsb::Allow c_allow = f.allow.from(q0);  // this chunk's bitmap indices
        // route of each query of the chunk: by_route[1] = graph, by_route[0] = exact scan
        std::vector<uint32_t> by_route[2];
        for (uint32_t i = 0; i < nb; ++i) by_route[graph_of_filter[f.h_fidx ? f.h_fidx[q0 + i] : 0]].push_back(i);
        if (by_route[0].empty() || by_route[1].empty()) {
            ST(search_block(v, sc, qv, k, o, s, by_route[0].empty(), c_allow));
            continue;
        }
        // mixed routes: each route runs on a compact block of its own queries (rows and bitmap indices gathered like
        // the certificate fallback's), and its [n][k] results are scattered back to the caller's rows
        const uint32_t n_max = (uint32_t)std::max(by_route[0].size(), by_route[1].size());
        CU(sc.rt_map.ensure((size_t)nb * 4));
        CU(sc.rt.ensure(n_max, row_bytes));
        CU(sc.rt_fidx.ensure((size_t)n_max * 4));
        CU(sc.rt_keys.ensure((size_t)n_max * k * 8));
        CU(sc.rt_dists.ensure((size_t)n_max * k * 4));
        CU(sc.rt_counts.ensure((size_t)n_max * 4));
        TopK r_out;
        r_out.keys = sc.rt_keys.as<uint64_t>();
        r_out.dists = sc.rt_dists.as<float>();
        r_out.counts = sc.rt_counts.as<uint32_t>();
        uint32_t* d_map[2] = {sc.rt_map.as<uint32_t>(), sc.rt_map.as<uint32_t>() + by_route[0].size()};
        CU(cudaMemcpyAsync(d_map[0], by_route[0].data(), by_route[0].size() * 4, cudaMemcpyHostToDevice, s));
        CU(cudaMemcpyAsync(d_map[1], by_route[1].data(), by_route[1].size() * 4, cudaMemcpyHostToDevice, s));
        for (int r = 1; r >= 0; --r) {
            const uint32_t n = (uint32_t)by_route[r].size();
            vsbi::gather_rows(qv, d_map[r], n, sc.rt, s);
            vsb::Allow r_allow;
            ST(gather_allow(c_allow, d_map[r], n, sc.rt_fidx, s, r_allow));
            CU(cudaGetLastError());
            ST(search_block(v, sc, sc.rt.view(n), k, r_out, s, r == 1, r_allow));
            vsb::launch_scatter_topk(r_out.keys, r_out.dists, r_out.counts, d_map[r], n, k, o.keys, o.dists, o.counts, s);
            CU(cudaGetLastError());
        }
    }
    ST(end_search(s, v));
    return VSB_OK;
}

namespace vsbi {

std::vector<uint64_t> filter_population(const HostFilters& hf) {
    std::vector<uint64_t> pop(hf.bitmaps ? hf.n : 0, 0);
    const size_t words = (size_t)((hf.bits + 31) / 32), full = (size_t)(hf.bits / 32);
    for (size_t f = 0; f < pop.size(); ++f) {
        const uint32_t* w = hf.bitmaps + f * words;
        for (size_t i = 0; i < full; ++i) pop[f] += (uint64_t)__builtin_popcount(w[i]);
        if (hf.bits % 32) pop[f] += (uint64_t)__builtin_popcount(w[full] & ((1u << (hf.bits % 32)) - 1));
    }
    return pop;
}

vsb_status upload_filters(Scratch& sc, const HostFilters& hf, const uint64_t* pop, const uint32_t* d_fidx, cudaStream_t s,
                          Filters& f) {
    if (hf.bitmaps == nullptr) return VSB_OK;
    const size_t bytes = (size_t)hf.n * ((hf.bits + 31) / 32) * 4;
    CU(sc.allow.ensure(std::max<size_t>(bytes, 16)));
    CU(cudaMemcpyAsync(sc.allow.p, hf.bitmaps, bytes, cudaMemcpyHostToDevice, s));
    f.allow = vsb::Allow{sc.allow.as<uint32_t>(), hf.bits, d_fidx};
    f.n = hf.n;
    f.h_fidx = hf.of_query;
    f.pop = pop;
    return VSB_OK;
}

cudaError_t Staging::carve(DevBuf& buf, size_t q_bytes, uint64_t nq, uint32_t k, bool with_fidx) {
    auto al = [](size_t v) { return (v + 255) / 256 * 256; };
    keys_bytes = (size_t)nq * k * 8;
    dists_bytes = (size_t)nq * k * 4;
    counts_bytes = (size_t)nq * 4;
    const size_t fidx_bytes = with_fidx ? (size_t)nq * 4 : 0;
    const cudaError_t e = buf.ensure(al(q_bytes) + al(keys_bytes) + al(dists_bytes) + al(counts_bytes) + al(fidx_bytes));
    if (e != cudaSuccess) return e;
    uint8_t* p = buf.as<uint8_t>();
    q = q_bytes ? reinterpret_cast<float*>(p) : nullptr;
    keys = reinterpret_cast<uint64_t*>(p += al(q_bytes));
    dists = reinterpret_cast<float*>(p += al(keys_bytes));
    counts = reinterpret_cast<uint32_t*>(p += al(dists_bytes));
    fidx = with_fidx ? reinterpret_cast<uint32_t*>(p + al(counts_bytes)) : nullptr;
    return cudaSuccess;
}

cudaError_t Staging::read(PinBuf& pin, cudaStream_t s, uint64_t* keys_out, float* dists_out, uint32_t* counts_out) const {
    auto al = [](size_t v) { return (v + 255) / 256 * 256; };
    HostReadback rb(pin, s);
    cudaError_t e = cudaSuccess;
    if (!host_is_pinned(keys_out) || !host_is_pinned(dists_out) || (counts_out && !host_is_pinned(counts_out)))
        e = rb.reserve(al(keys_bytes) + al(dists_bytes) + al(counts_bytes));
    if (e == cudaSuccess) e = rb.copy(keys_out, keys, keys_bytes);
    if (e == cudaSuccess) e = rb.copy(dists_out, dists, dists_bytes);
    if (e == cudaSuccess && counts_out) e = rb.copy(counts_out, counts, counts_bytes);
    return e == cudaSuccess ? rb.finish() : e;
}

}  // namespace vsbi

vsb_status vsb_index::search_host(const float* queries, uint64_t nq, uint32_t k, uint64_t* keys_out,
                                  float* dists_out, uint32_t* counts_out, bool exact, const vsbi::HostFilters& hf) {
    if (nq == 0) return VSB_OK;
    if (k == 0) return fail(VSB_EINVAL, "k must be > 0");
    if (queries == nullptr || keys_out == nullptr || dists_out == nullptr) return fail(VSB_EINVAL, "null buffer");
    const size_t in_bytes = (size_t)nq * dim * 4;
    const std::vector<uint64_t> pop = vsbi::filter_population(hf);
    vsbi::Filters f;
    vsbi::Staging st;  // per-query bitmap indices travel with the queries
    if (nq >= 1024) {
        // Large batches are PIPELINED across concurrent callers (the reference serves ann requests from a worker
        // pool, worker.rs:44-118): each call takes one of two staging slots, uploads its queries on the slot's copy
        // stream, runs its kernels on the search stream under search_mu, and downloads its results on the copy
        // stream again — so one caller's H2D / D2H overlaps another caller's kernels.
        CU(cudaSetDevice(device));
        int si = -1;
        {
            std::unique_lock<std::mutex> lk(slot_mu);
            slot_cv.wait(lk, [&] { return !slots[0].busy || !slots[1].busy; });
            si = slots[0].busy ? 1 : 0;
            slots[si].busy = true;
        }
        HostSlot& sl = slots[si];
        struct Release {
            vsb_index* ix;
            int si;
            ~Release() {
                std::lock_guard<std::mutex> lk(ix->slot_mu);
                ix->slots[si].busy = false;
                ix->slot_cv.notify_one();
            }
        } release{this, si};
        if (sl.cs == nullptr) {
            CU(cudaStreamCreateWithFlags(&sl.cs, cudaStreamNonBlocking));
            CU(cudaEventCreateWithFlags(&sl.ev_in, cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&sl.ev_done, cudaEventDisableTiming));
        }
        CU(st.carve(sl.buf, in_bytes, nq, k, hf.of_query != nullptr));
        CU(cudaMemcpyAsync(st.q, queries, in_bytes, cudaMemcpyHostToDevice, sl.cs));
        if (st.fidx) CU(cudaMemcpyAsync(st.fidx, hf.of_query, (size_t)nq * 4, cudaMemcpyHostToDevice, sl.cs));
        CU(cudaEventRecord(sl.ev_in, sl.cs));
        {
            std::lock_guard<std::mutex> g(search_mu);
            ST(vsbi::upload_filters(ss, hf, pop.data(), st.fidx, stream, f));
            CU(cudaStreamWaitEvent(stream, sl.ev_in, 0));
            ST(search_dev(st.q, nq, k, st.keys, st.dists, st.counts, stream, exact, f));
            CU(cudaEventRecord(sl.ev_done, stream));
        }
        CU(cudaStreamWaitEvent(sl.cs, sl.ev_done, 0));
        CU(st.read(sl.pin, sl.cs, keys_out, dists_out, counts_out));
        return VSB_OK;
    }
    std::lock_guard<std::mutex> g(search_mu);
    CU(cudaSetDevice(device));
    ST(begin_search(stream));
    CU(st.carve(ss.q_in, in_bytes, nq, k, hf.of_query != nullptr));
    CU(cudaMemcpyAsync(st.q, queries, in_bytes, cudaMemcpyHostToDevice, stream));
    if (st.fidx) CU(cudaMemcpyAsync(st.fidx, hf.of_query, (size_t)nq * 4, cudaMemcpyHostToDevice, stream));
    ST(vsbi::upload_filters(ss, hf, pop.data(), st.fidx, stream, f));
    ST(search_dev(st.q, nq, k, st.keys, st.dists, st.counts, stream, exact, f));
    CU(st.read(ss.pin, stream, keys_out, dists_out, counts_out));
    reap_inflight(true);
    return VSB_OK;
}
