// index_range.cu — range search (vsb_search_range): every live row within a per-query distance bound, exact.
//
// Per chunk of queries: K0 converts them; the K1 tiles (tensor cores from tc_min_rows rows on, SIMT below and for
// integer rows) run a COUNT pass against bound = max_distance + the candidate stage's error margin; the counts come
// back to the host, which cuts the chunk into sub-chunks whose candidates fit kRangeEntryBudget; per sub-chunk a FILL
// pass appends the candidates, a canonical re-evaluation (K3's arithmetic) keeps the rows within max_distance, a
// segmented sort orders each query's rows by (distance, key) and the kept rows go to the host.
#include <algorithm>
#include <chrono>

#include "index_impl.h"

using vsbi::DevBuf;
using vsbi::fail;

namespace {

// Candidate entries one fill pass holds on the device.  Each costs 32 bytes (the entry, its key and distance, and the
// sort's second copy of both), so the budget is 512 MB; a query that alone has more runs alone with the buffers grown.
constexpr uint64_t kRangeEntryBudget = 1ull << 24;
constexpr uint64_t kRangeChunk = 65536;  // queries converted at a time

inline size_t al256(size_t v) { return (v + 255) / 256 * 256; }

// exclusive prefix sum of v[0..n) (+ total at [n]) into out
template <class F>
void scan_into(uint32_t n, std::vector<uint32_t>& out, F value) {
    out.resize(n + 1);
    uint32_t acc = 0;
    for (uint32_t i = 0; i < n; ++i) {
        out[i] = acc;
        acc += value(i);
    }
    out[n] = acc;
}

}  // namespace

vsb_status vsb_index::search_range(const float* queries, uint64_t nq, const float* max_distance, const vsbi::HostFilters& hf,
                                   uint64_t capacity, uint64_t* keys_out, float* dists_out, vsbi::RangeResult& out) {
    out.off.assign(1, 0);
    out.keys.clear();
    out.dists.clear();
    out.in_place = false;
    if (nq == 0) return VSB_OK;
    std::lock_guard<std::mutex> g(search_mu);
    CU(cudaSetDevice(device));
    last_search_ns.store(std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now().time_since_epoch()).count(),
                         std::memory_order_relaxed);
    const vsbi::View v = snapshot();
    const uint32_t n_rows = v.n_slots;
    if (n_rows == 0) {
        out.off.assign(nq + 1, 0);
        return VSB_OK;
    }
    cudaStream_t s = stream;
    ST(begin_search(s));
    vsbi::Scratch& sc = ss;
    const std::vector<uint64_t> pop = vsbi::filter_population(hf);
    vsbi::Filters f;
    ST(vsbi::upload_filters(sc, hf, pop.data(), nullptr, s, f));
    out.off.reserve(nq + 1);

    // Tensor-core tiles for float rows from tc_min_rows on (f32 rows as TF32), SIMT tiles otherwise.  The margin is the
    // exact search's certificate bound, so every row whose canonical distance is <= max_distance is a candidate.
    const bool tc_shape = tc_enabled && vsb::exact_tc_supported(storage, metric) && n_rows >= tc_min_rows;
    const float rel = cert_rel(tc_shape && storage == VSB_F32), sum = cert_sum();

    // per-chunk arrays: max_distance, bound, count, cursor, kept [nb]; segment / group / output offsets [nb + 1];
    // the block's max row norm and the mismatch counter
    const uint32_t qc = (uint32_t)std::min<uint64_t>(kRangeChunk, nq);
    const size_t qa = al256((size_t)qc * 4), qo = al256((size_t)(qc + 1) * 4);
    const size_t deny_bytes = v.any_tombstone ? al256((size_t)(n_rows + 31) / 32 * 4) : 0;
    CU(sc.rg_q.ensure(5 * qa + 3 * qo + 256 + deny_bytes));
    uint8_t* qbase = sc.rg_q.as<uint8_t>();
    float* d_maxd = reinterpret_cast<float*>(qbase);
    float* d_thr = reinterpret_cast<float*>(qbase + qa);
    uint32_t* d_count = reinterpret_cast<uint32_t*>(qbase + 2 * qa);
    uint32_t* d_cursor = reinterpret_cast<uint32_t*>(qbase + 3 * qa);
    uint32_t* d_kept = reinterpret_cast<uint32_t*>(qbase + 4 * qa);
    uint32_t* d_seg = reinterpret_cast<uint32_t*>(qbase + 5 * qa);
    uint32_t* d_grp = reinterpret_cast<uint32_t*>(qbase + 5 * qa + qo);
    uint32_t* d_out = reinterpret_cast<uint32_t*>(qbase + 5 * qa + 2 * qo);
    float* d_xmax = reinterpret_cast<float*>(qbase + 5 * qa + 3 * qo);
    uint32_t* d_mismatch = reinterpret_cast<uint32_t*>(d_xmax + 1);
    // The tombstones are a live bitmap that vsb_remove writes while searches run.  Both candidate passes test ONE copy
    // of it, taken here, so a concurrent remove can never make the fill pass find fewer rows than the count pass.
    const uint32_t* deny = nullptr;
    if (v.any_tombstone) {
        uint32_t* d_deny = reinterpret_cast<uint32_t*>(qbase + 5 * qa + 3 * qo + 256);
        CU(cudaMemcpyAsync(d_deny, v.st->deny.p, (size_t)(n_rows + 31) / 32 * 4, cudaMemcpyDeviceToDevice, s));
        deny = d_deny;
    }
    vsb::launch_max_norm(v.st->rows.nrm.as<float>(), 0, n_rows, d_xmax, s);

    // K0 + the per-query bound of the chunk of queries [q0, q0 + nb) into sc.q / d_maxd / d_thr
    auto prepare = [&](uint64_t q0, uint32_t nb) -> vsb_status {
        CU(sc.q_in.ensure((size_t)nb * dim * 4));
        CU(cudaMemcpyAsync(sc.q_in.p, queries + q0 * dim, (size_t)nb * dim * 4, cudaMemcpyHostToDevice, s));
        CU(cudaMemcpyAsync(d_maxd, max_distance + q0, (size_t)nb * 4, cudaMemcpyHostToDevice, s));
        CU(sc.q.ensure(nb, row_bytes));
        vsb::launch_convert_rows(storage, sc.q_in.as<float>(), nb, dim, sc.q.rows.as<uint8_t>(), row_bytes, sc.q.sq.as<float>(),
                                 sc.q.nrm.as<float>(), s);
        vsb::launch_range_bound(storage, metric, sc.q.nrm.as<float>(), d_maxd, nb, d_xmax, rel, sum, d_thr, s);
        CU(cudaGetLastError());
        return VSB_OK;
    };
    auto params = [&](uint32_t nb) {
        vsb::ExactParams p = exact_in(v, sc.q.view(nb), 0, n_rows, f.allow);
        p.deny = deny;
        return p;
    };
    auto splits = [&](bool tc, uint32_t n) {
        return tc ? vsb::exact_tc_pick_splits(n, n_rows, sm_count, 32) : vsb::exact_pick_splits(n, n_rows, sm_count);
    };

    // 1. count passes of every chunk (the fill passes take the same path, so both see the same candidate-stage bits)
    std::vector<uint32_t> h_count(nq);
    bool tc = tc_shape;
    uint64_t n_cand = 0;
    for (uint64_t q0 = 0; q0 < nq; q0 += kRangeChunk) {
        const uint32_t nb = (uint32_t)std::min<uint64_t>(kRangeChunk, nq - q0);
        ST(prepare(q0, nb));
        vsb::ExactParams p = params(nb);
        CU(cudaMemsetAsync(d_count, 0, (size_t)nb * 4, s));
        vsb::RangeParams rc;
        rc.thr = d_thr;
        rc.count = d_count;
        p.n_splits = splits(tc, nb);
        if (tc && !vsb::launch_range_candidates_tc(p, rc, s)) {
            // the TMA descriptors could not be encoded: the SIMT tiles serve the whole call, unless earlier chunks
            // already ran on the tensor cores
            if (q0 > 0) return fail(VSB_ECUDA, "range search: the tensor-core count pass could not be launched");
            tc = false;
        }
        if (!tc) {
            p.n_splits = splits(false, nb);
            vsb::launch_range_candidates(p, rc, s);
        }
        CU(cudaGetLastError());
        CU(vsbi::HostReadback::read(sc.pin, s, h_count.data() + q0, d_count, (size_t)nb * 4));
        for (uint32_t i = 0; i < nb; ++i) n_cand += h_count[q0 + i];
    }
    // Kept rows are a subset of the candidates: when all candidates fit, the kept rows go straight to the caller's
    // buffers.  Otherwise they are collected here and copied only if their total fits, since the caller's buffers must
    // stay untouched when the call returns VSB_EFULL.
    out.in_place = keys_out != nullptr && n_cand <= capacity;

    std::vector<uint32_t> h_kept, h_seg, h_grp, h_out;
    bool over = false;  // the total has passed `capacity`: only the counts are finished
    size_t max_entry_bytes = 0;
    for (uint64_t q0 = 0; q0 < nq; q0 += kRangeChunk) {
        const uint32_t nb = (uint32_t)std::min<uint64_t>(kRangeChunk, nq - q0);
        if (nq > kRangeChunk) {  // one chunk: its queries, bounds and counts are still on the device
            ST(prepare(q0, nb));
            CU(cudaMemcpyAsync(d_count, h_count.data() + q0, (size_t)nb * 4, cudaMemcpyHostToDevice, s));
        }
        const vsb::RowsView qv = sc.q.view(nb);
        const vsb::ExactParams p = params(nb);
        const uint32_t* cnt = h_count.data() + q0;

        for (uint32_t a = 0; a < nb;) {
            // 2. sub-chunk [a, b): as many queries as the budget holds, at least one
            uint64_t n_ent = 0;
            uint32_t b = a;
            while (b < nb && (b == a || n_ent + cnt[b] <= kRangeEntryBudget)) n_ent += cnt[b++];
            if (n_ent > 0x7FFFFFFFull)
                return fail(VSB_EOOM, "range search: query %llu has %llu candidate rows (at most 2^31 - 1)",
                            (unsigned long long)(q0 + a), (unsigned long long)n_ent);
            const uint32_t n = b - a, ne = (uint32_t)n_ent;
            h_kept.assign(n, 0);
            uint64_t* emit_keys = nullptr;  // the kept rows of this sub-chunk, compacted (reusing the entry buffers)
            float* emit_dists = nullptr;
            uint32_t* sorted_dord = nullptr;
            uint64_t* sorted_key = nullptr;
            if (ne > 0) {
                scan_into(n, h_seg, [&](uint32_t i) { return cnt[a + i]; });
                scan_into(n, h_grp, [&](uint32_t i) { return (cnt[a + i] + 3) / 4; });
                CU(cudaMemcpyAsync(d_seg, h_seg.data(), (size_t)(n + 1) * 4, cudaMemcpyHostToDevice, s));
                CU(cudaMemcpyAsync(d_grp, h_grp.data(), (size_t)(n + 1) * 4, cudaMemcpyHostToDevice, s));
                const size_t e8 = al256((size_t)ne * 8), e4 = al256((size_t)ne * 4);
                max_entry_bytes = std::max(max_entry_bytes, 3 * e8 + 2 * e4);
                CU(sc.rg_e.ensure(3 * e8 + 2 * e4));
                uint8_t* ebase = sc.rg_e.as<uint8_t>();
                uint64_t* cand = reinterpret_cast<uint64_t*>(ebase);
                uint64_t* key = reinterpret_cast<uint64_t*>(ebase + e8);
                uint64_t* key_alt = reinterpret_cast<uint64_t*>(ebase + 2 * e8);
                uint32_t* dord = reinterpret_cast<uint32_t*>(ebase + 3 * e8);
                uint32_t* dord_alt = reinterpret_cast<uint32_t*>(ebase + 3 * e8 + e4);
                const size_t temp_bytes = vsb::range_sort_temp_bytes(ne, n);
                CU(sc.rg_sort.ensure(temp_bytes));
                CU(cudaMemsetAsync(d_cursor, 0, (size_t)n * 4, s));
                CU(cudaMemsetAsync(d_kept, 0, (size_t)n * 4, s));
                CU(cudaMemsetAsync(d_mismatch, 0, 4, s));

                // 3. fill pass
                vsb::ExactParams pf = p;
                pf.q = qv.slice(a, n);
                pf.n_splits = splits(tc, n);
                vsb::RangeParams rf;
                rf.thr = d_thr + a;
                rf.count = d_count + a;
                rf.off = d_seg;
                rf.cursor = d_cursor;
                rf.out = cand;
                if (tc) {
                    if (!vsb::launch_range_candidates_tc(pf, rf, s))
                        return fail(VSB_ECUDA, "range search: the tensor-core fill pass could not be launched");
                } else {
                    vsb::launch_range_candidates(pf, rf, s);
                }
                CU(cudaGetLastError());
                // 4. canonical re-evaluation (and the per-query cursor == count check)
                vsb::launch_range_eval(pf, d_maxd + a, d_count + a, d_cursor, d_seg, d_grp, h_grp[n], cand, key, dord, d_kept,
                                       d_mismatch, s);
                CU(cudaGetLastError());
                // 5. per-query sort by (distance, key)
                if (!over) CU(vsb::launch_range_sort(dord, key, dord_alt, key_alt, ne, d_seg, n, sc.rg_sort.p, temp_bytes, s));
                uint32_t mismatch = 0;
                vsbi::HostReadback rb(sc.pin, s);
                CU(rb.reserve((size_t)n * 4 + 4));
                CU(rb.copy(h_kept.data(), d_kept, (size_t)n * 4));
                CU(rb.copy(&mismatch, d_mismatch, 4));
                CU(rb.finish());
                if (mismatch != 0)
                    return fail(VSB_ECUDA, "range search: for %u queries the fill pass appended a different number of rows "
                                           "than the count pass counted", mismatch);
                sorted_dord = dord;
                sorted_key = key;
                emit_keys = cand;
                emit_dists = reinterpret_cast<float*>(dord_alt);
            }
            const uint64_t base = out.off.back();
            for (uint32_t i = 0; i < n; ++i) out.off.push_back(out.off.back() + h_kept[i]);
            const uint64_t n_kept = out.off.back() - base;
            if (out.off.back() > capacity) over = true;
            if (!over && n_kept > 0) {
                // 6. the kept rows, compacted in query order, to the host at their offsets
                scan_into(n, h_out, [&](uint32_t i) { return h_kept[i]; });
                CU(cudaMemcpyAsync(d_out, h_out.data(), (size_t)(n + 1) * 4, cudaMemcpyHostToDevice, s));
                vsb::launch_range_emit(sorted_dord, sorted_key, d_seg, d_out, n, (uint32_t)n_kept, emit_keys, emit_dists, s);
                CU(cudaGetLastError());
                uint64_t* k_dst = keys_out + base;
                float* d_dst = dists_out + base;
                if (!out.in_place) {
                    out.keys.resize(base + n_kept);
                    out.dists.resize(base + n_kept);
                    k_dst = out.keys.data() + base;
                    d_dst = out.dists.data() + base;
                }
                vsbi::HostReadback rb(sc.pin, s);
                CU(rb.reserve((size_t)n_kept * 12));
                CU(rb.copy(k_dst, emit_keys, (size_t)n_kept * 8));
                CU(rb.copy(d_dst, emit_dists, (size_t)n_kept * 4));
                CU(rb.finish());
            }
            a = b;
        }
    }
    ST(end_search(s, v));
    reap_inflight(true);
    // like every search scratch buffer the entry buffers stay allocated for the next call, up to the budget's size; a
    // call in which one query alone exceeded the budget gives its larger buffers back
    if (max_entry_bytes > kRangeEntryBudget * 32 + 1024) {
        sc.rg_e.release();
        sc.rg_sort.release();
        sc.pin.release();
    }
    return VSB_OK;
}
