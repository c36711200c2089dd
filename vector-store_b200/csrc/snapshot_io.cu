// snapshot_io.cu — N3 (SURVEY §8f): flat-file snapshot of one shard.  The reference rebuilds its in-memory index
// from a full table scan on every restart (db_cdc/checkpoint_saver.rs:103-112, SURVEY F7); keys / tombstones /
// rows / graph in one file make restart O(read).  A sharded handle writes one file per shard (sharded.cu).
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <vector>

#include "index_impl.h"
#include "sharded.h"

using vsbi::fail;

namespace {
struct SnapHeader {
    char magic[8];  // "VSB200S2"
    vsb_options opt;
    uint64_t n_slots, n_graphed, capacity;
    uint32_t row_bytes, graph_stride, degree;
    // runtime state that is not derivable from the data
    uint32_t itopk, max_iters, n_seeds, search_width, stream_threshold;
    uint64_t churn_since_refine;
};

bool write_dev(FILE* f, const void* dptr, size_t bytes, std::vector<uint8_t>& stage) {
    const size_t CH = stage.size();
    for (size_t off = 0; off < bytes; off += CH) {
        const size_t nb = std::min(CH, bytes - off);
        if (cudaMemcpy(stage.data(), static_cast<const uint8_t*>(dptr) + off, nb, cudaMemcpyDeviceToHost) != cudaSuccess) return false;
        if (fwrite(stage.data(), 1, nb, f) != nb) return false;
    }
    return true;
}
// `check`: called on every chunk before it is uploaded (range validation of the graph)
template <class Check>
bool read_dev(FILE* f, void* dptr, size_t bytes, std::vector<uint8_t>& stage, Check check) {
    const size_t CH = stage.size();
    for (size_t off = 0; off < bytes; off += CH) {
        const size_t nb = std::min(CH, bytes - off);
        if (fread(stage.data(), 1, nb, f) != nb) return false;
        if (!check(stage.data(), nb)) return false;
        if (cudaMemcpy(static_cast<uint8_t*>(dptr) + off, stage.data(), nb, cudaMemcpyHostToDevice) != cudaSuccess) return false;
    }
    return true;
}
}  // namespace

namespace vsbi {

vsb_status save_single(vsb_index* ix, const char* path) {
    // a snapshot is a mutator-consistent state: taken under mut_mu from the working view
    std::lock_guard<std::mutex> g(ix->mut_mu);
    CU(cudaSetDevice(ix->device));
    const View& v = ix->w;
    FILE* f = fopen(path, "wb");
    if (!f) return fail(VSB_EINVAL, "cannot open %s for writing", path);
    SnapHeader h{};
    memcpy(h.magic, "VSB200S2", 8);
    h.opt = ix->opt;
    h.n_slots = v.n_slots;
    h.n_graphed = v.n_graphed;
    h.capacity = v.st ? v.st->capacity : 0;
    h.row_bytes = ix->row_bytes;
    h.graph_stride = ix->graph_stride;
    h.degree = ix->degree;
    h.itopk = ix->itopk;
    h.max_iters = ix->max_iters;
    h.n_seeds = ix->n_seeds;
    h.search_width = ix->search_width;
    h.stream_threshold = ix->stream_threshold;
    h.churn_since_refine = ix->churn_since_refine;
    std::vector<uint8_t> stage((size_t)64 << 20);
    const size_t n = v.n_slots;
    bool ok = fwrite(&h, sizeof h, 1, f) == 1;
    ok = ok && fwrite(ix->h_deny.data(), 4, (n + 31) / 32, f) == (n + 31) / 32;
    if (n) {
        ok = ok && write_dev(f, v.st->keys.p, n * 8, stage);
        const vsbi::RowBuf& rows = v.st->rows;
        ok = ok && write_dev(f, rows.rows.p, n * ix->row_bytes, stage);
        ok = ok && write_dev(f, rows.sq.p, n * 4, stage);
        ok = ok && write_dev(f, rows.nrm.p, n * 4, stage);
    }
    if (v.n_graphed) ok = ok && write_dev(f, v.gr->g.p, (size_t)v.n_graphed * ix->graph_stride * 4, stage);
    ok = (fclose(f) == 0) && ok;
    if (!ok) return fail(VSB_ECUDA, "short write or copy failure while saving %s", path);
    return VSB_OK;
}

vsb_status load_single(const char* path, int32_t device, vsb_index** out) {
    *out = nullptr;
    FILE* f = fopen(path, "rb");
    if (!f) return fail(VSB_EINVAL, "cannot open %s", path);
    SnapHeader h{};
    if (fread(&h, sizeof h, 1, f) != 1 || memcmp(h.magic, "VSB200S2", 8) != 0) {
        fclose(f);
        return fail(VSB_EINVAL, "%s is not a vsb200 snapshot (format VSB200S2)", path);
    }
    h.opt.device = device;
    h.opt.n_devices = 0;
    vsb_index* ix = nullptr;
    vsb_status st = create_single(&h.opt, &ix);
    if (st != VSB_OK) {
        fclose(f);
        return st;
    }
    auto bail = [&](vsb_status code, const char* what) {
        fclose(f);
        destroy_single(ix);
        return fail(code, "%s while loading %s", what, path);
    };
    // the header is untrusted input: every count that later indexes device memory is checked here
    if (h.row_bytes != ix->row_bytes || h.graph_stride != ix->graph_stride || h.degree != ix->degree)
        return bail(VSB_EINVAL, "layout mismatch");
    if (h.n_slots >= (1ull << 28) || h.capacity >= (1ull << 28) || h.n_slots > std::max<uint64_t>(h.capacity, 1) ||
        h.n_graphed > h.n_slots)
        return bail(VSB_EINVAL, "inconsistent row counts in the header");
    const size_t n = (size_t)h.n_slots;  // nobody else holds this handle yet: no locking needed
    if (ix->reserve(std::max<uint64_t>(h.capacity, std::max<uint64_t>(n, 1))) != VSB_OK) return bail(VSB_EOOM, "reserve failed");
    std::vector<uint8_t> stage((size_t)64 << 20);
    std::vector<uint64_t> h_keys(n);
    bool ok = fread(ix->h_deny.data(), 4, (n + 31) / 32, f) == (n + 31) / 32;
    ok = ok && fread(h_keys.data(), 8, n, f) == n;
    if (!ok) return bail(VSB_EINVAL, "truncated file");
    vsbi::Store& store = *ix->w.st;
    auto no_check = [](const uint8_t*, size_t) { return true; };
    if (n) {
        if (cudaMemcpy(store.keys.p, h_keys.data(), n * 8, cudaMemcpyHostToDevice) != cudaSuccess ||
            cudaMemcpy(store.deny.p, ix->h_deny.data(), ((n + 31) / 32) * 4, cudaMemcpyHostToDevice) != cudaSuccess)
            return bail(VSB_ECUDA, "upload failed");
        ok = read_dev(f, store.rows.rows.p, n * ix->row_bytes, stage, no_check);
        ok = ok && read_dev(f, store.rows.sq.p, n * 4, stage, no_check);
        ok = ok && read_dev(f, store.rows.nrm.p, n * 4, stage, no_check);
    }
    if (ok && h.n_graphed) {
        auto gr = std::make_shared<vsbi::Graph>();
        gr->cap_rows = std::max<uint64_t>(store.capacity, h.n_graphed);
        if (gr->g.alloc((size_t)gr->cap_rows * ix->graph_stride * 4) != cudaSuccess) return bail(VSB_EOOM, "graph allocation failed");
        bool in_range = true;
        const uint32_t limit = (uint32_t)h.n_graphed;
        auto check_ids = [&](const uint8_t* p, size_t nb) {
            const uint32_t* ids = reinterpret_cast<const uint32_t*>(p);
            for (size_t i = 0; i < nb / 4; ++i)
                if (ids[i] != vsb::kInvalidSlot && ids[i] >= limit) {
                    in_range = false;
                    return false;
                }
            return true;
        };
        ok = read_dev(f, gr->g.p, (size_t)h.n_graphed * ix->graph_stride * 4, stage, check_ids);
        if (!in_range) return bail(VSB_EINVAL, "graph edge out of range");
        ix->w.gr = gr;
    }
    if (!ok) return bail(VSB_EINVAL, "truncated file or copy failure");
    fclose(f);
    ix->w.n_slots = (uint32_t)n;
    ix->w.n_graphed = (uint32_t)h.n_graphed;
    uint64_t live = 0;
    for (size_t i = 0; i < n; ++i) {
        if (ix->h_deny[i >> 5] >> (i & 31) & 1u) {
            ix->w.any_tombstone = true;
            ix->n_tombstones += 1;
            continue;
        }
        ix->key2slot.emplace(h_keys[i], (uint32_t)i);
        ++live;
    }
    ix->live = live;
    ix->itopk = std::min<uint32_t>(std::max<uint32_t>(h.itopk, 32), 1024);
    ix->max_iters = h.max_iters;
    ix->n_seeds = std::min<uint32_t>(std::max<uint32_t>(h.n_seeds, 1), 32);
    ix->search_width = std::min<uint32_t>(std::max<uint32_t>(h.search_width, 1), 4);
    ix->stream_threshold = h.stream_threshold;
    ix->churn_since_refine = h.churn_since_refine;
    // the traversal copies are derived data: regenerated instead of stored
    if ((n && ix->derive_traversal(store, store.rows.rows.as<float>(), ix->row_bytes / 4, 0, (uint32_t)n) != VSB_OK) ||
        (ix->w.n_graphed && ix->sample_seeds(ix->w.n_graphed) != VSB_OK)) {
        destroy_single(ix);
        return VSB_ECUDA;
    }
    cudaStreamSynchronize(ix->mstream);
    ix->publish();
    *out = ix;
    return VSB_OK;
}

}  // namespace vsbi

extern "C" vsb_status vsb_save(vsb_index* ix, const char* path) {
    if (!ix || !path) return fail(VSB_EINVAL, "null argument");
    if (ix->sharded) return vsbi::sharded_save(ix, path);
    return vsbi::save_single(ix, path);
}

extern "C" vsb_status vsb_load(const char* path, int32_t device, vsb_index** out) {
    if (!path || !out) return fail(VSB_EINVAL, "null argument");
    return vsbi::load_single(path, device, out);
}
