// index.cu — lifecycle, mutations and the C ABI of libvsb200 (include/vsb200.h).
// The object model and the concurrency contract are described in index_impl.h; the search building blocks
// live in index_search.cu, the graph build in index_build.cu, snapshots in snapshot_io.cu, the multi-device
// router in sharded.cu.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <new>
#include <unordered_set>

#include <nvtx3/nvToolsExt.h>

#include "index_impl.h"
#include "sharded.h"

namespace vsb {
std::atomic<uint64_t> g_kernel_launches{0};
std::atomic<uint64_t> g_tc_launches{0};
}  // namespace vsb

namespace vsbi {

static thread_local std::string g_last_error;

vsb_status fail(vsb_status st, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_last_error = buf;
    return st;
}

// one allocator stream per device (see DevBuf); the device's default pool is told to keep what it is given back
cudaStream_t pool_stream(int device) {
    static std::mutex mu;
    static cudaStream_t streams[64] = {};
    std::lock_guard<std::mutex> g(mu);
    if (device < 0 || device >= 64) return nullptr;
    if (streams[device] == nullptr) {
        int cur = -1;
        cudaGetDevice(&cur);
        if (cur != device) cudaSetDevice(device);
        cudaStreamCreateWithFlags(&streams[device], cudaStreamNonBlocking);
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
            uint64_t keep = ~0ull;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        }
        if (cur != device && cur >= 0) cudaSetDevice(cur);
    }
    return streams[device];
}

static int64_t now_ns() {
    return std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

MutGuard::MutGuard(vsb_index* ix) : lock(ix->mut_mu) {
    const bool searching = ix->mstream_green != nullptr && now_ns() - ix->last_search_ns.load(std::memory_order_relaxed) < 2000000000ll;
    ix->mstream = searching ? ix->mstream_green : ix->mstream_full;
}

uint32_t storage_row_bytes(int storage, uint32_t dim) {
    uint64_t bits = 0;
    switch (storage) {
        case VSB_F32: bits = (uint64_t)dim * 32; break;
        case VSB_F16:
        case VSB_BF16: bits = (uint64_t)dim * 16; break;
        case VSB_I8: bits = (uint64_t)dim * 8; break;
        default: bits = dim; break;
    }
    return (uint32_t)(((bits + 127) / 128) * 16);
}

}  // namespace vsbi

using vsbi::DevBuf;
using vsbi::fail;
using vsbi::round_up;

// ---- phase timing of the search path --------------------------------------------------------------------------
void vsb_index::t_begin(int phase, cudaStream_t s) {
    if (!timing) return;
    Timed t;
    t.phase = phase;
    cudaEventCreate(&t.a);
    cudaEventCreate(&t.b);
    cudaEventRecord(t.a, s);
    timed.push_back(t);
}
void vsb_index::t_end(cudaStream_t s) {
    if (!timing) return;
    cudaEventRecord(timed.back().b, s);
}
void vsb_index::t_resolve() {
    for (auto& t : timed) {
        float ms = 0.f;
        if (cudaEventSynchronize(t.b) == cudaSuccess && cudaEventElapsedTime(&ms, t.a, t.b) == cudaSuccess) {
            phase_ns[t.phase] += (uint64_t)((double)ms * 1e6);
            phase_launches[t.phase] += 1;
        }
        cudaEventDestroy(t.a);
        cudaEventDestroy(t.b);
    }
    timed.clear();
}

// ---- search-side stream hand-over and view lifetime -------------------------------------------------------------
// The scratch set is shared by consecutive searches: a search on another stream than the previous one waits
// (on the device, not on the host) for the event the previous search recorded.  The legacy default stream
// (nullptr) is a stream like any other here.
void vsb_index::reap_inflight(bool wait) {
    while (!inflight.empty()) {
        InFlight& f = inflight.front();
        if (wait) cudaEventSynchronize(f.done);
        else if (cudaEventQuery(f.done) != cudaSuccess) break;
        cudaEventDestroy(f.done);
        inflight.pop_front();
    }
}

vsb_status vsb_index::begin_search(cudaStream_t s) {
    reap_inflight(false);
    if (!inflight.empty() && inflight.back().stream != s) CU(cudaStreamWaitEvent(s, inflight.back().done, 0));
    return VSB_OK;
}

vsb_status vsb_index::end_search(cudaStream_t s, const vsbi::View& v) {
    InFlight f;
    CU(cudaEventCreateWithFlags(&f.done, cudaEventDisableTiming));
    CU(cudaEventRecord(f.done, s));
    f.stream = s;
    f.view = v;
    inflight.push_back(std::move(f));
    return VSB_OK;
}

size_t vsb_index::hbm_bytes() {
    vsbi::View v = snapshot();
    size_t s = ss.bytes() + ms.bytes() + slots[0].buf.bytes + slots[1].buf.bytes;
    if (v.st) s += v.st->bytes();
    if (v.gr) s += v.gr->g.bytes;
    if (v.sd) s += v.sd->bytes();
    return s;
}

// ---- mutators (mut_mu held by the caller) -----------------------------------------------------------------------
vsb_status vsb_index::new_store(uint64_t cap, std::shared_ptr<vsbi::Store>& out) {
    auto st = std::make_shared<vsbi::Store>();
    const uint64_t words = (cap + 31) / 32;
    st->capacity = cap;
    CU(st->rows.alloc(cap, row_bytes));
    CU(st->keys.alloc((size_t)cap * 8));
    CU(st->deny.alloc((size_t)words * 4));
    if (trav16) CU(st->bf16.alloc(cap, row_bytes16));
    if (trav8) CU(st->i8.alloc(cap, row_bytes8));
    CU(cudaMemsetAsync(st->deny.p, 0, (size_t)words * 4, mstream));
    out = std::move(st);
    return VSB_OK;
}

vsb_status vsb_index::reserve(uint64_t cap) {
    const uint64_t have = w.st ? w.st->capacity : 0;
    if (cap <= have) return VSB_OK;
    if (cap >= (1ull << 28)) return fail(VSB_EINVAL, "capacity %llu exceeds the 2^28 rows one shard holds", (unsigned long long)cap);
    CU(cudaSetDevice(device));
    nvtxRangePushA("vsb_reserve");
    std::shared_ptr<vsbi::Store> ns;
    vsb_status st = new_store(cap, ns);
    if (st != VSB_OK) {
        nvtxRangePop();
        return st;
    }
    const size_t n = w.n_slots;
    if (n > 0) {
        const vsbi::Store& o = *w.st;
        auto cp = [&](const DevBuf& dst, const DevBuf& src, size_t bytes) {
            return cudaMemcpyAsync(dst.p, src.p, bytes, cudaMemcpyDeviceToDevice, mstream);
        };
        for (auto b : vsbi::kStoreRows) {
            const vsbi::RowBuf &from = o.*b, &to = (*ns).*b;
            if (from.row_bytes == 0) continue;
            CU(cp(to.rows, from.rows, n * from.row_bytes));
            CU(cp(to.sq, from.sq, n * 4));
            CU(cp(to.nrm, from.nrm, n * 4));
        }
        CU(cp(ns->keys, o.keys, n * 8));
        CU(cp(ns->deny, o.deny, ((n + 31) / 32) * 4));
    }
    CU(cudaStreamSynchronize(mstream));
    w.st = ns;
    h_deny.resize((cap + 31) / 32, 0u);
    {
        std::lock_guard<std::mutex> g(map_mu);
        key2slot.reserve((size_t)cap);
    }
    publish();
    nvtxRangePop();
    return VSB_OK;
}

// row_status == nullptr: all-or-nothing (vsb_add).  Otherwise per-row verdicts (vsb_add_each).
vsb_status vsb_index::add(const uint64_t* k, const float* r, uint64_t n, int32_t* row_status, uint64_t* n_added,
                          bool rows_on_device) {
    if (n_added) *n_added = 0;
    if (n == 0) return VSB_OK;
    if (k == nullptr || r == nullptr) return fail(VSB_EINVAL, "null keys/rows");
    const uint64_t cap = w.st ? w.st->capacity : 0;
    std::vector<uint64_t> take;  // indices of the rows to insert (each mode with rejects only)
    uint64_t nv = n;
    {
        std::unordered_set<uint64_t> batch;
        if (n > 1) batch.reserve((size_t)n);
        bool any_reject = false;
        for (uint64_t i = 0; i < n; ++i) {
            int32_t verdict = VSB_OK;
            if (k[i] == 0xFFFFFFFFFFFFFFFFull) verdict = VSB_EINVAL;
            else if (key2slot.count(k[i]) || (n > 1 && !batch.insert(k[i]).second)) verdict = VSB_EDUPKEY;
            if (row_status == nullptr) {
                if (verdict == VSB_EINVAL) return fail(VSB_EINVAL, "key UINT64_MAX is reserved");
                if (verdict == VSB_EDUPKEY) return fail(VSB_EDUPKEY, "duplicate key %llu", (unsigned long long)k[i]);
            } else {
                row_status[i] = verdict;
                any_reject |= verdict != VSB_OK;
            }
        }
        if (any_reject) {
            for (uint64_t i = 0; i < n; ++i)
                if (row_status[i] == VSB_OK) take.push_back(i);
            nv = take.size();
            if (nv == 0) return VSB_OK;
        }
    }
    if (live + nv > cap)
        return fail(VSB_EFULL, "size %llu + %llu exceeds capacity %llu: reserve capacity ahead of insertions",
                    (unsigned long long)live, (unsigned long long)nv, (unsigned long long)cap);
    CU(cudaSetDevice(device));
    if ((uint64_t)w.n_slots + nv > cap) {
        // usearch reuses the slots of removed vectors; here the slot space is reclaimed by a compaction that keeps the
        // graph (edges are renumbered, edges to removed rows dropped) — a few ms of HBM copies per GB
        ST(compact(true));
    }
    vsbi::Store& st = *w.st;
    std::vector<float> gathered;
    std::vector<uint64_t> gathered_keys;
    const float* src = r;
    const uint64_t* src_keys = k;
    if (!take.empty()) {
        if (rows_on_device) return fail(VSB_EINVAL, "vsb_add_dev is all-or-nothing");
        gathered.resize((size_t)nv * dim);
        gathered_keys.resize((size_t)nv);
        for (uint64_t j = 0; j < nv; ++j) {
            std::memcpy(&gathered[(size_t)j * dim], r + take[j] * dim, (size_t)dim * 4);
            gathered_keys[j] = k[take[j]];
        }
        src = gathered.data();
        src_keys = gathered_keys.data();
    }
    // rows already in HBM (vsb_add_dev): one pass; host rows: 256 MB chunks through the staging buffer
    const uint64_t chunk_rows = rows_on_device ? nv : std::max<uint64_t>(1, (256ull << 20) / ((uint64_t)dim * 4));
    for (uint64_t b = 0; b < nv; b += chunk_rows) {
        const uint64_t nb = std::min(chunk_rows, nv - b);
        const float* d_src = src + b * dim;
        if (!rows_on_device) {
            CU(ms.q_in.ensure(nb * dim * 4));
            CU(cudaMemcpyAsync(ms.q_in.p, src + b * dim, nb * dim * 4, cudaMemcpyHostToDevice, mstream));
            d_src = ms.q_in.as<float>();
        }
        const uint32_t s0 = w.n_slots + (uint32_t)b;
        vsb::launch_convert_rows(storage, d_src, (uint32_t)nb, dim, st.rows.rows.as<uint8_t>() + (size_t)s0 * row_bytes,
                                 row_bytes, st.rows.sq.as<float>() + s0, st.rows.nrm.as<float>() + s0, mstream);
        CU(cudaGetLastError());
        ST(derive_traversal(st, d_src, dim, s0, (uint32_t)nb));
        CU(cudaMemcpyAsync(st.keys.as<uint64_t>() + s0, src_keys + b, nb * 8, cudaMemcpyHostToDevice, mstream));
        CU(cudaStreamSynchronize(mstream));  // q_in is reused by the next chunk
    }
    {
        std::lock_guard<std::mutex> g(map_mu);
        for (uint64_t i = 0; i < nv; ++i) key2slot.emplace(src_keys[i], w.n_slots + (uint32_t)i);
    }
    w.n_slots += (uint32_t)nv;
    live += nv;
    if (n_added) *n_added = nv;
    publish();  // searchable from here on (brute-force tail)
    if (w.n_graphed > 0 && stream_threshold > 0 && w.n_slots - w.n_graphed >= stream_threshold) {
        ST(stream_insert());
        publish();
    }
    return VSB_OK;
}

vsb_status vsb_index::derive_traversal(vsbi::Store& st, const float* src, uint32_t in_stride, uint32_t s0, uint32_t n) {
    if (trav16) {
        vsb::launch_convert_rows(VSB_BF16, src, n, in_stride, st.bf16.rows.as<uint8_t>() + (size_t)s0 * row_bytes16, row_bytes16,
                                 st.bf16.sq.as<float>() + s0, st.bf16.nrm.as<float>() + s0, mstream);
        CU(cudaGetLastError());
    }
    if (trav8) {
        vsb::launch_convert_rows_i8s(src, n, dim, in_stride, st.i8.rows.as<uint8_t>() + (size_t)s0 * row_bytes8, row_bytes8,
                                     st.i8.sq.as<float>() + s0, st.i8.nrm.as<float>() + s0, mstream);
        CU(cudaGetLastError());
    }
    return VSB_OK;
}

vsb_status vsb_index::remove(const uint64_t* k, uint64_t n, uint64_t* removed) {
    uint64_t cnt = 0;
    uint32_t lo_word = 0xFFFFFFFFu, hi_word = 0;
    {
        std::lock_guard<std::mutex> g(map_mu);
        for (uint64_t i = 0; i < n; ++i) {
            auto it = key2slot.find(k[i]);
            if (it == key2slot.end()) continue;
            const uint32_t slot = it->second;
            h_deny[slot >> 5] |= 1u << (slot & 31);
            lo_word = std::min(lo_word, slot >> 5);
            hi_word = std::max(hi_word, slot >> 5);
            key2slot.erase(it);
            ++cnt;
        }
    }
    if (cnt) {
        CU(cudaSetDevice(device));
        // tombstones are a live bitmap: a search that runs concurrently sees either state of a word
        CU(cudaMemcpyAsync(w.st->deny.as<uint32_t>() + lo_word, h_deny.data() + lo_word, (size_t)(hi_word - lo_word + 1) * 4,
                           cudaMemcpyHostToDevice, mstream));
        CU(cudaStreamSynchronize(mstream));
        live -= cnt;
        n_tombstones += cnt;
        w.any_tombstone = true;
        churn_since_refine += cnt;
        publish();
    }
    if (removed) *removed = cnt;
    return VSB_OK;
}

// Tombstone compaction: live rows are gathered to the front in slot order into a NEW store (the old one keeps
// serving running searches), the key map is renumbered, the tombstone bitmap cleared.  keep_graph: the graph rows
// are renumbered too (edges to removed rows dropped), so the index stays navigable without a rebuild.
vsb_status vsb_index::compact(bool keep_graph) {
    const uint32_t n_old = w.n_slots;
    std::vector<uint32_t> live_slots;
    live_slots.reserve((size_t)live);
    for (uint32_t i = 0; i < n_old; ++i)
        if (!(h_deny[i >> 5] >> (i & 31) & 1u)) live_slots.push_back(i);
    const uint32_t m = (uint32_t)live_slots.size();
    if (m == n_old) {
        w.any_tombstone = false;
        n_tombstones = 0;
        return VSB_OK;
    }
    nvtxRangePushA("vsb_compact");
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    cudaEventRecord(e0, mstream);
    const vsbi::Store& o = *w.st;
    std::shared_ptr<vsbi::Store> ns;
    ST(new_store(o.capacity, ns));
    DevBuf d_slots, d_map;
    CU(d_slots.alloc(std::max<size_t>((size_t)m * 4, 16)));
    CU(cudaMemcpyAsync(d_slots.p, live_slots.data(), (size_t)m * 4, cudaMemcpyHostToDevice, mstream));
    for (auto b : vsbi::kStoreRows)
        if ((o.*b).row_bytes) vsbi::gather_rows((o.*b).view(n_old), d_slots.as<uint32_t>(), m, (*ns).*b, mstream);
    vsb::launch_gather_u64(o.keys.as<uint64_t>(), d_slots.as<uint32_t>(), m, ns->keys.as<uint64_t>(), mstream);
    CU(cudaGetLastError());
    std::vector<uint32_t> old2new((size_t)n_old, vsb::kInvalidSlot);
    for (uint32_t i = 0; i < m; ++i) old2new[live_slots[i]] = i;
    uint32_t new_graphed = 0;
    std::shared_ptr<vsbi::Graph> ng;
    if (keep_graph && w.n_graphed > 0) {
        new_graphed = (uint32_t)(std::lower_bound(live_slots.begin(), live_slots.end(), w.n_graphed) - live_slots.begin());
        CU(d_map.alloc((size_t)n_old * 4));
        CU(cudaMemcpyAsync(d_map.p, old2new.data(), (size_t)n_old * 4, cudaMemcpyHostToDevice, mstream));
        ng = std::make_shared<vsbi::Graph>();
        ng->cap_rows = o.capacity;
        CU(ng->g.alloc((size_t)o.capacity * graph_stride * 4));
        vsb::launch_remap_graph(w.gr->g.as<uint32_t>(), w.n_graphed, graph_stride, d_map.as<uint32_t>(), ng->g.as<uint32_t>(), mstream);
        CU(cudaGetLastError());
    }
    CU(cudaStreamSynchronize(mstream));
    {
        std::lock_guard<std::mutex> g(map_mu);
        for (auto& kv : key2slot) kv.second = old2new[kv.second];
    }
    std::fill(h_deny.begin(), h_deny.end(), 0u);
    w.st = ns;
    w.n_slots = m;
    w.n_graphed = new_graphed;
    w.gr = ng;
    w.any_tombstone = false;
    n_tombstones = 0;
    if (new_graphed > 0) ST(sample_seeds(new_graphed));
    else w.sd.reset();
    cudaEventRecord(e1, mstream);
    cudaEventSynchronize(e1);
    float ms_ = 0.f;
    cudaEventElapsedTime(&ms_, e0, e1);
    bstats.compact_ns += (uint64_t)((double)ms_ * 1e6);
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    nvtxRangePop();
    return VSB_OK;
}

// ------------------------------------------------------------------------------------------------
namespace vsbi {

vsb_status create_single(const vsb_options* o, vsb_index** out) {
    *out = nullptr;
    int metric = o->metric;
    // usearch.rs:450-464: B1 always uses Hamming; Hamming without B1 is rejected (usearch.rs:480-485)
    if (o->storage == VSB_B1) metric = VSB_HAMMING;
    else if (metric == VSB_HAMMING) return fail(VSB_EINVAL, "Binary space type requires B1 quantization.");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(VSB_ECUDA, "no usable CUDA device (%s): vsb200 has no CPU fallback", cudaGetErrorString(e));
    int dev = o->device;
    if (dev < 0) CU(cudaGetDevice(&dev));
    if (dev >= ndev) return fail(VSB_EINVAL, "device %d out of range (%d devices)", dev, ndev);
    CU(cudaSetDevice(dev));
    vsb_index* ix = new (std::nothrow) vsb_index();
    if (!ix) return fail(VSB_EOOM, "host allocation failed");
    ix->opt = *o;
    ix->opt.n_devices = 0;
    ix->dim = o->dimensions;
    ix->metric = metric;
    ix->storage = o->storage;
    ix->device = dev;
    ix->row_bytes = storage_row_bytes(o->storage, o->dimensions);
    const uint32_t M = o->connectivity ? o->connectivity : 16;
    const uint32_t ef_add = o->expansion_add ? o->expansion_add : 128;
    const uint32_t ef_search = o->expansion_search ? o->expansion_search : 64;
    ix->degree = std::min<uint32_t>(std::max<uint32_t>(2 * M, 8), 64);
    ix->graph_stride = round_up(ix->degree, 32);
    ix->k_init = std::min<uint32_t>(std::max<uint32_t>(ef_add / 2, ix->degree), 128);
    ix->itopk = std::min<uint32_t>(round_up(ef_search, 32), 1024);
    ix->trav16 = (o->flags & VSB_FLAG_BF16_TRAVERSAL) != 0 && o->storage == VSB_F32;
    ix->row_bytes16 = storage_row_bytes(VSB_BF16, o->dimensions);
    ix->trav8 = (o->flags & VSB_FLAG_I8_TRAVERSAL) != 0 && o->storage == VSB_F32 && o->metric == VSB_COS;
    if (ix->trav8) ix->trav16 = true;  // the bf16 copy feeds the build and the seed tiles
    ix->row_bytes8 = storage_row_bytes(VSB_I8, o->dimensions);
    if (const char* v = getenv("VSB_DISABLE_TC")) ix->tc_enabled = !(v[0] == '1');
    if (const char* v = getenv("VSB_DISABLE_CERT")) ix->cert_enabled = !(v[0] == '1');
    if (const char* v = getenv("VSB_CERT_KP")) ix->cert_kp = (uint32_t)strtoul(v, nullptr, 10);
    if (const char* v = getenv("VSB_ALLPAIRS_MAX")) ix->allpairs_max = (uint32_t)strtoul(v, nullptr, 10);
    if (const char* v = getenv("VSB_ALLPAIRS_PREFIX")) ix->allpairs_prefix = (uint32_t)strtoul(v, nullptr, 10);
    if (o->flags & VSB_FLAG_BUILD_REFINE) ix->refine_passes = 1;
    if (const char* v = getenv("VSB_REFINE_PASSES")) ix->refine_passes = (uint32_t)strtoul(v, nullptr, 10);
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, dev) == cudaSuccess) ix->sm_count = prop.multiProcessorCount;
    // searches on a high-priority stream, mutators (build, streaming insert, refinement) on a low-priority one:
    // when both have CTAs pending, the block scheduler serves the search first
    int prio_lo = 0, prio_hi = 0;
    cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
    e = cudaStreamCreateWithPriority(&ix->stream, cudaStreamNonBlocking, prio_hi);
    if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&ix->mstream_full, cudaStreamNonBlocking, prio_lo);
    if (e != cudaSuccess) {
        destroy_single(ix);
        return fail(VSB_ECUDA, "cudaStreamCreate: %s", cudaGetErrorString(e));
    }
    ix->mstream = ix->mstream_full;
    // SMs the mutators never touch while searches are active; without a green context the mutators stay on the plain
    // low-priority stream
    constexpr unsigned kSearchSmReserve = 12;
    unsigned sms = 0;
    if (make_green_stream(dev, kSearchSmReserve, prio_lo, &ix->mstream_green, &ix->green_ctx, &sms)) ix->green_sms = sms;
    CU(cudaSetDevice(dev));
    ix->w.st = std::make_shared<Store>();
    ix->publish();
    *out = ix;
    return VSB_OK;
}

void destroy_single(vsb_index* ix) {
    if (!ix) return;
    cudaSetDevice(ix->device);
    cudaDeviceSynchronize();
    ix->t_resolve();
    ix->reap_inflight(true);
    for (auto& sl : ix->slots) {
        if (sl.cs) cudaStreamDestroy(sl.cs);
        if (sl.ev_in) cudaEventDestroy(sl.ev_in);
        if (sl.ev_done) cudaEventDestroy(sl.ev_done);
    }
    if (ix->stream) cudaStreamDestroy(ix->stream);
    if (ix->mstream_full) cudaStreamDestroy(ix->mstream_full);
    if (ix->mstream_green) cudaStreamDestroy(ix->mstream_green);
    if (ix->green_ctx) destroy_green(ix->green_ctx);
    delete ix;
}

}  // namespace vsbi

extern "C" {

vsb_status vsb_create(const vsb_options* o, vsb_index** out) {
    if (o == nullptr || out == nullptr) return fail(VSB_EINVAL, "null options/out");
    *out = nullptr;
    if (o->dimensions == 0) return fail(VSB_EINVAL, "dimensions must be > 0");
    if (o->storage < VSB_F32 || o->storage > VSB_B1) return fail(VSB_EINVAL, "unknown storage scalar %d", o->storage);
    if (o->metric < VSB_L2SQ || o->metric > VSB_HAMMING) return fail(VSB_EINVAL, "unknown metric %d", o->metric);
    if (o->n_devices < 0 || o->n_devices > 8) return fail(VSB_EINVAL, "n_devices must be in 0..8");
    if (o->n_devices > 1) return vsbi::create_sharded(o, out);
    vsb_options one = *o;
    if (o->n_devices == 1) one.device = o->device_ids[0];
    return vsbi::create_single(&one, out);
}

void vsb_destroy(vsb_index* ix) {
    if (!ix) return;
    if (ix->sharded) {
        vsbi::destroy_sharded(ix);
        return;
    }
    vsbi::destroy_single(ix);
}

vsb_status vsb_reserve(vsb_index* ix, uint64_t capacity) {
    if (!ix) return fail(VSB_EINVAL, "null index");
    if (ix->sharded) return vsbi::sharded_reserve(ix, capacity);
    vsbi::MutGuard g(ix);
    return ix->reserve(capacity);
}

uint64_t vsb_capacity(const vsb_index* ix) {
    if (!ix) return 0;
    if (ix->sharded) return vsbi::sharded_capacity(ix);
    return ix->capacity_atomic.load();
}
uint64_t vsb_size(const vsb_index* ix) {
    if (!ix) return 0;
    if (ix->sharded) return vsbi::sharded_size(ix);
    return ix->live_atomic.load();
}

vsb_status vsb_add(vsb_index* ix, const uint64_t* keys, const float* rows, uint64_t n) {
    if (!ix) return fail(VSB_EINVAL, "null index");
    if (ix->sharded) return vsbi::sharded_add(ix, keys, rows, n, nullptr, nullptr);
    vsbi::MutGuard g(ix);
    return ix->add(keys, rows, n, nullptr, nullptr);
}

vsb_status vsb_add_dev(vsb_index* ix, const uint64_t* keys, const float* d_rows, uint64_t n) {
    if (!ix) return fail(VSB_EINVAL, "null index");
    if (ix->sharded) return fail(VSB_EINVAL, "vsb_add_dev takes rows that already live on the index's device: add to a shard handle");
    vsbi::MutGuard g(ix);
    CU(cudaSetDevice(ix->device));
    CU(cudaDeviceSynchronize());  // the rows were produced on a stream of the caller's
    return ix->add(keys, d_rows, n, nullptr, nullptr, true);
}

vsb_status vsb_add_each(vsb_index* ix, const uint64_t* keys, const float* rows, uint64_t n, int32_t* row_status,
                        uint64_t* n_added) {
    if (!ix) return fail(VSB_EINVAL, "null index");
    std::vector<int32_t> local;
    if (row_status == nullptr) {
        local.resize((size_t)n);
        row_status = local.data();
    }
    if (ix->sharded) return vsbi::sharded_add(ix, keys, rows, n, row_status, n_added);
    vsbi::MutGuard g(ix);
    return ix->add(keys, rows, n, row_status, n_added);
}

vsb_status vsb_remove(vsb_index* ix, const uint64_t* keys, uint64_t n, uint64_t* n_removed) {
    if (!ix) return fail(VSB_EINVAL, "null index");
    if (n_removed) *n_removed = 0;
    if (n == 0) return VSB_OK;
    if (!keys) return fail(VSB_EINVAL, "null keys");
    if (ix->sharded) return vsbi::sharded_remove(ix, keys, n, n_removed);
    vsbi::MutGuard g(ix);
    return ix->remove(keys, n, n_removed);
}

int vsb_contains(const vsb_index* cix, uint64_t key) {
    if (!cix) return 0;
    vsb_index* ix = const_cast<vsb_index*>(cix);
    if (ix->sharded) return vsbi::sharded_contains(ix, key);
    std::lock_guard<std::mutex> g(ix->map_mu);
    return ix->key2slot.count(key) ? 1 : 0;
}

vsb_status vsb_build(vsb_index* ix) {
    if (!ix) return fail(VSB_EINVAL, "null index");
    if (ix->sharded) return vsbi::sharded_build(ix);
    vsbi::MutGuard g(ix);
    nvtxRangePushA("vsb_build");
    const auto t0 = std::chrono::steady_clock::now();
    const vsb_status st = ix->build();
    ix->bstats.total_ns = (uint64_t)std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now() - t0).count();
    if (st == VSB_OK) ix->publish();
    else ix->w = ix->snapshot();  // a failed build leaves the published generation in charge
    nvtxRangePop();
    return st;
}

vsb_status vsb_insert_pending(vsb_index* ix) {
    if (!ix) return fail(VSB_EINVAL, "null index");
    if (ix->sharded) return vsbi::sharded_insert_pending(ix);
    vsbi::MutGuard g(ix);
    const vsb_status st = ix->stream_insert();
    if (st == VSB_OK) ix->publish();
    return st;
}

vsb_status vsb_export_graph(vsb_index* ix, uint32_t* rows_out, uint64_t* keys_out, uint64_t* n_graphed,
                            uint32_t* stride) {
    if (!ix) return fail(VSB_EINVAL, "null index");
    if (ix->sharded) return fail(VSB_EINVAL, "vsb_export_graph works on one shard; a sharded handle has one graph per device");
    const vsbi::View v = ix->snapshot();
    if (n_graphed) *n_graphed = v.n_graphed;
    if (stride) *stride = ix->graph_stride;
    CU(cudaSetDevice(ix->device));
    if (rows_out && v.n_graphed)
        CU(cudaMemcpy(rows_out, v.gr->g.p, (size_t)v.n_graphed * ix->graph_stride * 4, cudaMemcpyDeviceToHost));
    if (keys_out && v.n_graphed) CU(cudaMemcpy(keys_out, v.st->keys.p, (size_t)v.n_graphed * 8, cudaMemcpyDeviceToHost));
    return VSB_OK;
}

vsb_status vsb_set_search_params(vsb_index* ix, const vsb_search_params* p) {
    if (!ix || !p) return fail(VSB_EINVAL, "null argument");
    if (ix->sharded) return vsbi::sharded_set_search_params(ix, p);
    {
        std::lock_guard<std::mutex> g(ix->search_mu);
        if (p->expansion_search) ix->itopk = std::min<uint32_t>(round_up(p->expansion_search, 32), 1024);
        if (p->max_iterations) ix->max_iters = p->max_iterations >= 1000000u ? 0 : p->max_iterations;  // >= 1e6: back to auto
        if (p->n_seeds) ix->n_seeds = std::min<uint32_t>(p->n_seeds, 32);
        if (p->min_graph_size) ix->min_graph_size = p->min_graph_size;
        if (p->search_width) ix->search_width = std::min<uint32_t>(p->search_width, 4);
        if (p->traversal) ix->native_traversal = p->traversal == 2;
        if (p->filter_exact_below_pct) ix->filter_min_pct = p->filter_exact_below_pct == 0xFFFFFFFFu ? 0 : std::min<uint32_t>(p->filter_exact_below_pct, 101);
    }
    if (p->stream_threshold || p->expansion_add) {
        std::lock_guard<std::mutex> g(ix->mut_mu);
        if (p->stream_threshold) ix->stream_threshold = p->stream_threshold == 0xFFFFFFFFu ? 0 : p->stream_threshold;
        if (p->expansion_add) ix->ef_add_rt = p->expansion_add;
    }
    return VSB_OK;
}

vsb_status vsb_set_instrumented(vsb_index* ix, int on) {
    if (!ix) return fail(VSB_EINVAL, "null index");
    if (ix->sharded) return vsbi::sharded_set_instrumented(ix, on);
    std::lock_guard<std::mutex> g(ix->search_mu);
    ix->instrumented = on != 0;
    return VSB_OK;
}

vsb_status vsb_set_kernel_timing(vsb_index* ix, int on) {
    if (!ix) return fail(VSB_EINVAL, "null index");
    if (ix->sharded) return vsbi::sharded_set_kernel_timing(ix, on);
    std::lock_guard<std::mutex> g(ix->search_mu);
    cudaSetDevice(ix->device);
    ix->t_resolve();
    ix->timing = on != 0;
    if (on) {
        for (int i = 0; i < vsb_index::PH_COUNT; ++i) ix->phase_ns[i] = ix->phase_launches[i] = 0;
    }
    return VSB_OK;
}

vsb_status vsb_get_stats(vsb_index* ix, vsb_stats* out) {
    if (!ix || !out) return fail(VSB_EINVAL, "null argument");
    if (ix->sharded) return vsbi::sharded_get_stats(ix, out);
    std::lock_guard<std::mutex> g(ix->search_mu);
    const vsbi::View v = ix->snapshot();
    out->kernel_launches = vsb::g_kernel_launches.load();
    out->distance_evals = ix->last_evals;
    out->parent_expansions = ix->last_parents;
    out->queries = ix->last_queries;
    out->n_slots = v.n_slots;
    out->n_graphed = v.n_graphed;
    out->graph_degree = ix->degree;
    out->row_bytes = ix->row_bytes;
    out->n_seed_rows = v.sd ? v.sd->n : 0;
    out->hbm_bytes = ix->hbm_bytes();
    cudaSetDevice(ix->device);
    ix->t_resolve();
    out->convert_ns = ix->phase_ns[vsb_index::PH_CONVERT];
    out->seed_ns = ix->phase_ns[vsb_index::PH_SEED];
    out->graph_search_ns = ix->phase_ns[vsb_index::PH_GRAPH];
    out->exact_ns = ix->phase_ns[vsb_index::PH_EXACT];
    out->merge_ns = ix->phase_ns[vsb_index::PH_MERGE];
    out->convert_launches = ix->phase_launches[vsb_index::PH_CONVERT];
    out->seed_launches = ix->phase_launches[vsb_index::PH_SEED];
    out->graph_search_launches = ix->phase_launches[vsb_index::PH_GRAPH];
    out->exact_launches = ix->phase_launches[vsb_index::PH_EXACT];
    out->merge_launches = ix->phase_launches[vsb_index::PH_MERGE];
    out->tc_launches = vsb::g_tc_launches.load();
    out->exact_certified = ix->cert_ok;
    out->exact_fallback = ix->cert_fallback;
    out->exact_scanned = ix->cert_scanned;
    out->extra_seeds = v.sd ? v.sd->extra : 0;
    return VSB_OK;
}

vsb_status vsb_get_build_stats(vsb_index* ix, vsb_build_stats* out) {
    if (!ix || !out) return fail(VSB_EINVAL, "null argument");
    if (ix->sharded) return vsbi::sharded_get_build_stats(ix, out);
    std::lock_guard<std::mutex> g(ix->mut_mu);
    *out = ix->bstats;
    return VSB_OK;
}

vsb_status vsb_get_options(vsb_index* ix, vsb_options* out) {
    if (!ix || !out) return fail(VSB_EINVAL, "null argument");
    *out = ix->opt;
    return VSB_OK;
}

vsb_status vsb_search(vsb_index* ix, const float* queries, uint64_t q, uint32_t k, uint64_t* keys, float* distances,
                      uint32_t* counts) {
    if (!ix) return fail(VSB_EINVAL, "null index");
    if (ix->sharded) return vsbi::sharded_search_host(ix, queries, q, k, keys, distances, counts, false);
    return ix->search_host(queries, q, k, keys, distances, counts, false);
}

vsb_status vsb_search_exact(vsb_index* ix, const float* queries, uint64_t q, uint32_t k, uint64_t* keys,
                            float* distances, uint32_t* counts) {
    if (!ix) return fail(VSB_EINVAL, "null index");
    if (ix->sharded) return vsbi::sharded_search_host(ix, queries, q, k, keys, distances, counts, true);
    return ix->search_host(queries, q, k, keys, distances, counts, true);
}

vsb_status vsb_search_filtered(vsb_index* ix, const float* queries, uint64_t q, uint32_t k,
                               const uint32_t* allow_bitmap, uint64_t bitmap_bits, uint64_t* keys, float* distances,
                               uint32_t* counts) {
    if (!ix) return fail(VSB_EINVAL, "null index");
    if (!allow_bitmap) return fail(VSB_EINVAL, "null bitmap");
    vsbi::HostFilters hf;
    hf.bitmaps = allow_bitmap;
    hf.n = 1;
    hf.bits = bitmap_bits;
    if (ix->sharded) return vsbi::sharded_search_host(ix, queries, q, k, keys, distances, counts, false, hf);
    return ix->search_host(queries, q, k, keys, distances, counts, false, hf);
}

vsb_status vsb_search_filtered_multi(vsb_index* ix, const float* queries, uint64_t q, uint32_t k,
                                     const uint32_t* allow_bitmaps, uint32_t n_filters, uint64_t bitmap_bits,
                                     const uint32_t* filter_of_query, uint64_t* keys, float* distances, uint32_t* counts) {
    if (!ix) return fail(VSB_EINVAL, "null index");
    if (!queries || !allow_bitmaps || !filter_of_query || !keys || !distances) return fail(VSB_EINVAL, "null argument");
    if (n_filters == 0 || n_filters > q)
        return fail(VSB_EINVAL, "n_filters = %u must be in [1, q = %llu]", n_filters, (unsigned long long)q);
    for (uint64_t i = 0; i < q; ++i)
        if (filter_of_query[i] >= n_filters)
            return fail(VSB_EINVAL, "filter_of_query[%llu] = %u >= n_filters = %u", (unsigned long long)i, filter_of_query[i],
                        n_filters);
    vsbi::HostFilters hf;
    hf.bitmaps = allow_bitmaps;
    hf.n = n_filters;
    hf.bits = bitmap_bits;
    hf.of_query = filter_of_query;
    if (ix->sharded) return vsbi::sharded_search_host(ix, queries, q, k, keys, distances, counts, false, hf);
    return ix->search_host(queries, q, k, keys, distances, counts, false, hf);
}

vsb_status vsb_search_range(vsb_index* ix, const float* queries, uint64_t q, const float* max_distance,
                            const uint32_t* allow_bitmap, uint64_t bitmap_bits, uint64_t capacity, uint64_t* keys,
                            float* distances, uint64_t* offsets) {
    if (!ix) return fail(VSB_EINVAL, "null index");
    if (!queries || !max_distance || !offsets) return fail(VSB_EINVAL, "null queries, max_distance or offsets");
    if (capacity > 0 && (!keys || !distances)) return fail(VSB_EINVAL, "null keys or distances with capacity %llu",
                                                           (unsigned long long)capacity);
    for (uint64_t i = 0; i < q; ++i)
        if (std::isnan(max_distance[i])) return fail(VSB_EINVAL, "max_distance[%llu] is NaN", (unsigned long long)i);
    vsbi::HostFilters hf;
    hf.bitmaps = allow_bitmap;
    hf.n = allow_bitmap ? 1 : 0;
    hf.bits = bitmap_bits;
    vsbi::RangeResult r;
    ST(ix->sharded ? vsbi::sharded_search_range(ix, queries, q, max_distance, hf, capacity, r)
                   : ix->search_range(queries, q, max_distance, hf, capacity, keys, distances, r));
    std::memcpy(offsets, r.off.data(), (size_t)(q + 1) * 8);
    const uint64_t total = r.off[q];
    if (total > capacity)
        return fail(VSB_EFULL, "range search: %llu rows do not fit capacity %llu", (unsigned long long)total,
                    (unsigned long long)capacity);
    if (total > 0 && !r.in_place) {
        std::memcpy(keys, r.keys.data(), (size_t)total * 8);
        std::memcpy(distances, r.dists.data(), (size_t)total * 4);
    }
    return VSB_OK;
}

vsb_status vsb_search_dev(vsb_index* ix, const float* d_queries, uint64_t q, uint32_t k, uint64_t* d_keys,
                          float* d_distances, uint32_t* d_counts, void* stream, int exact) {
    if (!ix) return fail(VSB_EINVAL, "null index");
    if (ix->sharded)
        return vsbi::sharded_search_dev(ix, d_queries, q, k, d_keys, d_distances, d_counts, static_cast<cudaStream_t>(stream), exact != 0);
    std::lock_guard<std::mutex> g(ix->search_mu);
    return ix->search_dev(d_queries, q, k, d_keys, d_distances, d_counts, static_cast<cudaStream_t>(stream), exact != 0);
}

vsb_status vsb_merge_topk_dev(const uint64_t* d_keys, const float* d_distances, uint32_t parts, uint64_t q, uint32_t k,
                              uint64_t* d_out_keys, float* d_out_distances, uint32_t* d_out_counts, int device,
                              void* stream) {
    if (!d_keys || !d_distances || !d_out_keys || !d_out_distances) return fail(VSB_EINVAL, "null buffer");
    if (parts == 0 || k == 0 || (uint64_t)parts * k > 2048) return fail(VSB_EINVAL, "parts*k must be in [1, 2048]");
    if (device >= 0) CU(cudaSetDevice(device));
    vsb::launch_merge_topk(d_keys, d_distances, parts, q, k, d_out_keys, d_out_distances, d_out_counts,
                           static_cast<cudaStream_t>(stream));
    CU(cudaGetLastError());
    return VSB_OK;
}

vsb_status vsb_merge_topk_strided_dev(const uint64_t* d_keys, const float* d_distances, uint32_t parts,
                                      uint64_t key_part_stride, uint64_t dist_part_stride, uint64_t q, uint32_t k,
                                      uint64_t* d_out_keys, float* d_out_distances, uint32_t* d_out_counts, int device,
                                      void* stream) {
    if (!d_keys || !d_distances || !d_out_keys || !d_out_distances) return fail(VSB_EINVAL, "null buffer");
    if (parts == 0 || k == 0 || (uint64_t)parts * k > 2048) return fail(VSB_EINVAL, "parts*k must be in [1, 2048]");
    if (device >= 0) CU(cudaSetDevice(device));
    vsb::launch_merge_topk(d_keys, d_distances, parts, q, k, d_out_keys, d_out_distances, d_out_counts,
                           static_cast<cudaStream_t>(stream), key_part_stride, dist_part_stride);
    CU(cudaGetLastError());
    return VSB_OK;
}

void vsb_f32_to_b1x8(const float* v, uint64_t n, uint8_t* out) {
    const uint64_t nb = (n + 7) / 8;
    for (uint64_t j = 0; j < nb; ++j) {
        uint8_t b = 0;
        for (uint64_t i = 0; i < 8 && 8 * j + i < n; ++i)
            if (v[8 * j + i] > 0.0f) b |= (uint8_t)(1u << i);
        out[j] = b;
    }
}

const char* vsb_last_error(void) { return vsbi::g_last_error.c_str(); }
const char* vsb_version(void) { return "vsb200-0.2.0"; }

}  // extern "C"
