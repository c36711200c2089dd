// sharded.cu — multi-GPU inside the library (SURVEY §8e): one process, one sub-index per device behind ONE handle.
//
// The reference's analogue is the per-partition index map of the actor (vs_index/usearch.rs:704-705): an index is
// a set of independent sub-indexes and k-NN over a disjoint union is the merge of the per-part top-k.  Here:
//   * mutations are routed by a hash of the key (streaming-friendly: no rebalancing, shards stay within a few
//     percent of each other); every shard builds its own graph over its own rows, no cross-shard edges;
//   * a search runs on every shard at once (one worker thread per device issues that device's launches);
//     the query block is copied device-to-device over NVLink, and every shard's kernels STORE their top-k straight
//     into the gather buffer of device 0 through a peer-mapped pointer — there is no all-gather, no staging copy;
//   * device 0 waits (stream-side, cudaStreamWaitEvent) for the shards' events and runs the K8 merge.
// VSB_ENCCL is returned when the devices cannot map each other's memory.
#include <algorithm>
#include <condition_variable>
#include <cstring>
#include <functional>
#include <string>
#include <thread>
#include <unordered_set>

#include "sharded.h"

namespace vsbi {

struct Worker {
    std::thread th;
    std::mutex mu;
    std::condition_variable cv;
    std::function<void()> job;
    bool has_job = false, stop = false, done = true;
};

struct Sharded {
    std::vector<vsb_index*> shards;
    std::vector<int> devices;
    std::vector<std::unique_ptr<Worker>> workers;
    std::mutex mut;     // router-level mutations
    std::mutex search;  // router-level searches (gather buffers)
    uint64_t cap_requested = 0;
    // device 0
    cudaStream_t stream0 = nullptr;
    cudaEvent_t q_ready = nullptr;
    DevBuf g_keys, g_dists, out_buf, q0;
    PinBuf pin;  // pinned staging of the merged results for pageable callers
    // per shard
    std::vector<DevBuf> qbuf, allow, fidx;
    std::vector<cudaEvent_t> done_ev;

    uint32_t G() const { return (uint32_t)shards.size(); }
    uint32_t route(uint64_t key) const {
        uint64_t z = key + 0x9E3779B97F4A7C15ull;  // splitmix64 finaliser: adjacent row ids spread evenly
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
        z ^= z >> 31;
        return (uint32_t)(z % shards.size());
    }

    // fork-join over the shard workers; returns the first failure
    vsb_status for_each(const std::function<vsb_status(uint32_t)>& fn) {
        const uint32_t g = G();
        std::vector<vsb_status> rc(g, VSB_OK);
        std::vector<std::string> msg(g);
        for (uint32_t i = 0; i < g; ++i) {
            Worker& wk = *workers[i];
            std::lock_guard<std::mutex> l(wk.mu);
            wk.job = [&, i] {
                rc[i] = fn(i);
                if (rc[i] != VSB_OK) msg[i] = vsb_last_error();
            };
            wk.has_job = true;
            wk.done = false;
            wk.cv.notify_all();
        }
        for (uint32_t i = 0; i < g; ++i) {
            Worker& wk = *workers[i];
            std::unique_lock<std::mutex> l(wk.mu);
            wk.cv.wait(l, [&] { return wk.done; });
        }
        for (uint32_t i = 0; i < g; ++i)
            if (rc[i] != VSB_OK) return fail(rc[i], "shard %u (device %d): %s", i, devices[i], msg[i].c_str());
        return VSB_OK;
    }
};

static void worker_loop(Worker* wk, int device) {
    cudaSetDevice(device);
    std::unique_lock<std::mutex> l(wk->mu);
    while (true) {
        wk->cv.wait(l, [&] { return wk->has_job || wk->stop; });
        if (wk->stop) return;
        auto job = std::move(wk->job);
        wk->has_job = false;
        l.unlock();
        job();
        l.lock();
        wk->done = true;
        wk->cv.notify_all();
    }
}

vsb_status create_sharded(const vsb_options* o, vsb_index** out) {
    *out = nullptr;
    const uint32_t G = (uint32_t)o->n_devices;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(VSB_ECUDA, "no usable CUDA device (%s): vsb200 has no CPU fallback", cudaGetErrorString(e));
    std::unordered_set<int> seen;
    for (uint32_t i = 0; i < G; ++i) {
        const int d = o->device_ids[i];
        if (d < 0 || d >= ndev) return fail(VSB_EINVAL, "device_ids[%u] = %d out of range (%d devices)", i, d, ndev);
        if (!seen.insert(d).second) return fail(VSB_EINVAL, "device %d listed twice", d);
    }
    const int dev0 = o->device_ids[0];
    // every shard stores into device 0's gather buffer and reads device 0's query block: peer mapping both ways
    for (uint32_t i = 1; i < G; ++i) {
        const int d = o->device_ids[i];
        int a = 0, b = 0;
        cudaDeviceCanAccessPeer(&a, d, dev0);
        cudaDeviceCanAccessPeer(&b, dev0, d);
        if (!a || !b) return fail(VSB_ENCCL, "devices %d and %d cannot map each other's memory (no NVLink/PCIe P2P)", dev0, d);
        cudaSetDevice(d);
        e = cudaDeviceEnablePeerAccess(dev0, 0);
        if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
        else if (e != cudaSuccess) return fail(VSB_ENCCL, "cudaDeviceEnablePeerAccess(%d -> %d): %s", d, dev0, cudaGetErrorString(e));
        cudaSetDevice(dev0);
        e = cudaDeviceEnablePeerAccess(d, 0);
        if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
        else if (e != cudaSuccess) return fail(VSB_ENCCL, "cudaDeviceEnablePeerAccess(%d -> %d): %s", dev0, d, cudaGetErrorString(e));
    }
    vsb_index* ix = new (std::nothrow) vsb_index();
    if (!ix) return fail(VSB_EOOM, "host allocation failed");
    ix->opt = *o;
    ix->dim = o->dimensions;
    ix->device = dev0;
    ix->sharded = new Sharded();
    Sharded& S = *ix->sharded;
    for (uint32_t i = 0; i < G; ++i) {
        vsb_options one = *o;
        one.n_devices = 0;
        one.device = o->device_ids[i];
        vsb_index* sh = nullptr;
        const vsb_status st = create_single(&one, &sh);
        if (st != VSB_OK) {
            destroy_sharded(ix);
            return st;
        }
        S.shards.push_back(sh);
        S.devices.push_back(one.device);
    }
    ix->metric = S.shards[0]->metric;
    ix->storage = S.shards[0]->storage;
    ix->row_bytes = S.shards[0]->row_bytes;
    ix->degree = S.shards[0]->degree;
    ix->graph_stride = S.shards[0]->graph_stride;
    S.qbuf.resize(G);
    S.allow.resize(G);
    S.fidx.resize(G);
    S.done_ev.resize(G, nullptr);
    cudaSetDevice(dev0);
    int prio_lo = 0, prio_hi = 0;
    cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
    if (cudaStreamCreateWithPriority(&S.stream0, cudaStreamNonBlocking, prio_hi) != cudaSuccess ||
        cudaEventCreateWithFlags(&S.q_ready, cudaEventDisableTiming) != cudaSuccess) {
        destroy_sharded(ix);
        return fail(VSB_ECUDA, "router stream/event creation failed");
    }
    for (uint32_t i = 0; i < G; ++i) {
        cudaSetDevice(S.devices[i]);
        if (cudaEventCreateWithFlags(&S.done_ev[i], cudaEventDisableTiming) != cudaSuccess) {
            destroy_sharded(ix);
            return fail(VSB_ECUDA, "event creation failed on device %d", S.devices[i]);
        }
        S.workers.emplace_back(new Worker());
        Worker* wk = S.workers.back().get();
        wk->th = std::thread(worker_loop, wk, S.devices[i]);
    }
    cudaSetDevice(dev0);
    *out = ix;
    return VSB_OK;
}

void destroy_sharded(vsb_index* ix) {
    if (!ix) return;
    Sharded& S = *ix->sharded;
    for (auto& wk : S.workers) {
        {
            std::lock_guard<std::mutex> l(wk->mu);
            wk->stop = true;
            wk->cv.notify_all();
        }
        if (wk->th.joinable()) wk->th.join();
    }
    for (uint32_t i = 0; i < S.shards.size(); ++i) {
        cudaSetDevice(S.devices[i]);
        cudaDeviceSynchronize();
        if (i < S.done_ev.size() && S.done_ev[i]) cudaEventDestroy(S.done_ev[i]);
        if (i < S.qbuf.size()) S.qbuf[i].release();
        if (i < S.allow.size()) S.allow[i].release();
        if (i < S.fidx.size()) S.fidx[i].release();
    }
    cudaSetDevice(ix->device);
    cudaDeviceSynchronize();
    S.g_keys.release();
    S.g_dists.release();
    S.out_buf.release();
    S.q0.release();
    if (S.q_ready) cudaEventDestroy(S.q_ready);
    if (S.stream0) cudaStreamDestroy(S.stream0);
    for (vsb_index* sh : S.shards) destroy_single(sh);
    delete ix->sharded;
    ix->sharded = nullptr;
    delete ix;
}

static uint64_t shard_capacity_for(uint64_t total, uint32_t G) {
    const uint64_t even = (total + G - 1) / G;
    return even + even / 20 + 64;  // hash routing keeps shards within a few sigma of n/G; growth covers the rest
}

vsb_status sharded_reserve(vsb_index* ix, uint64_t capacity) {
    Sharded& S = *ix->sharded;
    std::lock_guard<std::mutex> g(S.mut);
    if (capacity <= S.cap_requested) return VSB_OK;
    const uint64_t per = shard_capacity_for(capacity, S.G());
    ST(S.for_each([&](uint32_t i) {
        MutGuard l(S.shards[i]);
        return S.shards[i]->reserve(per);
    }));
    S.cap_requested = capacity;
    return VSB_OK;
}

uint64_t sharded_capacity(const vsb_index* ix) { return ix->sharded->cap_requested; }

uint64_t sharded_size(const vsb_index* ix) {
    uint64_t s = 0;
    for (vsb_index* sh : ix->sharded->shards) s += sh->live_atomic.load();
    return s;
}

int sharded_contains(vsb_index* ix, uint64_t key) {
    Sharded& S = *ix->sharded;
    vsb_index* sh = S.shards[S.route(key)];
    std::lock_guard<std::mutex> g(sh->map_mu);
    return sh->key2slot.count(key) ? 1 : 0;
}

vsb_status sharded_add(vsb_index* ix, const uint64_t* keys, const float* rows, uint64_t n, int32_t* row_status,
                       uint64_t* n_added) {
    if (n_added) *n_added = 0;
    if (n == 0) return VSB_OK;
    if (!keys || !rows) return fail(VSB_EINVAL, "null keys/rows");
    Sharded& S = *ix->sharded;
    std::lock_guard<std::mutex> g(S.mut);
    const uint32_t G = S.G();
    const uint32_t dim = ix->dim;
    if (row_status == nullptr) {
        // all-or-nothing across shards: reject before anything is written
        std::unordered_set<uint64_t> batch;
        batch.reserve((size_t)n);
        for (uint64_t i = 0; i < n; ++i) {
            if (keys[i] == 0xFFFFFFFFFFFFFFFFull) return fail(VSB_EINVAL, "key UINT64_MAX is reserved");
            if (!batch.insert(keys[i]).second || sharded_contains(ix, keys[i]))
                return fail(VSB_EDUPKEY, "duplicate key %llu", (unsigned long long)keys[i]);
        }
    }
    if (sharded_size(ix) + n > S.cap_requested && row_status == nullptr)
        return fail(VSB_EFULL, "size %llu + %llu exceeds capacity %llu: reserve capacity ahead of insertions",
                    (unsigned long long)sharded_size(ix), (unsigned long long)n, (unsigned long long)S.cap_requested);
    std::vector<std::vector<uint64_t>> idx(G);
    for (uint64_t i = 0; i < n; ++i) idx[S.route(keys[i])].push_back(i);
    std::vector<uint64_t> added(G, 0);
    ST(S.for_each([&](uint32_t s) -> vsb_status {
        const std::vector<uint64_t>& mine = idx[s];
        if (mine.empty()) return VSB_OK;
        std::vector<uint64_t> k2(mine.size());
        std::vector<float> r2(mine.size() * (size_t)dim);
        std::vector<int32_t> st2(mine.size(), VSB_OK);
        for (size_t j = 0; j < mine.size(); ++j) {
            k2[j] = keys[mine[j]];
            std::memcpy(&r2[j * dim], rows + mine[j] * dim, (size_t)dim * 4);
        }
        vsb_index* sh = S.shards[s];
        MutGuard l(sh);
        const uint64_t cap = sh->w.st ? sh->w.st->capacity : 0;
        if (sh->live + mine.size() > cap) ST(sh->reserve((sh->live + mine.size()) + (sh->live + mine.size()) / 8 + 64));
        const vsb_status rc = sh->add(k2.data(), r2.data(), mine.size(), row_status ? st2.data() : nullptr, &added[s]);
        if (row_status)
            for (size_t j = 0; j < mine.size(); ++j) row_status[mine[j]] = st2[j];
        return rc;
    }));
    if (n_added)
        for (uint32_t s = 0; s < G; ++s) *n_added += added[s];
    return VSB_OK;
}

vsb_status sharded_remove(vsb_index* ix, const uint64_t* keys, uint64_t n, uint64_t* n_removed) {
    Sharded& S = *ix->sharded;
    std::lock_guard<std::mutex> g(S.mut);
    const uint32_t G = S.G();
    std::vector<std::vector<uint64_t>> ks(G);
    for (uint64_t i = 0; i < n; ++i) ks[S.route(keys[i])].push_back(keys[i]);
    std::vector<uint64_t> removed(G, 0);
    ST(S.for_each([&](uint32_t s) -> vsb_status {
        if (ks[s].empty()) return VSB_OK;
        MutGuard l(S.shards[s]);
        return S.shards[s]->remove(ks[s].data(), ks[s].size(), &removed[s]);
    }));
    if (n_removed)
        for (uint32_t s = 0; s < G; ++s) *n_removed += removed[s];
    return VSB_OK;
}

vsb_status sharded_build(vsb_index* ix) {
    Sharded& S = *ix->sharded;
    std::lock_guard<std::mutex> g(S.mut);
    return S.for_each([&](uint32_t s) { return vsb_build(S.shards[s]); });
}

vsb_status sharded_insert_pending(vsb_index* ix) {
    Sharded& S = *ix->sharded;
    std::lock_guard<std::mutex> g(S.mut);
    return S.for_each([&](uint32_t s) { return vsb_insert_pending(S.shards[s]); });
}

vsb_status sharded_set_search_params(vsb_index* ix, const vsb_search_params* p) {
    for (vsb_index* sh : ix->sharded->shards) ST(vsb_set_search_params(sh, p));
    return VSB_OK;
}
vsb_status sharded_set_instrumented(vsb_index* ix, int on) {
    for (vsb_index* sh : ix->sharded->shards) ST(vsb_set_instrumented(sh, on));
    return VSB_OK;
}
vsb_status sharded_set_kernel_timing(vsb_index* ix, int on) {
    for (vsb_index* sh : ix->sharded->shards) ST(vsb_set_kernel_timing(sh, on));
    return VSB_OK;
}

vsb_status sharded_get_stats(vsb_index* ix, vsb_stats* out) {
    std::memset(out, 0, sizeof *out);
    bool first = true;
    for (vsb_index* sh : ix->sharded->shards) {
        vsb_stats s;
        ST(vsb_get_stats(sh, &s));
        uint64_t* acc = reinterpret_cast<uint64_t*>(out);
        const uint64_t* one = reinterpret_cast<const uint64_t*>(&s);
        const size_t nf = sizeof(vsb_stats) / 8;
        for (size_t f = 0; f < nf; ++f) acc[f] += one[f];
        if (!first) {  // not additive: process-wide counters and per-shard constants
            out->kernel_launches = s.kernel_launches;
            out->tc_launches = s.tc_launches;
            out->graph_degree = s.graph_degree;
            out->row_bytes = s.row_bytes;
            out->queries = s.queries;
        }
        first = false;
    }
    // phase times are per-device and concurrent: report the mean over the shards
    const uint64_t G = ix->sharded->G();
    for (uint64_t* f : {&out->convert_ns, &out->seed_ns, &out->graph_search_ns, &out->exact_ns, &out->merge_ns,
                        &out->convert_launches, &out->seed_launches, &out->graph_search_launches, &out->exact_launches,
                        &out->merge_launches})
        *f /= G;
    out->hbm_bytes += ix->sharded->g_keys.bytes + ix->sharded->g_dists.bytes + ix->sharded->out_buf.bytes + ix->sharded->q0.bytes;
    return VSB_OK;
}

vsb_status sharded_get_build_stats(vsb_index* ix, vsb_build_stats* out) {
    std::memset(out, 0, sizeof *out);
    for (vsb_index* sh : ix->sharded->shards) {
        vsb_build_stats s;
        ST(vsb_get_build_stats(sh, &s));
        out->rows += s.rows;
        out->allpairs_rows += s.allpairs_rows;
        out->allpairs_flops += s.allpairs_flops;
        out->stream_rows += s.stream_rows;
        out->stream_evals += s.stream_evals;
        out->stream_parents += s.stream_parents;
        out->refine_rows += s.refine_rows;
        out->refine_evals += s.refine_evals;
        out->refine_parents += s.refine_parents;
        // shards build concurrently: times are the slowest shard's
        out->allpairs_ns = std::max(out->allpairs_ns, s.allpairs_ns);
        out->prune_ns = std::max(out->prune_ns, s.prune_ns);
        out->stream_ns = std::max(out->stream_ns, s.stream_ns);
        out->refine_ns = std::max(out->refine_ns, s.refine_ns);
        out->seeds_ns = std::max(out->seeds_ns, s.seeds_ns);
        out->compact_ns = std::max(out->compact_ns, s.compact_ns);
        out->total_ns = std::max(out->total_ns, s.total_ns);
        out->traversal_row_bytes = s.traversal_row_bytes;
    }
    return VSB_OK;
}

// Common body: queries are in `d_q` on device 0, valid once `ready` has fired; results land in o_* on device 0,
// ordered on `s0`.  hf: optional host bitmaps and per-query bitmap indices (uploaded to every shard); pop: admissible
// rows of each bitmap, split evenly over the shards for the route selection.
static vsb_status fan_out(vsb_index* ix, const float* d_q, cudaEvent_t ready, uint64_t nq, uint32_t k, uint64_t* o_keys,
                          float* o_dists, uint32_t* o_counts, cudaStream_t s0, bool exact, const HostFilters& hf,
                          const std::vector<uint64_t>& pop) {
    Sharded& S = *ix->sharded;
    const uint32_t G = S.G();
    const int dev0 = S.devices[0];
    if ((uint64_t)G * k > 2048) return fail(VSB_EINVAL, "shards*k must be <= 2048 for the merge");
    CU(cudaSetDevice(dev0));
    CU(S.g_keys.ensure((size_t)G * nq * k * 8, true));
    CU(S.g_dists.ensure((size_t)G * nq * k * 4, true));
    uint64_t* gk = S.g_keys.as<uint64_t>();
    float* gd = S.g_dists.as<float>();
    const size_t q_bytes = (size_t)nq * ix->dim * 4;
    const size_t allow_words = hf.bitmaps ? (size_t)((hf.bits + 31) / 32) * hf.n : 0;
    std::vector<uint64_t> shard_pop(pop.size());
    for (size_t f = 0; f < pop.size(); ++f) shard_pop[f] = pop[f] / G;
    ST(S.for_each([&](uint32_t i) -> vsb_status {
        vsb_index* sh = S.shards[i];
        CU(cudaSetDevice(S.devices[i]));
        std::lock_guard<std::mutex> l(sh->search_mu);
        cudaStream_t si = sh->stream;
        CU(cudaStreamWaitEvent(si, ready, 0));
        const float* q_local = d_q;
        if (i != 0) {
            CU(S.qbuf[i].ensure(q_bytes));
            CU(cudaMemcpyPeerAsync(S.qbuf[i].p, S.devices[i], d_q, dev0, q_bytes, si));  // NVLink, device to device
            q_local = S.qbuf[i].as<float>();
        }
        Filters f;
        if (hf.bitmaps) {
            CU(S.allow[i].ensure(std::max<size_t>(allow_words * 4, 16)));
            CU(cudaMemcpyAsync(S.allow[i].p, hf.bitmaps, allow_words * 4, cudaMemcpyHostToDevice, si));
            f.d_allow = S.allow[i].as<uint32_t>();
            f.bits = hf.bits;
            f.n = hf.n;
            f.pop = shard_pop.data();
            if (hf.of_query) {
                CU(S.fidx[i].ensure((size_t)nq * 4));
                CU(cudaMemcpyAsync(S.fidx[i].p, hf.of_query, (size_t)nq * 4, cudaMemcpyHostToDevice, si));
                f.d_fidx = S.fidx[i].as<uint32_t>();
                f.h_fidx = hf.of_query;
            }
        }
        // the shard's last kernel stores into device 0's gather buffer (peer-mapped): part i of [G][nq][k]
        ST(sh->search_dev(q_local, nq, k, gk + (size_t)i * nq * k, gd + (size_t)i * nq * k, nullptr, si, exact, f));
        CU(cudaEventRecord(S.done_ev[i], si));
        return VSB_OK;
    }));
    CU(cudaSetDevice(dev0));
    for (uint32_t i = 0; i < G; ++i) CU(cudaStreamWaitEvent(s0, S.done_ev[i], 0));
    vsb::launch_merge_topk(gk, gd, G, nq, k, o_keys, o_dists, o_counts, s0);
    CU(cudaGetLastError());
    return VSB_OK;
}

vsb_status sharded_search_dev(vsb_index* ix, const float* d_queries, uint64_t nq, uint32_t k, uint64_t* d_keys,
                              float* d_dists, uint32_t* d_counts, cudaStream_t stream, bool exact) {
    if (nq == 0) return VSB_OK;
    if (k == 0) return fail(VSB_EINVAL, "k must be > 0");
    if (!d_queries || !d_keys || !d_dists) return fail(VSB_EINVAL, "null buffer");
    Sharded& S = *ix->sharded;
    std::lock_guard<std::mutex> g(S.search);
    CU(cudaSetDevice(S.devices[0]));
    CU(cudaEventRecord(S.q_ready, stream));
    return fan_out(ix, d_queries, S.q_ready, nq, k, d_keys, d_dists, d_counts, stream, exact, HostFilters(), {});
}

vsb_status sharded_search_host(vsb_index* ix, const float* queries, uint64_t nq, uint32_t k, uint64_t* keys, float* dists,
                               uint32_t* counts, bool exact, const HostFilters& hf) {
    if (nq == 0) return VSB_OK;
    if (k == 0) return fail(VSB_EINVAL, "k must be > 0");
    if (!queries || !keys || !dists) return fail(VSB_EINVAL, "null buffer");
    Sharded& S = *ix->sharded;
    std::lock_guard<std::mutex> g(S.search);
    CU(cudaSetDevice(S.devices[0]));
    const size_t q_bytes = (size_t)nq * ix->dim * 4;
    const size_t kb = (size_t)nq * k * 8, db = (size_t)nq * k * 4, cb = (size_t)nq * 4;
    auto al = [](size_t v) { return (v + 255) / 256 * 256; };
    CU(S.q0.ensure(q_bytes, true));
    CU(S.out_buf.ensure(al(kb) + al(db) + al(cb)));
    uint64_t* ok = S.out_buf.as<uint64_t>();
    float* od = reinterpret_cast<float*>(S.out_buf.as<uint8_t>() + al(kb));
    uint32_t* oc = reinterpret_cast<uint32_t*>(S.out_buf.as<uint8_t>() + al(kb) + al(db));
    CU(cudaMemcpyAsync(S.q0.p, queries, q_bytes, cudaMemcpyHostToDevice, S.stream0));
    CU(cudaEventRecord(S.q_ready, S.stream0));
    std::vector<uint64_t> pop(hf.bitmaps ? hf.n : 0, 0);
    const size_t words = (size_t)((hf.bits + 31) / 32);
    for (size_t f = 0; f < pop.size(); ++f)
        for (size_t i = 0; i < words; ++i) pop[f] += (uint64_t)__builtin_popcount(hf.bitmaps[f * words + i]);
    ST(fan_out(ix, S.q0.as<float>(), S.q_ready, nq, k, ok, od, oc, S.stream0, exact, hf, pop));
    vsbi::HostReadback rb(S.pin, S.stream0);  // pageable destinations are staged (index_impl.h)
    CU(rb.reserve(al(kb) + al(db) + al(cb)));
    CU(rb.copy(keys, ok, kb));
    CU(rb.copy(dists, od, db));
    if (counts) CU(rb.copy(counts, oc, cb));
    CU(rb.finish());
    return VSB_OK;
}

vsb_status sharded_save(vsb_index* ix, const char* path) {
    Sharded& S = *ix->sharded;
    std::lock_guard<std::mutex> g(S.mut);
    return S.for_each([&](uint32_t s) {
        const std::string p = std::string(path) + ".shard" + std::to_string(s);
        return save_single(S.shards[s], p.c_str());
    });
}

}  // namespace vsbi
