// index_impl.h — the index object behind the C ABI of include/vsb200.h (internal to libvsb200).
//
// Mirrors what `ThreadedUsearchIndex` + `usearch::Index` are to the reference
// (crates/vector-store/src/vs_index/usearch.rs:162-251): opaque u64 keys, unique keys (multi=false), explicit
// capacity (`reserve`), add / remove / search, a live count.
//
// Concurrency (replaces the reader/writer gate `mod operation`, usearch.rs:515-624):
//   * every search works on a VIEW: shared_ptr's to the row store, the graph and the entry-point sample plus the
//     counts that were current when the search began.  A view is immutable in everything a search depends on;
//   * mutators (reserve / add / remove / build / insert_pending) are serialised by `mut_mu`, work on their own
//     stream and their own scratch, prepare NEW buffers where a buffer has to change shape (reserve, compaction,
//     graph rebuild, seed resampling) and PUBLISH the next view with a pointer swap under `pub_mu` (held for
//     nanoseconds).  Searches never wait for a mutator; buffers die with the last view that references them;
//   * the only in-place writes to published buffers are single 32-bit words whose old and new values are both
//     valid for a reader: tombstone bits (remove) and reverse-edge slots of existing graph rows (K7);
//   * searches are serialised among themselves by `search_mu` (they share one scratch set and one GPU).
//
// HBM layout (per shard):
//   Store : rows [cap][row_bytes], sq/nrm [cap] f32, keys [cap] u64, deny [cap/32] u32 (+ bf16 / int8 traversal copies)
//   Graph : [cap][stride] u32 fixed-degree neighbour rows; rows >= n_graphed are the brute-force tail
//   Seeds : contiguous copy of the entry-point sample ("upper layer")
#pragma once
#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <memory>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/vsb200.h"
#include "kernels.h"

namespace vsbi {

vsb_status fail(vsb_status st, const char* fmt, ...);

#define CU(expr)                                                                                             \
    do {                                                                                                     \
        cudaError_t e_ = (expr);                                                                             \
        if (e_ != cudaSuccess)                                                                               \
            return vsbi::fail(e_ == cudaErrorMemoryAllocation ? VSB_EOOM : VSB_ECUDA, "%s: %s (%s:%d)", #expr, \
                              cudaGetErrorString(e_), __FILE__, __LINE__);                                   \
    } while (0)

#define ST(expr)                     \
    do {                             \
        vsb_status s_ = (expr);      \
        if (s_ != VSB_OK) return s_; \
    } while (0)

// Device memory comes from the device's stream-ordered pool (cudaMallocAsync on a dedicated allocator stream that is
// drained before the pointer is handed out, so the block is valid on every stream) and goes back with cudaFreeAsync:
// cudaMalloc / cudaFree serialise on the context and cudaFree waits for the whole device, which would stall every
// running search whenever a mutator drops a temporary.  The pool keeps freed blocks (release threshold = max), so a
// steady mutation stream allocates without ever reaching the driver.  Callers release a buffer only after the work
// that used it has been synchronised (every mutator phase ends with an event wait); growing a scratch buffer that
// un-synchronised kernels may still read drains the device first.  `plain` buffers (cudaMalloc) are for memory that
// other devices or processes map: the router's gather buffers and the IPC exchange.
cudaStream_t pool_stream(int device);  // index.cu

// Experiment knob (VSB_PLAIN_ALLOC_MB): buffers of at least this many MB come from cudaMalloc instead of the pool
// (page size / TLB reach of a 15 GB row store).  0 = never (default).
inline size_t big_alloc_threshold() {
    static const size_t t = [] {
        const char* e = getenv("VSB_PLAIN_ALLOC_MB");
        const size_t mb = e ? (size_t)strtoull(e, nullptr, 10) : 0;
        return mb ? mb << 20 : ~(size_t)0;
    }();
    return t;
}

struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
    int dev = -1;
    bool plain = false;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    DevBuf(DevBuf&& o) noexcept : p(o.p), bytes(o.bytes), dev(o.dev), plain(o.plain) {
        o.p = nullptr;
        o.bytes = 0;
    }
    DevBuf& operator=(DevBuf&& o) noexcept {
        if (this != &o) {
            release();
            p = o.p;
            bytes = o.bytes;
            dev = o.dev;
            plain = o.plain;
            o.p = nullptr;
            o.bytes = 0;
        }
        return *this;
    }
    ~DevBuf() { release(); }
    void release() {
        if (p) {
            int cur = -1;
            cudaGetDevice(&cur);
            if (cur != dev) cudaSetDevice(dev);
            if (plain) cudaFree(p);
            else cudaFreeAsync(p, pool_stream(dev));
            if (cur != dev && cur >= 0) cudaSetDevice(cur);
        }
        p = nullptr;
        bytes = 0;
    }
    // exact-size allocation on the current device (contents undefined)
    cudaError_t alloc(size_t want, bool plain_memory = false) {
        release();
        const size_t sz = want ? want : 16;
        cudaGetDevice(&dev);
        plain = plain_memory || sz >= big_alloc_threshold();
        cudaError_t e;
        if (plain) {
            e = cudaMalloc(&p, sz);
        } else {
            cudaStream_t ps = pool_stream(dev);
            e = cudaMallocAsync(&p, sz, ps);
            if (e == cudaSuccess) e = cudaStreamSynchronize(ps);
        }
        if (e != cudaSuccess) {
            p = nullptr;
            return e;
        }
        bytes = sz;
        return cudaSuccess;
    }
    // grow-only scratch (contents not preserved)
    cudaError_t ensure(size_t want, bool plain_memory = false) {
        if (want <= bytes) return cudaSuccess;
        if (p) cudaDeviceSynchronize();  // kernels of an un-synchronised search may still read the old block
        return alloc(want + want / 4, plain_memory);
    }
    template <class T>
    T* as() const { return static_cast<T*>(p); }
};

inline uint32_t round_up(uint32_t v, uint32_t m) { return (v + m - 1) / m * m; }

// Device -> host copies never go straight into PAGEABLE memory: for such a destination cudaMemcpyAsync waits INSIDE the
// call — holding the context lock — until the stream has reached the copy, and every other thread's CUDA call queues up
// behind it.  Measured in config C5: while a refinement pass read back its 16-byte work counters after each K4 launch,
// every concurrent batch-1 search took one whole launch (21 ms) instead of 0.3 ms.  Pageable destinations are staged
// through a pinned buffer (the async copy returns at once, the wait is a cudaStreamSynchronize, which blocks nobody
// else); destinations the caller pinned (cudaHostAlloc / cudaHostRegister, e.g. bench.py's e2e buffers) are written
// directly.
struct PinBuf {
    void* p = nullptr;
    size_t bytes = 0;
    PinBuf() = default;
    PinBuf(const PinBuf&) = delete;
    PinBuf& operator=(const PinBuf&) = delete;
    ~PinBuf() {
        if (p) cudaFreeHost(p);
    }
    cudaError_t ensure(size_t want) {
        if (want <= bytes) return cudaSuccess;
        if (p) cudaFreeHost(p);
        p = nullptr;
        bytes = 0;
        const size_t sz = std::max<size_t>(want + want / 4, 4096);
        const cudaError_t e = cudaHostAlloc(&p, sz, cudaHostAllocDefault);
        if (e == cudaSuccess) bytes = sz;
        else p = nullptr;
        return e;
    }
};

inline bool host_is_pinned(const void* ptr) {
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, ptr) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return at.type == cudaMemoryTypeHost || at.type == cudaMemoryTypeManaged;
}

// A batch of device -> host copies on one stream followed by one synchronisation.  reserve() the total first.
class HostReadback {
    PinBuf& pin;
    cudaStream_t s;
    struct Item {
        void* dst;
        size_t off, bytes;
    };
    Item items[4];
    int n_items = 0;
    size_t used = 0;

   public:
    HostReadback(PinBuf& pin_, cudaStream_t s_) : pin(pin_), s(s_) {}
    cudaError_t reserve(size_t total) { return pin.ensure(total + 4 * 256); }
    cudaError_t copy(void* dst, const void* src_dev, size_t bytes) {
        if (bytes == 0) return cudaSuccess;
        if (host_is_pinned(dst)) return cudaMemcpyAsync(dst, src_dev, bytes, cudaMemcpyDeviceToHost, s);
        if (n_items == 4 || used + bytes > pin.bytes) return cudaErrorInvalidValue;
        items[n_items++] = Item{dst, used, bytes};
        const cudaError_t e = cudaMemcpyAsync(static_cast<uint8_t*>(pin.p) + used, src_dev, bytes, cudaMemcpyDeviceToHost, s);
        used += (bytes + 255) / 256 * 256;
        return e;
    }
    cudaError_t finish() {
        const cudaError_t e = cudaStreamSynchronize(s);
        if (e != cudaSuccess) return e;
        for (int i = 0; i < n_items; ++i) std::memcpy(items[i].dst, static_cast<uint8_t*>(pin.p) + items[i].off, items[i].bytes);
        n_items = 0;
        used = 0;
        return cudaSuccess;
    }
};

// capacity-sized per-row arrays; reserve / compaction build a NEW store and publish it
struct Store {
    uint64_t capacity = 0;
    DevBuf rows, sq, nrm, keys, deny;
    DevBuf rows16, sq16, nrm16;  // VSB_FLAG_BF16_TRAVERSAL: bf16 copy of the rows for K4
    DevBuf rows8, sq8, nrm8;     // VSB_FLAG_I8_TRAVERSAL: scaled-int8 copy
    size_t bytes() const {
        return rows.bytes + sq.bytes + nrm.bytes + keys.bytes + deny.bytes + rows16.bytes + sq16.bytes + nrm16.bytes +
               rows8.bytes + sq8.bytes + nrm8.bytes;
    }
};

struct Graph {
    DevBuf g;  // [cap_rows][stride] u32
    uint64_t cap_rows = 0;
};

struct Seeds {
    DevBuf rows, sq, nrm, slots;
    DevBuf rows16, sq16, nrm16;  // bf16 shadow of the seed block (f32 storage only)
    uint32_t n = 0, extra = 0;
    uint32_t sampled_rows = 0;  // rows the sample was drawn from (the streaming insert re-samples when the graph has doubled)
    size_t bytes() const { return rows.bytes + sq.bytes + nrm.bytes + slots.bytes + rows16.bytes + sq16.bytes + nrm16.bytes; }
};

struct View {
    std::shared_ptr<Store> st;
    std::shared_ptr<Graph> gr;
    std::shared_ptr<Seeds> sd;
    uint32_t n_slots = 0, n_graphed = 0;
    bool any_tombstone = false;
};

// per-caller-class scratch: one set for searches (under search_mu), one for mutators (under mut_mu)
struct Scratch {
    DevBuf q_in, q_rows, q_sq, q_nrm, q16_rows, q16_sq, q16_nrm, q8_rows, q8_sq, q8_nrm;
    DevBuf part, seed_part, tmp_keys, tmp_dists, rr_packed, counters, allow;
    DevBuf cert_state, fb_map, fb_rows, fb_sq, fb_nrm, fb_fidx;  // certified exact search
    // filtered searches whose bitmaps take different routes: each route's queries, bitmap indices and results
    DevBuf rt_map, rt_rows, rt_sq, rt_nrm, rt_fidx, rt_keys, rt_dists, rt_counts;
    DevBuf thr_part, thr, thr_cnt;                       // sampled list bounds of the all-pairs build (exact_block)
    PinBuf pin;                                          // pinned staging of this caller class's read-backs
    size_t bytes() const {
        const DevBuf* all[] = {&q_in, &q_rows, &q_sq, &q_nrm, &q16_rows, &q16_sq, &q16_nrm, &q8_rows, &q8_sq, &q8_nrm, &part,
                               &seed_part, &tmp_keys, &tmp_dists, &rr_packed, &counters, &allow, &cert_state, &fb_map,
                               &fb_rows, &fb_sq, &fb_nrm, &fb_fidx, &rt_map, &rt_rows, &rt_sq, &rt_nrm, &rt_fidx,
                               &rt_keys, &rt_dists, &rt_counts, &thr_part, &thr, &thr_cnt};
        size_t s = 0;
        for (auto* b : all) s += b->bytes;
        return s;
    }
};

// A filtered call as the caller hands it over: n bitmaps over (key & 2^48-1) back to back in host memory,
// ceil(bits / 32) words each; query i is filtered by bitmap of_query[i] (null: bitmap 0 for every query).
struct HostFilters {
    const uint32_t* bitmaps = nullptr;  // null: unfiltered search
    uint32_t n = 0;
    uint64_t bits = 0;
    const uint32_t* of_query = nullptr;
};

// The same call once the bitmaps are on the device: what search_dev needs to route and run it.
struct Filters {
    const uint32_t* d_allow = nullptr;  // [n][ceil(bits / 32)] (null: unfiltered search)
    uint64_t bits = 0;
    uint32_t n = 0;
    const uint32_t* d_fidx = nullptr;  // [nq] bitmap index per query (null: bitmap 0 for every query)
    const uint32_t* h_fidx = nullptr;  // host copy of d_fidx (route selection); null exactly when d_fidx is
    const uint64_t* pop = nullptr;     // host [n]: admissible rows per bitmap (route selection)
};

struct Sharded;  // sharded.cu: the multi-device router behind the same handle type

}  // namespace vsbi

struct vsb_index {
    // ---- immutable after vsb_create ----
    vsb_options opt{};
    uint32_t dim = 0, row_bytes = 0, row_bytes16 = 0, row_bytes8 = 0;
    int metric = 0, storage = 0, device = 0, sm_count = 148;
    uint32_t degree = 32, graph_stride = 32, k_init = 64;
    bool trav16 = false, trav8 = false;
    uint32_t rr_mult8 = 4;
    bool tc_enabled = true;       // tcgen05 path for the dense distance tiles (VSB_DISABLE_TC=1 turns it off)
    uint32_t tc_min_rows = 8192;  // below this the SIMT K1 is used (launch + pipeline fill dominate)
    bool cert_enabled = true;     // VSB_DISABLE_CERT=1: exact f32 search always on the SIMT tiles
    uint32_t cert_kp = 128, cert_kp16 = 32;
    bool reach_fix = true;
    uint32_t reach_budget = 1024;
    uint32_t allpairs_max = 262144, allpairs_prefix = 131072;
    // refinement passes at the end of vsb_build (VSB_REFINE_PASSES).  0 by default: with detour-pruned K7 links a pass buys
    // ~2 % QPS at equal recall and costs 1.7x the rest of the build (10 M x 768: 5.7 s -> 16.6 s, profiles/r2_*)
    uint32_t refine_passes = 0;
    bool sampled_bounds = true;  // all-pairs kNN lists start from sampled bounds (VSB_TC_SAMPLED_BOUNDS=0 turns it off)
    bool churn_refine = true;  // one refinement pass after 10 % of the graph has churned (VSB_CHURN_REFINE=0 turns it off)
    uint32_t build_search_width = 4;  // parents per K4 iteration in the streaming insert / refinement searches (VSB_BUILD_SW): 10 M x 768 build 6.1 s at 2, 5.6 s at 4, same graph quality
    vsbi::Sharded* sharded = nullptr;  // n_devices > 1: every entry point forwards to the router (owned; sharded.cu)

    // ---- published state ----
    std::mutex pub_mu;
    vsbi::View cur;
    std::atomic<uint64_t> live_atomic{0}, capacity_atomic{0};
    vsbi::View snapshot() {
        std::lock_guard<std::mutex> g(pub_mu);
        return cur;
    }

    // ---- search side (search_mu) ----
    std::mutex search_mu;
    cudaStream_t stream = nullptr;  // default search stream (high priority)
    vsbi::Scratch ss;
    struct InFlight {
        cudaEvent_t done;
        cudaStream_t stream;
        vsbi::View view;
    };
    std::deque<InFlight> inflight;  // views of searches whose kernels may still be running
    // host-pointer searches of >= 1024 queries: two staging slots with their own copy stream (search_host)
    struct HostSlot {
        vsbi::DevBuf buf;
        vsbi::PinBuf pin;
        cudaStream_t cs = nullptr;
        cudaEvent_t ev_in = nullptr, ev_done = nullptr;
        bool busy = false;
    };
    std::mutex slot_mu;
    std::condition_variable slot_cv;
    HostSlot slots[2];
    // runtime parameters (set under search_mu)
    uint32_t itopk = 64, max_iters = 0, n_seeds = 32, min_graph_size = 4096, search_width = 1;
    uint32_t filter_min_pct = 2;  // filtered ANN: below this share of admissible rows the exact bitmap scan is used
    bool native_traversal = false;  // runtime override of VSB_FLAG_*_TRAVERSAL: K4 walks the stored rows themselves
    bool instrumented = false;
    uint64_t last_evals = 0, last_parents = 0, last_queries = 0;
    uint64_t cert_ok = 0, cert_fallback = 0, cert_scanned = 0;
    enum Phase { PH_CONVERT = 0, PH_SEED, PH_GRAPH, PH_EXACT, PH_MERGE, PH_COUNT };
    bool timing = false;
    struct Timed {
        cudaEvent_t a, b;
        int phase;
    };
    std::vector<Timed> timed;
    uint64_t phase_ns[PH_COUNT] = {0, 0, 0, 0, 0};
    uint64_t phase_launches[PH_COUNT] = {0, 0, 0, 0, 0};
    void t_begin(int phase, cudaStream_t s);
    void t_end(cudaStream_t s);
    void t_resolve();
    vsb_status begin_search(cudaStream_t s);
    vsb_status end_search(cudaStream_t s, const vsbi::View& v);
    void reap_inflight(bool wait);

    // ---- mutator side (mut_mu) ----
    std::mutex mut_mu;
    cudaStream_t mstream = nullptr;  // the stream the running mutator uses: mstream_green while searches are active
    cudaStream_t mstream_full = nullptr, mstream_green = nullptr;  // low priority on all SMs / green context (green.cu)
    void* green_ctx = nullptr;
    uint32_t green_sms = 0;
    std::atomic<int64_t> last_search_ns{0};  // steady-clock time of the latest search (mutators pick their stream by it)
    vsbi::Scratch ms;
    vsbi::View w;                    // the mutators' working view; `publish()` makes it current
    uint64_t live = 0;
    std::mutex map_mu;               // key2slot readers (vsb_contains) vs the mutator that edits it
    std::unordered_map<uint64_t, uint32_t> key2slot;
    std::vector<uint32_t> h_deny;
    uint64_t n_tombstones = 0;
    uint64_t churn_since_refine = 0;  // rows streamed in + rows removed since the graph was last (re)built / refined
    uint32_t stream_threshold = 4096; // un-graphed tail rows that trigger an automatic streaming insert
    bool in_build = false;
    uint32_t ef_add_rt = 0;           // 0 = options.expansion_add
    // build accounting (vsb_build_stats): CUDA-event phase times + the algorithmic work of each phase
    vsb_build_stats bstats{};
    void publish() {
        std::lock_guard<std::mutex> g(pub_mu);
        cur = w;
        live_atomic.store(live);
        capacity_atomic.store(w.st ? w.st->capacity : 0);
    }

    size_t hbm_bytes();
    vsb::RowsView rows_view(const vsbi::View& v) const;

    vsb_status new_store(uint64_t cap, std::shared_ptr<vsbi::Store>& out);
    vsb_status reserve(uint64_t cap);
    vsb_status add(const uint64_t* k, const float* r, uint64_t n, int32_t* row_status, uint64_t* n_added,
                   bool rows_on_device = false);
    vsb_status remove(const uint64_t* k, uint64_t n, uint64_t* removed);
    vsb_status compact(bool keep_graph);
    vsb_status build();
    vsb_status graph_from_knn(const uint64_t* knn, uint32_t n, uint32_t kin, const uint32_t* deny_bm);
    vsb_status refine_graph();
    vsb_status stream_insert();
    vsb_status sample_seeds(uint32_t n_rows, bool ensure_reach = true);

    // search building blocks: run on stream `s` with scratch `sc` against view `v`
    vsb_status exact_block(const vsbi::View& v, vsbi::Scratch& sc, const vsb::RowsView& q, const vsb::RowsView& x,
                           uint32_t x_lo, uint32_t x_hi, const uint32_t* deny_bm, const uint64_t* key_arr,
                           const uint32_t* allow_bm, uint64_t allow_bits, const uint32_t* allow_of_q, uint32_t k,
                           uint64_t* out_keys,
                           float* out_dists, uint32_t* out_counts, uint64_t* out_packed, int64_t self_base,
                           cudaStream_t s, bool approx_ok, const vsb::RowsView* shadow_q = nullptr,
                           const vsb::RowsView* shadow_x = nullptr);
    struct GraphRun {
        uint32_t itopk = 64, max_iters = 0, n_seeds = 32, search_width = 1;
        bool count = false;  // instrumented launch (E / P counters)
        bool native = false; // ignore the traversal copies
        const uint32_t* allow = nullptr;  // filtered ANN: bitmap over (key & 2^48-1)
        uint64_t allow_bits = 0;
        const uint32_t* allow_of_q = nullptr;  // [nb] bitmap index per query (null: bitmap 0)
    };
    vsb_status graph_block(const vsbi::View& v, vsbi::Scratch& sc, const GraphRun& run, const vsb::RowsView& qv,
                           uint32_t nb, uint32_t k, uint64_t* g_keys, float* g_dists, uint32_t* counts_out,
                           uint64_t* packed_out, const vsb::RowsView* q16_in, cudaStream_t s, long long self_base,
                           bool timed_phases, uint64_t* evals_out = nullptr, uint64_t* parents_out = nullptr);
    // one chunk of converted queries on one route: the graph (with the brute-force tail and the K8 merge) or the
    // exact scan; allow_bm != null filters it (per query through allow_of_q)
    vsb_status search_block(const vsbi::View& v, vsbi::Scratch& sc, const vsb::RowsView& qv, uint32_t nb, uint32_t k,
                            uint64_t* o_keys, float* o_dists, uint32_t* o_counts, cudaStream_t s, bool graph,
                            const uint32_t* allow_bm, uint64_t allow_bits, const uint32_t* allow_of_q);
    vsb_status search_dev(const float* d_q, uint64_t nq, uint32_t k, uint64_t* d_keys, float* d_dists,
                          uint32_t* d_counts, cudaStream_t s, bool exact, const vsbi::Filters& f = vsbi::Filters());
    vsb_status search_host(const float* queries, uint64_t nq, uint32_t k, uint64_t* keys_out, float* dists_out,
                           uint32_t* counts_out, bool exact, const vsbi::HostFilters& hf = vsbi::HostFilters());
};

namespace vsbi {
// green.cu
bool make_green_stream(int device, unsigned reserve_sms, int priority, cudaStream_t* stream_out, void** ctx_out,
                       unsigned* sms_out);
void destroy_green(void* ctx);
// Mutator entry: takes mut_mu and picks the stream — the green-context stream (a few SMs stay free for searches) if a
// search ran within the last two seconds, the whole device otherwise (a bulk build with nobody searching).
struct MutGuard {
    std::lock_guard<std::mutex> lock;
    explicit MutGuard(vsb_index* ix);
};
uint32_t storage_row_bytes(int storage, uint32_t dim);
// index.cu: creates an un-sharded handle on opt.device (shared by vsb_create, the router and vsb_load)
vsb_status create_single(const vsb_options* o, vsb_index** out);
void destroy_single(vsb_index* ix);
}  // namespace vsbi
