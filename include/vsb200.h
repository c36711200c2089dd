/*
 * vsb200.h — C ABI of libvsb200.so, the B200-native (sm_100a) ANN engine that
 * replaces the USearch index behind scylladb/vector-store's index actor.
 *
 * Drop-in boundary.  In the reference the engine is reached through the
 * crate-private trait `UsearchIndex` (crates/vector-store/src/vs_index/usearch.rs:142-160)
 * whose only implementation forwards to the `usearch` crate's cxx FFI
 * (usearch.rs:169-251).  Every entry point below names the reference call it
 * replaces.  All functions are thread-safe on one handle, copy their inputs
 * before returning, never call back into the host and never fall back to a CPU
 * path: if no CUDA device is usable `vsb_create` fails with VSB_ECUDA.
 *
 * Conventions
 *   - keys are opaque u64 (reference PrimaryId: 16-bit epoch | 48-bit row id,
 *     table/primary_id.rs:27-62); all 64 bits are stored and returned.
 *   - vectors cross the boundary as row-major f32, exactly like
 *     `usearch::Index::add(key, &[f32])` / `search(&[f32], k)`; the cast to the
 *     storage scalar (f32/f16/bf16/i8/b1) happens on the device, on add AND on
 *     the query.
 *   - results: per query `k` slots, ascending by (distance, key); unused slots
 *     hold key = UINT64_MAX and distance = +inf; `counts[q]` = valid entries.
 *   - k (the reference's `Limit`, an unbounded NonZeroUsize): vsb_search accepts k <= 1024 whether or not
 *     un-graphed rows exist (of the brute-force tail at most its 200 best rows take part in a result);
 *     vsb_search_exact and the exact bitmap scan accept k <= 200 and return VSB_EINVAL above that.
 *   - "_dev" variants take DEVICE pointers and a `cudaStream_t` (as void*) and
 *     never synchronise; they are what bench.py times for the in-HBM number
 *     and what the multi-GPU path feeds straight into the NCCL all-gather.
 */
#ifndef VSB200_H
#define VSB200_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct vsb_index vsb_index;

typedef enum {
    VSB_OK = 0,
    VSB_EINVAL = 1,  /* bad argument / unsupported option combination          */
    VSB_EDIM = 2,    /* reference: vs_index::Error::WrongEmbeddingDimension     */
    VSB_EDUPKEY = 3, /* usearch multi=false: add of an existing key             */
    VSB_EFULL = 4,   /* usearch: "Reserve capacity ahead of insertions!"        */
    VSB_EOOM = 5,    /* HBM budget exhausted (reference: memory.rs Allocate::Cannot) */
    VSB_ECUDA = 6,   /* CUDA runtime/driver failure, incl. "no device"          */
    VSB_ENCCL = 7    /* multi-GPU plumbing: peer access / IPC mapping between shards unavailable */
} vsb_status;

/* usearch.rs:480-485  SpaceType -> MetricKind */
typedef enum { VSB_L2SQ = 0, VSB_COS = 1, VSB_IP = 2, VSB_HAMMING = 3 } vsb_metric;
/* usearch.rs:503-513  Quantization -> ScalarKind */
typedef enum { VSB_F32 = 0, VSB_F16 = 1, VSB_BF16 = 2, VSB_I8 = 3, VSB_B1 = 4 } vsb_scalar;

/* replaces usearch::IndexOptions as filled at usearch.rs:74-82 (A1/A2 in SURVEY §8a).
 * 0 in connectivity / expansion_* selects the reference defaults 16 / 128 / 64
 * (crates/vector-store/src/lib.rs:394-437). */
typedef struct {
    uint32_t dimensions;
    int32_t metric;           /* vsb_metric; VSB_B1 storage forces VSB_HAMMING (usearch.rs:450-464) */
    int32_t storage;          /* vsb_scalar */
    uint32_t connectivity;    /* M; the flat graph uses degree 2M like HNSW level 0 */
    uint32_t expansion_add;   /* build-time candidate width (kNN list length before pruning) */
    uint32_t expansion_search;/* beam width (itopk) of the graph search; ef = max(this, k) */
    int32_t device;           /* CUDA device ordinal; -1 = current device */
    uint32_t flags;           /* VSB_FLAG_* */
    uint64_t seed;            /* seed for the entry-point sample; 0 = default */
    /* Multi-GPU inside the library (SURVEY §8e; the reference's analogue is the per-partition index map,
     * usearch.rs:704-705).  n_devices <= 1: one index on `device`.  n_devices in 2..8: the handle is a ROUTER
     * over one sub-index per listed device, all in this process: mutations are routed by a hash of the key,
     * every search runs on every shard, each shard's kernels store their top-k straight into the gather
     * buffer of device_ids[0] over NVLink peer memory, and one K8 merge on that device produces the answer. */
    int32_t n_devices;
    int32_t device_ids[8];
} vsb_options;

#define VSB_FLAG_NONE 0u
/* f32 storage only: keep a bf16 copy of every row for the graph traversal (K4 reads half the bytes);
 * the best candidates are then re-ranked on the f32 rows (K3), so returned distances stay the
 * canonical fp32 distances of the stored vectors.  Costs +50 % HBM for the rows. */
#define VSB_FLAG_BF16_TRAVERSAL 1u
/* f32 storage + cosine only (ignored otherwise): the search walks a scaled-int8 copy of the rows (per-row
 * scale max|x|/127, a quarter of the f32 bytes, dp4a arithmetic) and re-ranks 4k candidates on the f32 rows,
 * so returned distances are still the canonical fp32 ones.  Implies VSB_FLAG_BF16_TRAVERSAL (the bf16 copy
 * keeps serving the build and the seed tiles); +25 % HBM for the rows on top of it. */
#define VSB_FLAG_I8_TRAVERSAL 2u
/* vsb_build ends with one refinement pass: every row searches the finished graph for its own nearest rows (K4, beam =
 * expansion_add) and the lists go through the pruning pipeline again.  The streamed (K7) graph needs a ~15 % wider
 * beam for the same recall (1 M x 768: ef 224 instead of 192, 10 % fewer QPS; 10 M x 768 bf16: 2-4 %); the pass
 * costs 1.7-1.9x the rest of the build.  Off by default; VSB_REFINE_PASSES overrides. */
#define VSB_FLAG_BUILD_REFINE 4u

/* Runtime tunables of the graph search (all 0 = keep current). */
typedef struct {
    uint32_t expansion_search; /* itopk; rounded up to a multiple of 32, <= 1024 */
    uint32_t max_iterations;   /* beam-search iterations per query; 0 = keep, >= 1000000 = automatic */
    uint32_t n_seeds;          /* entry points taken from the seed layer, <= 32 */
    uint32_t min_graph_size;   /* below this many live vectors search is brute force */
    uint32_t search_width;     /* parents expanded per iteration, 1..4 */
    uint32_t stream_threshold; /* un-graphed rows that make vsb_add link them into the graph (K7);
                                  default 4096; UINT32_MAX = never (only vsb_insert_pending / vsb_build) */
    uint32_t filter_exact_below_pct; /* filtered search: if fewer than this percentage of the live rows is
                                  admissible the exact bitmap scan is used instead of the graph (default 2;
                                  100 = always exact, UINT32_MAX = never) */
    uint32_t expansion_add;    /* beam width of the streaming insert / refinement searches; 0 = keep */
    uint32_t traversal;        /* 0 = keep, 1 = the traversal copy the index was created with (default),
                                  2 = walk the stored rows themselves (native scalar) although a copy exists */
    uint32_t reserved;
} vsb_search_params;

/* Counters the roofline arithmetic is computed from (SURVEY §8d). */
typedef struct {
    uint64_t kernel_launches;      /* kernels launched by this handle since creation */
    uint64_t distance_evals;       /* graph-search distance evaluations (last instrumented search) */
    uint64_t parent_expansions;    /* graph-search parent expansions (last instrumented search) */
    uint64_t queries;              /* queries in the last instrumented search */
    uint64_t n_slots;              /* rows resident in HBM (live + tombstoned) */
    uint64_t n_graphed;            /* rows covered by the graph; the rest is the brute-force tail */
    uint64_t graph_degree;         /* R */
    uint64_t row_bytes;            /* bytes per stored vector (16-byte padded) */
    uint64_t n_seed_rows;          /* rows in the entry-point sample */
    uint64_t hbm_bytes;            /* device bytes held by this handle */
    /* CUDA-event timing of the search phases on their launch stream (vsb_set_kernel_timing):
     * summed nanoseconds and launch counts since timing was switched on. */
    uint64_t convert_ns, seed_ns, graph_search_ns, exact_ns, merge_ns;
    uint64_t convert_launches, seed_launches, graph_search_launches, exact_launches, merge_launches;
    uint64_t tc_launches;          /* distance-tile launches that ran on tcgen05 (exact_tc.cu), process-wide */
    /* exact search on float rows: queries whose tiled candidate stage (TF32 / 16-bit tensor-core tiles, fp32
     * SIMT tiles) was PROVEN to contain the canonical top-k; queries the first stage could not certify; and
     * queries that went all the way to the canonical full scan (near-ties below fp32 summation noise) */
    uint64_t exact_certified, exact_fallback, exact_scanned;
    /* entry points added because a graph component held no seed of the regular sample (every live graph node
     * is reachable from the seed set after a build) */
    uint64_t extra_seeds;
} vsb_stats;

/* Work and CUDA-event time of each phase of the last vsb_build (plus the streaming inserts / refinements
 * since): what bench.py's `build_roofline` is computed from (SURVEY §8d: tensor part = 2*P^2*D flop of the
 * all-pairs stage; HBM part = E * row_bytes of the K4 passes behind K7 and the refinement). */
typedef struct {
    uint64_t rows;                 /* rows the last vsb_build covered */
    uint64_t allpairs_rows;        /* P: rows of the exact all-pairs kNN stage (K1 on tcgen05 + K3) */
    uint64_t allpairs_flops;       /* 2 * P^2 * D */
    uint64_t allpairs_ns;
    uint64_t prune_ns;             /* K6: detour pruning + reverse edges + row assembly (all passes) */
    uint64_t stream_rows;          /* rows linked by K7 */
    uint64_t stream_evals;         /* K4 distance evaluations behind them */
    uint64_t stream_parents;
    uint64_t stream_ns;
    uint64_t refine_rows;          /* rows searched by the refinement passes */
    uint64_t refine_evals;
    uint64_t refine_parents;
    uint64_t refine_ns;
    uint64_t seeds_ns;             /* entry-point sampling + reachability */
    uint64_t compact_ns;           /* tombstone compaction */
    uint64_t total_ns;             /* the whole vsb_build call, host clock */
    uint64_t traversal_row_bytes;  /* bytes one K4 distance evaluation reads during the build */
} vsb_build_stats;

/* usearch.rs:172  usearch::Index::new(&options) */
vsb_status vsb_create(const vsb_options* options, vsb_index** out);
/* drop of ThreadedUsearchIndex / UsearchIndex::stop (usearch.rs:250) */
void vsb_destroy(vsb_index* index);

/* usearch.rs:181-185  reserve_capacity_and_threads(size, threads).  Exclusive in the reference (it drains every
 * search, usearch.rs:601-605); here the grown buffers are filled on the mutator stream and published with a
 * pointer swap, so searches keep running on the old buffers meanwhile. */
vsb_status vsb_reserve(vsb_index* index, uint64_t capacity);
/* usearch.rs:187-189  capacity() */
uint64_t vsb_capacity(const vsb_index* index);
/* the AtomicUsize the actor keeps for Count (usearch.rs:866-877) */
uint64_t vsb_size(const vsb_index* index);

/* usearch.rs:191-197  add(key, &[f32]) — batched: n rows of `dimensions` f32.
 * All-or-nothing: a duplicate key (in the index or inside the batch) fails the
 * whole call with VSB_EDUPKEY; size+n > capacity fails with VSB_EFULL.
 * Added vectors are searchable as soon as the call returns (brute-force tail). */
vsb_status vsb_add(vsb_index* index, const uint64_t* keys, const float* rows, uint64_t n);
/* Same as vsb_add, with the n x dimensions f32 rows already resident in HBM on the index's device (`d_rows` is a
 * device pointer; `keys` stays a host pointer).  For bulk loads whose vectors are produced on the GPU (bench.py's
 * on-device corpus generator, config C4: a billion rows never exist in host memory).  Single-device handles only. */
vsb_status vsb_add_dev(vsb_index* index, const uint64_t* keys, const float* d_rows, uint64_t n);
/* Same, but row by row like the reference's one-message-per-vector ingest (usearch.rs:1020-1033): a duplicate
 * or reserved key fails only its own row.  row_status (nullable) receives VSB_OK / VSB_EDUPKEY / VSB_EINVAL
 * per row, *n_added (nullable) the number of rows inserted.  VSB_EFULL if the valid rows do not fit. */
vsb_status vsb_add_each(vsb_index* index, const uint64_t* keys, const float* rows, uint64_t n,
                        int32_t* row_status, uint64_t* n_added);
/* usearch.rs:199-201  remove(key) -> usize.  Unknown keys are skipped.  The slot of a removed row is
 * reclaimed by the next compaction (vsb_build, a refinement pass, or automatically when vsb_add finds the
 * slot space exhausted while size < capacity), so capacity is accounted in LIVE rows like usearch's. */
vsb_status vsb_remove(vsb_index* index, const uint64_t* keys, uint64_t n, uint64_t* n_removed);
/* usearch has no equivalent: `contains` for the host-side mirror's duplicate checks. */
int vsb_contains(const vsb_index* index, uint64_t key);

/* Bulk (re)build of the graph over every live vector added so far (A5, K5+K6).
 * Until it is called (and for vectors added after it) search is exact brute force
 * over the un-graphed tail, merged with the graph result. */
vsb_status vsb_build(vsb_index* index);

/* K7 streaming insert: links every vector added since the last build / insert into the existing graph
 * (the batched equivalent of usearch's per-vector HNSW insert, usearch.rs:191-197).  vsb_add calls
 * it by itself once `stream_threshold` rows are pending.  No-op before the first vsb_build. */
vsb_status vsb_insert_pending(vsb_index* index);

/* Copies the graph rows [n_graphed][stride] (u32 slot ids, UINT32_MAX padded) and the slot->key
 * table to host memory; `stride` = 32-rounded degree.  Snapshot/debug hook (SURVEY §8f N3) and the
 * bit-exact graph parity test.  Either output may be NULL; *n_graphed / *stride are always set. */
vsb_status vsb_export_graph(vsb_index* index, uint32_t* rows_out, uint64_t* keys_out,
                            uint64_t* n_graphed, uint32_t* stride);

vsb_status vsb_set_search_params(vsb_index* index, const vsb_search_params* params);
vsb_status vsb_get_stats(vsb_index* index, vsb_stats* out);
vsb_status vsb_get_build_stats(vsb_index* index, vsb_build_stats* out);
/* the options the handle was created with (after a vsb_load: the snapshot's) */
vsb_status vsb_get_options(vsb_index* index, vsb_options* out);
/* Re-runs nothing: switches the graph-search kernel to its counting build for the
 * next searches (identical algorithm; counters off by default for timing runs). */
vsb_status vsb_set_instrumented(vsb_index* index, int on);
/* Brackets each search phase with cudaEventRecord on the launch stream and accumulates the
 * elapsed times into vsb_stats (resolved in vsb_get_stats).  Switching on resets the sums. */
vsb_status vsb_set_kernel_timing(vsb_index* index, int on);

/* usearch.rs:203-222  search(&[f32], k) -> Matches{keys, distances}; batched over q queries. */
vsb_status vsb_search(vsb_index* index, const float* queries, uint64_t q, uint32_t k,
                      uint64_t* keys, float* distances, uint32_t* counts);
/* exact brute force (ground truth; bit-exact vs oracle/exact.c) */
vsb_status vsb_search_exact(vsb_index* index, const float* queries, uint64_t q, uint32_t k,
                            uint64_t* keys, float* distances, uint32_t* counts);
/* usearch.rs:224-248  filtered_search(&[f32], k, |key| -> bool).  The host predicate
 * becomes a bitmap over the table's row ids: bit (key & (2^48-1)) set = admissible
 * (rows >= bitmap_bits are inadmissible).  Like the reference the graph is TRAVERSED through
 * inadmissible rows and only admissible ones enter the result (K4 with the bitmap); when fewer than
 * filter_exact_below_pct percent of the live rows are admissible, or no graph exists, the exact
 * bitmap scan (K1+K3 under the bitmap, recall 1.0) answers instead. */
vsb_status vsb_search_filtered(vsb_index* index, const float* queries, uint64_t q, uint32_t k,
                               const uint32_t* allow_bitmap, uint64_t bitmap_bits,
                               uint64_t* keys, float* distances, uint32_t* counts);
/* filtered_search for q queries that each carry their own predicate.  allow_bitmaps: n_filters bitmaps
 * back to back, each ceil(bitmap_bits/32) words, same bit convention as vsb_search_filtered; query i is
 * filtered by bitmap filter_of_query[i] (< n_filters).  Per filter, the same rule as vsb_search_filtered
 * picks the graph or the exact bitmap scan, so one call may use both; results come back in the caller's
 * query order.  With n_filters = 1 the results are those of vsb_search_filtered.  VSB_EINVAL for a null
 * pointer (counts may be NULL), n_filters == 0, n_filters > q or any filter_of_query[i] >= n_filters. */
vsb_status vsb_search_filtered_multi(vsb_index* index, const float* queries, uint64_t q, uint32_t k,
                                     const uint32_t* allow_bitmaps, uint32_t n_filters, uint64_t bitmap_bits,
                                     const uint32_t* filter_of_query,
                                     uint64_t* keys, float* distances, uint32_t* counts);

/* Range search: for query i, every live row whose canonical distance is <= max_distance[i] and, when allow_bitmap is
 * not NULL, whose bit (key & (2^48-1)) is set (same convention as vsb_search_filtered), ascending by (distance, key).
 * CSR output: query i's rows are keys/distances[offsets[i] .. offsets[i+1]), offsets has q+1 entries.
 * capacity = entries keys/distances can hold.  If the total exceeds it: VSB_EFULL, offsets fully written
 * (offsets[q] = entries needed), keys/distances untouched; VSB_EFULL costs the full computation.  Exact on every
 * storage and metric: the rows and the fp32 distance bits are those of a canonical brute force (oracle/exact.c).
 * Graph and un-graphed rows alike.  max_distance[i] = +inf returns every admissible live row.  VSB_EINVAL before
 * anything runs for a NULL queries / max_distance / offsets, NULL keys or distances with capacity > 0, or a NaN
 * max_distance[i]. */
vsb_status vsb_search_range(vsb_index* index, const float* queries, uint64_t q, const float* max_distance,
                            const uint32_t* allow_bitmap, uint64_t bitmap_bits,
                            uint64_t capacity, uint64_t* keys, float* distances, uint64_t* offsets);

/* Device-resident variants: d_* are device pointers on the index's device,
 * `stream` is a cudaStream_t.  No host synchronisation, except `exact` != 0 (brute force) on float rows,
 * which reads the certification count back (see vsb_stats.exact_certified). */
vsb_status vsb_search_dev(vsb_index* index, const float* d_queries, uint64_t q, uint32_t k,
                          uint64_t* d_keys, float* d_distances, uint32_t* d_counts,
                          void* stream, int exact);
/* K8 shard merge: `parts` result blocks laid out [parts][q][k] (exactly what an
 * all-gather of per-shard vsb_search_dev outputs produces) -> [q][k], by (distance, key). */
vsb_status vsb_merge_topk_dev(const uint64_t* d_keys, const float* d_distances, uint32_t parts,
                              uint64_t q, uint32_t k, uint64_t* d_out_keys, float* d_out_distances,
                              uint32_t* d_out_counts, int device, void* stream);

/* ---- N2: micro-batcher (what a Rust shim would put into the actor's recv loop, vs_index/mod.rs:30-45).
 * Many threads call vsb_batcher_search with ONE query each (the reference's VsIndexSearch::Ann message,
 * vs_index/actor.rs:38-56); a dispatcher thread coalesces up to max_batch requests, or whatever arrived
 * within max_wait_us of the first, into one vsb_search and hands every caller its own row back. */
typedef struct vsb_batcher vsb_batcher;
vsb_status vsb_batcher_create(vsb_index* index, uint32_t dimensions, uint32_t max_batch, uint32_t max_wait_us,
                              vsb_batcher** out);
void vsb_batcher_destroy(vsb_batcher* batcher);
vsb_status vsb_batcher_search(vsb_batcher* batcher, const float* query, uint32_t k, uint64_t* keys,
                              float* distances, uint32_t* count);
vsb_status vsb_batcher_stats(vsb_batcher* batcher, uint64_t* n_queries, uint64_t* n_batches);

/* single-vector ingest through the batcher (the reference's VsIndexModify::AddVector, one vector per message,
 * monitor_items.rs:255-353): the row is copied into a staging block and the call returns; the dispatcher
 * applies staged rows with ONE vsb_add_each per flush (max_batch rows or max_wait_us after the first), so the
 * per-row H2D + stream sync of vsb_add(n=1) is paid once per block.  Like the reference's fire-and-forget add,
 * failures of individual rows are counted, not returned.  vsb_batcher_flush waits until everything staged so
 * far is searchable. */
vsb_status vsb_batcher_add(vsb_batcher* batcher, uint64_t key, const float* row);
vsb_status vsb_batcher_flush(vsb_batcher* batcher, uint64_t* n_added, uint64_t* n_failed);

/* ---- A13: the actor's partition state (vs_index/usearch.rs:626-895) as an object: a map PartitionId -> index with the
 * reference's lazy creation, capacity growth (+1 000 000 slots for a global index, +1 000 for a local one, whenever
 * fewer than free_threshold + n slots are free; usearch.rs:442-443, 655-665), per-IndexId live counters (Count),
 * empty answers for unknown partitions and the FilteredAnn -> Ann downgrade (allow_bitmap == NULL).
 * PartitionId = IndexId << 48 | partition number, bit 63 = global index (table/partition_id.rs:11-44).
 * free_threshold 0 = 64 (the reference uses its channel depth, 3 x workers). */
typedef struct vsb_set vsb_set;
vsb_status vsb_set_create(const vsb_options* options, uint32_t free_threshold, vsb_set** out);
void vsb_set_destroy(vsb_set* set);
vsb_status vsb_set_add(vsb_set* set, uint64_t partition_id, const uint64_t* keys, const float* rows, uint64_t n,
                       uint64_t* n_added);
vsb_status vsb_set_remove(vsb_set* set, uint64_t partition_id, const uint64_t* keys, uint64_t n, uint64_t* n_removed);
vsb_status vsb_set_remove_partition(vsb_set* set, uint64_t partition_id);
vsb_status vsb_set_search(vsb_set* set, uint64_t partition_id, const float* queries, uint64_t q, uint32_t k,
                          const uint32_t* allow_bitmap, uint64_t bitmap_bits, uint64_t* keys, float* distances,
                          uint32_t* counts);
uint64_t vsb_set_count(const vsb_set* set, uint16_t index_id);
uint64_t vsb_set_partitions(const vsb_set* set);
vsb_index* vsb_set_index(vsb_set* set, uint64_t partition_id);

/* ---- multi-process sharding (one rank per GPU, e.g. under torchrun): exchange of the per-shard top-k over
 * NVLink peer memory instead of an NCCL all-gather.  Every rank creates an exchange on its device, the ranks
 * swap the 64-byte CUDA-IPC handles with whatever plumbing the host has (torch.distributed in bench.py), and
 * vsb_xchg_allgather_merge then (1) stores this rank's [q][k] keys+distances into EVERY rank's gather buffer
 * with plain peer stores, (2) raises a per-rank step flag, (3) runs the K8 merge, which spins on the flags of
 * all ranks before it reads.  No collective library call and no host synchronisation in the step. */
typedef struct vsb_xchg vsb_xchg;
#define VSB_XCHG_HANDLE_BYTES 64
vsb_status vsb_xchg_create(int32_t device, uint32_t world, uint32_t rank, uint64_t max_queries, uint32_t max_k,
                           uint64_t aux_bytes_per_rank, vsb_xchg** out);
void vsb_xchg_destroy(vsb_xchg* x);
/* writes VSB_XCHG_HANDLE_BYTES bytes: this rank's gather-buffer handle */
vsb_status vsb_xchg_local_handle(vsb_xchg* x, void* handle_out);
/* `handles` = world x VSB_XCHG_HANDLE_BYTES bytes in rank order (own entry ignored); VSB_ENCCL if a peer
 * buffer cannot be mapped (no P2P / IPC between the devices) */
vsb_status vsb_xchg_open(vsb_xchg* x, const void* handles);
vsb_status vsb_xchg_allgather_merge(vsb_xchg* x, const uint64_t* d_keys, const float* d_distances, uint64_t q,
                                    uint32_t k, uint64_t* d_out_keys, float* d_out_distances,
                                    uint32_t* d_out_counts, void* stream);
/* All-gather of one opaque block per rank over the same peer stores (bench.py's e2e leg: every rank uploads 1/N of
 * the query batch over its own PCIe link and the slices are exchanged over NVLink).  bytes_per_rank: multiple of 16,
 * <= aux_bytes_per_rank of vsb_xchg_create.  *d_gathered (nullable) = device pointer to the world blocks in rank
 * order, aux_bytes_per_rank apart, valid (stream-ordered) until a peer's second-next call; d_copy_out (nullable) =
 * caller's device buffer that receives the blocks back to back (use it when gathers are pipelined). */
vsb_status vsb_xchg_allgather_bytes(vsb_xchg* x, const void* d_src, uint64_t bytes_per_rank, void** d_gathered,
                                    void* d_copy_out, void* stream);
/* synchronises `stream` and reports VSB_ENCCL if the watchdog of a merge gave up on a rank (~2 s) */
vsb_status vsb_xchg_check(vsb_xchg* x, void* stream);

/* ---- N3: snapshot.  The reference rebuilds its in-memory index from a full table scan on every restart
 * (db_cdc/checkpoint_saver.rs:103-112, SURVEY F7); a flat file of keys / tombstones / rows / graph makes
 * restart O(read).  vsb_load creates a new handle on `device` (-1 = current). */
vsb_status vsb_save(vsb_index* index, const char* path);
vsb_status vsb_load(const char* path, int32_t device, vsb_index** out);

/* Same merge for parts that are NOT stored back to back: part p's keys start at d_keys + p*key_part_stride
 * (u64 elements), its distances at d_distances + p*dist_part_stride (f32 elements).  Lets one all-gather of a
 * per-rank record [q*k keys | q*k distances] feed the merge directly. */
vsb_status vsb_merge_topk_strided_dev(const uint64_t* d_keys, const float* d_distances, uint32_t parts,
                                      uint64_t key_part_stride, uint64_t dist_part_stride, uint64_t q, uint32_t k,
                                      uint64_t* d_out_keys, float* d_out_distances, uint32_t* d_out_counts,
                                      int device, void* stream);

/* A11: usearch.rs:1179-1205  f32_to_b1x8 (host utility, same bit order) */
void vsb_f32_to_b1x8(const float* v, uint64_t n, uint8_t* out /* ceil(n/8) bytes */);

/* thread-local message of the last failing call on this thread */
const char* vsb_last_error(void);
/* "vsb200-x.y.z" — what VsIndexFactory::index_engine_version would report (usearch.rs:109-114) */
const char* vsb_version(void);

#ifdef __cplusplus
}
#endif
#endif /* VSB200_H */
