// sharded.h — the multi-device router behind a vsb_index handle created with n_devices > 1 (internal).
#pragma once
#include "index_impl.h"

namespace vsbi {

vsb_status create_sharded(const vsb_options* o, vsb_index** out);
void destroy_sharded(vsb_index* ix);
vsb_status sharded_reserve(vsb_index* ix, uint64_t capacity);
uint64_t sharded_capacity(const vsb_index* ix);
uint64_t sharded_size(const vsb_index* ix);
vsb_status sharded_add(vsb_index* ix, const uint64_t* keys, const float* rows, uint64_t n, int32_t* row_status,
                       uint64_t* n_added);
vsb_status sharded_remove(vsb_index* ix, const uint64_t* keys, uint64_t n, uint64_t* n_removed);
int sharded_contains(vsb_index* ix, uint64_t key);
vsb_status sharded_build(vsb_index* ix);
vsb_status sharded_insert_pending(vsb_index* ix);
vsb_status sharded_set_search_params(vsb_index* ix, const vsb_search_params* p);
vsb_status sharded_set_instrumented(vsb_index* ix, int on);
vsb_status sharded_set_kernel_timing(vsb_index* ix, int on);
vsb_status sharded_get_stats(vsb_index* ix, vsb_stats* out);
vsb_status sharded_get_build_stats(vsb_index* ix, vsb_build_stats* out);
vsb_status sharded_search_host(vsb_index* ix, const float* queries, uint64_t nq, uint32_t k, uint64_t* keys,
                               float* dists, uint32_t* counts, bool exact, const HostFilters& hf = HostFilters());
vsb_status sharded_search_dev(vsb_index* ix, const float* d_queries, uint64_t nq, uint32_t k, uint64_t* d_keys,
                              float* d_dists, uint32_t* d_counts, cudaStream_t stream, bool exact);
// every shard's range search, merged per query by (distance, key); capacity as in search_range
vsb_status sharded_search_range(vsb_index* ix, const float* queries, uint64_t nq, const float* max_distance,
                                const HostFilters& hf, uint64_t capacity, RangeResult& out);
vsb_status sharded_save(vsb_index* ix, const char* path);

// snapshot_io.cu
vsb_status save_single(vsb_index* ix, const char* path);
vsb_status load_single(const char* path, int32_t device, vsb_index** out);

}  // namespace vsbi
