//! Raw bindings to `libvsb200.so` — one declaration per entry point of `include/vsb200.h`, same order.
//!
//! NOT COMPILED in the vsb200 repository's image (no cargo/rustc there); `tests/test_abi.py` checks that every
//! symbol the header declares is declared here and that the struct field lists match.  The safe wrapper lives in
//! `crates/vector-store/src/vs_index/gpu.rs`.
#![allow(non_camel_case_types)]

use std::os::raw::{c_char, c_int, c_void};

#[repr(C)]
pub struct vsb_index {
    _private: [u8; 0],
}
#[repr(C)]
pub struct vsb_batcher {
    _private: [u8; 0],
}
#[repr(C)]
pub struct vsb_set {
    _private: [u8; 0],
}
#[repr(C)]
pub struct vsb_xchg {
    _private: [u8; 0],
}

pub type vsb_status = c_int;
pub const VSB_OK: vsb_status = 0;
pub const VSB_EINVAL: vsb_status = 1;
pub const VSB_EDIM: vsb_status = 2;
pub const VSB_EDUPKEY: vsb_status = 3;
pub const VSB_EFULL: vsb_status = 4;
pub const VSB_EOOM: vsb_status = 5;
pub const VSB_ECUDA: vsb_status = 6;
pub const VSB_ENCCL: vsb_status = 7;

pub const VSB_L2SQ: i32 = 0;
pub const VSB_COS: i32 = 1;
pub const VSB_IP: i32 = 2;
pub const VSB_HAMMING: i32 = 3;

pub const VSB_F32: i32 = 0;
pub const VSB_F16: i32 = 1;
pub const VSB_BF16: i32 = 2;
pub const VSB_I8: i32 = 3;
pub const VSB_B1: i32 = 4;

pub const VSB_FLAG_NONE: u32 = 0;
/// f32 storage: the graph walk reads a bf16 copy, the best candidates are re-ranked on the f32 rows
pub const VSB_FLAG_BF16_TRAVERSAL: u32 = 1;
/// f32 storage + cosine: the graph walk reads a scaled-int8 copy, fp32 re-rank
pub const VSB_FLAG_I8_TRAVERSAL: u32 = 2;
/// vsb_build ends with one refinement pass (better graph, 1.7-1.9x the build time)
pub const VSB_FLAG_BUILD_REFINE: u32 = 4;

pub const VSB_XCHG_HANDLE_BYTES: usize = 64;

#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct vsb_options {
    pub dimensions: u32,
    pub metric: i32,
    pub storage: i32,
    pub connectivity: u32,
    pub expansion_add: u32,
    pub expansion_search: u32,
    pub device: i32,
    pub flags: u32,
    pub seed: u64,
    pub n_devices: i32,
    pub device_ids: [i32; 8],
}

#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct vsb_search_params {
    pub expansion_search: u32,
    pub max_iterations: u32,
    pub n_seeds: u32,
    pub min_graph_size: u32,
    pub search_width: u32,
    pub stream_threshold: u32,
    pub filter_exact_below_pct: u32,
    pub expansion_add: u32,
    pub traversal: u32,
    pub reserved: u32,
}

#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct vsb_stats {
    pub kernel_launches: u64,
    pub distance_evals: u64,
    pub parent_expansions: u64,
    pub queries: u64,
    pub n_slots: u64,
    pub n_graphed: u64,
    pub graph_degree: u64,
    pub row_bytes: u64,
    pub n_seed_rows: u64,
    pub hbm_bytes: u64,
    pub convert_ns: u64,
    pub seed_ns: u64,
    pub graph_search_ns: u64,
    pub exact_ns: u64,
    pub merge_ns: u64,
    pub convert_launches: u64,
    pub seed_launches: u64,
    pub graph_search_launches: u64,
    pub exact_launches: u64,
    pub merge_launches: u64,
    pub tc_launches: u64,
    pub exact_certified: u64,
    pub exact_fallback: u64,
    pub exact_scanned: u64,
    pub extra_seeds: u64,
}

#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct vsb_build_stats {
    pub rows: u64,
    pub allpairs_rows: u64,
    pub allpairs_flops: u64,
    pub allpairs_ns: u64,
    pub prune_ns: u64,
    pub stream_rows: u64,
    pub stream_evals: u64,
    pub stream_parents: u64,
    pub stream_ns: u64,
    pub refine_rows: u64,
    pub refine_evals: u64,
    pub refine_parents: u64,
    pub refine_ns: u64,
    pub seeds_ns: u64,
    pub compact_ns: u64,
    pub total_ns: u64,
    pub traversal_row_bytes: u64,
}

unsafe extern "C" {
    pub fn vsb_create(options: *const vsb_options, out: *mut *mut vsb_index) -> vsb_status;
    pub fn vsb_destroy(index: *mut vsb_index);
    pub fn vsb_reserve(index: *mut vsb_index, capacity: u64) -> vsb_status;
    pub fn vsb_capacity(index: *const vsb_index) -> u64;
    pub fn vsb_size(index: *const vsb_index) -> u64;
    pub fn vsb_add(index: *mut vsb_index, keys: *const u64, rows: *const f32, n: u64) -> vsb_status;
    pub fn vsb_add_dev(index: *mut vsb_index, keys: *const u64, d_rows: *const f32, n: u64) -> vsb_status;
    pub fn vsb_add_each(
        index: *mut vsb_index,
        keys: *const u64,
        rows: *const f32,
        n: u64,
        row_status: *mut i32,
        n_added: *mut u64,
    ) -> vsb_status;
    pub fn vsb_remove(index: *mut vsb_index, keys: *const u64, n: u64, n_removed: *mut u64) -> vsb_status;
    pub fn vsb_contains(index: *const vsb_index, key: u64) -> c_int;
    pub fn vsb_build(index: *mut vsb_index) -> vsb_status;
    pub fn vsb_insert_pending(index: *mut vsb_index) -> vsb_status;
    pub fn vsb_export_graph(
        index: *mut vsb_index,
        rows_out: *mut u32,
        keys_out: *mut u64,
        n_graphed: *mut u64,
        stride: *mut u32,
    ) -> vsb_status;
    pub fn vsb_set_search_params(index: *mut vsb_index, params: *const vsb_search_params) -> vsb_status;
    pub fn vsb_get_stats(index: *mut vsb_index, out: *mut vsb_stats) -> vsb_status;
    pub fn vsb_get_build_stats(index: *mut vsb_index, out: *mut vsb_build_stats) -> vsb_status;
    pub fn vsb_get_options(index: *mut vsb_index, out: *mut vsb_options) -> vsb_status;
    pub fn vsb_set_instrumented(index: *mut vsb_index, on: c_int) -> vsb_status;
    pub fn vsb_set_kernel_timing(index: *mut vsb_index, on: c_int) -> vsb_status;
    pub fn vsb_search(
        index: *mut vsb_index,
        queries: *const f32,
        q: u64,
        k: u32,
        keys: *mut u64,
        distances: *mut f32,
        counts: *mut u32,
    ) -> vsb_status;
    pub fn vsb_search_exact(
        index: *mut vsb_index,
        queries: *const f32,
        q: u64,
        k: u32,
        keys: *mut u64,
        distances: *mut f32,
        counts: *mut u32,
    ) -> vsb_status;
    pub fn vsb_search_filtered(
        index: *mut vsb_index,
        queries: *const f32,
        q: u64,
        k: u32,
        allow_bitmap: *const u32,
        bitmap_bits: u64,
        keys: *mut u64,
        distances: *mut f32,
        counts: *mut u32,
    ) -> vsb_status;
    pub fn vsb_search_filtered_multi(
        index: *mut vsb_index,
        queries: *const f32,
        q: u64,
        k: u32,
        allow_bitmaps: *const u32,
        n_filters: u32,
        bitmap_bits: u64,
        filter_of_query: *const u32,
        keys: *mut u64,
        distances: *mut f32,
        counts: *mut u32,
    ) -> vsb_status;
    pub fn vsb_search_dev(
        index: *mut vsb_index,
        d_queries: *const f32,
        q: u64,
        k: u32,
        d_keys: *mut u64,
        d_distances: *mut f32,
        d_counts: *mut u32,
        stream: *mut c_void,
        exact: c_int,
    ) -> vsb_status;
    pub fn vsb_merge_topk_dev(
        d_keys: *const u64,
        d_distances: *const f32,
        parts: u32,
        q: u64,
        k: u32,
        d_out_keys: *mut u64,
        d_out_distances: *mut f32,
        d_out_counts: *mut u32,
        device: c_int,
        stream: *mut c_void,
    ) -> vsb_status;
    pub fn vsb_batcher_create(
        index: *mut vsb_index,
        dimensions: u32,
        max_batch: u32,
        max_wait_us: u32,
        out: *mut *mut vsb_batcher,
    ) -> vsb_status;
    pub fn vsb_batcher_destroy(batcher: *mut vsb_batcher);
    pub fn vsb_batcher_search(
        batcher: *mut vsb_batcher,
        query: *const f32,
        k: u32,
        keys: *mut u64,
        distances: *mut f32,
        count: *mut u32,
    ) -> vsb_status;
    pub fn vsb_batcher_stats(batcher: *mut vsb_batcher, n_queries: *mut u64, n_batches: *mut u64) -> vsb_status;
    pub fn vsb_batcher_add(batcher: *mut vsb_batcher, key: u64, row: *const f32) -> vsb_status;
    pub fn vsb_batcher_flush(batcher: *mut vsb_batcher, n_added: *mut u64, n_failed: *mut u64) -> vsb_status;
    pub fn vsb_set_create(options: *const vsb_options, free_threshold: u32, out: *mut *mut vsb_set) -> vsb_status;
    pub fn vsb_set_destroy(set: *mut vsb_set);
    pub fn vsb_set_add(
        set: *mut vsb_set,
        partition_id: u64,
        keys: *const u64,
        rows: *const f32,
        n: u64,
        n_added: *mut u64,
    ) -> vsb_status;
    pub fn vsb_set_remove(
        set: *mut vsb_set,
        partition_id: u64,
        keys: *const u64,
        n: u64,
        n_removed: *mut u64,
    ) -> vsb_status;
    pub fn vsb_set_remove_partition(set: *mut vsb_set, partition_id: u64) -> vsb_status;
    pub fn vsb_set_search(
        set: *mut vsb_set,
        partition_id: u64,
        queries: *const f32,
        q: u64,
        k: u32,
        allow_bitmap: *const u32,
        bitmap_bits: u64,
        keys: *mut u64,
        distances: *mut f32,
        counts: *mut u32,
    ) -> vsb_status;
    pub fn vsb_set_count(set: *const vsb_set, index_id: u16) -> u64;
    pub fn vsb_set_partitions(set: *const vsb_set) -> u64;
    pub fn vsb_set_index(set: *mut vsb_set, partition_id: u64) -> *mut vsb_index;
    pub fn vsb_xchg_create(
        device: i32,
        world: u32,
        rank: u32,
        max_queries: u64,
        max_k: u32,
        aux_bytes_per_rank: u64,
        out: *mut *mut vsb_xchg,
    ) -> vsb_status;
    pub fn vsb_xchg_destroy(x: *mut vsb_xchg);
    pub fn vsb_xchg_local_handle(x: *mut vsb_xchg, handle_out: *mut c_void) -> vsb_status;
    pub fn vsb_xchg_open(x: *mut vsb_xchg, handles: *const c_void) -> vsb_status;
    pub fn vsb_xchg_allgather_merge(
        x: *mut vsb_xchg,
        d_keys: *const u64,
        d_distances: *const f32,
        q: u64,
        k: u32,
        d_out_keys: *mut u64,
        d_out_distances: *mut f32,
        d_out_counts: *mut u32,
        stream: *mut c_void,
    ) -> vsb_status;
    pub fn vsb_xchg_allgather_bytes(
        x: *mut vsb_xchg,
        d_src: *const c_void,
        bytes_per_rank: u64,
        d_gathered: *mut *mut c_void,
        d_copy_out: *mut c_void,
        stream: *mut c_void,
    ) -> vsb_status;
    pub fn vsb_xchg_check(x: *mut vsb_xchg, stream: *mut c_void) -> vsb_status;
    pub fn vsb_save(index: *mut vsb_index, path: *const c_char) -> vsb_status;
    pub fn vsb_load(path: *const c_char, device: i32, out: *mut *mut vsb_index) -> vsb_status;
    pub fn vsb_merge_topk_strided_dev(
        d_keys: *const u64,
        d_distances: *const f32,
        parts: u32,
        key_part_stride: u64,
        dist_part_stride: u64,
        q: u64,
        k: u32,
        d_out_keys: *mut u64,
        d_out_distances: *mut f32,
        d_out_counts: *mut u32,
        device: c_int,
        stream: *mut c_void,
    ) -> vsb_status;
    pub fn vsb_f32_to_b1x8(v: *const f32, n: u64, out: *mut u8);
    pub fn vsb_last_error() -> *const c_char;
    pub fn vsb_version() -> *const c_char;
}

/// `vsb_last_error()` of the calling thread as an owned string.
pub fn last_error() -> String {
    // SAFETY: the library returns a pointer to a NUL-terminated thread-local buffer that stays valid until the next
    // failing call on this thread.
    unsafe {
        let p = vsb_last_error();
        if p.is_null() {
            String::new()
        } else {
            std::ffi::CStr::from_ptr(p).to_string_lossy().into_owned()
        }
    }
}

/// `vsb_version()`, e.g. "vsb200-0.2.0 (sm_100a)".
pub fn version() -> String {
    // SAFETY: static NUL-terminated string.
    unsafe { std::ffi::CStr::from_ptr(vsb_version()).to_string_lossy().into_owned() }
}
