"""`GpuIndex` — host-side mirror of the reference's inner seam, the private trait `UsearchIndex`
(crates/vector-store/src/vs_index/usearch.rs:142-160: reserve / capacity / add / remove / search /
filtered_search / stop), implemented over the C ABI of libvsb200.so.  The single-vector methods
keep the reference's names and error behaviour; the `*_batch` methods expose the batched ABI."""
from __future__ import annotations

import ctypes as C
import enum

import numpy as np

from . import native
from .native import VsbBuildStats, VsbOptions, VsbSearchParams, VsbStats, check, lib


class Metric(enum.IntEnum):  # usearch MetricKind as mapped at usearch.rs:480-501
    L2sq = 0
    Cos = 1
    IP = 2
    Hamming = 3


class Scalar(enum.IntEnum):  # usearch ScalarKind, usearch.rs:503-513
    F32 = 0
    F16 = 1
    BF16 = 2
    I8 = 3
    B1 = 4


INVALID_KEY = np.uint64(0xFFFFFFFFFFFFFFFF)


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


class GpuIndex:
    def __init__(self, dimensions: int, metric: Metric = Metric.Cos, storage: Scalar = Scalar.F32,
                 connectivity: int = 0, expansion_add: int = 0, expansion_search: int = 0, device: int = -1,
                 seed: int = 0, bf16_traversal: bool = False, i8_traversal: bool = False, devices=None,
                 build_refine: bool = False):
        """devices: list of 2..8 CUDA ordinals -> ONE handle over one shard per device (vsb_options.n_devices)."""
        self._lib = lib()
        # VSB_FLAG_BF16_TRAVERSAL | VSB_FLAG_I8_TRAVERSAL | VSB_FLAG_BUILD_REFINE
        flags = (1 if bf16_traversal else 0) | (2 if i8_traversal else 0) | (4 if build_refine else 0)
        devs = list(devices) if devices else []
        opt = VsbOptions(dimensions, int(metric), int(storage), connectivity, expansion_add, expansion_search,
                         device, flags, seed, len(devs), (C.c_int32 * 8)(*(devs + [0] * (8 - len(devs)))))
        h = C.c_void_p()
        check(self._lib.vsb_create(C.byref(opt), C.byref(h)))
        self._h = h
        self.dimensions = dimensions
        self.metric = Metric.Hamming if storage == Scalar.B1 else Metric(metric)
        self.storage = Scalar(storage)

    # ---- UsearchIndex trait (usearch.rs:142-160) ----
    def reserve(self, size: int) -> None:
        check(self._lib.vsb_reserve(self._h, size))

    def capacity(self) -> int:
        return int(self._lib.vsb_capacity(self._h))

    def add(self, primary_id: int, vector) -> None:
        self.add_batch(np.array([primary_id], dtype=np.uint64), np.asarray(vector, dtype=np.float32)[None, :])

    def remove(self, primary_id: int) -> bool:
        return self.remove_batch(np.array([primary_id], dtype=np.uint64)) != 0

    def search(self, vector, limit: int):
        """-> list[(primary_id, distance)] ascending; fewer than `limit` when the index is small."""
        keys, dists, counts = self.search_batch(np.asarray(vector, dtype=np.float32)[None, :], limit)
        return [(int(keys[0, i]), float(dists[0, i])) for i in range(int(counts[0]))]

    def filtered_search(self, vector, limit: int, predicate):
        """The reference passes a host closure |PrimaryId| -> bool (usearch.rs:224-248); the device needs a
        bitmap, so the closure is evaluated once per live row id here (host side) and uploaded."""
        raise NotImplementedError("use filtered_search_bitmap (the actor mirror builds the bitmap)")

    def filtered_search_bitmap(self, vector, limit: int, allow_bitmap: np.ndarray, bitmap_bits: int):
        q = np.ascontiguousarray(np.asarray(vector, dtype=np.float32)[None, :])
        self._check_dim(q)
        bm = np.ascontiguousarray(allow_bitmap, dtype=np.uint32)
        keys = np.empty((1, limit), dtype=np.uint64)
        dists = np.empty((1, limit), dtype=np.float32)
        counts = np.empty(1, dtype=np.uint32)
        check(self._lib.vsb_search_filtered(self._h, _ptr(q), 1, limit, _ptr(bm), bitmap_bits, _ptr(keys),
                                            _ptr(dists), _ptr(counts)))
        return [(int(keys[0, i]), float(dists[0, i])) for i in range(int(counts[0]))]

    def stop(self) -> None:
        self.close()

    # ---- batched ABI ----
    def _check_dim(self, a: np.ndarray) -> None:
        if a.ndim != 2 or a.shape[1] != self.dimensions:
            raise native.VsbError(native.VSB_EDIM, f"expected dimension {self.dimensions}, got {a.shape}")

    def size(self) -> int:
        return int(self._lib.vsb_size(self._h))

    def __len__(self) -> int:
        return self.size()

    def contains(self, key: int) -> bool:
        return bool(self._lib.vsb_contains(self._h, key))

    def add_batch(self, keys, rows) -> None:
        rows = np.ascontiguousarray(rows, dtype=np.float32)
        keys = np.ascontiguousarray(keys, dtype=np.uint64)
        self._check_dim(rows)
        if keys.shape[0] != rows.shape[0]:
            raise native.VsbError(native.VSB_EINVAL, "keys/rows length mismatch")
        check(self._lib.vsb_add(self._h, _ptr(keys), _ptr(rows), rows.shape[0]))

    def add_dev(self, keys, d_rows: int, n: int) -> None:
        """rows already in HBM on the index's device (raw device pointer to n x dimensions f32)"""
        keys = np.ascontiguousarray(keys, dtype=np.uint64)
        if keys.shape[0] != n:
            raise native.VsbError(native.VSB_EINVAL, "keys/rows length mismatch")
        check(self._lib.vsb_add_dev(self._h, _ptr(keys), d_rows, n))

    def add_each(self, keys, rows):
        """Row-by-row semantics of the reference's one-message-per-vector ingest (usearch.rs:1020-1033): a duplicate
        or reserved key fails only its own row.  -> (n_added, per-row status array)."""
        rows = np.ascontiguousarray(rows, dtype=np.float32)
        keys = np.ascontiguousarray(keys, dtype=np.uint64)
        self._check_dim(rows)
        if keys.shape[0] != rows.shape[0]:
            raise native.VsbError(native.VSB_EINVAL, "keys/rows length mismatch")
        status = np.zeros(rows.shape[0], dtype=np.int32)
        n = C.c_uint64(0)
        check(self._lib.vsb_add_each(self._h, _ptr(keys), _ptr(rows), rows.shape[0], _ptr(status), C.byref(n)))
        return int(n.value), status

    def remove_batch(self, keys) -> int:
        keys = np.ascontiguousarray(keys, dtype=np.uint64)
        n = C.c_uint64(0)
        check(self._lib.vsb_remove(self._h, _ptr(keys), keys.shape[0], C.byref(n)))
        return int(n.value)

    def build(self) -> None:
        check(self._lib.vsb_build(self._h))

    def insert_pending(self) -> None:
        check(self._lib.vsb_insert_pending(self._h))

    def export_graph(self):
        """-> (rows u32 [n_graphed, stride], keys u64 [n_graphed])"""
        n = C.c_uint64(0)
        stride = C.c_uint32(0)
        check(self._lib.vsb_export_graph(self._h, None, None, C.byref(n), C.byref(stride)))
        rows = np.empty((n.value, stride.value), dtype=np.uint32)
        keys = np.empty(n.value, dtype=np.uint64)
        if n.value:
            check(self._lib.vsb_export_graph(self._h, _ptr(rows), _ptr(keys), C.byref(n), C.byref(stride)))
        return rows, keys

    def set_search_params(self, expansion_search: int = 0, max_iterations: int = 0, n_seeds: int = 0,
                          min_graph_size: int = 0, search_width: int = 0, stream_threshold: int = 0,
                          filter_exact_below_pct: int = 0, expansion_add: int = 0, traversal: int = 0) -> None:
        p = VsbSearchParams(expansion_search, max_iterations, n_seeds, min_graph_size, search_width, stream_threshold,
                            filter_exact_below_pct, expansion_add, traversal, 0)
        check(self._lib.vsb_set_search_params(self._h, C.byref(p)))

    def set_instrumented(self, on: bool) -> None:
        check(self._lib.vsb_set_instrumented(self._h, int(on)))

    def set_kernel_timing(self, on: bool) -> None:
        check(self._lib.vsb_set_kernel_timing(self._h, int(on)))

    def stats(self) -> dict:
        s = VsbStats()
        check(self._lib.vsb_get_stats(self._h, C.byref(s)))
        return {n: int(getattr(s, n)) for n, _ in VsbStats._fields_}

    def build_stats(self) -> dict:
        s = VsbBuildStats()
        check(self._lib.vsb_get_build_stats(self._h, C.byref(s)))
        return {n: int(getattr(s, n)) for n, _ in VsbBuildStats._fields_}

    def search_batch(self, queries, k: int, exact: bool = False, out=None):
        q = np.ascontiguousarray(queries, dtype=np.float32)
        self._check_dim(q)
        n = q.shape[0]
        if out is None:
            keys = np.empty((n, k), dtype=np.uint64)
            dists = np.empty((n, k), dtype=np.float32)
            counts = np.empty(n, dtype=np.uint32)
        else:
            keys, dists, counts = out
        fn = self._lib.vsb_search_exact if exact else self._lib.vsb_search
        check(fn(self._h, _ptr(q), n, k, _ptr(keys), _ptr(dists), _ptr(counts)))
        return keys, dists, counts

    def search_filtered(self, queries, k: int, allow_mask):
        """Batched filtered search: allow_mask[i] (bool) admits the row whose id (key & 2^48-1) is i."""
        q = np.ascontiguousarray(queries, dtype=np.float32)
        self._check_dim(q)
        mask = np.asarray(allow_mask, dtype=bool)
        bm = np.packbits(mask, bitorder="little")
        bm = np.concatenate([bm, np.zeros((-len(bm)) % 4, np.uint8)]).view(np.uint32)
        n = q.shape[0]
        keys = np.empty((n, k), dtype=np.uint64)
        dists = np.empty((n, k), dtype=np.float32)
        counts = np.empty(n, dtype=np.uint32)
        check(self._lib.vsb_search_filtered(self._h, _ptr(q), n, k, _ptr(bm), len(mask), _ptr(keys), _ptr(dists),
                                            _ptr(counts)))
        return keys, dists, counts

    def search_filtered_multi(self, queries, k: int, masks, filter_of_query):
        """Batched filtered search with one filter per query: masks is an [n_filters][bits] bool array (row i of a
        mask admits the row whose id, key & 2^48-1, is i) and query j is filtered by masks[filter_of_query[j]]."""
        q = np.ascontiguousarray(queries, dtype=np.float32)
        self._check_dim(q)
        m = np.asarray(masks, dtype=bool)
        if m.ndim != 2:
            raise ValueError("masks must be [n_filters][bits]")
        bm = np.packbits(m, axis=1, bitorder="little")
        bm = np.concatenate([bm, np.zeros((m.shape[0], (-bm.shape[1]) % 4), np.uint8)], axis=1)
        bm = np.ascontiguousarray(bm).view(np.uint32)
        fq = np.ascontiguousarray(filter_of_query, dtype=np.uint32)
        n = q.shape[0]
        if fq.shape != (n,):
            raise ValueError("filter_of_query must hold one index per query")
        keys = np.empty((n, k), dtype=np.uint64)
        dists = np.empty((n, k), dtype=np.float32)
        counts = np.empty(n, dtype=np.uint32)
        check(self._lib.vsb_search_filtered_multi(self._h, _ptr(q), n, k, _ptr(bm), m.shape[0], m.shape[1], _ptr(fq),
                                                  _ptr(keys), _ptr(dists), _ptr(counts)))
        return keys, dists, counts

    def search_range(self, queries, max_distance, allow_mask=None):
        """Range search, exact: for query i every live row whose distance is <= max_distance[i] (and, with allow_mask,
        whose id key & 2^48-1 is admitted, as in search_filtered), ascending by (distance, key).  max_distance is a
        scalar or one value per query (+inf returns every admissible row).  -> (offsets u64 [n + 1], keys u64 [total],
        dists f32 [total]); query i's rows are keys[offsets[i]:offsets[i + 1]].  The result size is not known before
        the call: the first attempt has room for 256 rows per query, and if that is too small (VSB_EFULL, which
        costs a full search) the call is made once more with exactly offsets[-1] rows of room."""
        q = np.ascontiguousarray(queries, dtype=np.float32)
        self._check_dim(q)
        n = q.shape[0]
        r = np.ascontiguousarray(np.broadcast_to(np.asarray(max_distance, dtype=np.float32), (n,)))
        bm, bits = None, 0
        if allow_mask is not None:
            mask = np.asarray(allow_mask, dtype=bool)
            bm = np.packbits(mask, bitorder="little")
            bm = np.concatenate([bm, np.zeros((-len(bm)) % 4, np.uint8)]).view(np.uint32)
            bits = len(mask)
        offsets = np.zeros(n + 1, dtype=np.uint64)
        cap = 256 * n
        for attempt in range(2):
            keys = np.empty(cap, dtype=np.uint64)
            dists = np.empty(cap, dtype=np.float32)
            st = self._lib.vsb_search_range(self._h, _ptr(q), n, _ptr(r), _ptr(bm), bits, cap, _ptr(keys), _ptr(dists),
                                            _ptr(offsets))
            if st == native.VSB_EFULL and attempt == 0:
                cap = int(offsets[-1])
                continue
            check(st)
            break
        total = int(offsets[-1])
        return offsets, keys[:total], dists[:total]

    def search_raw(self, q_ptr: int, n: int, k: int, keys_ptr: int, dists_ptr: int, counts_ptr: int,
                   exact: bool = False) -> None:
        """Host-pointer call without NumPy marshalling (bench e2e leg uses pinned torch buffers)."""
        fn = self._lib.vsb_search_exact if exact else self._lib.vsb_search
        check(fn(self._h, q_ptr, n, k, keys_ptr, dists_ptr, counts_ptr))

    def search_dev(self, d_queries: int, n: int, k: int, d_keys: int, d_dists: int, d_counts: int, stream: int,
                   exact: bool = False) -> None:
        """Device-pointer call (ints = raw CUDA pointers / cudaStream_t), never synchronises."""
        check(self._lib.vsb_search_dev(self._h, d_queries, n, k, d_keys, d_dists, d_counts or None, stream or None,
                                       int(exact)))

    def save(self, path: str) -> None:
        check(self._lib.vsb_save(self._h, path.encode()))

    @classmethod
    def load(cls, path: str, device: int = -1) -> "GpuIndex":
        l = lib()
        h = C.c_void_p()
        check(l.vsb_load(path.encode(), device, C.byref(h)))
        self = cls.__new__(cls)
        self._lib, self._h = l, h
        opt = VsbOptions()
        check(l.vsb_get_options(h, C.byref(opt)))  # dimensions / metric / storage come from the snapshot header
        self.dimensions = int(opt.dimensions)
        self.storage = Scalar(opt.storage)
        self.metric = Metric.Hamming if self.storage == Scalar.B1 else Metric(opt.metric)
        return self

    def close(self) -> None:
        if getattr(self, "_h", None):
            self._lib.vsb_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def merge_topk_dev(d_keys: int, d_dists: int, parts: int, q: int, k: int, d_out_keys: int, d_out_dists: int,
                   d_out_counts: int, device: int, stream: int) -> None:
    check(lib().vsb_merge_topk_dev(d_keys, d_dists, parts, q, k, d_out_keys, d_out_dists, d_out_counts or None,
                                   device, stream or None))


class Batcher:
    """N2 micro-batcher: `search(query, k)` may be called from many threads; calls are coalesced on the C++ side."""

    def __init__(self, index: GpuIndex, max_batch: int = 1024, max_wait_us: int = 200):
        self._lib = lib()
        self._index = index  # keep the index alive
        b = C.c_void_p()
        check(self._lib.vsb_batcher_create(index._h, index.dimensions, max_batch, max_wait_us, C.byref(b)))
        self._b = b
        self._dim = index.dimensions

    def add(self, key: int, row) -> None:
        """fire-and-forget single-vector add (VsIndexModify::AddVector): staged, applied in blocks"""
        r = np.ascontiguousarray(row, dtype=np.float32).ravel()
        if r.shape[0] != self._dim:
            raise native.VsbError(native.VSB_EDIM, f"expected dimension {self._dim}, got {r.shape[0]}")
        check(self._lib.vsb_batcher_add(self._b, int(key), _ptr(r)))

    def flush(self):
        """-> (rows added, rows rejected) since creation; returns once everything staged so far is searchable"""
        ok, bad = C.c_uint64(0), C.c_uint64(0)
        check(self._lib.vsb_batcher_flush(self._b, C.byref(ok), C.byref(bad)))
        return int(ok.value), int(bad.value)

    def search(self, query, k: int):
        q = np.ascontiguousarray(query, dtype=np.float32).ravel()
        if q.shape[0] != self._dim:
            raise native.VsbError(native.VSB_EDIM, f"expected dimension {self._dim}, got {q.shape[0]}")
        keys = np.empty(k, dtype=np.uint64)
        dists = np.empty(k, dtype=np.float32)
        cnt = C.c_uint32(0)
        check(self._lib.vsb_batcher_search(self._b, _ptr(q), k, _ptr(keys), _ptr(dists), C.byref(cnt)))
        return keys[:cnt.value], dists[:cnt.value]

    def stats(self):
        nq, nb = C.c_uint64(0), C.c_uint64(0)
        check(self._lib.vsb_batcher_stats(self._b, C.byref(nq), C.byref(nb)))
        return int(nq.value), int(nb.value)

    def close(self) -> None:
        if getattr(self, "_b", None):
            self._lib.vsb_batcher_destroy(self._b)
            self._b = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def merge_topk_strided_dev(d_keys: int, d_dists: int, parts: int, key_part_stride: int, dist_part_stride: int, q: int,
                           k: int, d_out_keys: int, d_out_dists: int, d_out_counts: int, device: int,
                           stream: int) -> None:
    check(lib().vsb_merge_topk_strided_dev(d_keys, d_dists, parts, key_part_stride, dist_part_stride, q, k, d_out_keys,
                                           d_out_dists, d_out_counts or None, device, stream or None))


class IndexSet:
    """A13: the actor's partition map as the library keeps it (vsb_set_*, csrc/index_set.cu): lazily created
    per-partition indexes, the reference's capacity growth, per-IndexId counters, empty answers for unknown partitions.
    partition_id = index_id << 48 | partition number; bit 63 set = global index (table/partition_id.rs:11-44)."""

    def __init__(self, dimensions: int, metric: Metric = Metric.Cos, storage: Scalar = Scalar.F32, connectivity: int = 0,
                 expansion_add: int = 0, expansion_search: int = 0, device: int = -1, bf16_traversal: bool = False,
                 free_threshold: int = 0):
        self._lib = lib()
        opt = VsbOptions(dimensions, int(metric), int(storage), connectivity, expansion_add, expansion_search, device,
                         1 if bf16_traversal else 0, 0, 0, (C.c_int32 * 8)(*([0] * 8)))
        h = C.c_void_p()
        check(self._lib.vsb_set_create(C.byref(opt), free_threshold, C.byref(h)))
        self._h = h
        self.dimensions = dimensions

    def add(self, partition_id: int, keys, rows) -> int:
        k = np.ascontiguousarray(keys, dtype=np.uint64)
        r = np.ascontiguousarray(rows, dtype=np.float32).reshape(len(k), self.dimensions)
        added = C.c_uint64(0)
        check(self._lib.vsb_set_add(self._h, partition_id, _ptr(k), _ptr(r), len(k), C.byref(added)))
        return int(added.value)

    def remove(self, partition_id: int, keys) -> int:
        k = np.ascontiguousarray(keys, dtype=np.uint64)
        removed = C.c_uint64(0)
        check(self._lib.vsb_set_remove(self._h, partition_id, _ptr(k), len(k), C.byref(removed)))
        return int(removed.value)

    def remove_partition(self, partition_id: int) -> None:
        check(self._lib.vsb_set_remove_partition(self._h, partition_id))

    def search(self, partition_id: int, queries, k: int, allow_mask=None):
        q = np.ascontiguousarray(queries, dtype=np.float32).reshape(-1, self.dimensions)
        n = q.shape[0]
        keys = np.empty((n, k), dtype=np.uint64)
        dists = np.empty((n, k), dtype=np.float32)
        counts = np.empty(n, dtype=np.uint32)
        bm, bits = None, 0
        if allow_mask is not None:
            mask = np.asarray(allow_mask, dtype=bool)
            bm = np.packbits(mask, bitorder="little")
            bm = np.concatenate([bm, np.zeros((-len(bm)) % 4, np.uint8)]).view(np.uint32)
            bits = len(mask)
        check(self._lib.vsb_set_search(self._h, partition_id, _ptr(q), n, k, _ptr(bm), bits, _ptr(keys), _ptr(dists),
                                       _ptr(counts)))
        return keys, dists, counts

    def count(self, index_id: int) -> int:
        return int(self._lib.vsb_set_count(self._h, index_id))

    def partitions(self) -> int:
        return int(self._lib.vsb_set_partitions(self._h))

    def capacity(self, partition_id: int) -> int:
        h = self._lib.vsb_set_index(self._h, partition_id)
        return int(self._lib.vsb_capacity(h)) if h else 0

    def close(self) -> None:
        if getattr(self, "_h", None):
            self._lib.vsb_set_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Exchange:
    """Per-shard top-k exchange between one-process-per-GPU ranks over NVLink peer memory (vsb_xchg_*, csrc/xchg.cu).
    `allgather_bytes(local: bytes) -> list[bytes]` is the host plumbing that swaps the 64-byte IPC handles
    (torch.distributed.all_gather_object in bench.py)."""

    def __init__(self, device: int, world: int, rank: int, max_queries: int, max_k: int, allgather_bytes,
                 aux_bytes_per_rank: int = 0):
        self._lib = lib()
        x = C.c_void_p()
        check(self._lib.vsb_xchg_create(device, world, rank, max_queries, max_k, aux_bytes_per_rank, C.byref(x)))
        self._x = x
        mine = C.create_string_buffer(native.XCHG_HANDLE_BYTES)
        check(self._lib.vsb_xchg_local_handle(self._x, mine))
        handles = allgather_bytes(mine.raw)
        blob = C.create_string_buffer(b"".join(handles), world * native.XCHG_HANDLE_BYTES)
        check(self._lib.vsb_xchg_open(self._x, blob))

    def allgather_merge(self, d_keys: int, d_dists: int, q: int, k: int, d_out_keys: int, d_out_dists: int,
                        d_out_counts: int, stream: int) -> None:
        check(self._lib.vsb_xchg_allgather_merge(self._x, d_keys, d_dists, q, k, d_out_keys, d_out_dists,
                                                 d_out_counts or None, stream or None))

    def allgather_rows(self, d_src: int, bytes_per_rank: int, stream: int, d_copy_out: int = 0) -> int:
        """-> device pointer to the world blocks in rank order (aux_bytes_per_rank apart); d_copy_out: the blocks are
        also copied back to back into that device buffer (pipelined gathers must not read the window later)"""
        out = C.c_void_p()
        check(self._lib.vsb_xchg_allgather_bytes(self._x, d_src, bytes_per_rank, C.byref(out), d_copy_out or None,
                                                 stream or None))
        return int(out.value)

    def check(self, stream: int) -> None:
        check(self._lib.vsb_xchg_check(self._x, stream or None))

    def close(self) -> None:
        if getattr(self, "_x", None):
            self._lib.vsb_xchg_destroy(self._x)
            self._x = None
