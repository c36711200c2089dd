"""Host-side mirror of the reference's index actor for the GPU backend — what
`crates/vector-store/src/vs_index/gpu.rs` would be (INTEGRATION.md), written against the same
interface so the parity tests read like the reference's own (vs_index/usearch.rs:1207-1665).

Mirrored behaviour (file:line in the reference):
  * VsIndexConfiguration                         vs_index/factory.rs:20-28, defaults lib.rs:394-480
  * metric_kind / quantization mapping           vs_index/usearch.rs:450-513
  * lazy per-partition index creation            vs_index/usearch.rs:744-779
  * capacity growth: +1_000_000 (global) / +1_000 (local) when free < threshold
                                                 vs_index/usearch.rs:442-443, 655-665, 908-921
  * add/remove failures are logged and swallowed vs_index/usearch.rs:1028-1030, 1042
  * Count from a counter, never from the index   vs_index/usearch.rs:866-877
  * unknown partition => empty result            vs_index/usearch.rs:787-802
  * wrong dimension => WrongEmbeddingDimension   vs_index/validator.rs:12-26
  * every hit passes Distance::try_from          vs_index/usearch.rs:219
  * memory gate: adds dropped while Cannot       vs_index/usearch.rs:1157-1177
The message transport (tokio mpsc/oneshot) is replaced by direct synchronous calls; the batched
calls (`add_vectors`, `ann_batch`) are what the Rust shim's micro-batcher would issue."""
from __future__ import annotations

import enum
import logging
from dataclasses import dataclass, field

import numpy as np

from . import native
from .distance import Distance, SpaceType
from .index import GpuIndex, Metric, Scalar

log = logging.getLogger("vsb200.actor")

RESERVE_INCREMENT_GLOBAL = 1_000_000  # usearch.rs:442
RESERVE_INCREMENT_LOCAL = 1_000       # usearch.rs:443


class Quantization(enum.Enum):
    F32 = "f32"
    F16 = "f16"
    BF16 = "bf16"
    I8 = "i8"
    B1 = "b1"


class WrongEmbeddingDimension(ValueError):
    """vs_index::Error::WrongEmbeddingDimension -> HTTP 400 (httproutes.rs:855-856)."""


@dataclass
class VsIndexConfiguration:
    key: str
    dimensions: int
    connectivity: int = 16           # lib.rs:394-407
    expansion_add: int = 128         # lib.rs:409-422
    expansion_search: int = 64       # lib.rs:424-437
    space_type: SpaceType = SpaceType.Cosine
    quantization: Quantization = Quantization.F32


_SCALAR = {Quantization.F32: Scalar.F32, Quantization.F16: Scalar.F16, Quantization.BF16: Scalar.BF16,
           Quantization.I8: Scalar.I8, Quantization.B1: Scalar.B1}


def metric_kind(quantization: Quantization, space_type: SpaceType) -> Metric:
    """usearch.rs:450-501."""
    if quantization is Quantization.B1:
        return Metric.Hamming
    if space_type is SpaceType.Cosine:
        return Metric.Cos
    if space_type is SpaceType.Euclidean:
        return Metric.L2sq
    if space_type is SpaceType.DotProduct:
        return Metric.IP
    raise ValueError("Binary space type requires B1 quantization.")


_SPACE_OF_METRIC = {Metric.Cos: SpaceType.Cosine, Metric.L2sq: SpaceType.Euclidean, Metric.IP: SpaceType.DotProduct,
                    Metric.Hamming: SpaceType.Hamming}


@dataclass
class _Partition:
    idx: GpuIndex
    is_global: bool
    size: int = 0
    capacity: int = 0

    def needs_more_capacity(self, free_threshold: int) -> int | None:
        if self.capacity - self.size < free_threshold:
            return self.capacity + (RESERVE_INCREMENT_GLOBAL if self.is_global else RESERVE_INCREMENT_LOCAL)
        return None


GLOBAL_PARTITION = 0


@dataclass
class IndexActor:
    config: VsIndexConfiguration
    device: int = -1
    free_threshold: int = 24  # perf::channel_size() = 3 x workers (perf.rs:20-24) on an 8-thread box
    reserve_increment: int | None = None  # tests shrink the 1M-row global increment
    partitions: dict = field(default_factory=dict)
    can_allocate: bool = True  # memory.rs Allocate::{Can,Cannot}
    size: int = 0

    def __post_init__(self):
        self.metric = metric_kind(self.config.quantization, self.config.space_type)
        self.space = _SPACE_OF_METRIC[self.metric]

    # ---- VsIndexModifyExt (actor.rs:63-76) ----
    def _partition(self, partition_id: int) -> _Partition:
        p = self.partitions.get(partition_id)
        if p is None:
            c = self.config
            idx = GpuIndex(c.dimensions, self.metric, _SCALAR[c.quantization], c.connectivity, c.expansion_add,
                           c.expansion_search, self.device)
            p = _Partition(idx, partition_id == GLOBAL_PARTITION)
            self.partitions[partition_id] = p
        return p

    def _grow(self, p: _Partition, incoming: int) -> None:
        while True:
            want = p.needs_more_capacity(self.free_threshold + incoming)
            if want is None:
                return
            if self.reserve_increment is not None:
                want = p.capacity + max(self.reserve_increment, incoming + self.free_threshold)
            p.idx.reserve(want)
            p.capacity = p.idx.capacity()

    def add_vector(self, partition_id: int, primary_id: int, embedding) -> None:
        self.add_vectors(partition_id, [primary_id], np.asarray(embedding, dtype=np.float32)[None, :])

    def add_vectors(self, partition_id: int, primary_ids, embeddings) -> None:
        if not self.can_allocate:  # usearch.rs:1157-1177: silently dropped
            return
        emb = np.asarray(embeddings, dtype=np.float32)
        if emb.ndim != 2 or emb.shape[1] != self.config.dimensions:
            log.warning("add_vector: wrong dimension %s for index %s", emb.shape, self.config.key)
            return
        p = self._partition(partition_id)
        try:
            self._grow(p, emb.shape[0])
            # row-by-row verdicts like the reference's one-message-per-vector loop (usearch.rs:1020-1033): a duplicate or
            # reserved key fails only its own row, the rest of the batch is indexed
            added, status = p.idx.add_each(np.asarray(primary_ids, dtype=np.uint64), emb)
        except native.VsbError as e:  # logged and swallowed, usearch.rs:1028-1030
            log.warning("add_vector failed for index %s: %s", self.config.key, e)
            return
        if added != emb.shape[0]:
            bad = np.flatnonzero(status)
            log.warning("add_vector: %d of %d rows rejected for index %s (first: key %s, status %d)", len(bad),
                        emb.shape[0], self.config.key, np.asarray(primary_ids)[bad[0]], int(status[bad[0]]))
        p.size += added
        self.size += added

    def remove_vector(self, partition_id: int, primary_id: int) -> None:
        p = self.partitions.get(partition_id)
        if p is None:
            return
        try:
            removed = p.idx.remove(primary_id)
        except native.VsbError as e:  # usearch.rs:1042
            log.warning("remove_vector failed for index %s: %s", self.config.key, e)
            return
        if removed:
            p.size -= 1
            self.size -= 1

    def remove_partition(self, partition_id: int) -> None:  # usearch.rs:888-893
        p = self.partitions.pop(partition_id, None)
        if p is not None:
            self.size -= p.size
            p.idx.stop()

    def build(self) -> None:
        """GPU-only step: bulk graph build once the full scan has delivered its rows (INTEGRATION.md)."""
        for p in self.partitions.values():
            p.idx.build()

    # ---- VsIndexSearchExt (actor.rs:78-90) ----
    def _validate(self, embedding: np.ndarray) -> None:
        if embedding.shape[-1] != self.config.dimensions:
            raise WrongEmbeddingDimension(
                f"Wrong embedding dimension: expected {self.config.dimensions}, got {embedding.shape[-1]}")

    def _to_hits(self, keys, dists, count):
        out_k, out_d = [], []
        for i in range(int(count)):
            d = Distance.try_from(float(dists[i]), self.space, self.config.dimensions)  # Err => whole query fails
            out_k.append(int(keys[i]))
            out_d.append(d)
        return out_k, out_d

    MAX_LIMIT = 1024  # vsb_search's k ceiling (include/vsb200.h); the reference's Limit is unbounded

    def ann(self, embedding, limit: int, partition_id: int = GLOBAL_PARTITION):
        e = np.asarray(embedding, dtype=np.float32)
        self._validate(e)
        p = self.partitions.get(partition_id)
        if p is None:
            return [], []
        # a Limit above the engine's ceiling is served with the ceiling (never an error: usearch returns what it has)
        keys, dists, counts = p.idx.search_batch(e[None, :], min(limit, self.MAX_LIMIT))
        return self._to_hits(keys[0], dists[0], counts[0])

    def ann_batch(self, embeddings, limit: int, partition_id: int = GLOBAL_PARTITION):
        e = np.asarray(embeddings, dtype=np.float32)
        self._validate(e)
        p = self.partitions.get(partition_id)
        if p is None:
            return [([], []) for _ in range(e.shape[0])]
        keys, dists, counts = p.idx.search_batch(e, limit)
        return [self._to_hits(keys[i], dists[i], counts[i]) for i in range(e.shape[0])]

    def filtered_ann(self, embedding, limit: int, predicate, max_row_id: int,
                     partition_id: int = GLOBAL_PARTITION):
        """`predicate(primary_id) -> bool` mirrors the reference closure (usearch.rs:1108-1154); it is
        evaluated per table row id (low 48 bits of the key, table/primary_id.rs:27-62) into a bitmap.
        `predicate=None` is the reference's downgrade: a FilteredAnn whose restrictions are fully consumed by the
        local partition key becomes a plain Ann on that partition (usearch.rs:844-862)."""
        if predicate is None:
            return self.ann(embedding, limit, partition_id)
        e = np.asarray(embedding, dtype=np.float32)
        self._validate(e)
        p = self.partitions.get(partition_id)
        if p is None:
            return [], []
        bits = max_row_id + 1
        bm = np.zeros((bits + 31) // 32, dtype=np.uint32)
        for row in range(bits):
            if predicate(row):
                bm[row >> 5] |= np.uint32(1 << (row & 31))
        hits = p.idx.filtered_search_bitmap(e, limit, bm, bits)
        keys = np.array([h[0] for h in hits], dtype=np.uint64)
        dists = np.array([h[1] for h in hits], dtype=np.float32)
        return self._to_hits(keys, dists, len(hits))

    def filtered_ann_batch(self, embeddings, limit: int, predicates, max_row_id: int,
                           partition_id: int = GLOBAL_PARTITION):
        """A run of FilteredAnn requests on one partition in one call, as the Rust backend coalesces them:
        predicates[i] filters embeddings[i]; each predicate becomes a bitmap over the row ids, identical bitmaps are
        sent once, and every request gets what `filtered_ann` would return for it.  A None predicate is a plain Ann."""
        e = np.asarray(embeddings, dtype=np.float32)
        self._validate(e)
        n = e.shape[0]
        if len(predicates) != n:
            raise ValueError("one predicate per embedding")
        p = self.partitions.get(partition_id)
        if p is None:
            return [([], []) for _ in range(n)]
        out = [None] * n
        plain = [i for i in range(n) if predicates[i] is None]
        for i in plain:
            out[i] = self.ann(e[i], limit, partition_id)
        filtered = [i for i in range(n) if predicates[i] is not None]
        if filtered:
            bits = max_row_id + 1
            rows = np.arange(bits)
            masks, index_of, fq = [], {}, []
            for i in filtered:
                m = np.fromiter((bool(predicates[i](int(r))) for r in rows), dtype=bool, count=bits)
                j = index_of.setdefault(m.tobytes(), len(masks))
                if j == len(masks):
                    masks.append(m)
                fq.append(j)
            keys, dists, counts = p.idx.search_filtered_multi(e[filtered], limit, np.stack(masks), fq)
            for r, i in enumerate(filtered):
                out[i] = self._to_hits(keys[r], dists[r], counts[r])
        return out

    def count(self) -> int:
        return self.size

    def stop(self) -> None:
        for p in self.partitions.values():
            p.idx.stop()
        self.partitions.clear()


def new_index_factory_gpu(device: int = -1):
    """Mirror of `new_index_factory_usearch` (vs_index/mod.rs:47-53): returns create_index(config)."""
    def create_index(config: VsIndexConfiguration) -> IndexActor:
        return IndexActor(config, device=device)
    create_index.index_engine_version = native.version
    return create_index
