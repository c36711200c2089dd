/*
 * crates/vector-store/src/vs_index/gpu.rs — the vsb200 (B200) backend of the index actor.
 *
 * NOT COMPILED in the vsb200 repository's image (no cargo/rustc there).  It is the source a maintainer adds next to
 * `usearch.rs`; registration: `mod gpu;` in vs_index/mod.rs:6-11, `new_index_factory_gpu` beside
 * `new_index_factory_usearch` (vs_index/mod.rs:47-68, bottom of this file), and one more branch in the backend
 * pick at lib.rs:766-775 (`else if config.use_gpu { new_index_factory_gpu(config_rx, worker, memory) }`).
 *
 * What stays exactly as in usearch.rs: the two mpsc channels and the search-first `recv` (vs_index/mod.rs:30-45),
 * the lazily created per-partition indexes and the +1 000 000 / +1 000 capacity growth (usearch.rs:626-670), the
 * memory gate for AddVector (usearch.rs:1157-1177), `Count` answered from a counter, empty results for unknown
 * partitions, the FilteredAnn -> Ann downgrade when the partition lookup consumed every restriction
 * (usearch.rs:844-862), swallowed add/remove errors (usearch.rs:1020-1050), `Distance::try_from` on every hit.
 *
 * What changes: the reference hands ONE message to ONE worker and takes a reader/writer permit per message
 * (usearch.rs:515-624).  A GPU wants batches and needs no gate (libvsb200 searches a published view while mutators
 * prepare the next one), so the loop drains what is already queued and coalesces RUNS of compatible messages:
 *   Ann x n on one partition         -> one vsb_search(q = n)
 *   FilteredAnn x n on one partition -> one vsb_search_filtered_multi(q = n), one bitmap per distinct predicate
 *   AddVector x n on one partition   -> one vsb_add_each(n)     (per-row status: one bad row fails alone)
 *   RemoveVector x n                 -> one vsb_remove(n)
 * Order inside a partition is preserved (an update is RemoveVector followed by AddVector of the same row).
 */

use crate::Dimensions;
use crate::Distance;
use crate::Filter;
use crate::IndexKey;
use crate::Limit;
use crate::PrimaryKey;
use crate::Quantization;
use crate::SpaceType;
use crate::Vector;
use crate::memory::Allocate;
use crate::memory::Memory;
use crate::memory::MemoryExt;
use crate::perf;
use crate::table::IndexId;
use crate::table::PartitionId;
use crate::table::PrimaryId;
use crate::table::Table;
use crate::table::TableSearch;
use crate::vs_index::Message;
use crate::vs_index::VsIndexModify;
use crate::vs_index::VsIndexSearch;
use crate::vs_index::actor::AnnR;
use crate::vs_index::factory::VsIndexConfiguration;
use crate::vs_index::factory::VsIndexFactory;
use crate::vs_index::validator;
use crate::worker::Worker;
use crate::worker::WorkerExt;
use anyhow::anyhow;
use anyhow::bail;
use std::collections::BTreeMap;
use std::collections::HashMap;
use std::sync::Arc;
use std::sync::Mutex;
use std::sync::RwLock;
use std::sync::atomic::AtomicUsize;
use std::sync::atomic::Ordering;
use tokio::sync::mpsc;
use tokio::sync::oneshot;
use tokio::sync::watch;
use tracing::Instrument;
use tracing::debug;
use tracing::error;
use tracing::error_span;
use tracing::trace;
use tracing::warn;
use vsb200_sys as sys;

const RESERVE_INCREMENT_GLOBAL: usize = 1_000_000; // usearch.rs:442
const RESERVE_INCREMENT_LOCAL: usize = 1_000; // usearch.rs:443
const MAX_RUN: usize = 1024; // messages coalesced into one library call
const ROW_MASK: u64 = (1u64 << 48) - 1; // PrimaryId = epoch << 48 | row idx (table/primary_id.rs:27-62)

fn check(rc: sys::vsb_status) -> anyhow::Result<()> {
    match rc {
        sys::VSB_OK => Ok(()),
        sys::VSB_EDIM => Err(validator::Error::WrongEmbeddingDimension.into()),
        _ => Err(anyhow!("vsb200: {}", sys::last_error())),
    }
}

/// metric / storage mapping, same rule as usearch.rs:450-513: B1 forces Hamming, Hamming needs B1.
fn metric_of(quantization: Quantization, space_type: SpaceType) -> anyhow::Result<i32> {
    match (quantization, space_type) {
        (Quantization::B1, _) => Ok(sys::VSB_HAMMING),
        (_, SpaceType::Hamming) => bail!("Hamming space type is only supported with B1 quantization"),
        (_, SpaceType::Euclidean) => Ok(sys::VSB_L2SQ),
        (_, SpaceType::Cosine) => Ok(sys::VSB_COS),
        (_, SpaceType::DotProduct) => Ok(sys::VSB_IP),
    }
}

fn storage_of(quantization: Quantization) -> i32 {
    match quantization {
        Quantization::F32 => sys::VSB_F32,
        Quantization::F16 => sys::VSB_F16,
        Quantization::BF16 => sys::VSB_BF16,
        Quantization::I8 => sys::VSB_I8,
        Quantization::B1 => sys::VSB_B1,
    }
}

/// One partition's index in HBM.  Every vsb_* call is thread-safe on one handle.
struct GpuIndex {
    h: *mut sys::vsb_index,
    space: SpaceType,
    dimensions: Dimensions,
    /// rows currently in the index, as a bitmap over the row idx (low 48 bits of the key): the universe a filter
    /// predicate is evaluated over when a FilteredAnn request is turned into an allow-bitmap
    live_rows: Mutex<Vec<u32>>,
}

// SAFETY: the handle is an opaque pointer to a library object whose entry points lock internally.
unsafe impl Send for GpuIndex {}
unsafe impl Sync for GpuIndex {}

impl Drop for GpuIndex {
    fn drop(&mut self) {
        // SAFETY: created by vsb_create, destroyed once.
        unsafe { sys::vsb_destroy(self.h) }
    }
}

impl GpuIndex {
    fn new(options: &sys::vsb_options, space: SpaceType, dimensions: Dimensions) -> anyhow::Result<Self> {
        let mut h = std::ptr::null_mut();
        // SAFETY: plain-old-data options, out pointer to a local.
        check(unsafe { sys::vsb_create(options, &mut h) })?;
        Ok(Self {
            h,
            space,
            dimensions,
            live_rows: Mutex::new(Vec::new()),
        })
    }

    fn reserve(&self, size: usize) -> anyhow::Result<()> {
        check(unsafe { sys::vsb_reserve(self.h, size as u64) }) // replaces usearch.rs:181-185
    }

    fn capacity(&self) -> usize {
        unsafe { sys::vsb_capacity(self.h) as usize }
    }

    fn mark_rows(&self, keys: impl Iterator<Item = u64>, live: bool) {
        let mut bm = self.live_rows.lock().unwrap();
        for key in keys {
            let row = (key & ROW_MASK) as usize;
            if live && row / 32 >= bm.len() {
                bm.resize(row / 32 + 1, 0);
            }
            if let Some(word) = bm.get_mut(row / 32) {
                if live {
                    *word |= 1u32 << (row % 32);
                } else {
                    *word &= !(1u32 << (row % 32));
                }
            }
        }
    }

    /// n rows in one call; returns how many were inserted (a duplicate or reserved key fails alone, usearch.rs:191-197)
    fn add_many(&self, keys: &[u64], rows: &[f32]) -> anyhow::Result<usize> {
        let mut status = vec![0i32; keys.len()];
        let mut added = 0u64;
        check(unsafe {
            sys::vsb_add_each(
                self.h,
                keys.as_ptr(),
                rows.as_ptr(),
                keys.len() as u64,
                status.as_mut_ptr(),
                &mut added,
            )
        })?;
        for (key, st) in keys.iter().zip(&status) {
            if *st != sys::VSB_OK {
                warn!("row {key} was not inserted (vsb status {st})");
            }
        }
        self.mark_rows(
            keys.iter().zip(&status).filter(|(_, st)| **st == sys::VSB_OK).map(|(key, _)| *key),
            true,
        );
        Ok(added as usize)
    }

    /// returns how many of the keys were present (usearch.rs:199-201)
    fn remove_many(&self, keys: &[u64]) -> anyhow::Result<usize> {
        let mut removed = 0u64;
        check(unsafe { sys::vsb_remove(self.h, keys.as_ptr(), keys.len() as u64, &mut removed) })?;
        self.mark_rows(keys.iter().copied(), false);
        Ok(removed as usize)
    }

    fn unpack(
        &self,
        keys: &[u64],
        dists: &[f32],
        count: usize,
    ) -> anyhow::Result<Vec<(PrimaryId, Distance)>> {
        keys.iter()
            .zip(dists)
            .take(count)
            .map(|(key, dist)| {
                // distance.rs:58-105 unchanged: the library already clamps to the ranges it checks
                Distance::try_from((*dist, self.space, Some(self.dimensions))).map(|d| (PrimaryId::from(*key), d))
            })
            .collect()
    }

    /// q queries of `dimensions` floats each, one k for all; per query the (id, distance) pairs in ascending order
    fn search_many(&self, queries: &[f32], q: usize, k: usize) -> anyhow::Result<Vec<Vec<(PrimaryId, Distance)>>> {
        let (mut keys, mut dists, mut counts) = (vec![0u64; q * k], vec![0f32; q * k], vec![0u32; q]);
        check(unsafe {
            sys::vsb_search(
                self.h,
                queries.as_ptr(),
                q as u64,
                k as u32,
                keys.as_mut_ptr(),
                dists.as_mut_ptr(),
                counts.as_mut_ptr(),
            )
        })?; // replaces usearch.rs:203-222
        (0..q)
            .map(|i| self.unpack(&keys[i * k..(i + 1) * k], &dists[i * k..(i + 1) * k], counts[i] as usize))
            .collect()
    }

    /// The host predicate of usearch.rs:224-248 becomes a bitmap over row ids, built once per request over the rows
    /// that are in the index, and the graph is traversed on the device with the bit tested where a result is emitted.
    /// A run of q requests is one call: `predicate(i, id)` is request i's predicate, identical bitmaps are sent once,
    /// every request is answered with its own bitmap and k, and the answers come back in request order.
    fn search_filtered_many(
        &self,
        queries: &[f32],
        q: usize,
        k: usize,
        predicate: impl Fn(usize, PrimaryId) -> bool,
    ) -> anyhow::Result<Vec<Vec<(PrimaryId, Distance)>>> {
        let (allow, n_filters, words, filter_of_query) = {
            let live = self.live_rows.lock().unwrap();
            let words = live.len();
            let mut allow: Vec<u32> = Vec::new();
            let mut seen: HashMap<Vec<u32>, u32> = HashMap::new();
            let mut filter_of_query = Vec::with_capacity(q);
            for i in 0..q {
                let bitmap: Vec<u32> = live
                    .iter()
                    .enumerate()
                    .map(|(w, word)| {
                        let mut out = 0u32;
                        let mut bits = *word;
                        while bits != 0 {
                            let b = bits.trailing_zeros();
                            bits &= bits - 1;
                            // the epoch is not part of the row id the table is asked about (Idx::idx masks it off)
                            if predicate(i, PrimaryId::from((w as u64) * 32 + b as u64)) {
                                out |= 1u32 << b;
                            }
                        }
                        out
                    })
                    .collect();
                let next = seen.len() as u32;
                let f = *seen.entry(bitmap).or_insert_with_key(|bitmap| {
                    allow.extend_from_slice(bitmap);
                    next
                });
                filter_of_query.push(f);
            }
            (allow, seen.len(), words, filter_of_query)
        };
        let (mut keys, mut dists, mut counts) = (vec![0u64; q * k], vec![0f32; q * k], vec![0u32; q]);
        check(unsafe {
            sys::vsb_search_filtered_multi(
                self.h,
                queries.as_ptr(),
                q as u64,
                k as u32,
                allow.as_ptr(),
                n_filters as u32,
                (words * 32) as u64,
                filter_of_query.as_ptr(),
                keys.as_mut_ptr(),
                dists.as_mut_ptr(),
                counts.as_mut_ptr(),
            )
        })?;
        (0..q)
            .map(|i| self.unpack(&keys[i * k..(i + 1) * k], &dists[i * k..(i + 1) * k], counts[i] as usize))
            .collect()
    }
}

struct PartitionState {
    partition_id: PartitionId,
    size: AtomicUsize,
    capacity: AtomicUsize,
    capacity_increment: usize,
    free_threshold: usize,
    idx: GpuIndex,
}

impl PartitionState {
    fn new(partition_id: PartitionId, idx: GpuIndex) -> Self {
        Self {
            partition_id,
            size: AtomicUsize::new(0),
            capacity: AtomicUsize::new(0),
            capacity_increment: if partition_id.index_id().is_global() {
                RESERVE_INCREMENT_GLOBAL
            } else {
                RESERVE_INCREMENT_LOCAL
            },
            // a coalesced run may add MAX_RUN rows at once, the reference adds one per message
            free_threshold: usize::from(perf::channel_size()).max(MAX_RUN),
            idx,
        }
    }

    /// usearch.rs:655-665, with room for a whole run
    fn needs_more_capacity(&self, incoming: usize) -> Option<usize> {
        let capacity = self.capacity.load(Ordering::Relaxed);
        let size = self.size.load(Ordering::Relaxed);
        (capacity - size < self.free_threshold + incoming)
            .then(|| capacity + self.capacity_increment.max(incoming + self.free_threshold))
    }
}

struct IndexState {
    size: Arc<AtomicUsize>,
}

/// A run of messages that one library call serves.
enum Run {
    Add {
        partition: Arc<PartitionState>,
        keys: Vec<u64>,
        rows: Vec<f32>,
        // the reference drops AsyncInProgress when the add finished; the rows are searchable when vsb_add_each returns
        in_progress: Vec<crate::AsyncInProgress>,
    },
    Remove {
        partition: Arc<PartitionState>,
        keys: Vec<u64>,
        in_progress: Vec<crate::AsyncInProgress>,
    },
    Ann {
        partition: Arc<PartitionState>,
        queries: Vec<f32>,
        limits: Vec<usize>,
        txs: Vec<oneshot::Sender<AnnR>>,
    },
    FilteredAnn {
        partition: Arc<PartitionState>,
        queries: Vec<f32>,
        filters: Vec<Filter>,
        limits: Vec<usize>,
        txs: Vec<oneshot::Sender<AnnR>>,
    },
}

fn to_primary_keys(
    partition: &PartitionState,
    table: &RwLock<impl TableSearch>,
    hits: Vec<(PrimaryId, Distance)>,
) -> (Vec<PrimaryKey>, Vec<Distance>) {
    let table = table.read().unwrap();
    hits.into_iter()
        .filter_map(|(primary_id, distance)| {
            table
                .primary_key(partition.partition_id, primary_id)
                .or_else(|| {
                    debug!(
                        "hit {primary_id:?} of partition {:?} has no primary key any more, dropped from the answer",
                        partition.partition_id
                    );
                    None
                })
                .map(|primary_key| (primary_key, distance))
        })
        .unzip()
}

fn execute(run: Run, table: &RwLock<impl TableSearch>, index_size: &AtomicUsize) {
    match run {
        Run::Add {
            partition,
            keys,
            rows,
            in_progress,
        } => {
            match partition.idx.add_many(&keys, &rows) {
                Err(err) => warn!("a run of {} inserts failed as a whole: {err}", keys.len()),
                Ok(added) => {
                    partition.size.fetch_add(added, Ordering::Relaxed);
                    index_size.fetch_add(added, Ordering::Relaxed);
                }
            }
            drop(in_progress);
        }
        Run::Remove {
            partition,
            keys,
            in_progress,
        } => {
            match partition.idx.remove_many(&keys) {
                Err(err) => warn!("a run of {} removals failed as a whole: {err}", keys.len()),
                Ok(removed) => {
                    partition.size.fetch_sub(removed, Ordering::Relaxed);
                    index_size.fetch_sub(removed, Ordering::Relaxed);
                }
            }
            drop(in_progress);
        }
        Run::Ann {
            partition,
            queries,
            limits,
            txs,
        } => {
            let k = limits.iter().copied().max().unwrap_or(1);
            match partition.idx.search_many(&queries, txs.len(), k) {
                Err(err) => {
                    let msg = err.to_string();
                    for tx in txs {
                        tx.send(Err(anyhow!("batched search failed: {msg}")))
                            .unwrap_or_else(|_| trace!("the requester of an ann went away"));
                    }
                }
                Ok(per_query) => {
                    for ((hits, limit), tx) in per_query.into_iter().zip(limits).zip(txs) {
                        let hits = hits.into_iter().take(limit).collect();
                        tx.send(Ok(to_primary_keys(&partition, table, hits)))
                            .unwrap_or_else(|_| trace!("the requester of an ann went away"));
                    }
                }
            }
        }
        Run::FilteredAnn {
            partition,
            queries,
            filters,
            limits,
            txs,
        } => {
            let id_ok = |i: usize, primary_id: PrimaryId| {
                let table = table.read().unwrap();
                filters[i]
                    .restrictions
                    .iter()
                    .all(|restriction| table.is_valid_for(partition.partition_id, primary_id, restriction))
            };
            let k = limits.iter().copied().max().unwrap_or(1);
            match partition.idx.search_filtered_many(&queries, txs.len(), k, id_ok) {
                Err(err) => {
                    let msg = err.to_string();
                    for tx in txs {
                        tx.send(Err(anyhow!("filtered search failed: {msg}")))
                            .unwrap_or_else(|_| trace!("the requester of an ann went away"));
                    }
                }
                Ok(per_query) => {
                    for ((hits, limit), tx) in per_query.into_iter().zip(limits).zip(txs) {
                        let hits = hits.into_iter().take(limit).collect();
                        tx.send(Ok(to_primary_keys(&partition, table, hits)))
                            .unwrap_or_else(|_| trace!("the requester of an ann went away"));
                    }
                }
            }
        }
    }
}

/// The memory gate of usearch.rs:1157-1177 for a drained batch: while the monitor says `Cannot`, AddVector messages
/// are dropped (everything else passes); the refusal is logged once per Can -> Cannot edge.
struct MemoryGate {
    rx: watch::Receiver<Allocate>,
    refused_before: bool,
}

impl MemoryGate {
    fn admits(&mut self, msg: &Message, key: &IndexKey) -> bool {
        let is_add = matches!(msg, Message::Modify(VsIndexModify::AddVector { .. }));
        if !is_add {
            return true;
        }
        let refused = *self.rx.borrow() == Allocate::Cannot;
        if refused && !self.refused_before {
            error!("index {key}: vectors are being dropped, the memory monitor forbids new allocations");
        }
        self.refused_before = refused;
        !refused
    }
}

/// Appends `msg` to the last run if it is compatible, else starts a new run.  Mirrors `preprocess`
/// (usearch.rs:744-896) for the partition lookup, lazy creation, the Ann replies for unknown partitions, Count,
/// RemovePartition and the FilteredAnn -> Ann downgrade.
#[allow(clippy::too_many_arguments)]
fn enqueue(
    runs: &mut Vec<Run>,
    msg: Message,
    index_fn: &impl Fn() -> anyhow::Result<GpuIndex>,
    states: &mut BTreeMap<IndexId, IndexState>,
    partitions: &mut BTreeMap<PartitionId, Arc<PartitionState>>,
    table: &RwLock<impl TableSearch>,
    dimensions: Dimensions,
) {
    let same = |a: &Arc<PartitionState>, b: &Arc<PartitionState>| Arc::ptr_eq(a, b);
    match msg {
        Message::Modify(VsIndexModify::AddVector {
            partition_id,
            primary_id,
            embedding,
            in_progress,
        }) => {
            let partition = match partitions.get(&partition_id) {
                Some(partition) => Arc::clone(partition),
                None => {
                    let idx = match index_fn() {
                        Ok(idx) => idx,
                        Err(err) => {
                            error!("partition {partition_id:?}: no index could be created on the GPU: {err}");
                            return;
                        }
                    };
                    let partition = Arc::new(PartitionState::new(partition_id, idx));
                    partitions.insert(partition_id, Arc::clone(&partition));
                    partition
                }
            };
            states.entry(partition_id.index_id()).or_insert_with(|| IndexState {
                size: Arc::new(AtomicUsize::new(0)),
            });
            if embedding.as_slice().len() != dimensions.0.get() {
                warn!("add: wrong embedding dimension for primary id {primary_id:?}");
                return;
            }
            let key: u64 = primary_id.into();
            if let Some(Run::Add {
                partition: p,
                keys,
                rows,
                in_progress: ips,
            }) = runs.last_mut()
                && same(p, &partition)
                && keys.len() < MAX_RUN
            {
                keys.push(key);
                rows.extend_from_slice(embedding.as_slice());
                ips.push(in_progress);
                return;
            }
            runs.push(Run::Add {
                partition,
                keys: vec![key],
                rows: embedding.as_slice().to_vec(),
                in_progress: vec![in_progress],
            });
        }

        Message::Modify(VsIndexModify::RemoveVector {
            partition_id,
            primary_id,
            in_progress,
        }) => {
            let Some(partition) = partitions.get(&partition_id).map(Arc::clone) else {
                return;
            };
            let key: u64 = primary_id.into();
            if let Some(Run::Remove {
                partition: p,
                keys,
                in_progress: ips,
            }) = runs.last_mut()
                && same(p, &partition)
                && keys.len() < MAX_RUN
            {
                keys.push(key);
                ips.push(in_progress);
                return;
            }
            runs.push(Run::Remove {
                partition,
                keys: vec![key],
                in_progress: vec![in_progress],
            });
        }

        Message::Modify(VsIndexModify::RemovePartition { partition_id }) => {
            // runs queued before this message still hold their Arc; the index is destroyed when the last one drops
            partitions.remove(&partition_id);
        }

        Message::Search(VsIndexSearch::Count { index_key, tx }) => {
            let Some(index_id) = table.read().unwrap().index_id(&index_key) else {
                let err = anyhow!("count: {index_key:?} is not a known index");
                warn!("{err}");
                _ = tx.send(Err(err));
                return;
            };
            _ = tx.send(Ok(states
                .get(&index_id)
                .map(|state| state.size.load(Ordering::Relaxed))
                .unwrap_or(0)));
        }

        Message::Search(VsIndexSearch::Ann {
            index_key,
            embedding,
            limit,
            tx,
        }) => {
            let partition = table
                .read()
                .unwrap()
                .partition_id(&index_key, None)
                .and_then(|(partition_id, _)| partitions.get(&partition_id).map(Arc::clone));
            let Some(partition) = partition else {
                warn!("ann on {index_key:?}: no such partition yet, answering with no hits");
                _ = tx.send(Ok((vec![], vec![])));
                return;
            };
            push_ann(runs, partition, embedding, limit, tx, dimensions);
        }

        Message::Search(VsIndexSearch::FilteredAnn {
            index_key,
            embedding,
            filter,
            limit,
            tx,
        }) => {
            let found = table
                .read()
                .unwrap()
                .partition_id(&index_key, Some(filter.restrictions))
                .and_then(|(partition_id, restrictions)| {
                    partitions.get(&partition_id).map(|p| (Arc::clone(p), restrictions))
                });
            let Some((partition, restrictions)) = found else {
                debug!("filtered ann on {index_key:?}: no such partition yet, answering with no hits");
                _ = tx.send(Ok((vec![], vec![])));
                return;
            };
            match restrictions {
                // the partition key consumed every restriction: a plain ANN over that partition (usearch.rs:844-862)
                None => push_ann(runs, partition, embedding, limit, tx, dimensions),
                Some(restrictions) => {
                    if let Err(err) = validator::embedding_dimensions(&embedding, dimensions) {
                        _ = tx.send(Err(err));
                        return;
                    }
                    let filter = Filter {
                        restrictions,
                        allow_filtering: filter.allow_filtering,
                    };
                    // consecutive FilteredAnn requests on one partition share one call, like Ann runs (push_ann)
                    if let Some(Run::FilteredAnn {
                        partition: p,
                        queries,
                        filters,
                        limits,
                        txs,
                    }) = runs.last_mut()
                        && same(p, &partition)
                        && txs.len() < MAX_RUN
                    {
                        queries.extend_from_slice(embedding.as_slice());
                        filters.push(filter);
                        limits.push(limit.0.get());
                        txs.push(tx);
                        return;
                    }
                    runs.push(Run::FilteredAnn {
                        partition,
                        queries: embedding.as_slice().to_vec(),
                        filters: vec![filter],
                        limits: vec![limit.0.get()],
                        txs: vec![tx],
                    });
                }
            }
        }
    }
}

fn push_ann(
    runs: &mut Vec<Run>,
    partition: Arc<PartitionState>,
    embedding: Vector,
    limit: Limit,
    tx: oneshot::Sender<AnnR>,
    dimensions: Dimensions,
) {
    if let Err(err) = validator::embedding_dimensions(&embedding, dimensions) {
        tx.send(Err(err))
            .unwrap_or_else(|_| trace!("the requester of an ann went away"));
        return;
    }
    if let Some(Run::Ann {
        partition: p,
        queries,
        limits,
        txs,
    }) = runs.last_mut()
        && Arc::ptr_eq(p, &partition)
        && txs.len() < MAX_RUN
    {
        queries.extend_from_slice(embedding.as_slice());
        limits.push(limit.0.get());
        txs.push(tx);
        return;
    }
    runs.push(Run::Ann {
        partition,
        queries: embedding.as_slice().to_vec(),
        limits: vec![limit.0.get()],
        txs: vec![tx],
    });
}

fn new(
    index_fn: impl Fn() -> anyhow::Result<GpuIndex> + Send + Sync + 'static,
    index_key: IndexKey,
    dimensions: Dimensions,
    table: Arc<RwLock<impl TableSearch + Send + Sync + 'static>>,
    worker: async_channel::Sender<Worker>,
    memory: mpsc::Sender<Memory>,
) -> anyhow::Result<(mpsc::Sender<VsIndexModify>, mpsc::Sender<VsIndexSearch>)> {
    let (tx_modify, mut rx_modify) = mpsc::channel(perf::channel_size().into());
    let (tx_search, mut rx_search) = mpsc::channel(perf::channel_size().into());

    tokio::spawn(
        {
            let index_key = index_key.clone();
            async move {
                debug!("starting");
                let mut states: BTreeMap<IndexId, IndexState> = BTreeMap::new();
                let mut partitions: BTreeMap<PartitionId, Arc<PartitionState>> = BTreeMap::new();
                let mut gate = MemoryGate {
                    rx: memory.subscribe_allocate().await,
                    refused_before: false,
                };

                // vs_index::recv waits for the first message (searches first); everything already queued behind
                // it is drained without waiting, searches first again, up to MAX_RUN per kind
                while let Some(first) = crate::vs_index::recv(&mut rx_search, &mut rx_modify).await {
                    let mut batch = vec![first];
                    while batch.len() < MAX_RUN {
                        match rx_search.try_recv() {
                            Ok(msg) => batch.push(Message::Search(msg)),
                            Err(_) => break,
                        }
                    }
                    while batch.len() < 2 * MAX_RUN {
                        match rx_modify.try_recv() {
                            Ok(msg) => batch.push(Message::Modify(msg)),
                            Err(_) => break,
                        }
                    }

                    let mut runs = Vec::new();
                    for msg in batch {
                        if !gate.admits(&msg, &index_key) {
                            continue;
                        }
                        enqueue(
                            &mut runs,
                            msg,
                            &index_fn,
                            &mut states,
                            &mut partitions,
                            table.as_ref(),
                            dimensions,
                        );
                    }

                    for run in runs {
                        // capacity ahead of insertions (usearch.rs:908-921); vsb_reserve publishes a new store and
                        // never blocks the searches running on the old one, so no exclusive permit is needed
                        if let Run::Add { partition, keys, .. } = &run
                            && let Some(capacity) = partition.needs_more_capacity(keys.len())
                        {
                            let partition = Arc::clone(partition);
                            worker
                                .spawn_blocking(move || match partition.idx.reserve(capacity) {
                                    Err(err) => error!("growing a partition to {capacity} slots failed: {err}"),
                                    Ok(()) => partition.capacity.store(partition.idx.capacity(), Ordering::Relaxed),
                                })
                                .await;
                        }
                        let index_id = match &run {
                            Run::Add { partition, .. }
                            | Run::Remove { partition, .. }
                            | Run::Ann { partition, .. }
                            | Run::FilteredAnn { partition, .. } => partition.partition_id.index_id(),
                        };
                        let size = states
                            .entry(index_id)
                            .or_insert_with(|| IndexState {
                                size: Arc::new(AtomicUsize::new(0)),
                            })
                            .size
                            .clone();
                        let table = Arc::clone(&table);
                        // modifies of one actor run in order on the worker pool's blocking lane; searches overlap
                        // them freely (the library serves them from the published view)
                        match run {
                            run @ (Run::Ann { .. } | Run::FilteredAnn { .. }) => {
                                worker
                                    .spawn_non_blocking(move || execute(run, table.as_ref(), &size))
                                    .await
                            }
                            run => worker.spawn_blocking(move || execute(run, table.as_ref(), &size)).await,
                        }
                    }
                }
                debug!("finished");
            }
        }
        .instrument(error_span!("gpu", "{index_key}")),
    );

    Ok((tx_modify, tx_search))
}

pub struct GpuIndexFactory {
    worker: async_channel::Sender<Worker>,
    memory: mpsc::Sender<Memory>,
    /// CUDA ordinals: one entry = one GPU per partition index, several = every index sharded over them
    devices: Vec<i32>,
}

impl VsIndexFactory for GpuIndexFactory {
    fn create_index(
        &self,
        index: VsIndexConfiguration,
        table: Arc<RwLock<Table>>,
    ) -> anyhow::Result<(mpsc::Sender<VsIndexModify>, mpsc::Sender<VsIndexSearch>)> {
        let mut options = sys::vsb_options {
            dimensions: index.dimensions.0.get() as u32,
            metric: metric_of(index.quantization, index.space_type)?,
            storage: storage_of(index.quantization),
            connectivity: index.connectivity.0 as u32,
            expansion_add: index.expansion_add.0 as u32,
            expansion_search: index.expansion_search.0 as u32,
            device: self.devices.first().copied().unwrap_or(-1),
            // f32 rows: walk a bf16 copy and re-rank on the f32 rows — same results, half the bytes per hop
            flags: if index.quantization == Quantization::F32 {
                sys::VSB_FLAG_BF16_TRAVERSAL
            } else {
                sys::VSB_FLAG_NONE
            },
            ..Default::default()
        };
        if self.devices.len() > 1 {
            options.n_devices = self.devices.len().min(8) as i32;
            for (slot, device) in options.device_ids.iter_mut().zip(&self.devices) {
                *slot = *device;
            }
        }
        let (space, dimensions) = (index.space_type, index.dimensions);
        new(
            move || GpuIndex::new(&options, space, dimensions),
            index.key,
            index.dimensions,
            table,
            self.worker.clone(),
            self.memory.clone(),
        )
    }

    fn index_engine_version(&self) -> String {
        sys::version()
    }
}

/// vs_index/mod.rs: `pub(crate) fn new_index_factory_gpu(...)` forwards here.
pub fn new_gpu(
    devices: Vec<i32>,
    worker: async_channel::Sender<Worker>,
    memory: mpsc::Sender<Memory>,
) -> anyhow::Result<GpuIndexFactory> {
    if devices.len() > 8 {
        bail!("vsb200 shards one index over at most 8 devices");
    }
    Ok(GpuIndexFactory {
        worker,
        memory,
        devices,
    })
}
