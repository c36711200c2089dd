"""GPU parity tests: the CUDA path, called through the C ABI (ctypes), against the CPU oracle on the
same seeded inputs.  Bit-exact for ids, keys, integer graph rows AND for fp32 distances (the
kernels and oracle/exact.c share one defined summation order); ANN recall is measured against
exact ground truth and compared with the USearch-equivalent CPU HNSW at the same M/ef."""
import threading

import numpy as np
import pytest

import oracle as O
from conftest import embedding_like, sift_like
from oracle import graph_oracle

pytestmark = pytest.mark.gpu

INVALID = np.uint64(0xFFFFFFFFFFFFFFFF)


def V():
    import vector_store_b200 as v
    return v


def make_index(x, keys, metric, storage, **kw):
    v = V()
    idx = v.GpuIndex(x.shape[1], v.Metric(metric), v.Scalar(storage), **kw)
    idx.reserve(len(x) + 64)
    idx.add_batch(keys, x)
    return idx


def assert_bit_equal(gk, gd, gc, ok, od, oc):
    assert np.array_equal(gc, oc)
    assert np.array_equal(gk, ok)
    assert np.array_equal(gd.view(np.uint32), od.view(np.uint32)), \
        f"max |diff| = {np.nanmax(np.abs(gd[np.isfinite(od)] - od[np.isfinite(od)]))}"


PAIRS = [(s, m) for s in (O.F32, O.F16, O.BF16, O.I8) for m in (O.L2SQ, O.COS, O.IP)] + [(O.B1, O.HAMMING)]


@pytest.mark.parametrize("storage,metric", PAIRS)
def test_exact_bit_parity_ragged(storage, metric):
    rng = np.random.default_rng(100 + storage * 7 + metric)
    n, dim, nq, k = 5003, 100, 37, 10  # dim not a multiple of any chunk size, n/nq not tile multiples
    x = rng.standard_normal((n, dim)).astype(np.float32)
    if storage == O.I8:
        x = np.clip(x * 0.4, -1.2, 1.2).astype(np.float32)
    q = rng.standard_normal((nq, dim)).astype(np.float32) * (0.4 if storage == O.I8 else 1.0)
    keys = rng.permutation(n).astype(np.uint64) + np.uint64(1 << 48)  # epoch bits set, key order != slot order
    idx = make_index(x, keys, metric, storage)
    gk, gd, gc = idx.search_batch(q, k, exact=True)
    ok, od, oc, _ = O.exact_topk(x, q, k, metric, storage, keys=keys)
    assert_bit_equal(gk, gd, gc, ok, od, oc)
    # un-built index: the ANN entry point is the brute-force tail => identical
    gk2, gd2, gc2 = idx.search_batch(q, k)
    assert_bit_equal(gk2, gd2, gc2, ok, od, oc)
    space = {O.L2SQ: V().SpaceType.Euclidean, O.COS: V().SpaceType.Cosine, O.IP: V().SpaceType.DotProduct,
             O.HAMMING: V().SpaceType.Hamming}[metric]
    for d in gd.ravel():
        V().Distance.try_from(float(d), space, dim)  # output contract distance.rs:58-105


def test_exact_ties_by_key_sift_shaped():
    n, dim, nq, k = 20000, 128, 64, 10
    x = sift_like(n, dim)
    x[5000:5040] = x[4000]  # 41 identical rows straddle any k boundary
    q = sift_like(nq, dim, seed=4321)
    q[0] = x[4000]
    rng = np.random.default_rng(5)
    keys = rng.permutation(n).astype(np.uint64)
    idx = make_index(x, keys, O.L2SQ, O.F32)
    gk, gd, gc = idx.search_batch(q, k, exact=True)
    ok, od, oc, _ = O.exact_topk(x, q, k, O.L2SQ, O.F32, keys=keys)
    assert_bit_equal(gk, gd, gc, ok, od, oc)
    assert np.all(gd[0] == 0.0) and list(gk[0]) == sorted(gk[0])


@pytest.mark.parametrize("k", [1, 33, 100, 200])
def test_exact_k_variants_and_small_index(k):
    rng = np.random.default_rng(k)
    x = rng.standard_normal((150, 24)).astype(np.float32)
    q = rng.standard_normal((5, 24)).astype(np.float32)
    keys = np.arange(150, dtype=np.uint64) * 3
    idx = make_index(x, keys, O.COS, O.F32)
    gk, gd, gc = idx.search_batch(q, k, exact=True)
    ok, od, oc, _ = O.exact_topk(x, q, k, O.COS, O.F32, keys=keys)
    assert_bit_equal(gk, gd, gc, ok, od, oc)
    assert np.all(gc == min(k, 150))
    assert np.all(np.diff(gd[:, :min(k, 150)], axis=1) >= 0)


def test_tombstones_and_filtered_search():
    rng = np.random.default_rng(11)
    n, dim = 4000, 48
    x = rng.standard_normal((n, dim)).astype(np.float32)
    q = rng.standard_normal((20, dim)).astype(np.float32)
    keys = np.arange(n, dtype=np.uint64) | np.uint64(3 << 48)  # epoch 3, row id = i
    idx = make_index(x, keys, O.L2SQ, O.BF16)
    dead = rng.choice(n, 900, replace=False)
    assert idx.remove_batch(keys[dead]) == 900
    assert idx.remove_batch(keys[dead[:10]]) == 0  # already gone
    assert idx.size() == n - 900
    alive = np.ones(n, np.uint8)
    alive[dead] = 0
    gk, gd, gc = idx.search_batch(q, 10, exact=True)
    ok, od, oc, _ = O.exact_topk(x, q, 10, O.L2SQ, O.BF16, keys=keys, alive=alive)
    assert_bit_equal(gk, gd, gc, ok, od, oc)
    # N1: bitmap predicate over row ids (low 48 bits of the key)
    allow_rows = rng.random(n) < 0.05
    bm = np.zeros((n + 31) // 32, np.uint32)
    for r in np.nonzero(allow_rows)[0]:
        bm[r >> 5] |= np.uint32(1 << (r & 31))
    alive2 = (alive.astype(bool) & allow_rows).astype(np.uint8)
    ok2, od2, oc2, _ = O.exact_topk(x, q[:1], 10, O.L2SQ, O.BF16, keys=keys, alive=alive2)
    hits = idx.filtered_search_bitmap(q[0], 10, bm, n)
    assert [h[0] for h in hits] == [int(v) for v in ok2[0][:oc2[0]]]
    assert np.array_equal(np.array([h[1] for h in hits], np.float32).view(np.uint32),
                          od2[0][:oc2[0]].view(np.uint32))


def test_merge_topk_kernel_matches_numpy():
    import torch
    from importlib import import_module
    index_mod = import_module("vector_store_b200.host.index")
    rng = np.random.default_rng(2)
    parts, nq, k = 5, 300, 10
    d = np.sort(rng.integers(0, 50, size=(parts, nq, k)).astype(np.float32), axis=2)  # many ties
    keys = rng.permutation(parts * nq * k).astype(np.uint64).reshape(parts, nq, k)
    keys[:, :, 7:] = INVALID
    d[:, :, 7:] = np.inf
    order = np.lexsort((keys, d), axis=2) if False else None
    for p in range(parts):  # make each list ascending by (dist, key)
        for i in range(nq):
            o = np.lexsort((keys[p, i], d[p, i]))
            keys[p, i], d[p, i] = keys[p, i][o], d[p, i][o]
    tk = torch.from_numpy(keys.view(np.int64)).cuda()
    td = torch.from_numpy(d).cuda()
    ok = torch.empty((nq, k), dtype=torch.int64, device="cuda")
    od = torch.empty((nq, k), dtype=torch.float32, device="cuda")
    oc = torch.empty(nq, dtype=torch.int32, device="cuda")
    index_mod.merge_topk_dev(tk.data_ptr(), td.data_ptr(), parts, nq, k, ok.data_ptr(), od.data_ptr(), oc.data_ptr(),
                             0, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    gk = ok.cpu().numpy().view(np.uint64)
    gd = od.cpu().numpy()
    for i in range(nq):
        ak = keys[:, i, :].ravel()
        ad = d[:, i, :].ravel()
        o = np.lexsort((ak, ad))[:k]
        assert np.array_equal(gk[i], ak[o]) and np.array_equal(gd[i], ad[o])
    assert np.all(oc.cpu().numpy() == k)
    # strided form: one record per part [q*k keys | q*k distances], as a single all-gather delivers it
    rec = torch.empty(parts * nq * k * 12, dtype=torch.uint8, device="cuda")
    for p in range(parts):
        base = p * nq * k * 12
        rec[base:base + nq * k * 8].view(torch.int64).copy_(tk[p].reshape(-1))
        rec[base + nq * k * 8:base + nq * k * 12].view(torch.float32).copy_(td[p].reshape(-1))
    ok2 = torch.empty_like(ok)
    od2 = torch.empty_like(od)
    index_mod.merge_topk_strided_dev(rec.data_ptr(), rec.data_ptr() + nq * k * 8, parts, nq * k * 12 // 8,
                                     nq * k * 12 // 4, nq, k, ok2.data_ptr(), od2.data_ptr(), 0, 0,
                                     torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert torch.equal(ok2, ok) and torch.equal(od2, od)


# ---- reference golden vectors through the actor mirror (reads like the reference's own tests) ----------
def cfg(dim, space="Euclidean", quant="F32", **kw):
    v = V()
    return v.VsIndexConfiguration("vector.store", dim, space_type=v.SpaceType[space],
                                  quantization=v.Quantization[quant], **kw)


def new_actor(config):
    a = V().new_index_factory_gpu()(config)
    a.reserve_increment = 1000
    return a


def test_g1_add_or_replace_size_ann():
    # vs_index/usearch.rs:1298-1458
    a = new_actor(cfg(3))
    a.add_vector(0, 1, [1.0, 1.0, 1.0])
    a.add_vector(0, 2, [2.0, -2.0, 2.0])
    a.add_vector(0, 3, [3.0, 3.0, 3.0])
    assert a.count() == 3
    keys, dists = a.ann([2.2, -2.2, 2.2], 1)
    assert keys == [2] and len(dists) == 1
    a.remove_vector(0, 3)
    assert a.count() == 2
    a.add_vector(0, 3, [2.1, -2.1, 2.1])
    assert a.count() == 3
    assert a.ann([2.2, -2.2, 2.2], 1)[0] == [3]
    a.remove_vector(0, 3)
    assert a.count() == 2
    assert a.ann([2.2, -2.2, 2.2], 1)[0] == [2]
    a.stop()


def test_g2_similarity_scores_are_decreasing_and_correctly_converted():
    # tests/integration/vs_index.rs:1746-1887
    v = V()
    a = new_actor(cfg(1))
    for pk, x in ((10, 0.0), (11, 1.0), (13, 3.0)):
        a.add_vector(0, pk, [x])
    keys, dists = a.ann([0.0], 3)
    assert keys == [10, 11, 13] and [float(d) for d in dists] == [0.0, 1.0, 9.0]
    scores = [v.SimilarityScore.from_distance(d).value for d in dists]
    assert np.allclose(scores, [1.0, 0.5, 0.1], atol=1e-5) and scores[0] > scores[1] > scores[2]


def test_g3_g10_simple_ann_wrong_dim_and_empty():
    # tests/integration/vs_index.rs:226-311, 441-480, 1889-1951
    v = V()
    a = new_actor(cfg(3))
    assert a.ann([1.0, 2.0, 3.0], 5) == ([], []) and a.count() == 0
    a.add_vector(0, 1, [1.0, 1.0, 1.0])
    a.add_vector(0, 2, [2.0, -2.0, 2.0])
    a.add_vector(0, 3, [3.0, 3.0, 3.0])
    assert a.ann([2.1, -2.0, 2.0], 1)[0] == [2]
    with pytest.raises(v.WrongEmbeddingDimension):
        a.ann([1.0, 2.0], 1)
    a.add_vector(0, 4, [1.0, 2.0])  # wrong dimension on add: logged and dropped
    assert a.count() == 3
    a.add_vector(0, 1, [9.0, 9.0, 9.0])  # duplicate key: logged and swallowed (usearch multi=false)
    assert a.count() == 3
    assert a.ann([1.0, 1.0, 1.0], 5)[0] == [1, 2, 3] or len(a.ann([1.0, 1.0, 1.0], 5)[0]) == 3
    a.can_allocate = False  # memory gate: usearch.rs:1460-1524 allocate_parameter_works
    a.add_vector(0, 5, [5.0, 5.0, 5.0])
    assert a.count() == 3
    a.remove_partition(0)
    assert a.count() == 0 and a.ann([1.0, 1.0, 1.0], 5) == ([], [])


def test_g4_quantization_is_effectively_applied():
    # tests/integration/quantization.rs:40-124
    def dist(quant):
        a = new_actor(cfg(3, quant=quant))
        a.add_vector(0, 1, [0.9, 0.1, 0.1])
        return float(a.ann([1.0, 0.0, 0.0], 1)[1][0])
    assert dist("F32") < 0.1
    assert dist("I8") > 300 and dist("I8") == 507.0


@pytest.mark.parametrize("quant", ["F32", "F16", "BF16", "I8", "B1"])
def test_g5_g6_self_distance_zero(quant):
    # tests/integration/quantization.rs:175-259 (dim 1536) and :293-358 (B1, dim 100)
    for dim in (1536, 100):
        a = new_actor(cfg(dim, quant=quant))
        x = np.full(dim, 0.5, np.float32)
        a.add_vector(0, 1, x)
        a.add_vector(0, 2, -x)
        keys, dists = a.ann(x, 1)
        assert keys == [1] and float(dists[0]) == 0.0
        keys, dists = a.filtered_ann(x, 2, lambda row: row == 1, max_row_id=2)  # "IN" filter variant
        assert keys == [1] and float(dists[0]) == 0.0


def test_g9_similarity_function_semantics():
    # crates/validator/src/similarity_functions.rs:113-178
    rows = {1: [1, 0, 0], 2: [0, 1, 0], 3: [0, 0, 1], 4: [2, 0, 0]}
    expect_first = {"Euclidean": {1}, "Cosine": {1, 4}, "DotProduct": {4}}
    for space, first in expect_first.items():
        a = new_actor(cfg(3, space=space))
        for pk, x in rows.items():
            a.add_vector(0, pk, np.array(x, np.float32))
        keys, dists = a.ann([1.0, 0.0, 0.0], 4)
        d0 = float(dists[0])
        assert {k for k, d in zip(keys, dists) if float(d) == d0} == first


def test_g11_concurrent_add_and_search():
    # vs_index/usearch.rs:1526-1607: 2 x cores concurrent adds + searches at dim 1024, exact final count
    dim, per = 1024, 40
    a = new_actor(cfg(dim))
    a.reserve_increment = 4096
    a.add_vector(0, 10 ** 6, np.ones(dim, np.float32))
    errors = []
    lock = threading.Lock()

    def adder(t):
        rng = np.random.default_rng(t)
        for i in range(per):
            with lock:  # the reference's actor loop serialises dispatch; the engine calls run concurrently
                pass
            try:
                a.partitions[0].idx.add(t * 1000 + i, rng.standard_normal(dim).astype(np.float32))
            except Exception as e:  # noqa: BLE001
                errors.append(e)

    def searcher(t):
        rng = np.random.default_rng(100 + t)
        for _ in range(per):
            try:
                a.partitions[0].idx.search(rng.standard_normal(dim).astype(np.float32), 5)
            except Exception as e:  # noqa: BLE001
                errors.append(e)

    a.partitions[0].idx.reserve(8 * per + 64)
    ts = [threading.Thread(target=adder, args=(t,)) for t in range(8)] + \
         [threading.Thread(target=searcher, args=(t,)) for t in range(8)]
    [t.start() for t in ts]
    [t.join() for t in ts]
    assert not errors, errors[:3]
    assert a.partitions[0].idx.size() == 8 * per + 1


# ---- graph build + ANN ------------------------------------------------------------------------------
def test_graph_build_bit_exact_vs_oracle():
    rng = np.random.default_rng(21)
    n, dim = 1500, 32
    x = rng.standard_normal((n, dim)).astype(np.float32)
    keys = rng.permutation(n).astype(np.uint64)
    idx = make_index(x, keys, O.L2SQ, O.F32, connectivity=8, expansion_add=32)  # R = 16, k_init = 16
    dead = rng.choice(n, 100, replace=False)
    idx.remove_batch(keys[dead])
    idx.set_search_params(min_graph_size=1000)
    idx.build()
    rows, gkeys = idx.export_graph()
    alive = np.ones(n, bool)
    alive[dead] = False
    # vsb_build compacts tombstoned rows away: the graph is over the live rows in their original order
    assert rows.shape == (n - 100, 32) and np.array_equal(gkeys, keys[alive])
    want = graph_oracle.build_graph(x[alive], k_init=16, R=16, metric=O.L2SQ, storage=O.F32, keys=keys[alive], stride=32)
    assert np.array_equal(rows, want), f"{(rows != want).any(axis=1).sum()} rows differ"


@pytest.mark.parametrize("storage,metric,dim,clusters", [(O.F32, O.COS, 96, 32), (O.BF16, O.COS, 768, 64),
                                                         (O.F32, O.L2SQ, 128, 0)])
def test_ann_recall_vs_cpu_hnsw(storage, metric, dim, clusters):
    n, nq, k = 30000, 500, 10
    if clusters:
        x = embedding_like(n, dim, n_clusters=clusters)
        q = embedding_like(nq, dim, seed=4321, n_clusters=clusters)
    else:
        x, q = sift_like(n, dim), sift_like(nq, dim, seed=4321)
    keys = np.arange(n, dtype=np.uint64)
    idx = make_index(x, keys, metric, storage)  # defaults M=16 / ef_add=128 / ef_search=64
    idx.build()
    st = idx.stats()
    assert st["n_graphed"] == n and st["graph_degree"] == 32
    tk, td, tc = idx.search_batch(q, k, exact=True)
    gk, gd, gc = idx.search_batch(q, k)
    recall_gpu = O.recall_at_k(gk, tk)
    h = O.HnswCpu(dim, metric, n, storage=storage)
    h.add(keys, x)
    hk, _ = h.search(q, k)
    recall_cpu = O.recall_at_k(hk, tk)
    print(f"recall@10 gpu={recall_gpu:.4f} cpu_hnsw={recall_cpu:.4f} (storage={storage} metric={metric} dim={dim})")
    assert np.all(gc == k)
    assert np.all(np.diff(gd, axis=1) >= 0)
    if clusters:  # iid 128-d data has no neighbourhood structure: ef=64 gives ~0.66 for HNSW too
        assert recall_gpu >= 0.95
    # parity bar: the same M/ef must not do worse than the CPU HNSW (whose parallel build is not
    # deterministic: +-0.01 run to run on the iid case)
    assert recall_gpu >= recall_cpu - (0.01 if clusters else 0.025)
    # distances of ANN hits are the canonical exact distances of those rows
    od = O.distance_matrix(x[gk[0].astype(np.int64)], q[:1], metric, storage)[0]
    assert np.array_equal(gd[0].view(np.uint32), od.view(np.uint32))


def test_ann_sees_vectors_added_and_removed_after_build():
    n, dim = 20000, 64
    x = embedding_like(n + 200, dim, n_clusters=16)
    keys = np.arange(n + 200, dtype=np.uint64)
    idx = make_index(x[:n], keys[:n], O.COS, O.F32)
    idx.reserve(n + 1000)
    idx.build()
    idx.add_batch(keys[n:], x[n:])  # un-graphed tail
    gk, gd, gc = idx.search_batch(x[n:n + 50], 3)
    assert np.array_equal(gk[:, 0], keys[n:n + 50]) and np.all(gd[:, 0] <= 1e-6)
    gk, _, _ = idx.search_batch(x[:50], 1)
    assert np.array_equal(gk[:, 0], keys[:50])
    idx.remove_batch(keys[:50])
    gk, _, gc = idx.search_batch(x[:50], 5)
    assert not np.isin(gk, keys[:50]).any() and np.all(gc == 5)
    assert idx.size() == n + 200 - 50


def test_c1_full_size_properties():
    # BASELINE config #1: 100k x 128 f32 L2sq, k=10 — size-independent properties + oracle on a query subset
    n, dim, k = 100_000, 128, 10
    x = sift_like(n, dim)
    q = sift_like(256, dim, seed=4321)
    keys = np.arange(n, dtype=np.uint64)
    idx = make_index(x, keys, O.L2SQ, O.F32)
    gk, gd, gc = idx.search_batch(np.concatenate([q, x[:64]]), k, exact=True)
    assert np.all(gc == k) and np.all(np.diff(gd, axis=1) >= 0)
    assert np.all(gd[256:, 0] == 0.0)                        # a stored row is its own nearest neighbour
    gk2, gd2, _ = idx.search_batch(np.concatenate([q, x[:64]]), k, exact=True)
    assert np.array_equal(gk, gk2) and np.array_equal(gd, gd2)  # idempotent / deterministic
    ok, od, oc, _ = O.exact_topk(x, q[:32], k, O.L2SQ, O.F32, keys=keys)
    assert_bit_equal(gk[:32], gd[:32], gc[:32], ok, od, oc)
    idx.build()
    ak, ad, ac = idx.search_batch(q, k)
    recall = O.recall_at_k(ak, gk[:256])
    idx.set_search_params(expansion_search=512)
    ak2, _, _ = idx.search_batch(q, k)
    recall_hi = O.recall_at_k(ak2, gk[:256])
    print(f"C1 100k x 128 L2sq recall@10: ef=64 {recall:.4f}, ef=512 {recall_hi:.4f}")
    assert recall_hi >= recall and recall_hi >= 0.9


@pytest.mark.parametrize("storage,dim", [(O.F32, 96), (O.BF16, 768)])
def test_small_batch_paths_cta_per_query(storage, dim):
    # batch <= 256 runs the CTA-per-query kernel (K4b); batch < 16 also uses the seed-scan kernel
    n, k = 30000, 10
    x = embedding_like(n, dim, n_clusters=32)
    q = embedding_like(300, dim, seed=4321, n_clusters=32)
    keys = np.arange(n, dtype=np.uint64) + np.uint64(5 << 48)
    idx = make_index(x, keys, O.COS, storage)
    idx.build()
    tk, td, _ = idx.search_batch(q, k, exact=True)
    big_k, big_d, _ = idx.search_batch(q, k)  # warp-per-query kernel (batch 300)
    for nq in (1, 5, 16, 100, 256):
        gk, gd, gc = idx.search_batch(q[:nq], k)
        assert np.all(gc == k) and np.all(np.diff(gd, axis=1) >= 0)
        r = O.recall_at_k(gk, tk[:nq])
        print(f"batch {nq}: recall@10 = {r:.4f}")
        assert r >= 0.9 if nq < 16 else r >= 0.95
        od = O.distance_matrix(x[(gk[0] - np.uint64(5 << 48)).astype(np.int64)], q[:1], O.COS, storage)[0]
        assert np.array_equal(gd[0].view(np.uint32), od.view(np.uint32))
    assert O.recall_at_k(big_k, tk) >= 0.95


def test_bf16_traversal_flag_keeps_fp32_distances():
    # VSB_FLAG_BF16_TRAVERSAL: K4 walks a bf16 copy, K3 re-ranks on the f32 rows => canonical f32 distances
    n, dim, k = 30000, 768, 10
    x = embedding_like(n, dim, n_clusters=64)
    q = embedding_like(400, dim, seed=4321, n_clusters=64)
    keys = np.arange(n, dtype=np.uint64)
    v = V()
    idx = v.GpuIndex(dim, v.Metric.Cos, v.Scalar.F32, bf16_traversal=True)
    idx.reserve(n + 100)
    idx.add_batch(keys, x)
    idx.build()
    tk, td, _ = idx.search_batch(q, k, exact=True)
    ok, od, _, _ = O.exact_topk(x, q[:8], k, O.COS, O.F32, keys=keys)
    assert np.array_equal(tk[:8], ok) and np.array_equal(td[:8].view(np.uint32), od.view(np.uint32))
    for nq in (400, 3):
        gk, gd, gc = idx.search_batch(q[:nq], k)
        r = O.recall_at_k(gk, tk[:nq])
        print(f"bf16 traversal, batch {nq}: recall@10 = {r:.4f}")
        assert np.all(gc == k) and np.all(np.diff(gd, axis=1) >= 0) and r >= 0.95
        d0 = O.distance_matrix(x[gk[0].astype(np.int64)], q[:1], O.COS, O.F32)[0]
        assert np.array_equal(gd[0].view(np.uint32), d0.view(np.uint32))
    idx.add_batch(np.arange(n, n + 50, dtype=np.uint64), q[:50])  # tail + traversal copy stay in sync
    gk, gd, _ = idx.search_batch(q[:50], 1)
    assert np.array_equal(gk[:, 0], np.arange(n, n + 50, dtype=np.uint64))


def test_i8_traversal_flag_keeps_fp32_distances_and_recall():
    # VSB_FLAG_I8_TRAVERSAL: K4 walks a scaled-int8 copy (cosine, f32 storage), K3 re-ranks 4k candidates on the
    # f32 rows => canonical f32 distances; recall must stay with the bf16 traversal's
    n, dim, k = 30000, 768, 10
    x = embedding_like(n, dim, n_clusters=64)
    q = embedding_like(400, dim, seed=4321, n_clusters=64)
    keys = np.arange(n, dtype=np.uint64)
    v = V()
    recalls = {}
    for mode in ("bf16", "i8"):
        idx = v.GpuIndex(dim, v.Metric.Cos, v.Scalar.F32, bf16_traversal=True, i8_traversal=(mode == "i8"))
        idx.reserve(n + 100)
        idx.add_batch(keys[: n // 2], x[: n // 2])
        idx.remove_batch(keys[100:200])                       # compaction at build carries the int8 copy along
        idx.add_batch(keys[n // 2:], x[n // 2:])
        idx.build()
        alive = np.ones(n, np.uint8)
        alive[100:200] = 0
        tk, td, _ = idx.search_batch(q, k, exact=True)
        ok, od, _, _ = O.exact_topk(x, q[:8], k, O.COS, O.F32, keys=keys, alive=alive)
        assert np.array_equal(tk[:8], ok) and np.array_equal(td[:8].view(np.uint32), od.view(np.uint32))
        for nq in (400, 3):
            gk, gd, gc = idx.search_batch(q[:nq], k)
            r = O.recall_at_k(gk, tk[:nq])
            print(f"{mode} traversal, batch {nq}: recall@10 = {r:.4f}")
            assert np.all(gc == k) and np.all(np.diff(gd, axis=1) >= 0) and r >= 0.95
            d0 = O.distance_matrix(x[gk[0].astype(np.int64)], q[:1], O.COS, O.F32)[0]
            assert np.array_equal(gd[0].view(np.uint32), d0.view(np.uint32))
            recalls[(mode, nq)] = r
        idx.add_batch(np.arange(n, n + 50, dtype=np.uint64), q[:50])  # streamed rows get their int8 copy too
        idx.insert_pending()
        gk, gd, _ = idx.search_batch(q[:50], 1)
        assert np.array_equal(gk[:, 0], np.arange(n, n + 50, dtype=np.uint64))
        idx.close()
    assert recalls[("i8", 400)] >= recalls[("bf16", 400)] - 0.01
    # the flag is ignored (bf16 / native traversal) where the scaled-int8 cosine trick does not apply
    idx = v.GpuIndex(64, v.Metric.L2sq, v.Scalar.F32, i8_traversal=True)
    idx.reserve(5000)
    xs = embedding_like(5000, 64, n_clusters=8)
    idx.add_batch(np.arange(5000, dtype=np.uint64), xs)
    idx.build()
    gk, _, _ = idx.search_batch(xs[:20], 1)
    assert np.array_equal(gk[:, 0], np.arange(20, dtype=np.uint64))
    idx.close()


def test_streaming_insert_k7():
    # C5-shaped: build on 70 % of the data, stream the rest in (K7), delete some, recall stays high
    n, dim, k = 40000, 96, 10
    x = embedding_like(n, dim, n_clusters=32)
    q = embedding_like(500, dim, seed=4321, n_clusters=32)
    keys = np.arange(n, dtype=np.uint64)
    n0 = 28000
    idx = make_index(x[:n0], keys[:n0], O.COS, O.F32)
    idx.reserve(n + 64)
    idx.build()
    idx.set_search_params(stream_threshold=2048)
    for b in range(n0, n, 1000):      # CDC-style batches; every 2048 pending rows trigger a K7 insert
        idx.add_batch(keys[b:b + 1000], x[b:b + 1000])
    st = idx.stats()
    assert st["n_graphed"] >= n - 2048 and st["n_slots"] == n
    idx.insert_pending()
    assert idx.stats()["n_graphed"] == n
    dead = np.arange(0, n, 17)
    idx.remove_batch(keys[dead])
    tk, _, _ = idx.search_batch(q, k, exact=True)
    gk, gd, gc = idx.search_batch(q, k)
    r = O.recall_at_k(gk, tk)
    idx.build()                        # full rebuild as the yardstick
    bk, _, _ = idx.search_batch(q, k)
    r_rebuilt = O.recall_at_k(bk, tk)
    print(f"recall@10 after streaming 30% of the rows in: {r:.4f}; after full rebuild: {r_rebuilt:.4f}")
    assert np.all(gc == k) and not np.isin(gk, keys[dead]).any()
    assert r >= 0.93 and r >= r_rebuilt - 0.04
    # streamed rows are reachable through the graph (not only through the tail)
    idx.set_search_params(expansion_search=128)
    sk, sd, _ = idx.search_batch(x[n - 100:], 1)
    print(f"streamed rows found as their own top-1: {np.mean(sk[:, 0] == keys[n - 100:]):.3f}")
    assert np.mean(sk[:, 0] == keys[n - 100:]) >= 0.9


def test_hybrid_build_allpairs_prefix_plus_streaming():
    # above VSB_ALLPAIRS_MAX rows vsb_build all-pairs-builds a prefix and streams the rest in (K7)
    import os
    n, dim, k = 50000, 96, 10
    x = embedding_like(n, dim, n_clusters=32)
    q = embedding_like(500, dim, seed=4321, n_clusters=32)
    keys = np.arange(n, dtype=np.uint64)
    os.environ["VSB_ALLPAIRS_MAX"] = "20000"
    os.environ["VSB_ALLPAIRS_PREFIX"] = "20000"
    try:
        idx = make_index(x, keys, O.COS, O.BF16)
    finally:
        del os.environ["VSB_ALLPAIRS_MAX"]
        del os.environ["VSB_ALLPAIRS_PREFIX"]
    idx.build()
    st = idx.stats()
    assert st["n_graphed"] == n
    tk, _, _ = idx.search_batch(q, k, exact=True)
    gk, _, gc = idx.search_batch(q, k)
    r = O.recall_at_k(gk, tk)
    print(f"hybrid build (20k all-pairs + 30k streamed + refine): recall@10 = {r:.4f}")
    assert np.all(gc == k) and r >= 0.93


def test_streamed_build_is_deterministic(monkeypatch):
    # K7 links the rows beyond the all-pairs prefix in batches of 8192, and the reverse links of one batch compete for
    # the same old rows: two builds of the same rows must still give the same graph bit for bit, and the same results
    n, dim, k = 60000, 64, 10
    x = embedding_like(n, dim, n_clusters=32)
    q = embedding_like(500, dim, seed=4321, n_clusters=32)
    keys = np.arange(n, dtype=np.uint64)
    monkeypatch.setenv("VSB_ALLPAIRS_MAX", "10000")                   # read when the index is created
    monkeypatch.setenv("VSB_ALLPAIRS_PREFIX", "10000")
    runs = []
    for _ in range(2):
        idx = make_index(x, keys, O.COS, O.BF16)
        idx.build()
        assert idx.build_stats()["stream_rows"] == n - 10000
        rows, _ = idx.export_graph()
        runs.append((rows, idx.search_batch(q, k)))
        idx.close()
    (g0, r0), (g1, r1) = runs
    assert np.array_equal(g0, g1), f"{(g0 != g1).any(axis=1).sum()} rows differ"
    assert all(np.array_equal(a, b) for a, b in zip(r0, r1))


def test_snapshot_roundtrip(tmp_path):
    # N3: save / load reproduces exact and ANN results (keys, tombstones, rows, graph)
    n, dim, k = 20000, 64, 10
    x = embedding_like(n, dim, n_clusters=16)
    q = embedding_like(200, dim, seed=4321, n_clusters=16)
    keys = (np.arange(n, dtype=np.uint64) * 3) | np.uint64(9 << 48)
    v = V()
    idx = v.GpuIndex(dim, v.Metric.Cos, v.Scalar.F32, bf16_traversal=True)
    idx.reserve(n + 500)
    idx.add_batch(keys, x)
    idx.remove_batch(keys[::13])
    idx.build()
    idx.add_batch(keys[:100] + np.uint64(1), x[:100] * 0.5 + 0.01)  # un-graphed tail
    e0 = idx.search_batch(q, k, exact=True)
    a0 = idx.search_batch(q, k)
    path = str(tmp_path / "index.vsb")
    idx.save(path)
    size0 = idx.size()
    idx.close()
    idx2 = v.GpuIndex.load(path)
    assert idx2.size() == size0
    e1 = idx2.search_batch(q, k, exact=True)
    a1 = idx2.search_batch(q, k)
    for a, b in zip(e0 + a0, e1 + a1):
        assert np.array_equal(a, b)
    assert not idx2.contains(int(keys[0])) and idx2.contains(int(keys[1]))
    idx2.add_batch(np.array([123456789], np.uint64), q[:1])  # a loaded index keeps working
    assert idx2.search(q[0], 1)[0][0] == 123456789


def test_micro_batcher_coalesces_concurrent_single_queries():
    # N2: 32 threads x 40 single-query calls -> far fewer vsb_search calls, identical rows
    n, dim, k = 30000, 96, 10
    x = embedding_like(n, dim, n_clusters=32)
    q = embedding_like(32 * 40, dim, seed=4321, n_clusters=32)
    v = V()
    idx = make_index(x, np.arange(n, dtype=np.uint64), O.COS, O.F32)
    idx.build()
    want_k, want_d, _ = idx.search_batch(q, k)
    b = v.Batcher(idx, max_batch=256, max_wait_us=500)
    got = [None] * len(q)
    errors = []

    def worker(t):
        try:
            for i in range(t * 40, (t + 1) * 40):
                got[i] = b.search(q[i], k)
        except Exception as e:  # noqa: BLE001
            errors.append(e)

    ts = [threading.Thread(target=worker, args=(t,)) for t in range(32)]
    [t.start() for t in ts]
    [t.join() for t in ts]
    assert not errors, errors[:2]
    nq, nb = b.stats()
    print(f"batcher: {nq} queries in {nb} batches (avg {nq / max(nb, 1):.1f} per vsb_search)")
    assert nq == len(q) and nb < nq / 4
    # same rows as the direct batched call (small batches take the CTA-per-query kernel: compare as sets + recall)
    agree = np.mean([len(np.intersect1d(got[i][0], want_k[i])) / k for i in range(len(q))])
    assert agree >= 0.97
    for i in range(0, len(q), 97):
        assert np.all(np.diff(got[i][1]) >= 0) and len(got[i][0]) == k
    b.close()


def test_build_compacts_tombstones():
    rng = np.random.default_rng(3)
    n, dim, k = 12000, 48, 10
    x = embedding_like(n, dim, n_clusters=8)
    q = embedding_like(100, dim, seed=4321, n_clusters=8)
    keys = rng.permutation(n).astype(np.uint64) | np.uint64(1 << 48)
    idx = make_index(x, keys, O.COS, O.BF16)
    dead = rng.choice(n, 5000, replace=False)
    idx.remove_batch(keys[dead])
    assert idx.stats()["n_slots"] == n and idx.size() == n - 5000
    idx.build()
    st = idx.stats()
    assert st["n_slots"] == n - 5000 and st["n_graphed"] == n - 5000 and idx.size() == n - 5000
    alive = np.ones(n, np.uint8)
    alive[dead] = 0
    gk, gd, gc = idx.search_batch(q, k, exact=True)
    ok, od, oc, _ = O.exact_topk(x, q, k, O.COS, O.BF16, keys=keys, alive=alive)
    assert_bit_equal(gk, gd, gc, ok, od, oc)
    ak, _, _ = idx.search_batch(q, k)
    assert O.recall_at_k(ak, ok) >= 0.95 and not np.isin(ak, keys[dead]).any()
    idx.add_batch(keys[dead[:10]], x[dead[:10]])   # a removed key can come back (new epoch in the reference)
    assert idx.size() == n - 4990 and idx.contains(int(keys[dead[0]]))
    gk2, _, _ = idx.search_batch(x[dead[:10]], 1)
    assert np.array_equal(gk2[:, 0], keys[dead[:10]])


def test_c2_full_size_properties():
    # BASELINE config #2 at full size: 1M x 768 f32 cosine — size-independent properties + recall vs exact
    n, dim, k = 1_000_000, 768, 10
    v = V()
    idx = v.GpuIndex(dim, v.Metric.Cos, v.Scalar.F32, bf16_traversal=True)
    idx.reserve(n)
    first = None
    for c0 in range(0, n, 100_000):
        xc = embedding_like(100_000, dim, seed=1234 + c0 // 100_000)
        if first is None:
            first = xc[:256].copy()
        idx.add_batch(np.arange(c0, c0 + len(xc), dtype=np.uint64), xc)
    assert idx.size() == n
    idx.build()
    st = idx.stats()
    assert st["n_graphed"] == n and st["hbm_bytes"] > n * (3072 + 1536)
    q = embedding_like(2000, dim, seed=4321)
    idx.set_search_params(expansion_search=192, search_width=2)
    tk, td, tc = idx.search_batch(q, k, exact=True)
    gk, gd, gc = idx.search_batch(q, k)
    gk2, gd2, _ = idx.search_batch(q, k)
    assert np.array_equal(gk, gk2) and np.array_equal(gd, gd2)          # deterministic
    assert np.all(gc == k) and np.all(tc == k)
    assert np.all(np.diff(gd, axis=1) >= 0) and np.all(np.diff(td, axis=1) >= 0)
    assert np.all((gd >= 0) & (gd <= 2))                                # distance.rs:66-69
    r = O.recall_at_k(gk, tk)
    print(f"C2 1M x 768 recall@10 at ef=192: {r:.4f}")
    assert r >= 0.94  # streamed (K7) graph, no optional refinement pass (VSB_REFINE_PASSES=0 default)
    # every hit's distance is the canonical fp32 distance of that stored row (checked on the oracle for 3 queries)
    for i in range(3):
        rows = np.stack([embedding_like(100_000, dim, seed=1234 + int(key) // 100_000)[int(key) % 100_000]
                         for key in gk[i][:3]])
        od = O.distance_matrix(rows, q[i:i + 1], O.COS, O.F32)[0]
        assert np.array_equal(gd[i][:3].view(np.uint32), od.view(np.uint32))
    sk, sd, _ = idx.search_batch(first, 1, exact=True)                  # a stored row is its own nearest neighbour
    assert np.array_equal(sk[:, 0], np.arange(256, dtype=np.uint64)) and np.all(sd[:, 0] <= 1e-6)


@pytest.mark.parametrize("storage,metric", [(O.BF16, O.L2SQ), (O.BF16, O.IP), (O.F16, O.COS), (O.F16, O.L2SQ)])
def test_tensor_core_traversal_returns_canonical_distances(storage, metric):
    """16-bit float rows, a batch above the small-batch limit and a beam >= 96: K4 multiplies the rows with mma.sync
    (group_reduce_mma) and ranks by candidate-grade sums, K3 re-ranks what is returned.  Whatever the traversal
    arithmetic, the hits must carry the canonical distances of the oracle, ascending, no key twice, recall >= 0.95.
    200 dimensions = 400-byte rows: the last 16-byte chunk row of a lane group is ragged (zero-filled fragments)."""
    n, dim, nq, k = 60_000, 200, 600, 10
    x = embedding_like(n, dim, n_clusters=40)
    q = embedding_like(nq, dim, seed=4321, n_clusters=40)
    keys = np.arange(n, dtype=np.uint64) + np.uint64(7)
    idx = make_index(x, keys, metric, storage)
    idx.build()
    idx.set_search_params(expansion_search=128, search_width=4)
    gk, gd, gc = idx.search_batch(q, k)
    tk, td, tc = idx.search_batch(q, k, exact=True)
    assert np.all(gc == k)
    assert np.all(np.diff(gd, axis=1) >= 0)
    assert all(len(set(row.tolist())) == k for row in gk)
    recall = O.recall_at_k(gk, tk)
    print(f"tensor-core traversal storage={storage} metric={metric}: recall@10 = {recall:.4f}")
    assert recall >= 0.95
    for i in (0, 1, nq - 1):
        od = O.distance_matrix(x[(gk[i] - np.uint64(7)).astype(np.int64)], q[i:i + 1], metric, storage)[0]
        assert np.array_equal(gd[i].view(np.uint32), od.view(np.uint32))
    # a batch-1 call (CTA-per-query kernel, SIMT evaluation, no re-rank) returns the same canonical distances for its hits
    sk, sd, _ = idx.search_batch(q[:1], k)
    od = O.distance_matrix(x[(sk[0] - np.uint64(7)).astype(np.int64)], q[:1], metric, storage)[0]
    assert np.array_equal(sd[0].view(np.uint32), od.view(np.uint32))
    idx.close()


def test_c_abi_client_replays_reference_scenario(tmp_path):
    # a plain C program (tests/abi_client.c) drives G1 through the C ABI — no Python in the data path
    import subprocess
    from test_abi import _build_c_client
    exe = _build_c_client(tmp_path)
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0 and "scenario passed" in r.stdout, r.stdout + r.stderr
    # the same scenario on ONE handle sharded over every GPU of the box (vsb_options.n_devices), still plain C
    import torch
    n = min(torch.cuda.device_count(), 8)
    if n >= 2:
        r = subprocess.run([exe, str(n)], capture_output=True, text=True)
        assert r.returncode == 0 and "sharded handle" in r.stdout, r.stdout + r.stderr


# ---- edge cases the reference's tests touch: empty / tiny / oversized inputs, growth, everything deleted ---------
def test_edge_cases_tiny_and_degenerate_inputs():
    v = V()
    # dim 1, k larger than the index, duplicate vectors (ties by key)
    idx = v.GpuIndex(1, v.Metric.L2sq, v.Scalar.F32)
    idx.reserve(8)
    idx.add_batch(np.array([30, 10, 20], np.uint64), np.array([[1.0], [1.0], [1.0]], np.float32))
    keys, dists, counts = idx.search_batch(np.array([[1.0]], np.float32), 5)
    assert list(keys[0][:3]) == [10, 20, 30] and counts[0] == 3 and np.all(dists[0][:3] == 0)
    assert keys[0][3] == np.uint64(0xFFFFFFFFFFFFFFFF) and np.isinf(dists[0][3])
    # zero queries is a no-op; zero vectors in cosine space follow the 0 / 1 convention
    k0, d0, c0 = idx.search_batch(np.zeros((0, 1), np.float32), 3)
    assert k0.shape == (0, 3)
    cidx = v.GpuIndex(4, v.Metric.Cos, v.Scalar.F32)
    cidx.reserve(4)
    cidx.add_batch(np.array([1, 2], np.uint64), np.array([[0, 0, 0, 0], [1, 0, 0, 0]], np.float32))
    ck, cd, _ = cidx.search_batch(np.array([[0, 0, 0, 0], [2, 0, 0, 0]], np.float32), 2)
    assert list(ck[0]) == [1, 2] and list(cd[0]) == [0.0, 1.0]      # both-zero -> 0, one-zero -> 1
    assert list(ck[1]) == [2, 1] and list(cd[1]) == [0.0, 1.0]
    # capacity errors and growth keep the contents
    with pytest.raises(v.VsbError) as e:
        idx.add_batch(np.arange(100, 110, dtype=np.uint64), np.zeros((10, 1), np.float32))
    assert e.value.status == 4  # VSB_EFULL
    idx.reserve(64)
    idx.add_batch(np.arange(100, 110, dtype=np.uint64), np.arange(10, dtype=np.float32)[:, None])
    assert idx.size() == 13 and idx.search(np.array([9.0], np.float32), 1)[0][0] == 109
    with pytest.raises(v.VsbError) as e:
        idx.search_batch(np.zeros((1, 2), np.float32), 1)
    assert e.value.status == 2  # VSB_EDIM
    with pytest.raises(v.VsbError):
        v.GpuIndex(8, v.Metric.Hamming, v.Scalar.F32)                # "Binary space type requires B1 quantization."
    assert v.GpuIndex(8, v.Metric.Cos, v.Scalar.B1).metric == v.Metric.Hamming   # usearch.rs:450-464


def test_everything_deleted_then_refilled():
    n, dim = 9000, 32
    x = embedding_like(n, dim, n_clusters=8)
    keys = np.arange(n, dtype=np.uint64)
    idx = make_index(x, keys, O.COS, O.F32)
    idx.build()
    idx.remove_batch(keys)
    assert idx.size() == 0
    k, d, c = idx.search_batch(x[:5], 3)
    assert np.all(c == 0) and np.all(k == np.uint64(0xFFFFFFFFFFFFFFFF))
    idx.build()                                                       # compacts to an empty index
    assert idx.stats()["n_slots"] == 0
    idx.add_batch(keys[:100] | np.uint64(1 << 48), x[:100])          # new epoch of the same rows
    k, d, c = idx.search_batch(x[:5], 1)
    assert np.array_equal(k[:, 0], keys[:5] | np.uint64(1 << 48)) and np.all(c == 1)


def test_wide_rows_fall_back_to_exact_search_and_large_k():
    # rows wider than K4 supports (> 6144 bytes) are served by the exact path; k up to 200 works there
    rng = np.random.default_rng(1)
    n, dim = 6000, 2000
    x = rng.standard_normal((n, dim)).astype(np.float32)
    keys = np.arange(n, dtype=np.uint64)
    idx = make_index(x, keys, O.IP, O.F32)
    idx.build()
    assert idx.stats()["n_graphed"] == 0
    q = rng.standard_normal((3, dim)).astype(np.float32)
    gk, gd, gc = idx.search_batch(q, 200)
    ok, od, oc, _ = O.exact_topk(x, q, 200, O.IP, O.F32, keys=keys)
    assert_bit_equal(gk, gd, gc, ok, od, oc)
    for d in gd.ravel():
        V().Distance.try_from(float(d), V().SpaceType.DotProduct, dim)   # negative IP distances are valid


def test_golden_fixture_file_through_the_c_abi():
    # tests/golden/index_path_goldens.json: the same cases the oracle is pinned on, through libvsb200
    from golden_cases import METRIC, STORAGE, check_case, load_cases
    v = V()
    for cid, c, keys, rows, q in load_cases():
        m, s = METRIC[c["metric"]], STORAGE[c["storage"]]
        idx = v.GpuIndex(rows.shape[1], v.Metric(m), v.Scalar(s))
        idx.reserve(len(keys))
        idx.add_batch(keys, rows)
        for exact in (False, True):
            kk, dd, cc = idx.search_batch(q[None, :], c["k"], exact=exact)
            check_case(c, kk[0][:cc[0]], dd[0][:cc[0]], O.HAMMING if s == O.B1 else m)
        idx.close()


def test_every_cluster_is_reachable_from_the_entry_points():
    # well separated clusters give a kNN graph of disconnected components; a component without a seed of the regular
    # sample used to be invisible to the search (recall 0 for its queries).  After a build every live node must be
    # reachable: extra seeds are promoted, one per lost component.
    rng = np.random.default_rng(12)
    dim, per, n_clusters, k = 64, 120, 400, 10              # 48 000 rows, ~1 750 seeds: many clusters get no seed
    centers = 20.0 * rng.standard_normal((n_clusters, dim)).astype(np.float32)
    x = (centers[:, None, :] + rng.standard_normal((n_clusters, per, dim)).astype(np.float32)).reshape(-1, dim)
    perm = rng.permutation(len(x))
    x = np.ascontiguousarray(x[perm])
    q = (centers + rng.standard_normal((n_clusters, dim)).astype(np.float32))   # one query per cluster
    keys = np.arange(len(x), dtype=np.uint64)
    idx = make_index(x, keys, O.L2SQ, O.F32)
    idx.build()
    st = idx.stats()
    print(f"seed rows {st['n_seed_rows']}, extra seeds {st['extra_seeds']}")
    tk, _, _ = idx.search_batch(q, k, exact=True)
    gk, _, gc = idx.search_batch(q, k)
    per_query = np.array([len(np.intersect1d(gk[i], tk[i])) for i in range(len(q))]) / k
    assert st["extra_seeds"] > 0
    assert per_query.min() >= 0.5 and per_query.mean() >= 0.95, (per_query.min(), per_query.mean())
