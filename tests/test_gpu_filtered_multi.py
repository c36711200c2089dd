"""vsb_search_filtered_multi: many queries with different allow-bitmaps in one call.

Every query is checked under ITS OWN filter: exact-route answers bit for bit against the oracle, graph-route answers
for admissibility and recall; n_filters = 1 must be vsb_search_filtered, and a group of queries sharing a filter must
get what a separate vsb_search_filtered call gives that group."""
import numpy as np
import pytest

import oracle as O
from conftest import embedding_like

pytestmark = pytest.mark.gpu

INVALID = np.uint64(0xFFFFFFFFFFFFFFFF)
ROW = np.uint64(0xFFFFFFFFFFFF)


def V():
    import vector_store_b200 as v
    return v


def assert_bit_equal(gk, gd, gc, ok, od, oc):
    assert np.array_equal(gc, oc)
    assert np.array_equal(gk, ok)
    assert np.array_equal(gd.view(np.uint32), od.view(np.uint32))


def row_ids(keys):
    return (np.asarray(keys, dtype=np.uint64) & ROW).astype(np.int64)


def alive_of(keys, mask):
    """oracle `alive` per corpus row for a mask over row ids"""
    return mask[row_ids(keys)].astype(np.uint8)


def check_exact_per_query(x, keys, q, k, metric, storage, masks, fq, gk, gd, gc, queries=None):
    """each query (or each of `queries`) equals the oracle under its own mask"""
    sel = np.arange(len(q)) if queries is None else np.asarray(queries)
    for f in np.unique(fq[sel]):
        qi = sel[fq[sel] == f]
        ok, od, oc, _ = O.exact_topk(x, q[qi], k, metric, storage, keys=keys, alive=alive_of(keys, masks[f]))
        assert_bit_equal(gk[qi], gd[qi], gc[qi], ok, od, oc)


def modulo_masks(n_rows, F):
    """bitmap j admits only the row ids == j (mod F)"""
    r = np.arange(n_rows)
    return np.stack([(r % F) == j for j in range(F)])


# ---- exact route, bit for bit -------------------------------------------------------------------------------------
@pytest.mark.parametrize("storage,metric,n,dim,F", [
    (O.F32, O.COS, 20000, 128, 7),     # tensor-core candidates + certificate
    (O.I8, O.L2SQ, 5003, 100, 5),      # SIMT tiles
    (O.B1, O.HAMMING, 5003, 100, 3),   # SIMT tiles
])
def test_exact_route_every_query_under_its_own_filter(storage, metric, n, dim, F):
    rng = np.random.default_rng(n + F)
    x = rng.standard_normal((n, dim)).astype(np.float32)
    if storage == O.I8:
        x = np.clip(x * 0.4, -1.2, 1.2).astype(np.float32)
    nq, k = 150, 10
    q = rng.standard_normal((nq, dim)).astype(np.float32) * (0.4 if storage == O.I8 else 1.0)
    keys = rng.permutation(n).astype(np.uint64) + np.uint64(1 << 48)  # row id != slot, epoch bits set
    v = V()
    idx = v.GpuIndex(dim, v.Metric(metric), v.Scalar(storage))
    idx.reserve(n)
    idx.add_batch(keys, x)
    masks = modulo_masks(n, F)
    fq = (np.arange(nq) % F).astype(np.uint32)
    gk, gd, gc = idx.search_filtered_multi(q, k, masks, fq)
    idx.close()
    valid = gk != INVALID
    assert np.all(row_ids(gk[valid]) % F == np.broadcast_to(fq[:, None], gk.shape)[valid])
    check_exact_per_query(x, keys, q, k, metric, storage, masks, fq, gk, gd, gc)


# ---- certificate fallbacks with per-query filters -----------------------------------------------------------------
def test_certificate_fallbacks_follow_each_querys_filter():
    # the near-tie corpus of test_certificate_rejects_near_ties_and_the_fallback_is_exact, four disjoint filters.
    # F times the rows, so that each filter admits as many rows as that test's whole corpus: every query then meets
    # near-tie clusters longer than the candidate lists, which the certificate must refuse.
    rng = np.random.default_rng(77)
    F = 4
    n, dim, nq, k = 10000 * F, 64, 96, 10
    base = rng.standard_normal((40, dim)).astype(np.float32)
    x = base[rng.integers(0, 40, n)] * (1.0 + 1e-6 * rng.standard_normal((n, 1)).astype(np.float32))
    x += (1e-6 * rng.standard_normal((n, dim))).astype(np.float32)
    x[:50] = x[50:100]
    q = base[rng.integers(0, 40, nq)] + (1e-3 * rng.standard_normal((nq, dim))).astype(np.float32)
    keys = rng.permutation(n).astype(np.uint64)
    masks = modulo_masks(n, F)
    fq = rng.integers(0, F, nq).astype(np.uint32)
    v = V()
    for metric in (O.L2SQ, O.COS, O.IP):
        idx = v.GpuIndex(dim, v.Metric(metric), v.Scalar.F32)
        idx.reserve(n)
        idx.add_batch(keys, x)
        s0 = idx.stats()
        gk, gd, gc = idx.search_filtered_multi(q, k, masks, fq)
        s1 = idx.stats()
        idx.close()
        fb, sc = s1["exact_fallback"] - s0["exact_fallback"], s1["exact_scanned"] - s0["exact_scanned"]
        print(f"metric {metric}: fallback {fb}, scanned {sc} of {nq}")
        assert fb > 0 and sc > 0
        check_exact_per_query(x, keys, q, k, metric, O.F32, masks, fq, gk, gd, gc)


# ---- graph route, mixed routes, one filter, groups (one built index) ----------------------------------------------
N_G, DIM_G = 100_000, 96


@pytest.fixture(scope="module")
def built():
    x = embedding_like(N_G, DIM_G, n_clusters=64)
    keys = np.arange(N_G, dtype=np.uint64) | np.uint64(2 << 48)
    v = V()
    idx = v.GpuIndex(DIM_G, v.Metric.Cos, v.Scalar.F32)
    idx.reserve(N_G)
    idx.add_batch(keys, x)
    idx.build()
    idx.set_search_params(expansion_search=192, search_width=2)
    yield idx, x, keys
    idx.close()


def random_masks(rng, selectivities, n=N_G):
    return np.stack([rng.random(n) < s for s in selectivities])


def check_graph_answers(gk, gd, gc, masks, fq, k):
    rows = row_ids(gk)
    valid = gk != INVALID
    for i in range(len(gk)):
        assert masks[fq[i]][rows[i][valid[i]]].all(), f"query {i}: a row outside its own filter"
    assert np.all(gc == k) and np.all(np.diff(gd, axis=1) >= 0)


def test_graph_route_per_query_filters(built):
    idx, x, keys = built
    rng = np.random.default_rng(11)
    k = 10
    q = embedding_like(1000, DIM_G, seed=4321, n_clusters=64)
    masks = random_masks(rng, [0.5, 0.4, 0.3, 0.2, 0.15, 0.1, 0.07, 0.05])
    fq = rng.integers(0, len(masks), len(q)).astype(np.uint32)
    idx.set_kernel_timing(True)
    gk, gd, gc = idx.search_filtered_multi(q, k, masks, fq)
    st = idx.stats()
    idx.set_kernel_timing(False)
    assert st["graph_search_launches"] >= 1
    check_graph_answers(gk, gd, gc, masks, fq, k)
    idx.set_search_params(expansion_search=192, search_width=2, filter_exact_below_pct=100)
    try:
        tk, _, _ = idx.search_filtered_multi(q, k, masks, fq)   # yardstick: every filter on the exact bitmap scan
    finally:
        idx.set_search_params(expansion_search=192, search_width=2, filter_exact_below_pct=2)
    r = O.recall_at_k(gk, tk)
    print(f"per-query filters on the graph: recall@10 vs exact filtered = {r:.4f}")
    assert r >= 0.95


def test_mixed_routes_in_one_call(built):
    idx, x, keys = built
    rng = np.random.default_rng(12)
    k = 10
    q = embedding_like(400, DIM_G, seed=99, n_clusters=64)
    sel = [0.01, 0.3, 0.005, 0.1]              # 1 % and 0.5 %: exact scan (below 2 %); 30 % and 10 %: graph
    masks = random_masks(rng, sel)
    fq = rng.integers(0, len(masks), len(q)).astype(np.uint32)   # routes interleaved in the caller's order
    gk, gd, gc = idx.search_filtered_multi(q, k, masks, fq)
    exact_q = np.flatnonzero(np.isin(fq, [0, 2]))
    graph_q = np.flatnonzero(np.isin(fq, [1, 3]))
    assert len(exact_q) and len(graph_q)
    check_exact_per_query(x, keys, q, k, O.COS, O.F32, masks, fq, gk, gd, gc, queries=exact_q)
    check_graph_answers(gk[graph_q], gd[graph_q], gc[graph_q], masks, fq[graph_q], k)
    idx.set_search_params(expansion_search=192, search_width=2, filter_exact_below_pct=100)
    try:
        tk, _, _ = idx.search_filtered_multi(q[graph_q], k, masks, fq[graph_q])
    finally:
        idx.set_search_params(expansion_search=192, search_width=2, filter_exact_below_pct=2)
    r = O.recall_at_k(gk[graph_q], tk)
    print(f"mixed call: {len(exact_q)} exact-route + {len(graph_q)} graph-route queries, graph recall@10 = {r:.4f}")
    assert r >= 0.95


@pytest.mark.parametrize("selectivity,nq", [
    (0.5, 300),      # graph route
    (0.01, 300),     # exact route
    (0.01, 1500),    # >= 1024 queries: the pipelined host path
    (0.5, 70_000),   # more than one 65 536-query chunk
])
def test_one_filter_equals_search_filtered(built, selectivity, nq):
    idx, x, keys = built
    rng = np.random.default_rng(nq)
    q = embedding_like(nq, DIM_G, seed=nq, n_clusters=64)
    mask = rng.random(N_G) < selectivity
    a = idx.search_filtered(q, 10, mask)
    b = idx.search_filtered_multi(q, 10, mask[None, :], np.zeros(nq, np.uint32))
    assert_bit_equal(*b, *a)


def test_filter_groups_equal_separate_calls(built):
    idx, x, keys = built
    rng = np.random.default_rng(13)
    k = 10
    masks = random_masks(rng, [0.4, 0.01, 0.1, 0.015])   # two graph-route, two exact-route filters
    q = embedding_like(4 * 32, DIM_G, seed=7, n_clusters=64)
    fq = rng.permutation(np.repeat(np.arange(4, dtype=np.uint32), 32))
    gk, gd, gc = idx.search_filtered_multi(q, k, masks, fq)
    for f in range(4):
        qi = np.flatnonzero(fq == f)
        assert_bit_equal(gk[qi], gd[qi], gc[qi], *idx.search_filtered(q[qi], k, masks[f]))


def test_one_filter_with_tail_and_tombstones():
    n, dim, k = 20_000, 64, 10
    x = embedding_like(n + 2000, dim, n_clusters=32)
    keys = np.arange(n + 2000, dtype=np.uint64)
    q = embedding_like(300, dim, seed=5, n_clusters=32)
    rng = np.random.default_rng(3)
    v = V()
    idx = v.GpuIndex(dim, v.Metric.L2sq, v.Scalar.F32)
    idx.reserve(n + 2000)
    idx.add_batch(keys[:n], x[:n])
    idx.build()
    idx.add_batch(keys[n:], x[n:])               # below the streaming threshold: an un-graphed tail
    assert idx.remove_batch(keys[rng.choice(n + 2000, 500, replace=False)]) == 500
    assert idx.stats()["n_graphed"] < idx.size()
    for sel in (0.5, 0.01):
        mask = rng.random(n + 2000) < sel
        a = idx.search_filtered(q, k, mask)
        b = idx.search_filtered_multi(q, k, mask[None, :], np.zeros(len(q), np.uint32))
        assert_bit_equal(*b, *a)
    idx.close()


# ---- bad input ------------------------------------------------------------------------------------------------------
def test_bad_filter_arguments_are_rejected():
    v = V()
    n, dim = 1000, 32
    x = embedding_like(n, dim)
    idx = v.GpuIndex(dim, v.Metric.L2sq, v.Scalar.F32)
    idx.reserve(n)
    idx.add_batch(np.arange(n, dtype=np.uint64), x)
    q = x[:4]
    masks = np.ones((2, n), bool)
    for m, fq in ((masks, [0, 1, 2, 0]),                      # filter index >= n_filters
                  (masks[:0], [0, 0, 0, 0]),                  # n_filters = 0
                  (np.ones((5, n), bool), [0, 1, 2, 3])):     # n_filters > q
        with pytest.raises(v.VsbError) as e:
            idx.search_filtered_multi(q, 5, m, np.asarray(fq, np.uint32))
        assert e.value.status == 1  # VSB_EINVAL
    idx.close()


# ---- sharded handle -------------------------------------------------------------------------------------------------
def test_sharded_handle_matches_single_device_on_the_exact_route():
    import torch
    g = min(torch.cuda.device_count(), 8)
    if g < 2:
        pytest.skip("needs two or more GPUs")
    n, dim, k, F = 40_000, 96, 10, 6
    x = embedding_like(n, dim, n_clusters=32)
    q = embedding_like(300, dim, seed=4321, n_clusters=32)
    keys = np.arange(n, dtype=np.uint64) | np.uint64(1 << 48)
    masks = modulo_masks(n, F)
    fq = (np.arange(len(q)) % F).astype(np.uint32)
    v = V()
    out = []
    for devices in (None, list(range(g))):
        idx = v.GpuIndex(dim, v.Metric.Cos, v.Scalar.F32, devices=devices)
        idx.reserve(n)
        idx.add_batch(keys, x)
        out.append(idx.search_filtered_multi(q, k, masks, fq))
        idx.close()
    assert_bit_equal(*out[1], *out[0])
    check_exact_per_query(x, keys, q, k, O.COS, O.F32, masks, fq, *out[0])


# ---- actor mirror ---------------------------------------------------------------------------------------------------
def test_actor_filtered_ann_batch_equals_one_call_per_query():
    v = V()
    dim, n = 48, 3000
    cfg = v.VsIndexConfiguration("vector.store", dim, space_type=v.SpaceType.Euclidean,
                                 quantization=v.Quantization.F32)
    a = v.new_index_factory_gpu()(cfg)
    a.reserve_increment = 4000
    x = embedding_like(n, dim, n_clusters=8)
    a.add_vectors(0, list(range(n)), x)
    q = embedding_like(12, dim, seed=2, n_clusters=8)
    preds = [(lambda r, m=m: r % 3 == m) for m in (0, 1, 2)] * 3 + [lambda r: r < 500, None, lambda r: r % 3 == 0]
    got = a.filtered_ann_batch(q, 7, preds, max_row_id=n - 1)
    for i in range(len(q)):
        want = a.filtered_ann(q[i], 7, preds[i], max_row_id=n - 1)
        assert got[i][0] == want[0]
        assert [float(d) for d in got[i][1]] == [float(d) for d in want[1]]
    a.stop()
