"""vsb_search_range: every live row within a per-query distance bound, exact.

The reference is a canonical brute force (oracle/exact.c): for each query the rows whose canonical distance is <= r,
ordered by (distance, key), with the same fp32 distance bits.  Corpora above and below tc_min_rows (8192) exercise the
tensor-core and the SIMT candidate stages."""
import ctypes as C

import numpy as np
import pytest

import oracle as O

pytestmark = pytest.mark.gpu

ROW = np.uint64(0xFFFFFFFFFFFF)
VSB_OK, VSB_EINVAL, VSB_EFULL = 0, 1, 4
SENTINEL_KEY = np.uint64(0xDEADBEEFDEADBEEF)


def V():
    import vector_store_b200 as v
    return v


def corpus(n, dim, seed, storage=O.F32, dup=True):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((n, dim)).astype(np.float32)
    if storage == O.I8:
        x = np.clip(x * 0.4, -1.2, 1.2).astype(np.float32)
    if dup:
        x[100:110] = x[50]  # eleven identical rows: every query sees an eleven-way distance tie
    keys = rng.permutation(n).astype(np.uint64) + np.uint64(1 << 48)  # key order != slot order, epoch bits set
    return x, keys


def queries(nq, dim, seed, storage=O.F32):
    q = np.random.default_rng(seed).standard_normal((nq, dim)).astype(np.float32)
    return q * (0.4 if storage == O.I8 else 1.0)


def make_index(x, keys, metric, storage):
    v = V()
    m = v.Metric.Hamming if storage == O.B1 else v.Metric(metric)
    idx = v.GpuIndex(x.shape[1], m, v.Scalar(storage), device=0)
    idx.reserve(len(x) + 2000)
    idx.add_batch(keys, x)
    return idx


def oracle_range(D, keys, r, alive=None):
    """CSR answer of the canonical brute force: D = distance matrix [nq, n] (oracle), r [nq]"""
    off = [0]
    ks, ds = [], []
    for i in range(D.shape[0]):
        sel = D[i] <= r[i]
        if alive is not None:
            sel &= alive.astype(bool)
        idx = np.nonzero(sel)[0]
        order = np.lexsort((keys[idx], D[i, idx]))
        ks.append(keys[idx][order])
        ds.append(D[i, idx][order])
        off.append(off[-1] + len(idx))
    return (np.array(off, dtype=np.uint64), np.concatenate(ks).astype(np.uint64) if ks else np.zeros(0, np.uint64),
            np.concatenate(ds).astype(np.float32) if ds else np.zeros(0, np.float32))


def assert_same(got, want):
    go, gk, gd = got
    wo, wk, wd = want
    assert np.array_equal(go, wo), "offsets differ"
    assert np.array_equal(gk, wk), "keys differ"
    assert np.array_equal(gd.view(np.uint32), wd.view(np.uint32)), "distance bits differ"


def kth(D, k):
    """each query's own k-th canonical distance (1-based)"""
    return np.sort(D, axis=1)[:, k - 1].astype(np.float32)


def raw_range(idx, q, r, capacity, bm=None, bits=0, keys=None, dists=None, offsets=None):
    """the C call with caller-owned buffers -> (status, offsets, keys, dists)"""
    q = np.ascontiguousarray(q, dtype=np.float32)
    r = np.ascontiguousarray(r, dtype=np.float32)
    if keys is None:
        keys = np.full(max(capacity, 1), SENTINEL_KEY, np.uint64)
        dists = np.full(max(capacity, 1), -7.0, np.float32)
    if offsets is None:
        offsets = np.full(len(q) + 1, 12345, np.uint64)
    p = lambda a: a.ctypes.data_as(C.c_void_p) if a is not None else None  # noqa: E731
    st = idx._lib.vsb_search_range(idx._h, p(q), len(q), p(r), p(bm), bits, capacity, p(keys), p(dists), p(offsets))
    return st, offsets, keys, dists


# ---- 1. bit-exact across storages and metrics, both candidate stages --------------------------------------------
CASES = [(O.F32, O.COS), (O.F32, O.L2SQ), (O.F32, O.IP), (O.F16, O.L2SQ), (O.BF16, O.COS), (O.BF16, O.IP),
         (O.I8, O.L2SQ), (O.I8, O.COS), (O.B1, O.HAMMING)]


@pytest.mark.parametrize("n", [3000, 9000])
@pytest.mark.parametrize("storage,metric", CASES)
def test_bit_exact_against_the_oracle(storage, metric, n):
    dim, nq = 72, 24
    x, keys = corpus(n, dim, 10 + storage * 5 + metric, storage)
    q = queries(nq, dim, 99 + n, storage)
    idx = make_index(x, keys, metric, storage)
    D = O.distance_matrix(x, q, metric, storage)
    radii = [kth(D, 1), kth(D, 100), kth(D, 3000), np.zeros(nq, np.float32), np.full(nq, np.inf, np.float32)]
    for r in radii:
        assert_same(idx.search_range(q, r), oracle_range(D, keys, r))
    idx.close()


# ---- 2. at the bound ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("storage", [O.F32, O.BF16])
def test_rows_tied_at_the_bound(storage):
    """r = a distance eleven rows share returns all eleven; the next float below returns none of them"""
    n, dim, nq = 9000, 96, 16  # >= 8192 rows: tensor-core candidate stage (TF32 for f32 rows)
    x, keys = corpus(n, dim, 3, storage)
    q = queries(nq, dim, 4, storage)
    idx = make_index(x, keys, O.COS, storage)
    D = O.distance_matrix(x, q, O.COS, storage)
    tied = keys[[50] + list(range(100, 110))]
    r = D[:, 50].copy()
    got = idx.search_range(q, r)
    assert_same(got, oracle_range(D, keys, r))
    for i in range(nq):
        assert set(tied) <= set(got[1][got[0][i]:got[0][i + 1]].tolist())
    below = np.nextafter(r, np.float32(-np.inf)).astype(np.float32)
    got = idx.search_range(q, below)
    assert_same(got, oracle_range(D, keys, below))
    for i in range(nq):
        assert not set(tied) & set(got[1][got[0][i]:got[0][i + 1]].tolist())
    idx.close()


# ---- 3. tombstones, the build and the tail ------------------------------------------------------------------------
def test_tombstones_build_and_tail():
    n, dim, nq = 9000, 64, 20
    storage, metric = O.BF16, O.L2SQ
    x, keys = corpus(n + 1500, dim, 21, storage)
    q = queries(nq, dim, 22, storage)
    idx = make_index(x[:n], keys[:n], metric, storage)
    removed = keys[np.random.default_rng(1).choice(n, 700, replace=False)]
    assert idx.remove_batch(removed) == 700
    alive = np.ones(n + 1500, np.uint8)
    alive[np.isin(keys, removed)] = 0
    D = O.distance_matrix(x, q, metric, storage)
    r = kth(D[:, :n], 400)
    before = idx.search_range(q, r)
    assert not np.isin(before[1], removed).any()
    assert_same(before, oracle_range(D[:, :n], keys[:n], r, alive[:n]))
    idx.build()
    assert_same(idx.search_range(q, r), before)
    idx.set_search_params(stream_threshold=1 << 30)  # the new rows stay an un-graphed tail
    idx.add_batch(keys[n:], x[n:])
    assert idx.stats()["n_graphed"] < idx.size()
    assert_same(idx.search_range(q, r), oracle_range(D, keys, r, alive))
    idx.close()


# ---- 4. filter ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [3000, 9000])
def test_filter_against_the_oracle(n):
    dim, nq = 64, 16
    x, keys = corpus(n, dim, 31)
    keys = np.arange(n, dtype=np.uint64)[np.random.default_rng(2).permutation(n)] | np.uint64(1 << 48)
    q = queries(nq, dim, 32)
    idx = make_index(x, keys, O.COS, O.F32)
    D = O.distance_matrix(x, q, O.COS, O.F32)
    rid = (keys & ROW).astype(np.int64)
    mask = np.random.default_rng(3).random(n) < 0.3
    r = kth(D, 2000)
    assert_same(idx.search_range(q, r, allow_mask=mask), oracle_range(D, keys, r, mask[rid]))
    # bits at and past bitmap_bits are inadmissible, stray bits of the last word included
    bits = n - 45                        # bits % 32 != 0
    bm = np.zeros((n + 31) // 32, np.uint32)
    bm[: (bits + 31) // 32] = 0xFFFFFFFF  # every row admitted by the words, the tail only by stray bits
    st, off, k_, d_ = raw_range(idx, q, r, 10_000_000, bm=bm, bits=bits)
    assert st == VSB_OK
    total = int(off[-1])
    assert_same((off, k_[:total], d_[:total]), oracle_range(D, keys, r, (rid < bits)))
    idx.close()


# ---- 5. capacity and argument checks ------------------------------------------------------------------------------
def test_capacity_and_invalid_arguments():
    n, dim, nq = 9000, 64, 12
    x, keys = corpus(n, dim, 41)
    q = queries(nq, dim, 42)
    idx = make_index(x, keys, O.L2SQ, O.F32)
    D = O.distance_matrix(x, q, O.L2SQ, O.F32)
    r = kth(D, 500)
    want = oracle_range(D, keys, r)
    total = int(want[0][-1])
    st, off, k_, d_ = raw_range(idx, q, r, total - 1)
    assert st == VSB_EFULL
    assert np.array_equal(off, want[0])
    assert (k_ == SENTINEL_KEY).all() and (d_ == -7.0).all()
    st, off, k_, d_ = raw_range(idx, q, r, total)
    assert st == VSB_OK
    assert_same((off, k_, d_), want)
    # q == 0 writes offsets[0] = 0
    st, off, _, _ = raw_range(idx, q[:0], r[:0], 0, offsets=np.full(1, 9, np.uint64))
    assert st == VSB_OK and off[0] == 0
    # VSB_EINVAL before anything runs
    p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    kb, db, ob = np.zeros(8, np.uint64), np.zeros(8, np.float32), np.zeros(nq + 1, np.uint64)
    qq = np.ascontiguousarray(q)
    lib, h = idx._lib, idx._h
    assert lib.vsb_search_range(h, None, nq, p(r), None, 0, 8, p(kb), p(db), p(ob)) == VSB_EINVAL
    assert lib.vsb_search_range(h, p(qq), nq, None, None, 0, 8, p(kb), p(db), p(ob)) == VSB_EINVAL
    assert lib.vsb_search_range(h, p(qq), nq, p(r), None, 0, 8, p(kb), p(db), None) == VSB_EINVAL
    assert lib.vsb_search_range(h, p(qq), nq, p(r), None, 0, 8, None, p(db), p(ob)) == VSB_EINVAL
    assert lib.vsb_search_range(h, p(qq), nq, p(r), None, 0, 8, p(kb), None, p(ob)) == VSB_EINVAL
    r_nan = r.copy()
    r_nan[3] = np.nan
    assert lib.vsb_search_range(h, p(qq), nq, p(r_nan), None, 0, 8, p(kb), p(db), p(ob)) == VSB_EINVAL
    with pytest.raises(V().VsbError):
        idx.search_range(q, r_nan)
    # capacity 0 with null buffers is a valid way to ask for the counts
    ob[:] = 0
    assert lib.vsb_search_range(h, p(qq), nq, p(r), None, 0, 0, None, None, p(ob)) == VSB_EFULL
    assert np.array_equal(ob, want[0])
    # the binding retries once with the exact size
    got = idx.search_range(q, np.full(nq, np.inf, np.float32))
    assert int(got[0][-1]) == nq * n and len(got[1]) == nq * n
    idx.close()


# ---- 6. sub-chunks ------------------------------------------------------------------------------------------------
def test_candidates_beyond_the_device_budget():
    """4000 queries x 9000 rows with r = +inf: 36 M candidates, more than twice the 2^24 entries one fill pass holds
    on the device, so the queries run in three sub-chunks.  Needs about 2 GB of host memory (the 36 M results held by
    the library and by the caller at 12 bytes each, plus the oracle's 4000 x 9000 distance matrix)."""
    n, dim, nq = 9000, 32, 4000
    x, keys = corpus(n, dim, 51, O.BF16)
    q = queries(nq, dim, 52)
    idx = make_index(x, keys, O.COS, O.BF16)
    off, gk, gd = idx.search_range(q, np.inf)
    assert np.array_equal(off, np.arange(nq + 1, dtype=np.uint64) * n)
    D = O.distance_matrix(x, q, O.COS, O.BF16)
    for i in range(0, nq, 7):
        order = np.lexsort((keys, D[i]))
        assert np.array_equal(gk[i * n:(i + 1) * n], keys[order])
        assert np.array_equal(gd[i * n:(i + 1) * n].view(np.uint32), D[i, order].view(np.uint32))
    idx.close()


# ---- 7. sharded handle --------------------------------------------------------------------------------------------
def test_sharded_handle_matches_single_device():
    import torch
    g = min(torch.cuda.device_count(), 8)
    if g < 2:
        pytest.skip("needs two or more GPUs")
    n, dim, nq = 20_000, 64, 32
    x, keys = corpus(n, dim, 61)
    q = queries(nq, dim, 62)
    D = O.distance_matrix(x, q, O.COS, O.F32)
    r = kth(D, 300)
    mask = np.random.default_rng(4).random(n) < 0.5
    v = V()
    out = []
    for devices in (None, list(range(g))):
        idx = v.GpuIndex(dim, v.Metric.Cos, v.Scalar.F32, devices=devices)
        idx.reserve(n)
        idx.add_batch(keys, x)
        out.append((idx.search_range(q, r), idx.search_range(q, r, allow_mask=mask)))
        idx.close()
    for a, b in zip(out[0], out[1]):
        assert_same(b, a)
    assert_same(out[0][0], oracle_range(D, keys, r))


# ---- 8. tombstones written while range searches run ---------------------------------------------------------------
def test_rows_removed_between_and_during_range_searches():
    """vsb_remove writes the live tombstone bitmap without waiting for searches.  A call's count and fill passes see
    one copy of it, so a remove landing mid-call never breaks the call: its answer is the brute force over a live set
    between the one before the call and the one after it."""
    import threading
    n, dim, nq = 9000, 64, 64
    x, keys = corpus(n, dim, 71)
    q = queries(nq, dim, 72)
    idx = make_index(x, keys, O.COS, O.BF16)
    D = O.distance_matrix(x, q, O.COS, O.BF16)
    r = kth(D, 1500)
    alive = np.ones(n, np.uint8)
    # between two calls
    gone = keys[np.random.default_rng(5).choice(n, 300, replace=False)]
    assert_same(idx.search_range(q, r), oracle_range(D, keys, r, alive))
    idx.remove_batch(gone)
    alive[np.isin(keys, gone)] = 0
    assert_same(idx.search_range(q, r), oracle_range(D, keys, r, alive))
    # during calls: one thread removes in small batches while this one searches
    order = np.random.default_rng(6).permutation(keys[alive.astype(bool)])[:3000]
    done = threading.Event()

    def remover():
        for c in range(0, len(order), 50):
            idx.remove_batch(order[c:c + 50])
        done.set()

    th = threading.Thread(target=remover)
    before = alive.copy()
    th.start()
    calls = 0
    while not done.is_set() or calls < 2:
        got = idx.search_range(q, r)
        calls += 1
        ok_rows = oracle_range(D, keys, r, before)  # the largest answer a call can give
        for i in range(nq):
            gk = got[1][got[0][i]:got[0][i + 1]]
            wk = ok_rows[1][ok_rows[0][i]:ok_rows[0][i + 1]]
            wd = ok_rows[2][ok_rows[0][i]:ok_rows[0][i + 1]]
            keep = np.isin(wk, gk)
            assert keep.sum() == len(gk)          # only rows of the larger live set, each once
            assert np.array_equal(wk[keep], gk)   # in the brute force's (distance, key) order
            assert np.array_equal(wd[keep].view(np.uint32), got[2][got[0][i]:got[0][i + 1]].view(np.uint32))
            assert np.isin(wk[~keep], order).all()  # what is missing was removed
    th.join()
    alive[np.isin(keys, order)] = 0
    assert_same(idx.search_range(q, r), oracle_range(D, keys, r, alive))
    idx.close()


# ---- 9. more queries than one chunk -------------------------------------------------------------------------------
def test_more_queries_than_one_chunk():
    """70 000 queries: two chunks of at most 65 536, whose offsets continue across the chunk boundary"""
    n, dim, nq = 1000, 16, 70_000
    x, keys = corpus(n, dim, 81)
    q = queries(nq, dim, 82)
    idx = make_index(x, keys, O.L2SQ, O.F32)
    D = O.distance_matrix(x, q, O.L2SQ, O.F32)
    r = kth(D, 8)
    assert_same(idx.search_range(q, r), oracle_range(D, keys, r))
    idx.close()
