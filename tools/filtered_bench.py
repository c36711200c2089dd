"""Filtered ANN throughput: one call per query vs one call per filter vs one vsb_search_filtered_multi call.

Corpus: bench.py's own (embedding_mix rows generated in HBM, cosine, bf16 by default, 10 M x 768).  Queries: 10 000,
each restricted by one of F distinct filters (F in --filters).  Filter j admits a pseudo-random share of the row ids
drawn from {50 %, 10 %, 5 %, 1 %} (j mod 4), so the 1 % filters take the exact bitmap scan and the rest the graph.

Arms, each timed with a host clock around calls that return results to host memory:
  a  one vsb_search_filtered(q = 1) per query from --threads host threads (a backend that cannot coalesce)
  b  one vsb_search_filtered per distinct filter, over that filter's queries
  c  one vsb_search_filtered_multi over all queries

Per arm and F, one JSON line: queries/s, recall@10 on a query sample against the exact filtered search
(filter_exact_below_pct = 100), bytes of bitmap uploaded per call, and the card's name and power limit read in the
same run.  Usage: python tools/filtered_bench.py [--rows N] [--filters 1,16,256,10000]
"""
import argparse
import json
import os
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SELECTIVITIES = (0.5, 0.1, 0.05, 0.01)


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        power = float(out.splitlines()[0])
    except Exception:
        power = None
    return name, power


def base_bitmaps(rows, seed):
    """one packed bitmap (uint32 words) per selectivity; filter j is base j % 4 rotated by a per-filter word offset"""
    rng = np.random.default_rng(seed)
    words = (rows + 31) // 32
    out = []
    for s in SELECTIVITIES:
        m = rng.random(words * 32) < s
        m[rows:] = False
        out.append(np.packbits(m, bitorder="little").view(np.uint32))
    return out


def filter_bitmap(bases, j, rows):
    b = np.roll(bases[j % len(bases)], (j * 7919) % len(bases[0]))
    if rows % 32:
        b[-1] &= np.uint32((1 << (rows % 32)) - 1)
    return b


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--dim", type=int, default=768)
    ap.add_argument("--storage", default="bf16", choices=["bf16", "f16", "f32"])
    ap.add_argument("--queries", type=int, default=10_000)
    ap.add_argument("--filters", default="1,16,256,10000")
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--threads", type=int, default=8)
    ap.add_argument("--recall-sample", type=int, default=200)
    ap.add_argument("--ef", type=int, default=0, help="expansion_search (0: the index default)")
    ap.add_argument("--max-bitmap-gb", type=float, default=16.0,
                    help="skip an F whose bitmap block would exceed this many GB of host memory")
    a = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("filtered_bench.py measures the GPU and needs one")
    import vector_store_b200 as v
    from vector_store_b200.host import datasets as ds

    torch.cuda.set_device(0)
    name, power = card()
    scalar = {"f32": v.Scalar.F32, "bf16": v.Scalar.BF16, "f16": v.Scalar.F16}[a.storage]
    clusters = 2560 if a.rows == 10_000_000 else max(16, int(round(256 * a.rows / 1e6)))
    stream = torch.cuda.current_stream().cuda_stream

    # ---- corpus (same generator and seed as bench.py) + graph ----
    idx = v.GpuIndex(a.dim, v.Metric.Cos, scalar, device=0)
    idx.reserve(a.rows)
    CH = 500_000
    buf = torch.empty((min(CH, a.rows), a.dim), dtype=torch.float32, device="cuda")
    for c0 in range(0, a.rows, CH):
        nb = min(CH, a.rows - c0)
        ds.embedding_mix_dev(buf.data_ptr(), nb, a.dim, row0=c0, seed=1234, n_clusters=clusters, stream=stream)
        torch.cuda.synchronize()
        idx.add_dev(np.arange(c0, c0 + nb, dtype=np.uint64), buf.data_ptr(), nb)
    del buf
    t0 = time.perf_counter()
    idx.build()
    t_build = time.perf_counter() - t0
    qb = torch.empty((a.queries, a.dim), dtype=torch.float32, device="cuda")
    ds.embedding_mix_dev(qb.data_ptr(), a.queries, a.dim, row0=0, seed=4321, n_clusters=clusters, stream=stream)
    torch.cuda.synchronize()
    q = qb.cpu().numpy()
    del qb
    if a.ef:
        idx.set_search_params(expansion_search=a.ef)
    print(json.dumps({"setup": True, "rows": a.rows, "dim": a.dim, "storage": a.storage, "queries": a.queries,
                      "build_s": round(t_build, 2), "gpu": name, "power_limit_w": power}), flush=True)

    bases = base_bitmaps(a.rows, seed=17)
    words = len(bases[0])
    rng = np.random.default_rng(5)
    sample = np.sort(rng.choice(a.queries, min(a.recall_sample, a.queries), replace=False))
    k = a.k
    h = idx._h
    lib = idx._lib

    def ptr(x):
        return x.ctypes.data

    def one_call(qi, fi, block, out_k, out_d, out_c):
        st = lib.vsb_search_filtered(h, ptr(q[qi]), 1, k, ptr(block[fi]), a.rows, ptr(out_k[qi]), ptr(out_d[qi]),
                                     ptr(out_c[qi:qi + 1]))
        if st != 0:
            raise RuntimeError(f"vsb_search_filtered failed with status {st}")

    for F in [int(s) for s in a.filters.split(",")]:
        if F > a.queries:
            continue
        gb = F * words * 4 / 1e9
        base = {"F": F, "rows": a.rows, "queries": a.queries, "gpu": name, "power_limit_w": power}
        if gb > a.max_bitmap_gb:
            for arm in ("a_per_query", "b_per_filter", "c_multi"):
                print(json.dumps({**base, "arm": arm, "qps": "not measured",
                                  "note": f"bitmap block {gb:.1f} GB > --max-bitmap-gb"}), flush=True)
            continue
        block = np.stack([filter_bitmap(bases, j, a.rows) for j in range(F)])  # [F][words]
        fq = (np.arange(a.queries) % F).astype(np.uint32)
        rng.shuffle(fq)

        # exact filtered yardstick on the sample
        idx.set_search_params(filter_exact_below_pct=100)
        tk = np.empty((len(sample), k), np.uint64)
        td = np.empty((len(sample), k), np.float32)
        tc = np.empty(len(sample), np.uint32)
        qs = np.ascontiguousarray(q[sample])
        used, fs = np.unique(fq[sample], return_inverse=True)  # the sample's own filters (n_filters <= q)
        sub = np.ascontiguousarray(block[used])
        fs = np.ascontiguousarray(fs, dtype=np.uint32)
        st = lib.vsb_search_filtered_multi(h, ptr(qs), len(sample), k, ptr(sub), len(used), a.rows, ptr(fs), ptr(tk),
                                           ptr(td), ptr(tc))
        del sub
        idx.set_search_params(filter_exact_below_pct=2)
        if st != 0:
            raise RuntimeError("exact yardstick failed")

        def report(arm, keys, secs, calls, bytes_per_call):
            import oracle as O
            print(json.dumps({**base, "arm": arm, "qps": round(a.queries / secs, 1), "seconds": round(secs, 4),
                              "calls": calls, "bitmap_bytes_per_call": int(bytes_per_call),
                              "recall_at_10": round(O.recall_at_k(keys[sample], tk), 4)}), flush=True)

        out_k = np.empty((a.queries, k), np.uint64)
        out_d = np.empty((a.queries, k), np.float32)
        out_c = np.empty(a.queries, np.uint32)

        # (a) one q = 1 call per query from a pool of host threads (warm-up: one call per filter route)
        for fi in range(min(F, 4)):
            one_call(int(np.flatnonzero(fq == fi)[0]), fi, block, out_k, out_d, out_c)
        t0 = time.perf_counter()
        with ThreadPoolExecutor(a.threads) as ex:
            list(ex.map(lambda i: one_call(i, int(fq[i]), block, out_k, out_d, out_c), range(a.queries)))
        report("a_per_query", out_k, time.perf_counter() - t0, a.queries, words * 4)

        # (b) one call per distinct filter
        groups = [np.flatnonzero(fq == f) for f in range(F)]
        qg = [np.ascontiguousarray(q[g]) for g in groups]
        gk = [np.empty((len(g), k), np.uint64) for g in groups]
        gd = [np.empty((len(g), k), np.float32) for g in groups]
        gc = [np.empty(len(g), np.uint32) for g in groups]
        t0 = time.perf_counter()
        for f, g in enumerate(groups):
            if lib.vsb_search_filtered(h, ptr(qg[f]), len(g), k, ptr(block[f]), a.rows, ptr(gk[f]), ptr(gd[f]),
                                       ptr(gc[f])) != 0:
                raise RuntimeError("vsb_search_filtered failed")
        secs = time.perf_counter() - t0
        out_k[:] = 0
        for f, g in enumerate(groups):
            out_k[g] = gk[f]
        report("b_per_filter", out_k, secs, F, words * 4)

        # (c) one vsb_search_filtered_multi call (a first untimed call warms the route scratch)
        lib.vsb_search_filtered_multi(h, ptr(q), a.queries, k, ptr(block), F, a.rows, ptr(fq), ptr(out_k),
                                      ptr(out_d), ptr(out_c))
        t0 = time.perf_counter()
        if lib.vsb_search_filtered_multi(h, ptr(q), a.queries, k, ptr(block), F, a.rows, ptr(fq), ptr(out_k),
                                         ptr(out_d), ptr(out_c)) != 0:
            raise RuntimeError("vsb_search_filtered_multi failed")
        report("c_multi", out_k, time.perf_counter() - t0, 1, F * words * 4 + a.queries * 4)
        del block
    idx.close()


if __name__ == "__main__":
    main()
