"""Range search (vsb_search_range) throughput and where its time goes.

Corpus: bench.py's own (embedding_mix rows generated in HBM, cosine, bf16 by default, 10 M x 768).  Queries: 10 000
from the same generator.  Radii: one per run, the median over a 64-query sample of the distance to the 10th, 100th and
1000th neighbour (computed here with torch on the regenerated rows; the benchmark's parameter, not the measured path).

Per radius, one JSON line:
  queries/s        host clock around one vsb_search_range call that returns to host memory (after one warm-up call
                   whose total sizes the caller's buffers)
  rows_per_query   rows returned per query
  *_ms             device time of the count pass, the fill pass(es), the canonical re-evaluation and the two
                   segmented sort passes, from a separate torch.profiler run of one call (kernels in launch order: the
                   first K1 range launch of the call is the count pass, the later ones are fill passes)
  exact_k100_ms    host clock around vsb_search_exact(k = 100) on the same batch, for scale
and the card's name and power limit, read in the same run.  Usage: python tools/range_bench.py [--rows N]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


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


def kernel_times(fn):
    """device ms per phase of one call of fn, from torch.profiler's CUDA kernel records"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    ev = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA),
                key=lambda e: e.time_range.start)
    t = {"count_ms": 0.0, "fill_ms": 0.0, "eval_ms": 0.0, "sort_ms": 0.0, "emit_ms": 0.0}
    seen_count = False
    for e in ev:
        us = e.time_range.elapsed_us()
        n = e.name
        if "exact_candidates" in n:
            t["fill_ms" if seen_count else "count_ms"] += us / 1e3
            seen_count = True
        elif "range_eval" in n:
            t["eval_ms"] += us / 1e3
        elif "Segmented" in n or "segmented" in n:
            t["sort_ms"] += us / 1e3
        elif "range_emit" in n:
            t["emit_ms"] += us / 1e3
    return {k: round(v, 3) for k, v in t.items()}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--dim", type=int, default=768)
    ap.add_argument("--storage", default="bf16", choices=["bf16", "f16", "f32"])
    ap.add_argument("--queries", type=int, default=10_000)
    ap.add_argument("--neighbours", default="10,100,1000")
    a = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("range_bench.py measures the GPU and needs one")
    import vector_store_b200 as v
    from vector_store_b200.host import datasets as ds
    from vector_store_b200.host.native import check

    torch.cuda.set_device(0)
    name, power = card()
    scalar = {"f32": v.Scalar.F32, "bf16": v.Scalar.BF16, "f16": v.Scalar.F16}[a.storage]
    tdt = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}[a.storage]
    clusters = 2560 if a.rows == 10_000_000 else max(16, int(round(256 * a.rows / 1e6)))
    stream = torch.cuda.current_stream().cuda_stream
    ks = [int(s) for s in a.neighbours.split(",")]

    qb = torch.empty((a.queries, a.dim), dtype=torch.float32, device="cuda")
    ds.embedding_mix_dev(qb.data_ptr(), a.queries, a.dim, row0=0, seed=4321, n_clusters=clusters, stream=stream)
    torch.cuda.synchronize()
    q = qb.cpu().numpy()
    qs = qb[:64].to(tdt).float()
    qs = qs / qs.norm(dim=1, keepdim=True)
    del qb

    # ---- corpus (same generator and seed as bench.py); the sample's kmax nearest cosine distances on the way ----
    idx = v.GpuIndex(a.dim, v.Metric.Cos, scalar, device=0)
    idx.reserve(a.rows)
    CH = 500_000
    kmax = max(ks)
    best = torch.full((qs.shape[0], kmax), float("inf"), device="cuda")
    buf = torch.empty((min(CH, a.rows), a.dim), dtype=torch.float32, device="cuda")
    for c0 in range(0, a.rows, CH):
        nb = min(CH, a.rows - c0)
        ds.embedding_mix_dev(buf.data_ptr(), nb, a.dim, row0=c0, seed=1234, n_clusters=clusters, stream=stream)
        torch.cuda.synchronize()
        idx.add_dev(np.arange(c0, c0 + nb, dtype=np.uint64), buf.data_ptr(), nb)
        x = buf[:nb].to(tdt).float()
        d = 1.0 - qs @ (x / x.norm(dim=1, keepdim=True).clamp_min(1e-30)).T
        best = torch.topk(torch.cat([best, d], dim=1), kmax, dim=1, largest=False).values
    del buf
    torch.cuda.synchronize()
    print(json.dumps({"setup": True, "rows": a.rows, "dim": a.dim, "storage": a.storage, "queries": a.queries,
                      "gpu": name, "power_limit_w": power}), flush=True)

    nq = a.queries
    kk = np.empty((nq, 100), np.uint64)
    kd = np.empty((nq, 100), np.float32)
    kc = np.empty(nq, np.uint32)
    idx.search_batch(q, 100, exact=True, out=(kk, kd, kc))
    t0 = time.perf_counter()
    idx.search_batch(q, 100, exact=True, out=(kk, kd, kc))
    exact_ms = (time.perf_counter() - t0) * 1e3

    for k in ks:
        radius = float(best[:, k - 1].median().item())
        off, _, _ = idx.search_range(q, radius)   # warm-up; its total sizes the buffers of the timed calls
        cap = int(off[-1])
        r = np.full(nq, radius, np.float32)
        keys = np.empty(max(cap, 1), np.uint64)
        dists = np.empty(max(cap, 1), np.float32)
        p = lambda x: x.ctypes.data_as(C.c_void_p)  # noqa: E731

        def call():
            check(idx._lib.vsb_search_range(idx._h, p(q), nq, p(r), None, 0, cap, p(keys), p(dists), p(off)))

        t0 = time.perf_counter()
        call()
        dt = time.perf_counter() - t0
        phases = kernel_times(call)
        print(json.dumps({"neighbour": k, "radius": radius, "queries_per_s": round(nq / dt, 1),
                          "rows_per_query": round(int(off[-1]) / nq, 1), "call_ms": round(dt * 1e3, 2), **phases,
                          "exact_k100_ms": round(exact_ms, 2), "gpu": name, "power_limit_w": power}), flush=True)
    idx.close()


if __name__ == "__main__":
    main()
