#!/usr/bin/env python
"""bench.py — headline benchmark of the B200-native index path (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            our arm   (one rank per GPU under torchrun)
  python bench.py --impl reference --gpus N --steps K ...  CPU arm   (USearch-equivalent HNSW restatement)

Workload (config.workload): BASELINE configs[2], the configuration north_star's target is quoted on — 10 M x 768
bf16 cosine, embedding-shaped synthetic vectors (counter-based mixture generator, rows drawn in HBM by
tools/synth/synth.cu; NumPy twin for the CPU arm), k = 10.  `--config c2` selects configs[1] (1 M x 768 f32).
One STEP = `--batches-per-step` (16) query batches of 10 000 through the ANN search path at the smallest
expansion_search / iteration budget that reaches recall@10 >= 0.95 against exact ground truth.
  value    queries/s with the query batches already resident in HBM (vsb_search_dev, CUDA events)
  e2e      the same through the host-pointer C ABI call (vsb_search) from two host threads: pinned H2D of every
           batch and D2H of keys+distances inside the timed region
  roofline graph_search_kernel (K4): algorithmic bytes = Q*(E*(row_bytes+4) + P*R*4), E/P counted by the
           instrumented kernel, duration from CUDA events on the launch stream
  build_roofline  tensor part (all-pairs kNN on tcgen05) and HBM part (K4 passes behind K7 + refinement)
Multi-GPU (N > 1): the corpus is split into N row-range shards (strong scaling, fixed global corpus and query
set); every rank searches every query on its shard; the per-shard top-k are exchanged by peer stores over NVLink
(vsb_xchg_*, `--exchange p2p`) or by ONE NCCL all-gather (`--exchange nccl`) and merged by K8.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC_NAME = "ann_search_qps_at_recall10_ge_0.95"
UNIT = "queries/s"
EF_SWEEP = (32, 64, 96, 128, 160, 192, 224, 256, 320, 384, 512, 768, 1024)  # both arms pick the smallest that reaches the target
CONFIGS = {  # BASELINE.json configs[2] (the north_star target) and configs[1]
    "c3": dict(n=10_000_000, storage="bf16", clusters=2560, traversal="native", name="configs[2]"),
    "c2": dict(n=1_000_000, storage="f32", clusters=256, traversal="bf16", name="configs[1]"),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c3", choices=sorted(CONFIGS))
    ap.add_argument("--n", "--rows", dest="n", type=int, default=None)  # torchrun's own parser trips over a bare --n
    ap.add_argument("--dim", type=int, default=768)
    ap.add_argument("--batch", type=int, default=10_000)
    ap.add_argument("--batches-per-step", type=int, default=16)
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--storage", default=None, choices=["f32", "bf16", "f16"])
    ap.add_argument("--clusters", type=int, default=None,
                    help="mixture components of the synthetic corpus (256 per million rows)")
    ap.add_argument("--target-recall", type=float, default=0.95)
    ap.add_argument("--cpu-sample", type=int, default=1_000_000, help="corpus rows of the bounded CPU-baseline sample")
    ap.add_argument("--search-width", type=int, default=0, help="parents per K4 iteration (1..4); 0 = pick the faster of 2 and 4")
    ap.add_argument("--traversal", default=None, choices=["bf16", "i8", "native"],
                    help="f32 storage: traverse a bf16 (or scaled-int8) copy and re-rank the best candidates on the f32 rows")
    ap.add_argument("--exchange", default="p2p", choices=["p2p", "nccl"])
    ap.add_argument("--cpu-queries", type=int, default=2_000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--refine", action="store_true", help="VSB_FLAG_BUILD_REFINE: vsb_build ends with one refinement pass")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the keys and distances the last timed step returned to DIR/*.npy "
                         "(pin --search-width when comparing two builds: it is otherwise picked by timing)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    cfg = CONFIGS[a.config]
    if a.n is None:
        a.n = cfg["n"]
    if a.storage is None:
        a.storage = cfg["storage"]
    if a.clusters is None:
        a.clusters = cfg["clusters"] if a.n == cfg["n"] else max(16, int(round(256 * a.n / 1e6)))
    if a.traversal is None:
        a.traversal = cfg["traversal"] if a.storage == "f32" else "native"
    if a.storage != "f32":
        a.traversal = "native"
    a.config_name = cfg["name"] if a.n == cfg["n"] else f"{cfg['name']} shape at {a.n} rows"
    return a


def workload_name(a):
    return (f"{a.n}x{a.dim} {a.storage} cosine embedding-shaped synthetic, {a.clusters} mixture components "
            f"(BASELINE {a.config_name}), k={a.k}, query batch {a.batch}")


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), float(d.get("bf16_tflops", 1666.4)), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, 1666.0, "fallback (B200_PROFILING.md)"


DUMP_BUDGET = 64 << 20  # bytes --dump-outputs may write


def dump_outputs(out_dir, keys, dists, budget=DUMP_BUDGET):
    """One step's results, [queries, k] each, for an output-by-output comparison of two builds: keys.npy (float64: keys
    below 2^53 are exact, the empty-slot key 2^64 - 1 reads 2^64), distances.npy (float32) and query_rows.npy (float64,
    the query of each row, numbered through the step's batches).  Above `budget` bytes a fixed seeded sample of the
    queries is written.  Inputs, graph build and search are deterministic: the same arguments give the same arrays."""
    keys = np.asarray(keys, dtype=np.uint64)
    dists = np.asarray(dists, dtype=np.float32)
    n, k = keys.shape
    rows = np.arange(n)
    per_row = k * (8 + 4) + 8
    if n * per_row > budget - 1024:  # 1024: the three .npy headers
        rows = np.sort(np.random.default_rng(0).choice(n, (budget - 1024) // per_row, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "keys.npy"), keys[rows].astype(np.float64))
    np.save(os.path.join(out_dir, "distances.npy"), dists[rows])
    np.save(os.path.join(out_dir, "query_rows.npy"), rows.astype(np.float64))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region.  The sampler is started before the
    warm-up so it is already streaming when the timed region begins; samples are matched to the region by their
    own timestamps."""
    Q = "timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown," \
        "clocks_event_reasons.sw_power_cap"

    def __init__(self, device: int):
        self.device, self.proc, self.lines = device, None, []
        self.t0 = self.t1 = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.device), "-lms", "20"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.1)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = []
        for t_recv, ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                rows.append((t_recv, float(f[1]), float(f[2]), float(f[3]), f[4:8]))
            except ValueError:
                continue
        inside = [r for r in rows if self.t0 is not None and self.t0 - 0.03 <= r[0] <= self.t1 + 0.03]
        note = None
        if not inside and rows:  # region shorter than the sampling period: take the samples closest to it
            mid = 0.5 * ((self.t0 or 0) + (self.t1 or 0))
            inside = sorted(rows, key=lambda r: abs(r[0] - mid))[:3]
            note = (f"no nvidia-smi sample fell inside the {(self.t1 - self.t0) * 1e3:.0f} ms timed region: "
                    "nearest samples used")
        reasons = set()
        for r in inside:
            for nm, val in zip(names, r[4]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        out = {"sm_mhz": float(np.median([r[1] for r in inside])) if inside else None,
               "sm_max_mhz": max(r[2] for r in inside) if inside else None,
               "power_w_max": max(r[3] for r in inside) if inside else None, "samples": len(inside),
               "reasons": sorted(reasons)}
        if note:
            out["note"] = note
        return out


# --------------------------------------------------------------------------------------------------
def cpu_hnsw_run(a, steps, warmup, full_line):
    """The CPU arm: USearch-equivalent HNSW (oracle/hnsw_cpu.cpp) on the host cores, bounded sample."""
    import oracle as O
    from importlib import import_module
    ds = import_module("vector_store_b200.host.datasets")
    threads = os.cpu_count() or 1
    n = min(a.cpu_sample, a.n)
    # rows [0, n) of the SAME counter-based stream the GPU arm generates in HBM (NumPy twin, bit for bit)
    x = ds.embedding_mix(n, a.dim, row0=0, seed=1234, n_clusters=a.clusters)
    q = ds.embedding_mix(a.cpu_queries, a.dim, row0=0, seed=4321, n_clusters=a.clusters)
    st = O.BF16 if a.storage == "bf16" else O.F32
    h = O.HnswCpu(a.dim, O.COS, n, 16, 128, 64, storage=st, threads=threads)
    t0 = time.perf_counter()
    h.add(np.arange(n, dtype=np.uint64), x)
    build_s = time.perf_counter() - t0
    # ground truth for the operating-point search: sgemm on the (unit-norm) vectors
    NR = min(1000, len(q))  # queries behind the recall estimate (200 left the chosen ef noisy by one step)
    tk = np.empty((NR, a.k), np.uint64)
    for r0 in range(0, NR, 200):
        sims = q[r0:r0 + 200] @ x.T
        tk[r0:r0 + 200] = np.argsort(-sims, axis=1, kind="stable")[:, :a.k].astype(np.uint64)
        del sims
    # smallest ef reaching the target recall (same rule as the GPU arm)
    ef_used, recall = 64, 0.0
    for ef in range(16, 513, 16):
        h.set_ef(ef)
        hk, _ = h.search(q[:NR], a.k)
        recall = O.recall_at_k(hk, tk)
        ef_used = ef
        if recall >= a.target_recall:
            break
    for _ in range(warmup):
        h.search(q, a.k)
    t0 = time.perf_counter()
    for _ in range(steps):
        hk, hd = h.search(q, a.k)
    dt = time.perf_counter() - t0
    if full_line and a.dump_outputs:
        dump_outputs(a.dump_outputs, hk, hd)
    qps = steps * len(q) / dt
    lat = []
    for i in range(200):
        t1 = time.perf_counter()
        h.search_one(q[i], a.k)
        lat.append(time.perf_counter() - t1)
    sub = "all" if n == a.n else "the first"
    note = "" if n == a.n else (f"; an HNSW over the full {a.n} rows costs MORE per query (~log n hops), so this sample "
                                "flatters the CPU arm")
    sample = (f"HNSW M=16/ef_add=128 built on {sub} {n} corpus rows (of {a.n}), {len(q)} queries per step, "
              f"ef_search={ef_used} (recall@10={recall:.3f} on {NR} queries); USearch-equivalent CPU restatement, "
              f"not USearch 2.22.0{note}")
    base = {"value": qps, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
            "build_vectors_per_s": n / build_s, "recall_at_10": recall, "ef_search": ef_used,
            "p50_batch1_ms": float(np.percentile(lat, 50) * 1e3), "p99_batch1_ms": float(np.percentile(lat, 99) * 1e3)}
    if not full_line:
        return base
    return {"metric": METRIC_NAME, "value": qps, "unit": UNIT, "n_gpus": a.gpus, "steps": steps, "warmup": warmup,
            "ms_per_step": dt / steps * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": a.storage, "data": "synthetic", "impl": "reference",
            "config": {"workload": workload_name(a), "index": "M=16 ef_add=128", "sample": sample},
            "cpu_baseline": base,
            "e2e": {"value": qps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}


# --------------------------------------------------------------------------------------------------
def main():
    a = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if a.impl == "reference":
        if rank == 0:
            print(json.dumps(cpu_hnsw_run(a, a.steps, a.warmup, True)), flush=True)
        return 0

    import torch
    import torch.distributed as dist
    from importlib import import_module

    import vector_store_b200 as v
    ds = import_module("vector_store_b200.host.datasets")
    shard = import_module("vector_store_b200.host.shard")
    index_mod = import_module("vector_store_b200.host.index")

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: vsb200 has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    scalar = {"f32": v.Scalar.F32, "bf16": v.Scalar.BF16, "f16": v.Scalar.F16}[a.storage]
    lo, hi = shard.shard_range(a.n, rank, world)
    n_local = hi - lo
    k, B, R = a.k, a.batch, a.batches_per_step
    dim = a.dim
    stream = torch.cuda.current_stream().cuda_stream
    trav8 = a.storage == "f32" and a.traversal == "i8"
    trav16 = a.storage == "f32" and a.traversal in ("bf16", "i8")

    def gen_rows(buf, row0, n, seed):
        """rows [row0, row0+n) of the counter-based corpus stream into the device tensor `buf` (tools/synth)"""
        ds.embedding_mix_dev(buf.data_ptr(), n, dim, row0=row0, seed=seed, n_clusters=a.clusters, stream=stream)

    # ---- process warm-up (untimed): a 40k-row index exercises every kernel once, so CUDA's lazy module
    # loading and the first cudaMalloc's are not billed to the timed build below ----
    wbuf = torch.empty((40_000, dim), dtype=torch.float32, device=dev)
    gen_rows(wbuf, 0, 40_000, 7)
    torch.cuda.synchronize()
    warm = v.GpuIndex(dim, v.Metric.Cos, scalar, device=local_rank, bf16_traversal=trav16, i8_traversal=trav8)
    warm.reserve(40_000)
    warm.add_dev(np.arange(30_000, dtype=np.uint64), wbuf.data_ptr(), 30_000)
    warm.build()
    warm.add_dev(np.arange(30_000, 40_000, dtype=np.uint64), wbuf[30_000:].data_ptr(), 10_000)
    warm.insert_pending()
    wx = wbuf[:1000].cpu().numpy()
    warm.search_batch(wx, k)
    warm.search_batch(wx[:4], k)
    warm.close()
    del warm, wbuf

    # ---- host-pointer ingest rate (what the reference's add path would see): 100k rows through vsb_add ----
    host_add_rows_per_s = None
    if rank == 0:
        hb = torch.empty((100_000, dim), dtype=torch.float32, device=dev)
        gen_rows(hb, 0, 100_000, 1234)
        hx = hb.cpu().numpy()
        del hb
        tmp = v.GpuIndex(dim, v.Metric.Cos, scalar, device=local_rank, bf16_traversal=trav16, i8_traversal=trav8)
        tmp.reserve(100_000)
        t0 = time.perf_counter()
        tmp.add_batch(np.arange(100_000, dtype=np.uint64), hx)
        host_add_rows_per_s = 100_000 / (time.perf_counter() - t0)
        tmp.close()
        del tmp, hx

    # ---- corpus shard: generated in HBM chunk by chunk and ingested from there ----
    idx = v.GpuIndex(dim, v.Metric.Cos, scalar, device=local_rank, bf16_traversal=trav16, i8_traversal=trav8,
                     build_refine=a.refine)
    idx.reserve(n_local)
    CH = 500_000
    gbuf = torch.empty((min(CH, n_local), dim), dtype=torch.float32, device=dev)
    barrier()
    t_gen = t_add = 0.0
    for c0 in range(lo, hi, CH):
        nb = min(CH, hi - c0)
        t0 = time.perf_counter()
        gen_rows(gbuf, c0, nb, 1234)
        torch.cuda.synchronize()
        t_gen += time.perf_counter() - t0
        t0 = time.perf_counter()
        idx.add_dev(np.arange(c0, c0 + nb, dtype=np.uint64), gbuf.data_ptr(), nb)
        t_add += time.perf_counter() - t0
    del gbuf
    torch.cuda.empty_cache()
    barrier()
    t0 = time.perf_counter()
    idx.build()
    barrier()
    t_build = time.perf_counter() - t0
    bs = idx.build_stats()
    # clock sampler: started long before the timed region (nvidia-smi needs a second or two to come up on an
    # 8-GPU box) and only on rank 0, whose line is the one reported
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    build_vps = a.n / (t_add + t_build)  # rows resident in HBM -> graph ready, whole job (max over ranks via the barriers)

    # ---- query pool: NB distinct batches, pinned on the host and resident on the device ----
    NB = 4
    q_host, q_dev = [], []
    for b in range(NB):
        qd = torch.empty((B, dim), dtype=torch.float32, device=dev)
        gen_rows(qd, 0, B, 4321 + b)
        torch.cuda.synchronize()
        q_dev.append(qd)
        q_host.append(qd.cpu().pin_memory())
    out_k0 = out_k = torch.empty((B, k), dtype=torch.int64, device=dev)
    out_d0 = out_d = torch.empty((B, k), dtype=torch.float32, device=dev)
    keys_l = torch.empty((B, k), dtype=torch.int64, device=dev)
    dists_l = torch.empty((B, k), dtype=torch.float32, device=dev)
    assert world == 1 or B % world == 0, "query batch must divide evenly over the ranks"
    assert (B * k) % 2 == 0, "B*k must be even (16-byte peer stores / 8-byte aligned records)"
    xchg = None
    slice_rows = B // world
    if world > 1 and a.exchange == "p2p":
        def ag(blob):
            out = [None] * world
            dist.all_gather_object(out, blob)
            return out
        xchg = index_mod.Exchange(local_rank, world, rank, B, k, ag, aux_bytes_per_rank=slice_rows * dim * 4)
    # NCCL variant: per-rank record [B*k keys (8 B) | B*k distances (4 B)] -> ONE all-gather per batch
    rec_bytes = B * k * 12
    if world > 1 and xchg is None:
        rec_local = torch.empty(rec_bytes, dtype=torch.uint8, device=dev)
        rec_all = torch.empty(world * rec_bytes, dtype=torch.uint8, device=dev)
        keys_l = rec_local[:B * k * 8].view(torch.int64).view(B, k)
        dists_l = rec_local[B * k * 8:].view(torch.float32).view(B, k)
    xt = []  # (event before, event after) around the exchange of timed batches
    # value leg, N > 1: the exchange + merge of batch j (latency-bound, ~0.1 ms, a few CTAs) runs on its own high-priority
    # stream under the seed tiles / K4 of batch j + 1; two sets of per-shard result buffers
    pipe = None
    if xchg is not None:
        pipe = {"stream": torch.cuda.Stream(priority=-1), "j": 0,
                "k": [torch.empty((B, k), dtype=torch.int64, device=dev) for _ in range(2)],
                "d": [torch.empty((B, k), dtype=torch.float32, device=dev) for _ in range(2)],
                "searched": [torch.cuda.Event() for _ in range(2)], "exchanged": [torch.cuda.Event() for _ in range(2)]}

    def search_batch_pipelined(q_ptr, timed, out=None):
        out_k, out_d = out if out is not None else (out_k0, out_d0)
        p = pipe["j"] % 2
        pipe["j"] += 1
        main = torch.cuda.current_stream()
        main.wait_event(pipe["exchanged"][p])  # the exchange of batch j - 2 has read this buffer pair
        idx.search_dev(q_ptr, B, k, pipe["k"][p].data_ptr(), pipe["d"][p].data_ptr(), 0, stream, False)
        pipe["searched"][p].record(main)
        sx = pipe["stream"]
        with torch.cuda.stream(sx):
            sx.wait_event(pipe["searched"][p])
            if timed:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(sx)
            xchg.allgather_merge(pipe["k"][p].data_ptr(), pipe["d"][p].data_ptr(), B, k, out_k.data_ptr(), out_d.data_ptr(), 0,
                                 sx.cuda_stream)
            if timed:
                e1.record(sx)
                xt.append((e0, e1))
            pipe["exchanged"][p].record(sx)

    def search_batch_dev(q_ptr, exact=False, timed=False, out=None):
        """device-resident batch: local shard search [+ exchange + K8 merge]; result in out_k/out_d (or `out`)"""
        out_k, out_d = out if out is not None else (out_k0, out_d0)
        if world == 1:
            idx.search_dev(q_ptr, B, k, out_k.data_ptr(), out_d.data_ptr(), 0, stream, exact)
            return
        idx.search_dev(q_ptr, B, k, keys_l.data_ptr(), dists_l.data_ptr(), 0, stream, exact)
        if timed:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        if xchg is not None:
            xchg.allgather_merge(keys_l.data_ptr(), dists_l.data_ptr(), B, k, out_k.data_ptr(), out_d.data_ptr(), 0, stream)
        else:
            dist.all_gather_into_tensor(rec_all, rec_local)
            index_mod.merge_topk_strided_dev(rec_all.data_ptr(), rec_all.data_ptr() + B * k * 8, world, rec_bytes // 8,
                                             rec_bytes // 4, B, k, out_k.data_ptr(), out_d.data_ptr(), 0, local_rank, stream)
        if timed:
            e1.record()
            xt.append((e0, e1))

    # ---- exact ground truth (GPU brute force; bit-exact vs the oracle at this size by tests/test_gpu_round2.py) ----
    gt = []
    for b in range(NB):
        search_batch_dev(q_dev[b].data_ptr(), exact=True)
        torch.cuda.synchronize()
        gt.append(out_k.cpu().numpy().copy())

    def recall_of(b):
        got = out_k.cpu().numpy()
        hits = 0
        for i in range(0, B, max(1, B // 2000)):  # 2000-query sample per batch
            hits += len(np.intersect1d(got[i], gt[b][i]))
        return hits / (len(range(0, B, max(1, B // 2000))) * k)

    # ---- operating point: smallest expansion_search (list size, multiples of 32) with recall@10 >= target,
    # then the smallest iteration budget at that list size that still reaches it (the GPU's fine knob;
    # the CPU arm gets an equally fine sweep of its own knob, ef in steps of 16) ----
    tune_target = a.target_recall + 0.004  # margin: tuned on batch 0, reported on the timed batches

    def tune(sw):
        sweep = []
        ef_used, ef_prev = None, 0
        for ef in EF_SWEEP:
            idx.set_search_params(expansion_search=ef, search_width=sw, max_iterations=10 ** 6)
            search_batch_dev(q_dev[0].data_ptr())
            torch.cuda.synchronize()
            r = recall_of(0)
            sweep.append({"ef": ef, "recall_at_10": round(r, 4)})
            ef_used = ef
            if r >= tune_target:
                break
            ef_prev = ef
        lo_it, hi_it = max(1, ef_prev // sw), ef_used // sw + 8
        while lo_it < hi_it:  # recall is monotone in the iteration budget
            mid = (lo_it + hi_it) // 2
            idx.set_search_params(max_iterations=mid)
            search_batch_dev(q_dev[0].data_ptr())
            torch.cuda.synchronize()
            if recall_of(0) >= tune_target:
                hi_it = mid
            else:
                lo_it = mid + 1
        idx.set_search_params(max_iterations=hi_it)
        sweep.append({"ef": ef_used, "search_width": sw, "max_iterations": hi_it})
        # cost of this operating point: 3 batches, device time
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        search_batch_dev(q_dev[1].data_ptr())
        barrier()
        e0.record()
        for i in range(3):
            search_batch_dev(q_dev[i % NB].data_ptr())
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1) / 3], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return {"ef": ef_used, "max_iterations": hi_it, "search_width": sw, "ms_per_batch": float(t.item()), "sweep": sweep}

    cands = [tune(sw) for sw in ((2, 4) if a.search_width == 0 else (a.search_width,))]
    op = min(cands, key=lambda c: c["ms_per_batch"])
    ef_used, max_iters_used, sw_used = op["ef"], op["max_iterations"], op["search_width"]
    idx.set_search_params(expansion_search=ef_used, search_width=sw_used, max_iterations=max_iters_used)

    # ---- instrumented pass: E (distance evaluations) and P (parent expansions) per query ----
    idx.set_instrumented(True)
    idx.search_dev(q_dev[1].data_ptr(), B, k, keys_l.data_ptr(), dists_l.data_ptr(), 0, stream, False)
    torch.cuda.synchronize()
    st = idx.stats()
    idx.set_instrumented(False)
    E = st["distance_evals"] / max(st["queries"], 1)
    P = st["parent_expansions"] / max(st["queries"], 1)
    trav_row_bytes = st["row_bytes"] // 4 if trav8 else (st["row_bytes"] // 2 if trav16 else st["row_bytes"])
    bytes_per_query = E * (trav_row_bytes + 4) + P * st["graph_degree"] * 4  # +4: the row's norm (cosine)

    # ---- timed region 1: inputs resident in HBM ----
    def dev_step(timed=False, outs=None):
        for j in range(R):
            out = None if outs is None else outs[j]
            if pipe is not None:
                search_batch_pipelined(q_dev[j % NB].data_ptr(), timed, out)
            else:
                search_batch_dev(q_dev[j % NB].data_ptr(), timed=timed, out=out)
        if pipe is not None:
            torch.cuda.current_stream().wait_stream(pipe["stream"])  # the step ends when its last exchange has merged

    # --dump-outputs: every batch of the last timed step writes its own result buffers (the last batch the usual ones,
    # which recall_of reads), so the whole step's results are still there after it
    last_outs = None
    if a.dump_outputs:
        last_outs = [(torch.empty((B, k), dtype=torch.int64, device=dev), torch.empty((B, k), dtype=torch.float32, device=dev))
                     for _ in range(R - 1)] + [(out_k0, out_d0)]

    for i in range(a.warmup):
        dev_step()
    barrier()
    launches0 = idx.stats()["kernel_launches"]
    idx.set_kernel_timing(True)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    torch.cuda.profiler.start()  # ncu --profile-from-start off captures exactly the timed region
    sampler.mark_begin()
    ev0.record()
    for i in range(a.steps):
        dev_step(timed=True, outs=last_outs if i == a.steps - 1 else None)
    ev1.record()
    barrier()
    sampler.mark_end()
    torch.cuda.profiler.stop()
    ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop()
    st = idx.stats()
    idx.set_kernel_timing(False)
    n_batches = a.steps * R
    launches = st["kernel_launches"] - launches0 + (n_batches if world > 1 and xchg is None else 0)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value = n_batches * B / (ms * 1e-3)
    recall_timed = recall_of((R - 1) % NB)
    if last_outs is not None and rank == 0:
        dump_outputs(a.dump_outputs, torch.cat([o[0] for o in last_outs]).cpu().numpy().view(np.uint64),
                     torch.cat([o[1] for o in last_outs]).cpu().numpy())

    k4_ms = st["graph_search_ns"] / 1e6 / max(st["graph_search_launches"], 1)
    peak, tensor_peak, peak_src = load_peaks()
    achieved = B * bytes_per_query / (k4_ms * 1e-3) / 1e9 if k4_ms > 0 else 0.0
    phase_ms = {p: st[p + "_ns"] / 1e6 / n_batches for p in ("convert", "seed", "graph_search", "exact", "merge")}
    if xt:
        phase_ms["exchange_and_merge"] = float(np.mean([e0.elapsed_time(e1) for e0, e1 in xt]))
    traffic = None  # DRAM bytes of one K4 launch from the committed ncu --set full capture, same configuration only
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "k4_traffic.json")))
        for ent in tr if isinstance(tr, list) else [tr]:
            if all(ent.get(k_) == v_ for k_, v_ in (("n", a.n), ("n_gpus", world), ("dim", dim), ("storage", a.storage),
                                                      ("traversal", a.traversal), ("batch", B), ("k", k),
                                                      ("expansion_search", ef_used), ("search_width", sw_used))) \
                    and abs(ent.get("max_iterations", -99) - max_iters_used) <= 2:
                traffic = ent["dram_bytes_read"] + ent["dram_bytes_write"]
    except Exception:
        pass

    # ---- native-f32 traversal of the same index (configs[1] only): the like-for-like f32 line ----
    native_f32 = None
    if trav16 and world == 1:
        cur = (ef_used, sw_used, max_iters_used)
        idx.set_search_params(traversal=2)
        opn = tune(sw_used)
        idx.set_kernel_timing(True)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for j in range(2 * R):
            search_batch_dev(q_dev[j % NB].data_ptr())
        e1.record()
        torch.cuda.synchronize()
        stn = idx.stats()
        idx.set_kernel_timing(False)
        rn = recall_of((2 * R - 1) % NB)
        idx.set_instrumented(True)
        idx.search_dev(q_dev[1].data_ptr(), B, k, keys_l.data_ptr(), dists_l.data_ptr(), 0, stream, False)
        torch.cuda.synchronize()
        sti = idx.stats()
        idx.set_instrumented(False)
        En = sti["distance_evals"] / max(sti["queries"], 1)
        Pn = sti["parent_expansions"] / max(sti["queries"], 1)
        bpq = En * (st["row_bytes"] + 4) + Pn * st["graph_degree"] * 4
        k4n = stn["graph_search_ns"] / 1e6 / max(stn["graph_search_launches"], 1)
        native_f32 = {"value": 2 * R * B / (e0.elapsed_time(e1) * 1e-3), "unit": UNIT, "recall_at_10": round(rn, 4),
                      "expansion_search": opn["ef"], "max_iterations": opn["max_iterations"],
                      "k4_ms_per_launch": k4n, "roofline_frac": B * bpq / (k4n * 1e-3) / 1e9 / peak if k4n > 0 else None,
                      "note": "K4 walks the f32 rows themselves (no bf16 copy, no re-rank)"}
        idx.set_search_params(traversal=1, expansion_search=cur[0], search_width=cur[1], max_iterations=cur[2])

    # ---- timed region 2: end to end through the host-pointer C ABI ----
    h_keys = [torch.empty((B, k), dtype=torch.int64).pin_memory() for _ in range(2)]
    h_dists = [torch.empty((B, k), dtype=torch.float32).pin_memory() for _ in range(2)]
    h_counts = [torch.empty((B,), dtype=torch.int32).pin_memory() for _ in range(2)]

    def e2e_batches(batches, t):
        for b in batches:
            idx.search_raw(q_host[b % NB].data_ptr(), B, k, h_keys[t].data_ptr(), h_dists[t].data_ptr(),
                           h_counts[t].data_ptr())

    def e2e_step():
        if world == 1:
            # two host threads (the reference serves ann requests from a worker pool): the library overlaps one
            # call's H2D / D2H with the other call's kernels
            ts = [threading.Thread(target=e2e_batches, args=(range(t, R, 2), t)) for t in range(2)]
            [x.start() for x in ts]
            [x.join() for x in ts]
            return
        # every shard needs every query: each rank uploads 1/N of the batch from its pinned buffer over its own
        # PCIe link and the slices are exchanged over NVLink (job-wide H2D = one batch, not N batches).  The batches
        # of a step are pipelined over three streams (upload + gather | search + exchange | download), two buffers
        # each, exactly what the two host threads do to the single-GPU library call.
        s0, s1 = shard.shard_range(B, rank, world)
        main = torch.cuda.current_stream()
        for j in range(R):
            p = j % 2
            with torch.cuda.stream(s_up):
                s_up.wait_event(ev_s[p])        # search j-2 has consumed q_priv[p]
                q_slices[p].copy_(q_host[j % NB][s0:s1], non_blocking=True)
                if xchg is not None:
                    # gathered into a private block: the exchange's window is overwritten by peers two gathers later
                    xchg.allgather_rows(q_slices[p].data_ptr(), slice_rows * dim * 4, s_up.cuda_stream, q_priv[p].data_ptr())
                else:
                    dist.all_gather_into_tensor(q_priv[p], q_slices[p])
                ev_q[p].record(s_up)
            main.wait_event(ev_q[p])
            main.wait_event(ev_d[p])            # download j-2 has drained outs[p]
            search_batch_dev(q_priv[p].data_ptr(), out=outs[p])
            ev_s[p].record(main)
            with torch.cuda.stream(s_down):
                s_down.wait_event(ev_s[p])
                h_keys[p].copy_(outs[p][0], non_blocking=True)
                h_dists[p].copy_(outs[p][1], non_blocking=True)
                ev_d[p].record(s_down)
        torch.cuda.synchronize()

    if world > 1:
        # high priority: the gather / copy kernels of batch j+1 must get a CTA slot while K4 of batch j fills every SM,
        # or the upload lands on the critical path instead of under the search
        s_up, s_down = torch.cuda.Stream(priority=-1), torch.cuda.Stream(priority=-1)
        q_slices = [torch.empty((slice_rows, dim), dtype=torch.float32, device=dev) for _ in range(2)]
        q_priv = [torch.empty((B, dim), dtype=torch.float32, device=dev) for _ in range(2)]
        outs = [(torch.empty((B, k), dtype=torch.int64, device=dev), torch.empty((B, k), dtype=torch.float32, device=dev))
                for _ in range(2)]
        ev_q = [torch.cuda.Event() for _ in range(2)]
        ev_s = [torch.cuda.Event() for _ in range(2)]
        ev_d = [torch.cuda.Event() for _ in range(2)]

    for i in range(a.warmup):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for i in range(a.steps):
        e2e_step()
    barrier()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_s = float(t.item())
    if xchg is not None:
        xchg.check(stream)
    e2e = {"value": n_batches * B / e2e_s, "unit": UNIT, "h2d_bytes_per_step": R * B * dim * 4,
           "d2h_bytes_per_step": R * (B * k * 12 * world + (B * 4 if world == 1 else 0)), "ms_per_step": e2e_s / a.steps * 1e3,
           "callers": 2 if world == 1 else 1}

    # ---- p99 batch-1 latency through the host ABI (rank 0 shard only when sharded) ----
    lat = []
    q1 = q_host[2]
    if world == 1:
        for i in range(320):
            t1 = time.perf_counter()
            idx.search_raw(q1[i:i + 1].data_ptr(), 1, k, h_keys[0].data_ptr(), h_dists[0].data_ptr(), h_counts[0].data_ptr())
            lat.append(time.perf_counter() - t1)
        lat = lat[20:]

    # ---- build roofline (vsb_build_stats: CUDA-event phase times + the work of each phase) ----
    ap_tf = bs["allpairs_flops"] / max(bs["allpairs_ns"], 1) / 1e3  # flop/ns -> TFLOP/s
    hbm_bytes_build = ((bs["stream_evals"] + bs["refine_evals"]) * (bs["traversal_row_bytes"] + 4) +
                       (bs["stream_parents"] + bs["refine_parents"]) * st["graph_degree"] * 4)
    hbm_ns = bs["stream_ns"] + bs["refine_ns"]
    build_roofline = {
        "tensor": {"kernel": "exact_candidates_tc_kernel (K1-TC, all-pairs kNN lists)", "rows": bs["allpairs_rows"],
                   "flops": bs["allpairs_flops"], "ms": bs["allpairs_ns"] / 1e6, "achieved": ap_tf, "peak": tensor_peak,
                   "unit": "TFLOP/s", "frac": ap_tf / tensor_peak},
        "hbm": {"kernel": "graph_search_kernel (K4) behind K7 streaming insert + refinement", "bytes": hbm_bytes_build,
                "ms": hbm_ns / 1e6, "achieved": hbm_bytes_build / max(hbm_ns, 1), "peak": peak, "unit": "GB/s",
                "frac": hbm_bytes_build / max(hbm_ns, 1) / peak,
                "distance_evals_per_row": (bs["stream_evals"] + bs["refine_evals"]) / max(bs["rows"], 1)},
        "phase_s": {"allpairs": bs["allpairs_ns"] / 1e9, "prune_reverse_merge": bs["prune_ns"] / 1e9,
                    "stream_insert": bs["stream_ns"] / 1e9, "refine": bs["refine_ns"] / 1e9, "seeds": bs["seeds_ns"] / 1e9,
                    "compact": bs["compact_ns"] / 1e9, "total": bs["total_ns"] / 1e9},
        "note": "per-rank figures of rank 0" if world > 1 else "1 GPU",
    }
    trav_txt = ("scaled-int8 copy of the f32 rows for the graph traversal, fp32 re-rank of 4k candidates on the f32 rows"
                if trav8 else "bf16 copy of the f32 rows for the graph traversal, fp32 re-rank of the best candidates on "
                "the f32 rows" if trav16 else "native storage scalar")
    line = {
        "metric": METRIC_NAME, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": a.storage, "data": "synthetic",
        "config": {"workload": workload_name(a), "step": f"{R} query batches of {B}",
                   "index": "M=16 (degree 32) ef_add=128; build = exact all-pairs kNN on a 131072-row prefix (tcgen05) + "
                            "K7 streaming insert (detour-pruned links)" +
                            (f" + {bs['refine_rows'] // max(bs['rows'], 1)} K4/K6 refinement pass(es)" if bs["refine_rows"] else
                             "; no refinement pass (VSB_REFINE_PASSES=0)"),
                   "traversal": trav_txt, "expansion_search": ef_used, "search_width": sw_used,
                   "max_iterations": max_iters_used, "recall_at_10": round(recall_timed, 4),
                   "operating_points": [{kk: c[kk] for kk in ("ef", "max_iterations", "search_width", "ms_per_batch")} for c in cands],
                   "ef_sweep": op["sweep"],
                   "parallelism": (f"corpus sharded over {world} GPU(s); per-shard top-k exchanged by "
                                   f"{'peer stores over NVLink (vsb_xchg)' if xchg is not None else 'one NCCL all-gather'}"
                                   " + K8 merge") if world > 1 else "1 GPU",
                   "l2_policy": f"corpus shard {n_local * st['row_bytes'] / 1e9:.2f} GB >> 126 MB L2; {NB} query batches rotate"},
        "clocks": clocks,
        "e2e": e2e,
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "kernel": "graph_search_kernel (K4)", "achieved": achieved, "peak": peak,
                     "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                     "algorithmic_bytes_per_launch": B * bytes_per_query, "peak_source": peak_src,
                     "kernel_ms_per_launch": k4_ms, "distance_evals_per_query": E, "parent_expansions_per_query": P,
                     "bytes_per_query": bytes_per_query, "phase_ms_per_batch": phase_ms},
        "build_vectors_per_s": build_vps,
        "build_s": {"add_convert": t_add, "graph": t_build, "generate_in_hbm": t_gen},
        "build_roofline": build_roofline,
        "hbm_bytes": st["hbm_bytes"],
    }
    if host_add_rows_per_s:
        line["host_ingest"] = {"vsb_add_rows_per_s": host_add_rows_per_s,
                               "build_vectors_per_s_with_host_ingest": a.n / (a.n / host_add_rows_per_s / world + t_build),
                               "note": "vsb_add of 100k host rows (pageable, H2D + convert) measured; the second figure "
                                       "charges every row that rate instead of the in-HBM ingest"}
    if native_f32:
        line["native_f32"] = native_f32
    if lat:
        line["p50_batch1_ms"] = float(np.percentile(lat, 50) * 1e3)
        line["p99_batch1_ms"] = float(np.percentile(lat, 99) * 1e3)
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        line["cpu_baseline"] = cpu_hnsw_run(a, 3, 1, False)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if xchg is not None:
        barrier()
        xchg.close()
    idx.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
