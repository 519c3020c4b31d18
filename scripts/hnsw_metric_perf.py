#!/usr/bin/env python
"""Walk throughput of the HNSW search kernel per metric, on ONE graph.

  python scripts/hnsw_metric_perf.py [--rows 1000000 --dim 768 --queries 20000 --k 10 --ef 64 --out profiles/...json]

Builds one graph with the GPU batch builder under EUCLIDEAN (the builder serves cosine / Euclid only), then walks that
same graph with EUCLIDEAN, MANHATTAN, CHEBYSHEV, HAMMING and MINKOWSKI(2) through sdb_hnsw_search_device (queries and
results in HBM).  Per metric: best-of-3 device time (CUDA events on the library's stream, after a warm-up), QPS, the
mean visit counters of one untimed sdb_hnsw_search on the same queries, the touched bytes they imply
(visited * (4D + 4) + expanded * deg * 4) per second and their fraction of 7.7 TB/s, and 8 queries checked against the
CPU walk on the same graph (ids equal; distances equal, Minkowski within 1e-12 relative).  Recall is not reported: the
graph was built for Euclid.  Visit counts differ between metrics, so compare them by touched bytes/s, not by QPS.
Hamming walks a {0, 1} copy of the corpus and queries (x > 0), as the reference's generator draws {0, 1} vectors for
it: on continuous data every Hamming distance equals D and the walk stops at once.
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
sys.path.insert(0, os.path.join(ROOT, "tests"))

HBM_TBS = 7.7  # HGX B200 data sheet, one GPU


class _MinkowskiRow:
    """Distance::calculate(element, query) for Minkowski(p), computed by the oracle on demand (the walk touches few rows)"""

    def __init__(self, vectors, q, p):
        self.v, self.q, self.p = vectors, np.ascontiguousarray(q, np.float64), p

    def __getitem__(self, e):
        from oracle import pyoracle as O
        O.lib().orc_set_minkowski_order(C.c_double(self.p))
        try:
            return float(O.knn_topk(self.v[e:e + 1], self.q, "minkowski", 1)[1][0])
        finally:
            O.lib().orc_set_minkowski_order(C.c_double(3.0))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=1_000_000)
    ap.add_argument("--dim", type=int, default=768)
    ap.add_argument("--queries", type=int, default=20_000)
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--ef", type=int, default=64)
    ap.add_argument("--m", type=int, default=16)
    ap.add_argument("--sigma", type=float, default=0.15)
    ap.add_argument("--check", type=int, default=8, help="queries per metric checked against the CPU walk")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "hnsw_metric_perf_1Mx768.json"))
    a = ap.parse_args()

    import torch
    from oracle import pyoracle as O
    from surrealdb_b200 import Context, HnswIndex
    from surrealdb_b200 import _lib as L
    from surrealdb_b200.hnsw_build import build_layers
    from test_oracle_hnsw_metrics import walk_csr

    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()[0]
    ctx = Context(0)
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(0x5DB00003)
    n, dim = a.rows, a.dim
    centers = torch.nn.functional.normalize(torch.randn((4096, dim), generator=g, device=dev), dim=1)

    def sample(cnt):  # the data of bench_extra.py hnsw: 4096 unit-norm centroids + gaussian noise of total norm sigma
        out = torch.empty((cnt, dim), dtype=torch.float32, device=dev)
        for r0 in range(0, cnt, 1 << 20):
            r1 = min(cnt, r0 + (1 << 20))
            c = torch.randint(0, 4096, (r1 - r0,), generator=g, device=dev)
            out[r0:r1] = centers[c] + (a.sigma / dim ** 0.5) * torch.randn((r1 - r0, dim), generator=g, device=dev)
        return out

    x = sample(n)
    queries = sample(a.queries)
    t0 = time.perf_counter()
    layers, entry, _ = build_layers(ctx, x, n, dim, "EUCLIDEAN", m=a.m, m0=2 * a.m, seed=7)
    build_s = time.perf_counter() - t0
    deg0 = float(np.diff(layers[0][0].astype(np.int64)).mean())
    layers_dev = [(torch.from_numpy(rp.astype(np.int64)).to(dev), torch.from_numpy(ci.astype(np.int32)).to(dev))
                  for rp, ci in layers]
    x_bin = (x > 0).float()
    q_bin = (queries > 0).float()
    stream = torch.cuda.ExternalStream(ctx.stream())
    d_ids = torch.empty((a.queries, a.k), dtype=torch.int64, device=dev)
    d_dist = torch.empty((a.queries, a.k), dtype=torch.float64, device=dev)
    d_cnt = torch.empty((a.queries,), dtype=torch.int32, device=dev)
    rows = []
    for metric, p in (("EUCLIDEAN", 3.0), ("MANHATTAN", 3.0), ("CHEBYSHEV", 3.0), ("HAMMING", 3.0), ("MINKOWSKI", 2.0)):
        xv, qv = (x_bin, q_bin) if metric == "HAMMING" else (x, queries)
        torch.cuda.synchronize()
        idx = HnswIndex.from_device(ctx, xv, layers_dev, entry, metric, minkowski_order=p)

        def search():
            L.check(L.lib().sdb_hnsw_search_device(idx.h, C.c_void_p(qv.data_ptr()), a.queries, a.k, a.ef,
                                                   C.c_void_p(d_ids.data_ptr()), C.c_void_p(d_dist.data_ptr()),
                                                   C.c_void_p(d_cnt.data_ptr())))
        search()  # warm-up (module load, visited tables)
        times = []
        for _ in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record(stream)
            search()
            e1.record(stream)
            e1.synchronize()
            times.append(e0.elapsed_time(e1))
        ms = min(times)
        qh = qv.cpu().numpy()
        ids, dist, cnt, ctr = idx.search_graph(qh, a.k, a.ef, counters=True)  # untimed: the visit counters
        same_dev = bool(np.array_equal(d_ids.cpu().numpy().astype(np.uint64), ids))
        visited, expanded = float(ctr[:, 0].mean()), float(ctr[:, 1].mean())
        byts = a.queries * (visited * (4.0 * dim + 4.0) + expanded * deg0 * 4.0)
        # parity on a few queries: the CPU walk on the same graph
        xh = xv.cpu().numpy()
        graph = {"vectors": xh, "layers": layers, "entry_point": entry, "metric": metric.lower()}
        ok = True
        for q in range(a.check):
            if metric == "MINKOWSKI":
                oi, od, oc = walk_csr(graph, _MinkowskiRow(xh, qh[q], p), a.k, a.ef)
                ok &= bool(np.allclose(dist[q, : cnt[q]], od, rtol=1e-12, atol=0.0))
            else:
                oi, od, oc = O.hnsw_search_csr(graph, qh[q], a.k, a.ef)
                ok &= dist[q, : cnt[q]].tobytes() == od.tobytes()
            ok &= list(ids[q, : cnt[q]]) == list(oi) and (int(ctr[q, 0]), int(ctr[q, 1])) == oc
        del idx
        row = {"metric": metric if metric != "MINKOWSKI" else "MINKOWSKI(2)", "qps": a.queries / (ms * 1e-3),
               "device_ms_best": ms, "device_ms_all": times, "visited_per_query": visited, "expanded_per_query": expanded,
               "touched_bytes": byts, "touched_GBps": byts / (ms * 1e-3) / 1e9,
               "frac_of_7p7TBps": byts / (ms * 1e-3) / (HBM_TBS * 1e12), "device_results_equal_host_call": same_dev,
               "cpu_walk_parity_queries": a.check, "cpu_walk_parity": bool(ok)}
        if metric == "HAMMING":
            row["data"] = "corpus and queries rounded to {0, 1} (x > 0)"
        rows.append(row)
        print(json.dumps(row), flush=True)
    eu = rows[0]["touched_GBps"]
    for r in rows:
        r["touched_rate_vs_euclidean"] = r["touched_GBps"] / eu
    out = {"bench": "hnsw_metric_perf", "gpu": gpu, "kernel": "hnsw_search_kernel via sdb_hnsw_search_device",
           "config": {"rows": n, "dim": dim, "queries": a.queries, "k": a.k, "ef": a.ef, "m": a.m, "m0": 2 * a.m,
                      "graph": "GPU batch builder (hnsw_build.build_layers) under EUCLIDEAN, walked with every metric",
                      "data": f"4096 unit-norm centroids + gaussian noise of total norm {a.sigma}", "build_s": build_s,
                      "layers": len(layers), "mean_degree_layer0": deg0,
                      "timing": "best of 3 after one warm-up, CUDA events on the library stream"},
           "rows": rows}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({"gpu": gpu, "out": a.out}), flush=True)
    assert all(r["cpu_walk_parity"] and r["device_results_equal_host_call"] for r in rows)


if __name__ == "__main__":
    main()
