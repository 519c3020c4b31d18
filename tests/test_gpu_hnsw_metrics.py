"""HNSW walk on the GPU with MANHATTAN, CHEBYSHEV, HAMMING and MINKOWSKI vs the CPU restatement on the SAME graph:
element ids, their order and the visit counters must be identical; f64 distances bit for bit, except Minkowski
(pow(): CUDA's libm against the platform's, rtol 1e-12).  The reference walks come from test_oracle_hnsw_metrics."""
import numpy as np
import pytest

from oracle import kvformats as K
from oracle import pyoracle as O
from test_oracle_hnsw_metrics import (build, distance_table, graph_metric, minkowski_f32, reference_collection,
                                      reference_walk)

pytestmark = pytest.mark.gpu

NEW_METRICS = [("manhattan", 3.0), ("chebyshev", 3.0), ("hamming", 3.0), ("minkowski", 2.0), ("minkowski", 3.0),
               ("minkowski", 1.5)]


@pytest.fixture(scope="module")
def ctx():
    from surrealdb_b200 import Context
    return Context(0)


def sample(rng, metric, shape):
    if metric == "hamming":  # {0, 1}-valued: heavy ties, the FIFO rules of the queues decide
        return rng.integers(0, 2, shape).astype(np.float32)
    return rng.uniform(-20, 20, shape).astype(np.float32)


def same_dist(metric, got, want):
    if metric == "minkowski":
        return np.allclose(got, want, rtol=1e-12, atol=0.0)
    return got.tobytes() == want.tobytes()


def check(metric, p, g, idx, queries, k, ef, **kw):
    ids, dist, cnt, ctr = idx.search_graph(queries, k, ef, counters=True, **kw)
    for q in range(queries.shape[0]):
        oi, od, oc = reference_walk(g, metric, queries[q], k, ef, p, **kw)
        assert cnt[q] == oi.size, (metric, p, k, ef, q)
        assert list(ids[q, : cnt[q]]) == list(oi), (metric, p, k, ef, q)
        assert same_dist(metric, dist[q, : cnt[q]], od), (metric, p, k, ef, q, dist[q, : cnt[q]], od)
        assert (int(ctr[q, 0]), int(ctr[q, 1])) == oc, (metric, p, k, ef, q)
    return ids, cnt


@pytest.mark.parametrize("metric,p", NEW_METRICS)
@pytest.mark.parametrize("dim", [5, 20, 96, 100])
def test_walk_parity_random_graphs(ctx, metric, p, dim):
    from surrealdb_b200.hnsw import HnswIndex
    rng = np.random.default_rng(dim + len(metric) + int(4 * p))
    data = sample(rng, metric, (1500, dim))
    g = build(data, graph_metric(metric), m=8, efc=60)
    idx = HnswIndex(ctx, g["vectors"], g["layers"], g["entry_point"], metric, minkowski_order=p)
    queries = sample(rng, metric, (70, dim))
    for k, ef in ((10, 10), (10, 40), (1, 1), (25, 64), (10, 150)):
        check(metric, p, g, idx, queries, k, ef)


@pytest.mark.parametrize("metric,p", NEW_METRICS[:4])
def test_filtered_walk_parity(ctx, metric, p):
    from surrealdb_b200.hnsw import HnswIndex
    rng = np.random.default_rng(77)
    dim = 24
    data = sample(rng, metric, (3000, dim))
    g = build(data, graph_metric(metric), m=8, efc=60)
    idx = HnswIndex(ctx, g["vectors"], g["layers"], g["entry_point"], metric, minkowski_order=p)
    queries = sample(rng, metric, (48, dim))
    for sel in (1.0, 0.5, 0.2, 0.08, 0.0):
        truthy = (rng.random(3000) < sel).astype(np.uint8)
        for k, ef in ((10, 40), (3, 8), (10, 10)):
            try:
                ids, cnt = check(metric, p, g, idx, queries, k, ef, truthy=truthy)
            except Exception as e:  # documented: a filter too selective for the on-chip window -> caller's CPU path
                if "SDB_EOVERFLOW" not in str(e):
                    raise
                assert sel < 0.2, (sel, k, ef, str(e))
                continue
            for q in range(queries.shape[0]):
                assert all(truthy[int(e)] for e in ids[q, : cnt[q]])


@pytest.mark.parametrize("metric,p", NEW_METRICS[:4])
def test_pending_updates(ctx, metric, p):
    # HnswIndex::knn_search with a pending log (hnsw/index.rs:270-335,372-420): moved, deleted and new vectors; the new
    # vectors are ranked with Distance::calculate(query, vector) on the GPU (sdb_hnsw_distance_f32)
    from surrealdb_b200.hnsw import HnswIndex
    rng = np.random.default_rng(78)
    dim, n = 24, 900
    data = sample(rng, metric, (n, dim))
    g = build(data, graph_metric(metric), m=8, efc=60)
    idx = HnswIndex(ctx, g["vectors"], g["layers"], g["entry_point"], metric, minkowski_order=p)
    q = sample(rng, metric, (dim,))
    k, ef = 10, 40
    table = distance_table(metric, data, q, p)
    near = np.argsort(table, kind="stable")[:30]
    if metric == "hamming":
        moved = {int(e): np.abs(data[e] - (rng.random(dim) < 0.1)).astype(np.float32) for e in near[::2]}
        fresh = q.copy()
        fresh[0] = 1.0 - fresh[0]
    else:
        moved = {int(e): (data[e] + rng.normal(0, 0.05, dim)).astype(np.float32) for e in near[::2]}
        fresh = q + np.float32(0.01)
    for e, v in moved.items():
        idx.add_pending(e, [data[e]], [v])
    idx.add_pending(5, [data[5]], [])
    idx.add_pending("person:new", [], [fresh])
    idx.add_pending("person:gone", [], [q])
    idx.add_pending("person:gone", [q], [])
    got = idx.knn_search(q, k, ef)
    # ---- the same flow restated with the CPU pieces ----
    news = list(moved.items()) + [("person:new", fresh)]
    gpu_d = idx._typed_distances(q, np.stack([v for _, v in news]))
    entries = set()
    key = HnswIndex._vid_key

    def offer(d, vid):
        if len(entries) >= k and d > max(e[0] for e in entries):
            return
        entries.add((d, key(vid), vid))
        while len(entries) > k:
            entries.remove(max(entries, key=lambda e: (e[0], e[1])))
    for (vid, v), dg in zip(news, gpu_d):
        d = minkowski_f32(q, v, p) if metric == "minkowski" else O.vec_distance_f32(metric, q, v)
        assert same_dist(metric, np.array([dg]), np.array([d])), (metric, vid, dg, d)
        offer(float(dg) if metric == "minkowski" else d, vid)
    mask = np.zeros(n, np.uint8)
    mask[list(set(moved) | {5})] = 1
    oi, od, _ = reference_walk(g, metric, q, k, ef, p, all_docs_pending=mask)
    ids, dist, cnt = idx.search_graph(q[None, :], k, ef, all_docs_pending=mask)
    assert list(ids[0, : cnt[0]]) == list(oi) and same_dist(metric, dist[0, : cnt[0]], od)
    for e, d in zip(ids[0, : cnt[0]], dist[0, : cnt[0]]):
        offer(float(d), int(e))
    want = [(vid, d) for d, _, vid in sorted(entries, key=lambda e: (e[0], e[1]))]
    assert got == want, (metric, got, want)
    assert any(vid == "person:new" for vid, _ in got) and all(vid != "person:gone" for vid, _ in got)


@pytest.mark.parametrize("metric,p", [("manhattan", 3.0), ("minkowski", 2.0)])
def test_index_loaded_from_raw_kv_values(ctx, metric, p):
    from surrealdb_b200.hnsw import HnswIndex
    rng = np.random.default_rng(11)
    dim = 48
    data = rng.uniform(-20, 20, (1200, dim)).astype(np.float32)
    g = build(data, graph_metric(metric), m=8, efc=60, seed=5)
    n = data.shape[0]
    he = [(e, K.ser_vector("F32", g["vectors"][e])) for e in range(n)]
    hn = []
    for rp, ci in g["layers"]:
        hn.append([(e, K.node_to_val(ci[rp[e]:rp[e + 1]])) for e in range(n) if rp[e + 1] > rp[e]])
    state = K.hnsw_state(int(g["entry_point"]), n, (n, 0), tuple((1, 0) for _ in g["layers"][1:]))
    idx = HnswIndex.from_kv(ctx, dim, state, he, hn, metric, minkowski_order=p)
    assert idx.n_bad == 0 and idx.n == n
    queries = rng.uniform(-20, 20, (40, dim)).astype(np.float32)
    for k, ef in ((10, 40), (5, 5)):
        check(metric, p, g, idx, queries, k, ef)


@pytest.mark.parametrize("metric", ["chebyshev", "hamming", "manhattan", "minkowski"])
@pytest.mark.parametrize("flags", [(False, False), (True, False), (False, True), (True, True)])
def test_reference_tests_hnsw_matrix_on_the_gpu(ctx, metric, flags):
    # tests_hnsw (hnsw/mod.rs:752-791) searched through HnswIndex.knn_search: every vector finds itself, and the result
    # holds min(knn, 30) entries for knn in 1..19 at ef = 80
    from surrealdb_b200.hnsw import HnswIndex
    data = reference_collection(metric, seed=len(metric) + 2 * flags[0] + flags[1])
    h = O.Hnsw(data.shape[1], graph_metric(metric), m=24, m0=48, efc=500, extend_candidates=flags[0],
               keep_pruned_connections=flags[1], seed=7)
    for v in data:
        h.insert(v)
    assert h.check_props()
    g = h.export()
    idx = HnswIndex(ctx, g["vectors"], g["layers"], g["entry_point"], metric, minkowski_order=2.0)
    for i, v in enumerate(data):
        for knn in range(1, 20):
            res = idx.knn_search(v, knn, 80)
            assert len(res) == min(knn, 30), (metric, i, knn)
            assert any(np.array_equal(data[vid], v) for vid, _ in res), (metric, i, knn)


def test_minkowski_order_on_a_loaded_handle(ctx):
    from surrealdb_b200 import SdbError
    from surrealdb_b200.hnsw import HnswIndex
    rng = np.random.default_rng(21)
    data = rng.uniform(-20, 20, (1000, 16)).astype(np.float32)
    g = build(data, "euclidean", m=8, efc=60)
    idx = HnswIndex(ctx, g["vectors"], g["layers"], g["entry_point"], "MINKOWSKI")  # default order 3
    queries = rng.uniform(-20, 20, (24, 16)).astype(np.float32)
    check("minkowski", 3.0, g, idx, queries, 10, 40)
    for p in (1.5, 1.0, 4.0):
        idx.set_minkowski_order(p)
        check("minkowski", p, g, idx, queries, 10, 40)
        d = idx._typed_distances(queries[0], data[:50])
        assert np.allclose(d, [minkowski_f32(queries[0], v, p) for v in data[:50]], rtol=1e-12, atol=0.0)
    with pytest.raises(SdbError, match="SDB_EINVAL"):
        idx.set_minkowski_order(float("nan"))
    check("minkowski", 4.0, g, idx, queries, 10, 40)  # a refused order leaves the handle as it was


@pytest.mark.parametrize("metric", ["manhattan", "chebyshev"])
def test_degenerate_values(ctx, metric):
    # elements with a NaN or +-inf component: ids and counters equal the oracle's, including where NaN distances queue
    # (after every number, FIFO among themselves); distances bit for bit (a Manhattan NaN is the positive 0x7FF8...)
    from surrealdb_b200.hnsw import HnswIndex
    rng = np.random.default_rng(5 + len(metric))
    dim = 20
    data = rng.uniform(-20, 20, (1200, dim)).astype(np.float32)
    g = build(data, metric, m=8, efc=60)
    vec = g["vectors"].copy()
    bad = rng.choice(1200, 120, replace=False)
    for j, e in enumerate(bad):
        vec[e, rng.integers(0, dim)] = (np.nan, np.inf, -np.inf)[j % 3]
    g = dict(g, vectors=vec)
    idx = HnswIndex(ctx, vec, g["layers"], g["entry_point"], metric)
    queries = rng.uniform(-20, 20, (40, dim)).astype(np.float32)
    queries[1, 3] = np.inf
    queries[2, 0] = np.nan
    saw_nan = False
    for k, ef in ((10, 40), (25, 64), (1, 1)):
        ids, dist, cnt, ctr = idx.search_graph(queries, k, ef, counters=True)
        for q in range(queries.shape[0]):
            oi, od, oc = O.hnsw_search_csr(g, queries[q], k, ef)
            assert list(ids[q, : cnt[q]]) == list(oi), (metric, k, ef, q)
            assert dist[q, : cnt[q]].tobytes() == od.tobytes(), (metric, k, ef, q, dist[q, : cnt[q]], od)
            assert (int(ctr[q, 0]), int(ctr[q, 1])) == oc, (metric, k, ef, q)
            saw_nan |= bool(np.isnan(od).any())
    assert saw_nan or metric == "chebyshev"  # Chebyshev never takes a NaN difference


@pytest.mark.parametrize("metric", ["PEARSON", "JACCARD"])
def test_similarity_metrics_keep_the_cpu_path(ctx, metric):
    from surrealdb_b200 import SdbError
    from surrealdb_b200.hnsw import HnswIndex
    data = np.random.default_rng(1).uniform(-1, 1, (50, 8)).astype(np.float32)
    g = build(data, "euclidean", m=4, efc=20)
    with pytest.raises(SdbError, match="SDB_EUNSUPPORTED") as e:
        HnswIndex(ctx, g["vectors"], g["layers"], g["entry_point"], metric)
    assert metric in str(e.value)
    n = data.shape[0]
    he = [(i, K.ser_vector("F32", data[i])) for i in range(n)]
    hn = [[(i, K.node_to_val(ci[rp[i]:rp[i + 1]])) for i in range(n) if rp[i + 1] > rp[i]] for rp, ci in g["layers"]]
    state = K.hnsw_state(int(g["entry_point"]), n, (n, 0), tuple((1, 0) for _ in g["layers"][1:]))
    with pytest.raises(SdbError, match="SDB_EUNSUPPORTED"):
        HnswIndex.from_kv(ctx, 8, state, he, hn, metric)
