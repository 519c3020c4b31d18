"""HNSW with the MANHATTAN, CHEBYSHEV, HAMMING and MINKOWSKI distances, on the CPU.

The C oracle restates the F32 typed Manhattan, Chebyshev and Hamming metrics and walks / builds graphs with them.  It has
no F32 typed Minkowski (its Minkowski is the brute-force one, `orc_knn_topk`), so this module restates

  * Minkowski on F32 vectors (idx/trees/vector.rs:389-399) in Python with the platform libm's pow, and checks it bit
    for bit against the oracle's brute-force Minkowski on f32 rows (same formula: the query is f32, widened);
  * the CSR walk of Hnsw::knn_search / knn_search_with_filter / the pending-docs walk (hnsw/mod.rs:459-548,
    hnsw/layer.rs:76-306) over a precomputed distance table, and checks it against the oracle's walk for the metrics
    the oracle has -- so the same walk can serve as the reference for Minkowski.

The reference's own HNSW matrix (`tests_hnsw`, hnsw/mod.rs:752-791, find_collection_hnsw :618-662) is restated for
Chebyshev, Hamming, Manhattan and Minkowski(2).
"""
import bisect
import ctypes as C
import math
import struct

import numpy as np
import pytest

from oracle import pyoracle as O

F64_MAX = 1.7976931348623157e308


# ---------------------------------------------------------------- distances
def minkowski_f32(a, b, p):
    """vector.rs:389-399 for VectorType::F32: sum |(f64)a - (f64)b|^p sequentially in f64, then ^(1/p)"""
    s = 0.0
    for x, y in zip(np.asarray(a, np.float32).tolist(), np.asarray(b, np.float32).tolist()):
        s += math.pow(abs(x - y), p)
    return math.pow(s, 1.0 / p)


def distance_table(metric, vectors, q, p=3.0):
    """Distance::calculate(element, query) for every element (f64).  Minkowski: the oracle's brute-force Minkowski over
    f32 rows with the query widened to f64 -- the F32 typed formula (test_minkowski_kats checks it bit for bit)."""
    vectors = np.ascontiguousarray(vectors, np.float32)
    q = np.ascontiguousarray(q, np.float32)
    n = vectors.shape[0]
    if metric == "minkowski":
        O.lib().orc_set_minkowski_order(C.c_double(p))
        try:
            rows, dist = O.knn_topk(vectors, q.astype(np.float64), "minkowski", n)
        finally:
            O.lib().orc_set_minkowski_order(C.c_double(3.0))
        out = np.empty(n, np.float64)
        out[rows.astype(np.int64)] = dist
        return out
    return np.array([O.vec_distance_f32(metric, vectors[e], q) for e in range(n)], np.float64)


# ---------------------------------------------------------------- the walk over a distance table
def _key(d):  # f64::total_cmp
    b = struct.unpack("<q", struct.pack("<d", d))[0]
    return b ^ 0x7FFFFFFFFFFFFFFF if b < 0 else b


class _Dpq:
    """DoublePriorityQueue (idx/trees/knn.rs:15-123): ascending total_cmp key, FIFO inside a key; pop_last takes the
    newest of the farthest"""

    def __init__(self, other=None):
        self.e = list(other.e) if other else []
        self.seq = other.seq if other else 0

    def push(self, d, i):
        bisect.insort(self.e, (_key(d), self.seq, d, i))
        self.seq += 1

    def pop_first(self):
        return self.e.pop(0)[2:]

    def pop_last(self):
        return self.e.pop()[2:]

    def last_dist(self):
        return self.e[-1][2] if self.e else F64_MAX


def walk_csr(graph, dist, k, ef, truthy=None, all_docs_pending=None):
    """Hnsw::knn_search (truthy = None) / knn_search_with_filter over an exported graph, with dist[e] =
    Distance::calculate(element e, query).  -> (ids, dist, (visited, expanded)), like pyoracle.hnsw_search_csr."""
    layers, ep = graph["layers"], int(graph["entry_point"])
    if ep < 0 or k == 0:
        return np.zeros(0, np.uint64), np.zeros(0, np.float64), (0, 0)
    ctr = [1, 0]
    ep_d = float(dist[ep])

    def search(rp, ci, ep, ep_d, ef, flt):
        visited = {ep}
        cand = _Dpq()
        cand.push(ep_d, ep)
        w = _Dpq()
        if flt is None or flt[ep]:
            w.push(ep_d, ep)
        fq = w.last_dist()
        while cand.e:
            cd, c = cand.pop_first()
            if cd > fq:
                break
            ctr[1] += 1
            for e in ci[int(rp[c]):int(rp[c + 1])].tolist():
                if e in visited:
                    continue
                visited.add(e)
                ed = float(dist[e])
                ctr[0] += 1
                if ed < fq or len(w.e) < ef:
                    if flt is not None:
                        cand.push(ed, e)
                        if flt[e]:  # add_if_truthy
                            w.push(ed, e)
                            if len(w.e) > ef:
                                w.pop_last()
                            fq = w.last_dist()
                    else:
                        if all_docs_pending is None or not all_docs_pending[e]:  # layer.rs:209
                            cand.push(ed, e)
                        w.push(ed, e)
                        if len(w.e) > ef:
                            w.pop_last()
                        fq = w.last_dist()
        return w

    for l in range(len(layers) - 1, 0, -1):  # search_ep: never filtered
        w = search(layers[l][0], layers[l][1], ep, ep_d, 1, None)
        if w.e:
            ep_d, ep = w.e[0][2], w.e[0][3]
    w = search(layers[0][0], layers[0][1], ep, ep_d, ef, truthy)
    res = w.e[:k]
    return (np.array([e[3] for e in res], np.uint64), np.array([e[2] for e in res], np.float64), tuple(ctr))


def reference_walk(graph, metric, q, k, ef, p=3.0, truthy=None, all_docs_pending=None):
    """the oracle's walk where it has the metric, the walk above over the Minkowski table otherwise"""
    if metric != "minkowski":
        g = dict(graph, metric=metric)
        return O.hnsw_search_csr(g, q, k, ef, truthy=truthy, all_docs_pending=all_docs_pending)
    return walk_csr(graph, distance_table("minkowski", graph["vectors"], q, p), k, ef, truthy, all_docs_pending)


def build(data, metric, m, efc, seed=1, **kw):
    h = O.Hnsw(data.shape[1], metric, m=m, efc=efc, seed=seed, **kw)
    for v in data:
        h.insert(v)
    assert h.check_props()
    return h.export()


def graph_metric(metric):
    """the oracle's builder has no F32 Minkowski: Minkowski graphs are built under EUCLIDEAN (Minkowski(2) orders the
    elements like Euclid up to rounding).  The walk is what is checked; it does not depend on how the graph was made."""
    return "euclidean" if metric == "minkowski" else metric


def reference_collection(metric, seed):
    """RandomItemGenerator (knn.rs:625-644) shapes of tests_hnsw: 30 unique vectors, floats in [-20, 20] at dim 5;
    Hamming: integers in {0, 1} at dim 20"""
    rng = np.random.default_rng(seed)
    rows, seen = [], set()
    while len(rows) < 30:
        v = (rng.integers(0, 2, 20) if metric == "hamming" else rng.uniform(-20, 20, 5)).astype(np.float32)
        if v.tobytes() not in seen:
            seen.add(v.tobytes())
            rows.append(v)
    return np.stack(rows)


# ---------------------------------------------------------------- tests
@pytest.mark.parametrize("p", [1.0, 2.0, 3.0, 1.5])
@pytest.mark.parametrize("dim", [1, 5, 20, 100])
def test_minkowski_kats(p, dim):
    rng = np.random.default_rng(int(p * 10) + dim)
    a = rng.uniform(-20, 20, (40, dim)).astype(np.float32)
    q = rng.uniform(-20, 20, dim).astype(np.float32)
    a[3] = q  # distance 0
    a[4, 0] = q[0] + np.float32(1e-6)
    table = distance_table("minkowski", a, q, p)
    for e in range(a.shape[0]):
        want = minkowski_f32(a[e], q, p)
        assert table[e] == want, (p, dim, e, table[e], want)
        assert minkowski_f32(q, a[e], p) == want  # symmetric bit for bit: calculate(query, vector) is the same
    assert table[3] == 0.0
    # the order does not leak: the oracle's brute force is back at its default
    rows, d = O.knn_topk(a, q.astype(np.float64), "minkowski", 1)
    assert d[0] == 0.0
    assert minkowski_f32([1, 2, 3], [2, 3, 4], 3.0) == O.num_metric("minkowski", [1.0, 2.0, 3.0], [2.0, 3.0, 4.0], 3.0)[1]


@pytest.mark.parametrize("metric", ["euclidean", "manhattan", "chebyshev", "hamming"])
def test_walk_restatement_equals_the_oracle_walk(metric):
    # the Python walk over a distance table reproduces the oracle's walk (ids, distances, counters) for every metric the
    # oracle has, plain, filtered and with pending docs: it is then trusted as the Minkowski reference
    rng = np.random.default_rng(len(metric))
    dim = 20 if metric == "hamming" else 12
    data = (rng.integers(0, 2, (500, dim)) if metric == "hamming" else rng.uniform(-20, 20, (500, dim))).astype(np.float32)
    g = build(data, metric, m=8, efc=40)
    truthy = (rng.random(500) < 0.3).astype(np.uint8)
    pending = (rng.random(500) < 0.2).astype(np.uint8)
    for q in (rng.integers(0, 2, (6, dim)) if metric == "hamming" else rng.uniform(-20, 20, (6, dim))).astype(np.float32):
        table = distance_table(metric, data, q)
        for k, ef in ((10, 10), (1, 1), (10, 40)):
            for kw in ({}, {"truthy": truthy}, {"all_docs_pending": pending}):
                oi, od, oc = O.hnsw_search_csr(g, q, k, ef, **kw)
                pi, pd, pc = walk_csr(g, table, k, ef, **kw)
                assert list(pi) == list(oi) and pd.tobytes() == od.tobytes() and pc == oc, (metric, k, ef, kw)


@pytest.mark.parametrize("metric", ["chebyshev", "hamming", "manhattan", "minkowski"])
@pytest.mark.parametrize("flags", [(False, False), (True, False), (False, True), (True, True)])
def test_reference_tests_hnsw_matrix(metric, flags):
    # tests_hnsw: new_params(dim, F32, dist, m = 24, efc = 500, extend, keep), 30 vectors inserted (check_hnsw_properties
    # after each), then every vector searched with knn in 1..min(20, 30) at ef = 80: it finds itself and the result
    # holds min(knn, 30) entries
    data = reference_collection(metric, seed=len(metric) + 2 * flags[0] + flags[1])
    h = O.Hnsw(data.shape[1], graph_metric(metric), m=24, m0=48, efc=500, extend_candidates=flags[0],
               keep_pruned_connections=flags[1], seed=7)
    for v in data:
        h.insert(v)
        assert h.check_props()
    g = h.export()
    for i, v in enumerate(data):
        table = distance_table(metric, data, v, 2.0)
        for knn in range(1, 20):
            ids, dist, _ = walk_csr(g, table, knn, 80)
            assert len(ids) == min(knn, 30), (metric, i, knn)
            assert any(np.array_equal(data[int(e)], v) for e in ids), (metric, i, knn)
            if metric != "minkowski":
                oi, od = h.search(v, knn, 80)
                assert list(oi) == list(ids) and od.tobytes() == dist.tobytes()
