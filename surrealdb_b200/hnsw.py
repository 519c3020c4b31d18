"""Host-side mirror of the HNSW search path on top of the C ABI.

  HnswIndex.load(...)                 what the Rust shim hands over after HnswFlavor::check_state
                                      (idx/trees/hnsw/mod.rs:187-224): element vectors + per-layer adjacency
  HnswIndex.search_graph(q, k, ef)    Hnsw::knn_search (hnsw/mod.rs:459-482) -> [(dist, element)] ascending
  HnswIndex.knn_search(q, k, ef)      HnswIndex::knn_search (hnsw/index.rs:270-335): pending updates first
                                      (search_pendings, :372-420), then the graph with the pending-docs bitmap,
                                      element -> docs expansion through KnnResultBuilder semantics
                                      (idx/trees/knn.rs:363-437): final order (distance, VectorId), <= k
  HnswIndex.add_pending(...)          the Hp log (VectorPendingUpdate, hnsw/mod.rs:88-113) as the Rust shim streams it
  HnswIndex.check_state(state)        Hnsw::check_state (hnsw/mod.rs:187-224): is the device copy still current?

Metrics (DIST of the index): COSINE, EUCLIDEAN, MANHATTAN, CHEBYSHEV, HAMMING and MINKOWSKI (minkowski_order, default
3) in the reference's F32 typed arithmetic.  PEARSON and JACCARD raise SdbError(SDB_EUNSUPPORTED): such indexes keep
the reference's CPU path.
"""
import ctypes as C

import numpy as np

from . import _lib as L


class KnnResultBuilder:
    """idx/trees/knn.rs:363-437: a BTreeSet<(FloatKey(dist), VectorId)> capped at knn entries."""

    def __init__(self, knn, vid_key):
        self.knn, self.vid_key, self.items = int(knn), vid_key, []  # items: sorted [(dist, key(vid), vid)]

    def check_add(self, dist):  # accept unless the list is full and the distance is farther than the last
        return not (len(self.items) >= self.knn and self.items and dist > self.items[-1][0])

    def add_vector_id_result(self, dist, vid):
        ent = (dist, self.vid_key(vid), vid)
        if not any(e[0] == ent[0] and e[1] == ent[1] for e in self.items):  # a set: an equal pair collapses
            self.items.append(ent)
            self.items.sort(key=lambda e: (e[0], e[1]))
        if len(self.items) > self.knn:
            self.items.pop()

    def collect(self):
        return [(d, vid) for d, _, vid in self.items]


class HnswIndex:
    def __init__(self, ctx, vectors, layers, entry_point, metric="EUCLIDEAN", elem_docs=None, minkowski_order=3.0):
        """vectors (n, dim) f32; layers = [(row_ptr u64[n+1], col_idx u32[e]), ...] layer 0 first;
        elem_docs: optional list of doc-id lists per element (identical vectors share one element:
        hnsw/docs.rs:161-176); default = one doc per element with the same id.  minkowski_order: the p of
        DIST MINKOWSKI p (ignored by the other metrics)."""
        vec = np.ascontiguousarray(vectors, np.float32)
        self.n, self.dim = vec.shape
        self.ctx, self.metric = ctx, metric.upper()
        self.elem_docs = elem_docs
        self.pendings = []
        self.versions = None
        nl = len(layers)
        rps = [np.ascontiguousarray(l[0], np.uint64) for l in layers]
        cis = [np.ascontiguousarray(l[1] if len(l[1]) else np.zeros(1, np.uint32), np.uint32) for l in layers]
        RP = (C.c_void_p * nl)(*[a.ctypes.data for a in rps])
        CI = (C.c_void_p * nl)(*[a.ctypes.data for a in cis])
        self.h = C.c_void_p()
        L.check(L.lib().sdb_hnsw_load(ctx.h, self.dim, L.METRIC[self.metric], self.n, C.c_void_p(vec.ctypes.data), nl,
                                      RP, CI, int(entry_point), C.byref(self.h)))
        self.set_minkowski_order(minkowski_order)

    @classmethod
    def from_device(cls, ctx, x_dev, layers_dev, entry_point, metric="EUCLIDEAN", elem_docs=None, minkowski_order=3.0):
        """wraps device-resident vectors and CSR layers WITHOUT copying them (sdb_hnsw_load_device): x_dev is a torch CUDA
        float32 (n, dim) tensor, layers_dev = [(row_ptr int64 (n+1), col_idx int32)] layer 0 first.  The tensors must
        stay alive (they are kept on the object)."""
        self = cls.__new__(cls)
        self.ctx, self.metric, self.elem_docs = ctx, metric.upper(), elem_docs
        self.n, self.dim = int(x_dev.shape[0]), int(x_dev.shape[1])
        self.pendings, self.versions = [], None
        self._keep = (x_dev, layers_dev)
        nl = len(layers_dev)
        RP = (C.c_void_p * nl)(*[t[0].data_ptr() for t in layers_dev])
        CI = (C.c_void_p * nl)(*[t[1].data_ptr() for t in layers_dev])
        self.h = C.c_void_p()
        L.check(L.lib().sdb_hnsw_load_device(ctx.h, self.dim, L.METRIC[self.metric], self.n, C.c_void_p(x_dev.data_ptr()), nl,
                                             RP, CI, int(entry_point), C.byref(self.h)))
        self.set_minkowski_order(minkowski_order)
        return self

    @classmethod
    def from_kv(cls, ctx, dim, state_value, he_items, hn_items_per_layer, metric="EUCLIDEAN", elem_docs=None,
                minkowski_order=3.0):
        """Loads the index straight from raw KV values (staging.py): `state_value` = the Hs value, `he_items` =
        [(element id, He value)], `hn_items_per_layer[l]` = [(node id, Hn value)] of layer l (0 first), each in key
        order.  Decoding happens on the GPU (sdb_hnsw_load_staged).  Mirrors Hnsw::check_state + HnswLayer::load
        (hnsw/mod.rs:187-224, hnsw/layer.rs:505-560) for indexes without legacy Hl chunks."""
        from . import staging as S
        st = S.parse_hnsw_state(state_value)
        if st["layer0"]["chunks"] or any(l["chunks"] for l in st["layers"]):
            raise L.SdbError(L.SDB_EUNSUPPORTED, "legacy Hl chunks present: run the reference's migration first")
        nl = 1 + len(st["layers"])
        if len(hn_items_per_layer) != nl:
            raise L.SdbError(L.SDB_EINVAL, f"state names {nl} layers, {len(hn_items_per_layer)} given")
        self = cls.__new__(cls)
        self.ctx, self.metric, self.dim, self.elem_docs = ctx, metric.upper(), int(dim), elem_docs
        self.pendings = []
        self.versions = [st["layer0"]["version"]] + [l["version"] for l in st["layers"]]
        self.n = int(st["next_element_id"])
        vb, vo, vi = S.pack_values(he_items)
        packs = [S.pack_values(it) for it in hn_items_per_layer]
        NB = (C.c_void_p * nl)(*[p[0].ctypes.data for p in packs])
        NO = (C.c_void_p * nl)(*[p[1].ctypes.data for p in packs])
        NI = (C.c_void_p * nl)(*[p[2].ctypes.data for p in packs])
        NN = (C.c_uint64 * nl)(*[len(it) for it in hn_items_per_layer])
        self.h = C.c_void_p()
        bad = C.c_uint64(0)
        ep = -1 if st["enter_point"] is None else int(st["enter_point"])
        L.check(L.lib().sdb_hnsw_load_staged(ctx.h, self.dim, L.METRIC[self.metric], self.n, C.c_void_p(vb.ctypes.data),
                                             C.c_void_p(vo.ctypes.data), C.c_void_p(vi.ctypes.data), len(he_items), nl,
                                             NB, NO, NI, NN, ep, C.byref(self.h), C.byref(bad)))
        self.n_bad = bad.value
        self.set_minkowski_order(minkowski_order)
        return self

    def set_minkowski_order(self, order):
        """the p of Distance::Minkowski(p) (sdb_hnsw_set_minkowski_order); may change between searches.  NaN raises
        SdbError(SDB_EINVAL).  Ignored by the other metrics."""
        L.check(L.lib().sdb_hnsw_set_minkowski_order(self.h, float(order)))

    # ---- freshness: layer versions (Hs) and the pending log (Hp) ---------------------------------------------------
    def check_state(self, state_value):
        """Hnsw::check_state (hnsw/mod.rs:187-224): the persisted HnswState carries one version per layer; a layer
        whose version differs from the loaded one must be reloaded.  Returns True when the device copy is current,
        False when the caller has to rebuild it (HnswIndex.from_kv) before searching."""
        from . import staging as S
        st = S.parse_hnsw_state(state_value)
        cur = [st["layer0"]["version"]] + [l["version"] for l in st["layers"]]
        return self.versions is not None and cur == self.versions and int(st["next_element_id"]) == self.n

    def add_pending(self, vector_id, old_vectors, new_vectors):
        """one VectorPendingUpdate of the Hp range, in key order (hnsw/index.rs:424-452).  vector_id: an int (VectorId::
        DocId) or any other hashable (VectorId::RecordKey); new_vectors empty = deletion."""
        self.pendings.append((vector_id, [np.asarray(v, np.float32) for v in old_vectors],
                              [np.asarray(v, np.float32) for v in new_vectors]))

    def clear_pendings(self):
        """index_pendings applied the log (hnsw/index.rs:138-211): the caller reloads the graph and drops the log"""
        self.pendings = []

    @staticmethod
    def _vid_key(vid):
        """VectorId ordering (derive(PartialOrd, Ord), hnsw/mod.rs:109-113): every DocId sorts before every RecordKey"""
        return (0, int(vid)) if isinstance(vid, (int, np.integer)) else (1, vid)

    def _typed_distances(self, query, vectors):
        """Distance::calculate(&search.pt, &vector) for F32 vectors with the index's metric and Minkowski order, on the
        GPU (sdb_hnsw_distance_f32)"""
        q = np.ascontiguousarray(query, np.float32)
        v = np.ascontiguousarray(vectors, np.float32).reshape(-1, self.dim)
        out = np.zeros(v.shape[0], np.float64)
        L.check(L.lib().sdb_hnsw_distance_f32(self.h, C.c_void_p(q.ctypes.data), C.c_void_p(v.ctypes.data), v.shape[0],
                                              C.c_void_p(out.ctypes.data)))
        return out

    def search_graph(self, queries, k, ef, counters=False, truthy=None, all_docs_pending=None):
        """truthy: optional predicate mask, one byte per element (Hnsw::knn_search_with_filter, hnsw/mod.rs:488-515).
        all_docs_pending: optional mask, one byte per element: every document of the element has a pending update
        (the pending_docs argument of Hnsw::knn_search evaluated per element, hnsw/layer.rs:209,320-339)."""
        q = np.ascontiguousarray(queries, np.float32)
        if q.ndim == 1:
            q = q[None, :]
        if q.shape[1] != self.dim:  # Error::InvalidVectorDimension  idx/trees/vector.rs:643-652
            raise L.SdbError(L.SDB_EDIM, f"Incorrect vector dimension ({q.shape[1]}). Expected a vector of {self.dim} dimension.")
        nq = q.shape[0]
        ids = np.zeros((nq, max(k, 1)), np.uint64)
        dist = np.zeros((nq, max(k, 1)), np.float64)
        cnt = np.zeros(nq, np.uint32)
        ctr = np.zeros((nq, 2), np.uint64)
        if truthy is not None and all_docs_pending is not None:
            # add_if_truthy ignores an element whose documents are all pending (layer.rs:287-296)
            truthy = np.asarray(truthy, np.uint8) & (np.asarray(all_docs_pending, np.uint8) == 0)
        elif all_docs_pending is not None:
            m = np.ascontiguousarray(all_docs_pending, np.uint8)
            if m.shape != (self.n,):
                raise L.SdbError(L.SDB_EINVAL, f"pending mask must have one byte per element ({self.n})")
            L.check(L.lib().sdb_hnsw_search_pending(self.h, C.c_void_p(q.ctypes.data), nq, int(k), int(ef),
                                                    C.c_void_p(m.ctypes.data), C.c_void_p(ids.ctypes.data),
                                                    C.c_void_p(dist.ctypes.data), C.c_void_p(cnt.ctypes.data),
                                                    C.c_void_p(ctr.ctypes.data)))
            return (ids, dist, cnt, ctr) if counters else (ids, dist, cnt)
        if truthy is not None:
            t = np.ascontiguousarray(truthy, np.uint8)
            if t.shape != (self.n,):
                raise L.SdbError(L.SDB_EINVAL, f"predicate mask must have one byte per element ({self.n})")
            L.check(L.lib().sdb_hnsw_search_filtered(self.h, C.c_void_p(q.ctypes.data), nq, int(k), int(ef),
                                                     C.c_void_p(t.ctypes.data), C.c_void_p(ids.ctypes.data),
                                                     C.c_void_p(dist.ctypes.data), C.c_void_p(cnt.ctypes.data),
                                                     C.c_void_p(ctr.ctypes.data)))
        else:
            L.check(L.lib().sdb_hnsw_search(self.h, C.c_void_p(q.ctypes.data), nq, int(k), int(ef),
                                            C.c_void_p(ids.ctypes.data), C.c_void_p(dist.ctypes.data),
                                            C.c_void_p(cnt.ctypes.data), C.c_void_p(ctr.ctypes.data)))
        if counters:
            return ids, dist, cnt, ctr
        return ids, dist, cnt

    def knn_search(self, query, k, ef, truthy_docs=None):
        """-> [(vector id, distance)] ordered by (distance, VectorId), at most k  (one query).  Mirrors
        HnswIndex::knn_search (hnsw/index.rs:270-335):
          1. search_pendings (:372-420): the Hp log is folded per VectorId (a later deletion removes it, a later
             update replaces it); every surviving new vector is ranked with Distance::calculate and offered to the
             KnnResultBuilder; the DocIds seen in ANY pending update form the pending_docs bitmap.
          2. search_graph (:341-364) with that bitmap: an element whose docs are all pending is kept in w but not
             expanded (unfiltered) / ignored by add_if_truthy (filtered); add_graph_results adds ALL docs of each
             neighbour (:454-475).
        truthy_docs: optional set of vector ids passing the WHERE condition (cond_filter): an element enters the result
        window if ANY of its docs is truthy (HnswTruthyDocumentFilter::check_any_doc_truthy, hnsw/filter.rs:52-62); a
        pending vector is skipped unless its id is truthy (check_vector_id_truthy).  The executor re-applies the
        WHERE clause downstream."""
        builder = KnnResultBuilder(k, self._vid_key)
        # ---- 1. pendings ----
        all_existing_docs, non_deleted = set(), {}
        for vid, _old, new in self.pendings:
            if isinstance(vid, (int, np.integer)):
                all_existing_docs.add(int(vid))
            if len(new) == 0:
                non_deleted.pop(vid, None)
            else:
                non_deleted[vid] = new
        pending_docs = None
        if all_existing_docs or non_deleted:
            for vid, vectors in non_deleted.items():  # (HashMap iteration order: the builder's set makes it irrelevant)
                if truthy_docs is not None and vid not in truthy_docs:
                    continue
                for d in self._typed_distances(query, np.stack(vectors)):
                    if builder.check_add(float(d)):
                        builder.add_vector_id_result(float(d), vid)
            if all_existing_docs:
                pending_docs = all_existing_docs
        # ---- 2. graph ----
        docs_of = (lambda e: [e]) if self.elem_docs is None else (lambda e: self.elem_docs[e])
        truthy = None
        if truthy_docs is not None:
            truthy = np.zeros(self.n, np.uint8)
            for e in range(self.n):
                truthy[e] = any(d in truthy_docs for d in docs_of(e))
        all_pending = None
        if pending_docs:
            all_pending = np.zeros(self.n, np.uint8)
            for e in range(self.n):
                dl = docs_of(e)
                all_pending[e] = all(int(d) in pending_docs for d in dl)  # an element without docs counts as pending
        ids, dist, cnt = self.search_graph(np.asarray(query, np.float32)[None, :], k, ef, truthy=truthy,
                                           all_docs_pending=all_pending)
        for j in range(int(cnt[0])):
            d, e = float(dist[0, j]), int(ids[0, j])
            if builder.check_add(d):
                for doc in docs_of(e):
                    builder.add_vector_id_result(d, int(doc))
        return [(vid, d) for d, vid in builder.collect()]

    def close(self):
        if self.h:
            L.lib().sdb_hnsw_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
