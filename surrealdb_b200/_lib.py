"""ctypes loader of the C-ABI library (surrealdb_b200/csrc/libsdbgpu.so, declared in include/sdbgpu.h).

There is NO CPU fallback: if the shared library is missing this module raises, and if no B200 is
visible every call returns SDB_ECUDA which is raised as SdbError.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "csrc", "libsdbgpu.so")

(SDB_OK, SDB_EINVAL, SDB_EDIM, SDB_ENOMEM, SDB_ECUDA, SDB_ECANCELLED, SDB_EUNSUPPORTED, SDB_EOVERFLOW,
 SDB_ENCCL) = range(9)
STATUS_NAMES = ["SDB_OK", "SDB_EINVAL", "SDB_EDIM", "SDB_ENOMEM", "SDB_ECUDA", "SDB_ECANCELLED",
                "SDB_EUNSUPPORTED", "SDB_EOVERFLOW", "SDB_ENCCL"]
COMM_ID_BYTES = 128
METRIC = {"CHEBYSHEV": 0, "COSINE": 1, "EUCLIDEAN": 2, "HAMMING": 3, "JACCARD": 4, "MANHATTAN": 5,
          "MINKOWSKI": 6, "PEARSON": 7}
DTYPE = {"F32": 0, "F64": 1}
VECTOR_FN = {"SIMILARITY_COSINE": 16, "DOT": 17, "MAGNITUDE": 18}
SCREEN = {"AUTO": 0, "SIMT_F32": 1, "TC_BF16": 2, "NONE_EXACT": 3, "TC_INT8": 4}

# every symbol include/sdbgpu.h declares (tests/test_abi_symbols.py cross-checks this list with the header)
ABI_SYMBOLS = [
    "sdb_ctx_create", "sdb_ctx_destroy", "sdb_last_error", "sdb_version", "sdb_pinned_alloc", "sdb_pinned_free",
    "sdb_ctx_cancel", "sdb_ctx_cancel_reset", "sdb_debug_schedule", "sdb_ctx_kernel_launches", "sdb_ctx_stream", "sdb_corpus_create", "sdb_corpus_destroy", "sdb_corpus_append",
    "sdb_corpus_append_device", "sdb_corpus_append_synthetic", "sdb_corpus_set_skip", "sdb_corpus_remove", "sdb_corpus_finalize",
    "sdb_corpus_rows", "sdb_corpus_read_rows", "sdb_corpus_set_minkowski_order", "sdb_corpus_set_screen", "sdb_corpus_set_schedule", "sdb_corpus_set_exact", "sdb_knn_bruteforce", "sdb_knn_bruteforce_device",
    "sdb_knn_last_stats", "sdb_knn_submit", "sdb_knn_submit_device", "sdb_knn_wait", "sdb_comm_unique_id",
    "sdb_comm_init_rank", "sdb_comm_size", "sdb_comm_rank", "sdb_ctx_create_multi", "sdb_corpus_set_row_base",
    "sdb_knn_sharded_submit", "sdb_knn_sharded_submit_device", "sdb_knn_sharded_wait", "sdb_knn_sharded_multi",
    "sdb_corpus_project", "sdb_topk_merge_device", "sdb_hnsw_load", "sdb_hnsw_load_device", "sdb_hnsw_search_device", "sdb_hnsw_select_neighbors_ids", "sdb_hnsw_destroy", "sdb_stage_decode_vectors", "sdb_stage_decode_nodes", "sdb_hnsw_load_staged", "sdb_hnsw_search", "sdb_hnsw_search_filtered", "sdb_hnsw_search_pending", "sdb_vec_distance_f32", "sdb_hnsw_distance_f32", "sdb_hnsw_set_minkowski_order", "sdb_hnsw_select_neighbors",
    "sdb_graph_load_csr", "sdb_graph_load_csr_shard", "sdb_graph_destroy", "sdb_graph_expand", "sdb_graph_expand_device", "sdb_device_free", "sdb_graph_collect", "sdb_free",
]


class SdbError(RuntimeError):
    def __init__(self, status, message):
        super().__init__(f"{STATUS_NAMES[status] if 0 <= status < len(STATUS_NAMES) else status}: {message}")
        self.status = status


class KnnStats(C.Structure):
    _fields_ = [("screen_used", C.c_uint32), ("n_passes", C.c_uint32), ("n_fallback", C.c_uint32),
                ("n_special_rows", C.c_uint32), ("n_candidates", C.c_uint64), ("n_reranked", C.c_uint64),
                ("kernel_launches", C.c_uint64), ("screen_ms", C.c_float), ("total_ms", C.c_float),
                ("n_survivors", C.c_uint64), ("n_repaired", C.c_uint32), ("reserved0", C.c_uint32)]


_lib = None


def lib():
    """Loads libsdbgpu.so or fails loudly."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise ImportError(f"{SO_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(make -C surrealdb_b200/csrc).  There is no CPU fallback.")
    L = C.CDLL(SO_PATH)
    vp, u64, u32, i32 = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int
    L.sdb_last_error.restype = C.c_char_p
    L.sdb_version.restype = C.c_char_p
    L.sdb_pinned_alloc.restype = vp
    L.sdb_pinned_alloc.argtypes = [C.c_size_t]
    L.sdb_pinned_free.argtypes = [vp]
    L.sdb_ctx_create.argtypes = [i32, C.POINTER(vp)]
    L.sdb_ctx_destroy.argtypes = [vp]
    L.sdb_ctx_cancel.argtypes = [vp]
    L.sdb_ctx_cancel.restype = None
    L.sdb_ctx_cancel_reset.argtypes = [vp]
    L.sdb_ctx_cancel_reset.restype = None
    L.sdb_ctx_kernel_launches.restype = u64
    L.sdb_ctx_kernel_launches.argtypes = [vp]
    L.sdb_ctx_stream.restype = vp
    L.sdb_ctx_stream.argtypes = [vp]
    L.sdb_corpus_create.argtypes = [vp, u32, i32, i32, u64, C.POINTER(vp)]
    L.sdb_corpus_destroy.argtypes = [vp]
    L.sdb_corpus_append.argtypes = [vp, vp, u64]
    L.sdb_corpus_append_device.argtypes = [vp, vp, u64]
    L.sdb_corpus_append_synthetic.argtypes = [vp, u64, u64, u64]
    L.sdb_corpus_set_skip.argtypes = [vp, vp, u64]
    L.sdb_corpus_remove.argtypes = [vp, vp, u64]
    L.sdb_corpus_finalize.argtypes = [vp]
    L.sdb_corpus_rows.restype = u64
    L.sdb_corpus_rows.argtypes = [vp]
    L.sdb_corpus_read_rows.argtypes = [vp, u64, u64, vp]
    L.sdb_corpus_set_screen.argtypes = [vp, i32]
    L.sdb_corpus_set_exact.argtypes = [vp, i32]
    L.sdb_corpus_set_minkowski_order.argtypes = [vp, C.c_double]
    L.sdb_corpus_set_schedule.argtypes = [vp, i32]
    L.sdb_knn_bruteforce.argtypes = [vp, vp, u32, u32, vp, vp, vp, vp]
    L.sdb_knn_bruteforce_device.argtypes = [vp, vp, u32, u32, u64, vp, vp, vp]
    L.sdb_knn_submit.argtypes = [vp, vp, u32, u32, vp, vp, vp, C.POINTER(u32)]
    L.sdb_knn_submit_device.argtypes = [vp, vp, u32, u32, u64, vp, vp, vp, C.POINTER(u32)]
    L.sdb_knn_wait.argtypes = [vp, u32]
    L.sdb_comm_unique_id.argtypes = [vp]
    L.sdb_comm_init_rank.argtypes = [vp, i32, i32, vp]
    L.sdb_comm_size.argtypes = [vp]
    L.sdb_comm_rank.argtypes = [vp]
    L.sdb_ctx_create_multi.argtypes = [vp, i32, vp]
    L.sdb_corpus_set_row_base.argtypes = [vp, u64]
    L.sdb_knn_sharded_submit.argtypes = [vp, vp, u32, u32, vp, vp, vp, C.POINTER(u32)]
    L.sdb_knn_sharded_submit_device.argtypes = [vp, vp, u32, u32, vp, vp, vp, C.POINTER(u32)]
    L.sdb_knn_sharded_wait.argtypes = [vp, u32]
    L.sdb_knn_sharded_multi.argtypes = [vp, i32, vp, u32, u32, vp, vp, vp]
    L.sdb_corpus_project.argtypes = [vp, vp, i32, vp]
    L.sdb_knn_last_stats.argtypes = [vp, C.POINTER(KnnStats)]
    L.sdb_topk_merge_device.argtypes = [vp, u32, u32, u32, vp, vp, vp, u64, u64, u64, vp, vp, vp]
    L.sdb_hnsw_load.argtypes = [vp, u32, i32, u64, vp, u32, vp, vp, C.c_int64, C.POINTER(vp)]
    L.sdb_hnsw_load_device.argtypes = [vp, u32, i32, u64, vp, u32, vp, vp, C.c_int64, C.POINTER(vp)]
    L.sdb_hnsw_search_device.argtypes = [vp, vp, u32, u32, u32, vp, vp, vp]
    L.sdb_hnsw_select_neighbors_ids.argtypes = [vp, vp, u32, i32, vp, u64, vp, vp, u32, u32, i32, vp, vp]
    L.sdb_hnsw_destroy.argtypes = [vp]
    L.sdb_stage_decode_vectors.argtypes = [vp, vp, vp, vp, u64, u32, i32, u64, vp, vp, C.POINTER(u64)]
    L.sdb_stage_decode_nodes.argtypes = [vp, vp, vp, vp, u64, u64, C.POINTER(vp), C.POINTER(vp), C.POINTER(u64)]
    L.sdb_hnsw_load_staged.argtypes = [vp, u32, i32, u64, vp, vp, vp, u64, u32, vp, vp, vp, vp, C.c_int64, C.POINTER(vp),
                                       C.POINTER(u64)]
    L.sdb_hnsw_search.argtypes = [vp, vp, u32, u32, u32, vp, vp, vp, vp]
    L.sdb_hnsw_search_filtered.argtypes = [vp, vp, u32, u32, u32, vp, vp, vp, vp, vp]
    L.sdb_hnsw_search_pending.argtypes = [vp, vp, u32, u32, u32, vp, vp, vp, vp, vp]
    L.sdb_vec_distance_f32.argtypes = [vp, i32, u32, vp, vp, u64, vp]
    L.sdb_hnsw_distance_f32.argtypes = [vp, vp, vp, u64, vp]
    L.sdb_hnsw_set_minkowski_order.argtypes = [vp, C.c_double]
    L.sdb_hnsw_select_neighbors.argtypes = [vp, vp, u32, i32, u64, u64, vp, vp, u32, u32, i32, vp, vp]
    L.sdb_graph_load_csr.argtypes = [vp, u64, vp, vp, C.POINTER(vp)]
    L.sdb_graph_load_csr_shard.argtypes = [vp, u64, u64, u64, vp, vp, C.POINTER(vp)]
    L.sdb_graph_destroy.argtypes = [vp]
    L.sdb_graph_expand.argtypes = [vp, u32, vp, u64, u32, C.POINTER(vp), C.POINTER(u64)]
    L.sdb_graph_expand_device.argtypes = [vp, u32, vp, u64, u32, C.POINTER(vp), C.POINTER(u64)]
    L.sdb_device_free.argtypes = [vp, vp]
    L.sdb_graph_collect.argtypes = [vp, vp, u64, u32, u32, i32, C.POINTER(vp), C.POINTER(u64)]
    L.sdb_free.argtypes = [vp]
    _lib = L
    return L


def check(status):
    if status != SDB_OK:
        raise SdbError(status, lib().sdb_last_error().decode("utf-8", "replace"))
