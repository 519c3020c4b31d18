/*
 * sdbgpu.h -- C ABI of the B200-native KNN / HNSW / graph-expansion engine.
 *
 * This is the drop-in boundary for SurrealDB's vector-similarity and graph-scan hot path
 * (SURVEY.md section 8b).  The reference has NO FFI of its own (pure Rust, SURVEY F4/F5), so each
 * entry point below names the Rust-internal seam it replaces; INTEGRATION.md shows the
 * `extern "C"` block and the operator wrappers a maintainer adds behind a `gpu-knn` cargo feature.
 * Paths are relative to surrealdb/core/src in the reference checkout.
 *
 * Conventions
 *  - plain pointers and sizes only; no C++/torch types cross the boundary.
 *  - every function is thread-safe per handle family: concurrent searches on one corpus/hnsw/graph
 *    handle are serialised internally (one in-flight search per handle); mutation
 *    (append/finalize) must not race with searches -- the same RW discipline the reference applies
 *    to its HNSW graph (idx/trees/hnsw/index.rs:55,224,350).
 *  - errors: integer status + thread-local message (sdb_last_error); nothing unwinds across the ABI.
 *  - "rows" are scan positions: the caller appends vectors in the reference's scan order (record-key
 *    byte order, i.e. what TableScan yields) and maps returned row numbers back to RecordIds.
 *  - NO CPU FALLBACK: if no CUDA device is usable every entry point fails with SDB_ECUDA.
 */
#ifndef SDBGPU_H
#define SDBGPU_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct sdb_ctx sdb_ctx;       /* one CUDA device: streams, scratch, TMA driver entry points   */
typedef struct sdb_corpus sdb_corpus; /* device-resident N x D vector column (+ norms, screen copy)    */
typedef struct sdb_hnsw sdb_hnsw;     /* device-resident HNSW layers (CSR) + element vectors           */
typedef struct sdb_graph sdb_graph;   /* device-resident CSR adjacency of one (direction, edge table)  */

typedef enum {
  SDB_OK = 0,
  SDB_EINVAL = 1,     /* bad argument                                                               */
  SDB_EDIM = 2,       /* dimension mismatch -> Error::InvalidVectorDimension (idx/trees/vector.rs:643) */
  SDB_ENOMEM = 3,
  SDB_ECUDA = 4,      /* CUDA runtime/driver failure, or no sm_100 device                           */
  SDB_ECANCELLED = 5, /* cancel flag observed -> Error::QueryCancelled (exec/operators/knn_topk.rs:186) */
  SDB_EUNSUPPORTED = 6,
  SDB_EOVERFLOW = 7,  /* caller-provided output capacity too small / too many batches in flight      */
  SDB_ENCCL = 8       /* NCCL failure (multi-GPU entry points)                                      */
} sdb_status;

/* catalog::Distance (catalog/schema/index.rs:247-284).  COSINE and EUCLIDEAN are screened on the tensor cores and
 * re-ranked exactly; the other six run through the exact kernel (sequential f64, Distance::compute op for op). */
typedef enum {
  SDB_CHEBYSHEV = 0,
  SDB_COSINE = 1,
  SDB_EUCLIDEAN = 2,
  SDB_HAMMING = 3,
  SDB_JACCARD = 4,
  SDB_MANHATTAN = 5,
  SDB_MINKOWSKI = 6,
  SDB_PEARSON = 7
} sdb_metric;

/* element type of the rows handed to sdb_corpus_append (catalog VectorType, index.rs:321-334).
 * Brute-force KnnTopK holds Vec<Number>: F64 covers arbitrary Number::Float rows, F32 covers rows whose
 * values are f32-representable (the BASELINE configs) and enables the low-precision screen. */
typedef enum { SDB_F32 = 0, SDB_F64 = 1 } sdb_dtype;

/* which screening kernel sdb_knn_bruteforce uses (results are identical for all; this only moves the performance
 * point).  AUTO: cosine corpora whose normalised rows quantise well (largest relative int8 error <= 0.02 once the few
 * outlier rows are set aside) start on the int8 tensor-core screen, everything else on the bf16 one; queries whose
 * proof fails climb to finer screens (bf16, then the f32 stream) before the exact kernel. */
typedef enum {
  SDB_SCREEN_AUTO = 0,
  SDB_SCREEN_SIMT_F32 = 1,   /* f32 streaming SIMT kernel                                             */
  SDB_SCREEN_TC_BF16 = 2,    /* tcgen05 kind::f16, bf16 operands                                        */
  SDB_SCREEN_NONE_EXACT = 3, /* no screen: exact f64 kernel for every query                              */
  SDB_SCREEN_TC_INT8 = 4     /* tcgen05 kind::i8, int8 copy of the normalised rows (cosine); falls back to bf16 */
} sdb_screen;

/* counters of the last brute-force call on a corpus (diagnostics / bench roofline arithmetic) */
typedef struct {
  uint32_t screen_used;      /* sdb_screen actually run                                        */
  uint32_t n_passes;         /* threshold-refinement passes of the screen                      */
  uint32_t n_fallback;       /* queries re-run through the exact kernel (verification failed)  */
  uint32_t n_special_rows;   /* rows with zero / non-finite norm (always exact-ranked)         */
  uint64_t n_candidates;     /* largest candidate set of any query that reached the exact re-rank */
  uint64_t n_reranked;       /* exact f64 distances computed by the re-rank kernel             */
  uint64_t kernel_launches;  /* kernels launched by this call                                  */
  float screen_ms;           /* device time of the screening kernels (CUDA events)             */
  float total_ms;            /* device time of the whole call                                  */
  uint64_t n_survivors;      /* screened rows that passed a threshold and were gathered (all queries) */
  uint32_t n_repaired;       /* queries whose proof failed on the batch's screen and succeeded on a finer one
                                (re-screened as a small batch of their own; never reached the exact kernel) */
  uint32_t reserved0;
} sdb_knn_stats;

/* ---- context -------------------------------------------------------------------------------- */
sdb_status sdb_ctx_create(int device, sdb_ctx** out);
void sdb_ctx_destroy(sdb_ctx*);
const char* sdb_last_error(void); /* thread-local; valid until the next call on this thread */
const char* sdb_version(void);
void* sdb_pinned_alloc(size_t bytes); /* cudaHostAlloc: staging buffers for append / queries */
void sdb_pinned_free(void*);
/* Cancellation of whatever runs on this context, from any thread: the counterpart of the reference's ctx.is_done()
 * polls (exec/operators/knn_topk.rs:186, idx/trees/hnsw/index.rs:437, hnsw/layer.rs:533).  Brute force polls between
 * kernel phases and before every exact fallback, the HNSW walk before every query (inside the kernel), graph expansion
 * before every hop / BFS level.  A cancelled call returns SDB_ECANCELLED and its outputs are undefined.  The flag stays
 * up until sdb_ctx_cancel_reset.  (sdb_knn_bruteforce additionally takes a per-call flag.) */
void sdb_ctx_cancel(sdb_ctx*);
void sdb_ctx_cancel_reset(sdb_ctx*);
/* total kernels launched through this context since creation (bench's gpu_launches) */
/* Host-only diagnostic (needs no GPU): the sequence of corpus tiles (256 rows each) the screen of one batch visits --
 * the streaming schedule's main launch (its probe tiles are returned separately) or, with streaming = 0, the passes of
 * the multi-pass schedule.  No reference seam; exists so that "every tile is screened exactly once" can be tested on
 * the CPU for any corpus size.  out_tiles / out_probe_tiles may be NULL (counts only). */
sdb_status sdb_debug_schedule(uint64_t n_rows, uint32_t cand_cap, uint32_t k, uint32_t nq, int streaming,
                              uint32_t* out_tiles, uint64_t cap_tiles, uint64_t* out_n, uint32_t* out_probe_tiles,
                              uint32_t cap_probe, uint32_t* out_n_probe);
uint64_t sdb_ctx_kernel_launches(const sdb_ctx*);
/* the cudaStream_t every kernel of this context is launched on (so a harness can bracket calls with
 * CUDA events on the launching stream) */
void* sdb_ctx_stream(const sdb_ctx*);

/* ---- brute-force KNN: replaces KnnTopK::execute (exec/operators/knn_topk.rs:166-267) and the
 *      legacy QueryExecutor::knn (idx/planner/executor.rs:283-311) ----------------------------- */
sdb_status sdb_corpus_create(sdb_ctx*, uint32_t dim, sdb_dtype, sdb_metric, uint64_t capacity_rows, sdb_corpus** out);
void sdb_corpus_destroy(sdb_corpus*);
/* rows: host memory (pinned preferred), row-major n x dim of the corpus dtype, in scan order. */
sdb_status sdb_corpus_append(sdb_corpus*, const void* rows, uint64_t n);
/* same, rows already in device memory of this context's device */
sdb_status sdb_corpus_append_device(sdb_corpus*, const void* d_rows, uint64_t n);
/* synthetic rows generated in HBM by the counter-based generator shared with the oracle
 * (element (r, c) = gen(seed, (first_row + r) * dim + c)); bench/test input only. */
sdb_status sdb_corpus_append_synthetic(sdb_corpus*, uint64_t seed, uint64_t first_row, uint64_t n);
/* rows the reference would skip (field missing / non-numeric / dimension mismatch:
 * extract_vector, knn_topk.rs:274-288; residual WHERE filter, planner/select.rs:1642-1652).
 * skip[i] != 0 excludes row i.  May be called again to change the mask. */
sdb_status sdb_corpus_set_skip(sdb_corpus*, const uint8_t* skip, uint64_t n);
/* Tombstones: the rows (scan positions) are excluded from every later search, as if the reference's TableScan no
 * longer yielded them (a DELETE, or the old version of an UPDATE whose new version is appended at the end of the
 * column).  Works on a finalized corpus without re-finalizing (skip mask + NaN screening norm + zeroed int8 row) and
 * before finalize (skip mask only).  Must not race with searches.  Row numbers of the remaining rows do not change;
 * the caller compacts (new corpus) when the tombstones pile up, or when the table version moved (KnnTopK has no
 * persistent state of its own: the cached column is keyed by (ns, db, table, field, table version), SURVEY 8f-1). */
sdb_status sdb_corpus_remove(sdb_corpus*, const uint64_t* row_ids, uint64_t n);
/* builds per-row exact f64 magnitudes, f32 screening norms, the bf16 screen copy and the special-row
 * list.  Must be called after the last append and before searching. */
sdb_status sdb_corpus_finalize(sdb_corpus*);
uint64_t sdb_corpus_rows(const sdb_corpus*);
/* copies rows [first_row, first_row + n) of the device-resident master copy back to host memory (n x dim of the
 * corpus dtype): lets a harness check results against exactly the bytes the kernels read */
sdb_status sdb_corpus_read_rows(sdb_corpus*, uint64_t first_row, uint64_t n, void* out);
/* order p of Distance::Minkowski(p) (catalog/schema/index.rs:247-284; fnc/util/math/vector.rs:163-174); default 3.
 * MINKOWSKI goes through pow(): CUDA's libm here, the platform libm in the reference -- each call agrees to within an
 * ulp or two, so Minkowski distances are equal to ~1e-14 relative rather than bit for bit (every other metric is
 * bit-exact). */
sdb_status sdb_corpus_set_minkowski_order(sdb_corpus*, double order);
sdb_status sdb_corpus_set_screen(sdb_corpus*, sdb_screen);
/* schedule of the tensor-core screens (results are identical; tuning / A-B only).  streaming = 1 (default): a scored
 * sample seeds the thresholds, then ONE launch streams the rest of the corpus while refiner warps raise the thresholds
 * inside the kernel.  streaming = 0: the multi-pass schedule (a launch + a selection kernel per geometric pass). */
sdb_status sdb_corpus_set_schedule(sdb_corpus*, int streaming);
/* exact = 1 (default): results are proven identical to the reference (queries whose proof fails are re-run by the exact
 * kernel).  exact = 0: opt-in approximate mode -- the exactly re-ranked best candidates of the screen are returned
 * without the proof / fallback (used by the index builder, where near-duplicate clusters would otherwise send every
 * query to the exact kernel). */
sdb_status sdb_corpus_set_exact(sdb_corpus*, int exact);
/* queries: nq x dim f64 (the reference's query is Vec<Number>; Number::Float values).
 * out_rows / out_dist: nq x k, nearest first, ties by scan order; out_count[q] <= k.
 * cancel_flag (nullable) is polled between kernel phases.  */
sdb_status sdb_knn_bruteforce(sdb_corpus*, const double* queries, uint32_t nq, uint32_t k, uint64_t* out_rows,
                              double* out_dist, uint32_t* out_count, const volatile int* cancel_flag);
/* device-resident variant: d_queries / d_out_* are device pointers; results are complete when the
 * call returns.  row_base is added to every returned row (global id of a row-sharded corpus). */
sdb_status sdb_knn_bruteforce_device(sdb_corpus*, const double* d_queries, uint32_t nq, uint32_t k,
                                     uint64_t row_base, uint64_t* d_out_rows, double* d_out_dist,
                                     uint32_t* d_out_count);
sdb_status sdb_knn_last_stats(const sdb_corpus*, sdb_knn_stats* out);

/* ---- asynchronous batches.  submit enqueues a whole batch (query preparation, screen, exact re-rank, proof, result
 * copy) on the context's stream WITHOUT any host synchronisation and returns a ticket; wait blocks until that batch is
 * complete (and, for the rare query whose proof failed, runs the exact kernel).  Up to 4 batches may be in flight per
 * corpus, so the host can prepare / transfer batch i+1 while batch i computes -- the shape in which concurrent
 * SurrealQL queries arrive at KnnTopK::execute (one operator instance per query, exec/operators/knn_topk.rs:166).
 * Buffers handed to submit must stay valid until the matching wait returns.  Host variant: `queries` and `out_*` are
 * host buffers (pinned for overlap); the H2D copy runs on a separate copy stream.  Tickets complete in any order. */
sdb_status sdb_knn_submit(sdb_corpus*, const double* queries, uint32_t nq, uint32_t k, uint64_t* out_rows,
                          double* out_dist, uint32_t* out_count, uint32_t* ticket);
sdb_status sdb_knn_submit_device(sdb_corpus*, const double* d_queries, uint32_t nq, uint32_t k, uint64_t row_base,
                                 uint64_t* d_out_rows, double* d_out_dist, uint32_t* d_out_count, uint32_t* ticket);
sdb_status sdb_knn_wait(sdb_corpus*, uint32_t ticket);

/* ---- multi-GPU brute force (SURVEY 8e): the corpus is row-sharded, every shard searches its rows, ONE NCCL
 * all-gather moves the per-shard top-k blocks and a merge kernel on every rank produces the global top-k by
 * (distance, global row).  NCCL lives inside the library (bound at run time with dlopen, so single-GPU users need
 * none); everything is enqueued on the context's stream without host synchronisation.
 *   one process per GPU : rank 0 calls sdb_comm_unique_id and hands the 128 bytes to the other ranks out of band;
 *                         every rank calls sdb_comm_init_rank on its context (collective).
 *   one process, N GPUs : sdb_ctx_create_multi creates the N contexts and their communicator (ncclCommInitAll);
 *                         sdb_knn_sharded_multi drives all shards from the calling thread.
 * A corpus becomes a shard by sdb_corpus_set_row_base(first global row).  sdb_knn_sharded_* are COLLECTIVE: every
 * rank must call them with the same queries, nq and k, in the same order.  Exactness across ranks: each block carries
 * the number of queries its rank must still repair on the host (failed proof, special queries); every rank sees every
 * header after the all-gather, so all ranks agree on whether a repair round (local exact re-runs, second all-gather
 * and merge) is needed -- no extra collective. */
#define SDB_COMM_ID_BYTES 128
sdb_status sdb_comm_unique_id(uint8_t* id128);
sdb_status sdb_comm_init_rank(sdb_ctx*, int nranks, int rank, const uint8_t* id128);
int sdb_comm_size(const sdb_ctx*);
int sdb_comm_rank(const sdb_ctx*);
sdb_status sdb_ctx_create_multi(const int* devices, int ndev, sdb_ctx** out /* [ndev] */);
sdb_status sdb_corpus_set_row_base(sdb_corpus*, uint64_t first_global_row);
sdb_status sdb_knn_sharded_submit(sdb_corpus*, const double* queries, uint32_t nq, uint32_t k, uint64_t* out_rows,
                                  double* out_dist, uint32_t* out_count, uint32_t* ticket);
sdb_status sdb_knn_sharded_submit_device(sdb_corpus*, const double* d_queries, uint32_t nq, uint32_t k,
                                         uint64_t* d_out_rows, double* d_out_dist, uint32_t* d_out_count,
                                         uint32_t* ticket);
sdb_status sdb_knn_sharded_wait(sdb_corpus*, uint32_t ticket);
/* one process, N GPUs: shards[i] lives on the i-th context of sdb_ctx_create_multi; queries / out_* are host buffers */
sdb_status sdb_knn_sharded_multi(sdb_corpus* const* shards, int n_shards, const double* queries, uint32_t nq, uint32_t k,
                                 uint64_t* out_rows, double* out_dist, uint32_t* out_count);
/* ---- projected scalar vector functions over a whole column (SURVEY 8f-4): replaces a per-row evaluation of
 *      vector::distance::* / vector::similarity::* / vector::dot / vector::magnitude (fnc/vector.rs:25-143,
 *      fnc/util/math/vector.rs:61-314) in `SELECT vector::similarity::cosine(emb, $q) FROM t`.
 * fn: an sdb_metric id (= what Distance::compute returns for it: COSINE -> cosine DISTANCE, PEARSON -> the
 * similarity, JACCARD -> the similarity, MINKOWSKI with the corpus' order) or one of sdb_vector_fn.  out: host, one f64 per row in scan order,
 * bit-identical to the reference's sequential f64 arithmetic; skipped rows get NaN.  query: host, dim doubles
 * (ignored for SDB_FN_MAGNITUDE). */
typedef enum { SDB_FN_SIMILARITY_COSINE = 16, SDB_FN_DOT = 17, SDB_FN_MAGNITUDE = 18 } sdb_vector_fn;
sdb_status sdb_corpus_project(sdb_corpus*, const double* query, int fn, double* out);

/* merges `n_lists` per-shard result lists (each nq x k; list l's entry j of query q is valid iff
 * j < d_counts[l*stride_counts + q]) into the global top-k by (distance, row); all pointers are device
 * pointers.  stride_* = distance in ELEMENTS between consecutive lists (0 = dense: nq*k, nq*k, nq), so the
 * lists can sit inside the per-rank blocks of ONE NCCL all-gather buffer.  This is the merge step after
 * the all-gather of per-shard candidates. */
sdb_status sdb_topk_merge_device(sdb_ctx*, uint32_t n_lists, uint32_t nq, uint32_t k, const uint64_t* d_rows,
                                 const double* d_dist, const uint32_t* d_counts, uint64_t stride_rows,
                                 uint64_t stride_dist, uint64_t stride_counts, uint64_t* d_out_rows,
                                 double* d_out_dist, uint32_t* d_out_count);

/* ---- HNSW search: replaces Hnsw::knn_search (idx/trees/hnsw/mod.rs:459-482) called from
 *      HnswIndex::search_graph (idx/trees/hnsw/index.rs:341-364) ------------------------------- */
/* vectors: n_elems x dim f32 (element id = row).  Layer l adjacency is CSR over element ids;
 * row_ptr[l] has n_elems+1 entries; neighbours keep the stored order (graph.rs:104-125).
 * Metrics: the F32 typed arithmetic of Distance::calculate (idx/trees/vector.rs:221-410,659-672) for COSINE, EUCLIDEAN,
 * MANHATTAN, CHEBYSHEV, HAMMING and MINKOWSKI (order: sdb_hnsw_set_minkowski_order), bit-exact except MINKOWSKI, whose
 * pow() agrees with the platform libm to an ulp or two per call.  PEARSON and JACCARD return SDB_EUNSUPPORTED (the index
 * keeps the reference's CPU path).  The loaders below accept the same metrics. */
sdb_status sdb_hnsw_load(sdb_ctx*, uint32_t dim, sdb_metric, uint64_t n_elems, const float* vectors,
                         uint32_t n_layers, const uint64_t* const* row_ptr, const uint32_t* const* col_idx,
                         int64_t entry_point, sdb_hnsw** out);
/* Device-resident variants for index construction (SURVEY 8f-2): vectors and per-layer CSR arrays are DEVICE pointers
 * that the handle BORROWS (nothing is copied; the caller keeps them alive and unchanged while the handle exists), and
 * the search takes device queries / writes device results.  The incremental builder re-wraps the growing graph with
 * sdb_hnsw_load_device after every insertion batch and uses the walk kernel itself as the insertion search
 * (Hnsw::insert -> HnswLayer::search_multi with efc, hnsw/mod.rs:297-377, hnsw/layer.rs:342-387). */
sdb_status sdb_hnsw_load_device(sdb_ctx*, uint32_t dim, sdb_metric, uint64_t n_elems, const float* d_vectors,
                                uint32_t n_layers, const uint64_t* const* d_row_ptr, const uint32_t* const* d_col_idx,
                                int64_t entry_point, sdb_hnsw** out);
sdb_status sdb_hnsw_search_device(sdb_hnsw*, const float* d_queries, uint32_t nq, uint32_t k, uint32_t ef,
                                  uint64_t* d_out_elems, double* d_out_dist, uint32_t* d_out_count);
void sdb_hnsw_destroy(sdb_hnsw*);
/* Filtered search: replaces Hnsw::knn_search_with_filter (hnsw/mod.rs:488-515; HnswLayer::search_single_with_filter /
 * search_with_filter / add_if_truthy, hnsw/layer.rs:111-149,226-306) when the WHERE condition has been evaluated
 * ahead of time into a predicate mask: truthy[e] != 0 iff HnswTruthyDocumentFilter::check_any_doc_truthy
 * (hnsw/filter.rs:52-136) holds for element e (host, n_elems bytes).  The descent through the upper layers is
 * unfiltered, as in the reference.  SDB_EOVERFLOW = the filter is too selective for the on-chip candidate window
 * (the caller keeps the CPU path for that query). */
sdb_status sdb_hnsw_search_filtered(sdb_hnsw*, const float* queries, uint32_t nq, uint32_t k, uint32_t ef,
                                    const uint8_t* truthy, uint64_t* out_elems, double* out_dist, uint32_t* out_count,
                                    uint64_t* out_counters);

/* Search while pending updates exist: Hnsw::knn_search(.., pending_docs = Some(bitmap)) (hnsw/mod.rs:459-482).
 * all_docs_pending[e] != 0 iff EVERY document of element e is in the pending bitmap that
 * HnswIndex::search_pendings (hnsw/index.rs:372-420) returned (are_all_docs_in_pending, hnsw/layer.rs:320-339),
 * evaluated by the caller per element (host, n_elems bytes).  Such an element still enters the result window but is
 * never expanded (layer.rs:209), in every layer.  The filtered search needs no extra entry point: add_if_truthy
 * ignores those elements (layer.rs:287-296), i.e. the caller clears their bits in the `truthy` mask. */
sdb_status sdb_hnsw_search_pending(sdb_hnsw*, const float* queries, uint32_t nq, uint32_t k, uint32_t ef,
                                   const uint8_t* all_docs_pending, uint64_t* out_elems, double* out_dist,
                                   uint32_t* out_count, uint64_t* out_counters);

/* Distance::calculate for VectorType::F32 vectors (idx/trees/vector.rs:243-289,659-672) applied to vectors that are
 * not part of the graph: the new_vectors of pending updates, which HnswIndex::search_pendings ranks by brute force
 * (hnsw/index.rs:398-404).  query: dim floats, vectors: n x dim floats, out: n doubles (all host memory).  Same
 * arithmetic as the walk kernel (cosine: f32 8-lane accumulation, f64 finish; euclid: sequential f32 sum of squares).
 * F32 typed metrics served here: cosine / euclid (sdb_hnsw_distance_f32 serves every metric of the walk). */
sdb_status sdb_vec_distance_f32(sdb_ctx*, sdb_metric, uint32_t dim, const float* query, const float* vectors, uint64_t n,
                                double* out);
/* The same for an index: Distance::calculate(query, vector) with the handle's metric and Minkowski order -- what
 * HnswIndex::search_pendings computes for the new vectors of pending updates (hnsw/index.rs:398-407).  Uses the folds
 * of the walk kernel, so a vector gets the same distance through the graph and through the pending log. */
sdb_status sdb_hnsw_distance_f32(sdb_hnsw*, const float* query, const float* vectors, uint64_t n, double* out);
/* order p of an SDB_MINKOWSKI index (Distance::Minkowski(p)); default 3, as for sdb_corpus_set_minkowski_order.  NaN
 * returns SDB_EINVAL.  May be called between searches: nothing precomputed depends on it.  Ignored by other metrics. */
sdb_status sdb_hnsw_set_minkowski_order(sdb_hnsw*, double order);

/* ---- staging: the reference's persisted HNSW state -> device (SURVEY 8a row a14).  These replace the per-key
 *      decode loops of HnswLayer::load (idx/trees/hnsw/layer.rs:526-540, UndirectedGraph::load_node
 *      idx/trees/graph.rs:117-126) and HnswElements::get_vector (hnsw/elements.rs:95-128, Vector::from(
 *      SerializedVector) idx/trees/vector.rs:93-103).  The caller range-scans the KV store and hands over the raw
 *      VALUE bytes, concatenated: value i occupies blob[off[i] .. off[i+1]).  Blobs may be pageable or pinned host
 *      memory.  *n_bad (nullable) counts values that failed validation (bad header, length != dim, target id out
 *      of range, value not representable in the output type, edge to an unknown element); those values are skipped.
 * He values: revisioned SerializedVector {F64,F32,I64,I32,I16}; elem_ids[i] = destination row (NULL: row i).
 * d_out_rows: DEVICE buffer n_rows x dim of out_dtype (SDB_F32 / SDB_F64); d_present (device, nullable) gets 1 per
 * decoded row. */
sdb_status sdb_stage_decode_vectors(sdb_ctx*, const uint8_t* blob, const uint64_t* off, const uint64_t* elem_ids,
                                    uint64_t n, uint32_t dim, sdb_dtype out_dtype, uint64_t n_rows, void* d_out_rows,
                                    uint8_t* d_present, uint64_t* n_bad);
/* Hn values of ONE layer (BE u16 count + BE u64 neighbour ids), node_ids[i] = the key's node id.  Output: CSR over
 * element ids 0..n_elems-1 in stored neighbour order, first occurrence kept (DynamicSet::insert); host arrays owned
 * by the library (sdb_free). */
sdb_status sdb_stage_decode_nodes(sdb_ctx*, const uint8_t* blob, const uint64_t* off, const uint64_t* node_ids,
                                  uint64_t n, uint64_t n_elems, uint64_t** out_row_ptr, uint32_t** out_col_idx,
                                  uint64_t* n_bad);
/* Both of the above fused with sdb_hnsw_load: raw He values + per-layer Hn values in, device-resident index out
 * (no host-side CSR is ever materialised).  entry_point / n_layers come from the Hs state (hnsw/mod.rs:61-72). */
sdb_status sdb_hnsw_load_staged(sdb_ctx*, uint32_t dim, sdb_metric, uint64_t n_elems, const uint8_t* vec_blob,
                                const uint64_t* vec_off, const uint64_t* vec_ids, uint64_t n_vec, uint32_t n_layers,
                                const uint8_t* const* node_blob, const uint64_t* const* node_off,
                                const uint64_t* const* node_ids, const uint64_t* n_nodes, int64_t entry_point,
                                sdb_hnsw** out, uint64_t* n_bad);
/* queries nq x dim f32; out nq x k (element id, f64 distance) ascending; out_counters (nullable)
 * nq x 2 = {distance evaluations, expanded nodes} per query. */
sdb_status sdb_hnsw_search(sdb_hnsw*, const float* queries, uint32_t nq, uint32_t k, uint32_t ef,
                           uint64_t* out_elems, double* out_dist, uint32_t* out_count, uint64_t* out_counters);

/* Index-construction helper (SURVEY 8f-2, "next" row): Heuristic::select, standard variant
 * (idx/trees/hnsw/heuristic.rs:61-81,201-216), applied in parallel to pre-ranked candidate lists.
 * d_vectors: n x dim f32 (device) of the layer's members; d_cand: n x kc candidate member indices, nearest first
 * (e.g. the rows written by sdb_knn_bruteforce_device; the element itself is skipped), d_cand_cnt: valid entries per
 * row.  For every element: if it has <= m_max candidates all are taken, otherwise candidates are visited nearest-first
 * and e is accepted iff no already accepted r is closer to e than the element is (e_dist > dist(e,r) rejects), until
 * m_max are accepted.  presorted = 0: the candidates are first ordered by their distance to the element
 * (build_priority_list, layer.rs:389-405 -- the re-selection of an over-full node).  d_out: n x m_max member indices,
 * d_out_cnt: accepted count.  All pointers are device pointers. */
sdb_status sdb_hnsw_select_neighbors(sdb_ctx*, const float* d_vectors, uint32_t dim, sdb_metric, uint64_t row0, uint64_t n,
                                     const uint64_t* d_cand, const uint32_t* d_cand_cnt, uint32_t kc, uint32_t m_max,
                                     int presorted, uint32_t* d_out, uint32_t* d_out_cnt);

/* the same selection for an explicit list of elements (d_elem_ids[i] = row of element i in d_vectors): the re-selection
 * of over-full neighbours after a batch of insertions (hnsw/layer.rs:362-378) touches scattered elements */
sdb_status sdb_hnsw_select_neighbors_ids(sdb_ctx*, const float* d_vectors, uint32_t dim, sdb_metric,
                                         const uint32_t* d_elem_ids, uint64_t n, const uint64_t* d_cand,
                                         const uint32_t* d_cand_cnt, uint32_t kc, uint32_t m_max, int presorted,
                                         uint32_t* d_out, uint32_t* d_out_cnt);

/* ---- graph expansion: replaces GraphEdgeScan::execute (exec/operators/scan/graph.rs:168-283)
 *      driven by LookupPart (exec/parts/lookup.rs:139-170) and the +collect recursion
 *      (exec/operators/recursion/collect.rs:74-143) -------------------------------------------- */
sdb_status sdb_graph_load_csr(sdb_ctx*, uint64_t n_rows, const uint64_t* row_ptr, const uint32_t* col_idx,
                              sdb_graph** out);
/* Row-sharded adjacency (SURVEY 8e, "one exchange per hop"): this rank holds rows [row_lo, row_hi) of the
 * n_rows_total-row CSR -- row_ptr has row_hi - row_lo + 1 entries rebased to row_ptr[0] = 0, col_idx the matching
 * slice.  sdb_graph_expand / _device / sdb_graph_collect on shard handles are COLLECTIVE over the context's
 * communicator (sdb_comm_init_rank / sdb_ctx_create_multi): every rank passes the same frontier and receives the
 * complete result, identical -- order and duplicates included -- to the unsharded call.  Per hop every rank expands
 * the sources it owns into their positions of the global output (positions = prefix sum of the all-reduced degree
 * array) and one all-reduce assembles the next frontier; +collect de-duplicates the assembled level on every rank.
 * One thread (or process) per rank: the calls synchronise with the host between hops. */
sdb_status sdb_graph_load_csr_shard(sdb_ctx*, uint64_t n_rows_total, uint64_t row_lo, uint64_t row_hi,
                                    const uint64_t* row_ptr, const uint32_t* col_idx, sdb_graph** out);
void sdb_graph_destroy(sdb_graph*);
/* applies hops[0..n_hops) in order to the frontier (multiset semantics: duplicates kept, frontier
 * order preserved, per-source limit honoured; 0 = no limit).  *out_ids is library-owned host
 * memory (free with sdb_free). */
sdb_status sdb_graph_expand(sdb_graph* const* hops, uint32_t n_hops, const uint32_t* frontier, uint64_t n_frontier,
                            uint32_t per_source_limit, uint32_t** out_ids, uint64_t* out_n);
/* device-resident variant: d_frontier and *d_out_ids are device pointers; *d_out_ids is library-owned (sdb_device_free) */
sdb_status sdb_graph_expand_device(sdb_graph* const* hops, uint32_t n_hops, const uint32_t* d_frontier, uint64_t n_frontier,
                                   uint32_t per_source_limit, uint32_t** d_out_ids, uint64_t* out_n);
void sdb_device_free(sdb_ctx*, void* d_ptr);
/* +collect BFS: first-seen dedup, emits from min_depth, start only marked seen when inclusive. */
sdb_status sdb_graph_collect(sdb_graph*, const uint32_t* start, uint64_t n_start, uint32_t min_depth,
                             uint32_t max_depth, int inclusive, uint32_t** out_ids, uint64_t* out_n);
void sdb_free(void*);

#ifdef __cplusplus
}
#endif
#endif
