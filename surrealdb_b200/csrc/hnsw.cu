// hnsw.cu -- K3: HNSW layer walk, one warp per query, strict-parity with the reference's sequential search.
//
// Replaces Hnsw::knn_search (idx/trees/hnsw/mod.rs:459-482): search_ep greedy descent (mod.rs:521-548) and
// HnswLayer::search (hnsw/layer.rs:184-223) with its two DoublePriorityQueues (idx/trees/knn.rs:15-123) and
// visited set.  Parity rules reproduced exactly:
//   * candidates popped nearest-first, FIFO among equal distances; stop when nearest candidate > farthest kept
//   * neighbours visited in STORED order; admitted iff d < f or |w| < ef; w trimmed with pop_last (newest of
//     the farthest); f re-read after every admission
//   * distances are the typed-f32 kernels of idx/trees/vector.rs:221-410: cosine = ndarray 8-lane f32 dot and
//     sums, finished in f64; euclid = sequential f32 sum of squares, f64 sqrt (same op order as the oracle);
//     manhattan / chebyshev / hamming = sequential f32 (integer) folds widened to f64; minkowski = sequential f64
//     sum of |a-b|^p, then ^(1/p).  PEARSON and JACCARD are not served (the index keeps the reference's CPU path).
// Batched candidate expansion: the <=32 neighbours of the popped candidate are de-duplicated against the
// per-query visited table with warp-parallel CAS, their vectors are gathered with coalesced transposed loads
// (one lane per neighbour walks its row in order), and only the admission step is serial.
// Queue trick (result-neutral): once w is full, candidates farther than f can never be expanded (f only
// shrinks), so they are dropped from the candidate array, which bounds it to 2*ef entries.
//
// Algorithmic bytes per query = visited * (4*dim + 4) + expanded * 4*deg, both counters are returned.
#include <algorithm>

#include "exactmath.cuh"
#include "internal.cuh"
#include "rowwalk.cuh"

namespace sdb {

struct Hnsw {
  Ctx* ctx = nullptr;
  uint32_t dim = 0;
  sdb_metric metric = SDB_EUCLIDEAN;
  double minkowski_p = 3.0;  // order of SDB_MINKOWSKI (sdb_hnsw_set_minkowski_order); nothing precomputed depends on it
  uint64_t n = 0;
  uint32_t n_layers = 0;
  int64_t entry = -1;
  float* d_vec = nullptr;
  float* d_sumsq = nullptr;
  double* d_norm = nullptr;  // sqrt((double)sumsq): the per-element factor of the cosine denominator (vector.rs:246)
  std::vector<uint64_t*> rp;
  std::vector<uint32_t*> ci;
  const uint64_t** d_rp = nullptr;
  const uint32_t** d_ci = nullptr;
  uint64_t* d_visited = nullptr;
  uint32_t table_log2 = 0, n_tables = 0;
  uint32_t gen = 1;  // generations consumed so far (each warp uses gen_base + its own counter)
  bool borrowed = false;  // sdb_hnsw_load_device: vectors and CSR arrays belong to the caller
  std::mutex mu;
};

constexpr int HN_WARPS = 4;
constexpr uint64_t KEY_MAX = 0xFFEFFFFFFFFFFFFFull;  // dist_key(f64::MAX)

__device__ __forceinline__ double key_to_double(uint64_t key) {
  const uint64_t b = (key >> 63) ? (key & 0x7fffffffffffffffull) : ~key;
  return __longlong_as_double((long long)b);
}

// ndarray-style 8-lane f32 sum of squares of every row (load time).  8 threads per row, thread j owns the partial sum
// over the columns 8i+j (a sequential chain, as in ndarray's unrolled fold); the 8 threads of a row read one 32-byte
// sector per step.  Also writes sqrt((double)sumsq), the element's factor of the cosine denominator.
__global__ void hnsw_sumsq_kernel(const float* __restrict__ vec, uint32_t dim, uint64_t n, float* __restrict__ out,
                                  double* __restrict__ norm) {
  const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const uint64_t r = t >> 3;
  const uint32_t j = (uint32_t)t & 7u;
  const bool valid = r < n;
  const float* a = vec + (valid ? r : 0) * dim + j;
  const uint32_t steps = dim >> 3;
  float p = 0.f;
  if (valid)
    for (uint32_t i = 0; i < steps; i++) {
      const float v = __ldg(a + 8u * i);
      p = __fadd_rn(p, __fmul_rn(v, v));
    }
  const float sj = __fadd_rn(p, __shfl_down_sync(0xffffffffu, p, 4));
  const float s1 = __shfl_down_sync(0xffffffffu, sj, 1);
  const float s2 = __shfl_down_sync(0xffffffffu, sj, 2);
  const float s3 = __shfl_down_sync(0xffffffffu, sj, 3);
  if (valid && j == 0) {
    float sum = __fadd_rn(0.f, sj);
    sum = __fadd_rn(sum, s1);
    sum = __fadd_rn(sum, s2);
    sum = __fadd_rn(sum, s3);
    const float* row = vec + r * dim;
    for (uint32_t c = dim & ~7u; c < dim; c++) sum = __fadd_rn(sum, __fmul_rn(__ldg(row + c), __ldg(row + c)));
    out[r] = sum;
    if (norm) norm[r] = __dsqrt_rn((double)sum);
  }
}

// The metrics whose F32 form is ONE fold over the columns in column order (idx/trees/vector.rs), as a per-column
// policy: step(x, q) takes column c of the element and of the query, finish() widens / finishes to f64.  Only
// round-to-nearest intrinsics, so nothing is contracted into an FMA (Rust/LLVM does not fuse either).  All four
// metrics are symmetric bit for bit in (x, q), so calculate(element, query) (the walk, hnsw/elements.rs:128-139) and
// calculate(query, vector) (the pending log, hnsw/index.rs:407) give the same value.
template <int METRIC>
struct RowFold;
// EUCLID  l2_dist: sequential f32 sum of (a-b)^2, f64 sqrt
template <>
struct RowFold<SDB_EUCLIDEAN> {
  float s = 0.f;
  __device__ __forceinline__ void step(float x, float q, double) {
    const float d = __fsub_rn(x, q);
    s = __fadd_rn(s, __fmul_rn(d, d));
  }
  __device__ __forceinline__ double finish(double) const { return __dsqrt_rn((double)s); }
};
// MANHATTAN  l1_dist (vector.rs:380): sequential f32 sum of |a-b|, widened.  |.| clears the sign, so a NaN result is
// positive on the reference's x86-64; it is returned as the canonical 0x7FF8... there (the GPU's own NaN bits differ)
template <>
struct RowFold<SDB_MANHATTAN> {
  float s = 0.f;
  __device__ __forceinline__ void step(float x, float q, double) { s = __fadd_rn(s, fabsf(__fsub_rn(x, q))); }
  __device__ __forceinline__ double finish(double) const {
    return s != s ? __longlong_as_double(0x7FF8000000000000ll) : (double)s;
  }
};
// CHEBYSHEV  linf_dist (vector.rs:221-223): max = 0; if diff > max { max = diff } -- a NaN difference is never taken,
// so the fold does not depend on the column order
template <>
struct RowFold<SDB_CHEBYSHEV> {
  float m = 0.f;
  __device__ __forceinline__ void step(float x, float q, double) {
    const float d = fabsf(__fsub_rn(x, q));
    if (d > m) m = d;
  }
  __device__ __forceinline__ double finish(double) const { return (double)m; }
};
// HAMMING  (vector.rs:292-311): count of a != b as FLOAT comparisons (NaN != NaN counts, -0.0 == 0.0 does not)
template <>
struct RowFold<SDB_HAMMING> {
  uint32_t c = 0;
  __device__ __forceinline__ void step(float x, float q, double) { c += x != q ? 1u : 0u; }
  __device__ __forceinline__ double finish(double) const { return (double)c; }
};
// MINKOWSKI(p)  (vector.rs:389-399): s += |(f64)a - (f64)b|^p in sequential f64, then s^(1/p).  pow() is CUDA's libm
// here and the platform libm in the reference: an ulp or two apart per call (DESIGN section 8)
template <>
struct RowFold<SDB_MINKOWSKI> {
  ExactAcc a;
  __device__ __forceinline__ void step(float x, float q, double p) { a.minkowski_step((double)x, (double)q, p); }
  __device__ __forceinline__ double finish(double p) const { return pow(a.acc, __ddiv_rn(1.0, p)); }
};

// Distance::calculate for VectorType::F32 (idx/trees/vector.rs:221-410,659-672), one thread per vector: the typed
// metric of the walk applied to vectors that are NOT part of the graph -- the new_vectors of pending updates that
// HnswIndex::search_pendings ranks by brute force (hnsw/index.rs:398-404).  Same lane structure and the same folds as
// the walk, so a vector gets the same distance whether it is reached through the graph or through the pending log.
// p: the Minkowski order (unused by the other metrics).
template <int METRIC>
__global__ void typed_distance_kernel(const float* __restrict__ q, const float* __restrict__ vecs, uint32_t dim, uint64_t n,
                                      double p, double* __restrict__ out) {
  const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  const float* a = vecs + r * dim;
  if (METRIC == SDB_COSINE) {
    float p[8] = {0, 0, 0, 0, 0, 0, 0, 0}, pa[8] = {0, 0, 0, 0, 0, 0, 0, 0}, pq[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    uint32_t i = 0;
    for (; i + 8 <= dim; i += 8)
#pragma unroll
      for (int j = 0; j < 8; j++) {
        p[j] = __fadd_rn(p[j], __fmul_rn(a[i + j], q[i + j]));
        pa[j] = __fadd_rn(pa[j], __fmul_rn(a[i + j], a[i + j]));
        pq[j] = __fadd_rn(pq[j], __fmul_rn(q[i + j], q[i + j]));
      }
    float dot = 0.f, sa = 0.f, sq = 0.f;
#pragma unroll
    for (int j = 0; j < 4; j++) {
      dot = __fadd_rn(dot, __fadd_rn(p[j], p[j + 4]));
      sa = __fadd_rn(sa, __fadd_rn(pa[j], pa[j + 4]));
      sq = __fadd_rn(sq, __fadd_rn(pq[j], pq[j + 4]));
    }
    for (; i < dim; i++) {
      dot = __fadd_rn(dot, __fmul_rn(a[i], q[i]));
      sa = __fadd_rn(sa, __fmul_rn(a[i], a[i]));
      sq = __fadd_rn(sq, __fmul_rn(q[i], q[i]));
    }
    const double na = __dsqrt_rn((double)sa), nb = __dsqrt_rn((double)sq);
    // calculate(a = search.pt, b = vector): dot and the product of norms are symmetric
    out[r] = __dsub_rn(1.0, __ddiv_rn((double)dot, __dmul_rn(na, nb)));
  } else {
    RowFold<METRIC == SDB_COSINE ? SDB_EUCLIDEAN : METRIC> f;
    for (uint32_t i = 0; i < dim; i++) f.step(a[i], q[i], p);
    out[r] = f.finish(p);
  }
}

// distance of this lane's row (or NO_ROW) to the query held in shared memory; all 32 lanes must call.
// Scratch of the distance phase, per warp.  One lane per row (every metric but cosine): a 32 x 33 float transposing
// tile.  Cosine: 32 compacted row ids + 32 f64 results (the rows are read straight from global memory, see
// warp_distance<SDB_COSINE>).
__host__ __device__ constexpr size_t hn_tile_bytes(bool cosine) { return cosine ? 32 * 4 + 32 * 8 : sizeof(float) * 32 * 33; }

// COSINE.  ndarray's f32 dot (a6; oracle orc_nd_dot_f32) keeps 8 running sums p_j over the columns 8i+j, each one a
// strictly sequential chain over i, and folds them as ((((0+(p0+p4))+(p1+p5))+(p2+p6))+(p3+p7)) followed by the <8
// tail columns.  The 8 chains of a row are independent, so a row is given to 8 LANES (lane j = chain j) and a warp
// works on 4 rows at a time -- two such quads interleaved when more than 4 rows are new, so every lane carries two
// independent chains.  Lane (g, j) reads x[row_g][8i+j] directly from global memory: the 8 lanes of a row cover one 32-byte
// sector and the 4 rows of a quad 4 sectors, i.e. a request moves as many bytes as a fully coalesced one; no shared-memory
// transposition, 8 x fewer dependent steps per row than one lane per row (the walk was bound by issue latency: ncu r1,
// 30 % issue-active at 13 cycles per instruction, ~6.7k instructions per expanded node).
template <int METRIC>
__device__ __forceinline__ double warp_distance(const float* __restrict__ vec, const double* __restrict__ norm,
                                                uint32_t dim, uint32_t my_row, const float* s_q, double q_norm,
                                                float (*tile)[33], double p);

// Cosine keeps the query TRANSPOSED in shared memory: qT[j * qs + i] = q[8i + j] (chain j contiguous), qs = hn_q_stride
// = 4 mod 32 words so the 8 lanes of a row read 8 different bank groups with one LDS.128 per 4 steps; the < 8 tail
// columns follow at qT[8 * qs ...].
__host__ __device__ constexpr uint32_t hn_q_stride(uint32_t dim) { return (((dim >> 3) + 27u) / 32u) * 32u + 4u; }
__host__ __device__ constexpr size_t hn_q_floats(uint32_t dim, bool cosine) {
  return cosine ? (size_t)8 * hn_q_stride(dim) + 8 : (size_t)((dim + 3) & ~3u);
}

template <>
__device__ __forceinline__ double warp_distance<SDB_COSINE>(const float* __restrict__ vec, const double* __restrict__ norm,
                                                            uint32_t dim, uint32_t my_row, const float* s_q, double q_norm,
                                                            float (*tile)[33], double) {
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t d8 = dim & ~7u, steps = dim >> 3, qs = hn_q_stride(dim);
  uint32_t* ids = reinterpret_cast<uint32_t*>(tile);
  double* res = reinterpret_cast<double*>(ids + 32);
  const uint32_t vmask = __ballot_sync(0xffffffffu, my_row != NO_ROW);
  const uint32_t n_rows = __popc(vmask);
  const uint32_t ci = __popc(vmask & ((1u << lane) - 1u));  // compact index of this lane's row
  if (my_row != NO_ROW) ids[ci] = my_row;
  __syncwarp();
  const uint32_t grp = lane >> 3, j = lane & 7u;
  const float* qj = s_q + j * qs;
  const uint32_t row_bytes = dim * 4u;
  for (uint32_t g0 = 0; g0 < n_rows; g0 += 8) {
    const uint32_t ia = g0 + grp, ib = g0 + 4 + grp;
    const bool va = ia < n_rows, vb = ib < n_rows;
    const uint32_t ra = va ? ids[ia] : 0u, rb = vb ? ids[ib] : 0u;
    const float* xa = vec + (size_t)ra * dim + j;
    const float* xb = vec + (size_t)rb * dim + j;
    // ask L2 for every line of the rows of this round up front (lane j: lines j, j+8, ...): the first loads below pay
    // the DRAM latency once, the later ones find their sectors in L2
    if (va)
      for (uint32_t off = j * 128u; off < row_bytes; off += 8u * 128u)
        asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const char*>(xa - j) + off));
    if (vb)
      for (uint32_t off = j * 128u; off < row_bytes; off += 8u * 128u)
        asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const char*>(xb - j) + off));
    double na = 0.0, nb = 0.0;
    if (va && j == 0) na = __ldg(norm + ra);
    if (vb && j == 0) nb = __ldg(norm + rb);
    float pa = 0.f, pb = 0.f;
    uint32_t i = 0;
    if (g0 + 4 < n_rows) {  // (warp-uniform) two quads
      for (; i + 8 <= steps; i += 8) {
        float a[8], b[8];
#pragma unroll
        for (int u = 0; u < 8; u++) {
          a[u] = va ? __ldg(xa + 8u * (i + u)) : 0.f;
          b[u] = vb ? __ldg(xb + 8u * (i + u)) : 0.f;
        }
        const float4 q0 = *reinterpret_cast<const float4*>(qj + i), q1 = *reinterpret_cast<const float4*>(qj + i + 4);
        const float qv[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
#pragma unroll
        for (int u = 0; u < 8; u++) {
          pa = __fadd_rn(pa, __fmul_rn(a[u], qv[u]));
          pb = __fadd_rn(pb, __fmul_rn(b[u], qv[u]));
        }
      }
      for (; i < steps; i++) {
        const float qv = qj[i];
        pa = __fadd_rn(pa, __fmul_rn(va ? __ldg(xa + 8u * i) : 0.f, qv));
        pb = __fadd_rn(pb, __fmul_rn(vb ? __ldg(xb + 8u * i) : 0.f, qv));
      }
    } else {  // one quad: deeper unroll for the same number of loads in flight
      for (; i + 16 <= steps; i += 16) {
        float a[16];
#pragma unroll
        for (int u = 0; u < 16; u++) a[u] = va ? __ldg(xa + 8u * (i + u)) : 0.f;
#pragma unroll
        for (int v4 = 0; v4 < 4; v4++) {
          const float4 q4 = *reinterpret_cast<const float4*>(qj + i + 4 * v4);
          pa = __fadd_rn(pa, __fmul_rn(a[4 * v4 + 0], q4.x));
          pa = __fadd_rn(pa, __fmul_rn(a[4 * v4 + 1], q4.y));
          pa = __fadd_rn(pa, __fmul_rn(a[4 * v4 + 2], q4.z));
          pa = __fadd_rn(pa, __fmul_rn(a[4 * v4 + 3], q4.w));
        }
      }
      for (; i < steps; i++) pa = __fadd_rn(pa, __fmul_rn(va ? __ldg(xa + 8u * i) : 0.f, qj[i]));
    }
    // fold: s_j = p_j + p_(j+4) on lanes j < 4, then the sequential sum on the quad's lane 0
#pragma unroll
    for (int h = 0; h < 2; h++) {
      const float p = h ? pb : pa;
      const float sj = __fadd_rn(p, __shfl_down_sync(0xffffffffu, p, 4));
      const float s1 = __shfl_down_sync(0xffffffffu, sj, 1);
      const float s2 = __shfl_down_sync(0xffffffffu, sj, 2);
      const float s3 = __shfl_down_sync(0xffffffffu, sj, 3);
      const bool v = h ? vb : va;
      if (v && j == 0) {
        const uint32_t row = h ? rb : ra;
        float dot = __fadd_rn(0.f, sj);
        dot = __fadd_rn(dot, s1);
        dot = __fadd_rn(dot, s2);
        dot = __fadd_rn(dot, s3);
        for (uint32_t c = d8; c < dim; c++)
          dot = __fadd_rn(dot, __fmul_rn(__ldg(vec + (size_t)row * dim + c), s_q[8u * qs + (c - d8)]));
        res[h ? ib : ia] = __dsub_rn(1.0, __ddiv_rn((double)dot, __dmul_rn(h ? nb : na, q_norm)));
      }
    }
  }
  __syncwarp();
  return my_row != NO_ROW ? res[ci] : 0.0;
}

// EUCLID, MANHATTAN, CHEBYSHEV, HAMMING, MINKOWSKI.  Each folds its columns strictly sequentially (RowFold<METRIC>):
// one chain per row, so a row stays on ONE lane and the rows of a round are transposed through shared memory
// (coalesced fetches, 64 columns a step).  p: the Minkowski order.
template <int METRIC>
__device__ __forceinline__ double warp_distance(const float* __restrict__ vec, const double* __restrict__ norm,
                                                uint32_t dim, uint32_t my_row, const float* s_q, double q_norm,
                                                float (*tile)[33], double p) {
  const uint32_t lane = threadIdx.x & 31u;
  RowFold<METRIC> f;
  // Only a handful of the <=32 neighbours of an expanded node are new (6 on average): the valid rows are compacted and
  // handled in rounds of 16; the 32 x 33 float scratch is viewed as 16 rows x (64 columns + 2 padding words), so one
  // step moves 64 columns of every row of the round -- up to 32 independent loads per lane in flight per wait instead
  // of 4.  The padding words park the compacted row ids.
  float(*t)[66] = reinterpret_cast<float(*)[66]>(tile);
  const uint32_t vmask = __ballot_sync(0xffffffffu, my_row != NO_ROW);
  const uint32_t n_rows = __popc(vmask);
  const uint32_t ci = __popc(vmask & ((1u << lane) - 1u));  // compact index of this lane's row
  if (my_row != NO_ROW) t[ci & 15u][64 + (ci >> 4)] = __uint_as_float(my_row);
  __syncwarp();
  {
    const uint32_t row_bytes = dim * 4u;
    for (uint32_t r = 0; r < n_rows; r++) {
      const char* base = reinterpret_cast<const char*>(vec + (size_t)__float_as_uint(t[r & 15u][64 + (r >> 4)]) * dim);
      for (uint32_t off = lane * 128u; off < row_bytes; off += 32u * 128u)
        asm volatile("prefetch.global.L2 [%0];" ::"l"(base + off));
    }
  }
  for (uint32_t g0 = 0; g0 < n_rows; g0 += 16) {
    const uint32_t nr = n_rows - g0 < 16u ? n_rows - g0 : 16u;
    const bool mine = my_row != NO_ROW && (ci >> 4) == (g0 >> 4);
    const float* x = t[ci & 15u];
    for (uint32_t c0 = 0; c0 < dim; c0 += 64) {
      const bool in0 = c0 + lane < dim, in1 = c0 + 32 + lane < dim;
#pragma unroll 4
      for (uint32_t r = 0; r < nr; r++) {
        const float* src = vec + (size_t)__float_as_uint(t[r][64 + (g0 >> 4)]) * dim + c0 + lane;  // broadcast id read
        const float v0 = in0 ? __ldg(src) : 0.f;
        const float v1 = in1 ? __ldg(src + 32) : 0.f;
        t[r][lane] = v0;
        t[r][lane + 32] = v1;
      }
      __syncwarp();
      if (mine) {
        const uint32_t lim = dim - c0 < 64u ? dim - c0 : 64u;
        for (uint32_t jj = 0; jj < lim; jj++) f.step(x[jj], s_q[c0 + jj], p);
      }
      __syncwarp();
    }
  }
  if (my_row == NO_ROW) return 0.0;
  return f.finish(p);
}

// sorted (ascending key, FIFO inside a key) array insert by the whole warp; entries live in [head, n).  One pass from
// the top: every 32-entry chunk above the insertion point moves up by one; the chunk that holds an entry <= key fixes the
// position (the new entry goes AFTER its equals).
__device__ __forceinline__ uint32_t sorted_insert(uint64_t* keys, uint32_t* ids, uint32_t head, uint32_t n, uint64_t key,
                                                  uint32_t id) {
  const uint32_t lane = threadIdx.x & 31u;
  uint32_t pos = head;
  for (uint32_t hi = n; hi > head;) {
    const uint32_t lo = hi - head > 32u ? hi - 32u : head;
    const uint32_t i = lo + lane;
    uint64_t k = 0;
    uint32_t v = 0;
    const bool in = i < hi;
    if (in) {
      k = keys[i];
      v = ids[i];
    }
    const uint32_t le = __ballot_sync(0xffffffffu, in && k <= key);
    __syncwarp();  // every lane has read its entry before a neighbour overwrites it
    if (in && k > key) {
      keys[i + 1] = k;
      ids[i + 1] = v;
    }
    __syncwarp();
    if (le) {
      pos = lo + __popc(le);
      break;
    }
    hi = lo;
  }
  if (lane == 0) {
    keys[pos] = key;
    ids[pos] = id;
  }
  __syncwarp();
  return n + 1;
}

struct HnswParams {
  const float* vec;
  const double* norm;     // sqrt((double)sumsq) per element (cosine)
  const uint64_t* const* rp;
  const uint32_t* const* ci;
  uint32_t dim, n_layers;
  int64_t entry;
  const float* queries;
  uint32_t nq, k, ef;
  uint32_t ccap;          // capacity of the candidate window (entries)
  const uint8_t* truthy;  // non-null: knn_search_with_filter -- one byte per element (layer 0 only)
  const uint8_t* noexp;   // non-null: pending docs -- noexp[e] != 0: every document of element e has a pending update;
                          // the element still enters w but is never expanded (layer.rs:209, every layer)
  uint64_t* visited;
  uint32_t table_log2;
  uint32_t gen_base, gens_per_warp;
  uint64_t* out_elems;
  double* out_dist;
  uint32_t* out_count;
  uint64_t* out_counters;
  uint32_t* overflow;
  const int* cancel;  // mapped host flag (sdb_ctx_cancel): polled before every query
  double minkowski_p;  // order of SDB_MINKOWSKI
};

template <int METRIC, int MINB>
__global__ void __launch_bounds__(HN_WARPS * 32, MINB) hnsw_search_kernel(HnswParams P) {
  constexpr bool COSINE = METRIC == SDB_COSINE;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t ccap = P.ccap, wcap = P.ef + 2;
  // per-warp shared layout
  const size_t per_warp = sizeof(float) * hn_q_floats(P.dim, COSINE) + hn_tile_bytes(COSINE) + (sizeof(uint64_t) + sizeof(uint32_t)) * (ccap + wcap) + 64;
  uint8_t* base = smem_raw + (size_t)warp * ((per_warp + 15) & ~size_t(15));
  // query first (16-byte aligned: LDS.128), then the distance scratch, the 8-byte keys, the 4-byte ids
  float* s_q = reinterpret_cast<float*>(base);
  float(*tile)[33] = reinterpret_cast<float(*)[33]>(s_q + ((hn_q_floats(P.dim, COSINE) + 3) & ~size_t(3)));
  uint64_t* c_key = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(tile) + hn_tile_bytes(COSINE));
  uint64_t* w_key = c_key + ccap;
  uint32_t* c_id = reinterpret_cast<uint32_t*>(w_key + wcap);
  uint32_t* w_id = c_id + ccap;

  const uint32_t gwarp = blockIdx.x * HN_WARPS + warp;
  const uint32_t n_warps = gridDim.x * HN_WARPS;
  uint64_t* table = P.visited + ((size_t)gwarp << P.table_log2);
  const uint32_t mask = (1u << P.table_log2) - 1u;
  uint32_t gen = P.gen_base + gwarp * P.gens_per_warp;

  for (uint32_t q = gwarp; q < P.nq; q += n_warps) {
    if (*reinterpret_cast<const volatile int*>(P.cancel)) break;  // uniform per warp: every lane reads the same word
    // stage the query (cosine: transposed, see hn_q_stride) and its 8-lane sum of squares
    double q_norm = 0.0;
    if (COSINE) {
      const uint32_t qs = hn_q_stride(P.dim), d8 = P.dim & ~7u, steps = P.dim >> 3;
      const float* qg = P.queries + (size_t)q * P.dim;
      for (uint32_t c = lane; c < P.dim; c += 32) {
        const float v = qg[c];
        if (c < d8) s_q[(c & 7u) * qs + (c >> 3)] = v;
        else s_q[8u * qs + (c - d8)] = v;
      }
      __syncwarp();
      float p = 0.f;
      if (lane < 8)
        for (uint32_t i = 0; i < steps; i++) {
          const float v = s_q[lane * qs + i];
          p = __fadd_rn(p, __fmul_rn(v, v));
        }
      const float sj = __fadd_rn(p, __shfl_down_sync(0xffffffffu, p, 4));
      const float s1 = __shfl_down_sync(0xffffffffu, sj, 1);
      const float s2 = __shfl_down_sync(0xffffffffu, sj, 2);
      const float s3 = __shfl_down_sync(0xffffffffu, sj, 3);
      float q_sumsq = __fadd_rn(0.f, sj);
      q_sumsq = __fadd_rn(q_sumsq, s1);
      q_sumsq = __fadd_rn(q_sumsq, s2);
      q_sumsq = __fadd_rn(q_sumsq, s3);
      for (uint32_t c = d8; c < P.dim; c++) {
        const float v = s_q[8u * qs + (c - d8)];
        q_sumsq = __fadd_rn(q_sumsq, __fmul_rn(v, v));
      }
      q_norm = __dsqrt_rn((double)__shfl_sync(0xffffffffu, q_sumsq, 0));
    } else {
      for (uint32_t c = lane; c < P.dim; c += 32) s_q[c] = P.queries[(size_t)q * P.dim + c];
      __syncwarp();
    }
    uint64_t n_visited = 0, n_expanded = 0;
    uint32_t n_out = 0;
    if (P.entry >= 0) {
      uint32_t ep = (uint32_t)P.entry;
      double ep_d = warp_distance<METRIC>(P.vec, P.norm, P.dim, lane == 0 ? ep : NO_ROW, s_q, q_norm, tile, P.minkowski_p);
      ep_d = __shfl_sync(0xffffffffu, ep_d, 0);
      n_visited++;
      for (int32_t layer = (int32_t)P.n_layers - 1; layer >= 0; layer--) {
        const uint32_t ef = layer == 0 ? P.ef : 1u;
        const uint64_t* rp = P.rp[layer];
        const uint32_t* ci = P.ci[layer];
        gen++;
        // search_single: visited = {ep}; candidates = w = {(ep_d, ep)}        layer.rs:76-90
        uint32_t head = 0, cn = 0, wn = 0;
        {
          const uint64_t my = ((uint64_t)gen << 32) | ep;
          if (lane == 0) {
            uint32_t slot = (ep * 2654435761u) & mask;
            while ((table[slot] >> 32) == gen) slot = (slot + 1) & mask;
            table[slot] = my;
          }
          __syncwarp();
        }
        // search_single_with_filter (layer.rs:111-149): w starts with ep only if one of its documents is truthy
        const uint8_t* truthy = layer == 0 ? P.truthy : nullptr;
        cn = sorted_insert(c_key, c_id, head, cn, dist_key(ep_d), ep);
        double fd = 1.7976931348623157e308;  // w.peek_last_dist().unwrap_or(f64::MAX)
        if (!truthy || truthy[ep]) {
          wn = sorted_insert(w_key, w_id, 0, wn, dist_key(ep_d), ep);
          fd = ep_d;
        }
        while (head < cn) {
          const uint64_t ckey = c_key[head];
          const uint32_t cid = c_id[head];
          head++;
          if (key_to_double(ckey) > fd) break;  // cq_dist > fq_dist
          n_expanded++;
          const uint64_t beg = rp[cid], end = rp[cid + 1];
          for (uint64_t b0 = beg; b0 < end; b0 += 32) {
            const uint32_t nb = b0 + lane < end ? __ldg(ci + b0 + lane) : NO_ROW;
            bool is_new = false;
            if (nb != NO_ROW) {  // visited.insert(e_id)
              const uint64_t my = ((uint64_t)gen << 32) | nb;
              uint32_t slot = (nb * 2654435761u) & mask;
              for (uint32_t probes = 0;; probes++) {
                const uint64_t cur = *reinterpret_cast<volatile uint64_t*>(table + slot);
                if (cur == my) break;
                if ((uint32_t)(cur >> 32) != gen) {
                  const uint64_t old = atomicCAS(reinterpret_cast<unsigned long long*>(table + slot),
                                                 (unsigned long long)cur, (unsigned long long)my);
                  if (old == cur) {
                    is_new = true;
                    break;
                  }
                  if (old == my) break;
                  if ((uint32_t)(old >> 32) != gen) continue;
                }
                if (probes > mask) {  // table full: report, treat as visited
                  *P.overflow = 1;
                  break;
                }
                slot = (slot + 1) & mask;
              }
            }
            const uint32_t new_mask = __ballot_sync(0xffffffffu, is_new);
            if (!new_mask) continue;
            n_visited += __popc(new_mask);
            const double d = warp_distance<METRIC>(P.vec, P.norm, P.dim, is_new ? nb : NO_ROW, s_q, q_norm, tile, P.minkowski_p);
            // admission in stored order                                     layer.rs:205-217
            uint32_t m = new_mask;
            while (m) {
              const int i = __ffs(m) - 1;
              m &= m - 1;
              const double di = __shfl_sync(0xffffffffu, d, i);
              const uint32_t idi = __shfl_sync(0xffffffffu, nb, i);
              if (di < fd || wn < ef) {
                const uint64_t key = dist_key(di);
                if (cn >= ccap) {  // slide the live window down (or, if truly full, drop the farthest tie)
                  if (head > 0) {
                    for (uint32_t lo = head; lo < cn; lo += 32) {
                      const uint32_t j = lo + lane;
                      uint64_t kk = 0;
                      uint32_t vv = 0;
                      if (j < cn) { kk = c_key[j]; vv = c_id[j]; }
                      __syncwarp();
                      if (j < cn) { c_key[j - head] = kk; c_id[j - head] = vv; }
                      __syncwarp();
                    }
                    cn -= head;
                    head = 0;
                  }
                  if (cn >= ccap) {
                    cn = ccap - 1;
                    *P.overflow = 2;
                  }
                }
                if (!P.noexp || !P.noexp[idi]) cn = sorted_insert(c_key, c_id, head, cn, key, idi);
                if (!truthy || truthy[idi]) {  // add_if_truthy  layer.rs:277-306
                  wn = sorted_insert(w_key, w_id, 0, wn, key, idi);
                  if (wn > ef) wn--;  // pop_last
                  fd = key_to_double(w_key[wn - 1]);
                }
                if (wn == ef) {  // candidates beyond f can never be expanded any more
                  const uint64_t fkey = w_key[wn - 1];
                  while (cn > head && c_key[cn - 1] > fkey) cn--;
                }
              }
            }
          }
        }
        // next layer starts from w.peek_first()                                mod.rs:530-538
        if (wn) {
          ep = w_id[0];
          ep_d = key_to_double(w_key[0]);
        }
        if (layer == 0) {
          n_out = wn < P.k ? wn : P.k;  // to_vec_limit(k)
          for (uint32_t i = lane; i < n_out; i += 32) {
            P.out_elems[(size_t)q * P.k + i] = w_id[i];
            P.out_dist[(size_t)q * P.k + i] = key_to_double(w_key[i]);
          }
        }
        __syncwarp();
      }
    }
    if (lane == 0) {
      P.out_count[q] = n_out;
      if (P.out_counters) {
        P.out_counters[2 * (size_t)q] = n_visited;
        P.out_counters[2 * (size_t)q + 1] = n_expanded;
      }
    }
  }
}

// ---- construction helper: Heuristic::select over pre-ranked candidates, one warp per element ------------------------
template <bool COSINE>
__device__ __forceinline__ float warp_pair_dist(const float* a_smem, float a_n2, const float* __restrict__ b, uint32_t dim) {
  const uint32_t lane = threadIdx.x & 31u;
  float dot = 0.f, n2 = 0.f;
  for (uint32_t c = lane; c < dim; c += 32) {
    const float x = a_smem[c], y = __ldg(b + c);
    if (COSINE) {
      dot = fmaf(x, y, dot);
      n2 = fmaf(y, y, n2);
    } else {
      const float d = x - y;
      dot = fmaf(d, d, dot);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    dot += __shfl_xor_sync(0xffffffffu, dot, o);
    if (COSINE) n2 += __shfl_xor_sync(0xffffffffu, n2, o);
  }
  return COSINE ? 1.f - dot * rsqrtf(a_n2 * n2) : dot;  // euclid: squared distance (same ordering)
}

template <bool COSINE>
__global__ void __launch_bounds__(128) hnsw_select_kernel(const float* __restrict__ vec, uint32_t dim, uint64_t row0, uint64_t n,
                                                          const uint32_t* __restrict__ elem_ids,
                                                          const uint64_t* __restrict__ cand, const uint32_t* __restrict__ cand_cnt,
                                                          uint32_t kc, uint32_t m_max, int presorted, uint32_t* __restrict__ out,
                                                          uint32_t* __restrict__ out_cnt) {
  extern __shared__ float s_sel[];
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* s_q = s_sel + (size_t)warp * (2 * dim + 2 * kc);
  float* s_e = s_q + dim;
  float* s_d = s_e + dim;                                   // [kc] distances (unsorted mode)
  uint32_t* s_ord = reinterpret_cast<uint32_t*>(s_d + kc);  // [kc] visiting order
  const uint64_t i = (uint64_t)blockIdx.x * 4 + warp;  // element index inside this batch
  if (i >= n) return;
  const uint64_t self = elem_ids ? (uint64_t)elem_ids[i] : row0 + i;
  const float* q = vec + self * dim;
  float qn2 = 0.f;
  for (uint32_t c = lane; c < dim; c += 32) {
    const float x = __ldg(q + c);
    s_q[c] = x;
    qn2 = fmaf(x, x, qn2);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) qn2 += __shfl_xor_sync(0xffffffffu, qn2, o);
  __syncwarp();
  const uint64_t* cl = cand + i * kc;
  uint32_t nc = cand_cnt[i] < kc ? cand_cnt[i] : kc;
  uint32_t n_real = 0;  // candidates other than the element itself
  for (uint32_t j = 0; j < nc; j++) n_real += cl[j] != self;
  // visiting order: as given (nearest first) or by computed distance (build_priority_list, layer.rs:389-405)
  if (presorted) {
    for (uint32_t j = lane; j < nc; j += 32) s_ord[j] = j;
  } else {
    for (uint32_t j = 0; j < nc; j++) {
      const float d = cl[j] == self ? 3.0e38f : warp_pair_dist<COSINE>(s_q, qn2, vec + cl[j] * dim, dim);
      if (lane == 0) s_d[j] = d;
    }
    __syncwarp();
    for (uint32_t j = lane; j < nc; j += 32) {
      const float dj = s_d[j];
      uint32_t rank = 0;
      for (uint32_t t = 0; t < nc; t++) rank += (s_d[t] < dj) || (s_d[t] == dj && t < j);
      s_ord[rank] = j;
    }
  }
  __syncwarp();
  uint32_t* o = out + i * m_max;
  uint32_t acc = 0;
  const bool take_all = n_real <= m_max;
  for (uint32_t jj = 0; jj < nc && acc < m_max; jj++) {
    const uint32_t j = s_ord[jj];
    const uint64_t e = cl[j];
    if (e == self) continue;
    bool ok = true;
    if (!take_all) {
      const float* ev = vec + e * dim;
      float en2 = 0.f;
      for (uint32_t c = lane; c < dim; c += 32) {
        const float x = __ldg(ev + c);
        s_e[c] = x;
        en2 = fmaf(x, x, en2);
      }
#pragma unroll
      for (int o2 = 16; o2 > 0; o2 >>= 1) en2 += __shfl_xor_sync(0xffffffffu, en2, o2);
      __syncwarp();
      const float e_dist = warp_pair_dist<COSINE>(s_q, qn2, ev, dim);
      for (uint32_t r = 0; r < acc && ok; r++) {
        const float r_dist = warp_pair_dist<COSINE>(s_e, en2, vec + (uint64_t)o[r] * dim, dim);
        if (e_dist > r_dist) ok = false;  // is_closer: heuristic.rs:209-211
      }
      __syncwarp();
    }
    if (ok) {
      if (lane == 0) o[acc] = (uint32_t)e;
      acc++;
      __syncwarp();
    }
  }
  if (lane == 0) out_cnt[i] = acc;
}

// ---- load-time validation (ADVICE r1): adjacency supplied across the ABI is used for device indexing, so it is
// range-checked once here instead of trusted.  bad[0] counts row_ptr violations (non-monotone / beyond the edge count),
// bad[1] counts neighbour ids >= n_elems.
__global__ void csr_validate_kernel(const uint64_t* __restrict__ rp, const uint32_t* __restrict__ ci, uint64_t n_rows,
                                    uint64_t n_edges, uint64_t id_limit, unsigned long long* __restrict__ bad) {
  const uint64_t step = (uint64_t)gridDim.x * blockDim.x;
  const uint64_t t0 = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  for (uint64_t r = t0; r < n_rows; r += step)
    if (rp[r] > rp[r + 1] || rp[r + 1] > n_edges) atomicAdd(bad, 1ull);
  if (t0 == 0 && n_rows && rp[0] != 0) atomicAdd(bad, 1ull);
  for (uint64_t e = t0; e < n_edges; e += step)
    if ((uint64_t)ci[e] >= id_limit) atomicAdd(bad + 1, 1ull);
}

sdb_status csr_check(Ctx* ctx, const uint64_t* d_rp, const uint32_t* d_ci, uint64_t n_rows, uint64_t n_edges,
                     uint64_t id_limit, unsigned long long counts[2], const char* what, cudaStream_t st) {
  unsigned long long* d_bad = nullptr;
  SDB_CUDA(cudaMallocAsync(&d_bad, 16, st));
  cudaMemsetAsync(d_bad, 0, 16, st);
  const uint64_t work = n_rows > n_edges ? n_rows : n_edges;
  const unsigned grid = (unsigned)std::min<uint64_t>((work + 255) / 256 + 1, (uint64_t)ctx->sm_count * 16);
  csr_validate_kernel<<<grid, 256, 0, st>>>(d_rp, d_ci, n_rows, n_edges, id_limit, d_bad);
  count_launch(ctx);
  unsigned long long h_bad[2] = {0, 0};
  cudaError_t e = cudaMemcpyAsync(h_bad, d_bad, 16, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  cudaFreeAsync(d_bad, st);
  if (e != cudaSuccess) {
    set_error("%s: validation failed to run: %s", what, cudaGetErrorString(e));
    return SDB_ECUDA;
  }
  counts[0] = h_bad[0];
  counts[1] = h_bad[1];
  return SDB_OK;
}
sdb_status csr_validate(Ctx* ctx, const uint64_t* d_rp, const uint32_t* d_ci, uint64_t n_rows, uint64_t n_edges,
                        uint64_t id_limit, const char* what, cudaStream_t st) {
  unsigned long long h_bad[2] = {0, 0};
  SDB_TRY(csr_check(ctx, d_rp, d_ci, n_rows, n_edges, id_limit, h_bad, what, st));
  if (h_bad[0] || h_bad[1]) {
    set_error("%s: malformed CSR (%llu row_ptr violations, %llu neighbour ids out of range)", what, h_bad[0], h_bad[1]);
    return SDB_EINVAL;
  }
  return SDB_OK;
}

// ---- edges to elements without a vector: the reference marks such a neighbour visited and computes nothing
// (elements.get_vector -> None, hnsw/layer.rs:204), which is equivalent to the edge not being there.  Staged loads
// therefore drop them from the device CSR: count, scan, fill.
__global__ void csr_present_degree_kernel(const uint64_t* __restrict__ rp, const uint32_t* __restrict__ ci,
                                          const uint8_t* __restrict__ present, uint64_t n_rows,
                                          uint64_t* __restrict__ deg) {
  const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r > n_rows) return;
  uint64_t d = 0;
  if (r < n_rows && present[r])  // an absent element is never expanded either
    for (uint64_t e = rp[r]; e < rp[r + 1]; e++) d += present[ci[e]] ? 1 : 0;
  deg[r] = d;  // deg[n_rows] = 0: the scan's total
}
__global__ void csr_present_fill_kernel(const uint64_t* __restrict__ rp, const uint32_t* __restrict__ ci,
                                        const uint8_t* __restrict__ present, uint64_t n_rows,
                                        const uint64_t* __restrict__ rp2, uint32_t* __restrict__ ci2) {
  const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_rows || !present[r]) return;
  uint64_t o = rp2[r];
  for (uint64_t e = rp[r]; e < rp[r + 1]; e++) {
    const uint32_t v = ci[e];
    if (present[v]) ci2[o++] = v;  // stored order kept
  }
}

}  // namespace sdb

struct sdb_hnsw : sdb::Hnsw {};
using namespace sdb;

extern "C" void sdb_hnsw_destroy(sdb_hnsw* h);

// the metrics the walk serves (F32 typed arithmetic): COSINE (8 lanes per row), EUCLIDEAN, MANHATTAN, CHEBYSHEV, HAMMING
// and MINKOWSKI (one lane per row).  PEARSON and JACCARD are similarities used as distances; the reference's own HNSW
// tests leave them disabled (idx/trees/hnsw/mod.rs:752-791) and Jaccard's F32 form is asymmetric in its arguments, so
// indexes declared with them keep the reference's CPU path.
static sdb_status hnsw_check_metric(sdb_metric metric, const char* what) {
  switch (metric) {
    case SDB_COSINE:
    case SDB_EUCLIDEAN:
    case SDB_MANHATTAN:
    case SDB_CHEBYSHEV:
    case SDB_HAMMING:
    case SDB_MINKOWSKI:
      return SDB_OK;
    case SDB_PEARSON:
    case SDB_JACCARD:
      set_error("%s: %s is a similarity used as a distance and is not implemented on the GPU walk (the index keeps the "
                "reference's CPU path)", what, metric == SDB_PEARSON ? "PEARSON" : "JACCARD");
      return SDB_EUNSUPPORTED;
    default:
      set_error("%s: metric %d not implemented on the GPU path", what, (int)metric);
      return SDB_EUNSUPPORTED;
  }
}

// common tail of the loaders: per-layer pointer tables + cached |x|^2 (cosine / euclid only: the other metrics need no
// per-element precomputation)
static sdb_status hnsw_finish(sdb_hnsw* h, sdb_hnsw** out) {
  Ctx* ctx = h->ctx;
  cudaStream_t st = ctx->stream;
  auto fail = [&](const char* what, sdb_status rc) {
    set_error("hnsw load: %s failed: %s", what, cudaGetErrorString(cudaGetLastError()));
    sdb_hnsw_destroy(h);
    return rc;
  };
  const uint32_t n_layers = h->n_layers;
  if (cudaMalloc(&h->d_rp, sizeof(void*) * n_layers) != cudaSuccess) return fail("layer table", SDB_ENOMEM);
  if (cudaMalloc(&h->d_ci, sizeof(void*) * n_layers) != cudaSuccess) return fail("layer table", SDB_ENOMEM);
  if (cudaMemcpyAsync(h->d_rp, h->rp.data(), sizeof(void*) * n_layers, cudaMemcpyHostToDevice, st) != cudaSuccess ||
      cudaMemcpyAsync(h->d_ci, h->ci.data(), sizeof(void*) * n_layers, cudaMemcpyHostToDevice, st) != cudaSuccess)
    return fail("layer table copy", SDB_ECUDA);
  if (h->n && (h->metric == SDB_COSINE || h->metric == SDB_EUCLIDEAN)) {
    if (cudaMalloc(&h->d_norm, sizeof(double) * h->n) != cudaSuccess) return fail("norms", SDB_ENOMEM);
    hnsw_sumsq_kernel<<<(unsigned)((h->n * 8 + 127) / 128), 128, 0, st>>>(h->d_vec, h->dim, h->n, h->d_sumsq, h->d_norm);
    count_launch(ctx);
  }
  if (cudaStreamSynchronize(st) != cudaSuccess || cudaGetLastError() != cudaSuccess) return fail("finish", SDB_ECUDA);
  *out = h;
  return SDB_OK;
}

extern "C" {

void sdb_hnsw_destroy(sdb_hnsw* h) {
  if (!h) return;
  cudaSetDevice(h->ctx->device);
  if (!h->borrowed) {
    cudaFree(h->d_vec);
    for (auto p : h->rp) cudaFree(p);
    for (auto p : h->ci) cudaFree(p);
  }
  cudaFree(h->d_sumsq);
  cudaFree(h->d_norm);
  cudaFree(h->d_rp);
  cudaFree(h->d_ci);
  cudaFree(h->d_visited);
  delete h;
}

sdb_status sdb_hnsw_load(sdb_ctx* ctx, uint32_t dim, sdb_metric metric, uint64_t n_elems, const float* vectors,
                         uint32_t n_layers, const uint64_t* const* row_ptr, const uint32_t* const* col_idx,
                         int64_t entry_point, sdb_hnsw** out) {
  if (!ctx || !out || dim == 0 || dim > 65535 || n_elems >= 0xFFFFFFF0ull || (n_elems && !vectors) || !n_layers ||
      !row_ptr || !col_idx || entry_point >= (int64_t)n_elems)
    return SDB_EINVAL;
  {
    const sdb_status mrc = hnsw_check_metric(metric, "sdb_hnsw_load");
    if (mrc != SDB_OK) return mrc;
  }
  *out = nullptr;
  std::lock_guard<std::mutex> guard(ctx->mu);
  SDB_CUDA(cudaSetDevice(ctx->device));
  sdb_hnsw* h = new sdb_hnsw();
  h->ctx = ctx;
  h->dim = dim;
  h->metric = metric;
  h->n = n_elems;
  h->n_layers = n_layers;
  h->entry = entry_point;
  cudaStream_t st = ctx->stream;
  auto fail = [&](const char* what) {
    set_error("hnsw load: %s failed: %s", what, cudaGetErrorString(cudaGetLastError()));
    sdb_hnsw_destroy(h);
    return SDB_ENOMEM;
  };
  const uint64_t nn = n_elems ? n_elems : 1;
  if (cudaMalloc(&h->d_vec, sizeof(float) * nn * dim) != cudaSuccess) return fail("vectors");
  if (cudaMalloc(&h->d_sumsq, sizeof(float) * nn) != cudaSuccess) return fail("sumsq");
  if (n_elems) SDB_CUDA(cudaMemcpyAsync(h->d_vec, vectors, sizeof(float) * n_elems * dim, cudaMemcpyHostToDevice, st));
  for (uint32_t l = 0; l < n_layers; l++) {
    const uint64_t e = n_elems ? row_ptr[l][n_elems] : 0;
    uint64_t* drp = nullptr;
    uint32_t* dci = nullptr;
    if (cudaMalloc(&drp, sizeof(uint64_t) * (n_elems + 1)) != cudaSuccess) return fail("row_ptr");
    h->rp.push_back(drp);
    if (cudaMalloc(&dci, sizeof(uint32_t) * (e ? e : 1)) != cudaSuccess) return fail("col_idx");
    h->ci.push_back(dci);
    SDB_CUDA(cudaMemcpyAsync(drp, row_ptr[l], sizeof(uint64_t) * (n_elems + 1), cudaMemcpyHostToDevice, st));
    if (e) SDB_CUDA(cudaMemcpyAsync(dci, col_idx[l], sizeof(uint32_t) * e, cudaMemcpyHostToDevice, st));
    const sdb_status vrc = csr_validate(ctx, drp, dci, n_elems, e, n_elems, "sdb_hnsw_load", st);
    if (vrc != SDB_OK) {
      sdb_hnsw_destroy(h);
      return vrc;
    }
  }
  return hnsw_finish(h, out);
}

sdb_status sdb_hnsw_load_device(sdb_ctx* ctx, uint32_t dim, sdb_metric metric, uint64_t n_elems, const float* d_vectors,
                                uint32_t n_layers, const uint64_t* const* d_row_ptr, const uint32_t* const* d_col_idx,
                                int64_t entry_point, sdb_hnsw** out) {
  if (!ctx || !out || dim == 0 || dim > 65535 || n_elems >= 0xFFFFFFF0ull || (n_elems && !d_vectors) || !n_layers ||
      !d_row_ptr || !d_col_idx || entry_point >= (int64_t)n_elems)
    return SDB_EINVAL;
  {
    const sdb_status mrc = hnsw_check_metric(metric, "sdb_hnsw_load_device");
    if (mrc != SDB_OK) return mrc;
  }
  *out = nullptr;
  std::lock_guard<std::mutex> guard(ctx->mu);
  SDB_CUDA(cudaSetDevice(ctx->device));
  sdb_hnsw* h = new sdb_hnsw();
  h->ctx = ctx;
  h->dim = dim;
  h->metric = metric;
  h->n = n_elems;
  h->n_layers = n_layers;
  h->entry = entry_point;
  h->borrowed = true;  // nothing is copied: the caller keeps vectors and adjacency alive while the handle exists
  h->d_vec = const_cast<float*>(d_vectors);
  for (uint32_t l = 0; l < n_layers; l++) {
    h->rp.push_back(const_cast<uint64_t*>(d_row_ptr[l]));
    h->ci.push_back(const_cast<uint32_t*>(d_col_idx[l]));
  }
  if (cudaMalloc(&h->d_sumsq, sizeof(float) * (n_elems ? n_elems : 1)) != cudaSuccess) {
    set_error("hnsw load: sumsq allocation failed: %s", cudaGetErrorString(cudaGetLastError()));
    sdb_hnsw_destroy(h);
    return SDB_ENOMEM;
  }
  return hnsw_finish(h, out);
}

sdb_status sdb_hnsw_load_staged(sdb_ctx* ctx, uint32_t dim, sdb_metric metric, uint64_t n_elems,
                                const uint8_t* vec_blob, const uint64_t* vec_off, const uint64_t* vec_ids, uint64_t n_vec,
                                uint32_t n_layers, const uint8_t* const* node_blob, const uint64_t* const* node_off,
                                const uint64_t* const* node_ids, const uint64_t* n_nodes, int64_t entry_point,
                                sdb_hnsw** out, uint64_t* n_bad) {
  if (!ctx || !out || dim == 0 || dim > 65535 || n_elems >= 0xFFFFFFF0ull || !n_layers || !node_blob || !node_off ||
      !node_ids || !n_nodes || entry_point >= (int64_t)n_elems || (n_vec && (!vec_blob || !vec_off)))
    return SDB_EINVAL;
  {
    const sdb_status mrc = hnsw_check_metric(metric, "sdb_hnsw_load_staged");
    if (mrc != SDB_OK) return mrc;
  }
  *out = nullptr;
  // The walk kernels implement the reference's typed metrics for VectorType::F32 only (idx/trees/vector.rs:243-289
  // computes F64 / I64 / I32 / I16 vectors in their own arithmetic).  A value of another SerializedVector variant
  // would load -- the decoder converts it -- but be searched with the wrong arithmetic, so the load refuses it instead
  // of reporting success (ADVICE r1).  Header = revision varint (1) + variant varint: one byte each.
  for (uint64_t v = 0; v < n_vec; v++) {
    const uint64_t a = vec_off[v], b = vec_off[v + 1];
    if (b >= a + 2 && vec_blob[a] == 1 && vec_blob[a + 1] != 1 && vec_blob[a + 1] <= 4) {
      static const char* names[] = {"F64", "F32", "I64", "I32", "I16"};
      set_error("sdb_hnsw_load_staged: He value %llu holds a %s vector; the GPU walk implements the F32 typed metrics only "
                "(the index keeps the reference's CPU path)", (unsigned long long)v, names[vec_blob[a + 1]]);
      return SDB_EUNSUPPORTED;
    }
  }
  std::lock_guard<std::mutex> guard(ctx->mu);
  SDB_CUDA(cudaSetDevice(ctx->device));
  sdb_hnsw* h = new sdb_hnsw();
  h->ctx = ctx;
  h->dim = dim;
  h->metric = metric;
  h->n = n_elems;
  h->n_layers = n_layers;
  h->entry = entry_point;
  cudaStream_t st = ctx->stream;
  const uint64_t nn = n_elems ? n_elems : 1;
  uint64_t bad_total = 0, bad = 0;
  sdb_status rc = SDB_OK;
  uint8_t* d_present = nullptr;
  if (cudaMalloc(&d_present, nn) != cudaSuccess || cudaMemsetAsync(d_present, 0, nn, st) != cudaSuccess) {
    set_error("hnsw load: present-mask allocation failed: %s", cudaGetErrorString(cudaGetLastError()));
    rc = SDB_ENOMEM;
  }
  if (cudaMalloc(&h->d_vec, sizeof(float) * nn * dim) != cudaSuccess ||
      cudaMalloc(&h->d_sumsq, sizeof(float) * nn) != cudaSuccess) {
    set_error("hnsw load: vector allocation failed: %s", cudaGetErrorString(cudaGetLastError()));
    rc = SDB_ENOMEM;
  }
  // elements without an He value keep all-zero vectors; they are unreachable unless an Hn value names them
  if (rc == SDB_OK && cudaMemsetAsync(h->d_vec, 0, sizeof(float) * nn * dim, st) != cudaSuccess) rc = SDB_ECUDA;
  if (rc == SDB_OK)
    rc = stage_decode_vectors(ctx, vec_blob, vec_off, vec_ids, n_vec, dim, SDB_F32, n_elems, h->d_vec, d_present, &bad, st);
  bad_total += bad;
  uint64_t n_dropped = 0;
  for (uint32_t l = 0; l < n_layers && rc == SDB_OK; l++) {
    uint64_t* drp = nullptr;
    uint32_t* dci = nullptr;
    uint64_t ne = 0;
    bad = 0;
    rc = stage_decode_nodes(ctx, node_blob[l], node_off[l], node_ids[l], n_nodes[l], n_elems, &drp, &dci, &ne, &bad, st);
    if (rc == SDB_OK) {
      bad_total += bad;
      // drop edges from / to elements that have no He value ("edge to an unknown element")
      uint64_t *rp2 = nullptr, *d_tot = nullptr;
      uint32_t* ci2 = nullptr;
      uint64_t kept = 0;
      const unsigned g1 = (unsigned)((n_elems + 1 + 255) / 256);
      if (cudaMalloc(&rp2, 8 * (n_elems + 1)) != cudaSuccess || cudaMalloc(&d_tot, 8) != cudaSuccess) rc = SDB_ENOMEM;
      if (rc == SDB_OK) {
        csr_present_degree_kernel<<<g1, 256, 0, st>>>(drp, dci, d_present, n_elems, rp2);
        count_launch(ctx);
        rc = exclusive_scan(ctx, rp2, rp2, n_elems + 1, d_tot, st);
      }
      if (rc == SDB_OK && (cudaMemcpyAsync(&kept, d_tot, 8, cudaMemcpyDeviceToHost, st) != cudaSuccess ||
                           cudaStreamSynchronize(st) != cudaSuccess))
        rc = SDB_ECUDA;
      if (rc == SDB_OK && cudaMalloc(&ci2, 4 * (kept ? kept : 1)) != cudaSuccess) rc = SDB_ENOMEM;
      if (rc == SDB_OK && n_elems) {
        csr_present_fill_kernel<<<g1, 256, 0, st>>>(drp, dci, d_present, n_elems, rp2, ci2);
        count_launch(ctx);
        if (cudaStreamSynchronize(st) != cudaSuccess) rc = SDB_ECUDA;
      }
      cudaFree(d_tot);
      if (rc == SDB_OK) {
        n_dropped += ne - kept;
        cudaFree(drp);
        cudaFree(dci);
        h->rp.push_back(rp2);
        h->ci.push_back(ci2);
      } else {
        if (rc == SDB_ENOMEM) set_error("hnsw load: CSR filter allocation failed");
        cudaFree(rp2);
        cudaFree(ci2);
        cudaFree(drp);
        cudaFree(dci);
      }
    }
  }
  bad_total += n_dropped;
  if (n_bad) *n_bad = bad_total;
  uint8_t ep_present = 1;
  if (rc == SDB_OK && entry_point >= 0 && n_elems &&
      cudaMemcpy(&ep_present, d_present + entry_point, 1, cudaMemcpyDeviceToHost) != cudaSuccess)
    rc = SDB_ECUDA;
  cudaFree(d_present);
  if (rc == SDB_OK && !ep_present) {
    set_error("sdb_hnsw_load_staged: the entry point %lld has no He value", (long long)entry_point);
    rc = SDB_EINVAL;
  }
  if (rc != SDB_OK) {
    sdb_hnsw_destroy(h);
    return rc;
  }
  return hnsw_finish(h, out);
}

sdb_status sdb_hnsw_select_neighbors(sdb_ctx* ctx, const float* d_vectors, uint32_t dim, sdb_metric metric, uint64_t row0,
                                     uint64_t n, const uint64_t* d_cand, const uint32_t* d_cand_cnt, uint32_t kc,
                                     uint32_t m_max, int presorted, uint32_t* d_out, uint32_t* d_out_cnt) {
  if (!ctx || !d_vectors || !d_cand || !d_cand_cnt || !d_out || !d_out_cnt || !dim || !kc || !m_max) return SDB_EINVAL;
  if (metric != SDB_COSINE && metric != SDB_EUCLIDEAN) return SDB_EUNSUPPORTED;
  if (n == 0) return SDB_OK;
  std::lock_guard<std::mutex> guard(ctx->mu);
  SDB_CUDA(cudaSetDevice(ctx->device));
  const size_t smem = sizeof(float) * (2 * (size_t)dim + 2 * kc) * 4;
  auto kern = metric == SDB_COSINE ? hnsw_select_kernel<true> : hnsw_select_kernel<false>;
  SDB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<(unsigned)((n + 3) / 4), 128, smem, ctx->stream>>>(d_vectors, dim, row0, n, nullptr, d_cand, d_cand_cnt, kc, m_max, presorted, d_out, d_out_cnt);
  count_launch(ctx);
  SDB_CUDA(cudaGetLastError());
  SDB_CUDA(cudaStreamSynchronize(ctx->stream));
  return SDB_OK;
}

sdb_status sdb_hnsw_select_neighbors_ids(sdb_ctx* ctx, const float* d_vectors, uint32_t dim, sdb_metric metric,
                                         const uint32_t* d_elem_ids, uint64_t n, const uint64_t* d_cand,
                                         const uint32_t* d_cand_cnt, uint32_t kc, uint32_t m_max, int presorted,
                                         uint32_t* d_out, uint32_t* d_out_cnt) {
  if (!ctx || !d_vectors || !d_elem_ids || !d_cand || !d_cand_cnt || !d_out || !d_out_cnt || !dim || !kc || !m_max) return SDB_EINVAL;
  if (metric != SDB_COSINE && metric != SDB_EUCLIDEAN) return SDB_EUNSUPPORTED;
  if (n == 0) return SDB_OK;
  std::lock_guard<std::mutex> guard(ctx->mu);
  SDB_CUDA(cudaSetDevice(ctx->device));
  const size_t smem = sizeof(float) * (2 * (size_t)dim + 2 * kc) * 4;
  auto kern = metric == SDB_COSINE ? hnsw_select_kernel<true> : hnsw_select_kernel<false>;
  SDB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<(unsigned)((n + 3) / 4), 128, smem, ctx->stream>>>(d_vectors, dim, 0, n, d_elem_ids, d_cand, d_cand_cnt, kc, m_max, presorted, d_out, d_out_cnt);
  count_launch(ctx);
  SDB_CUDA(cudaGetLastError());
  SDB_CUDA(cudaStreamSynchronize(ctx->stream));
  return SDB_OK;
}

static sdb_status hnsw_search_impl(sdb_hnsw* h, const float* queries, uint32_t nq, uint32_t k, uint32_t ef,
                                   const uint8_t* truthy, const uint8_t* noexp, uint64_t* out_elems, double* out_dist,
                                   uint32_t* out_count, uint64_t* out_counters, bool device_io = false) {
  if (!h || (nq && (!queries || !out_count)) || (nq && k && (!out_elems || !out_dist))) return SDB_EINVAL;
  if (nq == 0) return SDB_OK;
  if (k == 0 || ef == 0) {  // to_vec_limit(0) underflows in the reference; we return nothing
    if (device_io) {
      SDB_CUDA(cudaSetDevice(h->ctx->device));
      SDB_CUDA(cudaMemsetAsync(out_count, 0, sizeof(uint32_t) * nq, h->ctx->stream));
      SDB_CUDA(cudaStreamSynchronize(h->ctx->stream));
    } else {
      memset(out_count, 0, sizeof(uint32_t) * nq);
    }
    return SDB_OK;
  }
  if (ef > 4096) {
    set_error("hnsw: ef %u > 4096 unsupported", ef);
    return SDB_EUNSUPPORTED;
  }
  Ctx* ctx = h->ctx;
  std::lock_guard<std::mutex> guard(h->mu);
  SDB_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  // unfiltered: live candidates are a subset of w plus ties, 2*ef+34 is ample.  Filtered: every admitted element is a
  // candidate but only truthy ones enter w, so the window is sized for a selectivity down to ~1/16 (more = EOVERFLOW)
  uint32_t ccap = 2 * ef + 34;
  const uint32_t wcap = ef + 2;
  if (truthy) {
    ccap = 16 * ef + 34;
    if (ccap < 1024) ccap = 1024;
    const size_t fixed = sizeof(float) * hn_q_floats(h->dim, h->metric == SDB_COSINE) + hn_tile_bytes(h->metric == SDB_COSINE) + 12 * (size_t)wcap + 64 + 16;
    const size_t room = (220 * 1024) / HN_WARPS;
    if (fixed + 12 * (size_t)ccap > room) ccap = room > fixed + 12 * (2 * (size_t)ef + 34) ? (uint32_t)((room - fixed) / 12) : 2 * ef + 34;
  }
  size_t per_warp = sizeof(float) * hn_q_floats(h->dim, h->metric == SDB_COSINE) + hn_tile_bytes(h->metric == SDB_COSINE) + 12 * (size_t)(ccap + wcap) + 64;
  per_warp = (per_warp + 15) & ~size_t(15);
  const size_t smem = per_warp * HN_WARPS;
  if (smem > 220 * 1024) {
    set_error("hnsw: dim %u / ef %u need %zu bytes of shared memory per block", h->dim, ef, smem);
    return SDB_EUNSUPPORTED;
  }
  // cosine: 8 lanes per row keep ~16 loads in flight per lane; 80 registers (6 blocks per SM) holds that without spills
  const int occ = getenv("SDB_HNSW_OCC") ? atoi(getenv("SDB_HNSW_OCC")) : 6;  // measured r2 (1M x 768, ef 64): 6 -> 1.40M QPS, 4 -> 1.32M, 8 -> 1.02M (spills)
  void (*kern)(HnswParams);
  switch (h->metric) {
    case SDB_COSINE:
      kern = occ >= 8 ? hnsw_search_kernel<SDB_COSINE, 8> : occ <= 4 ? hnsw_search_kernel<SDB_COSINE, 4> : hnsw_search_kernel<SDB_COSINE, 6>;
      break;
    case SDB_MANHATTAN: kern = hnsw_search_kernel<SDB_MANHATTAN, 1>; break;
    case SDB_CHEBYSHEV: kern = hnsw_search_kernel<SDB_CHEBYSHEV, 1>; break;
    case SDB_HAMMING: kern = hnsw_search_kernel<SDB_HAMMING, 1>; break;
    case SDB_MINKOWSKI: kern = hnsw_search_kernel<SDB_MINKOWSKI, 1>; break;
    default: kern = hnsw_search_kernel<SDB_EUCLIDEAN, 1>; break;  // the loaders admit no other metric
  }
  SDB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  // the walk gets nothing from L1 (0.7 % hit rate): give the whole array to shared memory, or the driver's default
  // carve-out (135 KB) caps the kernel at 5 blocks per SM
  SDB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
  int per_sm = 1;
  SDB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, HN_WARPS * 32, smem));
  if (per_sm < 1) per_sm = 1;
  uint32_t grid = (uint32_t)(ctx->sm_count * per_sm);
  if (grid > (nq + HN_WARPS - 1) / HN_WARPS) grid = (nq + HN_WARPS - 1) / HN_WARPS;
  // visited tables: one per resident warp; 16 x the worst-case expansion of a typical walk, >= 2^13 slots
  uint32_t tl = 13;
  while ((1u << tl) < ef * 64u * 4u && tl < 20) tl++;
  if (truthy) tl = tl + 3 > 18 ? (tl > 18 ? tl : 18) : tl + 3;  // filtered walks visit ~1/selectivity more elements
  const uint32_t n_tables = grid * HN_WARPS;
  if (!h->d_visited || h->table_log2 != tl || h->n_tables < n_tables) {
    cudaFree(h->d_visited);
    h->d_visited = nullptr;
    SDB_CUDA(cudaMalloc(&h->d_visited, sizeof(uint64_t) * ((size_t)n_tables << tl)));
    SDB_CUDA(cudaMemsetAsync(h->d_visited, 0, sizeof(uint64_t) * ((size_t)n_tables << tl), st));
    h->table_log2 = tl;
    h->n_tables = n_tables;
    h->gen = 1;
  }
  const uint32_t q_per_warp = (nq + n_tables - 1) / n_tables;
  const uint32_t gens_per_warp = q_per_warp * h->n_layers + 1;
  if ((uint64_t)h->gen + (uint64_t)gens_per_warp * n_tables >= 0xFFFFFFF0ull) {  // generation counter wrap
    SDB_CUDA(cudaMemsetAsync(h->d_visited, 0, sizeof(uint64_t) * ((size_t)h->n_tables << tl), st));
    h->gen = 1;
  }
  float* d_q = nullptr;
  uint64_t* d_elems = nullptr;
  double* d_dist = nullptr;
  uint32_t* d_cnt = nullptr;
  uint64_t* d_ctr = nullptr;
  uint32_t* d_ovf = nullptr;
  if (device_io) {  // queries and outputs already live on the device (index construction): no staging
    d_q = const_cast<float*>(queries);
    d_elems = out_elems;
    d_dist = out_dist;
    d_cnt = out_count;
  } else {
    SDB_CUDA(cudaMallocAsync(&d_q, sizeof(float) * (size_t)nq * h->dim, st));
    SDB_CUDA(cudaMallocAsync(&d_elems, sizeof(uint64_t) * (size_t)nq * k, st));
    SDB_CUDA(cudaMallocAsync(&d_dist, sizeof(double) * (size_t)nq * k, st));
    SDB_CUDA(cudaMallocAsync(&d_cnt, sizeof(uint32_t) * nq, st));
    SDB_CUDA(cudaMemcpyAsync(d_q, queries, sizeof(float) * (size_t)nq * h->dim, cudaMemcpyHostToDevice, st));
  }
  SDB_CUDA(cudaMallocAsync(&d_ctr, sizeof(uint64_t) * 2 * nq, st));
  SDB_CUDA(cudaMallocAsync(&d_ovf, 4, st));
  SDB_CUDA(cudaMemsetAsync(d_ovf, 0, 4, st));
  uint8_t* d_noexp = nullptr;
  if (noexp) {
    SDB_CUDA(cudaMallocAsync(&d_noexp, h->n ? h->n : 1, st));
    SDB_CUDA(cudaMemcpyAsync(d_noexp, noexp, h->n, cudaMemcpyHostToDevice, st));
  }
  uint8_t* d_truthy = nullptr;
  if (truthy) {
    SDB_CUDA(cudaMallocAsync(&d_truthy, h->n ? h->n : 1, st));
    SDB_CUDA(cudaMemcpyAsync(d_truthy, truthy, h->n, cudaMemcpyHostToDevice, st));
  }
  HnswParams P;
  P.ccap = ccap;
  P.truthy = d_truthy;
  P.noexp = d_noexp;
  P.vec = h->d_vec;
  P.norm = h->d_norm;
  P.rp = h->d_rp;
  P.ci = h->d_ci;
  P.dim = h->dim;
  P.n_layers = h->n_layers;
  P.entry = h->entry;
  P.queries = d_q;
  P.nq = nq;
  P.k = k;
  P.ef = ef;
  P.visited = h->d_visited;
  P.table_log2 = tl;
  P.gen_base = h->gen;
  P.gens_per_warp = gens_per_warp;
  P.cancel = ctx->d_cancel;
  P.out_elems = d_elems;
  P.out_dist = d_dist;
  P.out_count = d_cnt;
  P.out_counters = d_ctr;
  P.overflow = d_ovf;
  P.minkowski_p = h->minkowski_p;
  kern<<<grid, HN_WARPS * 32, smem, st>>>(P);
  count_launch(ctx);
  h->gen += gens_per_warp * n_tables;
  uint32_t ovf = 0;
  if (!device_io) {
    SDB_CUDA(cudaMemcpyAsync(out_elems, d_elems, sizeof(uint64_t) * (size_t)nq * k, cudaMemcpyDeviceToHost, st));
    SDB_CUDA(cudaMemcpyAsync(out_dist, d_dist, sizeof(double) * (size_t)nq * k, cudaMemcpyDeviceToHost, st));
    SDB_CUDA(cudaMemcpyAsync(out_count, d_cnt, sizeof(uint32_t) * nq, cudaMemcpyDeviceToHost, st));
  }
  if (out_counters)
    SDB_CUDA(cudaMemcpyAsync(out_counters, d_ctr, sizeof(uint64_t) * 2 * nq, device_io ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, st));
  SDB_CUDA(cudaMemcpyAsync(&ovf, d_ovf, 4, cudaMemcpyDeviceToHost, st));
  if (!device_io) {
    cudaFreeAsync(d_q, st);
    cudaFreeAsync(d_elems, st);
    cudaFreeAsync(d_dist, st);
    cudaFreeAsync(d_cnt, st);
  }
  cudaFreeAsync(d_ctr, st);
  cudaFreeAsync(d_ovf, st);
  if (d_truthy) cudaFreeAsync(d_truthy, st);
  if (d_noexp) cudaFreeAsync(d_noexp, st);
  SDB_CUDA(cudaStreamSynchronize(st));
  SDB_CUDA(cudaGetLastError());
  if (ctx_cancelled(ctx)) {  // warps stop taking new queries once the flag is up: the outputs are incomplete
    set_error("query cancelled");
    return SDB_ECANCELLED;
  }
  if (ovf == 1) {
    set_error("hnsw: visited table overflow (ef too large, or filter too selective, for the per-query table)");
    return SDB_EOVERFLOW;
  }
  if (ovf == 2) {
    set_error("hnsw: candidate window overflow (filter too selective for ef %u): use the CPU path for this query", ef);
    return SDB_EOVERFLOW;
  }
  return SDB_OK;
}

// Distance::calculate(query, vector) for n host vectors on the context's stream (sdb_vec_distance_f32 /
// sdb_hnsw_distance_f32); the metric has been validated by the caller
static sdb_status typed_distances(Ctx* ctx, sdb_metric metric, double p, uint32_t dim, const float* query,
                                  const float* vectors, uint64_t n, double* out, const char* what) {
  std::lock_guard<std::mutex> guard(ctx->mu);
  SDB_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  float *d_q = nullptr, *d_v = nullptr;
  double* d_o = nullptr;
  auto run = [&]() -> sdb_status {
    SDB_CUDA(cudaMallocAsync(&d_q, sizeof(float) * dim, st));
    SDB_CUDA(cudaMallocAsync(&d_v, sizeof(float) * n * dim, st));
    SDB_CUDA(cudaMallocAsync(&d_o, sizeof(double) * n, st));
    SDB_CUDA(cudaMemcpyAsync(d_q, query, sizeof(float) * dim, cudaMemcpyHostToDevice, st));
    SDB_CUDA(cudaMemcpyAsync(d_v, vectors, sizeof(float) * n * dim, cudaMemcpyHostToDevice, st));
    const unsigned grid = (unsigned)((n + 127) / 128);
    switch (metric) {
      case SDB_COSINE: typed_distance_kernel<SDB_COSINE><<<grid, 128, 0, st>>>(d_q, d_v, dim, n, p, d_o); break;
      case SDB_MANHATTAN: typed_distance_kernel<SDB_MANHATTAN><<<grid, 128, 0, st>>>(d_q, d_v, dim, n, p, d_o); break;
      case SDB_CHEBYSHEV: typed_distance_kernel<SDB_CHEBYSHEV><<<grid, 128, 0, st>>>(d_q, d_v, dim, n, p, d_o); break;
      case SDB_HAMMING: typed_distance_kernel<SDB_HAMMING><<<grid, 128, 0, st>>>(d_q, d_v, dim, n, p, d_o); break;
      case SDB_MINKOWSKI: typed_distance_kernel<SDB_MINKOWSKI><<<grid, 128, 0, st>>>(d_q, d_v, dim, n, p, d_o); break;
      default: typed_distance_kernel<SDB_EUCLIDEAN><<<grid, 128, 0, st>>>(d_q, d_v, dim, n, p, d_o); break;
    }
    count_launch(ctx);
    SDB_CUDA(cudaGetLastError());
    SDB_CUDA(cudaMemcpyAsync(out, d_o, sizeof(double) * n, cudaMemcpyDeviceToHost, st));
    return SDB_OK;
  };
  const sdb_status rc = run();
  if (d_q) cudaFreeAsync(d_q, st);
  if (d_v) cudaFreeAsync(d_v, st);
  if (d_o) cudaFreeAsync(d_o, st);
  if (cudaStreamSynchronize(st) != cudaSuccess && rc == SDB_OK) {
    set_error("%s: %s", what, cudaGetErrorString(cudaGetLastError()));
    return SDB_ECUDA;
  }
  return rc;
}

sdb_status sdb_vec_distance_f32(sdb_ctx* ctx, sdb_metric metric, uint32_t dim, const float* query, const float* vectors,
                                uint64_t n, double* out) {
  if (!ctx || !dim || (n && (!query || !vectors || !out))) return SDB_EINVAL;
  if (metric != SDB_COSINE && metric != SDB_EUCLIDEAN) {
    set_error("sdb_vec_distance_f32: metric %d not implemented on the GPU path", (int)metric);
    return SDB_EUNSUPPORTED;
  }
  if (n == 0) return SDB_OK;
  return typed_distances(ctx, metric, 3.0, dim, query, vectors, n, out, "sdb_vec_distance_f32");
}

sdb_status sdb_hnsw_distance_f32(sdb_hnsw* h, const float* query, const float* vectors, uint64_t n, double* out) {
  if (!h || (n && (!query || !vectors || !out))) return SDB_EINVAL;
  if (n == 0) return SDB_OK;
  double p;
  {
    std::lock_guard<std::mutex> guard(h->mu);
    p = h->minkowski_p;
  }
  return typed_distances(h->ctx, h->metric, p, h->dim, query, vectors, n, out, "sdb_hnsw_distance_f32");
}

sdb_status sdb_hnsw_set_minkowski_order(sdb_hnsw* h, double order) {
  if (!h || !(order == order)) return SDB_EINVAL;
  std::lock_guard<std::mutex> guard(h->mu);  // a search in flight keeps the order it started with
  h->minkowski_p = order;
  return SDB_OK;
}

sdb_status sdb_hnsw_search(sdb_hnsw* h, const float* queries, uint32_t nq, uint32_t k, uint32_t ef, uint64_t* out_elems,
                           double* out_dist, uint32_t* out_count, uint64_t* out_counters) {
  return hnsw_search_impl(h, queries, nq, k, ef, nullptr, nullptr, out_elems, out_dist, out_count, out_counters);
}

sdb_status sdb_hnsw_search_device(sdb_hnsw* h, const float* d_queries, uint32_t nq, uint32_t k, uint32_t ef,
                                  uint64_t* d_out_elems, double* d_out_dist, uint32_t* d_out_count) {
  return hnsw_search_impl(h, d_queries, nq, k, ef, nullptr, nullptr, d_out_elems, d_out_dist, d_out_count, nullptr, true);
}

sdb_status sdb_hnsw_search_pending(sdb_hnsw* h, const float* queries, uint32_t nq, uint32_t k, uint32_t ef,
                                   const uint8_t* all_docs_pending, uint64_t* out_elems, double* out_dist,
                                   uint32_t* out_count, uint64_t* out_counters) {
  if (!all_docs_pending) {
    set_error("sdb_hnsw_search_pending: the pending mask is NULL (use sdb_hnsw_search)");
    return SDB_EINVAL;
  }
  return hnsw_search_impl(h, queries, nq, k, ef, nullptr, all_docs_pending, out_elems, out_dist, out_count, out_counters);
}

sdb_status sdb_hnsw_search_filtered(sdb_hnsw* h, const float* queries, uint32_t nq, uint32_t k, uint32_t ef,
                                    const uint8_t* truthy, uint64_t* out_elems, double* out_dist, uint32_t* out_count,
                                    uint64_t* out_counters) {
  if (!truthy) {
    set_error("sdb_hnsw_search_filtered: truthy mask is NULL (use sdb_hnsw_search)");
    return SDB_EINVAL;
  }
  return hnsw_search_impl(h, queries, nq, k, ef, truthy, nullptr, out_elems, out_dist, out_count, out_counters);
}

}  // extern "C"
