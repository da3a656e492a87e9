// Device-side graph construction: edge list / COO / CSR / dense -> CSR + CSR^T + row-length-
// binned schedule.  Replaces the host scipy pipeline of the reference
//   pygcn/utils.py:360-368  (edge list -> A, symmetrise by max, + I)
//   pygcn/utils.py:390-397  (normalize: D^-1 M, fp64)
//   pygcn/utils.py:407-414  (sparse_mx_to_torch_sparse_tensor: COO int64 / fp32)
// and the per-call coalesce + COO->CSR that torch.spmm performs inside ATen (layers.py:34).
// Index layout and values are bit-exact with the reference (tests/test_gpu_parity.py).
// One-off work per adjacency: CUB radix sort / scan / reduce-by-key are used as plumbing.
#include <cub/cub.cuh>

#include <new>
#include <vector>

#include "common.cuh"

namespace gcnb {
namespace {

constexpr int kT = 256;
constexpr double kDenseRouteMinDensity = 0.10;
inline unsigned blocks_for(int64_t n) { return (unsigned)(n > 0 ? ceil_div(n, kT) : 1); }

struct DevBuf {
  void* p = nullptr;
  ~DevBuf() { if (p) cudaFree(p); }
  int alloc(size_t bytes) {
    if (p) { cudaFree(p); p = nullptr; }
    if (bytes == 0) bytes = 16;
    GCNB_CUDA(cudaMalloc(&p, bytes));
    return GCNB_OK;
  }
  template <typename T> T* as() { return reinterpret_cast<T*>(p); }
  void* release() { void* q = p; p = nullptr; return q; }
};

template <typename T>
int graph_alloc(gcnb_graph* g, T** out, int64_t count) {
  // + 16 bytes: the TMA-staged SpMM widens its copy windows to 16-byte boundaries
  size_t bytes = (size_t)(count > 0 ? count : 1) * sizeof(T) + 16;
  bytes = (bytes + 255) & ~(size_t)255;
  void* p = nullptr;
  GCNB_CUDA(cudaMalloc(&p, bytes));
  *out = reinterpret_cast<T*>(p);
  g->device_bytes += (int64_t)bytes;
  return GCNB_OK;
}

// ---------------------------------------------------------------- small kernels

// rowptr[r] = first position i in the (sorted) row-id array with ids[i] >= r ; rowptr[n] = nnz
__global__ void rowptr_from_sorted_kernel(const int32_t* __restrict__ ids, int64_t nnz, int64_t n,
                                          int32_t* __restrict__ rowptr) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r > n) return;
  int64_t lo = 0, hi = nnz;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (ids[mid] < r) lo = mid + 1; else hi = mid;
  }
  rowptr[r] = (int32_t)lo;
}

__global__ void expand_rows_kernel(const int32_t* __restrict__ rowptr, int64_t n, int64_t nnz,
                                   int32_t* __restrict__ rows) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= nnz) return;
  int64_t lo = 0, hi = n;  // largest r with rowptr[r] <= e
  while (hi - lo > 1) {
    const int64_t mid = (lo + hi) >> 1;
    if (rowptr[mid] <= e) lo = mid; else hi = mid;
  }
  rows[e] = (int32_t)lo;
}

__global__ void iota_kernel(int32_t* p, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = (int32_t)i;
}

// int64 COO -> int32 + range check + sortedness check (flags[0] = out of range, flags[1] = unsorted)
__global__ void coo_convert_kernel(int64_t nnz, int64_t n_rows, int64_t n_cols,
                                   const int64_t* __restrict__ row, const int64_t* __restrict__ col,
                                   int32_t* __restrict__ row32, int32_t* __restrict__ col32,
                                   uint64_t* __restrict__ key, int* __restrict__ flags) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= nnz) return;
  const int64_t r = row[e], c = col[e];
  if (r < 0 || r >= n_rows || c < 0 || c >= n_cols) { flags[0] = 1; return; }
  row32[e] = (int32_t)r;
  col32[e] = (int32_t)c;
  const uint64_t k = ((uint64_t)r << 32) | (uint64_t)c;
  key[e] = k;
  if (e > 0) {
    const uint64_t kp = ((uint64_t)row[e - 1] << 32) | (uint64_t)col[e - 1];
    if (kp > k) flags[1] = 1;
  }
}

__global__ void gather_coo_kernel(int64_t nnz, const int32_t* __restrict__ perm,
                                  const uint64_t* __restrict__ sorted_key,
                                  const float* __restrict__ val_in, int32_t* __restrict__ row32,
                                  int32_t* __restrict__ col32, float* __restrict__ val_out) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= nnz) return;
  const uint64_t k = sorted_key[e];
  row32[e] = (int32_t)(k >> 32);
  col32[e] = (int32_t)(k & 0xffffffffu);
  val_out[e] = val_in[perm[e]];
}

__global__ void csr_convert_kernel(int64_t n_rows, int64_t n_cols, int64_t nnz,
                                   const int64_t* __restrict__ crow, const int64_t* __restrict__ col,
                                   int32_t* __restrict__ rowptr, int32_t* __restrict__ col32,
                                   int* __restrict__ flags) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i <= n_rows) {
    const int64_t v = crow[i];
    if (v < 0 || v > nnz || (i > 0 && crow[i - 1] > v) || (i == 0 && v != 0) ||
        (i == n_rows && v != nnz))
      flags[0] = 1;
    rowptr[i] = (int32_t)v;
  }
  if (i < nnz) {
    const int64_t c = col[i];
    if (c < 0 || c >= n_cols) flags[0] = 1;
    col32[i] = (int32_t)c;
  }
}

// transpose gather: entry i of CSR^T comes from entry perm[i] of the CSR
__global__ void transpose_gather_kernel(int64_t nnz, const int32_t* __restrict__ perm,
                                        const int32_t* __restrict__ rows,
                                        const float* __restrict__ val, int32_t* __restrict__ t_col,
                                        float* __restrict__ t_val) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nnz) return;
  const int32_t p = perm[i];
  t_col[i] = rows[p];
  t_val[i] = val[p];
}

__global__ void compare_i32_kernel(const int32_t* a, const int32_t* b, int64_t n, int* differs) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && a[i] != b[i]) *differs = 1;
}

// degree statistics: hist[0..4] bins, hist[5] = number of long rows, maxdeg via atomicMax
__global__ void degree_stats_kernel(const int32_t* __restrict__ rowptr, int64_t n,
                                    unsigned long long* __restrict__ hist, int* __restrict__ maxdeg,
                                    int32_t* __restrict__ long_flag, int32_t* __restrict__ long_chunks) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  const int deg = rowptr[r + 1] - rowptr[r];
  int b = 0;
  if (deg >= GCNB_BIN_EDGE_4) b = 4;
  else if (deg >= GCNB_BIN_EDGE_3) b = 3;
  else if (deg >= GCNB_BIN_EDGE_2) b = 2;
  else if (deg >= GCNB_BIN_EDGE_1) b = 1;
  atomicAdd(hist + b, 1ull);
  atomicMax(maxdeg, deg);
  const int is_long = deg >= kLongRowThreshold;
  long_flag[r] = is_long;
  long_chunks[r] = is_long ? (deg + kLongChunk - 1) / kLongChunk : 0;
}

// compaction of long rows: pos = exclusive scan of long_flag ; chunk_pos = exclusive scan of long_chunks
__global__ void long_rows_fill_kernel(int64_t n, const int32_t* __restrict__ long_flag,
                                      const int32_t* __restrict__ pos,
                                      const int32_t* __restrict__ chunk_pos,
                                      int32_t* __restrict__ long_rows,
                                      int32_t* __restrict__ long_chunk_ptr) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  if (long_flag[r]) {
    long_rows[pos[r]] = (int32_t)r;
    long_chunk_ptr[pos[r]] = chunk_pos[r];
  }
}

// rows [r0, r1) x cols [c0, c1) of a CSR: count, then fill (storage order preserved)
__global__ void block_count_kernel(int64_t r0, int64_t n_rows, int32_t c0, int32_t c1,
                                   const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                   int32_t* __restrict__ counts) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_rows) return;
  int cnt = 0;
  for (int e = rowptr[r0 + r]; e < rowptr[r0 + r + 1]; ++e) {
    const int c = col[e];
    cnt += (c >= c0 && c < c1);
  }
  counts[r] = cnt;
}

__global__ void block_fill_kernel(int64_t r0, int64_t n_rows, int32_t c0, int32_t c1, int32_t shift,
                                  const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                  const float* __restrict__ val, const int32_t* __restrict__ new_rowptr,
                                  int32_t* __restrict__ new_col, float* __restrict__ new_val,
                                  int32_t* __restrict__ new_rows) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_rows) return;
  int o = new_rowptr[r];
  for (int e = rowptr[r0 + r]; e < rowptr[r0 + r + 1]; ++e) {
    const int c = col[e];
    if (c >= c0 && c < c1) {
      new_col[o] = c - c0 + shift;
      new_val[o] = val[e];
      new_rows[o] = (int32_t)r;
      ++o;
    }
  }
}

// same as block_count/fill, but columns are remapped through the partition bounds (all-gather layout)
__device__ __forceinline__ int part_of(const int64_t* __restrict__ bounds, int n_parts, int c) {
  int lo = 0, hi = n_parts;  // largest q with bounds[q] <= c
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (bounds[mid] <= c) lo = mid; else hi = mid;
  }
  return lo;
}

__global__ void gathered_count_kernel(int64_t r0, int64_t n_rows, int n_parts,
                                      const int64_t* __restrict__ bounds, unsigned long long include,
                                      const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                      int32_t* __restrict__ counts) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_rows) return;
  int cnt = 0;
  for (int e = rowptr[r0 + r]; e < rowptr[r0 + r + 1]; ++e) cnt += (int)((include >> part_of(bounds, n_parts, col[e])) & 1ull);
  counts[r] = cnt;
}

__global__ void gathered_fill_kernel(int64_t r0, int64_t n_rows, int n_parts,
                                     const int64_t* __restrict__ bounds, unsigned long long include, int64_t pad_rows,
                                     const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                     const float* __restrict__ val, const int32_t* __restrict__ new_rowptr,
                                     int32_t* __restrict__ new_col, float* __restrict__ new_val,
                                     int32_t* __restrict__ new_rows) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_rows) return;
  int o = new_rowptr[r];
  for (int e = rowptr[r0 + r]; e < rowptr[r0 + r + 1]; ++e) {
    const int c = col[e];
    const int q = part_of(bounds, n_parts, c);
    if ((include >> q) & 1ull) {
      new_col[o] = (int32_t)((int64_t)q * pad_rows + (c - bounds[q]));
      new_val[o] = val[e];
      new_rows[o] = (int32_t)r;
      ++o;
    }
  }
}

// zero-padded copy of a dense matrix and of its transpose (dense route)
__global__ void dense_copy_kernel(int64_t n_rows, int64_t n_cols, const float* __restrict__ a, int64_t lda,
                                  float* __restrict__ fwd, int64_t ld_fwd, float* __restrict__ bwd, int64_t ld_bwd) {
  __shared__ float tile[32][33];
  const int64_t c0 = (int64_t)blockIdx.x * 32, r0 = (int64_t)blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int64_t r = r0 + i, c = c0 + threadIdx.x;
    float v = 0.f;
    if (r < n_rows && c < n_cols) v = a[r * lda + c];
    if (r < n_rows && c < ld_fwd) fwd[r * ld_fwd + c] = v;
    tile[i][threadIdx.x] = v;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int64_t c = c0 + i, r = r0 + threadIdx.x;  // bwd[c][r] = a[r][c]
    if (c < n_cols && r < ld_bwd) bwd[c * ld_bwd + r] = tile[threadIdx.x][i];
  }
}

__global__ void sum_i32_kernel(const int32_t* __restrict__ v, int64_t n, unsigned long long* out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && v[i] != 0) atomicAdd(out, (unsigned long long)v[i]);
}

// dense -> CSR: one warp per row
__global__ void dense_count_kernel(int64_t n_rows, int64_t n_cols, const float* __restrict__ a,
                                   int64_t lda, int32_t* __restrict__ counts) {
  const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= n_rows) return;
  int cnt = 0;
  for (int64_t c0 = 0; c0 < n_cols; c0 += 32) {
    const int64_t c = c0 + lane;
    const bool nz = (c < n_cols) && (a[row * lda + c] != 0.f);
    cnt += __popc(__ballot_sync(0xffffffffu, nz));
  }
  if (lane == 0) counts[row] = cnt;
}

__global__ void dense_fill_kernel(int64_t n_rows, int64_t n_cols, const float* __restrict__ a,
                                  int64_t lda, const int32_t* __restrict__ rowptr,
                                  int32_t* __restrict__ col, float* __restrict__ val) {
  const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= n_rows) return;
  int out = rowptr[row];
  for (int64_t c0 = 0; c0 < n_cols; c0 += 32) {
    const int64_t c = c0 + lane;
    float v = 0.f;
    if (c < n_cols) v = a[row * lda + c];
    const bool nz = (v != 0.f);
    const unsigned m = __ballot_sync(0xffffffffu, nz);
    if (nz) {
      const int off = __popc(m & ((1u << lane) - 1u));
      col[out + off] = (int32_t)c;
      val[out + off] = v;
    }
    out += __popc(m);
  }
}

// ---------------------------------------------------------------- edge-list pipeline kernels

__global__ void edge_keys_kernel(int64_t n_edges, int64_t n, const int32_t* __restrict__ src,
                                 const int32_t* __restrict__ dst, uint64_t* __restrict__ key,
                                 int* __restrict__ flags) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n_edges) return;
  const int64_t s = src[e], d = dst[e];
  if (s < 0 || s >= n || d < 0 || d >= n) { flags[0] = 1; key[e] = 0; return; }
  key[e] = (uint64_t)s * (uint64_t)n + (uint64_t)d;
}

// payload of one candidate entry: mx = multiplicity seen from A or A^T, diag = identity part
struct EntryVal {
  float mx;
  float diag;
};
struct EntryCombine {
  __host__ __device__ EntryVal operator()(const EntryVal& a, const EntryVal& b) const {
    EntryVal r;
    r.mx = a.mx > b.mx ? a.mx : b.mx;  // element-wise max(A, A^T)  (utils.py:365)
    r.diag = a.diag + b.diag;          // + I                       (utils.py:368)
    return r;
  }
};

__global__ void emit_entries_kernel(int64_t n_unique, int64_t n, const uint64_t* __restrict__ ukey,
                                    const int32_t* __restrict__ ucount, int symmetrize,
                                    int self_loops, uint64_t* __restrict__ key,
                                    unsigned long long* __restrict__ payload) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t n_dir = symmetrize ? 2 * n_unique : n_unique;
  const int64_t total = n_dir + (self_loops ? n : 0);
  if (i >= total) return;
  EntryVal v;
  uint64_t k;
  if (i < n_unique) {
    k = ukey[i];
    v.mx = (float)ucount[i];  // duplicate edges are summed by the COO->CSR conversion (utils.py:360)
    v.diag = 0.f;
  } else if (i < n_dir) {
    const uint64_t k0 = ukey[i - n_unique];
    k = (k0 % (uint64_t)n) * (uint64_t)n + (k0 / (uint64_t)n);
    v.mx = (float)ucount[i - n_unique];
    v.diag = 0.f;
  } else {
    const uint64_t d = (uint64_t)(i - n_dir);
    k = d * (uint64_t)n + d;
    v.mx = 0.f;
    v.diag = 1.f;
  }
  key[i] = k;
  unsigned long long p;
  memcpy(&p, &v, sizeof(p));
  payload[i] = p;
}

__global__ void entries_to_csr_kernel(int64_t nnz, int64_t n, const uint64_t* __restrict__ key,
                                      const EntryVal* __restrict__ ev, int32_t* __restrict__ rows,
                                      int32_t* __restrict__ col, double* __restrict__ val64) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= nnz) return;
  const uint64_t k = key[e];
  rows[e] = (int32_t)(k / (uint64_t)n);
  col[e] = (int32_t)(k % (uint64_t)n);
  val64[e] = (double)ev[e].mx + (double)ev[e].diag;  // A (fp32) + I (fp64) upcasts to fp64
}

// normalize (utils.py:390-397): rowsum in storage order (fp64), r_inv = 1/rowsum with inf -> 0,
// value = r_inv * value, then the fp64 -> fp32 cast of utils.py:409.
__global__ void normalize_rows_kernel(int64_t n, const int32_t* __restrict__ rowptr,
                                      const double* __restrict__ val64, int normalize,
                                      float* __restrict__ val) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  const int s = rowptr[r], e = rowptr[r + 1];
  double r_inv = 1.0;
  if (normalize) {
    double sum = 0.0;
    for (int i = s; i < e; ++i) sum += val64[i];
    r_inv = 1.0 / sum;
    if (isinf(r_inv)) r_inv = 0.0;
  }
  for (int i = s; i < e; ++i) val[i] = (float)(normalize ? r_inv * val64[i] : val64[i]);
}

__global__ void export_coo_kernel(int64_t nnz, int64_t n_rows, const int32_t* __restrict__ rowptr,
                                  const int32_t* __restrict__ col, const float* __restrict__ val,
                                  int64_t* __restrict__ indices, float* __restrict__ values) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= nnz) return;
  int64_t lo = 0, hi = n_rows;
  while (hi - lo > 1) {
    const int64_t mid = (lo + hi) >> 1;
    if (rowptr[mid] <= e) lo = mid; else hi = mid;
  }
  indices[e] = lo;
  indices[nnz + e] = col[e];
  values[e] = val[e];
}

// ---- fp64 handles: the same pipeline carries val64 beside val, gathered with the same permutations; val = fp32(val64)
__global__ void gather_coo_f64_kernel(int64_t nnz, const int32_t* __restrict__ perm, const uint64_t* __restrict__ sorted_key,
                                      const double* __restrict__ val_in, int32_t* __restrict__ row32,
                                      int32_t* __restrict__ col32, double* __restrict__ val64, float* __restrict__ val) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= nnz) return;
  const uint64_t k = sorted_key[e];
  row32[e] = (int32_t)(k >> 32);
  col32[e] = (int32_t)(k & 0xffffffffu);
  const double v = val_in[perm[e]];
  val64[e] = v;
  val[e] = (float)v;
}

// dst[i] = src[perm[i]] (the transpose's values)
__global__ void permute_f64_kernel(int64_t nnz, const int32_t* __restrict__ perm, const double* __restrict__ src,
                                   double* __restrict__ dst) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nnz) dst[i] = src[perm[i]];
}

__global__ void round_f64_kernel(int64_t nnz, const double* __restrict__ val64, float* __restrict__ val) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nnz) val[i] = (float)val64[i];
}

__global__ void dense_count_f64_kernel(int64_t n_rows, int64_t n_cols, const double* __restrict__ a, int64_t lda,
                                       int32_t* __restrict__ counts) {
  const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= n_rows) return;
  int cnt = 0;
  for (int64_t c0 = 0; c0 < n_cols; c0 += 32) {
    const int64_t c = c0 + lane;
    cnt += __popc(__ballot_sync(0xffffffffu, (c < n_cols) && (a[row * lda + c] != 0.0)));
  }
  if (lane == 0) counts[row] = cnt;
}

__global__ void dense_fill_f64_kernel(int64_t n_rows, int64_t n_cols, const double* __restrict__ a, int64_t lda,
                                      const int32_t* __restrict__ rowptr, int32_t* __restrict__ col,
                                      double* __restrict__ val64, float* __restrict__ val) {
  const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= n_rows) return;
  int out = rowptr[row];
  for (int64_t c0 = 0; c0 < n_cols; c0 += 32) {
    const int64_t c = c0 + lane;
    const double v = (c < n_cols) ? a[row * lda + c] : 0.0;
    const bool nz = (v != 0.0);
    const unsigned m = __ballot_sync(0xffffffffu, nz);
    if (nz) {
      const int off = __popc(m & ((1u << lane) - 1u));
      col[out + off] = (int32_t)c;
      val64[out + off] = v;
      val[out + off] = (float)v;
    }
    out += __popc(m);
  }
}

// normalize_rows_kernel that also keeps the fp64 values r_inv * value (utils.py:397, before the cast of utils.py:409)
__global__ void normalize_rows_keep_f64_kernel(int64_t n, const int32_t* __restrict__ rowptr, double* __restrict__ val64,
                                               int normalize, float* __restrict__ val) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  const int s = rowptr[r], e = rowptr[r + 1];
  double r_inv = 1.0;
  if (normalize) {
    double sum = 0.0;
    for (int i = s; i < e; ++i) sum += val64[i];
    r_inv = 1.0 / sum;
    if (isinf(r_inv)) r_inv = 0.0;
  }
  for (int i = s; i < e; ++i) {
    const double v = normalize ? r_inv * val64[i] : val64[i];
    val64[i] = v;
    val[i] = (float)v;
  }
}

int bits_for(uint64_t max_value) {
  int b = 1;
  while (b < 64 && (max_value >> b) != 0) ++b;
  return b;
}

// pair[i] = (col[i], bits of val[i])
__global__ void interleave_kernel(int64_t nnz, const int32_t* __restrict__ col, const float* __restrict__ val,
                                  uint2* __restrict__ pair) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nnz) pair[i] = make_uint2((uint32_t)col[i], __float_as_uint(val[i]));
}

// ---- tags of the pair stream (common.cuh: heat class of the column, end-of-row flag) and the entry-balanced
// ---- items of the streaming SpMM
__global__ void col_count_kernel(int64_t nnz, const int32_t* __restrict__ col, int32_t* __restrict__ cnt) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nnz) atomicAdd(cnt + col[i], 1);  // integer counts: order-independent
}

struct HeatThresholds { int32_t t[15]; };  // class c <=> count > t[c] (t non-increasing in c)

// pair[i].x |= class(col) << 27
__global__ void tag_class_kernel(int64_t nnz, const int32_t* __restrict__ cnt, HeatThresholds th,
                                 uint2* __restrict__ pair) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nnz) return;
  const uint32_t c = pair[i].x;
  const int32_t k = cnt[c];
  uint32_t cls = kPairColdClass;
#pragma unroll
  for (int j = 14; j >= 0; --j)
    if (k > th.t[j]) cls = (uint32_t)j;
  pair[i].x = c | (cls << kPairClassShift);
}

// the last stored entry of every non-empty row carries kPairRowEnd
__global__ void tag_row_end_kernel(int64_t n, const int32_t* __restrict__ rowptr, uint2* __restrict__ pair) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  const int s = rowptr[r], e = rowptr[r + 1];
  if (e > s) pair[e - 1].x |= kPairRowEnd;
}

// items[i] = row holding stored entry i * kStreamItem | (that row began before the item ? 1 << 31 : 0)
__global__ void stream_items_kernel(int64_t n_items, int64_t n, const int32_t* __restrict__ rowptr,
                                    uint32_t* __restrict__ items) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_items) return;
  const int e = (int)(i * kStreamItem);
  int64_t lo = 0, hi = n;  // last r in [0, n) with rowptr[r] <= e  (rowptr[0] = 0 <= e); empty rows share a value
  while (hi - lo > 1) {    // with their successor, so the last such r is the row that holds entry e
    const int64_t mid = (lo + hi) >> 1;
    if (rowptr[mid] <= e) lo = mid; else hi = mid;
  }
  items[i] = (uint32_t)lo | (rowptr[lo] < e ? 0x80000000u : 0u);
}

int build_pairs(gcnb_graph* g, const int32_t* col, const float* val, uint2** out, cudaStream_t st) {
  GCNB_TRY(graph_alloc(g, out, g->nnz + 2));  // + slack: stages are copied two entries at a time
  GCNB_CUDA(cudaMemsetAsync(*out, 0, (size_t)(g->nnz + 2) * sizeof(uint2), st));
  if (g->nnz > 0) {
    interleave_kernel<<<blocks_for(g->nnz), kT, 0, st>>>(g->nnz, col, val, *out);
    GCNB_LAUNCH_CHECK();
  }
  return GCNB_OK;
}

// Tags `pair` (n_rows x n_cols view, CSR rowptr / col) and builds the view's stream items.
int build_stream_schedule(gcnb_graph* g, const int32_t* rowptr, const int32_t* col, int64_t n_rows, int64_t n_cols,
                          uint2* pair, CsrView* view, uint32_t** items_out, cudaStream_t st) {
  const int64_t nnz = g->nnz;
  view->pair_tagged = false;
  view->n_stream_items = 0;
  view->stream_items = nullptr;
  *items_out = nullptr;
  if (nnz == 0 || n_cols > (1ll << kPairColBits) || n_rows == 0) return GCNB_OK;
  // heat classes: class c = among the 1024 * 2^c most referenced columns (strictly more references than the
  // column at that rank)
  DevBuf cnt, sorted, temp;
  GCNB_TRY(cnt.alloc((size_t)n_cols * 4));
  GCNB_TRY(sorted.alloc((size_t)n_cols * 4));
  GCNB_CUDA(cudaMemsetAsync(cnt.p, 0, (size_t)n_cols * 4, st));
  col_count_kernel<<<blocks_for(nnz), kT, 0, st>>>(nnz, col, cnt.as<int32_t>());
  GCNB_LAUNCH_CHECK();
  size_t tb = 0;
  GCNB_CUDA(cub::DeviceRadixSort::SortKeysDescending(nullptr, tb, cnt.as<int32_t>(), sorted.as<int32_t>(), (int)n_cols, 0, 32, st));
  GCNB_TRY(temp.alloc(tb));
  GCNB_CUDA(cub::DeviceRadixSort::SortKeysDescending(temp.p, tb, cnt.as<int32_t>(), sorted.as<int32_t>(), (int)n_cols, 0, 32, st));
  HeatThresholds th;
  for (int c = 0; c < 15; ++c) {
    const int64_t rank = 1024ll << c;
    th.t[c] = 0x7fffffff;  // nothing qualifies ...
    if (rank < n_cols) {
      GCNB_CUDA(cudaMemcpyAsync(&th.t[c], sorted.as<int32_t>() + rank, 4, cudaMemcpyDeviceToHost, st));
    } else {
      th.t[c] = -1;        // ... or, when the class holds every column, everything does
    }
  }
  GCNB_CUDA(cudaStreamSynchronize(st));
  tag_class_kernel<<<blocks_for(nnz), kT, 0, st>>>(nnz, cnt.as<int32_t>(), th, pair);
  GCNB_LAUNCH_CHECK();
  tag_row_end_kernel<<<blocks_for(n_rows), kT, 0, st>>>(n_rows, rowptr, pair);
  GCNB_LAUNCH_CHECK();
  view->pair_tagged = true;
  const int64_t n_items = ceil_div(nnz, kStreamItem);
  GCNB_TRY(graph_alloc(g, items_out, n_items));
  stream_items_kernel<<<blocks_for(n_items), kT, 0, st>>>(n_items, n_rows, rowptr, *items_out);
  GCNB_LAUNCH_CHECK();
  view->n_stream_items = n_items;
  view->stream_items = *items_out;
  return GCNB_OK;
}

// ---------------------------------------------------------------- schedule + transpose

int build_schedule(gcnb_graph* g, const int32_t* rowptr, int64_t n, CsrView* view,
                   int32_t** long_rows_out, int32_t** long_chunk_ptr_out, cudaStream_t st) {
  DevBuf hist, maxdeg, flag, chunks, pos, cpos, temp;
  GCNB_TRY(hist.alloc(6 * sizeof(unsigned long long)));
  GCNB_TRY(maxdeg.alloc(sizeof(int)));
  GCNB_TRY(flag.alloc((size_t)(n + 1) * 4));
  GCNB_TRY(chunks.alloc((size_t)(n + 1) * 4));
  GCNB_TRY(pos.alloc((size_t)(n + 1) * 4));
  GCNB_TRY(cpos.alloc((size_t)(n + 1) * 4));
  GCNB_CUDA(cudaMemsetAsync(hist.p, 0, 6 * sizeof(unsigned long long), st));
  GCNB_CUDA(cudaMemsetAsync(maxdeg.p, 0, sizeof(int), st));
  GCNB_CUDA(cudaMemsetAsync(flag.p, 0, (size_t)(n + 1) * 4, st));
  GCNB_CUDA(cudaMemsetAsync(chunks.p, 0, (size_t)(n + 1) * 4, st));
  if (n > 0) {
    degree_stats_kernel<<<blocks_for(n), kT, 0, st>>>(rowptr, n, hist.as<unsigned long long>(),
                                                      maxdeg.as<int>(), flag.as<int32_t>(),
                                                      chunks.as<int32_t>());
    GCNB_LAUNCH_CHECK();
  }
  size_t tb = 0;
  GCNB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tb, flag.as<int32_t>(), pos.as<int32_t>(), (int)(n + 1), st));
  GCNB_TRY(temp.alloc(tb));
  GCNB_CUDA(cub::DeviceScan::ExclusiveSum(temp.p, tb, flag.as<int32_t>(), pos.as<int32_t>(), (int)(n + 1), st));
  GCNB_CUDA(cub::DeviceScan::ExclusiveSum(temp.p, tb, chunks.as<int32_t>(), cpos.as<int32_t>(), (int)(n + 1), st));
  unsigned long long h[6];
  int md = 0, n_long = 0, n_chunks = 0;
  GCNB_CUDA(cudaMemcpyAsync(h, hist.p, sizeof(h), cudaMemcpyDeviceToHost, st));
  GCNB_CUDA(cudaMemcpyAsync(&md, maxdeg.p, sizeof(int), cudaMemcpyDeviceToHost, st));
  GCNB_CUDA(cudaMemcpyAsync(&n_long, pos.as<int32_t>() + n, 4, cudaMemcpyDeviceToHost, st));
  GCNB_CUDA(cudaMemcpyAsync(&n_chunks, cpos.as<int32_t>() + n, 4, cudaMemcpyDeviceToHost, st));
  GCNB_CUDA(cudaStreamSynchronize(st));
  for (int b = 0; b < GCNB_NUM_BINS; ++b) view->bin_rows[b] = (int64_t)h[b];
  view->max_degree = md;
  view->n_long_rows = n_long;
  view->n_long_chunks = n_chunks;
  *long_rows_out = nullptr;
  *long_chunk_ptr_out = nullptr;
  if (n_long > 0) {
    GCNB_TRY(graph_alloc(g, long_rows_out, n_long));
    GCNB_TRY(graph_alloc(g, long_chunk_ptr_out, n_long + 1));
    long_rows_fill_kernel<<<blocks_for(n), kT, 0, st>>>(n, flag.as<int32_t>(), pos.as<int32_t>(),
                                                        cpos.as<int32_t>(), *long_rows_out,
                                                        *long_chunk_ptr_out);
    GCNB_LAUNCH_CHECK();
    GCNB_CUDA(cudaMemcpyAsync(*long_chunk_ptr_out + n_long, &n_chunks, 4, cudaMemcpyHostToDevice, st));
    GCNB_CUDA(cudaStreamSynchronize(st));
  }
  view->long_rows = *long_rows_out;
  view->long_chunk_ptr = *long_chunk_ptr_out;
  return GCNB_OK;
}

// g->rowptr/col/val hold a CSR whose rows are in order; `rows` = expanded row ids (device, nnz).
int finalize(gcnb_graph* g, const int32_t* rows, cudaStream_t st, bool with_transpose = true) {
  const int64_t nnz = g->nnz;
  if (!with_transpose) {
    g->has_transpose = false;
    g->pattern_symmetric = false;
    g->fwd.n_rows = g->n_rows; g->fwd.n_cols = g->n_cols; g->fwd.nnz = nnz;
    g->fwd.rowptr = g->rowptr; g->fwd.col = g->col; g->fwd.val = g->val;
    GCNB_TRY(build_pairs(g, g->col, g->val, &g->pair, st));
    g->fwd.pair = g->pair;
    g->bwd = CsrView();
    GCNB_TRY(build_schedule(g, g->rowptr, g->n_rows, &g->fwd, &g->long_rows, &g->long_chunk_ptr, st));
    GCNB_TRY(build_stream_schedule(g, g->rowptr, g->col, g->n_rows, g->n_cols, g->pair, &g->fwd, &g->stream_items, st));
    GCNB_CUDA(cudaStreamSynchronize(st));
    return GCNB_OK;
  }
  // ---- transpose: stable radix sort of entry ids by column
  DevBuf key_out, perm_in, perm_out, temp, differs;
  GCNB_TRY(key_out.alloc((size_t)nnz * 4));
  GCNB_TRY(perm_in.alloc((size_t)nnz * 4));
  GCNB_TRY(perm_out.alloc((size_t)nnz * 4));
  GCNB_TRY(graph_alloc(g, &g->t_rowptr, g->n_cols + 1));
  GCNB_TRY(graph_alloc(g, &g->t_col, nnz));
  GCNB_TRY(graph_alloc(g, &g->t_val, nnz));
  if (nnz > 0) {
    iota_kernel<<<blocks_for(nnz), kT, 0, st>>>(perm_in.as<int32_t>(), nnz);
    GCNB_LAUNCH_CHECK();
    size_t tb = 0;
    const int end_bit = bits_for((uint64_t)(g->n_cols > 0 ? g->n_cols - 1 : 0));
    GCNB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tb, g->col, key_out.as<int32_t>(),
                                              perm_in.as<int32_t>(), perm_out.as<int32_t>(), nnz, 0,
                                              end_bit, st));
    GCNB_TRY(temp.alloc(tb));
    GCNB_CUDA(cub::DeviceRadixSort::SortPairs(temp.p, tb, g->col, key_out.as<int32_t>(),
                                              perm_in.as<int32_t>(), perm_out.as<int32_t>(), nnz, 0,
                                              end_bit, st));
    transpose_gather_kernel<<<blocks_for(nnz), kT, 0, st>>>(nnz, perm_out.as<int32_t>(), rows, g->val,
                                                            g->t_col, g->t_val);
    GCNB_LAUNCH_CHECK();
  }
  if (g->val64) {
    GCNB_TRY(graph_alloc(g, &g->t_val64, nnz));
    if (nnz > 0) {
      permute_f64_kernel<<<blocks_for(nnz), kT, 0, st>>>(nnz, perm_out.as<int32_t>(), g->val64, g->t_val64);
      GCNB_LAUNCH_CHECK();
    }
  }
  rowptr_from_sorted_kernel<<<blocks_for(g->n_cols + 1), kT, 0, st>>>(key_out.as<int32_t>(), nnz,
                                                                      g->n_cols, g->t_rowptr);
  GCNB_LAUNCH_CHECK();
  // ---- symmetric pattern?  then CSR^T can share rowptr/col with the CSR (values differ)
  g->pattern_symmetric = false;
  if (g->n_rows == g->n_cols) {
    GCNB_TRY(differs.alloc(sizeof(int)));
    GCNB_CUDA(cudaMemsetAsync(differs.p, 0, sizeof(int), st));
    compare_i32_kernel<<<blocks_for(g->n_rows + 1), kT, 0, st>>>(g->rowptr, g->t_rowptr, g->n_rows + 1,
                                                                 differs.as<int>());
    if (nnz > 0)
      compare_i32_kernel<<<blocks_for(nnz), kT, 0, st>>>(g->col, g->t_col, nnz, differs.as<int>());
    GCNB_LAUNCH_CHECK();
    int d = 1;
    GCNB_CUDA(cudaMemcpyAsync(&d, differs.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    GCNB_CUDA(cudaStreamSynchronize(st));
    if (d == 0) {
      g->pattern_symmetric = true;
      g->device_bytes -= (int64_t)((((size_t)(g->n_cols + 1) * 4 + 16 + 255) & ~(size_t)255) +
                                   (((size_t)(nnz > 0 ? nnz : 1) * 4 + 16 + 255) & ~(size_t)255));
      cudaFree(g->t_rowptr);
      cudaFree(g->t_col);
      g->t_rowptr = g->rowptr;
      g->t_col = g->col;
    }
  }
  // ---- views + schedules
  g->fwd.n_rows = g->n_rows; g->fwd.n_cols = g->n_cols; g->fwd.nnz = nnz;
  g->fwd.rowptr = g->rowptr; g->fwd.col = g->col; g->fwd.val = g->val;
  g->bwd.n_rows = g->n_cols; g->bwd.n_cols = g->n_rows; g->bwd.nnz = nnz;
  g->bwd.rowptr = g->t_rowptr; g->bwd.col = g->t_col; g->bwd.val = g->t_val;
  GCNB_TRY(build_pairs(g, g->col, g->val, &g->pair, st));
  GCNB_TRY(build_pairs(g, g->t_col, g->t_val, &g->t_pair, st));
  g->fwd.pair = g->pair;
  g->bwd.pair = g->t_pair;
  GCNB_TRY(build_schedule(g, g->rowptr, g->n_rows, &g->fwd, &g->long_rows, &g->long_chunk_ptr, st));
  GCNB_TRY(build_schedule(g, g->t_rowptr, g->n_cols, &g->bwd, &g->t_long_rows, &g->t_long_chunk_ptr, st));
  GCNB_TRY(build_stream_schedule(g, g->rowptr, g->col, g->n_rows, g->n_cols, g->pair, &g->fwd, &g->stream_items, st));
  GCNB_TRY(build_stream_schedule(g, g->t_rowptr, g->t_col, g->n_cols, g->n_rows, g->t_pair, &g->bwd, &g->t_stream_items, st));
  GCNB_CUDA(cudaStreamSynchronize(st));
  return GCNB_OK;
}

int check_dims(int64_t n_rows, int64_t n_cols, int64_t nnz) {
  GCNB_REQUIRE(n_rows >= 0 && n_cols >= 0 && nnz >= 0, "graph: negative size");
  GCNB_REQUIRE(n_rows < (1ll << 31) - 1 && n_cols < (1ll << 31) - 1, "graph: more than 2^31-2 rows/cols");
  GCNB_REQUIRE(nnz < (1ll << 31) - 1, "graph: more than 2^31-2 stored entries per handle (partition the graph)");
  return GCNB_OK;
}

gcnb_graph* new_graph(int64_t n_rows, int64_t n_cols, int64_t nnz) {
  gcnb_graph* g = new (std::nothrow) gcnb_graph();
  if (!g) return nullptr;
  cudaGetDevice(&g->device);
  g->n_rows = n_rows; g->n_cols = n_cols; g->nnz = nnz;
  return g;
}

int read_flags(DevBuf& flags, int* h, int count, cudaStream_t st) {
  GCNB_CUDA(cudaMemcpyAsync(h, flags.p, sizeof(int) * count, cudaMemcpyDeviceToHost, st));
  GCNB_CUDA(cudaStreamSynchronize(st));
  return GCNB_OK;
}

// f64: an fp64 handle, values from val64 (val unused)
int from_coo_impl(gcnb_graph* g, const int64_t* row, const int64_t* col, const float* val, cudaStream_t st,
                  bool f64 = false, const double* val64 = nullptr) {
  const int64_t nnz = g->nnz;
  DevBuf rows32, key, flags;
  GCNB_TRY(rows32.alloc((size_t)nnz * 4));
  GCNB_TRY(key.alloc((size_t)nnz * 8));
  GCNB_TRY(flags.alloc(2 * sizeof(int)));
  GCNB_CUDA(cudaMemsetAsync(flags.p, 0, 2 * sizeof(int), st));
  GCNB_TRY(graph_alloc(g, &g->rowptr, g->n_rows + 1));
  GCNB_TRY(graph_alloc(g, &g->col, nnz));
  GCNB_TRY(graph_alloc(g, &g->val, nnz));
  if (f64) GCNB_TRY(graph_alloc(g, &g->val64, nnz));
  int hf[2] = {0, 0};
  if (nnz > 0) {
    GCNB_REQUIRE(row && col && (f64 ? val64 != nullptr : val != nullptr), "graph_from_coo: null input");
    coo_convert_kernel<<<blocks_for(nnz), kT, 0, st>>>(nnz, g->n_rows, g->n_cols, row, col,
                                                       rows32.as<int32_t>(), g->col, key.as<uint64_t>(),
                                                       flags.as<int>());
    GCNB_LAUNCH_CHECK();
    GCNB_TRY(read_flags(flags, hf, 2, st));
    GCNB_REQUIRE(hf[0] == 0, "graph_from_coo: index out of range for a %lld x %lld matrix",
                 (long long)g->n_rows, (long long)g->n_cols);
    if (hf[1]) {  // not in (row, col) order: stable sort, duplicates keep their relative order
      DevBuf key_out, perm_in, perm_out, temp;
      GCNB_TRY(key_out.alloc((size_t)nnz * 8));
      GCNB_TRY(perm_in.alloc((size_t)nnz * 4));
      GCNB_TRY(perm_out.alloc((size_t)nnz * 4));
      iota_kernel<<<blocks_for(nnz), kT, 0, st>>>(perm_in.as<int32_t>(), nnz);
      size_t tb = 0;
      const int end_bit = 32 + bits_for((uint64_t)(g->n_rows > 0 ? g->n_rows - 1 : 0));
      GCNB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tb, key.as<uint64_t>(), key_out.as<uint64_t>(),
                                                perm_in.as<int32_t>(), perm_out.as<int32_t>(), nnz, 0,
                                                end_bit, st));
      GCNB_TRY(temp.alloc(tb));
      GCNB_CUDA(cub::DeviceRadixSort::SortPairs(temp.p, tb, key.as<uint64_t>(), key_out.as<uint64_t>(),
                                                perm_in.as<int32_t>(), perm_out.as<int32_t>(), nnz, 0,
                                                end_bit, st));
      if (f64)
        gather_coo_f64_kernel<<<blocks_for(nnz), kT, 0, st>>>(nnz, perm_out.as<int32_t>(), key_out.as<uint64_t>(), val64,
                                                              rows32.as<int32_t>(), g->col, g->val64, g->val);
      else
        gather_coo_kernel<<<blocks_for(nnz), kT, 0, st>>>(nnz, perm_out.as<int32_t>(), key_out.as<uint64_t>(),
                                                          val, rows32.as<int32_t>(), g->col, g->val);
      GCNB_LAUNCH_CHECK();
      GCNB_CUDA(cudaStreamSynchronize(st));
    } else if (f64) {
      GCNB_CUDA(cudaMemcpyAsync(g->val64, val64, (size_t)nnz * 8, cudaMemcpyDeviceToDevice, st));
      round_f64_kernel<<<blocks_for(nnz), kT, 0, st>>>(nnz, g->val64, g->val);
      GCNB_LAUNCH_CHECK();
    } else {
      GCNB_CUDA(cudaMemcpyAsync(g->val, val, (size_t)nnz * 4, cudaMemcpyDeviceToDevice, st));
    }
  }
  rowptr_from_sorted_kernel<<<blocks_for(g->n_rows + 1), kT, 0, st>>>(rows32.as<int32_t>(), nnz, g->n_rows,
                                                                      g->rowptr);
  GCNB_LAUNCH_CHECK();
  return finalize(g, rows32.as<int32_t>(), st);
}

int from_csr_impl(gcnb_graph* g, const int64_t* crow, const int64_t* col, const float* val, cudaStream_t st,
                  bool f64 = false, const double* val64 = nullptr) {
  const int64_t nnz = g->nnz;
  GCNB_REQUIRE(crow != nullptr && (nnz == 0 || (col && (f64 ? val64 != nullptr : val != nullptr))), "graph_from_csr: null input");
  DevBuf rows32, flags;
  GCNB_TRY(rows32.alloc((size_t)nnz * 4));
  GCNB_TRY(flags.alloc(2 * sizeof(int)));
  GCNB_CUDA(cudaMemsetAsync(flags.p, 0, 2 * sizeof(int), st));
  GCNB_TRY(graph_alloc(g, &g->rowptr, g->n_rows + 1));
  GCNB_TRY(graph_alloc(g, &g->col, nnz));
  GCNB_TRY(graph_alloc(g, &g->val, nnz));
  if (f64) GCNB_TRY(graph_alloc(g, &g->val64, nnz));
  const int64_t span = (g->n_rows + 1 > nnz) ? g->n_rows + 1 : nnz;
  csr_convert_kernel<<<blocks_for(span), kT, 0, st>>>(g->n_rows, g->n_cols, nnz, crow, col, g->rowptr,
                                                      g->col, flags.as<int>());
  GCNB_LAUNCH_CHECK();
  int hf[2] = {0, 0};
  GCNB_TRY(read_flags(flags, hf, 2, st));
  GCNB_REQUIRE(hf[0] == 0, "graph_from_csr: malformed crow_indices / col_indices");
  if (nnz > 0) {
    if (f64) {
      GCNB_CUDA(cudaMemcpyAsync(g->val64, val64, (size_t)nnz * 8, cudaMemcpyDeviceToDevice, st));
      round_f64_kernel<<<blocks_for(nnz), kT, 0, st>>>(nnz, g->val64, g->val);
      GCNB_LAUNCH_CHECK();
    } else {
      GCNB_CUDA(cudaMemcpyAsync(g->val, val, (size_t)nnz * 4, cudaMemcpyDeviceToDevice, st));
    }
    expand_rows_kernel<<<blocks_for(nnz), kT, 0, st>>>(g->rowptr, g->n_rows, nnz, rows32.as<int32_t>());
    GCNB_LAUNCH_CHECK();
  }
  return finalize(g, rows32.as<int32_t>(), st);
}

int from_dense_impl(gcnb_graph** out, int64_t n_rows, int64_t n_cols, const float* a, int64_t lda,
                    cudaStream_t st) {
  GCNB_REQUIRE(a != nullptr || n_rows * n_cols == 0, "graph_from_dense: null input");
  GCNB_REQUIRE(lda >= n_cols, "graph_from_dense: lda < n_cols");
  DevBuf counts, rowptr, temp;
  GCNB_TRY(counts.alloc((size_t)(n_rows + 1) * 4));
  GCNB_TRY(rowptr.alloc((size_t)(n_rows + 1) * 4));
  GCNB_CUDA(cudaMemsetAsync(counts.p, 0, (size_t)(n_rows + 1) * 4, st));
  if (n_rows > 0) {
    dense_count_kernel<<<blocks_for(n_rows * 32), kT, 0, st>>>(n_rows, n_cols, a, lda, counts.as<int32_t>());
    GCNB_LAUNCH_CHECK();
  }
  // guard int32 overflow of the scan with a 64-bit sum first
  DevBuf total;
  GCNB_TRY(total.alloc(8));
  GCNB_CUDA(cudaMemsetAsync(total.p, 0, 8, st));
  if (n_rows > 0) {
    sum_i32_kernel<<<blocks_for(n_rows), kT, 0, st>>>(counts.as<int32_t>(), n_rows, total.as<unsigned long long>());
    GCNB_LAUNCH_CHECK();
  }
  int64_t nnz = 0;
  GCNB_CUDA(cudaMemcpyAsync(&nnz, total.p, 8, cudaMemcpyDeviceToHost, st));
  GCNB_CUDA(cudaStreamSynchronize(st));
  GCNB_TRY(check_dims(n_rows, n_cols, nnz));
  size_t tb2 = 0;
  GCNB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tb2, counts.as<int32_t>(), rowptr.as<int32_t>(), (int)(n_rows + 1), st));
  GCNB_TRY(temp.alloc(tb2));
  GCNB_CUDA(cub::DeviceScan::ExclusiveSum(temp.p, tb2, counts.as<int32_t>(), rowptr.as<int32_t>(), (int)(n_rows + 1), st));
  gcnb_graph* g = new_graph(n_rows, n_cols, nnz);
  GCNB_REQUIRE(g != nullptr, "graph: host allocation failed");
  *out = g;
  DevBuf rows32;
  GCNB_TRY(rows32.alloc((size_t)nnz * 4));
  GCNB_TRY(graph_alloc(g, &g->rowptr, n_rows + 1));
  GCNB_TRY(graph_alloc(g, &g->col, nnz));
  GCNB_TRY(graph_alloc(g, &g->val, nnz));
  GCNB_CUDA(cudaMemcpyAsync(g->rowptr, rowptr.p, (size_t)(n_rows + 1) * 4, cudaMemcpyDeviceToDevice, st));
  if (n_rows > 0 && nnz > 0) {
    dense_fill_kernel<<<blocks_for(n_rows * 32), kT, 0, st>>>(n_rows, n_cols, a, lda, g->rowptr, g->col, g->val);
    GCNB_LAUNCH_CHECK();
    expand_rows_kernel<<<blocks_for(nnz), kT, 0, st>>>(g->rowptr, n_rows, nnz, rows32.as<int32_t>());
    GCNB_LAUNCH_CHECK();
  }
  GCNB_TRY(finalize(g, rows32.as<int32_t>(), st));
  // Dense route: above this density the tensor-core product over the dense matrix beats the CSR
  // gather (N^2*4 B streamed from HBM vs nnz*F*4 B gathered through L2).
  const double density = (n_rows > 0 && n_cols > 0) ? (double)nnz / ((double)n_rows * (double)n_cols) : 0.0;
  if (density >= kDenseRouteMinDensity && n_rows >= 64 && n_cols >= 64) {
    g->ld_fwd = ceil_div(n_cols, 4) * 4;
    g->ld_bwd = ceil_div(n_rows, 4) * 4;
    GCNB_TRY(graph_alloc(g, &g->dense_fwd, n_rows * g->ld_fwd));
    GCNB_TRY(graph_alloc(g, &g->dense_bwd, n_cols * g->ld_bwd));
    GCNB_CUDA(cudaMemsetAsync(g->dense_fwd, 0, (size_t)n_rows * g->ld_fwd * 4, st));
    GCNB_CUDA(cudaMemsetAsync(g->dense_bwd, 0, (size_t)n_cols * g->ld_bwd * 4, st));
    dim3 grid((unsigned)ceil_div(g->ld_fwd > n_cols ? g->ld_fwd : n_cols, 32),
              (unsigned)ceil_div(g->ld_bwd > n_rows ? g->ld_bwd : n_rows, 32));
    dense_copy_kernel<<<grid, dim3(32, 8), 0, st>>>(n_rows, n_cols, a, lda, g->dense_fwd, g->ld_fwd, g->dense_bwd,
                                                    g->ld_bwd);
    GCNB_LAUNCH_CHECK();
    GCNB_CUDA(cudaStreamSynchronize(st));
  }
  return GCNB_OK;
}

// fp64 dense adjacency: scanned into CSR (an fp64 handle never takes the dense route)
int from_dense_f64_impl(gcnb_graph** out, int64_t n_rows, int64_t n_cols, const double* a, int64_t lda, cudaStream_t st) {
  GCNB_REQUIRE(a != nullptr || n_rows * n_cols == 0, "graph_from_dense_f64: null input");
  GCNB_REQUIRE(lda >= n_cols, "graph_from_dense_f64: lda < n_cols");
  GCNB_REQUIRE((reinterpret_cast<uintptr_t>(a) & 7u) == 0, "graph_from_dense_f64: input not 8-byte aligned");
  DevBuf counts, rowptr, temp, total;
  GCNB_TRY(counts.alloc((size_t)(n_rows + 1) * 4));
  GCNB_TRY(rowptr.alloc((size_t)(n_rows + 1) * 4));
  GCNB_TRY(total.alloc(8));
  GCNB_CUDA(cudaMemsetAsync(counts.p, 0, (size_t)(n_rows + 1) * 4, st));
  GCNB_CUDA(cudaMemsetAsync(total.p, 0, 8, st));
  if (n_rows > 0) {
    dense_count_f64_kernel<<<blocks_for(n_rows * 32), kT, 0, st>>>(n_rows, n_cols, a, lda, counts.as<int32_t>());
    GCNB_LAUNCH_CHECK();
    sum_i32_kernel<<<blocks_for(n_rows), kT, 0, st>>>(counts.as<int32_t>(), n_rows, total.as<unsigned long long>());
    GCNB_LAUNCH_CHECK();
  }
  int64_t nnz = 0;
  GCNB_CUDA(cudaMemcpyAsync(&nnz, total.p, 8, cudaMemcpyDeviceToHost, st));
  GCNB_CUDA(cudaStreamSynchronize(st));
  GCNB_TRY(check_dims(n_rows, n_cols, nnz));
  size_t tb = 0;
  GCNB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tb, counts.as<int32_t>(), rowptr.as<int32_t>(), (int)(n_rows + 1), st));
  GCNB_TRY(temp.alloc(tb));
  GCNB_CUDA(cub::DeviceScan::ExclusiveSum(temp.p, tb, counts.as<int32_t>(), rowptr.as<int32_t>(), (int)(n_rows + 1), st));
  gcnb_graph* g = new_graph(n_rows, n_cols, nnz);
  GCNB_REQUIRE(g != nullptr, "graph: host allocation failed");
  *out = g;
  DevBuf rows32;
  GCNB_TRY(rows32.alloc((size_t)nnz * 4));
  GCNB_TRY(graph_alloc(g, &g->rowptr, n_rows + 1));
  GCNB_TRY(graph_alloc(g, &g->col, nnz));
  GCNB_TRY(graph_alloc(g, &g->val, nnz));
  GCNB_TRY(graph_alloc(g, &g->val64, nnz));
  GCNB_CUDA(cudaMemcpyAsync(g->rowptr, rowptr.p, (size_t)(n_rows + 1) * 4, cudaMemcpyDeviceToDevice, st));
  if (n_rows > 0 && nnz > 0) {
    dense_fill_f64_kernel<<<blocks_for(n_rows * 32), kT, 0, st>>>(n_rows, n_cols, a, lda, g->rowptr, g->col, g->val64,
                                                                  g->val);
    GCNB_LAUNCH_CHECK();
    expand_rows_kernel<<<blocks_for(nnz), kT, 0, st>>>(g->rowptr, n_rows, nnz, rows32.as<int32_t>());
    GCNB_LAUNCH_CHECK();
  }
  return finalize(g, rows32.as<int32_t>(), st);
}

int from_edges_impl(gcnb_graph** out, int64_t n, int64_t n_edges, const int32_t* src, const int32_t* dst,
                    int flags_in, cudaStream_t st) {
  GCNB_REQUIRE(n_edges == 0 || (src && dst), "graph_from_edges: null input");
  const int symmetrize = (flags_in & GCNB_BUILD_SYMMETRIZE) ? 1 : 0;
  const int self_loops = (flags_in & GCNB_BUILD_SELF_LOOPS) ? 1 : 0;
  const int normalize = (flags_in & GCNB_BUILD_ROW_NORMALIZE) ? 1 : 0;
  const int64_t max_entries = 2 * n_edges + n;
  GCNB_TRY(check_dims(n, n, max_entries));
  const int key_bits = bits_for(n > 0 ? (uint64_t)n * (uint64_t)n - 1 : 0);

  // 1. keys (src*n + dst), sorted; run-length encode -> unique (i,j) with multiplicity
  DevBuf key, key_sorted, flags, temp, ukey, ucount, nruns;
  GCNB_TRY(key.alloc((size_t)n_edges * 8));
  GCNB_TRY(key_sorted.alloc((size_t)n_edges * 8));
  GCNB_TRY(ukey.alloc((size_t)n_edges * 8));
  GCNB_TRY(ucount.alloc((size_t)n_edges * 4));
  GCNB_TRY(nruns.alloc(8));
  GCNB_TRY(flags.alloc(2 * sizeof(int)));
  GCNB_CUDA(cudaMemsetAsync(flags.p, 0, 2 * sizeof(int), st));
  GCNB_CUDA(cudaMemsetAsync(nruns.p, 0, 8, st));
  int64_t n_unique = 0;
  if (n_edges > 0) {
    edge_keys_kernel<<<blocks_for(n_edges), kT, 0, st>>>(n_edges, n, src, dst, key.as<uint64_t>(), flags.as<int>());
    GCNB_LAUNCH_CHECK();
    int hf[2];
    GCNB_TRY(read_flags(flags, hf, 2, st));
    GCNB_REQUIRE(hf[0] == 0, "graph_from_edges: node id out of range [0, %lld)", (long long)n);
    size_t tb = 0, tb2 = 0;
    GCNB_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, tb, key.as<uint64_t>(), key_sorted.as<uint64_t>(), n_edges, 0, key_bits, st));
    GCNB_CUDA(cub::DeviceRunLengthEncode::Encode(nullptr, tb2, key_sorted.as<uint64_t>(), ukey.as<uint64_t>(),
                                                 ucount.as<int32_t>(), nruns.as<int>(), (int)n_edges, st));
    GCNB_TRY(temp.alloc(tb > tb2 ? tb : tb2));
    GCNB_CUDA(cub::DeviceRadixSort::SortKeys(temp.p, tb, key.as<uint64_t>(), key_sorted.as<uint64_t>(), n_edges, 0, key_bits, st));
    GCNB_CUDA(cub::DeviceRunLengthEncode::Encode(temp.p, tb2, key_sorted.as<uint64_t>(), ukey.as<uint64_t>(),
                                                 ucount.as<int32_t>(), nruns.as<int>(), (int)n_edges, st));
    int nr = 0;
    GCNB_CUDA(cudaMemcpyAsync(&nr, nruns.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    GCNB_CUDA(cudaStreamSynchronize(st));
    n_unique = nr;
  }

  // 2. candidate entries: (i,j), (j,i) when symmetrising, (i,i) for + I; sort; reduce by key
  const int64_t n_cand = (symmetrize ? 2 : 1) * n_unique + (self_loops ? n : 0);
  DevBuf ckey, ckey_sorted, cval, cval_sorted, rkey, rval, temp2;
  GCNB_TRY(ckey.alloc((size_t)n_cand * 8));
  GCNB_TRY(ckey_sorted.alloc((size_t)n_cand * 8));
  GCNB_TRY(cval.alloc((size_t)n_cand * 8));
  GCNB_TRY(cval_sorted.alloc((size_t)n_cand * 8));
  GCNB_TRY(rkey.alloc((size_t)n_cand * 8));
  GCNB_TRY(rval.alloc((size_t)n_cand * 8));
  int64_t nnz = 0;
  if (n_cand > 0) {
    emit_entries_kernel<<<blocks_for(n_cand), kT, 0, st>>>(n_unique, n, ukey.as<uint64_t>(), ucount.as<int32_t>(),
                                                           symmetrize, self_loops, ckey.as<uint64_t>(),
                                                           cval.as<unsigned long long>());
    GCNB_LAUNCH_CHECK();
    size_t tb = 0, tb2 = 0;
    GCNB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tb, ckey.as<uint64_t>(), ckey_sorted.as<uint64_t>(),
                                              cval.as<unsigned long long>(), cval_sorted.as<unsigned long long>(),
                                              n_cand, 0, key_bits, st));
    GCNB_CUDA(cub::DeviceReduce::ReduceByKey(nullptr, tb2, ckey_sorted.as<uint64_t>(), rkey.as<uint64_t>(),
                                             cval_sorted.as<EntryVal>(), rval.as<EntryVal>(), nruns.as<int>(),
                                             EntryCombine(), (int)n_cand, st));
    GCNB_TRY(temp2.alloc(tb > tb2 ? tb : tb2));
    GCNB_CUDA(cub::DeviceRadixSort::SortPairs(temp2.p, tb, ckey.as<uint64_t>(), ckey_sorted.as<uint64_t>(),
                                              cval.as<unsigned long long>(), cval_sorted.as<unsigned long long>(),
                                              n_cand, 0, key_bits, st));
    GCNB_CUDA(cub::DeviceReduce::ReduceByKey(temp2.p, tb2, ckey_sorted.as<uint64_t>(), rkey.as<uint64_t>(),
                                             cval_sorted.as<EntryVal>(), rval.as<EntryVal>(), nruns.as<int>(),
                                             EntryCombine(), (int)n_cand, st));
    int nr = 0;
    GCNB_CUDA(cudaMemcpyAsync(&nr, nruns.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    GCNB_CUDA(cudaStreamSynchronize(st));
    nnz = nr;
  }

  // 3. CSR arrays, fp64 values, row normalisation, fp32 cast
  gcnb_graph* g = new_graph(n, n, nnz);
  GCNB_REQUIRE(g != nullptr, "graph: host allocation failed");
  *out = g;
  DevBuf rows32, val64;
  GCNB_TRY(rows32.alloc((size_t)nnz * 4));
  GCNB_TRY(val64.alloc((size_t)nnz * 8));
  GCNB_TRY(graph_alloc(g, &g->rowptr, n + 1));
  GCNB_TRY(graph_alloc(g, &g->col, nnz));
  GCNB_TRY(graph_alloc(g, &g->val, nnz));
  const bool keep_f64 = (flags_in & GCNB_BUILD_KEEP_F64) != 0;
  if (keep_f64) GCNB_TRY(graph_alloc(g, &g->val64, nnz));
  if (nnz > 0) {
    entries_to_csr_kernel<<<blocks_for(nnz), kT, 0, st>>>(nnz, n, rkey.as<uint64_t>(), rval.as<EntryVal>(),
                                                          rows32.as<int32_t>(), g->col, val64.as<double>());
    GCNB_LAUNCH_CHECK();
  }
  rowptr_from_sorted_kernel<<<blocks_for(n + 1), kT, 0, st>>>(rows32.as<int32_t>(), nnz, n, g->rowptr);
  GCNB_LAUNCH_CHECK();
  if (n > 0 && keep_f64) {
    if (nnz > 0) GCNB_CUDA(cudaMemcpyAsync(g->val64, val64.p, (size_t)nnz * 8, cudaMemcpyDeviceToDevice, st));
    normalize_rows_keep_f64_kernel<<<blocks_for(n), kT, 0, st>>>(n, g->rowptr, g->val64, normalize, g->val);
    GCNB_LAUNCH_CHECK();
  } else if (n > 0) {
    normalize_rows_kernel<<<blocks_for(n), kT, 0, st>>>(n, g->rowptr, val64.as<double>(), normalize, g->val);
    GCNB_LAUNCH_CHECK();
  }
  return finalize(g, rows32.as<int32_t>(), st);
}

}  // namespace
}  // namespace gcnb

// ------------------------------------------------------------------------------------ C ABI
using namespace gcnb;

extern "C" void gcnb_graph_free(gcnb_graph* g) {
  if (!g) return;
  int cur = 0;
  cudaGetDevice(&cur);
  if (cur != g->device) cudaSetDevice(g->device);
  if (!g->pattern_symmetric) {
    if (g->t_rowptr) cudaFree(g->t_rowptr);
    if (g->t_col) cudaFree(g->t_col);
  }
  cudaFree(g->rowptr);
  cudaFree(g->col);
  cudaFree(g->val);
  cudaFree(g->t_val);
  cudaFree(g->pair);
  cudaFree(g->t_pair);
  cudaFree(g->long_rows);
  cudaFree(g->long_chunk_ptr);
  cudaFree(g->t_long_rows);
  cudaFree(g->t_long_chunk_ptr);
  cudaFree(g->stream_items);
  cudaFree(g->t_stream_items);
  cudaFree(g->dense_fwd);
  cudaFree(g->dense_bwd);
  cudaFree(g->val64);
  cudaFree(g->t_val64);
  if (cur != g->device) cudaSetDevice(cur);
  delete g;
}

#define GCNB_BUILD_EPILOGUE(status)      \
  do {                                   \
    if ((status) != GCNB_OK) {           \
      if (*out) gcnb_graph_free(*out);   \
      *out = nullptr;                    \
    }                                    \
    return (status);                     \
  } while (0)

extern "C" int gcnb_graph_from_edges(int64_t n, int64_t n_edges, const int32_t* d_src, const int32_t* d_dst,
                                     int flags, void* stream, gcnb_graph** out) {
  GCNB_REQUIRE(out != nullptr, "graph_from_edges: out is null");
  *out = nullptr;
  GCNB_REQUIRE(n >= 0 && n_edges >= 0, "graph_from_edges: negative size");
  GCNB_TRY(gcnb_check_device());
  const int s = from_edges_impl(out, n, n_edges, d_src, d_dst, flags, (cudaStream_t)stream);
  GCNB_BUILD_EPILOGUE(s);
}

extern "C" int gcnb_graph_from_coo(int64_t n_rows, int64_t n_cols, int64_t nnz, const int64_t* d_row,
                                   const int64_t* d_col, const float* d_val, void* stream, gcnb_graph** out) {
  GCNB_REQUIRE(out != nullptr, "graph_from_coo: out is null");
  *out = nullptr;
  GCNB_TRY(check_dims(n_rows, n_cols, nnz));
  GCNB_TRY(gcnb_check_device());
  *out = new_graph(n_rows, n_cols, nnz);
  GCNB_REQUIRE(*out != nullptr, "graph: host allocation failed");
  const int s = from_coo_impl(*out, d_row, d_col, d_val, (cudaStream_t)stream);
  GCNB_BUILD_EPILOGUE(s);
}

extern "C" int gcnb_graph_from_csr(int64_t n_rows, int64_t n_cols, int64_t nnz, const int64_t* d_crow,
                                   const int64_t* d_col, const float* d_val, void* stream, gcnb_graph** out) {
  GCNB_REQUIRE(out != nullptr, "graph_from_csr: out is null");
  *out = nullptr;
  GCNB_TRY(check_dims(n_rows, n_cols, nnz));
  GCNB_TRY(gcnb_check_device());
  *out = new_graph(n_rows, n_cols, nnz);
  GCNB_REQUIRE(*out != nullptr, "graph: host allocation failed");
  const int s = from_csr_impl(*out, d_crow, d_col, d_val, (cudaStream_t)stream);
  GCNB_BUILD_EPILOGUE(s);
}

extern "C" int gcnb_graph_from_dense(int64_t n_rows, int64_t n_cols, const float* d_a, int64_t lda,
                                     void* stream, gcnb_graph** out) {
  GCNB_REQUIRE(out != nullptr, "graph_from_dense: out is null");
  *out = nullptr;
  GCNB_TRY(check_dims(n_rows, n_cols, 0));
  GCNB_TRY(gcnb_check_device());
  const int s = from_dense_impl(out, n_rows, n_cols, d_a, lda, (cudaStream_t)stream);
  GCNB_BUILD_EPILOGUE(s);
}

extern "C" int gcnb_graph_from_coo_f64(int64_t n_rows, int64_t n_cols, int64_t nnz, const int64_t* d_row,
                                       const int64_t* d_col, const double* d_val, void* stream, gcnb_graph** out) {
  GCNB_REQUIRE(out != nullptr, "graph_from_coo_f64: out is null");
  *out = nullptr;
  GCNB_TRY(check_dims(n_rows, n_cols, nnz));
  GCNB_REQUIRE((reinterpret_cast<uintptr_t>(d_val) & 7u) == 0, "graph_from_coo_f64: values not 8-byte aligned");
  GCNB_TRY(gcnb_check_device());
  *out = new_graph(n_rows, n_cols, nnz);
  GCNB_REQUIRE(*out != nullptr, "graph: host allocation failed");
  const int s = from_coo_impl(*out, d_row, d_col, nullptr, (cudaStream_t)stream, true, d_val);
  GCNB_BUILD_EPILOGUE(s);
}

extern "C" int gcnb_graph_from_csr_f64(int64_t n_rows, int64_t n_cols, int64_t nnz, const int64_t* d_crow,
                                       const int64_t* d_col, const double* d_val, void* stream, gcnb_graph** out) {
  GCNB_REQUIRE(out != nullptr, "graph_from_csr_f64: out is null");
  *out = nullptr;
  GCNB_TRY(check_dims(n_rows, n_cols, nnz));
  GCNB_REQUIRE((reinterpret_cast<uintptr_t>(d_val) & 7u) == 0, "graph_from_csr_f64: values not 8-byte aligned");
  GCNB_TRY(gcnb_check_device());
  *out = new_graph(n_rows, n_cols, nnz);
  GCNB_REQUIRE(*out != nullptr, "graph: host allocation failed");
  const int s = from_csr_impl(*out, d_crow, d_col, nullptr, (cudaStream_t)stream, true, d_val);
  GCNB_BUILD_EPILOGUE(s);
}

extern "C" int gcnb_graph_from_dense_f64(int64_t n_rows, int64_t n_cols, const double* d_a, int64_t lda, void* stream,
                                         gcnb_graph** out) {
  GCNB_REQUIRE(out != nullptr, "graph_from_dense_f64: out is null");
  *out = nullptr;
  GCNB_TRY(check_dims(n_rows, n_cols, 0));
  GCNB_TRY(gcnb_check_device());
  const int s = from_dense_f64_impl(out, n_rows, n_cols, d_a, lda, (cudaStream_t)stream);
  GCNB_BUILD_EPILOGUE(s);
}

extern "C" int gcnb_graph_block(const gcnb_graph* g, int transpose, int64_t r0, int64_t r1, int64_t c0,
                                int64_t c1, int64_t col_shift, int64_t n_cols_out, void* stream,
                                gcnb_graph** out) {
  GCNB_REQUIRE(out != nullptr, "graph_block: out is null");
  *out = nullptr;
  GCNB_REQUIRE(g != nullptr, "graph_block: null graph");
  GCNB_REQUIRE(!transpose || g->has_transpose, "graph_block: handle has no transpose");
  const CsrView& v = transpose ? g->bwd : g->fwd;
  GCNB_REQUIRE(0 <= r0 && r0 <= r1 && r1 <= v.n_rows, "graph_block: bad row range");
  GCNB_REQUIRE(0 <= c0 && c0 <= c1 && c1 <= v.n_cols, "graph_block: bad column range");
  GCNB_REQUIRE(col_shift >= 0 && n_cols_out >= (c1 - c0) + col_shift, "graph_block: bad column shift");
  GCNB_TRY(check_dims(r1 - r0, n_cols_out, 0));
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t nr = r1 - r0;
  auto impl = [&]() -> int {
    DevBuf counts, rowptr, temp, total;
    GCNB_TRY(counts.alloc((size_t)(nr + 1) * 4));
    GCNB_TRY(rowptr.alloc((size_t)(nr + 1) * 4));
    GCNB_TRY(total.alloc(8));
    GCNB_CUDA(cudaMemsetAsync(counts.p, 0, (size_t)(nr + 1) * 4, st));
    GCNB_CUDA(cudaMemsetAsync(total.p, 0, 8, st));
    if (nr > 0) {
      block_count_kernel<<<blocks_for(nr), kT, 0, st>>>(r0, nr, (int32_t)c0, (int32_t)c1, v.rowptr, v.col,
                                                        counts.as<int32_t>());
      sum_i32_kernel<<<blocks_for(nr), kT, 0, st>>>(counts.as<int32_t>(), nr, total.as<unsigned long long>());
      GCNB_LAUNCH_CHECK();
    }
    size_t tb = 0;
    GCNB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tb, counts.as<int32_t>(), rowptr.as<int32_t>(), (int)(nr + 1), st));
    GCNB_TRY(temp.alloc(tb));
    GCNB_CUDA(cub::DeviceScan::ExclusiveSum(temp.p, tb, counts.as<int32_t>(), rowptr.as<int32_t>(), (int)(nr + 1), st));
    int64_t nnz = 0;
    GCNB_CUDA(cudaMemcpyAsync(&nnz, total.p, 8, cudaMemcpyDeviceToHost, st));
    GCNB_CUDA(cudaStreamSynchronize(st));
    gcnb_graph* b = new_graph(nr, n_cols_out, nnz);
    GCNB_REQUIRE(b != nullptr, "graph: host allocation failed");
    *out = b;
    DevBuf rows32;
    GCNB_TRY(rows32.alloc((size_t)nnz * 4));
    GCNB_TRY(graph_alloc(b, &b->rowptr, nr + 1));
    GCNB_TRY(graph_alloc(b, &b->col, nnz));
    GCNB_TRY(graph_alloc(b, &b->val, nnz));
    GCNB_CUDA(cudaMemcpyAsync(b->rowptr, rowptr.p, (size_t)(nr + 1) * 4, cudaMemcpyDeviceToDevice, st));
    if (nr > 0 && nnz > 0) {
      block_fill_kernel<<<blocks_for(nr), kT, 0, st>>>(r0, nr, (int32_t)c0, (int32_t)c1, (int32_t)col_shift,
                                                       v.rowptr, v.col, v.val, b->rowptr, b->col, b->val,
                                                       rows32.as<int32_t>());
      GCNB_LAUNCH_CHECK();
    }
    return finalize(b, rows32.as<int32_t>(), st, /*with_transpose=*/false);
  };
  const int s = impl();
  GCNB_BUILD_EPILOGUE(s);
}

extern "C" int gcnb_graph_block_gathered(const gcnb_graph* g, int transpose, int64_t r0, int64_t r1, int n_parts,
                                         const int64_t* h_bounds, int64_t pad_rows, int exclude_part, void* stream,
                                         gcnb_graph** out) {
  GCNB_REQUIRE(n_parts >= 1 && n_parts <= 64, "graph_block_gathered: 1..64 parts");
  unsigned long long include = (n_parts == 64) ? ~0ull : ((1ull << n_parts) - 1ull);
  if (exclude_part >= 0 && exclude_part < n_parts) include &= ~(1ull << exclude_part);
  return gcnb_graph_block_sources(g, transpose, r0, r1, n_parts, h_bounds, pad_rows, include, stream, out);
}

extern "C" int gcnb_graph_block_sources(const gcnb_graph* g, int transpose, int64_t r0, int64_t r1, int n_parts,
                                        const int64_t* h_bounds, int64_t pad_rows, unsigned long long include_mask,
                                        void* stream, gcnb_graph** out) {
  GCNB_REQUIRE(out != nullptr, "graph_block_gathered: out is null");
  *out = nullptr;
  GCNB_REQUIRE(g != nullptr && h_bounds != nullptr && n_parts >= 1 && n_parts <= 64, "graph_block_gathered: bad argument");
  GCNB_REQUIRE(!transpose || g->has_transpose, "graph_block_gathered: handle has no transpose");
  const CsrView& v = transpose ? g->bwd : g->fwd;
  GCNB_REQUIRE(0 <= r0 && r0 <= r1 && r1 <= v.n_rows, "graph_block_gathered: bad row range");
  GCNB_REQUIRE(h_bounds[0] == 0 && h_bounds[n_parts] == v.n_cols, "graph_block_gathered: bounds must cover the columns");
  for (int q = 0; q < n_parts; ++q)
    GCNB_REQUIRE(h_bounds[q] <= h_bounds[q + 1] && h_bounds[q + 1] - h_bounds[q] <= pad_rows,
                 "graph_block_gathered: part %d larger than pad_rows", q);
  const int64_t n_cols_out = (int64_t)n_parts * pad_rows;
  GCNB_TRY(check_dims(r1 - r0, n_cols_out, 0));
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t nr = r1 - r0;
  auto impl = [&]() -> int {
    DevBuf counts, rowptr, temp, total, bounds;
    GCNB_TRY(counts.alloc((size_t)(nr + 1) * 4));
    GCNB_TRY(rowptr.alloc((size_t)(nr + 1) * 4));
    GCNB_TRY(total.alloc(8));
    GCNB_TRY(bounds.alloc((size_t)(n_parts + 1) * 8));
    GCNB_CUDA(cudaMemcpyAsync(bounds.p, h_bounds, (size_t)(n_parts + 1) * 8, cudaMemcpyHostToDevice, st));
    GCNB_CUDA(cudaMemsetAsync(counts.p, 0, (size_t)(nr + 1) * 4, st));
    GCNB_CUDA(cudaMemsetAsync(total.p, 0, 8, st));
    if (nr > 0) {
      gathered_count_kernel<<<blocks_for(nr), kT, 0, st>>>(r0, nr, n_parts, bounds.as<int64_t>(), include_mask,
                                                           v.rowptr, v.col, counts.as<int32_t>());
      sum_i32_kernel<<<blocks_for(nr), kT, 0, st>>>(counts.as<int32_t>(), nr, total.as<unsigned long long>());
      GCNB_LAUNCH_CHECK();
    }
    size_t tb = 0;
    GCNB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tb, counts.as<int32_t>(), rowptr.as<int32_t>(), (int)(nr + 1), st));
    GCNB_TRY(temp.alloc(tb));
    GCNB_CUDA(cub::DeviceScan::ExclusiveSum(temp.p, tb, counts.as<int32_t>(), rowptr.as<int32_t>(), (int)(nr + 1), st));
    int64_t nnz = 0;
    GCNB_CUDA(cudaMemcpyAsync(&nnz, total.p, 8, cudaMemcpyDeviceToHost, st));
    GCNB_CUDA(cudaStreamSynchronize(st));
    gcnb_graph* b = new_graph(nr, n_cols_out, nnz);
    GCNB_REQUIRE(b != nullptr, "graph: host allocation failed");
    *out = b;
    DevBuf rows32;
    GCNB_TRY(rows32.alloc((size_t)nnz * 4));
    GCNB_TRY(graph_alloc(b, &b->rowptr, nr + 1));
    GCNB_TRY(graph_alloc(b, &b->col, nnz));
    GCNB_TRY(graph_alloc(b, &b->val, nnz));
    GCNB_CUDA(cudaMemcpyAsync(b->rowptr, rowptr.p, (size_t)(nr + 1) * 4, cudaMemcpyDeviceToDevice, st));
    if (nr > 0 && nnz > 0) {
      gathered_fill_kernel<<<blocks_for(nr), kT, 0, st>>>(r0, nr, n_parts, bounds.as<int64_t>(), include_mask, pad_rows,
                                                          v.rowptr, v.col, v.val, b->rowptr, b->col, b->val,
                                                          rows32.as<int32_t>());
      GCNB_LAUNCH_CHECK();
    }
    return finalize(b, rows32.as<int32_t>(), st, /*with_transpose=*/false);
  };
  const int s = impl();
  GCNB_BUILD_EPILOGUE(s);
}

extern "C" int gcnb_graph_get_info(const gcnb_graph* g, gcnb_graph_info* info) {
  GCNB_REQUIRE(g != nullptr && info != nullptr, "graph_get_info: null argument");
  info->n_rows = g->n_rows;
  info->n_cols = g->n_cols;
  info->nnz = g->nnz;
  for (int b = 0; b < GCNB_NUM_BINS; ++b) {
    info->bin_rows[b] = g->fwd.bin_rows[b];
    info->t_bin_rows[b] = g->bwd.bin_rows[b];
  }
  info->max_degree = g->fwd.max_degree;
  info->t_max_degree = g->bwd.max_degree;
  info->n_long_chunks = g->fwd.n_long_chunks;
  info->t_n_long_chunks = g->bwd.n_long_chunks;
  info->pattern_symmetric = g->pattern_symmetric ? 1 : 0;
  info->dense_route = g->dense_fwd ? 1 : 0;
  info->device_bytes = g->device_bytes;
  info->d_rowptr = g->rowptr;
  info->d_col = g->col;
  info->d_val = g->val;
  info->d_t_rowptr = g->t_rowptr;
  info->d_t_col = g->t_col;
  info->d_t_val = g->t_val;
  return GCNB_OK;
}

extern "C" int gcnb_graph_export_coo(const gcnb_graph* g, int64_t* d_indices, float* d_values, void* stream) {
  GCNB_REQUIRE(g != nullptr, "graph_export_coo: null graph");
  if (g->nnz == 0) return GCNB_OK;
  GCNB_REQUIRE(d_indices != nullptr && d_values != nullptr, "graph_export_coo: null output");
  export_coo_kernel<<<blocks_for(g->nnz), kT, 0, (cudaStream_t)stream>>>(g->nnz, g->n_rows, g->rowptr, g->col,
                                                                         g->val, d_indices, d_values);
  GCNB_LAUNCH_CHECK();
  return GCNB_OK;
}

extern "C" int gcnb_graph_export_csr(const gcnb_graph* g, int transpose, int32_t* d_rowptr, int32_t* d_col,
                                     float* d_val, void* stream) {
  GCNB_REQUIRE(g != nullptr && d_rowptr != nullptr, "graph_export_csr: null argument");
  const CsrView& v = transpose ? g->bwd : g->fwd;
  cudaStream_t st = (cudaStream_t)stream;
  GCNB_CUDA(cudaMemcpyAsync(d_rowptr, v.rowptr, (size_t)(v.n_rows + 1) * 4, cudaMemcpyDeviceToDevice, st));
  if (v.nnz > 0) {
    GCNB_REQUIRE(d_col != nullptr && d_val != nullptr, "graph_export_csr: null output");
    GCNB_CUDA(cudaMemcpyAsync(d_col, v.col, (size_t)v.nnz * 4, cudaMemcpyDeviceToDevice, st));
    GCNB_CUDA(cudaMemcpyAsync(d_val, v.val, (size_t)v.nnz * 4, cudaMemcpyDeviceToDevice, st));
  }
  return GCNB_OK;
}

extern "C" int gcnb_graph_export_csr_f64(const gcnb_graph* g, int transpose, int32_t* d_rowptr, int32_t* d_col,
                                         double* d_val64, void* stream) {
  GCNB_REQUIRE(g != nullptr && d_rowptr != nullptr, "graph_export_csr_f64: null argument");
  if (g->val64 == nullptr) {
    set_error("graph_export_csr_f64: the handle has no fp64 values (it was built from fp32 data)");
    return GCNB_E_UNSUPPORTED;
  }
  GCNB_REQUIRE(!transpose || g->has_transpose, "graph_export_csr_f64: handle has no transpose");
  const CsrView& v = transpose ? g->bwd : g->fwd;
  cudaStream_t st = (cudaStream_t)stream;
  GCNB_CUDA(cudaMemcpyAsync(d_rowptr, v.rowptr, (size_t)(v.n_rows + 1) * 4, cudaMemcpyDeviceToDevice, st));
  if (v.nnz > 0) {
    GCNB_REQUIRE(d_col != nullptr && d_val64 != nullptr, "graph_export_csr_f64: null output");
    GCNB_CUDA(cudaMemcpyAsync(d_col, v.col, (size_t)v.nnz * 4, cudaMemcpyDeviceToDevice, st));
    GCNB_CUDA(cudaMemcpyAsync(d_val64, transpose ? g->t_val64 : g->val64, (size_t)v.nnz * 8, cudaMemcpyDeviceToDevice, st));
  }
  return GCNB_OK;
}
