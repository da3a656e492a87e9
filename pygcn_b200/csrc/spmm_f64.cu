// fp64 tier: SpMM over the fp64 values of a graph handle (val64 / t_val64) and the fp64 column sums of the layer's
// backward.  These kernels share nothing with the fp32 ones, so the fp32 SASS is untouched by this file.
//
// SpMM: a group of G lanes per row (G = 32 for panels of more than 32 columns; 4 / 8 / 8 lanes -- several rows per warp
// -- for panels of <= 8 / 16 / 32 columns; panels wider than 128 columns run in passes of 128).  Lane l of a group owns
// the column pairs l, l + G, ... and holds CH of them in registers; a stored entry costs one 16-byte load per pair when the panel rows are 16-byte aligned (ldb even), two 8-byte loads
// otherwise.  Entries are read G at a time, one per lane, and broadcast with shuffles.  Rows of more than 1024 entries
// are skipped here and run on the handle's long-row schedule: one warp per 1024-entry chunk writes an fp64 partial row
// to the workspace, and an ordered fix-up adds a row's partials chunk by chunk -- no atomics, so every result is
// bit-reproducible.
#include "common.cuh"

namespace gcnb {
namespace {

constexpr int kThreads = 256;

__device__ __forceinline__ double finish64(double acc, const Epilogue64& ep, int64_t row, int64_t j, const double* out,
                                           int64_t ldo) {
  if (ep.accumulate) acc += out[row * ldo + j];
  if (ep.bias) acc += ep.bias[j];
  if (ep.relu) acc = fmax(acc, 0.0);
  if (ep.mask) acc = ep.mask[row * ep.ld_mask + j] ? acc * ep.mask_scale : 0.0;
  return acc;
}

// acc[u] += sum over entries [s, e) of val * b[col, j + 2 G u .. + 1], j = 2 * lane (columns past f are read only
// when they are panel padding inside ldb, and never stored)
// U > 1 (16-byte path): the gathers of U entries are issued before any of them is added, so U * CH loads per lane are
// in flight; the adds still run entry by entry, so the result does not depend on U.
template <int G, int CH, bool VEC, int U>
__device__ __forceinline__ void gather_range(double (&acc)[CH][2], int s, int e, int lane, unsigned gmask,
                                             const int32_t* __restrict__ col, const double* __restrict__ val,
                                             const double* __restrict__ b, int64_t ldb, int64_t j0, int64_t f) {
  for (int p0 = s; p0 < e; p0 += G) {
    int c_mine = 0;
    double v_mine = 0.0;
    if (p0 + lane < e) {
      c_mine = __ldg(col + p0 + lane);
      v_mine = __ldg(val + p0 + lane);
    }
    const int cnt = min(G, e - p0);
    int t = 0;
    if (VEC && U > 1) {
      for (; t + U <= cnt; t += U) {
        double v[U];
        double2 x[U][CH];
#pragma unroll
        for (int q = 0; q < U; ++q) {
          const int c = __shfl_sync(gmask, c_mine, t + q, G);
          v[q] = __shfl_sync(gmask, v_mine, t + q, G);
          const double* src = b + (int64_t)c * ldb;
#pragma unroll
          for (int u = 0; u < CH; ++u) {
            const int64_t j = j0 + 2 * lane + 2 * G * u;
            x[q][u] = j < f ? __ldg(reinterpret_cast<const double2*>(src + j)) : make_double2(0.0, 0.0);
          }
        }
#pragma unroll
        for (int q = 0; q < U; ++q)
#pragma unroll
          for (int u = 0; u < CH; ++u) {
            acc[u][0] = fma(v[q], x[q][u].x, acc[u][0]);
            acc[u][1] = fma(v[q], x[q][u].y, acc[u][1]);
          }
      }
    }
#pragma unroll 1  // one entry in flight per lane measured fastest on wide panels (products F = 256: 16.2 ms, 2 per lane
    for (; t < cnt; ++t) {  // 17.0-17.3 ms, 4 per lane 20.5 ms; B200 at 1000 W, profiles/r03_fp64_spmm_variants.txt)
      const int c = __shfl_sync(gmask, c_mine, t, G);
      const double v = __shfl_sync(gmask, v_mine, t, G);
      const double* src = b + (int64_t)c * ldb;
#pragma unroll
      for (int u = 0; u < CH; ++u) {
        const int64_t j = j0 + 2 * lane + 2 * G * u;
        if (j < f) {
          if (VEC) {
            const double2 x = __ldg(reinterpret_cast<const double2*>(src + j));
            acc[u][0] = fma(v, x.x, acc[u][0]);
            acc[u][1] = fma(v, x.y, acc[u][1]);
          } else {
            acc[u][0] = fma(v, __ldg(src + j), acc[u][0]);
            if (j + 1 < f) acc[u][1] = fma(v, __ldg(src + j + 1), acc[u][1]);
          }
        }
      }
    }
  }
}

template <int G, int CH, bool VEC, int U>
__global__ void __launch_bounds__(kThreads) spmm_f64_rows_kernel(int64_t n_rows, const int32_t* __restrict__ rowptr,
                                                                const int32_t* __restrict__ col,
                                                                const double* __restrict__ val, const double* __restrict__ b,
                                                                int64_t ldb, int64_t f, Epilogue64 ep, double* out,
                                                                int64_t ldo) {
  const int64_t row = ((int64_t)blockIdx.x * kThreads + threadIdx.x) / G;
  const int lane = threadIdx.x % G;
  if (row >= n_rows) return;  // whole groups leave together
  const int s = rowptr[row], e = rowptr[row + 1];
  if (e - s >= kLongRowThreshold) return;  // long-row schedule
  const unsigned gmask = (G == 32) ? 0xffffffffu : (((1u << G) - 1u) << ((threadIdx.x & 31) / G * G));
  for (int64_t j0 = 0; j0 < f; j0 += 2 * G * CH) {
    double acc[CH][2] = {};
    gather_range<G, CH, VEC, U>(acc, s, e, lane, gmask, col, val, b, ldb, j0, f);
#pragma unroll
    for (int u = 0; u < CH; ++u)
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int64_t j = j0 + 2 * lane + 2 * G * u + h;
        if (j < f) out[row * ldo + j] = finish64(acc[u][h], ep, row, j, out, ldo);
      }
  }
}

// one warp per chunk of a long row: partial[chunk, 0:f] = sum over the chunk's entries
template <bool VEC>
__global__ void __launch_bounds__(kThreads, 4) spmm_f64_long_chunk_kernel(
    int64_t n_chunks, int64_t n_long, const int32_t* __restrict__ long_rows, const int32_t* __restrict__ chunk_ptr,
    const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, const double* __restrict__ val,
    const double* __restrict__ b, int64_t ldb, int64_t f, double* __restrict__ partial) {
  const int64_t chunk = ((int64_t)blockIdx.x * kThreads + threadIdx.x) / 32;
  const int lane = threadIdx.x % 32;
  if (chunk >= n_chunks) return;
  int64_t lo = 0, hi = n_long;  // the long row whose chunks hold this one: last q with chunk_ptr[q] <= chunk
  while (hi - lo > 1) {
    const int64_t mid = (lo + hi) >> 1;
    if (chunk_ptr[mid] <= chunk) lo = mid; else hi = mid;
  }
  const int row = long_rows[lo];
  const int s = rowptr[row] + (int)(chunk - chunk_ptr[lo]) * kLongChunk;
  const int e = min(s + kLongChunk, rowptr[row + 1]);
  for (int64_t j0 = 0; j0 < f; j0 += 64) {
    double acc[1][2] = {};
    gather_range<32, 1, VEC, 1>(acc, s, e, lane, 0xffffffffu, col, val, b, ldb, j0, f);
    const int64_t j = j0 + 2 * lane;
    if (j < f) partial[chunk * f + j] = acc[0][0];
    if (j + 1 < f) partial[chunk * f + j + 1] = acc[0][1];
  }
}

// out[long row, j] = epilogue(sum of the row's chunk partials, chunk by chunk)
__global__ void __launch_bounds__(kThreads) spmm_f64_long_fixup_kernel(int64_t n_long, const int32_t* __restrict__ long_rows,
                                                                      const int32_t* __restrict__ chunk_ptr,
                                                                      const double* __restrict__ partial, int64_t f,
                                                                      Epilogue64 ep, double* out, int64_t ldo) {
  const int64_t j = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  if (j >= f) return;
  for (int64_t q = blockIdx.y; q < n_long; q += gridDim.y) {  // any number of long rows
    double acc = 0.0;
    for (int c = chunk_ptr[q]; c < chunk_ptr[q + 1]; ++c) acc += partial[(int64_t)c * f + j];
    const int64_t row = long_rows[q];
    out[row * ldo + j] = finish64(acc, ep, row, j, out, ldo);
  }
}

template <int G, int CH, int U = 1>
int launch_rows(const CsrView& a, const double* val, const double* b, int64_t ldb, int64_t f, bool vec,
                const Epilogue64& ep, double* out, int64_t ldo, cudaStream_t st) {
  const unsigned blocks = (unsigned)ceil_div(a.n_rows * G, kThreads);
  if (vec)
    spmm_f64_rows_kernel<G, CH, true, U><<<blocks, kThreads, 0, st>>>(a.n_rows, a.rowptr, a.col, val, b, ldb, f, ep, out, ldo);
  else
    spmm_f64_rows_kernel<G, CH, false, 1><<<blocks, kThreads, 0, st>>>(a.n_rows, a.rowptr, a.col, val, b, ldb, f, ep, out,
                                                                       ldo);
  GCNB_LAUNCH_CHECK();
  return GCNB_OK;
}

// -------------------------------------------------------------------------------- column sums
// Block = 32 columns x 8 row lanes over one slab of rows; each lane adds its rows in order, the 8 lanes are added in
// order, and the slab partials are added slab by slab: a fixed order, so the sums are reproducible.
constexpr int kColsumMaxSlabs = 512;
constexpr int kColsumRowsPerSlab = 256;

int64_t colsum_f64_slabs(int64_t n_rows) {
  const int64_t s = ceil_div(n_rows, kColsumRowsPerSlab);
  return s < 1 ? 1 : (s > kColsumMaxSlabs ? kColsumMaxSlabs : s);
}

__global__ void __launch_bounds__(kThreads) colsum_f64_partial_kernel(
    int64_t n_rows, int64_t f, int64_t rows_per_slab, const double* __restrict__ g, int64_t ldg,
    const double* __restrict__ y, int64_t ldy, double* gm, int64_t ldgm, const uint8_t* __restrict__ mask,
    int64_t ld_mask, double mask_scale, double* __restrict__ partial) {
  __shared__ double red[8][32];
  const int64_t j = (int64_t)blockIdx.x * 32 + threadIdx.x;
  const int64_t r0 = (int64_t)blockIdx.y * rows_per_slab;
  const int64_t r1 = min(r0 + rows_per_slab, n_rows);
  double s = 0.0;
  if (j < f) {
    for (int64_t r = r0 + threadIdx.y; r < r1; r += 8) {
      double v = g[r * ldg + j];
      if (mask != nullptr) v = mask[r * ld_mask + j] ? v * mask_scale : 0.0;  // dropout came last in the forward
      if (y != nullptr) v = (y[r * ldy + j] > 0.0) ? v : 0.0;
      if (gm != nullptr) gm[r * ldgm + j] = v;
      s += v;
    }
  }
  red[threadIdx.y][threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.y == 0 && j < f) {
    double t = red[0][threadIdx.x];
#pragma unroll
    for (int i = 1; i < 8; ++i) t += red[i][threadIdx.x];
    partial[(int64_t)blockIdx.y * f + j] = t;
  }
}

__global__ void __launch_bounds__(kThreads) colsum_f64_reduce_kernel(int64_t n_slabs, int64_t f,
                                                                    const double* __restrict__ partial,
                                                                    double* __restrict__ out) {
  const int64_t j = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  if (j >= f) return;
  double t = partial[j];
  for (int64_t s = 1; s < n_slabs; ++s) t += partial[s * f + j];
  out[j] = t;
}

}  // namespace

size_t spmm_f64_workspace_bytes(const CsrView& a, int64_t f) {
  if (a.n_long_chunks == 0 || f <= 0) return 0;
  return ((size_t)a.n_long_chunks * (size_t)f * sizeof(double) + 255) & ~(size_t)255;
}

int spmm_f64_launch(const CsrView& a, const double* val, const double* b, int64_t ldb, int64_t f,
                    const Epilogue64& ep, double* out, int64_t ldo, void* ws, size_t ws_bytes, cudaStream_t st) {
  GCNB_REQUIRE(val != nullptr, "spmm_f64: the graph handle has no fp64 values (build it from fp64 data)");
  GCNB_REQUIRE(f >= 0 && f < (1ll << 31), "spmm_f64: width out of range");
  if (a.n_rows == 0 || f == 0) return GCNB_OK;
  GCNB_REQUIRE(out != nullptr && ldo >= f, "spmm_f64: null output or ldo < f");
  GCNB_REQUIRE(a.nnz == 0 || (b != nullptr && ldb >= f), "spmm_f64: null dense operand or ldb < f");
  GCNB_REQUIRE((double)a.n_cols * (double)(ldb > 0 ? ldb : 1) < 9.2e18 && (double)a.n_rows * (double)ldo < 9.2e18,
               "spmm_f64: operand extent overflows 64-bit indexing");
  GCNB_REQUIRE(ep.bias == nullptr || (reinterpret_cast<uintptr_t>(ep.bias) & 7u) == 0, "spmm_f64: bias not 8-byte aligned");
  GCNB_REQUIRE(ep.mask == nullptr || ep.ld_mask >= f, "spmm_f64: dropout mask leading dimension smaller than width");
  GCNB_REQUIRE(((reinterpret_cast<uintptr_t>(b) | reinterpret_cast<uintptr_t>(out)) & 7u) == 0,
               "spmm_f64: operands must be 8-byte aligned");
  const size_t need = spmm_f64_workspace_bytes(a, f);
  GCNB_REQUIRE(ws_bytes >= need && (need == 0 || ws != nullptr), "spmm_f64: workspace too small (%zu < %zu)", ws_bytes, need);
  GCNB_REQUIRE((reinterpret_cast<uintptr_t>(ws) & 7u) == 0, "spmm_f64: workspace not 8-byte aligned");
  const bool vec = ldb % 2 == 0 && (reinterpret_cast<uintptr_t>(b) & 15u) == 0;
  if (f <= 8) GCNB_TRY((launch_rows<4, 1>(a, val, b, ldb, f, vec, ep, out, ldo, st)));
  else if (f <= 16) GCNB_TRY((launch_rows<8, 1>(a, val, b, ldb, f, vec, ep, out, ldo, st)));
  else if (f <= 32) GCNB_TRY((launch_rows<8, 2, 4>(a, val, b, ldb, f, vec, ep, out, ldo, st)));  // CBG F = 32: 0.240 ms
  // (16 lanes x 1 pair: 0.27 ms; with 1 entry in flight: 0.28 ms)
  else if (f <= 64) GCNB_TRY((launch_rows<32, 1>(a, val, b, ldb, f, vec, ep, out, ldo, st)));
  else if (f <= 128) GCNB_TRY((launch_rows<32, 2>(a, val, b, ldb, f, vec, ep, out, ldo, st)));
  else {
    // wider panels in passes of 128 columns: each pass re-reads the (col, val) stream but gathers half-width rows
    // (products F = 256: 16.2 ms, against 20.3 ms in one pass of 256 columns and 20.9 ms in passes of 64, with the loads
    // of that measurement; profiles/r03_fp64_spmm_variants.txt)
    for (int64_t f0 = 0; f0 < f; f0 += 128) {
      Epilogue64 e = ep;
      if (e.bias) e.bias += f0;
      if (e.mask) e.mask += f0;
      const int64_t fw = f - f0 < 128 ? f - f0 : 128;
      if (fw <= 64) GCNB_TRY((launch_rows<32, 1>(a, val, b + f0, ldb, fw, vec, e, out + f0, ldo, st)));
      else GCNB_TRY((launch_rows<32, 2>(a, val, b + f0, ldb, fw, vec, e, out + f0, ldo, st)));
    }
  }
  if (a.n_long_chunks > 0) {
    double* partial = reinterpret_cast<double*>(ws);
    const unsigned blocks = (unsigned)ceil_div(a.n_long_chunks * 32, kThreads);
    if (vec)
      spmm_f64_long_chunk_kernel<true><<<blocks, kThreads, 0, st>>>(a.n_long_chunks, a.n_long_rows, a.long_rows,
                                                                    a.long_chunk_ptr, a.rowptr, a.col, val, b, ldb, f,
                                                                    partial);
    else
      spmm_f64_long_chunk_kernel<false><<<blocks, kThreads, 0, st>>>(a.n_long_chunks, a.n_long_rows, a.long_rows,
                                                                     a.long_chunk_ptr, a.rowptr, a.col, val, b, ldb, f,
                                                                     partial);
    GCNB_LAUNCH_CHECK();
    const unsigned gy = (unsigned)(a.n_long_rows < 65535 ? a.n_long_rows : 65535);
    spmm_f64_long_fixup_kernel<<<dim3((unsigned)ceil_div(f, kThreads), gy), kThreads, 0, st>>>(
        a.n_long_rows, a.long_rows, a.long_chunk_ptr, partial, f, ep, out, ldo);
    GCNB_LAUNCH_CHECK();
  }
  return GCNB_OK;
}

size_t colsum_f64_workspace_bytes(int64_t n_rows, int64_t f) {
  return (size_t)colsum_f64_slabs(n_rows) * (size_t)(f > 0 ? f : 0) * sizeof(double) + 256;
}

int colsum_f64_launch(int64_t n_rows, int64_t f, const double* g, int64_t ldg, const double* y, int64_t ldy, double* gm,
                      int64_t ldgm, double* out, void* ws, size_t ws_bytes, cudaStream_t st, const uint8_t* mask,
                      int64_t ld_mask, double mask_scale) {
  GCNB_REQUIRE(n_rows >= 0 && f > 0 && f < (1ll << 31) && (int64_t)ceil_div(f, 32) < (1ll << 31),
               "colsum_f64: shape out of range");
  GCNB_REQUIRE(out != nullptr || gm != nullptr, "colsum_f64: null output (and no gm to stage)");
  GCNB_REQUIRE(n_rows == 0 || (g != nullptr && ldg >= f), "colsum_f64: bad gradient operand");
  GCNB_REQUIRE(y == nullptr || (gm != nullptr && ldy >= f), "colsum_f64: bad mask operands");
  GCNB_REQUIRE(gm == nullptr || ldgm >= f, "colsum_f64: ldgm < width");
  GCNB_REQUIRE(mask == nullptr || (gm != nullptr && ld_mask >= f), "colsum_f64: dropout mask needs gm and ld_mask >= width");
  GCNB_REQUIRE(((reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(gm) |
                 reinterpret_cast<uintptr_t>(out)) & 7u) == 0, "colsum_f64: operands must be 8-byte aligned");
  const size_t need = colsum_f64_workspace_bytes(n_rows, f);
  GCNB_REQUIRE(ws != nullptr && ws_bytes >= need, "colsum_f64: workspace too small (%zu < %zu)", ws_bytes, need);
  GCNB_REQUIRE((reinterpret_cast<uintptr_t>(ws) & 7u) == 0, "colsum_f64: workspace not 8-byte aligned");
  const int64_t slabs = colsum_f64_slabs(n_rows);
  const int64_t rows_per_slab = n_rows > 0 ? ceil_div(n_rows, slabs) : 1;
  double* partial = reinterpret_cast<double*>(ws);
  colsum_f64_partial_kernel<<<dim3((unsigned)ceil_div(f, 32), (unsigned)slabs), dim3(32, 8), 0, st>>>(
      n_rows, f, rows_per_slab, g, ldg, y, ldy, gm, ldgm, mask, ld_mask, mask_scale, partial);
  GCNB_LAUNCH_CHECK();
  if (out != nullptr) {  // (null: only the staged / masked copy gm is wanted)
    colsum_f64_reduce_kernel<<<(unsigned)ceil_div(f, kThreads), kThreads, 0, st>>>(slabs, f, partial, out);
    GCNB_LAUNCH_CHECK();
  }
  return GCNB_OK;
}

}  // namespace gcnb
