// Column sum of the upstream gradient (db of `output + self.bias`, pygcn/layers.py:36), with
// the ReLU mask of the fused epilogue applied on the fly when requested, plus the L2 flush
// helper the benchmark uses.  Two-phase deterministic reduction (no atomics).
#include "common.cuh"
#include "ptx.cuh"

namespace gcnb {
namespace {

constexpr int kThreads = 256;
constexpr int kMaxBlocks = 4 * kNumSMs;

// Phase 1: block b reduces rows [b*rows_per_block, ...) -> partial[b][0:f] (fp64)
__global__ void __launch_bounds__(kThreads)
colsum_partial_kernel(int64_t n_rows, int f, int cw, int64_t rows_per_block,
                      const float* __restrict__ g, int64_t ldg, const float* __restrict__ y,
                      int64_t ldy, float* __restrict__ gm, int64_t ldgm,
                      double* __restrict__ partial, const uint8_t* __restrict__ mask, int64_t ld_mask,
                      float mask_scale) {
  // (fp64 accumulators AND fp64 block partials: a column of the upstream gradient is 10^6 terms of either sign that
  // cancel to ~sqrt(N) of their mass; the kernel is memory-bound, the DADDs are free, and db then carries fp32
  // rounding of the RESULT only -- a partial rounded to fp32 would lose what the other blocks' partials cancel)
  __shared__ double red[kThreads];
  const int tx = threadIdx.x % cw;  // column lane
  const int ty = threadIdx.x / cw;  // row lane
  const int rl = kThreads / cw;
  const int64_t r0 = (int64_t)blockIdx.x * rows_per_block;
  const int64_t r1 = (r0 + rows_per_block < n_rows) ? (r0 + rows_per_block) : n_rows;
  for (int j0 = 0; j0 < f; j0 += cw) {
    const int j = j0 + tx;
    double acc = 0.0;
    if (j < f) {
      int64_t r = r0 + ty;
      double a4[4] = {0.0, 0.0, 0.0, 0.0};
      for (; r + 3 * rl < r1; r += 4 * rl) {  // four rows in flight per thread
        float v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = g[(r + u * rl) * ldg + j];
        if (mask != nullptr) {  // backward of the dropout epilogue comes first (it was applied last)
#pragma unroll
          for (int u = 0; u < 4; ++u) v[u] = mask[(r + u * rl) * ld_mask + j] ? v[u] * mask_scale : 0.f;
        }
        if (y != nullptr) {
#pragma unroll
          for (int u = 0; u < 4; ++u) v[u] = (y[(r + u * rl) * ldy + j] > 0.f) ? v[u] : 0.f;
        }
        if (gm != nullptr) {
#pragma unroll
          for (int u = 0; u < 4; ++u) gm[(r + u * rl) * ldgm + j] = v[u];
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) a4[u] += v[u];
      }
      for (; r < r1; r += rl) {
        float v = g[r * ldg + j];
        if (mask != nullptr) v = mask[r * ld_mask + j] ? v * mask_scale : 0.f;
        if (y != nullptr) v = (y[r * ldy + j] > 0.f) ? v : 0.f;
        if (gm != nullptr) gm[r * ldgm + j] = v;  // masked gradient, or a plain copy when y == NULL
        a4[0] += v;
      }
      acc = (a4[0] + a4[1]) + (a4[2] + a4[3]);
    }
    red[threadIdx.x] = acc;
    __syncthreads();
    if (ty == 0 && j < f) {
      double s = 0.0;
      for (int t = 0; t < rl; ++t) s += red[t * cw + tx];
      partial[(int64_t)blockIdx.x * f + j] = s;
    }
    __syncthreads();
  }
}

// Vectorised single-launch variant (f % 4 == 0, 16-byte aligned operands): every thread owns one float4
// column chunk and walks rows with four 16-byte loads in flight; the CTA's partial sums go to scratch and
// the LAST CTA to arrive (atomic ticket) adds all partials in block order -- one launch instead of two,
// still run-to-run deterministic (the order of the final additions is fixed, only who does them varies).
__global__ void __launch_bounds__(kThreads)
colsum_vec_kernel(int64_t n_rows, int f4, int cw, int64_t rows_per_block, const float4* __restrict__ g, int64_t ldg4,
                  const float4* __restrict__ y, int64_t ldy4, float4* __restrict__ gm, int64_t ldgm4,
                  double2* __restrict__ partial, unsigned int* __restrict__ ticket, float* __restrict__ out,
                  const uchar4* __restrict__ mask, int64_t ld_mask4, float mask_scale) {
  __shared__ double red[kThreads][4];  // fp64 accumulation and fp64 partials, see colsum_partial_kernel
  __shared__ bool is_last;
  const int tx = threadIdx.x % cw;  // float4 column chunk
  const int ty = threadIdx.x / cw;  // row lane
  const int rl = kThreads / cw;
  const int64_t r0 = (int64_t)blockIdx.x * rows_per_block;
  const int64_t r1 = (r0 + rows_per_block < n_rows) ? (r0 + rows_per_block) : n_rows;
  auto load = [&](int64_t r) {
    float4 v = g[r * ldg4 + tx];
    if (mask != nullptr) {  // backward of the dropout epilogue comes first (it was applied last)
      const uchar4 m = mask[r * ld_mask4 + tx];
      v.x = m.x ? v.x * mask_scale : 0.f; v.y = m.y ? v.y * mask_scale : 0.f;
      v.z = m.z ? v.z * mask_scale : 0.f; v.w = m.w ? v.w * mask_scale : 0.f;
    }
    if (y != nullptr) {
      const float4 o = y[r * ldy4 + tx];
      v.x = o.x > 0.f ? v.x : 0.f; v.y = o.y > 0.f ? v.y : 0.f;
      v.z = o.z > 0.f ? v.z : 0.f; v.w = o.w > 0.f ? v.w : 0.f;
    }
    if (gm != nullptr) gm[r * ldgm4 + tx] = v;  // masked gradient, or a plain copy when y == NULL
    return v;
  };
  double acc[4] = {0.0, 0.0, 0.0, 0.0};
  if (tx < f4) {
    int64_t r = r0 + ty;
    for (; r + 3 * rl < r1; r += 4 * rl) {
      float4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u] = load(r + u * rl);
#pragma unroll
      for (int u = 0; u < 4; ++u) { acc[0] += v[u].x; acc[1] += v[u].y; acc[2] += v[u].z; acc[3] += v[u].w; }
    }
    for (; r < r1; r += rl) {
      const float4 v = load(r);
      acc[0] += v.x; acc[1] += v.y; acc[2] += v.z; acc[3] += v.w;
    }
  }
#pragma unroll
  for (int c = 0; c < 4; ++c) red[threadIdx.x][c] = acc[c];
  __syncthreads();
  if (ty == 0 && tx < f4) {
    double s[4] = {0.0, 0.0, 0.0, 0.0};
    for (int t = 0; t < rl; ++t)
#pragma unroll
      for (int c = 0; c < 4; ++c) s[c] += red[t * cw + tx][c];
    partial[2 * ((int64_t)blockIdx.x * f4 + tx)] = make_double2(s[0], s[1]);
    partial[2 * ((int64_t)blockIdx.x * f4 + tx) + 1] = make_double2(s[2], s[3]);
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) is_last = (atomicAdd(ticket, 1u) == gridDim.x - 1);
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  // final pass: row lane ty adds the partials of blocks ty, ty + rl, ... ; then the lanes in order
#pragma unroll
  for (int c = 0; c < 4; ++c) acc[c] = 0.0;
  if (tx < f4) {
    for (int b = ty; b < (int)gridDim.x; b += rl) {
      const double2 v = partial[2 * ((int64_t)b * f4 + tx)], w = partial[2 * ((int64_t)b * f4 + tx) + 1];
      acc[0] += v.x; acc[1] += v.y; acc[2] += w.x; acc[3] += w.y;
    }
  }
#pragma unroll
  for (int c = 0; c < 4; ++c) red[threadIdx.x][c] = acc[c];
  __syncthreads();
  if (ty == 0 && tx < f4) {
    double s[4] = {0.0, 0.0, 0.0, 0.0};
    for (int t = 0; t < rl; ++t)
#pragma unroll
      for (int c = 0; c < 4; ++c) s[c] += red[t * cw + tx][c];
    reinterpret_cast<float4*>(out)[tx] = make_float4((float)s[0], (float)s[1], (float)s[2], (float)s[3]);
  }
}

// Lane ty of a part sum adds parts ty, ty + lanes, ...: four loads in flight, added in a fixed order (T = float for
// the tiles of a split product, double for the column-sum partials).
template <typename T, int kLanes>
__device__ __forceinline__ T sum_parts(const T* __restrict__ p, int64_t stride, int64_t i, int n_parts, int ty) {
  T a0 = 0, a1 = 0, a2 = 0, a3 = 0;
  int s = ty;
  for (; s + 3 * kLanes < n_parts; s += 4 * kLanes) {
    a0 += p[(int64_t)s * stride + i];
    a1 += p[(int64_t)(s + kLanes) * stride + i];
    a2 += p[(int64_t)(s + 2 * kLanes) * stride + i];
    a3 += p[(int64_t)(s + 3 * kLanes) * stride + i];
  }
  for (; s < n_parts; s += kLanes) a0 += p[(int64_t)s * stride + i];
  return (a0 + a1) + (a2 + a3);
}

// out[i / n, i % n] = sum over parts of the fp32 partial[s][i] for i < m * n, and -- when xout is given -- one more
// row: xout[j] = sum over parts of the fp64 xpart[s][j], rounded to fp32 once (column sums).  32 outputs x 8
// part-lanes per CTA, fixed-order tree (an fp32 lane sum goes through the fp64 shared array unchanged).
__global__ void __launch_bounds__(kThreads)
reduce_partials_kernel(int64_t total, int64_t n, int n_parts, const float* __restrict__ partial,
                       float* __restrict__ out, int64_t ldo, int64_t m, const double* __restrict__ xpart,
                       float* __restrict__ xout) {
  __shared__ double red[8][33];
  const int tx = threadIdx.x & 31;
  const int ty = threadIdx.x >> 5;
  const int64_t i = (int64_t)blockIdx.x * 32 + tx;
  const int64_t mn = m * n;
  double acc = 0.0;
  if (i < total) acc = (i < mn) ? (double)sum_parts<float, 8>(partial, mn, i, n_parts, ty)
                                : sum_parts<double, 8>(xpart, n, i - mn, n_parts, ty);
  red[ty][tx] = acc;
  __syncthreads();
  if (ty == 0 && i < total) {
    if (i < mn) {
      float v = 0.f;
#pragma unroll
      for (int t = 0; t < 8; ++t) v += (float)red[t][tx];
      out[(i / n) * ldo + (i % n)] = v;
    } else {
      double v = 0.0;
#pragma unroll
      for (int t = 0; t < 8; ++t) v += red[t][tx];
      xout[i - mn] = (float)v;
    }
  }
}

// The same sum for many parts (split-K over 148-296 CTAs): 32 part-lanes per output float4, so a lane adds ~10
// parts whose loads are all in flight together (the kernel above walks 37 dependent rounds of L2 latency for the
// CBG dW: 8.7 us for 2.4 MB).  Lane p adds parts p, p+32, ... in order, then lanes are added in order: fixed.
template <bool PDL>  // (the programmatic-dependent-launch instantiation, common.cuh)
__global__ void __launch_bounds__(kThreads)
reduce_partials_vec_kernel(int64_t total4, int64_t n4, int n_parts, const float4* __restrict__ partial,
                           float* __restrict__ out, int64_t ldo, int64_t m, const double2* __restrict__ xpart,
                           float* __restrict__ xout) {
  __shared__ float4 red[32][8];
  __shared__ double2 xred[32][8][2];
  if constexpr (PDL) {
    pdl_launch_dependents();
    pdl_wait();  // the partial tiles are the previous kernel's output
  }
  const int tx = threadIdx.x & 7;
  const int ty = threadIdx.x >> 3;
  const int64_t i = (int64_t)blockIdx.x * 8 + tx;
  const int64_t mn4 = m * n4;
  if (i < mn4) {  // (warp-uniform except in the one warp that straddles row m)
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    int s = ty;
    for (; s + 96 < n_parts; s += 128) {
      const float4 v0 = __ldg(partial + (int64_t)s * mn4 + i);
      const float4 v1 = __ldg(partial + (int64_t)(s + 32) * mn4 + i);
      const float4 v2 = __ldg(partial + (int64_t)(s + 64) * mn4 + i);
      const float4 v3 = __ldg(partial + (int64_t)(s + 96) * mn4 + i);
      acc.x = (((acc.x + v0.x) + v1.x) + v2.x) + v3.x;
      acc.y = (((acc.y + v0.y) + v1.y) + v2.y) + v3.y;
      acc.z = (((acc.z + v0.z) + v1.z) + v2.z) + v3.z;
      acc.w = (((acc.w + v0.w) + v1.w) + v2.w) + v3.w;
    }
    for (; s < n_parts; s += 32) {
      const float4 v = __ldg(partial + (int64_t)s * mn4 + i);
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
    red[ty][tx] = acc;
  } else if (i < total4) {  // the fp64 column-sum row
    double a[4] = {0.0, 0.0, 0.0, 0.0};
    for (int s = ty; s < n_parts; s += 32) {
      const double2 v = __ldg(xpart + 2 * ((int64_t)s * n4 + (i - mn4))), w = __ldg(xpart + 2 * ((int64_t)s * n4 + (i - mn4)) + 1);
      a[0] += v.x; a[1] += v.y; a[2] += w.x; a[3] += w.y;
    }
    xred[ty][tx][0] = make_double2(a[0], a[1]);
    xred[ty][tx][1] = make_double2(a[2], a[3]);
  }
  __syncthreads();
  if (ty == 0 && i < mn4) {
    float4 v = red[0][tx];
#pragma unroll
    for (int t = 1; t < 32; ++t) {
      const float4 r = red[t][tx];
      v.x += r.x; v.y += r.y; v.z += r.z; v.w += r.w;
    }
    *reinterpret_cast<float4*>(out + (i / n4) * ldo + 4 * (i % n4)) = v;
  } else if (ty == 0 && i < total4) {
    double a[4] = {0.0, 0.0, 0.0, 0.0};
    for (int t = 0; t < 32; ++t) {
      a[0] += xred[t][tx][0].x; a[1] += xred[t][tx][0].y; a[2] += xred[t][tx][1].x; a[3] += xred[t][tx][1].y;
    }
    *reinterpret_cast<float4*>(xout + 4 * (i - mn4)) = make_float4((float)a[0], (float)a[1], (float)a[2], (float)a[3]);
  }
}

__global__ void __launch_bounds__(kThreads)
bias_act_kernel(int64_t n_rows, int f, float* __restrict__ out, int64_t ldo, Epilogue ep) {
  const int64_t total = n_rows * f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / f;
    const int j = (int)(i % f);
    float v = out[r * ldo + j];
    if (ep.bias) v += __ldg(ep.bias + j);
    if (ep.relu) v = fmaxf(v, 0.f);
    if (ep.mask) v = __ldg(ep.mask + r * ep.ld_mask + j) ? v * ep.mask_scale : 0.f;
    out[r * ldo + j] = v;
  }
}

__global__ void __launch_bounds__(kThreads)
pad_copy_kernel(int64_t n_rows, int w, int w4, const float* __restrict__ src, int64_t ld_src, float* __restrict__ dst,
                int64_t ld_dst) {
  const int64_t total = n_rows * w4;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / w4;
    const int j = (int)(i % w4);
    dst[r * ld_dst + j] = (j < w) ? __ldg(src + r * ld_src + j) : 0.f;
  }
}

__global__ void __launch_bounds__(kThreads) zero_kernel(float* out, int f) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < f) out[j] = 0.f;
}

__global__ void __launch_bounds__(kThreads) flush_kernel(float4* buf, size_t n4, float v) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride)
    buf[i] = make_float4(v, v, v, v);
}

int colsum_blocks(int64_t n_rows) {
  int64_t b = ceil_div(n_rows, 128);
  if (b > kMaxBlocks) b = kMaxBlocks;
  return (int)(b < 1 ? 1 : b);
}

}  // namespace

size_t colsum_workspace_bytes(int64_t n_rows, int64_t f) {
  // fp64 partials [blocks][f] (32-byte aligned rows) + the arrival ticket of the single-launch variant
  return (size_t)colsum_blocks(n_rows) * (size_t)(ceil_div(f, 4) * 4) * sizeof(double) + 256;
}

int colsum_launch(int64_t n_rows, int64_t f, const float* g, int64_t ldg, const float* y,
                  int64_t ldy, float* gm, int64_t ldgm, float* out, void* ws, size_t ws_bytes,
                  cudaStream_t st, const uint8_t* mask, int64_t ld_mask, float mask_scale) {
  GCNB_REQUIRE(f > 0 && f < (1 << 24), "colsum: width out of range");
  GCNB_REQUIRE(out != nullptr, "colsum: null output");
  if (n_rows == 0) {
    zero_kernel<<<(unsigned)ceil_div(f, kThreads), kThreads, 0, st>>>(out, (int)f);
    GCNB_LAUNCH_CHECK();
    return GCNB_OK;
  }
  GCNB_REQUIRE(g != nullptr && ldg >= f, "colsum: bad gradient operand");
  GCNB_REQUIRE(y == nullptr || (gm != nullptr && ldy >= f), "colsum: bad mask operands");
  GCNB_REQUIRE(gm == nullptr || ldgm >= f, "colsum: ldgm < width");
  GCNB_REQUIRE(mask == nullptr || (gm != nullptr && ld_mask >= f), "colsum: dropout mask needs gm and ld_mask >= width");
  const int nb = colsum_blocks(n_rows);
  const size_t need = colsum_workspace_bytes(n_rows, f);
  GCNB_REQUIRE(ws != nullptr && ws_bytes >= need, "colsum: workspace too small (%zu < %zu)", ws_bytes, need);
  GCNB_REQUIRE((reinterpret_cast<uintptr_t>(ws) & 7u) == 0, "colsum: workspace not 8-byte aligned (fp64 partials)");
  const int64_t rows_per_block = ceil_div(n_rows, nb);
  auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; };
  const bool vec = f % 4 == 0 && f <= 4 * kThreads && al16(g) && ldg % 4 == 0 && al16(out) && al16(ws) &&
                   (y == nullptr || (al16(y) && ldy % 4 == 0)) && (gm == nullptr || (al16(gm) && ldgm % 4 == 0)) &&
                   (mask == nullptr || ((reinterpret_cast<uintptr_t>(mask) & 3u) == 0 && ld_mask % 4 == 0));
  if (vec) {
    const int f4 = (int)(f / 4);
    int cw4 = 1;
    while (cw4 < f4) cw4 <<= 1;
    unsigned int* ticket = reinterpret_cast<unsigned int*>(reinterpret_cast<char*>(ws) + (need - 256));
    GCNB_CUDA(cudaMemsetAsync(ticket, 0, sizeof(unsigned int), st));
    colsum_vec_kernel<<<nb, kThreads, 0, st>>>(
        n_rows, f4, cw4, rows_per_block, reinterpret_cast<const float4*>(g), ldg / 4, reinterpret_cast<const float4*>(y),
        ldy / 4, reinterpret_cast<float4*>(gm), ldgm / 4, reinterpret_cast<double2*>(ws), ticket, out,
        reinterpret_cast<const uchar4*>(mask), ld_mask / 4, mask_scale);
    GCNB_LAUNCH_CHECK();
    return GCNB_OK;
  }
  int cw = 32;
  while (cw < f && cw < kThreads) cw <<= 1;
  colsum_partial_kernel<<<nb, kThreads, 0, st>>>(n_rows, (int)f, cw, rows_per_block, g, ldg, y, ldy, gm,
                                                 ldgm, reinterpret_cast<double*>(ws), mask, ld_mask, mask_scale);
  GCNB_LAUNCH_CHECK();
  return reduce_partials_launch(0, f, nb, nullptr, nullptr, 0, st, reinterpret_cast<const double*>(ws), out);
}

int pad_copy_launch(int64_t n_rows, int64_t w, const float* src, int64_t ld_src, float* dst, int64_t ld_dst,
                    cudaStream_t st) {
  if (n_rows == 0 || w == 0) return GCNB_OK;
  const int64_t w4 = ceil_div(w, 4) * 4;
  GCNB_REQUIRE(ld_dst >= w4 && ld_src >= w, "pad_copy: bad leading dimension");
  int64_t blocks = ceil_div(n_rows * w4, kThreads * 4);
  if (blocks > 16 * kNumSMs) blocks = 16 * kNumSMs;
  if (blocks < 1) blocks = 1;
  pad_copy_kernel<<<(unsigned)blocks, kThreads, 0, st>>>(n_rows, (int)w, (int)w4, src, ld_src, dst, ld_dst);
  GCNB_LAUNCH_CHECK();
  return GCNB_OK;
}

// dst[r, 0:ld8] = bf16(src[r, 0:f]) (round to nearest even), zero past f: one thread per 8 output elements
// (16-byte store); rows of dst are 16-byte aligned (ld_dst % 8 == 0).  src rows may be unaligned / strided.
__global__ void __launch_bounds__(kThreads)
to_bf16_kernel(int64_t n_rows, int f, int c8, const float* __restrict__ src, int64_t ld_src, uint16_t* __restrict__ dst,
               int64_t ld_dst, int vec_in) {
  const int64_t total = n_rows * c8;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / c8;
    const int q = (int)(i % c8);
    const float* p = src + r * ld_src + 8 * q;
    float v[8];
    if (vec_in && 8 * q + 8 <= f) {
      const float4 a = __ldg(reinterpret_cast<const float4*>(p));
      const float4 b = __ldg(reinterpret_cast<const float4*>(p + 4));
      v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
    } else {
#pragma unroll
      for (int t = 0; t < 8; ++t) v[t] = (8 * q + t < f) ? __ldg(p + t) : 0.f;
    }
    uint32_t w[4];
#pragma unroll
    for (int t = 0; t < 4; ++t)  // cvt.rn.bf16x2.f32 d, hi, lo: element 2t in the low half
      asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(w[t]) : "f"(v[2 * t + 1]), "f"(v[2 * t]));
    *reinterpret_cast<uint4*>(dst + r * ld_dst + 8 * q) = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

int to_bf16_launch(int64_t n_rows, int64_t f, const float* src, int64_t ld_src, uint16_t* dst, int64_t ld_dst,
                   cudaStream_t st) {
  if (n_rows == 0 || f == 0) return GCNB_OK;
  const int64_t c8 = ceil_div(f, 8);
  GCNB_REQUIRE(src != nullptr && dst != nullptr, "to_bf16: null operand");
  GCNB_REQUIRE(ld_src >= f && ld_dst >= 8 * c8 && ld_dst % 8 == 0 && (reinterpret_cast<uintptr_t>(dst) & 15u) == 0,
               "to_bf16: destination rows must be 16-byte aligned with ld a multiple of 8 and >= 8*ceil(f/8)");
  const int vec_in = ((reinterpret_cast<uintptr_t>(src) & 15u) == 0) && (ld_src % 4 == 0);
  int64_t blocks = ceil_div(n_rows * c8, kThreads);
  if (blocks > 16 * kNumSMs) blocks = 16 * kNumSMs;
  to_bf16_kernel<<<(unsigned)blocks, kThreads, 0, st>>>(n_rows, (int)f, (int)c8, src, ld_src, dst, ld_dst, vec_in);
  GCNB_LAUNCH_CHECK();
  return GCNB_OK;
}

int bias_act_launch(int64_t n_rows, int64_t f, float* out, int64_t ldo, const Epilogue& ep, cudaStream_t st) {
  if (n_rows == 0 || f == 0 || (ep.bias == nullptr && !ep.relu && ep.mask == nullptr)) return GCNB_OK;
  int64_t blocks = ceil_div(n_rows * f, kThreads);
  if (blocks > kMaxBlocks) blocks = kMaxBlocks;
  bias_act_kernel<<<(unsigned)blocks, kThreads, 0, st>>>(n_rows, (int)f, out, ldo, ep);
  GCNB_LAUNCH_CHECK();
  return GCNB_OK;
}

int reduce_partials_launch(int64_t m, int64_t n, int n_parts, const float* partial, float* out,
                           int64_t ldo, cudaStream_t st, const double* xpart, float* xout) {
  const int64_t total = (m + (xout ? 1 : 0)) * n;
  if (total == 0) return GCNB_OK;
  auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; };
  if (n_parts >= 16 && n % 4 == 0 && ldo % 4 == 0 && al16(partial) && al16(out) && al16(xpart) && al16(xout)) {
    if (pdl_enabled()) {  // opt-in (common.cuh)
      GCNB_CUDA(launch_pdl(reduce_partials_vec_kernel<true>, dim3((unsigned)ceil_div(total / 4, 8)), dim3(kThreads), 0, st,
                           total / 4, n / 4, n_parts, reinterpret_cast<const float4*>(partial), out, ldo, m,
                           reinterpret_cast<const double2*>(xpart), xout));
      return GCNB_OK;
    }
    reduce_partials_vec_kernel<false><<<(unsigned)ceil_div(total / 4, 8), kThreads, 0, st>>>(
        total / 4, n / 4, n_parts, reinterpret_cast<const float4*>(partial), out, ldo, m,
        reinterpret_cast<const double2*>(xpart), xout);
    GCNB_LAUNCH_CHECK();
    return GCNB_OK;
  }
  reduce_partials_kernel<<<(unsigned)ceil_div(total, 32), kThreads, 0, st>>>(total, n, n_parts, partial, out, ldo, m,
                                                                            xpart, xout);
  GCNB_LAUNCH_CHECK();
  return GCNB_OK;
}

}  // namespace gcnb

extern "C" int gcnb_l2_flush(void* d_buf, size_t bytes, void* stream) {
  using namespace gcnb;
  GCNB_REQUIRE(d_buf != nullptr && bytes >= 16, "l2_flush: bad buffer");
  static unsigned tick = 0;
  flush_kernel<<<4 * kNumSMs, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<float4*>(d_buf),
                                                              bytes / 16, (float)(++tick));
  GCNB_LAUNCH_CHECK();
  return GCNB_OK;
}
