// Skinny fp32 GEMMs on CUDA cores for the narrow layers of the reference's real workloads
// (CBG 64->32, the fork's 8->32 / 32->32, Cora's 16->7):
//     rows:  C[M,N]  = A[M,K] . B[K,N]          support = X W (pygcn/layers.py:33), dX = dS W^T
//     tn  :  C[Mo,N] = sum_r X[r,0:Mo]^T Y[r,0:N]   dW = X^T dS   (MmBackward0, SURVEY.md 3.2)
// with K (resp. Mo) <= 64 and N <= 64.  These products are HBM-bound streams over M = number of nodes
// with a few dozen FMAs per loaded float: a tensor-core pipeline (operand split into tf32 hi/lo,
// swizzled shared-memory tiles, TMEM) only adds latency here -- the tcgen05 kernels stay for the
// shapes that are dense contractions (Reddit 602->256, products 100->256 / 256->256).
//
// One lane owns one output column: the small operand (a column of B, resp. the accumulators of one
// column of C) lives in its registers; rows of the streamed operands are staged global -> shared with
// 16-byte cp.async (double-buffered, 8 rows per stage and warp) and read back as broadcast LDS.128.
// Exact fp32 FMA accumulation in a fixed order: bit-stable run to run.
#include <stdlib.h>

#include "common.cuh"
#include "ptx.cuh"

namespace gcnb {
namespace {

constexpr int kWarps = 8;
constexpr int kThreads = kWarps * 32;
constexpr int kStageRows = 8;
constexpr unsigned kFull = 0xffffffffu;

// ---------------------------------------------------------------------------------------------- rows
// KMAX: padded K (multiple of 4); NC: output columns per lane (N <= 32 * NC).
template <int KMAX, int NC>
__global__ void __launch_bounds__(kThreads)
skinny_rows_kernel(int64_t M, int N, int K, const float* __restrict__ a, int64_t lda, const float* __restrict__ b,
                   int64_t b_rs, int64_t b_cs, float* __restrict__ c, int64_t ldc) {
  constexpr int K4 = KMAX / 4;
  __shared__ __align__(16) float stage[kWarps][2][kStageRows][KMAX];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // B (any strides) -> shared memory once per CTA, zero past K / N; then this lane's columns -> registers
  {
    float* bs = &stage[0][0][0][0];  // KMAX * 32 * NC floats <= the staging array (kWarps*2*8*KMAX)
    for (int i = threadIdx.x; i < KMAX * 32 * NC; i += kThreads) {
      const int k = i / (32 * NC), col = i % (32 * NC);
      bs[i] = (k < K && col < N) ? __ldg(b + (int64_t)k * b_rs + (int64_t)col * b_cs) : 0.f;
    }
    __syncthreads();
  }
  float w[KMAX][NC];
  {
    const float* bs = &stage[0][0][0][0];
#pragma unroll
    for (int k = 0; k < KMAX; ++k)
#pragma unroll
      for (int j = 0; j < NC; ++j) w[k][j] = bs[k * 32 * NC + lane + 32 * j];
  }
  __syncthreads();  // the staging array is reused for rows below
  const int64_t gw = (int64_t)blockIdx.x * kWarps + warp;
  const int64_t nw = (int64_t)gridDim.x * kWarps;
  const int64_t n_stages = (M + kStageRows - 1) / kStageRows;
  // stage s covers rows [s*8, s*8+8): lane l copies float4 #(l % K4) of row (l / K4) (+ 32/K4 per step)
  auto fetch = [&](int64_t s, int buf) {
    constexpr int kCopies = (kStageRows * K4 + 31) / 32;
#pragma unroll
    for (int t = 0; t < kCopies; ++t) {
      const int i = lane + 32 * t;
      const int r = i / K4, q = i % K4;
      if (i < kStageRows * K4) {
        const int64_t row = s * kStageRows + r;
        const int kleft = K - 4 * q;  // floats of this chunk that exist
        const uint32_t bytes = (row < M && kleft > 0) ? (uint32_t)(kleft >= 4 ? 16 : 4 * kleft) : 0u;
        cp_async16_zfill(smem_u32(&stage[warp][buf][r][4 * q]), a + (row < M ? row : 0) * lda + 4 * q, bytes);
      }
    }
    cp_async_commit();
  };
  int buf = 0;
  if (gw < n_stages) fetch(gw, 0);
  for (int64_t s = gw; s < n_stages; s += nw) {
    if (s + nw < n_stages) fetch(s + nw, buf ^ 1); else cp_async_commit();
    cp_async_wait<1>();
    __syncwarp();
#pragma unroll 2
    for (int r = 0; r < kStageRows; ++r) {
      const int64_t row = s * kStageRows + r;
      float acc[NC];
#pragma unroll
      for (int j = 0; j < NC; ++j) acc[j] = 0.f;
#pragma unroll
      for (int q = 0; q < K4; ++q) {
        const float4 x = *reinterpret_cast<const float4*>(&stage[warp][buf][r][4 * q]);  // broadcast
#pragma unroll
        for (int j = 0; j < NC; ++j) {
          acc[j] = fmaf(x.x, w[4 * q + 0][j], acc[j]);
          acc[j] = fmaf(x.y, w[4 * q + 1][j], acc[j]);
          acc[j] = fmaf(x.z, w[4 * q + 2][j], acc[j]);
          acc[j] = fmaf(x.w, w[4 * q + 3][j], acc[j]);
        }
      }
      if (row < M) {
#pragma unroll
        for (int j = 0; j < NC; ++j) {
          const int col = lane + 32 * j;
          if (col < N) c[row * ldc + col] = acc[j];
        }
      }
    }
    __syncwarp();
    buf ^= 1;
  }
  cp_async_wait<0>();
}

// ---------------------------------------------------------------------------------------------- tn
// C_partial[cta][Mo][N] = sum over this CTA's rows of X[r, 0:Mo]^T Y[r, 0:N];  MMAX = padded Mo, N <= 32.
// GSUM: a third operand G [R, N] rides along and its column sums (db = colsum(G), the AddBackward0 of
// pygcn/layers.py:36) land in gpartial[cta][N], in fp64 like every column sum (elementwise.cu) -- the layer's backward
// then needs no colsum kernel when no mask has to be applied to G first (one launch and one 12.8 MB pass less on the
// CBG shape).
// PDL: the programmatic-dependent-launch instantiation (common.cuh); y is the previous kernel's output, so the wait
// comes first and only the launch latency and the CTA scheduling overlap.
template <int MMAX, bool GSUM, bool PDL = false>
__global__ void __launch_bounds__(kThreads)
skinny_tn_kernel(int64_t R, int Mo, int N, const float* __restrict__ x, int64_t ldx, const float* __restrict__ y,
                 int64_t ldy, const float* __restrict__ gx, int64_t ldg, float* __restrict__ partial,
                 double* __restrict__ gpartial) {
  if constexpr (PDL) {
    pdl_launch_dependents();
    pdl_wait();
  }
  constexpr int M4 = MMAX / 4;
  extern __shared__ __align__(16) float skinny_smem[];
  float (*xs)[2][kStageRows][MMAX] = reinterpret_cast<float (*)[2][kStageRows][MMAX]>(skinny_smem);
  float (*ys)[2][kStageRows][32] = reinterpret_cast<float (*)[2][kStageRows][32]>(skinny_smem + kWarps * 2 * kStageRows * MMAX);
  float (*gs)[2][kStageRows][32] = reinterpret_cast<float (*)[2][kStageRows][32]>(
      skinny_smem + kWarps * 2 * kStageRows * (MMAX + 32));  // only touched when GSUM
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double gacc = 0.0;  // fp64: a column sum of G cancels to ~sqrt(rows) of its mass (elementwise.cu)
  float acc[MMAX];
#pragma unroll
  for (int k = 0; k < MMAX; ++k) acc[k] = 0.f;
  const int64_t gw = (int64_t)blockIdx.x * kWarps + warp;
  const int64_t nw = (int64_t)gridDim.x * kWarps;
  const int64_t n_stages = (R + kStageRows - 1) / kStageRows;
  const int n4 = (N + 3) >> 2;
  auto fetch = [&](int64_t s, int buf) {
    constexpr int kCopies = (kStageRows * M4 + 31) / 32;
#pragma unroll
    for (int t = 0; t < kCopies; ++t) {
      const int i = lane + 32 * t;
      const int r = i / M4, q = i % M4;
      if (i < kStageRows * M4) {
        const int64_t row = s * kStageRows + r;
        const int left = Mo - 4 * q;
        const uint32_t bytes = (row < R && left > 0) ? (uint32_t)(left >= 4 ? 16 : 4 * left) : 0u;
        cp_async16_zfill(smem_u32(&xs[warp][buf][r][4 * q]), x + (row < R ? row : 0) * ldx + 4 * q, bytes);
      }
    }
    {  // Y: 8 rows x 8 float4 = 64 copies, two per lane
#pragma unroll
      for (int t = 0; t < 2; ++t) {
        const int i = lane + 32 * t;
        const int r = i >> 3, q = i & 7;
        const int64_t row = s * kStageRows + r;
        const int left = N - 4 * q;
        const uint32_t bytes = (row < R && q < n4 && left > 0) ? (uint32_t)(left >= 4 ? 16 : 4 * left) : 0u;
        cp_async16_zfill(smem_u32(&ys[warp][buf][r][4 * q]), y + (row < R ? row : 0) * ldy + 4 * q, bytes);
        if constexpr (GSUM)
          cp_async16_zfill(smem_u32(&gs[warp][buf][r][4 * q]), gx + (row < R ? row : 0) * ldg + 4 * q, bytes);
      }
    }
    cp_async_commit();
  };
  int buf = 0;
  if (gw < n_stages) fetch(gw, 0);
  for (int64_t s = gw; s < n_stages; s += nw) {
    if (s + nw < n_stages) fetch(s + nw, buf ^ 1); else cp_async_commit();
    cp_async_wait<1>();
    __syncwarp();
#pragma unroll 2
    for (int r = 0; r < kStageRows; ++r) {
      const float yv = ys[warp][buf][r][lane];  // zero-filled past N and past R
      if constexpr (GSUM) gacc += (double)gs[warp][buf][r][lane];
#pragma unroll
      for (int q = 0; q < M4; ++q) {
        const float4 xv = *reinterpret_cast<const float4*>(&xs[warp][buf][r][4 * q]);  // broadcast
        acc[4 * q + 0] = fmaf(xv.x, yv, acc[4 * q + 0]);
        acc[4 * q + 1] = fmaf(xv.y, yv, acc[4 * q + 1]);
        acc[4 * q + 2] = fmaf(xv.z, yv, acc[4 * q + 2]);
        acc[4 * q + 3] = fmaf(xv.w, yv, acc[4 * q + 3]);
      }
    }
    __syncwarp();
    buf ^= 1;
  }
  cp_async_wait<0>();
  __syncthreads();
  // CTA reduction in a fixed order: warp w adds into the shared tile in turn (w = 0 initialises)
  float* tile = &xs[0][0][0][0];  // MMAX * 32 floats + 32 doubles <= the xs array (kWarps*2*8*MMAX floats)
  double* gtile = reinterpret_cast<double*>(tile + MMAX * 32);
  for (int wv = 0; wv < kWarps; ++wv) {
    if (warp == wv) {
#pragma unroll
      for (int k = 0; k < MMAX; ++k) {
        const float prev = (wv == 0) ? 0.f : tile[k * 32 + lane];
        tile[k * 32 + lane] = prev + acc[k];
      }
      if constexpr (GSUM) gtile[lane] = ((wv == 0) ? 0.0 : gtile[lane]) + gacc;
    }
    __syncthreads();
  }
  float* dst = partial + (int64_t)blockIdx.x * Mo * N;
  for (int i = threadIdx.x; i < Mo * N; i += kThreads) dst[i] = tile[(i / N) * 32 + (i % N)];
  if constexpr (GSUM)
    if (threadIdx.x < N) gpartial[(int64_t)blockIdx.x * N + threadIdx.x] = gtile[threadIdx.x];
}

inline bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

}  // namespace

// ---------------------------------------------------------------------------------------------- host side
bool gemm_skinny_rows_eligible(int64_t m, int64_t n, int64_t k, const float* a, int64_t a_rs, int64_t a_cs) {
  if (m < 4096 || n < 1 || k < 1 || a_cs != 1 || a_rs % 4 != 0 || !al16(a)) return false;
  if (n <= 32) return k <= 64;
  return n <= 64 && k <= 32;
}

int gemm_skinny_rows_launch(int64_t m, int64_t n, int64_t k, const float* a, int64_t lda, const float* b, int64_t b_rs,
                            int64_t b_cs, float* c, int64_t ldc, cudaStream_t st) {
  // persistent: two CTAs per SM (the register budget allows no more), each warp walks its stages
  int64_t grid = ceil_div(ceil_div(m, kStageRows), kWarps);
  if (grid > 2 * kNumSMs) grid = 2 * kNumSMs;
#define GCNB_SKINNY_ROWS(KMAX_, NC_)                                                                              \
  skinny_rows_kernel<KMAX_, NC_><<<(unsigned)grid, kThreads, 0, st>>>(m, (int)n, (int)k, a, lda, b, b_rs, b_cs, c, ldc)
  if (n <= 32) {
    if (k <= 8) GCNB_SKINNY_ROWS(8, 1);
    else if (k <= 16) GCNB_SKINNY_ROWS(16, 1);
    else if (k <= 32) GCNB_SKINNY_ROWS(32, 1);
    else GCNB_SKINNY_ROWS(64, 1);
  } else {
    if (k <= 8) GCNB_SKINNY_ROWS(8, 2);
    else if (k <= 16) GCNB_SKINNY_ROWS(16, 2);
    else GCNB_SKINNY_ROWS(32, 2);
  }
#undef GCNB_SKINNY_ROWS
  GCNB_LAUNCH_CHECK();
  return GCNB_OK;
}

bool gemm_skinny_tn_eligible(int64_t m, int64_t n, int64_t r, const float* x, int64_t ldx, const float* y, int64_t ldy) {
  return r >= 4096 && m >= 1 && m <= 64 && n >= 1 && n <= 32 && ldx % 4 == 0 && ldy % 4 == 0 && al16(x) && al16(y);
}

static int skinny_tn_ctas(int64_t r) {
  int64_t g = ceil_div(ceil_div(r, kStageRows), kWarps);
  static int per_sm = 0;  // GCNB_SKINNY_TN_CTAS = CTAs per SM (tuning knob; one partial tile per CTA)
  if (per_sm == 0) {
    const char* e = getenv("GCNB_SKINNY_TN_CTAS");
    per_sm = (e && atoi(e) > 0) ? atoi(e) : 2;
  }
  if (g > (int64_t)per_sm * kNumSMs) g = (int64_t)per_sm * kNumSMs;
  return (int)(g < 1 ? 1 : g);
}

// fp32 partial tiles [ctas][m][n], then (256-byte aligned) the fp64 column sums of the fused db [ctas][n]
static size_t skinny_tn_tile_bytes(int64_t m, int64_t n, int64_t r) {
  return ((size_t)skinny_tn_ctas(r) * (size_t)m * (size_t)n * sizeof(float) + 255) & ~(size_t)255;
}

size_t gemm_skinny_tn_workspace_bytes(int64_t m, int64_t n, int64_t r) {
  return skinny_tn_tile_bytes(m, n, r) + (size_t)skinny_tn_ctas(r) * (size_t)n * sizeof(double);
}

// per-device opt-in above the static 48 KB limit (MMAX = 64 with the third operand: 64 KB)
template <int MMAX, bool GSUM, bool PDL>
static int skinny_tn_allow_smem(size_t smem) {
  if (smem <= 48 * 1024) return GCNB_OK;
  static bool done[64] = {};
  int dev = 0;
  GCNB_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64 || !done[dev]) {
    GCNB_CUDA(cudaFuncSetAttribute(skinny_tn_kernel<MMAX, GSUM, PDL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (dev >= 0 && dev < 64) done[dev] = true;
  }
  return GCNB_OK;
}

template <int MMAX, bool GSUM>
static int skinny_tn_launch_t(int ctas, int64_t r, int m, int n, const float* x, int64_t ldx, const float* y, int64_t ldy,
                              const float* gx, int64_t ldg, float* partial, double* gpartial, cudaStream_t st) {
  const size_t smem = (size_t)kWarps * 2 * kStageRows * (MMAX + 32 + (GSUM ? 32 : 0)) * sizeof(float);
  if (pdl_enabled()) {  // opt-in (common.cuh)
    GCNB_TRY((skinny_tn_allow_smem<MMAX, GSUM, true>(smem)));
    GCNB_CUDA(launch_pdl(skinny_tn_kernel<MMAX, GSUM, true>, dim3((unsigned)ctas), dim3(kThreads), smem, st, r, m, n, x, ldx,
                         y, ldy, gx, ldg, partial, gpartial));
    return GCNB_OK;
  }
  GCNB_TRY((skinny_tn_allow_smem<MMAX, GSUM, false>(smem)));
  skinny_tn_kernel<MMAX, GSUM><<<ctas, kThreads, smem, st>>>(r, m, n, x, ldx, y, ldy, gx, ldg, partial, gpartial);
  GCNB_LAUNCH_CHECK();
  return GCNB_OK;
}

// gx != nullptr: also db[0:n] = column sums of G [r, n] (row stride ldg), fused into the same pass
int gemm_skinny_tn_launch(int64_t m, int64_t n, int64_t r, const float* x, int64_t ldx, const float* y, int64_t ldy,
                          float* c, int64_t ldc, void* ws, size_t ws_bytes, cudaStream_t st, const float* gx, int64_t ldg,
                          float* db) {
  const int ctas = skinny_tn_ctas(r);
  GCNB_REQUIRE(ws != nullptr && ws_bytes >= gemm_skinny_tn_workspace_bytes(m, n, r), "gemm(skinny tn): workspace too small");
  GCNB_REQUIRE(gx == nullptr || (db != nullptr && ldg % 4 == 0 && ldg >= n && al16(gx) && al16(ws)),
               "gemm(skinny tn): the fused column sum needs 16-byte aligned rows of G and workspace, and an output");
  float* partial = reinterpret_cast<float*>(ws);
  double* gpartial = reinterpret_cast<double*>(reinterpret_cast<char*>(ws) + skinny_tn_tile_bytes(m, n, r));
  int status;
#define GCNB_SKINNY_TN(MMAX_)                                                                                              \
  status = gx ? (skinny_tn_launch_t<MMAX_, true>(ctas, r, (int)m, (int)n, x, ldx, y, ldy, gx, ldg, partial, gpartial, st)) \
              : (skinny_tn_launch_t<MMAX_, false>(ctas, r, (int)m, (int)n, x, ldx, y, ldy, nullptr, 0, partial, nullptr, st))
  if (m <= 8) GCNB_SKINNY_TN(8);
  else if (m <= 16) GCNB_SKINNY_TN(16);
  else if (m <= 32) GCNB_SKINNY_TN(32);
  else GCNB_SKINNY_TN(64);
#undef GCNB_SKINNY_TN
  GCNB_TRY(status);
  return reduce_partials_launch(m, n, ctas, partial, c, ldc, st, gx ? gpartial : nullptr, gx ? db : nullptr);
}

}  // namespace gcnb
