// fp32 CUDA-core GEMM with generic operand strides: the bit-faithful (fp32 FMA accumulate)
// path for  support = X W  (pygcn/layers.py:33),  dW = X^T dS  and  dX = dS W^T
// (MmBackward0, SURVEY.md 3.2).  Used for shapes where tensor cores are pointless
// (Cora L2 is 16x7) and as the always-available exact tier next to the tcgen05 kernels.
//
// Block tile BM x BN, K step 16, 256 threads, TM x TN register tile per thread.  A reduction
// longer than kSplitK is split across gridDim.z; partial tiles go to scratch and are added in
// split order by a second kernel (deterministic, no atomics).
#include "common.cuh"

namespace gcnb {
namespace {

constexpr int BK = 16;
constexpr int kThreads = 256;
constexpr int64_t kSplitChunk = 512;  // K elements per split when splitting

template <int BM, int BN>
__global__ void __launch_bounds__(kThreads)
gemm_fp32_kernel(int m, int n, int64_t k, const float* __restrict__ a, int64_t a_rs, int64_t a_cs,
                 const float* __restrict__ b, int64_t b_rs, int64_t b_cs, float* __restrict__ c,
                 int64_t ldc, int64_t k_per_split, int64_t split_stride) {
  constexpr int TM = BM / 16;
  constexpr int TN = BN / 16;
  __shared__ float As[BK][BM + 4];
  __shared__ float Bs[BK][BN + 4];
  const int tid = threadIdx.x;
  const int tx = tid % 16;  // along N
  const int ty = tid / 16;  // along M
  const int m0 = blockIdx.x * BM;
  const int n0 = blockIdx.y * BN;
  const int64_t k_begin = (int64_t)blockIdx.z * k_per_split;
  const int64_t k_end = (k_begin + k_per_split < k) ? (k_begin + k_per_split) : k;
  const bool a_k_contig = (a_cs == 1);
  const bool b_n_contig = (b_cs == 1);

  float acc[TM][TN];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

  for (int64_t k0 = k_begin; k0 < k_end; k0 += BK) {
    // A tile: BM x BK
    for (int idx = tid; idx < BM * BK; idx += kThreads) {
      int mm, kk;
      if (a_k_contig) { kk = idx % BK; mm = idx / BK; } else { mm = idx % BM; kk = idx / BM; }
      const int gm = m0 + mm;
      const int64_t gk = k0 + kk;
      float v = 0.f;
      if (gm < m && gk < k_end) v = __ldg(a + (int64_t)gm * a_rs + gk * a_cs);
      As[kk][mm] = v;
    }
    // B tile: BK x BN
    for (int idx = tid; idx < BK * BN; idx += kThreads) {
      int nn, kk;
      if (b_n_contig) { nn = idx % BN; kk = idx / BN; } else { kk = idx % BK; nn = idx / BK; }
      const int gn = n0 + nn;
      const int64_t gk = k0 + kk;
      float v = 0.f;
      if (gn < n && gk < k_end) v = __ldg(b + gk * b_rs + (int64_t)gn * b_cs);
      Bs[kk][nn] = v;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      float av[TM], bv[TN];
#pragma unroll
      for (int i = 0; i < TM; ++i) av[i] = As[kk][ty * TM + i];
#pragma unroll
      for (int j = 0; j < TN; ++j) bv[j] = Bs[kk][tx * TN + j];
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    __syncthreads();
  }

  float* cbase = c + (int64_t)blockIdx.z * split_stride;
#pragma unroll
  for (int i = 0; i < TM; ++i) {
    const int gm = m0 + ty * TM + i;
    if (gm >= m) continue;
#pragma unroll
    for (int j = 0; j < TN; ++j) {
      const int gn = n0 + tx * TN + j;
      if (gn < n) cbase[(int64_t)gm * ldc + gn] = acc[i][j];
    }
  }
}

int num_splits(int64_t m, int64_t n, int64_t k) {
  // split whenever the output tiles alone cannot fill the GPU and the reduction is long enough
  // to share (dW = X^T dS: a handful of tiles, K = number of nodes)
  const int64_t tiles = ceil_div(m, 64) * ceil_div(n, 64);
  if (k < 512 || tiles >= kNumSMs) return 1;
  const int64_t chunk = (k >= 64 * kSplitChunk) ? kSplitChunk : 128;
  int64_t s = ceil_div(k, chunk);
  const int64_t cap = ceil_div(4 * kNumSMs, tiles);
  if (s > cap) s = cap;
  return (int)(s < 1 ? 1 : s);
}

}  // namespace

size_t gemm_fp32_workspace_bytes(int64_t m, int64_t n, int64_t k) {
  const int s = num_splits(m, n, k);
  return s > 1 ? (size_t)s * (size_t)m * (size_t)n * sizeof(float) : 0;
}

int gemm_fp32_launch(int64_t m, int64_t n, int64_t k, const float* a, int64_t a_rs, int64_t a_cs,
                     const float* b, int64_t b_rs, int64_t b_cs, float* c, int64_t ldc, void* ws,
                     size_t ws_bytes, cudaStream_t st) {
  GCNB_REQUIRE(m >= 0 && n >= 0 && k >= 0, "gemm: negative dimension");
  GCNB_REQUIRE(m < (1ll << 31) && n < (1ll << 31), "gemm: m/n too large");
  GCNB_REQUIRE(ldc >= n, "gemm: ldc < n");
  if (m == 0 || n == 0) return GCNB_OK;
  GCNB_REQUIRE(c != nullptr && (k == 0 || (a != nullptr && b != nullptr)), "gemm: null operand");
  const int splits = num_splits(m, n, k);
  const size_t need = gemm_fp32_workspace_bytes(m, n, k);
  GCNB_REQUIRE(need == 0 || (ws != nullptr && ws_bytes >= need), "gemm: workspace too small (%zu < %zu)",
               ws_bytes, need);
  int64_t k_per_split = k;
  float* dst = c;
  int64_t dst_ld = ldc;
  int64_t split_stride = 0;
  if (splits > 1) {
    k_per_split = ceil_div(ceil_div(k, splits), BK) * BK;
    dst = reinterpret_cast<float*>(ws);
    dst_ld = n;
    split_stride = m * n;
  }
  if (k_per_split == 0) k_per_split = BK;
  const int real_splits = (splits > 1) ? (int)ceil_div(k, k_per_split) : 1;
  // N tiles go on grid y, which holds at most 65535: wider products run as several launches of column panels
#define GCNB_GEMM_LAUNCH(BM_, BN_)                                                                     \
  do {                                                                                                 \
    const int64_t panel = 65535ll * BN_;                                                               \
    for (int64_t n0 = 0; n0 < n; n0 += panel) {                                                        \
      const int64_t nc = (n - n0 < panel) ? n - n0 : panel;                                            \
      dim3 grid((unsigned)ceil_div(m, BM_), (unsigned)ceil_div(nc, BN_), (unsigned)real_splits);       \
      gemm_fp32_kernel<BM_, BN_><<<grid, kThreads, 0, st>>>((int)m, (int)nc, k, a, a_rs, a_cs,         \
                                                            b + n0 * b_cs, b_rs, b_cs, dst + n0, dst_ld, \
                                                            k_per_split, split_stride);                \
      if (n0 + nc < n) GCNB_LAUNCH_CHECK();                                                            \
    }                                                                                                  \
  } while (0)
  if (m <= 64) {
    if (n <= 16) GCNB_GEMM_LAUNCH(64, 16);
    else if (n <= 32) GCNB_GEMM_LAUNCH(64, 32);
    else GCNB_GEMM_LAUNCH(64, 64);
  } else {
    if (n <= 16) GCNB_GEMM_LAUNCH(128, 16);
    else if (n <= 32) GCNB_GEMM_LAUNCH(128, 32);
    else GCNB_GEMM_LAUNCH(128, 64);
  }
#undef GCNB_GEMM_LAUNCH
  GCNB_LAUNCH_CHECK();
  if (splits > 1) {
    GCNB_TRY(reduce_partials_launch(m, n, real_splits, dst, c, ldc, st));
  }
  return GCNB_OK;
}

}  // namespace gcnb
