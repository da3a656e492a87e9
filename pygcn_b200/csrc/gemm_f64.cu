// fp64 tier: C = A B (+ bias) (ReLU) (dropout) with generic strides, on the fp64 tensor cores.
//
// tcgen05 has no fp64 kind, so the product runs on mma.sync.aligned.m8n8k4.row.col.f64 (DMMA.8x8x4).  A CTA of four
// warps computes a 64 x 64 tile (two warps a 64 x 32 tile for outputs of <= 32 columns), each warp a 32 x 32 block of
// 4 x 4 MMA tiles.  Operand tiles of 16 K columns are staged through shared memory by 8-byte cp.async with zero fill, two
// stages deep.  One element per copy is what makes any (row stride, column stride) pair work -- X W, dW = X^T dS and
// dX = dS W^T all run here -- and the thread-to-element map follows whichever stride is 1 so that a warp's copies
// stay coalesced.  Long reductions (dW reduces over every node) are split along K: each split writes an fp64 partial
// tile to the workspace and a second kernel adds the splits in ascending order, so results are bit-reproducible.
#include "common.cuh"

namespace gcnb {
namespace {

constexpr int kBK = 16;
constexpr int kPad = 4;  // shared-memory row padding (doubles): fragment loads take the minimum two wavefronts
constexpr int kMaxSplits = 64;
constexpr int64_t kMinKPerSplit = 256;

__device__ __forceinline__ void cp_async8(void* smem, const double* g, bool pred) {
  const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;\n" ::"r"(s), "l"(g), "r"(pred ? 8 : 0));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

__device__ __forceinline__ void dmma(double (&d)[2], double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};\n"
               : "+d"(d[0]), "+d"(d[1])
               : "d"(a), "d"(b));
}

__device__ __forceinline__ double ep_apply(double v, const Epilogue64& ep, int64_t i, int64_t j) {
  if (ep.bias) v += ep.bias[j];
  if (ep.relu) v = fmax(v, 0.0);
  if (ep.mask) v = ep.mask[i * ep.ld_mask + j] ? v * ep.mask_scale : 0.0;
  return v;
}

template <int BM, int BN>
struct GemmTile {
  static constexpr int kWarpsM = BM / 32;
  static constexpr int kThreads = 32 * kWarpsM * (BN / 32);  // one 32 x 32 block per warp
  double a[2][BM][kBK + kPad];
  double b[2][kBK][BN + kPad];
};

// grid: x = M tiles, y = N tiles, z = K splits.  splits == 1: C = epilogue(A B); else partial[z, i, j] (no epilogue).
template <int BM, int BN>
__global__ void __launch_bounds__(GemmTile<BM, BN>::kThreads) gemm_f64_dmma_kernel(
    int64_t m, int64_t n, int64_t k, const double* __restrict__ a, int64_t a_rs, int64_t a_cs,
    const double* __restrict__ b, int64_t b_rs, int64_t b_cs, double* __restrict__ c, int64_t ldc, int64_t k_per_split,
    Epilogue64 ep, double* __restrict__ partial) {
  __shared__ __align__(16) GemmTile<BM, BN> sm;
  constexpr int kThreads = GemmTile<BM, BN>::kThreads;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t m0 = (int64_t)blockIdx.x * BM, n0 = (int64_t)blockIdx.y * BN;
  const int64_t kb = (int64_t)blockIdx.z * k_per_split;
  const int64_t ke = min(k, kb + k_per_split);
  const int n_kt = ke > kb ? (int)((ke - kb + kBK - 1) / kBK) : 0;
  const bool a_kfast = a_cs == 1;  // consecutive threads walk K (row-major A) or M (A = X^T)
  const bool b_nfast = b_cs == 1;  // consecutive threads walk N (row-major B) or K (B = W^T)

  auto load = [&](int stage, int kt) {
    const int64_t k0 = kb + (int64_t)kt * kBK;
#pragma unroll
    for (int t = 0; t < BM * kBK / kThreads; ++t) {
      const int idx = tid + t * kThreads;
      const int r = a_kfast ? idx / kBK : idx % BM;
      const int kk = a_kfast ? idx % kBK : idx / BM;
      const int64_t gi = m0 + r, gk = k0 + kk;
      const bool ok = gi < m && gk < ke;
      cp_async8(&sm.a[stage][r][kk], ok ? a + gi * a_rs + gk * a_cs : a, ok);
    }
#pragma unroll
    for (int t = 0; t < kBK * BN / kThreads; ++t) {
      const int idx = tid + t * kThreads;
      const int kk = b_nfast ? idx / BN : idx % kBK;
      const int jj = b_nfast ? idx % BN : idx / kBK;
      const int64_t gk = k0 + kk, gj = n0 + jj;
      const bool ok = gk < ke && gj < n;
      cp_async8(&sm.b[stage][kk][jj], ok ? b + gk * b_rs + gj * b_cs : b, ok);
    }
    cp_async_commit();
  };

  const int wm = warp % GemmTile<BM, BN>::kWarpsM, wn = warp / GemmTile<BM, BN>::kWarpsM;
  double acc[4][4][2] = {};
  if (n_kt > 0) load(0, 0);
  for (int kt = 0; kt < n_kt; ++kt) {
    const int s = kt & 1;
    if (kt + 1 < n_kt) {
      load(s ^ 1, kt + 1);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < kBK; kk += 4) {
      double af[4], bf[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) af[i] = sm.a[s][wm * 32 + i * 8 + (lane >> 2)][kk + (lane & 3)];
#pragma unroll
      for (int j = 0; j < 4; ++j) bf[j] = sm.b[s][kk + (lane & 3)][wn * 32 + j * 8 + (lane >> 2)];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) dmma(acc[i][j], af[i], bf[j]);
    }
    __syncthreads();
  }
  // accumulator (i, j, h) is C[row, col]: row = 8 i + lane / 4, col = 8 j + 2 (lane % 4) + h inside the warp tile
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int64_t gi = m0 + wm * 32 + i * 8 + (lane >> 2);
        const int64_t gj = n0 + wn * 32 + j * 8 + 2 * (lane & 3) + h;
        if (gi < m && gj < n) {
          if (partial != nullptr)
            partial[((int64_t)blockIdx.z * m + gi) * n + gj] = acc[i][j][h];
          else
            c[gi * ldc + gj] = ep_apply(acc[i][j][h], ep, gi, gj);
        }
      }
}

// C[i, j] = epilogue(sum over z ascending of partial[z, i, j])
__global__ void __launch_bounds__(256) gemm_f64_reduce_kernel(int64_t m, int64_t n, int splits,
                                                             const double* __restrict__ partial, double* __restrict__ c,
                                                             int64_t ldc, Epilogue64 ep) {
  const int64_t idx = (int64_t)blockIdx.x * 256 + threadIdx.x;
  const int64_t total = m * n;
  if (idx >= total) return;
  double t = partial[idx];
  for (int z = 1; z < splits; ++z) t += partial[(int64_t)z * total + idx];
  const int64_t i = idx / n, j = idx % n;
  c[i * ldc + j] = ep_apply(t, ep, i, j);
}

struct GemmPlan {
  int bm, bn;
  int64_t mt, nt;
  int splits;
  int64_t k_per_split;
};

GemmPlan plan(int64_t m, int64_t n, int64_t k) {
  GemmPlan p;
  p.bm = 64;
  p.bn = n <= 32 ? 32 : 64;
  p.mt = ceil_div(m, p.bm);
  p.nt = ceil_div(n, p.bn);
  const int64_t tiles = p.mt * p.nt;
  int64_t s = 1;
  if (k > 2 * kMinKPerSplit && tiles < 2 * kNumSMs) {
    s = ceil_div(2 * kNumSMs, tiles);
    const int64_t by_k = k / kMinKPerSplit;
    if (s > by_k) s = by_k;
    if (s > kMaxSplits) s = kMaxSplits;
    if (s < 1) s = 1;
  }
  p.k_per_split = ceil_div(ceil_div(k, s), kBK) * kBK;
  p.splits = (int)(k > 0 ? ceil_div(k, p.k_per_split) : 1);
  return p;
}

}  // namespace

size_t gemm_f64_workspace_bytes(int64_t m, int64_t n, int64_t k) {
  if (m <= 0 || n <= 0 || k <= 0) return 0;
  const GemmPlan p = plan(m, n, k);
  if (p.splits <= 1) return 0;
  return ((size_t)p.splits * (size_t)m * (size_t)n * sizeof(double) + 255) & ~(size_t)255;
}

int gemm_f64_launch(int64_t m, int64_t n, int64_t k, const double* a, int64_t a_rs, int64_t a_cs, const double* b,
                    int64_t b_rs, int64_t b_cs, double* c, int64_t ldc, const Epilogue64& ep, void* ws, size_t ws_bytes,
                    cudaStream_t st) {
  GCNB_REQUIRE(m >= 0 && n >= 0 && k >= 0, "gemm_f64: negative dimension");
  GCNB_REQUIRE(ldc >= n, "gemm_f64: ldc < n");
  if (m == 0 || n == 0) return GCNB_OK;
  GCNB_REQUIRE(c != nullptr, "gemm_f64: null output");
  GCNB_REQUIRE(k == 0 || (a != nullptr && b != nullptr), "gemm_f64: null operand");
  GCNB_REQUIRE(a_rs >= 0 && a_cs >= 0 && b_rs >= 0 && b_cs >= 0, "gemm_f64: negative stride");
  GCNB_REQUIRE(((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b) | reinterpret_cast<uintptr_t>(c) |
                 reinterpret_cast<uintptr_t>(ep.bias)) & 7u) == 0, "gemm_f64: operands must be 8-byte aligned");
  GCNB_REQUIRE(ep.mask == nullptr || ep.ld_mask >= n, "gemm_f64: dropout mask leading dimension smaller than n");
  GCNB_REQUIRE((double)m * (double)(ldc) < 9.2e18 && (double)m * (double)n * kMaxSplits < 9.2e18,
               "gemm_f64: operand extent overflows 64-bit indexing");
  const GemmPlan p = plan(m, n, k);
  GCNB_REQUIRE(p.mt < (1ll << 31) && p.nt < 65536, "gemm_f64: too many tiles (n > %lld)", 65535ll * p.bn);
  const size_t need = gemm_f64_workspace_bytes(m, n, k);
  GCNB_REQUIRE(ws_bytes >= need && (need == 0 || ws != nullptr), "gemm_f64: workspace too small (%zu < %zu)", ws_bytes, need);
  GCNB_REQUIRE((reinterpret_cast<uintptr_t>(ws) & 7u) == 0, "gemm_f64: workspace not 8-byte aligned");
  double* partial = p.splits > 1 ? reinterpret_cast<double*>(ws) : nullptr;
  const dim3 grid((unsigned)p.mt, (unsigned)p.nt, (unsigned)p.splits);
  if (p.bn == 32)
    gemm_f64_dmma_kernel<64, 32><<<grid, GemmTile<64, 32>::kThreads, 0, st>>>(m, n, k, a, a_rs, a_cs, b, b_rs, b_cs, c,
                                                                              ldc, p.k_per_split, ep, partial);
  else
    gemm_f64_dmma_kernel<64, 64><<<grid, GemmTile<64, 64>::kThreads, 0, st>>>(m, n, k, a, a_rs, a_cs, b, b_rs, b_cs, c,
                                                                              ldc, p.k_per_split, ep, partial);
  GCNB_LAUNCH_CHECK();
  if (partial != nullptr) {
    gemm_f64_reduce_kernel<<<(unsigned)ceil_div(m * n, 256), 256, 0, st>>>(m, n, p.splits, partial, c, ldc, ep);
    GCNB_LAUNCH_CHECK();
  }
  return GCNB_OK;
}

}  // namespace gcnb
