// tcgen05 (5th-gen tensor core) GEMMs for the dense contractions of the GCN layer, fp32 in /
// fp32 out with fp32-level accuracy through the 3-term TF32 split ("3xTF32"):
//     a = a_hi + a_lo,  b = b_hi + b_lo   (lo = a - hi, exact)
//     a*b ~= a_lo*b_hi + a_hi*b_lo + a_hi*b_hi          (fp32 accumulate in TMEM)
//
//   mode R ("rows"):  C[M,N] = A[M,K] * B[K,N], A row-major with K contiguous, M huge, K/N small
//                     support = X W (pygcn/layers.py:33) and dX = dS W^T (MmBackward0).
//                     B is tiny: a pre-pass packs it once into hi/lo images (hi = cvt.rna.tf32) that
//                     already have the UMMA shared-memory layout, the main kernel pulls them with
//                     cp.async.bulk (TMA, mbarrier complete_tx); A arrives in K-major tiles by TMA
//                     tensor-map loads and is split in shared memory (hi = the raw words, truncated).
//   mode T ("tn"):    C[M,N] = sum_r X[r,M]^T * Y[r,N]: both operands row-major with the
//                     reduction index outermost (dW = X^T dS).  Rows are split across CTAs
//                     (split-K); both operands arrive by TMA as MN-major tiles and are split
//                     the same way; partial tiles are reduced in a fixed order (deterministic).
//
// K-major operand tiles in shared memory have the canonical SWIZZLE_128B layout (rows of 32 tf32 = 128 B,
// 16-byte chunk c of row r stored at chunk c ^ (r & 7), 8-row groups 1024 B apart), accumulators live in
// TMEM (128 lanes x N columns fp32), tcgen05.mma is issued by one thread, completion is tracked with
// tcgen05.commit -> mbarrier, the epilogue reads TMEM with tcgen05.ld.  Both kernels are warp-specialised
// (TMA producer, splitters, MMA issuer, epilogue), one CTA per SM, with as many operand stages as fit.
#include <cuda.h>  // CUtensorMap types only: the encoder is fetched with cudaGetDriverEntryPoint (no libcuda link)
#include <string.h>

#include "common.cuh"
#include "ptx.cuh"

namespace gcnb {
namespace {

constexpr int BM = 128;       // UMMA M
constexpr int BKF = 32;        // floats per K block (one 128-byte swizzle row)
constexpr int kTileBytes = BM * 128;  // one 128-row operand tile (hi or lo)
constexpr int kChunkBlocks = 8;  // K blocks (of 32) accumulated inside TMEM before a drain
constexpr int kTnDrainBlocks = 16;  // K blocks (of 32 rows) accumulated in TMEM between drains

__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// K-major SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor):
// start>>4 [0,14) | LBO>>4 [16,30) (=1, unused) | SBO>>4 [32,46) (=1024 B) | version=1 [46,48) | layout=2 [61,64)
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// MN-major descriptor for 32-bit operands: the only swizzled MN-major layout tf32 has is
// SWIZZLE_128B_BASE32B (cute Layout_MN_SW128_32B_Atom): atoms of 4 K-rows x 128 B (32 contiguous
// M/N elements), 32-byte chunk c of row r stored at chunk c ^ (r & 3).
// LBO = byte stride between consecutive 32-element M/N groups, SBO = byte stride between 4-row K groups
__device__ __forceinline__ uint64_t make_desc_mn(uint32_t smem_addr, uint32_t lbo, uint32_t sbo) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)((lbo >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)1 << 61;  // SWIZZLE_128B_BASE32B
  return d;
}
// kind::tf32 instruction descriptor (cute::UMMA::InstrDescriptor): D=f32, A=B=tf32;
// mn_major sets a_major_/b_major_ (bits 15/16) for MN-major operands
__host__ __device__ inline uint32_t make_idesc(int n, bool mn_major = false) {
  return (1u << 4) | (2u << 7) | (2u << 10) | (mn_major ? (3u << 15) : 0u) | ((uint32_t)(n >> 3) << 17) |
         ((uint32_t)(BM >> 4) << 24);
}

__device__ __forceinline__ void split_tf32(float v, float& hi, float& lo) {
  uint32_t h;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(h) : "f"(v));
  hi = __uint_as_float(h);
  lo = v - hi;
}

// byte offset of (row r, float column k) inside a K-major SW128 tile
__device__ __forceinline__ uint32_t sw128_off(int r, int k) {
  return (uint32_t)(r * 128 + ((((k >> 2) ^ (r & 7)) << 4) | ((k & 3) << 2)));
}

// One K block: 4 K-steps of 8 tf32, 3 MMAs each.  first = first K block of the tile.
__device__ __forceinline__ void issue_kblock(uint32_t tmem_d, uint32_t a_hi, uint32_t a_lo, uint32_t b_hi,
                                             uint32_t b_lo, uint32_t idesc, bool first) {
  const uint64_t dah = make_desc(a_hi), dal = make_desc(a_lo), dbh = make_desc(b_hi), dbl = make_desc(b_lo);
#pragma unroll
  for (int ks = 0; ks < BKF / 8; ++ks) {
    const uint64_t adv = (uint64_t)((ks * 32) >> 4);  // 32 bytes per K step inside the swizzle row
    umma_tf32(tmem_d, dal + adv, dbh + adv, idesc, (first && ks == 0) ? 0u : 1u);
    umma_tf32(tmem_d, dah + adv, dbl + adv, idesc, 1u);
    umma_tf32(tmem_d, dah + adv, dbh + adv, idesc, 1u);
  }
}

// ------------------------------------------------------------------ B packing (mode R)
// image[(nt * nkb + kb)][n][32 floats, swizzled]; zero padded in n and k.
// (PDL: the programmatic-dependent-launch instantiation, common.cuh)
template <bool PDL>
__global__ void __launch_bounds__(256)
pack_b_kernel(int64_t K, int64_t N, int npad, int n_tiles, int nkb, const float* __restrict__ b, int64_t b_rs,
              int64_t b_cs, float* __restrict__ img_hi, float* __restrict__ img_lo) {
  if constexpr (PDL) {
    pdl_launch_dependents();
    pdl_wait();  // B (the weights) may have been written by the previous kernel of the stream
  }
  const int64_t total = (int64_t)n_tiles * nkb * npad * BKF;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int kk = (int)(i % BKF);
    const int n = (int)((i / BKF) % npad);
    const int64_t blk = i / ((int64_t)BKF * npad);
    const int kb = (int)(blk % nkb);
    const int nt = (int)(blk / nkb);
    const int64_t gk = (int64_t)kb * BKF + kk;
    const int64_t gn = (int64_t)nt * npad + n;
    float v = 0.f;
    if (gk < K && gn < N) v = __ldg(b + gk * b_rs + gn * b_cs);
    float hi, lo;
    split_tf32(v, hi, lo);
    const int64_t dst = blk * ((int64_t)npad * BKF) + (sw128_off(n, kk) >> 2);
    img_hi[dst] = hi;
    img_lo[dst] = lo;
  }
}

// ------------------------------------------------------------------ mode R kernel
// A moved through registers (HBM -> LDG -> split -> STS) keeps only one or two 16 KB K blocks ahead per thread
// (16-48 KB in flight per SM): such a kernel measured 1.7 TB/s on the shapes that are pure streams
// (papers100M-shaped 13.8 M x 128 -> 128: 8.2 ms for 14.1 GB).  Here the copy engine does the streaming and the
// SM only does arithmetic:
//   warp  5    TMA producer: one thread issues cp.async.bulk.tensor.2d per (M tile, K block): a 128 x 32 fp32
//              box of A, SWIZZLE_128B, lands in stage s as the K-major UMMA tile; rows / columns past the
//              matrix are zero-filled by the tensor map.  With ns stages, (ns-1) x 16 KB stay in flight.
//              When the packed B does not fit in shared memory, its (hi, lo) K block rides in the same stage.
//   warps 6-9  splitters: wait raw_full[s]; a_lo = a - tf32(a) written to the stage's second tile at the SAME
//              byte offsets (the swizzle is a property of the address, so no index arithmetic); the raw tile
//              itself is the hi operand -- kind::tf32 reads the upper 19 bits of each word, i.e. truncates, and
//              a - trunc(a) is exact in fp32.
//   warp  4    MMA issuer (one thread): 12 tcgen05.mma per K block into one of two TMEM accumulators,
//              tcgen05.commit -> empty[s] / acc_full[a].
//   warps 0-3  epilogue: tcgen05.ld 32 columns -> registers -> per-warp shared staging (row stride 36 floats,
//              conflict free) -> global stores in which 8 lanes write one full 128-byte line of a C row
//              (lane-per-row stores would touch 32 lines per instruction).
constexpr int kTmaThreads = 320;
constexpr int kEpiLd = 36;
constexpr int kTmaMaxStages = 8;

__device__ __forceinline__ void tma_load_2d(uint32_t dst, const void* tmap, int c0, int c1, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
      "l"(tmap), "r"(c0), "r"(c1), "r"(bar)
      : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

struct alignas(64) TmaDesc { uint8_t bytes[128]; };  // CUtensorMap (opaque, 128 bytes, 64-byte aligned)

template <bool PDL>
__global__ void __launch_bounds__(kTmaThreads, 1)
gemm_tc_rows_tma_kernel(const __grid_constant__ TmaDesc tmap_a, int64_t M, int N, int K,
                        const float* __restrict__ img_hi, const float* __restrict__ img_lo, float* __restrict__ c,
                        int64_t ldc, int npad, int nkb, int tmem_cols, int vec_ok, int ns, int b_resident,
                        const float* __restrict__ ep_bias, int ep_relu) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gen = smem_raw + (base - smem_u32(smem_raw));
  // layout: [ns x (a_raw 16K, a_lo 16K, (b_hi, b_lo when streamed))] [resident B: nkb x (b_hi, b_lo)]
  //         [epilogue staging 4 x 32 x 36 floats] [barriers]
  const uint32_t b_bytes = (uint32_t)npad * 128;
  const uint32_t stage_bytes = 2u * kTileBytes + (b_resident ? 0u : 2u * b_bytes);
  const uint32_t off_b = (uint32_t)ns * stage_bytes;
  const uint32_t off_epi = off_b + (b_resident ? (uint32_t)nkb * 2u * b_bytes : 0u);
  const uint32_t off_bar = (off_epi + 4u * 32u * kEpiLd * 4u + 1023u) & ~1023u;
  auto bar_raw = [&](int s_) { return base + off_bar + 8u * (uint32_t)s_; };
  auto bar_split = [&](int s_) { return base + off_bar + 64u + 8u * (uint32_t)s_; };
  auto bar_empty = [&](int s_) { return base + off_bar + 128u + 8u * (uint32_t)s_; };
  const uint32_t bar_b = base + off_bar + 192u;
  auto bar_acc_full = [&](int a_) { return base + off_bar + 200u + 8u * (uint32_t)a_; };
  auto bar_acc_empty = [&](int a_) { return base + off_bar + 216u + 8u * (uint32_t)a_; };
  const uint32_t tmem_slot_off = off_bar + 232u;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0) {
    for (int i = 0; i < ns; ++i) { mbar_init(bar_raw(i), 1); mbar_init(bar_split(i), 4); mbar_init(bar_empty(i), 1); }
    mbar_init(bar_b, 1);
    for (int i = 0; i < 2; ++i) { mbar_init(bar_acc_full(i), 1); mbar_init(bar_acc_empty(i), 4); }
    fence_barrier_init();
  }
  if (warp == 4) {
    __syncwarp();
    tmem_alloc(base + tmem_slot_off, (uint32_t)tmem_cols);
  }
  if constexpr (PDL) pdl_launch_dependents();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(gen + tmem_slot_off);
  // barriers initialised and TMEM allocated while the previous kernel (the pack of B) drains; A, the packed B and C
  // are touched only from here on
  if constexpr (PDL) pdl_wait();

  const int nt = blockIdx.y;
  const int n0 = nt * npad;
  const int n_cols = min(npad, N - n0);
  const int64_t m_tiles = (M + BM - 1) / BM;
  const int64_t my_tiles = (m_tiles > (int64_t)blockIdx.x) ? (m_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
  const int64_t n_items = my_tiles * nkb;
  const int chunks_per_tile = (nkb + kChunkBlocks - 1) / kChunkBlocks;

  if (warp == 5) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      if (b_resident) {
        mbar_expect_tx(bar_b, 2 * b_bytes * (uint32_t)nkb);
        for (int kb = 0; kb < nkb; ++kb) {
          const int64_t blk = (int64_t)nt * nkb + kb;
          bulk_g2s(base + off_b + (uint32_t)kb * 2 * b_bytes, img_hi + blk * ((int64_t)npad * BKF), b_bytes, bar_b);
          bulk_g2s(base + off_b + (uint32_t)kb * 2 * b_bytes + b_bytes, img_lo + blk * ((int64_t)npad * BKF), b_bytes, bar_b);
        }
      }
      int64_t item = 0;
      for (int64_t t = 0; t < my_tiles; ++t) {
        const int64_t m0 = ((int64_t)blockIdx.x + t * gridDim.x) * BM;
        for (int kb = 0; kb < nkb; ++kb, ++item) {
          const int s = (int)(item % ns);
          const uint32_t use = (uint32_t)(item / ns);
          if (use > 0) mbar_wait(bar_empty(s), (use - 1) & 1);
          const uint32_t st_base = base + (uint32_t)s * stage_bytes;
          mbar_expect_tx(bar_raw(s), (uint32_t)kTileBytes + (b_resident ? 0u : 2u * b_bytes));
          tma_load_2d(st_base, &tmap_a, kb * BKF, (int)m0, bar_raw(s));
          if (!b_resident) {
            const int64_t blk = (int64_t)nt * nkb + kb;
            bulk_g2s(st_base + 2u * kTileBytes, img_hi + blk * ((int64_t)npad * BKF), b_bytes, bar_raw(s));
            bulk_g2s(st_base + 2u * kTileBytes + b_bytes, img_lo + blk * ((int64_t)npad * BKF), b_bytes, bar_raw(s));
          }
        }
      }
    }
  } else if (warp >= 6) {
    // ===================== splitters =====================
    const int pt = tid - 192;  // 0..127
    for (int64_t item = 0; item < n_items; ++item) {
      const int s = (int)(item % ns);
      const uint32_t use = (uint32_t)(item / ns);
      mbar_wait(bar_raw(s), use & 1);
      uint8_t* raw = gen + (uint32_t)s * stage_bytes;
      uint8_t* lo_t = raw + kTileBytes;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const uint32_t off = 16u * (uint32_t)(pt + 128 * j);
        const float4 v = *reinterpret_cast<const float4*>(raw + off);
        float4 lo;
        lo.x = v.x - __uint_as_float(__float_as_uint(v.x) & 0xffffe000u);
        lo.y = v.y - __uint_as_float(__float_as_uint(v.y) & 0xffffe000u);
        lo.z = v.z - __uint_as_float(__float_as_uint(v.z) & 0xffffe000u);
        lo.w = v.w - __uint_as_float(__float_as_uint(v.w) & 0xffffe000u);
        *reinterpret_cast<float4*>(lo_t + off) = lo;
      }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_split(s));
    }
  } else if (warp == 4) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      const uint32_t idesc = make_idesc(npad);
      if (b_resident) mbar_wait(bar_b, 0);
      int64_t item = 0;
      uint32_t chunk_ctr = 0;
      for (int64_t t = 0; t < my_tiles; ++t) {
        for (int kb = 0; kb < nkb; ++kb, ++item) {
          const int ab = (int)(chunk_ctr & 1u);
          const uint32_t j_use = chunk_ctr >> 1;
          if (kb % kChunkBlocks == 0 && j_use > 0) mbar_wait(bar_acc_empty(ab), (j_use - 1) & 1);
          const int s = (int)(item % ns);
          const uint32_t use = (uint32_t)(item / ns);
          mbar_wait(bar_split(s), use & 1);
          tc_fence_after();
          const uint32_t a_hi = base + (uint32_t)s * stage_bytes;
          const uint32_t bh = b_resident ? base + off_b + (uint32_t)kb * 2 * b_bytes : a_hi + 2u * kTileBytes;
          issue_kblock(tmem_base + (uint32_t)ab * (uint32_t)npad, a_hi, a_hi + kTileBytes, bh, bh + b_bytes, idesc,
                       kb % kChunkBlocks == 0);
          umma_commit(bar_empty(s));
          if (kb == nkb - 1 || kb % kChunkBlocks == kChunkBlocks - 1) {
            umma_commit(bar_acc_full(ab));
            ++chunk_ctr;
          }
        }
      }
    }
  } else {
    // ===================== epilogue =====================
    float* stg = reinterpret_cast<float*>(gen + off_epi) + warp * 32 * kEpiLd;
    uint32_t chunk_ctr = 0;
    for (int64_t t = 0; t < my_tiles; ++t) {
      const int64_t m0 = ((int64_t)blockIdx.x + t * gridDim.x) * BM + warp * 32;
      for (int ch = 0; ch < chunks_per_tile; ++ch, ++chunk_ctr) {
        const int ab = (int)(chunk_ctr & 1u);
        mbar_wait(bar_acc_full(ab), (chunk_ctr >> 1) & 1);
        tc_fence_after();
        const bool add = ch > 0;
        // fused epilogue of the layer's aggregate-first order (out = (A X) W + bias, ReLU): applied with the last K chunk
        const bool fin_ep = (ch == chunks_per_tile - 1) && (ep_bias != nullptr || ep_relu != 0);
        for (int cb = 0; cb < n_cols; cb += 32) {
          uint32_t r[32];
          __syncwarp();
          tmem_ld32(tmem_base + (uint32_t)ab * (uint32_t)npad + ((uint32_t)(warp * 32) << 16) + (uint32_t)cb, r);
#pragma unroll
          for (int q = 0; q < 8; ++q)
            *reinterpret_cast<uint4*>(stg + lane * kEpiLd + 4 * q) = make_uint4(r[4 * q], r[4 * q + 1], r[4 * q + 2], r[4 * q + 3]);
          __syncwarp();
          const int q = lane & 7;
          const int col = cb + 4 * q;  // column inside this N tile
          float bv[4] = {0.f, 0.f, 0.f, 0.f};
          if (fin_ep && ep_bias != nullptr) {
#pragma unroll
            for (int t2 = 0; t2 < 4; ++t2)
              if (col + t2 < n_cols) bv[t2] = __ldg(ep_bias + n0 + col + t2);
          }
          // Fast path (whole 32 x 32 blocks of an aligned C): 128-bit stores without per-store predicates.  The general
          // loop below costs ~40 instructions and several dependent branches per store and made the epilogue the
          // floor of every 256-wide product (7.9 us per 128 x 256 tile whatever K: profiles/r02_gemm_k_sweep.txt); it
          // keeps the last rows and a ragged last column block (47 classes).
          if (vec_ok && m0 + 32 <= M && cb + 32 <= n_cols) {  // (warp-uniform)
            const float* sp = stg + (lane >> 3) * kEpiLd + 4 * q;
            float* dp = c + (m0 + (lane >> 3)) * ldc + n0 + col;
            if (!add && !fin_ep) {
#pragma unroll
              for (int i = 0; i < 8; ++i)
                *reinterpret_cast<float4*>(dp + (int64_t)(4 * i) * ldc) = *reinterpret_cast<const float4*>(sp + 4 * i * kEpiLd);
            } else {
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                float4 v = *reinterpret_cast<const float4*>(sp + 4 * i * kEpiLd);
                float* dst = dp + (int64_t)(4 * i) * ldc;
                if (add) {
                  const float4 p = *reinterpret_cast<const float4*>(dst);
                  v.x += p.x; v.y += p.y; v.z += p.z; v.w += p.w;
                }
                if (fin_ep) {
                  v.x += bv[0]; v.y += bv[1]; v.z += bv[2]; v.w += bv[3];
                  if (ep_relu) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
                }
                *reinterpret_cast<float4*>(dst) = v;
              }
            }
            continue;
          }
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int rr = 4 * i + (lane >> 3);
            float4 v = *reinterpret_cast<const float4*>(stg + rr * kEpiLd + 4 * q);
            const int64_t row = m0 + rr;
            if (row < M && col < n_cols) {
              float* dst = c + row * ldc + n0 + col;
              if (vec_ok && col + 4 <= n_cols) {
                if (add) {
                  const float4 p = *reinterpret_cast<const float4*>(dst);
                  v.x += p.x; v.y += p.y; v.z += p.z; v.w += p.w;
                }
                if (fin_ep) {
                  v.x += bv[0]; v.y += bv[1]; v.z += bv[2]; v.w += bv[3];
                  if (ep_relu) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
                }
                *reinterpret_cast<float4*>(dst) = v;
              } else {
                const float e[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int t2 = 0; t2 < 4; ++t2)
                  if (col + t2 < n_cols) {
                    float o = add ? dst[t2] + e[t2] : e[t2];
                    if (fin_ep) {
                      o += bv[t2];
                      if (ep_relu) o = fmaxf(o, 0.f);
                    }
                    dst[t2] = o;
                  }
              }
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_acc_empty(ab));
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 4) {
    __syncwarp();
    tmem_dealloc(tmem_base, (uint32_t)tmem_cols);
  }
}

// ------------------------------------------------------------------ mode T kernel, TMA-fed
// C_partial[split][128-row M tile][npad] = sum over the split's rows r of X[r, m0:m0+128]^T Y[r, 0:npad]
// with the same division of labour as gemm_tc_rows_tma_kernel.  Both operands are MN-major (a reduction row
// holds contiguous M resp. N elements), so the UMMA tiles are SWIZZLE_128B_BASE32B atoms of 4 reduction rows x
// 32 elements -- exactly what a tensor map with CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B writes for a box of 32
// floats x 32 rows.  One K block (32 reduction rows) = 4 boxes of X (M groups, 4 KB apart) + npad/32 boxes of
// Y; columns past the matrices' widths and rows past R arrive as zeros.  K step ks of a block starts 1 KB
// into every box (two 4-row K groups of 512 B), LBO = 4096 (next M/N group), SBO = 512 (next K group).
__global__ void __launch_bounds__(kTmaThreads, 1)
gemm_tc_tn_tma_kernel(const __grid_constant__ TmaDesc tmap_x, const __grid_constant__ TmaDesc tmap_y, int64_t R, int M,
                      int N, float* __restrict__ c, int64_t ldc, int64_t split_stride, int64_t rows_per_split, int npad,
                      int tmem_cols, int vec_ok, int ns) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gen = smem_raw + (base - smem_u32(smem_raw));
  // stage: [x_raw 16K][y_raw npad*128][x_lo 16K][y_lo npad*128]  (raw | lo halves have the same internal offsets)
  const uint32_t y_bytes = (uint32_t)npad * 128;
  const uint32_t half = (uint32_t)kTileBytes + y_bytes;
  const uint32_t stage_bytes = 2u * half;
  const uint32_t off_epi = (uint32_t)ns * stage_bytes;
  const uint32_t off_bar = (off_epi + 4u * 32u * kEpiLd * 4u + 1023u) & ~1023u;
  auto bar_raw = [&](int s_) { return base + off_bar + 8u * (uint32_t)s_; };
  auto bar_split = [&](int s_) { return base + off_bar + 64u + 8u * (uint32_t)s_; };
  auto bar_empty = [&](int s_) { return base + off_bar + 128u + 8u * (uint32_t)s_; };
  auto bar_acc_full = [&](int a_) { return base + off_bar + 200u + 8u * (uint32_t)a_; };
  auto bar_acc_empty = [&](int a_) { return base + off_bar + 216u + 8u * (uint32_t)a_; };
  const uint32_t tmem_slot_off = off_bar + 232u;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0) {
    for (int i = 0; i < ns; ++i) { mbar_init(bar_raw(i), 1); mbar_init(bar_split(i), 4); mbar_init(bar_empty(i), 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(bar_acc_full(i), 1); mbar_init(bar_acc_empty(i), 4); }
    fence_barrier_init();
  }
  if (warp == 4) {
    __syncwarp();
    tmem_alloc(base + tmem_slot_off, (uint32_t)tmem_cols);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(gen + tmem_slot_off);

  const int m0 = blockIdx.x * BM;  // (M tiles on x: y would cap them at 65535, M at 8.4 M)
  const int64_t r_begin = (int64_t)blockIdx.y * rows_per_split;
  const int64_t r_end = min(R, r_begin + rows_per_split);
  const int nkb = (r_end > r_begin) ? (int)((r_end - r_begin + BKF - 1) / BKF) : 0;
  const int n_chunks = (nkb + kTnDrainBlocks - 1) / kTnDrainBlocks;
  const int ng = npad >> 5;
  float* cdst = c + (int64_t)blockIdx.y * split_stride;

  if (warp == 5) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      for (int kb = 0; kb < nkb; ++kb) {
        const int s = kb % ns;
        const uint32_t use = (uint32_t)(kb / ns);
        if (use > 0) mbar_wait(bar_empty(s), (use - 1) & 1);
        const uint32_t st_base = base + (uint32_t)s * stage_bytes;
        const int r0 = (int)(r_begin + (int64_t)kb * BKF);
        mbar_expect_tx(bar_raw(s), half);
#pragma unroll
        for (int mg = 0; mg < 4; ++mg) tma_load_2d(st_base + (uint32_t)mg * 4096u, &tmap_x, m0 + 32 * mg, r0, bar_raw(s));
        for (int g = 0; g < ng; ++g)
          tma_load_2d(st_base + (uint32_t)kTileBytes + (uint32_t)g * 4096u, &tmap_y, 32 * g, r0, bar_raw(s));
      }
    }
  } else if (warp >= 6) {
    // ===================== splitters =====================
    const int pt = tid - 192;  // 0..127
    const int n16 = (int)(half >> 4);  // 16-byte chunks of the raw half (multiple of 128)
    for (int kb = 0; kb < nkb; ++kb) {
      const int s = kb % ns;
      const uint32_t use = (uint32_t)(kb / ns);
      mbar_wait(bar_raw(s), use & 1);
      uint8_t* raw = gen + (uint32_t)s * stage_bytes;
      uint8_t* lo_t = raw + half;
#pragma unroll 4
      for (int i = pt; i < n16; i += 128) {
        const uint32_t off = 16u * (uint32_t)i;
        const float4 v = *reinterpret_cast<const float4*>(raw + off);
        float4 lo;
        lo.x = v.x - __uint_as_float(__float_as_uint(v.x) & 0xffffe000u);
        lo.y = v.y - __uint_as_float(__float_as_uint(v.y) & 0xffffe000u);
        lo.z = v.z - __uint_as_float(__float_as_uint(v.z) & 0xffffe000u);
        lo.w = v.w - __uint_as_float(__float_as_uint(v.w) & 0xffffe000u);
        *reinterpret_cast<float4*>(lo_t + off) = lo;
      }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_split(s));
    }
  } else if (warp == 4) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      const uint32_t idesc = make_idesc(npad, true);
      uint32_t chunk_ctr = 0;
      for (int kb = 0; kb < nkb; ++kb) {
        const int ab = (int)(chunk_ctr & 1u);
        const uint32_t j_use = chunk_ctr >> 1;
        const bool first = (kb % kTnDrainBlocks) == 0;
        if (first && j_use > 0) mbar_wait(bar_acc_empty(ab), (j_use - 1) & 1);
        const int s = kb % ns;
        const uint32_t use = (uint32_t)(kb / ns);
        mbar_wait(bar_split(s), use & 1);
        tc_fence_after();
        const uint32_t xh = base + (uint32_t)s * stage_bytes, yh = xh + (uint32_t)kTileBytes;
        const uint32_t xl = xh + half, yl = yh + half;
        const uint32_t d = tmem_base + (uint32_t)ab * (uint32_t)npad;
#pragma unroll
        for (int ks = 0; ks < BKF / 8; ++ks) {
          const uint32_t o = (uint32_t)ks * 1024u;
          const uint64_t dxh = make_desc_mn(xh + o, 4096u, 512u), dxl = make_desc_mn(xl + o, 4096u, 512u);
          const uint64_t dyh = make_desc_mn(yh + o, 4096u, 512u), dyl = make_desc_mn(yl + o, 4096u, 512u);
          umma_tf32(d, dxl, dyh, idesc, (first && ks == 0) ? 0u : 1u);
          umma_tf32(d, dxh, dyl, idesc, 1u);
          umma_tf32(d, dxh, dyh, idesc, 1u);
        }
        umma_commit(bar_empty(s));
        if (kb == nkb - 1 || (kb % kTnDrainBlocks) == kTnDrainBlocks - 1) {
          umma_commit(bar_acc_full(ab));
          ++chunk_ctr;
        }
      }
    }
  } else {
    // ===================== epilogue: partial tile rows m0 + 32*warp .. (TMEM lane = m) =====================
    float* stg = reinterpret_cast<float*>(gen + off_epi) + warp * 32 * kEpiLd;
    const int q = lane & 7;
    if (nkb == 0) {  // an empty split still owns its partial tile
      for (int i = lane; i < 32 * N; i += 32) {
        const int row = m0 + warp * 32 + i / N;
        if (row < M) cdst[(int64_t)row * ldc + (i % N)] = 0.f;
      }
    }
    for (int ch = 0; ch < n_chunks; ++ch) {
      const int ab = ch & 1;
      mbar_wait(bar_acc_full(ab), (uint32_t)(ch >> 1) & 1u);
      tc_fence_after();
      const bool add = ch > 0;
      for (int cb = 0; cb < N; cb += 32) {
        uint32_t r[32];
        __syncwarp();
        tmem_ld32(tmem_base + (uint32_t)ab * (uint32_t)npad + ((uint32_t)(warp * 32) << 16) + (uint32_t)cb, r);
#pragma unroll
        for (int qq = 0; qq < 8; ++qq)
          *reinterpret_cast<uint4*>(stg + lane * kEpiLd + 4 * qq) = make_uint4(r[4 * qq], r[4 * qq + 1], r[4 * qq + 2], r[4 * qq + 3]);
        __syncwarp();
        const int col = cb + 4 * q;
        // Fast path for whole 32 x 32 blocks: the eight read-modify-write groups of a block are independent -- all
        // loads first, then the adds, then the stores.  In the general loop below every group waits for its own load
        // behind a chain of predicates (~700 cycles each): a drain of a 128 x 256 tile then outlasts the 16 K blocks
        // of MMAs it is meant to hide behind.
        if (vec_ok && m0 + warp * 32 + 32 <= M && cb + 32 <= N) {  // (warp-uniform)
          const float* sp = stg + (lane >> 3) * kEpiLd + 4 * q;
          float* dp = cdst + (int64_t)(m0 + warp * 32 + (lane >> 3)) * ldc + col;
          float4 v[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) v[i] = *reinterpret_cast<const float4*>(sp + 4 * i * kEpiLd);
          if (add) {
            float4 pv[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) pv[i] = *reinterpret_cast<const float4*>(dp + (int64_t)(4 * i) * ldc);
#pragma unroll
            for (int i = 0; i < 8; ++i) { v[i].x += pv[i].x; v[i].y += pv[i].y; v[i].z += pv[i].z; v[i].w += pv[i].w; }
          }
#pragma unroll
          for (int i = 0; i < 8; ++i) *reinterpret_cast<float4*>(dp + (int64_t)(4 * i) * ldc) = v[i];
          continue;
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int rr = 4 * i + (lane >> 3);
          float4 v = *reinterpret_cast<const float4*>(stg + rr * kEpiLd + 4 * q);
          const int row = m0 + warp * 32 + rr;
          if (row < M && col < N) {
            float* dst = cdst + (int64_t)row * ldc + col;
            if (vec_ok && col + 4 <= N) {
              if (add) {
                const float4 p = *reinterpret_cast<const float4*>(dst);
                v.x += p.x; v.y += p.y; v.z += p.z; v.w += p.w;
              }
              *reinterpret_cast<float4*>(dst) = v;
            } else {
              const float e[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
              for (int t2 = 0; t2 < 4; ++t2)
                if (col + t2 < N) dst[t2] = add ? dst[t2] + e[t2] : e[t2];
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_acc_empty(ab));
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 4) {
    __syncwarp();
    tmem_dealloc(tmem_base, (uint32_t)tmem_cols);
  }
}

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
inline int tmem_cols_for(int npad) {
  int c = 32;
  while (c < npad) c <<= 1;
  return c;
}

// the 227 KB dynamic shared memory opt-in is a per-device attribute of the function: once per (kernel, device)
int allow_big_smem(const void* kernel, int slot) {
  static bool done[3][64] = {};
  int dev = 0;
  GCNB_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64 || !done[slot][dev]) {
    GCNB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    if (dev >= 0 && dev < 64) done[slot][dev] = true;
  }
  return GCNB_OK;
}

struct TmaPlan { int npad, n_tiles, nkb, ns, b_resident; size_t img_floats; uint32_t smem; };
TmaPlan tma_plan(int64_t n, int64_t k) {
  TmaPlan p;
  p.npad = n >= 256 ? 256 : (int)(ceil_div(n, 32) * 32);
  p.n_tiles = (int)ceil_div(n, p.npad);
  p.nkb = (int)ceil_div(k, BKF);
  p.img_floats = (size_t)p.n_tiles * p.nkb * p.npad * BKF;
  const size_t b_total = (size_t)p.nkb * 2 * p.npad * 128;
  const size_t epi = 4 * 32 * kEpiLd * sizeof(float);
  const size_t budget = 227 * 1024 - epi - 1024 /*barriers*/ - 2048 /*alignment*/;
  size_t stage = 2 * kTileBytes;
  if (b_total + 3 * stage <= budget) {
    p.b_resident = 1;
    p.ns = (int)((budget - b_total) / stage);
  } else {
    p.b_resident = 0;
    stage += 2 * (size_t)p.npad * 128;
    p.ns = (int)(budget / stage);
  }
  if (p.ns > kTmaMaxStages) p.ns = kTmaMaxStages;
  const size_t off_epi = (size_t)p.ns * stage + (p.b_resident ? b_total : 0);
  const size_t off_bar = (off_epi + epi + 1023) & ~(size_t)1023;
  p.smem = (uint32_t)(off_bar + 256 + 1024);
  return p;
}

// cuTensorMapEncodeTiled through the runtime's driver entry point table
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
    else
      (void)cudaGetLastError();
  }
  return fn;
}
// A [M, K] fp32 row-major (lda floats) as boxes of 128 rows x 32 floats, SWIZZLE_128B, zero fill outside
bool make_tmap_a(TmaDesc* out, const float* a, int64_t m, int64_t k, int64_t lda) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (!fn || m >= (1ll << 31)) return false;
  CUtensorMap tm;
  const cuuint64_t gdim[2] = {(cuuint64_t)k, (cuuint64_t)m};
  const cuuint64_t gstride[1] = {(cuuint64_t)lda * sizeof(float)};
  const cuuint32_t box[2] = {(cuuint32_t)BKF, (cuuint32_t)BM};
  const cuuint32_t estr[2] = {1, 1};
  if (fn(&tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(a), gdim, gstride, box, estr,
         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
    return false;
  static_assert(sizeof(CUtensorMap) == sizeof(TmaDesc), "CUtensorMap is 128 bytes");
  memcpy(out, &tm, sizeof(tm));
  return true;
}

// X [R, W] fp32 row-major (ld floats) as boxes of 32 floats x 32 rows, SWIZZLE_128B_ATOM_32B (the MN-major UMMA atom)
bool make_tmap_mn(TmaDesc* out, const float* x, int64_t rows, int64_t width, int64_t ld) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (!fn || rows >= (1ll << 31) || width >= (1ll << 31)) return false;
  CUtensorMap tm;
  const cuuint64_t gdim[2] = {(cuuint64_t)width, (cuuint64_t)rows};
  const cuuint64_t gstride[1] = {(cuuint64_t)ld * sizeof(float)};
  const cuuint32_t box[2] = {32u, (cuuint32_t)BKF};
  const cuuint32_t estr[2] = {1, 1};
  if (fn(&tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(x), gdim, gstride, box, estr,
         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
    return false;
  memcpy(out, &tm, sizeof(tm));
  return true;
}

struct TnTmaPlan { int npad, m_tiles, ns; int64_t splits, rows_per_split; uint32_t smem; };
TnTmaPlan tn_tma_plan(int64_t m, int64_t n, int64_t r) {
  TnTmaPlan p;
  p.npad = (int)(ceil_div(n, 32) * 32);
  p.m_tiles = (int)ceil_div(m, BM);
  int64_t s = kNumSMs / p.m_tiles;  // one CTA per SM
  const int64_t max_s = ceil_div(r, 4 * BKF);
  if (s > max_s) s = max_s;
  if (s < 1) s = 1;
  p.rows_per_split = ceil_div(ceil_div(r, s), BKF) * BKF;
  p.splits = ceil_div(r, p.rows_per_split);
  if (p.splits < 1) p.splits = 1;
  const size_t epi = 4 * 32 * kEpiLd * sizeof(float);
  const size_t budget = 227 * 1024 - epi - 1024 - 2048;
  const size_t stage = 2 * ((size_t)kTileBytes + (size_t)p.npad * 128);
  p.ns = (int)(budget / stage);
  if (p.ns > kTmaMaxStages) p.ns = kTmaMaxStages;
  const size_t off_bar = ((size_t)p.ns * stage + epi + 1023) & ~(size_t)1023;
  p.smem = (uint32_t)(off_bar + 256 + 1024);
  return p;
}

}  // namespace

// ------------------------------------------------------------------ host side
bool gemm_tc_rows_eligible(int64_t m, int64_t n, int64_t k, const float* a, int64_t a_rs, int64_t a_cs,
                           const float* c, int64_t ldc) {
  (void)c; (void)ldc;
  return m > 0 && n > 0 && k > 0 && a_cs == 1 && (a_rs % 4 == 0) && (k % 4 == 0) && aligned16(a) &&
         k <= (1 << 20) && n <= (1 << 20) && encode_tiled_fn() != nullptr;
}

size_t gemm_tc_rows_workspace_bytes(int64_t m, int64_t n, int64_t k) {
  (void)m;
  return 2 * tma_plan(n, k).img_floats * sizeof(float) + 256;
}

int gemm_tc_rows_launch(int64_t m, int64_t n, int64_t k, const float* a, int64_t lda, const float* b, int64_t b_rs,
                        int64_t b_cs, float* c, int64_t ldc, void* ws, size_t ws_bytes, cudaStream_t st,
                        const float* ep_bias, int ep_relu) {
  GCNB_REQUIRE(ws != nullptr && ws_bytes >= gemm_tc_rows_workspace_bytes(m, n, k) && aligned16(ws),
               "gemm(tc rows): workspace too small or unaligned");
  const TmaPlan t = tma_plan(n, k);
  GCNB_REQUIRE(t.ns >= 2, "gemm(tc rows): fewer than two operand stages fit in shared memory");
  float* hi = reinterpret_cast<float*>(ws);
  float* lo = hi + ((t.img_floats + 31) & ~(size_t)31);
  int pg = (int)ceil_div((int64_t)t.img_floats, 256);
  if (pg > 4 * kNumSMs) pg = 4 * kNumSMs;
  const int vec = (ldc % 4 == 0) && aligned16(c);
  const int tmem_cols = tmem_cols_for(2 * t.npad);
  const bool pdl = pdl_enabled();  // opt-in: both kernels start while their predecessor drains (common.cuh)
  if (pdl) {
    GCNB_CUDA(launch_pdl(pack_b_kernel<true>, dim3((unsigned)pg), dim3(256), 0, st, k, n, t.npad, t.n_tiles, t.nkb, b,
                         b_rs, b_cs, hi, lo));
    GCNB_TRY(allow_big_smem(reinterpret_cast<const void*>(gemm_tc_rows_tma_kernel<true>), 2));
  } else {
    pack_b_kernel<false><<<pg, 256, 0, st>>>(k, n, t.npad, t.n_tiles, t.nkb, b, b_rs, b_cs, hi, lo);
    GCNB_LAUNCH_CHECK();
    GCNB_TRY(allow_big_smem(reinterpret_cast<const void*>(gemm_tc_rows_tma_kernel<false>), 0));
  }
  // The tensor map takes 32-bit row coordinates: a taller A runs in chunks of whole 128-row tiles, each with a map of
  // its own.  A row's result does not depend on the chunk it is in.
  const int64_t chunk_rows = (1ll << 31) - BM;
  for (int64_t m0 = 0; m0 < m; m0 += chunk_rows) {
    const int64_t mc = (m - m0 < chunk_rows) ? m - m0 : chunk_rows;
    TmaDesc tmap;
    GCNB_REQUIRE(make_tmap_a(&tmap, a + m0 * lda, mc, k, lda), "gemm(tc rows): tensor map encoding failed");
    const int64_t mt = ceil_div(mc, BM);
    int64_t gx = kNumSMs / t.n_tiles;
    if (gx < 1) gx = 1;
    if (gx > mt) gx = mt;
    const dim3 grid((unsigned)gx, (unsigned)t.n_tiles);
    if (pdl) {
      GCNB_CUDA(launch_pdl(gemm_tc_rows_tma_kernel<true>, grid, dim3(kTmaThreads), t.smem, st, tmap, mc, (int)n, (int)k,
                           (const float*)hi, (const float*)lo, c + m0 * ldc, ldc, t.npad, t.nkb, tmem_cols, vec, t.ns,
                           t.b_resident, ep_bias, ep_relu));
    } else {
      gemm_tc_rows_tma_kernel<false><<<grid, kTmaThreads, t.smem, st>>>(tmap, mc, (int)n, (int)k, hi, lo, c + m0 * ldc,
                                                                       ldc, t.npad, t.nkb, tmem_cols, vec, t.ns,
                                                                       t.b_resident, ep_bias, ep_relu);
      GCNB_LAUNCH_CHECK();
    }
  }
  return GCNB_OK;
}

// narrow "rows" products with K >= 32 measure faster on the tensor-core kernel than on the CUDA-core skinny kernel
// (CBG 64->32 X W: 23.1 vs 26.6 us in the step's graph; 8->32: 16.6 vs 12.3)
bool gemm_tc_rows_beats_skinny(int64_t k) { return k >= 32 && encode_tiled_fn() != nullptr; }

// dW-shaped product: C[M,N] = sum_r X[r, 0:M]^T Y[r, 0:N].  The kernel zero-fills past the widths itself; the
// tensor maps take 32-bit coordinates.
bool gemm_tc_tn_eligible(int64_t m, int64_t n, int64_t r, const float* x, int64_t ldx, const float* y, int64_t ldy) {
  return m > 0 && n > 0 && r > 0 && n <= 256 && m < (1ll << 31) && r < (1ll << 31) && (ldx % 4 == 0) &&
         (ldy % 4 == 0) && aligned16(x) && aligned16(y) && encode_tiled_fn() != nullptr;
}

size_t gemm_tc_tn_workspace_bytes(int64_t m, int64_t n, int64_t r) {
  const TnTmaPlan t = tn_tma_plan(m, n, r);
  return t.splits > 1 ? (size_t)t.splits * (size_t)m * (size_t)n * sizeof(float) : 0;
}

int gemm_tc_tn_launch(int64_t m, int64_t n, int64_t r, const float* x, int64_t ldx, const float* y, int64_t ldy,
                      float* c, int64_t ldc, void* ws, size_t ws_bytes, cudaStream_t st) {
  const TnTmaPlan t = tn_tma_plan(m, n, r);
  const size_t need = gemm_tc_tn_workspace_bytes(m, n, r);
  GCNB_REQUIRE(need == 0 || (ws != nullptr && ws_bytes >= need && aligned16(ws)), "gemm(tc tn): workspace too small");
  GCNB_REQUIRE(t.ns >= 2, "gemm(tc tn): fewer than two operand stages fit in shared memory");
  TmaDesc tx, ty;
  GCNB_REQUIRE(make_tmap_mn(&tx, x, r, m, ldx) && make_tmap_mn(&ty, y, r, n, ldy),
               "gemm(tc tn): tensor map encoding failed");
  float* dst = (t.splits > 1) ? reinterpret_cast<float*>(ws) : c;
  const int64_t ld = (t.splits > 1) ? n : ldc;
  const int64_t stride = (t.splits > 1) ? m * n : 0;
  const int vec = (ld % 4 == 0) && aligned16(dst);
  GCNB_TRY(allow_big_smem(reinterpret_cast<const void*>(gemm_tc_tn_tma_kernel), 1));
  gemm_tc_tn_tma_kernel<<<dim3((unsigned)t.m_tiles, (unsigned)t.splits), kTmaThreads, t.smem, st>>>(
      tx, ty, r, (int)m, (int)n, dst, ld, stride, t.rows_per_split, t.npad, tmem_cols_for(2 * t.npad), vec, t.ns);
  GCNB_LAUNCH_CHECK();
  if (t.splits > 1) GCNB_TRY(reduce_partials_launch(m, n, (int)t.splits, dst, c, ldc, st));
  return GCNB_OK;
}

}  // namespace gcnb
