// CSR SpMM for the GCN layer:  out = A * B (+ bias) (ReLU)     -- pygcn/layers.py:34-36,
// and, on the CSR of A^T, the backward product dS = A^T * G     -- SURVEY.md 3.2.
//
// HBM/L2-bound gather kernel, no tensor cores (the work is nnz*F FMAs on gathered rows):
//   * one warp per row for rows below the long-row threshold; the warp's 32 lanes are split
//     into G = 32/LPR "slots" of LPR lanes, every slot gathers a different stored entry's
//     feature row with 128-bit loads (LPR = lanes needed to cover F floats as float4),
//     so one LDG.128 instruction moves G feature rows;
//   * col/val of 32 stored entries are fetched with one coalesced load per lane and
//     broadcast with shuffles;
//   * rows in the long bin (deg >= GCNB_BIN_EDGE_4) are split into chunks of kLongChunk
//     entries, one warp per chunk writes a partial row to scratch, a fix-up kernel adds the
//     partials in chunk order (atomic-free, run-to-run deterministic);
//   * bias add and ReLU are fused in the epilogue.
#include <stdlib.h>

#include <algorithm>
#include <type_traits>

#include "common.cuh"
#include "ptx.cuh"

namespace gcnb {

namespace {

constexpr int kWarpsPerCta = 8;
constexpr unsigned kFull = 0xffffffffu;

// The dense operand ("panel") is fp32, or -- the reduced-precision tier (<= 2e-2, BASELINE north_star) -- bf16:
// a gathered row is then half the bytes, which is what the kernel is bound by (L2 -> SM gather traffic for
// narrow rows, HBM for panels that do not fit L2).  Accumulation and output stay fp32.  Every 16-byte load
// carries kElems elements and feeds kAcc float4 accumulators.
template <bool BF16>
struct Panel {
  static constexpr int kElems = BF16 ? 8 : 4;
  static constexpr int kAcc = BF16 ? 2 : 1;
  static constexpr int kElemBytes = BF16 ? 2 : 4;
  using elem_t = typename std::conditional<BF16, uint16_t, float>::type;
  using vec_t = typename std::conditional<BF16, uint4, float4>::type;  // one 16-byte load
  static __host__ __device__ __forceinline__ int chunks(int f) { return (f + kElems - 1) / kElems; }
  static __device__ __forceinline__ vec_t ldg(const elem_t* p) { return __ldg(reinterpret_cast<const vec_t*>(p)); }
};

__device__ __forceinline__ uint4 ldg_u4(const char* p) { return __ldg(reinterpret_cast<const uint4*>(p)); }
__device__ __forceinline__ float4 ldg_f4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }

__device__ __forceinline__ void fma4(float4& acc, float v, const float4& x) {
  acc.x = fmaf(v, x.x, acc.x);
  acc.y = fmaf(v, x.y, acc.y);
  acc.z = fmaf(v, x.z, acc.z);
  acc.w = fmaf(v, x.w, acc.w);
}
// acc[0..kAcc) += v * (the elements of one 16-byte chunk); bf16 -> fp32 is a shift / a mask
__device__ __forceinline__ void fma_vec(float4* acc, float v, const float4& x) { fma4(acc[0], v, x); }
__device__ __forceinline__ void fma_vec(float4* acc, float v, const uint4& x) {
  fma4(acc[0], v, make_float4(__uint_as_float(x.x << 16), __uint_as_float(x.x & 0xffff0000u),
                              __uint_as_float(x.y << 16), __uint_as_float(x.y & 0xffff0000u)));
  fma4(acc[1], v, make_float4(__uint_as_float(x.z << 16), __uint_as_float(x.z & 0xffff0000u),
                              __uint_as_float(x.w << 16), __uint_as_float(x.w & 0xffff0000u)));
}
template <bool BF16>
__device__ __forceinline__ void fma_chunk(float4* acc, float v, const uint4& x) {
  if constexpr (!BF16) {
    fma4(acc[0], v, make_float4(__uint_as_float(x.x), __uint_as_float(x.y), __uint_as_float(x.z), __uint_as_float(x.w)));
  } else {
    fma4(acc[0], v, make_float4(__uint_as_float(x.x << 16), __uint_as_float(x.x & 0xffff0000u),
                                __uint_as_float(x.y << 16), __uint_as_float(x.y & 0xffff0000u)));
    fma4(acc[1], v, make_float4(__uint_as_float(x.z << 16), __uint_as_float(x.z & 0xffff0000u),
                                __uint_as_float(x.w << 16), __uint_as_float(x.w & 0xffff0000u)));
  }
}

// U gathered rows per lane in flight: all loads are issued before the first FMA (memory-level
// parallelism is what this kernel lives on).  Entry s = (j + u) * G + slot of the current block
// of cnt; slots past the end of the row carry v = 0 / c = 0: their gather of row 0 is harmless,
// their FMA is skipped (0 * Inf would put a NaN that is not in the product into the row).
template <int LPR, int CH, int U, bool BF16>
__device__ __forceinline__ void gather_batch(float4 (&acc)[CH * Panel<BF16>::kAcc], int c, float v, int j, int slot,
                                             int cnt, const typename Panel<BF16>::elem_t* __restrict__ b,
                                             const int (&qoff)[CH], int64_t ldb) {
  constexpr int G = 32 / LPR;
  constexpr int A = Panel<BF16>::kAcc;
  int cc[U];
  float vv[U];
  typename Panel<BF16>::vec_t x[U][CH];
#pragma unroll
  for (int u = 0; u < U; ++u) {
    const int s = (j + u) * G + slot;
    cc[u] = __shfl_sync(kFull, c, s);
    vv[u] = __shfl_sync(kFull, v, s);
  }
#pragma unroll
  for (int u = 0; u < U; ++u) {
    const typename Panel<BF16>::elem_t* rowp = b + (int64_t)cc[u] * ldb;
#pragma unroll
    for (int k = 0; k < CH; ++k) x[u][k] = Panel<BF16>::ldg(rowp + qoff[k]);
  }
#pragma unroll
  for (int u = 0; u < U; ++u)
    if ((j + u) * G + slot < cnt) {
#pragma unroll
      for (int k = 0; k < CH; ++k) fma_vec(&acc[k * A], vv[u], x[u][k]);
    }
}

// Accumulate stored entries [start, end) of one row into acc (per-lane partial sums).
// LPR lanes cover one gathered row; CH float4 chunks per lane (CH > 1 only when LPR == 32).
// Lanes whose float4 index is past the row width read a clamped (valid) address and build a
// value that is never stored.
// b / ldb in elements of the panel type; nch = 16-byte chunks per panel row.
template <int LPR, int CH, bool BF16>
__device__ __forceinline__ void accumulate_range(float4 (&acc)[CH * Panel<BF16>::kAcc], int start, int end,
                                                 const int32_t* __restrict__ col,
                                                 const float* __restrict__ val,
                                                 const typename Panel<BF16>::elem_t* __restrict__ b, int64_t ldb,
                                                 int nch, int lane) {
  constexpr int G = 32 / LPR;
  constexpr int U = (LPR * CH >= 64) ? (8 / CH > 0 ? 8 / CH : 1) : (LPR < 8 ? LPR : 8);
  const int slot = lane / LPR;
  const int sub = lane % LPR;
  // chunk k of this lane is float4 index k*LPR + sub; clamp so that every chunk is readable
  int qoff[CH];
#pragma unroll
  for (int k = 0; k < CH; ++k) qoff[k] = Panel<BF16>::kElems * min(k * LPR + sub, nch - 1);
  int c = 0;
  float v = 0.f;
  if (start + lane < end) {
    c = __ldg(col + start + lane);
    v = __ldg(val + start + lane);
  }
  for (int base = start; base < end; base += 32) {
    // prefetch the next block of 32 (col, val) pairs while this one is consumed
    int cn = 0;
    float vn = 0.f;
    if (base + 32 + lane < end) {
      cn = __ldg(col + base + 32 + lane);
      vn = __ldg(val + base + 32 + lane);
    }
    const int cnt = min(32, end - base);
    const int jmax = (cnt + G - 1) / G;  // entries past cnt have v = 0, c = 0 and are skipped by gather_batch
    int j = 0;
    for (; j + U <= jmax; j += U) gather_batch<LPR, CH, U, BF16>(acc, c, v, j, slot, cnt, b, qoff, ldb);
    if (U > 4 && j + 4 <= jmax) { gather_batch<LPR, CH, (U > 4 ? 4 : 1), BF16>(acc, c, v, j, slot, cnt, b, qoff, ldb); j += 4; }
    if (U > 2 && j + 2 <= jmax) { gather_batch<LPR, CH, (U > 2 ? 2 : 1), BF16>(acc, c, v, j, slot, cnt, b, qoff, ldb); j += 2; }
    if (U > 1 && j < jmax) { gather_batch<LPR, CH, 1, BF16>(acc, c, v, j, slot, cnt, b, qoff, ldb); j += 1; }
    c = cn;
    v = vn;
  }
}

template <int LPR, int CH>  // CH = number of float4 accumulators per lane here
__device__ __forceinline__ void reduce_slots(float4 (&acc)[CH]) {
#pragma unroll
  for (int off = LPR; off < 32; off <<= 1) {
#pragma unroll
    for (int k = 0; k < CH; ++k) {
      acc[k].x += __shfl_xor_sync(kFull, acc[k].x, off);
      acc[k].y += __shfl_xor_sync(kFull, acc[k].y, off);
      acc[k].z += __shfl_xor_sync(kFull, acc[k].z, off);
      acc[k].w += __shfl_xor_sync(kFull, acc[k].w, off);
    }
  }
}

__device__ __forceinline__ void store_row_chunk(float* out_row, int64_t row, int q, int f, bool vec_out,
                                                float4 a, const Epilogue& ep) {
  float r[4] = {a.x, a.y, a.z, a.w};
  if (ep.accumulate) {  // out += A*B (column-blocked multi-GPU SpMM adds one source block at a time)
    if (vec_out) {
      const float4 o = *reinterpret_cast<const float4*>(out_row + 4 * q);
      r[0] += o.x; r[1] += o.y; r[2] += o.z; r[3] += o.w;
    } else {
#pragma unroll
      for (int t = 0; t < 4; ++t)
        if (4 * q + t < f) r[t] += out_row[4 * q + t];
    }
  }
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    const int c = 4 * q + t;
    if (c < f) {
      if (ep.bias) r[t] += __ldg(ep.bias + c);
      if (ep.relu) r[t] = fmaxf(r[t], 0.f);
      if (ep.mask) r[t] = __ldg(ep.mask + row * ep.ld_mask + c) ? r[t] * ep.mask_scale : 0.f;
    }
  }
  if (vec_out) {
    *reinterpret_cast<float4*>(out_row + 4 * q) = make_float4(r[0], r[1], r[2], r[3]);
  } else {
#pragma unroll
    for (int t = 0; t < 4; ++t)
      if (4 * q + t < f) out_row[4 * q + t] = r[t];
  }
}

// the kAcc float4 results of 16-byte panel chunk q -> output columns [q * kElems, (q + 1) * kElems)
template <bool BF16>
__device__ __forceinline__ void store_panel_chunk(float* out_row, int64_t row, int q, int f, bool vec_out,
                                                  const float4* acc, const Epilogue& ep) {
  constexpr int A = Panel<BF16>::kAcc;
#pragma unroll
  for (int t = 0; t < A; ++t)
    if (4 * (q * A + t) < f) store_row_chunk(out_row, row, q * A + t, f, vec_out, acc[t], ep);
}

// One warp per row.  Rows of the long bin are skipped when skip_long is set.  b / ldb in elements of the panel type.
template <int LPR, int CH, bool BF16>
__global__ void __launch_bounds__(kWarpsPerCta * 32)
spmm_rows_vec_kernel(int n_rows, const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                     const float* __restrict__ val, const void* __restrict__ b, int64_t ldb, int f,
                     Epilogue ep, float* __restrict__ out, int64_t ldo, int vec_out, int skip_long) {
  constexpr int A = Panel<BF16>::kAcc;
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5);
  if (row >= n_rows) return;
  const int start = __ldg(rowptr + row);
  const int end = __ldg(rowptr + row + 1);
  if (skip_long && end - start >= kLongRowThreshold) return;
  const int nch = Panel<BF16>::chunks(f);
  float4 acc[CH * A];
#pragma unroll
  for (int k = 0; k < CH * A; ++k) acc[k] = make_float4(0.f, 0.f, 0.f, 0.f);
  accumulate_range<LPR, CH, BF16>(acc, start, end, col, val, reinterpret_cast<const typename Panel<BF16>::elem_t*>(b), ldb,
                                  nch, lane);
  reduce_slots<LPR, CH * A>(acc);
  if (lane < LPR) {
    float* out_row = out + (int64_t)row * ldo;
#pragma unroll
    for (int k = 0; k < CH; ++k) {
      const int q = k * LPR + lane;
      if (q < nch) store_panel_chunk<BF16>(out_row, row, q, f, vec_out, &acc[k * A], ep);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Group-per-row kernel (widths up to 64 floats): the G = 32/LPR lane groups of a warp each walk
// their OWN row, so one LDG.128 instruction still moves G feature rows but there is no cross-slot
// reduction, G rows' start-up latencies overlap, and short rows do not idle most of the warp.
//
// What bounds it (ncu, profiles/): the L1/TEX pipe -- every gathered 128-byte line is a wavefront
// there, and so is every shared-memory access and every global load of the index/value stream.  So
// the (col, val) pairs are staged with as few L1 operations as possible: the graph keeps them
// interleaved (CsrView::pair), a stage of 32 pairs per group is copied global->shared with 16-byte
// cp.async.cg (two pairs per copy, no registers held, L1 bypassed), and a batch of U entries is read
// back with U/2 broadcast LDS.128.  Each gather is then one IMAD.WIDE.U32 (col * row bytes + lane
// base) + one LDG.128 + 4 FFMA; the shuffle kernel above spends ~15 instructions per gather on 64-bit
// index arithmetic and shuffles.  Per-row accumulation order is the stored order, run-to-run
// deterministic.
constexpr int kStageEntries = 32;
// the largest power of two <= `want` for which `groups` double-buffered stages of (E + 2) pairs fit 48 KB
constexpr int stage_entries(int want, int groups) {
  int e = want;
  while (e > 2 && groups * 2 * (e + 2) * 8 > 48 * 1024) e /= 2;
  return e;
}

// (OR of one word of every gathered row) & never, where `never` is a kernel argument that is always
// 0 at run time (the compiler cannot know).  OR-ing it into the accumulators makes every FFMA of a
// batch depend on ALL the batch's gathers, i.e. all U gathers are in flight together.  Left alone,
// ptxas interleaves gathers and FFMAs assuming a short load latency and keeps 2-3 rows in flight per
// lane; the L2 gather rate needs several hundred rows in flight per SM (tools/microbench/gather_bw.cu).
template <int U>
__device__ __forceinline__ uint32_t all_landed(const uint4 (&x)[U], uint32_t never) {
  uint32_t g = 0u;
#pragma unroll
  for (int u = 0; u < U; ++u) g |= x[u].w;
  return g & never;
}

// W = warps per CTA, SE = entries per stage (tuning variants: smaller CTAs free their slots in finer steps at the
// tail of the grid; longer stages halve the per-stage bookkeeping of a ~100-entry row)
// PDL: the programmatic-dependent-launch instantiation (common.cuh): the row pointers and the first stage of (col,val)
// pairs -- constant for the life of the graph handle -- are fetched while the previous kernel of the stream drains;
// the wait sits in front of the first gather of the dense operand.
template <int LPR, int U, int MINB, bool BF16, int W = kWarpsPerCta, int SE = kStageEntries, bool PDL = false>
__global__ void __launch_bounds__(W * 32, MINB)
spmm_group_kernel(int n_rows, const int32_t* __restrict__ rowptr, const uint2* __restrict__ pair, int last_pair,
                  const void* __restrict__ b, uint32_t ldb_bytes, int f, Epilogue ep, float* __restrict__ out,
                  int64_t ldo, int vec_out, int skip_long, uint32_t never, uint32_t col_mask) {
  constexpr int G = 32 / LPR;
  constexpr int A = Panel<BF16>::kAcc;
  constexpr int E = stage_entries(SE, W * G) < 2 * LPR ? 2 * LPR : stage_entries(SE, W * G);  // static shared memory stays < 48 KB (32 entries for LPR >= 4, else 16)
  constexpr int NC = E / (2 * LPR);  // 16-byte copies (two pairs) per lane and stage
  static_assert(E % U == 0 && U % 2 == 0 && NC >= 1, "batches of U entries must divide the stage");
  // +2 pairs of padding per buffer: buffers stay 16-byte aligned and consecutive groups start
  // 2*(E+2)*2 = 136 words apart, i.e. 8 banks, so the G broadcast LDS.128 of one instruction hit
  // disjoint banks
  constexpr uint32_t kBufBytes = 8u * (E + 2);
  __shared__ __align__(16) uint2 stage[W][G][2][E + 2];
  if constexpr (PDL) pdl_launch_dependents();
  // Register diet (the budget decides how many warps x gathers fly per SM): inside the loops only
  // e (next entry to stage), left (entries not yet consumed, counted from the 2-aligned window start),
  // the two buffer addresses, the lane's base pointer and the accumulators live; row / width data are
  // rebuilt at the end.
  const int sub = (threadIdx.x & 31) % LPR;
  int e, left, lead;
  {
    const int lane = threadIdx.x & 31;
    const int row = (blockIdx.x * W + (threadIdx.x >> 5)) * G + lane / LPR;
    int start = 0, end = 0;
    if (row < n_rows) {
      start = __ldg(rowptr + row);
      end = __ldg(rowptr + row + 1);
      if (skip_long && end - start >= kLongRowThreshold) end = start;
    }
    lead = start & 1;  // the stage window starts at an even entry (16-byte aligned pair address)
    e = start - lead + 2 * sub;
    left = end - start + lead;
    if (end == start) left = 0;
  }
  uint64_t bl;  // lane's base: column chunk `sub` of row 0 (lanes past the width read a clamped, valid chunk)
  {
    bl = reinterpret_cast<uint64_t>(b) + 16u * (uint32_t)min(sub, Panel<BF16>::chunks(f) - 1);
    asm volatile("" : "+l"(bl));  // keep it in a register pair (ptxas would rebuild it per gather)
  }
  uint32_t cur = smem_u32(&stage[threadIdx.x >> 5][((threadIdx.x & 31) / LPR)][0][0]);
  uint32_t nxt = cur + kBufBytes;

  // stage <- the next E pairs of this group's row, global -> shared; pairs past the row's end are
  // zero-filled (col 0, val 0) and gathered but not accumulated.  `ahead` = entries not yet staged, counted
  // from this lane's first one.
  auto fetch = [&](uint32_t dst_buf, int ahead) {
#pragma unroll
    for (int k = 0; k < NC; ++k) {
      const int a = ahead - 2 * LPR * k;
      const uint32_t bytes = a >= 2 ? 16u : (a == 1 ? 8u : 0u);
      // (zero-byte copies past the row's end still carry an address: keep it inside the array)
      cp_async16_zfill(dst_buf + 16u * (uint32_t)(sub + LPR * k), pair + min(e + 2 * LPR * k, last_pair), bytes);
    }
    cp_async_commit();
    e += E;
  };
  auto pairs_at = [&](int j) {  // pairs j, j + 1 of the current stage: (col, val, col, val)
    uint4 q;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(q.x), "=r"(q.y), "=r"(q.z), "=r"(q.w) : "r"(cur + 8u * (uint32_t)j));
    return q;
  };
  auto gather = [&](uint32_t c) {  // one IMAD.WIDE.U32: c * row bytes + lane base
    uint4 x;
    asm volatile("ld.global.nc.v4.u32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(x.x), "=r"(x.y), "=r"(x.z), "=r"(x.w)
                 : "l"(bl + (uint64_t)c * ldb_bytes));
    return x;
  };
  fetch(cur, left - 2 * sub);
  if constexpr (PDL) pdl_wait();  // the dense operand (and, for the accumulate epilogue, out) may come from the previous kernel
  float4 acc[A];
#pragma unroll
  for (int t = 0; t < A; ++t) acc[t] = make_float4(0.f, 0.f, 0.f, 0.f);
  while (!__all_sync(kFull, left <= 0)) {
    fetch(nxt, left - E - 2 * sub);  // next stage flies while this one is consumed
    cp_async_wait<1>();              // this lane's copies for the current stage have landed ...
    __syncwarp();                    // ... and so have the other lanes'
    // live entries of this stage: [lead, cnt) -- with an odd row start the first stage's first pair belongs to
    // the previous row
    const int cnt = min(max(left, 0), E);
    const int cmax = __reduce_max_sync(kFull, cnt);
    // (unroll 1: with the batches unrolled ptxas software-pipelines them with 2-3 gathers in flight)
#pragma unroll 1
    for (int j = 0; j < cmax; j += U) {
      // groups whose row has ended sit the batch out (a divergent branch, reconverged below); inside a
      // live batch the entries past the row's end (and the previous row's pair in front of an odd start)
      // are still gathered -- at most U harmless loads per row, all of a batch in flight together -- but
      // their FMAs are predicated off: a zero value times an Inf / NaN of the gathered row is NaN
      if (j < cnt) {
        uint4 q[U / 2];
        uint4 x[U];
#pragma unroll
        for (int h = 0; h < U / 2; ++h) q[h] = pairs_at(j + 2 * h);  // j + u < E because U divides E
#pragma unroll
        for (int h = 0; h < U / 2; ++h) {
          x[2 * h] = gather(q[h].x & col_mask);  // the column word may carry tags (common.cuh kPairColMask)
          x[2 * h + 1] = gather(q[h].z & col_mask);
        }
        const uint32_t zero = all_landed(x, never);
#pragma unroll
        for (int t = 0; t < A; ++t) {
          acc[t].x = __uint_as_float(__float_as_uint(acc[t].x) | zero);
          acc[t].y = __uint_as_float(__float_as_uint(acc[t].y) | zero);
          acc[t].z = __uint_as_float(__float_as_uint(acc[t].z) | zero);
          acc[t].w = __uint_as_float(__float_as_uint(acc[t].w) | zero);
        }
#pragma unroll
        for (int h = 0; h < U / 2; ++h) {
          if (j + 2 * h >= lead && j + 2 * h < cnt) fma_chunk<BF16>(acc, __uint_as_float(q[h].y), x[2 * h]);
          if (j + 2 * h + 1 < cnt) fma_chunk<BF16>(acc, __uint_as_float(q[h].w), x[2 * h + 1]);
        }
      }
    }
    __syncwarp();  // all lanes are done with `cur` before the next iteration's copies overwrite it
    lead = 0;
    left -= E;
    const uint32_t t = cur;
    cur = nxt;
    nxt = t;
  }
  cp_async_wait<0>();
  {
    const int lane = threadIdx.x & 31;
    const int row = (blockIdx.x * W + (threadIdx.x >> 5)) * G + lane / LPR;
    if (row >= n_rows || sub >= Panel<BF16>::chunks(f)) return;
    if (skip_long && __ldg(rowptr + row + 1) - __ldg(rowptr + row) >= kLongRowThreshold) return;
    store_panel_chunk<BF16>(out + (int64_t)row * ldo, row, sub, f, vec_out, acc, ep);
  }
}

// ---------------------------------------------------------------------------------------------
// TMA-staged variant: the column-index and value streams of a row are pulled into shared memory
// with cp.async.bulk (1-D TMA, mbarrier complete_tx) one chunk ahead of their use, instead of
// being loaded into registers and broadcast with shuffles.  Each warp owns a two-slot ring
// (2 x (132 int32 + 132 fp32)) and walks rows gw, gw + W, ...; the copy window is widened to
// 16-byte boundaries (the CSR arrays are padded).  The gathers of feature rows are unchanged.
constexpr int kTmaChunk = 128;           // stored entries per staged chunk
constexpr int kTmaSlot = kTmaChunk + 4;  // + alignment slack; 528 bytes per array

template <int LPR, int CH, int U>
__device__ __forceinline__ void gather_batch_smem(float4 (&acc)[CH], const int32_t* __restrict__ cols,
                                                  const float* __restrict__ vals, int s0, int cnt, int slot,
                                                  const float* __restrict__ b, const int (&qoff)[CH], int64_t ldb) {
  constexpr int G = 32 / LPR;
  int cc[U];
  float vv[U];
  bool ok[U];
  float4 x[U][CH];
#pragma unroll
  for (int u = 0; u < U; ++u) {
    const int s = s0 + u * G + slot;  // entry index inside the current block of 32
    ok[u] = s < cnt;
    cc[u] = ok[u] ? cols[s] : 0;
    vv[u] = ok[u] ? vals[s] : 0.f;
  }
#pragma unroll
  for (int u = 0; u < U; ++u) {
    const float* rowp = b + (int64_t)cc[u] * ldb;
#pragma unroll
    for (int k = 0; k < CH; ++k) x[u][k] = ldg_f4(rowp + qoff[k]);
  }
#pragma unroll
  for (int u = 0; u < U; ++u)
    if (ok[u]) {  // (the gather of row 0 past the row's end is harmless, 0 * Inf in the sum is not)
#pragma unroll
      for (int k = 0; k < CH; ++k) fma4(acc[k], vv[u], x[u][k]);
    }
}

template <int LPR, int CH>
__global__ void __launch_bounds__(kWarpsPerCta * 32)
spmm_rows_tma_kernel(int n_rows, const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                     const float* __restrict__ val, const float* __restrict__ b, int64_t ldb, int f,
                     Epilogue ep, float* __restrict__ out, int64_t ldo, int vec_out, int skip_long) {
  constexpr int G = 32 / LPR;
  constexpr int U = (LPR * CH >= 64) ? (8 / CH > 0 ? 8 / CH : 1) : (LPR < 8 ? LPR : 8);
  __shared__ __align__(16) int32_t col_s[kWarpsPerCta][2][kTmaSlot];
  __shared__ __align__(16) float val_s[kWarpsPerCta][2][kTmaSlot];
  __shared__ __align__(8) unsigned long long bars[kWarpsPerCta][2];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int slot = lane / LPR, sub = lane % LPR;
  const uint32_t bar[2] = {smem_u32(&bars[warp][0]), smem_u32(&bars[warp][1])};
  if (lane == 0) {
    mbar_init(bar[0], 1);
    mbar_init(bar[1], 1);
    fence_barrier_init();
  }
  __syncthreads();
  const int f4 = (f + 3) >> 2;
  int qoff[CH];
#pragma unroll
  for (int k = 0; k < CH; ++k) qoff[k] = 4 * min(k * LPR + sub, f4 - 1);

  const int W = gridDim.x * kWarpsPerCta;
  // item = one chunk of one row: entries [e0, e1) of row `row` whose range ends at row_end
  int row = blockIdx.x * kWarpsPerCta + warp - W, e0 = 0, e1 = 0, row_end = 0;
  bool valid = true;
  auto next_row = [&](int& r, int& a0, int& a1, int& rend) -> bool {
    for (;;) {
      r += W;
      if (r >= n_rows) return false;
      const int s_ = __ldg(rowptr + r), e_ = __ldg(rowptr + r + 1);
      if (skip_long && e_ - s_ >= kLongRowThreshold) continue;
      a0 = s_;
      rend = e_;
      a1 = min(s_ + kTmaChunk, e_);
      return true;
    }
  };
  auto issue = [&](int a0, int a1, int stage) {
    if (a1 > a0 && lane == 0) {
      const int w0 = a0 & ~3, w1 = (a1 + 3) & ~3;
      const uint32_t bytes = (uint32_t)(w1 - w0) * 4u;
      mbar_expect_tx(bar[stage], 2 * bytes);
      bulk_g2s(smem_u32(&col_s[warp][stage][0]), col + w0, bytes, bar[stage]);
      bulk_g2s(smem_u32(&val_s[warp][stage][0]), val + w0, bytes, bar[stage]);
    }
  };
  valid = next_row(row, e0, e1, row_end);
  int stage = 0;
  uint32_t phase[2] = {0u, 0u};
  if (valid) issue(e0, e1, 0);
  float4 acc[CH];
#pragma unroll
  for (int k = 0; k < CH; ++k) acc[k] = make_float4(0.f, 0.f, 0.f, 0.f);
  while (valid) {
    // the item after this one (next chunk of the row, or the first chunk of the warp's next row)
    int nrow = row, ne0, ne1, nend = row_end;
    bool nvalid = true;
    if (e1 < row_end) {
      ne0 = e1;
      ne1 = min(e1 + kTmaChunk, row_end);
    } else {
      nvalid = next_row(nrow, ne0, ne1, nend);
    }
    if (nvalid) issue(ne0, ne1, stage ^ 1);
    if (e1 > e0) {
      mbar_wait(bar[stage], phase[stage]);
      phase[stage] ^= 1u;
      const int32_t* cols = &col_s[warp][stage][e0 & 3];
      const float* vals = &val_s[warp][stage][e0 & 3];
      const int n = e1 - e0;
      for (int base = 0; base < n; base += 32) {
        const int cnt = min(32, n - base);
        const int jmax = (cnt + G - 1) / G;
        int j = 0;
        for (; j + U <= jmax; j += U)
          gather_batch_smem<LPR, CH, U>(acc, cols + base, vals + base, j * G, cnt, slot, b, qoff, ldb);
        if (U > 4 && j + 4 <= jmax) {
          gather_batch_smem<LPR, CH, (U > 4 ? 4 : 1)>(acc, cols + base, vals + base, j * G, cnt, slot, b, qoff, ldb);
          j += 4;
        }
        if (U > 2 && j + 2 <= jmax) {
          gather_batch_smem<LPR, CH, (U > 2 ? 2 : 1)>(acc, cols + base, vals + base, j * G, cnt, slot, b, qoff, ldb);
          j += 2;
        }
        if (U > 1 && j < jmax) gather_batch_smem<LPR, CH, 1>(acc, cols + base, vals + base, j * G, cnt, slot, b, qoff, ldb);
      }
    }
    if (e1 == row_end) {  // row finished: combine the slots, epilogue, reset
      reduce_slots<LPR, CH>(acc);
      if (lane < LPR) {
        float* out_row = out + (int64_t)row * ldo;
#pragma unroll
        for (int k = 0; k < CH; ++k) {
          const int q = k * LPR + lane;
          if (q < f4) store_row_chunk(out_row, row, q, f, vec_out, acc[k], ep);
        }
      }
#pragma unroll
      for (int k = 0; k < CH; ++k) acc[k] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    __syncwarp();  // every lane is done with this slot before lane 0 lets TMA overwrite it
    row = nrow; e0 = ne0; e1 = ne1; row_end = nend; valid = nvalid;
    stage ^= 1;
  }
}

// Long-row bin, phase 1: one warp per chunk of kLongChunk stored entries -> partial row.
template <int LPR, int CH, bool BF16>
__global__ void __launch_bounds__(kWarpsPerCta * 32)
spmm_long_partial_kernel(int n_long_rows, int n_chunks, const int32_t* __restrict__ long_rows,
                         const int32_t* __restrict__ long_chunk_ptr,
                         const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                         const float* __restrict__ val, const void* __restrict__ b, int64_t ldb,
                         int f, float* __restrict__ partial, int ldp) {
  constexpr int A = Panel<BF16>::kAcc;
  const int lane = threadIdx.x & 31;
  const int ch = blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5);
  if (ch >= n_chunks) return;
  int lo = 0, hi = n_long_rows;  // last li with long_chunk_ptr[li] <= ch
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(long_chunk_ptr + mid) <= ch) lo = mid; else hi = mid;
  }
  const int row = __ldg(long_rows + lo);
  const int local = ch - __ldg(long_chunk_ptr + lo);
  const int row_start = __ldg(rowptr + row);
  const int row_end = __ldg(rowptr + row + 1);
  const int start = row_start + local * kLongChunk;
  const int end = min(start + kLongChunk, row_end);
  const int nch = Panel<BF16>::chunks(f);
  const int f4 = (f + 3) >> 2;
  float4 acc[CH * A];
#pragma unroll
  for (int k = 0; k < CH * A; ++k) acc[k] = make_float4(0.f, 0.f, 0.f, 0.f);
  accumulate_range<LPR, CH, BF16>(acc, start, end, col, val, reinterpret_cast<const typename Panel<BF16>::elem_t*>(b), ldb,
                                  nch, lane);
  reduce_slots<LPR, CH * A>(acc);
  if (lane < LPR) {
    float* prow = partial + (int64_t)ch * ldp;
#pragma unroll
    for (int k = 0; k < CH; ++k) {
      const int q = k * LPR + lane;
#pragma unroll
      for (int t = 0; t < A; ++t)
        if (q * A + t < f4) *reinterpret_cast<float4*>(prow + 4 * (q * A + t)) = acc[k * A + t];
    }
  }
}

// Long-row bin, phase 2: one warp per long row adds its partial rows in chunk order.
__global__ void __launch_bounds__(kWarpsPerCta * 32)
spmm_long_fixup_kernel(int n_long_rows, const int32_t* __restrict__ long_rows,
                       const int32_t* __restrict__ long_chunk_ptr, const float* __restrict__ partial,
                       int ldp, int f, Epilogue ep, float* __restrict__ out, int64_t ldo) {
  const int lane = threadIdx.x & 31;
  const int li = blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5);
  if (li >= n_long_rows) return;
  const int row = __ldg(long_rows + li);
  const int c0 = __ldg(long_chunk_ptr + li);
  const int c1 = __ldg(long_chunk_ptr + li + 1);
  for (int j = lane; j < f; j += 32) {
    float acc = 0.f;
    for (int c = c0; c < c1; ++c) acc += partial[(int64_t)c * ldp + j];
    if (ep.accumulate) acc += out[(int64_t)row * ldo + j];
    if (ep.bias) acc += __ldg(ep.bias + j);
    if (ep.relu) acc = fmaxf(acc, 0.f);
    if (ep.mask) acc = __ldg(ep.mask + (int64_t)row * ep.ld_mask + j) ? acc * ep.mask_scale : 0.f;
    out[(int64_t)row * ldo + j] = acc;
  }
}

// Fully generic fallback: any f / ld / alignment.  One warp per row, lanes over columns.
__global__ void __launch_bounds__(kWarpsPerCta * 32)
spmm_rows_scalar_kernel(int n_rows, const int32_t* __restrict__ rowptr,
                        const int32_t* __restrict__ col, const float* __restrict__ val,
                        const float* __restrict__ b, int64_t ldb, int f,
                        Epilogue ep, float* __restrict__ out, int64_t ldo) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5);
  if (row >= n_rows) return;
  const int start = __ldg(rowptr + row);
  const int end = __ldg(rowptr + row + 1);
  for (int f0 = 0; f0 < f; f0 += 32) {
    const int j = f0 + lane;
    float acc = 0.f;
    for (int base = start; base < end; base += 32) {
      const int e = base + lane;
      int c = 0;
      float v = 0.f;
      if (e < end) {
        c = __ldg(col + e);
        v = __ldg(val + e);
      }
      const int cnt = min(32, end - base);
      for (int s = 0; s < cnt; ++s) {
        const int cc = __shfl_sync(kFull, c, s);
        const float vv = __shfl_sync(kFull, v, s);
        if (j < f) acc = fmaf(vv, __ldg(b + (int64_t)cc * ldb + j), acc);
      }
    }
    if (j < f) {
      if (ep.accumulate) acc += out[(int64_t)row * ldo + j];
      if (ep.bias) acc += __ldg(ep.bias + j);
      if (ep.relu) acc = fmaxf(acc, 0.f);
      if (ep.mask) acc = __ldg(ep.mask + (int64_t)row * ep.ld_mask + j) ? acc * ep.mask_scale : 0.f;
      out[(int64_t)row * ldo + j] = acc;
    }
  }
}

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// Which kernel serves the short-row bins.  Default (auto): the group-per-row kernel when the shape
// suits it, the warp-per-row shuffle kernel otherwise.  Environment GCNB_SPMM_KERNEL = rows | group |
// tma and GCNB_SPMM_GROUP_VARIANT = 0..4 set the initial value; gcnb_set_tuning() changes it at run
// time (tests force each kernel on small graphs).
int g_spmm_kernel = -1;   // 0 auto, 1 rows, 2 group (forced), 3 tma
int g_group_variant = -2;  // -1 auto
int g_pdl = -1;            // programmatic dependent launch of the layer's kernel chain: 0 off (default), 1 on

void tuning_init() {
  if (g_spmm_kernel < 0) {
    const char* e = getenv("GCNB_SPMM_KERNEL");
    g_spmm_kernel = !e ? 0 : (e[0] == 'r' ? 1 : (e[0] == 'g' ? 2 : (e[0] == 't' ? 3 : 0)));
    const char* s = getenv("GCNB_SPMM_STAGING");  // older spelling of the tma switch
    if (s && (s[0] == 't' || s[0] == 'T')) g_spmm_kernel = 3;
  }
  if (g_group_variant == -2) {
    const char* e = getenv("GCNB_SPMM_GROUP_VARIANT");
    g_group_variant = e ? atoi(e) : -1;
  }
  if (g_pdl < 0) {
    const char* e = getenv("GCNB_PDL");
    g_pdl = (e && atoi(e) > 0) ? 1 : 0;
  }
}
bool spmm_use_tma() { tuning_init(); return g_spmm_kernel == 3; }
int spmm_group_variant() { tuning_init(); return g_group_variant; }

// Long-row bin: chunk partials, then the ordered fix-up (both no-ops when the bin is empty).
template <int LPR, int CH, bool BF16>
int launch_long(const CsrView& a, const void* b, int64_t ldb, int f, const Epilogue& ep, float* out,
                int64_t ldo, float* partial, int ldp, cudaStream_t st) {
  if (a.n_long_rows == 0) return GCNB_OK;
  const int g1 = (int)ceil_div(a.n_long_chunks, kWarpsPerCta);
  spmm_long_partial_kernel<LPR, CH, BF16><<<g1, kWarpsPerCta * 32, 0, st>>>(
      (int)a.n_long_rows, (int)a.n_long_chunks, a.long_rows, a.long_chunk_ptr, a.rowptr, a.col, a.val, b, ldb, f,
      partial, ldp);
  GCNB_LAUNCH_CHECK();
  const int g2 = (int)ceil_div(a.n_long_rows, kWarpsPerCta);
  spmm_long_fixup_kernel<<<g2, kWarpsPerCta * 32, 0, st>>>((int)a.n_long_rows, a.long_rows, a.long_chunk_ptr, partial,
                                                          ldp, f, ep, out, ldo);
  GCNB_LAUNCH_CHECK();
  return GCNB_OK;
}

template <int LPR, int CH, bool BF16>
int launch_vec(const CsrView& a, const void* b, int64_t ldb, int f, const Epilogue& ep, float* out,
               int64_t ldo, bool vec_out, float* partial, int ldp, cudaStream_t st) {
  constexpr int kEB = Panel<BF16>::kElemBytes;
  const bool has_long = a.n_long_rows > 0;
  const int grid = (int)ceil_div(a.n_rows, kWarpsPerCta);
  if constexpr (LPR >= 2 && LPR <= 16 && CH == 1) {
    constexpr int G = 32 / LPR;
    // one row per lane group needs enough rows to fill the machine with warps, and rows short enough
    // that a group's serial walk is not the critical path (few long rows: warp-per-row splits them)
    const bool shape_ok = a.n_rows >= (int64_t)kNumSMs * 16 * G && a.nnz <= a.n_rows * 384;
    tuning_init();
    const bool want_group = g_spmm_kernel == 2 || (g_spmm_kernel == 0 && (shape_ok || g_group_variant >= 0));
    if (grid > 0 && a.pair != nullptr && want_group && ldb * kEB < (1ll << 32)) {
#define GCNB_GROUP_ARGS                                                                                 \
  (int)a.n_rows, a.rowptr, a.pair, (int)(a.nnz & ~1ll), b, (uint32_t)(ldb * kEB), f, ep, out, ldo, \
      vec_out ? 1 : 0, has_long ? 1 : 0, 0u, a.pair_tagged ? kPairColMask : 0xffffffffu
#define GCNB_GROUP_LAUNCH_W(U_, MINB_, W_, SE_)                                                                      \
  spmm_group_kernel<LPR, U_, MINB_, BF16, W_, SE_><<<(int)ceil_div(a.n_rows, (int64_t)(W_) * G), (W_) * 32, 0, st>>>( \
      GCNB_GROUP_ARGS)
// the PDL instantiation exists for the auto variants only
#define GCNB_GROUP_LAUNCH_PDL(U_, MINB_, W_, SE_)                                                                 \
  GCNB_CUDA(launch_pdl(spmm_group_kernel<LPR, U_, MINB_, BF16, W_, SE_, true>,                                    \
                       dim3((unsigned)ceil_div(a.n_rows, (int64_t)(W_) * G)), dim3((W_) * 32), 0, st, GCNB_GROUP_ARGS))
#define GCNB_GROUP_LAUNCH(U_, MINB_) GCNB_GROUP_LAUNCH_W(U_, MINB_, kWarpsPerCta, kStageEntries)
      // (gathers in flight per lane, CTAs per SM the register budget must allow).  Measured on B200
      // (gpurun_out/probe_sweep8.log): 128/256-byte rows like many warps with 4 gathers each, narrower
      // rows fewer warps with 8.  GCNB_SPMM_GROUP_VARIANT overrides (tuning knob).
      int variant = spmm_group_variant();
      // auto (profiles/r01_spmm_variant_sweep_w_se_*.txt): 2-warp CTAs and 16-entry stages -- slots are handed to the
      // next rows in finer steps, the first stage of a row is half as long, and 24 x 2.3 KB of staging leave more
      // of the SM's L1 to the gathers: 4-6 % over the 8-warp / 32-entry shapes (variants 2 and 0) on every
      // measured graph
      // (bf16 panels with 64-byte rows stay on variant 0: 75.3 us per CBG launch there, 77.3 us with variant 14,
      // profiles/r01_launches_v10_summary.txt vs _v12_)
      if (variant < 0) variant = (LPR >= 8) ? 13 : ((LPR == 4 && !BF16) ? 14 : 0);
      const bool pdl = pdl_enabled() && spmm_group_variant() < 0;
      if (pdl) {
        if (variant == 13) GCNB_GROUP_LAUNCH_PDL(4, 24, 2, 16);
        else if (variant == 14) GCNB_GROUP_LAUNCH_PDL(8, 16, 2, 16);
        else GCNB_GROUP_LAUNCH_PDL(8, 4, kWarpsPerCta, kStageEntries);
      } else
      switch (variant) {
        case 1: GCNB_GROUP_LAUNCH(8, 3); break;
        case 2: GCNB_GROUP_LAUNCH(4, 6); break;
        case 3: GCNB_GROUP_LAUNCH(16, 2); break;
        case 4: GCNB_GROUP_LAUNCH(4, 5); break;
        case 5: GCNB_GROUP_LAUNCH(4, 7); break;                       // 56 warps per SM (a few spilled registers)
        case 6: GCNB_GROUP_LAUNCH_W(4, 12, 4, kStageEntries); break;  // 4-warp CTAs, same 48 warps per SM
        case 7: GCNB_GROUP_LAUNCH_W(4, 6, kWarpsPerCta, 64); break;   // 64-entry stages
        case 8: GCNB_GROUP_LAUNCH_W(4, 12, 4, 64); break;             // both
        case 9: GCNB_GROUP_LAUNCH_W(8, 8, 4, kStageEntries); break;   // variant 0 with 4-warp CTAs
        case 10: GCNB_GROUP_LAUNCH_W(4, 24, 2, kStageEntries); break; // 2-warp CTAs
        case 11: GCNB_GROUP_LAUNCH_W(8, 16, 2, kStageEntries); break;
        case 12: GCNB_GROUP_LAUNCH_W(4, 12, 4, 16); break;            // 16-entry stages
        case 13: GCNB_GROUP_LAUNCH_W(4, 24, 2, 16); break;
        case 14: GCNB_GROUP_LAUNCH_W(8, 16, 2, 16); break;
        case 15: GCNB_GROUP_LAUNCH_W(8, 8, 4, 16); break;
        default: GCNB_GROUP_LAUNCH(8, 4); break;
      }
#undef GCNB_GROUP_LAUNCH
#undef GCNB_GROUP_LAUNCH_W
#undef GCNB_GROUP_LAUNCH_PDL
#undef GCNB_GROUP_ARGS
      GCNB_LAUNCH_CHECK();
      return launch_long<LPR, CH, BF16>(a, b, ldb, f, ep, out, ldo, partial, ldp, st);
    }
  }
  if (grid > 0 && !BF16 && spmm_use_tma()) {
    // persistent: 6 CTAs per SM walk the rows with a per-warp TMA ring for the index/value streams
    int pgrid = 6 * kNumSMs;
    if (pgrid > grid) pgrid = grid;
    spmm_rows_tma_kernel<LPR, CH><<<pgrid, kWarpsPerCta * 32, 0, st>>>(
        (int)a.n_rows, a.rowptr, a.col, a.val, reinterpret_cast<const float*>(b), ldb, f, ep, out, ldo, vec_out ? 1 : 0,
        has_long ? 1 : 0);
    GCNB_LAUNCH_CHECK();
  } else if (grid > 0) {
    spmm_rows_vec_kernel<LPR, CH, BF16><<<grid, kWarpsPerCta * 32, 0, st>>>(
        (int)a.n_rows, a.rowptr, a.col, a.val, b, ldb, f, ep, out, ldo, vec_out ? 1 : 0, has_long ? 1 : 0);
    GCNB_LAUNCH_CHECK();
  }
  return launch_long<LPR, CH, BF16>(a, b, ldb, f, ep, out, ldo, partial, ldp, st);
}

inline int partial_ld(int64_t f) { return (int)(ceil_div(f, 4) * 4); }

}  // namespace

bool pdl_enabled() {
  tuning_init();
  return g_pdl > 0;
}

int spmm_set_tuning(int key, int value) {
  tuning_init();
  if (key == GCNB_TUNE_SPMM_KERNEL) {
    GCNB_REQUIRE(value >= 0 && value <= 3, "set_tuning: spmm kernel must be 0..3");
    g_spmm_kernel = value;
  } else if (key == GCNB_TUNE_SPMM_GROUP_VARIANT) {
    GCNB_REQUIRE(value >= -1 && value <= 15, "set_tuning: group variant must be -1..15");
    g_group_variant = value;
  } else if (key == GCNB_TUNE_PDL) {
    GCNB_REQUIRE(value == 0 || value == 1, "set_tuning: PDL must be 0 or 1");
    g_pdl = value;
  } else if (key == GCNB_TUNE_SPMM_STREAM) {
    GCNB_REQUIRE(value >= 0 && value <= 2, "set_tuning: stream mode must be 0..2");
    spmm_stream_set(key, value);
  } else if (key == GCNB_TUNE_STREAM_HOT_MB) {
    GCNB_REQUIRE(value >= 0 && value <= 126, "set_tuning: hot-row L2 budget must be 0..126 MB");
    spmm_stream_set(key, value);
  } else if (key == GCNB_TUNE_STREAM_HINT) {
    GCNB_REQUIRE(value >= 0 && value <= 2, "set_tuning: stream hint mode must be 0..2");
    spmm_stream_set(key, value);
  } else if (key == GCNB_TUNE_STREAM_MIN_ROW_BYTES) {
    GCNB_REQUIRE(value >= 16 && value <= 1024, "set_tuning: stream row threshold must be 16..1024 bytes");
    spmm_stream_set(key, value);
  } else if (key == GCNB_TUNE_STREAM_BATCH) {
    GCNB_REQUIRE(value == 0 || value == 2 || value == 4 || value == 8, "set_tuning: stream rows in flight must be 0, 2, 4 or 8");
    spmm_stream_set(key, value);
  } else {
    GCNB_REQUIRE(false, "set_tuning: unknown key %d", key);
  }
  return GCNB_OK;
}

size_t spmm_workspace_bytes(const CsrView& a, int64_t f) {
  // (the streaming kernel works on column panels of at most 256 floats / 512 bf16: spmm_launch_t)
  const size_t stream = spmm_stream_mode() != 0 ? spmm_stream_workspace_bytes(a, f < 512 ? f : 512) : 0;
  const size_t lng = a.n_long_chunks == 0 ? 0 : (size_t)a.n_long_chunks * (size_t)partial_ld(f) * sizeof(float);
  return stream > lng ? stream : lng;
}

namespace {
template <bool BF16>
int spmm_launch_t(const CsrView& a, const void* bv, int64_t ldb, int64_t f, const Epilogue& ep, float* out,
                  int64_t ldo, void* ws, size_t ws_bytes, cudaStream_t st) {
  using elem_t = typename std::conditional<BF16, uint16_t, float>::type;
  constexpr int kE = Panel<BF16>::kElems;
  const elem_t* b = reinterpret_cast<const elem_t*>(bv);
  GCNB_REQUIRE(f > 0 && f <= (1 << 20), "spmm: feature width %lld out of range", (long long)f);
  GCNB_REQUIRE(ldb >= f && ldo >= f, "spmm: leading dimension smaller than width");
  GCNB_REQUIRE(a.n_rows < (1ll << 31), "spmm: too many rows");
  if (a.n_rows == 0) return GCNB_OK;
  GCNB_REQUIRE(b != nullptr && out != nullptr, "spmm: null operand");
  const size_t need = spmm_workspace_bytes(a, f);
  GCNB_REQUIRE(need == 0 || (ws != nullptr && ws_bytes >= need && aligned16(ws)),
               "spmm: workspace too small (%zu < %zu) or unaligned", ws_bytes, need);
  float* partial = reinterpret_cast<float*>(ws);
  const int ldp = partial_ld(f);
  const int nch = (int)ceil_div(f, kE);  // 16-byte chunks per panel row
  // vector gathers need 16-byte aligned rows of b that are readable up to nch whole chunks
  const bool vec_in = aligned16(b) && (ldb % kE == 0) && (ldb >= (int64_t)nch * kE);
  const bool vec_out = aligned16(out) && (ldo % 4 == 0) && (f % 4 == 0);
  if (!vec_in) {
    if constexpr (BF16) {
      GCNB_REQUIRE(false, "spmm(bf16 panel): rows must be 16-byte aligned with ld a multiple of 8 and >= 8*ceil(f/8)");
    } else {
      // generic path handles long rows too (a warp walks the whole row)
      const int grid = (int)ceil_div(a.n_rows, kWarpsPerCta);
      spmm_rows_scalar_kernel<<<grid, kWarpsPerCta * 32, 0, st>>>(
          (int)a.n_rows, a.rowptr, a.col, a.val, b, ldb, (int)f, ep, out, ldo);
      GCNB_LAUNCH_CHECK();
      return GCNB_OK;
    }
  }
  // wide panel rows on graphs whose every row is non-empty: the streaming kernel (spmm_stream.cu), at most 64
  // 16-byte chunks per pass
  tuning_init();
  if (g_spmm_kernel == 0 && spmm_stream_eligible(a, 16 * (int64_t)(nch < 64 ? nch : 64), nch < 64 ? nch : 64, BF16)) {
    const int64_t pw = 64 * kE;
    for (int64_t f0 = 0; f0 < f; f0 += pw) {
      const int64_t fw = (f - f0 < pw) ? (f - f0) : pw;
      Epilogue e2 = ep;
      if (e2.bias) e2.bias += f0;
      if (e2.mask) e2.mask += f0;
      GCNB_TRY(spmm_stream_launch(a, b + f0, ldb * (int64_t)sizeof(elem_t), (int)fw, BF16, e2, out + f0, ldo, vec_out,
                                  ws, ws_bytes, st));
    }
    return GCNB_OK;
  }
#define GCNB_SPMM_CASE(LPR, CH) \
  return launch_vec<LPR, CH, BF16>(a, b, ldb, (int)f, ep, out, ldo, vec_out, partial, ldp, st)
  if (nch <= 1) GCNB_SPMM_CASE(1, 1);
  if (nch <= 2) GCNB_SPMM_CASE(2, 1);
  if (nch <= 4) GCNB_SPMM_CASE(4, 1);
  if (nch <= 8) GCNB_SPMM_CASE(8, 1);
  if (nch <= 16) GCNB_SPMM_CASE(16, 1);
  if (nch <= 32) GCNB_SPMM_CASE(32, 1);
  if (nch <= 64) GCNB_SPMM_CASE(32, 2);
  if (nch <= 128) GCNB_SPMM_CASE(32, 4);
#undef GCNB_SPMM_CASE
  // wider than 128 chunks: column panels of 128 chunks (512 floats / 1024 bf16)
  const int64_t pw = 128 * kE;
  for (int64_t f0 = 0; f0 < f; f0 += pw) {
    const int64_t fw = (f - f0 < pw) ? (f - f0) : pw;
    Epilogue e2 = ep;
    if (e2.bias) e2.bias += f0;
    if (e2.mask) e2.mask += f0;
    GCNB_TRY(spmm_launch_t<BF16>(a, b + f0, ldb, fw, e2, out + f0, ldo, ws, ws_bytes, st));
  }
  return GCNB_OK;
}
}  // namespace

int spmm_launch(const CsrView& a, const float* b, int64_t ldb, int64_t f, const Epilogue& ep, float* out,
                int64_t ldo, void* ws, size_t ws_bytes, cudaStream_t st) {
  return spmm_launch_t<false>(a, b, ldb, f, ep, out, ldo, ws, ws_bytes, st);
}

int spmm_bf16_launch(const CsrView& a, const uint16_t* b, int64_t ldb, int64_t f, const Epilogue& ep, float* out,
                     int64_t ldo, void* ws, size_t ws_bytes, cudaStream_t st) {
  return spmm_launch_t<true>(a, b, ldb, f, ep, out, ldo, ws, ws_bytes, st);
}

}  // namespace gcnb
