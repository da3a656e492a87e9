// Shared helpers for libgcnb200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "gcnb200.h"

namespace gcnb {

void set_error(const char* fmt, ...);

#define GCNB_CUDA(expr)                                                                     \
  do {                                                                                      \
    cudaError_t _e = (expr);                                                                \
    if (_e != cudaSuccess) {                                                                \
      ::gcnb::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__,   \
                        __LINE__);                                                          \
      return (_e == cudaErrorMemoryAllocation) ? GCNB_E_NOMEM : GCNB_E_CUDA;                \
    }                                                                                       \
  } while (0)

#define GCNB_REQUIRE(cond, ...)        \
  do {                                 \
    if (!(cond)) {                     \
      ::gcnb::set_error(__VA_ARGS__);  \
      return GCNB_E_INVALID;           \
    }                                  \
  } while (0)

#define GCNB_TRY(expr)              \
  do {                              \
    int _s = (expr);                \
    if (_s != GCNB_OK) return _s;   \
  } while (0)

// every kernel launch of the library passes through here (or launch_pdl): gcnb_launch_count() reports the total, which
// is how bench.py counts the launches of one step instead of claiming a number
void count_launch();
#define GCNB_LAUNCH_CHECK()          \
  do {                               \
    ::gcnb::count_launch();          \
    GCNB_CUDA(cudaGetLastError());   \
  } while (0)

constexpr int kNumSMs = 148;  // B200

// Programmatic dependent launch of the layer's kernel chain (pack W, X.W, SpMM | SpMM^T, dW, split-K reduce):
// OFF by default; GCNB_PDL=1 or gcnb_set_tuning(GCNB_TUNE_PDL, 1) turns it on.  Each kernel of the chain then runs
// its PDL instantiation: `griddepcontrol.launch_dependents` first, so that the next kernel's CTAs take the SM slots
// this grid frees in its last wave, and `griddepcontrol.wait` before the first access to anything an earlier kernel
// of the stream may have written.  Only data that is constant for the life of the graph handle (rowptr, the
// (col,val) pairs) is touched before the wait.
bool pdl_enabled();

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                              Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  count_launch();
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

// One CSR (either the adjacency or its transpose) plus its row-length-binned schedule.
struct CsrView {
  int64_t n_rows = 0, n_cols = 0, nnz = 0;
  const int32_t* rowptr = nullptr;
  const int32_t* col = nullptr;
  const float* val = nullptr;
  // the same entries as (col, val bits) pairs, 16-byte aligned: what the group-per-row SpMM stages
  // (one 16-byte cp.async moves two entries; with separate arrays it takes four 4-byte copies)
  const uint2* pair = nullptr;
  // schedule: rows whose degree exceeds the long-row threshold are split into chunks of
  // kLongChunk stored entries; each chunk is one warp work item writing a partial row.
  int64_t n_long_rows = 0;
  int64_t n_long_chunks = 0;
  const int32_t* long_rows = nullptr;       // [n_long_rows] row ids (ascending)
  const int32_t* long_chunk_ptr = nullptr;  // [n_long_rows+1] prefix of chunks per long row
  int64_t max_degree = 0;
  int64_t bin_rows[GCNB_NUM_BINS] = {0, 0, 0, 0, 0};
  // Entry-balanced ("merge-style") schedule of the streaming SpMM (spmm_stream.cu): item i = stored entries
  // [i * kStreamItem, (i + 1) * kStreamItem); stream_items[i] = the row holding the item's first entry, bit 31 set
  // when that row began in an earlier item.  pair_tagged: the pair stream carries, in the upper bits of the column
  // word, the heat class of the column (bits 27..30, kPairClassShift) and an end-of-row flag (bit 31).
  int64_t n_stream_items = 0;
  const uint32_t* stream_items = nullptr;
  bool pair_tagged = false;
};

// Tags in the column word of a (col, val) pair (graphs with n_cols <= 2^27; wider ones keep plain columns):
//   bits 0..26  column
//   bits 27..30 heat class c of the column: it is among the 1024 * 2^c most referenced columns of the view
//               (kPairColdClass = not among the 16 M most referenced); the streaming SpMM asks L2 to keep the rows
//               of the hottest classes (evict_last) -- on a power-law graph a few % of the panel rows take most of
//               the gathers
//   bit  31     the entry is the last one of its row
constexpr int kPairColBits = 27;
constexpr uint32_t kPairColMask = (1u << kPairColBits) - 1u;
constexpr int kPairClassShift = kPairColBits;
constexpr uint32_t kPairColdClass = 15u;
constexpr uint32_t kPairRowEnd = 0x80000000u;
constexpr int kStreamItem = 1024;  // stored entries per work item of the streaming SpMM

// Fused SpMM epilogue:  out = dropout(relu(acc (+ out) (+ bias)))   -- pygcn/layers.py:36, the caller's
// F.relu (models.py:49,53,56) and upstream pygcn's F.dropout on the layer output.
struct Epilogue {
  const float* bias = nullptr;    // [f] or null
  int relu = 0;
  int accumulate = 0;             // add the previous contents of out first
  const uint8_t* mask = nullptr;  // [n_rows, ld_mask] keep-mask (0 / non-zero) or null
  int64_t ld_mask = 0;
  float mask_scale = 1.f;         // 1 / (1 - p)
};

constexpr int kLongRowThreshold = GCNB_BIN_EDGE_4;  // deg >= this -> split
constexpr int kLongChunk = 1024;

int spmm_launch(const CsrView& a, const float* b, int64_t ldb, int64_t f, const Epilogue& ep, float* out,
                int64_t ldo, void* ws, size_t ws_bytes, cudaStream_t stream);
// the same product with a bf16 panel (the <= 2e-2 tier): b is [n_cols, ldb] bf16, ldb % 8 == 0, 16-byte aligned
int spmm_bf16_launch(const CsrView& a, const uint16_t* b, int64_t ldb, int64_t f, const Epilogue& ep, float* out,
                     int64_t ldo, void* ws, size_t ws_bytes, cudaStream_t stream);
int to_bf16_launch(int64_t n_rows, int64_t f, const float* src, int64_t ld_src, uint16_t* dst, int64_t ld_dst,
                   cudaStream_t stream);
size_t spmm_workspace_bytes(const CsrView& a, int64_t f);
int spmm_set_tuning(int key, int value);

// streaming SpMM (spmm_stream.cu): TMA row gathers over the entry-balanced items of the view
bool spmm_stream_eligible(const CsrView& a, int64_t row_bytes, int nch, bool bf16);
size_t spmm_stream_workspace_bytes(const CsrView& a, int64_t f);
int spmm_stream_launch(const CsrView& a, const void* b, int64_t ldb_bytes, int f, bool bf16, const Epilogue& ep,
                       float* out, int64_t ldo, bool vec_out, void* ws, size_t ws_bytes, cudaStream_t stream);
int spmm_stream_mode();         // 0 off, 1 auto (default), 2 forced wherever eligible
void spmm_stream_set(int key, int value);

int gemm_fp32_launch(int64_t m, int64_t n, int64_t k, const float* a, int64_t a_rs, int64_t a_cs,
                     const float* b, int64_t b_rs, int64_t b_cs, float* c, int64_t ldc, void* ws,
                     size_t ws_bytes, cudaStream_t stream);
size_t gemm_fp32_workspace_bytes(int64_t m, int64_t n, int64_t k);

// tcgen05 3xTF32 kernels (gemm_tc.cu)
bool gemm_tc_rows_eligible(int64_t m, int64_t n, int64_t k, const float* a, int64_t a_rs, int64_t a_cs,
                           const float* c, int64_t ldc);
size_t gemm_tc_rows_workspace_bytes(int64_t m, int64_t n, int64_t k);
// ep_bias / ep_relu: C = act(A B + bias), applied by the kernel's epilogue
int gemm_tc_rows_launch(int64_t m, int64_t n, int64_t k, const float* a, int64_t lda, const float* b,
                        int64_t b_rs, int64_t b_cs, float* c, int64_t ldc, void* ws, size_t ws_bytes,
                        cudaStream_t stream, const float* ep_bias = nullptr, int ep_relu = 0);
bool gemm_tc_rows_beats_skinny(int64_t k);
bool gemm_tc_tn_eligible(int64_t m, int64_t n, int64_t r, const float* x, int64_t ldx, const float* y,
                         int64_t ldy);
size_t gemm_tc_tn_workspace_bytes(int64_t m, int64_t n, int64_t r);
int gemm_tc_tn_launch(int64_t m, int64_t n, int64_t r, const float* x, int64_t ldx, const float* y,
                      int64_t ldy, float* c, int64_t ldc, void* ws, size_t ws_bytes, cudaStream_t stream);

// CUDA-core kernels for narrow products over many rows (gemm_skinny.cu): K (resp. M) <= 64, N <= 64
bool gemm_skinny_rows_eligible(int64_t m, int64_t n, int64_t k, const float* a, int64_t a_rs, int64_t a_cs);
int gemm_skinny_rows_launch(int64_t m, int64_t n, int64_t k, const float* a, int64_t lda, const float* b, int64_t b_rs,
                            int64_t b_cs, float* c, int64_t ldc, cudaStream_t stream);
bool gemm_skinny_tn_eligible(int64_t m, int64_t n, int64_t r, const float* x, int64_t ldx, const float* y, int64_t ldy);
size_t gemm_skinny_tn_workspace_bytes(int64_t m, int64_t n, int64_t r);
// gx / db: optional third operand G [r, n] whose column sums are produced in the same pass (db = colsum(G))
int gemm_skinny_tn_launch(int64_t m, int64_t n, int64_t r, const float* x, int64_t ldx, const float* y, int64_t ldy,
                          float* c, int64_t ldc, void* ws, size_t ws_bytes, cudaStream_t stream,
                          const float* gx = nullptr, int64_t ldg = 0, float* db = nullptr);

int colsum_launch(int64_t n_rows, int64_t f, const float* g, int64_t ldg, const float* y,
                  int64_t ldy, float* gm, int64_t ldgm, float* out, void* ws, size_t ws_bytes,
                  cudaStream_t stream, const uint8_t* mask = nullptr, int64_t ld_mask = 0,
                  float mask_scale = 1.f);
size_t colsum_workspace_bytes(int64_t n_rows, int64_t f);

// out[(i / n) * ldo + i % n] = sum_{s < n_parts} partial[s * total + i], s ascending inside a fixed
// 8-lane tree (deterministic).  total = m * n.
// out[r, 0:f] = (accumulate ? out : 0) ... in place: out = act(out + bias)
// dst[r, 0:w4] = (src[r, 0:w], 0 ...) for r < n_rows, w4 = 4*ceil(w/4): zero-padded, 16-byte aligned rows
int pad_copy_launch(int64_t n_rows, int64_t w, const float* src, int64_t ld_src, float* dst, int64_t ld_dst,
                    cudaStream_t stream);

int bias_act_launch(int64_t n_rows, int64_t f, float* out, int64_t ldo, const Epilogue& ep, cudaStream_t stream);

// xout != nullptr: also xout[0:n] = the sum over parts of the fp64 xpart[n_parts][n], rounded to fp32 once (column
// sums); m may then be 0
int reduce_partials_launch(int64_t m, int64_t n, int n_parts, const float* partial, float* out,
                           int64_t ldo, cudaStream_t stream, const double* xpart = nullptr, float* xout = nullptr);

// ---- fp64 tier (spmm_f64.cu, gemm_f64.cu): the same products and epilogue on fp64 operands, over the fp64 values a
// handle keeps when it was built from fp64 data (gcnb_graph::val64 / t_val64)
struct Epilogue64 {
  const double* bias = nullptr;   // [f] or null
  int relu = 0;
  int accumulate = 0;             // add the previous contents of out first
  const uint8_t* mask = nullptr;  // [n_rows, ld_mask] keep-mask (0 / non-zero) or null
  int64_t ld_mask = 0;
  double mask_scale = 1.0;
};

// val: the view's fp64 values (g->val64 for g->fwd, g->t_val64 for g->bwd)
int spmm_f64_launch(const CsrView& a, const double* val, const double* b, int64_t ldb, int64_t f,
                    const Epilogue64& ep, double* out, int64_t ldo, void* ws, size_t ws_bytes, cudaStream_t stream);
size_t spmm_f64_workspace_bytes(const CsrView& a, int64_t f);
int gemm_f64_launch(int64_t m, int64_t n, int64_t k, const double* a, int64_t a_rs, int64_t a_cs, const double* b,
                    int64_t b_rs, int64_t b_cs, double* c, int64_t ldc, const Epilogue64& ep, void* ws, size_t ws_bytes,
                    cudaStream_t stream);
size_t gemm_f64_workspace_bytes(int64_t m, int64_t n, int64_t k);
int colsum_f64_launch(int64_t n_rows, int64_t f, const double* g, int64_t ldg, const double* y, int64_t ldy, double* gm,
                      int64_t ldgm, double* out, void* ws, size_t ws_bytes, cudaStream_t stream,
                      const uint8_t* mask = nullptr, int64_t ld_mask = 0, double mask_scale = 1.0);
size_t colsum_f64_workspace_bytes(int64_t n_rows, int64_t f);

}  // namespace gcnb

struct gcnb_graph {
  int device = 0;
  int64_t n_rows = 0, n_cols = 0, nnz = 0;
  int32_t* rowptr = nullptr;
  int32_t* col = nullptr;
  float* val = nullptr;
  int32_t* t_rowptr = nullptr;  // may alias rowptr when the pattern is symmetric
  int32_t* t_col = nullptr;     // may alias col
  float* t_val = nullptr;
  uint2* pair = nullptr;    // interleaved (col, val) of the CSR, [nnz]
  uint2* t_pair = nullptr;  // interleaved (t_col, t_val) of the CSR of the transpose, [nnz]
  bool pattern_symmetric = false;
  bool has_transpose = true;  // false for row/column blocks cut by gcnb_graph_block
  // dense route (adjacency given as a dense matrix whose density makes the CSR gather the slower
  // path): zero-padded copies of A [n_rows, ld_fwd] and A^T [n_cols, ld_bwd], ld = 4*ceil(./4)
  float* dense_fwd = nullptr;
  float* dense_bwd = nullptr;
  int64_t ld_fwd = 0, ld_bwd = 0;
  int32_t* long_rows = nullptr;
  int32_t* long_chunk_ptr = nullptr;
  int32_t* t_long_rows = nullptr;
  int32_t* t_long_chunk_ptr = nullptr;
  uint32_t* stream_items = nullptr;
  uint32_t* t_stream_items = nullptr;
  gcnb::CsrView fwd, bwd;
  int64_t device_bytes = 0;
  // fp64 values of the CSR and of the CSR of A^T, in the order of val / t_val (whose entries are their fp32 rounding);
  // only on handles built from fp64 data (gcnb_graph_from_*_f64, GCNB_BUILD_KEEP_F64), null otherwise
  double* val64 = nullptr;
  double* t_val64 = nullptr;
};
