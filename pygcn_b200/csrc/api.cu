// extern "C" entry points of libgcnb200.so (see include/gcnb200.h).
#include <stdarg.h>
#include <string.h>

#include "common.cuh"

namespace gcnb {

static thread_local char g_error[1024] = "";

static long long g_launch_count = 0;
void count_launch() { __atomic_add_fetch(&g_launch_count, 1, __ATOMIC_RELAXED); }

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_error, sizeof(g_error), fmt, ap);
  va_end(ap);
}

namespace {

inline size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

constexpr double kTcMinWork = 1.0e7;  // m*n*k below this: launch overhead dominates, keep the CUDA-core kernel

// which kernel serves a product: 0 = CUDA-core fp32, 1 = tcgen05 rows, 2 = tcgen05 tn
int gemm_route(int64_t m, int64_t n, int64_t k, const float* a, int64_t a_rs, int64_t a_cs, const float* b,
               int64_t b_rs, int64_t b_cs, const float* c, int64_t ldc, int precision) {
  if (precision == GCNB_GEMM_FP32) return 0;
  if (precision == GCNB_GEMM_AUTO && (double)m * (double)n * (double)k < kTcMinWork) return 0;
  if (gemm_tc_rows_eligible(m, n, k, a, a_rs, a_cs, c, ldc)) return 1;
  if (a_rs == 1 && b_cs == 1 && gemm_tc_tn_eligible(m, n, k, a, a_cs, b, b_rs)) return 2;
  return 0;
}

// Widths that are not a multiple of 4 floats (Reddit's 602 features) break the 16-byte loads of the
// tensor-core kernels.  For products big enough to matter the operand is copied once into scratch with
// rows zero-padded to the next multiple of 4 (one extra read + write of it: 0.17 ms for Reddit's X,
// against 4.4 ms for the CUDA-core kernel) and the tensor-core kernel runs on the copy.
constexpr double kPadMinWork = 1.0e8;
inline int64_t pad4(int64_t v) { return ceil_div(v, 4) * 4; }
// 1: A [m,k] row-major with k % 4 != 0 -> rows kernel on a padded copy; 2: A = X^T with X [k rows, m cols],
// m % 4 != 0 -> tn kernel on a padded copy of X; 0: no
int gemm_pad_route(int64_t m, int64_t n, int64_t k, int64_t a_rs, int64_t a_cs, const float* b, int64_t b_rs,
                   int64_t b_cs, int precision) {
  if (precision == GCNB_GEMM_FP32 || (double)m * (double)n * (double)k < kPadMinWork) return 0;
  if (a_cs == 1 && k % 4 != 0 && k <= (1 << 20) && n <= (1 << 20)) return 1;
  if (a_rs == 1 && b_cs == 1 && m % 4 != 0 && n <= 256 && b_rs % 4 == 0 && b_rs >= pad4(n) &&
      (reinterpret_cast<uintptr_t>(b) & 15u) == 0)
    return 2;
  return 0;
}
size_t gemm_pad_bytes(int64_t m, int64_t n, int64_t k, int precision) {
  if (precision == GCNB_GEMM_FP32 || (double)m * (double)n * (double)k < kPadMinWork) return 0;
  size_t r = 0;
  if (k % 4 != 0) r = (size_t)m * (size_t)pad4(k) * sizeof(float);
  if (m % 4 != 0) {
    const size_t t = (size_t)k * (size_t)pad4(m) * sizeof(float);
    if (t > r) r = t;
  }
  return r ? align256(r) : 0;
}

// fuse: optional (bias, ReLU) the TMA-fed tensor-core rows kernel applies in its epilogue; *fused says whether it did
int gemm_dispatch(int64_t m, int64_t n, int64_t k, const float* a, int64_t a_rs, int64_t a_cs,
                  const float* b, int64_t b_rs, int64_t b_cs, float* c, int64_t ldc, int precision,
                  void* ws, size_t ws_bytes, cudaStream_t st, const Epilogue* fuse = nullptr, bool* fused = nullptr) {
  const float* fb = fuse ? fuse->bias : nullptr;
  const int fr = fuse ? fuse->relu : 0;
  if (fused) *fused = false;
  GCNB_REQUIRE(precision == GCNB_GEMM_FP32 || precision == GCNB_GEMM_TF32X3 || precision == GCNB_GEMM_AUTO,
               "gemm: unknown precision %d", precision);
  GCNB_REQUIRE(m >= 0 && n >= 0 && k >= 0, "gemm: negative dimension");
  GCNB_REQUIRE(ldc >= n, "gemm: ldc < n");
  if (m == 0 || n == 0) return GCNB_OK;
  // narrow products over many rows (CBG 64->32, the fork's 8->32): HBM-bound streams, exact fp32 on CUDA
  // cores beats the tensor-core pipeline's fixed costs; "tf32x3" still forces the tcgen05 kernels
  if (precision != GCNB_GEMM_TF32X3) {
    if (gemm_skinny_rows_eligible(m, n, k, a, a_rs, a_cs) &&
        !(precision == GCNB_GEMM_AUTO && (double)m * (double)n * (double)k >= kTcMinWork && gemm_tc_rows_beats_skinny(k) &&
          gemm_tc_rows_eligible(m, n, k, a, a_rs, a_cs, c, ldc)))
      return gemm_skinny_rows_launch(m, n, k, a, a_rs, b, b_rs, b_cs, c, ldc, st);
    if (a_rs == 1 && b_cs == 1 && gemm_skinny_tn_eligible(m, n, k, a, a_cs, b, b_rs) && ws != nullptr &&
        ws_bytes >= gemm_skinny_tn_workspace_bytes(m, n, k))
      return gemm_skinny_tn_launch(m, n, k, a, a_cs, b, b_rs, c, ldc, ws, ws_bytes, st);
  }
  switch (gemm_route(m, n, k, a, a_rs, a_cs, b, b_rs, b_cs, c, ldc, precision)) {
    case 1:
      if (fused) *fused = true;
      return gemm_tc_rows_launch(m, n, k, a, a_rs, b, b_rs, b_cs, c, ldc, ws, ws_bytes, st, fb, fr);
    case 2:
      return gemm_tc_tn_launch(m, n, k, a, a_cs, b, b_rs, c, ldc, ws, ws_bytes, st);
    default:
      break;
  }
  const int pr = gemm_pad_route(m, n, k, a_rs, a_cs, b, b_rs, b_cs, precision);
  const size_t pad_bytes = gemm_pad_bytes(m, n, k, precision);
  if (pr != 0 && pad_bytes != 0 && ws != nullptr && ws_bytes > pad_bytes) {
    float* pad = reinterpret_cast<float*>(ws);
    char* rest = reinterpret_cast<char*>(ws) + pad_bytes;
    const size_t rest_bytes = ws_bytes - pad_bytes;
    if (pr == 1) {
      const int64_t k4 = pad4(k);
      GCNB_TRY(pad_copy_launch(m, k, a, a_rs, pad, k4, st));
      if (gemm_tc_rows_eligible(m, n, k4, pad, k4, 1, c, ldc) && rest_bytes >= gemm_tc_rows_workspace_bytes(m, n, k)) {
        if (fused) *fused = true;
        return gemm_tc_rows_launch(m, n, k, pad, k4, b, b_rs, b_cs, c, ldc, rest, rest_bytes, st, fb, fr);
      }
    } else {
      const int64_t m4 = pad4(m);
      GCNB_TRY(pad_copy_launch(k, m, a, a_cs, pad, m4, st));  // X [k rows, m cols], row stride a_cs
      if (gemm_tc_tn_eligible(m, n, k, pad, m4, b, b_rs) &&
          rest_bytes >= gemm_tc_tn_workspace_bytes(m, n, k))
        return gemm_tc_tn_launch(m, n, k, pad, m4, b, b_rs, c, ldc, rest, rest_bytes, st);
    }
  }
  return gemm_fp32_launch(m, n, k, a, a_rs, a_cs, b, b_rs, b_cs, c, ldc, ws, ws_bytes, st);
}

// C = dropout(relu(A B + bias)): the epilogue rides in the GEMM when the kernel that runs can take it, and is one
// in-place pass over C otherwise (small / unaligned shapes); a dropout mask is always that pass
int gemm_dispatch_ep(int64_t m, int64_t n, int64_t k, const float* a, int64_t a_rs, int64_t a_cs, const float* b,
                     int64_t b_rs, int64_t b_cs, float* c, int64_t ldc, int precision, void* ws, size_t ws_bytes,
                     cudaStream_t st, const Epilogue& ep) {
  bool fused = false;
  GCNB_TRY(gemm_dispatch(m, n, k, a, a_rs, a_cs, b, b_rs, b_cs, c, ldc, precision, ws, ws_bytes, st, &ep, &fused));
  Epilogue rest = ep;
  if (fused) {
    rest.bias = nullptr;
    rest.relu = 0;
  }
  return bias_act_launch(m, n, c, ldc, rest, st);
}

// conservative: large enough for whichever kernel the route picks at call time
size_t gemm_ws(int64_t m, int64_t n, int64_t k, int precision) {
  size_t w = gemm_fp32_workspace_bytes(m, n, k);
  if (m <= 64 && n <= 32 && k >= 4096) {
    const size_t sk = gemm_skinny_tn_workspace_bytes(m, n, k);
    if (sk > w) w = sk;
  }
  if (precision != GCNB_GEMM_FP32 && m > 0 && n > 0 && k > 0) {
    const size_t r = gemm_tc_rows_workspace_bytes(m, n, k);
    const size_t t = (n <= 256) ? gemm_tc_tn_workspace_bytes(m, n, k) : 0;
    if (r > w) w = r;
    if (t > w) w = t;
    w = align256(w) + gemm_pad_bytes(m, n, k, precision);
  }
  return (w + 255) & ~(size_t)255;
}

// out = op(A) * B (+ bias) (relu) for a graph handle: CSR SpMM, or -- for handles on the dense route --
// a tensor-core GEMM over the zero-padded dense copy:  C[M,F] = sum_r X[r,M]^T B[r,F]  with X = A^T
// (forward) or A (transpose), i.e. the split-K "tn" kernel in both directions.
size_t graph_matmul_ws(const gcnb_graph* g, bool transpose, int64_t f) {
  const CsrView& v = transpose ? g->bwd : g->fwd;
  size_t w = spmm_workspace_bytes(v, f);
  if (g->dense_fwd) {
    const int64_t m = transpose ? g->n_cols : g->n_rows, r = transpose ? g->n_rows : g->n_cols;
    const int64_t fw = f < 256 ? f : 256;
    size_t a = gemm_fp32_workspace_bytes(m, fw, r);
    size_t b = gemm_tc_tn_workspace_bytes(m, fw, r);
    if (a > w) w = a;
    if (b > w) w = b;
  }
  return w;
}

int graph_matmul(const gcnb_graph* g, bool transpose, const float* b, int64_t ldb, int64_t f, const Epilogue& ep,
                 float* out, int64_t ldo, void* ws, size_t ws_bytes, cudaStream_t st) {
  const CsrView& v = transpose ? g->bwd : g->fwd;
  GCNB_REQUIRE(ep.mask == nullptr || ep.ld_mask >= f, "spmm: dropout mask leading dimension smaller than width");
  if (!g->dense_fwd || ep.accumulate) {
    return spmm_launch(v, b, ldb, f, ep, out, ldo, ws, ws_bytes, st);
  }
  GCNB_REQUIRE(f > 0 && ldb >= f && ldo >= f, "spmm(dense route): bad width / leading dimension");
  const int64_t m = transpose ? g->n_cols : g->n_rows;   // output rows
  const int64_t r = transpose ? g->n_rows : g->n_cols;   // reduction length
  const float* x = transpose ? g->dense_fwd : g->dense_bwd;
  const int64_t ldx = transpose ? g->ld_fwd : g->ld_bwd;
  GCNB_REQUIRE(ws_bytes >= graph_matmul_ws(g, transpose, f), "spmm(dense route): workspace too small");
  // the tn kernel takes up to 256 output columns: wider operands (batched layers) go in column panels
  for (int64_t f0 = 0; f0 < f; f0 += 256) {
    const int64_t fw = (f - f0 < 256) ? (f - f0) : 256;
    // Small products (the fork's 2943 x 2943 adjacency, 32 columns) take the exact-fp32 CUDA-core kernel: a
    // row-normalised dense adjacency averages ~3000 terms that cancel to a few % of their mass, and the tensor-core
    // path's truncating TMEM accumulation then shows as 3e-6 ... 1e-5 of the result (cuBLAS fp32: 3e-7 ... 9e-7,
    // profiles/r02_debug_ref_models.txt) -- inside the bar, but the reference's fresh BatchNorm amplifies it 100x.
    const bool big = (double)m * (double)fw * (double)r >= 4.0e9;
    if (big && gemm_tc_tn_eligible(m, fw, r, x, ldx, b + f0, ldb) && (f0 % 4 == 0)) {
      GCNB_TRY(gemm_tc_tn_launch(m, fw, r, x, ldx, b + f0, ldb, out + f0, ldo, ws, ws_bytes, st));
    } else {
      GCNB_TRY(gemm_fp32_launch(m, fw, r, x, 1, ldx, b + f0, ldb, 1, out + f0, ldo, ws, ws_bytes, st));
    }
  }
  return bias_act_launch(m, f, out, ldo, ep, st);
}

Epilogue make_epilogue(const float* bias, bool relu, bool accumulate, const uint8_t* mask, int64_t ld_mask, float scale) {
  Epilogue ep;
  ep.bias = bias;
  ep.relu = relu ? 1 : 0;
  ep.accumulate = accumulate ? 1 : 0;
  ep.mask = mask;
  ep.ld_mask = ld_mask;
  ep.mask_scale = scale;
  return ep;
}

}  // namespace
}  // namespace gcnb

using namespace gcnb;

extern "C" int gcnb_version(void) { return GCNB_VERSION; }

extern "C" const char* gcnb_last_error(void) { return g_error; }

extern "C" long long gcnb_launch_count(void) { return __atomic_load_n(&g_launch_count, __ATOMIC_RELAXED); }

extern "C" int gcnb_check_device(void) {
  int dev = 0;
  GCNB_CUDA(cudaGetDevice(&dev));
  int major = 0;
  GCNB_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  if (major != 10) {
    set_error("libgcnb200 is built for sm_100a only; device %d has compute capability major %d", dev, major);
    return GCNB_E_UNSUPPORTED;
  }
  return GCNB_OK;
}

extern "C" int gcnb_set_tuning(int key, int value) { return spmm_set_tuning(key, value); }

extern "C" int gcnb_spmm(const gcnb_graph* g, int flags, const float* d_b, int64_t ldb, int64_t f,
                         const float* d_bias, float* d_out, int64_t ldo, void* d_ws, size_t ws_bytes,
                         void* stream) {
  GCNB_REQUIRE(g != nullptr, "spmm: null graph");
  GCNB_REQUIRE(!(flags & GCNB_SPMM_TRANSPOSE) || g->has_transpose, "spmm: this handle is a block without a transpose");
  return graph_matmul(g, (flags & GCNB_SPMM_TRANSPOSE) != 0, d_b, ldb, f,
                      make_epilogue(d_bias, (flags & GCNB_SPMM_RELU) != 0, (flags & GCNB_SPMM_ACCUMULATE) != 0, nullptr, 0,
                                    1.f),
                      d_out, ldo, d_ws, ws_bytes, (cudaStream_t)stream);
}

extern "C" int gcnb_spmm_bf16(const gcnb_graph* g, int flags, const uint16_t* d_b, int64_t ldb, int64_t f,
                              const float* d_bias, float* d_out, int64_t ldo, void* d_ws, size_t ws_bytes,
                              void* stream) {
  GCNB_REQUIRE(g != nullptr, "spmm_bf16: null graph");
  const bool transpose = (flags & GCNB_SPMM_TRANSPOSE) != 0;
  GCNB_REQUIRE(!transpose || g->has_transpose, "spmm_bf16: this handle is a block without a transpose");
  GCNB_REQUIRE(g->dense_fwd == nullptr, "spmm_bf16: handles on the dense route have no bf16 panel path (use gcnb_spmm)");
  return spmm_bf16_launch(transpose ? g->bwd : g->fwd, d_b, ldb, f,
                          make_epilogue(d_bias, (flags & GCNB_SPMM_RELU) != 0, (flags & GCNB_SPMM_ACCUMULATE) != 0,
                                        nullptr, 0, 1.f),
                          d_out, ldo, d_ws, ws_bytes, (cudaStream_t)stream);
}

extern "C" int gcnb_to_bf16(int64_t n_rows, int64_t f, const float* d_src, int64_t ld_src, uint16_t* d_dst,
                            int64_t ld_dst, void* stream) {
  return to_bf16_launch(n_rows, f, d_src, ld_src, d_dst, ld_dst, (cudaStream_t)stream);
}

extern "C" size_t gcnb_spmm_workspace_bytes(const gcnb_graph* g, int flags, int64_t f) {
  if (!g) return 0;
  return graph_matmul_ws(g, (flags & GCNB_SPMM_TRANSPOSE) != 0, f);
}

extern "C" int gcnb_gemm(int64_t m, int64_t n, int64_t k, const float* d_a, int64_t a_rs, int64_t a_cs,
                         const float* d_b, int64_t b_rs, int64_t b_cs, float* d_c, int64_t ldc,
                         int precision, void* d_ws, size_t ws_bytes, void* stream) {
  return gemm_dispatch(m, n, k, d_a, a_rs, a_cs, d_b, b_rs, b_cs, d_c, ldc, precision, d_ws, ws_bytes,
                       (cudaStream_t)stream);
}

extern "C" int gcnb_gemm_ex(int64_t m, int64_t n, int64_t k, const float* d_a, int64_t a_rs, int64_t a_cs,
                            const float* d_b, int64_t b_rs, int64_t b_cs, float* d_c, int64_t ldc, const float* d_bias,
                            int relu, int precision, void* d_ws, size_t ws_bytes, void* stream) {
  return gemm_dispatch_ep(m, n, k, d_a, a_rs, a_cs, d_b, b_rs, b_cs, d_c, ldc, precision, d_ws, ws_bytes, (cudaStream_t)stream,
                          make_epilogue(d_bias, relu != 0, false, nullptr, 0, 1.f));
}

extern "C" size_t gcnb_gemm_workspace_bytes(int64_t m, int64_t n, int64_t k, int precision) {
  return gemm_ws(m, n, k, precision);
}

extern "C" int gcnb_colsum(int64_t n_rows, int64_t f, const float* d_g, int64_t ldg, const float* d_y,
                           int64_t ldy, float* d_gm, int64_t ldgm, float* d_out, void* d_ws,
                           size_t ws_bytes, void* stream) {
  return colsum_launch(n_rows, f, d_g, ldg, d_y, ldy, d_gm, ldgm, d_out, d_ws, ws_bytes,
                       (cudaStream_t)stream);
}

extern "C" size_t gcnb_colsum_workspace_bytes(int64_t n_rows, int64_t f) {
  return colsum_workspace_bytes(n_rows, f);
}

// ------------------------------------------------------------------------ layer level

extern "C" size_t gcnb_layer_workspace_bytes(const gcnb_graph* g, int64_t fin, int64_t fout, int precision) {
  if (!g) return 0;
  size_t s = 0;
  for (int64_t w : {fout, fin})  // (the aggregate-first order runs its SpMMs at width fin)
    for (bool t : {false, true}) {
      const size_t v = graph_matmul_ws(g, t, w);
      if (v > s) s = v;
    }
  size_t c = colsum_workspace_bytes(g->n_rows, fout);
  size_t d0 = gemm_ws(g->n_cols, fout, fin, precision);  // X W
  size_t d1 = gemm_ws(fin, fout, g->n_cols, precision);  // X^T dS
  size_t d2 = gemm_ws(g->n_cols, fin, fout, precision);  // dS W^T
  size_t d3 = gemm_ws(g->n_rows, fout, fin, precision);  // (A X) W and, transposed roles, G W^T
  size_t d4 = gemm_ws(g->n_rows, fin, fout, precision);
  size_t d5 = gemm_ws(fin, fout, g->n_rows, precision);  // (A X)^T G
  size_t d = d0 > d1 ? d0 : d1;
  d = d > d2 ? d : d2;
  d = d > d3 ? d : d3;
  d = d > d4 ? d : d4;
  d = d > d5 ? d : d5;
  // regions are used by different kernels of one call that run back to back on one stream,
  // but colsum / spmm / gemm scratch never overlap in time with themselves only -- keep them
  // disjoint to stay safe under future multi-stream use.
  return align256(s) + align256(c) + align256(d) + 256;
}

extern "C" int gcnb_layer_forward(const gcnb_graph* g, const float* d_x, int64_t ldx, const float* d_w,
                                  const float* d_bias, int64_t fin, int64_t fout, int flags, int precision,
                                  const uint8_t* d_mask, float mask_scale, float* d_support, float* d_out,
                                  void* d_ws, size_t ws_bytes, void* stream) {
  GCNB_REQUIRE(g != nullptr, "layer_forward: null graph");
  GCNB_REQUIRE(fin > 0 && fout > 0, "layer_forward: bad feature sizes %lld -> %lld", (long long)fin, (long long)fout);
  GCNB_REQUIRE(ldx >= fin, "layer_forward: ldx < in_features");
  cudaStream_t st = (cudaStream_t)stream;
  char* ws = reinterpret_cast<char*>(d_ws);
  if (flags & GCNB_LAYER_AGG_FIRST) {
    // out = (A X) W + bias: the SpMM gathers rows of X (width fin) instead of rows of X W (width fout) -- the order
    // that moves fewer bytes when fin < fout.  d_support receives A X [n_rows, 4*ceil(fin/4)], kept for backward.
    GCNB_REQUIRE(!g->dense_fwd, "layer_forward: the aggregate-first order is for CSR handles");
    const size_t s_bytes = align256(graph_matmul_ws(g, false, fin));
    const size_t d_bytes = gemm_ws(g->n_rows, fout, fin, precision);
    GCNB_REQUIRE(ws_bytes >= s_bytes + d_bytes && (s_bytes + d_bytes == 0 || ws != nullptr),
                 "layer_forward: workspace too small");
    const int64_t ldax = ceil_div(fin, 4) * 4;
    GCNB_TRY(graph_matmul(g, false, d_x, ldx, fin, Epilogue(), d_support, ldax, ws, s_bytes, st));
    return gemm_dispatch_ep(g->n_rows, fout, fin, d_support, ldax, 1, d_w, fout, 1, d_out, fout, precision, ws + s_bytes,
                            d_bytes, st, make_epilogue(d_bias, (flags & GCNB_LAYER_RELU) != 0, false, d_mask, fout, mask_scale));
  }
  const size_t s_bytes = align256(graph_matmul_ws(g, false, fout));
  const size_t d_bytes = gemm_ws(g->n_cols, fout, fin, precision);
  GCNB_REQUIRE(ws_bytes >= s_bytes + d_bytes && (s_bytes + d_bytes == 0 || ws != nullptr),
               "layer_forward: workspace too small");
  // support = X W                                   (pygcn/layers.py:33)
  const int64_t lds = ceil_div(fout, 4) * 4;
  GCNB_TRY(gemm_dispatch(g->n_cols, fout, fin, d_x, ldx, 1, d_w, fout, 1, d_support, lds, precision,
                         ws + s_bytes, d_bytes, st));
  // out = A support (+ bias) (relu)                  (pygcn/layers.py:34-36, models.py:49)
  return graph_matmul(g, false, d_support, lds, fout,
                      make_epilogue(d_bias, (flags & GCNB_LAYER_RELU) != 0, false, d_mask, fout, mask_scale), d_out,
                      fout, ws, s_bytes, st);
}

extern "C" int gcnb_layer_backward(const gcnb_graph* g, const float* d_x, int64_t ldx, const float* d_w,
                                   const float* d_g, int64_t ldg, const float* d_y, int64_t fin,
                                   int64_t fout, int flags, int precision, const uint8_t* d_mask,
                                   float mask_scale, float* d_gm, float* d_ds,
                                   float* d_dw, float* d_db, float* d_dx, int64_t lddx, void* d_ws,
                                   size_t ws_bytes, void* stream) {
  GCNB_REQUIRE(g != nullptr, "layer_backward: null graph");
  GCNB_REQUIRE(g->has_transpose, "layer_backward: this handle is a block without a transpose");
  GCNB_REQUIRE(fin > 0 && fout > 0, "layer_backward: bad feature sizes");
  GCNB_REQUIRE(ldg >= fout, "layer_backward: ldg < out_features");
  cudaStream_t st = (cudaStream_t)stream;
  const bool relu = (flags & GCNB_LAYER_RELU) != 0;
  const bool need_dx = (flags & GCNB_LAYER_NEED_DX) != 0;
  const bool need_dw = (flags & GCNB_LAYER_NEED_DW) != 0;
  const bool need_db = (flags & GCNB_LAYER_NEED_DB) != 0;
  GCNB_REQUIRE(!relu || (d_y != nullptr && d_gm != nullptr), "layer_backward: relu needs y and gm");
  GCNB_REQUIRE(d_mask == nullptr || d_gm != nullptr, "layer_backward: dropout mask needs gm");
  GCNB_REQUIRE(ws_bytes >= gcnb_layer_workspace_bytes(g, fin, fout, precision) && d_ws != nullptr,
               "layer_backward: workspace too small");
  char* ws = reinterpret_cast<char*>(d_ws);
  const bool agg_first = (flags & GCNB_LAYER_AGG_FIRST) != 0;
  const int64_t sw = agg_first ? fin : fout;  // width of this order's SpMMs
  const size_t s_bytes = align256(graph_matmul_ws(g, true, sw) > graph_matmul_ws(g, false, sw)
                                      ? graph_matmul_ws(g, true, sw)
                                      : graph_matmul_ws(g, false, sw));
  const size_t c_bytes = align256(colsum_workspace_bytes(g->n_rows, fout));
  void* ws_spmm = ws;
  void* ws_col = ws + s_bytes;
  void* ws_gemm = ws + s_bytes + c_bytes;
  const size_t g_bytes = ws_bytes - s_bytes - c_bytes;

  const float* gsrc = d_g;
  int64_t gld = ldg;
  // db = colsum(G) ; with the fused ReLU the mask is applied first: G <- G * [y > 0]
  const bool masked = relu || d_mask != nullptr;
  // d_gm [n_rows, ld4(fout)]: the staged copy of G the SpMM / dW product read -- the masked gradient, or a plain copy
  // when the caller's G has rows that are not 16-byte aligned (fout = 47: the scalar SpMM is 20x slower than one
  // extra pass over G)
  const int64_t lds_ = ceil_div(fout, 4) * 4;
  const bool stage = d_gm != nullptr;
  // Without a mask, db = colsum(G) rides in the narrow dW kernel (third operand, gemm_skinny.cu): G and dS have the
  // same number of rows when the adjacency is square, so the pass over (X, dS) adds G's column sums for free.
  const bool fuse_db = !agg_first && !masked && !stage && need_db && need_dw && precision != GCNB_GEMM_TF32X3 && g->n_rows == g->n_cols &&
                       d_db != nullptr && ldg % 4 == 0 && (reinterpret_cast<uintptr_t>(d_g) & 15u) == 0 &&
                       gemm_skinny_tn_eligible(fin, fout, g->n_cols, d_x, ldx, d_ds, lds_) &&
                       g_bytes >= gemm_skinny_tn_workspace_bytes(fin, fout, g->n_cols);
  if (!fuse_db && (masked || need_db || stage)) {
    float* db = d_db;
    GCNB_REQUIRE(db != nullptr || !need_db, "layer_backward: db requested but null");
    if (db == nullptr) db = reinterpret_cast<float*>(ws_gemm);  // discard
    // with ReLU + dropout the forward output y is 0 wherever relu clipped or the mask dropped, and
    // scale * relu(.) > 0 elsewhere, so [y > 0] is still the ReLU mask for the kept entries
    GCNB_TRY(colsum_launch(g->n_rows, fout, d_g, ldg, relu ? d_y : nullptr, fout, stage ? d_gm : nullptr,
                           lds_, db, ws_col, c_bytes, st, d_mask, fout, mask_scale));
    if (stage) {
      gsrc = d_gm;
      gld = lds_;
    }
  }
  if (!need_dw && !need_dx) return GCNB_OK;
  if (agg_first) {
    // forward was out = (A X) W + b with d_x = A X [n_rows, 4*ceil(fin/4)] kept from it:
    //   dW = (A X)^T G   -- no SpMM at all;   dX = A^T (G W^T)  -- one SpMM of width fin, only when asked for
    const int64_t ldax = ceil_div(fin, 4) * 4;
    GCNB_REQUIRE(ldx >= fin, "layer_backward: ld of the saved A X < in_features");
    if (need_dw) {
      GCNB_REQUIRE(d_dw != nullptr, "layer_backward: dW requested but null");
      GCNB_TRY(gemm_dispatch(fin, fout, g->n_rows, d_x, 1, ldx, gsrc, gld, 1, d_dw, fout, precision, ws_gemm, g_bytes, st));
    }
    if (need_dx) {
      GCNB_REQUIRE(d_dx != nullptr && lddx >= fin && d_ds != nullptr, "layer_backward: dX requested but null / lddx < in_features");
      GCNB_TRY(gemm_dispatch(g->n_rows, fin, fout, gsrc, gld, 1, d_w, 1, fout, d_ds, ldax, precision, ws_gemm, g_bytes, st));
      GCNB_TRY(graph_matmul(g, true, d_ds, ldax, fin, Epilogue(), d_dx, lddx, ws_spmm, s_bytes, st));
    }
    return GCNB_OK;
  }
  // dS = A^T G                                      (MmBackward0 of torch.spmm)
  const int64_t lds = ceil_div(fout, 4) * 4;
  GCNB_TRY(graph_matmul(g, true, gsrc, gld, fout, Epilogue(), d_ds, lds, ws_spmm, s_bytes, st));
  // dW = X^T dS                                     (MmBackward0 of torch.mm)
  if (need_dw) {
    GCNB_REQUIRE(d_dw != nullptr, "layer_backward: dW requested but null");
    if (fuse_db) {
      GCNB_TRY(gemm_skinny_tn_launch(fin, fout, g->n_cols, d_x, ldx, d_ds, lds, d_dw, fout, ws_gemm, g_bytes, st, d_g, ldg,
                                     d_db));
    } else {
      GCNB_TRY(gemm_dispatch(fin, fout, g->n_cols, d_x, 1, ldx, d_ds, lds, 1, d_dw, fout, precision, ws_gemm,
                             g_bytes, st));
    }
  }
  // dX = dS W^T
  if (need_dx) {
    GCNB_REQUIRE(d_dx != nullptr && lddx >= fin, "layer_backward: dX requested but null / lddx < in_features");
    GCNB_TRY(gemm_dispatch(g->n_cols, fin, fout, d_ds, lds, 1, d_w, 1, fout, d_dx, lddx, precision, ws_gemm,
                           g_bytes, st));
  }
  return GCNB_OK;
}

// ------------------------------------------------------------------------ fp64 tier

namespace gcnb {
namespace {

inline int64_t ld2(int64_t f) { return ceil_div(f, 2) * 2; }

int require_f64(const gcnb_graph* g, bool transpose, const char* what) {
  GCNB_REQUIRE(g != nullptr, "%s: null graph", what);
  GCNB_REQUIRE(g->val64 != nullptr,
               "%s: the graph handle has no fp64 values (build it with a gcnb_graph_from_*_f64 constructor or "
               "GCNB_BUILD_KEEP_F64)", what);
  GCNB_REQUIRE(!transpose || (g->has_transpose && g->t_val64 != nullptr), "%s: this handle has no transpose", what);
  return GCNB_OK;
}

int spmm_f64_graph(const gcnb_graph* g, bool transpose, const double* b, int64_t ldb, int64_t f, const Epilogue64& ep,
                   double* out, int64_t ldo, void* ws, size_t ws_bytes, cudaStream_t st) {
  return spmm_f64_launch(transpose ? g->bwd : g->fwd, transpose ? g->t_val64 : g->val64, b, ldb, f, ep, out, ldo, ws,
                         ws_bytes, st);
}

Epilogue64 make_epilogue64(const double* bias, bool relu, bool accumulate, const uint8_t* mask, int64_t ld_mask,
                           double scale) {
  Epilogue64 ep;
  ep.bias = bias;
  ep.relu = relu ? 1 : 0;
  ep.accumulate = accumulate ? 1 : 0;
  ep.mask = mask;
  ep.ld_mask = ld_mask;
  ep.mask_scale = scale;
  return ep;
}

struct LayerF64Ws {
  size_t s, c, d;
};

LayerF64Ws layer_f64_regions(const gcnb_graph* g, int64_t fin, int64_t fout) {
  LayerF64Ws r{0, 0, 0};
  for (int64_t w : {fout, fin})
    for (const CsrView* v : {&g->fwd, &g->bwd}) {
      const size_t b = spmm_f64_workspace_bytes(*v, w);
      if (b > r.s) r.s = b;
    }
  r.c = colsum_f64_workspace_bytes(g->n_rows, fout);
  const size_t d[6] = {gemm_f64_workspace_bytes(g->n_cols, fout, fin),   // X W
                       gemm_f64_workspace_bytes(fin, fout, g->n_cols),   // X^T dS
                       gemm_f64_workspace_bytes(g->n_cols, fin, fout),   // dS W^T
                       gemm_f64_workspace_bytes(g->n_rows, fout, fin),   // (A X) W
                       gemm_f64_workspace_bytes(g->n_rows, fin, fout),   // G W^T
                       gemm_f64_workspace_bytes(fin, fout, g->n_rows)};  // (A X)^T G
  for (size_t v : d)
    if (v > r.d) r.d = v;
  r.s = align256(r.s);
  r.c = align256(r.c);
  r.d = align256(r.d);
  return r;
}

}  // namespace
}  // namespace gcnb

extern "C" int gcnb_spmm_f64(const gcnb_graph* g, int flags, const double* d_b, int64_t ldb, int64_t f,
                             const double* d_bias, const uint8_t* d_mask, int64_t ld_mask, double mask_scale,
                             double* d_out, int64_t ldo, void* d_ws, size_t ws_bytes, void* stream) {
  const bool transpose = (flags & GCNB_SPMM_TRANSPOSE) != 0;
  GCNB_TRY(require_f64(g, transpose, "spmm_f64"));
  GCNB_REQUIRE((flags & ~(GCNB_SPMM_TRANSPOSE | GCNB_SPMM_RELU | GCNB_SPMM_ACCUMULATE)) == 0, "spmm_f64: unknown flags");
  return spmm_f64_graph(g, transpose, d_b, ldb, f,
                        make_epilogue64(d_bias, (flags & GCNB_SPMM_RELU) != 0, (flags & GCNB_SPMM_ACCUMULATE) != 0, d_mask,
                                        ld_mask, mask_scale),
                        d_out, ldo, d_ws, ws_bytes, (cudaStream_t)stream);
}

extern "C" size_t gcnb_spmm_f64_workspace_bytes(const gcnb_graph* g, int flags, int64_t f) {
  if (!g) return 0;
  return spmm_f64_workspace_bytes((flags & GCNB_SPMM_TRANSPOSE) ? g->bwd : g->fwd, f);
}

extern "C" int gcnb_gemm_f64(int64_t m, int64_t n, int64_t k, const double* d_a, int64_t a_rs, int64_t a_cs,
                             const double* d_b, int64_t b_rs, int64_t b_cs, double* d_c, int64_t ldc, void* d_ws,
                             size_t ws_bytes, void* stream) {
  return gemm_f64_launch(m, n, k, d_a, a_rs, a_cs, d_b, b_rs, b_cs, d_c, ldc, Epilogue64(), d_ws, ws_bytes,
                         (cudaStream_t)stream);
}

extern "C" int gcnb_gemm_f64_ex(int64_t m, int64_t n, int64_t k, const double* d_a, int64_t a_rs, int64_t a_cs,
                                const double* d_b, int64_t b_rs, int64_t b_cs, double* d_c, int64_t ldc,
                                const double* d_bias, int relu, void* d_ws, size_t ws_bytes, void* stream) {
  return gemm_f64_launch(m, n, k, d_a, a_rs, a_cs, d_b, b_rs, b_cs, d_c, ldc,
                         make_epilogue64(d_bias, relu != 0, false, nullptr, 0, 1.0), d_ws, ws_bytes, (cudaStream_t)stream);
}

extern "C" size_t gcnb_gemm_f64_workspace_bytes(int64_t m, int64_t n, int64_t k) { return gemm_f64_workspace_bytes(m, n, k); }

extern "C" int gcnb_colsum_f64(int64_t n_rows, int64_t f, const double* d_g, int64_t ldg, const double* d_y,
                               int64_t ldy, double* d_gm, int64_t ldgm, double* d_out, void* d_ws, size_t ws_bytes,
                               void* stream) {
  return colsum_f64_launch(n_rows, f, d_g, ldg, d_y, ldy, d_gm, ldgm, d_out, d_ws, ws_bytes, (cudaStream_t)stream);
}

extern "C" size_t gcnb_colsum_f64_workspace_bytes(int64_t n_rows, int64_t f) { return colsum_f64_workspace_bytes(n_rows, f); }

extern "C" size_t gcnb_layer_f64_workspace_bytes(const gcnb_graph* g, int64_t fin, int64_t fout) {
  if (!g) return 0;
  const LayerF64Ws r = layer_f64_regions(g, fin, fout);
  return r.s + r.c + r.d + 256;
}

extern "C" int gcnb_layer_forward_f64(const gcnb_graph* g, const double* d_x, int64_t ldx, const double* d_w,
                                      const double* d_bias, int64_t fin, int64_t fout, int flags, const uint8_t* d_mask,
                                      double mask_scale, double* d_support, double* d_out, void* d_ws, size_t ws_bytes,
                                      void* stream) {
  GCNB_TRY(require_f64(g, false, "layer_forward_f64"));
  GCNB_REQUIRE(fin > 0 && fout > 0 && fin < (1ll << 31) && fout < (1ll << 31), "layer_forward_f64: bad feature sizes %lld -> %lld",
               (long long)fin, (long long)fout);
  GCNB_REQUIRE(ldx >= fin, "layer_forward_f64: ldx < in_features");
  GCNB_REQUIRE(d_w != nullptr && d_support != nullptr && d_out != nullptr && (d_x != nullptr || g->n_cols == 0),
               "layer_forward_f64: null operand");
  const size_t need = gcnb_layer_f64_workspace_bytes(g, fin, fout);
  GCNB_REQUIRE(d_ws != nullptr && ws_bytes >= need, "layer_forward_f64: workspace too small (%zu < %zu)", ws_bytes, need);
  const LayerF64Ws r = layer_f64_regions(g, fin, fout);
  cudaStream_t st = (cudaStream_t)stream;
  char* ws = reinterpret_cast<char*>(d_ws);
  const Epilogue64 ep = make_epilogue64(d_bias, (flags & GCNB_LAYER_RELU) != 0, false, d_mask, fout, mask_scale);
  if (flags & GCNB_LAYER_AGG_FIRST) {  // out = (A X) W + bias; d_support receives A X [n_rows, ld2(fin)] for backward
    const int64_t ldax = ld2(fin);
    GCNB_TRY(spmm_f64_graph(g, false, d_x, ldx, fin, Epilogue64(), d_support, ldax, ws, r.s, st));
    return gemm_f64_launch(g->n_rows, fout, fin, d_support, ldax, 1, d_w, fout, 1, d_out, fout, ep, ws + r.s + r.c, r.d, st);
  }
  const int64_t lds = ld2(fout);  // support = X W ; out = A support (+ bias) (relu) (dropout)
  GCNB_TRY(gemm_f64_launch(g->n_cols, fout, fin, d_x, ldx, 1, d_w, fout, 1, d_support, lds, Epilogue64(), ws + r.s + r.c,
                           r.d, st));
  return spmm_f64_graph(g, false, d_support, lds, fout, ep, d_out, fout, ws, r.s, st);
}

extern "C" int gcnb_layer_backward_f64(const gcnb_graph* g, const double* d_x, int64_t ldx, const double* d_w,
                                       const double* d_g, int64_t ldg, const double* d_y, int64_t fin, int64_t fout,
                                       int flags, const uint8_t* d_mask, double mask_scale, double* d_gm, double* d_ds,
                                       double* d_dw, double* d_db, double* d_dx, int64_t lddx, void* d_ws,
                                       size_t ws_bytes, void* stream) {
  GCNB_TRY(require_f64(g, true, "layer_backward_f64"));
  GCNB_REQUIRE(fin > 0 && fout > 0 && fin < (1ll << 31) && fout < (1ll << 31), "layer_backward_f64: bad feature sizes");
  GCNB_REQUIRE(ldg >= fout && (d_g != nullptr || g->n_rows == 0), "layer_backward_f64: null G or ldg < out_features");
  const bool relu = (flags & GCNB_LAYER_RELU) != 0;
  const bool need_dx = (flags & GCNB_LAYER_NEED_DX) != 0;
  const bool need_dw = (flags & GCNB_LAYER_NEED_DW) != 0;
  const bool need_db = (flags & GCNB_LAYER_NEED_DB) != 0;
  const bool agg_first = (flags & GCNB_LAYER_AGG_FIRST) != 0;
  const bool masked = relu || d_mask != nullptr;
  GCNB_REQUIRE(!relu || d_y != nullptr, "layer_backward_f64: relu needs y");
  GCNB_REQUIRE(!masked || d_gm != nullptr, "layer_backward_f64: relu / dropout mask needs gm");
  GCNB_REQUIRE(!need_db || d_db != nullptr, "layer_backward_f64: db requested but null");
  GCNB_REQUIRE(!need_dw || d_dw != nullptr, "layer_backward_f64: dW requested but null");
  GCNB_REQUIRE(!need_dx || (d_dx != nullptr && lddx >= fin), "layer_backward_f64: dX requested but null / lddx < in_features");
  GCNB_REQUIRE(!(need_dw || need_dx) || ((d_x != nullptr || !need_dw) && ldx >= fin && d_w != nullptr),
               "layer_backward_f64: null X / W or ldx < in_features");
  GCNB_REQUIRE(!(agg_first ? need_dx : (need_dx || need_dw)) || d_ds != nullptr, "layer_backward_f64: null ds");
  const size_t need = gcnb_layer_f64_workspace_bytes(g, fin, fout);
  GCNB_REQUIRE(d_ws != nullptr && ws_bytes >= need, "layer_backward_f64: workspace too small (%zu < %zu)", ws_bytes, need);
  const LayerF64Ws r = layer_f64_regions(g, fin, fout);
  cudaStream_t st = (cudaStream_t)stream;
  char* ws = reinterpret_cast<char*>(d_ws);
  void* ws_spmm = ws;
  void* ws_col = ws + r.s;
  void* ws_gemm = ws + r.s + r.c;
  // db = colsum(G); with ReLU / dropout the masked gradient is staged in gm [n_rows, ld2(fout)] and read from there on
  const double* gsrc = d_g;
  int64_t gld = ldg;
  if (masked || need_db) {
    GCNB_TRY(colsum_f64_launch(g->n_rows, fout, d_g, ldg, relu ? d_y : nullptr, fout, masked ? d_gm : nullptr, ld2(fout),
                               need_db ? d_db : nullptr,
                               ws_col, r.c, st, d_mask, fout, mask_scale));
    if (masked) {
      gsrc = d_gm;
      gld = ld2(fout);
    }
  }
  if (!need_dw && !need_dx) return GCNB_OK;
  if (agg_first) {  // d_x = A X [n_rows, ld2(fin)] from the forward: dW = (A X)^T G ; dX = A^T (G W^T)
    if (need_dw)
      GCNB_TRY(gemm_f64_launch(fin, fout, g->n_rows, d_x, 1, ldx, gsrc, gld, 1, d_dw, fout, Epilogue64(), ws_gemm, r.d, st));
    if (need_dx) {
      const int64_t ldt = ld2(fin);
      GCNB_TRY(gemm_f64_launch(g->n_rows, fin, fout, gsrc, gld, 1, d_w, 1, fout, d_ds, ldt, Epilogue64(), ws_gemm, r.d, st));
      GCNB_TRY(spmm_f64_graph(g, true, d_ds, ldt, fin, Epilogue64(), d_dx, lddx, ws_spmm, r.s, st));
    }
    return GCNB_OK;
  }
  const int64_t lds = ld2(fout);  // dS = A^T G ; dW = X^T dS ; dX = dS W^T
  GCNB_TRY(spmm_f64_graph(g, true, gsrc, gld, fout, Epilogue64(), d_ds, lds, ws_spmm, r.s, st));
  if (need_dw)
    GCNB_TRY(gemm_f64_launch(fin, fout, g->n_cols, d_x, 1, ldx, d_ds, lds, 1, d_dw, fout, Epilogue64(), ws_gemm, r.d, st));
  if (need_dx)
    GCNB_TRY(gemm_f64_launch(g->n_cols, fin, fout, d_ds, lds, 1, d_w, 1, fout, d_dx, lddx, Epilogue64(), ws_gemm, r.d, st));
  return GCNB_OK;
}
