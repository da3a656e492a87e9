/*
 * gcnb200.h -- C ABI of libgcnb200.so: the B200 (sm_100a) implementation of the
 * graph-convolution layer hot path of LinChen-65/pygcn.
 *
 * The reference has no FFI of its own: its boundary for this path is the Python class
 * `GraphConvolution` (pygcn/layers.py:7-43) plus `torch.spmm`, and the host-side graph
 * helpers `normalize` / `sparse_mx_to_torch_sparse_tensor` (pygcn/utils.py:390-397,
 * 407-414).  Every entry point below names the reference line(s) it replaces; the Python
 * binding a pygcn maintainer would add is in INTEGRATION.md and shipped in
 * pygcn_b200/_lib.py.
 *
 * Conventions
 *   - every pointer named d_* is a DEVICE pointer on the current CUDA device; the library
 *     never frees or keeps caller memory past the call.
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, nothing
 *     synchronises unless stated ("sync" in the comment).
 *   - return value 0 = ok, otherwise one of GCNB_E_*; gcnb_last_error() returns a
 *     thread-local message for the last failing call on this thread.
 *   - dense matrices are fp32 row-major with an explicit leading dimension in ELEMENTS.
 *   - thread-safe: the only shared mutable state is inside a graph handle and is written
 *     only by the build call that creates it.
 */
#ifndef GCNB200_H_
#define GCNB200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GCNB_VERSION 200

#define GCNB_OK 0
#define GCNB_E_INVALID 1  /* bad argument (shape, null pointer, alignment, overflow)  */
#define GCNB_E_CUDA 2     /* a CUDA runtime call failed; message has the CUDA error    */
#define GCNB_E_NOMEM 3    /* device allocation failed                                  */
#define GCNB_E_UNSUPPORTED 4

typedef struct gcnb_graph gcnb_graph; /* opaque: CSR + CSR^T + row-length-binned schedule */

int gcnb_version(void);
const char* gcnb_last_error(void);
/* Number of kernels this library has launched in the process so far (every launch site counts itself): the
 * difference across one captured step is the step's launch count (bench.py "gpu_launches"). */
long long gcnb_launch_count(void);
/* 0 when the current device is compute capability 10.x (the only target of this build). */
int gcnb_check_device(void);

/* ------------------------------------------------------------------------------------
 * Graph construction.  One-off per adjacency; the handle is reused by every layer call.
 * ---------------------------------------------------------------------------------- */

/* flags for gcnb_graph_from_edges */
#define GCNB_BUILD_SYMMETRIZE 1    /* A <- max(A, A^T)                 pygcn/utils.py:365 */
#define GCNB_BUILD_SELF_LOOPS 2    /* A <- A + I (fp64)                pygcn/utils.py:368 */
#define GCNB_BUILD_ROW_NORMALIZE 4 /* A <- D^-1 A, fp64, inf -> 0      pygcn/utils.py:390-397 */
#define GCNB_BUILD_CORA_PIPELINE 7
#define GCNB_BUILD_KEEP_F64 8      /* also keep the fp64 values (before the cast of utils.py:409): an fp64 handle */

/* Row-length bins of the schedule (deg = stored entries in the row):
 *   0: deg == 0   1: 1..8   2: 9..32   3: 33..1024   4: > 1024 (split across warps)   */
#define GCNB_NUM_BINS 5
#define GCNB_BIN_EDGE_1 1
#define GCNB_BIN_EDGE_2 9
#define GCNB_BIN_EDGE_3 33
#define GCNB_BIN_EDGE_4 1025

/* Edge list -> normalised adjacency, on the device.  Replaces the Cora loader's graph
 * statements pygcn/utils.py:360-368 (duplicate edges summed, symmetrise by element-wise
 * max, + I), `normalize` (utils.py:390-397) and `sparse_mx_to_torch_sparse_tensor`
 * (utils.py:407-414).  Stored entries come out row-major with ascending columns, values
 * rounded fp64 -> fp32 exactly as `.astype(np.float32)` does.  sync. */
int gcnb_graph_from_edges(int64_t n, int64_t n_edges, const int32_t* d_src, const int32_t* d_dst,
                          int flags, void* stream, gcnb_graph** out);

/* torch sparse COO adjacency (int64 indices [2,nnz] given as two rows, fp32 values), any
 * order, duplicates allowed (they stay separate stored entries, which sums them exactly as
 * torch.spmm does for an uncoalesced tensor).  Replaces the per-call coalesce / COO->CSR that
 * `torch.spmm(adj, .)` (pygcn/layers.py:34) performs inside ATen.  sync. */
int gcnb_graph_from_coo(int64_t n_rows, int64_t n_cols, int64_t nnz, const int64_t* d_row,
                        const int64_t* d_col, const float* d_val, void* stream, gcnb_graph** out);

/* torch sparse CSR adjacency (int64 crow [n_rows+1], int64 col [nnz]).  sync. */
int gcnb_graph_from_csr(int64_t n_rows, int64_t n_cols, int64_t nnz, const int64_t* d_crow,
                        const int64_t* d_col, const float* d_val, void* stream, gcnb_graph** out);

/* Dense strided adjacency as the fork's live scripts pass it (pygcn/utils.py:124-132,
 * policy-generator.py:339): non-zeros are scanned into CSR on the device.  sync. */
int gcnb_graph_from_dense(int64_t n_rows, int64_t n_cols, const float* d_a, int64_t lda,
                          void* stream, gcnb_graph** out);

/* fp64 handles.  The same builds on double values: same sort, duplicate handling, transpose and schedule; the
 * handle keeps the fp64 values for the _f64 products below and, as val / t_val, their fp32 rounding (so the fp32
 * entry points, the exports and gcnb_graph_block work on it as on any handle).  A dense fp64 adjacency is scanned into
 * CSR: fp64 handles never take the dense route.  d_val / d_a 8-byte aligned.  sync. */
int gcnb_graph_from_coo_f64(int64_t n_rows, int64_t n_cols, int64_t nnz, const int64_t* d_row,
                            const int64_t* d_col, const double* d_val, void* stream, gcnb_graph** out);
int gcnb_graph_from_csr_f64(int64_t n_rows, int64_t n_cols, int64_t nnz, const int64_t* d_crow,
                            const int64_t* d_col, const double* d_val, void* stream, gcnb_graph** out);
int gcnb_graph_from_dense_f64(int64_t n_rows, int64_t n_cols, const double* d_a, int64_t lda,
                              void* stream, gcnb_graph** out);

void gcnb_graph_free(gcnb_graph* g);

typedef struct {
  int64_t n_rows, n_cols, nnz;
  int64_t bin_rows[GCNB_NUM_BINS]; /* rows per degree bin (forward CSR)            */
  int64_t t_bin_rows[GCNB_NUM_BINS];
  int64_t max_degree, t_max_degree;
  int64_t n_long_chunks, t_n_long_chunks; /* work items the long-row bin was split into */
  int32_t pattern_symmetric;       /* 1: CSR^T shares rowptr/col with CSR (values differ) */
  int32_t dense_route;             /* 1: built from a dense matrix of density >= 10 %: products run as
                                      tcgen05 GEMMs over zero-padded dense copies instead of the CSR */
  int64_t device_bytes;            /* HBM held by the handle                       */
  const int32_t* d_rowptr;         /* [n_rows+1]                                   */
  const int32_t* d_col;            /* [nnz]                                        */
  const float* d_val;              /* [nnz]                                        */
  const int32_t* d_t_rowptr;       /* [n_cols+1]  CSR of A^T                       */
  const int32_t* d_t_col;          /* [nnz]                                        */
  const float* d_t_val;            /* [nnz]                                        */
} gcnb_graph_info;

int gcnb_graph_get_info(const gcnb_graph* g, gcnb_graph_info* info);

/* Write the adjacency in the exact layout `sparse_mx_to_torch_sparse_tensor` returns
 * (pygcn/utils.py:407-414): d_indices int64 [2, nnz] (row 0 = row ids, row 1 = col ids),
 * d_values fp32 [nnz], row-major / columns ascending. */
int gcnb_graph_export_coo(const gcnb_graph* g, int64_t* d_indices, float* d_values, void* stream);

/* Sub-matrix of A (transpose = 0) or of A^T (transpose = 1): rows [r0, r1) x columns [c0, c1) as a
 * new handle with local row ids 0..r1-r0 and column ids shifted by -c0 (+ col_shift).  Used by the
 * 1-D row partition across GPUs (one block per source rank).  n_cols_out >= c1-c0+col_shift is the
 * column count recorded in the new handle.  sync. */
int gcnb_graph_block(const gcnb_graph* g, int transpose, int64_t r0, int64_t r1, int64_t c0, int64_t c1,
                     int64_t col_shift, int64_t n_cols_out, void* stream, gcnb_graph** out);

/* Rows [r0, r1) of A (or A^T) restricted to the columns owned by OTHER ranks, with column ids
 * remapped to the layout of an all-gathered panel of equal-sized (padded) blocks:
 *     col in [bounds[q], bounds[q+1])  ->  q * pad_rows + (col - bounds[q]),   q != exclude_part
 * h_bounds is a HOST array of n_parts+1 row boundaries.  The new handle has n_parts*pad_rows
 * columns.  With exclude_part < 0 no part is excluded (the whole row block, remapped).  sync. */
int gcnb_graph_block_gathered(const gcnb_graph* g, int transpose, int64_t r0, int64_t r1, int n_parts,
                              const int64_t* h_bounds, int64_t pad_rows, int exclude_part, void* stream,
                              gcnb_graph** out);

/* The same remap restricted to the source ranks whose bit is set in include_mask (n_parts <= 64): the
 * column block "sources S" of the row block, for the pipelined peer-memory exchange (one SpMM per
 * group of source ranks, started when their slots have landed).  sync. */
int gcnb_graph_block_sources(const gcnb_graph* g, int transpose, int64_t r0, int64_t r1, int n_parts,
                             const int64_t* h_bounds, int64_t pad_rows, unsigned long long include_mask, void* stream,
                             gcnb_graph** out);

/* Copy the device CSR (transpose = 0) or the CSR of A^T (transpose = 1) into caller
 * buffers: d_rowptr int32 [rows+1], d_col int32 [nnz], d_val fp32 [nnz]. */
int gcnb_graph_export_csr(const gcnb_graph* g, int transpose, int32_t* d_rowptr, int32_t* d_col,
                          float* d_val, void* stream);

/* gcnb_graph_export_csr with the fp64 values; GCNB_E_UNSUPPORTED for a handle that has none. */
int gcnb_graph_export_csr_f64(const gcnb_graph* g, int transpose, int32_t* d_rowptr, int32_t* d_col,
                              double* d_val64, void* stream);

/* ------------------------------------------------------------------------------------
 * Hot path kernels
 * ---------------------------------------------------------------------------------- */

#define GCNB_SPMM_TRANSPOSE 1 /* use A^T (backward of pygcn/layers.py:34)               */
#define GCNB_SPMM_RELU 2      /* fuse the caller's F.relu (pygcn/models.py:49,53,56)    */
#define GCNB_SPMM_ACCUMULATE 4 /* out += A*b before bias/relu (column-blocked multi-GPU SpMM) */

/* out[r, 0:f] = sum_e val[e] * b[col[e], 0:f]  (+ bias[0:f]) (then max(.,0))
 * `torch.spmm(adj, support)` + `output + self.bias` (pygcn/layers.py:34-36).
 * d_bias may be NULL.  b is [n_cols, f] (or [n_rows, f] with TRANSPOSE), ld in elements. */
int gcnb_spmm(const gcnb_graph* g, int flags, const float* d_b, int64_t ldb, int64_t f,
              const float* d_bias, float* d_out, int64_t ldo, void* d_ws, size_t ws_bytes,
              void* stream);
/* scratch for the partial rows of the split long-row bin (0 when the graph has none) */
size_t gcnb_spmm_workspace_bytes(const gcnb_graph* g, int flags, int64_t f);

/* Reduced-precision tier of the same product (BASELINE north_star: "2e-2 when bf16 features are used"): the
 * dense operand is bf16, so a gathered row is half the bytes the kernel is bound by; accumulation, bias, ReLU
 * and the output stay fp32.  d_b is [n_cols, ldb] bf16 with ldb a multiple of 8 and >= 8*ceil(f/8), rows
 * 16-byte aligned (gcnb_to_bf16 produces exactly that).  Not available for handles on the dense route. */
int gcnb_spmm_bf16(const gcnb_graph* g, int flags, const uint16_t* d_b, int64_t ldb, int64_t f,
                   const float* d_bias, float* d_out, int64_t ldo, void* d_ws, size_t ws_bytes, void* stream);
/* d_dst[r, 0:ld_dst] = bf16(d_src[r, 0:f]) round-to-nearest-even, zeros past f (the panel gcnb_spmm_bf16 gathers) */
int gcnb_to_bf16(int64_t n_rows, int64_t f, const float* d_src, int64_t ld_src, uint16_t* d_dst, int64_t ld_dst,
                 void* stream);

#define GCNB_GEMM_FP32 0    /* CUDA-core fp32 FMA (bit-faithful fp32 accumulate)          */
#define GCNB_GEMM_TF32X3 1  /* tcgen05 kind::tf32, 3-term split: fp32-level accuracy      */
#define GCNB_GEMM_AUTO 2    /* TF32X3 when the shape is tensor-core friendly, else FP32   */

/* c[m,n] = sum_k A(i,k) B(k,j) with element (i,k) of A at d_a[i*a_rs + k*a_cs] and (k,j) of
 * B at d_b[k*b_rs + j*b_cs]; c row-major with ldc.  Covers `torch.mm(input, weight)`
 * (pygcn/layers.py:33) and both MmBackward products (dW = X^T dS, dX = dS W^T).
 * d_ws / ws_bytes: scratch for split-K (see gcnb_gemm_workspace_bytes), may be NULL/0 when
 * that returns 0. */
int gcnb_gemm(int64_t m, int64_t n, int64_t k, const float* d_a, int64_t a_rs, int64_t a_cs,
              const float* d_b, int64_t b_rs, int64_t b_cs, float* d_c, int64_t ldc, int precision,
              void* d_ws, size_t ws_bytes, void* stream);
size_t gcnb_gemm_workspace_bytes(int64_t m, int64_t n, int64_t k, int precision);
/* The same product followed by  c = relu?(c + bias[j])  -- `+ self.bias` (pygcn/layers.py:36) and the caller's F.relu
 * (models.py:49) for the aggregate-first order (A X) W + b (GCNB_LAYER_AGG_FIRST), where the dense product comes
 * last.  The TMA-fed tcgen05 kernel applies it in its epilogue; other routes add one in-place pass over c.
 * d_bias may be NULL; workspace as gcnb_gemm. */
int gcnb_gemm_ex(int64_t m, int64_t n, int64_t k, const float* d_a, int64_t a_rs, int64_t a_cs, const float* d_b,
                 int64_t b_rs, int64_t b_cs, float* d_c, int64_t ldc, const float* d_bias, int relu, int precision,
                 void* d_ws, size_t ws_bytes, void* stream);

/* d_out[0:f] = sum_rows g[r, 0:f]  (AddBackward0 of `output + self.bias`, layers.py:36).
 * If d_y != NULL the ReLU mask of the fused epilogue is applied first and the masked
 * gradient is written to d_gm (may alias d_g):  gm = g * [y > 0].  With d_y == NULL and
 * d_gm != NULL, d_gm receives a copy of g (used to stage G into the padded all-gather panel). */
int gcnb_colsum(int64_t n_rows, int64_t f, const float* d_g, int64_t ldg, const float* d_y,
                int64_t ldy, float* d_gm, int64_t ldgm, float* d_out, void* d_ws, size_t ws_bytes,
                void* stream);
size_t gcnb_colsum_workspace_bytes(int64_t n_rows, int64_t f);

/* ------------------------------------------------------------------------------------
 * Layer-level entry points: what GraphConvolution.forward / its autograd backward bind to.
 * ---------------------------------------------------------------------------------- */

#define GCNB_LAYER_RELU 1     /* fused ReLU epilogue + mask in backward */
#define GCNB_LAYER_NEED_DX 2  /* compute dX (ctx.needs_input_grad[0])   */
#define GCNB_LAYER_NEED_DW 4
#define GCNB_LAYER_NEED_DB 8
/* Association order.  The reference computes A (X W) (pygcn/layers.py:33-34).  With this flag the layer computes
 * (A X) W + bias instead -- the same function and gradients to fp32 rounding (tests: <= 1e-5), chosen by the host
 * when in_features < out_features: the SpMM then gathers rows of X (fin wide) instead of rows of X W (fout wide), and
 * backward needs no SpMM for dW = (A X)^T G  (dX = A^T (G W^T), width fin, only when the input requires grad).
 * forward : d_support receives A X [n_rows, ld4(fin)] (keep it for backward); d_x must have 16-byte aligned rows.
 * backward: pass that A X as d_x (ldx = ld4(fin)); d_ds is scratch [n_rows, ld4(fin)] for G W^T (dX only). */
#define GCNB_LAYER_AGG_FIRST 16

/* forward of pygcn/layers.py:32-38:  support = X W ; out = A support (+ bias) (relu) (dropout)
 *   d_x [n_cols, fin] ld ldx ; d_w [fin, fout] contiguous ; d_bias [fout] or NULL
 *   d_mask: NULL, or a keep-mask uint8 [n_rows, fout] applied last in the epilogue together with
 *           mask_scale = 1/(1-p)  (upstream pygcn's F.dropout on the layer output; the fork has it
 *           commented out, pygcn/models.py:50,54)
 *   d_support [n_cols, ld4(fout)] scratch, ld4(f) = 4*ceil(f/4) (rows stay 16-byte aligned)
 *   d_out [n_rows, fout] contiguous ; d_ws: gcnb_layer_workspace_bytes() bytes */
int gcnb_layer_forward(const gcnb_graph* g, const float* d_x, int64_t ldx, const float* d_w,
                       const float* d_bias, int64_t fin, int64_t fout, int flags, int precision,
                       const uint8_t* d_mask, float mask_scale, float* d_support, float* d_out, void* d_ws,
                       size_t ws_bytes, void* stream);

/* backward (SURVEY.md 3.2): db = colsum(G) ; dS = A^T G ; dW = X^T dS ; dX = dS W^T
 *   d_g [n_rows, fout] ld ldg ; d_y = forward output (only read with GCNB_LAYER_RELU)
 *   d_ds [n_cols, ld4(fout)] scratch ; d_gm [n_rows, ld4(fout)] scratch or NULL: when given, G (masked by the ReLU /
 *   dropout mask, or as it is) is staged there with 16-byte aligned rows for the SpMM and the dW product -- required with
 *   RELU or a dropout mask, and what to pass when d_g's rows are not 16-byte aligned (fout % 4 != 0)
 *   d_mask / mask_scale: the same keep-mask the forward used (G is masked before anything else)
 *   d_dw [fin, fout], d_db [fout], d_dx [n_cols, fin] ld lddx: written when requested */
int gcnb_layer_backward(const gcnb_graph* g, const float* d_x, int64_t ldx, const float* d_w,
                        const float* d_g, int64_t ldg, const float* d_y, int64_t fin, int64_t fout,
                        int flags, int precision, const uint8_t* d_mask, float mask_scale, float* d_gm,
                        float* d_ds, float* d_dw,
                        float* d_db, float* d_dx, int64_t lddx, void* d_ws, size_t ws_bytes,
                        void* stream);
size_t gcnb_layer_workspace_bytes(const gcnb_graph* g, int64_t fin, int64_t fout, int precision);

/* ---- fp64 tier: the layer's products, column sums and layer entry points on double operands --------------------
 * What `model.double()` runs in the reference (torch.mm / torch.spmm on fp64).  Each mirrors the fp32 entry point of
 * the same name without the `precision` argument: the SpMM reads the handle's fp64 values (handles built by the _f64
 * constructors or with GCNB_BUILD_KEEP_F64; any other handle is refused with GCNB_E_INVALID), the dense products run on
 * the fp64 tensor cores (DMMA), the column sums add in fp64 in a fixed order.  Every result is bit-reproducible.
 * Operands are 8-byte aligned; panels whose rows are 16-byte aligned (even ld, 16-byte aligned base) are gathered with
 * 16-byte loads, so internal panels use ld2(f) = 2*ceil(f/2).  Workspaces: the matching *_workspace_bytes, 8-byte
 * aligned. */
/* gcnb_spmm with the dropout epilogue: out = dropout(relu(A b (+ out) (+ bias))), d_mask NULL or uint8 [rows, ld_mask] */
int gcnb_spmm_f64(const gcnb_graph* g, int flags, const double* d_b, int64_t ldb, int64_t f, const double* d_bias,
                  const uint8_t* d_mask, int64_t ld_mask, double mask_scale, double* d_out, int64_t ldo, void* d_ws,
                  size_t ws_bytes, void* stream);
size_t gcnb_spmm_f64_workspace_bytes(const gcnb_graph* g, int flags, int64_t f);
int gcnb_gemm_f64(int64_t m, int64_t n, int64_t k, const double* d_a, int64_t a_rs, int64_t a_cs, const double* d_b,
                  int64_t b_rs, int64_t b_cs, double* d_c, int64_t ldc, void* d_ws, size_t ws_bytes, void* stream);
int gcnb_gemm_f64_ex(int64_t m, int64_t n, int64_t k, const double* d_a, int64_t a_rs, int64_t a_cs, const double* d_b,
                     int64_t b_rs, int64_t b_cs, double* d_c, int64_t ldc, const double* d_bias, int relu, void* d_ws,
                     size_t ws_bytes, void* stream);
size_t gcnb_gemm_f64_workspace_bytes(int64_t m, int64_t n, int64_t k);
/* gcnb_colsum in fp64; d_out may be NULL when d_gm is given (only the masked / staged copy is written) */
int gcnb_colsum_f64(int64_t n_rows, int64_t f, const double* d_g, int64_t ldg, const double* d_y, int64_t ldy,
                    double* d_gm, int64_t ldgm, double* d_out, void* d_ws, size_t ws_bytes, void* stream);
size_t gcnb_colsum_f64_workspace_bytes(int64_t n_rows, int64_t f);
/* as gcnb_layer_forward / _backward with ld2 in place of ld4: d_support [n_cols, ld2(fout)] (AGG_FIRST: A X
 * [n_rows, ld2(fin)]), d_gm [n_rows, ld2(fout)] (required with RELU or a dropout mask), d_ds [n_cols, ld2(fout)]
 * (AGG_FIRST: [n_rows, ld2(fin)], dX only) */
int gcnb_layer_forward_f64(const gcnb_graph* g, const double* d_x, int64_t ldx, const double* d_w, const double* d_bias,
                           int64_t fin, int64_t fout, int flags, const uint8_t* d_mask, double mask_scale,
                           double* d_support, double* d_out, void* d_ws, size_t ws_bytes, void* stream);
int gcnb_layer_backward_f64(const gcnb_graph* g, const double* d_x, int64_t ldx, const double* d_w, const double* d_g,
                            int64_t ldg, const double* d_y, int64_t fin, int64_t fout, int flags, const uint8_t* d_mask,
                            double mask_scale, double* d_gm, double* d_ds, double* d_dw, double* d_db, double* d_dx,
                            int64_t lddx, void* d_ws, size_t ws_bytes, void* stream);
size_t gcnb_layer_f64_workspace_bytes(const gcnb_graph* g, int64_t fin, int64_t fout);

/* ---- (ReLU ->) fresh training-mode BatchNorm1d over the layer output (SURVEY.md 8f rank 2) ------------------------
 * Replaces pygcn/models.py:41-45 `GCN.apply_bn` (a NEW nn.BatchNorm1d(F) per call: affine weight 1 / bias 0, batch
 * statistics even under model.eval()) as the models apply it, `apply_bn(F.relu(gc(x, adj)))` (models.py:49,53), and
 * its autograd backward.  relu != 0 folds the caller's F.relu and its backward mask into the same two passes.
 *   forward : a = relu ? max(y, 0) : y;  mean_c, rstd_c = 1 / sqrt(biased var_c + eps) over the n_rows rows;
 *             out = (a - mean) * rstd;  d_mean / d_rstd [f] are kept by the caller for backward.
 *   backward: dy = [relu: y > 0] * rstd * (g - mean_rows(g) - xh * mean_rows(g * xh)), xh recomputed from y;
 *             d_gstat [2 * f] receives the two row means (scratch the caller owns).
 * One statistics pass (fp64 accumulation, per-CTA partials added in fixed order: deterministic) and one apply pass
 * each way.  d_ws: gcnb_fresh_bn_workspace_bytes(n_rows, f) bytes, 8-byte aligned.  Operands fp32 row-major with
 * leading dimensions; float4 path when f, the leading dimensions and the addresses allow it.
 * Written at the end of round 1: compiled, NOT yet run on hardware; not called by any other entry point. */
size_t gcnb_fresh_bn_workspace_bytes(int64_t n_rows, int64_t f);
int gcnb_fresh_bn_forward(int64_t n_rows, int64_t f, const float* d_y, int64_t ldy, int relu, float eps, float* d_out,
                          int64_t ldo, float* d_mean, float* d_rstd, void* d_ws, size_t ws_bytes, void* stream);
int gcnb_fresh_bn_backward(int64_t n_rows, int64_t f, const float* d_y, int64_t ldy, int relu, const float* d_g,
                           int64_t ldg, const float* d_mean, const float* d_rstd, float* d_dy, int64_t lddy,
                           float* d_gstat, void* d_ws, size_t ws_bytes, void* stream);

/* ---- peer-memory exchange for the row-partitioned multi-GPU layer (one process per GPU) ------------
 * The reference has no multi-GPU path (SURVEY.md 8e); these entry points replace the NCCL all-gather
 * of the X.W / G panels with our own push kernel over NVLink peer memory + per-source-rank flags, so
 * the SpMM over the column block of source q can start when slot q has landed.
 *   gcnb_symm_alloc : cudaMalloc + zero + CUDA IPC handle (GCNB_IPC_HANDLE_BYTES bytes, host memory)
 *   gcnb_symm_open  : map a peer's allocation into this process (peer access enabled); close / free
 *   gcnb_peer_epoch_bump : d_epoch[0] += 1, clears the n_peers arrival counters (1 tiny kernel)
 *   gcnb_peer_push  : copies [d_src, d_src+bytes) into peer_dst[k] for k = 0..n_peers-1 in that order with
 *                     P2P stores; per peer it first waits until *local_ack[k] >= epoch-1 (the peer has
 *                     finished reading the previous exchange), and afterwards stores *peer_flag[k] = epoch
 *                     with release semantics at system scope.  Pointer arrays are HOST arrays.
 *   gcnb_peer_wait  : one-thread kernel spinning (bounded, traps on timeout) until *d_flag >= *d_epoch
 *   gcnb_peer_ack   : *peer_ack = *d_epoch (release, system scope), after everything before it on the stream */
#define GCNB_MAX_PEERS 15
#define GCNB_IPC_HANDLE_BYTES 64
int gcnb_symm_alloc(size_t bytes, void** d_ptr, void* handle_out);
int gcnb_symm_open(const void* handle, void** d_ptr);
int gcnb_symm_close(void* d_ptr);
int gcnb_symm_free(void* d_ptr);
int gcnb_peer_epoch_bump(uint32_t* d_epoch, uint32_t* d_counters, int n_peers, void* stream);
int gcnb_peer_push(const void* d_src, size_t bytes, int n_peers, void* const* peer_dst, uint32_t* const* peer_flag,
                   const uint32_t* const* local_ack, const uint32_t* d_epoch, uint32_t* d_counters, int n_ctas,
                   void* stream);
int gcnb_peer_wait(const uint32_t* d_flag, const uint32_t* d_epoch, void* stream);
/* spins until *d_word >= *d_epoch - lag (lag = 1: the peer's ack of the previous exchange) */
int gcnb_peer_wait_lag(const uint32_t* d_word, const uint32_t* d_epoch, uint32_t lag, void* stream);
/* copy-engine transfer to / from mapped peer memory: cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault) */
int gcnb_peer_copy(void* dst, const void* src, size_t bytes, void* stream);
int gcnb_peer_ack(uint32_t* peer_ack, const uint32_t* d_epoch, void* stream);

/* ------------------------------------------------------------------------------------
 * Row-partitioned layer, exchange step (SURVEY.md 8b / 8e; nothing in the reference: it is single-GPU).
 * Needed-rows-only ("halo") exchange of a dense panel over an NCCL communicator the CALLER owns
 * (nccl_comm = an ncclComm_t; from torch: ProcessGroupNCCL._comm_ptr()).  NCCL is bound at run time.
 * gcnb_halo_create : h_send_counts / h_recv_counts [world] rows per peer (0 for the rank itself); d_send_rows the
 *                    local panel row ids to send, grouped by destination rank in rank order (copied);
 *                    h_recv_offsets [world] = first row of source q's rows in the compact panel.
 * gcnb_halo_pack   : d_sendbuf [send rows, f] <- the rows of d_panel (ld ldp) every peer reads, one kernel.
 * gcnb_halo_exchange: one grouped ncclSend / ncclRecv round on `stream`: d_compact [.., f] contiguous receives
 *                    source q's rows at row h_recv_offsets[q].  Both calls are stream-ordered and graph-capturable.
 * ---------------------------------------------------------------------------------- */
typedef struct gcnb_halo gcnb_halo;
int gcnb_halo_create(int rank, int world, const int64_t* h_send_counts, const int32_t* d_send_rows,
                     const int64_t* h_recv_counts, const int64_t* h_recv_offsets, void* stream, gcnb_halo** out);
void gcnb_halo_free(gcnb_halo* h);
int64_t gcnb_halo_send_rows(const gcnb_halo* h);
int64_t gcnb_halo_recv_rows(const gcnb_halo* h);
int gcnb_halo_nccl_available(void); /* 1 when libnccl.so.2 could be bound */
int gcnb_halo_pack(const gcnb_halo* h, const float* d_panel, int64_t ldp, int64_t f, float* d_sendbuf, void* stream);
int gcnb_halo_exchange(const gcnb_halo* h, void* nccl_comm, const float* d_sendbuf, int64_t f, float* d_compact,
                       void* stream);

/* Tuning knobs (process-wide, not thread-safe against concurrent launches; for tests and benchmarks).
 *   GCNB_TUNE_SPMM_KERNEL: 0 auto (default), 1 warp-per-row shuffle kernel, 2 group-per-row kernel,
 *                          3 TMA-staged warp-per-row kernel
 *   GCNB_TUNE_SPMM_GROUP_VARIANT: -1 auto, 0..15 = (gathers in flight, CTAs/SM, warps per CTA, stage entries) of
 *   the group kernel (spmm.cu) */
#define GCNB_TUNE_SPMM_KERNEL 1
#define GCNB_TUNE_SPMM_GROUP_VARIANT 2
/*   GCNB_TUNE_PDL: 0 (default) plain stream order; 1 = the layer's kernels are launched with programmatic
 *   stream serialization (each starts while its predecessor drains and waits on-device before touching its output) */
#define GCNB_TUNE_PDL 3
/*   The streaming SpMM (spmm_stream.cu: entry-balanced items, one warp per 1024 stored entries, L2 eviction hints):
 *   GCNB_TUNE_SPMM_STREAM: 0 off, 1 auto (default: panel rows of >= MIN_ROW_BYTES on graphs without empty rows),
 *                          2 wherever the view is eligible;
 *   GCNB_TUNE_STREAM_HOT_MB: L2 budget (MB, default 48) for the rows of the most referenced columns (evict_last);
 *   GCNB_TUNE_STREAM_HINT: 0 (default) no eviction hints, 1 hot rows evict_last, 2 + the other rows evict_first;
 *   GCNB_TUNE_STREAM_MIN_ROW_BYTES: auto threshold (default 256);  GCNB_TUNE_STREAM_BATCH: 0 auto, 2 / 4 / 8 gathered rows
 *   in flight per lane.  Environment: GCNB_SPMM_STREAM, GCNB_L2_HOT_MB, GCNB_STREAM_HINT, GCNB_STREAM_MIN_ROW_BYTES,
 *   GCNB_STREAM_BATCH. */
#define GCNB_TUNE_SPMM_STREAM 4
#define GCNB_TUNE_STREAM_HOT_MB 5
#define GCNB_TUNE_STREAM_HINT 6
#define GCNB_TUNE_STREAM_MIN_ROW_BYTES 7
#define GCNB_TUNE_STREAM_BATCH 8
int gcnb_set_tuning(int key, int value);

/* L2 flush helper for benchmarks: writes `bytes` of d_buf. */
int gcnb_l2_flush(void* d_buf, size_t bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GCNB200_H_ */
