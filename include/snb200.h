/*
 * snb200.h -- C ABI of libsnb200.so, the B200 (sm_100a) implementation of the structured-layer
 * hot path of MatthiasKi/structurednets.
 *
 * The reference has no FFI: its "operator interface" for this path is the forward()/autograd
 * backward of the nn.Modules in structurednets/layers/ (one .py per layer).  Each pair of entry points below
 * replaces one of those (file:line cited per function).  A maintainer of the reference binds them
 * with ctypes (see INTEGRATION.md for the stub).
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless its name ends in
 *     _host; the library owns no memory, allocates nothing and never synchronises the device;
 *   - every kernel is enqueued on `stream` (a cudaStream_t passed as void*);
 *   - return value 0 = ok, non-zero = error, message in sn_last_error_string() (thread local);
 *   - matrices are row-major; "ld" arguments are row strides in elements;
 *   - gradients are ACCUMULATED (+=) into grad buffers, like torch autograd does;
 *   - an empty batch (B == 0) is a no-op that returns 0: every entry that takes a batch size checks its plan and parameter
 *     arguments, then returns before it looks at any batch buffer (features, outputs, their gradients, activations and scratch
 *     sized by B), which may then be NULL or point anywhere.  Nothing is written, accumulated gradients included.
 */
#ifndef SNB200_H
#define SNB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* sn_stream_t; /* cudaStream_t */

#define SN_VERSION 100

int sn_version(void);
const char* sn_last_error_string(void);
/* number of kernels this library has launched since load / last reset (bench.py's gpu_launches) */
long long sn_launch_count(void);
void sn_reset_launch_count(void);
/* optional per-kernel timing with CUDA events on the launching stream: enable, run, synchronise the device, then read
 * "name count total_ms\n" lines (returns the length of the full report) */
void sn_timing_enable(int on);
int sn_timing_report(char* buf, int cap);

/* ------------------------------------------------------------------------------------------
 * SSS layer -- replaces SSSLayer.forward (layers/sss_layer.py:99-131) and its autograd backward.
 *
 * One stage descriptor per (direction, processing step).  Direction 0 = causal sweep (stages
 * 0..n-1), direction 1 = anticausal sweep (stages n-1..0); entry [dir*n + kk] describes the
 * kk-th stage that direction visits.  "state in" / "state out" are the state vectors entering /
 * leaving the stage in processing order.  Offsets off_* index the flat parameter buffer (floats):
 *   off_ys: (out_dim x d_in)   C_k  (causal)  or G_k (anticausal)
 *   off_yu: (out_dim x in_dim) D_k  (causal)  or -1  (anticausal: y_k does not see u_k)
 *   off_ss: (d_out x d_in)     A_k  (causal)  or E_k (anticausal)
 *   off_su: (d_out x in_dim)   B_k  (causal)  or F_k (anticausal)
 * ------------------------------------------------------------------------------------------ */
typedef struct sn_sss_stage {
    int32_t in_off, in_dim, out_off, out_dim;
    int32_t d_in, d_out;
    int32_t off_ys, off_yu, off_ss, off_su;
    int32_t pack_off; /* offset (floats) of this stage's block in the packed buffer */
    int32_t k;        /* natural stage index */
    int32_t reserved[4];
} sn_sss_stage;

/* A contiguous run of processing steps [kk_begin, kk_end) handled as one unit (state checkpoint
 * at kk_begin).  Chunks never straddle first_visit -> second_visit. */
typedef struct sn_sss_chunk {
    int32_t kk_begin, kk_end;
    int32_t col0, ncols;   /* input columns covered by the chunk  */
    int32_t row0, nrows;   /* output columns covered by the chunk */
    int32_t second_visit;  /* 1: the other direction already wrote y for these stages */
    int32_t kk_mid;        /* the forward stages its input columns in two halves: [kk_begin,kk_mid) and [kk_mid,kk_end) */
    int32_t col0_a, ncols_a, col0_b, ncols_b; /* input columns of the two halves */
    int32_t reserved[4];
} sn_sss_chunk;

typedef struct sn_sss_plan {
    int32_t nb_states, input_dim, output_dim;
    int32_t rows_pad, k_pad, d_pad; /* multiples of 4: max rows (out_dim+d_out), max K (d_in+in_dim), max state dim */
    int32_t nchunks;                /* per direction */
    int32_t chunk_in_max, chunk_out_max, chunk_len_max;
    int32_t nparams;                /* floats in the flat parameter buffer */
    int32_t half_in_max;            /* max input columns of a half chunk */
    const sn_sss_stage* stages; /* device, [2][nb_states] */
    const sn_sss_chunk* chunks; /* device, [2][nchunks]   */
} sn_sss_plan;

/* floats needed for the packed parameter copy / for the state checkpoints of a batch of B samples */
size_t sn_sss_packed_floats(const sn_sss_plan* plan_host);
size_t sn_sss_ckpt_floats(const sn_sss_plan* plan_host, int64_t B);
/* re-lays the flat parameters out per stage (transposed + row-major, zero padded); call once per
 * parameter update, before forward/backward */
int sn_sss_pack(const sn_sss_plan* plan_host, const float* params, float* packed, sn_stream_t stream);
/* y[B x output_dim] = SSS(x[B x input_dim]) + bias.  bias may be NULL.  ckpt may be NULL (inference);
 * otherwise it receives the chunk-entry states backward() needs. */
int sn_sss_forward(const sn_sss_plan* plan_host, const float* packed, const float* x, int64_t ldx,
                   float* y, int64_t ldy, const float* bias, float* ckpt, int64_t B, sn_stream_t stream);
/* grad_params (flat, same layout as params) += d loss / d params ; grad_bias (may be NULL) += column
 * sums of grad_y.  grad_x (may be NULL; row stride ldgx >= input_dim) receives d loss / d x (overwritten,
 * bitwise reproducible).  workspace: scratch of sn_sss_backward_workspace_floats() floats (packed per-stage
 * gradient accumulators).  grad_params may be NULL when grad_x is not (input gradient only, e.g. frozen
 * parameters); workspace may then be NULL too.  grad_params and grad_x both NULL is an error. */
size_t sn_sss_backward_workspace_floats(const sn_sss_plan* plan_host);
int sn_sss_backward(const sn_sss_plan* plan_host, const float* packed, const float* x, int64_t ldx,
                    const float* grad_y, int64_t ldgy, const float* ckpt, float* workspace, float* grad_params,
                    float* grad_bias, float* grad_x, int64_t ldgx, int64_t B, sn_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * SSS layer, tensor-core path (tcgen05 / TMEM / TMA, 3xTF32 = fp32-accurate) -- same contract as sn_sss_forward /
 * sn_sss_backward (layers/sss_layer.py:99-131 and its autograd backward), for layers whose stages have state
 * dimensions <= 16, <= 16 outputs and <= 160 inputs each, with input_dim and output_dim multiples of 4.
 * The stages are grouped into chunks of consecutive stages (<= 32 outputs, <= 160 inputs, <= 16 stages); the chunk
 * matrices are rebuilt from the flat parameters by sn_sss_tc_build (call once per parameter update).
 * `stages` is the same device table as sn_sss_plan.stages.  coef must be zero-initialised once by the caller
 * (padding entries are never written).  coef is owned by the caller and shared by the three calls: sn_sss_tc_build writes the
 * chunk matrices and the states of their construction, sn_sss_tc_forward adds the scans' coefficient tiles (packed on an auxiliary
 * stream beside its first GEMM), sn_sss_tc_backward reads all of them -- so a backward must see the coef (and params) of its own
 * forward: call build + forward again after a parameter update before calling backward.
 * Kernels: chunk-matrix construction and its backward, chunk scans: warp-level tensor cores (mma.sync tf32); the two batch GEMMs and
 * the optional chain-scan kernels: tcgen05 / TMEM / TMA.
 * ------------------------------------------------------------------------------------------ */
#define SN_SSS_TC_DS 16
#define SN_SSS_TC_PO 32
#define SN_SSS_TC_KB_MAX 5
#define SN_SSS_TC_LMAX 16
typedef struct sn_sss_tc_chunk {
    int32_t k_begin, k_end; /* natural stages [k_begin, k_end) */
    int32_t col0, ncols;    /* input columns  */
    int32_t row0, nrows;    /* output columns */
    int32_t nkb;            /* ceil(ncols / 32) */
    int32_t reserved;
} sn_sss_tc_chunk;
typedef struct sn_sss_tc_plan {
    int32_t nb_states, input_dim, output_dim, nchunks;
    int32_t rows_aligned; /* 1: every chunk's row0 is a multiple of 4 (16-byte y / grad_y accesses) */
    int32_t chunk_param_floats; /* largest number of parameters (floats) of one direction of one chunk; <= 40960 */
    int32_t reserved[2];        /* reserved[0] = 1: in the flat parameter buffer the entries of each of the lists A..G for consecutive
                                   stages are adjacent (the layout FlatParamsMixin produces): a chunk's parameters are 4 contiguous ranges */
    const sn_sss_stage* stages;    /* device, [2][nb_states] */
    const sn_sss_tc_chunk* chunks; /* device, [nchunks] */
} sn_sss_tc_plan;
size_t sn_sss_tc_coef_floats(const sn_sss_tc_plan* plan_host);
size_t sn_sss_tc_rbuf_floats(const sn_sss_tc_plan* plan_host, int64_t B);   /* forward scratch */
size_t sn_sss_tc_states_floats(const sn_sss_tc_plan* plan_host, int64_t B); /* chunk-boundary states kept for backward */
size_t sn_sss_tc_backward_workspace_floats(const sn_sss_tc_plan* plan_host, int64_t B);
int sn_sss_tc_build(const sn_sss_tc_plan* plan_host, const float* params, float* coef, sn_stream_t stream);
int sn_sss_tc_forward(const sn_sss_tc_plan* plan_host, const float* coef, const float* x, int64_t ldx, float* y, int64_t ldy,
                      const float* bias, float* rbuf, float* states, int64_t B, sn_stream_t stream);
int sn_sss_tc_backward(const sn_sss_tc_plan* plan_host, const float* params, const float* coef, const float* x, int64_t ldx,
                       const float* grad_y, int64_t ldgy, const float* states, float* workspace, float* grad_params, float* grad_bias,
                       float* grad_x /* nullable: gradient w.r.t. the input features, (B x input_dim), written */, int64_t ldgx,
                       int64_t B, sn_stream_t stream);
/* sn_sss_tc_backward: grad_params may be NULL when grad_x is not (input gradient only: the scans and the grad_x products run, the
 * parameter-gradient kernels do not; grad_bias is still accumulated when given).  Both NULL is an error.  workspace is always needed. */

/* ------------------------------------------------------------------------------------------
 * Low-rank layer, fp32 path -- replaces LRLayer.forward (layers/lr_layer.py:38-46) and its backward.
 *   left (out_dim x rank), right (rank x in_dim), hidden (B x rank, written by forward, read by backward),
 *   grad_hidden_ws: scratch (B x rank).  grad_left / grad_right / grad_bias are accumulated; grad_x may be NULL.
 * ------------------------------------------------------------------------------------------ */
int sn_lr_forward_f32(const float* x, int64_t ldx, const float* left, const float* right, const float* bias, float* hidden,
                      float* y, int64_t ldy, int64_t B, int in_dim, int out_dim, int rank, sn_stream_t stream);
int sn_lr_backward_f32(const float* x, int64_t ldx, const float* grad_y, int64_t ldgy, const float* left, const float* right,
                       const float* hidden, float* grad_hidden_ws, float* grad_left, float* grad_right, float* grad_bias,
                       float* grad_x, int64_t ldgx, int64_t B, int in_dim, int out_dim, int rank, sn_stream_t stream);

/* Low-rank layer, bf16 tensor-core path (tcgen05 / TMEM / TMA; BASELINE config C2).  All bf16 matrices are row-major
 * with 16-byte aligned rows (row pitch multiple of 8 elements).  sn_lr_tc_cast_params makes the bf16 copies
 * L (out x rank), L^T (rank x lt_ld) and R (rank x in) of the fp32 master parameters.  Backward scratch (bf16):
 * ghid (B x rank); gyt (out x ldt) and ht (rank x ldt), needed only with grad_left; ght (rank x ldt) and xt (in x ldt), needed
 * only with grad_right; ldt = B rounded up to 8;
 * grad_left / grad_right / grad_bias are fp32, accumulated, and each may be NULL.  grad_x (nullable, bf16, B x in, row
 * pitch ldgx >= in_dim and a multiple of 8) = ghid R, written, bitwise reproducible (no split-K); it needs right_bf16 (the
 * R of sn_lr_tc_cast_params) and right_t, scratch for R^T (in x rank); both may be NULL when grad_x is. */
int sn_lr_tc_cast_params(const float* left, const float* right, void* left_bf16, void* left_t_bf16, int64_t lt_ld, void* right_bf16,
                         int in_dim, int out_dim, int rank, sn_stream_t stream);
int sn_lr_tc_forward(const void* x, int64_t ldx, const void* left_bf16, const void* right_bf16, const float* bias, void* hidden, void* y,
                     int64_t ldy, int64_t B, int in_dim, int out_dim, int rank, sn_stream_t stream);
int sn_lr_tc_backward(const void* x, int64_t ldx, const void* grad_y, int64_t ldgy, const void* left_t_bf16, int64_t lt_ld,
                      const void* right_bf16, const void* hidden, void* ghid, void* gyt, void* ht, void* ght, void* xt, int64_t ldt,
                      void* right_t, float* grad_left, float* grad_right, float* grad_bias, void* grad_x, int64_t ldgx, int64_t B,
                      int in_dim, int out_dim, int rank, sn_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * H-matrix layer -- replaces HMatLayer.forward (layers/hmat_layer.py:34-49) and its backward.
 *   leaves: device table, 8 int32 per leaf {row_start, rows, col_start, cols, rank, off_left, off_right, 0};
 *   params: flat buffer holding left_lr (rows x rank) / right_lr (rank x cols) of every leaf at those offsets;
 *   grad_params has the same layout (accumulated).  sn_hmat_backward: grad_x (nullable; row pitch ldgx >= in_dim) = grad_y W,
 *   written; its leaves add through shared-memory atomics, so it agrees with other summation orders to rounding, not bitwise.
 *   grad_params may be NULL when grad_x is not (input gradient only: the leaf-gradient kernel does not run; grad_bias is still
 *   accumulated when given).  Both NULL is an error.
 * ------------------------------------------------------------------------------------------ */
int sn_hmat_forward(const int32_t* leaves, int nleaves, const float* params, const float* x, int64_t ldx, float* y, int64_t ldy,
                    const float* bias, int64_t B, int in_dim, int out_dim, sn_stream_t stream);
int sn_hmat_backward(const int32_t* leaves, int nleaves, const float* params, const float* x, int64_t ldx, const float* grad_y,
                     int64_t ldgy, float* grad_params, float* grad_bias, float* grad_x, int64_t ldgx, int64_t B, int in_dim, int out_dim,
                     sn_stream_t stream);
/* Dense-block path (default for layers whose dense matrix fits): W = the H-matrix as a dense (out_dim x in_dim) matrix built from
 * the leaves (max_rows = the tallest leaf), applied / differentiated with sn_dense_apply / sn_dense_weight_grad on the tensor cores,
 * and the dense gradient projected back onto the leaf factors (accumulated into grad_params). */
int sn_hmat_build_dense(const int32_t* leaves, int nleaves, int max_rows, const int32_t* slabs /* nullable: work list, see below */, int nslabs,
                        const float* params, float* W, int out_dim, int in_dim, sn_stream_t stream);
int sn_hmat_project_grad(const int32_t* leaves, int nleaves, const int32_t* slabs /* (leaf, first row) per 32 rows of every leaf */, int nslabs,
                         const float* params, const float* dW, int out_dim, int in_dim, float* grad_params, sn_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * PSM layer -- replaces PSMLayer.forward / forward_sparse (layers/psm_layer.py:36-60) and its backward,
 * with the intended factor order W = S_0 S_1 ... S_{n-1} (see csrc/psm.cu).  factors_host: host array of nf
 * descriptors; every pointer inside is a device pointer.  The static pattern is given twice in sliced-ELL form
 * (for S: `fwd`, for S^T: `tr`): rows sorted by length, slices of 32 rows, entry j of a slice's 32 rows contiguous.
 * `src` maps a packed entry to its index in the parameter's own COO value array (-1 = padding).  val_fwd / val_tr
 * ([fwd.total] / [tr.total]) and grad_packed ([fwd.total]) are scratch owned by the caller; grad_vals is COO-ordered
 * and accumulated.  Dimensions up to 65535 (column indices are 16 bit).
 * ------------------------------------------------------------------------------------------ */
typedef struct sn_psm_ell {
    int32_t nslices, total;        /* total = padded entry count = slice_off[nslices] */
    const int32_t* rowmap;         /* [nslices * 32] natural row of position p (-1: none) */
    const int32_t* slice_off;      /* [nslices + 1], multiples of 32 */
    const uint16_t* col;           /* [total] */
    const int32_t* src;            /* [total] */
} sn_psm_ell;
typedef struct sn_psm_factor {
    int32_t rows, cols, nnz, reserved;
    sn_psm_ell fwd, tr;
    const float* vals;
    float* grad_vals;
    float *val_fwd, *val_tr, *grad_packed;
} sn_psm_factor;
/* acts (nullable): sn_psm_acts_floats floats; the forward keeps the input of every factor but the last there ([B][cols_k] row-major,
 * factor 0 first) and the backward reads them instead of recomputing them from x.
 * sn_psm_backward: grad_x (nullable; row pitch ldgx >= in_dim) = grad_y S_0 .. S_{n-1}, written, bitwise reproducible.  The factor
 * gradient buffers (grad_vals, grad_packed of every factor) are all set or all NULL; all NULL is allowed only when grad_x is set
 * (input gradient only, e.g. frozen factors: the forward kernel runs on the transposed chain and acts is not read; grad_bias is
 * still accumulated when given).  val_tr is needed in both modes. */
size_t sn_psm_acts_floats(const sn_psm_factor* factors_host, int nf, int64_t B);
int sn_psm_forward(const sn_psm_factor* factors_host, int nf, const float* x, int64_t ldx, float* y, int64_t ldy, const float* bias,
                   float* acts, int64_t B, int in_dim, int out_dim, sn_stream_t stream);
int sn_psm_backward(const sn_psm_factor* factors_host, int nf, const float* x, int64_t ldx, const float* grad_y, int64_t ldgy,
                    const float* acts, float* grad_bias, float* grad_x, int64_t ldgx, int64_t B, int in_dim, int out_dim,
                    sn_stream_t stream);

/* Dense-product path of the PSM layer for large batches (csrc/psm.cu): the batch-independent product W = S_0 .. S_{n-1} is
 * multiplied out once per call (transposed prefix products, kept in `prefix` for the backward), applied / differentiated on the
 * tensor cores, and the dense gradient is projected back onto every factor's pattern.  The reference's default forward also
 * multiplies the densified factors with dense GEMMs (layers/psm_layer.py:47-60).  csr_* / csc_*: the pattern by rows / by
 * columns (ptr [rows + 1] / [cols + 1], idx = column / row index, src = index into the parameter's COO value array);
 * coo_row / coo_col: the COO indices as int32.  output_dim must be a multiple of 4. */
typedef struct sn_psm_dense_factor {
    int32_t rows, cols, nnz, reserved;
    const int32_t *csr_ptr, *csr_idx, *csr_src;
    const int32_t *csc_ptr, *csc_idx, *csc_src;
    const int32_t *coo_row, *coo_col;
    const float* vals;
    float* grad_vals;
} sn_psm_dense_factor;
size_t sn_psm_dense_prefix_floats(const sn_psm_dense_factor* factors_host, int nf, int out_dim);
size_t sn_psm_dense_backward_floats(const sn_psm_dense_factor* factors_host, int nf, int out_dim);
int sn_psm_dense_forward(const sn_psm_dense_factor* factors_host, int nf, const float* x, int64_t ldx, float* y, int64_t ldy,
                         const float* bias, float* prefix, int64_t B, int in_dim, int out_dim, sn_stream_t stream);
int sn_psm_dense_backward(const sn_psm_dense_factor* factors_host, int nf, const float* x, int64_t ldx, const float* grad_y,
                          int64_t ldgy, const float* prefix, float* work, float* grad_bias, int64_t B, int in_dim, int out_dim,
                          sn_stream_t stream);
/* grad_x = grad_y W (gradient w.r.t. the input features) from the product kept in `prefix` by sn_psm_dense_forward */
int sn_psm_dense_input_grad(const sn_psm_dense_factor* factors, int nf, const float* prefix, const float* grad_y, int64_t ldgy,
                            float* grad_x, int64_t ldgx, int64_t B, int in_dim, int out_dim, sn_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * LDR layer -- replaces build_weight_matrix_torch (approximators/ldr_approximator.py:29-39) + the matmul of
 * LDRLayer.forward (layers/ldr_layer.py:54-58) and their backward.  A, B: COO value arrays (float64) with a slot
 * map per entry into the banded layout {lo[n] | di[n] | up[n] | corner(0,n-1), corner(n-1,0)}; G, H: n x r float64.
 * The Krylov blocks KA_j = A^j G, KB_j = (B^T)^j H are built by recurrence (one kernel, float64) for j < max_terms, and
 * W = [KA_0 | KA_1 | ..][KB_0 | KB_1 | ..]^T is one tensor-core contraction whose length (the number of powers that matter,
 * found on the device) travels through `status` (device int[4]: {powers used, K, converged, max_terms}).  Nothing here
 * synchronises the stream; the caller reads `status` when it wants to know whether max_terms was enough.
 * The workspace (sn_ldr_workspace_bytes) keeps what sn_ldr_backward needs.  n must be a multiple of 4 and <= 4096.
 * ------------------------------------------------------------------------------------------ */
size_t sn_ldr_workspace_bytes(int n, int r, int max_terms);
int sn_ldr_build_weight(int n, int r, const double* A_vals, const int32_t* A_slot, int A_nnz, const double* B_vals,
                        const int32_t* B_slot, int B_nnz, const double* G, const double* H, void* workspace, int max_terms,
                        double rel_tol, float* W_out, int* status_dev, sn_stream_t stream);
int sn_ldr_backward(int n, int r, const float* dW, const int32_t* A_slot, int A_nnz, const int32_t* B_slot, int B_nnz,
                    void* workspace, int max_terms, const int* status_dev, double* gA_vals, double* gB_vals, double* gG,
                    double* gH, sn_stream_t stream);
/* y = x W^T + bias and dW += grad_y^T x (grad_bias += column sums): the dense apply shared by LDR and TL */
int sn_dense_apply(const float* W, int n_out, int n_in, const float* x, int64_t ldx, float* y, int64_t ldy, const float* bias,
                   int64_t B, sn_stream_t stream);
/* grad_x = grad_y W: gradient w.r.t. the input features for every layer that materialises its weight matrix */
int sn_dense_input_grad(const float* W, int n_out, int n_in, const float* grad_y, int64_t ldgy, float* grad_x, int64_t ldgx,
                        int64_t B, sn_stream_t stream);
int sn_dense_weight_grad(const float* x, int64_t ldx, const float* grad_y, int64_t ldgy, float* dW, int n_out, int n_in,
                         float* grad_bias, int64_t B, sn_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * bf16 features on the dense-product layers (PSM dense path, H-matrix dense-block path, LDR, TL), csrc/dense_bf16.cu:
 * W is still built in fp32 from the layer's parameters; these entries run the batch GEMMs on bf16 tensor cores (fp32
 * accumulation in TMEM).  x, grad_y, y, grad_x and the W copies are bf16 ("void*"), dW and the gradients fp32.  Every bf16
 * operand needs a 16-byte aligned base and a row pitch that is a multiple of 8 elements.
 *   sn_dense_cast_bf16: Mb = bf16(M) [rows][ldmb] and / or Mtb = bf16(M)^T [cols][ldmtb] (either nullable) in one pass over
 *     the fp32 M [rows][cols]; pad columns are zeroed.
 *   sn_dense_apply_bf16: y = x W^T + bias (bf16 store); Wb = W bf16 [n_out][ldwb].
 *   sn_dense_weight_grad_bf16: dW [n_out][lddw] += grad_y^T x in fp32 (split-K over the batch, fp32 reductions),
 *     grad_bias += column sums of grad_y.
 *   sn_dense_input_grad_bf16: grad_x = grad_y W (bf16 store); Wtb = W^T bf16 [n_in][ldwtb].
 * ------------------------------------------------------------------------------------------ */
int sn_dense_cast_bf16(const float* M, int rows, int cols, void* Mb, int64_t ldmb, void* Mtb, int64_t ldmtb, sn_stream_t stream);
int sn_dense_apply_bf16(const void* Wb, int64_t ldwb, int n_out, int n_in, const void* x, int64_t ldx, void* y, int64_t ldy,
                        const float* bias, int64_t B, sn_stream_t stream);
int sn_dense_weight_grad_bf16(const void* x, int64_t ldx, const void* grad_y, int64_t ldgy, float* dW, int64_t lddw, int n_out,
                              int n_in, float* grad_bias, int64_t B, sn_stream_t stream);
int sn_dense_input_grad_bf16(const void* Wtb, int64_t ldwtb, int n_out, int n_in, const void* grad_y, int64_t ldgy, void* grad_x,
                             int64_t ldgx, int64_t B, sn_stream_t stream);
/* PSM dense-product path with bf16 features: the prefix products and the projection of sn_psm_dense_forward / _backward, the
 * batch GEMMs above.  wb = W bf16 [out_dim][ldwb] and wtb = W^T bf16 [in_dim][ldwtb] (nullable) are written by the forward;
 * grad_x = sn_dense_input_grad_bf16(wtb, ...). */
int sn_psm_dense_forward_bf16(const sn_psm_dense_factor* factors_host, int nf, const void* x, int64_t ldx, void* y, int64_t ldy,
                              const float* bias, float* prefix, void* wb, int64_t ldwb, void* wtb, int64_t ldwtb, int64_t B,
                              int in_dim, int out_dim, sn_stream_t stream);
int sn_psm_dense_backward_bf16(const sn_psm_dense_factor* factors_host, int nf, const void* x, int64_t ldx, const void* grad_y,
                               int64_t ldgy, const float* prefix, float* work, float* grad_bias, int64_t B, int in_dim, int out_dim,
                               sn_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Toeplitz-like layer -- replaces the weight construction of TLLayer.forward (layers/tl_layer.py:11-18,59) and
 * its backward.  G (n x r), H (r x n) float32; K1 (n x rn) and K2 (rn x n) are scratch kept for the backward.
 * ------------------------------------------------------------------------------------------ */
int sn_tl_build_weight(int n, int r, const float* G, const float* H, float* K1, float* K2, float* W, sn_stream_t stream);
int sn_tl_backward(int n, int r, const float* dW, const float* K1, const float* K2, float* dK1, float* dK2, float* gG, float* gH,
                   sn_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Training-loop call sites (reference training_helpers.py:57-73, 139-153): fused loss + accuracy + logit gradient, and optimizer
 * steps over a layer's flat parameter / gradient buffers (csrc/train.cu).  loss_sum / correct are accumulated into.
 * ------------------------------------------------------------------------------------------ */
int sn_ce_loss(const float* logits, int64_t ld, const int64_t* targets, int64_t B, int C, float* loss_sum, int* correct,
               float* grad_logits /* nullable */, int64_t ldg, sn_stream_t stream);
int sn_mse_loss(const float* x, int64_t ld, const float* target, int64_t ldt, int64_t B, int C, float* loss_sum, int* correct,
                float* grad_x /* nullable */, int64_t ldg, sn_stream_t stream);
int sn_flat_sgd(float* params, const float* grads, int64_t n, float lr, float grad_scale, sn_stream_t stream);
int sn_flat_adam(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float beta1, float beta2,
                 float eps, float grad_scale, int* step_dev /* nullable */, int step_host, sn_stream_t stream);

/* ---- the path's only exchange step (SURVEY.md section 8e): one-shot all-reduce of the flat gradient buffer over NVLink peer memory.
 * The reference has no multi-GPU code (F6); this replaces torch.distributed.all_reduce(flat_grad) in the data-parallel step.
 * Every rank allocates one region (cudaMalloc), exports its 64-byte CUDA IPC handle, imports its peers' and then calls
 * sn_allreduce_oneshot_f32 once per step with the same n (<= capacity): data <- scale * sum over ranks, bit-identical on every rank.
 * regions: host array of `world` device pointers, regions[rank] = the own region.  Graph-capturable (epochs live in device memory). */
size_t sn_p2p_region_bytes(int64_t capacity_floats, int world);
int sn_p2p_alloc(void** region, int64_t capacity_floats, int world);
int sn_p2p_free(void* region);
int sn_p2p_export(const void* region, unsigned char* handle64);
int sn_p2p_import(const unsigned char* handle64, void** region);
int sn_p2p_close(void* region);
int sn_allreduce_oneshot_f32(float* data, int64_t n, void* const* regions, int rank, int world, int64_t capacity_floats, float scale,
                             sn_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* SNB200_H */
