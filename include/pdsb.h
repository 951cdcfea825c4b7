/*
 * pdsb.h — C ABI of the B200-native linear-regression engine (libpds_b200).
 *
 * This is the drop-in boundary for ONE hot path of abstractqqq/polars_ds_extension: the
 * lin_reg expression family.  Plain pointers and sizes only; no torch / C++ types.
 * Every entry point cites the reference interface it replaces (paths under /root/reference).
 *
 * Three layers, bottom-up:
 *   (1) device layer  pdsb_dev_*  : device pointers + a cudaStream_t (passed as void*).  This is what
 *       the roofline timing, ncu and the torch-allocated tests call, and what a Rust host that keeps
 *       frames resident on the GPU would bind.
 *   (2) host layer    pdsb_host_* : host (Arrow-buffer) pointers in, host buffers out; does the
 *       H2D packing, the device pipeline and the D2H.  This is the `extern "C"` shim the reference's
 *       `#[polars_expr] fn pl_lr*` bodies (src/num_ext/linear_regression.rs:419-1283) would call instead of
 *       `series_to_mat_for_lr` + `faer_*`.
 *   (3) plugin layer  _polars_plugin_pl_lr* : declared in polars_plugin_abi.h; the symbols Polars itself
 *       dlopen()s, so the .so replaces the reference cdylib for this path without any Rust.
 *
 * All functions return 0 on success, non-zero on error; pdsb_last_error() gives the message
 * (thread-local, NUL-terminated; same strings as the reference's PolarsError::ComputeError texts).
 */
#ifndef PDSB_H
#define PDSB_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PDSB_VERSION 0x000100 /* 0.1.0 */

/* ---- dtypes of an incoming Arrow primitive column (format chars of the Arrow C data interface) ---- */
enum pdsb_dtype {
  PDSB_F32 = 0, PDSB_F64 = 1, PDSB_I8 = 2, PDSB_U8 = 3, PDSB_I16 = 4, PDSB_U16 = 5,
  PDSB_I32 = 6, PDSB_U32 = 7, PDSB_I64 = 8, PDSB_U64 = 9, PDSB_BOOL = 10
};

/* solver strings of the reference: src/linear/lr/mod.rs:18-27 ("qr" | "svd" | "choleskey", else qr) */
enum pdsb_solver { PDSB_SOLVER_QR = 0, PDSB_SOLVER_SVD = 1, PDSB_SOLVER_CHOLESKEY = 2 };

/* what to do on the (p+bias)x(p+bias) normal equations; mirrors the dispatch at linear_regression.rs:436-498 */
enum pdsb_method {
  PDSB_METHOD_LSTSQ = 0, /* OLS / ridge: faer_solve_lr / faer_solve_lr_gated  (lr_solvers.rs:299-382) */
  PDSB_METHOD_CD    = 1, /* lasso / elastic net / positive ridge: faer_coordinate_descent (:426-538)   */
  PDSB_METHOD_NNLS  = 2, /* faer_nn_lr (:542-600)                                                      */
  PDSB_METHOD_RCOND = 3, /* faer_solve_lr_rcond (:216-258)                                             */
  PDSB_METHOD_INV   = 4  /* explicit inverse + solve: faer_qr_lr_with_inv (lr_online_solvers.rs:120-143),
                            pl_lin_reg_report (linear_regression.rs:854-858)                           */
};

/* status written per problem by the solve kernels */
enum pdsb_status { PDSB_OK = 0, PDSB_GATED = 1 /* rank gate fired -> null output */ };

const char* pdsb_last_error(void);
int pdsb_version(void);
/* number of this library's kernels launched so far on this process (bench.py's gpu_launches) */
int64_t pdsb_kernel_launch_count(void);
/* plugin layer: results exported to the caller whose buffers have not been released yet (ownership tests) */
int64_t pdsb_plugin_live_results(void);
/* which kernel handled the last pdsb_dev_moments_f32 call on this thread: 1 = tcgen05/TMA Gram kernel, 3 = register-moments
 * kernel (<= 10 features, one target, >= 65536 rows, no mask / weights), 0 = the generic path of k2_gram_simt.cu (FP64
 * tensor-core ring kernels for up to 64 aligned columns — f32 columns are widened on the fly —, SIMT register tiles otherwise) */
int pdsb_last_moments_path(void);
/* force a path for the f32 moments: 0 auto, 1 simt, 2 tcgen05 (tests / ncu) */
void pdsb_set_moments_path(int path);
/* make `device` current for the calling thread inside the library's (statically linked) CUDA runtime */
int pdsb_set_device(int device);
/* ---- multi-GPU (SURVEY.md §8e).  Rows shard naturally: every GPU builds the moments of its row range, ONE
 * ncclAllReduce(sum, f64) of (p+t+1)^2 values over NVLink joins them, every GPU solves redundantly and predicts its
 * own rows.  The Gram being sharded: get_xtx_with_lambda / build_xty (src/linear/lr/lr_solvers.rs:183-211, 262-278).
 * NCCL is bound at run time (dlopen of libnccl.so.2; PDS_B200_NCCL_LIB overrides the name).
 *
 * (i) device group, single process (a Polars process): the host layer splits every large pdsb_host_lin_reg call
 *     (>= PDS_B200_SHARD_MIN_ROWS rows, default 2^21) into one contiguous row shard per device; each shard is uploaded
 *     over its own PCIe link by its own worker thread.  Chosen by the environment variable PDS_B200_DEVICES
 *     ("8" = first 8, "all", or "0,2,5") or by pdsb_set_devices (n <= 1 returns to single-device operation). */
int pdsb_set_devices(const int* devices, int n);
int pdsb_device_group_size(void);
/* (ii) world communicator, one process per GPU (torchrun / Dask / Ray workers): rank 0 creates a 128-byte id, the
 *     launcher distributes it, every rank joins.  From then on every pdsb_host_lin_reg / plugin lin_reg call is
 *     COLLECTIVE: each rank passes its own rows and all ranks get the coefficients of the fit over the union (and the
 *     predictions of their own rows).  pdsb_comm_destroy leaves the communicator. */
int pdsb_comm_unique_id(void* out128);
int pdsb_comm_init_rank(int world_size, int rank, const void* id128);
void pdsb_comm_destroy(void);
int pdsb_comm_size(void);
int pdsb_nccl_version(void); /* 0 when NCCL could not be loaded */
/* device layer of (ii): in-place sum of `count` f64 values over the world communicator, enqueued on `stream`
 * (no-op without a communicator).  This is the one exchange of the row-sharded path: count = (p+t+1)^2. */
int pdsb_dev_allreduce_f64(double* buf, int64_t count, void* stream);
/* bytes of the calling thread's last host-layer upload that went through the pinned staging ring (pageable input) */
int64_t pdsb_last_staged_bytes(void);

/* tcgen05 kernel variant: 1 (default) the hi lanes of the A operand hold the raw data (the tensor core truncates fp32
 * to TF32 itself), 0 they clear the low 13 mantissa bits themselves (cross-check: must be bit-identical) */
void pdsb_set_tc_variant(int v);

/* =====================================================================================================
 * (1) device layer.  X is column-major [n x p] with leading dimension ldx (elements), Y is column-major
 *     [n x t] with ldy; `w` (nullable) are per-row weights, `mask` (nullable) a per-row 0/1 validity in the
 *     matrix dtype (masked rows must already be zero in X and Y; the packer guarantees it).
 * ===================================================================================================== */

/* Moments  M = [X | Y | 1]^T diag(w) [X | Y | 1], (q1 x q1) row-major f64 on the device, q1 = p+t+1.
 * The "1" column is `mask` when given.  One pass over the data: replaces get_xtx_with_lambda + build_xty
 * (lr_solvers.rs:183-211, 262-278), x.transpose()*w*x (linear_regression.rs:1026-1027), and the column sums
 * of faer_coordinate_descent (:483-484).  f32 data: 3xTF32 split on tcgen05 tensor cores, f64 reduction. */
int pdsb_dev_moments_f32(const float* X, int64_t ldx, const float* Y, int64_t ldy, const float* w,
                         const float* mask, int64_t n, int p, int t, double* M, void* stream);
int pdsb_dev_moments_f64(const double* X, int64_t ldx, const double* Y, int64_t ldy, const double* w,
                         const double* mask, int64_t n, int p, int t, double* M, void* stream);

/* Row-blocked frame: the library's native HBM layout for the f32 headline path.  A frame of `ncols` columns and n rows
 * stores element (row r, column c) at  frame[(r / 128) * ncols * 128 + c * 128 + (r % 128)]  — i.e. every block of
 * 128 rows x ncols columns is ONE contiguous run, so a 128-row stage of the Gram kernel is a single sequential
 * 512*ncols-byte read (measured on B200: a column-major frame caps the TMA pipeline at 4.3 TB/s with all arithmetic
 * removed, the blocked frame reaches 6.5 TB/s).  Rows >= n of the last block must be zero.  pdsb_frame_elems gives the
 * allocation size in elements; pdsb_dev_frame_from_colmajor_f32 converts a column-major matrix. */
#define PDSB_FRAME_ROWS 128
size_t pdsb_frame_elems(int64_t n, int ncols);
int pdsb_dev_frame_from_colmajor_f32(const float* src, int64_t ld, int64_t n, int ncols, float* frame, void* stream);
/* pdsb_dev_moments_f32 / pdsb_dev_predict_f32 on a frame: X = columns [xcol, xcol+p), Y = columns [ycol, ycol+t).
 * The tcgen05 kernel takes frames with ncols == p + t and X, Y adjacent in either order; other shapes use K2a. */
int pdsb_dev_moments_frame_f32(const float* frame, int64_t n, int ncols, int xcol, int p, int ycol, int t,
                               const float* mask, double* M, void* stream);
int pdsb_dev_predict_frame_f32(const float* frame, int64_t n, int ncols, int xcol, int p, int ycol, int t, int add_bias,
                               const float* mask, const double* beta, const int* status, float* pred, float* resid,
                               int64_t ldo, uint8_t* valid, double* ssr, void* stream);

typedef struct pdsb_solve_opts {
  int p, t;              /* features (bias excluded), targets                                          */
  int add_bias;          /* LRKwargs.bias (linear_regression.rs:29)                                     */
  int method;            /* enum pdsb_method                                                            */
  int solver;            /* enum pdsb_solver                                                            */
  int positive;          /* LRKwargs.positive                                                           */
  int max_iter;          /* LRKwargs.max_iter (the f32 twin's hard-coded 200/2000 are applied by caller)*/
  int f32_gate;          /* 1: evaluate logs of the gate the way the f32 twin would (tolerance in f32)  */
  double l1_reg, l2_reg; /* l2 is NOT scaled by n for ridge, IS scaled by n inside CD (lr_solvers.rs:442,479) */
  double tol;            /* CD / NNLS tolerance, or rcond for PDSB_METHOD_RCOND                          */
  double singular_x_tol; /* rank gate; <= 0 disables (linear_regression.rs:452)                         */
} pdsb_solve_opts;

/* Solve on device from the moments.  beta: [(p+bias) x t] column-major f64 (bias last, as the reference's
 * physical ones column makes it).  status: 1 int.  aux (nullable): method RCOND -> (p+bias) singular values
 * of X; method INV -> (p+bias)^2 inverse of X'X (+lambda), row-major. */
int pdsb_dev_solve(const double* M, const pdsb_solve_opts* opts, double* beta, int* status, double* aux,
                   void* stream);

/* pred = [X|1] beta, resid = Y - pred  (linear_regression.rs:782-785, 635-636; lr/mod.rs:146-174).
 * pred/resid are column-major [n x t] with leading dimension ldo.  Rows with mask==0 and every row when
 * *status != 0 get valid=0 (valid nullable: one byte per row).  ssr (nullable): 8 doubles; [k] = sum of squared
 * residuals of target k (< 4) over valid rows, [4+k] = the same weighted by w (linear_regression.rs:1037-1038). */
int pdsb_dev_predict_f32(const float* X, int64_t ldx, const float* Y, int64_t ldy, const float* w,
                         const float* mask, int64_t n, int p, int t, int add_bias, const double* beta,
                         const int* status, float* pred, float* resid, int64_t ldo, uint8_t* valid,
                         double* ssr, void* stream);
int pdsb_dev_predict_f64(const double* X, int64_t ldx, const double* Y, int64_t ldy, const double* w,
                         const double* mask, int64_t n, int p, int t, int add_bias, const double* beta,
                         const int* status, double* pred, double* resid, int64_t ldo, uint8_t* valid,
                         double* ssr, void* stream);

/* group_by(seg).agg(pds.lin_reg(...)) in ONE launch sequence: groups are contiguous row ranges
 * [offsets[g], offsets[g+1]) (device int64, n_groups+1 entries).  Batched per-group Gram + solve, one warp
 * per problem.  Replaces Polars calling _polars_plugin_pl_lr once per group (SURVEY 3.6; utils/mod.rs:81-84).
 * beta: [n_groups x (p+bias)] row-major f64; status: n_groups ints.  Only OLS / ridge (+gate). */
int pdsb_dev_grouped_lin_reg_f32(const float* X, int64_t ldx, const float* y, const int64_t* offsets,
                                 int64_t n_groups, int64_t n, int p, const pdsb_solve_opts* opts,
                                 double* beta, int* status, void* stream);
int pdsb_dev_grouped_lin_reg_f64(const double* X, int64_t ldx, const double* y, const int64_t* offsets,
                                 int64_t n_groups, int64_t n, int p, const pdsb_solve_opts* opts,
                                 double* beta, int* status, void* stream);

/* rolling_lin_reg / recursive_lin_reg: faer_rolling_lr, faer_rolling_skipping_lr, faer_recursive_lr
 * (lr_online_solvers.rs:148-301) + the output loops of pl_rolling_lr / pl_recursive_lr
 * (linear_regression.rs:1121-1283).  window > 0: row j (>= window-1) gets OLS/ridge on rows (j-window, j];
 * window == 0: expanding fit on rows [0, j] starting when `min_rows` valid rows have been seen.
 * Non-finite rows never contribute (OnlineLR::update, lr_online_solvers.rs:85-89).
 * skip != 0: row j is valid iff its window holds >= min_rows finite rows (skip-window policy); else every
 * j >= window-1 is valid.  coeffs: [n x (p+bias)] row-major (the list values), pred: [n], valid: [n] bytes. */
int pdsb_dev_online_lin_reg_f32(const float* X, int64_t ldx, const float* y, int64_t n, int p, int add_bias,
                                int64_t window, int64_t min_rows, int skip, double lambda, float* coeffs,
                                float* pred, uint8_t* valid, void* stream);
int pdsb_dev_online_lin_reg_f64(const double* X, int64_t ldx, const double* y, int64_t n, int p, int add_bias,
                                int64_t window, int64_t min_rows, int skip, double lambda, double* coeffs,
                                double* pred, uint8_t* valid, void* stream);

/* Row-sharded recursive_lin_reg (SURVEY.md §8e): the shard holding global rows [row0, row0 + n) continues the
 * expanding fit of the shards before it.  m0 = moments [X | y | 1]' [X | y | 1] ((p+2)^2 f64, row-major, as written by
 * pdsb_dev_moments_* with t = 1) summed over all preceding rows (null for the first shard). */
int pdsb_dev_recursive_shard_f32(const float* X, int64_t ldx, const float* y, int64_t n, int p, int add_bias,
                                 int64_t min_rows, int skip, double lambda, const double* m0, int64_t row0,
                                 float* coeffs, float* pred, uint8_t* valid, void* stream);
int pdsb_dev_recursive_shard_f64(const double* X, int64_t ldx, const double* y, int64_t n, int p, int add_bias,
                                 int64_t min_rows, int skip, double lambda, const double* m0, int64_t row0,
                                 double* coeffs, double* pred, uint8_t* valid, void* stream);

/* lin_reg_report statistics (pl_lin_reg_report / pl_wls_report, linear_regression.rs:822-1117).
 * se_type: 0 se, 1..4 hc0..hc3.  out: 8 rows x (p+bias) f64 row-major = beta, std_err, t, p, ci_lo, ci_hi,
 * and r2 / adj_r2 broadcast.  y_var is the ddof=1 variance Polars computes upstream (expr_linear.py:615). */
int pdsb_dev_report_f32(const float* X, int64_t ldx, const float* y, const float* w, const float* mask,
                        int64_t n, int p, int add_bias, int se_type, double y_var, double* out, void* stream);
int pdsb_dev_report_f64(const double* X, int64_t ldx, const double* y, const double* w, const double* mask,
                        int64_t n, int p, int add_bias, int se_type, double y_var, double* out, void* stream);

/* =====================================================================================================
 * (2) host layer: Arrow-style chunked columns in host memory.
 * ===================================================================================================== */
typedef struct pdsb_chunk {
  const void* data;        /* values buffer (Arrow buffers[1]), NOT yet offset                          */
  const uint8_t* validity; /* Arrow validity bitmap (buffers[0]) or NULL                                */
  int64_t offset;          /* Arrow `offset` (sliced arrays / groups)                                   */
  int64_t length;
} pdsb_chunk;

typedef struct pdsb_column {
  const char* name;
  int dtype;               /* enum pdsb_dtype */
  int n_chunks;
  const pdsb_chunk* chunks;
  int64_t null_count;      /* -1 = unknown (computed from bitmaps) */
} pdsb_column;

/* LRKwargs / MultiLRKwargs / SWWLRKwargs of the reference (linear_regression.rs:27-66), one struct. */
typedef struct pdsb_lr_kwargs {
  int bias;
  const char* null_policy; /* "raise"|"skip"|"zero"|"one"|"ignore"|"skip_window"|<float>  (linear/mod.rs:43-65) */
  const char* solver;
  double l1_reg, l2_reg, tol;
  int weighted;
  const char* std_err;     /* "se"|"hc0".."hc3" */
  int positive;
  int64_t max_iter;
  double singular_x_tol;
  int64_t last_target_idx; /* MultiLRKwargs */
  int64_t n;               /* SWWLRKwargs.n (window / start_with) */
  double lambda;           /* SWWLRKwargs.lambda */
  int64_t min_size;        /* SWWLRKwargs.min_size */
} pdsb_lr_kwargs;

/* Result buffers are owned by the library (pinned host memory from an internal pool); release with
 * pdsb_host_result_free.  Unused members are NULL/0. */
typedef struct pdsb_host_result {
  int is_f32;
  int64_t n_rows;          /* rows of row-wise outputs (pred/resid/online) */
  int n_coef;              /* p + bias */
  int n_targets;
  int gated;               /* 1 -> null coefficient list(s) / all-null predictions */
  void* coeffs;            /* [n_targets x n_coef] (lin_reg) or [n_rows x n_coef] (online), dtype T */
  void* singular_values;   /* [n_coef] T (w_rcond) */
  void* pred;              /* [n_targets x n_rows] T */
  void* resid;             /* [n_targets x n_rows] T */
  uint8_t* valid;          /* [n_rows] bytes, 1 = not null (NULL => all valid) */
  double* report;          /* 8 x n_coef f64 (see pdsb_dev_report_*) */
  void* _owner;            /* internal */
} pdsb_host_result;

void pdsb_host_result_free(pdsb_host_result* r);

/* pl_lr / pl_lr_pred / pl_lr_multi / pl_lr_multi_pred / pl_lr_w_rcond  (linear_regression.rs:419-820).
 * cols follow the reference's input order: [weights?] target(s) features...   want_pred selects the _pred twin.
 * rcond != 0 selects pl_lr_w_rcond.  f32 selects the `_f32` symbol family (linear_regression_f32.rs). */
int pdsb_host_lin_reg(const pdsb_column* cols, int n_cols, const pdsb_lr_kwargs* kw, int f32, int n_targets,
                      int want_pred, int w_rcond, pdsb_host_result* out);
/* pl_lin_reg_report / pl_wls_report: cols = [weights?] var(y) y features... */
int pdsb_host_report(const pdsb_column* cols, int n_cols, const pdsb_lr_kwargs* kw, int f32, int weighted,
                     pdsb_host_result* out);
/* pl_rolling_lr (rolling=1) / pl_recursive_lr (rolling=0): cols = y features... */
int pdsb_host_online(const pdsb_column* cols, int n_cols, const pdsb_lr_kwargs* kw, int f32, int rolling,
                     pdsb_host_result* out);
/* pl_logistic_coeffs (want_pred = 0) / pl_logistic_pred (want_pred = 1)  (src/num_ext/logistic_regression.rs:10-99,
 * solver src/linear/logistic/logistic_solver.rs:107-146): cols = y (0/1) features...; float64 only, like the reference.
 * coeffs: [n_coef] (bias last); pred: [n_rows] probabilities, valid marks the rows the null policy kept. */
int pdsb_host_logistic(const pdsb_column* cols, int n_cols, const pdsb_lr_kwargs* kw, int want_pred,
                       pdsb_host_result* out);
/* additive fast path for group_by().agg(lin_reg): cols = y features..., `group_offsets` host int64 [n_groups+1]
 * over contiguous (sorted-by-key) rows.  coeffs: [n_groups x n_coef], valid: [n_groups] (0 = gated). */
int pdsb_host_grouped_lin_reg(const pdsb_column* cols, int n_cols, const int64_t* group_offsets,
                              int64_t n_groups, const pdsb_lr_kwargs* kw, int f32, pdsb_host_result* out);

/* ---------------------------------------------------------------------------------------------------------
 * Dense-matrix callers of the same solvers: what the reference's PyO3 classes bind
 * (src/pymodels/py_lr.rs:21-224: PyLR, PyElasticNet, PyOnlineLR; numpy float64 matrices, numpy_faer.rs:10-66).
 * A pdsb_matrix is a HOST view with strides in elements.  Accepted layouts: C order (col_stride == 1),
 * F order (row_stride == 1), and any strided column vector; anything else -> "Input array is not contiguous."
 * Error strings follow LinalgErrors::to_string (src/linear/mod.rs:20-31).
 * --------------------------------------------------------------------------------------------------------- */
typedef struct pdsb_matrix {
  const double* data;
  int64_t n_rows, n_cols;
  int64_t row_stride, col_stride;
} pdsb_matrix;

enum pdsb_model { PDSB_MODEL_LR = 0, PDSB_MODEL_ELASTIC_NET = 1, PDSB_MODEL_ONLINE_LR = 2 };

/* LR::fit (lr_solvers.rs:64-73: faer_solve_lr, ungated; l2_reg = lambda on the non-bias diagonal; `solver` as
 * lr/mod.rs:18-27), ElasticNet::fit (:140-176: coordinate descent, l1/l2 scaled by n inside, tol, max_iter),
 * OnlineLR::fit (lr_online_solvers.rs:100-143: QR solve + explicit inverse of X'X + lambda I).
 * coeffs: n_cols + add_bias doubles, bias last.  inv (PDSB_MODEL_ONLINE_LR only): (n_cols + add_bias)^2, row-major. */
int pdsb_model_fit(int model, const pdsb_matrix* X, const pdsb_matrix* y, int add_bias, const char* solver,
                   double l1_reg, double l2_reg, double tol, int64_t max_iter, double* coeffs, double* inv);
/* LinearModel::predict (lr/mod.rs:146-174): out[r] = X[r,:] . coeffs[:p] + (has_bias ? coeffs[p] : 0) */
int pdsb_model_predict(const pdsb_matrix* X, const double* coeffs, int n_coef, int has_bias, double* out);

/* GLM (src/pymodels/py_glm.rs, src/linear/glm/glm_solvers.rs): a family and its canonical link —
 * gaussian: identity, poisson: log, binomial: logit, gamma: inverse; variances 1, mu, mu (1 - mu), mu^2. */
enum pdsb_glm_family { PDSB_GLM_GAUSSIAN = 0, PDSB_GLM_POISSON = 1, PDSB_GLM_BINOMIAL = 2, PDSB_GLM_GAMMA = 3 };
/* GLM::fit by IRLS (faer_irls, glm_solvers.rs:249-359): beta = 0, mu from y, then per iteration the weighted normal
 * equations X'WX beta = X'Wz by pivoted QR until max|beta - beta_new| < tol or max_iter solves (the last beta is
 * returned either way).  add_bias appends the ones column last, so the bias is coeffs[n_cols].  At most 64 columns.
 * coeffs: n_cols + add_bias doubles; *n_iter: the number of weighted least-squares solves. */
int pdsb_glm_fit(const pdsb_matrix* X, const pdsb_matrix* y, int add_bias, int family, int64_t max_iter, double tol,
                 double* coeffs, int64_t* n_iter);
/* GLM predict: g^-1(X coeffs[:p] + bias) (GLM::glm_predict), or the linear predictor itself when linear != 0 */
int pdsb_glm_predict(const pdsb_matrix* X, const double* coeffs, int n_coef, int has_bias, int family, int linear,
                     double* out);
/* Device layer of pdsb_glm_fit: X column-major [n x p] (ldx) and y [n] on the device; X's columns and y must be 16-byte
 * aligned and ldx even (else an error).  beta: device, p + add_bias doubles.  n_iter: HOST.  Each iteration is one
 * fused pass over X and y plus a solve on the moments; the call synchronises `stream` once per iteration to test
 * convergence, and returns when the fit is done. */
int pdsb_dev_glm_f64(const double* X, int64_t ldx, const double* y, int64_t n, int p, int add_bias, int family,
                     int64_t max_iter, double tol, double* beta, int64_t* n_iter, void* stream);

/* OnlineLR state ((X'X)^-1 and the coefficients) kept resident on the device between updates. */
typedef struct pdsb_online_lr pdsb_online_lr;
pdsb_online_lr* pdsb_online_lr_new(int n_coef, int has_bias);          /* NULL on failure (see pdsb_last_error) */
void pdsb_online_lr_free(pdsb_online_lr* h);
int pdsb_online_lr_set(pdsb_online_lr* h, const double* coeffs, const double* inv);   /* set_coeffs_bias_inverse :29-52 */
/* OnlineLR::update (:85-89) + woodbury_step (:307-332); c = +1 adds the row, -1 removes it.  A row with a
 * non-finite value is ignored.  Stream-ordered: returns without waiting for the device. */
int pdsb_online_lr_update(pdsb_online_lr* h, const double* x_row, double y, double c);
int pdsb_online_lr_get(pdsb_online_lr* h, double* coeffs /* nullable */, double* inv /* nullable */);

#ifdef __cplusplus
}
#endif
#endif /* PDSB_H */
