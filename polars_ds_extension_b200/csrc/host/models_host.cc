// Dense-matrix host layer: the second caller of the solvers (SURVEY.md §8f rank 1).
//
// Reference: PyLR / PyElasticNet / PyOnlineLR (/root/reference/src/pymodels/py_lr.rs:21-224) wrap
// LR::fit -> faer_solve_lr (src/linear/lr/lr_solvers.rs:64-73, 296-308; ungated, ridge on the non-bias diagonal),
// ElasticNet::fit -> faer_coordinate_descent (:140-176), OnlineLR::fit -> faer_qr_lr_with_inv
// (src/linear/online_lr/lr_online_solvers.rs:100-143), OnlineLR::update -> woodbury_step (:62-90, 307-332) and
// LinearModel::predict (src/linear/lr/mod.rs:146-174); the error strings are LinalgErrors::to_string
// (src/linear/mod.rs:20-31).  Inputs are numpy float64 matrices (numpy_faer.rs:10-66).
//
// Everything numeric runs on the device: upload -> (transpose to the column-major frame) -> K2a moments -> K3 solve,
// K10 strided predict, K10 Woodbury update on device-resident state.  No CPU arithmetic, no fallback.
#include <cstring>
#include <vector>

#include "../common.h"
#include "../kernels/kernels.h"
#include "host.h"
#include <mutex>

namespace pdsb {
namespace {

struct Bag {
  cudaStream_t s;
  std::vector<void*> ptrs;
  explicit Bag(cudaStream_t st) : s(st) {}
  ~Bag() { for (void* p : ptrs) dev_free(p, s); }
  double* alloc(size_t count) {
    void* p = nullptr;
    if (dev_alloc(&p, (count ? count : 1) * sizeof(double), s)) return nullptr;
    ptrs.push_back(p);
    return reinterpret_cast<double*>(p);
  }
};

inline int64_t pad_ld(int64_t n) { return (n + 31) & ~int64_t(31); }

int check_matrix(const pdsb_matrix* m) {
  if (!m || m->n_rows < 0 || m->n_cols < 0 || (m->n_rows > 0 && m->n_cols > 0 && !m->data)) {
    set_error("Input is not contiguous or is empty");
    return 1;
  }
  return 0;
}

// Host matrix -> device.  C order (col_stride 1) lands row-major and is transposed by K10 into the column-major
// destination; F order (row_stride 1) is copied column by column with one strided DMA.  Returns the device view
// actually usable by a strided reader in (*view, *vrs, *vcs) when `colmajor_dst` is null (predict path).
int upload(const pdsb_matrix& m, double* colmajor_dst, int64_t ld, Bag& bag, cudaStream_t s, const double** view,
           int64_t* vrs, int64_t* vcs) {
  const int64_t n = m.n_rows, p = m.n_cols;
  if (n == 0 || p == 0) return 0;
  if (m.col_stride == 1 && m.row_stride >= p) {
    double* raw = bag.alloc((size_t)n * p);
    if (!raw) return 1;
    PDSB_CUDA_OK(cudaMemcpy2DAsync(raw, (size_t)p * 8, m.data, (size_t)m.row_stride * 8, (size_t)p * 8, (size_t)n,
                                   cudaMemcpyHostToDevice, s));
    if (colmajor_dst) return gather_colmajor<double>(raw, p, 1, n, (int)p, colmajor_dst, ld, s);
    *view = raw; *vrs = p; *vcs = 1;
    return 0;
  }
  if (m.row_stride == 1 && m.col_stride >= n) {
    double* dst = colmajor_dst;
    int64_t dld = ld;
    if (!dst) { dld = pad_ld(n); dst = bag.alloc((size_t)dld * p); if (!dst) return 1; }
    PDSB_CUDA_OK(cudaMemcpy2DAsync(dst, (size_t)dld * 8, m.data, (size_t)m.col_stride * 8, (size_t)n * 8, (size_t)p,
                                   cudaMemcpyHostToDevice, s));
    if (!colmajor_dst) { *view = dst; *vrs = 1; *vcs = dld; }
    return 0;
  }
  if (p == 1 && m.row_stride >= 1) {   // a strided vector (a column of a C-order matrix)
    double* dst = colmajor_dst ? colmajor_dst : bag.alloc((size_t)n);
    if (!dst) return 1;
    PDSB_CUDA_OK(cudaMemcpy2DAsync(dst, 8, m.data, (size_t)m.row_stride * 8, 8, (size_t)n, cudaMemcpyHostToDevice, s));
    if (!colmajor_dst) { *view = dst; *vrs = 1; *vcs = n; }
    return 0;
  }
  set_error("Input array is not contiguous.");
  return 1;
}

}  // namespace
}  // namespace pdsb

using namespace pdsb;

struct pdsb_online_lr {
  int q, has_bias, device;
  double* inv;   // [q][q]
  double* w;     // [q]  (bias last)
  double* x;     // [q]  staging for one row
  bool fit;
  // the handle owns its stream and a lock: update / get / set from ANY thread are ordered on this one stream and never
  // race on inv / w / the single staging row (the Python OnlineLR object carries no thread affinity)
  cudaStream_t stream = nullptr;
  std::mutex mu;
};

extern "C" {

int pdsb_model_fit(int model, const pdsb_matrix* X, const pdsb_matrix* y, int add_bias, const char* solver,
                   double l1_reg, double l2_reg, double tol, int64_t max_iter, double* coeffs, double* inv) {
  if (require_device()) return 1;
  if (check_matrix(X) || check_matrix(y)) return 1;
  if (!coeffs || (model == PDSB_MODEL_ONLINE_LR && !inv)) { set_error("pdsb_model_fit: null output"); return 1; }
  const int64_t n = X->n_rows;
  const int p = (int)X->n_cols;
  if (n != y->n_rows) { set_error("Dimension mismatch."); return 1; }                   // lr/mod.rs:122-123
  if (y->n_cols != 1) { set_error("Dimension mismatch."); return 1; }
  if (n == 0 || p == 0) { set_error("Not enough rows / columns."); return 1; }
  if (model != PDSB_MODEL_ELASTIC_NET && n < p) { set_error("Not enough rows / columns."); return 1; }   // :124-126; EN: lr_solvers.rs:168-175
  cudaStream_t s, s2;
  if (thread_streams(&s, &s2)) return 1;
  Bag bag(s);
  const int q = p + (add_bias ? 1 : 0);
  const int64_t ld = pad_ld(n);
  double* dZ = bag.alloc((size_t)ld * (p + 1));
  double* dM = bag.alloc((size_t)(p + 2) * (p + 2));
  double* dbeta = bag.alloc((size_t)q);
  double* daux = bag.alloc((size_t)q * q + q);
  int* dstatus = reinterpret_cast<int*>(bag.alloc(2));
  if (!dZ || !dM || !dbeta || !daux || !dstatus) return 1;
  const double* v; int64_t a, b;
  if (upload(*X, dZ, ld, bag, s, &v, &a, &b)) return 1;
  if (upload(*y, dZ + (size_t)ld * p, ld, bag, s, &v, &a, &b)) return 1;
  if (moments_simt<double>(dZ, ld, dZ + (size_t)ld * p, ld, nullptr, nullptr, n, p, 1, dM, s)) return 1;

  pdsb_solve_opts o{};
  o.p = p; o.t = 1; o.add_bias = add_bias ? 1 : 0; o.solver = solver_from_string(solver ? solver : "qr");
  o.singular_x_tol = 0.0;                       // the model classes never gate (faer_solve_lr, not _gated)
  if (model == PDSB_MODEL_LR) { o.method = PDSB_METHOD_LSTSQ; o.l2_reg = l2_reg; }
  else if (model == PDSB_MODEL_ELASTIC_NET) {
    o.method = PDSB_METHOD_CD; o.l1_reg = l1_reg; o.l2_reg = l2_reg; o.tol = tol; o.max_iter = (int)max_iter; o.positive = 0;
  } else if (model == PDSB_MODEL_ONLINE_LR) { o.method = PDSB_METHOD_INV; o.l2_reg = l2_reg; }
  else { set_error("pdsb_model_fit: unknown model %d", model); return 1; }
  if (solve_from_moments(dM, o, dbeta, dstatus, model == PDSB_MODEL_ONLINE_LR ? daux : nullptr, s)) return 1;
  PDSB_CUDA_OK(cudaMemcpyAsync(coeffs, dbeta, (size_t)q * sizeof(double), cudaMemcpyDeviceToHost, s));
  if (model == PDSB_MODEL_ONLINE_LR)
    PDSB_CUDA_OK(cudaMemcpyAsync(inv, daux, (size_t)q * q * sizeof(double), cudaMemcpyDeviceToHost, s));
  PDSB_CUDA_OK(cudaStreamSynchronize(s));
  return 0;
}

}  // extern "C"

namespace {
// LinearModel::predict (lr/mod.rs:146-174), then g^-1 of `family` (-1: none)
int predict_matrix(const pdsb_matrix* X, const double* coeffs, int n_coef, int has_bias, int family, double* out) {
  if (require_device()) return 1;
  if (check_matrix(X)) return 1;
  if (n_coef < 1 || !coeffs) { set_error("Matrix is not learned yet."); return 1; }      // lr/mod.rs:149-150
  const int p = n_coef - (has_bias ? 1 : 0);
  if (X->n_cols != p) { set_error("Dimension mismatch."); return 1; }                  // :147-148
  const int64_t n = X->n_rows;
  if (n == 0) return 0;
  cudaStream_t s, s2;
  if (thread_streams(&s, &s2)) return 1;
  Bag bag(s);
  double* dbeta = bag.alloc((size_t)n_coef);
  double* dout = bag.alloc((size_t)n);
  if (!dbeta || !dout) return 1;
  PDSB_CUDA_OK(cudaMemcpyAsync(dbeta, coeffs, (size_t)n_coef * sizeof(double), cudaMemcpyHostToDevice, s));
  const double* view = nullptr; int64_t rs = 0, cs = 0;
  if (p > 0 && upload(*X, nullptr, 0, bag, s, &view, &rs, &cs)) return 1;
  if (predict_strided(view, rs, cs, n, p, dbeta, has_bias ? 1 : 0, family, dout, s)) return 1;
  PDSB_CUDA_OK(cudaMemcpyAsync(out, dout, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, s));
  PDSB_CUDA_OK(cudaStreamSynchronize(s));
  return 0;
}
}  // namespace

extern "C" {

int pdsb_model_predict(const pdsb_matrix* X, const double* coeffs, int n_coef, int has_bias, double* out) {
  return predict_matrix(X, coeffs, n_coef, has_bias, -1, out);
}

/* GLM::fit (glm_solvers.rs:213-237 -> faer_irls) on numpy matrices: upload to the padded column-major frame, IRLS on
 * the device (glm_host.cc) */
int pdsb_glm_fit(const pdsb_matrix* X, const pdsb_matrix* y, int add_bias, int family, int64_t max_iter, double tol,
                 double* coeffs, int64_t* n_iter) {
  if (require_device()) return 1;
  if (check_matrix(X) || check_matrix(y)) return 1;
  if (!coeffs || !n_iter) { set_error("pdsb_glm_fit: null output"); return 1; }
  const int64_t n = X->n_rows;
  const int p = (int)X->n_cols;
  if (n != y->n_rows || y->n_cols != 1) { set_error("Dimension mismatch."); return 1; }   // lr/mod.rs:122-123
  if (n == 0 || p == 0 || n < p) { set_error("Not enough rows / columns."); return 1; }   // :124-126
  if (p > 64) { set_error("glm: more than 64 features are not supported"); return 1; }
  cudaStream_t s, s2;
  if (thread_streams(&s, &s2)) return 1;
  Bag bag(s);
  const int q = p + (add_bias ? 1 : 0);
  const int64_t ld = pad_ld(n);
  double* dZ = bag.alloc((size_t)ld * (p + 1));
  double* dbeta = bag.alloc((size_t)q);
  if (!dZ || !dbeta) return 1;
  const double* v; int64_t a, b;
  if (upload(*X, dZ, ld, bag, s, &v, &a, &b)) return 1;
  if (upload(*y, dZ + (size_t)ld * p, ld, bag, s, &v, &a, &b)) return 1;
  if (glm_irls(dZ, ld, dZ + (size_t)ld * p, n, p, add_bias ? 1 : 0, family, max_iter, tol, dbeta, n_iter, s)) return 1;
  PDSB_CUDA_OK(cudaMemcpyAsync(coeffs, dbeta, (size_t)q * sizeof(double), cudaMemcpyDeviceToHost, s));
  PDSB_CUDA_OK(cudaStreamSynchronize(s));
  return 0;
}

int pdsb_glm_predict(const pdsb_matrix* X, const double* coeffs, int n_coef, int has_bias, int family, int linear,
                     double* out) {
  if (family < PDSB_GLM_GAUSSIAN || family > PDSB_GLM_GAMMA) { set_error("glm: unknown family %d", family); return 1; }
  return predict_matrix(X, coeffs, n_coef, has_bias, linear ? -1 : family, out);
}

pdsb_online_lr* pdsb_online_lr_new(int n_coef, int has_bias) {
  if (require_device()) return nullptr;
  if (n_coef < 1 || n_coef > 512) { set_error("online lin_reg state: %d coefficients not supported (1..512)", n_coef); return nullptr; }
  pdsb_online_lr* h = new pdsb_online_lr{n_coef, has_bias ? 1 : 0, 0, nullptr, nullptr, nullptr, false};
  cudaGetDevice(&h->device);
  double* blk = nullptr;
  if (cudaMalloc(&blk, ((size_t)n_coef * n_coef + 2 * (size_t)n_coef) * sizeof(double)) != cudaSuccess) {
    set_error("online lin_reg state: cudaMalloc failed");
    delete h;
    return nullptr;
  }
  h->inv = blk; h->w = blk + (size_t)n_coef * n_coef; h->x = h->w + n_coef;
  if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess) {
    set_error("pdsb_online_lr_new: stream creation failed");
    cudaFree(blk);
    delete h;
    return nullptr;
  }
  return h;
}

void pdsb_online_lr_free(pdsb_online_lr* h) {
  if (!h) return;
  if (h->stream) { cudaStreamSynchronize(h->stream); cudaStreamDestroy(h->stream); }
  cudaFree(h->inv);
  delete h;
}

/* coeffs: n_coef values (bias last), inv: n_coef^2 row-major  (OnlineLR::set_coeffs_bias_inverse, :29-52) */
int pdsb_online_lr_set(pdsb_online_lr* h, const double* coeffs, const double* inv) {
  if (!h || !coeffs || !inv) { set_error("pdsb_online_lr_set: null argument"); return 1; }
  std::lock_guard<std::mutex> lk(h->mu);
  cudaStream_t s = h->stream;
  PDSB_CUDA_OK(cudaMemcpyAsync(h->w, coeffs, (size_t)h->q * sizeof(double), cudaMemcpyHostToDevice, s));
  PDSB_CUDA_OK(cudaMemcpyAsync(h->inv, inv, (size_t)h->q * h->q * sizeof(double), cudaMemcpyHostToDevice, s));
  PDSB_CUDA_OK(cudaStreamSynchronize(s));
  h->fit = true;
  return 0;
}

/* x_row: the n_coef - has_bias feature values of ONE row; non-finite rows are ignored (OnlineLR::update :85-89) */
int pdsb_online_lr_update(pdsb_online_lr* h, const double* x_row, double y, double c) {
  if (!h || !x_row) { set_error("pdsb_online_lr_update: null argument"); return 1; }
  if (!h->fit) { set_error("Matrix is not learned yet."); return 1; }
  std::lock_guard<std::mutex> lk(h->mu);
  cudaStream_t s = h->stream;
  const int pf = h->q - h->has_bias;
  if (pf > 0) PDSB_CUDA_OK(cudaMemcpyAsync(h->x, x_row, (size_t)pf * sizeof(double), cudaMemcpyHostToDevice, s));
  if (woodbury_update(h->inv, h->w, h->q, h->has_bias, h->x, y, c, s)) return 1;
  return 0;   // stream-ordered on the handle's stream: the next update / get (from any thread) sees the new state
}

int pdsb_online_lr_get(pdsb_online_lr* h, double* coeffs, double* inv) {
  if (!h) { set_error("pdsb_online_lr_get: null handle"); return 1; }
  if (!h->fit) { set_error("Matrix is not learned yet."); return 1; }
  std::lock_guard<std::mutex> lk(h->mu);
  cudaStream_t s = h->stream;
  if (coeffs) PDSB_CUDA_OK(cudaMemcpyAsync(coeffs, h->w, (size_t)h->q * sizeof(double), cudaMemcpyDeviceToHost, s));
  if (inv) PDSB_CUDA_OK(cudaMemcpyAsync(inv, h->inv, (size_t)h->q * h->q * sizeof(double), cudaMemcpyDeviceToHost, s));
  PDSB_CUDA_OK(cudaStreamSynchronize(s));
  return 0;
}

}  // extern "C"
