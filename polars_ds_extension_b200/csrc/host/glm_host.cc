// GLM (gaussian / Poisson / binomial / gamma with their canonical links) by iteratively reweighted least squares:
// faer_irls (/root/reference/src/linear/glm/glm_solvers.rs:249-359) on the device.  Per iteration ONE pass over X and y
// (K2a-GLM: eta, mu, the IRLS weight and the working response in registers, fed straight into the FP64 tensor-core
// moments), the pivoted-QR solve of X'WX beta = X'Wz on those moments (K3; faer_weighted_lr, lr_solvers.rs:384-409: no
// ridge, no rank gate), and a download of the q coefficients for the convergence test max|beta - beta_new| < tol.
// No line search and no step halving: the reference has none; after max_iter iterations the last beta is returned.
#include <cmath>
#include <cstdint>
#include <vector>

#include "../common.h"
#include "../kernels/glm_link.h"
#include "../kernels/kernels.h"
#include "host.h"

namespace pdsb {

int glm_irls(const double* X, int64_t ldx, const double* y, int64_t n, int p, int add_bias, int family, int64_t max_iter,
             double tol, double* beta, int64_t* n_iter, cudaStream_t s) {
  if (family < glm::GAUSSIAN || family > glm::GAMMA) { set_error("glm: unknown family %d", family); return 1; }
  if (p > 64) { set_error("glm: more than 64 features are not supported"); return 1; }
  if (n < 1 || p < 1 || n < p) { set_error("Not enough rows / columns."); return 1; }
  if (max_iter < 1) { set_error("`max_iter` must be > 1."); return 1; }
  auto al16 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
  if (!X || !y || !beta || !al16(X) || !al16(y) || ldx % 2 != 0 || ldx < n) {
    set_error("glm: X and y need 16-byte aligned columns and an even leading dimension >= n");
    return 1;
  }
  const int q = p + (add_bias ? 1 : 0), q1 = p + 2;
  double* dM = nullptr;
  int* dstatus = nullptr;
  if (dev_alloc((void**)&dM, (size_t)(q1 * q1 + 4) * sizeof(double), s)) return 1;   // M, then [y | 1]' [y | 1]
  dstatus = reinterpret_cast<int*>(dM + q1 * q1);
  struct Free { double* p; cudaStream_t s; ~Free() { dev_free(p, s); } } free_m{dM, s};

  // mean(y) for the starting mu of every family but binomial: the moments of [y | 1] (p = 0), a fixed-order sum
  double mean_y = 0.0;
  if (family != glm::BINOMIAL) {
    double sums[4];
    if (moments_simt<double>(y, ldx, y, ldx, nullptr, nullptr, n, 0, 1, dM, s)) return 1;
    PDSB_CUDA_OK(cudaMemcpyAsync(sums, dM, sizeof(sums), cudaMemcpyDeviceToHost, s));
    PDSB_CUDA_OK(cudaStreamSynchronize(s));
    mean_y = sums[1] / (double)n;
  }
  PDSB_CUDA_OK(cudaMemsetAsync(beta, 0, (size_t)q * sizeof(double), s));
  pdsb_solve_opts o{};
  o.p = p; o.t = 1; o.add_bias = add_bias ? 1 : 0; o.method = PDSB_METHOD_LSTSQ; o.solver = PDSB_SOLVER_QR;
  o.l2_reg = 0.0; o.singular_x_tol = 0.0;
  std::vector<double> hb((size_t)q, 0.0), hn((size_t)q);
  int64_t it = 0;
  while (it < max_iter) {
    if (glm_moments(X, ldx, y, n, p, add_bias, family, beta, it == 0, mean_y, dM, s)) return 1;
    if (solve_from_moments(dM, o, beta, dstatus, nullptr, s)) return 1;
    PDSB_CUDA_OK(cudaMemcpyAsync(hn.data(), beta, (size_t)q * sizeof(double), cudaMemcpyDeviceToHost, s));
    PDSB_CUDA_OK(cudaStreamSynchronize(s));
    ++it;
    double max_diff = 0.0;                       // Rust's f64::max: a NaN difference is skipped
    for (int j = 0; j < q; ++j) max_diff = std::fmax(max_diff, std::fabs(hb[j] - hn[j]));
    hb.swap(hn);
    if (max_diff < tol) break;
  }
  *n_iter = it;
  return 0;
}

}  // namespace pdsb

using namespace pdsb;

extern "C" {

int pdsb_dev_glm_f64(const double* X, int64_t ldx, const double* y, int64_t n, int p, int add_bias, int family,
                     int64_t max_iter, double tol, double* beta, int64_t* n_iter, void* stream) {
  if (require_device()) return 1;
  if (!n_iter) { set_error("glm: null n_iter"); return 1; }
  return glm_irls(X, ldx, y, n, p, add_bias, family, max_iter, tol, beta, n_iter, (cudaStream_t)stream);
}

}  // extern "C"
