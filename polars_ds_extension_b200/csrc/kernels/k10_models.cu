// K10 — kernels behind the dense-matrix callers of the solvers: the reference's PyO3 classes PyLR / PyElasticNet /
// PyOnlineLR (/root/reference/src/pymodels/py_lr.rs:21-224) hand numpy float64 matrices of any stride
// (numpy_faer.rs:10-66) to LR::fit / ElasticNet::fit / OnlineLR::{fit, update} and LinearModel::predict
// (src/linear/lr/mod.rs:146-174).  Fit reuses K2a (moments) + K3 (solve); what is specific to this caller:
//   gather_colmajor   numpy row-major [n][p] -> the column-major frame the moment kernels read (tiled transpose)
//   predict_strided   pred = X beta + bias straight from the strided matrix (one pass, no transpose); for a GLM the
//                     inverse link of it (GLM::glm_predict, src/linear/glm/glm_solvers.rs)
//   woodbury_update   one rank-1 update / downdate of the device-resident (X'X)^-1 and beta
//                     (woodbury_step, src/linear/online_lr/lr_online_solvers.rs:307-332; OnlineLR::update :85-89)
#include "../common.h"
#include "kernels.h"
#include "glm_link.h"

namespace pdsb {

namespace {

constexpr int TILE = 32;

// dst[c * ld + r] = src[r * rs + c * cs]; reads and writes are both coalesced through a padded shared tile
template <typename T>
__global__ void __launch_bounds__(TILE * 8)
gather_colmajor_kernel(const T* __restrict__ src, int64_t rs, int64_t cs, int64_t n, int p, T* __restrict__ dst,
                       int64_t ld) {
  __shared__ T tile[TILE][TILE + 1];
  const int64_t r0 = (int64_t)blockIdx.x * TILE;
  const int c0 = blockIdx.y * TILE;
  // load: threadIdx.x walks the columns of a row (contiguous when cs == 1)
  for (int j = threadIdx.y; j < TILE; j += 8) {
    const int64_t r = r0 + j;
    const int c = c0 + threadIdx.x;
    if (r < n && c < p) tile[j][threadIdx.x] = src[r * rs + (int64_t)c * cs];
  }
  __syncthreads();
  // store: threadIdx.x walks the rows of a column (contiguous in the column-major destination)
  for (int j = threadIdx.y; j < TILE; j += 8) {
    const int c = c0 + j;
    const int64_t r = r0 + threadIdx.x;
    if (r < n && c < p) dst[(int64_t)c * ld + r] = tile[threadIdx.x][j];
  }
}

// one thread per row; beta (<= 256 coefficients) in shared memory
__global__ void __launch_bounds__(256)
predict_strided_kernel(const double* __restrict__ X, int64_t rs, int64_t cs, int64_t n, int p,
                       const double* __restrict__ beta, int has_bias, int family, double* __restrict__ out) {
  extern __shared__ double sb[];
  for (int i = threadIdx.x; i < p + has_bias; i += blockDim.x) sb[i] = beta[i];
  __syncthreads();
  const double bias = has_bias ? sb[p] : 0.0;
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (int64_t)gridDim.x * blockDim.x) {
    const double* row = X + r * rs;
    double acc = bias;
    for (int c = 0; c < p; ++c) acc = fma(row[(int64_t)c * cs], sb[c], acc);
    out[r] = glm::inv_rt(family, acc);
  }
}

// u = inv x';  z = 1 / (c + x u);  inv -= z u u';  w += z u (y - x w).   Single CTA, q <= 512.
// A row with a non-finite entry leaves the state untouched (OnlineLR::update, lr_online_solvers.rs:85-89).
__global__ void __launch_bounds__(128)
woodbury_kernel(double* __restrict__ inv, double* __restrict__ w, int q, int has_bias, const double* __restrict__ xin,
                double y, double c) {
  extern __shared__ double sm[];
  double* x = sm;            // q
  double* u = sm + q;        // q
  __shared__ double s_xu, s_xw;
  __shared__ int s_bad;
  const int tid = threadIdx.x;
  if (tid == 0) { s_bad = isfinite(y) ? 0 : 1; s_xu = 0.0; s_xw = 0.0; }
  __syncthreads();
  const int pf = q - has_bias;
  for (int i = tid; i < q; i += blockDim.x) {
    const double v = i < pf ? xin[i] : 1.0;     // the ones column is appended here (update_unchecked :64-75)
    x[i] = v;
    if (!isfinite(v)) s_bad = 1;
  }
  __syncthreads();
  if (s_bad) return;
  for (int i = tid; i < q; i += blockDim.x) {
    double acc = 0.0;
    for (int j = 0; j < q; ++j) acc = fma(inv[(size_t)i * q + j], x[j], acc);
    u[i] = acc;
  }
  __syncthreads();
  if (tid == 0) {
    double a = 0.0, b = 0.0;
    for (int i = 0; i < q; ++i) { a = fma(x[i], u[i], a); b = fma(x[i], w[i], b); }
    s_xu = a; s_xw = b;
  }
  __syncthreads();
  const double z = 1.0 / (c + s_xu);
  const double ydiff = y - s_xw;
  for (int idx = tid; idx < q * q; idx += blockDim.x) {
    const int i = idx / q, j = idx % q;
    inv[idx] -= z * u[i] * u[j];
  }
  for (int i = tid; i < q; i += blockDim.x) w[i] += z * u[i] * ydiff;
}

}  // namespace

template <typename T>
int gather_colmajor(const T* src, int64_t rs, int64_t cs, int64_t n, int p, T* dst, int64_t ld, cudaStream_t s) {
  if (n <= 0 || p <= 0) return 0;
  dim3 grid((unsigned)ceil_div(n, TILE), (unsigned)ceil_div(p, TILE));
  if (grid.y > 65535) { set_error("gather_colmajor: too many columns"); return 1; }
  gather_colmajor_kernel<T><<<grid, dim3(TILE, 8), 0, s>>>(src, rs, cs, n, p, dst, ld);
  PDSB_LAUNCH_OK();
  count_launch();
  return 0;
}
template int gather_colmajor<float>(const float*, int64_t, int64_t, int64_t, int, float*, int64_t, cudaStream_t);
template int gather_colmajor<double>(const double*, int64_t, int64_t, int64_t, int, double*, int64_t, cudaStream_t);

int predict_strided(const double* X, int64_t rs, int64_t cs, int64_t n, int p, const double* beta, int has_bias,
                    int family, double* out, cudaStream_t s) {
  if (n <= 0) return 0;
  const int64_t blocks = std::min<int64_t>(ceil_div(n, 256), (int64_t)sm_count() * 8);
  predict_strided_kernel<<<(unsigned)blocks, 256, (size_t)(p + 1) * sizeof(double), s>>>(X, rs, cs, n, p, beta, has_bias, family, out);
  PDSB_LAUNCH_OK();
  count_launch();
  return 0;
}

int woodbury_update(double* inv, double* w, int q, int has_bias, const double* x, double y, double c, cudaStream_t s) {
  if (q < 1 || q > 512) { set_error("online update: %d coefficients not supported (max 512)", q); return 1; }
  woodbury_kernel<<<1, 128, (size_t)2 * q * sizeof(double), s>>>(inv, w, q, has_bias, x, y, c);
  PDSB_LAUNCH_OK();
  count_launch();
  return 0;
}

}  // namespace pdsb
