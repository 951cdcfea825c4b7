// Internal launch wrappers of the device kernels (C++), used by the C-ABI layer in host/api.cc.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include "../../../include/pdsb.h"

namespace pdsb {

// K2a generic SIMT moments (f32 / f64, weights, mask)
template <typename T>
int moments_simt(const T* X, int64_t ldx, const T* Y, int64_t ldy, const T* w, const T* mask, int64_t n,
                 int p, int t, double* M, cudaStream_t s, int64_t bstride = 0 /* frame block stride (elements) or 0 */);

// K2a-GLM: moments [X | z | 1]' diag(w) [X | z | 1] of one IRLS iteration of `family` (enum pdsb_glm_family), (w, z)
// computed in the kernel from X, y and beta (first != 0: from mu_start(y, mean_y), beta not read).  p <= 64; X columns and
// y 16-byte aligned, ldx even.
int glm_moments(const double* X, int64_t ldx, const double* y, int64_t n, int p, int add_bias, int family,
                const double* beta, int first, double mean_y, double* M, cudaStream_t s);

// K2b tcgen05 + TMA moments, f32, 3xTF32 split (hi/lo), f64 flush; p <= 64 features, t <= 4 targets.  Returns 0 ok, 1 error,
// -1 "shape not supported by this kernel" (caller uses K2a).
int moments_tcgen05_f32(const float* X, int64_t ldx, const float* Y, int64_t ldy, const float* mask,
                        int64_t n, int p, int t, double* M, cudaStream_t s);
void set_tc_mode(int m);   // 1 raw hi operand (default), 0 the hi lanes clear the low 13 bits themselves (cross-check)
constexpr int FRAME_ROWS = 128;   // rows per block of the row-blocked frame layout: [block][column][FRAME_ROWS]
bool moments_tcgen05_frame_supported(int64_t n, int ncols, int xcol, int p, int ycol, int t);
int moments_tcgen05_frame_f32(const float* frame, int64_t n, int ncols, int xcol, int p, int ycol, int t, const float* mask,
                              double* M, cudaStream_t s);
bool moments_tcgen05_supported(const float* X, int64_t ldx, const float* Y, int64_t ldy, int64_t n, int p,
                               int t);

// K3 single-CTA solve on the moments
int solve_from_moments(const double* M, const pdsb_solve_opts& o, double* beta, int* status, double* aux,
                       cudaStream_t s);

// K4 predict / residual / SSR
template <typename T>
int predict_resid(const T* X, int64_t ldx, const T* Y, int64_t ldy, const T* w, const T* mask, int64_t n,
                  int p, int t, int add_bias, const double* beta, const int* status, T* pred, T* resid,
                  int64_t ldo, uint8_t* valid, double* ssr, cudaStream_t s, int64_t bstride = 0);

// K1 pack: src column chunk (any numeric dtype, optional validity bitmap) -> T column
// mode: 0 null->NaN, 1 null->fill, 2 null->0 (row masked elsewhere)
template <typename T>
int pack_chunk(const void* src, int src_dtype, const uint8_t* validity, int64_t bit_offset, int64_t len,
               T* dst, int mode, double fill, cudaStream_t s, int64_t bstride = 0, int64_t row0 = 0);
// column-major [n x ncols] (ld) -> row-blocked frame
template <typename T>
int to_frame(const T* src, int64_t ld, int64_t n, int ncols, T* frame, cudaStream_t s);
// rowmask[i] &= validity bit (rowmask pre-set to 1)
template <typename T>
int and_validity(const uint8_t* validity, int64_t bit_offset, int64_t len, T* rowmask, cudaStream_t s);
template <typename T>
int fill_value(T* dst, int64_t len, T v, cudaStream_t s);
// zero rows of a column where rowmask == 0
template <typename T>
int zero_masked(T* col, const T* rowmask, int64_t len, cudaStream_t s);
// dst[i] = sqrt(w[i]) * (mask ? mask[i] : 1)   (unused by the exact-weight path; kept for the tcgen05 WLS route)
template <typename T>
int count_mask(const T* rowmask, int64_t len, double* out, cudaStream_t s);

// K5 grouped (segmented) OLS / ridge, one warp per problem
template <typename T>
int grouped_lin_reg(const T* X, int64_t ldx, const T* y, const int64_t* offsets, int64_t n_groups,
                    int64_t n, int p, const pdsb_solve_opts& o, double* beta, int* status, cudaStream_t s);

// whole-frame moments for p <= 10 features and one target on K5's register kernel (0 ok, 1 error, -1 shape not taken)
template <typename T>
int moments_small(const T* X, int64_t ldx, const T* y, int64_t n, int p, double* M, cudaStream_t s);

// K6/K7 rolling + recursive
template <typename T>
int online_lin_reg(const T* X, int64_t ldx, const T* y, int64_t n, int p, int add_bias, int64_t window,
                   int64_t min_rows, int skip, double lambda, const double* m0 /* moments of the preceding rows or null */,
                   int64_t row0 /* global index of row 0 */, T* coeffs, T* pred, uint8_t* valid, cudaStream_t s);

// K10 dense-matrix callers (model classes): strided gather to column-major, strided predict, Woodbury update
template <typename T>
int gather_colmajor(const T* src, int64_t rs, int64_t cs, int64_t n, int p, T* dst, int64_t ld, cudaStream_t s);
// family: enum pdsb_glm_family whose inverse link is applied to X beta + bias; -1 (or gaussian) leaves it as is
int predict_strided(const double* X, int64_t rs, int64_t cs, int64_t n, int p, const double* beta, int has_bias,
                    int family, double* out, cudaStream_t s);
int woodbury_update(double* inv, double* w, int q, int has_bias, const double* x, double y, double c, cudaStream_t s);

// K11 logistic regression (IRLS row pass: weights, working response, summed log-loss per block; probabilities)
int irls_max_parts();
template <typename T>
int irls_rows(const T* X, int64_t ldx, const T* y, const T* mask, int64_t n, int p, int add_bias, const double* beta,
              T* w, T* z, double* loss_parts, int* n_parts, cudaStream_t s);
template <typename T>
int sigmoid_predict(const T* X, int64_t ldx, int64_t n, int p, int add_bias, const double* beta, T* out, cudaStream_t s);

// K9 report
template <typename T>
int report_stats(const T* X, int64_t ldx, const T* y, const T* w, const T* mask, int64_t n, int p,
                 int add_bias, int se_type, double y_var, double* out, cudaStream_t s);

}  // namespace pdsb
