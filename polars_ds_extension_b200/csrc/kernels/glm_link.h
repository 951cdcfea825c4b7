// GLM link and variance functions of the four canonical families, written as the reference writes them
// (/root/reference/src/linear/glm/link_functions.rs) and evaluated literally: no clamping, so saturation gives what the
// reference gives (Poisson with mu = 0: w = 1 / (inf * 0) = NaN).  One definition for the fused IRLS moments kernel, its
// tail, the predict kernel and the host.  Family codes are enum pdsb_glm_family.
#pragma once
#include <cmath>

namespace pdsb {
namespace glm {

enum Family { GAUSSIAN = 0, POISSON = 1, BINOMIAL = 2, GAMMA = 3 };

// g(mu): identity, log, logit, inverse
template <int F> __host__ __device__ __forceinline__ double link(double mu) {
  if constexpr (F == GAUSSIAN) return mu;
  else if constexpr (F == POISSON) return log(mu);
  else if constexpr (F == BINOMIAL) return log(mu / (1.0 - mu));
  else return 1.0 / mu;
}

// g^-1(eta); the logit inverse is exp(eta) / (1 + exp(eta)) as written (NaN once exp overflows)
template <int F> __host__ __device__ __forceinline__ double inv(double eta) {
  if constexpr (F == GAUSSIAN) return eta;
  else if constexpr (F == POISSON) return exp(eta);
  else if constexpr (F == BINOMIAL) { const double e = exp(eta); return e / (1.0 + e); }
  else return 1.0 / eta;
}

// g'(mu)
template <int F> __host__ __device__ __forceinline__ double deriv(double mu) {
  if constexpr (F == GAUSSIAN) return 1.0;
  else if constexpr (F == POISSON) return 1.0 / mu;
  else if constexpr (F == BINOMIAL) return 1.0 / (mu * (1.0 - mu));
  else { const double r = 1.0 / mu; return -(r * r); }
}

// V(mu)
template <int F> __host__ __device__ __forceinline__ double variance(double mu) {
  if constexpr (F == GAUSSIAN) return 1.0;
  else if constexpr (F == POISSON) return mu;
  else if constexpr (F == BINOMIAL) return mu * (1.0 - mu);
  else return mu * mu;
}

// mu of the first iteration (faer_irls, glm_solvers.rs:266-279): (y + 0.5) / 2 for binomial, (y + mean(y)) / 2 otherwise
template <int F> __host__ __device__ __forceinline__ double mu_start(double y, double mean_y) {
  if constexpr (F == BINOMIAL) return (y + 0.5) * 0.5;
  else return (y + mean_y) * 0.5;
}

// One IRLS row (glm_solvers.rs:289-304): from eta and mu, the weight w = 1 / (g'(mu)^2 V(mu)) and the working response
// z = eta + g'(mu) (y - mu)
template <int F> __host__ __device__ __forceinline__ void irls_row(double eta, double mu, double y, double& w, double& z) {
  const double d = deriv<F>(mu);
  w = 1.0 / (d * d * variance<F>(mu));
  z = eta + d * (y - mu);
}

// runtime family -> g^-1 (predict); identity returns eta untouched
__host__ __device__ __forceinline__ double inv_rt(int family, double eta) {
  switch (family) {
    case POISSON: return inv<POISSON>(eta);
    case BINOMIAL: return inv<BINOMIAL>(eta);
    case GAMMA: return inv<GAMMA>(eta);
    default: return eta;
  }
}

}  // namespace glm
}  // namespace pdsb
