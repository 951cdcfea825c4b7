"""CPU oracle of the GLM class: a NumPy restatement of the reference's `faer_irls`
(/root/reference/src/linear/glm/glm_solvers.rs:249-359) with the link and variance functions of
src/linear/glm/link_functions.rs, each line evaluated as the reference writes it.  The weighted least-squares step is
`oracle.lin_reg_oracle.faer_weighted_lr` (lr_solvers.rs:384-409: pivoted QR on X'WX, no ridge, no rank gate).

Test infrastructure only, like the rest of the oracle.
"""
from __future__ import annotations

from typing import Tuple

import numpy as np

from oracle.lin_reg_oracle import faer_weighted_lr

FAMILIES = {"gaussian": "gaussian", "normal": "gaussian", "poisson": "poisson", "binomial": "binomial",
            "logistic": "binomial", "gamma": "gamma"}


def link(f: str, mu):                                  # LinkFunction::link
    if f == "gaussian":
        return mu
    if f == "poisson":
        return np.log(mu)
    if f == "binomial":
        return np.log(mu / (1.0 - mu))
    return 1.0 / mu


def inv_link(f: str, eta):                             # LinkFunction::inv
    if f == "gaussian":
        return eta
    if f == "poisson":
        return np.exp(eta)
    if f == "binomial":
        e = np.exp(eta)
        return e / (1.0 + e)
    return 1.0 / eta


def deriv(f: str, mu):                                 # LinkFunction::deriv
    if f == "gaussian":
        return np.ones_like(mu)
    if f == "poisson":
        return 1.0 / mu
    if f == "binomial":
        return 1.0 / (mu * (1.0 - mu))
    r = 1.0 / mu
    return -(r * r)


def variance(f: str, mu):                              # VarianceFunction::variance
    if f == "gaussian":
        return np.ones_like(mu)
    if f == "poisson":
        return mu
    if f == "binomial":
        return mu * (1.0 - mu)
    return mu * mu


def faer_irls(X, y, family: str, add_bias: bool, max_iter: int, tol: float) -> Tuple[np.ndarray, int]:
    """(beta, n_iter): beta with the bias last when add_bias (GLM::fit_unchecked appends the ones column,
    glm_solvers.rs:213-237); n_iter = weighted least-squares solves performed."""
    f = FAMILIES[family]
    X = np.asarray(X, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64).reshape(-1)
    if add_bias:
        X = np.hstack([X, np.ones((X.shape[0], 1))])
    n = X.shape[0]
    beta = np.zeros(X.shape[1])
    with np.errstate(all="ignore"):
        if f == "binomial":                            # :266-272
            mu = (y + 0.5) * 0.5
        else:                                          # :273-279
            mu = (y + y.sum() / n) * 0.5
        eta = link(f, mu)
        n_iter = 0
        for _ in range(max_iter):
            d = deriv(f, mu)                           # :293-297
            w = 1.0 / ((d * d) * variance(f, mu))
            z = eta + d * (y - mu)                     # :301-305
            beta_new = faer_weighted_lr(X, z.reshape(-1, 1), w, "qr").reshape(-1)   # :308-313
            n_iter += 1
            eta = X @ beta_new                         # :316-330
            mu = inv_link(f, eta)                      # :333-335
            diff = np.abs(beta - beta_new)             # :338-341 (f64::max skips a NaN)
            max_diff = float(np.max(diff[~np.isnan(diff)], initial=0.0))
            beta = beta_new
            if max_diff < tol:                         # :344-348
                break
    return beta, n_iter


def predict(X, beta, add_bias: bool, family: str, linear: bool = False) -> np.ndarray:
    eta = np.asarray(X, dtype=np.float64) @ beta[: beta.size - int(add_bias)] + (beta[-1] if add_bias else 0.0)
    with np.errstate(all="ignore"):
        return (eta if linear else inv_link(FAMILIES[family], eta)).reshape(-1, 1)


# The data of the reference's test_glm_family (tests/test_linear_models.py:193-253): RandomState(42), n = 500, p = 4.
_GEN = {
    "gaussian": lambda X, rng: X @ np.array([1.0, -0.5, 0.3, 0.8]) + rng.randn(X.shape[0]) * 0.1,
    "binomial": lambda X, rng: rng.binomial(1, 1.0 / (1.0 + np.exp(-(X @ np.array([1.0, -0.5, 0.3, 0.8]))))).astype(float),
    "poisson": lambda X, rng: rng.poisson(np.exp(np.clip(X @ np.array([0.5, -0.25, 0.15, 0.4]), -2.0, 2.0))).astype(float),
    "gamma": lambda X, rng: rng.gamma(shape=2.0,
                                      scale=np.exp(np.clip(X @ np.array([0.3, -0.15, 0.09, 0.24]), -2.0, 2.0)) / 2.0),
}


def family_data(family: str):
    rng = np.random.RandomState(42)
    X = rng.randn(500, 4)
    return X, _GEN[family](X, rng)


def convergence_failure_data():
    """test_glm_convergence_failure (tests/test_linear_models.py:256-271)."""
    rng = np.random.RandomState(0)
    n, p = 200, 5
    X = rng.randn(n, p)
    y = np.exp(np.clip(X @ np.ones(p) * 0.2, -2, 2)) + rng.exponential(0.5, n)
    return X, y.reshape(-1, 1)


def mle(family: str, X, y) -> np.ndarray:
    """Independent maximum-likelihood fit with an intercept, returned as (coeffs..., bias): scikit-learn for the
    gaussian / binomial / Poisson families, scipy.optimize on the gamma log-likelihood (inverse link) otherwise.  All four
    links are canonical, so the maximiser is unique."""
    y = np.asarray(y, dtype=np.float64).reshape(-1)
    if family == "gaussian":
        from sklearn.linear_model import LinearRegression

        m = LinearRegression().fit(X, y)
    elif family == "binomial":
        from sklearn.linear_model import LogisticRegression

        m = LogisticRegression(C=np.inf, solver="newton-cholesky", tol=1e-14, max_iter=1000).fit(X, y)   # unpenalised
        return np.concatenate([m.coef_.ravel(), m.intercept_])
    elif family == "poisson":
        from sklearn.linear_model import PoissonRegressor

        m = PoissonRegressor(alpha=0.0, tol=1e-12, max_iter=10_000).fit(X, y)
    else:
        from scipy.optimize import minimize

        Xb = np.hstack([X, np.ones((X.shape[0], 1))])

        def nll(b):   # gamma with mu = 1 / eta, shape fixed: sum(y eta - log eta) up to constants
            eta = Xb @ b
            if np.any(eta <= 0):
                return np.inf, np.zeros_like(b)
            return float(np.sum(y * eta - np.log(eta))), Xb.T @ (y - 1.0 / eta)

        b0 = np.zeros(Xb.shape[1])
        b0[-1] = 1.0 / y.mean()
        r = minimize(nll, b0, jac=True, method="BFGS", options={"gtol": 1e-12, "maxiter": 10_000})
        return r.x
    return np.concatenate([np.ravel(m.coef_), [m.intercept_]])
