"""GLM without a GPU: the IRLS oracle (tests/glm_oracle.py, a restatement of the reference's faer_irls) against
independent maximum-likelihood fits on the data of the reference's test_glm_family, the reference's
convergence-failure case, the GLM class's constructor errors and repr, the loud failure of every numeric call without a
CUDA device, and the exported C symbols."""
import numpy as np
import pytest

from polars_ds_extension_b200.linear_models import GLM
from tests import glm_oracle as go

FAMILIES = ["gaussian", "binomial", "poisson", "gamma"]


@pytest.mark.parametrize("family", FAMILIES)
def test_oracle_matches_maximum_likelihood(family):
    X, y = go.family_data(family)
    beta, n_iter = go.faer_irls(X, y, family, add_bias=True, max_iter=200, tol=1e-8)
    ref = go.mle(family, X, y)
    assert n_iter < 200
    np.testing.assert_allclose(beta, ref, atol=1e-2)                  # the reference's tolerance against statsmodels
    np.testing.assert_allclose(beta, ref, rtol=1e-6, atol=1e-12)


def test_gaussian_glm_is_ols_in_two_iterations():
    X, y = go.family_data("gaussian")
    beta, n_iter = go.faer_irls(X, y, "normal", add_bias=True, max_iter=100, tol=1e-8)
    Xb = np.hstack([X, np.ones((X.shape[0], 1))])
    ols = np.linalg.lstsq(Xb, y, rcond=None)[0]
    assert n_iter == 2
    np.testing.assert_allclose(beta, ols, rtol=1e-12, atol=1e-13)


def test_oracle_convergence_failure_returns_finite_coefficients():
    X, y = go.convergence_failure_data()
    beta, n_iter = go.faer_irls(X, y, "poisson", add_bias=False, max_iter=1, tol=1e-12)
    assert n_iter == 1 and beta.shape == (5,) and np.all(np.isfinite(beta))


def test_constructor_errors_and_repr():
    with pytest.raises(NotImplementedError):
        GLM(solver="lbfgs")
    with pytest.raises(ValueError, match="`max_iter` must be > 1."):
        GLM(max_iter=0)
    with pytest.raises(NotImplementedError):
        GLM(family="tweedie")
    assert GLM(tol=-1e-6).tol == 1e-6
    assert repr(GLM()) == "GLM:\nLink: Identity\nVariance: Gaussian"
    assert repr(GLM(family="poisson")) == "GLM:\nLink: Log\nVariance: Poisson"
    assert repr(GLM(family="logistic")) == "GLM:\nLink: Logit\nVariance: Binomial"
    assert repr(GLM(family="gamma")) == "GLM:\nLink: Inverse\nVariance: Gamma"
    m = GLM(add_bias=True, feature_names_in_=["a"])
    assert not m.is_fit() and m.bias() == 0.0 and m.feature_names_in_ == ["a"]
    assert m.set_input_features(["b", "c"]).feature_names_in_ == ["b", "c"]
    with pytest.raises(ValueError, match="Matrix is not learned yet."):
        m.coeffs()
    with pytest.raises(ValueError, match="Matrix is not learned yet."):
        m.predict(np.zeros((2, 2)))


def test_numeric_calls_fail_loudly_without_gpu():
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    X, y = go.family_data("poisson")
    fitted = GLM(family="poisson", add_bias=True)
    fitted._fitted = np.array([0.1, 0.2, 0.3, 0.4, 0.5])
    for call in (lambda: GLM(family="poisson").fit(X, y), lambda: GLM().fit_df({"a": X[:, 0], "y": y}, ["a"], "y"),
                 lambda: fitted.predict(X), lambda: fitted.predict(X, linear=True)):
        with pytest.raises(ValueError, match="no usable CUDA device"):
            call()


def test_glm_symbols_are_exported():
    from polars_ds_extension_b200._lib import lib

    L = lib()
    for sym in ("pdsb_glm_fit", "pdsb_glm_predict", "pdsb_dev_glm_f64"):
        assert hasattr(L, sym), sym
