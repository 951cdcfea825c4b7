"""GLM on the B200: the fused IRLS moments kernel + pivoted-QR solve (pdsb_glm_fit / pdsb_dev_glm_f64) against the IRLS
oracle (tests/glm_oracle.py) and independent maximum-likelihood fits, on the reference's test_glm_family data, on
every tail shape of the 8-row batches and every feature-block count, and at size."""
import numpy as np
import pytest

from polars_ds_extension_b200.linear_models import GLM
from tests import glm_oracle as go

pytestmark = pytest.mark.gpu

FAMILIES = ["gaussian", "binomial", "poisson", "gamma"]


def _poisson_data(n, p, seed=0):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((n, p)) / np.sqrt(p)
    beta = rng.uniform(-0.5, 0.5, p)
    y = 1.0 + rng.poisson(np.exp(X @ beta + 0.3))
    return X, y.astype(np.float64)


def _close_to_oracle(m: GLM, X, y, family, add_bias, max_iter=100, tol=1e-8):
    beta, n_iter = go.faer_irls(X, y, family, add_bias, max_iter, tol)
    got = np.concatenate([m.coeffs(), [m.bias()]]) if add_bias else m.coeffs()
    np.testing.assert_allclose(got, beta, rtol=1e-6, atol=1e-9)
    assert m._n_iter == n_iter


@pytest.mark.parametrize("family", FAMILIES)
def test_families_match_mle_and_oracle(family):
    X, y = go.family_data(family)
    m = GLM(solver="irls", add_bias=True, family=family, max_iter=200, tol=1e-8).fit(X, y.reshape(-1, 1))
    ref = go.mle(family, X, y)
    np.testing.assert_allclose(m.coeffs(), ref[:-1], atol=1e-2)       # the reference's tolerance against statsmodels
    assert abs(m.bias() - ref[-1]) < 1e-2
    np.testing.assert_allclose(np.concatenate([m.coeffs(), [m.bias()]]), ref, rtol=1e-6, atol=1e-12)
    _close_to_oracle(m, X, y, family, True, 200, 1e-8)
    if family == "gaussian":
        assert m._n_iter == 2


def test_convergence_failure_returns_finite_coefficients():
    X, y = go.convergence_failure_data()
    m = GLM(solver="irls", add_bias=False, family="poisson", max_iter=1, tol=1e-12).fit(X, y)
    assert m._n_iter == 1 and np.all(np.isfinite(m.coeffs()))
    _close_to_oracle(m, X, y, "poisson", False, 1, 1e-12)


@pytest.mark.parametrize("p", [1, 8, 9, 31, 32, 33, 64])
@pytest.mark.parametrize("add_bias", [False, True])
def test_shapes(p, add_bias):
    for r in range(1, 8):                           # n = 8k + r: the fused tail kernel takes the last r rows
        X, y = _poisson_data(2048 + r, p, seed=p * 10 + r)
        _close_to_oracle(GLM(add_bias=add_bias, family="poisson").fit(X, y), X, y, "poisson", add_bias)
    X, y = _poisson_data(2048, p, seed=p)           # no tail
    _close_to_oracle(GLM(add_bias=add_bias, family="poisson").fit(X, y), X, y, "poisson", add_bias)


@pytest.mark.parametrize("family", ["gaussian", "poisson"])   # the fits of these few rows that have a maximiser
def test_fewer_than_eight_rows(family):
    for n in range(3, 8):                           # the tail kernel alone
        X, y = go.family_data(family)
        X, y = X[:n, :2], y[:n]
        _close_to_oracle(GLM(add_bias=False, family=family, max_iter=20).fit(X, y), X, y, family, False, 20)


def test_more_than_64_features_raises():
    X, y = _poisson_data(256, 65)
    with pytest.raises(ValueError, match="more than 64 features"):
        GLM(family="poisson").fit(X, y)


def test_input_layouts_and_null_policies():
    X, y = _poisson_data(5003, 12, seed=3)
    ref = GLM(add_bias=True, family="poisson").fit(X, y).coeffs()
    f = GLM(add_bias=True, family="poisson").fit(np.asfortranarray(X), y).coeffs()
    wide = np.hstack([X, np.ones((X.shape[0], 5))])
    s = GLM(add_bias=True, family="poisson").fit(wide[:, :12], y).coeffs()
    np.testing.assert_array_equal(f, ref)
    np.testing.assert_array_equal(s, ref)
    Xn = X.copy()
    Xn[::7, 3] = np.nan
    keep = ~np.isnan(Xn).any(axis=1)
    skipped = GLM(add_bias=True, family="poisson").fit(Xn, y, null_policy="skip")
    clean = GLM(add_bias=True, family="poisson").fit(X[keep], y[keep])
    np.testing.assert_array_equal(skipped.coeffs(), clean.coeffs())

    from polars_ds_extension_b200 import Frame

    names = [f"x{i}" for i in range(12)]
    df = Frame({n: X[:, i] for i, n in enumerate(names)} | {"y": y})
    m = GLM(add_bias=True, family="poisson").fit_df(df, names, "y")
    np.testing.assert_array_equal(m.coeffs(), ref)
    assert m.feature_names_in_ == names


@pytest.mark.parametrize("family", FAMILIES)
def test_predict(family):
    X, y = go.family_data(family)
    m = GLM(add_bias=True, family=family).fit(X, y)
    beta = np.concatenate([m.coeffs(), [m.bias()]])
    lin = m.predict(X, linear=True)
    assert lin.shape == (X.shape[0], 1)
    np.testing.assert_allclose(lin.ravel(), X @ m.coeffs() + m.bias(), rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(m.predict(X), go.predict(X, beta, True, family), rtol=1e-12, atol=1e-14)


def test_fits_are_bit_identical():
    X, y = _poisson_data(100_003, 20, seed=9)
    a = GLM(add_bias=True, family="poisson").fit(X, y)
    b = GLM(add_bias=True, family="poisson").fit(X, y)
    np.testing.assert_array_equal(a.coeffs(), b.coeffs())
    assert a.bias() == b.bias() and a._n_iter == b._n_iter


def test_device_api_equals_class():
    import torch

    from polars_ds_extension_b200 import device as dev

    X, y = _poisson_data(10_005, 17, seed=4)
    m = GLM(add_bias=True, family="poisson").fit(X, y)
    Xt = torch.from_numpy(np.ascontiguousarray(X.T)).cuda()          # (p, ld) with ld = n
    Xt = torch.nn.functional.pad(Xt, (0, 1))                          # even ld
    yt = torch.nn.functional.pad(torch.from_numpy(y).cuda(), (0, 1))
    beta, n_iter = dev.glm(Xt, yt, "poisson", add_bias=True, n=X.shape[0])
    got = beta.cpu().numpy()
    np.testing.assert_array_equal(got, np.concatenate([m.coeffs(), [m.bias()]]))
    assert n_iter == m._n_iter
    with pytest.raises(Exception, match="16-byte aligned"):
        dev.glm(Xt[:, 1:], yt[1:], "poisson", n=X.shape[0])


@pytest.mark.parametrize("family", ["poisson", "binomial"])
def test_at_size(family):
    rng = np.random.default_rng(11)
    n, p = 2_000_000, 32
    X = rng.standard_normal((n, p)) / np.sqrt(p)
    beta = rng.uniform(-1.0, 1.0, p)
    eta = X @ beta + 0.2
    y = rng.poisson(np.exp(eta)) if family == "poisson" else (rng.random(n) < 1.0 / (1.0 + np.exp(-eta)))
    y = y.astype(np.float64)
    m = GLM(add_bias=True, family=family).fit(X, y)
    _close_to_oracle(m, X, y, family, True)
