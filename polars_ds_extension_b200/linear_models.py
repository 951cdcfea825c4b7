"""Model classes over the B200 engine: `LR`, `ElasticNet`, `OnlineLR`, `GLM`.

Mirror of the reference's numpy-facing classes (/root/reference/python/polars_ds/linear_models.py:134-700), which are
thin wrappers over the PyO3 types PyLR / PyElasticNet / PyOnlineLR (src/pymodels/py_lr.rs:21-224).  Same constructor
arguments, method names, null policies and error messages; the arithmetic runs in libpds_b200 (`pdsb_model_fit`,
`pdsb_model_predict`, `pdsb_online_lr_*` in include/pdsb.h): moments + solve on the device, Woodbury updates on
device-resident state.  There is no CPU path: without the shared library or a CUDA device every fit / predict raises.

`GLM` (linear_models.py:700-950; PyGLM, src/pymodels/py_glm.rs) fits by IRLS on the device (`pdsb_glm_fit`): one fused
pass over X and y per iteration builds the weighted moments, a pivoted-QR solve on them gives the next iterate.

Data frames: `fit_df` / `predict_df` accept this package's Arrow-backed `Frame` (and a Polars frame when polars is
installed); MixedModel of the reference file is outside this engine's scope (SURVEY.md §8f).
"""
from __future__ import annotations

import ctypes as C
from typing import Any, List, Optional, Sequence, Tuple

import numpy as np

from ._lib import GLM_FAMILIES, MODEL_ELASTIC_NET, MODEL_LR, MODEL_ONLINE_LR, Matrix, lib
from .typing import LRSolverMethods, NullPolicy

__all__ = ["LR", "ElasticNet", "OnlineLR", "GLM"]


# ---------------------------------------------------------------------------------------------------------------
# host-side data preparation (the reference does this in Python as well: linear_models.py:45-131)
# ---------------------------------------------------------------------------------------------------------------
def _fill_value(null_policy: str) -> float:
    if null_policy == "zero":
        return 0.0
    if null_policy == "one":
        return 1.0
    try:
        v = float(null_policy)
    except Exception as e:  # same wording as linear_models.py:68-69
        raise ValueError(f"Unknown null_policy. Error: {e}")
    if not np.isfinite(v):
        raise ValueError("Unknown null_policy. Error: When null_policy is a number, it cannot be nan or infinite.")
    return v


def _handle_nans_in_np(X: np.ndarray, y: np.ndarray, null_policy: NullPolicy) -> Tuple[np.ndarray, np.ndarray]:
    """NaN handling for numpy inputs (linear_models.py:100-131): X is N x M, y is N x 1."""
    if null_policy == "ignore":
        return X, y
    if null_policy == "raise":
        if np.isnan(X).any() or np.isnan(y).any():
            raise ValueError("Nulls found in X or y.")
        return X, y
    y_nan = np.isnan(y).any(axis=1)
    if null_policy == "skip":
        keep = ~(np.isnan(X).any(axis=1) | y_nan)
        return X[keep], y[keep]
    fill = _fill_value(null_policy)
    return np.nan_to_num(X, nan=fill)[~y_nan], y[~y_nan]


def _as_matrix(a: Any) -> np.ndarray:
    m = np.asarray(a, dtype=np.float64)       # what the reference's _sanitize_np does (linear_models.py:71-97)
    if m.ndim == 1:
        m = m.reshape((-1, 1))
    if m.ndim != 2:
        raise ValueError("Dimension mismatch.")
    n, p = m.shape
    s0, s1 = m.strides
    row_major = s1 == 8 and s0 >= 8 * p          # C order, rows possibly padded (a column slice of a wider matrix)
    col_major = s0 == 8 and s1 >= 8 * n          # F order, columns possibly padded
    if not (row_major or col_major or n <= 1 or p <= 1 and s0 > 0):
        m = np.ascontiguousarray(m)              # the C ABI takes the two dense layouts and strided vectors
    return m


def _view(m: np.ndarray) -> Matrix:
    return Matrix(m.ctypes.data, m.shape[0], m.shape[1], m.strides[0] // 8 if m.shape[0] > 1 else max(m.shape[1], 1),
                  m.strides[1] // 8 if m.shape[1] > 1 else 1)


def _call(rc: int) -> None:
    if rc != 0:   # the PyO3 classes raise ValueError(LinalgErrors::to_string) (py_lr.rs:14-18)
        raise ValueError(lib().pdsb_last_error().decode("utf-8", "replace"))


def _fit(model: int, X: np.ndarray, y: np.ndarray, add_bias: bool, solver: str = "qr", l1: float = 0.0, l2: float = 0.0,
         tol: float = 1e-5, max_iter: int = 2000, want_inv: bool = False):
    Xm, ym = _as_matrix(X), _as_matrix(y)
    q = Xm.shape[1] + int(add_bias)
    coeffs = np.empty(q, dtype=np.float64)
    inv = np.empty((q, q), dtype=np.float64) if want_inv else None
    xv, yv = _view(Xm), _view(ym)
    _call(lib().pdsb_model_fit(model, C.byref(xv), C.byref(yv), int(add_bias), solver.encode(), float(l1), float(l2),
                               float(tol), int(max_iter), coeffs.ctypes.data, inv.ctypes.data if want_inv else None))
    return coeffs, inv


def _predict(X: np.ndarray, fitted: Optional[np.ndarray], has_bias: bool) -> np.ndarray:
    if fitted is None or fitted.size == 0:
        raise ValueError("Matrix is not learned yet.")
    Xm = _as_matrix(X)
    out = np.empty((Xm.shape[0], 1), dtype=np.float64)
    xv = _view(Xm)
    _call(lib().pdsb_model_predict(C.byref(xv), fitted.ctypes.data, int(fitted.size), int(has_bias), out.ctypes.data))
    return out


def _columns_of(df: Any, names: Sequence[str]) -> np.ndarray:
    """N x len(names) float64 matrix out of a Frame / Polars frame / mapping of arrays; nulls become NaN."""
    if hasattr(df, "lazy") and hasattr(df, "collect_schema"):          # polars, when installed
        return df.lazy().select(list(names)).collect().to_numpy().astype(np.float64)
    cols = df.columns if hasattr(df, "columns") and isinstance(df.columns, dict) else df
    out = []
    for n in names:
        c = cols[n]
        if hasattr(c, "to_numpy") and not isinstance(c, np.ndarray):
            try:
                c = c.to_numpy(zero_copy_only=False)
            except TypeError:
                c = c.to_numpy()
        a = np.asarray(c)
        if a.dtype == object:
            a = np.array([np.nan if v is None else v for v in a], dtype=np.float64)
        out.append(a.astype(np.float64))
    return np.column_stack(out) if out else np.empty((0, 0))


def _df_to_xy(df: Any, features: List[str], target: str, null_policy: NullPolicy) -> Tuple[np.ndarray, np.ndarray]:
    """Null policy for data frames (linear_models.py:45-68, 296-305): nulls, not NaNs, are what is handled."""
    Z = _columns_of(df, list(features) + [target])
    X, y = Z[:, :-1], Z[:, -1:]
    if null_policy == "ignore":
        return X, y
    if null_policy == "raise":
        if np.isnan(Z).any():
            raise ValueError("Nulls found in Dataframe.")
        return X, y
    return _handle_nans_in_np(X, y, null_policy)


def _with_prediction(df: Any, names: List[str], coeffs: np.ndarray, bias: float, name: str, predict):
    if len(names) <= 0:
        raise ValueError(
            "The linear model is not fitted on a dataframe, or no feature names have been given."
            "Not enough info to predict on a dataframe. Hint: try .fit_df() or .set_input_features()."
        )
    if hasattr(df, "lazy") and hasattr(df, "collect_schema"):          # polars: stays an expression, like the reference
        import polars as pl

        pred = pl.sum_horizontal(beta * pl.col(c) for c, beta in zip(names, coeffs))
        if bias != 0.0:
            pred = pred + bias
        return df.with_columns(pred.alias(name))
    return df.with_columns(**{name: predict(_columns_of(df, names)).ravel()})


class _Base:
    feature_names_in_: List[str]
    _fitted: Optional[np.ndarray]      # coefficients, bias last when _has_bias
    _has_bias: bool

    def is_fit(self) -> bool:
        return self._fitted is not None and self._fitted.size > 0

    def set_input_features(self, features: List[str]):
        self.feature_names_in_ = list(features)
        return self

    def coeffs(self) -> np.ndarray:
        """A copy of the coefficients (bias excluded)."""
        if not self.is_fit():
            raise ValueError("Matrix is not learned yet.")
        n = self._fitted.size - int(self._has_bias)
        return self._fitted[:n].copy()

    def bias(self) -> float:
        return float(self._fitted[-1]) if (self.is_fit() and self._has_bias) else 0.0

    def _set_coeffs_and_bias(self, coeffs, bias: float) -> None:
        # set_coeffs_and_bias (lr_solvers.rs:38-51): the bias is kept only when |bias| > eps
        c = np.ascontiguousarray(coeffs, dtype=np.float64).ravel()
        self._has_bias = abs(bias) > np.finfo(np.float64).eps
        self._fitted = np.concatenate([c, [bias]]) if self._has_bias else c.copy()

    def predict(self, X: np.ndarray) -> np.ndarray:
        return _predict(X, self._fitted, self._has_bias)

    def predict_df(self, df: Any, name: str = "prediction"):
        return _with_prediction(df, self.feature_names_in_, self.coeffs(), self.bias(), name, self.predict)

    def _describe(self, title: str) -> str:
        if not self.is_fit():
            return f"{title}\nNot fitted yet."
        return f"{title}\nCoefficients: {[round(float(x), 5) for x in self.coeffs()]}\nBias/Intercept: {self.bias()}\n"


class LR(_Base):
    """Ordinary least squares / ridge (linear_models.py:134-347; PyLR, py_lr.rs:21-80)."""

    def __init__(self, has_bias: bool = False, lambda_: float = 0.0, solver: LRSolverMethods = "qr",
                 feature_names_in_: Optional[List[str]] = None):
        self._has_bias = bool(has_bias)
        self.lambda_ = float(lambda_)
        self.solver = str(solver)
        self._fitted = None
        self.feature_names_in_ = [] if feature_names_in_ is None else list(feature_names_in_)

    @classmethod
    def from_values(cls, coeffs: List[float], bias: float = 0.0, feature_names_in_: Optional[List[str]] = None):
        m = cls(has_bias=(bias != 0.0), lambda_=0.0, solver="Not Solved", feature_names_in_=feature_names_in_)
        m._set_coeffs_and_bias(coeffs, float(bias))
        return m

    def __repr__(self) -> str:
        return self._describe("Linear Regression (Ridge) Model" if self.lambda_ > 0.0 else "Linear Regression Model")

    def fit(self, X: np.ndarray, y: np.ndarray, null_policy: NullPolicy = "ignore"):
        X_, y_ = _handle_nans_in_np(_as_matrix(X), _as_matrix(y).reshape((-1, 1)), null_policy)
        self._fitted, _ = _fit(MODEL_LR, X_, y_, self._has_bias, solver=self.solver, l2=self.lambda_)
        return self

    def fit_df(self, df: Any, features: List[str], target: str, null_policy: NullPolicy = "skip",
               show_report: bool = False):
        if show_report and self.lambda_ == 0.0:
            from .exprs.expr_linear import lin_reg_report

            frame = df if hasattr(df, "select") and hasattr(df, "columns") and isinstance(df.columns, dict) else None
            if frame is not None:
                print(frame.select(lin_reg_report(*features, target=target, add_bias=self._has_bias)))
        X, y = _df_to_xy(df, list(features), target, null_policy)
        self.feature_names_in_ = list(features)
        self._fitted, _ = _fit(MODEL_LR, X, y, self._has_bias, solver=self.solver, l2=self.lambda_)
        return self


class ElasticNet(_Base):
    """Elastic net by coordinate descent (linear_models.py:350-557; PyElasticNet, py_lr.rs:82-147).  Equivalent to
    scikit-learn's with alpha = l1_reg + l2_reg and l1_ratio = l1_reg / (l1_reg + l2_reg)."""

    def __init__(self, l1_reg: float, l2_reg: float, has_bias: bool = False, tol: float = 1e-5, max_iter: int = 2000,
                 feature_names_in_: Optional[List[str]] = None):
        if l1_reg <= 0.0 and l2_reg <= 0.0:
            raise ValueError("Cannot have both l1_reg and l2_reg <= 0.")
        self.l1_reg, self.l2_reg = float(l1_reg), float(l2_reg)
        self.tol, self.max_iter = float(tol), int(max_iter)
        self._has_bias = bool(has_bias)
        self._fitted = None
        self.feature_names_in_ = [] if feature_names_in_ is None else list(feature_names_in_)

    @classmethod
    def from_values(cls, coeffs: List[float], bias: float = 0.0, feature_names_in_: Optional[List[str]] = None):
        m = cls.__new__(cls)
        m.l1_reg = m.l2_reg = float("nan")       # ElasticNet::from_values (lr_solvers.rs:99-110)
        m.tol, m.max_iter = 1e-5, 2000
        m._fitted = None
        m.feature_names_in_ = [] if feature_names_in_ is None else list(feature_names_in_)
        m._set_coeffs_and_bias(coeffs, float(bias))
        return m

    def has_bias(self) -> bool:
        return self._has_bias

    def regularizers(self) -> Tuple[float, float]:
        return self.l1_reg, self.l2_reg

    def __repr__(self) -> str:
        return self._describe("ElasticNet Model")

    def _run(self, X, y):
        self._fitted, _ = _fit(MODEL_ELASTIC_NET, X, y, self._has_bias, l1=self.l1_reg, l2=self.l2_reg, tol=self.tol,
                               max_iter=self.max_iter)
        return self

    def fit(self, X: np.ndarray, y: np.ndarray, null_policy: NullPolicy = "ignore"):
        X_, y_ = _handle_nans_in_np(_as_matrix(X), _as_matrix(y).reshape((-1, 1)), null_policy)
        return self._run(X_, y_)

    def fit_df(self, df: Any, features: List[str], target: str, null_policy: NullPolicy = "skip"):
        X, y = _df_to_xy(df, list(features), target, null_policy)
        self.feature_names_in_ = list(features)
        return self._run(X, y)


class OnlineLR:
    """Online OLS / ridge: initial fit, then rank-1 Woodbury updates (linear_models.py:560-700; PyOnlineLR,
    py_lr.rs:149-224).  The inverse of X'X and the coefficients live on the device between updates; a row with a NaN
    is ignored by `update`."""

    def __init__(self, lambda_: float = 0.0, has_bias: bool = False):
        self.lambda_ = float(lambda_)
        self._has_bias = bool(has_bias)
        self._h: Optional[int] = None
        self._q = 0

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            try:
                lib().pdsb_online_lr_free(h)
            except Exception:
                pass

    def _state(self, q: int, has_bias: bool) -> int:
        if self._h and self._q == q and self._has_bias == has_bias:
            return self._h
        if self._h:
            lib().pdsb_online_lr_free(self._h)
            self._h = None
        h = lib().pdsb_online_lr_new(q, int(has_bias))
        if not h:
            raise ValueError(lib().pdsb_last_error().decode("utf-8", "replace"))
        self._h, self._q, self._has_bias = h, q, has_bias
        return h

    @classmethod
    def from_coeffs_bias_inverse(cls, coeffs: List[float], bias: float, inv: np.ndarray):
        c = np.ascontiguousarray(coeffs, dtype=np.float64).ravel()
        inv = np.ascontiguousarray(inv, dtype=np.float64)
        m = cls(lambda_=0.0, has_bias=(bias > 0.0))
        has_bias = abs(bias) > np.finfo(np.float64).eps
        full = np.concatenate([c, [bias]]) if has_bias else c
        # The reference compares len(coeffs) with inv.ncols() (lr_online_solvers.rs:35-36), which rejects every model
        # WITH a bias (its inverse has one more row/column); here the inverse must match coefficients + bias.
        if inv.ndim != 2 or inv.shape != (full.size, full.size):
            raise ValueError("Dimension mismatch.")
        _call(lib().pdsb_online_lr_set(m._state(full.size, has_bias), full.ctypes.data, inv.ctypes.data))
        return m

    def is_fit(self) -> bool:
        return bool(self._h)

    def __repr__(self) -> str:
        title = "Online Linear Regression (Ridge) Model" if self.lambda_ > 0.0 else "Online Linear Regression Model"
        if not self.is_fit():
            return f"{title}\nNot fitted yet."
        return f"{title}\nCoefficients: {[round(float(x), 5) for x in self.coeffs()]}\nBias/Intercept: {self.bias()}\n"

    def _get(self, want_inv: bool = False):
        if not self._h:
            raise ValueError("Matrix is not learned yet.")
        w = np.empty(self._q, dtype=np.float64)
        inv = np.empty((self._q, self._q), dtype=np.float64) if want_inv else None
        _call(lib().pdsb_online_lr_get(self._h, w.ctypes.data, inv.ctypes.data if want_inv else None))
        return w, inv

    def coeffs(self) -> np.ndarray:
        w, _ = self._get()
        return w[: self._q - int(self._has_bias)]

    def bias(self) -> float:
        if not self._h or not self._has_bias:
            return 0.0
        return float(self._get()[0][-1])

    def inv(self) -> np.ndarray:
        return self._get(want_inv=True)[1]

    def fit(self, X: np.ndarray, y: np.ndarray):
        Xm, ym = _as_matrix(X), _as_matrix(y).reshape((-1, 1))
        if np.isnan(Xm).any() or np.isnan(ym).any():
            raise ValueError("Online regression currently must fit without null for the initial fit.")
        w, inv = _fit(MODEL_ONLINE_LR, Xm, ym, self._has_bias, l2=self.lambda_, want_inv=True)
        _call(lib().pdsb_online_lr_set(self._state(w.size, self._has_bias), w.ctypes.data, inv.ctypes.data))
        return self

    def update(self, X: np.ndarray, y: Any, c: float = 1.0):
        if not self.is_fit():
            raise ValueError("You cannot update before the initial fit of the matrix.")
        x = np.ascontiguousarray(np.asarray(X, dtype=np.float64).reshape((1, -1)))
        if x.shape[1] != self._q - int(self._has_bias):
            raise ValueError("Dimension mismatch.")
        yv = float(np.asarray(y, dtype=np.float64).reshape((1, 1))[0, 0])
        _call(lib().pdsb_online_lr_update(self._h, x.ctypes.data, yv, float(c)))
        return self

    def predict(self, X: np.ndarray) -> np.ndarray:
        w, _ = self._get()
        return _predict(X, w, self._has_bias)


# GLM::to_string (glm_solvers.rs): the Debug names of the family's link and variance functions
_GLM_NAMES = {0: ("Identity", "Gaussian"), 1: ("Log", "Poisson"), 2: ("Logit", "Binomial"), 3: ("Inverse", "Gamma")}


class GLM(_Base):
    """Generalized linear model with the canonical link of its family, fit by IRLS (linear_models.py:700-950; PyGLM,
    py_glm.rs): gaussian / normal -> identity, poisson -> log, binomial / logistic -> logit, gamma -> inverse.  With
    `add_bias` the bias is the last coefficient.  At most 64 features."""

    def __init__(self, add_bias: bool = False, solver: str = "irls", family: str = "normal", max_iter: int = 100,
                 tol: float = 1e-8, feature_names_in_: Optional[List[str]] = None):
        if solver not in ["irls"]:
            raise NotImplementedError
        if max_iter < 1:
            raise ValueError("`max_iter` must be > 1.")
        if family not in ["gaussian", "normal", "poisson", "binomial", "logistic", "gamma"]:
            raise NotImplementedError
        self._has_bias = bool(add_bias)
        self.solver = solver
        self.family = family
        self.max_iter = int(max_iter)
        self.tol = abs(float(tol))
        self._family = GLM_FAMILIES[family]
        self._fitted = None
        self._n_iter = 0          # weighted least-squares solves of the last fit
        self.feature_names_in_ = [] if feature_names_in_ is None else list(feature_names_in_)

    def __repr__(self) -> str:
        # The reference calls PyGLM.describe(), which does not exist (AttributeError); this is GLM::to_string's text.
        link, variance = _GLM_NAMES[self._family]
        return f"GLM:\nLink: {link}\nVariance: {variance}"

    def _run(self, X: np.ndarray, y: np.ndarray):
        Xm, ym = _as_matrix(X), _as_matrix(y)
        coeffs = np.empty(Xm.shape[1] + int(self._has_bias), dtype=np.float64)
        it = C.c_int64(0)
        xv, yv = _view(Xm), _view(ym)
        _call(lib().pdsb_glm_fit(C.byref(xv), C.byref(yv), int(self._has_bias), self._family, self.max_iter, self.tol,
                                 coeffs.ctypes.data, C.byref(it)))
        self._fitted, self._n_iter = coeffs, int(it.value)
        return self

    def fit(self, X: np.ndarray, y: np.ndarray, null_policy: NullPolicy = "ignore"):
        X_, y_ = _handle_nans_in_np(_as_matrix(X), _as_matrix(y).reshape((-1, 1)), null_policy)
        return self._run(X_, y_)

    def fit_df(self, df: Any, features: List[str], target: str, null_policy: NullPolicy = "skip",
               show_report: bool = False):
        X, y = _df_to_xy(df, list(features), target, null_policy)
        self.feature_names_in_ = list(features)
        return self._run(X, y)

    def predict_df(self, df: Any, name: str = "prediction"):
        raise NotImplementedError("GLM.predict_df is not available (the reference leaves it out too)")

    def predict(self, X: np.ndarray, linear: bool = False) -> np.ndarray:
        """g^-1(X beta + bias) as an (n, 1) array; the linear predictor X beta + bias itself when `linear`."""
        if not self.is_fit():
            raise ValueError("Matrix is not learned yet.")
        Xm = _as_matrix(X)
        out = np.empty((Xm.shape[0], 1), dtype=np.float64)
        xv = _view(Xm)
        _call(lib().pdsb_glm_predict(C.byref(xv), self._fitted.ctypes.data, int(self._fitted.size), int(self._has_bias),
                                     self._family, int(bool(linear)), out.ctypes.data))
        return out
