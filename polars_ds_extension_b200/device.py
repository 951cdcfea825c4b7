"""torch-tensor front end of the device layer (pdsb_dev_*).  torch is plumbing here: it owns device memory and
streams (and torch.distributed carries the one collective of the multi-GPU path); all arithmetic is in the library.

Layout convention: a design matrix is a torch tensor of shape (p, ld) — p columns of ld >= n rows, row-major in
torch == column-major [ld x p] for the library.  Targets likewise (t, ld).
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Tuple

import torch

from ._lib import (GLM_FAMILIES, METHOD_CD, METHOD_INV, METHOD_LSTSQ, METHOD_NNLS, METHOD_RCOND, SOLVER_CHOLESKEY,
                   SOLVER_QR, SOLVER_SVD, SolveOpts, check, lib)


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream() -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _sfx(t: torch.Tensor) -> str:
    if t.dtype == torch.float32:
        return "f32"
    if t.dtype == torch.float64:
        return "f64"
    raise TypeError(f"unsupported dtype {t.dtype}")


def _ld(t: torch.Tensor) -> int:
    assert t.dim() == 2 and t.stride(1) == 1, "matrix must be (columns, rows) with contiguous rows"
    return t.stride(0) if t.shape[0] > 1 else t.shape[1]


def moments(X: torch.Tensor, Y: torch.Tensor, n: Optional[int] = None, w: Optional[torch.Tensor] = None,
            mask: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """M = [X|Y|1]^T diag(w) [X|Y|1] as a (q1, q1) float64 tensor, q1 = p + t + 1."""
    p, t = X.shape[0], Y.shape[0]
    n = X.shape[1] if n is None else n
    q1 = p + t + 1
    M = out if out is not None else torch.empty((q1, q1), dtype=torch.float64, device=X.device)
    fn = getattr(lib(), f"pdsb_dev_moments_{_sfx(X)}")
    check(fn(_ptr(X), _ld(X), _ptr(Y), _ld(Y), _ptr(w), _ptr(mask), n, p, t, _ptr(M), _stream()))
    return M


def solve(M: torch.Tensor, p: int, t: int = 1, add_bias: bool = False, method: int = METHOD_LSTSQ,
          solver: int = SOLVER_QR, l1_reg: float = 0.0, l2_reg: float = 0.0, tol: float = 0.0,
          singular_x_tol: float = 0.0, positive: bool = False, max_iter: int = 200, want_aux: bool = False,
          beta: Optional[torch.Tensor] = None, status: Optional[torch.Tensor] = None):
    q = p + int(add_bias)
    beta = beta if beta is not None else torch.empty((t, q), dtype=torch.float64, device=M.device)
    status = status if status is not None else torch.zeros(4, dtype=torch.int32, device=M.device)
    aux = torch.zeros(q * q + q, dtype=torch.float64, device=M.device) if want_aux else None
    o = SolveOpts(p=p, t=t, add_bias=int(add_bias), method=method, solver=solver, positive=int(positive),
                  max_iter=max_iter, f32_gate=0, l1_reg=l1_reg, l2_reg=l2_reg, tol=tol, singular_x_tol=singular_x_tol)
    check(lib().pdsb_dev_solve(_ptr(M), C.byref(o), _ptr(beta), _ptr(status), _ptr(aux), _stream()))
    return (beta, status, aux) if want_aux else (beta, status)


def predict(X: torch.Tensor, Y: torch.Tensor, beta: torch.Tensor, status: Optional[torch.Tensor], add_bias: bool,
            n: Optional[int] = None, mask: Optional[torch.Tensor] = None, w: Optional[torch.Tensor] = None,
            pred: Optional[torch.Tensor] = None, resid: Optional[torch.Tensor] = None,
            valid: Optional[torch.Tensor] = None, ssr: Optional[torch.Tensor] = None):
    p, t = X.shape[0], Y.shape[0]
    n = X.shape[1] if n is None else n
    ld = _ld(X)
    pred = pred if pred is not None else torch.empty((t, ld), dtype=X.dtype, device=X.device)
    resid = resid if resid is not None else torch.empty((t, ld), dtype=X.dtype, device=X.device)
    fn = getattr(lib(), f"pdsb_dev_predict_{_sfx(X)}")
    check(fn(_ptr(X), ld, _ptr(Y), _ld(Y), _ptr(w), _ptr(mask), n, p, t, int(add_bias), _ptr(beta), _ptr(status),
             _ptr(pred), _ptr(resid), _ld(pred), _ptr(valid), _ptr(ssr), _stream()))
    return pred, resid


def grouped_lin_reg(X: torch.Tensor, y: torch.Tensor, offsets: torch.Tensor, add_bias: bool = False,
                    l2_reg: float = 0.0, singular_x_tol: float = 0.0, solver: int = SOLVER_QR):
    p = X.shape[0]
    n = X.shape[1]
    ng = offsets.numel() - 1
    q = p + int(add_bias)
    beta = torch.empty((ng, q), dtype=torch.float64, device=X.device)
    status = torch.empty(ng, dtype=torch.int32, device=X.device)
    o = SolveOpts(p=p, t=1, add_bias=int(add_bias), method=METHOD_LSTSQ, solver=solver, l2_reg=l2_reg,
                  singular_x_tol=singular_x_tol)
    fn = getattr(lib(), f"pdsb_dev_grouped_lin_reg_{_sfx(X)}")
    check(fn(_ptr(X), _ld(X), _ptr(y), _ptr(offsets), ng, n, p, C.byref(o), _ptr(beta), _ptr(status), _stream()))
    return beta, status


def online_lin_reg(X: torch.Tensor, y: torch.Tensor, window: int, min_rows: int, add_bias: bool = False,
                   l2_reg: float = 0.0, skip: bool = False, n: Optional[int] = None,
                   coeffs: Optional[torch.Tensor] = None, pred: Optional[torch.Tensor] = None,
                   valid: Optional[torch.Tensor] = None):
    """window > 0: rolling_lin_reg; window == 0: recursive_lin_reg starting after `min_rows` rows."""
    p = X.shape[0]
    n = X.shape[1] if n is None else n
    q = p + int(add_bias)
    coeffs = coeffs if coeffs is not None else torch.empty((n, q), dtype=X.dtype, device=X.device)
    pred = pred if pred is not None else torch.empty(n, dtype=X.dtype, device=X.device)
    valid = valid if valid is not None else torch.empty(n, dtype=torch.uint8, device=X.device)
    fn = getattr(lib(), f"pdsb_dev_online_lin_reg_{_sfx(X)}")
    check(fn(_ptr(X), _ld(X), _ptr(y), n, p, int(add_bias), window, min_rows, int(skip), float(l2_reg), _ptr(coeffs),
             _ptr(pred), _ptr(valid), _stream()))
    return coeffs, pred, valid


def recursive_shard(X: torch.Tensor, y: torch.Tensor, min_rows: int, m0: Optional[torch.Tensor], row0: int,
                    add_bias: bool = False, l2_reg: float = 0.0, skip: bool = False):
    """recursive_lin_reg on the row shard that starts at global row `row0`; `m0` = float64 (p+2)^2 moments
    ([X | y | 1]) of all preceding rows (None for the first shard)."""
    p, n = X.shape
    q = p + int(add_bias)
    coeffs = torch.empty((n, q), dtype=X.dtype, device=X.device)
    pred = torch.empty(n, dtype=X.dtype, device=X.device)
    valid = torch.empty(n, dtype=torch.uint8, device=X.device)
    if m0 is not None:
        assert m0.dtype == torch.float64 and m0.is_contiguous() and m0.numel() == (p + 2) ** 2
    fn = getattr(lib(), f"pdsb_dev_recursive_shard_{_sfx(X)}")
    check(fn(_ptr(X), _ld(X), _ptr(y), n, p, int(add_bias), min_rows, int(skip), float(l2_reg),
             _ptr(m0) if m0 is not None else None, row0, _ptr(coeffs), _ptr(pred), _ptr(valid), _stream()))
    return coeffs, pred, valid


def glm(X: torch.Tensor, y: torch.Tensor, family: str = "normal", add_bias: bool = False, max_iter: int = 100,
        tol: float = 1e-8, n: Optional[int] = None) -> Tuple[torch.Tensor, int]:
    """GLM by IRLS on float64 tensors: X (p, ld), y (1, ld) or (ld,).  Returns (beta, n_iter): beta is a (p + add_bias,)
    float64 tensor on X's device, bias last; n_iter the number of weighted least-squares solves.  X's rows and y must
    start 16-byte aligned and ld must be even (torch allocations with an even ld are)."""
    if family not in GLM_FAMILIES:
        raise NotImplementedError(f"unknown GLM family {family!r}")
    p = X.shape[0]
    n = X.shape[1] if n is None else n
    yv = y.reshape(1, -1) if y.dim() == 1 else y
    beta = torch.empty(p + int(add_bias), dtype=torch.float64, device=X.device)
    it = C.c_int64(0)
    check(lib().pdsb_dev_glm_f64(_ptr(X), _ld(X), _ptr(yv), n, p, int(add_bias), GLM_FAMILIES[family], int(max_iter),
                                 float(tol), _ptr(beta), C.byref(it), _stream()))
    return beta, int(it.value)


FRAME_ROWS = 128


def frame_elems(n: int, ncols: int) -> int:
    return int(lib().pdsb_frame_elems(n, ncols))


def to_frame(Z: torch.Tensor, n: Optional[int] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Column-major (ncols, ld) float32 matrix -> row-blocked frame [block][column][128] (flat tensor)."""
    ncols = Z.shape[0]
    n = Z.shape[1] if n is None else n
    frame = out if out is not None else torch.empty(frame_elems(n, ncols), dtype=torch.float32, device=Z.device)
    check(lib().pdsb_dev_frame_from_colmajor_f32(_ptr(Z), _ld(Z), n, ncols, _ptr(frame), _stream()))
    return frame


def moments_frame(frame: torch.Tensor, n: int, ncols: int, xcol: int, p: int, ycol: int, t: int = 1,
                  mask: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    q1 = p + t + 1
    M = out if out is not None else torch.empty((q1, q1), dtype=torch.float64, device=frame.device)
    check(lib().pdsb_dev_moments_frame_f32(_ptr(frame), n, ncols, xcol, p, ycol, t, _ptr(mask), _ptr(M), _stream()))
    return M


def predict_frame(frame: torch.Tensor, n: int, ncols: int, xcol: int, p: int, ycol: int, t: int, beta: torch.Tensor,
                  status: Optional[torch.Tensor], add_bias: bool, pred: torch.Tensor, resid: torch.Tensor,
                  mask: Optional[torch.Tensor] = None, valid: Optional[torch.Tensor] = None,
                  ssr: Optional[torch.Tensor] = None):
    check(lib().pdsb_dev_predict_frame_f32(_ptr(frame), n, ncols, xcol, p, ycol, t, int(add_bias), _ptr(mask), _ptr(beta),
                                           _ptr(status), _ptr(pred), _ptr(resid), _ld(pred), _ptr(valid), _ptr(ssr),
                                           _stream()))
    return pred, resid


def launch_count() -> int:
    return int(lib().pdsb_kernel_launch_count())
