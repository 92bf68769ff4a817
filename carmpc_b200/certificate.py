"""Certificates of batched QP solves, and an independent device checker for them.

``BatchQP.solve(..., want_certificate=True)`` returns one float64 row per sample in the row space of the handle: the
general rows of ``ParametricQP`` (merged, u-independent rows removed), the box rows, then the u-independent rows.
``to_one_sided`` maps such rows onto the reference's own stack (``rows_x``: terminal rows, then state rows, each
``rows_x[i] (T x0 + S u) <= rows_b[i]``) plus the box, where a proof can be checked without the solver's setup by
``QPChecker`` (``carmpc_qp_checker_create`` / ``carmpc_qp_check``).

Sign convention everywhere: positive means "against the upper bound", negative "against the lower bound".  In a
one-sided stack every valid entry is therefore >= 0.
"""
from __future__ import annotations

import ctypes

import numpy as np

from . import _capi
from ._capi import check

#: thresholds of a passing status-0 check (the columns of ``QPChecker.check``)
KKT_TOL = {"primal": 1e-8, "stationarity": 1e-9, "wrong_side": 1e-9, "complementarity": 1e-8}
#: a Farkas ray proves infeasibility when its support value is below -SUPPORT_MARGIN * scale (kSupportMargin of
#: qp_check.cu, which derives it) and no mass sits against an infinite bound
SUPPORT_MARGIN = 4e-12
#: the exported box part of a ray must equal -G'y_g to this relative accuracy (the checker completes its own)
BOX_TOL = 1e-9


def _torch():
    import torch
    return torch


def _signed_index_add(torch, out, vals, src_hi, src_lo):
    """Scatter the columns of ``vals`` (two-sided rows) onto one-sided rows: a positive entry onto its upper row
    ``src_hi``, a negative one as its magnitude onto its lower row ``src_lo``; a negative entry of a row without a lower
    row stays negative on ``src_hi`` (a wrong sign the checker reports)."""
    if vals.shape[1] == 0:
        return
    dev = vals.device
    hi = torch.as_tensor(np.asarray(src_hi, dtype=np.int64), device=dev)
    lo = torch.as_tensor(np.asarray(src_lo, dtype=np.int64), device=dev)
    pos, neg = vals.clamp(min=0.0), vals.clamp(max=0.0)
    has_lo = lo >= 0
    out.index_add_(1, hi, pos + torch.where(has_lo, torch.zeros_like(neg), neg))
    if bool(has_lo.any()):
        out.index_add_(1, lo[has_lo], -neg[:, has_lo])


def to_one_sided(pq, cert):
    """(B, m + n + k) handle-space certificate rows -> (B, len(pq.rows_b) + n) rows of the one-sided stack ``rows_x``
    followed by the (two-sided) box.  A row that the merge dropped for a tighter duplicate gets 0."""
    torch = _torch()
    m, n, k = pq.m, pq.n, len(pq.pre_hi)
    if cert.dim() != 2 or cert.shape[1] != m + n + k:
        raise ValueError(f"certificate rows must have m + n + k = {m + n + k} entries")
    if k > 0 and len(pq.pre_src_hi) != k:
        raise ValueError("this ParametricQP carries no provenance of its u-independent rows (pre_src_hi / pre_src_lo)")
    R = len(pq.rows_b)
    out = torch.zeros((cert.shape[0], R + n), dtype=cert.dtype, device=cert.device)
    _signed_index_add(torch, out, cert[:, :m], pq.src_hi, pq.src_lo)
    _signed_index_add(torch, out, cert[:, m + n:], pq.pre_src_hi, pq.pre_src_lo)
    out[:, R:] = cert[:, m:m + n]
    return out


class QPChecker:
    """Float64 KKT / Farkas checker of a QP in the general two-sided form (``carmpc_qp_checker_create``)

        min 1/2 u'Hu + (F (x0 - xref))'u    lo - Gx x0 - Gc c <= G u <= hi - Gx x0 - Gc c ,   lb <= u <= ub

    It shares nothing with the solver: pass the reference's own matrices (``from_reference``) to check a solve against
    the problem the reference states."""

    def __init__(self, H, F, G, Gx, lo, hi, lb, ub, Gc=None):
        self._lib = _capi.load()
        self._h = ctypes.c_void_p()
        f = lambda a: np.ascontiguousarray(a, dtype=np.float64)
        H, F, lb, ub = f(H), f(F), f(lb).ravel(), f(ub).ravel()
        n = H.shape[0]
        G = f(G).reshape(-1, n)
        R = G.shape[0]
        Gx, lo, hi = f(Gx).reshape(R, 4), f(lo).ravel(), f(hi).ravel()
        Gc = None if Gc is None else f(Gc).ravel()
        if H.shape != (n, n) or F.shape != (n, 4) or lb.shape != (n,) or ub.shape != (n,) or lo.shape != (R,) \
                or hi.shape != (R,) or (Gc is not None and Gc.shape != (R,)):
            raise ValueError("inconsistent shapes")
        self.n, self.R = n, R
        self._keep = (H, F, G, Gx, Gc, lo, hi, lb, ub)
        p = lambda a: None if a is None or a.size == 0 else _capi.ptr(a)
        check(self._lib.carmpc_qp_checker_create(n, R, p(H), p(F), p(G), p(Gx), p(Gc), p(lo), p(hi), p(lb), p(ub),
                                                 ctypes.byref(self._h)))

    @classmethod
    def from_reference(cls, pq, Gc=None) -> "QPChecker":
        """The one-sided stack of ``pq`` as the reference states it: ``rows_x (T x0 + S u) <= rows_b`` and the box.
        ``Gc``: per one-sided row, the shift per unit of the disturbance (``rows_x @ ABd``), if any."""
        R = len(pq.rows_b)
        return cls(pq.H, pq.F, pq.rows_x @ pq.S, pq.rows_x @ pq.T, np.full(R, -np.inf), pq.rows_b, pq.lb, pq.ub, Gc=Gc)

    def close(self):
        if getattr(self, "_h", None):
            self._lib.carmpc_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, x0, x_ref, status, u_full, cert, c=None, stream=None):
        """Per sample 4 float64 (CUDA tensor (B, 4)); see ``carmpc_qp_check`` for the columns.  ``x0``: (4, B) SoA,
        ``cert``: (B, R + n) in this checker's row space (``to_one_sided`` for a one-sided reference stack)."""
        torch = _torch()
        B = x0.shape[1]
        for name, t, shape, dt in (("x0", x0, (4, B), torch.float64), ("status", status, (B,), torch.int32),
                                   ("u_full", u_full, (B, self.n), torch.float64),
                                   ("cert", cert, (B, self.R + self.n), torch.float64)):
            if not (t.is_cuda and t.dtype == dt and tuple(t.shape) == shape and t.is_contiguous()):
                raise ValueError(f"{name} must be a contiguous {dt} CUDA tensor of shape {shape}")
        if c is not None and not (c.is_cuda and c.dtype == torch.float64 and c.numel() == B and c.is_contiguous()):
            raise ValueError("c must be a contiguous float64 CUDA tensor of B entries")
        xref = np.ascontiguousarray(x_ref, dtype=np.float64)
        out = torch.empty((B, 4), dtype=torch.float64, device=x0.device)
        s = None if stream is None else ctypes.c_void_p(stream.cuda_stream)
        check(self._lib.carmpc_qp_check(self._h, x0.data_ptr(), _capi.ptr(xref), None if c is None else c.data_ptr(), B,
                                        status.data_ptr(), u_full.data_ptr(), cert.data_ptr(), out.data_ptr(), s))
        return out


def passes(status, resid, tol=None):
    """Boolean per sample: status 0 within ``tol`` (default ``KKT_TOL``) on all four columns, status 1 a proof whose
    exported box part matches (``BOX_TOL``); status 2 never passes.  Works on numpy arrays and torch tensors alike."""
    tol = KKT_TOL if tol is None else tol
    r = [resid[:, i] for i in range(4)]
    kkt = (r[0] <= tol["primal"]) & (r[1] <= tol["stationarity"]) & (r[2] <= tol["wrong_side"]) & \
        (r[3] <= tol["complementarity"])
    farkas = (r[3] == 0) & (r[0] < -SUPPORT_MARGIN * r[1]) & (r[2] <= BOX_TOL)
    return ((status == 0) & kkt) | ((status == 1) & farkas)
