"""Condensed MPC problem in the parametric form the CUDA solver takes.

The reference states one QP per initial state (``lib/mpc.py:318-332`` / ``:461-475``):

    min_u 1/2 u'Hu + (h (x0 - x_ref))'u
    s.t.  A_term (T x0 + S u) <= b_term          terminal set on x(N)          (:324-326)
          [I; -I] u <= [ub; -lb]                 input box                     (:327-329)
          A_state (T x0 + S u) <= b_state        state rows on x(1..N)         (:330-332)

Everything except x0 / x_ref is shared by the whole batch.  This module turns a controller's matrices
into the arrays of ``carmpc_qp_create`` (include/carmpc.h):

    lo - Gx p  <=  G u  <=  hi - Gx p      (general rows; p = x0, lo = -inf for one-sided rows)
    lb <= u <= ub                           (box; identity rows never enter a matrix product)
    pre_lo <= Px p <= pre_hi                (rows whose G part is identically zero: they do not depend
                                             on u, so they are a pure feasibility test on x0)

Two exact reductions are applied, neither changes the feasible set or the minimiser:
  * a pair of rows that are exact negatives of each other (psi <= pi/8 and -psi <= pi/8, parallel
    facets of the terminal set) becomes one two-sided row;
  * rows with no dependence on u (x(1) and y(1): the first block row of S has zero position rows)
    are moved to the pre-check.
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np


@dataclass
class ParametricQP:
    N: int
    H: np.ndarray          # (n, n)
    F: np.ndarray          # (n, 4)    q = F (x0 - x_ref)
    G: np.ndarray          # (m, n)
    Gx: np.ndarray         # (m, 4)
    lo: np.ndarray         # (m,)  -inf where one-sided
    hi: np.ndarray         # (m,)
    lb: np.ndarray         # (n,)  -inf when the input box is disabled
    ub: np.ndarray         # (n,)
    Gc: np.ndarray         # (m,)  shift per unit of the scalar disturbance estimate (zeros without one)
    Px: np.ndarray         # (k, 4)
    Pc: np.ndarray         # (k,)
    pre_lo: np.ndarray     # (k,)
    pre_hi: np.ndarray     # (k,)
    goal: np.ndarray       # (4,)  default x_ref
    T: np.ndarray          # ((N+1)*4, 4)   kept for host-side post-processing (x_horizon)
    S: np.ndarray          # ((N+1)*4, n)
    rows_x: np.ndarray     # (m_all, (N+1)*4)  every one-sided state-space row (terminal first, then state)
    rows_b: np.ndarray     # (m_all,)
    # provenance of each general row: index into the one-sided stack (hi side, lo side or -1)
    src_hi: np.ndarray
    src_lo: np.ndarray
    # the same for the u-independent rows (certificate.to_one_sided); empty: none recorded
    pre_src_hi: np.ndarray = field(default_factory=lambda: np.zeros(0, dtype=np.int64))
    pre_src_lo: np.ndarray = field(default_factory=lambda: np.zeros(0, dtype=np.int64))

    @property
    def n(self) -> int:
        return self.H.shape[0]

    @property
    def m(self) -> int:
        return self.G.shape[0]


def _merge_opposites(M: np.ndarray, b: np.ndarray):
    """Fold rows r, s with M[s] == -M[r] (exactly) into lo <= M[r] . <= hi.  Duplicate directions keep the
    tighter bound.  Returns (rows, lo, hi, src_hi, src_lo)."""
    keys = {}
    rows, lo, hi, src_hi, src_lo = [], [], [], [], []
    for r in range(len(b)):
        row = M[r] + 0.0                        # normalise -0.0
        key = row.tobytes()
        neg = (-row + 0.0).tobytes()
        if key in keys:
            k = keys[key]
            if b[r] < hi[k]:
                hi[k], src_hi[k] = b[r], r
        elif neg in keys:
            k = keys[neg]
            if -b[r] > lo[k]:
                lo[k], src_lo[k] = -b[r], r
        else:
            keys[key] = len(rows)
            rows.append(row)
            hi.append(b[r])
            lo.append(-np.inf)
            src_hi.append(r)
            src_lo.append(-1)
    return (np.array(rows).reshape(len(rows), M.shape[1]), np.array(lo), np.array(hi),
            np.array(src_hi, dtype=np.int64), np.array(src_lo, dtype=np.int64))


def build_parametric_qp(controller, merge_rows: bool = True) -> ParametricQP:
    """Condense ``controller`` (an ``lib.mpc.MPC`` instance) with its enabled constraint blocks."""
    N, n = controller.N, controller.N * controller.nu
    T, S = controller.T, controller.S
    stack_A, stack_b = [], []
    if controller.terminal_constraint_bool:
        A, b = controller.terminal_constraint()
        stack_A.append(A)
        stack_b.append(b)
    if controller.state_constraint_bool:
        A, b = controller.state_constraint()
        stack_A.append(A)
        stack_b.append(b)
    if stack_A:
        rows_x = np.vstack(stack_A)
        rows_b = np.hstack(stack_b).astype(float)
    else:
        rows_x = np.zeros((0, (N + 1) * 4))
        rows_b = np.zeros(0)
    G_all = rows_x @ S
    Gx_all = rows_x @ T
    # constant-disturbance controllers predict x_ = T x0 + S u + ABd d (lib/mpc.py:631-637): one more column
    if hasattr(controller, "disturbance_response"):
        Gc_all = rows_x @ controller.disturbance_response()
    else:
        Gc_all = np.zeros(len(rows_b))

    stacked = np.hstack((G_all, Gx_all, Gc_all[:, None]))
    if merge_rows:
        M, lo, hi, src_hi, src_lo = _merge_opposites(stacked, rows_b)
    else:
        M, lo, hi = stacked, np.full(len(rows_b), -np.inf), rows_b.copy()
        src_hi, src_lo = np.arange(len(rows_b)), np.full(len(rows_b), -1)
    G, Gx, Gc = M[:, :n], M[:, n:n + 4], M[:, n + 4]
    param_only = ~np.any(G != 0.0, axis=1)

    if controller.input_constraint_bool:
        ub = np.tile(np.asarray(controller.input_upper, dtype=float), N)
        lb = np.tile(np.asarray(controller.input_lower, dtype=float), N)
    else:
        ub, lb = np.full(n, np.inf), np.full(n, -np.inf)

    keep = ~param_only
    return ParametricQP(
        N=N, H=np.array(controller.H, dtype=float), F=np.array(controller.h, dtype=float),
        G=np.ascontiguousarray(G[keep]), Gx=np.ascontiguousarray(Gx[keep]), lo=lo[keep], hi=hi[keep],
        Gc=np.ascontiguousarray(Gc[keep]), lb=lb, ub=ub, Px=np.ascontiguousarray(Gx[param_only]),
        Pc=np.ascontiguousarray(Gc[param_only]), pre_lo=lo[param_only], pre_hi=hi[param_only],
        goal=np.array(controller.goal, dtype=float), T=T, S=S, rows_x=rows_x, rows_b=rows_b,
        src_hi=src_hi[keep], src_lo=src_lo[keep], pre_src_hi=src_hi[param_only], pre_src_lo=src_lo[param_only])
