"""Numpy restatement of the sensitivity kernel (carmpc_b200/csrc/qp_sensitivity.cu), for the tests.

It works on a QP in the general two-sided form of ``carmpc_qp_checker_create`` (the reference's one-sided stack is lo =
-inf), u-independent rows included as general rows whose G part is zero:

    min 1/2 u'Hu + (F (x0 - xref))'u    lo - Gx x0 - Gc c <= G u <= hi - Gx x0 - Gc c ,   lb <= u <= ub

with one certificate row per sample in that row space (general rows, then box; ``certificate.to_one_sided`` maps the
solver's rows onto the reference's stack).  Unlike the kernel it uses no Schur complement and no handle table: the
derivatives come from the full KKT system [H A_S'; A_S 0] solved by LU.  Flags follow the same rules and tolerances.
"""
import numpy as np

FEAS_TOL = 1e-8          # kFeasTol of the polish
SIGN_TOL = 1e-9          # kSignTol of the polish
PIVOT_SKIP = 1e-11       # a row whose H^-1-metric residual against the rows before it is below this share is dependent
MAX_ACTIVE = 64
DERIVATIVE, WEAK, DEPENDENT, TOO_MANY_ROWS = 1, 2, 4, 8


def distinct_rows(G, Gx, Gc, lo, hi):
    """False for a row that repeats an earlier one exactly (same G, Gx, Gc and bounds): the same half-space stated twice.
    The library's setup keeps one of them (condensed.py) and ``to_one_sided`` puts the multiplier on the first."""
    seen, keep = set(), np.ones(len(hi), dtype=bool)
    for i in range(len(hi)):
        key = np.concatenate((G[i], Gx[i], [Gc[i], lo[i], hi[i]])).tobytes()
        keep[i] = key not in seen
        seen.add(key)
    return keep


def sensitivity_numpy(H, F, G, Gx, lo, hi, lb, ub, x0, u, cert, status=None, Gc=None, c=None, rows=None, cond=None,
                      term_scale=None):
    """x0 (B, 4), u (B, n), cert (B, R + n).  Returns jac (B, rows, 5), grad (B, 5), flags (B,) like
    ``BatchQP.sensitivity``; columns are d/d(x, y, psi, v, c).  ``cond`` (optional (B,) array) receives the 2-norm
    condition number of M = A_S H^-1 A_S' over the independent rows (1 for an empty S).  ``term_scale`` (optional (B, 5)
    array) receives, per column, max_r (|Uu_rk| + sum_a |(A_S H^-1)_ar dlam_ak|): the size of the terms the kernel's
    J = Uu - (A_S H^-1)' dlam adds up, hence of its rounding error, also where they cancel to a column that is 0."""
    x0, u, cert = np.atleast_2d(x0), np.atleast_2d(u), np.atleast_2d(cert)
    B, n = u.shape
    R = G.shape[0]
    rows = n if rows is None else rows
    Gc = np.zeros(R) if Gc is None else np.asarray(Gc, dtype=float)
    c = np.zeros(B) if c is None else np.asarray(c, dtype=float)
    status = np.zeros(B, dtype=np.int32) if status is None else np.asarray(status)
    keep = distinct_rows(G, Gx, Gc, lo, hi)
    A_all = np.vstack((G, np.eye(n)))
    Ax_all = np.vstack((Gx, np.zeros((n, 4))))
    Ac_all = np.concatenate((Gc, np.zeros(n)))
    lo_all, hi_all = np.concatenate((lo, lb)), np.concatenate((hi, ub))
    Hinv = np.linalg.inv(H)
    jac = np.full((B, rows, 5), np.nan)
    grad = np.full((B, 5), np.nan)
    flags = np.zeros(B, dtype=np.int32)
    for b in range(B):
        if status[b] != 0:
            continue
        y = cert[b]
        S = np.flatnonzero(y != 0)
        lam = y[S]
        grad[b, :4] = F.T @ u[b] + Ax_all[S].T @ lam
        grad[b, 4] = Ac_all[S] @ lam
        if len(S) > MAX_ACTIVE:
            flags[b] = TOO_MANY_ROWS
            continue
        # classification: multipliers on S, every other row against its bounds
        weak = bool(np.any(~(np.abs(lam) > SIGN_TOL * (1.0 + np.abs(lam).max(initial=0.0)))))
        t = A_all @ u[b] + Ax_all @ x0[b] + Ac_all * c[b]
        out = np.ones(R + n, dtype=bool)
        out[S] = False
        out[:R] &= keep
        with np.errstate(invalid="ignore"):
            at = (t >= hi_all - FEAS_TOL) | (t <= lo_all + FEAS_TOL)
        weak = weak or bool(np.any(at & out))
        # independent subset in row order: the residual of each row against the rows kept before it, in the H^-1 metric
        AS = A_all[S]
        Msel = AS @ Hinv @ AS.T
        sel = []
        for a in range(len(S)):
            d0 = Msel[a, a]
            d = d0 - (Msel[a, sel] @ np.linalg.solve(Msel[np.ix_(sel, sel)], Msel[sel, a]) if sel else 0.0)
            if d > PIVOT_SKIP * d0:
                sel.append(a)
        if cond is not None:
            cond[b] = np.linalg.cond(Msel[np.ix_(sel, sel)]) if sel else 1.0
        sel = S[sel]
        dependent = len(sel) < len(S)
        # full KKT system [H A'; A 0] [du; dlam] = -[F e_k; Gx e_k] (k < 4), -[0; Gc] (k = 4)
        k = len(sel)
        AS = A_all[sel]
        K = np.zeros((n + k, n + k))
        K[:n, :n], K[:n, n:], K[n:, :n] = H, AS.T, AS
        rhs = np.zeros((n + k, 5))
        rhs[:n, :4] = -F
        rhs[n:, :4] = -Ax_all[sel]
        rhs[n:, 4] = -Ac_all[sel]
        sol = np.linalg.solve(K, rhs)
        jac[b] = sol[:rows]
        if term_scale is not None:
            Uu = np.hstack((-Hinv @ F, np.zeros((n, 1))))
            term_scale[b] = (np.abs(Uu) + np.abs(AS @ Hinv).T @ np.abs(sol[n:]))[:rows].max(axis=0)
        flags[b] = (WEAK if weak else 0) | (DEPENDENT if dependent else 0) | (DERIVATIVE if not (weak or dependent) else 0)
    return jac, grad, flags


def reference_stack(d, Gc=None):
    """The reference's one-sided stack from a ``tests/golden/qp_*.npz``: (H, F, G, Gx, lo, hi, lb, ub, Gc)."""
    n = d["S"].shape[1]
    A = np.vstack((d["At"], d["As"]))
    G, Gx, hi = A @ d["S"], A @ d["T"], np.hstack((d["bt"], d["bs"]))
    bi = d["bi"]
    return d["H"], d["h"], G, Gx, np.full(len(hi), -np.inf), hi, -bi[n:], bi[:n], (None if Gc is None else A @ Gc)
