"""CPU oracle of the disturbance-estimating controller (MPCOutputFBWithDisturbance): a plain numpy restatement of its
closed loop, built on ``oracle/carmpc_oracle.py`` (whose functions it uses unchanged).

TEST INFRASTRUCTURE ONLY.  The loop follows examples/run_MPCOutputFB.py:29-41 with the augmented observer of
lib/mpc.py:362-366; each step's QP is solved exactly (``qp_solve_exact``) on the bounds shifted by rows_x @ ABd * d^.
"""
from __future__ import annotations

import numpy as np

from oracle.carmpc_oracle import CondensedQP, plant_step, state_constraint, terminal_constraint
def disturbance_response(A, Bd, N):
    """ABd ((N+1)*4,) with x_ = T x0 + S u + ABd d: block k is sum_{i<k} A^i Bd (reference :631-635)."""
    out = np.zeros((N + 1, 4))
    acc = np.zeros(4)
    ak = np.asarray(Bd, dtype=float).copy()
    for k in range(1, N + 1):
        acc = acc + ak
        out[k] = acc
        ak = A @ ak
    return out.ravel()


class DisturbedQP(CondensedQP):
    """The condensed QP with the disturbance estimate d as a fifth parameter: states are (x0, d), and
    G u <= w - Gx x0 - Gd d with Gd = rows_x @ ABd (the input box does not move).  ``qp_solve_exact`` solves it as it
    stands: pass (B, 5) parameters and a 5-entry x_ref whose last entry is 0 (d does not enter the cost)."""

    def __init__(self, env_name, N, term_Ab, Bd, use_terminal=True, use_input=True, use_state=True):
        super().__init__(env_name, N, term_Ab, use_terminal, use_input, use_state)
        ABd = disturbance_response(self.A, Bd, N)
        blocks = []
        if use_terminal:
            blocks.append(terminal_constraint(term_Ab, N)[0] @ ABd)
        if use_input:
            blocks.append(np.zeros(4 * N))
        if use_state:
            blocks.append(state_constraint(env_name, N)[0] @ ABd)
        Gd = np.hstack(blocks) if blocks else np.zeros(0)
        self.Gx = np.hstack((self.Gx, Gd[:, None]))
        self.h = np.hstack((self.h, np.zeros((self.n, 1))))


def disturbance_observer_step(A, B, C, Bd, Cd, L1, L2, xhat, dhat, u_prev, y):
    """Batched MPCOutputFBWithDisturbance.luenberger_observer: xhat (B, 4), dhat (B,), u_prev (B, 2), y (B, 3)."""
    innov = y - xhat @ C.T - dhat[:, None] * Cd[None, :]
    x_new = xhat @ A.T + dhat[:, None] * Bd[None, :] + u_prev @ B.T + innov @ L1.T
    d_new = dhat + innov @ L2
    return x_new, d_new


def closed_loop_disturbance(A, B, C, Bd, Cd, L1, L2, x_init, steps, solve, Bd_plant=None, Cd_plant=None,
                            d_plant=None, xhat_init=None, dhat_init=None):
    """Monte-Carlo closed loop of the disturbance controller, order of examples/run_MPCOutputFB.py:29-41: plant step
    with the previous input, then the true disturbance (s += Bd_plant d_r, y = C s + Cd_plant d_r), augmented observer,
    QP at (x^, d^).  ``solve(x (B, 4), d (B,)) -> (u0 (B, 2), status)``.  A run stops at its first unsolved step.
    Returns final states, final d^, fail_step (-1 = none), the state trajectory (steps, R, 4) and d^ per step (steps, R)."""
    A, B, C = (np.asarray(a, dtype=float) for a in (A, B, C))
    Bd, Cd, L2 = (np.asarray(a, dtype=float).ravel() for a in (Bd, Cd, L2))
    L1 = np.asarray(L1, dtype=float).reshape(4, 3)
    x = np.array(x_init, dtype=float)
    R = len(x)
    Bp = np.zeros(4) if Bd_plant is None else np.asarray(Bd_plant, dtype=float).ravel()
    Cp = np.zeros(3) if Cd_plant is None else np.asarray(Cd_plant, dtype=float).ravel()
    dr = np.zeros(R) if d_plant is None else np.asarray(d_plant, dtype=float).ravel()
    xhat = x.copy() if xhat_init is None else np.array(xhat_init, dtype=float)
    dhat = np.zeros(R) if dhat_init is None else np.array(dhat_init, dtype=float)
    u = np.zeros((R, 2))
    fail = np.full(R, -1, dtype=np.int32)
    traj = np.zeros((steps, R, 4))
    dlog = np.zeros((steps, R))
    for k in range(steps):
        alive = fail < 0
        s = plant_step(x[alive], u[alive]) + dr[alive, None] * Bp[None, :]
        x[alive] = s
        y = s @ C.T + dr[alive, None] * Cp[None, :]
        xhat[alive], dhat[alive] = disturbance_observer_step(A, B, C, Bd, Cd, L1, L2, xhat[alive], dhat[alive], u[alive], y)
        idx = np.flatnonzero(alive)
        if len(idx):
            u_new, st = solve(xhat[idx], dhat[idx])
            bad = st != 0
            fail[idx[bad]] = k
            u[idx[~bad]] = u_new[~bad]
        traj[k] = x
        dlog[k] = dhat
    return x, dhat, fail, traj, dlog
