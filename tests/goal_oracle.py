"""CPU restatement of closed loops that stop at a goal (carmpc_closed_loop with a goal), built on
``oracle/carmpc_oracle.py`` (used unchanged).

TEST INFRASTRUCTURE ONLY.  ``closed_loop`` is ``oracle.carmpc_oracle.closed_loop`` with the goal test of the reference's
loops (examples/run_MPCStateFB.py): after the plant step and the controller step of step k, a run whose state is inside
the goal rows stops, unless its QP of step k was not solved, which stops it as a failure first.  ``outcome_from_traj``
derives the same verdicts from the trajectory of a loop without a goal.
"""
from __future__ import annotations

import numpy as np

from oracle.carmpc_oracle import C_OUT, observer_step, plant_step


def inside(rows, s):
    """(n,) bool: the states s (n, 4) are finite and satisfy every row [a | b] (rows, 5)."""
    rows = np.asarray(rows, dtype=float)
    s = np.atleast_2d(np.asarray(s, dtype=float))
    with np.errstate(invalid="ignore"):
        lhs = s @ rows[:, :4].T
        return np.isfinite(s).all(1) & (lhs <= rows[:, 4][None, :]).all(1)


def closed_loop(qp, x_init, steps, output_feedback, solve, rows):
    """The loop of ``oracle.carmpc_oracle.closed_loop`` with the goal: returns final states (R, 4), fail_step,
    arrival_step (R,) int32 (-1: none) and the state trajectory (steps, R, 4); stopped runs keep their state."""
    x = np.array(x_init, dtype=float)
    Bn = len(x)
    xhat = x.copy()
    u = np.zeros((Bn, 2))
    fail = np.full(Bn, -1, dtype=np.int32)
    arrival = np.full(Bn, -1, dtype=np.int32)
    traj = np.zeros((steps, Bn, 4))
    A, Bm = qp.A, qp.B
    for k in range(steps):
        alive = (fail < 0) & (arrival < 0)
        idx = np.flatnonzero(alive)
        if len(idx):
            x[idx] = plant_step(x[idx], u[idx])
            if output_feedback:
                xhat[idx] = observer_step(A, Bm, xhat[idx], u[idx], x[idx] @ C_OUT.T)
                est = xhat
            else:
                est = x
            u_new, st = solve(est[idx])
            bad = st != 0
            arrived = ~bad & inside(rows, x[idx])
            fail[idx[bad]] = k
            arrival[idx[arrived]] = k
            take = ~bad & ~arrived
            u[idx[take]] = u_new[take]
        traj[k] = x
    return x, fail, arrival, traj


def outcome_from_traj(traj, fail, rows):
    """(arrival_step, fail_step) a loop with the goal ``rows`` gives, from the trajectory (steps, R, 4) and fail_step of
    the same loop without a goal: the first step k at which the run was running (k <= fail, or fail < 0) and its state
    inside is its arrival, unless its QP of that step was not solved (k == fail), which stays a failure."""
    traj = np.asarray(traj, dtype=float)
    fail = np.asarray(fail)
    steps, R = traj.shape[:2]
    ins = inside(rows, traj.reshape(-1, 4)).reshape(steps, R)
    k = np.arange(steps)[:, None]
    ins &= (fail[None, :] < 0) | (k <= fail[None, :])
    first = np.where(ins.any(0), ins.argmax(0), -1)
    arrival = np.where((first >= 0) & (first != fail), first, -1).astype(np.int32)
    fail_out = np.where(arrival >= 0, -1, fail).astype(np.int32)
    return arrival, fail_out


def face_distance(traj, rows):
    """(steps, R): the smallest |b - a . s| over the rows, the distance (in row units) of each state to a goal face."""
    rows = np.asarray(rows, dtype=float)
    t = np.asarray(traj, dtype=float)
    return np.abs(rows[:, 4] - t @ rows[:, :4].T).min(-1)
