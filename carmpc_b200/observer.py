"""Gains of the augmented (state + constant disturbance) observer of ``MPCOutputFBWithDisturbance``.

The controller estimates a scalar constant disturbance d beside the state (``lib/mpc.py:362-366``):

    i = y - C x^ - Cd d^ ,   x^' = A x^ + Bd d^ + B u + L1 i ,   d^' = d^ + L2 . i

i.e. the predictor form of the augmented model  A^ = [[A, Bd], [0, 1]],  C^ = [C, Cd]  with gain L^ = [L1; L2'].  Its
estimation error evolves with A^ - L^ C^.  The reference hard-codes L1 (the plain observer's gain) and L2 = [1, 1, 1]; with
its Bd = 1_4, Cd = 1_3 and the shipped A, C that matrix has spectral radius 3.31, so the estimate diverges.  Reproducing
the reference takes ``reference_disturbance_gains``; running the offset-free experiment the controller was written for
takes a stable gain, e.g. ``augmented_observer_gain`` (steady-state Kalman predictor gain).
"""
from __future__ import annotations

import numpy as np
from scipy.linalg import solve_discrete_are


def augmented_model(A, C, Bd, Cd):
    """(A^ (5, 5), C^ (3, 5)) of the state + constant-disturbance model."""
    A = np.asarray(A, dtype=float)
    C = np.asarray(C, dtype=float)
    Bd = np.asarray(Bd, dtype=float).reshape(4)
    Cd = np.asarray(Cd, dtype=float).reshape(3)
    A_hat = np.zeros((5, 5))
    A_hat[:4, :4] = A
    A_hat[:4, 4] = Bd
    A_hat[4, 4] = 1.0
    C_hat = np.hstack((C, Cd[:, None]))
    return A_hat, C_hat


def observer_error_radius(A, C, Bd, Cd, L1, L2) -> float:
    """Spectral radius of A^ - L^ C^: below 1 the estimate of a constant disturbance converges."""
    A_hat, C_hat = augmented_model(A, C, Bd, Cd)
    L_hat = np.vstack((np.asarray(L1, dtype=float).reshape(4, 3), np.asarray(L2, dtype=float).reshape(1, 3)))
    return float(np.max(np.abs(np.linalg.eigvals(A_hat - L_hat @ C_hat))))


def reference_disturbance_gains(ctl):
    """``(Bd (4,), Cd (3,), L1 (4, 3), L2 (3,))`` of an ``MPCOutputFBWithDisturbance`` as float64 arrays (the reference's
    hard-coded values unless the caller changed them)."""
    return (np.asarray(ctl.Bd, dtype=float).reshape(4).copy(), np.asarray(ctl.Cd, dtype=float).reshape(3).copy(),
            np.asarray(ctl.L1, dtype=float).reshape(4, 3).copy(), np.asarray(ctl.L2, dtype=float).reshape(3).copy())


def augmented_observer_gain(A, C, Bd, Cd, W, V):
    """Steady-state predictor gain  L^ = A^ P C^' (C^ P C^' + V)^-1  of the augmented model, P from
    ``solve_discrete_are(A^', C^', W, V)``; W (5, 5) is the process noise of (x, d), V (3, 3) the measurement noise.
    Returns ``(L1 (4, 3), L2 (3,))``.  Raises ``ValueError`` when the augmented model is not detectable (e.g. a
    disturbance that neither moves the state nor shows in the output)."""
    A_hat, C_hat = augmented_model(A, C, Bd, Cd)
    W = np.asarray(W, dtype=float)
    V = np.asarray(V, dtype=float)
    try:
        P = solve_discrete_are(A_hat.T, C_hat.T, W, V)
    except (np.linalg.LinAlgError, ValueError) as exc:
        raise ValueError(f"no stabilising observer gain for this disturbance model: {exc}") from exc
    L_hat = A_hat @ P @ C_hat.T @ np.linalg.inv(C_hat @ P @ C_hat.T + V)
    return L_hat[:4].copy(), L_hat[4].copy()
