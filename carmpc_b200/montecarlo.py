"""Monte-Carlo closed loops with random noise, and the rows that say whether the true plant stayed safe.

``LoopNoise`` describes the process and measurement noise of ``BatchQP.closed_loop(..., noise=...)`` and
``BatchQP.closed_loop_disturbance(..., noise=...)``; ``plant_rows`` gives a controller's own state rows as a monitor for
the ``monitor=`` argument of the same calls.  The noise is drawn on the device (``carmpc_closed_loop_stochastic``,
Philox4x64-10 at counter (first_run + run, step, 0 / 1, 0), key (seed, 0)), so it depends only on the seed, the global run
id and the step: a run set split over calls or GPUs with ``first_run`` offsets draws what one call would.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from . import _capi


def _factor(a, name: str, dims: tuple) -> np.ndarray:
    """A std vector (diagonal factor) or a square factor, padded with zeros to 4 x 4."""
    a = np.asarray(a, dtype=np.float64)
    if a.ndim == 1 and a.shape[0] in dims:
        f = np.diag(a)
    elif a.ndim == 2 and a.shape[0] == a.shape[1] and a.shape[0] in dims:
        f = a
    else:
        shapes = " or ".join(f"({d},) / ({d}, {d})" for d in dims)
        raise ValueError(f"{name} must be a std vector or a factor of shape {shapes}, got {a.shape}")
    if not np.isfinite(f).all():
        raise ValueError(f"{name} must be finite")
    out = np.zeros((4, 4))
    out[:len(f), :len(f)] = f
    return out


@dataclass
class LoopNoise:
    """Gaussian noise of a closed loop.

    ``process``: (4,) std vector or (4, 4) factor ``Lw``; every step adds ``Lw z_w`` to the plant state after its Euler
    step.  ``measurement``: (3,) / (4,) std vector or (3, 3) / (4, 4) factor ``Lv`` (padded to 4 x 4); the controller sees
    ``s + Lv z_v`` (state feedback) or ``C s + (Lv z_v)[:3]`` (output feedback).  ``z_w``, ``z_v`` are standard normals.
    ``seed`` picks the stream, ``first_run`` is the global id of the call's run 0."""
    process: object
    measurement: object
    seed: int = 0
    first_run: int = 0

    def factors(self) -> tuple:
        """(Lw, Lv) as 4 x 4 float64 arrays."""
        return _factor(self.process, "process", (4,)), _factor(self.measurement, "measurement", (3, 4))

    def params(self) -> "_capi.LoopNoiseParams":
        """The ``carmpc_loop_noise`` struct of the C ABI."""
        if not 0 <= int(self.seed) < 1 << 64:
            raise ValueError("seed must be in [0, 2^64)")
        if int(self.first_run) < 0:
            raise ValueError("first_run must be >= 0")
        Lw, Lv = self.factors()
        p = _capi.LoopNoiseParams()
        p.seed = int(self.seed)
        p.first_run = int(self.first_run)
        p.Lw[:] = Lw.ravel().tolist()
        p.Lv[:] = Lv.ravel().tolist()
        return p


def plant_rows(controller, terminal_set: bool = False) -> np.ndarray:
    """The controller's state rows in absolute coordinates as (rows, 5) ``[A | b]``: its built-in rows
    (``state_const_A / b``: heading and speed limits), then the environment's (``env.constraints_A / b``: road edges,
    other cars), the rows ``MPC.state_constraint`` imposes on every predicted state; with ``terminal_set`` its terminal
    set follows."""
    A = [np.asarray(a, dtype=np.float64) for a in controller.state_const_A]
    b = [float(v) for v in controller.state_const_b]
    if controller.env is not None:
        A += [np.asarray(a, dtype=np.float64) for a in controller.env.constraints_A]
        b += [float(v) for v in controller.env.constraints_b]
    rows = np.hstack((np.vstack(A), np.asarray(b)[:, None]))
    if terminal_set:
        At, bt = controller.terminal_constraint()
        rows = np.vstack((rows, np.hstack((np.asarray(At, dtype=np.float64)[:, -4:], np.asarray(bt, dtype=np.float64)[:, None]))))
    return np.ascontiguousarray(rows)
