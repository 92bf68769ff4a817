"""Region of attraction of an MPC controller from its sampled feasibility map (SURVEY 8f-2).

The reference's exact route to the feasible set of the condensed QP is the Fourier-Motzkin projection of
``lib/in_adm_set.py:4-77``, which nothing calls because it is doubly exponential in the number of inputs
(2N = 40 for the shipped horizon).  Its sampled statement is what the GPU path produces anyway: one feasibility
flag per initial state (``BatchQP.solve`` status, i.e. ``OutsideTheRegionOfAttractionError`` of ``lib/mpc.py:336``
per state).  This module turns such a map into an H-representation ``A x <= b`` in the ``terminal_sets/*.npy``
conventions (absolute coordinates, unit-norm rows):

* ``feasibility_map(controller, axes)``       - flags of a tensor grid of initial states, solved on the GPU;
* ``boundary_layer(flags, shape)``            - feasible grid points with an infeasible (or missing) neighbour: the only
                                                candidates for hull vertices, a few percent of the grid;
* ``hull_polytope(points)``                   - convex hull -> merged, unit-normalised facets;
* ``region_of_attraction(controller, axes)``  - the three above in sequence;
* ``exact_feasible_set(G, Gx, w)``            - Fourier-Motzkin with LP redundancy removal after every elimination
                                                (tiny horizons only; the cross-check of the tests);
* ``closed_loop_map(controller, axes)``       - the region of attraction by closed-loop convergence (the paper's
                                                criterion): the nonlinear bicycle under the MPC law from every grid point,
                                                run on the GPU until it reaches the goal, its QP fails, or the steps end.

The feasible set F = {x0 : exists u, G u <= w - Gx x0} is convex, so  hull(feasible samples) is an inner
approximation of F and no infeasible sample may lie inside it - the property the tests check at every size.  The
closed-loop map is not convex in general, so it is returned as flags only, never hulled.
"""
from __future__ import annotations

from typing import Optional, Sequence

import numpy as np

from .lib import in_adm_set
from .lib.polytope_ops import Polytope, reduce as reduce_polytope


def default_seed_block(axes: Sequence[np.ndarray], max_step=(0.8, 0.5, 0.0, 0.0)) -> tuple:
    """Lattice block (points per axis) for the seeded solve: as many grid steps as fit into ``max_step`` state units
    along x and y (neighbours within ~0.75 m along the road / ~0.5 m across share their active set on the shipped
    problems: measured on the config-3 grid, blocks of 3 x 8 points = 0.75 m x 0.48 m are the fastest); psi and v are
    not blocked (their grids are coarse)."""
    block = []
    for a, span in zip(axes, max_step):
        a = np.asarray(a, dtype=float)
        step = float(np.abs(np.diff(a)).mean()) if len(a) > 1 else 0.0
        block.append(int(min(16, max(1, np.floor(span / step + 1e-9)))) if step > 0 and span > 0 else 1)
    return tuple(block)


def feasibility_map(controller, axes: Sequence[np.ndarray], x_ref=None, batch_solver=None, seeded: bool = True,
                    block=None, undecided: str = "raise") -> np.ndarray:
    """Feasibility flag of every point of the tensor grid ``axes`` (C order, x slowest ... v fastest): True where the
    controller's QP is feasible.  Solved on the GPU (no CPU fallback).  ``seeded`` (default) solves only a sub-lattice
    of anchors cold and certifies every other point from its anchor's active set / Farkas certificate
    (``carmpc_qp_solve`` with seeds: same flags, 1.7 - 4.6 x faster on 10^6-point maps).

    Every True is backed by a float64 KKT certificate and every False by a float64 Farkas certificate.  A point the
    solver could prove neither way (status 2: degenerate states within ~1e-7 of the boundary of the region) is not
    silently counted as outside: ``undecided`` = "raise" (default, as ``MPC.step`` does for the same status),
    "outside" or "inside"."""
    from .batch import BatchQP
    bq = batch_solver if batch_solver is not None else BatchQP.from_controller(controller)
    blk = None
    if seeded and bq.opts.polish:
        blk = tuple(int(v) for v in block) if block is not None else default_seed_block(axes)
    res = bq.solve_map_host(axes, block=blk, x_ref=x_ref, want_u0=False, want_objective=False)
    flags = res.status == 0
    n_undecided = int((res.status == 2).sum())
    if n_undecided:
        if undecided == "raise":
            raise RuntimeError(f"feasibility_map: {n_undecided} of {len(flags)} grid points are undecided (QP status 2); "
                               "pass undecided='outside' or 'inside' to classify them")
        if undecided == "inside":
            flags = flags | (res.status == 2)
        elif undecided != "outside":
            raise ValueError("undecided must be 'raise', 'outside' or 'inside'")
    return flags


def boundary_layer(flags: np.ndarray, shape: Sequence[int]) -> np.ndarray:
    """Flat indices of the feasible grid points that have an infeasible neighbour along some axis or sit on the edge
    of the grid.  Every vertex of the hull of the feasible points is among them."""
    f = np.asarray(flags, dtype=bool).reshape(shape)
    interior = f.copy()
    for ax, d in enumerate(shape):
        if d == 1:
            continue
        lo = [slice(None)] * len(shape)
        hi = [slice(None)] * len(shape)
        lo[ax], hi[ax] = slice(0, d - 1), slice(1, d)
        nb = np.zeros_like(f)
        nb[tuple(hi)] = f[tuple(lo)]                 # neighbour at index - 1 (False on the edge)
        interior &= nb
        nb = np.zeros_like(f)
        nb[tuple(lo)] = f[tuple(hi)]                 # neighbour at index + 1
        interior &= nb
    return np.flatnonzero(f & ~interior)


def hull_polytope(points: np.ndarray, merge_tol: float = 1e-9) -> tuple[np.ndarray, np.ndarray]:
    """Convex hull of ``points`` (k, d) as ``A x <= b`` with unit-norm rows; coplanar simplicial facets are merged.
    Degenerate (lower-dimensional) point sets are handled by hulling in the affine span and adding the equalities
    as pairs of opposite rows."""
    from scipy.spatial import ConvexHull
    P = np.unique(np.asarray(points, dtype=float), axis=0)
    if len(P) == 0:
        raise ValueError("no feasible sample: empty region of attraction")
    d = P.shape[1]
    centre = P.mean(axis=0)
    U, s, Vt = np.linalg.svd(P - centre, full_matrices=True)
    scale = max(float(s[0]) if len(s) else 0.0, 1.0)
    rank = int(np.sum(s > 1e-9 * scale))
    basis, normal = Vt[:rank], Vt[rank:]
    rows_A, rows_b = [], []
    if rank == 0:
        pass
    elif rank == 1:
        t = (P - centre) @ basis[0]
        rows_A += [basis[0], -basis[0]]
        rows_b += [t.max() + basis[0] @ centre, -t.min() - basis[0] @ centre]
    else:
        Y = (P - centre) @ basis.T
        eq = ConvexHull(Y).equations                 # [normal | offset], normal' y + offset <= 0, unit normals
        key = np.round(eq / merge_tol).astype(np.int64) if merge_tol > 0 else eq
        _, first = np.unique(key, axis=0, return_index=True)
        eq = eq[np.sort(first)]
        An = eq[:, :-1] @ basis                      # back to the ambient space (rows stay unit-norm)
        rows_A += list(An)
        rows_b += list(-eq[:, -1] + An @ centre)
    for nrm in normal:                               # the affine span itself
        rows_A += [nrm, -nrm]
        rows_b += [nrm @ centre, -(nrm @ centre)]
    return np.array(rows_A).reshape(-1, d), np.array(rows_b)


def region_of_attraction(controller, axes: Sequence[np.ndarray], x_ref=None, batch_solver=None,
                         save_path: Optional[str] = None):
    """Sampled region of attraction of ``controller`` over the tensor grid ``axes``.  Returns ``(A, b, flags)``;
    ``save_path`` writes ``[A | b]`` in the ``terminal_sets/*.npy`` layout (``lib/terminal_set.py:207-210``)."""
    from .grids import materialise_grid_host
    flags = feasibility_map(controller, axes, x_ref=x_ref, batch_solver=batch_solver)
    shape = [len(a) for a in axes]
    idx = boundary_layer(flags, shape)
    cols = materialise_grid_host(axes)
    pts = np.column_stack([c[idx] for c in cols])
    A, b = hull_polytope(pts)
    if save_path is not None:
        np.save(save_path, np.column_stack((A, b)))
    return A, b, flags


def exact_feasible_set(G: np.ndarray, Gx: np.ndarray, w: np.ndarray) -> tuple[np.ndarray, np.ndarray]:
    """Exact projection {x0 : exists u, G u <= w - Gx x0} by the reference's Fourier-Motzkin step
    (``lib/in_adm_set.py:4-40``), with an LP redundancy removal after every eliminated input so that the row count
    stays polynomial in practice.  Tiny horizons only."""
    C = np.asarray(Gx, dtype=float)                  # rows: C x0 + H u + phi <= 0
    H = np.asarray(G, dtype=float)
    phi = -np.asarray(w, dtype=float)
    for _ in range(H.shape[1]):
        aug = np.column_stack((C, H[:, :-1]))
        P, phi = in_adm_set.algorithm_1(aug, H[:, -1], phi)
        keep = np.sqrt(np.sum(P * P, axis=1)) > 1e-12
        if np.any(~keep & (phi > 1e-12)):
            raise ValueError("the admissible set is empty")
        red = reduce_polytope(Polytope(P[keep], -phi[keep]))
        P, phi = red.A, -red.b
        C, H = P[:, :C.shape[1]], P[:, C.shape[1]:]
    return C, -phi


def closed_loop_map(controller, axes: Sequence[np.ndarray], steps: int = 200, goal=None, x_ref=None, batch_solver=None,
                    noise=None) -> dict:
    """Closed-loop convergence from every point of the tensor grid ``axes`` (C order, x slowest ... v fastest): the
    nonlinear bicycle under ``controller``'s MPC law, in the order of the reference's loops (examples/run_MPCStateFB.py,
    run_MPCOutputFB.py), one run per grid point on the GPU (``BatchQP.closed_loop`` with a goal).  ``MPCStateFB`` runs
    state feedback; ``MPCOutputFB`` output feedback with its ``C`` and ``L``, the observer started at the true state.
    ``goal``: rows as for ``closed_loop`` (default ``montecarlo.goal_box(controller.goal, 0.1)``, the reference's test).
    ``noise``: an optional ``montecarlo.LoopNoise``.

    Returns flat C-order numpy arrays: ``reached`` (bool), ``arrival_step`` and ``fail_step`` (int32, -1 none) and
    ``outcome`` (int8): 0 reached the goal, 1 stopped by a QP that was not solved, 2 neither within ``steps``."""
    import torch
    from .batch import BatchQP
    from .grids import materialise_grid
    from .lib.mpc import MPCOutputFB, MPCStateFB
    from .lib.simulator import CarTrailerDimension
    from .montecarlo import goal_box
    if isinstance(controller, MPCOutputFB):
        C, L = controller.C, controller.L
    elif isinstance(controller, MPCStateFB):
        C = L = None
    else:
        raise TypeError("closed_loop_map needs an MPCStateFB or an MPCOutputFB controller")
    bq = batch_solver if batch_solver is not None else BatchQP.from_controller(controller)
    x0 = torch.stack(materialise_grid(axes, device="cuda")).contiguous()
    out = bq.closed_loop(x0, steps, controller.A, controller.B, x_ref=x_ref, C=C, L=L, dt=controller.dt,
                         l1=CarTrailerDimension.l1, noise=noise,
                         goal=goal_box(controller.goal, 0.1) if goal is None else goal)
    arrival = out["arrival_step"].cpu().numpy()
    fail = out["fail_step"].cpu().numpy()
    reached = arrival >= 0
    outcome = np.where(reached, 0, np.where(fail >= 0, 1, 2)).astype(np.int8)
    return {"reached": reached, "arrival_step": arrival, "fail_step": fail, "outcome": outcome}
