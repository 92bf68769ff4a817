"""Sampled region of attraction on the GPU (carmpc_b200/roa.py, SURVEY 8f-2): the feasibility map of a grid of initial
states, its hull polytope, and the exact Fourier-Motzkin set of lib/in_adm_set.py at a tiny horizon."""
import os

import numpy as np
import pytest

from conftest import GOLDEN, make_env, make_controller
from carmpc_b200 import roa
from carmpc_b200.grids import materialise_grid_host

pytestmark = pytest.mark.gpu


def _grid(nx, ny, npsi, nv):
    return [np.linspace(5.0, 30.0, nx), np.linspace(-3.0, 3.0, ny), np.linspace(-np.pi / 8, np.pi / 8, npsi),
            np.linspace(-1.0, 5.0, nv)]


def test_roa_hull_separates_feasible_from_infeasible_samples(tmp_path):
    """The feasible set is convex, so the hull of the feasible samples must contain every feasible sample and no
    infeasible one (N = 20, the reference's controller)."""
    c = make_controller(make_env("RoadOneCarEnv", [29.9, 1.5, 0, 0]), 20)
    axes = _grid(28, 24, 7, 8)
    path = str(tmp_path / "roa.npy")
    A, b, flags = roa.region_of_attraction(c, axes, save_path=path)
    pts = np.column_stack(materialise_grid_host(axes))
    assert 0.3 < flags.mean() < 0.99
    np.testing.assert_allclose(np.linalg.norm(A, axis=1), 1.0, atol=1e-12)
    worst = (pts @ A.T - b).max(axis=1)
    assert worst[flags].max() <= 1e-9
    assert (worst[~flags] <= 1e-9).sum() == 0, "an infeasible sample lies inside the hull of the feasible ones"
    Ab = np.load(path)
    assert Ab.shape == (len(b), 5) and np.array_equal(Ab[:, :4], A) and np.array_equal(Ab[:, 4], b)
    # the terminal set is inside the region of attraction (samples of it are feasible states)
    T = np.load(os.path.join(GOLDEN, "terminal_sets", "RoadOneCarEnv_29.9_1.5_0_0.npy"))
    in_term = np.all(pts @ T[:, :4].T <= T[:, 4], axis=1)
    assert in_term.sum() > 0 and flags[in_term].all()


def test_feasibility_map_matches_exact_projection_at_tiny_horizon():
    """N = 2: the GPU flags against the exact projection polytope (reference algorithm, lib/in_adm_set.py:4-40)."""
    from oracle import carmpc_oracle as orc
    c = make_controller(make_env("RoadOneCarEnv", [29.9, 1.5, 0, 0]), 2)
    T = np.load(os.path.join(GOLDEN, "terminal_sets", "RoadOneCarEnv_29.9_1.5_0_0.npy"))
    oq = orc.CondensedQP("RoadOneCarEnv", 2, T)
    C, d = roa.exact_feasible_set(oq.G, oq.Gx, oq.w)
    axes = [np.linspace(22.0, 38.0, 33), np.linspace(-0.5, 3.5, 21), np.linspace(-0.3, 0.3, 9), np.linspace(-2.5, 2.5, 11)]
    flags = roa.feasibility_map(c, axes)
    pts = np.column_stack(materialise_grid_host(axes))
    slack = (d[None, :] - pts @ C.T) / np.linalg.norm(C, axis=1)[None, :]
    inside = np.all(slack >= 0, axis=1)
    band = np.abs(slack).min(axis=1) <= 1e-6
    assert 50 < inside.sum() < len(pts) - 50
    np.testing.assert_array_equal(flags[~band], inside[~band])


def test_seeded_and_cold_feasibility_maps_are_identical():
    """The default map goes through the seeded carmpc_qp_solve (lattice anchors + active-set / Farkas reuse); its flags must
    equal the cold solve's point for point, for the default block and for odd ones."""
    c = make_controller(make_env("RoadOneCarEnv", [29.9, 1.5, 0, 0]), 20)
    axes = _grid(40, 48, 4, 5)
    from carmpc_b200.batch import BatchQP
    bq = BatchQP.from_controller(c)
    cold = roa.feasibility_map(c, axes, batch_solver=bq, seeded=False)
    assert 0.3 < cold.mean() < 0.99
    for block in (None, (1, 5, 1, 1), (4, 3, 2, 1), (7, 7, 4, 5)):
        flags = roa.feasibility_map(c, axes, batch_solver=bq, block=block)
        np.testing.assert_array_equal(flags, cold)
    st = bq.polish_stats()
    assert st["used_multiplier_map"] > 0 and sum(st["certified_after_rounds"]) > 0
