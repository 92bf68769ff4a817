"""Host logic of the sampled region of attraction (carmpc_b200/roa.py, SURVEY 8f-2): boundary layer, hull -> H-rep,
and the exact Fourier-Motzkin projection (lib/in_adm_set.py) cross-checked against the oracle's LP feasibility."""
import os

import numpy as np

from conftest import GOLDEN
from carmpc_b200 import roa


def _box_grid(n=9):
    ax = [np.linspace(-1, 1, n)] * 3
    g = np.stack(np.meshgrid(*ax, indexing="ij"), axis=-1).reshape(-1, 3)
    return ax, g


def test_boundary_layer_contains_all_hull_vertices():
    ax, g = _box_grid(11)
    A = np.array([[1, 1, 0], [-1, 2, 1], [0, -1, -1], [1, 0, -2], [-1, -1, 1.0]])
    b = np.array([0.9, 1.4, 0.8, 1.1, 1.2])
    flags = np.all(g @ A.T <= b, axis=1)
    idx = roa.boundary_layer(flags, [11, 11, 11])
    assert 0 < len(idx) < flags.sum()
    assert flags[idx].all()
    from scipy.spatial import ConvexHull
    full = ConvexHull(g[flags])
    verts = {tuple(p) for p in g[flags][full.vertices]}
    assert verts <= {tuple(p) for p in g[idx]}
    # interior points have all six neighbours feasible
    f3 = flags.reshape(11, 11, 11)
    inner = np.setdiff1d(np.flatnonzero(flags), idx)
    for k in inner[:50]:
        i, j, l = np.unravel_index(k, f3.shape)
        assert f3[i - 1, j, l] and f3[i + 1, j, l] and f3[i, j - 1, l] and f3[i, j + 1, l] and f3[i, j, l - 1] and f3[i, j, l + 1]


def test_hull_polytope_is_tight_inner_approximation():
    ax, g = _box_grid(13)
    A = np.array([[1, 1, 0], [-1, 2, 1], [0, -1, -1], [1, 0, -2], [-1, -1, 1.0], [0, 0, 1]])
    b = np.array([0.9, 1.4, 0.8, 1.1, 1.2, 0.5])
    flags = np.all(g @ A.T <= b, axis=1)
    Ah, bh = roa.hull_polytope(g[roa.boundary_layer(flags, [13] * 3)])
    np.testing.assert_allclose(np.linalg.norm(Ah, axis=1), 1.0, atol=1e-12)
    inside = np.all(g @ Ah.T <= bh + 1e-9, axis=1)
    np.testing.assert_array_equal(inside, flags)            # convex set: its samples' hull excludes every other sample
    # merged facets: far fewer rows than simplicial facets
    from scipy.spatial import ConvexHull
    assert len(bh) < len(ConvexHull(g[flags]).equations)


def test_hull_polytope_degenerate_sets():
    # the reference's own grid has psi fixed (lib/terminal_set.py:96-106): a 3-D set embedded in 4-D
    rng = np.random.default_rng(0)
    P = np.column_stack((rng.uniform(0, 1, (200, 2)), np.zeros(200), rng.uniform(2, 3, 200)))
    A, b = roa.hull_polytope(P)
    assert np.all(P @ A.T <= b + 1e-9)
    off = P[0] + np.array([0, 0, 1e-3, 0])
    assert not np.all(A @ off <= b + 1e-9)
    # a segment and a single point
    A, b = roa.hull_polytope(np.array([[0.0, 0, 0, 0], [1, 1, 0, 0], [0.5, 0.5, 0, 0]]))
    assert np.all(A @ np.array([0.25, 0.25, 0, 0]) <= b + 1e-12) and not np.all(A @ np.array([1.5, 1.5, 0, 0]) <= b + 1e-9)
    A, b = roa.hull_polytope(np.array([[1.0, 2, 3, 4]]))
    assert np.all(A @ np.array([1.0, 2, 3, 4]) <= b + 1e-12) and not np.all(A @ np.array([1.0, 2, 3, 4.01]) <= b + 1e-9)


def test_exact_projection_matches_lp_feasibility():
    """Fourier-Motzkin (the reference's lib/in_adm_set.py step) on the horizon-2 condensed QP of RoadOneCarEnv against
    the oracle's LP feasibility flag on random states; states within 1e-6 of the boundary are enumerated."""
    from oracle import carmpc_oracle as orc
    Ab = np.load(os.path.join(GOLDEN, "terminal_sets", "RoadOneCarEnv_29.9_1.5_0_0.npy"))
    oq = orc.CondensedQP("RoadOneCarEnv", 2, Ab)
    C, d = roa.exact_feasible_set(oq.G, oq.Gx, oq.w)
    assert C.shape[1] == 4 and 4 < len(d) < 200
    rng = np.random.default_rng(1)
    goal = np.array([29.9, 1.5, 0, 0])
    x0 = goal + rng.uniform(-1, 1, size=(400, 4)) * np.array([6.0, 1.6, 0.3, 2.5])
    feas, margin = orc.qp_feasible_lp(oq, x0)
    slack = (d[None, :] - x0 @ C.T) / np.linalg.norm(C, axis=1)[None, :]
    inside = np.all(slack >= 0, axis=1)
    band = (np.abs(slack).min(axis=1) <= 1e-6) | (np.abs(margin) <= 1e-6)
    assert 20 < inside.sum() < 380
    np.testing.assert_array_equal(inside[~band], np.asarray(feas, dtype=bool)[~band])


def test_lattice_seeds_form_a_single_level_forest():
    """Seed maps of the seeded carmpc_qp_solve: anchors name themselves, every follower names an anchor of its own block, and
    shard-local maps never point outside the shard (SURVEY 8e: contiguous index ranges per rank)."""
    from carmpc_b200.grids import lattice_seeds, shard_range
    dims = (12, 10, 3, 4)
    n = int(np.prod(dims))
    for block in ((3, 8, 1, 1), (1, 1, 1, 1), (5, 4, 2, 3), (20, 20, 20, 20)):
        s = lattice_seeds(dims, block=block)
        assert s.dtype == np.int32 and s.shape == (n,)
        anchors = np.flatnonzero(s == np.arange(n))
        assert np.array_equal(s[s], s), "a follower's seed must be an anchor"
        idx = np.stack(np.unravel_index(np.arange(n), dims), axis=1)
        same_block = np.all(idx // np.array(block) == idx[s] // np.array(block), axis=1)
        assert same_block.all()
        expected = int(np.prod([-(-d // min(b, d)) if b <= d else 1 for d, b in zip(dims, block)]))
        assert len(anchors) == expected
    for world in (2, 3):
        for rank in range(world):
            lo, hi = shard_range(n, rank, world)
            s = lattice_seeds(dims, block=(3, 8, 1, 1), start=lo, stop=hi)
            assert s.shape == (hi - lo,) and s.min() >= 0 and s.max() < hi - lo
            assert np.array_equal(s[s], s)


def test_default_seed_block_follows_the_grid_spacing():
    from carmpc_b200.grids import config3_axes, config2_axes
    assert roa.default_seed_block(config3_axes()) == (3, 8, 1, 1)
    assert roa.default_seed_block(config2_axes()) == (1, 7, 1, 1)
    assert roa.default_seed_block([np.array([1.0]), np.linspace(0, 1, 2), np.linspace(0, 1, 9), np.linspace(0, 1, 9)]) == (1, 1, 1, 1)
