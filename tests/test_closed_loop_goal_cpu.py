"""Closed loops that stop at a goal, without a GPU: the argument checks of carmpc_closed_loop's goal, montecarlo.goal_box
against the reference's arrival test, and the oracle's derivation of arrival and failure steps from a trajectory."""
import ctypes
import math

import numpy as np
import pytest

from conftest import make_env, make_controller


# ---- carmpc_closed_loop argument checks of the goal ---------------------------------------------------------------
@pytest.fixture(scope="module")
def handle():
    from carmpc_b200.batch import BatchQP
    return BatchQP.from_controller(make_controller(make_env("RoadEnv"), 10))


_BOX = np.array([[1.0, 0.0, 0.0, 0.0, 30.1], [-1.0, 0.0, 0.0, 0.0, -29.9]])


def _call(lib, qp, goal, runs=4, steps=3, monitor=None):
    mat = np.zeros(16)
    p = ctypes.c_void_p(16)
    return lib.carmpc_closed_loop(
        qp, 0, mat.ctypes.data, mat.ctypes.data, None, None, None, mat.ctypes.data, 0.2, 3.5, steps, 1, p, None, None,
        None, runs, p, None, p, None, None, None, None, ctypes.byref(monitor) if monitor is not None else None,
        ctypes.byref(goal) if goal is not None else None, None, None)


def _goal(rows=_BOX, n=None, arrival=True, row=False, per_step=False):
    from carmpc_b200 import _capi
    rows = np.ascontiguousarray(rows, dtype=np.float64) if rows is not None else None
    g = _capi.LoopRows(rows.ctypes.data if rows is not None else None, len(rows) if n is None else n,
                       64 if arrival else None, 96 if row else None, 128 if per_step else None)
    g._keep = rows                       # the rows must outlive the call
    return g


def test_goal_argument_errors(handle):
    from carmpc_b200 import _capi
    lib = _capi.load()
    h = handle._h
    err = lambda: lib.carmpc_last_error()   # noqa: E731
    for runs in (0, 4):                     # checked before the early return of an empty run set
        assert _call(lib, h, _goal(n=0), runs=runs) == -1 and b"goal rows" in err()
        assert _call(lib, h, _goal(np.tile(_BOX, (257, 1)), n=513), runs=runs) == -1 and b"goal rows" in err()
        assert _call(lib, h, _goal(arrival=False), runs=runs) == -1 and b"a goal needs d_step" in err()
        assert _call(lib, h, _goal(row=True), runs=runs) == -1 and b"a goal has no d_row" in err()
        assert _call(lib, h, _goal(rows=None, n=2), runs=runs) == -1 and b"null goal rows" in err()
        for bad in (math.nan, math.inf, -math.inf):
            for r, c in ((0, 4), (1, 0), (1, 3)):
                rows = _BOX.copy()
                rows[r, c] = bad
                assert _call(lib, h, _goal(rows), runs=runs) == -1 and b"finite" in err()
    # valid goals and no runs: nothing to do
    for g in _valid_goals():
        assert _call(lib, h, g, runs=0) == 0


def _valid_goals():
    return (_goal(), _goal(per_step=True), _goal(np.tile(_BOX, (256, 1)), n=512), None)


def test_monitor_and_goal_together_pass_the_checks(handle):
    """One row set as the monitor (every output set) and another as the goal: valid together, each checked as its use."""
    from carmpc_b200 import _capi
    lib = _capi.load()
    rows = np.ascontiguousarray(np.tile(_BOX, (2, 1)))
    monitor = _capi.LoopRows(rows.ctypes.data, len(rows), 256, 320, 384)
    assert _call(lib, handle._h, _goal(per_step=True), runs=0, monitor=monitor) == 0
    assert _call(lib, handle._h, _goal(arrival=False), runs=0, monitor=monitor) == -1
    assert b"a goal needs d_step" in lib.carmpc_last_error()


def test_goal_loop_on_a_host_only_handle_is_a_cuda_error(handle):
    """Valid goals and runs on a handle created without a CUDA device: the loop fails loudly instead of computing."""
    try:
        import torch
        if torch.cuda.is_available():
            pytest.skip("a CUDA device is present: handles are not host-only here")
    except ImportError:
        pass
    from carmpc_b200 import _capi
    lib = _capi.load()
    for g in _valid_goals():
        assert _call(lib, handle._h, g, runs=4) == -2 and b"without a CUDA device" in lib.carmpc_last_error()


# ---- goal_box -----------------------------------------------------------------------------------------------------
def test_goal_box_is_the_reference_test():
    """Random states around random goals: the rows (with the monitor's chain) agree with
    np.all(np.abs(s - g) <= tol) everywhere outside a 1e-12 band of the faces; a non-finite state is never inside."""
    import goal_oracle as go
    from carmpc_b200.montecarlo import goal_box
    rng = np.random.default_rng(3)
    compared = 0
    for tol in (0.1, 0.5, 1e-3):
        for _ in range(20):
            g = rng.uniform([-5, -3, -0.5, -1], [40, 3, 0.5, 5])
            rows = goal_box(g, tol)
            assert rows.shape == (8, 5) and np.isfinite(rows).all()
            s = g + rng.uniform(-2.5, 2.5, size=(4000, 4)) * tol
            s[::7] = g + tol * rng.choice([-1.0, 1.0], size=(len(s[::7]), 4))      # on the faces
            want = np.all(np.abs(s - g) <= tol, axis=1)
            got = go.inside(rows, s)
            band = (np.abs(np.abs(s - g) - tol) <= 1e-12).any(1)
            np.testing.assert_array_equal(got[~band], want[~band])
            compared += int((~band).sum())
            assert want[~band].any() and not want[~band].all()
    assert compared > 100_000
    rows = goal_box([1.0, 2.0, 0.0, 0.0])
    np.testing.assert_array_equal(rows[0], [1, 0, 0, 0, 1.1])
    np.testing.assert_array_equal(rows[1], [-1, 0, 0, 0, -1.0 + 0.1])
    for s in ([math.nan, 2, 0, 0], [1, math.inf, 0, 0], [1, 2, 0, -math.inf]):
        assert not go.inside(rows, np.array([s]))[0]
    assert go.inside(rows, np.array([[1.0, 2.0, 0.0, 0.0]]))[0]
    for bad in ([1, 2, 3], [1, 2, math.nan, 0]):
        with pytest.raises(ValueError):
            goal_box(bad)
    with pytest.raises(ValueError):
        goal_box([0, 0, 0, 0], tol=-1)


# ---- the oracle's derivation from a trajectory without a goal -----------------------------------------------------
def test_outcome_from_trajectory():
    """Hand-made trajectories (goal box 0 +- 0.1): arrival and failure at the same step is a failure; a run that passes
    through the box and leaves it arrived at its first step inside; a run that never enters, one that fails before it
    enters, one inside only after its failure, and a non-finite state."""
    import goal_oracle as go
    from carmpc_b200.montecarlo import goal_box
    rows = goal_box(np.zeros(4), 0.1)
    far, near = np.full(4, 1.0), np.full(4, 0.05)
    steps, R = 6, 6
    traj = np.tile(far, (steps, R, 1))
    fail = np.full(R, -1, dtype=np.int32)
    traj[3, 0] = near; fail[0] = 3                          # 0: inside at its failing step
    traj[2, 1] = near; traj[4:, 1] = near                   # 1: enters at 2, leaves, comes back
    #                                                         2: never inside
    fail[3] = 1; traj[1:, 3] = far; traj[4, 3] = near       # 3: inside only after its failure
    traj[5, 4] = near                                       # 4: arrives at the last step
    traj[:, 5] = np.nan; fail[5] = 0                        # 5: non-finite, fails at once
    arrival, fail_out = go.outcome_from_traj(traj, fail, rows)
    np.testing.assert_array_equal(arrival, [-1, 2, -1, -1, 5, -1])
    np.testing.assert_array_equal(fail_out, [3, -1, -1, 1, -1, 0])
    assert arrival.dtype == np.int32 and fail_out.dtype == np.int32
    d = go.face_distance(traj[:, :5], rows)
    assert d.shape == (steps, 5) and np.isclose(d[0, 0], 0.9) and np.isclose(d[2, 1], 0.05)


def test_oracle_loop_stops_at_the_goal():
    """The oracle's loop with a goal equals the derivation from its loop without one (state and output feedback,
    a scripted solver that fails one run at the step it would arrive)."""
    import goal_oracle as go
    from oracle import carmpc_oracle as orc
    from carmpc_b200.montecarlo import goal_box

    class Q:
        A = np.eye(4)
        B = np.zeros((4, 2))

    goal = np.array([3.0, 0.0, 0.0, 1.0])
    rows = goal_box(goal, 0.1)
    x_init = np.array([[0.0, 0, 0, 1], [1.0, 0, 0, 1], [2.45, 0, 0.05, 1], [0.0, 0, 0, 0]])

    def solve(x):                          # coast; a heading above 0.01 has no solution within 0.1 of x = 3
        st = ((np.abs(x[:, 0] - 3.0) <= 0.1) & (x[:, 2] > 0.01)).astype(np.int32)
        return np.zeros((len(x), 2)), st

    for ofb in (False, True):
        _, fail0, traj0 = orc.closed_loop(Q, x_init, goal, 25, ofb, solve)
        x, fail, arrival, traj = go.closed_loop(Q, x_init, 25, ofb, solve, rows)
        want_a, want_f = go.outcome_from_traj(traj0, fail0, rows)
        np.testing.assert_array_equal(arrival, want_a)
        np.testing.assert_array_equal(fail, want_f)
        if not ofb:
            np.testing.assert_array_equal(arrival, [14, 9, -1, -1])
            np.testing.assert_array_equal(fail, [-1, -1, 2, -1])
        for r in range(len(x_init)):
            end = arrival[r] if arrival[r] >= 0 else len(traj)
            np.testing.assert_array_equal(traj[:end, r], traj0[:end, r])
            if arrival[r] >= 0:
                assert (traj[arrival[r]:, r] == traj[arrival[r], r]).all()
                np.testing.assert_array_equal(x[r], traj[arrival[r], r])
