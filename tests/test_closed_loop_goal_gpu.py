"""Closed loops that stop at a goal (carmpc_closed_loop with a goal) on the GPU: a goal that is never met changes
nothing, bit for bit, in every mode and warm-start form; parity with the restated loop (exact QPs) on RoadEnv; at size
(10^4 runs x 200 steps, graph-replayed steps) the arrival and failure steps are those of the loop without a goal; the
map by closed-loop convergence against the reference's own loop; the example end to end."""
import importlib
import os
import sys

import numpy as np
import pytest

from conftest import GOLDEN, ROOT, make_env, make_controller

pytestmark = pytest.mark.gpu
EXAMPLES = os.path.join(ROOT, "examples")

X_REF = np.array([30.0, 1.5, 0.0, 0.0])
BOX_LO, BOX_HI = [0, -2.5, -0.2, 0], [10, 2.5, 0.2, 3]
NEVER = np.array([[0.0, 0.0, 0.0, 0.0, -1.0]])          # 0 . s <= -1: no state is inside
W_AUG = np.diag([1e-2] * 4 + [1e-3])
V_OUT = 1e-2 * np.eye(3)


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "the GPU tests need a CUDA device"
    return torch


@pytest.fixture(scope="module")
def plain():
    from carmpc_b200.batch import BatchQP
    ctl = make_controller(make_env("RoadEnv"), 20, cls="MPCOutputFB", init_state=[0, 0, 0, 0])
    return ctl, BatchQP.from_controller(ctl)


@pytest.fixture(scope="module")
def dist():
    from carmpc_b200.batch import BatchQP
    from carmpc_b200.observer import augmented_observer_gain
    ctl = make_controller(make_env("RoadEnv"), 20, cls="MPCOutputFBWithDisturbance", init_state=[0, 0, 0, 0])
    ctl.Bd = np.ones(4)
    L1, L2 = augmented_observer_gain(ctl.A, ctl.C, np.ones(4), np.ones(3), W_AUG, V_OUT)
    return ctl, BatchQP.from_controller(ctl), (np.ones(4), np.ones(3), L1, L2)


@pytest.fixture(scope="module")
def onecar():
    """State-feedback controller on RoadOneCarEnv (the reference's default goal) and its handle."""
    from carmpc_b200.batch import BatchQP
    ctl = make_controller(make_env("RoadOneCarEnv"), 20)
    return ctl, BatchQP.from_controller(ctl)


@pytest.fixture()
def examples_on_path():
    """examples/ importable for one test; afterwards its modules are forgotten (their import sets the terminal-set
    directory, which other tests rely on) and the directory is restored."""
    from carmpc_b200.lib import terminal_set as ts
    saved, before = ts.TERMINAL_SET_DIR, set(sys.modules)
    sys.path.insert(0, EXAMPLES)
    yield
    sys.path.remove(EXAMPLES)
    for name in set(sys.modules) - before:
        if os.path.dirname(os.path.abspath(getattr(sys.modules[name], "__file__", None) or "")) == EXAMPLES:
            del sys.modules[name]
    ts.TERMINAL_SET_DIR = saved


def _x_init(torch, R, seed, lo=BOX_LO, hi=BOX_HI):
    g = torch.Generator(device="cpu").manual_seed(seed)
    lo, hi = torch.tensor(lo, dtype=torch.float64), torch.tensor(hi, dtype=torch.float64)
    return (lo[:, None] + (hi - lo)[:, None] * torch.rand((4, R), generator=g, dtype=torch.float64)).cuda().contiguous()


# ---- 1. a goal never met changes nothing ----------------------------------------------------------------------------
@pytest.mark.parametrize("warm_start", [0, 1, 2])
def test_unreachable_goal_changes_nothing(torch_cuda, plain, dist, warm_start):
    """Modes 0, 1 and 2, with neither, either or both of noise and monitor (every instantiation of the step kernel),
    2000 runs x 60 steps: every output of the loop and total_iters are torch.equal to the loop without a goal;
    arrival_step is -1 and arrivals_per_step 0."""
    torch = torch_cuda
    from carmpc_b200.lib.mpc import _C_XYV, _L_OBSERVER
    from carmpc_b200.montecarlo import LoopNoise, plant_rows
    ctl, bq = plain
    dctl, dbq, (Bd, Cd, L1, L2) = dist
    R, T = 2000, 60
    x0 = _x_init(torch, R, 1)
    d_r = ((torch.rand(R, generator=torch.Generator().manual_seed(2), dtype=torch.float64) - 0.5) * 0.02).cuda()
    rows = plant_rows(ctl)
    keys = ("final", "fail_step", "traj", "inputs", "violation_step", "violation_row", "violations_per_step", "dhat",
            "dhat_traj")

    def same(ref, o, what):
        assert o["total_iters"] == ref["total_iters"], what
        for k in keys:
            if k in ref:
                assert torch.equal(o[k], ref[k]), (what, k)
        assert (o["arrival_step"] == -1).all() and (o["arrivals_per_step"] == 0).all(), what
        assert o["arrivals_per_step"].shape == (T,)

    noisy = LoopNoise([0.02, 0.02, 0.004, 0.02], [0.03, 0.03, 0.03, 0.03], seed=9)
    for noise, monitor in ((None, None), (noisy, None), (None, rows), (noisy, rows)):
        for mode in (0, 1):
            C, L = (_C_XYV, _L_OBSERVER) if mode else (None, None)
            kw = dict(x_ref=X_REF, C=C, L=L, warm_start=warm_start, want_traj=True, want_inputs=True, noise=noise,
                      monitor=monitor)
            ref = bq.closed_loop(x0, T, ctl.A, ctl.B, **kw)
            ok = (ref["fail_step"] < 0).float().mean().item()
            assert 0.05 < ok < 0.95
            same(ref, bq.closed_loop(x0, T, ctl.A, ctl.B, goal=NEVER, **kw), (mode, noise is None, monitor is None))
        dkw = dict(x_ref=X_REF, Bd_plant=np.ones(4), d_plant=d_r, warm_start=warm_start, want_traj=True,
                   want_inputs=True, want_dhat=True, noise=noise, monitor=monitor)
        ref = dbq.closed_loop_disturbance(x0, T, dctl.A, dctl.B, dctl.C, Bd, Cd, L1, L2, **dkw)
        o = dbq.closed_loop_disturbance(x0, T, dctl.A, dctl.B, dctl.C, Bd, Cd, L1, L2, goal=(NEVER[:, :4], NEVER[:, 4]),
                                        **dkw)
        same(ref, o, (2, noise is None, monitor is None))


# ---- 2. oracle parity -----------------------------------------------------------------------------------------------
def test_matches_the_restated_loop_with_a_goal(torch_cuda, plain):
    """RoadEnv, 16 runs x 60 steps started in the goal's lane, state and output feedback, against the restated loop
    with exact QPs: arrival_step and fail_step equal, trajectories and final states within 1e-6."""
    torch = torch_cuda
    import goal_oracle as go
    from oracle import carmpc_oracle as orc
    from carmpc_b200.montecarlo import goal_box
    ctl, bq = plain
    oq = orc.CondensedQP("RoadEnv", 20, np.load(os.path.join(GOLDEN, "terminal_sets", "RoadEnv_30_1.5_0_0.npy")))

    def exact(x):
        u, obj, st, *_ = orc.qp_solve_exact(oq, x, X_REF)
        return u[:, :2], st

    R, T = 16, 60
    rows = goal_box(X_REF, 0.1)
    x_init = np.random.default_rng(0).uniform([20, 1.45, -0.01, 0], [29, 1.55, 0.01, 2], size=(R, 4))
    x0 = torch.from_numpy(np.ascontiguousarray(x_init.T)).cuda()
    for output_feedback in (False, True):
        want_x, want_fail, want_arr, want_traj = go.closed_loop(oq, x_init, T, output_feedback, exact, rows)
        assert (want_arr >= 0).sum() >= R // 2
        out = bq.closed_loop(x0, T, ctl.A, ctl.B, x_ref=X_REF, C=orc.C_OUT if output_feedback else None,
                             L=orc.L_OBS if output_feedback else None, want_traj=True, want_inputs=True, goal=rows)
        np.testing.assert_array_equal(out["arrival_step"].cpu().numpy(), want_arr)
        np.testing.assert_array_equal(out["fail_step"].cpu().numpy(), want_fail)
        assert np.abs(out["traj"].cpu().numpy().transpose(0, 2, 1) - want_traj).max() <= 1e-6
        np.testing.assert_allclose(out["final"].cpu().numpy().T, want_x, atol=1e-6)
        np.testing.assert_array_equal(out["arrivals_per_step"].cpu().numpy(),
                                      np.bincount(want_arr[want_arr >= 0], minlength=T))


# ---- 3. at size, against the loop without a goal -------------------------------------------------------------------
@pytest.mark.parametrize("noisy", [False, True])
def test_at_size_against_the_loop_without_a_goal(torch_cuda, onecar, noisy):
    """RoadOneCarEnv, 10^4 runs x 200 steps, warm_start 1 (graph-replayed steps): arrival_step and fail_step are those
    derived from the trajectory of the loop without a goal (runs that come within 1e-9 of a goal face before they
    stop are counted, and few); trajectories agree up to the arrival within 1e-9 and stay frozen after it, the input
    log keeps the last applied input; arrivals_per_step is the histogram of arrival_step.  With noise the same holds:
    the draws depend only on (run, step)."""
    torch = torch_cuda
    import goal_oracle as go
    from carmpc_b200.montecarlo import LoopNoise, goal_box
    ctl, bq = onecar
    R, T = 10_000, 200
    g = np.asarray(ctl.goal, dtype=float)
    rows = goal_box(g, 0.1)
    x0 = _x_init(torch, R, 7, lo=[12.0, g[1] - 0.3, -0.05, 0.0], hi=[29.0, g[1] + 0.3, 0.05, 3.0])
    noise = LoopNoise([1e-3, 1e-3, 1e-4, 1e-3], [1e-3] * 4, seed=4) if noisy else None
    kw = dict(warm_start=1, want_traj=True, want_inputs=True, noise=noise)
    ref = bq.closed_loop(x0, T, ctl.A, ctl.B, **kw)
    out = bq.closed_loop(x0, T, ctl.A, ctl.B, goal=rows, **kw)
    traj0 = ref["traj"].cpu().numpy().transpose(0, 2, 1)
    fail0 = ref["fail_step"].cpu().numpy()
    traj = out["traj"].cpu().numpy().transpose(0, 2, 1)
    inputs = out["inputs"].cpu().numpy().transpose(0, 2, 1)
    arr = out["arrival_step"].cpu().numpy()
    fail = out["fail_step"].cpu().numpy()
    want_arr, want_fail = go.outcome_from_traj(traj0, fail0, rows)

    # runs whose state comes within 1e-9 of a goal face while they still run (both loops' verdicts are then fragile)
    stop = np.where(want_arr >= 0, want_arr, np.where(want_fail >= 0, want_fail, T - 1))
    running = np.arange(T)[:, None] <= stop[None, :]
    band = ((go.face_distance(traj0, rows) <= 1e-9) & running).any(0)
    assert band.sum() <= 5, f"{band.sum()} runs within 1e-9 of a goal face"
    np.testing.assert_array_equal(arr[~band], want_arr[~band])
    np.testing.assert_array_equal(fail[~band], want_fail[~band])
    reached = arr >= 0
    assert 0.3 * R < reached.sum() < R, reached.sum()
    assert ((arr >= 0) & (fail >= 0)).sum() == 0

    np.testing.assert_array_equal(out["arrivals_per_step"].cpu().numpy(), np.bincount(arr[reached], minlength=T))
    for r in np.flatnonzero(~band):
        end = arr[r] + 1 if arr[r] >= 0 else T
        assert np.abs(traj[:end, r] - traj0[:end, r]).max() <= 1e-9, r
    final = out["final"].cpu().numpy().T
    idx = np.flatnonzero(reached)
    k = arr[idx]
    frozen = traj[:, idx] == traj[k, idx][None]
    assert frozen[np.arange(T)[:, None] >= k[None, :]].all()
    np.testing.assert_array_equal(final[idx], traj[k, idx])
    last_u = np.where((k > 0)[:, None], inputs[np.maximum(k - 1, 0), idx], 0.0)
    kept = inputs[:, idx] == last_u[None]
    assert kept.all(-1)[np.arange(T)[:, None] >= k[None, :]].all()
    assert out["total_iters"] <= ref["total_iters"]


# ---- 4. the map against the reference's own loop -------------------------------------------------------------------
def test_closed_loop_map_against_the_reference_loop(torch_cuda, onecar, examples_on_path):
    """A 4 x 3 x 1 x 1 map of RoadOneCarEnv (state feedback, 151 steps = the reference's 30 s) against
    examples/run_MPCStateFB.py started at each grid point: arrival at step k is a reference run of k + 1 plant steps
    that reached the goal, a failure at step k one of k + 1 steps that did not, and neither the full length."""
    from carmpc_b200 import roa
    from carmpc_b200.lib.configuration import DT_SIMULATION
    ctl, bq = onecar
    g = np.asarray(ctl.goal, dtype=float)
    steps = int(30.0 / DT_SIMULATION) + 1
    axes = [np.array([6.0, 15.0, 22.0, 27.0]), np.array([g[1] - 2.6, g[1] - 0.05, g[1] + 0.6]), np.array([0.0]),
            np.array([1.0])]
    m = roa.closed_loop_map(ctl, axes, steps=steps, batch_solver=bq)
    assert set(m) == {"reached", "arrival_step", "fail_step", "outcome"}
    assert m["outcome"].shape == (12,)
    np.testing.assert_array_equal(m["reached"], m["arrival_step"] >= 0)
    np.testing.assert_array_equal(m["outcome"], np.where(m["reached"], 0, np.where(m["fail_step"] >= 0, 1, 2)))
    assert m["reached"].any()
    from carmpc_b200.grids import materialise_grid_host
    run = importlib.import_module("run_MPCStateFB")
    for i, p in enumerate(np.column_stack(materialise_grid_host(axes))):
        states, _, _, reached = run.main(["--env", "RoadOneCarEnv", "--start", *[repr(float(v)) for v in p]])
        a, f = int(m["arrival_step"][i]), int(m["fail_step"][i])
        if a >= 0:
            assert reached and len(states) == a + 1, (p, a, len(states))
        elif f >= 0:
            assert not reached and len(states) == f + 1, (p, f, len(states))
        else:
            assert not reached and len(states) == steps, (p, len(states))


# ---- 5. the example -------------------------------------------------------------------------------------------------
def test_closed_loop_roa_example_runs(examples_on_path, capsys):
    res = importlib.import_module("closed_loop_roa").main(["--points", "4", "3", "--steps", "40"])
    out = capsys.readouterr().out
    assert "reached" in out and "feasible" in out
    assert res["outcome"].shape == (12,) and res["feasible"].shape == (12,)
    assert np.bincount(res["outcome"], minlength=3).sum() == 12
