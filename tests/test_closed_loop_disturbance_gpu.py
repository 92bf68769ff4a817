"""Closed loops of the disturbance-estimating output-feedback controller (carmpc_closed_loop_disturbance) on RoadEnv,
horizon 20: parity with the oracle's loop (exact QPs on the disturbance-shifted bounds), the reference's unstable gains,
reduction to the plain output-feedback loop, config-4 size, and the offset-free property the controller is for."""
import os

import numpy as np
import pytest

from conftest import GOLDEN, make_env, make_controller

pytestmark = pytest.mark.gpu

W_AUG = np.diag([1e-2] * 4 + [1e-3])
V_OUT = 1e-2 * np.eye(3)
X_REF = np.array([30.0, 1.5, 0.0, 0.0])
BOX_LO, BOX_HI = [0, -2.5, -0.2, 0], [10, 2.5, 0.2, 3]


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "the GPU tests need a CUDA device"
    return torch


def _setup(Bd):
    """Controller, solver handle and oracle QP for the disturbance model Bd (the handle's Gc is rows_x @ ABd(Bd))."""
    from carmpc_b200.batch import BatchQP
    import disturbance_oracle as dorc
    from oracle import carmpc_oracle as orc
    ctl = make_controller(make_env("RoadEnv"), 20, cls="MPCOutputFBWithDisturbance", init_state=[0, 0, 0, 0])
    ctl.Bd = np.asarray(Bd, dtype=float)
    bq = BatchQP.from_controller(ctl)
    Ab = np.load(os.path.join(GOLDEN, "terminal_sets", "RoadEnv_30_1.5_0_0.npy"))
    dq = dorc.DisturbedQP("RoadEnv", 20, Ab, ctl.Bd)

    def exact(x, d):
        u, obj, st, *_ = orc.qp_solve_exact(dq, np.hstack((x, d[:, None])), np.append(X_REF, 0.0))
        return u[:, :2], st

    return ctl, bq, exact


def _oracle(ctl, exact, gains, x_init, steps, Bd_p, Cd_p, d_r):
    import disturbance_oracle as dorc
    from oracle import carmpc_oracle as orc
    Bd, Cd, L1, L2 = gains
    return dorc.closed_loop_disturbance(ctl.A, ctl.B, ctl.C, Bd, Cd, L1, L2, x_init, steps, exact, Bd_p, Cd_p, d_r)


def _gpu(torch, bq, ctl, gains, x_init, steps, Bd_p, Cd_p, d_r, **kw):
    Bd, Cd, L1, L2 = gains
    x0 = torch.from_numpy(np.ascontiguousarray(np.asarray(x_init).T)).cuda()
    d = torch.from_numpy(np.ascontiguousarray(d_r, dtype=np.float64)).cuda() if d_r is not None else None
    return bq.closed_loop_disturbance(x0, steps, ctl.A, ctl.B, ctl.C, Bd, Cd, L1, L2, x_ref=X_REF, Bd_plant=Bd_p,
                                      Cd_plant=Cd_p, d_plant=d, **kw)


def _assert_matches(out, want, min_alive):
    want_x, want_d, want_fail, want_traj, want_dlog = want
    fail = out["fail_step"].cpu().numpy()
    np.testing.assert_array_equal(fail, want_fail)
    alive = want_fail < 0
    assert alive.sum() >= min_alive
    traj = out["traj"].cpu().numpy().transpose(0, 2, 1)
    assert np.abs(traj - want_traj).max() <= 1e-6
    np.testing.assert_allclose(out["final"].cpu().numpy().T, want_x, atol=1e-6)
    np.testing.assert_allclose(out["dhat"].cpu().numpy(), want_d, atol=1e-6)
    np.testing.assert_allclose(out["dhat_traj"].cpu().numpy(), want_dlog, atol=1e-6)


@pytest.mark.parametrize("source", ["process", "sensor"])
def test_matches_the_oracle_with_stable_gains(torch_cuda, source):
    """16 runs x 25 steps, Bd = 1_4, Cd = 1_3 with the steady-state predictor gain; a per-run constant disturbance enters
    the plant state (Bd_p = 1_4) or its output (Cd_p = 1_3).  fail_step equal, trajectories / d^ / finals within 1e-6."""
    from carmpc_b200.observer import augmented_observer_gain
    ctl, bq, exact = _setup(np.ones(4))
    L1, L2 = augmented_observer_gain(ctl.A, ctl.C, np.ones(4), np.ones(3), W_AUG, V_OUT)
    gains = (np.ones(4), np.ones(3), L1, L2)
    rng = np.random.default_rng(0)
    R, steps = 16, 25
    x_init = rng.uniform(BOX_LO, BOX_HI, size=(R, 4))
    d_proc, d_sens = rng.uniform(-0.02, 0.02, size=R), rng.uniform(-0.1, 0.1, size=R)
    if source == "process":
        Bd_p, Cd_p, d_r = np.ones(4), np.zeros(3), d_proc
    else:
        Bd_p, Cd_p, d_r = np.zeros(4), np.ones(3), d_sens
    want = _oracle(ctl, exact, gains, x_init, steps, Bd_p, Cd_p, d_r)
    out = _gpu(torch_cuda, bq, ctl, gains, x_init, steps, Bd_p, Cd_p, d_r, want_traj=True, want_inputs=True,
               want_dhat=True)
    _assert_matches(out, want, min_alive=R // 4)
    assert out["total_iters"] > 0
    assert np.abs(out["dhat"].cpu().numpy()).max() > 0


def test_reference_gains_diverge_and_stop_where_the_reference_raises(torch_cuda):
    """The reference's L1 / L2 = [1, 1, 1] (spectral radius 3.31): the estimate runs away and every run stops at the step
    at which the oracle's QP becomes infeasible."""
    from carmpc_b200.observer import reference_disturbance_gains
    ctl, bq, exact = _setup(np.ones(4))
    gains = reference_disturbance_gains(ctl)
    rng = np.random.default_rng(0)
    R, steps = 16, 25
    x_init = rng.uniform(BOX_LO, BOX_HI, size=(R, 4))
    d_r = rng.uniform(-0.02, 0.02, size=R)
    want = _oracle(ctl, exact, gains, x_init, steps, np.ones(4), np.zeros(3), d_r)
    assert (want[2] >= 0).all()
    out = _gpu(torch_cuda, bq, ctl, gains, x_init, steps, np.ones(4), np.zeros(3), d_r, want_traj=True, want_dhat=True)
    _assert_matches(out, want, min_alive=0)


def test_zero_disturbance_terms_reduce_to_the_output_feedback_loop(torch_cuda):
    """L2 = 0, Bd = Cd = Bd_p = Cd_p = 0, d^ = 0 on the same handle (its Gc is not zero): every c term is an exact zero,
    so the loop is bit for bit carmpc_closed_loop's output feedback (mode 1, graph-replayed steps included)."""
    torch = torch_cuda
    from carmpc_b200.lib.mpc import _C_XYV, _L_OBSERVER
    ctl, bq, _ = _setup(np.ones(4))
    R, T = 2000, 60
    g = torch.Generator(device="cpu").manual_seed(1)
    lo, hi = torch.tensor(BOX_LO, dtype=torch.float64), torch.tensor(BOX_HI, dtype=torch.float64)
    x_init = (lo[:, None] + (hi - lo)[:, None] * torch.rand((4, R), generator=g, dtype=torch.float64)).cuda().contiguous()
    ref = bq.closed_loop(x_init, T, ctl.A, ctl.B, x_ref=X_REF, C=_C_XYV, L=_L_OBSERVER, want_traj=True, want_inputs=True)
    out = bq.closed_loop_disturbance(x_init, T, ctl.A, ctl.B, _C_XYV, np.zeros(4), np.zeros(3), _L_OBSERVER, np.zeros(3),
                                     x_ref=X_REF, want_traj=True, want_inputs=True, want_dhat=True)
    assert torch.equal(out["fail_step"], ref["fail_step"])
    assert torch.equal(out["final"], ref["final"])
    assert torch.equal(out["traj"], ref["traj"]) and torch.equal(out["inputs"], ref["inputs"])
    assert out["total_iters"] == ref["total_iters"]
    assert int((out["dhat_traj"] != 0).sum()) == 0
    ok = (ref["fail_step"] < 0).float().mean().item()
    assert 0.05 < ok < 0.95


def test_config4_size(torch_cuda):
    """10^5 runs x 200 steps with a process disturbance: two calls identical, graph-replayed (warm_start 1) and host-sized
    (warm_start 2) steps agree, a run started from a non-finite d^ fails at step 0 and leaves every other run as it was."""
    torch = torch_cuda
    from carmpc_b200.observer import augmented_observer_gain
    ctl, bq, _ = _setup(np.ones(4))
    L1, L2 = augmented_observer_gain(ctl.A, ctl.C, np.ones(4), np.ones(3), W_AUG, V_OUT)
    R, T = 100_000, 200
    g = torch.Generator(device="cpu").manual_seed(0)
    lo, hi = torch.tensor(BOX_LO, dtype=torch.float64), torch.tensor(BOX_HI, dtype=torch.float64)
    x_init = (lo[:, None] + (hi - lo)[:, None] * torch.rand((4, R), generator=g, dtype=torch.float64)).cuda().contiguous()
    d_r = ((torch.rand(R, generator=g, dtype=torch.float64) - 0.5) * 0.02).cuda()

    def run(**kw):
        return bq.closed_loop_disturbance(x_init, T, ctl.A, ctl.B, ctl.C, np.ones(4), np.ones(3), L1, L2, x_ref=X_REF,
                                          Bd_plant=np.ones(4), d_plant=d_r, **kw)

    a, b = run(), run()
    for k in ("final", "dhat", "fail_step"):
        assert torch.equal(a[k], b[k]), k
    ok = a["fail_step"] < 0
    assert 0.01 < ok.float().mean().item() < 0.99
    assert torch.isfinite(a["dhat"][ok]).all() and torch.isfinite(a["final"][:, ok]).all()

    c = run(warm_start=2)
    same = c["fail_step"] == a["fail_step"]
    assert same.float().mean().item() >= 0.999
    both = same & ok
    assert (c["final"][:, both] - a["final"][:, both]).abs().max().item() <= 1e-6
    assert (c["dhat"][both] - a["dhat"][both]).abs().max().item() <= 1e-6

    bad = 17
    dh0 = torch.zeros(R, dtype=torch.float64, device="cuda")
    dh0[bad] = float("nan")
    n = run(dhat_init=dh0)
    assert int(n["fail_step"][bad]) == 0
    keep = torch.ones(R, dtype=torch.bool, device="cuda")
    keep[bad] = False
    assert torch.equal(n["fail_step"][keep], a["fail_step"][keep])
    assert torch.equal(n["final"][:, keep], a["final"][:, keep]) and torch.equal(n["dhat"][keep], a["dhat"][keep])


def test_sensor_offset_is_removed(torch_cuda):
    """The experiment the controller exists for: a constant sensor offset (Cd_p = 1_3, d_r = 0.05) with the output-only
    disturbance model Bd = 0, Cd = 1_3 and a stable gain.  Against plain output feedback on the same plant (L2 = 0,
    Bd = Cd = 0), d^ converges to the offset and x, v end nearer the goal.  The thresholds are the oracle's on the same
    runs (200 steps, exact QPs)."""
    torch = torch_cuda
    from carmpc_b200.lib.mpc import _C_XYV, _L_OBSERVER
    from carmpc_b200.observer import augmented_observer_gain
    ctl, bq, exact = _setup(np.zeros(4))
    L1, L2 = augmented_observer_gain(ctl.A, ctl.C, np.zeros(4), np.ones(3), W_AUG, V_OUT)
    dist = (np.zeros(4), np.ones(3), L1, L2)
    plain = (np.zeros(4), np.zeros(3), _L_OBSERVER.astype(float), np.zeros(3))
    rng = np.random.default_rng(1)
    R, steps, offset = 12, 200, 0.05
    x_init = rng.uniform(BOX_LO, BOX_HI, size=(R, 4))
    d_r = np.full(R, offset)
    res = {}
    for name, gains in (("dist", dist), ("plain", plain)):
        want = _oracle(ctl, exact, gains, x_init, steps, np.zeros(4), np.ones(3), d_r)
        out = _gpu(torch, bq, ctl, gains, x_init, steps, np.zeros(4), np.ones(3), d_r, want_traj=True, want_dhat=True)
        _assert_matches(out, want, min_alive=1)
        res[name] = (want, out)
    (wd, od), (wp, op) = res["dist"], res["plain"]
    alive_d, alive_p = wd[2] < 0, wp[2] < 0
    assert alive_d.sum() >= R // 2
    # oracle thresholds: how close d^ gets to the offset, how far x, v stay from the goal with / without the estimate
    d_err_oracle = np.abs(wd[1][alive_d] - offset).max()
    assert d_err_oracle < 0.1 * offset
    gd = od["dhat"].cpu().numpy()[alive_d]
    assert np.abs(gd - offset).max() <= d_err_oracle + 1e-6
    both = alive_d & alive_p
    assert both.sum() >= 1
    fd = np.abs(od["final"].cpu().numpy().T - X_REF)[:, [0, 3]]
    fp = np.abs(op["final"].cpu().numpy().T - X_REF)[:, [0, 3]]
    wfd = np.abs(wd[0] - X_REF)[:, [0, 3]]
    assert (fd[alive_d] <= wfd[alive_d].max(axis=0) + 1e-6).all()
    assert (fd[both].sum(1) < fp[both].sum(1)).all()
    assert (np.abs(wd[0] - X_REF)[both][:, [0, 3]].sum(1) < np.abs(wp[0] - X_REF)[both][:, [0, 3]].sum(1)).all()
