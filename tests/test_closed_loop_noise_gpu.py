"""Closed loops with random process and measurement noise and a monitor of the true plant (carmpc_closed_loop) on RoadEnv,
horizon 20: zero noise factors and a monitor leave the loop bit for bit as it is without them; the device draws are the
restated Philox4x64-10 normals; parity with the restated noisy loop (exact QPs) in the three modes; the monitor's outputs
equal the C membership oracle's on the stored trajectories; reproducibility across calls and run-set splits; config-4
size."""
import os

import numpy as np
import pytest

from conftest import GOLDEN, make_env, make_controller

pytestmark = pytest.mark.gpu

X_REF = np.array([30.0, 1.5, 0.0, 0.0])
BOX_LO, BOX_HI = [0, -2.5, -0.2, 0], [10, 2.5, 0.2, 3]
W_AUG = np.diag([1e-2] * 4 + [1e-3])
V_OUT = 1e-2 * np.eye(3)
# process noise: a full factor (row-major order matters); measurement noise as std vectors
LW = np.array([[0.02, 0.0, 0.0, 0.0], [0.005, 0.02, 0.0, 0.0], [0.0, 0.001, 0.004, 0.0], [0.003, 0.0, 0.0, 0.02]])
SV_STATE = [0.03, 0.03, 0.004, 0.03]
SV_OUT = [0.03, 0.03, 0.03]


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "the GPU tests need a CUDA device"
    return torch


@pytest.fixture(scope="module")
def plain():
    """Output-feedback controller, its handle and the oracle's exact QP."""
    from carmpc_b200.batch import BatchQP
    from oracle import carmpc_oracle as orc
    ctl = make_controller(make_env("RoadEnv"), 20, cls="MPCOutputFB", init_state=[0, 0, 0, 0])
    Ab = np.load(os.path.join(GOLDEN, "terminal_sets", "RoadEnv_30_1.5_0_0.npy"))
    oq = orc.CondensedQP("RoadEnv", 20, Ab)

    def exact(x, d):
        u, obj, st, *_ = orc.qp_solve_exact(oq, x, X_REF)
        return u[:, :2], st

    return ctl, BatchQP.from_controller(ctl), exact


@pytest.fixture(scope="module")
def dist():
    """Disturbance-estimating controller (Bd = 1_4), its handle, the oracle's exact disturbed QP and stable gains."""
    from carmpc_b200.batch import BatchQP
    from carmpc_b200.observer import augmented_observer_gain
    import disturbance_oracle as dorc
    from oracle import carmpc_oracle as orc
    ctl = make_controller(make_env("RoadEnv"), 20, cls="MPCOutputFBWithDisturbance", init_state=[0, 0, 0, 0])
    ctl.Bd = np.ones(4)
    Ab = np.load(os.path.join(GOLDEN, "terminal_sets", "RoadEnv_30_1.5_0_0.npy"))
    dq = dorc.DisturbedQP("RoadEnv", 20, Ab, ctl.Bd)

    def exact(x, d):
        u, obj, st, *_ = orc.qp_solve_exact(dq, np.hstack((x, d[:, None])), np.append(X_REF, 0.0))
        return u[:, :2], st

    L1, L2 = augmented_observer_gain(ctl.A, ctl.C, np.ones(4), np.ones(3), W_AUG, V_OUT)
    return ctl, BatchQP.from_controller(ctl), exact, (np.ones(4), np.ones(3), L1, L2)


def _x_init(torch, R, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    lo, hi = torch.tensor(BOX_LO, dtype=torch.float64), torch.tensor(BOX_HI, dtype=torch.float64)
    return (lo[:, None] + (hi - lo)[:, None] * torch.rand((4, R), generator=g, dtype=torch.float64)).cuda().contiguous()


def _alive_at(fail, steps):
    """(steps, R) bool: the run was still running at the start of step k."""
    k = np.arange(steps)[:, None]
    return (fail[None, :] < 0) | (fail[None, :] >= k)


def _process_draws(out, x_init):
    """w_k = traj[k] - Euler(traj[k-1], u_log[k-1]) ((steps, R, 4); traj[-1] = x_init, u_log[-1] = 0)."""
    from oracle.carmpc_oracle import plant_step
    traj = out["traj"].cpu().numpy().transpose(0, 2, 1)
    u = out["inputs"].cpu().numpy().transpose(0, 2, 1)
    prev = np.concatenate((x_init.cpu().numpy().T[None], traj[:-1]))
    uprev = np.concatenate((np.zeros_like(u[:1]), u[:-1]))
    return np.stack([traj[k] - plant_step(prev[k], uprev[k]) for k in range(len(traj))])


def _assert_draws(out, x_init, Lw, seed, first_run=0):
    import noise_oracle as no
    w = _process_draws(out, x_init)
    steps, R = w.shape[:2]
    alive = _alive_at(out["fail_step"].cpu().numpy(), steps)
    ids = first_run + np.arange(R)
    for k in range(steps):
        want = no.normals(seed, ids, k, 0) @ Lw.T
        assert np.abs(w[k][alive[k]] - want[alive[k]]).max() <= 1e-12, k
    return alive


# ---- 1. off is off ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("warm_start", [0, 1, 2])
def test_zero_noise_and_monitor_change_nothing(torch_cuda, plain, dist, warm_start):
    """Zero noise factors, a monitor, or both change nothing: torch.equal to the plain loop in modes 0, 1 and 2, 2000
    runs x 60 steps (graph-replayed steps with warm_start 1)."""
    torch = torch_cuda
    from carmpc_b200.lib.mpc import _C_XYV, _L_OBSERVER
    from carmpc_b200.montecarlo import LoopNoise, plant_rows
    ctl, bq, _ = plain
    dctl, dbq, _, gains = dist
    R, T = 2000, 60
    x0 = _x_init(torch, R, 1)
    d_r = ((torch.rand(R, generator=torch.Generator().manual_seed(2), dtype=torch.float64) - 0.5) * 0.02).cuda()
    zero = LoopNoise(np.zeros(4), np.zeros(4), seed=5)
    rows = plant_rows(ctl)
    keys = ("final", "fail_step", "traj", "inputs")

    for mode in (0, 1):
        C, L = (_C_XYV, _L_OBSERVER) if mode else (None, None)
        ref = bq.closed_loop(x0, T, ctl.A, ctl.B, x_ref=X_REF, C=C, L=L, warm_start=warm_start, want_traj=True,
                             want_inputs=True)
        ok = (ref["fail_step"] < 0).float().mean().item()
        assert 0.05 < ok < 0.95
        for noise, monitor in ((zero, None), (None, rows), (zero, rows)):
            o = bq.closed_loop(x0, T, ctl.A, ctl.B, x_ref=X_REF, C=C, L=L, warm_start=warm_start, want_traj=True,
                               want_inputs=True, noise=noise, monitor=monitor)
            for k in keys:
                assert torch.equal(o[k], ref[k]), (mode, k, noise is None)

    Bd, Cd, L1, L2 = gains
    dkw = dict(x_ref=X_REF, Bd_plant=np.ones(4), d_plant=d_r, warm_start=warm_start, want_traj=True, want_inputs=True,
               want_dhat=True)
    ref = dbq.closed_loop_disturbance(x0, T, dctl.A, dctl.B, dctl.C, Bd, Cd, L1, L2, **dkw)
    o = dbq.closed_loop_disturbance(x0, T, dctl.A, dctl.B, dctl.C, Bd, Cd, L1, L2, noise=zero, monitor=rows, **dkw)
    for k in keys + ("dhat", "dhat_traj"):
        assert torch.equal(o[k], ref[k]), k


# ---- 2. the draws -----------------------------------------------------------------------------------------------------
def test_process_draws_are_the_specified_ones(torch_cuda, plain):
    """State feedback with process noise only: w_k = traj[k] - Euler(traj[k-1], u_log[k-1]) equals Lw z_w of the
    restatement within 1e-12 for every running run and step, with warm_start 0 / 1 (graph-replayed steps) / 2."""
    torch = torch_cuda
    from carmpc_b200.montecarlo import LoopNoise
    ctl, bq, _ = plain
    R, T, seed = 700, 60, 12345
    x0 = _x_init(torch, R, 3)
    noise = LoopNoise(LW, np.zeros(4), seed=seed)
    for ws in (0, 1, 2):
        out = bq.closed_loop(x0, T, ctl.A, ctl.B, x_ref=X_REF, warm_start=ws, want_traj=True, want_inputs=True,
                             noise=noise)
        alive = _assert_draws(out, x0, LW, seed)
        assert alive[-1].sum() >= R // 20, ws


# ---- 3. oracle parity -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", [0, 1, 2])
def test_matches_the_restated_noisy_loop(torch_cuda, plain, dist, mode):
    """16 runs x 25 steps with process and measurement noise and the plant rows as monitor: fail_step and violation_step
    equal to the restated loop's (exact QPs), trajectories within 1e-6."""
    torch = torch_cuda
    import noise_oracle as no
    from carmpc_b200.lib.mpc import _C_XYV, _L_OBSERVER
    from carmpc_b200.montecarlo import LoopNoise, plant_rows
    R, T, seed = 16, 25, 2024
    x_init = np.random.default_rng(0).uniform(BOX_LO, BOX_HI, size=(R, 4))
    x0 = torch.from_numpy(np.ascontiguousarray(x_init.T)).cuda()
    if mode == 2:
        ctl, bq, exact, gains = dist
        d_r = np.random.default_rng(1).uniform(-0.01, 0.01, size=R)
        noise = LoopNoise(LW, SV_OUT, seed=seed)
    else:
        ctl, bq, exact = plain
        noise = LoopNoise(LW, SV_STATE if mode == 0 else SV_OUT, seed=seed)
    Lw, Lv = noise.factors()
    rows = plant_rows(ctl)
    if mode == 2:
        Bd, Cd, L1, L2 = gains
        want = no.noisy_closed_loop(2, ctl.A, ctl.B, ctl.C, None, x_init, T, exact, Lw, Lv, seed, monitor=rows,
                                    dist=(Bd, Cd, L1, L2, np.ones(4), np.zeros(3), d_r))
        out = bq.closed_loop_disturbance(x0, T, ctl.A, ctl.B, ctl.C, Bd, Cd, L1, L2, x_ref=X_REF, Bd_plant=np.ones(4),
                                         d_plant=torch.from_numpy(d_r).cuda(), want_traj=True, want_inputs=True,
                                         want_dhat=True, noise=noise, monitor=rows)
        np.testing.assert_allclose(out["dhat_traj"].cpu().numpy(), want["dhat_traj"], atol=1e-6)
    else:
        C, L = (_C_XYV, _L_OBSERVER) if mode else (None, None)
        want = no.noisy_closed_loop(mode, ctl.A, ctl.B, C, L, x_init, T, exact, Lw, Lv, seed, monitor=rows)
        out = bq.closed_loop(x0, T, ctl.A, ctl.B, x_ref=X_REF, C=C, L=L, want_traj=True, want_inputs=True, noise=noise,
                             monitor=rows)
    fail = out["fail_step"].cpu().numpy()
    np.testing.assert_array_equal(fail, want["fail_step"])
    np.testing.assert_array_equal(out["violation_step"].cpu().numpy(), want["violation_step"])
    assert np.abs(out["traj"].cpu().numpy().transpose(0, 2, 1) - want["traj"]).max() <= 1e-6
    np.testing.assert_allclose(out["final"].cpu().numpy().T, want["final"], atol=1e-6)
    assert (fail < 0).sum() >= 2
    assert out["total_iters"] > 0


# ---- 4. monitor bits --------------------------------------------------------------------------------------------------
def test_monitor_outputs_equal_the_membership_oracle(torch_cuda, plain):
    """2000 runs x 60 steps of output feedback with noise, monitored against the plant rows and the terminal set (so that
    most runs violate some row at some step): violation_step, violation_row and violations_per_step recomputed from the
    stored trajectory with oracle.c_oracle.membership_bits (the same fma chain; one row at a time for the row)."""
    torch = torch_cuda
    from oracle import c_oracle
    from carmpc_b200.lib.mpc import _C_XYV, _L_OBSERVER
    from carmpc_b200.montecarlo import LoopNoise, plant_rows
    ctl, bq, _ = plain
    R, T = 2000, 60
    x0 = _x_init(torch, R, 4)
    rows = plant_rows(ctl, terminal_set=True)
    out = bq.closed_loop(x0, T, ctl.A, ctl.B, x_ref=X_REF, C=_C_XYV, L=_L_OBSERVER, want_traj=True,
                         noise=LoopNoise(3 * LW, SV_OUT, seed=9), monitor=rows)
    traj = out["traj"].cpu().numpy()                                  # (T, 4, R)
    pts = [np.ascontiguousarray(traj[:, c].ravel()) for c in range(4)]
    n = T * R

    def outside(Ab):
        bits, _ = c_oracle.membership_bits(Ab, *pts)
        return ~c_oracle.unpack_bits(bits, n).reshape(T, R)

    viol = outside(rows)
    per_row = np.stack([outside(rows[r:r + 1]) for r in range(len(rows))])     # (rows, T, R)
    assert np.array_equal(viol, per_row.any(0))
    viol &= _alive_at(out["fail_step"].cpu().numpy(), T)
    first = np.where(viol.any(0), np.argmax(viol, axis=0), -1)
    row = np.where(first >= 0, np.argmax(per_row[:, np.maximum(first, 0), np.arange(R)], axis=0), -1)
    np.testing.assert_array_equal(out["violation_step"].cpu().numpy(), first)
    np.testing.assert_array_equal(out["violation_row"].cpu().numpy(), row)
    np.testing.assert_array_equal(out["violations_per_step"].cpu().numpy(), viol.sum(1))
    assert (first >= 0).sum() > R // 2 and len(np.unique(row[row >= 0])) >= 2


# ---- 5. reproducibility -----------------------------------------------------------------------------------------------
def test_reproducible_across_calls_and_run_set_splits(torch_cuda, plain):
    """Two calls are bit-identical; the same runs split into two calls with first_run offsets draw the same noise and
    give equal fail_step / violation_step, trajectories within 1e-9."""
    torch = torch_cuda
    from carmpc_b200.montecarlo import LoopNoise, plant_rows
    ctl, bq, _ = plain
    R, T, seed, cut = 1000, 60, 77, 389
    x0 = _x_init(torch, R, 5)
    rows = plant_rows(ctl)

    def run(x, first_run=0):
        return bq.closed_loop(x, T, ctl.A, ctl.B, x_ref=X_REF, want_traj=True, want_inputs=True, monitor=rows,
                              noise=LoopNoise(LW, SV_STATE, seed=seed, first_run=first_run))

    a, b = run(x0), run(x0)
    for k in a:
        if k != "total_iters":
            assert torch.equal(a[k], b[k]), k
    assert a["total_iters"] == b["total_iters"]
    parts = [(0, run(x0[:, :cut].contiguous())), (cut, run(x0[:, cut:].contiguous(), first_run=cut))]
    for off, p in parts:
        sl = slice(off, off + p["fail_step"].numel())
        _assert_draws(p, x0[:, sl], LW, seed, first_run=off)
        assert torch.equal(p["fail_step"], a["fail_step"][sl])
        assert torch.equal(p["violation_step"], a["violation_step"][sl])
        assert (p["traj"] - a["traj"][:, :, sl]).abs().max().item() <= 1e-9
    assert (a["violation_step"] >= 0).any()


# ---- 6. config-4 size -------------------------------------------------------------------------------------------------
def test_config4_size(torch_cuda, plain):
    """10^5 runs x 200 steps of output feedback with noise and the plant rows: finite results, violations per step never
    above the runs still running, two calls identical."""
    torch = torch_cuda
    from carmpc_b200.lib.mpc import _C_XYV, _L_OBSERVER
    from carmpc_b200.montecarlo import LoopNoise, plant_rows
    ctl, bq, _ = plain
    R, T = 100_000, 200
    x0 = _x_init(torch, R, 0)

    def run():
        return bq.closed_loop(x0, T, ctl.A, ctl.B, x_ref=X_REF, C=_C_XYV, L=_L_OBSERVER, monitor=plant_rows(ctl),
                              noise=LoopNoise(LW, SV_OUT, seed=1))

    a, b = run(), run()
    for k in ("final", "fail_step", "violation_step", "violation_row", "violations_per_step"):
        assert torch.equal(a[k], b[k]), k
    fail = a["fail_step"].cpu().numpy()
    ok = fail < 0
    assert 0.01 < ok.mean() < 0.99
    assert torch.isfinite(a["final"]).all()
    per = a["violations_per_step"].cpu().numpy()
    running = _alive_at(fail, T).sum(1)
    assert (per >= 0).all() and (per <= running).all()
    vs = a["violation_step"].cpu().numpy()
    assert (np.bincount(vs[vs >= 0], minlength=T) <= per).all()
    assert ((vs >= 0) == (a["violation_row"].cpu().numpy() >= 0)).all()
