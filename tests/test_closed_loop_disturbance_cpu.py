"""Disturbance-estimating output feedback without a GPU: the oracle's augmented observer against the controller's own,
the observer-gain helper (and the instability of the reference's gains), argument checks of
carmpc_closed_loop_disturbance."""
import ctypes
import math

import numpy as np
import pytest

from conftest import make_env, make_controller

W_AUG = np.diag([1e-2] * 4 + [1e-3])
V_OUT = 1e-2 * np.eye(3)


@pytest.fixture(scope="module")
def ctl():
    return make_controller(make_env("RoadEnv"), 20, cls="MPCOutputFBWithDisturbance", init_state=[5, -1.5, 0, 0])


def test_oracle_observer_step_is_the_controllers(ctl):
    """oracle.disturbance_observer_step == MPCOutputFBWithDisturbance.luenberger_observer, state by state."""
    import disturbance_oracle as dorc
    from carmpc_b200.observer import reference_disturbance_gains
    Bd, Cd, L1, L2 = reference_disturbance_gains(ctl)
    rng = np.random.default_rng(3)
    R = 50
    xhat = rng.uniform([0, -2.5, -0.3, 0], [30, 2.5, 0.3, 5], size=(R, 4))
    dhat = rng.uniform(-0.5, 0.5, size=R)
    u = rng.uniform([-2, -0.39], [2, 0.39], size=(R, 2))
    y = rng.uniform([0, -2.5, 0], [30, 2.5, 5], size=(R, 3))
    xn, dn = dorc.disturbance_observer_step(ctl.A, ctl.B, ctl.C.astype(float), Bd, Cd, L1, L2, xhat, dhat, u, y)
    for r in range(R):
        ctl.x_estimate, ctl.d_estimate, ctl.previous_u = xhat[r].copy(), float(dhat[r]), u[r].copy()
        want_x, want_d = ctl.luenberger_observer(y[r])
        np.testing.assert_allclose(xn[r], want_x, rtol=1e-13, atol=1e-12)
        assert abs(dn[r] - want_d) <= 1e-12 * max(1.0, abs(want_d))


def test_oracle_disturbed_qp_shifts_the_bounds_by_rows_times_ABd(ctl):
    """DisturbedQP: the fifth parameter moves exactly the state-space rows, by rows_x @ ABd (the controller's own
    disturbance_response), and leaves the input box and the cost alone."""
    import os
    from conftest import GOLDEN
    import disturbance_oracle as dorc
    from oracle import carmpc_oracle as orc
    Ab = np.load(os.path.join(GOLDEN, "terminal_sets", "RoadEnv_30_1.5_0_0.npy"))
    dq = dorc.DisturbedQP("RoadEnv", 20, Ab, ctl.Bd)
    np.testing.assert_allclose(dorc.disturbance_response(dq.A, ctl.Bd, 20), ctl.disturbance_response(), atol=1e-12)
    x = np.array([[10.0, 0.5, 0.1, 2.0, 0.0], [10.0, 0.5, 0.1, 2.0, 0.3]])
    shift = dq.rhs(x[1:]) - dq.rhs(x[:1])
    rows = np.vstack((orc.terminal_constraint(Ab, 20)[0], np.zeros((80, 84)), orc.state_constraint("RoadEnv", 20)[0]))
    np.testing.assert_allclose(shift[0], -0.3 * rows @ ctl.disturbance_response(), atol=1e-12)
    assert np.all(shift[0, len(Ab):len(Ab) + 80] == 0)
    np.testing.assert_array_equal(dq.lin(x[1:], np.zeros(5)), dq.lin(x[:1], np.zeros(5)))


def test_helper_gain_is_stable_and_the_reference_gain_is_not(ctl):
    """rho(A^ - L^ C^) < 1 for the steady-state predictor gain of both disturbance models (Bd = 1_4 / 0, Cd = 1_3);
    the reference's hard-coded L1, L2 = [1, 1, 1] give 3.31: its estimate diverges."""
    from carmpc_b200.observer import augmented_observer_gain, observer_error_radius, reference_disturbance_gains
    Bd, Cd, L1, L2 = reference_disturbance_gains(ctl)
    np.testing.assert_array_equal(Bd, np.ones(4))
    np.testing.assert_array_equal(Cd, np.ones(3))
    np.testing.assert_array_equal(L2, np.ones(3))
    rho_ref = observer_error_radius(ctl.A, ctl.C, Bd, Cd, L1, L2)
    assert rho_ref > 1.0 and abs(rho_ref - 3.31) < 0.01
    for bd, want in ((np.ones(4), 0.60), (np.zeros(4), 0.95)):
        g1, g2 = augmented_observer_gain(ctl.A, ctl.C, bd, np.ones(3), W_AUG, V_OUT)
        assert g1.shape == (4, 3) and g2.shape == (3,)
        rho = observer_error_radius(ctl.A, ctl.C, bd, np.ones(3), g1, g2)
        assert rho < 1.0 and abs(rho - want) < 0.01
    # a disturbance that neither moves the state nor shows in the output cannot be estimated
    with pytest.raises(ValueError):
        augmented_observer_gain(ctl.A, ctl.C, np.zeros(4), np.zeros(3), W_AUG, V_OUT)


def _call(lib, qp, dm, runs=4, steps=3, warm_start=1, dt=0.2, l1=3.5, A=True, ptr=16):
    mat = np.zeros(16)
    p = ctypes.c_void_p(ptr)
    return lib.carmpc_closed_loop_disturbance(qp, mat.ctypes.data if A else None, mat.ctypes.data, mat.ctypes.data,
                                              ctypes.byref(dm) if dm is not None else None, mat.ctypes.data, dt, l1,
                                              steps, warm_start, p, None, None, None, runs, p, None, p, None, None, None,
                                              None, None)


def _model():
    from carmpc_b200 import _capi
    dm = _capi.DisturbanceModel()
    dm.Bd[:] = [1.0] * 4
    dm.Cd[:] = [1.0] * 3
    dm.L2[:] = [0.1] * 3
    return dm


def test_entry_point_argument_errors(ctl):
    from carmpc_b200 import _capi
    from carmpc_b200.batch import BatchQP
    lib = _capi.load()
    bq = BatchQP.from_controller(ctl)
    dm = _model()
    assert _call(lib, None, dm) == -1 and b"QP handle" in lib.carmpc_last_error()
    assert _call(lib, bq._h, None) == -1
    assert _call(lib, bq._h, dm, A=False) == -1
    assert _call(lib, bq._h, dm, runs=-1) == -1
    assert _call(lib, bq._h, dm, steps=-1) == -1
    assert _call(lib, bq._h, dm, warm_start=3) == -1
    assert _call(lib, bq._h, dm, dt=0.0) == -1
    assert _call(lib, bq._h, dm, l1=-1.0) == -1
    assert _call(lib, bq._h, dm, ptr=0) == -1                  # runs > 0 needs x_init, final, fail_step
    for field, idx in (("L1", 5), ("L2", 0), ("Bd", 3), ("Cd", 1), ("Bd_plant", 2), ("Cd_plant", 0)):
        for bad in (math.nan, math.inf):
            m = _model()
            getattr(m, field)[idx] = bad
            assert _call(lib, bq._h, m) == -1 and b"finite" in lib.carmpc_last_error()
    # no runs: nothing to do, whatever the pointers
    total = ctypes.c_int64(7)
    mat = np.zeros(16)
    assert lib.carmpc_closed_loop_disturbance(bq._h, mat.ctypes.data, mat.ctypes.data, mat.ctypes.data, ctypes.byref(dm),
                                              mat.ctypes.data, 0.2, 3.5, 5, 1, None, None, None, None, 0, None, None,
                                              None, None, None, None, ctypes.byref(total), None) == 0
    assert total.value == 0


def test_host_only_handle_is_a_cuda_error(ctl):
    """A handle created without a CUDA device keeps its host setup; the loop fails loudly instead of computing."""
    try:
        import torch
        if torch.cuda.is_available():
            pytest.skip("a CUDA device is present: handles are not host-only here")
    except ImportError:
        pass
    from carmpc_b200 import _capi
    from carmpc_b200.batch import BatchQP
    lib = _capi.load()
    bq = BatchQP.from_controller(ctl)
    assert _call(lib, bq._h, _model()) == -2
    assert b"without a CUDA device" in lib.carmpc_last_error()
