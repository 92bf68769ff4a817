"""Noisy closed loops without a GPU: the Philox4x64-10 / Box-Muller restatement against numpy.random.Philox and the
normal distribution, the noise factors of montecarlo.LoopNoise, montecarlo.plant_rows against MPC.state_constraint, and
the argument checks of carmpc_closed_loop_stochastic."""
import ctypes
import math

import numpy as np
import pytest

from conftest import make_env, make_controller

ENVS = ("RoadEnv", "RoadOneCarEnv", "RoadMultipleCarsEnv")


def test_restated_generator_is_numpy_philox():
    """Random keys and counters, counters whose lowest words are 0 (the borrow of counter - 1 runs through them) and the
    top of the range; key 0 / counter 0 gives the published block."""
    import noise_oracle as no
    rng = np.random.default_rng(11)
    counters = [[0, 0, 0, 0], [0, 5, 1, 0], [0, 0, 0, 1], [1, 0, 0, 0], [2 ** 64 - 1, 2 ** 64 - 1, 0, 0],
                [2 ** 64 - 1] * 4, [123456, 199, 1, 0]]
    counters += [[int(v) for v in rng.integers(0, 2 ** 64, 4, dtype=np.uint64)] for _ in range(40)]
    keys = [[0, 0], [2 ** 64 - 1, 2 ** 64 - 1]] + [[int(v) for v in rng.integers(0, 2 ** 64, 2, dtype=np.uint64)]
                                                  for _ in range(10)]
    for c in counters:
        for k in keys:
            mine = no.philox4x64_10(*[np.uint64(v) for v in c], np.uint64(k[0]), np.uint64(k[1]))
            assert [int(w) for w in mine] == [int(w) for w in no.numpy_philox_block(c, k)], (c, k)
    zero = no.philox4x64_10(*[np.uint64(0)] * 6)
    assert [int(w) for w in zero] == [0x16554d9eca36314c, 0xdb20fe9d672d0fdc, 0xd7e772cee186176b, 0x7e68b68aec7ba23b]
    # the batched form is the scalar form, element by element
    runs = np.array([0, 1, 2 ** 40, 2 ** 63 + 5], dtype=np.uint64)
    batch = no.philox4x64_10(runs, np.uint64(7), np.uint64(1), np.uint64(0), np.uint64(99), np.uint64(0))
    for i, r in enumerate(runs):
        one = no.numpy_philox_block([int(r), 7, 1, 0], [99, 0])
        assert [int(w[i]) for w in batch] == [int(w) for w in one]


def test_box_muller_edges():
    """ua = 1 (a >> 11 all ones) gives exactly 0; ua = 2^-53 gives the largest radius, sqrt(106 ln 2); ub = 0 is cos 1."""
    import noise_oracle as no
    top = np.array([np.uint64(2 ** 64 - 1)])
    z0, z1 = no.box_muller(top, np.array([np.uint64(12345) << np.uint64(11)]))
    assert z0[0] == 0.0 and z1[0] == 0.0
    z0, z1 = no.box_muller(np.array([np.uint64(0)]), np.array([np.uint64(0)]))
    assert z0[0] == pytest.approx(math.sqrt(106 * math.log(2)), rel=1e-15) and z1[0] == 0.0


def test_restated_normals_are_standard_normal():
    """10^6 draws (250 000 runs x 4 components, one step): mean, covariance and a KS test."""
    from scipy import stats
    import noise_oracle as no
    z = no.normals(0, np.arange(250_000), 3, 0)
    assert np.abs(z.mean(0)).max() < 1e-2                  # 5 standard errors
    assert np.abs(np.cov(z.T) - np.eye(4)).max() < 1e-2
    assert stats.kstest(z.ravel(), "norm").pvalue > 1e-3
    # the two streams and neighbouring steps are different draws
    w = no.normals(0, np.arange(1000), 3, 1)
    assert abs(np.corrcoef(z[:1000].ravel(), w.ravel())[0, 1]) < 0.1
    assert not np.array_equal(no.normals(0, np.arange(10), 4, 0), z[:10])


def test_noise_factors_from_std_vectors_and_factors():
    from carmpc_b200.montecarlo import LoopNoise
    Lw, Lv = LoopNoise([0.1, 0.2, 0.01, 0.05], [0.3, 0.4, 0.5]).factors()
    np.testing.assert_array_equal(Lw, np.diag([0.1, 0.2, 0.01, 0.05]))
    np.testing.assert_array_equal(Lv, np.diag([0.3, 0.4, 0.5, 0.0]))
    F = np.arange(9.0).reshape(3, 3)
    _, Lv = LoopNoise(np.zeros(4), F).factors()
    np.testing.assert_array_equal(Lv[:3, :3], F)
    assert not Lv[3].any() and not Lv[:, 3].any()
    G = np.arange(16.0).reshape(4, 4)
    Lw, Lv = LoopNoise(G, G.T).factors()
    np.testing.assert_array_equal(Lw, G)
    np.testing.assert_array_equal(Lv, G.T)
    p = LoopNoise(G, np.ones(4), seed=2 ** 64 - 1, first_run=10 ** 12).params()
    assert p.seed == 2 ** 64 - 1 and p.first_run == 10 ** 12
    assert list(p.Lw) == G.ravel().tolist() and list(p.Lv) == np.eye(4).ravel().tolist()
    for bad in (np.ones(3), np.ones((3, 3)), np.ones(5), np.ones((4, 3)), [0.1, math.nan, 0, 0]):
        with pytest.raises(ValueError):
            LoopNoise(bad, np.ones(3)).factors()
    for bad in (np.ones(2), np.ones((2, 2)), np.ones((4, 3)), [math.inf, 0, 0]):
        with pytest.raises(ValueError):
            LoopNoise(np.ones(4), bad).factors()
    with pytest.raises(ValueError):
        LoopNoise(np.ones(4), np.ones(3), first_run=-1).params()
    with pytest.raises(ValueError):
        LoopNoise(np.ones(4), np.ones(3), seed=-1).params()


@pytest.mark.parametrize("env_name", ENVS)
def test_plant_rows_are_the_rows_state_constraint_imposes_on_x1(env_name):
    """plant_rows(controller) == the rows of MPC.state_constraint() that act on x(1) (row i N of each row type), in the
    same order; terminal_set=True appends the controller's terminal set."""
    from carmpc_b200.montecarlo import plant_rows
    ctl = make_controller(make_env(env_name), 10)
    A, b = ctl.state_constraint()
    N = ctl.N
    types = len(b) // N
    first = np.arange(types) * N
    assert np.all(A[first][:, :4] == 0) and np.all(A[first][:, 8:] == 0)
    rows = plant_rows(ctl)
    assert rows.shape == (types, 5) and rows.flags["C_CONTIGUOUS"]
    np.testing.assert_array_equal(rows[:, :4], A[first, 4:8])
    np.testing.assert_array_equal(rows[:, 4], b[first])
    At, bt = ctl.terminal_constraint()
    full = plant_rows(ctl, terminal_set=True)
    np.testing.assert_array_equal(full[:types], rows)
    np.testing.assert_array_equal(full[types:, :4], At[:, -4:])
    np.testing.assert_array_equal(full[types:, 4], bt)


def test_monitor_argument_forms():
    from carmpc_b200.batch import BatchQP
    Ab = np.arange(10.0).reshape(2, 5)
    np.testing.assert_array_equal(BatchQP._monitor_rows(Ab), Ab)
    np.testing.assert_array_equal(BatchQP._monitor_rows((Ab[:, :4], Ab[:, 4])), Ab)
    for bad in (np.zeros((0, 5)), np.zeros((513, 5)), np.zeros((3, 4)), np.full((2, 5), math.nan),
                (np.zeros((2, 4)), np.zeros(3))):
        with pytest.raises(ValueError):
            BatchQP._monitor_rows(bad)


# ---- carmpc_closed_loop_stochastic argument checks ----------------------------------------------------------------
@pytest.fixture(scope="module")
def handle():
    from carmpc_b200.batch import BatchQP
    ctl = make_controller(make_env("RoadEnv"), 10, cls="MPCOutputFBWithDisturbance", init_state=[5, -1.5, 0, 0])
    return BatchQP.from_controller(ctl)


def _model():
    from carmpc_b200 import _capi
    dm = _capi.DisturbanceModel()
    dm.Bd[:] = [1.0] * 4
    dm.Cd[:] = [1.0] * 3
    dm.L2[:] = [0.1] * 3
    return dm


def _noise(**kw):
    from carmpc_b200 import _capi
    nz = _capi.LoopNoiseParams()
    nz.Lw[:] = (0.01 * np.eye(4)).ravel().tolist()
    nz.Lv[:] = (0.02 * np.eye(4)).ravel().tolist()
    for k, v in kw.items():
        setattr(nz, k, v)
    return nz


_ROWS = np.array([[0.0, 1.0, 0.0, 0.0, 2.5], [0.0, -1.0, 0.0, 0.0, 2.5]])


def _call(lib, qp, mode=1, dm="model", noise="noise", rows=_ROWS, monitor_rows=None, outs=(True, True, True), runs=4,
          steps=3, warm_start=1, dt=0.2, l1=3.5, C=True, L=True, ptr=16):
    mat = np.zeros(16)
    p = ctypes.c_void_p(ptr)
    if isinstance(dm, str):
        dm = _model()
    if isinstance(noise, str):
        noise = _noise()
    if monitor_rows is None:
        monitor_rows = len(rows) if rows is not None else 0
    rows_ptr = np.ascontiguousarray(rows).ctypes.data if rows is not None else None
    vs, vr, vp = (ctypes.c_void_p(64) if o else None for o in outs)
    return lib.carmpc_closed_loop_stochastic(
        qp, mode, mat.ctypes.data, mat.ctypes.data, mat.ctypes.data if C else None, mat.ctypes.data if L else None,
        ctypes.byref(dm) if dm is not None else None, mat.ctypes.data, dt, l1, steps, warm_start, p, None, None, None, runs,
        p, None, p, None, None, None, ctypes.byref(noise) if noise is not None else None, rows_ptr, monitor_rows, vs, vr,
        vp, None, None)


def test_entry_point_argument_errors(handle):
    from carmpc_b200 import _capi
    lib = _capi.load()
    h = handle._h
    err = lambda: lib.carmpc_last_error()   # noqa: E731
    assert _call(lib, None) == -1 and b"QP handle" in err()
    for mode in (-1, 3):
        assert _call(lib, h, mode=mode) == -1
    assert _call(lib, h, mode=2, dm=None) == -1 and b"disturbance model" in err()
    assert _call(lib, h, mode=1, L=False) == -1
    assert _call(lib, h, mode=2, C=False) == -1
    assert _call(lib, h, runs=-1) == -1
    assert _call(lib, h, steps=-1) == -1
    assert _call(lib, h, warm_start=3) == -1
    assert _call(lib, h, dt=0.0) == -1 and _call(lib, h, l1=-1.0) == -1
    assert _call(lib, h, ptr=0) == -1                       # runs > 0 needs x_init, final, fail_step
    # non-finite noise factors and gains
    for field in ("Lw", "Lv"):
        for idx in (0, 7, 15):
            for bad in (math.nan, math.inf, -math.inf):
                nz = _noise()
                getattr(nz, field)[idx] = bad
                assert _call(lib, h, noise=nz) == -1 and b"finite" in err()
    for field, idx in (("L1", 5), ("L2", 0), ("Bd", 3), ("Cd", 1), ("Bd_plant", 2), ("Cd_plant", 0)):
        m = _model()
        getattr(m, field)[idx] = math.nan
        assert _call(lib, h, mode=2, dm=m) == -1 and b"finite" in err()
    assert _call(lib, h, noise=_noise(first_run=-1)) == -1 and b"first_run" in err()
    assert _call(lib, h, noise=_noise(first_run=2 ** 63 - 2)) == -1           # first_run + runs overflows
    # monitor rows
    assert _call(lib, h, monitor_rows=0) == -1 and b"monitor_rows" in err()
    assert _call(lib, h, rows=np.tile(_ROWS, (257, 1)), monitor_rows=513) == -1
    for bad in (math.nan, math.inf):
        r = _ROWS.copy()
        r[1, 4] = bad
        assert _call(lib, h, rows=r) == -1 and b"finite" in err()
        r = _ROWS.copy()
        r[0, 2] = bad
        assert _call(lib, h, rows=r) == -1
    for outs in ((True, False, False), (False, True, False), (False, False, True)):
        assert _call(lib, h, rows=None, outs=outs) == -1 and b"without monitor rows" in err()
    assert _call(lib, h, rows=None, monitor_rows=2, outs=(False, False, False)) == -1
    # no runs: nothing to do once the arguments are valid
    total = ctypes.c_int64(7)
    mat = np.zeros(16)
    assert lib.carmpc_closed_loop_stochastic(h, 0, mat.ctypes.data, mat.ctypes.data, None, None, None, mat.ctypes.data,
                                             0.2, 3.5, 5, 1, None, None, None, None, 0, None, None, None, None, None,
                                             None, None, None, 0, None, None, None, ctypes.byref(total), None) == 0
    assert total.value == 0


def test_host_only_handle_is_a_cuda_error(handle):
    """Valid arguments on a handle created without a CUDA device: the loop fails loudly instead of computing."""
    try:
        import torch
        if torch.cuda.is_available():
            pytest.skip("a CUDA device is present: handles are not host-only here")
    except ImportError:
        pass
    from carmpc_b200 import _capi
    lib = _capi.load()
    for mode in (0, 1, 2):
        assert _call(lib, handle._h, mode=mode) == -2
        assert b"without a CUDA device" in lib.carmpc_last_error()
    assert _call(lib, handle._h, noise=None, rows=None, outs=(False, False, False)) == -2
