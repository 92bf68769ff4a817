"""No call leaves state behind on a QP handle: whatever a certified, seeded or closed-loop call asks for is passed with
that call, so a cold solve after them computes and reports exactly what it did before them."""
import numpy as np
import pytest

from conftest import make_env, make_controller

pytestmark = pytest.mark.gpu

X_REF = np.array([30.0, 1.5, 0.0, 0.0])
W_AUG = np.diag([1e-2] * 4 + [1e-3])
V_OUT = 1e-2 * np.eye(3)
BOX_LO, BOX_HI = [0, -2.5, -0.2, 0], [10, 2.5, 0.2, 3]
LW = np.diag([0.02, 0.02, 0.004, 0.02])
SV_STATE = [0.03, 0.03, 0.004, 0.03]


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "the GPU tests need a CUDA device"
    return torch


@pytest.fixture(scope="module")
def handle():
    """Disturbance-estimating controller (Bd = 1_4) on RoadEnv, horizon 20: one handle with a disturbance column."""
    from carmpc_b200.batch import BatchQP
    ctl = make_controller(make_env("RoadEnv"), 20, cls="MPCOutputFBWithDisturbance", init_state=[0, 0, 0, 0])
    ctl.Bd = np.ones(4)
    return ctl, BatchQP.from_controller(ctl)


@pytest.fixture(scope="module")
def grid(torch_cuda):
    """A 20 x 24 x 4 x 4 subset of the config-3 grid, its lattice seeds and a per-state disturbance."""
    torch = torch_cuda
    from carmpc_b200.grids import config3_axes, lattice_seeds, materialise_grid
    axes = config3_axes(20, 24, 4, 4)
    x0 = torch.stack(materialise_grid(axes, device="cuda")).contiguous()
    seed = torch.from_numpy(lattice_seeds([len(a) for a in axes], block=(2, 6, 1, 1))).cuda()
    c = torch.from_numpy(np.random.default_rng(5).uniform(-0.02, 0.02, size=x0.shape[1])).cuda()
    return x0, seed, c


def _bits(t):
    import torch
    return t.contiguous().view(torch.int64) if t.dtype == torch.float64 else t


def test_a_cold_solve_is_the_same_after_every_other_kind_of_call(torch_cuda, handle, grid):
    torch = torch_cuda
    from carmpc_b200.montecarlo import LoopNoise, plant_rows
    from carmpc_b200.observer import augmented_observer_gain
    ctl, bq = handle
    x0, seed, c = grid

    def cold():
        out = bq.solve(x0, x_ref=X_REF, c=c, want_u_full=True)
        torch.cuda.synchronize()
        return out, bq.polish_stats(), bq.last_stats()

    first, first_hist, first_last = cold()
    st = first["status"].cpu().numpy()
    assert (st == 0).sum() > len(st) // 10 and (st == 1).sum() > 0

    cert = bq.solve(x0, x_ref=X_REF, c=c, want_u_full=True, want_certificate=True)
    seeded = bq.solve(x0, x_ref=X_REF, c=c, want_u_full=True, seed=seed, want_certificate=True)
    torch.cuda.synchronize()
    assert seeded["seeded"] > 0
    del cert, seeded                           # the certificate buffers are freed before the calls below

    R, T = 256, 30
    g = torch.Generator(device="cpu").manual_seed(7)
    lo, hi = torch.tensor(BOX_LO, dtype=torch.float64), torch.tensor(BOX_HI, dtype=torch.float64)
    x_init = (lo[:, None] + (hi - lo)[:, None] * torch.rand((4, R), generator=g, dtype=torch.float64)).cuda().contiguous()
    d_r = torch.from_numpy(np.random.default_rng(3).uniform(-0.01, 0.01, size=R)).cuda()
    L1, L2 = augmented_observer_gain(ctl.A, ctl.C, np.ones(4), np.ones(3), W_AUG, V_OUT)
    loop = bq.closed_loop_disturbance(x_init, T, ctl.A, ctl.B, ctl.C, np.ones(4), np.ones(3), L1, L2, x_ref=X_REF,
                                      Bd_plant=np.ones(4), d_plant=d_r, warm_start=1)
    assert loop["total_iters"] > 0
    noisy = bq.closed_loop(x_init, T, ctl.A, ctl.B, x_ref=X_REF, warm_start=1,
                           noise=LoopNoise(LW, SV_STATE, seed=11), monitor=plant_rows(ctl))
    assert noisy["total_iters"] > 0

    again, again_hist, again_last = cold()
    for k in ("u0", "objective", "status", "iters", "u_full"):
        assert torch.equal(_bits(again[k]), _bits(first[k])), k
    assert again_hist == first_hist
    assert again_last == first_last
