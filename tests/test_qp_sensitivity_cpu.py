"""Sensitivities of batched QP solutions without a GPU: the numpy restatement (sensitivity_check.py) against central finite
differences of the oracle's exact QP, its flags on hand-built QPs, and the argument errors of carmpc_qp_sensitivity."""
import ctypes
import os

import numpy as np
import pytest

from conftest import GOLDEN, TERMINAL_SETS
from sensitivity_check import DEPENDENT, DERIVATIVE, WEAK, reference_stack, sensitivity_numpy


# ---------------------------------------------------------------------------------------------------------------------
# hand-built QPs around a known KKT point (shared with test_qp_sensitivity_gpu.py)
def hand_built_cases():
    """name -> (problem dict in the restatement's two-sided form, x0, u, certificate row, expected flags).  Rows whose G
    part is zero are u-independent rows; every problem has xref = 0."""
    rng = np.random.default_rng(3)
    n = 3
    Mr = rng.normal(size=(n, n))
    H = Mr @ Mr.T + n * np.eye(n)
    x0 = np.array([0.7, -0.4, 0.2, 1.1])
    u = np.array([0.3, -0.2, 0.5])
    G0 = np.array([[1.0, 0.5, -0.3], [0.2, -1.0, 0.4], [-0.6, 0.3, 1.0]])
    Gx0 = rng.normal(size=(3, 4))
    Gc0 = np.array([0.5, -0.2, 0.1])

    def build(G, Gx, Gc, active, lam, box_active=(), lam_b=(), at_bound=(), box_at=(), lo_finite=()):
        t = G @ u + Gx @ x0
        hi, lo = t + 1.0, np.full(len(t), -np.inf)
        for i in lo_finite:
            lo[i] = t[i] - 2.0
        for i in list(active) + list(at_bound):
            hi[i] = t[i]
        lb, ub = u - 1.0, u + 1.0
        for j in list(box_active) + list(box_at):
            ub[j] = u[j]
        y = np.zeros(len(t) + n)
        y[list(active)] = lam
        y[[len(t) + j for j in box_active]] = lam_b
        q = -(H @ u + G.T @ y[:len(t)] + y[len(t):])
        F = np.outer(q, x0) / (x0 @ x0)
        return dict(H=H, F=F, G=G, Gx=Gx, Gc=Gc, lo=lo, hi=hi, lb=lb, ub=ub), y

    cases = {}
    p, y = build(G0, Gx0, Gc0, [], [], lo_finite=[2])
    cases["interior"] = (p, y, DERIVATIVE)
    p, y = build(G0, Gx0, Gc0, [0], [0.8], lo_finite=[2])
    cases["one strongly active row"] = (p, y, DERIVATIVE)
    p, y = build(G0, Gx0, Gc0, [0], [0.8], at_bound=[1])
    cases["weakly active row (at its bound, no multiplier)"] = (p, y, WEAK)
    p, y = build(G0, Gx0, Gc0, [0, 1], [0.8, 1e-13])
    cases["weakly active row (multiplier below the sign tolerance)"] = (p, y, WEAK)
    G = np.vstack((G0, 2.0 * G0[:1]))
    Gx = np.vstack((Gx0, 2.0 * Gx0[:1]))
    Gc = np.concatenate((Gc0, 2.0 * Gc0[:1]))
    p, y = build(G, Gx, Gc, [0, 3], [0.5, 0.15])
    cases["duplicated (dependent) rows"] = (p, y, DEPENDENT)
    p, y = build(G0, Gx0, Gc0, [], [], box_active=[1], lam_b=[0.3])
    cases["bound on the box only"] = (p, y, DERIVATIVE)
    p, y = build(G0, Gx0, Gc0, [], [], box_active=[1], lam_b=[0.3], box_at=[2])
    cases["box row at its bound without a multiplier"] = (p, y, WEAK)
    G = np.vstack((G0, np.zeros((1, n))))
    Gx = np.vstack((Gx0, rng.normal(size=(1, 4))))
    Gc = np.concatenate((Gc0, [0.3]))
    p, y = build(G, Gx, Gc, [0], [0.8], at_bound=[3])
    cases["u-independent row at its bound"] = (p, y, WEAK)
    p, y = build(G, Gx, Gc, [0], [0.8])
    cases["u-independent row inside its bounds"] = (p, y, DERIVATIVE)
    return {k: (p, x0, u, y, f) for k, (p, y, f) in cases.items()}


def _restate(p, x0, u, y, c=0.0):
    return sensitivity_numpy(p["H"], p["F"], p["G"], p["Gx"], p["lo"], p["hi"], p["lb"], p["ub"], x0[None], u[None],
                             y[None], Gc=p["Gc"], c=np.array([c]))


@pytest.mark.parametrize("name", list(hand_built_cases()))
def test_restatement_sets_the_expected_flag_on_hand_built_qps(name):
    p, x0, u, y, want = hand_built_cases()[name]
    jac, grad, flags = _restate(p, x0, u, y)
    assert flags[0] == want, (name, flags[0])
    assert np.isfinite(jac).all() and np.isfinite(grad).all()
    # the point is a KKT point of the stated problem: H u + F x0 + A'y = 0
    R = len(p["hi"])
    assert np.abs(p["H"] @ u + p["F"] @ x0 + p["G"].T @ y[:R] + y[R:]).max() <= 1e-12


def test_restatement_on_hand_built_qps_equals_its_own_finite_differences():
    """On the nondegenerate cases the affine piece of S is the solution: re-solving the equality-constrained QP at p +- h
    reproduces J and dV exactly (central differences of an affine map and of a quadratic)."""
    for name, (p, x0, u, y, want) in hand_built_cases().items():
        if want != DERIVATIVE:
            continue
        R, n = len(p["hi"]), len(u)
        S = np.flatnonzero(y != 0)
        A = np.vstack((p["G"], np.eye(n)))[S]
        Ax = np.vstack((p["Gx"], np.zeros((n, 4))))[S]
        Ac = np.concatenate((p["Gc"], np.zeros(n)))[S]
        b = A @ u + Ax @ x0                                  # the active bounds (c = 0 at the centre)

        def solve(xx, cc):
            K = np.block([[p["H"], A.T], [A, np.zeros((len(S), len(S)))]])
            sol = np.linalg.solve(K, np.concatenate((-p["F"] @ xx, b - Ax @ xx - Ac * cc)))
            uu = sol[:n]
            return uu, 0.5 * uu @ p["H"] @ uu + (p["F"] @ xx) @ uu

        jac, grad, _ = _restate(p, x0, u, y)
        h = 1e-4
        for k in range(5):
            e = np.zeros(5)
            e[k] = h
            (up, vp), (um, vm) = solve(x0 + e[:4], e[4]), solve(x0 - e[:4], -e[4])
            np.testing.assert_allclose((up - um) / (2 * h), jac[0, :, k], rtol=0, atol=1e-9, err_msg=name)
            assert abs((vp - vm) / (2 * h) - grad[0, k]) <= 1e-8 * max(1.0, abs(grad[0, k])), name


# ---------------------------------------------------------------------------------------------------------------------
def _oracle_polished(oq, X, goal):
    """u and the oracle's own active-set multipliers (its row order: terminal, input box [I; -I], state rows)."""
    from oracle import carmpc_oracle as orc
    ua, ya, st = orc.qp_solve_admm(oq, X, goal)
    U, L, ok = np.zeros_like(ua), np.zeros_like(ya), np.zeros(len(X), dtype=bool)
    for k in range(len(X)):
        U[k], L[k], ok[k] = orc.qp_polish(oq, X[k:k + 1], goal, ua[k], ya[k])
    return U, L, ok & (st == 0)


def test_restatement_equals_central_differences_of_the_oracle_qp():
    """RoadOneCarEnv N = 10: J and dV of the restatement (golden matrices, the oracle's certificate on the reference's
    one-sided stack) equal central differences of oracle.qp_solve_exact at states whose nine solves share the centre's
    active set and whose restatement flag is DERIVATIVE."""
    from oracle import carmpc_oracle as orc
    d = np.load(os.path.join(GOLDEN, "qp_RoadOneCarEnv_N10.npz"))
    H, F, G, Gx, lo, hi, lb, ub, _ = reference_stack(d)
    goal = d["goal"]
    Ab = np.load(os.path.join(TERMINAL_SETS, "RoadOneCarEnv_29.9_1.5_0_0.npy"))
    oq = orc.CondensedQP("RoadOneCarEnv", 10, Ab)
    n, nt = oq.n, len(d["bt"])
    np.testing.assert_allclose(oq.H, H, rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(np.vstack((oq.G[:nt], oq.G[nt + 2 * n:])), G, rtol=1e-12, atol=1e-12)
    rng = np.random.default_rng(7)
    X = goal + rng.uniform(-1, 1, size=(120, 4)) * np.array([8.0, 1.2, 0.2, 2.0])
    U, L, ok = _oracle_polished(oq, X, goal)
    cert = np.hstack((L[:, :nt], L[:, nt + 2 * n:], L[:, nt:nt + n] - L[:, nt + n:nt + 2 * n]))
    jac, grad, flags = sensitivity_numpy(H, F, G, Gx, lo, hi, lb, ub, X, U, cert, status=np.where(ok, 0, 1))
    h = 1e-4
    cand = np.flatnonzero(ok & (flags == DERIVATIVE))[:12]
    assert len(cand) >= 8, f"only {len(cand)} nondegenerate states"
    checked = 0
    for b in cand:
        P = np.repeat(X[b][None], 8, axis=0)
        for k in range(4):
            P[2 * k, k] += h
            P[2 * k + 1, k] -= h
        Up, Lp, okp = _oracle_polished(oq, P, goal)
        if not okp.all() or not all(np.array_equal(Lp[i] != 0, L[b] != 0) for i in range(8)):
            continue                                    # a perturbation crosses a piece boundary
        ue, obje, ste, _, _ = orc.qp_solve_exact(oq, P, goal)
        assert (ste == 0).all()
        fd = np.stack([(ue[2 * k] - ue[2 * k + 1]) / (2 * h) for k in range(4)], axis=1)
        scale = np.maximum(np.abs(jac[b, :, :4]).max(axis=0), 1e-3)
        err = np.abs(fd - jac[b, :, :4]).max(axis=0) / scale
        assert err.max() <= 1e-6, (b, err)
        fdv = np.array([(obje[2 * k] - obje[2 * k + 1]) / (2 * h) for k in range(4)])
        assert np.abs(fdv - grad[b, :4]).max() <= 1e-6 * max(1.0, np.abs(grad[b, :4]).max()), (b, fdv, grad[b])
        assert np.all(jac[b, :, 4] == 0) and grad[b, 4] == 0      # no disturbance term in this controller
        checked += 1
    assert checked >= 6, f"only {checked} states away from piece boundaries"


# ---------------------------------------------------------------------------------------------------------------------
def test_sensitivity_rejects_bad_arguments_without_a_gpu():
    from carmpc_b200 import _capi
    from carmpc_b200.batch import BatchQP
    from carmpc_b200.condensed import build_parametric_qp
    from conftest import make_controller, make_env
    lib = _capi.load()
    pq = build_parametric_qp(make_controller(make_env("RoadEnv"), 3))
    bq = BatchQP(pq)
    fake = 4096                                          # never dereferenced: every call below fails before device work
    args = lambda rows, x0=fake, st=fake, u=fake, cert=fake, flags=fake: (x0, None, 4, st, u, cert, rows, None, None, flags,
                                                                         None)
    assert lib.carmpc_qp_sensitivity(None, *args(2)) == -1
    assert lib.carmpc_qp_sensitivity(bq._h, *args(0)) == -1
    assert b"rows" in lib.carmpc_last_error()
    assert lib.carmpc_qp_sensitivity(bq._h, *args(bq.n + 1)) == -1
    for missing in ("x0", "st", "u", "cert", "flags"):
        assert lib.carmpc_qp_sensitivity(bq._h, *args(2, **{missing: None})) == -1, missing
    assert lib.carmpc_qp_sensitivity(bq._h, fake, None, -1, fake, fake, fake, 2, None, None, fake, None) == -1
    if not _has_device():                                # a host-only handle: CARMPC_ERR_CUDA, like the solve calls
        assert lib.carmpc_qp_sensitivity(bq._h, *args(2)) == -2
        assert b"without a CUDA device" in lib.carmpc_last_error()
    bq0 = BatchQP(pq, polish=0)
    assert lib.carmpc_qp_sensitivity(bq0._h, *args(2)) == -1
    assert b"polish" in lib.carmpc_last_error()
    # an empty batch is a no-op even on a host-only handle
    assert lib.carmpc_qp_sensitivity(bq._h, None, None, 0, None, None, None, 2, None, None, None, None) == 0


def _has_device():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False
