"""Certificates of batched QP solves without a GPU: the numpy restatement of the checker kernel on hand-built KKT points and
Farkas rays (and their corruptions), the mapping of handle-space certificates onto the reference's one-sided stacks, and
the argument errors of the new entry points."""
import ctypes
import os

import numpy as np
import pytest

from cert_check import check_numpy
from conftest import golden, make_env, make_controller


def _passes(status, resid):
    from carmpc_b200.certificate import passes
    return passes(np.asarray(status), resid)


def _kkt_case(seed=0):
    """A strictly convex QP built around a known KKT point: two rows active at their upper bound, one at its lower bound,
    one box entry at its upper bound, the rest inactive; some rows one-sided."""
    rng = np.random.default_rng(seed)
    n, R = 5, 7
    M = rng.normal(size=(n, n))
    H = M @ M.T + n * np.eye(n)
    G, Gx = rng.normal(size=(R, n)), rng.normal(size=(R, 4))
    x0, xref = rng.normal(size=4), rng.normal(size=4)
    u = rng.normal(size=n)
    s = Gx @ x0
    gu = G @ u
    hi, lo = gu + s + 1.0, gu + s - 1.0
    lo[[1, 4]] = -np.inf                             # one-sided rows
    hi[0], hi[1], lo[2] = gu[0] + s[0], gu[1] + s[1], gu[2] + s[2]
    lam = np.zeros(R)
    lam[0], lam[1], lam[2] = 0.7, 1.3, -0.4
    lb, ub = u - 1.0, u + 1.0
    ub[3] = u[3]
    lam_b = np.zeros(n)
    lam_b[3] = 0.25
    q = -(H @ u + G.T @ lam + lam_b)
    dx = x0 - xref
    F = np.outer(q, dx) / (dx @ dx)
    prob = dict(H=H, F=F, G=G, Gx=Gx, lo=lo, hi=hi, lb=lb, ub=ub)
    return prob, x0, xref, u, np.concatenate((lam, lam_b))


def _farkas_case():
    """Infeasible: row 0 is G_0 u <= 1 and row 1 the opposite -G_0 u <= -2; row 2 asks more of G_2 u than the box allows."""
    n = 3
    H, F = np.eye(n), np.zeros((n, 4))
    G = np.array([[1.0, 2.0, -1.0], [-1.0, -2.0, 1.0], [1.0, -1.0, 0.5]])
    Gx = np.zeros((3, 4))
    Gx[0, 0] = 0.5
    Gx[1, 0] = -0.5                                  # the shift cancels in y = (1, 1, 0)
    lo = np.full(3, -np.inf)
    hi = np.array([1.0, -2.0, -10.0])
    lb, ub = -np.ones(n), np.ones(n)
    prob = dict(H=H, F=F, G=G, Gx=Gx, lo=lo, hi=hi, lb=lb, ub=ub)
    ray_a = np.array([1.0, 1.0, 0.0, 0.0, 0.0, 0.0])       # G'y_g = 0: support 1 - 2 = -1
    ray_b = np.concatenate(([0.0, 0.0, 1.0], -G[2]))       # support -10 - min_box G_2 u = -10 + 2.5
    return prob, ray_a, ray_b


def _run(prob, x0, xref, status, u, cert):
    return check_numpy(prob["H"], prob["F"], prob["G"], prob["Gx"], prob["lo"], prob["hi"], prob["lb"], prob["ub"],
                       np.atleast_2d(x0), xref, np.atleast_1d(status), np.atleast_2d(u), np.atleast_2d(cert))


def test_numpy_checker_accepts_a_kkt_point_and_rejects_each_corruption():
    prob, x0, xref, u, cert = _kkt_case()
    r = _run(prob, x0, xref, 0, u, cert)
    assert _passes([0], r)[0], r
    assert r[0, 0] <= 1e-14 and r[0, 1] <= 1e-13 and r[0, 2] == 0 and r[0, 3] <= 1e-14
    corrupt = {}
    c = cert.copy(); c[1] = -c[1]; corrupt["flipped sign, one-sided row"] = c
    c = cert.copy(); c[0] = -c[0]; corrupt["flipped sign, two-sided row"] = c
    c = cert.copy(); c[5] = 0.3; corrupt["multiplier on an inactive row"] = c
    c = cert.copy(); c[1] = 0.0; corrupt["missing active-row multiplier"] = c
    c = cert.copy(); c[7 + 3] = 0.0; corrupt["missing active box multiplier"] = c
    for name, c in corrupt.items():
        r = _run(prob, x0, xref, 0, u, c)
        assert not _passes([0], r)[0], (name, r)
    # a point that is not optimal for the given multipliers
    r = _run(prob, x0, xref, 0, u + 1e-3, cert)
    assert not _passes([0], r)[0]


def test_numpy_checker_accepts_farkas_rays_and_rejects_each_corruption():
    prob, ray_a, ray_b = _farkas_case()
    x0, xref, u = np.array([0.3, 0.0, 0.0, 0.0]), np.zeros(4), np.full(3, np.nan)
    for ray, want in ((ray_a, -1.0), (ray_b, -7.5)):
        r = _run(prob, x0, xref, 1, u, ray)
        assert _passes([1], r)[0], r
        assert abs(r[0, 0] - want) <= 1e-12 and r[0, 2] == 0 and r[0, 3] == 0
    c = ray_b.copy(); c[3] += 1e-3
    assert not _passes([1], _run(prob, x0, xref, 1, u, c))[0], "perturbed box part"
    c = ray_a.copy(); c[1] = 0.0                               # box completion makes it a ray of row 0 alone: support > 0
    r = _run(prob, x0, xref, 1, u, np.concatenate((c[:3], -prob["G"].T @ c[:3])))
    assert r[0, 0] > 0 and not _passes([1], r)[0], "positive support"
    c = ray_a.copy(); c[0] = -1.0                              # against the infinite lower bound of a one-sided row
    r = _run(prob, x0, xref, 1, u, c)
    assert r[0, 3] > 0 and not _passes([1], r)[0]
    # status 2 is NaN and never passes
    r = _run(prob, x0, xref, 2, u, ray_a)
    assert np.isnan(r).all() and not _passes([2], r)[0]


def _parametric(tag, env, goal, N):
    from carmpc_b200.condensed import build_parametric_qp
    return build_parametric_qp(make_controller(make_env(env, goal), N))


@pytest.mark.parametrize("tag,env,goal", [("RoadEnv", "RoadEnv", None), ("RoadOneCarEnv", "RoadOneCarEnv", [29.9, 1.5, 0, 0]),
                                          ("RoadOneCarEnvDefault", "RoadOneCarEnv", None),
                                          ("RoadMultipleCarsEnv", "RoadMultipleCarsEnv", None)])
@pytest.mark.parametrize("N", [1, 3, 20])
def test_to_one_sided_round_trips_on_the_golden_stacks(tag, env, goal, N):
    """A handle-space certificate and its one-sided image act the same on u and on x0 (G'y and Gx'y agree), rows of the
    one-sided stack only receive entries >= 0 from multipliers on the right side, and the u-independent rows point at
    rows of the stack whose S part is exactly zero."""
    import torch
    from carmpc_b200.certificate import to_one_sided
    g = golden(f"constraints_{tag}_N{N}.npz")
    pq = _parametric(tag, env, goal, N)
    np.testing.assert_array_equal(pq.rows_x, np.vstack((g["At"], g["As"])))
    np.testing.assert_array_equal(pq.rows_b, np.hstack((g["bt"], g["bs"])))
    m, n, k = pq.m, pq.n, len(pq.pre_hi)
    assert len(pq.pre_src_hi) == k and len(pq.pre_src_lo) == k
    G1, Gx1 = pq.rows_x @ pq.S, pq.rows_x @ pq.T
    for src in (pq.pre_src_hi, pq.pre_src_lo[pq.pre_src_lo >= 0]):
        assert np.all(G1[src] == 0.0)
    rng = np.random.default_rng(N)
    cert = rng.normal(size=(6, m + n + k))
    cert[0] = np.abs(cert[0]) * (rng.random(m + n + k) < 0.2)        # a sparse "upper side only" row
    one = to_one_sided(pq, torch.from_numpy(cert)).numpy()
    R = len(pq.rows_b)
    assert one.shape == (6, R + n)
    Ghandle = np.vstack((pq.G, np.eye(n), np.zeros((k, n))))
    Gxhandle = np.vstack((pq.Gx, np.zeros((n, 4)), pq.Px))
    np.testing.assert_allclose(one[:, :R] @ G1 + one[:, R:], cert @ Ghandle, rtol=0, atol=1e-9 * max(1.0, np.abs(G1).max()))
    np.testing.assert_allclose(one[:, :R] @ Gx1, cert @ Gxhandle, rtol=0, atol=1e-9 * max(1.0, np.abs(Gx1).max()))
    assert np.all(one[0] >= 0.0)
    # a row dropped for a tighter duplicate receives nothing
    used = set(pq.src_hi) | set(pq.src_lo[pq.src_lo >= 0]) | set(pq.pre_src_hi) | set(pq.pre_src_lo[pq.pre_src_lo >= 0])
    dropped = np.array(sorted(set(range(R)) - used), dtype=int)
    assert np.all(one[:, dropped] == 0.0)


def test_to_one_sided_rejects_a_wrong_width():
    import torch
    from carmpc_b200.certificate import to_one_sided
    pq = _parametric("RoadEnv", "RoadEnv", None, 3)
    with pytest.raises(ValueError):
        to_one_sided(pq, torch.zeros((2, pq.m + pq.n)))


def test_checker_and_solve_reject_bad_arguments_without_a_gpu():
    from carmpc_b200 import _capi
    from carmpc_b200.certificate import QPChecker
    lib = _capi.load()
    h = ctypes.c_void_p()
    I2, F2, z = np.eye(2), np.zeros((2, 4)), np.zeros(2)
    p = _capi.ptr
    assert lib.carmpc_qp_checker_create(0, 0, p(I2), p(F2), None, None, None, None, None, p(z), p(z), ctypes.byref(h)) == -1
    assert lib.carmpc_qp_checker_create(2, 0, None, p(F2), None, None, None, None, None, p(z), p(z), ctypes.byref(h)) == -1
    assert b"null" in lib.carmpc_last_error()
    assert lib.carmpc_qp_checker_create(2, 1, p(I2), p(F2), None, None, None, None, None, p(z), p(z), ctypes.byref(h)) == -1
    assert lib.carmpc_qp_checker_create(2, 20000, p(I2), p(F2), None, None, None, None, None, p(z), p(z), ctypes.byref(h)) == -1
    bad = np.array([[1.0, np.nan], [0.0, 1.0]])
    assert lib.carmpc_qp_checker_create(2, 0, p(bad), p(F2), None, None, None, None, None, p(z), p(z), ctypes.byref(h)) == -1
    xref = np.zeros(4)
    assert lib.carmpc_qp_check(None, None, p(xref), None, 1, None, None, None, None, None) == -1
    fake = ctypes.c_void_p(64)            # never dereferenced: every call below is refused before any device work

    def solve(qp, seed=None, warm=None, cert=None, batch=1):
        return lib.carmpc_qp_solve(qp, None, p(xref), None, seed, batch, None, None, None, None, None, warm, 0, 0, cert, None,
                                   None)

    assert solve(None, cert=fake) == -1
    # a well-formed checker can be created without a device (its check calls then fail)
    chk = QPChecker(I2, F2, np.ones((1, 2)), np.zeros((1, 4)), [-np.inf], [1.0], -np.ones(2), np.ones(2))
    assert chk.R == 1 and chk._h
    # the polish is what produces certificates and reuses seeds: a handle without it is refused
    from carmpc_b200.batch import BatchQP
    pq = _parametric("RoadEnv", "RoadEnv", None, 3)
    bq = BatchQP(pq, polish=0)
    for kw in (dict(cert=fake), dict(seed=fake), dict(cert=fake, batch=0), dict(seed=fake, batch=0)):
        assert solve(bq._h, **kw) == -1, kw
        assert b"polish" in lib.carmpc_last_error()
    # a warm state is a starting point of its own: not with seeds or certificates, on any handle
    for handle in (bq, BatchQP(pq)):
        for kw in (dict(seed=fake), dict(cert=fake), dict(seed=fake, cert=fake)):
            for batch in (1, 0):
                assert solve(handle._h, warm=fake, batch=batch, **kw) == -1, (kw, batch)
                assert b"d_warm" in lib.carmpc_last_error()
