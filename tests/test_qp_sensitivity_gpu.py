"""Derivatives of batched MPC solutions on the device (``BatchQP.sensitivity``, ``solve_differentiable``), checked against
the numpy restatement on the reference's own matrices (``tests/golden/qp_<env>_N<k>.npz``), against central finite
differences of the solver itself, and through torch autograd."""
import os

import numpy as np
import pytest

from conftest import GOLDEN, make_controller, make_env
from sensitivity_check import DEPENDENT, DERIVATIVE, WEAK, reference_stack, sensitivity_numpy
from test_qp_sensitivity_cpu import hand_built_cases

pytestmark = pytest.mark.gpu

GOAL = {"RoadOneCarEnv": [29.9, 1.5, 0, 0], "RoadMultipleCarsEnv": None, "RoadEnv": None}
ENVS = [("RoadOneCarEnv", 20), ("RoadEnv", 20), ("RoadMultipleCarsEnv", 20), ("RoadOneCarEnv", 10),
        ("RoadOneCarEnv", 40), ("RoadOneCarEnv", 80)]


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "the GPU tests need a CUDA device"
    return torch


def _setup(env_name, N, cls="MPCStateFB", **kw):
    from carmpc_b200.batch import BatchQP
    c = make_controller(make_env(env_name, GOAL[env_name]), N, cls=cls, **kw)
    return c, BatchQP.from_controller(c)


def _grid(torch, goal):
    """The config-3 grid, shifted along x to the environment's goal (it is laid out for the RoadOneCarEnv goal)."""
    from carmpc_b200.grids import config3_axes, materialise_grid
    axes = config3_axes()
    axes = [axes[0] + (goal[0] - 29.9)] + list(axes[1:])
    return torch.stack(materialise_grid(axes, device="cuda")).contiguous(), axes


def _restate(torch, bq, env_name, N, x0, out, idx, c=None, Gc=None, cond=None, term_scale=None):
    from carmpc_b200.certificate import to_one_sided
    d = np.load(os.path.join(GOLDEN, f"qp_{env_name}_N{N}.npz"))
    H, F, G, Gx, lo, hi, lb, ub, Gcr = reference_stack(d, Gc)
    np.testing.assert_array_equal(bq.pq.rows_x, np.vstack((d["At"], d["As"])))
    ii = torch.from_numpy(idx).cuda()
    one = to_one_sided(bq.pq, out["certificate"][ii]).cpu().numpy()
    return sensitivity_numpy(H, F, G, Gx, lo, hi, lb, ub, x0[:, ii].cpu().numpy().T, out["u_full"][ii].cpu().numpy(), one,
                             status=out["status"][ii].cpu().numpy(), Gc=Gcr,
                             c=None if c is None else c[ii].cpu().numpy(), cond=cond, term_scale=term_scale)


def _compare(jk, gk, fk, jr, gr, fr, label, tol=1e-8, cond=None, term_scale=None):
    """Kernel against restatement on the samples with a Jacobian: flags exactly; dV relative to the sample's largest
    gradient entry; J per column relative to the larger of its largest entry and the size of the terms it is computed
    from (``term_scale``: J = Uu - (A_S H^-1)' dlam can cancel to a column that is exactly 0, e.g. inputs pinned by
    rows that do not depend on that coordinate, where both sides return rounding noise of the terms' size).  The J bound
    is 1e-8, or 1e-14 cond(M) where M is so badly conditioned that the two ways of solving (Schur complement and factor
    vs. full KKT by LU) may differ by more: each loses about cond(M) * 2^-53 of that scale."""
    np.testing.assert_array_equal(fk, fr, err_msg=f"{label}: flags")
    has = np.isfinite(jr).all(axis=(1, 2))
    assert np.array_equal(has, np.isfinite(jk).all(axis=(1, 2))), label
    colmax = np.abs(jr[has]).max(axis=1)                                         # (S, 5)
    scale = colmax if term_scale is None else np.maximum(colmax, term_scale[has])
    scale = np.maximum(scale, np.finfo(float).tiny)
    bound = np.full(int(has.sum()), tol) if cond is None else np.maximum(tol, 1e-14 * cond[has])
    abs_err = np.abs(jk[has] - jr[has]).max(axis=1)                              # (S, 5)
    err_s = (abs_err / scale).max(axis=1, initial=0.0)
    cancel = ((colmax < 1e-6 * scale) & (scale > np.finfo(float).tiny)).any(axis=1)
    print(f"{label}: {int(has.sum())} samples, max J error {err_s.max(initial=0.0):.2e} (bound 1e-8 or 1e-14 cond(M); "
          f"max cond(M) {(cond[has].max(initial=1.0) if cond is not None else float('nan')):.2e}), "
          f"{int(cancel.sum())} samples with a column that cancels to ~0 (max absolute error there "
          f"{abs_err[cancel].max(initial=0.0):.2e})")
    gs = np.maximum(np.abs(gr[has]).max(axis=1, keepdims=True), 1.0)
    gerr = (np.abs(gk[has] - gr[has]) / gs).max(initial=0.0)
    print(f"{label}: max dV error {gerr:.2e}")
    bad = np.flatnonzero(err_s > bound)
    assert len(bad) == 0 and gerr <= tol, (label, len(bad), err_s[bad[:5]], colmax[bad[:5]], scale[bad[:5]],
                                           abs_err[bad[:5]], gerr)


@pytest.mark.parametrize("env_name,N", ENVS)
def test_kernel_equals_the_restatement_on_grid_states(torch_cuda, env_name, N):
    """10^4 strided states of the config-3 grid, and every WEAK / DEPENDENT state of the grid up to 2,000 more."""
    torch = torch_cuda
    c, bq = _setup(env_name, N)
    g = np.array(c.goal, dtype=float)
    x0, _ = _grid(torch, g)
    out = bq.solve(x0, want_u_full=True, want_certificate=True)
    s = bq.sensitivity(x0, out)
    st = out["status"].cpu().numpy()
    flags = s["flags"].cpu().numpy()
    counts = {k: int(((flags & v) != 0).sum()) for k, v in (("derivative", DERIVATIVE), ("weak", WEAK),
                                                           ("dependent", DEPENDENT))}
    print(f"{env_name} N={N} grid of {len(st)}: solved {int((st == 0).sum())}, flags {counts}, "
          f"too many rows {int(((flags & 8) != 0).sum())}")
    assert np.all(flags[st != 0] == 0) and np.all(flags[st == 0] != 0) and not (flags & 8).any()
    assert torch.isnan(s["jac"][out["status"] != 0]).all() and torch.isnan(s["grad_objective"][out["status"] != 0]).all()
    B = x0.shape[1]
    idx = np.arange(0, B, B // 10000)[:10000]
    odd = np.flatnonzero((flags & (WEAK | DEPENDENT)) != 0)
    idx = np.union1d(idx, odd[np.linspace(0, len(odd) - 1, min(2000, len(odd))).astype(int)] if len(odd) else odd)
    cond, ts = np.ones(len(idx)), np.zeros((len(idx), 5))
    jr, gr, fr = _restate(torch, bq, env_name, N, x0, out, idx, cond=cond, term_scale=ts)
    ii = torch.from_numpy(idx).cuda()
    _compare(s["jac"][ii].cpu().numpy(), s["grad_objective"][ii].cpu().numpy(), flags[idx], jr, gr, fr,
             f"{env_name} N={N}", cond=cond, term_scale=ts)
    assert (st[idx] == 0).sum() >= 2000


def _finite_differences(torch, bq, x0, out, s, c=None, h=1e-4, want=2000, label=""):
    """Central differences of the solver over x0 +- h e_k (and c +- h) on DERIVATIVE states whose nine (eleven) solves
    share the centre's certificate support."""
    flags = s["flags"].cpu().numpy()
    idx = np.flatnonzero(flags == DERIVATIVE)
    idx = idx[np.linspace(0, len(idx) - 1, min(len(idx), 2 * want)).astype(int)]
    ii = torch.from_numpy(idx).cuda()
    xc = x0[:, ii]
    cc = None if c is None else c[ii]
    K = 5 if c is not None else 4
    xs, cs = [], []
    for k in range(K):
        for sgn in (1.0, -1.0):
            xp = xc.clone()
            cp = None if cc is None else cc.clone()
            if k < 4:
                xp[k] += sgn * h
            else:
                cp += sgn * h
            xs.append(xp)
            cs.append(cp)
    X = torch.cat(xs, dim=1).contiguous()
    C = None if c is None else torch.cat(cs).contiguous()
    o = bq.solve(X, c=C, want_u_full=True, want_certificate=True)
    nb = len(idx)
    sup0 = out["certificate"][ii] != 0
    same = (out["status"][ii] == 0).clone()
    for r in range(2 * K):
        sl = slice(r * nb, (r + 1) * nb)
        same &= (o["status"][sl] == 0) & (o["certificate"][sl] != 0).eq(sup0).all(dim=1)
    keep = same.cpu().numpy()
    assert keep.sum() >= want, f"{label}: only {int(keep.sum())} states away from piece boundaries"
    u = o["u_full"].cpu().numpy().reshape(2 * K, nb, -1)
    v = o["objective"].cpu().numpy().reshape(2 * K, nb)
    jac = s["jac"][ii].cpu().numpy()
    grad = s["grad_objective"][ii].cpu().numpy()
    # per column relative to its largest entry, floored by the unconstrained gain Uu = -H^-1 F (its largest entry; the
    # largest of all four for the disturbance column): a column that cancels to ~0 is compared at the size of its terms
    uu = np.abs(np.linalg.solve(bq.pq.H, -bq.pq.F)).max(axis=0)
    floor = np.append(uu, uu.max())
    worst_j = worst_v = 0.0
    for k in range(K):
        fd = (u[2 * k] - u[2 * k + 1]) / (2 * h)
        fv = (v[2 * k] - v[2 * k + 1]) / (2 * h)
        scale = np.maximum(np.abs(jac[:, :, k]).max(axis=1), floor[k])
        worst_j = max(worst_j, (np.abs(fd - jac[:, :, k]).max(axis=1) / scale)[keep].max())
        worst_v = max(worst_v, (np.abs(fv - grad[:, k]) / np.maximum(np.abs(grad).max(axis=1), 1.0))[keep].max())
    print(f"{label}: {int(keep.sum())} of {nb} states, max relative FD error J {worst_j:.2e}, dV {worst_v:.2e}")
    # the solver's u is accurate to ~1e-11 on a fixed active set: over h = 1e-4 that is ~1e-7 of an O(1) entry
    assert worst_j <= 1e-5 and worst_v <= 1e-5, (label, worst_j, worst_v)


@pytest.mark.parametrize("env_name,N", ENVS)
def test_kernel_equals_central_differences_of_the_solver(torch_cuda, env_name, N):
    torch = torch_cuda
    c, bq = _setup(env_name, N)
    x0, _ = _grid(torch, np.array(c.goal, dtype=float))
    out = bq.solve(x0, want_u_full=True, want_certificate=True)
    s = bq.sensitivity(x0, out)
    _finite_differences(torch, bq, x0, out, s, label=f"{env_name} N={N}")


def test_disturbance_handle_kernel_equals_restatement_and_central_differences(torch_cuda):
    torch = torch_cuda
    d = np.load(os.path.join(GOLDEN, "disturbance.npz"))
    c, bq = _setup("RoadEnv", 20, cls="MPCOutputFBWithDisturbance", init_state=[20, 0.5, 0, 2])
    x_ref = np.array(c.goal, dtype=float)
    rng = np.random.default_rng(5)
    B = 100000
    x0 = torch.from_numpy(np.ascontiguousarray((x_ref + rng.uniform(-1, 1, size=(B, 4)) * [14.0, 1.6, 0.3, 3.0]).T)).cuda()
    dist = torch.from_numpy(rng.uniform(-0.05, 0.05, size=B)).cuda()
    out = bq.solve(x0, c=dist, want_u_full=True, want_certificate=True)
    s = bq.sensitivity(x0, out, c=dist)
    assert (s["jac"][:, :, 4][out["status"] == 0] != 0).any(), "the disturbance column is zero everywhere"
    idx = np.arange(0, B, 10)
    cond, ts = np.ones(len(idx)), np.zeros((len(idx), 5))
    jr, gr, fr = _restate(torch, bq, "RoadEnv", 20, x0, out, idx, c=dist, Gc=d["ABd_N20"], cond=cond, term_scale=ts)
    ii = torch.from_numpy(idx).cuda()
    _compare(s["jac"][ii].cpu().numpy(), s["grad_objective"][ii].cpu().numpy(), s["flags"][ii].cpu().numpy(), jr, gr,
             fr, "RoadEnv N=20 disturbance", cond=cond, term_scale=ts)
    _finite_differences(torch, bq, x0, out, s, c=dist, label="RoadEnv N=20 disturbance")


def test_kernel_sets_the_restatement_flags_on_hand_built_qps(torch_cuda):
    torch = torch_cuda
    from carmpc_b200.batch import BatchQP
    from carmpc_b200.condensed import ParametricQP
    for name, (p, x0, u, y, want) in hand_built_cases().items():
        R, n = len(p["hi"]), len(u)
        pre = ~np.any(p["G"] != 0, axis=1)
        z = np.zeros(0)
        pq = ParametricQP(N=1, H=p["H"], F=p["F"], G=p["G"][~pre], Gx=p["Gx"][~pre], lo=p["lo"][~pre], hi=p["hi"][~pre],
                          lb=p["lb"], ub=p["ub"], Gc=p["Gc"][~pre], Px=p["Gx"][pre], Pc=p["Gc"][pre], pre_lo=p["lo"][pre],
                          pre_hi=p["hi"][pre], goal=np.zeros(4), T=z, S=z, rows_x=z, rows_b=z, src_hi=z, src_lo=z)
        bq = BatchQP(pq)
        cert = np.concatenate((y[:R][~pre], y[R:], y[:R][pre]))
        X = torch.from_numpy(np.ascontiguousarray(x0[:, None])).cuda()
        out = {"status": torch.zeros(1, dtype=torch.int32, device="cuda"),
               "u_full": torch.from_numpy(u[None].copy()).cuda(), "certificate": torch.from_numpy(cert[None]).cuda()}
        s = bq.sensitivity(X, out)
        ts = np.zeros((1, 5))
        jr, gr, fr = sensitivity_numpy(p["H"], p["F"], p["G"], p["Gx"], p["lo"], p["hi"], p["lb"], p["ub"], x0[None],
                                       u[None], y[None], Gc=p["Gc"], term_scale=ts)
        assert int(s["flags"][0]) == fr[0] == want, (name, int(s["flags"][0]), fr[0])
        _compare(s["jac"].cpu().numpy(), s["grad_objective"].cpu().numpy(), s["flags"].cpu().numpy(), jr, gr, fr, name,
                 tol=1e-10, term_scale=ts)


def test_seeded_and_cold_solves_give_the_same_jacobian(torch_cuda):
    torch = torch_cuda
    from carmpc_b200.grids import lattice_seeds
    c, bq = _setup("RoadOneCarEnv", 20)
    x0, axes = _grid(torch, np.array(c.goal, dtype=float))
    seed = torch.from_numpy(lattice_seeds([len(a) for a in axes], block=(3, 8, 1, 1))).cuda()
    cold = bq.solve(x0, want_u_full=True, want_certificate=True)
    seeded = bq.solve(x0, want_u_full=True, want_certificate=True, seed=seed)
    sc, ss = bq.sensitivity(x0, cold), bq.sensitivity(x0, seeded)
    both = (sc["flags"] == DERIVATIVE) & (ss["flags"] == DERIVATIVE)
    assert int(both.sum()) > 10 ** 5
    jc, js = sc["jac"][both], ss["jac"][both]
    # per column relative to its largest entry, or to the unconstrained gain Uu = -H^-1 F where it cancels to ~0
    uu = np.abs(np.linalg.solve(bq.pq.H, -bq.pq.F)).max(axis=0)
    floor = torch.from_numpy(np.append(uu, 1.0)).cuda()
    scale = torch.maximum(jc.abs().amax(dim=1, keepdim=True), floor)
    err = ((jc - js).abs() / scale).max().item()
    gerr = ((sc["grad_objective"][both] - ss["grad_objective"][both]).abs()
            / sc["grad_objective"][both].abs().amax(dim=1, keepdim=True).clamp(min=1.0)).max().item()
    print(f"seeded vs cold: {int(both.sum())} states, max J difference {err:.2e}, dV {gerr:.2e}")
    assert err <= 1e-8 and gerr <= 1e-8


def test_leading_rows_equal_the_full_jacobian(torch_cuda):
    torch = torch_cuda
    c, bq = _setup("RoadOneCarEnv", 40)
    x0, _ = _grid(torch, np.array(c.goal, dtype=float))
    x0 = x0[:, ::7].contiguous()
    out = bq.solve(x0, want_u_full=True, want_certificate=True)
    full, two = bq.sensitivity(x0, out), bq.sensitivity(x0, out, rows=2)
    assert two["jac"].shape == (x0.shape[1], 2, 5)
    ok = out["status"] == 0
    assert torch.equal(full["jac"][ok, :2], two["jac"][ok])
    assert torch.equal(full["flags"], two["flags"]) and torch.equal(full["grad_objective"][ok], two["grad_objective"][ok])


def test_autograd_layer(torch_cuda):
    torch = torch_cuda
    from carmpc_b200.sensitivity import solve_differentiable
    c, bq = _setup("RoadEnv", 20, cls="MPCOutputFBWithDisturbance", init_state=[20, 0.5, 0, 2])
    g0 = np.array(c.goal, dtype=float)
    rng = np.random.default_rng(9)
    B = 4000
    x0 = torch.from_numpy(np.ascontiguousarray((g0 + rng.uniform(-1, 1, size=(B, 4)) * [14.0, 1.6, 0.3, 3.0]).T)).cuda()
    dist = torch.from_numpy(rng.uniform(-0.05, 0.05, size=B)).cuda()
    out = bq.solve(x0, c=dist, want_u_full=True, want_certificate=True)
    s = bq.sensitivity(x0, out, c=dist)
    st = out["status"]
    ok = st == 0
    assert int(ok.sum()) > 500 and int((~ok).sum()) > 100
    # backward = J' g_u + g_v dV on solved samples (masked loss: infeasible samples get exactly zero)
    xg, cg = x0.clone().requires_grad_(True), dist.clone().requires_grad_(True)
    u, v = solve_differentiable(bq, xg, cg)
    gu = torch.randn_like(u).masked_fill(~ok[:, None], 0.0)
    gv = torch.randn_like(v).masked_fill(~ok, 0.0)
    (torch.where(ok[:, None], u, 0.0) * gu).sum().backward(inputs=[xg, cg], retain_graph=True)
    want = torch.einsum("bn,bnk->bk", gu[ok], s["jac"][ok])
    assert torch.allclose(xg.grad.t()[ok], want[:, :4], rtol=1e-12, atol=1e-12)
    assert torch.allclose(cg.grad[ok], want[:, 4], rtol=1e-12, atol=1e-12)
    assert torch.all(xg.grad[:, ~ok] == 0) and torch.all(cg.grad[~ok] == 0)
    xg.grad, cg.grad = None, None
    (torch.where(ok, v, 0.0) * gv).sum().backward(inputs=[xg, cg], retain_graph=True)
    want = gv[ok, None] * s["grad_objective"][ok]
    assert torch.allclose(xg.grad.t()[ok], want[:, :4], rtol=1e-12, atol=1e-12)
    assert torch.all(xg.grad[:, ~ok] == 0)
    # unmasked: samples without a derivative are NaN, the others stay exact
    xg.grad, cg.grad = None, None
    u.sum().backward(inputs=[xg])
    assert torch.isnan(xg.grad[:, ~ok]).all() and torch.isfinite(xg.grad[:, ok]).all()
    # gradcheck on 8 nondegenerate states, x0 and c in float64
    idx = torch.nonzero(s["flags"] == DERIVATIVE).flatten()[:8 * 50:50]
    assert len(idx) == 8
    xs, cs = x0[:, idx].contiguous().requires_grad_(True), dist[idx].contiguous().requires_grad_(True)
    assert torch.autograd.gradcheck(lambda a, b: solve_differentiable(bq, a, b), (xs, cs), eps=1e-6, atol=1e-6,
                                    rtol=1e-5, nondet_tol=1e-12)
    # no input requires grad: the forward pass computes no Jacobian and returns plain tensors
    u2, v2 = solve_differentiable(bq, x0, dist)
    assert not u2.requires_grad and torch.equal(u2[ok], out["u_full"][ok])
