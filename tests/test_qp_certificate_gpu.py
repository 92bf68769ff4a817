"""Certificates of batched QP solves on the device, checked against the reference's own QP.

The solver exports, per sample, the multipliers of its float64 KKT certificate or the Farkas ray of its infeasibility
proof (``BatchQP.solve(want_certificate=True)``).  Here they are mapped onto the reference's one-sided stack and checked
by the independent checker kernel (``QPChecker``) on matrices read only from ``tests/golden/qp_<env>_N<k>.npz`` (the
reference controller's H, h, T, S and constraint stacks): every decided state of every grid, not a sample of it.
"""
import os

import numpy as np
import pytest

from conftest import GOLDEN, make_env, make_controller

pytestmark = pytest.mark.gpu

GOAL = {"RoadOneCarEnv": [29.9, 1.5, 0, 0], "RoadMultipleCarsEnv": None, "RoadEnv": None}


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "the GPU tests need a CUDA device"
    return torch


class Reference:
    """The reference's QP from its golden matrices: one-sided rows [At; As] (T x0 + S u) <= [bt; bs], box from Ai / bi."""

    def __init__(self, env_name, N, Gc=None):
        d = np.load(os.path.join(GOLDEN, f"qp_{env_name}_N{N}.npz"))
        n = d["S"].shape[1]
        A = np.vstack((d["At"], d["As"]))
        self.H, self.F, self.goal = d["H"], d["h"], d["goal"]
        self.G, self.Gx, self.hi = A @ d["S"], A @ d["T"], np.hstack((d["bt"], d["bs"]))
        self.lo = np.full(len(self.hi), -np.inf)
        Ai, bi = d["Ai"], d["bi"]
        np.testing.assert_array_equal(Ai, np.vstack((np.eye(n), -np.eye(n))))
        self.ub, self.lb = bi[:n], -bi[n:]
        self.rows = A
        self.Gc = None if Gc is None else A @ Gc

    def checker(self):
        from carmpc_b200.certificate import QPChecker
        return QPChecker(self.H, self.F, self.G, self.Gx, self.lo, self.hi, self.lb, self.ub, Gc=self.Gc)

    def numpy(self, x0, xref, status, u, cert, c=None):
        from cert_check import check_numpy
        return check_numpy(self.H, self.F, self.G, self.Gx, self.lo, self.hi, self.lb, self.ub, x0, xref, status, u,
                           cert, Gc=self.Gc, c=c)


def _setup(env_name, N, cls="MPCStateFB", **kw):
    from carmpc_b200.batch import BatchQP
    c = make_controller(make_env(env_name, GOAL[env_name]), N, cls=cls, **kw)
    return c, BatchQP.from_controller(c)


def _bits(t):
    import torch
    return t.contiguous().view(torch.int64) if t.dtype == torch.float64 else t


def _assert_bit_identical(a, b):
    import torch
    for k in ("u0", "objective", "status", "iters", "u_full"):
        if k in a:
            assert torch.equal(_bits(a[k]), _bits(b[k])), f"{k} differs with certificates on"


def _grid(torch, goal, shift=True):
    from carmpc_b200.grids import config3_axes, materialise_grid
    axes = config3_axes()
    if shift:
        axes = [axes[0] + (goal[0] - 29.9)] + list(axes[1:])      # the grid is laid out for the RoadOneCarEnv goal
    return torch.stack(materialise_grid(axes, device="cuda")).contiguous(), axes


def _check_all(torch, ref, bq, x0, out, xref, c=None, label=""):
    """Every status-0 state passes the KKT test and every status-1 state the Farkas test, in the reference's row space."""
    from carmpc_b200.certificate import passes, to_one_sided
    one = to_one_sided(bq.pq, out["certificate"])
    chk = ref.checker()
    resid = chk.check(x0, xref, out["status"], out["u_full"], one, c=c)
    st = out["status"]
    ok = passes(st, resid)
    decided = st != 2
    bad = torch.nonzero(decided & ~ok).flatten()
    n2 = int((st == 2).sum())
    r = resid.cpu().numpy()
    s = st.cpu().numpy()
    kkt = r[s == 0]
    far = r[s == 1]
    info = {"states": int(st.numel()), "solved": int((s == 0).sum()), "infeasible": int((s == 1).sum()), "undecided": n2,
            "primal": float(kkt[:, 0].max(initial=0)), "stationarity": float(kkt[:, 1].max(initial=0)),
            "wrong_side": float(kkt[:, 2].max(initial=0)), "complementarity": float(kkt[:, 3].max(initial=0)),
            "worst_support_over_scale": float((far[:, 0] / far[:, 1]).max(initial=-np.inf)),
            "box_residual": float(far[:, 2].max(initial=0))}
    print(f"{label}: {info}")
    if len(bad):
        i = bad[:5].cpu().numpy()
        raise AssertionError(f"{label}: {len(bad)} decided states fail their certificate check, e.g. {i}: status "
                             f"{s[i]}, residuals {r[i]}")
    return one, resid, info


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("env_name,N", [("RoadOneCarEnv", 20), ("RoadEnv", 20), ("RoadMultipleCarsEnv", 20),
                                        ("RoadOneCarEnv", 10), ("RoadOneCarEnv", 40), ("RoadOneCarEnv", 80)])
def test_certified_solve_is_bit_identical_to_the_plain_solve(torch_cuda, env_name, N):
    torch = torch_cuda
    from carmpc_b200.grids import lattice_seeds
    c, bq = _setup(env_name, N)
    g = np.array(c.goal, dtype=float)
    axes = [np.linspace(g[0] - 22.0, g[0] + 0.5, 30), np.linspace(-3.0, 3.0, 41), np.linspace(-0.3, 0.3, 5),
            np.linspace(-1.0, 4.0, 5)]
    from carmpc_b200.grids import materialise_grid
    x0 = torch.stack(materialise_grid(axes, device="cuda")).contiguous()
    B = x0.shape[1]
    plain = bq.solve(x0, want_u_full=True)
    cert = bq.solve(x0, want_u_full=True, want_certificate=True)
    _assert_bit_identical(plain, cert)
    assert cert["certificate"].shape == (B, bq.m + bq.n + len(bq.pq.pre_hi))
    st = plain["status"].cpu().numpy()
    assert (st == 0).sum() > B // 10 and (st == 1).sum() > B // 50
    seed = torch.from_numpy(lattice_seeds([len(a) for a in axes], block=(3, 8, 1, 1))).cuda()
    plain_s = bq.solve(x0, want_u_full=True, seed=seed)
    cert_s = bq.solve(x0, want_u_full=True, seed=seed, want_certificate=True)
    _assert_bit_identical(plain_s, cert_s)
    assert plain_s["seeded"] == cert_s["seeded"]
    ref = Reference(env_name, N)
    np.testing.assert_array_equal(bq.pq.rows_x, ref.rows)
    for out, label in ((cert, "cold"), (cert_s, "seeded")):
        _check_all(torch, ref, bq, x0, out, g, label=f"{env_name} N={N} {label}")


def test_checker_kernel_equals_the_numpy_checker_and_flags_every_corruption(torch_cuda):
    torch = torch_cuda
    from carmpc_b200.certificate import passes, to_one_sided
    c, bq = _setup("RoadOneCarEnv", 20)
    g = np.array(c.goal, dtype=float)
    ref = Reference("RoadOneCarEnv", 20)
    rng = np.random.default_rng(4)
    x0 = torch.from_numpy(np.ascontiguousarray((g + rng.uniform(-1, 1, size=(8000, 4)) * [14.0, 1.6, 0.3, 3.0]).T)).cuda()
    out = bq.solve(x0, want_u_full=True, want_certificate=True)
    one = to_one_sided(bq.pq, out["certificate"])
    st = out["status"].clone()
    u = out["u_full"].clone()
    R = ref.G.shape[0]
    s = st.cpu().numpy()
    sol, inf = np.flatnonzero(s == 0), np.flatnonzero(s == 1)
    assert len(sol) > 500 and len(inf) > 500
    # corrupted copies, appended to the batch: each must fail the check
    cor_rows, cor_idx, kinds = [], [], []
    on = one.cpu().numpy()
    for i in sol[:400]:
        lam = on[i, :R]
        if not (lam > 0).any():
            continue
        a = int(np.argmax(lam))
        r = on[i].copy(); r[a] = -r[a]; cor_rows.append(r); cor_idx.append(i); kinds.append("flipped sign")
        r = on[i].copy(); r[a] = 0.0; cor_rows.append(r); cor_idx.append(i); kinds.append("missing active multiplier")
        inactive = np.flatnonzero(lam == 0)
        r = on[i].copy(); r[inactive[len(inactive) // 2]] = max(1.0, lam[a]); cor_rows.append(r); cor_idx.append(i)
        kinds.append("multiplier on an inactive row")
    for i in inf[:400]:
        y = on[i]
        r = y.copy(); r[R:] += 1e-3 * max(1.0, np.abs(y[R:]).max()); cor_rows.append(r); cor_idx.append(i)
        kinds.append("perturbed box part")
        r = -y; cor_rows.append(r); cor_idx.append(i); kinds.append("reversed ray")
    cor_idx = np.array(cor_idx)
    ci = torch.from_numpy(cor_idx).cuda()
    x_all = torch.cat((x0, x0[:, ci]), dim=1).contiguous()
    st_all = torch.cat((st, st[ci])).contiguous()
    u_all = torch.cat((u, u[ci])).contiguous()
    cert_all = torch.cat((one, torch.from_numpy(np.array(cor_rows)).cuda())).contiguous()
    resid = ref.checker().check(x_all, g, st_all, u_all, cert_all).cpu().numpy()
    want = ref.numpy(x_all.cpu().numpy().T, g, st_all.cpu().numpy(), u_all.cpu().numpy(), cert_all.cpu().numpy())
    sa = st_all.cpu().numpy()
    dec = sa != 2
    np.testing.assert_array_equal(np.isnan(resid), np.isnan(want))
    for col in range(4):
        a, b = resid[dec, col], want[dec, col]
        scale = np.where(sa[dec] == 1, np.maximum(np.abs(want[dec, 1]), 1e-300), 1.0) if col in (0,) else 1.0
        err = np.abs(a - b) / np.maximum(np.abs(b), 1.0)
        if col == 0:
            err = np.where(sa[dec] == 1, np.abs(a - b) / scale, err)
        assert err.max() <= 1e-9, f"column {col}: kernel and numpy differ by {err.max():.3e}"
    pk, pn = passes(sa, resid), passes(sa, want)
    np.testing.assert_array_equal(pk, pn)
    B = x0.shape[1]
    assert pk[:B][s != 2].all()
    flagged = ~pk[B:]
    for kind in sorted(set(kinds)):
        sel = np.array([k == kind for k in kinds])
        assert flagged[sel].all(), f"{kind}: {int((~flagged[sel]).sum())} of {int(sel.sum())} corrupted certificates pass"
    print({k: int(sum(1 for x in kinds if x == k)) for k in set(kinds)})


@pytest.mark.parametrize("N", [20, 10, 40, 80])
def test_every_config_grid_state_has_a_valid_certificate(torch_cuda, N):
    """Config 3 (N = 20) and config 5 (N = 10 / 40 / 80): all 10^6 states of the RoadOneCarEnv grid, cold; at N = 20 also
    the seeded lattice map.  The NNLS check of kkt_check.py and the phase-1 LP agree on subsets."""
    torch = torch_cuda
    from carmpc_b200.grids import lattice_seeds
    c, bq = _setup("RoadOneCarEnv", N)
    g = np.array(c.goal, dtype=float)
    ref = Reference("RoadOneCarEnv", N)
    x0, axes = _grid(torch, g, shift=False)
    assert x0.shape[1] == 10 ** 6
    out = bq.solve(x0, want_u_full=True, want_certificate=True)
    one, resid, info = _check_all(torch, ref, bq, x0, out, g, label=f"config grid N={N} cold")
    assert info["undecided"] <= (0 if N == 20 else 2)
    if N == 20:
        seed = torch.from_numpy(lattice_seeds([len(a) for a in axes], block=(3, 8, 1, 1))).cuda()
        outs = bq.solve(x0, want_u_full=True, want_certificate=True, seed=seed)
        _check_all(torch, ref, bq, x0, outs, g, label=f"config grid N={N} seeded")
        assert int((outs["status"] == 2).sum()) == 0
        # followers proven by their anchor's record carry exactly the anchor's exported ray
        st = outs["status"].cpu().numpy()
        sd = seed.cpu().numpy().astype(np.int64)
        fol = np.flatnonzero((sd != np.arange(len(sd))) & (st == 1) & (st[sd] == 1))
        cert = outs["certificate"]
        fi = torch.from_numpy(fol).cuda()
        same = (cert[fi] == cert[torch.from_numpy(sd[fol]).cuda()]).all(dim=1).cpu().numpy()
        print(f"infeasible followers of infeasible anchors: {len(fol)}, carrying the anchor's ray: {int(same.sum())}, "
              f"polish stats: {bq.polish_stats()['infeasible_by_anchor_certificate']}")
        assert same.sum() > 0
    # the evidence of kkt_check.py on a strided subset, and the phase-1 LP on infeasible states
    from kkt_check import ReferenceQP
    kref = ReferenceQP("RoadOneCarEnv", N)
    st = out["status"].cpu().numpy()
    n_sub = 2000 if N <= 40 else 500
    idx = np.arange(0, 10 ** 6, 10 ** 6 // n_sub)[:n_sub]
    sol = idx[st[idx] == 0]
    xs = x0.cpu().numpy().T
    u = out["u_full"].cpu().numpy()
    primal, stat, _ = kref.kkt(u[sol], xs[sol])
    assert primal.max() <= 1e-8 and stat.max() <= 1e-6
    inf = np.flatnonzero(st == 1)
    pick = inf[np.linspace(0, len(inf) - 1, 200 if N <= 40 else 40).astype(int)]
    slack = kref.feasibility_slack(xs[pick])
    assert np.all(slack <= 1e-6), f"LP finds a strictly feasible point for {int((slack > 1e-6).sum())} certified states"


@pytest.mark.parametrize("env_name", ["RoadEnv", "RoadMultipleCarsEnv"])
def test_every_shifted_grid_state_has_a_valid_certificate(torch_cuda, env_name):
    torch = torch_cuda
    c, bq = _setup(env_name, 20)
    g = np.array(c.goal, dtype=float)
    ref = Reference(env_name, 20)
    x0, _ = _grid(torch, g, shift=True)
    out = bq.solve(x0, want_u_full=True, want_certificate=True)
    _, _, info = _check_all(torch, ref, bq, x0, out, g, label=f"{env_name} shifted grid")
    assert info["undecided"] <= 300, "undecided states beyond DESIGN's count"


def test_per_sample_disturbance_batch_has_valid_certificates(torch_cuda):
    torch = torch_cuda
    d = np.load(os.path.join(GOLDEN, "disturbance.npz"))
    c, bq = _setup("RoadEnv", 20, cls="MPCOutputFBWithDisturbance", init_state=[20, 0.5, 0, 2])
    np.testing.assert_allclose(c.disturbance_response(), d["ABd_N20"], rtol=1e-12, atol=1e-12)
    ref = Reference("RoadEnv", 20, Gc=d["ABd_N20"])
    np.testing.assert_array_equal(bq.pq.rows_x, ref.rows)
    x_ref = np.array([30, 1.5, 0, 0.0])
    rng = np.random.default_rng(12)
    B = 200000
    x0 = torch.from_numpy(np.ascontiguousarray((x_ref + rng.uniform(-1, 1, size=(B, 4)) * [14.0, 1.6, 0.3, 3.0]).T)).cuda()
    dist = torch.from_numpy(rng.uniform(-0.05, 0.05, size=B)).cuda()
    plain = bq.solve(x0, x_ref=x_ref, c=dist, want_u_full=True)
    out = bq.solve(x0, x_ref=x_ref, c=dist, want_u_full=True, want_certificate=True)
    _assert_bit_identical(plain, out)
    _, _, info = _check_all(torch, ref, bq, x0, out, x_ref, c=dist, label="RoadEnv disturbance")
    assert info["solved"] > B // 10 and info["infeasible"] > B // 10
