"""The proof chain of the batched QP solver under starved solver budgets, against the exact oracle.

``qp_exact.cu`` promises that nothing leaves the library as solved without a float64 KKT certificate and nothing as
infeasible without a float64 Farkas certificate.  The stages that keep that promise (float64 verification of float32
"infeasible" verdicts, the Farkas filter before the second pass, the second ADMM pass, the final polish, the Farkas
decision on max_iter samples, the float64 fallback and its strict polish) see almost no samples with the default
options.  Here public solver options push whole batches down them, on the problems the project ships:

  starved   max_iter = check_every = 10: both ADMM passes stop after 10 iterations.  The polish still certifies most
            states from that iterate; the rest, one to a few percent of a batch (194, 330 and 883 of 20000 at horizon 20
            / 20 / 40), go through the float64 fallback and its strict polish
  loose     eps_abs = eps_rel = 0.3: the float32 ADMM stops early on a poor active set, which the polish must repair
            (certified_after_rounds[r >= 1]) or hand to the second pass (handed_to_admm)
  shy       eps_prim_inf = 2: the float32 infeasibility test (support <= -eps_prim_inf * sum |terms|) can never fire
            (|support| <= sum |terms|), so every infeasible state is settled by a Farkas certificate of its own ADMM state
            (before the second pass, or after it as a max_iter sample) or by the fallback.  A small eps_prim_inf would
            do the opposite: it makes the float32 test accept any negative support.
  eager     eps_prim_inf = -0.5: the float32 test then accepts positive support values, i.e. it calls feasible states
            infeasible (on a B200 with the polish off: 5 of 169 oracle-feasible RoadOneCarEnv states and 6 of 146
            RoadMultipleCarsEnv ones, horizon 20); the float64 verification must refuse every such verdict (after each
            ADMM pass), and the second pass or the fallback settles the samples.  At -1 the test sits on its own edge
            (|support| = sum |terms| whenever all terms share a sign), where the float32 rounding of the two sums decides
            and iteration counts vary from call to call.

Every (configuration, problem) pair asserts that its stage was reached (a polish_stats() counter above a floor measured
on a B200 with margin), then: flags equal to the oracle outside the 1e-6 slack band, status-2 samples bounded and
carrying NaN outputs and a zero certificate row, solutions within BASELINE's tolerances of the oracle and within 1e-7
of the default handle's, every decided sample's certificate accepted by the independent checker on the reference's own
matrices, consistent iteration and fallback bookkeeping, and bit-identical repeated calls (the fallback's work list is
built with atomicAdd, so its order varies from call to call; results must not).
"""
import os

import numpy as np
import pytest

from conftest import GOLDEN, make_env, make_controller
from test_qp_gpu import FIXTURE, GOAL, U_TOL, OBJ_RTOL, _config_states, _assert_same_solution
from test_qp_certificate_gpu import Reference, _check_all

pytestmark = pytest.mark.gpu

CONFIGS = {"starved": dict(max_iter=10, check_every=10), "loose": dict(eps_abs=0.3, eps_rel=0.3),
           "shy": dict(eps_prim_inf=2.0), "eager": dict(eps_prim_inf=-0.5)}

# name -> (environment, horizon, states, oracle subset)
PROBLEMS = {"onecar20": ("RoadOneCarEnv", 20, 20000, 400), "multi20": ("RoadMultipleCarsEnv", 20, 20000, 400),
            "road40": ("RoadEnv", 40, 20000, 300), "onecar80": ("RoadOneCarEnv", 80, 4000, 160),
            "onecar1": ("RoadOneCarEnv", 1, 4000, 400)}

CASES = [(c, p) for c in ("starved", "loose", "shy", "eager") for p in ("onecar20", "multi20")] + \
        [("starved", p) for p in ("road40", "onecar80", "onecar1")]

# The stage each configuration loads, as the counters that prove it ran, and the floor each must exceed per problem.
LOAD = {"starved": ("fallback_solved", "fallback_infeasible"),
        "loose": ("repaired", "handed_to_admm"),
        "shy": ("max_iter_settled_by_own_certificate", "infeasible_before_second_pass", "fallback_infeasible"),
        "eager": ("fallback_solved",)}
# Measured on a B200 (the sum of the LOAD counters): starved 194 / 330 / 883 / 57 / 10 (onecar20 / multi20 / road40 /
# onecar80 / onecar1), 419 with the disturbance; loose 7028 / 4772; shy 4166 / 2013; eager 499 / 109.
FLOOR = {("starved", "onecar20"): 100, ("starved", "multi20"): 160, ("starved", "road40"): 400, ("starved", "onecar80"): 25,
         ("starved", "onecar1"): 4, ("loose", "onecar20"): 3000, ("loose", "multi20"): 2000, ("shy", "onecar20"): 2000,
         ("shy", "multi20"): 1000, ("eager", "onecar20"): 250, ("eager", "multi20"): 50, ("starved", "disturbance"): 200}
# Undecided (status 2) samples allowed per batch.  Measured on a B200: 1 for starved / road40, 2 for starved / disturbance,
# 4 on the RoadMultipleCarsEnv grid of the seeded test, none elsewhere.
UNDECIDED = {("starved", "road40"): 5, ("starved", "disturbance"): 8, ("starved", "multi20 grid"): 15}
UNDECIDED_DEFAULT = 3


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "the GPU tests need a CUDA device"
    return torch


class _PQReference:
    """For a problem without golden matrices: the checker on the controller's own one-sided stack."""

    def __init__(self, pq):
        self.pq = pq

    def checker(self):
        from carmpc_b200.certificate import QPChecker
        return QPChecker.from_reference(self.pq)

    def numpy(self, x0, xref, status, u, cert, c=None):
        from cert_check import check_numpy
        pq = self.pq
        R = len(pq.rows_b)
        return check_numpy(pq.H, pq.F, pq.rows_x @ pq.S, pq.rows_x @ pq.T, np.full(R, -np.inf), pq.rows_b, pq.lb, pq.ub,
                           x0, xref, status, u, cert)


def _reference(env_name, N, pq):
    if os.path.isfile(os.path.join(GOLDEN, f"qp_{env_name}_N{N}.npz")):
        ref = Reference(env_name, N)
        np.testing.assert_array_equal(pq.rows_x, ref.rows)
        return ref
    return _PQReference(pq)


_PROBLEM_CACHE = {}


def _problem(torch, name):
    """Controller, states, the default handle's certified solve and the oracle on a strided subset (computed once)."""
    if name in _PROBLEM_CACHE:
        return _PROBLEM_CACHE[name]
    from carmpc_b200.batch import BatchQP
    from oracle import carmpc_oracle as orc
    env_name, N, n_states, n_oracle = PROBLEMS[name]
    c = make_controller(make_env(env_name, GOAL[env_name]), N)
    g = np.array(c.goal, dtype=float)
    oq = orc.CondensedQP(env_name, N, np.load(os.path.join(GOLDEN, "terminal_sets", FIXTURE[env_name])))
    x0 = _config_states(type("G", (), {"goal": g})(), n_states, seed=N + 1)
    x0_dev = torch.from_numpy(np.ascontiguousarray(x0.T)).cuda()
    default = BatchQP.from_controller(c)
    base = default.solve(x0_dev, want_u_full=True, want_certificate=True)
    sub = np.arange(0, n_states, n_states // n_oracle)[:n_oracle]
    oracle = orc.qp_solve_exact(oq, x0[sub], g)
    p = dict(c=c, g=g, oq=oq, x0=x0, x0_dev=x0_dev, base=base, sub=sub, oracle=oracle,
             ref=_reference(env_name, N, default.pq))
    _PROBLEM_CACHE[name] = p
    return p


def _stats(bq):
    s = bq.polish_stats()
    s["repaired"] = sum(s["certified_after_rounds"][1:])
    return s


def _host(out, k):
    return out[k].cpu().numpy()


def _assert_same_outputs(a, b):
    import torch
    for k in ("status", "iters", "u0", "objective", "u_full", "certificate"):
        x, y = a[k], b[k]
        if x.dtype == torch.float64:
            x, y = x.view(torch.int64), y.view(torch.int64)
        assert torch.equal(x, y), f"{k} differs between two identical calls"


def _assert_undecided_contract(out, label, bound):
    st = _host(out, "status")
    und = st == 2
    n2 = int(und.sum())
    assert n2 <= bound, f"{label}: {n2} undecided samples (bound {bound})"
    if n2:
        assert np.all(np.isnan(_host(out, "u0")[:, und])), f"{label}: an undecided sample carries a first input"
        assert np.all(np.isnan(_host(out, "u_full")[und])), f"{label}: an undecided sample carries an input sequence"
        assert np.all(np.isnan(_host(out, "objective")[und])), f"{label}: an undecided sample's objective is not NaN"
        assert np.all(_host(out, "certificate")[und] == 0.0), f"{label}: an undecided sample carries a certificate"
    inf = st == 1
    assert np.all(np.isposinf(_host(out, "objective")[inf])) and np.all(np.isnan(_host(out, "u0")[:, inf]))
    assert np.all(np.isnan(_host(out, "u_full")[inf]))
    return n2


def _assert_matches_oracle(out, p, label):
    """Flags outside the slack band equal the oracle's; solved samples within BASELINE's tolerances."""
    ue, obje, ste, polished, slack = p["oracle"]
    sub = p["sub"]
    st = _host(out, "status")[sub]
    band = np.abs(slack) <= 1e-6
    dec = (st != 2) & ~band
    np.testing.assert_array_equal(np.where(st[dec] == 0, 0, 1), ste[dec], err_msg=f"{label}: flags differ from the oracle")
    ok = (ste == 0) & ~band & polished & (st == 0)
    assert ok.sum() >= len(sub) // 10, f"{label}: too few solved oracle samples ({ok.sum()})"
    du = float(np.abs(_host(out, "u0").T[sub][ok] - ue[ok, :2]).max())
    duf = float(np.abs(_host(out, "u_full")[sub][ok] - ue[ok]).max())
    obj = _host(out, "objective")[sub]
    rel = float((np.abs(obj[ok] - obje[ok]) / np.maximum(1.0, np.abs(obje[ok]))).max())
    assert du <= U_TOL and duf <= U_TOL, f"{label}: inputs differ from the oracle by {max(du, duf)}"
    assert rel <= OBJ_RTOL, f"{label}: objectives differ from the oracle by {rel} (relative)"
    return du, rel


def _assert_matches_default(out, base, oq, x0, label):
    """Both are certified: solved samples agree to 1e-7, flags of decided samples agree outside the slack band."""
    from oracle import carmpc_oracle as orc
    sa, sb = _host(out, "status"), _host(base, "status")
    diff = np.flatnonzero((sa != sb) & (sa != 2) & (sb != 2))
    if len(diff):
        assert len(diff) <= 3, f"{label}: {len(diff)} flags differ from the default handle's"
        _, slack = orc.qp_feasible_lp(oq, x0[diff])
        assert np.all(np.abs(slack) <= 1e-6), f"{label}: flags differ outside the slack band: {slack}"
    ok = (sa == 0) & (sb == 0)
    du = float(np.abs(_host(out, "u0")[:, ok] - _host(base, "u0")[:, ok]).max(initial=0.0))
    duf = float(np.abs(_host(out, "u_full")[ok] - _host(base, "u_full")[ok]).max(initial=0.0))
    oa, ob = _host(out, "objective")[ok], _host(base, "objective")[ok]
    rel = float((np.abs(oa - ob) / np.maximum(1.0, np.abs(ob))).max(initial=0.0))
    assert du <= 1e-7 and duf <= 1e-7, f"{label}: inputs differ from the default handle by {max(du, duf)}"
    assert rel <= 1e-8, f"{label}: objectives differ from the default handle by {rel} (relative)"
    return du, rel


def _assert_numpy_certificates(torch, p, bq, out, label, c=None, n=300):
    """The numpy restatement of the checker accepts a few hundred decided samples (all kinds of verdict)."""
    from carmpc_b200.certificate import passes, to_one_sided
    st = _host(out, "status")
    dec = np.flatnonzero(st != 2)
    pick = dec[np.linspace(0, len(dec) - 1, min(n, len(dec))).astype(int)]
    one = to_one_sided(bq.pq, out["certificate"]).cpu().numpy()[pick]
    kw = {} if c is None else {"c": c[pick]}
    r = p["ref"].numpy(p["x0"][pick], p["g"], st[pick], _host(out, "u_full")[pick], one, **kw)
    bad = np.flatnonzero(~passes(st[pick], r))
    assert len(bad) == 0, f"{label}: numpy checker rejects samples {pick[bad[:5]]}: {r[bad[:5]]}"


def _assert_bookkeeping(bq, out, s, config, label):
    st = _host(out, "status")
    iters = _host(out, "iters")
    total, launches = bq.last_stats()
    assert total == int(iters.astype(np.int64).sum()), f"{label}: last_stats iterations {total} != sum of iters"
    settled = s["fallback_solved"] + s["fallback_infeasible"] + s["fallback_undecided"]
    # Every sample the fallback takes ends in exactly one of its three counters, and only the fallback leaves a sample
    # undecided (status 2) when the polish is on.  (A sample the float64 ADMM left at max_iter and the strict polish then
    # could not certify used to be counted twice.)
    assert s["fallback_undecided"] == int((st == 2).sum()), f"{label}: fallback_undecided {s['fallback_undecided']} != " \
                                                            f"{int((st == 2).sum())} undecided samples"
    # No counter holds the number of samples that entered the fallback.  A lower bound holds in every configuration: each
    # sample the final polish leaves uncertified (final_polish_uncertified) enters it, unless the Farkas decision proves
    # it infeasible first (max_iter_settled_by_own_certificate); the others come from second-pass "infeasible" verdicts
    # that the float64 verification refuses, which no counter records.
    lower = s["final_polish_uncertified"] - s["max_iter_settled_by_own_certificate"]
    assert settled >= lower, f"{label}: fallback counters {settled} below the {lower} samples the final polish handed it"
    # Under `starved` the number follows from the iteration counts: the two float32 passes give a sample at most
    # 2 * max_iter iterations, and the fallback adds at least one check interval (25 float64 iterations) to every sample
    # it takes.
    if config == "starved":
        entered = int((iters > 2 * CONFIGS["starved"]["max_iter"]).sum())
        assert settled == entered, f"{label}: fallback counters {settled} != {entered} samples it iterated on"
    return settled


def _run_case(torch, bq, p, label, floor, load, bound, c=None):
    x0 = p["x0_dev"]
    kw = {} if c is None else {"c": c, "x_ref": p["g"]}
    out = bq.solve(x0, want_u_full=True, want_certificate=True, **kw)
    s = _stats(bq)
    again = bq.solve(x0, want_u_full=True, want_certificate=True, **kw)
    assert _stats(bq) == s, f"{label}: polish_stats differ between two identical calls"
    _assert_same_outputs(out, again)
    n2 = _assert_undecided_contract(out, label, bound)
    print(f"\n{label}: stats {s}, launches {bq.last_stats()[1]}, undecided {n2}")
    reached = sum(s[k] for k in load)
    assert reached > floor, f"{label}: {' + '.join(load)} = {reached}, not above the floor {floor}: stage not reached"
    return out, s


@pytest.mark.parametrize("config,problem", CASES)
def test_forced_stage_keeps_the_proof_promise(torch_cuda, config, problem):
    torch = torch_cuda
    from carmpc_b200.batch import BatchQP
    p = _problem(torch, problem)
    label = f"{config} / {problem}"
    bq = BatchQP.from_controller(p["c"], **CONFIGS[config])
    bound = UNDECIDED.get((config, problem), UNDECIDED_DEFAULT)
    out, s = _run_case(torch, bq, p, label, FLOOR[(config, problem)], LOAD[config], bound)
    if problem == "road40":
        tm = bq.tensor_mode()
        print(f"{label}: tensor mode {tm['mode']}, samples on the tcgen05 kernel {tm['samples_last_solve']}")
        assert tm["samples_last_solve"] > 0, "the horizon-40 first pass did not run on the tcgen05 kernel"
    du_o, rel_o = _assert_matches_oracle(out, p, label)
    du_d, rel_d = _assert_matches_default(out, p["base"], p["oq"], p["x0"], label)
    _, _, info = _check_all(torch, p["ref"], bq, p["x0_dev"], out, p["g"], label=label)
    _assert_numpy_certificates(torch, p, bq, out, label)
    settled = _assert_bookkeeping(bq, out, s, config, label)
    print(f"{label}: oracle |du0| {du_o:.2e} rel dobj {rel_o:.2e}; default |du| {du_d:.2e} rel dobj {rel_d:.2e}; "
          f"fallback settled {settled}; certificates {info}")


def test_disturbance_batch_through_the_fallback(torch_cuda):
    """MPCOutputFBWithDisturbance with a per-sample disturbance c, starved.  The public entry points skip the Farkas
    filter and decision with a disturbance (they keep max_iter there), but the float64 verification and the fallback
    run on the shifted bounds: whatever they decide must carry a certificate valid for the shifted problem, and
    the flags must agree with the default handle's and with the oracle on the shifted problem."""
    torch = torch_cuda
    from carmpc_b200.batch import BatchQP
    from oracle import carmpc_oracle as orc
    d = np.load(os.path.join(GOLDEN, "disturbance.npz"))
    ctl = make_controller(make_env("RoadEnv"), 20, cls="MPCOutputFBWithDisturbance", init_state=[20, 0.5, 0, 2])
    np.testing.assert_allclose(ctl.disturbance_response(), d["ABd_N20"], rtol=1e-12, atol=1e-12)
    g = np.array([30, 1.5, 0, 0.0])
    B = 8000
    x0 = _config_states(type("G", (), {"goal": g})(), B, seed=23)
    rng = np.random.default_rng(23)
    cd = rng.uniform(-0.05, 0.05, size=B)
    Ab = np.load(os.path.join(GOLDEN, "terminal_sets", FIXTURE["RoadEnv"]))
    p = dict(x0=x0, x0_dev=torch.from_numpy(np.ascontiguousarray(x0.T)).cuda(), g=g,
             ref=Reference("RoadEnv", 20, Gc=d["ABd_N20"]))
    c = torch.from_numpy(cd).cuda()
    label = "starved / disturbance"
    bq = BatchQP.from_controller(ctl, **CONFIGS["starved"])
    out, s = _run_case(torch, bq, p, label, FLOOR[("starved", "disturbance")], LOAD["starved"],
                       UNDECIDED[("starved", "disturbance")], c=c)
    base = BatchQP.from_controller(ctl).solve(p["x0_dev"], x_ref=g, c=c, want_u_full=True, want_certificate=True)
    # the default handle's max_iter samples may be decided here and vice versa; decided flags must agree
    oq = orc.CondensedQP("RoadEnv", 20, Ab)
    sa, sb = _host(out, "status"), _host(base, "status")
    both = (sa != 2) & (sb != 2)
    diff = np.flatnonzero(both & (sa != sb))
    assert len(diff) <= 3, f"{label}: {len(diff)} flags differ from the default handle's"
    ok = (sa == 0) & (sb == 0)
    du = float(np.abs(_host(out, "u_full")[ok] - _host(base, "u_full")[ok]).max())
    assert du <= 1e-7, f"{label}: inputs differ from the default handle by {du}"
    _, _, info = _check_all(torch, p["ref"], bq, p["x0_dev"], out, g, c=c, label=label)
    _assert_numpy_certificates(torch, p, bq, out, label, c=cd)
    settled = _assert_bookkeeping(bq, out, s, "starved", label)
    # oracle on the shifted problem (bounds moved by rows @ ABd * c), a strided subset
    rows = np.vstack((orc.terminal_constraint(Ab, 20)[0], np.zeros((80, 84)), orc.state_constraint("RoadEnv", 20)[0]))
    Gd = rows @ d["ABd_N20"]
    n_ok = 0
    for i in np.arange(0, B, B // 80)[:80]:
        q = orc.CondensedQP("RoadEnv", 20, Ab)
        q.w = q.w - Gd * cd[i]
        ue, obje, ste, pol, slack = orc.qp_solve_exact(q, x0[i:i + 1], g)
        if abs(slack[0]) <= 1e-6 or sa[i] == 2:
            continue
        assert (sa[i] == 0) == (ste[0] == 0), f"{label}: state {i} flag {sa[i]}, oracle {ste[0]}"
        if ste[0] == 0 and pol[0]:
            n_ok += 1
            assert np.abs(_host(out, "u_full")[i] - ue[0]).max() <= U_TOL
            assert abs(_host(out, "objective")[i] - obje[0]) <= OBJ_RTOL * max(1.0, abs(obje[0]))
    assert n_ok >= 10
    print(f"{label}: differing decided flags {len(diff)}, |du| vs default {du:.2e}, fallback settled {settled}, "
          f"certificates {info}")


# ---------------------------------------------------------------------------------------------------------------------
# the other entry points under `starved`
# ---------------------------------------------------------------------------------------------------------------------
def _grid(torch, g):
    from carmpc_b200.grids import materialise_grid
    axes = [np.linspace(g[0] - 20.0, g[0] + 0.5, 24), np.linspace(-3.0, 3.0, 40), np.linspace(-0.3, 0.3, 3),
            np.linspace(-1.0, 4.0, 4)]
    return axes, torch.stack(materialise_grid(axes, device="cuda")).contiguous()


@pytest.mark.parametrize("problem", ["onecar20", "multi20"])
def test_starved_seeded_solve_and_map_match_the_cold_solve(torch_cuda, problem):
    torch = torch_cuda
    from carmpc_b200.batch import BatchQP
    from carmpc_b200.grids import lattice_seeds
    p = _problem(torch, problem)
    label = f"starved / {problem} grid"
    bq = BatchQP.from_controller(p["c"], **CONFIGS["starved"])
    axes, x0 = _grid(torch, p["g"])
    B = x0.shape[1]
    cold = bq.solve(x0, want_u_full=True, want_certificate=True)
    s_cold = _stats(bq)
    seed = torch.from_numpy(lattice_seeds([len(a) for a in axes], block=(2, 8, 1, 1))).cuda()
    warm = bq.solve(x0, want_u_full=True, want_certificate=True, seed=seed)
    s_warm = _stats(bq)
    print(f"\n{label}: cold stats {s_cold}\n{label}: seeded stats {s_warm}, seeded {warm['seeded']}")
    st = _host(cold, "status")
    assert (st == 0).sum() > B // 10 and (st == 1).sum() > 0, "the grid should cross the region-of-attraction boundary"
    # both solves reach the fallback (the seeded one through its anchors and through followers whose seed did not
    # certify); measured on a B200: 108 / 104 (onecar20) and 124 / 120 (multi20) settled, cold / seeded
    for s, tag in ((s_cold, "cold"), (s_warm, "seeded")):
        reached = s["fallback_solved"] + s["fallback_infeasible"]
        assert reached > FLOOR[("starved", problem)] // 4, f"{label} {tag}: the fallback settled only {reached} samples"
    bound = UNDECIDED.get(("starved", f"{problem} grid"), UNDECIDED_DEFAULT)
    for out, s, tag in ((cold, s_cold, "cold"), (warm, s_warm, "seeded")):
        n2 = _assert_undecided_contract(out, f"{label} {tag}", bound)
        assert s["fallback_undecided"] == n2, f"{label} {tag}: fallback_undecided {s['fallback_undecided']} != {n2}"
        _check_all(torch, p["ref"], bq, x0, out, p["g"], label=f"{label} {tag}")
    # undecided samples of either solve are left out of the comparison (bounded above)
    dec = torch.from_numpy(np.flatnonzero((st != 2) & (_host(warm, "status") != 2))).cuda()
    pick = lambda o: {k: (o[k][:, dec] if k == "u0" else o[k][dec]) for k in ("status", "u0", "objective", "u_full")}
    _assert_same_solution(pick(cold), pick(warm), p["oq"], x0[:, dec])
    assert warm["seeded"] > 0
    # the host-buffer map entry point: cold and seeded maps of the same grid give the batched solve's statuses
    for block in (None, (2, 8, 1, 1)):
        res = bq.solve_map_host(axes, block=block)
        np.testing.assert_array_equal(res.status, st, err_msg=f"{label}: map statuses (block {block}) differ")
        ok = st == 0
        assert np.abs(res.u0[ok] - _host(cold, "u0").T[ok]).max() <= 1e-7


_LOOP_CACHE = {}
# Runs of the closed-loop test, and the strided subset of them the oracle steps as well.  Warm-started steps mostly settle
# from the reused active set, so the float64 fallback sees only a few samples per hundred runs over 30 steps: the run
# count is what makes its device-sized form see enough of them.
LOOP_RUNS, LOOP_ORACLE_RUNS, LOOP_STEPS = 2048, 64, 30
# Samples the fallback settled in the device-sized steps (all but the first) of the warm_start = 1 loop, measured on a
# B200: LOOP_MEASURED (output feedback / state feedback).
LOOP_FLOOR = {True: 1, False: 1}


def _loop(bq, c, x_init, steps, output_feedback, warm_start):
    from oracle import carmpc_oracle as orc
    return bq.closed_loop(x_init, steps, c.A, c.B, C=orc.C_OUT if output_feedback else None,
                          L=orc.L_OBS if output_feedback else None, warm_start=warm_start, want_traj=True)


@pytest.mark.parametrize("warm_start", [1, 0])
@pytest.mark.parametrize("output_feedback", [True, False])
def test_starved_closed_loops_match_the_oracle(torch_cuda, output_feedback, warm_start):
    """warm_start = 1 runs every step after the first through the device-sized pipeline (sample counts stay on the
    device, the fallback's included); warm_start = 0 every step through the host-driven one.  A strided subset of the runs
    must step exactly as the oracle's loop with exact QP solutions: a run stops at the same step, and the trajectories
    agree to 1e-6.  With warm_start = 1 the fallback must have settled samples in the device-sized steps (the polish
    histogram accumulates over them; the first step is a host-driven solve, measured apart on a fresh handle), and all
    runs must step as the warm_start = 0 loop does."""
    torch = torch_cuda
    from carmpc_b200.batch import BatchQP
    from oracle import carmpc_oracle as orc
    c = make_controller(make_env("RoadEnv"), 20)
    g = np.array(c.goal, dtype=float)
    oq = orc.CondensedQP("RoadEnv", 20, np.load(os.path.join(GOLDEN, "terminal_sets", FIXTURE["RoadEnv"])))
    R, steps = LOOP_RUNS, LOOP_STEPS
    x_host = np.random.default_rng(31).uniform([0, -2.5, -0.2, 0], [10, 2.5, 0.2, 3], size=(R, 4))
    x_init = torch.from_numpy(np.ascontiguousarray(x_host.T)).cuda()
    sub = np.arange(0, R, R // LOOP_ORACLE_RUNS)[:LOOP_ORACLE_RUNS]
    if output_feedback not in _LOOP_CACHE:
        def exact(x):
            u, obj, st, *_ = orc.qp_solve_exact(oq, x, g)
            return u[:, :2], st
        _LOOP_CACHE[output_feedback] = orc.closed_loop(oq, x_host[sub], g, steps, output_feedback, exact)
    want_x, want_fail, want_traj = _LOOP_CACHE[output_feedback]
    bq = BatchQP.from_controller(c, **CONFIGS["starved"])
    out = _loop(bq, c, x_init, steps, output_feedback, warm_start)
    s = _stats(bq)
    fail = _host(out, "fail_step")
    traj = _host(out, "traj").transpose(0, 2, 1)
    label = f"closed loop (output feedback {output_feedback}, warm_start {warm_start})"
    print(f"\n{label}: failed runs {int((fail >= 0).sum())} of {R}, total iterations {out['total_iters']}")
    np.testing.assert_array_equal(fail[sub], want_fail, err_msg=f"{label}: runs stop at other steps than the oracle's")
    alive = want_fail < 0
    assert alive.sum() >= len(sub) // 4
    err = float(np.abs(traj[:, sub][:, alive] - want_traj[:, alive]).max())
    assert err <= 1e-6, f"{label}: trajectories differ from the oracle's by {err}"
    np.testing.assert_allclose(_host(out, "final").T[sub][alive], want_x[alive], atol=1e-6)
    if warm_start != 1:
        return
    first = BatchQP.from_controller(c, **CONFIGS["starved"])
    _loop(first, c, x_init, 1, output_feedback, warm_start)
    s1 = _stats(first)
    keys = ("fallback_solved", "fallback_infeasible", "fallback_undecided", "final_polish_uncertified")
    later = {k: s[k] - s1[k] for k in keys}
    print(f"{label}: first step {({k: s1[k] for k in keys})}, device-sized steps {later}")
    reached = later["fallback_solved"] + later["fallback_infeasible"]
    assert reached > LOOP_FLOOR[output_feedback], \
        f"{label}: the fallback settled {reached} samples in the device-sized steps, floor {LOOP_FLOOR[output_feedback]}"
    # every run steps as the host-driven loop does (both apply certified optima of the same QPs)
    ref = _loop(BatchQP.from_controller(c, **CONFIGS["starved"]), c, x_init, steps, output_feedback, 0)
    np.testing.assert_array_equal(fail, _host(ref, "fail_step"), err_msg=f"{label}: runs stop at other steps than with "
                                                                          "warm_start = 0")
    live = fail < 0
    err = float(np.abs(traj[:, live] - _host(ref, "traj").transpose(0, 2, 1)[:, live]).max())
    assert err <= 1e-6, f"{label}: trajectories differ from the warm_start = 0 loop's by {err}"
