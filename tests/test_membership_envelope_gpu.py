"""Terminal-set membership across its whole envelope, bit for bit against the C oracle (needs a B200).

The shipped terminal sets have 25 to 42 rows of modest scale, and the float32 screen of mode 1 is only sound if its
rounding-error bound covers every input.  These tests feed the kernels what the C ABI accepts but the shipped sets never
exercise: rows beyond or below the float32 range (part A), synthetic polytopes of 0 to 512 rows with mixed sparsity,
scales from 1e-3 to 1e3, exact ties and special coordinates (part B), and synthetic rollout forms up to the 512-row
screen limit (part C).  Every path that runs the screen is taken: the plain kernel, the bulk-async kernel (aligned,
n >= 65,536, ragged tail), unaligned views, the host pipeline and the implicit-grid kernel.  The reference is always the
float64 fma chain of oracle/c_oracle.py, compared with ==, bitset and count.
"""
import numpy as np
import pytest

from test_membership_screen_cpu import CASES, CASE_IDS, ROLLOUT, ROLLOUT_POINT, polytope

pytestmark = pytest.mark.gpu

BULK_N = 70 * 1024 + 37          # above the bulk-async threshold (64 chunks of 1024), with a ragged tail
SPECIALS = [np.nan, np.inf, -np.inf, 1e300, -1e300, 1e38, -0.0, 1e-310]


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "the GPU tests need a CUDA device"
    return torch


def _dev(torch, cols):
    return [torch.from_numpy(np.ascontiguousarray(c, dtype=np.float64)).cuda() for c in cols]


def _unaligned(torch, cols):
    """Views one element into their allocation: 8-byte aligned only, so the kernels take the scalar-load path."""
    out = []
    for c in cols:
        t = torch.from_numpy(np.concatenate(([0.0], np.asarray(c, dtype=np.float64)))).cuda()[1:]
        assert t.data_ptr() % 16 == 8
        out.append(t)
    return out


def _bits_np(bits):
    return bits.cpu().numpy().view(np.uint32)


def _tile(cols, n, rng, special_idx=()):
    """n samples: the given ones repeated in random order, each given sample also at the listed indices."""
    m = len(cols[0])
    idx = rng.integers(0, m, size=n)
    for j, i in enumerate(special_idx):
        idx[i] = j % m
    return [np.ascontiguousarray(c[idx]) for c in cols]


def _check_hrep(torch, ev, Ab, cols, paths, modes=(0, 1), what=""):
    """Every listed path and mode of a TerminalSetEvaluator against the oracle: bitset and count."""
    from oracle import c_oracle
    want_bits, want_cnt = c_oracle.membership_bits(Ab, *cols)
    for path in paths:
        for mode in modes:
            tag = f"{what} path={path} mode={mode}"
            if path == "host":
                bits, cnt = ev.contains_bits_host(*cols, mode=mode)
                np.testing.assert_array_equal(bits, want_bits, err_msg=tag)
                assert cnt == want_cnt, tag
                continue
            t = _unaligned(torch, cols) if path == "unaligned" else _dev(torch, cols)
            bits, cnt = ev.contains_bits(*t, mode=mode)
            np.testing.assert_array_equal(_bits_np(bits), want_bits, err_msg=tag)
            assert int(cnt.item()) == want_cnt, tag
    return want_bits, want_cnt


# ---- A. adversarial scaling ------------------------------------------------------------------------------------------
def _adversarial_samples(point, beta, n, rng):
    """n samples: benign random ones with the adversarial point at the start, around group and word edges, spread
    through the body and in the ragged tail."""
    scale = min(beta, 1.0)
    cols = [rng.uniform(-2, 2, n), rng.uniform(-2, 2, n), rng.uniform(-1.5, 1.5, n) * scale, rng.uniform(-1.5, 1.5, n) * scale]
    at = {0, 1, 31, 32, 33, 127, 128, 1023, 1024, n - 1, n - 2, n - 33}
    at |= set(range(5, n, 997))
    at = sorted(i for i in at if 0 <= i < n)
    for k in range(4):
        cols[k][at] = point[k]
    return cols, at


PATHS_A = ["plain", "bulk", "unaligned", "host"]


@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("path", PATHS_A)
@pytest.mark.parametrize("name,row,point,beta,expect", CASES, ids=CASE_IDS)
def test_adversarial_polytope(torch_cuda, name, row, point, beta, expect, path, mode):
    from carmpc_b200.batch import TerminalSetEvaluator, unpack_bits
    Ab = polytope(row, beta)
    rng = np.random.default_rng(1000 + CASE_IDS.index(name))
    n = 45 if path in ("plain", "host") else BULK_N
    cols, at = _adversarial_samples(point, beta, n, rng)
    ev = TerminalSetEvaluator(Ab)
    want_bits, _ = _check_hrep(torch_cuda, ev, Ab, cols, [path], modes=(mode,), what=name)
    assert (unpack_bits(want_bits, n)[at] == expect).all()


@pytest.mark.parametrize("name,row,point,beta,expect", CASES, ids=CASE_IDS)
def test_adversarial_polytope_grid(torch_cuda, name, row, point, beta, expect):
    """The implicit-grid kernel with the adversarial coordinates as axis values."""
    from carmpc_b200.batch import TerminalSetEvaluator, unpack_bits
    from oracle import c_oracle
    Ab = polytope(row, beta)
    axes = [np.array([point[0], 0.0, 1.0]), np.array([point[1], -1.0, 0.5]), np.array([point[2], 0.5 * min(beta, 1.0)]),
            np.array([point[3]])]
    n = 18
    cols = [c.ravel() for c in np.meshgrid(*axes, indexing="ij")]
    want_bits, want_cnt = c_oracle.membership_bits(Ab, *cols)
    ev = TerminalSetEvaluator(Ab)
    bits, cnt = ev.contains_grid_bits(axes)
    np.testing.assert_array_equal(_bits_np(bits), want_bits)
    assert int(cnt.item()) == want_cnt
    assert unpack_bits(want_bits, n)[0] == expect          # grid point 0 is the adversarial point


ROLLOUT_PATHS = ["plain", "bulk", "unaligned", "host", "first_violation"]


@pytest.mark.parametrize("path", ROLLOUT_PATHS)
def test_adversarial_rollout(torch_cuda, path):
    from carmpc_b200.batch import RolloutEvaluator, unpack_bits
    from oracle import c_oracle
    R = ROLLOUT
    ev = RolloutEvaluator(R["A_k"], R["A_con"], R["b_con"], R["A_in"], R["b_in"], R["goal"], R["k_steps"],
                          reduce_screen=False)
    assert len(ev.expanded()) == len(R["b_con"]) * (R["k_steps"] + 1)       # the float32 screen is on
    rng = np.random.default_rng(77)
    n = 45 if path in ("plain", "host", "first_violation") else BULK_N
    cols, at = _adversarial_samples(ROLLOUT_POINT, 1.0, n, rng)
    want_bits, want_first, want_cnt = c_oracle.rollout_bits(R["A_k"], R["A_con"], R["b_con"], R["A_in"], R["b_in"],
                                                            R["goal"], R["k_steps"], 0, *cols)
    assert unpack_bits(want_bits, n)[at].all()
    if path == "host":
        bits, cnt = ev.contains_bits_host(*cols)
        np.testing.assert_array_equal(bits, want_bits)
        assert cnt == want_cnt
        return
    t = _unaligned(torch_cuda, cols) if path == "unaligned" else _dev(torch_cuda, cols)
    if path == "first_violation":
        bits, cnt, first = ev.contains_bits(*t, want_first_violation=True)
        np.testing.assert_array_equal(first.cpu().numpy(), want_first)
    else:
        bits, cnt = ev.contains_bits(*t)
    np.testing.assert_array_equal(_bits_np(bits), want_bits)
    assert int(cnt.item()) == want_cnt


# ---- B. synthetic polytopes across the row range ---------------------------------------------------------------------
ROW_COUNTS = [0, 1, 2, 7, 8, 9, 63, 64, 65, 200, 511, 512]
ROW_CASES = [(r, "mixed") for r in ROW_COUNTS] + [(9, "zero_row_below_zero"), (64, "minus_inf_row")]


def synthetic_polytope(rows, variant, rng):
    """rows x 5 [A | b] around the origin, facets at distance about 0.7 to 3.

    Even rows are dyadic: a = s k (k small integers, s = 2^e with e in [-10, 10]) and b = tau s |k|^2, so that the point
    tau k lies exactly on the facet in float64 and in float32 alike.  Odd rows have non-dyadic coefficients.  The sparsity
    cycles through axis-aligned, 2-sparse and dense; every seventh row has no bound (b = +inf); rows 3 (b > 0) and, for
    an odd count, 5 (b = 0) are all zero.  Variants put a zero row with b < 0 or a row with b = -inf in: an empty set.
    Returns the rows and, for every dyadic row with a bound, its facet point tau k."""
    Ab = np.zeros((rows, 5))
    ties = []
    for r in range(rows):
        s = 2.0 ** rng.integers(-10, 11)
        nnz = (1, 2, 4)[r % 3]
        support = rng.choice(4, size=nnz, replace=False)
        if r == 3:
            Ab[r, 4] = 1.5 * s
            continue
        if r == 5 and rows % 2 == 1:
            continue                                         # 0 . p <= 0: an exact tie for every finite sample
        if r % 2 == 0:
            k = np.zeros(4)
            k[support] = rng.integers(1, 8, size=nnz) * rng.choice([-1.0, 1.0], size=nnz)
            kk = float(k @ k)
            tau = 2.0 ** -np.round(0.5 * np.log2(kk)) * (1 + rng.integers(0, 8) / 8)
            Ab[r, :4] = s * k
            Ab[r, 4] = tau * s * kk
            ties.append(tau * k)
        else:
            u = np.zeros(4)
            u[support] = rng.uniform(-1, 1, size=nnz)
            u[support] += np.sign(u[support]) * 0.05
            Ab[r, :4] = s * u
            Ab[r, 4] = s * np.linalg.norm(u) * rng.uniform(0.7, 3.0)
        if r % 7 == 6:
            Ab[r, 4] = np.inf
            if r % 2 == 0:
                ties.pop()
    if variant == "zero_row_below_zero":
        Ab[rows // 2] = (0.0, 0.0, 0.0, 0.0, -2.0 ** -20)
    elif variant == "minus_inf_row":
        Ab[rows // 2, 4] = -np.inf
    return Ab, np.array(ties).reshape(-1, 4)


def synthetic_samples(ties, rng, n_random=4000):
    """Random points (radius log-uniform over 0.05 .. 5), the exact facet points and 1 or 2 ulps either side of them in
    their largest coordinate, and special coordinates in every position."""
    d = rng.normal(size=(n_random, 4))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    pts = [d * np.exp(rng.uniform(np.log(0.05), np.log(5.0), size=(n_random, 1)))]
    if len(ties):
        pts.append(ties)
        j = np.argmax(np.abs(ties), axis=1)
        for steps in (1, 2, -1, -2):
            q = ties.copy()
            c = q[np.arange(len(q)), j]
            for _ in range(abs(steps)):
                c = np.nextafter(c, np.inf if steps > 0 else -np.inf)
            q[np.arange(len(q)), j] = c
            pts.append(q)
    base = rng.uniform(-0.1, 0.1, size=(len(SPECIALS) * 4, 4))
    for i, sp in enumerate(SPECIALS):
        for k in range(4):
            base[4 * i + k, k] = sp
    pts.append(base)
    pts.append(np.array([[sp] * 4 for sp in SPECIALS]))
    p = np.vstack(pts)
    return [np.ascontiguousarray(c) for c in p.T]


def _grid_axes(rng):
    """An implicit grid with one axis of 4096 points (the per-axis limit): dyadic values (facet coordinates of the
    axis-aligned dyadic rows among them) and specials; 4096 x 3 x 2 x 2 = 49,152 points."""
    x = np.concatenate((np.arange(-2047, 2047) / 512.0, [np.nan, 1e300]))
    assert len(x) == 4096
    return [x, np.array([-0.5, 1e-310, 0.75]), np.array([-0.0, 0.125]), np.array([0.0625, -1e38])]


@pytest.mark.parametrize("rows,variant", ROW_CASES, ids=[f"{r}-{v}" for r, v in ROW_CASES])
def test_synthetic_polytope(torch_cuda, rows, variant):
    from carmpc_b200.batch import TerminalSetEvaluator, unpack_bits
    from oracle import c_oracle
    torch = torch_cuda
    rng = np.random.default_rng(rows * 31 + len(variant))
    Ab, ties = synthetic_polytope(rows, variant, rng)
    small = synthetic_samples(ties, rng)
    n_small = len(small[0])
    big = _tile(small, BULK_N, rng, special_idx=range(n_small))
    ev = TerminalSetEvaluator(Ab)
    want_small, cnt_small = _check_hrep(torch, ev, Ab, small, ["plain", "unaligned", "host"], what=f"{rows} rows")
    _check_hrep(torch, ev, Ab, big, ["bulk", "unaligned", "host"], what=f"{rows} rows, {BULK_N} samples")
    if variant == "mixed":
        member = unpack_bits(want_small, n_small)
        assert 0 < cnt_small < n_small or rows <= 2
        if len(ties):
            # some facet points are members: ties decide, not only clear margins
            k = len(ties)
            on_facet = member[4000:4000 + k]
            assert on_facet.any() or rows > 200
    else:
        assert cnt_small == 0
    # the implicit-grid kernel
    axes = _grid_axes(rng)
    cols = [c.ravel() for c in np.meshgrid(*axes, indexing="ij")]
    want_bits, want_cnt = c_oracle.membership_bits(Ab, *cols)
    bits, cnt = ev.contains_grid_bits(axes)
    np.testing.assert_array_equal(_bits_np(bits), want_bits)
    assert int(cnt.item()) == want_cnt
    if rows in (64, 65):
        # the pilot re-orders up to 64 rows (and leaves 65 as they are): results must not depend on the order
        ev.tune(*_dev(torch, big))
        _check_hrep(torch, ev, Ab, small, ["plain"], what=f"{rows} rows after tune()")
        _check_hrep(torch, ev, Ab, big, ["bulk"], what=f"{rows} rows after tune()")
        bits, cnt = ev.contains_grid_bits(axes)
        np.testing.assert_array_equal(_bits_np(bits), want_bits)
    if rows == 512:
        # the largest shared-memory footprint of the bulk-async kernel, in every built staging geometry
        for geo in [(256, 3, 1), (128, 3, 1), (128, 4, 1), (128, 2, 2), (128, 3, 2), (256, 2, 1), (128, 2, 1), (256, 2, 2)]:
            ev.set_staging(*geo)
            _check_hrep(torch, ev, Ab, big, ["bulk"], modes=(1,), what=f"512 rows, staging {geo}")


# ---- C. synthetic rollout forms --------------------------------------------------------------------------------------
def synthetic_Ak(kind, rng):
    Q, _ = np.linalg.qr(rng.normal(size=(4, 4)))
    if kind == "contracting":
        return Q @ np.diag([0.9, -0.7, 0.5, 0.3]) @ Q.T
    if kind == "expanding":
        return Q @ np.diag([1.5, 0.9, -0.6, 0.4]) @ Q.T              # spectral radius 1.5
    assert kind == "nilpotent"
    return np.triu(rng.uniform(-1, 1, size=(4, 4)), 1)               # A^4 = 0: later expanded rows are zero


def synthetic_rows(m, rng):
    """m rows [a | b] of mixed sparsity, scales log-uniform over 1e-3 .. 1e3, facets at distance 0.5 to 3."""
    A = np.zeros((m, 4))
    for r in range(m):
        support = rng.choice(4, size=(1, 2, 4)[r % 3], replace=False)
        A[r, support] = rng.uniform(-1, 1, size=len(support)) + 0.05
    A *= np.exp(rng.uniform(np.log(1e-3), np.log(1e3), size=(m, 1)))
    b = np.linalg.norm(A, axis=1) * rng.uniform(0.5, 3.0, size=m)
    if m > 4:
        b[m // 3] = np.inf
    return A, b


# (s, rin, k_steps, input_every_step, A_k, nonzero goal): the screen holds s (k + 1) + rin (k + 1 or 1) expanded rows
ROLLOUT_FORMS = [
    (32, 0, 15, False, "contracting", False),       # 512 rows: the screen limit, screen on
    (32, 0, 16, False, "contracting", True),        # 544 rows: screen off, exact kernel only
    (16, 16, 15, True, "expanding", True),          # 512 rows, input rows at every step
    (0, 1, 5, False, "contracting", True),
    (1, 0, 5, True, "nilpotent", False),
    (256, 0, 1, False, "nilpotent", True),          # 512 rows
    (0, 256, 3, False, "expanding", False),         # input rows at t = 0 only: 256 rows
    (256, 256, 0, True, "contracting", True),       # 512 rows
    (1, 1, 7, True, "expanding", False),
    (0, 0, 4, False, "contracting", True),          # no rows at all: every sample is a member
]


def _rollout_samples(ev, rng, n_random=3000):
    goal = ev.goal
    d = rng.normal(size=(n_random, 4))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    pts = [goal + d * np.exp(rng.uniform(np.log(0.01), np.log(5.0), size=(n_random, 1)))]
    # points on the t = 0 facets and a few ulps-to-1e-9 away from them
    rows = np.vstack((ev.A_con, ev.A_in))
    bs = np.concatenate((ev.b_con, ev.b_in))
    for a, b in zip(rows, bs):
        if not np.isfinite(b):
            continue
        for _ in range(3):
            e = rng.uniform(-0.3, 0.3, 4)
            e = e + a * (b - a @ e) / (a @ a)
            for scale in (0.0, 1e-15, -1e-15, 1e-9, -1e-9):
                pts.append((goal + e + scale * a / np.linalg.norm(a))[None, :])
    base = goal + rng.uniform(-0.1, 0.1, size=(len(SPECIALS) * 4, 4))
    for i, sp in enumerate(SPECIALS):
        for k in range(4):
            base[4 * i + k, k] = sp
    pts.append(base)
    p = np.vstack(pts)
    return [np.ascontiguousarray(c) for c in p.T]


def _check_rollout(torch, ev, k, every, cols, what):
    from oracle import c_oracle
    want_bits, want_first, want_cnt = c_oracle.rollout_bits(ev.A_k, ev.A_con, ev.b_con, ev.A_in, ev.b_in, ev.goal, k,
                                                            int(every), *cols)
    t = _dev(torch, cols)
    bits, cnt = ev.contains_bits(*t)
    np.testing.assert_array_equal(_bits_np(bits), want_bits, err_msg=f"{what}: screened path")
    assert int(cnt.item()) == want_cnt, what
    bits, cnt, first = ev.contains_bits(*t, want_first_violation=True)
    np.testing.assert_array_equal(_bits_np(bits), want_bits, err_msg=f"{what}: step-by-step path")
    np.testing.assert_array_equal(first.cpu().numpy(), want_first, err_msg=f"{what}: first violation")
    assert int(cnt.item()) == want_cnt, what
    return want_cnt


@pytest.mark.parametrize("s,rin,k,every,kind,nonzero_goal", ROLLOUT_FORMS,
                         ids=[f"s{f[0]}-rin{f[1]}-k{f[2]}-{'every' if f[3] else 'first'}-{f[4]}" for f in ROLLOUT_FORMS])
def test_synthetic_rollout(torch_cuda, s, rin, k, every, kind, nonzero_goal):
    from carmpc_b200.batch import RolloutEvaluator
    rng = np.random.default_rng(s * 7 + rin * 11 + k + 3 * every)
    Ak = synthetic_Ak(kind, rng)
    A_con, b_con = synthetic_rows(s, rng)
    A_in, b_in = synthetic_rows(rin, rng)
    goal = np.array([30.0, 1.5, 0.1, 2.0]) if nonzero_goal else np.zeros(4)
    ev = RolloutEvaluator(Ak, A_con, b_con, A_in, b_in, goal, k, input_every_step=every, reduce_screen=False)
    total = s * (k + 1) + rin * (k + 1 if every else 1)
    assert len(ev.expanded()) == (total if 0 < total <= 512 else 0)
    small = _rollout_samples(ev, rng)
    n_small = len(small[0])
    cnt = _check_rollout(torch_cuda, ev, k, every, small, "small")
    big = _tile(small, BULK_N, rng, special_idx=range(n_small))
    _check_rollout(torch_cuda, ev, k, every, big, f"{BULK_N} samples")
    assert 0 < cnt < n_small or total == 0 or kind == "expanding"
    if total == 0:
        assert cnt == n_small


def test_synthetic_rollout_reduced_screen(torch_cuda):
    """The default reduce_screen=True: the float32 screen keeps the irredundant expanded rows and the library widens its
    acceptance band by the redundancy certificates of the dropped ones; decisions are still the float64 chain's."""
    from carmpc_b200.batch import RolloutEvaluator
    rng = np.random.default_rng(5)
    Ak = synthetic_Ak("contracting", rng)
    A_con = np.vstack((np.eye(4), -np.eye(4))) * np.array([0.5, 2.0, 8.0, 1.0])
    b_con = np.array([10.0, 5.0, 4.0, 6.0, 12.0, 3.0, 2.0, 4.0])
    A_in, b_in = synthetic_rows(4, rng)
    goal = np.array([30.0, 1.5, 0.0, 2.0])
    k = 5
    ev = RolloutEvaluator(Ak, A_con, b_con, A_in, b_in, goal, k)
    assert ev.expanded_rows == 8 * (k + 1) + 4 >= 24
    assert 0 < ev.screen_rows < ev.expanded_rows
    small = _rollout_samples(ev, rng)
    cnt = _check_rollout(torch_cuda, ev, k, False, small, "reduced screen")
    assert 0 < cnt < len(small[0])
    big = _tile(small, BULK_N, rng, special_idx=range(len(small[0])))
    _check_rollout(torch_cuda, ev, k, False, big, f"reduced screen, {BULK_N} samples")
