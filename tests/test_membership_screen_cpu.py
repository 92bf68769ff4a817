"""The adversarial terminal-set cases of tests/test_membership_envelope_gpu.py, checked exactly (no GPU needed).

Each case puts one row that the float32 screen of mode 1 cannot evaluate faithfully (a product or ``b`` beyond the
float32 range, a coefficient beyond it, a coordinate below its normal range) into a polytope of benign rows that the
point satisfies.  The GPU tests compare the kernels with the C oracle's float64 fma chain; here that oracle is compared
with an exact rational evaluation of ``a . p <= b`` (``fractions.Fraction``), row by row, and every row's exact margin is
checked to be non-zero, so the expected answers do not hinge on any rounding.
"""
from fractions import Fraction

import numpy as np
import pytest

INF = float("inf")

# (name, adversarial row [a | b], point (x, y, psi, v), scale of the benign rows' bounds, exact answer)
# The benign bounds are chosen per case so that the float32 screen of the unguarded kernel would commit to an answer:
# huge where it would wrongly say "inside" (the benign margins must clear its error bound), small where a wide bound
# would otherwise hide the wrong "outside".
CASES = [
    ("product_overflows_to_plus_inf", (-2.0 ** 100, 2.0 ** 100, 0.0, 0.0, -1.0), (2.0 ** 30, 2.0 ** 30, 0.0, 0.0), 1e35, False),
    ("product_overflows_to_minus_inf", (2.0 ** 100, -2.0 ** 100, 0.0, 0.0, 1.0), (2.0 ** 30, 2.0 ** 30, 0.0, 0.0), 1.0, True),
    ("bound_beyond_float32", (100.0, 0.0, 0.0, 0.0, -1e39), (-1e38, 0.0, 0.0, 0.0), 1.0, True),
    ("coefficient_beyond_float32", (1e39, 1.0, 0.0, 0.0, 0.0), (0.0, 1.0, 0.0, 0.0), 1e34, False),
    ("subnormal_float32_coordinate", (1e38, 0.0, 0.0, 0.0, 1.3e-7), (1.2e-45, 0.0, 0.0, 0.0), 1e-3, True),
    ("coordinate_below_float32", (1e20, 0.0, 0.0, 0.0, 5e-27), (1e-46, 0.0, 0.0, 0.0), 1e-22, False),
]
CASE_IDS = [c[0] for c in CASES]


def polytope(row, beta):
    """The adversarial row among benign ones: |psi| <= beta, |v| <= beta and a row without a bound."""
    benign = [(0.0, 0.0, 1.0, 0.0, beta), (0.0, 0.0, -1.0, 0.0, beta), (0.0, 0.0, 0.0, 1.0, beta),
              (0.0, 0.0, 0.0, -1.0, beta), (1.0, -1.0, 0.5, 2.0, INF)]
    return np.array(benign[:2] + [row] + benign[2:], dtype=np.float64)


# The screened rollout form: A_k = 0.5 I, the state row (2^100, -2^100, 0, 0) <= 1 among benign state rows, goal 0.
# Along the rollout e_t = 0.5^t p, so the row's value is exactly 0 at every step: a member.  Its float32 product at t = 0
# overflows to -inf, and the unguarded screen would call the point surely outside.
ROLLOUT = dict(
    A_k=0.5 * np.eye(4),
    A_con=np.array([[2.0 ** 100, -2.0 ** 100, 0.0, 0.0], [0.0, 0.0, 1.0, 0.0], [0.0, 0.0, 0.0, -1.0]]),
    b_con=np.array([1.0, 1.0, 1.0]),
    A_in=np.zeros((0, 4)),
    b_in=np.zeros(0),
    goal=np.zeros(4),
    k_steps=3,
)
ROLLOUT_POINT = (2.0 ** 30, 2.0 ** 30, 0.0, 0.0)


def _exact_margins(Ab, point):
    """b - a . p for every row, exactly; None for rows without a bound."""
    p = [Fraction(c) for c in point]
    out = []
    for row in Ab:
        if np.isinf(row[4]):
            assert row[4] > 0
            out.append(None)
            continue
        out.append(Fraction(float(row[4])) - sum(Fraction(float(a)) * c for a, c in zip(row[:4], p)))
    return out


def _oracle_member(Ab, point):
    from oracle import c_oracle
    bits, cnt = c_oracle.membership_bits(Ab, *[np.array([c]) for c in point])
    assert cnt in (0, 1)
    return bool(c_oracle.unpack_bits(bits, 1)[0])


@pytest.mark.parametrize("name,row,point,beta,expect", CASES, ids=CASE_IDS)
def test_adversarial_case_is_decided_by_exact_arithmetic(name, row, point, beta, expect):
    Ab = polytope(row, beta)
    margins = _exact_margins(Ab, point)
    # no row is a tie: the exact answer does not depend on how a correct evaluation rounds
    assert all(m is None or m != 0 for m in margins)
    exact = all(m is None or m > 0 for m in margins)
    assert exact == expect
    # the benign rows hold, so the adversarial row alone decides
    assert all(m is None or m > 0 for i, m in enumerate(margins) if i != 2)
    # the float64 chain of the oracle gets it right, row by row and for the whole polytope
    for r, m in zip(Ab, margins):
        assert _oracle_member(r[None, :], point) == (m is None or m > 0)
    assert _oracle_member(Ab, point) == expect


def test_adversarial_rows_are_beyond_what_the_float32_bound_assumed():
    """Each case really is outside the float32 evaluation's normal range, which is what makes it adversarial."""
    big, tiny = float(np.finfo(np.float32).max), float(np.finfo(np.float32).tiny)
    for name, row, point, beta, _ in CASES:
        a, b = np.array(row[:4]), row[4]
        p = np.array(point)
        products = np.abs(a) * np.abs(p)
        beyond = (products.max() > big or abs(b) > big or np.abs(a).max() > big
                  or np.any((p != 0) & (np.abs(p) < tiny)))
        assert beyond, name


def test_rollout_case_is_a_member_exactly():
    from oracle import c_oracle
    R = ROLLOUT
    Ak = [[Fraction(float(v)) for v in row] for row in R["A_k"]]
    e = [Fraction(c) - Fraction(float(g)) for c, g in zip(ROLLOUT_POINT, R["goal"])]
    member = True
    for t in range(R["k_steps"] + 1):
        for a, b in zip(R["A_con"], R["b_con"]):
            margin = Fraction(float(b)) - sum(Fraction(float(ai)) * ei for ai, ei in zip(a, e))
            assert margin != 0
            member &= margin > 0
        e = [sum(Ak[i][j] * e[j] for j in range(4)) for i in range(4)]
    assert member
    bits, first, cnt = c_oracle.rollout_bits(R["A_k"], R["A_con"], R["b_con"], R["A_in"], R["b_in"], R["goal"],
                                             R["k_steps"], 0, *[np.array([c]) for c in ROLLOUT_POINT])
    assert cnt == 1 and int(first[0]) == -1
    # the float32 product of the adversarial row at t = 0 overflows
    assert abs(R["A_con"][0, 0] * ROLLOUT_POINT[0]) > float(np.finfo(np.float32).max)
