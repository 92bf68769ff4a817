"""Option validation of ``carmpc_qp_create``, checked on the CPU (no device: the handle is created host-only).

The solver options reach the kernels unchanged, so a bad combination has to be refused at creation with a message that
names the rule, and the starved / loose / shy / eager configurations of tests/test_qp_proof_paths_gpu.py have to be
accepted as they are.
"""
import numpy as np
import pytest

from conftest import make_env, make_controller

GOAL = [29.9, 1.5, 0, 0]

# the forcing configurations of the proof-path tests (tests/test_qp_proof_paths_gpu.py)
FORCING = {"starved": dict(max_iter=10, check_every=10), "loose": dict(eps_abs=0.3, eps_rel=0.3),
           "shy": dict(eps_prim_inf=2.0), "eager": dict(eps_prim_inf=-0.5)}


@pytest.fixture(scope="module")
def pq20():
    from carmpc_b200.condensed import build_parametric_qp
    return build_parametric_qp(make_controller(make_env("RoadOneCarEnv", GOAL), 20))


@pytest.mark.parametrize("opts,match", [
    (dict(check_every=10, max_iter=9), "max_iter >= check_every"),
    (dict(check_every=10, max_iter=0), "max_iter >= check_every"),
    (dict(check_every=10, max_iter=-5), "max_iter >= check_every"),
    (dict(max_iter=9), "max_iter >= check_every"),          # automatic cadence at 40 variables: 10
    (dict(alpha=0.0), "alpha"),
    (dict(alpha=2.0), "alpha"),
    (dict(alpha=-1.0), "alpha"),
    (dict(scaling_iters=-1), "scaling_iters"),
    (dict(scaling_iters=101), "scaling_iters"),
])
def test_bad_options_are_refused_with_the_rule(pq20, opts, match):
    from carmpc_b200.batch import BatchQP
    from carmpc_b200._capi import CarmpcError
    with pytest.raises(CarmpcError, match=match):
        BatchQP(pq20, **opts)


def test_unknown_option_names_are_refused(pq20):
    from carmpc_b200.batch import BatchQP
    with pytest.raises(TypeError, match="max_iters"):
        BatchQP(pq20, max_iters=10)


@pytest.mark.parametrize("name", sorted(FORCING))
def test_forcing_configurations_are_accepted(pq20, name):
    from carmpc_b200.batch import BatchQP
    bq = BatchQP(pq20, **FORCING[name])
    for k, v in FORCING[name].items():
        assert getattr(bq.opts, k) == v
    # the handle is usable for inspection: the float64 scaling does not depend on these options
    ref = BatchQP(pq20)
    np.testing.assert_array_equal(bq.setup(0), ref.setup(0))
    np.testing.assert_array_equal(bq.setup(4), ref.setup(4))


def test_automatic_cadence_depends_on_the_problem_size():
    """check_every <= 0 picks 14 for n <= 20 variables, else 10: max_iter = 10 is refused at horizon 10 (20 variables)
    and accepted at horizon 20 (40 variables), and an explicit check_every = 10 makes it valid at horizon 10 too."""
    from carmpc_b200.batch import BatchQP
    from carmpc_b200._capi import CarmpcError
    from carmpc_b200.condensed import build_parametric_qp
    pq10 = build_parametric_qp(make_controller(make_env("RoadOneCarEnv", GOAL), 10))
    pq20 = build_parametric_qp(make_controller(make_env("RoadOneCarEnv", GOAL), 20))
    assert pq10.n == 20 and pq20.n == 40
    with pytest.raises(CarmpcError, match="max_iter >= check_every"):
        BatchQP(pq10, max_iter=10)
    with pytest.raises(CarmpcError, match="max_iter >= check_every"):
        BatchQP(pq10, max_iter=13, check_every=-3)
    BatchQP(pq10, max_iter=14)
    BatchQP(pq10, max_iter=10, check_every=10)
    BatchQP(pq20, max_iter=10)
    BatchQP(pq20, max_iter=1, check_every=1)
