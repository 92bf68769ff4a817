#!/usr/bin/env python
"""The region of attraction by closed-loop convergence (the paper's criterion, its Fig. 3 slice): from every point of an
(x, v) grid with y = psi = 0 the nonlinear bicycle runs under the state-feedback MPC until it reaches the goal box
(|s - goal| <= 0.1, the reference's test), its QP is not solved, or the steps end (``roa.closed_loop_map``, one batched
closed loop on the GPU).  Printed beside it: the one-step feasibility map of the same grid (``roa.feasibility_map``),
the cross table of the two, and the time of each.

    python examples/closed_loop_roa.py [--points 100 60] [--steps 200] [--env RoadOneCarEnv]
"""
import argparse
import time

import numpy as np

import _common
from carmpc_b200 import roa
from carmpc_b200.batch import BatchQP
from carmpc_b200.lib.configuration import DT_CONTROL, LINEARIZE_STATE, LINEARIZE_INPUT, N
from carmpc_b200.lib.mpc import MPCStateFB

OUTCOMES = ("reached", "QP not solved", "neither")


def main(argv=None):
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--env", default="RoadOneCarEnv")
    ap.add_argument("--points", type=int, nargs=2, default=[100, 60], metavar=("NX", "NV"))
    ap.add_argument("--steps", type=int, default=200)
    args = ap.parse_args(argv)
    env = _common.make_env(args.env)
    controller = MPCStateFB(dt=DT_CONTROL, N=N, lin_state=LINEARIZE_STATE, lin_input=LINEARIZE_INPUT, env=env)
    bq = BatchQP.from_controller(controller)
    nx, nv = args.points
    axes = [np.linspace(5.0, 30.0, nx), np.array([0.0]), np.array([0.0]), np.linspace(-1.0, 5.0, nv)]

    roa.closed_loop_map(controller, axes, steps=2, batch_solver=bq)          # warm-up: module load, workspace
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    m = roa.closed_loop_map(controller, axes, steps=args.steps, batch_solver=bq)
    t_loop = time.perf_counter() - t0
    t0 = time.perf_counter()
    feasible = roa.feasibility_map(controller, axes, batch_solver=bq, undecided="outside")
    t_map = time.perf_counter() - t0

    counts = np.bincount(m["outcome"], minlength=3)
    n = len(feasible)
    print(f"{args.env}, goal {np.round(controller.goal, 3)}, (x, v) grid {nx} x {nv} with y = psi = 0, {args.steps} steps")
    print(f"closed loop ({t_loop:.3f} s): " + ", ".join(f"{c} {name}" for c, name in zip(counts, OUTCOMES)))
    print(f"one-step QP feasibility ({t_map:.3f} s): {int(feasible.sum())} of {n} feasible")
    print(f"{'':>16s} {'feasible':>10s} {'infeasible':>10s}")
    for k, name in enumerate(OUTCOMES):
        row = m["outcome"] == k
        print(f"{name:>16s} {int((row & feasible).sum()):10d} {int((row & ~feasible).sum()):10d}")
    return {**m, "feasible": feasible}


if __name__ == "__main__":
    main()
