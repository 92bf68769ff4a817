"""Times closed loops that stop at a goal (``carmpc_closed_loop`` with a goal), in one process, with the GPU name and
power limit read in the same run.  Prints one JSON object.

1. Config 4 (RoadEnv, N = 20, output feedback, 10^5 runs x 200 steps against the nonlinear bicycle, the initial states of
   bench_qp.py's config 4) without a goal and with ``montecarlo.goal_box(goal, 0.1)``, alternating, ``--reps`` loops
   each: ms per loop (every repetition, min, median), total ADMM iterations, runs reached, runs failed.
2. ``roa.closed_loop_map`` on the 10^6-state config-3 grid (RoadOneCarEnv, goal (29.9, 1.5, 0, 0), state feedback) with
   200 steps against the same map with 100 steps, alternating: whether the late steps, where most runs have stopped,
   cost anything.

    python tools/time_goal_loop.py [--runs 100000] [--steps 200] [--reps 5] [--map-reps 3] [--out result.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def gpu_info():
    torch = __import__("torch")
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip()
    except Exception as exc:               # the timing stands without it; say why it is missing
        info["power_limit_and_max_sm_clock"] = f"not read: {exc}"
    return info


def _timed(torch, f):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    o = f()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, o


def _summary(times):
    return {"ms_per_loop": [round(t, 3) for t in times], "ms_min": round(min(times), 3),
            "ms_median": round(float(np.median(times)), 3)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--runs", type=int, default=100_000)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--map-reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this tool measures the GPU loop and has no CPU fallback")
    from conftest import make_env, make_controller
    from carmpc_b200 import roa
    from carmpc_b200.batch import BatchQP
    from carmpc_b200.grids import config3_axes, grid_size
    from carmpc_b200.lib.mpc import _C_XYV, _L_OBSERVER
    from carmpc_b200.montecarlo import goal_box

    res = {"gpu": gpu_info()}
    # ---- 1. config 4 with and without the goal
    ctl = make_controller(make_env("RoadEnv"), 20, cls="MPCOutputFB", init_state=[0, 0, 0, 0])
    bq = BatchQP.from_controller(ctl)
    R, T = args.runs, args.steps
    g = torch.Generator(device="cpu").manual_seed(0)
    lo = torch.tensor([0.0, -2.5, -0.2, 0.0], dtype=torch.float64)
    hi = torch.tensor([10.0, 2.5, 0.2, 3.0], dtype=torch.float64)
    x_init = (lo[:, None] + (hi - lo)[:, None] * torch.rand((4, R), generator=g, dtype=torch.float64)).cuda().contiguous()
    x_ref = np.array([30.0, 1.5, 0.0, 0.0])
    A, B = np.ascontiguousarray(ctl.A, dtype=float), np.ascontiguousarray(ctl.B, dtype=float)
    C, L = np.ascontiguousarray(_C_XYV, dtype=float), np.ascontiguousarray(_L_OBSERVER, dtype=float)
    rows = goal_box(x_ref, 0.1)
    arms = {
        "no_goal": lambda steps: bq.closed_loop(x_init, steps, A, B, x_ref=x_ref, C=C, L=L),
        "goal_box": lambda steps: bq.closed_loop(x_init, steps, A, B, x_ref=x_ref, C=C, L=L, goal=rows),
    }
    for f in arms.values():               # full-size warm-up: workspace allocation, module load, kernel attributes
        f(5)
    times = {k: [] for k in arms}
    last = {}
    for _ in range(args.reps):
        for name, f in arms.items():      # alternating, so that every arm sees the same state of the machine
            t, last[name] = _timed(torch, lambda: f(T))
            times[name].append(t)
    res["config4"] = {"workload": f"RoadEnv N = 20 output feedback, {R} runs x {T} steps vs the nonlinear bicycle"}
    for name in arms:
        o = last[name]
        res["config4"][name] = {**_summary(times[name]), "total_admm_iters": o["total_iters"],
                                "failed_runs": int((o["fail_step"] >= 0).sum().item())}
        if "arrival_step" in o:
            res["config4"][name]["reached_runs"] = int((o["arrival_step"] >= 0).sum().item())
    res["config4"]["min_ratio_goal_to_no_goal"] = res["config4"]["goal_box"]["ms_min"] / res["config4"]["no_goal"]["ms_min"]

    # ---- 2. the closed-loop map of the config-3 grid, 200 against 100 steps
    env = make_env("RoadOneCarEnv", [29.9, 1.5, 0, 0])
    sf = make_controller(env, 20)
    bq3 = BatchQP.from_controller(sf)
    axes = config3_axes()
    roa.closed_loop_map(sf, axes, steps=2, batch_solver=bq3)
    lengths = (T, T // 2)
    mt = {k: [] for k in lengths}
    maps = {}
    for _ in range(args.map_reps):
        for k in lengths:
            t, maps[k] = _timed(torch, lambda: roa.closed_loop_map(sf, axes, steps=k, batch_solver=bq3))
            mt[k].append(t)
    res["config3_map"] = {"workload": f"closed_loop_map, RoadOneCarEnv N = 20 state feedback, {grid_size(axes)} grid states"}
    for k in lengths:
        counts = np.bincount(maps[k]["outcome"], minlength=3)
        res["config3_map"][f"{k}_steps"] = {**_summary(mt[k]), "reached": int(counts[0]), "qp_not_solved": int(counts[1]),
                                            "neither": int(counts[2])}
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
