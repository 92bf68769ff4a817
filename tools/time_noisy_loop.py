"""Times config 4 (RoadEnv, N = 20, output feedback, 10^5 runs x 200 steps against the nonlinear bicycle) with noise and
monitor (``carmpc_closed_loop_stochastic``).  Four arms, alternating, in one process: the existing ``closed_loop``; the new
entry point with everything off; the monitor alone (the controller's plant rows); noise and monitor.  Prints one JSON
object: ms per loop (every repetition, min and median), ADMM iterations per solved QP, failed runs, runs with a
violation, with the GPU name and power limit read in the same run.

    python tools/time_noisy_loop.py [--runs 100000] [--steps 200] [--reps 5] [--out result.json]
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

PROCESS_STD = [0.02, 0.02, 0.004, 0.02]       # x, y, psi, v per step
MEASUREMENT_STD = [0.03, 0.03, 0.03]          # x, y, v


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


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--runs", type=int, default=100_000)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this tool measures the GPU loop and has no CPU fallback")
    from conftest import make_env, make_controller
    from carmpc_b200.batch import BatchQP
    from carmpc_b200.lib.mpc import _C_XYV, _L_OBSERVER
    from carmpc_b200.montecarlo import LoopNoise, plant_rows

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
    rows = plant_rows(ctl)
    noise = LoopNoise(PROCESS_STD, MEASUREMENT_STD, seed=0)

    def everything_off(steps):
        out = {"final": torch.empty((4, R), dtype=torch.float64, device="cuda"),
               "fail_step": torch.empty(R, dtype=torch.int32, device="cuda")}
        bq._closed_loop_stochastic(1, x_init, steps, A, B, C, L, None, x_ref, 0.2, 3.5, 1, None, None, None, out, None,
                                   None, None)
        return out

    arms = {
        "closed_loop": lambda steps: bq.closed_loop(x_init, steps, A, B, x_ref=x_ref, C=C, L=L),
        "stochastic_off": everything_off,
        "monitor_only": lambda steps: bq.closed_loop(x_init, steps, A, B, x_ref=x_ref, C=C, L=L, monitor=rows),
        "noise_and_monitor": lambda steps: bq.closed_loop(x_init, steps, A, B, x_ref=x_ref, C=C, L=L, monitor=rows,
                                                          noise=noise),
    }
    for f in arms.values():               # full-size warm-up: workspace allocation, module load, kernel attributes
        f(5)
    torch.cuda.synchronize()
    times = {k: [] for k in arms}
    last = {}
    for _ in range(args.reps):
        for name, f in arms.items():      # alternating, so that every arm sees the same state of the machine
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            o = f(T)
            torch.cuda.synchronize()
            times[name].append((time.perf_counter() - t0) * 1e3)
            last[name] = o
    res = {"workload": f"config 4: RoadEnv N = 20 output feedback, {R} runs x {T} steps vs the nonlinear bicycle",
           "gpu": gpu_info(),
           "noise": {"process_std": PROCESS_STD, "measurement_std": MEASUREMENT_STD, "seed": 0},
           "monitor_rows": len(rows)}
    for name in arms:
        o = last[name]
        fail = o["fail_step"]
        alive_steps = torch.where(fail < 0, torch.full_like(fail, T), fail + 1).sum().item()   # QPs solved per run
        res[name] = {"ms_per_loop": [round(t, 3) for t in times[name]], "ms_min": round(min(times[name]), 3),
                     "ms_median": round(float(np.median(times[name])), 3),
                     "admm_iters_per_qp": o["total_iters"] / max(1, alive_steps),
                     "failed_runs": int((fail >= 0).sum().item())}
        if "violation_step" in o:
            res[name]["runs_with_a_violation"] = int((o["violation_step"] >= 0).sum().item())
    res["ratio_min_to_closed_loop"] = {k: res[k]["ms_min"] / res["closed_loop"]["ms_min"] for k in arms}
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
