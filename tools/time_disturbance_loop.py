"""Times config 4 (RoadEnv, N = 20, 10^5 runs x 200 steps against the nonlinear bicycle) in the disturbance-estimating
mode (``BatchQP.closed_loop_disturbance``: Bd = 1_4, Cd = 1_3, steady-state predictor gain, per-run process disturbance)
and in plain output feedback (``BatchQP.closed_loop``), alternating, in one process.  Two more arms of the disturbance
mode (every disturbance term zero; stable gain without a plant disturbance) show where a difference comes from.  Prints
one JSON object: ms per loop (every repetition, min and median), ADMM iterations per solved QP, failed runs, with the GPU
name and power limit read in the same run.

    python tools/time_disturbance_loop.py [--runs 100000] [--steps 200] [--reps 5] [--out result.json]
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
    from carmpc_b200.observer import augmented_observer_gain, observer_error_radius

    ctl = make_controller(make_env("RoadEnv"), 20, cls="MPCOutputFBWithDisturbance", init_state=[0, 0, 0, 0])
    Bd, Cd = np.ones(4), np.ones(3)
    L1, L2 = augmented_observer_gain(ctl.A, ctl.C, Bd, Cd, np.diag([1e-2] * 4 + [1e-3]), 1e-2 * np.eye(3))
    bq_dist = BatchQP.from_controller(ctl)
    ofb = make_controller(make_env("RoadEnv"), 20, cls="MPCOutputFB", init_state=[0, 0, 0, 0])
    bq_ofb = BatchQP.from_controller(ofb)
    R, T = args.runs, args.steps
    g = torch.Generator(device="cpu").manual_seed(0)
    lo = torch.tensor([0.0, -2.5, -0.2, 0.0], dtype=torch.float64)
    hi = torch.tensor([10.0, 2.5, 0.2, 3.0], dtype=torch.float64)
    x_init = (lo[:, None] + (hi - lo)[:, None] * torch.rand((4, R), generator=g, dtype=torch.float64)).cuda().contiguous()
    d_r = ((torch.rand(R, generator=g, dtype=torch.float64) - 0.5) * 0.02).cuda()
    x_ref = np.array([30.0, 1.5, 0.0, 0.0])

    arms = {
        "disturbance": lambda steps: bq_dist.closed_loop_disturbance(
            x_init, steps, ctl.A, ctl.B, ctl.C, Bd, Cd, L1, L2, x_ref=x_ref, Bd_plant=np.ones(4), d_plant=d_r),
        "output_feedback": lambda steps: bq_ofb.closed_loop(x_init, steps, ofb.A, ofb.B, x_ref=x_ref, C=_C_XYV,
                                                            L=_L_OBSERVER),
        # where the difference comes from: the disturbance mode with every disturbance term zero (the output-feedback
        # loop computed by the new entry point, on the handle with Gc != 0), and with the stable gain but d_r = 0
        "disturbance_zero_terms": lambda steps: bq_dist.closed_loop_disturbance(
            x_init, steps, ctl.A, ctl.B, ctl.C, np.zeros(4), np.zeros(3), _L_OBSERVER, np.zeros(3), x_ref=x_ref),
        "disturbance_without_plant_disturbance": lambda steps: bq_dist.closed_loop_disturbance(
            x_init, steps, ctl.A, ctl.B, ctl.C, Bd, Cd, L1, L2, x_ref=x_ref),
    }
    for f in arms.values():               # full-size warm-up: workspace allocation, module load, kernel attributes
        f(5)
    torch.cuda.synchronize()
    times = {k: [] for k in arms}
    last = {}
    for _ in range(args.reps):
        for name, f in arms.items():      # alternating, so that both arms see the same state of the machine
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            o = f(T)
            torch.cuda.synchronize()
            times[name].append((time.perf_counter() - t0) * 1e3)
            last[name] = o
    res = {"workload": f"config 4: RoadEnv N = 20, {R} runs x {T} steps vs the nonlinear bicycle",
           "gpu": gpu_info(),
           "disturbance_model": {"Bd": "1_4", "Cd": "1_3", "gain": "steady-state predictor (W = diag(1e-2 1_4, 1e-3), V = 1e-2 I)",
                                 "observer_error_radius": observer_error_radius(ctl.A, ctl.C, Bd, Cd, L1, L2),
                                 "plant": "Bd_p = 1_4, d_r ~ U(-0.01, 0.01) per run"}}
    for name in arms:
        o = last[name]
        fail = o["fail_step"]
        alive_steps = torch.where(fail < 0, torch.full_like(fail, T), fail + 1).sum().item()   # QPs solved per run
        res[name] = {"ms_per_loop": [round(t, 3) for t in times[name]], "ms_min": round(min(times[name]), 3),
                     "ms_median": round(float(np.median(times[name])), 3),
                     "admm_iters_per_qp": o["total_iters"] / max(1, alive_steps),
                     "failed_runs": int((fail >= 0).sum().item())}
    res["ratio_min_to_output_feedback"] = {k: res[k]["ms_min"] / res["output_feedback"]["ms_min"] for k in arms}
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
