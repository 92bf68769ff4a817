"""Times what derivatives cost: the certified cold solve of the config-3 grid (RoadOneCarEnv, 10^6 states) alone, and
followed by the sensitivity pass (``BatchQP.sensitivity``) at ``rows = 2`` and at ``rows = n``, at N = 20 and N = 80.
The three arms alternate in one process and are timed with CUDA events; the sensitivity pass is also timed alone on the
solve's outputs.  Prints one JSON object with every repetition, the flag counts, and the GPU name and power limit read in
the same run.

    python tools/time_sensitivity.py [--reps 5] [--out result.json]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from time_disturbance_loop import gpu_info  # noqa: E402


def event_ms(torch, fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from conftest import make_env, make_controller
    from carmpc_b200.batch import BatchQP
    from carmpc_b200.grids import config3_axes, materialise_grid
    x0 = torch.stack(materialise_grid(config3_axes(), device="cuda")).contiguous()
    res = {"gpu": gpu_info(), "states": int(x0.shape[1])}
    for N in (20, 80):
        c = make_controller(make_env("RoadOneCarEnv", [29.9, 1.5, 0, 0]), N)
        q = BatchQP.from_controller(c)
        solve = lambda: q.solve(x0, want_u_full=True, want_certificate=True)
        arms = {"solve": lambda: solve(),
                "solve_rows2": lambda: q.sensitivity(x0, solve(), rows=2),
                "solve_rowsn": lambda: q.sensitivity(x0, solve())}
        for fn in arms.values():                     # warm-up of every shape the timed window uses
            fn()
        times = {k: [] for k in arms}
        for _ in range(args.reps):                   # alternating
            for k, fn in arms.items():
                times[k].append(event_ms(torch, fn))
        out = solve()
        alone = {"rows2": [], "rowsn": []}
        for _ in range(args.reps):
            alone["rows2"].append(event_ms(torch, lambda: q.sensitivity(x0, out, rows=2)))
            alone["rowsn"].append(event_ms(torch, lambda: q.sensitivity(x0, out)))
        flags = q.sensitivity(x0, out, rows=2)["flags"]
        res[f"N{N}"] = {
            "n": q.n, "m": q.m,
            **{f"{k}_ms": v for k, v in times.items()}, **{f"{k}_ms_min": min(v) for k, v in times.items()},
            **{f"sensitivity_{k}_alone_ms": v for k, v in alone.items()},
            **{f"sensitivity_{k}_alone_ms_min": min(v) for k, v in alone.items()},
            "solved": int((out["status"] == 0).sum()),
            "flags": {name: int(((flags & bit) != 0).sum()) for name, bit in
                      (("derivative", 1), ("weak", 2), ("dependent", 4), ("too_many_rows", 8))},
        }
        del out, flags
        torch.cuda.empty_cache()
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
