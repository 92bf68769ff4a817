"""Where the config-2 scan spends its time: the whole grid, its x < 30 half and its x >= 30 half timed on their own, and
10^8 uniform random samples (the distribution of the GPU tests, whose cost does not depend on the index), for one or
more builds of the library in one process, alternating (back-to-back launches, CUDA events).

    python tools/scan_halves.py [--rounds 3] [--steps 20] [--rollout] NAME=path/to/libcarmpc_b200.so ...

Without a library argument it times the library of this tree.  Every build must give the bits of the first one.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from carmpc_b200 import _capi, build  # noqa: E402
from carmpc_b200.batch import RolloutEvaluator, TerminalSetEvaluator  # noqa: E402
from carmpc_b200.grids import config2_axes, materialise_grid  # noqa: E402
from carmpc_b200.lib.environments import RoadMultipleCarsEnv  # noqa: E402

TERMINAL_SET = os.path.join(ROOT, "terminal_sets", "RoadMultipleCarsEnv_30_1.5_0_0.npy")


def load(path):
    """A fresh ctypes handle on the library at `path` (evaluators keep the library they were created with)."""
    build.LIB_PATH = os.path.abspath(path)
    _capi._lib = None
    return _capi.load(rebuild_if_stale=False)


def uniform_samples(n, seed=9):
    g = torch.Generator(device="cuda").manual_seed(seed)
    lo = torch.tensor([5.0, -3.2, -0.42, -1.2], dtype=torch.float64, device="cuda")
    hi = torch.tensor([55.0, 3.2, 0.42, 5.2], dtype=torch.float64, device="cuda")
    out = []
    for k in range(4):
        u = torch.rand(n, generator=g, dtype=torch.float64, device="cuda")
        out.append((lo[k] + (hi[k] - lo[k]) * u).contiguous())
    return out


def timed_ms(ev, cols, bits, count, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev.contains_bits(*cols, bits=bits, count=count)
    e0.record()
    for _ in range(steps):
        ev.contains_bits(*cols, bits=bits, count=count)
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("libs", nargs="*", help="NAME=path of a libcarmpc_b200.so")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rollout", action="store_true", help="also time the rollout form (k* = 16) on the whole grid")
    ap.add_argument("--staging", default="", help="threads,ring_slots,tiles_per_slot of the scan kernel (default: the library's)")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    libs = [a.split("=", 1) for a in args.libs] or [["this", build.LIB_PATH]]
    Ab = np.load(TERMINAL_SET)
    grid = materialise_grid(config2_axes(), device="cuda")
    n = grid[0].numel()
    half = n // 2 // 1024 * 1024                                  # x < 30 is the first half of the indices
    parts = {"all": (0, n), "x<30": (0, half), "x>=30": (half, n)}
    rnd = uniform_samples(n)
    bits = torch.empty((n + 31) // 32, dtype=torch.int32, device="cuda")
    count = torch.zeros(1, dtype=torch.int64, device="cuda")
    evs, ref = {}, {}
    for name, path in libs:
        load(path)
        ev, evr = TerminalSetEvaluator(Ab), TerminalSetEvaluator(Ab)
        if args.staging:
            for e in (ev, evr):
                e.set_staging(*[int(k) for k in args.staging.split(",")])
        ev.contains_bits(*grid, bits=bits, count=count)           # row order tuned on the whole grid, as in bench.py
        got = {"grid": (bits.clone(), int(count.item()))}
        evr.contains_bits(*rnd, bits=bits, count=count)
        got["uniform"] = (bits.clone(), int(count.item()))
        rv = None
        if args.rollout:
            rv = RolloutEvaluator.from_env(RoadMultipleCarsEnv(), 16)
            if args.staging:
                rv.set_staging(*[int(k) for k in args.staging.split(",")])
            rv.contains_bits(*grid, bits=bits, count=count)
            got["rollout"] = (bits.clone(), int(count.item()))
        for k, (b, c) in got.items():
            if k in ref:
                assert c == ref[k][1] and torch.equal(b, ref[k][0]), f"{name}: {k} bits differ from {libs[0][0]}"
            else:
                ref[k] = (b, c)
        evs[name] = (ev, evr, rv)
    times = {name: {} for name, _ in libs}
    for _ in range(args.rounds):
        for name, _ in libs:
            ev, evr, rv = evs[name]
            for part, (lo, hi) in parts.items():
                times[name].setdefault(part, []).append(timed_ms(ev, [t[lo:hi] for t in grid], bits, count, args.steps))
            times[name].setdefault("uniform", []).append(timed_ms(evr, rnd, bits, count, args.steps))
            if rv is not None:
                times[name].setdefault("rollout", []).append(timed_ms(rv, grid, bits, count, args.steps))
    props = torch.cuda.get_device_properties(0)
    print(f"# {props.name}; staging {args.staging or 'default'}; members: grid {ref['grid'][1]}, uniform {ref['uniform'][1]}; ms per launch, "
          f"mean of {args.rounds} alternating rounds of {args.steps} launches [min - max]", flush=True)
    for name, _ in libs:
        row = " | ".join(f"{k} {np.mean(v):.4f} [{min(v):.4f} - {max(v):.4f}]" for k, v in times[name].items())
        print(f"{name:>8}: {row}", flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump({"device": props.name, "times_ms": times}, f, indent=1)


if __name__ == "__main__":
    main()
