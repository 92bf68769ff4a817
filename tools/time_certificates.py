"""Times what certificates cost: the config-3 cold solve (RoadOneCarEnv, N = 20, the 10^6-state grid) without them, the
same solve with ``u_full`` with and without ``want_certificate``, alternating in one process, and the checker kernel
(``QPChecker``) on all 10^6 states at N = 20 and N = 80.  Prints one JSON object with every repetition and the GPU name
and power limit read in the same run.

``--lib PATH`` times another build of ``libcarmpc_b200.so`` (for example the parent commit's) for the plain solve only,
so that two builds can be compared in alternating processes.

    python tools/time_certificates.py [--reps 5] [--lib PATH] [--plain-only] [--out result.json]
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from time_disturbance_loop import gpu_info  # noqa: E402


def timed(fn, reps):
    torch = __import__("torch")
    fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        out.append(1e3 * (time.perf_counter() - t))
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--lib", default=None)
    ap.add_argument("--plain-only", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.lib:
        from carmpc_b200 import build
        import ctypes
        from carmpc_b200 import _capi
        build.LIB_PATH = os.path.abspath(args.lib)
        build.is_stale = lambda: False
        other = ctypes.CDLL(build.LIB_PATH)        # an older build lacks the newer entry points: type what it has
        _capi.SIGNATURES = {k: v for k, v in _capi.SIGNATURES.items() if hasattr(other, k)}
    import numpy as np
    import torch
    from conftest import make_env, make_controller
    from carmpc_b200.batch import BatchQP
    from carmpc_b200.grids import config3_axes, materialise_grid
    x0 = torch.stack(materialise_grid(config3_axes(), device="cuda")).contiguous()
    res = {"gpu": gpu_info(), "states": int(x0.shape[1]), "lib": args.lib or "tree"}
    bq = {}
    for N in (20, 80):
        c = make_controller(make_env("RoadOneCarEnv", [29.9, 1.5, 0, 0]), N)
        bq[N] = (c, BatchQP.from_controller(c))
    q20 = bq[20][1]
    res["cold_ms"] = timed(lambda: q20.solve(x0), args.reps)
    if not args.plain_only:
        plain, cert = [], []
        for _ in range(args.reps):                # alternating
            plain += timed(lambda: q20.solve(x0, want_u_full=True), 1)
            cert += timed(lambda: q20.solve(x0, want_u_full=True, want_certificate=True), 1)
        res["u_full_ms"], res["u_full_and_certificate_ms"] = plain, cert
        from carmpc_b200.certificate import to_one_sided
        for N, (c, q) in bq.items():
            out = q.solve(x0, want_u_full=True, want_certificate=True)
            one = to_one_sided(q.pq, out["certificate"])
            from test_qp_certificate_gpu import Reference
            chk = Reference("RoadOneCarEnv", N).checker()
            g = np.array(c.goal, dtype=float)
            res[f"certificate_width_N{N}"] = int(out["certificate"].shape[1])
            res[f"certificate_gb_N{N}"] = out["certificate"].numel() * 8 / 1e9
            res[f"to_one_sided_ms_N{N}"] = timed(lambda: to_one_sided(q.pq, out["certificate"]), args.reps)
            res[f"checker_ms_N{N}"] = timed(lambda: chk.check(x0, g, out["status"], out["u_full"], one), args.reps)
            del out, one
            torch.cuda.empty_cache()
    for k, v in list(res.items()):
        if k.endswith("_ms") or "_ms_" in k:
            res[k + "_min"] = min(v)
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
