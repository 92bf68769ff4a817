"""QP half of bench.py: BASELINE configs 3 (10^6 horizon-20 QPs), 5 (horizon sweep) and 4 (Monte-Carlo closed loop).

Imported by bench.py; returns a dict that goes under ``"qp"`` in the JSON line.  The CPU leg (numpy float64
OSQP-style ADMM of oracle/, the restatement of what cvxpy's default solver does for lib/mpc.py:334-335) is the only
place oracle/ is executed, as the baseline being timed.
"""
from __future__ import annotations

import io
import contextlib
import os
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))


def _controller(env_name, goal, N, cls="MPCStateFB", **kw):
    from carmpc_b200.lib import environments, mpc, terminal_set as ts
    from carmpc_b200.lib.configuration import DT_CONTROL, LINEARIZE_STATE, LINEARIZE_INPUT
    env = getattr(environments, env_name)()
    if goal is not None:
        env.set_goal(goal)
    ts.TERMINAL_SET_DIR = os.path.join(ROOT, "terminal_sets")
    with contextlib.redirect_stdout(io.StringIO()):
        return getattr(mpc, cls)(dt=DT_CONTROL, N=N, lin_state=LINEARIZE_STATE, lin_input=LINEARIZE_INPUT, env=env, **kw)


def cpu_qp_rate(n_states: int = 1500, seed: int = 0):
    """QPs/s of the numpy float64 ADMM oracle at cvxpy's default OSQP tolerances (eps 1e-5), config-3 states."""
    from oracle import carmpc_oracle as orc
    from carmpc_b200.grids import config3_axes, grid_size
    Ab = np.load(os.path.join(ROOT, "terminal_sets", "RoadOneCarEnv_29.9_1.5_0_0.npy"))
    oq = orc.CondensedQP("RoadOneCarEnv", 20, Ab)
    axes = config3_axes()
    n = grid_size(axes)
    idx = np.random.default_rng(seed).choice(n, n_states, replace=False)
    dims = [len(a) for a in axes]
    cols, stride = [], n
    for a, d in zip(axes, dims):
        stride //= d
        cols.append(a[(idx // stride) % d])
    x0 = np.stack(cols, axis=1)
    t0 = time.perf_counter()
    u, y, st, iters = orc.qp_solve_admm(oq, x0, np.array([29.9, 1.5, 0, 0]), eps=1e-5, eps_inf=1e-4, max_iter=4000,
                                        return_iters=True)
    dt = time.perf_counter() - t0
    return {"value": n_states / dt, "unit": "QPs/s", "cores": int(os.environ.get("OMP_NUM_THREADS", os.cpu_count() or 1)),
            "kind": "port", "sample": f"{n_states} random states of the config-3 grid, numpy float64 ADMM (OSQP iteration, "
            f"eps 1e-5, rho 30 unscaled), {dt:.1f} s", "mean_iters": float(iters.mean()),
            "feasible_frac": float((st == 0).mean())}


_SAMPLE_DIM = {"u0": 1, "objective": 0, "status": 0, "iters": 0}


def _time_solves(bq, x0, steps, warmup, torch, gather=None, barrier=None):
    """Average ms per step; a step is one batched solve of this rank's states and, when the states are sharded over
    several GPUs (``gather`` = total number of states), the all-gather of the per-sample results over NCCL."""
    from carmpc_b200.sharding import gather_samples

    def one():
        out = bq.solve(x0)
        it, la = bq.last_stats()
        full = gather_samples({k: out[k] for k in _SAMPLE_DIM}, gather, _SAMPLE_DIM) if gather else None
        return out, it, la, full

    for _ in range(warmup):
        out, _, _, full = one()
    if barrier is not None:
        barrier()
    torch.cuda.synchronize()
    t_iters, launches = 0, 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        out, it, la, full = one()
        t_iters += it
        launches += la
    e1.record()
    e1.synchronize()
    if full is not None:
        assert full["status"].numel() == gather and full["u0"].shape == (2, gather)
    return e0.elapsed_time(e1) / steps, t_iters / steps, launches, out


def run_qp_bench(args, rank, world, dev, barrier):
    import torch
    import torch.distributed as dist
    from carmpc_b200.batch import BatchQP, measure_peak
    from carmpc_b200.grids import config3_axes, materialise_grid

    from carmpc_b200.grids import grid_size, shard_range
    axes = config3_axes()
    B_all = min(args.qp_states, grid_size(axes))
    # strong scaling: the ONE 10^6-state grid is sharded over the ranks; per-sample results are all-gathered over NCCL
    lo, hi = shard_range(B_all, rank, world)
    x0 = torch.stack(materialise_grid(axes, device=dev, start=lo, stop=hi)).contiguous()          # (4, 10^6 / world)
    B = x0.shape[1]
    full_grid = B_all == grid_size(axes)
    gather = B_all if world > 1 else None
    steps, warmup = args.qp_steps, 3

    def max_over_ranks(v):
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(v):
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t)
        return float(t.item())

    c20 = _controller("RoadOneCarEnv", [29.9, 1.5, 0, 0], 20)
    bq = BatchQP.from_controller(c20)
    tiling = bq.tiling()
    barrier()
    ms, iters, launches, out = _time_solves(bq, x0, steps, warmup, torch, gather, barrier)
    ms_max = max_over_ranks(ms)
    ms_solve_only = max_over_ranks(_time_solves(bq, x0, steps, 0, torch)[0]) if world > 1 else ms_max
    status = out["status"]
    res = {
        "metric": "horizon-20 QPs/s", "value": B_all / (ms_max * 1e-3), "unit": "QPs/s", "ms_per_step": ms_max,
        "steps": steps, "warmup": warmup, "scaling": "strong" if world > 1 else "weak",
        "config": {"workload": "config 3: RoadOneCarEnv goal (29.9, 1.5, 0, 0), N = 20, 100x100x10x10 grid of initial "
                               "states, one condensed QP each, cold start; with N GPUs the grid is sharded and the per-sample "
                               "results (u0, objective, status, iterations) are all-gathered over NCCL inside the step",
                   "states_total": B_all, "states_per_gpu": B,
                   "tolerance": "ADMM float32 to 1e-3 (active set) + float64 polish with KKT check"},
        "solve_only_ms": ms_solve_only, "gather_ms": ms_max - ms_solve_only,
        "feasible_frac": float((status == 0).float().mean().item()),
        "max_iter_count": int((status == 2).sum().item()),
        "mean_admm_iters": iters / B, "gpu_launches": launches, "tiling": tiling, "polish": bq.polish_stats(),
    }
    if rank == 0:
        fp32_peak = measure_peak("fp32")
        flops_exec = iters * tiling["flop_per_iter"]
        flops_dense = iters * tiling["flop_per_iter_dense"]
        ms_k = ms_solve_only                              # this rank's solve without the gather (max over ranks), per GPU
        res["roofline"] = {"bound": "fp32-ffma", "achieved": flops_exec / (ms_k * 1e-3) / 1e12, "peak": fp32_peak,
                           "unit": "TFLOP/s", "frac": flops_exec / (ms_k * 1e-3) / 1e12 / fp32_peak,
                           "peak_source": "measured live (carmpc_measure_peak fp32 FFMA)",
                           "flop_per_iter_executed": tiling["flop_per_iter"],
                           "flop_per_iter_dense": tiling["flop_per_iter_dense"],
                           "dense_equivalent_tflops": flops_dense / (ms_k * 1e-3) / 1e12,
                           "note": "whole solve (ADMM + polish) time; executed flops exclude structural zeros"}
    # end to end through the host entry point (numpy AoS states in, numpy results out)
    xh_t = torch.empty((B, 4), dtype=torch.float64, pin_memory=True)            # states in pinned host memory, AoS
    xh_t.copy_(x0.t())
    xh = xh_t.numpy()
    bq.solve_host(xh, pinned=True)
    torch.cuda.synchronize()
    e2e_steps = 3
    dts = []
    for _ in range(e2e_steps):
        t0 = time.perf_counter()
        r = bq.solve_host(xh, pinned=True)
        dts.append(time.perf_counter() - t0)
    dt = float(np.median(dts))
    tt = torch.tensor([dt], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    res["e2e"] = {"value": B_all / float(tt.item()), "unit": "QPs/s", "h2d_bytes_per_step": B * 32,
                  "d2h_bytes_per_step": B * (16 + 8 + 4 + 4), "call": "carmpc_qp_solve_host (pinned host buffers)"}
    if rank == 0 and world == 1 and not args.skip_cpu:
        res["cpu_baseline"] = cpu_qp_rate()

    # ---- config 3 as a region-of-attraction MAP: anchors of a sub-lattice solved cold, every other grid point first tries its
    # anchor's certified active set in the float64 polish (carmpc_qp_solve with d_seed); identical results, fewer ADMM iterations
    if not args.skip_seeded and full_grid:
        from carmpc_b200.grids import lattice_seeds
        dims = [len(a) for a in axes]
        blocks = [tuple(int(v) for v in b.split("x")) for b in args.seed_blocks.split(",")]
        seeded = {}
        for blk in blocks:
            seed = torch.from_numpy(lattice_seeds(dims, block=blk, start=lo, stop=hi)).to(dev)
            for _ in range(2):
                o = bq.solve(x0, seed=seed)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            it_sum = 0
            e0.record()
            for _ in range(steps):
                o = bq.solve(x0, seed=seed)
                it_sum += bq.last_stats()[0]
                if gather:
                    from carmpc_b200.sharding import gather_samples
                    gather_samples({k: o[k] for k in _SAMPLE_DIM}, gather, _SAMPLE_DIM)
            e1.record()
            e1.synchronize()
            ms_s = e0.elapsed_time(e1) / steps
            ts = torch.tensor([ms_s], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(ts, op=dist.ReduceOp.MAX)
            same = bool((o["status"] == out["status"]).all().item())
            okm = out["status"] == 0
            du = float((o["u0"][:, okm] - out["u0"][:, okm]).abs().max().item())
            seeded["x".join(map(str, blk))] = {
                "qps": B_all / (float(ts.item()) * 1e-3), "ms": float(ts.item()),
                "anchors": int((seed == torch.arange(B, device=dev, dtype=torch.int32)).sum().item()),
                "certified_from_seed": o["seeded"], "mean_admm_iters": it_sum / steps / B,
                "flags_equal_cold": same, "max_du0_vs_cold": du, "polish": bq.polish_stats()}
        best = max(seeded, key=lambda k: seeded[k]["qps"])
        res["seeded_map"] = {"metric": "horizon-20 QPs/s (region-of-attraction map, active sets seeded from lattice anchors)",
                             "value": seeded[best]["qps"], "unit": "QPs/s", "ms_per_step": seeded[best]["ms"],
                             "block": best, "by_block": seeded,
                             "call": "carmpc_qp_solve with d_seed (same certified optima and flags as the cold solve)"}
    if not args.skip_seeded and full_grid and world == 1:
        # end to end for the map: grid axes on the host in, status / u0 / objective on the host out
        blk0 = blocks[0]
        bq.solve_map_host(axes, block=blk0, pinned=True)
        dts = []
        for _ in range(3):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            rm = bq.solve_map_host(axes, block=blk0, pinned=True)
            dts.append(time.perf_counter() - t0)
        tm = torch.tensor([float(np.median(dts))], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        map_e2e = {"value": B_all / float(tm.item()), "unit": "QPs/s", "h2d_bytes_per_step": int(sum(len(a) for a in axes) * 8),
                   "d2h_bytes_per_step": B * (16 + 8 + 4 + 4), "call": "carmpc_qp_map_host (grid axes in, status / u0 / objective / iters out)",
                   "flags_equal_cold": bool(np.array_equal(rm.status, out["status"].cpu().numpy()))}
        res["seeded_map"]["e2e"] = map_e2e

    # ---- config 4: output-feedback Monte-Carlo closed loop --------------------------------------------------------
    if not args.skip_closed_loop:
        from carmpc_b200.lib.mpc import _C_XYV as C_OUT, _L_OBSERVER as L_OBS
        ofb = _controller("RoadEnv", None, 20)
        bl = BatchQP.from_controller(ofb)
        R_all, T = args.cl_runs, args.cl_steps
        g = torch.Generator(device="cpu").manual_seed(0)
        blo = torch.tensor([0.0, -2.5, -0.2, 0.0], dtype=torch.float64)
        bhi = torch.tensor([10.0, 2.5, 0.2, 3.0], dtype=torch.float64)
        r_lo, r_hi = shard_range(R_all, rank, world)              # config 4 shards runs, not steps
        x_all = blo[:, None] + (bhi - blo)[:, None] * torch.rand((4, R_all), generator=g, dtype=torch.float64)
        x_init = x_all[:, r_lo:r_hi].to(dev).contiguous()
        R = x_init.shape[1]
        bl.closed_loop(x_init, 5, ofb.A, ofb.B, C=C_OUT, L=L_OBS)          # full-size warm-up (workspace allocation)
        dts = []
        for _ in range(3):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            o = bl.closed_loop(x_init, T, ofb.A, ofb.B, C=C_OUT, L=L_OBS)
            torch.cuda.synchronize()
            dts.append(time.perf_counter() - t0)
        dt = max_over_ranks(min(dts))
        fail = o["fail_step"]
        final = o["final"]
        goal = torch.tensor([30.0, 1.5, 0.0, 0.0], dtype=torch.float64, device=dev)
        ok = fail < 0
        reached = ((final - goal[:, None]).abs() <= 0.1).all(0) & ok
        n_ok = sum_over_ranks(float(ok.sum().item()))
        res["closed_loop"] = {"workload": f"config 4: RoadEnv output-feedback MPC, {R_all} runs x {T} steps vs nonlinear bicycle"
                                          + (f", runs sharded over {world} GPUs" if world > 1 else ""),
                              "closed_loop_steps_per_s": n_ok * T / dt, "runs_per_s": R_all / dt,
                              "seconds": dt, "never_infeasible_frac": n_ok / R_all,
                              "reached_goal_frac": sum_over_ranks(float(reached.sum().item())) / R_all,
                              "mean_admm_iters_per_qp": sum_over_ranks(float(o["total_iters"])) / max(1.0, n_ok * T)}
    # ---- config 5: horizon sweep ----------------------------------------------------------------------------
    if not args.skip_sweep:
        sweep = {}
        for N in (10, 20, 40, 80):
            cN = c20 if N == 20 else _controller("RoadOneCarEnv", [29.9, 1.5, 0, 0], N)
            bN = bq if N == 20 else BatchQP.from_controller(cN)
            ms_n, it_n, _, o = _time_solves(bN, x0, 2, 1, torch, gather, barrier)      # one full-size warm-up (workspace allocation)
            ms_n = max_over_ranks(ms_n)
            it_n = sum_over_ranks(it_n)
            tl = bN.tiling()
            tinfo = bN.tensor_mode()
            on_tensor = tinfo["samples_last_solve"] > 0
            ffma_ms = None
            if on_tensor:                      # the same solve on the FFMA tile kernel, for the comparison the default rests on
                bN.tensor_mode(0)
                ffma_ms = max_over_ranks(_time_solves(bN, x0, 2, 1, torch, gather, barrier)[0])
                bN.tensor_mode(1)
            seeded_n = None
            if not args.skip_seeded and full_grid:
                from carmpc_b200.grids import lattice_seeds
                blk = tuple(int(v) for v in args.seed_blocks.split(",")[0].split("x"))
                seed = torch.from_numpy(lattice_seeds([len(a) for a in axes], block=blk, start=lo, stop=hi)).to(dev)
                bN.solve(x0, seed=seed)
                torch.cuda.synchronize()
                s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s0.record()
                for _ in range(2):
                    os_ = bN.solve(x0, seed=seed)
                s1.record()
                s1.synchronize()
                ms_s = max_over_ranks(s0.elapsed_time(s1) / 2)
                seeded_n = {"qps": B_all / (ms_s * 1e-3), "ms": ms_s, "mean_iters": bN.last_stats()[0] / B,
                            "flags_equal_cold": bool((os_["status"] == o["status"]).all().item())}
            sweep[str(N)] = {"seeded_map": seeded_n, "qps": B_all / (ms_n * 1e-3), "ms": ms_n, "mean_iters": it_n / B_all,
                             "feasible_frac": float((o["status"] == 0).float().mean().item()),
                             "max_iter_count": int((o["status"] == 2).sum().item()),
                             "executed_tflops": it_n * tl["flop_per_iter"] / (ms_n * 1e-3) / 1e12,
                             "samples_per_lane": tl["samples_per_lane"], "matrices_in_smem": tl["matrices_in_smem"],
                             "admm_kernel": "tcgen05 kind::tf32, 3xTF32 split, 128-sample tiles" if on_tensor else "ffma tile kernel",
                             "tensor_form_available": tinfo["available"], "ffma_kernel_ms": ffma_ms}
            if on_tensor:       # dense multiply-adds the tensor pipe executes: three TF32 products per float32 product
                tf = 3 * it_n * tl["flop_per_iter_dense"] / (ms_n * 1e-3) / 1e12
                sweep[str(N)]["tensor_dense_tflops"] = tf
                sweep[str(N)]["tensor_roofline"] = {
                    "bound": "tensor", "achieved": tf, "peak": 1188.0 * world, "unit": "TFLOP/s", "frac": tf / (1188.0 * world),
                    "peak_source": "measured: sustained tcgen05.mma kind::tf32, 148 SMs (tools/tc_bench.cu, profiles/r02_tc_bench.txt)",
                    "note": "whole solve (ADMM + polish) time; the kernel is bound by the shared-memory port that feeds the K = 8 "
                            "MMAs, not by the tensor pipe (DESIGN.md section 4)"}
        res["horizon_sweep"] = sweep

    return res
