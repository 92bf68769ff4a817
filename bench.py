#!/usr/bin/env python
"""Benchmark of the CarMPC batch-evaluation hot path on B200 (contract: see the task brief / DESIGN.md).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

``--dump-outputs DIR`` writes what the last timed step computed as ``DIR/*.npy`` (see ``dump_outputs``): the inputs are
fixed, so two builds run with the same arguments can be compared output for output.

Headline line (one JSON object on stdout, rank 0): terminal-set samples/s on BASELINE config 2
(RoadMultipleCarsEnv H-rep, 100^4 = 10^8-point float64 SoA grid, resident in HBM).  One "step" = one
membership pass over the whole grid -> bitset + count.  With N > 1 GPUs the ONE grid is sharded over the ranks (strong
scaling) and the all-gather of the bitsets is part of the step (fused into the scan kernel over NVLink peer windows).
The same line carries the QP half of the metric under ``"qp"`` / ``"qp_summary"`` (config 3: 10^6 horizon-20 QPs).

``--impl reference`` times the reference's CPU path (its per-point membership test, restated in oracle/ because the
reference is pure Python with third-party solvers that are not installed) on the host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BYTES_PER_SAMPLE = 32.125          # 4 x float64 read + 1 bit written (SURVEY 8d)
TERMINAL_SET = os.path.join(ROOT, "terminal_sets", "RoadMultipleCarsEnv_30_1.5_0_0.npy")
QP_TERMINAL_SET = os.path.join(ROOT, "terminal_sets", "RoadOneCarEnv_29.9_1.5_0_0.npy")


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        with open(path) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, index: int, period_s: float = 0.01):
        self.index, self.period = index, period_s
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self._nv = None

    def _run(self):
        nv = self._nv
        while not self._stop.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
                mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self._h))
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(self.period)

    def __enter__(self):
        if self._nv is not None:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        if self._thread is not None:
            self._thread.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------------------
# workload description shared by both arms (the driver compares them)
# ------------------------------------------------------------------------------------------------------------
def workload_config():
    return {"workload": "config 2: RoadMultipleCarsEnv terminal set (42 rows, terminal_sets/RoadMultipleCarsEnv_30_1.5_0_0.npy) "
                        "on the 100^4 = 10^8-point float64 SoA grid (x, y, psi, v); one step = one membership pass over the "
                        "WHOLE grid -> bitset + member count; with N GPUs the grid is sharded over them",
            "samples_per_step": 100_000_000,
            "l2": "inputs (3.2 GB in total, 400 MB per GPU at 8 GPUs) exceed the 126 MB L2; no flush between iterations"}


# ------------------------------------------------------------------------------------------------------------
# CPU legs (the only places that execute oracle/)
# ------------------------------------------------------------------------------------------------------------
_HOST_GRID = None


def _host_grid():
    """The whole config-2 grid as four host SoA arrays (3.2 GB), built once per process."""
    global _HOST_GRID
    if _HOST_GRID is None:
        from carmpc_b200.grids import config2_axes
        axes = config2_axes()
        dims = [len(a) for a in axes]
        cols = []
        for k, a in enumerate(axes):
            shape = [1] * 4
            shape[k] = dims[k]
            cols.append(np.ascontiguousarray(np.broadcast_to(np.asarray(a, dtype=np.float64).reshape(shape), dims)).ravel())
        _HOST_GRID = cols
    return _HOST_GRID


def cpu_membership_pass(threads: int = 0):
    """One pass of the C restatement of lib/terminal_set.py:107-113 over the WHOLE 10^8 grid on all host threads;
    returns (seconds, threads, members)."""
    from oracle import c_oracle
    Ab = np.load(TERMINAL_SET)
    cols = _host_grid()
    threads = threads or c_oracle.max_threads()
    t0 = time.perf_counter()
    _, count = c_oracle.membership_bits(Ab, *cols, threads=threads)
    return time.perf_counter() - t0, threads, int(count)


def cpu_membership_rate(min_seconds: float):
    n = len(_host_grid()[0])
    cpu_membership_pass()                                  # warm-up (library build, page faults)
    t0, passes = time.perf_counter(), 0
    while True:
        _, threads, members = cpu_membership_pass()
        passes += 1
        dt = time.perf_counter() - t0
        if dt >= min_seconds:
            break
    return passes * n / dt, threads, f"{passes} passes over the full 10^8-point grid ({dt:.1f} s)", members


def cpu_pointwise_rate(points: int = 60000):
    """The reference's literal per-point Python loop (np.all(A @ point <= b)), one core."""
    from oracle import carmpc_oracle as orc
    Ab = np.load(TERMINAL_SET)
    cols = _host_grid()
    n = len(cols[0])
    idx = np.arange(0, n, n // points, dtype=np.int64)[:points]
    pts = np.stack([c[idx] for c in cols], axis=1)
    t0 = time.perf_counter()
    orc.membership_pointwise(Ab, pts)
    return points / (time.perf_counter() - t0)


def run_reference(args, rank: int, world: int):
    """The reference's own CPU implementation of the path (lib/terminal_set.py:107-113) on the box's host cores.  The
    reference is pure Python with nothing to compile (DESIGN.md section 2), so this is the C restatement in oracle/ on all
    host threads, on the SAME workload as the GPU arm: every step is one pass over the whole 10^8-point grid."""
    if rank != 0:
        return
    steps, warmup = args.steps, args.warmup
    n = len(_host_grid()[0])
    for _ in range(warmup):
        cpu_membership_pass()
    secs, members, threads = [], None, 0
    for _ in range(steps):
        dt, threads, members = cpu_membership_pass()
        secs.append(dt)
    value = n * steps / float(np.sum(secs))
    line = {
        "impl": "reference", "metric": "terminal-set samples/s", "value": value, "unit": "samples/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": float(np.mean(secs)) * 1e3,
        "higher_is_better": True, "scaling": "strong" if args.gpus > 1 else "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": workload_config(),
        "cpu_baseline": {"value": value, "unit": "samples/s", "cores": threads, "kind": "port",
                         "sample": f"{steps} passes over the full 10^8-point grid, one per step",
                         "pointwise_python_samples_per_s": cpu_pointwise_rate()},
        "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "members": members,
        "note": "the reference is pure Python (cvxpy / polytope not installed, nothing to build); this arm is the C "
                "restatement of lib/terminal_set.py:107-113 in oracle/ on all host threads",
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------------
def _pinned_copy_gbs(torch, dev, nbytes=1 << 30):
    """Measured host->device bandwidth of one pinned cudaMemcpyAsync (the link peak the end-to-end path is held against)."""
    src = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    dst = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    dst.copy_(src, non_blocking=True)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(3):
        dst.copy_(src, non_blocking=True)
    e1.record()
    e1.synchronize()
    return 3 * nbytes / (e0.elapsed_time(e1) * 1e-3) / 1e9


DUMP_SAMPLES = 1 << 22             # grid points drawn for flags_sample.npy (about 16 MB of float32)


def dump_outputs(out_dir: str, bits, members: int, n: int) -> None:
    """Writes what one membership step hands its caller (the bitset of the n grid points and the member count) as
    float arrays that two builds can be compared by with any tolerance:

    * ``members.npy``: the member count (float64, shape (1,));
    * ``group_members.npy``: members of every 1024-point group of the grid, in grid order (float64); a flag that
      differs changes one entry;
    * ``flags_sample.npy``: the 0 / 1 flags (float32) of the grid points
      ``np.unique(np.random.default_rng(0).integers(0, n, DUMP_SAMPLES))``, in that order."""
    import torch
    shifts = torch.arange(32, dtype=torch.int32, device=bits.device)
    flags = ((bits[:(n + 31) // 32, None] >> shifts) & 1).reshape(-1)[:n]
    groups = torch.nn.functional.pad(flags, (0, -n % 1024)).reshape(-1, 1024).sum(1)
    idx = torch.from_numpy(np.unique(np.random.default_rng(0).integers(0, n, DUMP_SAMPLES))).to(bits.device)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "members.npy"), np.array([members], dtype=np.float64))
    np.save(os.path.join(out_dir, "group_members.npy"), groups.cpu().numpy().astype(np.float64))
    np.save(os.path.join(out_dir, "flags_sample.npy"), flags[idx].cpu().numpy().astype(np.float32))


def run_ours(args, rank: int, world: int, local_rank: int):
    import torch
    import torch.distributed as dist
    from carmpc_b200.batch import TerminalSetEvaluator
    from carmpc_b200.grids import config2_axes, materialise_grid, materialise_grid_at, grid_size, shard_range
    from carmpc_b200.sharding import PeerWindow, contains_bits_sharded, gather_bitset, reduce_count

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    distributed = world > 1
    if distributed and not dist.is_initialized():
        # NCCL prints its version banner on stdout when the first communicator is created; the contract is ONE JSON
        # line on stdout, so fd 1 points at stderr until the communicator exists
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)

    def barrier():
        if distributed:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        if distributed:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    Ab = np.load(TERMINAL_SET)
    ev = TerminalSetEvaluator(Ab)
    if args.staging:
        ev.set_staging(*[int(t) for t in args.staging.split(",")])
    axes = config2_axes()
    n = grid_size(axes)
    words = (n + 31) // 32
    count = torch.zeros(1, dtype=torch.int64, device=dev)
    total = torch.zeros(1, dtype=torch.int64, device=dev)
    gather_mode, window, window_error = "none (single GPU)", None, None
    if distributed:
        try:
            window = PeerWindow(n, layout=args.layout)
            gather_mode = "fused: the scan kernel stores its bitset words into every rank's window over NVLink (CUDA IPC " \
                          "peer mappings), counts + completion flags by a one-warp exchange kernel; no NCCL call in the step"
        except Exception as exc:                              # no peer access on this box: NCCL carries the gather
            window_error = f"{type(exc).__name__}: {exc}"
        ok = torch.tensor([1 if window is not None else 0], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) == 0:
            window = None
            gather_mode = "nccl: all_gather_into_tensor of the bitset words + all_reduce of the count inside the step"
    # strong scaling: ONE 10^8-point grid.  Cyclic layout (default): its 1024-sample groups are dealt round-robin to the
    # ranks - the cost of a sample depends on where it lies (a warp leaves a tile as soon as all of it is rejected), so
    # contiguous slabs of the grid would leave the ranks with up to 1.8x different work.  Contiguous: rank r scans [lo, hi).
    if window is not None and args.layout == "cyclic":
        local_index = window.local_index(dev)
        x, y, psi, v = materialise_grid_at(axes, local_index)                    # 3.2 GB / world of float64 SoA
        n_local = int(local_index.numel())
        layout = f"cyclic: 1024-sample group g of the grid belongs to rank g % {world}"
    else:
        lo, hi = shard_range(n, rank, world, align=1024)
        n_local = hi - lo
        local_index = None
        x, y, psi, v = materialise_grid(axes, device=dev, start=lo, stop=hi)
        layout = "contiguous ranges of whole 1024-sample groups" if distributed else "whole grid"
    words_local = (n_local + 31) // 32
    bits = [torch.empty(max(words_local, 1), dtype=torch.int32, device=dev) for _ in range(2)]
    full_bits = torch.empty(world * ((shard_range(n, 0, world, align=1024)[1] + 31) // 32), dtype=torch.int32, device=dev) \
        if distributed else None
    launches = 0

    def step_nccl(i):
        # (with the cyclic layout the gathered words arrive in rank-major order: same traffic, not the same layout)
        ev.contains_bits(x, y, psi, v, mode=args.mode, bits=bits[i & 1], count=count)
        gather_bitset(bits[i & 1], n, out=full_bits, shard_align=1024)
        total.copy_(count)
        reduce_count(total)

    def step(i):
        nonlocal launches
        if not distributed:
            ev.contains_bits(x, y, psi, v, mode=args.mode, bits=bits[i & 1], count=total)
            launches += 1
        elif window is not None:
            contains_bits_sharded(ev, window, x, y, psi, v, mode=args.mode, total=total)
            launches += 2                                   # scan (+ stores to every peer) and the exchange kernel
        else:
            step_nccl(i)
            launches += 1

    for i in range(args.warmup):
        step(i)
    barrier()
    # At 8 GPUs a step is ~80 us of GPU work behind three Python -> ctypes -> launch round trips: the collective step (scan
    # kernel with the peer stores + exchange kernel; its launch arguments never change, the step counter lives on the
    # device) is captured once in a CUDA graph and replayed, so that the host does not bound the step rate.
    graph = None
    if distributed and window is not None and not args.no_graph:
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            contains_bits_sharded(ev, window, x, y, psi, v, mode=args.mode, total=total)
        eager_step = step

        def step(i):
            nonlocal launches
            graph.replay()
            launches += 2
        for i in range(2):
            step(i)
        barrier()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clocks:
        barrier()
        if distributed:
            # the ranks leave the host barrier tens of microseconds apart, which is a sizeable part of K steps of ~0.1 ms:
            # one more untimed collective step (its wait kernel is a device-side barrier) lines the GPUs up, and the
            # start event is enqueued right behind it
            step(0)
        launches = 0
        start.record()
        for i in range(args.steps):
            step(i)
        stop.record()
        barrier()
    ms = start.elapsed_time(stop)
    ms_total = max_over_ranks(ms)
    members = int(total.item())
    if window is not None:
        window.check()
    if args.dump_outputs and rank == 0:
        if not distributed:
            last_bits = bits[(args.steps - 1) & 1]
        else:
            last_bits = window.result_bits() if window is not None else full_bits
        dump_outputs(args.dump_outputs, last_bits, members, n)

    # ---- outside the timed steps: the gathered result of the last step against an independent evaluation -----------
    verify = None
    if distributed:
        ev.contains_bits(x, y, psi, v, mode=0, bits=bits[0], count=count)          # float64 kernel, this rank's samples
        ref_total = int(reduce_count(count.clone()).item())
        got = window.result_bits() if window is not None else full_bits[:words]
        gidx = local_index if local_index is not None else torch.arange(lo, hi, device=dev, dtype=torch.int64)
        lidx = torch.arange(n_local, device=dev, dtype=torch.int64)
        mine_gathered = (got[gidx >> 5] >> (gidx & 31).to(torch.int32)) & 1          # my samples, read back from the full bitset
        mine_local = (bits[0][lidx >> 5] >> (lidx & 31).to(torch.int32)) & 1
        same_local = bool(torch.equal(mine_gathered, mine_local))
        # every rank holds the same full bitset: compare a checksum of the words
        chk = got[:words].to(torch.int64).sum().reshape(1)
        chk_min, chk_max = chk.clone(), chk.clone()
        dist.all_reduce(chk_min, op=dist.ReduceOp.MIN)
        dist.all_reduce(chk_max, op=dist.ReduceOp.MAX)
        bits_set = int(np.unpackbits(got[:words].cpu().numpy().view(np.uint8)).sum())
        verify = {"my_samples_in_the_full_bitset_equal_float64_scan": same_local,
                  "full_bitset_identical_on_every_rank": int(chk_min.item()) == int(chk_max.item()),
                  "bits_set_in_full_bitset": bits_set, "count_equal": members == ref_total == bits_set, "members": ref_total}
        ok_all = torch.tensor([1 if (same_local and verify["full_bitset_identical_on_every_rank"] and verify["count_equal"]) else 0], device=dev)
        dist.all_reduce(ok_all, op=dist.ReduceOp.MIN)
        verify["all_ranks_ok"] = bool(int(ok_all.item()))
        assert verify["all_ranks_ok"], verify

    # ---- this rank's scan alone (no peers, no exchange): the kernel the roofline is about --------------------------------
    k_ms = []
    for i in range(min(args.steps, 50)):
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        ev.contains_bits(x, y, psi, v, mode=args.mode, bits=bits[0], count=count)
        s1.record()
        s1.synchronize()
        k_ms.append(s0.elapsed_time(s1))
    kernel_ms = max_over_ranks(float(np.mean(k_ms)))
    # back-to-back launches of the same kernel (what a step is at N = 1)
    barrier()
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record()
    for i in range(args.steps):
        ev.contains_bits(x, y, psi, v, mode=args.mode, bits=bits[0], count=count)
    s1.record()
    s1.synchronize()
    stream_ms = max_over_ranks(s0.elapsed_time(s1) / args.steps)

    # ---- where a collective step spends its time (graph replays: no host in the loop) -------------------------------------
    step_parts = None
    if distributed and window is not None and graph is not None:
        def replay_ms(fn, reps=100):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                fn()
            for _ in range(3):
                g.replay()
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(reps):
                g.replay()
            b.record()
            b.synchronize()
            return max_over_ranks(a.elapsed_time(b) / reps)
        t_scan = replay_ms(lambda: ev.contains_bits(x, y, psi, v, mode=args.mode, bits=bits[0], count=count))
        # scan with the stores into every rank's window + publish, no wait (ranks run free): a second window keeps the
        # protocol state of the timed one untouched
        w2 = PeerWindow(n, layout=args.layout)
        t_p2p = replay_ms(lambda: contains_bits_sharded(ev, w2, x, y, psi, v, mode=args.mode, total=total, defer_wait=True))
        barrier()
        t_full = replay_ms(lambda: contains_bits_sharded(ev, window, x, y, psi, v, mode=args.mode, total=total))
        step_parts = {"scan_local_ms": t_scan, "scan_with_peer_stores_and_publish_ms": t_p2p, "full_step_ms": t_full,
                      "note": "100 CUDA-graph replays each, max over ranks; full step = scan + peer stores + publish + wait for "
                              "every rank's flag (a device-side barrier per step)"}
        stream_ms = t_scan

    nccl_variant = None
    if distributed and window is not None:
        for i in range(3):
            step_nccl(i)
        barrier()
        s0.record()
        for i in range(args.steps):
            step_nccl(i)
        s1.record()
        barrier()
        nccl_ms = max_over_ranks(s0.elapsed_time(s1) / args.steps)
        nccl_variant = {"ms_per_step": nccl_ms, "value": n / (nccl_ms * 1e-3), "unit": "samples/s",
                        "what": "same sharded scan, bitset all_gather_into_tensor + count all_reduce over NCCL inside the step"}

    # ---- end to end through the host-buffer C-ABI call (pinned host SoA in, host bitset out) -----------------
    e2e = None
    if not args.skip_e2e:
        hn = min(args.e2e_samples, n_local)
        host = [torch.empty(hn, dtype=torch.float64, pin_memory=True).copy_(t[:hn]) for t in (x, y, psi, v)]
        hx, hy, hp, hv = [h.numpy() for h in host]
        ev.contains_bits_host(hx[:1 << 20], hy[:1 << 20], hp[:1 << 20], hv[:1 << 20], mode=args.mode)   # warm-up
        ev.contains_bits_host(hx, hy, hp, hv, mode=args.mode)
        barrier()
        t0 = time.perf_counter()
        e2e_steps = args.e2e_steps
        for _ in range(e2e_steps):
            hbits, hcount = ev.contains_bits_host(hx, hy, hp, hv, mode=args.mode)
        torch.cuda.synchronize()
        dt = max_over_ranks(time.perf_counter() - t0)
        hn_all = hn * world if hn == n_local else hn * world
        link_peak = _pinned_copy_gbs(torch, dev)
        link_gbs = hn * 32 * e2e_steps / dt / 1e9
        e2e = {"value": hn_all * e2e_steps / dt, "unit": "samples/s",
               "h2d_bytes_per_step": int(hn * 32), "d2h_bytes_per_step": int((hn + 31) // 32 * 4 + 8),
               "samples_per_step_per_gpu": hn, "steps": e2e_steps,
               "call": "carmpc_membership_bitset_host (pinned host SoA -> chunked H2D | kernel | D2H pipeline), each rank its shard",
               "roofline": {"bound": "host link (PCIe H2D)", "achieved": link_gbs, "peak": link_peak, "unit": "GB/s",
                            "frac": link_gbs / link_peak, "peak_source": "measured live: 1 GiB pinned cudaMemcpyAsync H2D, per GPU"}}
        del host

    # the same grid through the implicit-grid entry point: host axes in (3.2 KB), host bitset out (12.5 MB)
    e2e_grid = None
    if not args.skip_e2e and not distributed:
        gbits = torch.empty(words, dtype=torch.int32, device=dev)
        hbits = torch.empty(words, dtype=torch.int32, pin_memory=True)
        ev.contains_grid_bits(axes, bits=gbits, count=count)
        barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(20):
            ev.contains_grid_bits(axes, bits=gbits, count=count)
            hbits.copy_(gbits, non_blocking=True)
            torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / 20
        e2e_grid = {"value": n / dt, "unit": "samples/s", "h2d_bytes_per_step": int(sum(len(a) for a in axes) * 8),
                    "d2h_bytes_per_step": int(words * 4 + 8),
                    "call": "carmpc_membership_grid (axes on the host, coordinates generated in-kernel) + D2H of the bitset"}

    # ---- the rollout form of the same test (lib/terminal_set.py:53-59, 198-200 sampled): k* + 1 closed-loop steps, state rows
    # at every step, input rows at t = 0; float32 screen over the expanded rows + float64 step-by-step rollout ----------
    rollout = None
    if not args.skip_rollout:
        from carmpc_b200.batch import RolloutEvaluator
        from carmpc_b200.lib.environments import RoadMultipleCarsEnv
        k_star = 16
        rv = RolloutEvaluator.from_env(RoadMultipleCarsEnv(), k_star)
        rwin = None
        if window is not None:
            rwin = PeerWindow(n, layout=args.layout)
        rtotal = torch.zeros(1, dtype=torch.int64, device=dev)

        def rstep():
            if rwin is not None:
                contains_bits_sharded(rv, rwin, x, y, psi, v, total=rtotal)
            else:
                rv.contains_bits(x, y, psi, v, bits=bits[0], count=rtotal)
                if distributed:
                    gather_bitset(bits[0], n, out=full_bits, shard_align=1024)
                    reduce_count(rtotal)

        for _ in range(3):
            rstep()
        barrier()
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        r0.record()
        for _ in range(args.rollout_steps):
            rstep()
        r1.record()
        barrier()
        r_ms = max_over_ranks(r0.elapsed_time(r1) / args.rollout_steps)
        r_members = int(rtotal.item())
        rcount = torch.zeros(1, dtype=torch.int64, device=dev)
        r0.record()
        for _ in range(args.rollout_steps):
            rv.contains_bits(x, y, psi, v, bits=bits[0], count=rcount)
        r1.record()
        r1.synchronize()
        rk_ms = max_over_ranks(r0.elapsed_time(r1) / args.rollout_steps)
        # the plain float64 kernel (one sample per thread; selected when the first violated step is requested)
        exact_ms = None
        if not distributed:
            rv.contains_bits(x, y, psi, v, want_first_violation=True, bits=bits[0], count=rcount)
            torch.cuda.synchronize()
            r0.record()
            for _ in range(3):
                rv.contains_bits(x, y, psi, v, want_first_violation=True, bits=bits[0], count=rcount)
            r1.record()
            torch.cuda.synchronize()
            exact_ms = r0.elapsed_time(r1) / 3
        peak, _ = _peaks()
        s_rows, r_in = len(rv.b_con), len(rv.b_in)
        ach = n_local * BYTES_PER_SAMPLE / (rk_ms * 1e-3) / 1e9
        rollout = {"metric": "rollout-form terminal-set samples/s", "value": n / (r_ms * 1e-3), "unit": "samples/s",
                   "ms_per_step": r_ms, "steps": args.rollout_steps, "k_steps": k_star, "state_rows": s_rows, "input_rows": r_in,
                   "expanded_rows": s_rows * (k_star + 1) + r_in, "screen_rows": rv.screen_rows or rv.expanded_rows,
                   "screen_note": "the float32 screen holds the irredundant subset of the expanded rows (dual certificates for the "
                                  "dropped ones, verified by the library); band samples go to the float64 step-by-step rollout",
                   "members": r_members, "members_hrep": members,
                   "float64_kernel_ms": exact_ms,
                   "float64_kernel_note": "rollout_kernel, also writes the first violated step (4 B/sample)",
                   "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                                "launch_ms": rk_ms, "kernel": "membership_tma_kernel<1, rollout>",
                                "note": "this rank's scan alone, per GPU"},
                   "flop_per_sample_float64_form": (k_star + 1) * 8 * s_rows + 32 * k_star + 32}
        if rank == 0 and world == 1 and not args.skip_cpu:
            from oracle import c_oracle
            cols = [c[::50].copy() for c in _host_grid()]
            t0 = time.perf_counter()
            passes = 0
            while time.perf_counter() - t0 < 4.0:
                c_oracle.rollout_bits(rv.A_k, rv.A_con, rv.b_con, rv.A_in, rv.b_in, rv.goal, k_star, 0, *cols)
                passes += 1
            rollout["cpu_baseline"] = {"value": passes * len(cols[0]) / (time.perf_counter() - t0), "unit": "samples/s",
                                       "cores": c_oracle.max_threads(), "kind": "port",
                                       "sample": f"{passes} passes over every 50th point of the 10^8 grid"}

    qp = None
    if not args.skip_qp:
        try:
            from bench_qp import run_qp_bench
            qp = run_qp_bench(args, rank, world, dev, barrier)
        except Exception as exc:                                      # the QP half must never hide the headline
            qp = {"error": f"{type(exc).__name__}: {exc}"}

    if rank == 0:
        peak, peak_src = _peaks()
        # The dominant kernel is this rank's membership scan.  At N = 1 a step IS one launch of it, so its average
        # duration over the timed region (back-to-back launches, CUDA events on the launching stream) is ms / steps;
        # at N > 1 the step also holds the exchange kernel, so the scan is timed alone, back to back, right after.
        launch_ms = ms_total / args.steps if not distributed else stream_ms
        achieved = n_local * BYTES_PER_SAMPLE / (launch_ms * 1e-3) / 1e9
        cpu = None
        if world == 1 and not args.skip_cpu:
            rate, threads, sample, cpu_members = cpu_membership_rate(10.0)
            cpu = {"value": rate, "unit": "samples/s", "cores": threads, "kind": "port", "sample": sample,
                   "members_equal_gpu": cpu_members == members,
                   "pointwise_python_samples_per_s": cpu_pointwise_rate()}
        qp_summary = None
        if isinstance(qp, dict) and "value" in qp:
            qp_summary = {"metric": qp["metric"], "value": qp["value"], "unit": "QPs/s", "ms_per_step": qp["ms_per_step"],
                          "scaling": qp.get("scaling"), "roofline_frac": (qp.get("roofline") or {}).get("frac"),
                          "roofline_bound": (qp.get("roofline") or {}).get("bound"),
                          "e2e": (qp.get("e2e") or {}).get("value"),
                          "cpu_baseline": (qp.get("cpu_baseline") or {}).get("value"),
                          "seeded_map": (qp.get("seeded_map") or {}).get("value"),
                          "closed_loop_s": (qp.get("closed_loop") or {}).get("seconds"),
                          "sweep_qps": {k: v["qps"] for k, v in (qp.get("horizon_sweep") or {}).items()}}
        line = {
            "metric": "terminal-set samples/s", "value": n * args.steps / (ms_total * 1e-3),
            "unit": "samples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "strong" if distributed else "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": workload_config(),
            "clocks": clocks.summary(),
            "e2e": e2e,
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": n_local * 32.125 if not distributed else None,
                         "traffic_source": "ncu --set full: dram__bytes_read.sum + dram__bytes_write.sum per launch = "
                                           "algorithmic bytes (profiles/)",
                         "peak_source": peak_src, "launch_ms": launch_ms, "isolated_launch_ms": kernel_ms,
                         "kernel": "membership_tma_kernel<1, hrep>" if args.mode == 1 else "membership_kernel<0,true>",
                         "bytes_per_sample": BYTES_PER_SAMPLE, "samples_per_launch": n_local,
                         "algorithmic_bytes_per_launch": n_local * BYTES_PER_SAMPLE,
                         "note": "per GPU: this rank's scan of its shard"},
            "cpu_baseline": cpu,
            "qp_summary": qp_summary,
            "sharding": {"samples_per_gpu": n_local, "layout": layout, "gather": gather_mode, "window_error": window_error,
                         "step_launch": "CUDA graph replay (scan + exchange kernels captured once)" if graph is not None else "eager",
                         "scan_alone_ms": stream_ms, "step_overhead_ms": ms_total / args.steps - stream_ms,
                         "step_parts": step_parts, "verify": verify, "nccl_variant": nccl_variant,
                         "kernel_mode": "fp32 screen + fp64 re-check" if args.mode else "fp64", "members": members},
            "e2e_grid": e2e_grid,
            "rollout": rollout,
            "qp": qp,
        }
        print(json.dumps(line), flush=True)
    if distributed:
        dist.barrier()
        dist.destroy_process_group()


def main():
    sys.dont_write_bytecode = True     # the tree bench.py runs from may be read-only; it gets no bytecode caches either
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the member count and flags of the last timed step to DIR/*.npy (GPU arm, rank 0)")
    ap.add_argument("--mode", type=int, default=1, help="membership kernel: 0 = float64, 1 = float32 screen + float64 re-check")
    ap.add_argument("--layout", default="cyclic", choices=["cyclic", "contiguous"],
                    help="how the one sample set is sharded over the ranks (N > 1)")
    ap.add_argument("--no-graph", action="store_true", help="N > 1: launch every collective step from Python instead of replaying a CUDA graph")
    ap.add_argument("--staging", default="", help="threads,ring_slots,tiles_per_slot of the scan kernel (tuning)")
    ap.add_argument("--e2e-samples", type=int, default=100_000_000)
    ap.add_argument("--e2e-steps", type=int, default=4)
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--skip-qp", action="store_true")
    ap.add_argument("--skip-rollout", action="store_true")
    ap.add_argument("--rollout-steps", type=int, default=20)
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--qp-states", type=int, default=1_000_000)
    ap.add_argument("--qp-steps", type=int, default=5)
    ap.add_argument("--skip-sweep", action="store_true")
    ap.add_argument("--skip-seeded", action="store_true")
    ap.add_argument("--seed-blocks", default="2x8x1x1", help="comma-separated lattice blocks (points per axis) for the seeded map")
    ap.add_argument("--skip-closed-loop", action="store_true")
    ap.add_argument("--cl-runs", type=int, default=100_000)
    ap.add_argument("--cl-steps", type=int, default=200)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU arm (--impl ours)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world == 1 and args.gpus > 1:
        raise SystemExit("bench.py: launch with torch.distributed.run for --gpus > 1")
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
