"""Batched entry points over the CUDA library: the sampled forms of the reference's two hot loops.

* ``TerminalSetEvaluator`` - membership of very many states in an H-rep set ``{x : A x <= b}``
  (the test ``lib/terminal_set.py:107-113`` applies to one grid point at a time).
* ``RolloutEvaluator`` - the same set in its sampled LQR-rollout form (``lib/terminal_set.py:53-59,
  198-200``): constraint rows checked along x(t+1) = A_k x(t).
* ``BatchQP`` - one condensed MPC QP per initial state (``lib/mpc.py:318-335`` / ``:461-478``) and
  Monte-Carlo closed loops against the nonlinear plant (``lib/simulator.py:51-69``).

Device entry points take and return torch CUDA tensors (torch is only the allocator / stream owner);
``*_host`` entry points take numpy arrays and go through the library's own overlapped copy pipeline.
Nothing here computes on the CPU: without the CUDA library every call raises ``CarmpcError``.
"""
from __future__ import annotations

import ctypes
from dataclasses import dataclass
from typing import Optional

import numpy as np

from . import _capi
from ._capi import CarmpcError, check


def _torch():
    import torch
    return torch


def _f64(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float64)


def _stream_ptr(stream=None):
    torch = _torch()
    s = torch.cuda.current_stream() if stream is None else stream
    return ctypes.c_void_p(s.cuda_stream)


def unpack_bits(bits: np.ndarray, n: int) -> np.ndarray:
    """uint32 bitset -> bool[n]: bit (i & 31) of word (i >> 5) is sample i."""
    return np.unpackbits(np.ascontiguousarray(bits).view(np.uint8), bitorder="little")[:n].astype(bool)


class _Handle:
    def __init__(self):
        self._h = ctypes.c_void_p()
        self._lib = _capi.load()

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.carmpc_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class _ScanTuning:
    def set_staging(self, threads_per_cta: int = 256, ring_slots: int = 3, tiles_per_slot: int = 1) -> None:
        """Staging geometry of the bulk-async scan kernel (``carmpc_scan_staging``); results never depend on it."""
        check(self._lib.carmpc_scan_staging(self._h, int(threads_per_cta), int(ring_slots), int(tiles_per_slot)))


def _check_soa(x, y, psi, v):
    torch = _torch()
    n = x.numel()
    for t in (x, y, psi, v):
        if not (t.is_cuda and t.dtype == torch.float64 and t.is_contiguous() and t.numel() == n):
            raise ValueError("x, y, psi, v must be contiguous float64 CUDA tensors of equal length")
    return n


class TerminalSetEvaluator(_Handle, _ScanTuning):
    """``A x <= b`` for every sample; results as a bitset (1 bit per sample, warp-ballot packed)."""

    def __init__(self, A: np.ndarray, b: Optional[np.ndarray] = None):
        super().__init__()
        A = _f64(A)
        Ab = A if b is None else np.hstack((A, _f64(b).reshape(-1, 1)))
        if Ab.ndim != 2 or Ab.shape[1] != 5:
            raise ValueError("expected A (rows, 4) and b (rows,), or [A | b] (rows, 5)")
        self.Ab = np.ascontiguousarray(Ab)
        self.rows = len(Ab)
        check(self._lib.carmpc_polytope_create(_capi.ptr(self.Ab), self.rows, ctypes.byref(self._h)))

    @classmethod
    def from_file(cls, path: str) -> "TerminalSetEvaluator":
        """Load a ``terminal_sets/<env>_<goal>.npy`` H-rep (``[A | b]`` rows)."""
        return cls(np.load(path))

    # ---- device tensors in, device bitset out ------------------------------------------------
    def contains_bits(self, x, y, psi, v, mode: int = 1, bits=None, count=None, stream=None):
        """Returns ``(bits int32[ceil(n/32)], count int64[1])`` CUDA tensors; nothing is synchronised."""
        torch = _torch()
        n = _check_soa(x, y, psi, v)
        if bits is None:
            bits = torch.empty((n + 31) // 32, dtype=torch.int32, device=x.device)
        if count is None:
            count = torch.empty(1, dtype=torch.int64, device=x.device)
        check(self._lib.carmpc_membership_bitset(self._h, x.data_ptr(), y.data_ptr(), psi.data_ptr(), v.data_ptr(),
                                                 n, bits.data_ptr(), count.data_ptr(), mode, _stream_ptr(stream)))
        return bits, count

    def tune(self, x, y, psi, v, stream=None) -> None:
        """Adapt the row order to where these samples lie (done automatically on the first call with >= 2^20 samples);
        membership results never depend on it."""
        n = _check_soa(x, y, psi, v)
        check(self._lib.carmpc_polytope_tune(self._h, x.data_ptr(), y.data_ptr(), psi.data_ptr(), v.data_ptr(), n,
                                             _stream_ptr(stream)))

    def contains_grid_bits(self, axes, axis_to_state=(0, 1, 2, 3), bits=None, count=None, stream=None):
        """Membership on the implicit tensor grid ``axes[0] x axes[1] x axes[2] x axes[3]`` (C order); axis k carries
        state component ``axis_to_state[k]``.  No coordinate array is materialised."""
        torch = _torch()
        axes = [_f64(a).ravel() for a in axes]
        dims = (ctypes.c_int32 * 4)(*[len(a) for a in axes])
        a2s = (ctypes.c_int32 * 4)(*axis_to_state)
        n = int(np.prod([len(a) for a in axes]))
        cat = np.ascontiguousarray(np.concatenate(axes))
        if bits is None:
            bits = torch.empty((n + 31) // 32, dtype=torch.int32, device="cuda")
        if count is None:
            count = torch.empty(1, dtype=torch.int64, device="cuda")
        check(self._lib.carmpc_membership_grid(self._h, _capi.ptr(cat), dims, a2s, bits.data_ptr(), count.data_ptr(),
                                               _stream_ptr(stream)))     # the axes are copied before the call returns
        return bits, count

    # ---- host arrays in, host results out ---------------------------------------------------------
    def contains_bits_host(self, x, y, psi, v, mode: int = 1):
        """numpy SoA in -> ``(bits uint32[ceil(n/32)], count)``; copies overlap the kernel inside the library."""
        x, y, psi, v = _f64(x), _f64(y), _f64(psi), _f64(v)
        n = len(x)
        if not (len(y) == len(psi) == len(v) == n):
            raise ValueError("x, y, psi, v must have equal length")
        bits = np.zeros((n + 31) // 32, dtype=np.uint32)
        cnt = ctypes.c_int64(0)
        check(self._lib.carmpc_membership_bitset_host(self._h, _capi.ptr(x), _capi.ptr(y), _capi.ptr(psi),
                                                      _capi.ptr(v), n, _capi.ptr(bits), ctypes.byref(cnt), mode))
        return bits, int(cnt.value)

    def contains_host(self, x, y, psi, v, mode: int = 1) -> np.ndarray:
        """bool[n] membership of numpy SoA samples."""
        bits, _ = self.contains_bits_host(x, y, psi, v, mode)
        return unpack_bits(bits, len(np.atleast_1d(x)))


class RolloutEvaluator(_Handle, _ScanTuning):
    """Sampled form of the terminal set: e(0) = p - goal, e(t+1) = A_k e(t); state rows for t = 0..k_steps, input
    rows at t = 0 only (``input_every_step=False``, what the reference's construction does) or at every step."""

    def __init__(self, A_k, A_con, b_con, A_in, b_in, goal, k_steps: int, input_every_step: bool = False,
                 reduce_screen: bool = True):
        super().__init__()
        self.A_k, self.A_con, self.b_con = _f64(A_k), _f64(A_con).reshape(-1, 4), _f64(b_con).ravel()
        self.A_in, self.b_in, self.goal = _f64(A_in).reshape(-1, 4), _f64(b_in).ravel(), _f64(goal).ravel()
        self.k_steps = int(k_steps)
        check(self._lib.carmpc_rollout_create(_capi.ptr(self.A_k), _capi.ptr(self.A_con), _capi.ptr(self.b_con),
                                              len(self.b_con), _capi.ptr(self.A_in), _capi.ptr(self.b_in),
                                              len(self.b_in), _capi.ptr(self.goal), self.k_steps,
                                              1 if input_every_step else 0, ctypes.byref(self._h)))
        self.screen_rows = self.expanded_rows = 0
        if reduce_screen:
            self._reduce_screen()

    def expanded(self) -> np.ndarray:
        """The expanded rows ``g = a_r A_k^t`` of the float32 screen as the library built them: (rows, 5) = g, b'."""
        n = self._lib.carmpc_rollout_get_rows(self._h, None, 0)
        if n <= 0:
            return np.zeros((0, 5))
        rows = np.zeros((n, 5))
        check(min(0, self._lib.carmpc_rollout_get_rows(self._h, _capi.ptr(rows), rows.size)))
        return rows

    @staticmethod
    def irredundant_rows(rows: np.ndarray, abs_tol: float = 1e-9, n_dual: int = 4):
        """For expanded rows (m, 5) = g, b': the indices kept (ascending), and for every other row a redundancy certificate
        over kept rows - (m, n_dual) row indices and weights >= 0 with ``g_d = sum w_k g_k`` and ``sum w_k b_k <= b_d`` (the
        dual solution of ``max g_d . p`` over the kept rows; a vertex solution has at most four non-zero weights in R^4).
        Rows without a clean certificate are kept."""
        from scipy.optimize import linprog
        from .lib import polytope_ops as pc
        G, b = rows[:, :4], rows[:, 4]
        kept = set(int(i) for i in pc.reduce_indices(pc.Polytope(G, b, normalize=False), abs_tol))
        idx = np.zeros((len(rows), n_dual), dtype=np.int32)
        w = np.zeros((len(rows), n_dual))
        for _ in range(3):                                   # a dropped row without a clean certificate is kept instead
            order = np.array(sorted(kept), dtype=np.int64)
            again = False
            for d in range(len(rows)):
                if d in kept:
                    continue
                res = linprog(b[order], A_eq=G[order].T, b_eq=G[d], bounds=[(0, None)] * len(order), method="highs")
                lam = res.x if res.status == 0 else None
                nz = np.flatnonzero(lam > 1e-12) if lam is not None else np.zeros(0, dtype=np.int64)
                if lam is None or len(nz) == 0 or len(nz) > n_dual or res.fun - b[d] > 1e-6:
                    kept.add(d)
                    again = True
                    continue
                idx[d] = order[nz[0]]
                w[d] = 0.0
                idx[d, :len(nz)] = order[nz]
                w[d, :len(nz)] = lam[nz]
            if not again:
                break
        return np.array(sorted(kept), dtype=np.int32), idx, w

    def _reduce_screen(self) -> None:
        """Keeps only the irredundant expanded rows in the float32 screen (the operation ``lib/terminal_set.py:203`` applies
        to the same set) and hands the library one certificate per dropped row; the library verifies them and widens its
        acceptance band by what they leave open (``carmpc_rollout_reduce_screen``)."""
        rows = self.expanded()
        self.expanded_rows = self.screen_rows = len(rows)
        if len(rows) < 24 or not np.all(np.isfinite(rows)):
            return
        order, idx, w = self.irredundant_rows(rows)
        if len(order) >= len(rows):
            return
        check(self._lib.carmpc_rollout_reduce_screen(self._h, order.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), len(order),
                                                     idx.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), _capi.ptr(w), idx.shape[1]))
        self.screen_rows = len(order)

    @classmethod
    def from_env(cls, env, k_steps: int, input_every_step: bool = False) -> "RolloutEvaluator":
        """Rows exactly as ``calc_terminal_set`` builds them: unit-norm state rows shifted to the goal, and
        ``[I; -I] K`` input rows (``lib/terminal_set.py:145-161, 198-200``)."""
        from .lib.terminal_set import lqr_closed_loop
        from .lib import polytope_ops as pc
        _, A_k, A_con, b_con, A_in, b_in = lqr_closed_loop(env)
        goal = np.array(env.goal, dtype=float)
        pc_state = pc.Polytope(A_con, b_con).translation(-goal)
        pc_in = pc.Polytope(A_in, b_in)
        return cls(A_k, pc_state.A, pc_state.b, pc_in.A, pc_in.b, goal, k_steps, input_every_step)

    def contains_bits(self, x, y, psi, v, want_first_violation: bool = False, bits=None, count=None, stream=None):
        torch = _torch()
        n = _check_soa(x, y, psi, v)
        if bits is None:
            bits = torch.empty((n + 31) // 32, dtype=torch.int32, device=x.device)
        if count is None:
            count = torch.empty(1, dtype=torch.int64, device=x.device)
        first = torch.empty(n, dtype=torch.int32, device=x.device) if want_first_violation else None
        check(self._lib.carmpc_rollout_bitset(self._h, x.data_ptr(), y.data_ptr(), psi.data_ptr(), v.data_ptr(), n,
                                              bits.data_ptr(), first.data_ptr() if first is not None else None,
                                              count.data_ptr(), _stream_ptr(stream)))
        return (bits, count, first) if want_first_violation else (bits, count)

    def contains_bits_host(self, x, y, psi, v, want_first_violation: bool = False):
        x, y, psi, v = _f64(x), _f64(y), _f64(psi), _f64(v)
        n = len(x)
        bits = np.zeros((n + 31) // 32, dtype=np.uint32)
        first = np.zeros(n, dtype=np.int32) if want_first_violation else None
        cnt = ctypes.c_int64(0)
        check(self._lib.carmpc_rollout_bitset_host(self._h, _capi.ptr(x), _capi.ptr(y), _capi.ptr(psi), _capi.ptr(v), n,
                                                   _capi.ptr(bits), _capi.ptr(first), ctypes.byref(cnt)))
        return (bits, int(cnt.value), first) if want_first_violation else (bits, int(cnt.value))


def measure_peak(which: str) -> float:
    """Device micro-benchmarks: 'fp32' / 'fp64' FMA TFLOP/s (uniform multiplier), 'hbm' copy GB/s (read + write),
    'fp32_tile' TFLOP/s of a shared-memory-fed 8 x 8 register-tile product (both multiplicands in vector registers)."""
    idx = {"fp32": 0, "fp64": 1, "hbm": 2, "fp32_tile": 3}[which]
    val = ctypes.c_double(0.0)
    check(_capi.load().carmpc_measure_peak(idx, ctypes.byref(val)))
    return float(val.value)


# ----------------------------------------------------------------------------------------------------
# batched condensed MPC QP
# ----------------------------------------------------------------------------------------------------
@dataclass
class QPResult:
    """Per-sample results of a batched solve, in the layouts the reference uses for one sample."""
    u0: np.ndarray              # (B, 2)   first input of the optimal sequence (what ``.step`` returns)
    objective: np.ndarray       # (B,)     1/2 u'Hu + q'u  (the reference's ``cost``); +inf when infeasible
    status: np.ndarray          # (B,)     0 solved, 1 infeasible (outside the region of attraction), 2 max_iter
    iters: np.ndarray           # (B,)     ADMM iterations spent
    u_full: Optional[np.ndarray] = None     # (B, 2N)
    seeded: int = 0                         # map solves: samples certified from their anchor without ADMM iterations


class BatchQP(_Handle):
    """One condensed MPC QP per initial state, all on the GPU (``carmpc_qp_*``)."""

    def __init__(self, pq, **opts):
        super().__init__()
        self.pq = pq
        self.n, self.m = pq.n, pq.m
        o = _capi.QPOpts()
        self._lib.carmpc_qp_default_opts(ctypes.byref(o))
        for k, v in opts.items():
            if not hasattr(o, k):
                raise TypeError(f"unknown QP option {k!r}")
            setattr(o, k, v)
        self.opts = o
        arrs = [_f64(pq.H), _f64(pq.F), _f64(pq.G), _f64(pq.Gx), _f64(pq.Gc), _f64(pq.lo), _f64(pq.hi), _f64(pq.lb),
                _f64(pq.ub), _f64(pq.Px), _f64(pq.Pc), _f64(pq.pre_lo), _f64(pq.pre_hi)]
        self._keep = arrs
        check(self._lib.carmpc_qp_create(pq.n, pq.m, len(pq.pre_hi), *[_capi.ptr(a) if a.size else None for a in arrs],
                                         ctypes.byref(o), ctypes.byref(self._h)))

    @classmethod
    def from_controller(cls, controller, **opts) -> "BatchQP":
        """Condense an ``lib.mpc.MPC`` controller (its enabled constraint blocks, goal, horizon)."""
        from .condensed import build_parametric_qp
        return cls(build_parametric_qp(controller), **opts)

    # ---- introspection --------------------------------------------------------------------------
    def setup(self, which: int) -> np.ndarray:
        """Host view of the solver setup (see ``carmpc_qp_get_setup``)."""
        cnt = self._lib.carmpc_qp_get_setup(self._h, which, None, 0)
        if cnt < 0:
            check(cnt)
        out = np.zeros(cnt)
        got = self._lib.carmpc_qp_get_setup(self._h, which, _capi.ptr(out), cnt)
        if got < 0:
            check(got)
        return out

    def tiling(self) -> dict:
        t = self.setup(7)
        keys = ("samples_per_lane", "groups_a", "groups_b", "matrices_in_smem", "smem_bytes", "flop_per_iter",
                "flop_per_iter_dense", "k_total", "padded_rows", "padded_vars")
        return dict(zip(keys, t))

    def last_stats(self):
        """(sum of ADMM iterations over the samples of the last solve, kernel launches issued)."""
        a, b = ctypes.c_int64(0), ctypes.c_int64(0)
        check(self._lib.carmpc_qp_last_stats(self._h, ctypes.byref(a), ctypes.byref(b)))
        return int(a.value), int(b.value)

    def polish_stats(self) -> dict:
        """Histogram of the float64 polish over the last solve (``carmpc_qp_polish_stats``)."""
        h = (ctypes.c_int64 * 20)()
        check(self._lib.carmpc_qp_polish_stats(self._h, h))
        v = [int(x) for x in h]
        return {"certified_after_rounds": v[:10], "handed_to_admm": v[10], "used_multiplier_map": v[11],
                "certified_by_map_alone": v[12], "infeasible_by_anchor_certificate": v[13],
                "max_iter_settled_by_own_certificate": v[14], "infeasible_before_second_pass": v[15],
                "final_polish_uncertified": v[16], "fallback_solved": v[17], "fallback_infeasible": v[18],
                "fallback_undecided": v[19]}

    def tensor_mode(self, mode: int = -1) -> dict:
        """Selects (0 / 1) or queries (-1) the ADMM kernel of large first passes (``carmpc_qp_tensor_mode``): 1 = the
        tcgen05 kernel when the problem has a tensor-core form, 0 = the FFMA tile kernel."""
        info = (ctypes.c_int64 * 16)()
        check(self._lib.carmpc_qp_tensor_mode(self._h, int(mode), info))
        return {"mode": int(info[0]), "available": bool(info[1]), "parts": int(info[1]), "samples_last_solve": int(info[2]),
                "matrices_resident": bool(info[3]), "cycles": [int(v) for v in info[4:16]]}

    # ---- device tensors ---------------------------------------------------------------------------
    def solve(self, x0, x_ref=None, c=None, want_u_full: bool = False, warm=None, warm_in: bool = False,
              warm_out: bool = False, stream=None, seed=None, want_certificate: bool = False) -> dict:
        """``x0``: (4, B) float64 CUDA tensor (SoA).  Returns a dict of CUDA tensors: ``u0`` (2, B), ``objective``
        (B,), ``status`` (B,) int32, ``iters`` (B,) int32 and optionally ``u_full`` (B, 2N).

        ``seed`` (int32 CUDA tensor of B entries, e.g. ``grids.lattice_seeds``): sample ``i`` first tries the certified
        active set of sample ``seed[i]`` (an anchor: ``seed[a] == a``) and runs ADMM only if that does not certify;
        ``out["seeded"]`` counts the samples that needed no ADMM iteration.  Same results as the cold solve.

        ``want_certificate``: also ``out["certificate"]``, a (B, m + n + k) float64 CUDA tensor in the row space of the
        handle (``d_cert`` of ``carmpc_qp_solve``): the KKT multipliers of solved samples, the Farkas ray of infeasible ones,
        zeros for undecided ones.  The other outputs are bit-identical to a solve without it (not with ``warm``)."""
        torch = _torch()
        if not (x0.is_cuda and x0.dtype == torch.float64 and x0.dim() == 2 and x0.shape[0] == 4 and x0.is_contiguous()):
            raise ValueError("x0 must be a contiguous (4, B) float64 CUDA tensor")
        B = x0.shape[1]
        dev = x0.device
        xref = _f64(self.pq.goal if x_ref is None else x_ref)
        out = {"u0": torch.empty((2, B), dtype=torch.float64, device=dev),
               "objective": torch.empty(B, dtype=torch.float64, device=dev),
               "status": torch.empty(B, dtype=torch.int32, device=dev),
               "iters": torch.empty(B, dtype=torch.int32, device=dev)}
        if want_u_full:
            out["u_full"] = torch.empty((B, self.n), dtype=torch.float64, device=dev)
        if warm is not None and not (warm.is_cuda and warm.dtype == torch.float32 and warm.numel() == B * (self.m + self.n)):
            raise ValueError("warm must be a float32 CUDA tensor of B * (m + n) elements")
        if seed is not None:
            if warm is not None:
                raise ValueError("seed and warm are alternative starting points")
            if not (seed.is_cuda and seed.dtype == torch.int32 and seed.numel() == B and seed.is_contiguous()):
                raise ValueError("seed must be a contiguous int32 CUDA tensor of B entries")
        if want_certificate:
            if warm is not None:
                raise ValueError("certificates are exported by cold and seeded solves, not warm-started ones")
            out["certificate"] = torch.empty((B, self.m + self.n + len(self.pq.pre_hi)), dtype=torch.float64, device=dev)

        def p(t):
            return t.data_ptr() if t is not None else None

        seeded = ctypes.c_int64(0)
        check(self._lib.carmpc_qp_solve(
            self._h, x0.data_ptr(), _capi.ptr(xref), p(c), p(seed), B, out["u0"].data_ptr(), out["objective"].data_ptr(),
            out["status"].data_ptr(), out["iters"].data_ptr(), p(out.get("u_full")), p(warm), int(warm_in), int(warm_out),
            p(out.get("certificate")), ctypes.byref(seeded), _stream_ptr(stream)))
        if seed is not None:
            out["seeded"] = int(seeded.value)
        return out

    def sensitivity(self, x0, out, c=None, rows: Optional[int] = None, stream=None) -> dict:
        """Derivatives of a certified solve with respect to ``(x, y, psi, v, c)`` (``carmpc_qp_sensitivity``).

        ``out``: the dict of ``solve(x0, c=c, want_u_full=True, want_certificate=True)`` (cold or seeded) for the same
        ``x0`` and ``c``.  Returns CUDA tensors ``jac`` (B, rows, 5) = du/dp of the leading ``rows`` variables (default n;
        2 gives the local gain du0/dp), ``grad_objective`` (B, 5) = dV/dp and ``flags`` (B,) int32 (the bits of
        ``carmpc_b200.sensitivity``).  Samples with status != 0 get NaN and flags 0.  Nothing is synchronised."""
        torch = _torch()
        if not (x0.is_cuda and x0.dtype == torch.float64 and x0.dim() == 2 and x0.shape[0] == 4 and x0.is_contiguous()):
            raise ValueError("x0 must be a contiguous (4, B) float64 CUDA tensor")
        B = x0.shape[1]
        if "u_full" not in out or "certificate" not in out:
            raise ValueError("out must come from solve(..., want_u_full=True, want_certificate=True)")
        width = self.m + self.n + len(self.pq.pre_hi)
        for name, t, shape, dt in (("status", out["status"], (B,), torch.int32),
                                   ("u_full", out["u_full"], (B, self.n), torch.float64),
                                   ("certificate", out["certificate"], (B, width), torch.float64)):
            if not (t.is_cuda and t.dtype == dt and tuple(t.shape) == shape and t.is_contiguous()):
                raise ValueError(f"out[{name!r}] must be a contiguous {dt} CUDA tensor of shape {shape}")
        if c is not None and not (c.is_cuda and c.dtype == torch.float64 and c.numel() == B and c.is_contiguous()):
            raise ValueError("c must be a contiguous float64 CUDA tensor of B entries")
        rows = self.n if rows is None else int(rows)
        dev = x0.device
        res = {"jac": torch.empty((B, rows, 5), dtype=torch.float64, device=dev),
               "grad_objective": torch.empty((B, 5), dtype=torch.float64, device=dev),
               "flags": torch.empty(B, dtype=torch.int32, device=dev)}
        check(self._lib.carmpc_qp_sensitivity(
            self._h, x0.data_ptr(), c.data_ptr() if c is not None else None, B, out["status"].data_ptr(),
            out["u_full"].data_ptr(), out["certificate"].data_ptr(), rows, res["jac"].data_ptr(),
            res["grad_objective"].data_ptr(), res["flags"].data_ptr(), _stream_ptr(stream)))
        return res

    # ---- host arrays ---------------------------------------------------------------------------------
    def _host_result(self, B: int, want_u0=True, want_objective=True, want_u_full=False, pinned=False) -> QPResult:
        """Host result arrays; ``pinned``: page-locked buffers owned by this object and reused by the next call of the same
        size (device -> host copies then run at the full PCIe rate instead of through the driver's staging buffer)."""
        if not pinned:
            return QPResult(u0=np.zeros((B, 2)) if want_u0 else None, objective=np.zeros(B) if want_objective else None,
                            status=np.zeros(B, dtype=np.int32), iters=np.zeros(B, dtype=np.int32),
                            u_full=np.zeros((B, self.n)) if want_u_full else None)
        torch = _torch()
        cache = getattr(self, "_pinned", None)
        if cache is None or cache[0] != B:
            bufs = {"u0": torch.empty((B, 2), dtype=torch.float64, pin_memory=True),
                    "objective": torch.empty(B, dtype=torch.float64, pin_memory=True),
                    "status": torch.empty(B, dtype=torch.int32, pin_memory=True),
                    "iters": torch.empty(B, dtype=torch.int32, pin_memory=True)}
            cache = self._pinned = (B, bufs)
        bufs = cache[1]
        if want_u_full and "u_full" not in bufs:
            bufs["u_full"] = torch.empty((B, self.n), dtype=torch.float64, pin_memory=True)
        return QPResult(u0=bufs["u0"].numpy() if want_u0 else None, objective=bufs["objective"].numpy() if want_objective else None,
                        status=bufs["status"].numpy(), iters=bufs["iters"].numpy(),
                        u_full=bufs["u_full"].numpy() if want_u_full else None)

    def solve_host(self, x0, x_ref=None, want_u_full: bool = False, c=None, pinned: bool = False) -> QPResult:
        """``x0``: (B, 4) numpy states, as the reference passes them to ``.step`` one at a time.  ``pinned``: return the
        results in page-locked buffers that the next call of the same size overwrites."""
        x0 = _f64(np.atleast_2d(x0))
        if x0.shape[1] != 4:
            raise ValueError("x0 must be (B, 4)")
        B = len(x0)
        xref = _f64(self.pq.goal if x_ref is None else x_ref)
        res = self._host_result(B, want_u_full=want_u_full, pinned=pinned)
        cc = _f64(c) if c is not None else None
        check(self._lib.carmpc_qp_solve_host(self._h, _capi.ptr(x0), _capi.ptr(xref), _capi.ptr(cc), B,
                                             _capi.ptr(res.u0), _capi.ptr(res.objective), _capi.ptr(res.status),
                                             _capi.ptr(res.iters), _capi.ptr(res.u_full)))
        return res

    def solve_map_host(self, axes, block=None, x_ref=None, axis_to_state=(0, 1, 2, 3), want_u0: bool = True,
                       want_objective: bool = True, pinned: bool = False) -> QPResult:
        """Region-of-attraction map of the C-order tensor grid ``axes`` (four 1-D arrays; axis k is state component
        ``axis_to_state[k]``), numpy in / numpy out (``carmpc_qp_map_host``).  ``block``: points per axis of the lattice
        blocks for the seeded solve (None: every point cold).  ``result.seeded`` = points certified from their anchor.
        ``pinned``: results in page-locked buffers that the next call of the same size overwrites."""
        ax = [_f64(np.atleast_1d(a)) for a in axes]
        if len(ax) != 4:
            raise ValueError("axes must be four 1-D arrays")
        dims = (ctypes.c_int32 * 4)(*[len(a) for a in ax])
        a2s = (ctypes.c_int32 * 4)(*axis_to_state)
        blk = (ctypes.c_int32 * 4)(*[int(b) for b in block]) if block is not None else None
        flat = _f64(np.concatenate(ax))
        B = int(np.prod([len(a) for a in ax]))
        xref = _f64(self.pq.goal if x_ref is None else x_ref)
        res = self._host_result(B, want_u0=want_u0, want_objective=want_objective, pinned=pinned)
        seeded = ctypes.c_int64(0)
        check(self._lib.carmpc_qp_map_host(self._h, _capi.ptr(flat), dims, a2s, blk, _capi.ptr(xref), _capi.ptr(res.u0),
                                           _capi.ptr(res.objective), _capi.ptr(res.status), _capi.ptr(res.iters),
                                           ctypes.byref(seeded)))
        res.seeded = int(seeded.value)
        return res

    # ---- Monte-Carlo closed loop ------------------------------------------------------------------------
    @staticmethod
    def _monitor_rows(monitor) -> np.ndarray:
        """(rows, 5) [A | b] or (A, b) -> contiguous float64 (rows, 5)."""
        if isinstance(monitor, (tuple, list)) and len(monitor) == 2:
            A_, b_ = np.asarray(monitor[0], dtype=np.float64), np.asarray(monitor[1], dtype=np.float64).ravel()
            if A_.ndim != 2 or A_.shape[1] != 4 or len(b_) != len(A_):
                raise ValueError("monitor (A, b) must be (rows, 4) and (rows,)")
            rows = np.hstack((A_, b_[:, None]))
        else:
            rows = np.asarray(monitor, dtype=np.float64)
            if rows.ndim != 2 or rows.shape[1] != 5:
                raise ValueError("monitor must be (rows, 5) [A | b] or (A, b)")
        if not 1 <= len(rows) <= 512 or not np.isfinite(rows).all():
            raise ValueError("monitor must have 1 to 512 finite rows")
        return np.ascontiguousarray(rows)

    def _closed_loop(self, mode, x_init, steps, A, B, C, L, dm, x_ref, dt, l1, warm_start, xhat_init, dhat_init, d_plant,
                     want_traj, want_inputs, want_dhat, noise, monitor, goal, stream) -> dict:
        """``carmpc_closed_loop`` in ``mode`` 0, 1 or 2 (``dm``: a ``DisturbanceModel``): checks the device inputs,
        then returns the outputs the ``want_*`` flags, the mode, the monitor and the goal ask for, and ``total_iters``."""
        torch = _torch()
        if not (x_init.is_cuda and x_init.dtype == torch.float64 and x_init.dim() == 2 and x_init.shape[0] == 4
                and x_init.is_contiguous()):
            raise ValueError("x_init must be a contiguous (4, R) float64 CUDA tensor")
        R, dev = x_init.shape[1], x_init.device
        for name, t in (("d_plant", d_plant), ("dhat_init", dhat_init)):
            if t is not None and not (t.is_cuda and t.dtype == torch.float64 and t.numel() == R and t.is_contiguous()):
                raise ValueError(f"{name} must be a contiguous float64 CUDA tensor of R elements")
        if xhat_init is not None and not (xhat_init.is_cuda and xhat_init.dtype == torch.float64
                                          and tuple(xhat_init.shape) == (4, R) and xhat_init.is_contiguous()):
            raise ValueError("xhat_init must be a contiguous (4, R) float64 CUDA tensor")
        xref = _f64(self.pq.goal if x_ref is None else x_ref)
        A_, B_ = _f64(A), _f64(B)
        C_ = _f64(C) if C is not None else None
        L_ = _f64(L) if L is not None else None
        params = noise.params() if noise is not None else None
        rows = self._monitor_rows(monitor) if monitor is not None else None
        goal_rows = self._monitor_rows(goal) if goal is not None else None
        out = {"final": torch.empty((4, R), dtype=torch.float64, device=dev)}
        if mode == 2:
            out["dhat"] = torch.empty(R, dtype=torch.float64, device=dev)
        out["fail_step"] = torch.empty(R, dtype=torch.int32, device=dev)
        if want_traj:
            out["traj"] = torch.empty((steps, 4, R), dtype=torch.float64, device=dev)
        if want_inputs:
            out["inputs"] = torch.empty((steps, 2, R), dtype=torch.float64, device=dev)
        if want_dhat:
            out["dhat_traj"] = torch.empty((steps, R), dtype=torch.float64, device=dev)
        if rows is not None:
            out["violation_step"] = torch.empty(R, dtype=torch.int32, device=dev)
            out["violation_row"] = torch.empty(R, dtype=torch.int32, device=dev)
            out["violations_per_step"] = torch.empty(steps, dtype=torch.int32, device=dev)
        if goal_rows is not None:
            out["arrival_step"] = torch.empty(R, dtype=torch.int32, device=dev)
            out["arrivals_per_step"] = torch.empty(steps, dtype=torch.int32, device=dev)

        def p(key):
            return out[key].data_ptr() if key in out else None

        def loop_rows(Ab, step, row, per_step):
            if Ab is None:
                return None
            return ctypes.byref(_capi.LoopRows(Ab.ctypes.data, len(Ab), p(step), p(row), p(per_step)))

        total = ctypes.c_int64(0)
        check(self._lib.carmpc_closed_loop(
            self._h, mode, _capi.ptr(A_), _capi.ptr(B_), _capi.ptr(C_), _capi.ptr(L_),
            ctypes.byref(dm) if dm is not None else None, _capi.ptr(xref), float(dt), float(l1), int(steps),
            int(warm_start), x_init.data_ptr(), xhat_init.data_ptr() if xhat_init is not None else None,
            dhat_init.data_ptr() if dhat_init is not None else None, d_plant.data_ptr() if d_plant is not None else None,
            R, p("final"), p("dhat"), p("fail_step"), p("traj"), p("inputs"), p("dhat_traj"),
            ctypes.byref(params) if params is not None else None,
            loop_rows(rows, "violation_step", "violation_row", "violations_per_step"),
            loop_rows(goal_rows, "arrival_step", None, "arrivals_per_step"), ctypes.byref(total), _stream_ptr(stream)))
        out["total_iters"] = int(total.value)
        return out

    def closed_loop(self, x_init, steps: int, A, B, x_ref=None, C=None, L=None, xhat_init=None, dt: float = 0.2,
                    l1: float = 3.5, warm_start: bool = True, want_traj: bool = False, want_inputs: bool = False,
                    noise=None, monitor=None, goal=None, stream=None) -> dict:
        """Runs ``steps`` closed-loop steps for every column of ``x_init`` ((4, R) float64 CUDA tensor) against the
        nonlinear bicycle.  Output feedback when ``C`` and ``L`` are given (observer started at ``xhat_init`` or the
        true state), state feedback otherwise.  Returns ``final`` (4, R), ``fail_step`` (R,) int32 (-1: never
        infeasible), optionally ``traj`` (steps, 4, R) and ``inputs`` (steps, 2, R), and ``total_iters``.

        ``noise``: a ``carmpc_b200.montecarlo.LoopNoise`` (process and measurement noise drawn on the device).
        ``monitor``: (rows, 5) ``[A | b]`` or ``(A, b)``, e.g. ``montecarlo.plant_rows(controller)``; the true state is
        checked against it after every plant step and ``violation_step`` (R,), ``violation_row`` (R,) (-1: none) and
        ``violations_per_step`` (steps,) int32 are added to the result.  A violation does not stop a run.

        ``goal``: (rows, 5) ``[A | b]`` or ``(A, b)``, e.g. ``montecarlo.goal_box(controller.goal)``; a run whose true
        state satisfies every row after a plant step, and whose QP of that step is solved, stops there (the reference's
        loops break at the goal): its ``final`` state is that state and the step's input is not applied.  A QP that is not
        solved at the same step is a failure, as in the reference.  ``arrival_step`` (R,) (-1: none) and
        ``arrivals_per_step`` (steps,) int32 are added to the result."""
        return self._closed_loop(1 if C is not None else 0, x_init, steps, A, B, C, L, None, x_ref, dt, l1, warm_start,
                                 xhat_init, None, None, want_traj, want_inputs, False, noise, monitor, goal, stream)

    def closed_loop_disturbance(self, x_init, steps: int, A, B, C, Bd, Cd, L1, L2, x_ref=None, Bd_plant=None,
                                Cd_plant=None, d_plant=None, xhat_init=None, dhat_init=None, dt: float = 0.2,
                                l1: float = 3.5, warm_start=True, want_traj: bool = False, want_inputs: bool = False,
                                want_dhat: bool = False, noise=None, monitor=None, goal=None, stream=None) -> dict:
        """Closed loops of the disturbance-estimating output-feedback controller (``MPCOutputFBWithDisturbance``,
        ``carmpc_closed_loop`` mode 2): the loop of ``closed_loop`` with a scalar disturbance estimate ``d^`` kept
        beside ``x^`` by the augmented observer (``Bd`` (4,), ``Cd`` (3,), gains ``L1`` (4, 3), ``L2`` (3,); no defaults,
        see ``carmpc_b200.observer``), and the QP of each run taking ``d^`` as its disturbance.  This handle's ``Gc`` must
        come from a controller with the same ``Bd`` (or be zero).  The plant gets a constant disturbance ``d_plant`` per
        run ((R,) float64 CUDA tensor, None: 0) through ``Bd_plant`` (4,) after its Euler step and ``Cd_plant`` (3,) in its
        output (None: zeros).  ``dhat_init``: (R,) CUDA tensor (None: 0).  ``warm_start``: 0 / 1 (True) / 2 as in
        ``closed_loop``.  Returns ``final`` (4, R), ``dhat`` (R,), ``fail_step`` (R,) int32, ``total_iters`` and
        optionally ``traj`` (steps, 4, R), ``inputs`` (steps, 2, R), ``dhat_traj`` (steps, R).  ``noise``, ``monitor`` and
        ``goal`` as in ``closed_loop`` (the measurement noise adds to ``C s + Cd_plant d_r``)."""

        def vec(a, n, name):
            v = _f64(a).ravel()
            if v.size != n:
                raise ValueError(f"{name} must have {n} entries")
            return v

        dm = _capi.DisturbanceModel()
        dm.Bd[:] = vec(Bd, 4, "Bd").tolist()
        dm.Cd[:] = vec(Cd, 3, "Cd").tolist()
        dm.L1[:] = vec(L1, 12, "L1 (4 x 3)").tolist()
        dm.L2[:] = vec(L2, 3, "L2").tolist()
        dm.Bd_plant[:] = vec(np.zeros(4) if Bd_plant is None else Bd_plant, 4, "Bd_plant").tolist()
        dm.Cd_plant[:] = vec(np.zeros(3) if Cd_plant is None else Cd_plant, 3, "Cd_plant").tolist()
        return self._closed_loop(2, x_init, steps, A, B, C, None, dm, x_ref, dt, l1, warm_start, xhat_init, dhat_init,
                                 d_plant, want_traj, want_inputs, want_dhat, noise, monitor, goal, stream)
