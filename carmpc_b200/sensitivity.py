"""Batched MPC solutions as a differentiable torch layer.

``solve_differentiable(bq, x0, c)`` returns the optimal input sequences ``u_full`` (B, n) and objectives (B,) of one
certified solve, differentiable with respect to the states ``x0`` (4, B) and the per-sample disturbance ``c`` (B,).
The derivatives are exact on the critical region of each sample's certified active set (``BatchQP.sensitivity``,
``carmpc_qp_sensitivity``): no finite differences, one extra kernel pass, run only when an input requires grad.

A sample without a derivative (status != 0: infeasible or undecided) contributes NaN to the gradient when its upstream
gradient is non-zero and nothing when it is zero, so a loss that masks those states out has finite gradients and one that
does not is told.
"""
from __future__ import annotations

#: ``flags`` bits of ``BatchQP.sensitivity`` (carmpc.h, carmpc_qp_sensitivity)
DERIVATIVE = 1      # u* is differentiable here and the Jacobian is its derivative
WEAK = 2            # a row outside the active set is at its bound, or an active multiplier is ~0: one-sided derivative
DEPENDENT = 4       # linearly dependent active rows: the Jacobian comes from the independent subset
TOO_MANY_ROWS = 8   # more active rows than any solver certificate has: the Jacobian is NaN

_FUNCTION = None


def _certified_solve():
    global _FUNCTION
    if _FUNCTION is not None:
        return _FUNCTION
    import torch

    class CertifiedSolve(torch.autograd.Function):
        @staticmethod
        def forward(ctx, x0, c, bq, seed):
            x0 = x0.detach().contiguous()
            c = None if c is None else c.detach().contiguous()
            out = bq.solve(x0, c=c, want_u_full=True, want_certificate=True, seed=seed)
            ctx.has_c = c is not None
            if ctx.needs_input_grad[0] or ctx.needs_input_grad[1]:
                s = bq.sensitivity(x0, out, c=c)
                ctx.save_for_backward(s["jac"], s["grad_objective"], out["status"])
            return out["u_full"], out["objective"]

        @staticmethod
        def backward(ctx, g_u, g_v):
            jac, grad_v, status = ctx.saved_tensors
            bad = status != 0
            asked = (g_u != 0).any(dim=1) | (g_v != 0)
            # samples without a derivative: zeroed first (0 * NaN would poison the einsum), NaN where a gradient was asked
            g = torch.einsum("bn,bnk->bk", g_u.masked_fill(bad[:, None], 0.0), jac.masked_fill(bad[:, None, None], 0.0))
            g = g + g_v.masked_fill(bad, 0.0)[:, None] * grad_v.masked_fill(bad[:, None], 0.0)
            g = g.masked_fill((bad & asked)[:, None], float("nan"))
            return g[:, :4].t().contiguous(), (g[:, 4].contiguous() if ctx.has_c else None), None, None

    _FUNCTION = CertifiedSolve
    return _FUNCTION


def solve_differentiable(bq, x0, c=None, seed=None):
    """One certified solve of ``bq`` (a ``BatchQP`` with the polish) as a torch autograd function.

    ``x0``: (4, B) float64 CUDA tensor, ``c``: optional (B,) float64 CUDA tensor (the disturbance of
    ``MPCOutputFBWithDisturbance``), ``seed``: optional lattice seeds as in ``BatchQP.solve``.  Returns ``(u_full (B, n),
    objective (B,))``; both carry gradients to ``x0`` and ``c`` when those require grad."""
    return _certified_solve().apply(x0, c, bq, seed)
