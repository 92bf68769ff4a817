"""Numpy restatement of the certificate checker kernel (carmpc_b200/csrc/qp_check.cu), for the tests.

Same problem form, same row space, same four columns per sample; the sums run in numpy's order, so the kernel agrees with
it to rounding, not bit for bit.
"""
import numpy as np


def check_numpy(H, F, G, Gx, lo, hi, lb, ub, x0, xref, status, u, cert, Gc=None, c=None):
    """x0 (B, 4), u (B, n), cert (B, R + n); returns (B, 4) like ``QPChecker.check``."""
    x0, u, cert = np.atleast_2d(x0), np.atleast_2d(u), np.atleast_2d(cert)
    B, n = u.shape
    R = G.shape[0]
    y, yb = cert[:, :R], cert[:, R:]
    terms = np.abs(x0[:, None, :] * Gx[None, :, :]).sum(2)                   # (B, R)
    s = x0 @ Gx.T
    if Gc is not None and c is not None:
        s = s + c[:, None] * Gc[None, :]
        terms = terms + np.abs(c[:, None] * Gc[None, :])
    out = np.full((B, 4), np.nan)
    acc, aacc = y @ G, np.abs(y) @ np.abs(G)
    with np.errstate(invalid="ignore", over="ignore"):
        # ---- status 0 ----
        gu, ga = u @ G.T, np.abs(u) @ np.abs(G).T
        his, los = hi[None, :] - s, lo[None, :] - s
        sc = np.maximum(1.0, ga)
        scb = np.maximum(1.0, np.abs(u))
        primal = np.max(np.maximum(0.0, np.maximum(gu - his, los - gu)) / sc, axis=1, initial=0.0)
        primal = np.maximum(primal, np.max(np.maximum(0.0, np.maximum(u - ub, lb - u)) / scb, axis=1, initial=0.0))
        hu, q = u @ H.T, (x0 - xref) @ F.T
        stat = np.abs(hu + q + acc + yb).max(1) / np.maximum(1.0, np.maximum(np.abs(hu).max(1), np.abs(q).max(1)))
        lmax = np.maximum(1.0, np.abs(cert).max(1))

        def sides(lam, up_inf, lo_inf, slack_up, slack_lo, scale):
            wrong = np.where((lam > 0) & up_inf, lam, 0.0) + np.where((lam < 0) & lo_inf, -lam, 0.0)
            cpl = np.where((lam > 0) & ~up_inf, lam * np.abs(slack_up), 0.0) + \
                np.where((lam < 0) & ~lo_inf, -lam * np.abs(slack_lo), 0.0)
            return wrong.max(1, initial=0.0), (np.nan_to_num(cpl, posinf=np.inf) / scale).max(1, initial=0.0)

        wg, cg = sides(y, np.isinf(hi)[None, :], np.isinf(lo)[None, :], his - gu, gu - los, sc)
        wb, cb = sides(yb, np.isinf(ub)[None, :], np.isinf(lb)[None, :], ub[None, :] - u, u - lb[None, :], scb)
        kkt = np.stack((primal, stat, np.maximum(wg, wb) / lmax, np.maximum(cg, cb) / lmax), axis=1)
        finite = np.isfinite(u).all(1) & np.isfinite(cert).all(1)
        kkt[~finite] = np.nan
        # ---- status 1 ----
        ybc = -acc
        res = np.abs(acc + yb).max(1) / np.maximum(aacc.max(1), np.finfo(float).tiny)
        box_abs = np.maximum(np.abs(ub), np.abs(lb))
        scale = np.where(aacc != 0, aacc * box_abs[None, :], 0.0).sum(1)
        bnd_b = np.where(ybc > 0, ub[None, :], np.where(ybc < 0, lb[None, :], 0.0))
        inf_b = (ybc != 0) & np.isinf(bnd_b)
        sup = np.where((ybc != 0) & ~inf_b, ybc * bnd_b, 0.0).sum(1)
        wrong = np.where(inf_b, np.abs(ybc), 0.0).sum(1)
        bnd = np.where(y > 0, hi[None, :], np.where(y < 0, lo[None, :], 0.0))
        inf_g = (y != 0) & (np.isinf(bnd) | np.isnan(y))
        live = (y != 0) & ~inf_g
        sup = sup + np.where(live, y * (bnd - s), 0.0).sum(1)
        scale = scale + np.where(live, np.abs(y) * (np.abs(bnd) + terms), 0.0).sum(1)
        wrong = wrong + np.where(inf_g, np.abs(y), 0.0).sum(1)
        farkas = np.stack((sup, scale, res, wrong), axis=1)
    out[status == 0] = kkt[status == 0]
    out[status == 1] = farkas[status == 1]
    return out
