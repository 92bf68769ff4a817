"""CPU restatement of the closed loops' noise (carmpc_closed_loop_stochastic): Philox4x64-10 and the Box-Muller step in
numpy, and the noisy loop of the three modes with exact QPs, built on ``oracle/carmpc_oracle.py`` and
``tests/disturbance_oracle.py`` (both used unchanged).

TEST INFRASTRUCTURE ONLY.  The generator is checked against ``numpy.random.Philox`` (the same generator; it increments
its 256-bit counter before generating, so block c is ``Philox(key, counter=c - 1).random_raw(4)``).
"""
from __future__ import annotations

import numpy as np

from oracle.carmpc_oracle import plant_step

_U64 = np.uint64
M0, M1 = _U64(0xD2E7470EE14C6C93), _U64(0xCA5A826395121157)
W0, W1 = _U64(0x9E3779B97F4A7C15), _U64(0xBB67AE8584CAA73B)
_LO32 = _U64(0xFFFFFFFF)
_S32, _S11 = _U64(32), _U64(11)


def _mulhilo(m, b):
    """(hi, lo) of the 128-bit products m * b (m a uint64 scalar, b a uint64 array), from 32-bit halves."""
    ml, mh = m & _LO32, m >> _S32
    bl, bh = b & _LO32, b >> _S32
    ll, hl, lh, hh = ml * bl, mh * bl, ml * bh, mh * bh
    cross = (ll >> _S32) + (hl & _LO32) + lh          # < 2^64: no wrap
    return hh + (hl >> _S32) + (cross >> _S32), m * b


def philox4x64_10(c0, c1, c2, c3, k0, k1):
    """Philox4x64-10 of counters (c0..c3) under key (k0, k1); all arguments broadcast as uint64 arrays."""
    c = [np.array(v, dtype=np.uint64, copy=True) for v in np.broadcast_arrays(c0, c1, c2, c3)]
    k0 = np.array(k0, dtype=np.uint64)
    k1 = np.array(k1, dtype=np.uint64)
    with np.errstate(over="ignore"):
        for r in range(10):
            if r:
                k0, k1 = k0 + W0, k1 + W1
            hi0, lo0 = _mulhilo(M0, c[0])
            hi1, lo1 = _mulhilo(M1, c[2])
            c = [hi1 ^ c[1] ^ k0, lo1, hi0 ^ c[3] ^ k1, lo0]
    return c


def box_muller(a, b):
    """Two normals from two uint64 words: ua = ((a >> 11) + 1) 2^-53, ub = (b >> 11) 2^-53."""
    ua = ((a >> _S11) + _U64(1)).astype(np.float64) * 2.0 ** -53
    ub = (b >> _S11).astype(np.float64) * 2.0 ** -53
    r = np.sqrt(-2.0 * np.log(ua))
    t = np.pi * (2.0 * ub)
    return r * np.cos(t), r * np.sin(t)


def normals(seed, runs, step, stream):
    """(len(runs), 4) standard normals of the global run ids ``runs`` at ``step``; stream 0 process, 1 measurement."""
    runs = np.asarray(runs, dtype=np.uint64)
    x = philox4x64_10(runs, _U64(step), _U64(stream), _U64(0), _U64(seed), _U64(0))
    z0, z1 = box_muller(x[0], x[1])
    z2, z3 = box_muller(x[2], x[3])
    return np.stack((z0, z1, z2, z3), axis=1)


def numpy_philox_block(counter, key):
    """The same block from numpy.random.Philox (counter as four 64-bit words, least significant first)."""
    c = sum(int(v) << (64 * i) for i, v in enumerate(counter))
    prev = (c - 1) % (1 << 256)
    words = np.array([(prev >> (64 * i)) & ((1 << 64) - 1) for i in range(4)], dtype=np.uint64)
    bg = np.random.Philox(key=np.array([int(key[0]), int(key[1])], dtype=np.uint64), counter=words)
    return bg.random_raw(4)


def noisy_closed_loop(mode, A, B, C, L, x_init, steps, solve, Lw, Lv, seed, first_run=0, dist=None, monitor=None):
    """The loop of carmpc_closed_loop_stochastic for mode 0 (state feedback), 1 (output feedback, gain L) or 2
    (``dist`` = (Bd, Cd, L1, L2, Bd_plant, Cd_plant, d_plant)).  ``solve(x (B, 4), d (B,)) -> (u0 (B, 2), status)``.
    ``monitor``: (rows, 5) [A | b] checked with numpy's A @ s <= b.  Returns a dict of final, fail_step, traj (steps, R,
    4), inputs (steps, R, 2), dhat, dhat_traj and, with a monitor, violation_step, violation_row, violations_per_step."""
    from disturbance_oracle import disturbance_observer_step
    A, B = np.asarray(A, dtype=float), np.asarray(B, dtype=float)
    x = np.array(x_init, dtype=float)
    R = len(x)
    if mode == 2:
        Bd, Cd, L1, L2, Bp, Cp, dr = (np.asarray(a, dtype=float) for a in dist)
        C = np.asarray(C, dtype=float)
        L1 = L1.reshape(4, 3)
    elif mode == 1:
        C, L1 = np.asarray(C, dtype=float), np.asarray(L, dtype=float).reshape(4, 3)
        Bd, Cd, L2, Bp, Cp, dr = np.zeros(4), np.zeros(3), np.zeros(3), np.zeros(4), np.zeros(3), np.zeros(R)
    xhat = x.copy()
    dhat = np.zeros(R)
    u = np.zeros((R, 2))
    fail = np.full(R, -1, dtype=np.int32)
    traj, ulog, dlog = np.zeros((steps, R, 4)), np.zeros((steps, R, 2)), np.zeros((steps, R))
    vstep = np.full(R, -1, dtype=np.int32)
    vrow = np.full(R, -1, dtype=np.int32)
    per_step = np.zeros(steps, dtype=np.int32)
    for k in range(steps):
        idx = np.flatnonzero(fail < 0)
        ids = first_run + idx
        s = plant_step(x[idx], u[idx])
        if mode == 2:
            s = s + dr[idx, None] * Bp[None, :]
        s = s + normals(seed, ids, k, 0) @ np.asarray(Lw, dtype=float).T
        x[idx] = s
        if monitor is not None:
            ok = s @ monitor[:, :4].T <= monitor[None, :, 4]
            bad = ~ok.all(1)
            first = np.argmin(ok, axis=1)
            per_step[k] = int(bad.sum())
            new = bad & (vstep[idx] < 0)
            vstep[idx[new]] = k
            vrow[idx[new]] = first[new]
        v = normals(seed, ids, k, 1) @ np.asarray(Lv, dtype=float).T
        if mode == 0:
            est = s + v
        else:
            y = s @ C.T + dr[idx, None] * Cp[None, :] + v[:, :3]
            xhat[idx], dhat[idx] = disturbance_observer_step(A, B, C, Bd, Cd, L1, L2, xhat[idx], dhat[idx], u[idx], y)
            est = xhat[idx]
        if len(idx):
            u_new, st = solve(est, dhat[idx])
            failed = st != 0
            fail[idx[failed]] = k
            u[idx[~failed]] = u_new[~failed]
        traj[k], ulog[k], dlog[k] = x, u, dhat
    out = {"final": x, "fail_step": fail, "traj": traj, "inputs": ulog, "dhat": dhat, "dhat_traj": dlog}
    if monitor is not None:
        out.update(violation_step=vstep, violation_row=vrow, violations_per_step=per_step)
    return out
