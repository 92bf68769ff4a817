"""CPU model of how many float32 screen rows a 128-sample warp tile of the config-2 scan runs, per row-block schedule.

    python tools/scan_row_model.py [--every 41] [SCHEDULE ...]          e.g.  8   2,6,8   1,3,4,8   4,4,8

``screen32`` (csrc/membership.cu) runs the rows in blocks and, before each block, leaves the tile when every one of its
128 samples is already surely outside (float32 min margin below -beta(p)).  A schedule lists the block sizes; its last
entry repeats.  The model restates the library's row order (the sparsity sort of ``carmpc_polytope_create``, then the
greedy cover of ``tune_row_order`` over the same 65,536 strided pilot samples of the grid), evaluates every row of every
sample of every ``--every``-th tile of the 10^8-point grid in float64, and counts the rows the tile runs before its exit
(the padded row count when it never exits).  Decisions do not depend on the schedule; only the rows spent on them do.
The grid is in C order with x outermost, so the first half of the tiles is x < 30 m.
"""
from __future__ import annotations

import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from carmpc_b200.grids import config2_axes, grid_size   # noqa: E402

TERMINAL_SET = os.path.join(ROOT, "terminal_sets", "RoadMultipleCarsEnv_30_1.5_0_0.npy")
TILE = 128


def grid_points(axes, idx):
    dims = [len(a) for a in axes]
    stride = grid_size(axes)
    out = []
    for a, d in zip(axes, dims):
        stride //= d
        out.append(np.asarray(a, dtype=np.float64)[(idx // stride) % d])
    return np.stack(out, axis=1)


def sparsity_order(Ab):
    """carmpc_polytope_create: fewest non-zero coefficients first, then by pattern, stable."""
    pat = [sum(1 << k for k in range(4) if row[k] != 0.0) for row in Ab]
    return sorted(range(len(Ab)), key=lambda r: (bin(pat[r]).count("1"), pat[r]))


def greedy_order(Ab, pts):
    """tune_row_order: the row that rejects most of the pilot samples still alive comes next; the rest keeps its order."""
    rows = len(Ab)
    viol = ~(pts @ Ab[:, :4].T <= Ab[:, 4])
    alive = viol[viol.any(axis=1)]
    order, used = [], np.zeros(rows, bool)
    while len(alive) and len(order) < rows:
        cnt = np.where(used, -1, alive.sum(axis=0))
        best = int(np.argmax(cnt))                        # first of the largest, as the strict '>' of the library
        if cnt[best] <= 0:
            break
        used[best] = True
        order.append(best)
        alive = alive[~alive[:, best]]
    return order + [r for r in range(rows) if not used[r]]


def screen_beta(Ab):
    """beta0, beta1 of carmpc_polytope_create (surely outside: margin < -(beta0 + beta1 |p|_1))."""
    l1max = np.abs(Ab[:, :4]).sum(axis=1).max()
    fin = np.isfinite(Ab[:, 4])
    bmax = np.abs(Ab[fin, 4]).max() if fin.any() else 0.0
    u8, tiny = 8.0 * 2.0 ** -24, 2.0 ** -149
    return u8 * bmax * 1.000001 + l1max * tiny + 1e-37, u8 * l1max * 1.000001 + 1e-37


def tile_need(Ab, beta, pts):
    """Rows a tile must run before every sample is surely outside (inf: some sample never is)."""
    margin = Ab[:, 4] - pts @ Ab[:, :4].T                 # (samples, rows), rows in device order
    out = margin < -(beta[0] + beta[1] * np.abs(pts).sum(axis=1, keepdims=True))
    first = np.where(out.any(axis=1), out.argmax(axis=1) + 1, np.inf)
    return first.reshape(-1, TILE).max(axis=1)


def rows_run(need, schedule, rows_padded):
    bounds, r, k = [], 0, 0
    while r < rows_padded:
        r = min(r + schedule[min(k, len(schedule) - 1)], rows_padded)
        bounds.append(r)
        k += 1
    bounds = np.array(bounds, dtype=np.float64)
    pos = np.searchsorted(bounds, need)                   # first block boundary at or after the need
    return np.where(pos < len(bounds), bounds[np.minimum(pos, len(bounds) - 1)], rows_padded)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("schedules", nargs="*", default=["8", "2,6,8", "1,3,4,8", "4,4,8"])
    ap.add_argument("--every", type=int, default=41, help="model every k-th 128-sample tile of the grid")
    args = ap.parse_args()
    Ab = np.load(TERMINAL_SET)
    Ab = Ab[sparsity_order(Ab)]
    axes = config2_axes()
    n = grid_size(axes)
    n_sub = min(1 << 16, n)
    pilot = grid_points(axes, np.arange(n_sub, dtype=np.int64) * (n // n_sub))
    Ab = Ab[greedy_order(Ab, pilot)]
    beta = screen_beta(Ab)
    rows_padded = (len(Ab) + 7) & ~7
    tiles = np.arange(0, n // TILE, args.every, dtype=np.int64)
    need = np.concatenate([tile_need(Ab, beta, grid_points(axes, (t[:, None] * TILE + np.arange(TILE)).ravel()))
                           for t in np.array_split(tiles, max(1, len(tiles) // 2048))])
    low = tiles * TILE < n // 2
    print(f"# {len(tiles)} tiles (1 in {args.every} of {n // TILE}), {len(Ab)} rows padded to {rows_padded}")
    print(f"{'row-block schedule':<22} {'rows/tile, all':>15} {'x < 30':>8} {'x >= 30':>8}")
    for s in args.schedules:
        sched = [int(k) for k in s.split(",")]
        r = rows_run(need, sched, rows_padded)
        label = ", ".join(str(k) for k in sched) + ", ..."
        print(f"{label:<22} {r.mean():>15.2f} {r[low].mean():>8.2f} {r[~low].mean():>8.2f}")


if __name__ == "__main__":
    main()
