"""The bulk-async scan hands out its 1024-sample groups in an interleaved order when the row-order pilot sees the cost of
a sample vary along the index (ticket_group in csrc/membership.cu: 16 contiguous stripes, consecutive tickets in
different stripes).  The samples here are tensor grids in C order with x outermost, like config 2's, which the pilot
classifies that way (its costliest 1/16 of the index range is about 7x the cheapest), and uniform random samples, which
keep the index order.  Group counts around the stripe arithmetic - a multiple of the stripe count, one above and one
below it, neither, and ragged tails after the last whole group - must give the bits of the float64 kernel and of the C
oracle, through every staging geometry and through the fused sharded scan in both layouts (needs a B200)."""
import os

import numpy as np
import pytest

from conftest import GOLDEN
from test_sharded_gpu import _samples, _streams

pytestmark = pytest.mark.gpu

GEOMETRIES = [(256, 3, 1), (128, 3, 1), (128, 4, 1), (128, 2, 2), (128, 3, 2), (256, 2, 1), (128, 2, 1), (256, 2, 2)]
# (whole groups, samples after them); the bulk-async path takes calls of at least 64 groups
GROUP_COUNTS = [(64, 0), (65, 0), (79, 0), (80, 1), (100, 0), (111, 513), (127, 1023), (1000, 77)]


def _set():
    return np.load(os.path.join(GOLDEN, "terminal_sets", "RoadMultipleCarsEnv_30_1.5_0_0.npy"))


def _grid_samples(torch, n):
    """The first n points of a config-2-like grid (x outermost, 16 points on each other axis) spanning the whole x range."""
    from carmpc_b200.grids import materialise_grid
    k = -(-n // 4096)
    axes = [np.linspace(5.0, 55.0, k), np.linspace(-3.2, 3.2, 16), np.linspace(-0.42, 0.42, 16), np.linspace(-1.2, 5.2, 16)]
    return [t[:n].contiguous() for t in materialise_grid(axes, device="cuda")]


@pytest.mark.parametrize("samples", ["grid", "uniform"])
@pytest.mark.parametrize("groups,tail", GROUP_COUNTS)
def test_group_counts_around_the_stripes_give_the_oracles_bits(groups, tail, samples):
    import torch
    from carmpc_b200.batch import TerminalSetEvaluator
    from oracle import c_oracle
    Ab = _set()
    n = groups * 1024 + tail
    cols = _grid_samples(torch, n) if samples == "grid" else _samples(torch, n, seed=groups)
    want_bits, want_count = c_oracle.membership_bits(Ab, *[c.cpu().numpy() for c in cols])
    ref_bits, ref_count = TerminalSetEvaluator(Ab).contains_bits(*cols, mode=0)
    assert np.array_equal(ref_bits.cpu().numpy().view(np.uint32), want_bits) and int(ref_count.item()) == want_count
    for geometry in GEOMETRIES:
        ev = TerminalSetEvaluator(Ab)
        ev.set_staging(*geometry)
        ev.tune(*cols)                                      # the pilot picks the group order (and the row order)
        for _ in range(2):                                  # the work counter re-arms itself for the next launch
            bits, count = ev.contains_bits(*cols, mode=1)
            assert torch.equal(bits, ref_bits) and int(count.item()) == want_count, geometry


@pytest.mark.parametrize("layout", ["cyclic", "contiguous"])
@pytest.mark.parametrize("world,n", [(2, 2 * 79 * 1024 + 1024 + 300), (3, 3 * 66 * 1024 + 5), (2, 2 * 80 * 1024)])
def test_fused_sharded_scan_with_group_counts_around_the_stripes(world, n, layout):
    import torch
    from carmpc_b200.batch import TerminalSetEvaluator
    from carmpc_b200.sharding import PeerWindow, contains_bits_sharded, wait_sharded
    ev = TerminalSetEvaluator(_set())
    x, y, psi, v = _grid_samples(torch, n)
    want_bits, want_count = ev.contains_bits(x, y, psi, v, mode=0)
    want_bits, want_count = want_bits.clone(), int(want_count.item())
    ev.tune(x, y, psi, v)
    wins = PeerWindow.local_group(n, world, layout=layout)
    streams = _streams(torch, world)
    totals = [torch.zeros(1, dtype=torch.int64, device="cuda") for _ in range(world)]
    local = [[t[w.local_index("cuda")].contiguous() for t in (x, y, psi, v)] for w in wins]
    assert all(loc[0].numel() >= 64 * 1024 for loc in local)           # every rank's scan takes the bulk-async path
    torch.cuda.synchronize()
    for step in range(2):
        for r, w in enumerate(wins):
            with torch.cuda.stream(streams[r]):
                contains_bits_sharded(ev, w, *local[r], total=totals[r], defer_wait=True)
        for r, w in enumerate(wins):
            with torch.cuda.stream(streams[r]):
                wait_sharded(w, totals[r])
        torch.cuda.synchronize()
        for r, w in enumerate(wins):
            w.check()
            assert int(totals[r].item()) == want_count
            assert torch.equal(w.result_bits(), want_bits), f"rank {r} step {step}: gathered bitset differs"
