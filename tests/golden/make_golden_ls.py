"""Generate tests/golden/ls_tsp.npz (tests/test_two_opt.py) by executing rl4co's OWN, unmodified 2-opt local search
(rl4co/envs/routing/tsp/local_search.py, numba) through oracle/ref_standin.py, like make_golden.py does for the other
fixtures, whose helpers it uses.  Needs numba and the reference source:

    python tests/golden/make_golden_ls.py
"""

from __future__ import annotations

import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)

from make_golden import TensorDict, npy, seeded_instances  # noqa: E402


def _looped_two_opt(LS, dist, tours, max_iterations, count_ties=False):
    """_two_opt_python's loop (tsp/local_search.py:73-81) row by row around the reference's own two_opt_once, counting
    the moves it applies; with `count_ties`, also the scans whose smallest change < -1e-6 is attained by 2+ pairs."""
    out, moves, ties = tours.copy(), np.zeros(len(tours), np.int32), 0
    for b in range(len(tours)):
        t = out[b]
        it, min_change = 0, -1.0
        while min_change < -1e-6 and it < max_iterations:
            if count_ties:
                ties += _min_change_attained_twice(dist[b], t)
            min_change = LS.two_opt_once(dist[b], t, 0)
            moves[b] += min_change != 0.0
            it += 1
    return out, moves, ties


def _min_change_attained_twice(d, t):
    n = len(t)
    i, j = np.triu_indices(n, 1)
    keep = (i >= 1) & (i <= n - 2)
    i, j = i[keep], j[keep]
    prev, node_i, node_j, nxt = t[i - 1], t[i], t[j], t[(j + 1) % n]
    ok = (prev != node_j) & (nxt != node_i)
    change = ((d[prev, node_j] + d[node_i, nxt]) - d[prev, node_i]) - d[node_j, nxt]
    change = change[ok]
    return int(change.size > 0 and change.min() < -1e-6 and (change == change.min()).sum() >= 2)


def two_opt_fixture():
    """tests/test_two_opt.py: the reference's TSP local_search (tsp/local_search.py:16-81, numba) from random-permutation
    tours at max_iterations 0 / 1 / 7 / 1000, with per-row move counts.  Uniform instances are stored as seeds + CRC-32;
    the lattice instances (coordinates k / 8) are stored, and must contain scans with tied minimum changes."""
    import importlib

    LS = importlib.import_module("rl4co.envs.routing.tsp.local_search")
    out = {}
    cases = [(f"tsp{n}", n, batch, 600 + n) for n, batch in ((3, 64), (4, 64), (20, 64), (50, 48), (100, 48), (200, 32))]
    cases += [(f"lattice{n}", n, batch, 700 + n) for n, batch in ((50, 48), (100, 32))]
    for tag, n, batch, seed in cases:
        if tag.startswith("lattice"):
            g = torch.Generator().manual_seed(seed)
            locs = torch.randint(0, 8, (batch, n, 2), generator=g).float() / 8
            out[f"{tag}/locs"] = npy(locs)
        else:
            _, td0 = seeded_instances(out, tag, "tsp", n, batch, seed)
            locs = td0["locs"]
        g = torch.Generator().manual_seed(seed + 1)
        tours = torch.stack([torch.randperm(n, generator=g) for _ in range(batch)])
        out[f"{tag}/tours"] = npy(tours).astype(np.int16)
        dist = npy(LS.get_distance_matrix(locs)) + 1e9 * np.eye(n, dtype=np.float32)[None]
        ties = 0
        for mi in (0, 1, 7, 1000):
            res = LS.local_search(TensorDict({"locs": locs}, batch_size=[batch]), tours.clone(), max_iterations=mi)
            looped, moves, t = _looped_two_opt(LS, dist, npy(tours).astype(np.uint16), mi,
                                               count_ties=tag.startswith("lattice") and mi == 1000)
            ties += t
            assert (looped.astype(np.int64) == npy(res)).all(), (tag, mi)
            assert mi != 1000 or moves.max() < mi, "not converged"
            out[f"{tag}/out{mi}"] = npy(res).astype(np.int16)
            out[f"{tag}/moves{mi}"] = moves
        if tag.startswith("lattice"):
            assert ties > 0, f"{tag}: no scan with a tied minimum change"
            out[f"{tag}/tied_scans"] = np.int64(ties)
    return out


def main():
    data = two_opt_fixture()
    path = os.path.join(HERE, "ls_tsp.npz")
    np.savez_compressed(path, **data)
    print(f"ls_tsp: {len(data)} arrays, {os.path.getsize(path) / 1024:.0f} KiB")


if __name__ == "__main__":
    main()
