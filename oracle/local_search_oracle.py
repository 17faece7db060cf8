"""TEST INFRASTRUCTURE ONLY -- never imported by the product package.

rl4co's TSP 2-opt (rl4co/envs/routing/tsp/local_search.py) restated in plain torch, one vectorised scan per iteration
across the batch, with the reference's arithmetic and rules:

  * distances: get_distance_matrix(locs) (rl4co/utils/ops.py:93-100) on the CPU, plus 1e9 on the diagonal (:38);
  * one scan = two_opt_once (:47-70): pairs i = 1..n-2, j = i+1..n-1, skipped when tour[i-1] == tour[j] or
    tour[(j+1) % n] == tour[i]; change = ((D[prev, j] + D[i, next]) - D[prev, i]) - D[j, next] in fp32; the first pair
    in (i, j) order with the strictly smallest change < 0; tour[p..q] reversed only if delta < -1e-6 in double;
  * _two_opt_python (:73-81): scans repeat until one applies no move or max_iterations scans have run.

No numba: it runs wherever torch does.  The distance matrix is always built on the CPU (the reference's numbers);
the scans may run on a CUDA device, where the fp32 adds and the first-index argmin are the same.
"""

from __future__ import annotations

import torch

#: rows per block of the vectorised scan: bounds the [rows, n, n] temporaries
_ELEMS_PER_BLOCK = 1 << 23


def distance_matrix(locs: torch.Tensor) -> torch.Tensor:
    """[B, n, 2] -> [B, n, n] fp32: local_search.py:34-38 (get_distance_matrix + 1e9 * eye), on the CPU."""
    locs = locs.detach().to("cpu", torch.float32)
    d = (locs[..., :, None, :] - locs[..., None, :, :]).norm(p=2, dim=-1)
    return d + 1e9 * torch.eye(locs.shape[-2], dtype=torch.float32)


def scan_changes(D: torch.Tensor, tour: torch.Tensor) -> torch.Tensor:
    """All changes of one two_opt_once scan: [B, n-2, n] fp32 indexed [b, i-1, j]; +inf where the pair is not
    considered (j <= i or the skip rule)."""
    B, n = tour.shape
    P = D.gather(1, tour[:, :, None].expand(B, n, n)).gather(2, tour[:, None, :].expand(B, n, n))  # D[b, t[x], t[y]]
    ar = torch.arange(n, device=tour.device)
    nxt = torch.roll(ar, -1)  # (j + 1) % n
    i = ar[1:n - 1]
    new1 = P[:, i - 1, :]                                  # D[prev_i, node_j]
    new2 = P[:, i, :][:, :, nxt]                           # D[node_i, next_j]
    old1 = P[:, i - 1, i]                                  # D[prev_i, node_i]
    old2 = P[:, ar, nxt]                                   # D[node_j, next_j]
    change = ((new1 + new2) - old1[:, :, None]) - old2[:, None, :]
    valid = (ar[None, :] > i[:, None])[None] \
        & (tour[:, i - 1, None] != tour[:, None, :]) & (tour[:, None, nxt] != tour[:, i, None])
    return torch.where(valid, change, torch.full_like(change, float("inf")))


def _scan(D: torch.Tensor, tour: torch.Tensor):
    """two_opt_once on every row: (delta [B] fp32, p [B], q [B]); delta = +inf when no pair has change < 0."""
    B, n = tour.shape
    change = scan_changes(D, tour)
    change = torch.where(change < 0, change, torch.full_like(change, float("inf")))
    flat = change.reshape(B, -1).argmin(1)  # first minimum in (i, j) order
    delta = change.reshape(B, -1).gather(1, flat[:, None]).squeeze(1)
    return delta, flat // n + 1, flat % n


def _reverse(tour: torch.Tensor, p: torch.Tensor, q: torch.Tensor) -> torch.Tensor:
    ar = torch.arange(tour.shape[1], device=tour.device)[None]
    inside = (ar >= p[:, None]) & (ar <= q[:, None])
    return tour.gather(1, torch.where(inside, p[:, None] + q[:, None] - ar, ar.expand_as(tour)))


def local_search(locs: torch.Tensor, tours: torch.Tensor, max_iterations: int = 1000, device=None):
    """(tours [B, n] int64, moves [B] int32) on the CPU; moves = moves applied per row, -1 for a row holding a node
    index outside [0, n) (left unchanged).  `device` runs the scans there."""
    dev = torch.device("cpu") if device is None else torch.device(device)
    tours = tours.detach().to(dev, torch.int64).clone()
    B, n = tours.shape
    moves = torch.zeros(B, dtype=torch.int32, device=dev)
    bad = ((tours < 0) | (tours >= n)).any(1)
    moves[bad] = -1
    if n < 3 or max_iterations <= 0:
        return tours.cpu(), moves.cpu()
    D_all = distance_matrix(locs)
    rows_per_block = max(1, _ELEMS_PER_BLOCK // (n * n))
    good = (~bad).nonzero().squeeze(1).cpu()
    for s in range(0, good.numel(), rows_per_block):
        rows = good[s:s + rows_per_block].to(dev)
        D = D_all[rows.cpu()].to(dev)
        t = tours[rows]
        m = torch.zeros(rows.numel(), dtype=torch.int32, device=dev)
        active = torch.arange(rows.numel(), device=dev)
        for _ in range(max_iterations):
            delta, p, q = _scan(D[active], t[active])
            apply = delta.double() < -1e-6
            active = active[apply]
            if active.numel() == 0:
                break
            t[active] = _reverse(t[active], p[apply], q[apply])
            m[active] += 1
        tours[rows] = t
        moves[rows] = m
    return tours.cpu(), moves.cpu()


def tour_length(locs: torch.Tensor, tours: torch.Tensor) -> torch.Tensor:
    """Closed-tour length in float64 (for checks that a tour got no longer)."""
    x = locs.detach().cpu().double().gather(1, tours.cpu()[..., None].expand(*tours.shape, 2))
    return (x - x.roll(-1, 1)).norm(dim=-1).sum(-1)
