"""TSP 2-opt local search (FusedTSPEnv.local_search -> co_tsp_two_opt) against the reference's numba implementation
(rl4co/envs/routing/tsp/local_search.py), recorded in tests/golden/ls_tsp.npz by make_golden_ls.py, and
against the plain-torch oracle (oracle/local_search_oracle.py).  The algorithm is fp32 adds and compares only, so every
comparison is exact: tours and move counts."""

import ctypes

import numpy as np
import pytest
import torch

from conftest import GOLDEN_DIR, golden_case
from oracle import local_search_oracle as O

MAX_ITERATIONS = (0, 1, 7, 1000)


def _cases():
    z = np.load(f"{GOLDEN_DIR}/ls_tsp.npz")
    return sorted({k.split("/")[0] for k in z.files})


def _case(tag):
    z = np.load(f"{GOLDEN_DIR}/ls_tsp.npz")
    inst, outs, _ = golden_case(z, tag)
    locs = inst["locs"] if inst is not None else outs["locs"]
    want = {mi: (outs[f"out{mi}"].long(), outs[f"moves{mi}"]) for mi in MAX_ITERATIONS}
    return locs, outs["tours"].long(), want


def _td(locs):
    from rl4co_b200.tensordict import TensorDict

    return TensorDict({"locs": locs}, batch_size=[locs.shape[0]])


def _random_tours(B, n, seed, device="cpu"):
    g = torch.Generator().manual_seed(seed)
    return torch.stack([torch.randperm(n, generator=g) for _ in range(B)]).to(device)


def _kernel(locs, tours, max_iterations):
    from rl4co_b200 import native

    moves = torch.empty(tours.shape[0], dtype=torch.int32, device=tours.device)
    out = native.tsp_two_opt(locs, tours, max_iterations, moves=moves)
    return out, moves


# ----------------------------------------------------------------------------- CPU


@pytest.mark.parametrize("tag", _cases())
def test_oracle_reproduces_reference_fixture(tag):
    locs, tours, want = _case(tag)
    for mi, (w_tours, w_moves) in want.items():
        got, moves = O.local_search(locs, tours, mi)
        assert torch.equal(got, w_tours), (tag, mi)
        assert torch.equal(moves, w_moves), (tag, mi)


def test_lattice_fixture_exercises_ties():
    z = np.load(f"{GOLDEN_DIR}/ls_tsp.npz")
    assert all(int(z[f"lattice{n}/tied_scans"]) > 0 for n in (50, 100))


def test_abi_rejects_bad_arguments_without_a_gpu():
    from rl4co_b200 import native

    L = native.lib()
    fake = ctypes.c_void_p(256)
    assert L.co_tsp_two_opt(None, fake, fake, None, 4, 10, 5, None) == -1
    assert L.co_tsp_two_opt(fake, None, fake, None, 4, 10, 5, None) == -1
    assert L.co_tsp_two_opt(fake, fake, None, None, 4, 10, 5, None) == -1
    assert L.co_tsp_two_opt(fake, fake, fake, None, -1, 10, 5, None) == -1
    assert L.co_tsp_two_opt(fake, fake, fake, None, 4, -1, 5, None) == -1
    assert L.co_tsp_two_opt(fake, fake, fake, None, 4, 10, -1, None) == -1
    assert L.co_tsp_two_opt(fake, fake, fake, None, 4, 1025, 5, None) == -2
    assert b"1025" in L.co_last_error_string()
    assert L.co_tsp_two_opt(fake, fake, fake, None, 0, 10, 5, None) == 0  # B == 0: nothing to do


def test_cpu_tensors_raise():
    from rl4co_b200 import native
    from rl4co_b200.envs import FusedTSPEnv

    locs = torch.rand(3, 10, 2)
    with pytest.raises(native.NativeLibraryError):
        FusedTSPEnv.local_search(_td(locs), _random_tours(3, 10, 0))


def test_rejected_inputs():
    from rl4co_b200.envs import FusedTSPEnv, get_env

    locs = torch.rand(3, 10, 2)
    td = _td(locs)
    td.set("distances", torch.rand(3, 10, 10))
    with pytest.raises(NotImplementedError):
        FusedTSPEnv.local_search(td, _random_tours(3, 10, 0))
    with pytest.raises(ValueError):
        FusedTSPEnv.local_search(_td(locs), _random_tours(3, 9, 0))
    with pytest.raises(ValueError):
        FusedTSPEnv.local_search(_td(locs), _random_tours(2, 10, 0))
    with pytest.raises(ValueError):
        FusedTSPEnv.local_search(_td(locs), torch.arange(10))
    with pytest.raises(NotImplementedError):
        FusedTSPEnv.local_search(_td(torch.rand(1, 1025, 2)), _random_tours(1, 1025, 0))
    cvrp = get_env("cvrp", generator_params=dict(num_loc=10))
    with pytest.raises(NotImplementedError):
        cvrp.local_search(cvrp.reset(batch_size=[2]), torch.zeros(2, 12, dtype=torch.int64))


# ----------------------------------------------------------------------------- GPU


@pytest.mark.gpu
@pytest.mark.parametrize("tag", _cases())
def test_kernel_reproduces_reference_fixture(tag):
    from rl4co_b200.envs import FusedTSPEnv

    locs, tours, want = _case(tag)
    locs, tours = locs.cuda(), tours.cuda()
    for mi, (w_tours, w_moves) in want.items():
        got, moves = _kernel(locs, tours, mi)
        assert torch.equal(got.cpu(), w_tours), (tag, mi)
        assert torch.equal(moves.cpu(), w_moves), (tag, mi)
        assert torch.equal(FusedTSPEnv.local_search(_td(locs), tours, max_iterations=mi).cpu(), w_tours)
    # the reference's converged tours are fixed points
    got, moves = _kernel(locs, want[1000][0].cuda(), 1000)
    assert torch.equal(got.cpu(), want[1000][0]) and int(moves.abs().sum()) == 0


@pytest.mark.gpu
@pytest.mark.parametrize("n, B, max_iterations", [(100, 2048, 1000), (200, 256, 1000), (1000, 4, 50)])
def test_kernel_matches_oracle_seeded(n, B, max_iterations):
    g = torch.Generator().manual_seed(n)
    locs = torch.rand(B, n, 2, generator=g)
    tours = _random_tours(B, n, n + 1)
    got, moves = _kernel(locs.cuda(), tours.cuda(), max_iterations)
    want, w_moves = O.local_search(locs, tours, max_iterations, device="cuda")
    assert torch.equal(got.cpu(), want)
    assert torch.equal(moves.cpu(), w_moves)
    assert int(moves.min()) > 0


@pytest.mark.gpu
def test_n1000_converges_to_a_2opt_local_optimum():
    B, n = 4, 1000
    g = torch.Generator().manual_seed(5)
    locs = torch.rand(B, n, 2, generator=g)
    tours = _random_tours(B, n, 6)
    got, moves = _kernel(locs.cuda(), tours.cuda(), 100000)
    got = got.cpu()
    assert torch.equal(got.sort(1).values, torch.arange(n).expand(B, n))
    assert (O.tour_length(locs, got) <= O.tour_length(locs, tours)).all()
    change = O.scan_changes(O.distance_matrix(locs), got)
    assert float(change.min()) >= -1e-6
    assert (moves > 0).all()


@pytest.mark.gpu
def test_input_unmodified_and_bad_rows_passed_through():
    from rl4co_b200.envs import FusedTSPEnv

    B, n = 8, 50
    locs = torch.rand(B, n, 2, generator=torch.Generator().manual_seed(1)).cuda()
    tours = _random_tours(B, n, 2, "cuda")
    tours[3, 7] = n
    tours[5, 0] = -1
    before = tours.clone()
    got, moves = _kernel(locs, tours, 1000)
    assert torch.equal(tours, before)
    assert torch.equal(got[[3, 5]], before[[3, 5]])
    assert moves[3].item() == -1 and moves[5].item() == -1
    ok = [b for b in range(B) if b not in (3, 5)]
    assert (moves[ok] > 0).all()
    want, w_moves = O.local_search(locs.cpu(), before.cpu(), 1000)
    assert torch.equal(got.cpu(), want) and torch.equal(moves.cpu(), w_moves)
    assert torch.equal(FusedTSPEnv.local_search(_td(locs), before), got)


@pytest.mark.gpu
def test_int32_noncontiguous_and_empty_inputs():
    from rl4co_b200.envs import FusedTSPEnv

    B, n = 16, 60
    locs = torch.rand(B, n, 2, generator=torch.Generator().manual_seed(3)).cuda()
    tours = _random_tours(B, n, 4, "cuda")
    want = FusedTSPEnv.local_search(_td(locs), tours)
    wide = torch.zeros(B, 2 * n, dtype=torch.int32, device="cuda")
    wide[:, ::2] = tours.int()
    got = FusedTSPEnv.local_search(_td(locs), wide[:, ::2])
    assert got.dtype == torch.int64 and torch.equal(got, want)
    locs_nc = torch.zeros(B, n, 4, device="cuda")
    locs_nc[..., 1:3] = locs
    assert torch.equal(FusedTSPEnv.local_search(_td(locs_nc[..., 1:3]), tours, num_threads=4), want)
    empty = FusedTSPEnv.local_search(_td(torch.rand(0, n, 2, device="cuda")), torch.zeros(0, n, dtype=torch.int64,
                                                                                          device="cuda"))
    assert empty.shape == (0, n) and empty.dtype == torch.int64


@pytest.mark.gpu
def test_deterministic():
    B, n = 512, 100
    locs = torch.rand(B, n, 2, generator=torch.Generator().manual_seed(8)).cuda()
    tours = _random_tours(B, n, 9, "cuda")
    a, ma = _kernel(locs, tours, 1000)
    b, mb = _kernel(locs, tours, 1000)
    assert torch.equal(a, b) and torch.equal(ma, mb)
