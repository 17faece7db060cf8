"""2-opt local search benchmark: FusedTSPEnv.local_search (co_tsp_two_opt) at the sizes rl4co users run it.

    python tools/bench_two_opt.py [--steps 3] [--warmup 1] [--out profiles/r03_two_opt.json]

Workloads: TSP-20 and TSP-100 at B = 65 536, TSP-500 at B = 4 096, TSP-1000 at B = 512, all from random-permutation
tours (the most work per instance: every scan finds a move until the tour converges), and TSP-100 at B = 65 536 from
the project's greedy rollout tours on name-seeded weights (the "AM + 2-opt" evaluation step: few moves per tour).
Each call runs to convergence (max_iterations = 1000, the reference's default).

Per workload: ms per call (CUDA events around `steps` calls after `warmup` calls; every call reads the same input and
writes a new output), the moves applied (sum over rows), and pair evaluations per second, where one call evaluates
sum_rows scans * (N-1)(N-2)/2 pairs and scans = min(moves + 1, max_iterations).  The card name and power limit are read
in the same run.  The reference (tsp/local_search.py, numba on the host CPU) is timed on a bounded sample of the same
inputs only when numba imports and the staged reference is present; otherwise it is reported as not measured.
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

MAX_ITERATIONS = 1000
WORKLOADS = [  # name, N, B, tours
    ("tsp20_random", 20, 65536, "random"),
    ("tsp100_random", 100, 65536, "random"),
    ("tsp500_random", 500, 4096, "random"),
    ("tsp1000_random", 1000, 512, "random"),
    ("tsp100_greedy", 100, 65536, "greedy"),
]
REF_SAMPLE_ROWS = {20: 1024, 100: 256, 500: 16, 1000: 4}


def card_info() -> dict:
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        info["nvidia_smi"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "not read"
    except (OSError, subprocess.TimeoutExpired):
        info["nvidia_smi"] = "not read"
    return info


def random_tours(B, n, seed, device):
    g = torch.Generator(device=device).manual_seed(seed)
    return torch.rand(B, n, generator=g, device=device).argsort(1)


def greedy_tours(locs):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from conftest import name_seeded_weights

    from rl4co_b200.envs import get_env
    from rl4co_b200.policy import FusedAttentionModelPolicy

    n = locs.shape[1]
    env = get_env("tsp", generator_params=dict(num_loc=n))
    pol = FusedAttentionModelPolicy(env_name="tsp").to(locs.device).eval()
    pol.load_state_dict({k: v.to(locs.device) for k, v in name_seeded_weights(pol.state_dict(), 3).items()})
    from rl4co_b200.tensordict import TensorDict

    with torch.inference_mode():
        td = env.reset(TensorDict({"locs": locs}, batch_size=[locs.shape[0]], device=locs.device))
        return pol(td, env, phase="test", decode_type="greedy")["actions"].clone()


def reference_ms_per_instance(locs, tours):
    """Host time of the reference's numba local_search on a bounded sample (first call compiles: it is untimed)."""
    try:
        import numba  # noqa: F401
    except ImportError:
        return "not measured (numba is not installed on this host)"
    from oracle import ref_standin

    if not ref_standin.reference_available():
        return "not measured (the staged reference is not present)"
    ref = ref_standin.load()
    import importlib

    LS = importlib.import_module("rl4co.envs.routing.tsp.local_search")
    rows = REF_SAMPLE_ROWS[locs.shape[1]]
    l, t = locs[:rows].cpu(), tours[:rows].cpu()
    LS.local_search(ref.TensorDict({"locs": l[:2]}, batch_size=[2]), t[:2], max_iterations=MAX_ITERATIONS)
    t0 = time.perf_counter()
    LS.local_search(ref.TensorDict({"locs": l}, batch_size=[rows]), t, max_iterations=MAX_ITERATIONS)
    return {"rows": rows, "ms_per_instance": (time.perf_counter() - t0) * 1e3 / rows,
            "threads": min(os.cpu_count() or 1, 32)}


def run(name, n, B, kind, steps, warmup, ref_timing):
    from rl4co_b200 import native
    from rl4co_b200.envs import FusedTSPEnv
    from rl4co_b200.tensordict import TensorDict

    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev).manual_seed(n)
    locs = torch.rand(B, n, 2, generator=g, device=dev)
    tours = random_tours(B, n, n + 1, dev) if kind == "random" else greedy_tours(locs)
    td = TensorDict({"locs": locs}, batch_size=[B])
    moves = torch.empty(B, dtype=torch.int32, device=dev)
    native.tsp_two_opt(locs, tours, MAX_ITERATIONS, moves=moves)
    for _ in range(warmup):
        FusedTSPEnv.local_search(td, tours, MAX_ITERATIONS)
    torch.cuda.synchronize()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(steps):
        FusedTSPEnv.local_search(td, tours, MAX_ITERATIONS)
    end.record()
    end.synchronize()
    ms = start.elapsed_time(end) / steps
    m = moves.long()
    scans = torch.clamp(m + 1, max=MAX_ITERATIONS)
    pairs = int(scans.sum()) * (n - 1) * (n - 2) // 2
    res = {"workload": name, "N": n, "B": B, "tours": kind, "max_iterations": MAX_ITERATIONS, "ms_per_call": ms,
           "moves_sum": int(m.sum()), "moves_mean": float(m.float().mean()), "moves_max": int(m.max()),
           "pair_evals_per_call": pairs, "pair_evals_per_s": pairs / (ms * 1e-3), "steps": steps, "warmup": warmup}
    if ref_timing:
        res["reference_host"] = reference_ms_per_instance(locs, tours)
    print(json.dumps(res), flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--only", nargs="*", default=None, help="workload names")
    ap.add_argument("--no-reference", action="store_true")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_two_opt.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_two_opt needs a CUDA device")
    card = card_info()
    print(json.dumps(card), flush=True)
    results = [run(name, n, B, kind, a.steps, a.warmup, not a.no_reference)
               for name, n, B, kind in WORKLOADS if a.only is None or name in a.only]
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump({"card": card, "results": results}, f, indent=1)
    print(f"wrote {a.out}")


if __name__ == "__main__":
    main()
