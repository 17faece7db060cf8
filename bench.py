#!/usr/bin/env python
"""bench.py -- node-selections/sec of the AM rollout hot path (BASELINE.json metric).

Workloads (`--workload`, named in config.workload; default = north_star's headline):
  tsp100  TSP-100 AttentionModel greedy rollout, 65 536 instances PER GPU (weak scaling, BASELINE metric
          "node-selections/sec TSP-100 AM rollout @1/2/4/8 B200")
  c2      TSP-50 greedy, 4 096 instances per GPU            (BASELINE configs[1])
  c3      CVRP-50 sampling (in-kernel Philox), 4 096 per GPU (BASELINE configs[2])
  c4      TSP-100 POMO: 1 024 instances IN TOTAL x 8 dihedral augmentations x 100 starts, 6-layer
          instance-norm encoder, no graph context; instances sharded over the ranks (strong scaling)
  c5      CVRP-100 REINFORCE training step: 65 536 instances IN TOTAL sharded over the ranks (strong):
          sampling rollout + differentiable log-likelihood + loss + backward + gradient all-reduce +
          Adam, mean baseline over the GLOBAL batch through one {sum,count} all-reduce

  value : the step with inputs RESIDENT in HBM.
          rollout workloads: FusedAttentionModelDecoder._precompute_cache (one tcgen05 3xTF32 GEMM) + co_rollout
          (persistent kernel: context + glimpse + pointer + tanh/mask/log-softmax + selection + env step +
          incremental tour length, all T steps) from the resident encoder output;
          c4: cache GEMM + query-batched co_rollout (100 starts share K/V/L) + POMO max reductions;
          c5: the whole training step from the resident batch.
  e2e   : the call a user makes, from HOST buffers: pinned-host instance data -> H2D, policy / pomo_step /
          reinforce_step, D2H of the step's result.
  --impl reference : the reference's OWN policy (unmodified rl4co files, oracle/ref_runner.py) on the host CPU
          cores, same metric / workload on a bounded sample, all the host cores it can use.

Timing: CUDA events on the launching stream, barrier + synchronize on both sides, max over ranks.  The
resident inputs of the default workload (13.4 GB cache + 3.4 GB embeddings per rank) are far larger than the
126 MB L2, so no explicit L2 flush is needed between iterations (stated in config).  Outside the timed region a
parity gate re-checks a 1 024-row slice of the timed batch against the CPU oracle (`parity_gate` in the line).

--dump-outputs DIR writes what the last timed `value` step returned (rank 0) as DIR/<name>.npy, so that two
builds run with the same arguments (and therefore the same seeded inputs) can be compared output for output.
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# the benchmark may run from a read-only checkout: no bytecode caches in the tree, here or in the CPU-arm workers
sys.dont_write_bytecode = True
os.environ["PYTHONDONTWRITEBYTECODE"] = "1"

import torch  # noqa: E402

UNIT = "selections/s"
E = 128

WORKLOADS = {
    "tsp100": dict(env="tsp", n=100, batch=65536, per_gpu=True, decode="greedy", kind="rollout", policy={},
                   metric="node-selections/sec TSP-100 AM rollout", label="TSP-100 AM greedy rollout"),
    "c2": dict(env="tsp", n=50, batch=4096, per_gpu=True, decode="greedy", kind="rollout", policy={},
               metric="node-selections/sec TSP-50 AM rollout", label="TSP-50 AM greedy rollout"),
    "c3": dict(env="cvrp", n=50, batch=4096, per_gpu=True, decode="sampling", kind="rollout", policy={},
               metric="node-selections/sec CVRP-50 AM sampling rollout", label="CVRP-50 AM sampling rollout"),
    "c4": dict(env="tsp", n=100, batch=1024, per_gpu=False, decode="multistart_greedy", kind="pomo",
               policy=dict(num_encoder_layers=6, normalization="instance", use_graph_context=False),
               metric="node-selections/sec TSP-100 POMO 8-aug x 100-start", label="TSP-100 POMO 8 aug x 100 starts"),
    "c5": dict(env="cvrp", n=100, batch=65536, per_gpu=False, decode="sampling", kind="train", policy={},
               metric="node-selections/sec CVRP-100 AM REINFORCE step", label="CVRP-100 AM REINFORCE training step"),
}


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=5)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--workload", default="tsp100", choices=sorted(WORKLOADS))
    p.add_argument("--batch", type=int, default=None, help="override the workload's batch (per GPU or total, see workload)")
    p.add_argument("--cpu-batch", type=int, default=None, help="bounded CPU sample (instances per process)")
    p.add_argument("--micro-batch", type=int, default=8192, help="c5: instances per differentiable chunk")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-parity-gate", action="store_true")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="write the last timed step's outputs as DIR/<name>.npy (at most 64 MB in all)")
    args = p.parse_args()
    if args.steps < 1:
        p.error("--steps must be at least 1")
    return args


# ------------------------------------------------------------------------------------ output dump
DUMP_BYTES = 64 << 20


def _dump_dtype(t):
    """float32, or float64 where float32 would not hold the values exactly (float64 data, integers >= 2^24)."""
    if t.dtype == torch.float64:
        return torch.float64
    if t.dtype.is_floating_point or t.numel() == 0:
        return torch.float32
    return torch.float32 if int(t.abs().max()) < 2 ** 24 else torch.float64


def dump_outputs(res, out_dir, budget=DUMP_BYTES):
    """Write every tensor (and scalar) of a step's result as out_dir/<name>.npy.  When the whole set exceeds
    `budget`, the arrays that share the batch (leading) dimension are restricted to a fixed seeded sample of
    rows, the same rows for every array, and the sorted row indices go to out_dir/sample_rows.npy."""
    import numpy as np

    arrays = {}
    for k, v in res.items():
        if isinstance(v, torch.Tensor):
            arrays[k] = v.detach()
        elif isinstance(v, (int, float)) and not isinstance(v, bool):
            arrays[k] = torch.tensor(float(v), dtype=torch.float64)
    arrays = {k: v.to(_dump_dtype(v)) for k, v in arrays.items()}
    total = sum(v.numel() * v.element_size() for v in arrays.values())
    if total > budget:
        rows = max(v.shape[0] for v in arrays.values() if v.dim() > 0)
        batched = [k for k, v in arrays.items() if v.dim() > 0 and v.shape[0] == rows]
        fixed = total - sum(arrays[k].numel() * arrays[k].element_size() for k in batched)
        per_row = sum(arrays[k][0].numel() * arrays[k].element_size() for k in batched)
        keep = (budget - fixed - rows * 8) // per_row
        idx = torch.randperm(rows, generator=torch.Generator().manual_seed(0))[:keep].sort().values
        for k in batched:
            arrays[k] = arrays[k][idx.to(arrays[k].device)]
        arrays["sample_rows"] = idx.to(torch.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), v.cpu().numpy())
    return sorted(arrays)


# ------------------------------------------------------------------------------------ clocks
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100", "-i",
                 str(index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def mark(self):
        return time.time()

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons, power = [], None, set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        inside = [r for r in self.rows if t0 - 0.05 <= r[0] <= t1 + 0.05]
        extended = False
        if not inside and self.rows:  # timed region shorter than the 100 ms sampling period: nearest samples
            extended = True
            inside = sorted(self.rows, key=lambda r: min(abs(r[0] - t0), abs(r[0] - t1)))[:2]
        for ts, line in inside:
            parts = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(parts[0])); mx = float(parts[1]); power.append(float(parts[2]))
            except Exception:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        out = {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
               "samples": len(sm), "power_w_max": max(power) if power else None}
        if extended:
            out["note"] = "timed region shorter than the sampling period: the two samples nearest to it"
        return out


# ------------------------------------------------------------------------------------ common
def policy_kwargs(wl):
    kw = dict(embed_dim=128, num_heads=8, num_encoder_layers=3, normalization="batch", tanh_clipping=10.0)
    kw.update(wl["policy"])
    return kw


def algorithmic_bytes_per_instance(env_name, N, T, S=1):
    """SURVEY.md section 8d: read K,V,L + node table rows, graph ctx, coords (+demand); write
    actions (int64) + logp (f32) per step and reward + log-likelihood per trajectory (S per instance)."""
    b = N * 4 * E * 4 + E * 4 + N * 8 + S * (T * (8 + 4) + 4 + 4)
    if env_name == "cvrp":
        b += (N - 1) * 4
    return b


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f)["hbm_gbs"], "measured"
    except Exception:
        return 6650.0, "fallback"


def ncu_traffic(workload, instances):
    """dram__bytes_read+write of the dominant kernel from the committed `ncu --set full` capture, per instance,
    scaled to this launch (the kernel streams each instance exactly once)."""
    try:
        with open(os.path.join(ROOT, "profiles", "rollout_traffic.json")) as f:
            d = json.load(f)
        if workload in d:
            return d[workload]["dram_bytes_per_instance"] * instances
        if workload == "tsp100" and "dram_bytes_per_instance" in d:
            return d["dram_bytes_per_instance"] * instances
    except Exception:
        pass
    return None


# ------------------------------------------------------------------------------------ CPU arm
def cpu_reference(wl, batch, steps, warmup, multi_process=True):
    from oracle import ref_runner

    dk = {}
    if wl["kind"] == "pomo":
        dk = {"num_starts": wl["n"]}
    return ref_runner.time_reference(wl["env"], wl["n"], batch, wl["decode"], steps=steps, warmup=warmup,
                                     policy_kwargs=wl["policy"], decode_kwargs=dk, multi_process=multi_process,
                                     augment=8 if wl["kind"] == "pomo" else 0, train=wl["kind"] == "train")


def cpu_sample_batch(wl, override):
    if override:
        return override
    return {"rollout": 1024 if wl["n"] >= 100 else 2048, "pomo": 2, "train": 256}[wl["kind"]]


def cpu_baseline_obj(wl, r):
    scope = {"rollout": "policy-forward (encoder + decode loop + reward)",
             "pomo": "dihedral-8 augmentation + policy-forward multistart greedy",
             "train": "policy-forward sampling + REINFORCE loss + backward + Adam"}[wl["kind"]]
    return {"value": r["value"], "unit": UNIT, "cores": r["cores_used"], "kind": r["kind"],
            "sample": f"{wl['label']}, {scope}; {r['batch_per_step']} instances per step, torch CPU fp32, "
                      f"{r['layout']} on a {r['host_cores']}-core host (better of 1 process with its best thread count "
                      f"and P processes x T threads over all cores)",
            "single_process": r["single"], "multi_process": r.get("multi")}


def run_reference(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_reference(wl, cpu_sample_batch(wl, args.cpu_batch), steps=max(1, args.steps), warmup=min(args.warmup, 1))
    line = {
        "impl": "reference", "metric": wl["metric"], "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": max(1, args.steps), "warmup": min(args.warmup, 1), "ms_per_step": r["ms_per_step"],
        "higher_is_better": True, "scaling": "weak" if wl["per_gpu"] else "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": f"{wl['label']} (the reference's own rl4co files on the host CPU)",
                   "batch_per_step": r["batch_per_step"], "scope": "policy-forward"},
        "cpu_baseline": cpu_baseline_obj(wl, r),
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------ parity gate
def parity_gate(wl, policy, td_dev, h, res, rows=1024):
    """Outside the timed region: a `rows`-row slice of the batch that was just timed, against the CPU oracle
    (decode path from the GPU's own encoder output): teacher-forced log-likelihood / reward (<= 1e-5 relative,
    2e-5 absolute floor per log-prob) and, for greedy, the number of free-running trajectories that differ
    (near-tie flips).  Rows are the first `rows` instances (S = 1 workloads)."""
    from oracle import am_rollout_oracle as O

    env_name = wl["env"]
    rows = min(rows, h.shape[0])
    W = {k: v.detach().cpu() for k, v in policy.state_dict().items()}
    inst = {k: td_dev[k][:rows].cpu() for k in ("locs", "demand") if k in td_dev.keys()}
    if env_name == "cvrp":
        inst["depot"], inst["locs"] = inst["locs"][:, 0], inst["locs"][:, 1:]
    hh = h[:rows].cpu()
    acts = res["actions"][:rows].cpu()
    T = int(res["steps"][:rows].max().item())
    acts = acts[:, :T]
    torch.set_num_threads(min(16, os.cpu_count() or 1))
    ugc = wl["policy"].get("use_graph_context", True)
    with torch.inference_mode():
        ref = O.rollout(W, env_name, inst, hh, actions=acts, use_graph_context=ugc, faithful_copies=False)
        free = O.rollout(W, env_name, inst, hh, "greedy", use_graph_context=ugc, faithful_copies=False) \
            if wl["decode"] == "greedy" else None
    lp_gpu, lp_ref = res["logprobs"][:rows, :T].cpu(), ref["logprobs"]
    rw_gpu, rw_ref = res["reward"][:rows].cpu(), ref["reward"]
    lp_err = (lp_gpu - lp_ref).abs()
    lp_ok = bool((lp_err <= 1e-5 * lp_ref.abs() + 2e-5).all())
    rw_rel = ((rw_gpu - rw_ref).abs() / rw_ref.abs()).max().item()
    out = {"rows": rows, "checker": "oracle port (oracle/am_rollout_oracle.py), teacher-forced on the GPU's actions",
           "max_abs_logp_err": lp_err.max().item(), "max_rel_reward_err": rw_rel, "logp_ok": lp_ok,
           "reward_ok": rw_rel <= 1e-5, "ok": lp_ok and rw_rel <= 1e-5}
    if free is not None:
        same = (free["actions"][:, :T] == acts).all(1) if free["actions"].shape[1] >= T else torch.zeros(rows, dtype=torch.bool)
        out["free_running_rows_differing"] = int((~same).sum())
        out["free_running_flip_fraction"] = float((~same).float().mean())
    return out


# ------------------------------------------------------------------------------------ GPU arm
def run_ours(args, wl):
    import torch.distributed as dist

    from rl4co_b200 import native
    from rl4co_b200.distributed import shard_bounds
    from rl4co_b200.envs import get_env
    from rl4co_b200.policy import FusedAttentionModelPolicy
    from rl4co_b200.tensordict import TensorDict

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback for the product path)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    native.lib()

    env_name, n, kind = wl["env"], wl["n"], wl["kind"]
    total = args.batch if args.batch else wl["batch"]
    if wl["per_gpu"]:
        B, global_batch = total, total * world
    else:
        lo, hi = shard_bounds(total, rank, world)
        B, global_batch = hi - lo, total
    N = n + (1 if env_name == "cvrp" else 0)

    torch.manual_seed(0)
    policy = FusedAttentionModelPolicy(env_name=env_name, **policy_kwargs(wl)).to(dev)
    policy = policy.train() if kind == "train" else policy.eval()
    env = get_env(env_name, generator_params=dict(num_loc=n), check_solution=False)
    torch.manual_seed(1234 + rank)
    td_host = env.generator(B)
    pinned = {k: td_host[k].pin_memory() for k in td_host.keys()}
    stats = torch.zeros(2, dtype=torch.float64, device=dev)
    side = torch.cuda.Stream(device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def baseline_allreduce(reward):
        """REINFORCE mean baseline over the GLOBAL batch: {sum, count} in f64 (north_star).  The next step does
        not depend on it, so the NCCL all-reduce runs on a side stream and overlaps the next step's kernels
        (round 1 had it stream-serialised behind every rollout: every rank waited for the slowest rank)."""
        stats.zero_()
        native.reward_stats(reward, stats)
        if world > 1:
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                dist.all_reduce(stats)
        return stats

    def join_side():
        if world > 1:
            torch.cuda.current_stream().wait_stream(side)

    rollout_ev = []
    host_out = {}

    def to_host(name, t):
        if name not in host_out or host_out[name].shape != t.shape:
            host_out[name] = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
        host_out[name].copy_(t, non_blocking=True)

    def h2d():
        return TensorDict({k: v.to(dev, non_blocking=True) for k, v in pinned.items()}, batch_size=[B])

    # ------------------------------------------------------------------ workload-specific steps
    gate_ctx = {}
    if kind == "rollout":
        with torch.inference_mode():
            td_dev = env.reset(TensorDict({k: v.to(dev) for k, v in pinned.items()}, batch_size=[B]))
            h, _ = policy.encoder(td_dev)
            h = h.contiguous()
        mode = native.SELECT_GREEDY if "greedy" in wl["decode"] else native.SELECT_SAMPLE_PHILOX

        def value_step(record=False):
            with torch.inference_mode():
                cached = policy.decoder._precompute_cache(h)
                if record:
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                res = native.rollout(env_name, mode, cached.rollout_cache, cached.graph_context_or_none,
                                     cached.q_placeholder, cached.w_capacity, td_dev["locs"],
                                     td_dev["demand"] if env_name == "cvrp" else None,
                                     td_dev["vehicle_capacity"].reshape(-1) if env_name == "cvrp" else None, B, N,
                                     tanh_clipping=10.0, seed=1, node_emb=h if env_name == "tsp" else None,
                                     w_first=cached.w_first)
                if record:
                    e1.record()
                    rollout_ev.append((e0, e1))
                baseline_allreduce(res["reward"])
            return res

        def e2e_step():
            with torch.inference_mode():
                td = env.reset(h2d())
                out = policy(td, env, phase="test", decode_type=wl["decode"], **({"seed": 1} if "sampling" in wl["decode"] else {}))
                baseline_allreduce(out["reward"])
                for k in ("actions", "reward", "log_likelihood"):
                    to_host(k, out[k])
                join_side()
                torch.cuda.current_stream().synchronize()  # the results are on the host when the step returns
            return ("actions", "reward", "log_likelihood")

        gate_ctx = dict(td=td_dev, h=h)
        S_kernel, kernel_name, scope = 1, "co::rollout_kernel", \
            "precompute_cache GEMM + persistent rollout kernel from resident encoder output"
    elif kind == "pomo":
        from rl4co_b200.ops import StateAugmentation, unbatchify
        from rl4co_b200.reinforce import pomo_step

        n_aug, n_start = 8, n
        with torch.inference_mode():
            td_dev = env.reset(TensorDict({k: v.to(dev) for k, v in pinned.items()}, batch_size=[B]))
            td_aug = StateAugmentation(num_augment=n_aug)(td_dev)
            h, _ = policy.encoder(td_aug)
            h = h.contiguous()

        def value_step(record=False):
            with torch.inference_mode():
                cached = policy.decoder._precompute_cache(h, first_table=True)
                if record:
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                res = native.rollout(env_name, native.SELECT_GREEDY, cached.rollout_cache, None, cached.q_placeholder,
                                     None, td_aug["locs"], None, None, n_aug * B, N, num_starts=n_start,
                                     forced_start=True, num_loc=n, tanh_clipping=10.0)
                if record:
                    e1.record()
                    rollout_ev.append((e0, e1))
                r = unbatchify(res["reward"], (n_aug, n_start))  # pomo/model.py:103-136
                res["max_aug_reward"] = r.max(-1)[0].max(1)[0]
            return res

        def e2e_step():
            td = env.reset(h2d())
            out = pomo_step(policy, env, td, num_augment=n_aug, num_starts=n_start, phase="test")
            with torch.inference_mode():
                to_host("reward", out["reward"])
                to_host("max_aug_reward", out["max_aug_reward"])
                torch.cuda.current_stream().synchronize()
            return ("reward", "max_aug_reward")

        S_kernel, kernel_name, scope = n_start, "co::rollout_ms_kernel", \
            "precompute_cache GEMM + query-batched rollout kernel (100 starts share K/V/L) + POMO max reductions"
    else:  # train
        from rl4co_b200.reinforce import get_reinforce_baseline, reinforce_step

        opt = torch.optim.Adam(policy.parameters(), lr=1e-4)
        bl = get_reinforce_baseline("mean")
        td_dev = env.reset(TensorDict({k: v.to(dev) for k, v in pinned.items()}, batch_size=[B]))
        step_no = [0]

        def value_step(record=False, td=None):
            step_no[0] += 1
            return reinforce_step(policy, env, td_dev if td is None else td, bl, opt, seed=step_no[0],
                                  micro_batch=args.micro_batch, matmul_precision="medium")

        def e2e_step():
            out = value_step(td=env.reset(h2d()))
            to_host("loss", out["loss"].reshape(1))
            to_host("reward_mean", out["reward"].mean().reshape(1))
            torch.cuda.current_stream().synchronize()
            return ("loss", "reward_mean")

        S_kernel, kernel_name, scope = 1, "co::rollout_kernel", \
            ("whole REINFORCE step from the resident batch: sampling rollout (persistent kernel) + differentiable "
             "teacher-forced log-likelihood + loss + backward + gradient all-reduce + Adam; autograd GEMMs at "
             "float32_matmul_precision('medium') like the reference trainer (rl4co/utils/trainer.py:89-90)")

    # ---- warm-up (the clock sampler starts here so that nvidia-smi is already streaming when timing begins)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    for _ in range(max(args.warmup, 3)):
        res = value_step()
    join_side()
    torch.cuda.synchronize()
    if kind == "train":
        sel_per_step_rank = float(res["actions"].numel()) if "steps" not in res else float(res["steps"].sum().item())
    else:
        sel_per_step_rank = float(res["steps"].sum().item())  # exact number of (decode -> select -> env.step) iterations

    # ---- timed: value
    launch0 = native.LAUNCH_COUNT
    barrier()
    t_mark0 = sampler.mark() if sampler else 0
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        res = value_step(record=True) if kind != "train" else value_step()
    join_side()
    ev1.record()
    barrier()
    t_mark1 = sampler.mark() if sampler else 0
    ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop(t_mark0, t_mark1) if sampler else None
    n_launch = native.LAUNCH_COUNT - launch0
    dumped = dump_outputs(res, args.dump_outputs) if args.dump_outputs and rank == 0 else None
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    sel = torch.tensor([sel_per_step_rank], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(sel)
    ms_total = t.item()
    sel_total_per_step = sel.item()
    value = sel_total_per_step * args.steps / (ms_total * 1e-3)
    if kind == "train":
        torch.cuda.synchronize()
        k_ms_avg = res["rollout_events"][0].elapsed_time(res["rollout_events"][1]) if "rollout_events" in res else float("nan")
    else:
        k_ms = sorted(a.elapsed_time(b) for a, b in rollout_ev)
        k_ms_avg = sum(k_ms) / len(k_ms)

    # ---- timed: e2e
    e2e = None
    if not args.no_e2e:
        for _ in range(2):
            e2e_step()
        barrier()
        launch1 = native.LAUNCH_COUNT
        ev0.record()
        for _ in range(args.steps):
            keys = e2e_step()
        ev1.record()
        barrier()
        e2e_launches = native.LAUNCH_COUNT - launch1
        t2 = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t2, op=dist.ReduceOp.MAX)
        h2d_b = sum(v.numel() * v.element_size() for v in pinned.values())
        d2h_b = sum(host_out[k].numel() * host_out[k].element_size() for k in keys)
        e2e = {"value": sel_total_per_step * args.steps / (t2.item() * 1e-3), "unit": UNIT,
               "h2d_bytes_per_step": h2d_b, "d2h_bytes_per_step": d2h_b, "ms_per_step": t2.item() / args.steps,
               "gpu_launches": e2e_launches, "d2h": list(keys),
               "scope": {"rollout": "policy(td_host, env): H2D + encoder + cache GEMM + rollout + D2H(actions,reward,ll)",
                         "pomo": "pomo_step(td_host): H2D + dihedral-8 + 6-layer encoder + cache GEMM + multistart rollout + "
                                 "max reductions + D2H(reward[B,8,100], max_aug_reward)",
                         "train": "reinforce_step(td_host): H2D + full training step + D2H(loss, mean reward)"}[kind]}

    # ---- parity gate (outside the timed region, rank 0)
    gate = None
    if rank == 0 and kind == "rollout" and not args.no_parity_gate:
        try:
            gate = parity_gate(wl, policy, gate_ctx["td"], gate_ctx["h"], res)
        except Exception as exc:  # the gate must never hide the measurement; it reports its own failure
            gate = {"ok": False, "error": repr(exc)}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_kind = measured_peaks()
    inst_kernel = B * (8 if kind == "pomo" else 1)
    T_avg = sel_per_step_rank / (inst_kernel * S_kernel)
    roofline = None
    if kind != "train":
        bytes_per_launch = algorithmic_bytes_per_instance(env_name, N, T_avg, S_kernel) * inst_kernel
        achieved = bytes_per_launch / (k_ms_avg * 1e-3) / 1e9
        roofline = {"bound": "hbm", "kernel": kernel_name, "achieved": achieved, "peak": peak, "unit": "GB/s",
                    "frac": achieved / peak, "peak_source": f"{peak_kind} (MEASURED_PEAKS.json hbm_gbs)",
                    "traffic": ncu_traffic(args.workload, inst_kernel), "kernel_ms": k_ms_avg,
                    "algorithmic_bytes_per_launch": bytes_per_launch,
                    "kernel_share_of_step": k_ms_avg * args.steps / ms_total,
                    "cycles_per_selection_per_sm": (k_ms_avg * 1e-3 * (clocks["sm_mhz"] or 1965.0) * 1e6 * 148
                                                    / sel_per_step_rank) if clocks else None,
                    "note": "latency/issue-bound on-chip loop (one instance per SM); HBM roofline shown as required, "
                            "see DESIGN.md 4.1"}

    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        try:
            r = cpu_reference(wl, cpu_sample_batch(wl, args.cpu_batch), steps=2, warmup=1)
            cpu_baseline = cpu_baseline_obj(wl, r)
        except Exception as exc:
            cpu_baseline = {"value": None, "unit": UNIT, "cores": 0, "kind": "unavailable", "sample": repr(exc)}

    line = {
        "metric": wl["metric"], "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_total / args.steps, "higher_is_better": True,
        "scaling": "weak" if wl["per_gpu"] else "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{wl['label']}, " + (f"batch {B} per GPU" if wl["per_gpu"] else f"{global_batch} instances sharded over {world} GPU(s)"),
                   "workload_key": args.workload, "global_batch": global_batch, "nodes": N,
                   "parallelism": f"dp{world} (instances sharded, no data-path collective; "
                                  + ("baseline {sum,count} + gradient all-reduce" if kind == "train" else "baseline {sum,count} all-reduce on a side stream") + ")",
                   "value_scope": scope,
                   "l2_policy": "resident inputs per rank exceed the 126 MB L2; no flush needed",
                   "policy": f"AttentionModelPolicy E=128 H=8 {policy_kwargs(wl)} random-init seed 0"},
        "clocks": clocks, "e2e": e2e, "gpu_launches": n_launch, "roofline": roofline, "cpu_baseline": cpu_baseline,
        "selections_per_step": sel_total_per_step, "parity_gate": gate,
    }
    if dumped is not None:
        line["dumped_outputs"] = {"dir": args.dump_outputs, "arrays": dumped}
    if kind == "train":
        line["train_step"] = {"sampling_phase_ms": k_ms_avg, "micro_batch": args.micro_batch,
                              "chunks": res.get("chunks"), "loss": float(res["loss"]),
                              "collectives": "NCCL all-reduce {sum,count} f64 (baseline) + one flat gradient all-reduce (2.8 MB)"}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, wl)
    else:
        run_ours(args, wl)


if __name__ == "__main__":
    main()
