"""Small end-to-end run of every kernel family for compute-sanitizer (memcheck / racecheck / initcheck)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from rl4co_b200 import native
from rl4co_b200.envs import get_env
from rl4co_b200.policy import FusedAttentionModelPolicy
from rl4co_b200.reinforce import pomo_step

dev = torch.device("cuda:0")
CASES = (("tsp", 20), ("cvrp", 20), ("sdvrp", 20), ("tsp", 50), ("cvrp", 100), ("tsp", 100))
if os.environ.get("SAN_ONLY"):
    CASES = tuple(c for c in CASES if c[0] == os.environ["SAN_ONLY"])
for env_name, n in CASES:
    torch.manual_seed(0)
    env = get_env(env_name, generator_params=dict(num_loc=n), check_solution=True)
    pol = FusedAttentionModelPolicy(env_name=env_name, num_encoder_layers=1).to(dev).eval()
    with torch.inference_mode():
        td = env.reset(env.generator(300).to(dev))
        for dt, kw in (("greedy", {}), ("sampling", {"seed": 1}), ("multistart_greedy", {"num_starts": 3})):
            out = pol(td, env, decode_type=dt, **kw)
        out = pol(td, env, decode_type="greedy", fused_rollout=False)   # stepping kernels
        pol(td, env, actions=out["actions"])                             # evaluate mode
    print(env_name, n, "ok", out["reward"].mean().item())
# large-M GEMM path (pipe) + generic
a = torch.randn(20000, 128, device=dev); w = torch.randn(384, 128, device=dev)
hi, lo = native.split_tf32(w)
native.gemm_tf32x3(a, hi, lo, bias=torch.randn(384, device=dev), relu=True)
a = torch.randn(300, 512, device=dev); w = torch.randn(128, 512, device=dev)
hi, lo = native.split_tf32(w)
native.gemm_tf32x3(a, hi, lo, residual=torch.randn(300, 128, device=dev))
torch.cuda.synchronize()
print("gemm ok")
# orienteering: stepping kernels only (co_op_step / co_op_action_mask / co_op_reward)
env = get_env("op", generator_params=dict(num_loc=20), check_solution=True)
pol = FusedAttentionModelPolicy(env_name="op", num_encoder_layers=1).to(dev).eval()
with torch.inference_mode():
    for kw in (dict(decode_type="greedy"), dict(decode_type="sampling"), dict(decode_type="sampling", fused_rollout=False)):
        out = pol(env.reset(env.generator(300).to(dev)), env, **kw)
print("op ok", out["reward"].mean().item())
env = get_env("pctsp", generator_params=dict(num_loc=20), check_solution=True)
pol = FusedAttentionModelPolicy(env_name="pctsp", num_encoder_layers=1).to(dev).eval()
with torch.inference_mode():
    for kw in (dict(decode_type="greedy"), dict(decode_type="sampling"), dict(decode_type="sampling", fused_rollout=False)):
        out = pol(env.reset(env.generator(300).to(dev)), env, **kw)
print("pctsp ok", out["reward"].mean().item())
# training-step attention kernels (forward, dQ, dK/dV) with a mask and strided key / value views; instance norm
from rl4co_b200 import attention_train as AT

torch.manual_seed(1)
q = torch.randn(6, 131, 128, device=dev, requires_grad=True)
cache = torch.randn(6, 101, 512, device=dev, requires_grad=True)
mask = torch.rand(6, 131, 101, device=dev) < 0.5
mask[..., 0] = True
AT.attention(q, cache[..., :128], cache[..., 128:256], mask).square().sum().backward()
qkv = torch.randn(5, 100, 384, device=dev, requires_grad=True)
AT.self_attention_packed(qkv).sum().backward()
native.instance_norm(torch.randn(9, 100, 128, device=dev), torch.ones(128, device=dev), torch.zeros(128, device=dev))
torch.cuda.synchronize()
print("attention / norm ok")
# 2-opt local search: random tours to convergence, a row with an out-of-range node, a capped TSP-1000 run
from rl4co_b200.envs import FusedTSPEnv
from rl4co_b200.tensordict import TensorDict

for B, n, iters in ((64, 50, 1000), (2, 1000, 20)):
    locs = torch.rand(B, n, 2, device=dev)
    tours = torch.rand(B, n, device=dev).argsort(1)
    tours[0, 1] = n
    moves = torch.empty(B, dtype=torch.int32, device=dev)
    out = native.tsp_two_opt(locs, tours, iters, moves=moves)
    FusedTSPEnv.local_search(TensorDict({"locs": locs[1:]}, batch_size=[B - 1]), tours[1:], iters)
    torch.cuda.synchronize()
    print("two_opt", n, "ok", moves.tolist()[:4])
