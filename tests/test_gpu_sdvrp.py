"""GPU: the first sibling env (SURVEY.md 8f-4) -- SDVRP (rl4co/envs/routing/sdvrp/env.py) with its dynamic embedding
(nn/env_embeddings/dynamic.py:60-78) on the stepping kernels, against fixtures recorded from the unmodified reference
(`env_sdvrp*.npz`, `am_sdvrp*.npz`) and against the CPU oracle."""

import pytest
import torch

from conftest import env_of
from oracle import am_rollout_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
RTOL, ATOL_LP, TIE_TOL = 1e-5, 2e-5, 1e-4


def _policy(weights, **kw):
    from rl4co_b200.policy import FusedAttentionModelPolicy

    pol = FusedAttentionModelPolicy(env_name="sdvrp", num_encoder_layers=1, **kw)
    pol.decoder.cache_gemm = "cublas"
    sd = pol.state_dict()
    for k, v in weights.items():
        assert k in sd and sd[k].shape == v.shape, f"reference parameter {k} has no counterpart"
    pol.load_state_dict({**sd, **weights})
    return pol.to(DEV).eval()


class _FixedEncoder(torch.nn.Module):
    def __init__(self, h):
        super().__init__()
        self.h = h

    def forward(self, td):
        return self.h, self.h


@pytest.mark.parametrize("name", ["env_sdvrp20", "env_sdvrp50"])
@pytest.mark.parametrize("inplace", [False, True])
def test_sdvrp_env_kernels_bit_exact(golden, name, inplace):
    from rl4co_b200.envs import get_env
    from rl4co_b200.tensordict import TensorDict

    g = golden(name)
    inst = g.inst(DEV)
    B = inst["locs"].shape[0]
    env = get_env("sdvrp", generator_params=dict(num_loc=inst["locs"].shape[1]), inplace=inplace)
    td = env.reset(TensorDict(inst, batch_size=[B]))
    assert torch.equal(td["action_mask"].cpu(), g["action_mask"][0])
    actions = g["actions"].to(DEV)
    for t in range(actions.shape[1]):
        td.set("action", actions[:, t].contiguous())
        td = env.step(td)["next"]
        assert torch.equal(td["action_mask"].cpu(), g["action_mask"][t + 1]), f"mask step {t}"
        assert torch.equal(td["done"].cpu(), g["done"][t])
        assert torch.equal(td["demand_with_depot"].cpu(), g["demand_with_depot"][t])
        assert torch.equal(td["used_capacity"].cpu(), g["used_capacity"][t])
        assert torch.equal(td["current_node"].cpu().reshape(-1), g["current_node"][t])
    r = env.get_reward(td, actions)  # includes check_solution_validity
    torch.testing.assert_close(r.cpu(), g["reward"], rtol=RTOL, atol=1e-6)
    bad = actions.clone()
    bad[0, -1] = 0
    bad[0, bad[0].nonzero().reshape(-1)[-1]] = 0  # drop the last customer visit: demand stays unserved
    with pytest.raises(AssertionError):
        env.check_solution_validity(td, bad)


@pytest.mark.parametrize("name", ["am_sdvrp20", "am_sdvrp50"])
def test_sdvrp_decoder_step_vs_reference_logits(golden, name):
    """decoder.forward with the dynamic embedding, teacher-forced along the reference's greedy path: raw logits
    against the logits the reference recorded, masks bit-exact."""
    from rl4co_b200.envs import get_env
    from rl4co_b200.tensordict import TensorDict

    g = golden(name)
    pol = _policy(g.weights())
    inst = g.inst(DEV)
    B = inst["locs"].shape[0]
    env = get_env("sdvrp", generator_params=dict(num_loc=inst["locs"].shape[1]))
    td = env.reset(TensorDict(inst, batch_size=[B]))
    td, env, cached = pol.decoder.pre_decoder_hook(td, env, g["h"].to(DEV))
    ref_logits, ref_actions = g["greedy_logits"], g["greedy_actions"]
    for t in range(ref_actions.shape[1]):
        logits, mask = pol.decoder(td, cached, 0)
        torch.testing.assert_close(logits.cpu(), ref_logits[t], rtol=1e-4, atol=2e-5)
        assert torch.equal(mask.cpu(), g["greedy_masks"][t])
        td.set("action", ref_actions[:, t].to(DEV).contiguous())
        td = env.step(td)["next"]


@pytest.mark.parametrize("name", ["am_sdvrp20", "am_sdvrp50"])
@pytest.mark.parametrize("mode", ["greedy", "sampling", "evaluate"])
@pytest.mark.parametrize("fused", [True, False])
def test_sdvrp_policy_vs_golden(golden, name, mode, fused, monkeypatch):
    """Both execution paths against the reference fixtures: the persistent kernel (ENV = sdvrp behind the mask
    functor, dynamic embedding folded into per-step scalars) and the stepping kernels."""
    from rl4co_b200 import decoding
    from rl4co_b200.envs import get_env
    from rl4co_b200.tensordict import TensorDict

    g = golden(name)
    pol = _policy(g.weights())
    inst = g.inst(DEV)
    B = inst["locs"].shape[0]
    env = get_env("sdvrp", generator_params=dict(num_loc=inst["locs"].shape[1]), check_solution=True)
    td = env.reset(TensorDict(inst, batch_size=[B]))
    pol.encoder = _FixedEncoder(g["h"].to(DEV))
    kw = {}
    N = inst["locs"].shape[1] + 1
    if mode == "sampling" and fused:  # recorded-noise protocol, padded to the kernel's step bound
        q = g["sampling_noise"]
        qpad = torch.ones(3 * (N - 1) + 2, q.shape[1], q.shape[2])
        qpad[: q.shape[0]] = q
        kw = dict(decode_type="sampling", noise=qpad.to(DEV))
    elif mode == "sampling":  # stepping path: serve the Exp(1) draws torch.multinomial consumed, one per step
        served = iter(g["sampling_noise"].to(DEV).unbind(0))
        monkeypatch.setattr(decoding.Sampling, "_noise", lambda self, logits: next(served).contiguous())
        kw = dict(decode_type="sampling")
    elif mode == "evaluate":
        kw = dict(actions=g["eval_actions"].to(DEV))
    else:
        kw = dict(decode_type="greedy")
    with torch.inference_mode():
        out = pol(td, env, phase="test", return_sum_log_likelihood=False, fused_rollout=fused, **kw)
    key = {"greedy": "greedy", "sampling": "sampling", "evaluate": "eval"}[mode]
    ra, rl, rr = g[f"{key}_actions"], g[f"{key}_logprobs"], g[f"{key}_reward"]
    if mode == "evaluate":
        assert torch.equal(out["actions"].cpu(), ra)
        same = torch.ones(B, dtype=torch.bool)
    else:
        same = (out["actions"].cpu()[:, : ra.shape[1]] == ra).all(1) if out["actions"].shape[1] >= ra.shape[1] \
            else torch.zeros(B, dtype=torch.bool)
        assert same.float().mean() >= 0.75  # near-tie flips (fp32 re-association) are checked by the oracle test below
    T = ra.shape[1]
    torch.testing.assert_close(out["log_likelihood"].cpu()[:, :T][same], rl[same], rtol=RTOL, atol=ATOL_LP)
    torch.testing.assert_close(out["reward"].cpu()[same], rr[same], rtol=RTOL, atol=1e-6)


@pytest.mark.parametrize("fused", [True, False])
@pytest.mark.parametrize("n,batch", [(20, 64), (50, 64), (100, 32), (5, 40)])
def test_sdvrp_policy_vs_prefix_oracle(n, batch, fused):
    """Seeded larger cases: every GPU choice is the oracle's (near-)best for the same prefix, log-probs / reward
    agree, tours are valid."""
    from rl4co_b200.envs import get_env
    from rl4co_b200.policy import FusedAttentionModelPolicy

    torch.manual_seed(n)
    env = get_env("sdvrp", generator_params=dict(num_loc=n), check_solution=True)
    pol = FusedAttentionModelPolicy(env_name="sdvrp", num_encoder_layers=1).to(DEV).eval()
    pol.decoder.cache_gemm = "cublas"
    with torch.no_grad():
        pol.decoder.dynamic_embedding.projection.weight.mul_(3.0)
    td_host = env.generator(batch)
    with torch.inference_mode():
        td = env.reset(td_host.to(DEV))
        h, _ = pol.encoder(td)
        out = pol(td, env, phase="test", decode_type="greedy", return_sum_log_likelihood=False, encoder_output=(h, h),
                  fused_rollout=fused)
    W = {k: v.detach().cpu() for k, v in pol.state_dict().items()}
    inst = {k: td_host[k] for k in ("locs", "depot", "demand")}
    acts = out["actions"].cpu()
    with torch.inference_mode():
        ref = O.rollout(W, "sdvrp", inst, h.cpu(), actions=acts, return_trace=True, faithful_copies=False)
    torch.testing.assert_close(out["log_likelihood"].cpu(), ref["logprobs"], rtol=RTOL, atol=ATOL_LP)
    torch.testing.assert_close(out["reward"].cpu(), ref["reward"], rtol=RTOL, atol=1e-6)
    for t, full in enumerate(ref["trace"]["logprobs"]):
        chosen = full.gather(1, acts[:, t][:, None]).squeeze(1)
        assert (full.max(1)[0] - chosen < TIE_TOL).all(), f"step {t}: GPU arg-max is not the oracle's (near-)best"


def test_sdvrp_under_the_reference_loop():
    """Drop-in: the reference's own ConstructivePolicy.forward + DecodingStrategy on its SDVRP env, as recorded in
    tests/golden/dropin.npz, reproduced by FusedSDVRPEnv and the CUDA decoder on the same weights, instances and
    greedy decoding."""
    import os

    import numpy as np

    from test_gpu_dropin import check_forward_against_reference

    ref = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "dropin.npz"))
    *_, want = check_forward_against_reference(ref, "sdvrp20_greedy", "sdvrp", 20, 1, "greedy", sample_seed=None, phase="test")


def test_sdvrp_fused_equals_stepping_and_multisample():
    """Persistent kernel == stepping kernels on the same instances (greedy); in-kernel Philox sampling gives valid
    split-delivery tours and reproducible draws."""
    from rl4co_b200.envs import get_env
    from rl4co_b200.policy import FusedAttentionModelPolicy

    torch.manual_seed(9)
    env = get_env("sdvrp", generator_params=dict(num_loc=50), check_solution=True)
    pol = FusedAttentionModelPolicy(env_name="sdvrp", num_encoder_layers=1).to(DEV).eval()
    pol.decoder.cache_gemm = "cublas"
    with torch.inference_mode():
        td = env.reset(env.generator(256).to(DEV))
        a = pol(td, env, phase="test", decode_type="greedy", return_sum_log_likelihood=False)
        b = pol(td, env, phase="test", decode_type="greedy", return_sum_log_likelihood=False, fused_rollout=False)
        T = min(a["actions"].shape[1], b["actions"].shape[1])
        same = (a["actions"][:, :T] == b["actions"][:, :T]).all(1)
        assert same.float().mean() >= 0.95
        torch.testing.assert_close(a["reward"][same], b["reward"][same], rtol=RTOL, atol=1e-6)
        torch.testing.assert_close(a["log_likelihood"][:, :T][same], b["log_likelihood"][:, :T][same], rtol=RTOL, atol=ATOL_LP)
        s1 = pol(td, env, phase="train", decode_type="sampling", seed=4)   # check_solution=True validates the tours
        s2 = pol(td, env, phase="train", decode_type="sampling", seed=4)
        s3 = pol(td, env, phase="train", decode_type="sampling", seed=5)
    assert torch.equal(s1["actions"], s2["actions"]) and not torch.equal(s1["actions"], s3["actions"])
    assert torch.isfinite(s1["log_likelihood"]).all() and (s1["log_likelihood"] < 0).all()


@pytest.mark.gpu
def test_sdvrp_multistart_trajectories_share_an_instance():
    """S > 1 trajectories of one instance inside the persistent kernel: split deliveries consume the demand in place, so
    every further trajectory must start from the original demands again -- valid tours for every start
    (check_solution=True) and the same trajectories as the stepping kernels (sdvrp/env.py:55-116, ops.py:128-149)."""
    from rl4co_b200.envs import get_env
    from rl4co_b200.policy import FusedAttentionModelPolicy

    torch.manual_seed(11)
    for n, starts in ((20, 3), (50, 5)):
        env = get_env("sdvrp", generator_params=dict(num_loc=n), check_solution=True)
        pol = FusedAttentionModelPolicy(env_name="sdvrp", num_encoder_layers=1).to(DEV).eval()
        pol.decoder.cache_gemm = "cublas"
        with torch.inference_mode():
            td = env.reset(env.generator(64).to(DEV))
            a = pol(td, env, phase="test", decode_type="multistart_greedy", num_starts=starts)
            b = pol(td, env, phase="test", decode_type="multistart_greedy", num_starts=starts, fused_rollout=False)
        T = min(a["actions"].shape[1], b["actions"].shape[1])
        same = (a["actions"][:, :T] == b["actions"][:, :T]).all(1)
        assert same.float().mean() >= 0.9
        torch.testing.assert_close(a["reward"][same], b["reward"][same], rtol=RTOL, atol=1e-6)
        torch.testing.assert_close(a["log_likelihood"][same], b["log_likelihood"][same], rtol=RTOL, atol=ATOL_LP * 3)
