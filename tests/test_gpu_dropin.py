"""The drop-in claim against the reference's own loop: what rl4co's unmodified `rollout()` helper
(rl4co/utils/decoding.py:85-106) and `ConstructivePolicy.forward` (rl4co/models/common/constructive/base.py:154-263)
computed on seeded instances and name-seeded weights, recorded in tests/golden/dropin.npz
(tests/golden/make_golden.py), must be reproduced by the CUDA env and the CUDA decoder: bit-identical masks / done
flags along the reference's trajectories, and the same trajectories, log-likelihoods and rewards up to fp32
re-association (sampling replays the Exp(1) draws torch.multinomial took, regenerated from the recorded seed)."""

import os

import numpy as np
import pytest
import torch

from conftest import golden_case

pytestmark = pytest.mark.gpu

RTOL, ATOL_LP = 1e-5, 2e-5


@pytest.fixture(scope="module")
def ref():
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "dropin.npz"))


@pytest.fixture(scope="module")
def dev():
    from rl4co_b200 import native

    native.lib()
    return torch.device("cuda:0")


def _td(inst, dev):
    from rl4co_b200.tensordict import TensorDict

    B = next(iter(inst.values())).shape[0]
    return TensorDict({k: v.to(dev) for k, v in inst.items()}, batch_size=[B])


def _pad(a, T):
    return torch.nn.functional.pad(a, (0, T - a.shape[1]))


def check_forward_against_reference(ref, tag, name, n, layers, decode_type, sample_seed=None, phase="test",
                                    min_same=0.9):
    """The project's policy (CUDA env + decoder; strict-fp32 cache GEMM) on a recorded reference forward."""
    from rl4co_b200.envs import get_env
    from rl4co_b200.policy import FusedAttentionModelPolicy

    dev = torch.device("cuda:0")
    inst, want, W = golden_case(ref, tag)
    env = get_env(name, generator_params=dict(num_loc=n), check_solution=True)
    pol = FusedAttentionModelPolicy(env_name=name, num_encoder_layers=layers)
    pol.load_state_dict(W)
    pol.decoder.cache_gemm = "cublas"
    pol = pol.to(dev).eval()
    td0 = _td(inst, dev)
    if "sampling" in decode_type:
        # the reference drew one [B, N] Exp(1) block per step from the seeded torch generator
        B, N, T = want["actions"].shape[0], env.reset(td0.clone())["action_mask"].shape[-1], want["actions"].shape[1]
        torch.manual_seed(sample_seed)
        q = torch.stack([torch.empty(B, N).exponential_(1) for _ in range(T)])
        kw = {"noise": torch.cat([q, torch.ones(3 * N, B, N)]).to(dev)}  # rows past the reference's T are never read
    else:
        kw = {"fused_rollout": False}  # the step-at-a-time loop, like the reference's
    with torch.inference_mode():
        o = pol(env.reset(td0.clone()), env, phase=phase, decode_type=decode_type, return_sum_log_likelihood=False, **kw)
    T = max(o["actions"].shape[1], want["actions"].shape[1])
    same = (_pad(o["actions"].cpu(), T) == _pad(want["actions"], T)).all(1)
    # fp32 re-association between the reference's torch ops and the kernels can flip a genuine near-tie (and, for
    # sampling, a draw that lands on a bin edge); everything that follows the same trajectory must agree to tolerance
    assert same.float().mean() >= min_same
    ll, reward = o["log_likelihood"].cpu(), o["reward"].cpu()
    torch.testing.assert_close(ll.sum(-1)[same], want["ll"][same], rtol=RTOL, atol=4 * ATOL_LP)
    torch.testing.assert_close(reward[same], want["reward"][same], rtol=RTOL, atol=1e-6)
    if "logprobs" in want:
        rows = same[: want["logprobs"].shape[0]]
        Tw = want["logprobs"].shape[1]
        torch.testing.assert_close(_pad(ll[: rows.shape[0]], Tw)[rows][:, :Tw], want["logprobs"][rows],
                                   rtol=RTOL, atol=ATOL_LP)
    return pol, env, td0, want


@pytest.mark.parametrize("name,n", [("tsp", 20), ("cvrp", 20), ("tsp", 50), ("cvrp", 50)])
def test_reference_rollout_helper_drives_fused_env(ref, dev, name, n):
    """decoding.py:85-106 `rollout(env, td, random_policy)` as recorded from the reference env: the CUDA env, stepped
    along the same actions, gives bit-identical action masks and done flags at every step and the same rewards."""
    from rl4co_b200.envs import get_env

    inst, want, _ = golden_case(ref, f"env_{name}{n}")
    env = get_env(name, generator_params=dict(num_loc=n), check_solution=True)
    td = env.reset(_td(inst, dev))
    assert torch.equal(td["action_mask"].cpu(), want["action_mask"][0])
    actions = want["actions"].to(dev)
    for t in range(actions.shape[1]):
        td.set("action", actions[:, t].contiguous())
        td = env.step(td)["next"]
        assert torch.equal(td["action_mask"].cpu(), want["action_mask"][t + 1]), f"mask step {t}"
        assert torch.equal(td["done"].cpu().reshape(want["done"][t].shape), want["done"][t]), f"done step {t}"
    torch.testing.assert_close(env.get_reward(td, actions).cpu(), want["reward"], rtol=RTOL, atol=1e-6)


@pytest.mark.parametrize("name,n", [("tsp", 20), ("cvrp", 20), ("tsp", 50), ("cvrp", 50)])
@pytest.mark.parametrize("decode_type", ["greedy", "sampling", "multistart_greedy"])
def test_reference_policy_forward_drives_fused_env_and_decoder(ref, dev, name, n, decode_type):
    """The reference's ConstructivePolicy.forward on the reference env / decoder, against the CUDA env + decoder."""
    pol, env, td0, want = check_forward_against_reference(
        ref, f"fwd_{name}{n}_{decode_type}", name, n, 2, decode_type, sample_seed=3,
        min_same=0.9 if decode_type != "sampling" else 0.75)
    if "multistart" in decode_type:
        return
    # teacher-forced on the reference's actions: every row comparable
    with torch.inference_mode():
        e = pol(env.reset(td0.clone()), env, phase="test", actions=want["actions"].to(dev), fused_rollout=False,
                return_sum_log_likelihood=False)
    torch.testing.assert_close(e["log_likelihood"].sum(-1).cpu(), want["eval_ll"], rtol=RTOL, atol=4 * ATOL_LP)
    torch.testing.assert_close(e["reward"].cpu(), want["eval_reward"], rtol=RTOL, atol=1e-6)
    rows = want["eval_logprobs"].shape[0]
    torch.testing.assert_close(e["log_likelihood"][:rows].cpu(), want["eval_logprobs"], rtol=RTOL, atol=ATOL_LP)


def test_fused_envs_register_as_torchrl_envs(monkeypatch):
    """FusedEnvBase is a (virtual) subclass of torchrl.envs.EnvBase whenever torchrl is importable (here a stand-in
    module whose EnvBase is an ABC, as torchrl's is)."""
    import abc
    import sys
    import types

    class EnvBase(abc.ABC):
        pass

    torchrl, envs = types.ModuleType("torchrl"), types.ModuleType("torchrl.envs")
    torchrl.__path__, envs.EnvBase, torchrl.envs = [], EnvBase, envs
    monkeypatch.setitem(sys.modules, "torchrl", torchrl)
    monkeypatch.setitem(sys.modules, "torchrl.envs", envs)
    from rl4co_b200.envs import FusedTSPEnv, _register_with_torchrl

    assert _register_with_torchrl()
    assert isinstance(FusedTSPEnv(), EnvBase)
