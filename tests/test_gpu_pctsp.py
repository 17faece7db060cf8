"""GPU: the third sibling env (SURVEY.md 8f-4) -- the prize-collecting TSP (rl4co/envs/routing/pctsp/env.py,
PCTSPInitEmbedding init.py:221-251, PCTSPContext context.py:184-198) on the stepping kernels and inside the persistent kernel
(ENV = pctsp behind the mask functor: depot rule on the collected prize, reward = saved penalties - length - all penalties),
against fixtures recorded from the unmodified reference (`env_pctsp*.npz`, `am_pctsp*.npz`) and against the CPU oracle."""

import pytest
import torch

from oracle import am_rollout_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
RTOL, ATOL_LP = 1e-5, 2e-5


def _policy(weights):
    from rl4co_b200.policy import FusedAttentionModelPolicy

    pol = FusedAttentionModelPolicy(env_name="pctsp", num_encoder_layers=1)
    pol.decoder.cache_gemm = "cublas"
    sd = pol.state_dict()
    for k, v in weights.items():
        assert k in sd and sd[k].shape == v.shape, f"reference parameter {k} has no counterpart"
    pol.load_state_dict({**sd, **weights})
    return pol.to(DEV).eval()


@pytest.mark.parametrize("name", ["env_pctsp20", "env_pctsp50"])
@pytest.mark.parametrize("inplace", [False, True])
def test_pctsp_env_kernels_bit_exact(golden, name, inplace):
    """co_pctsp_step / co_pctsp_action_mask along the reference's random-policy traces: masks, visited, collected prize,
    running penalty and done bit for bit; the reward to 1e-5."""
    from rl4co_b200.envs import get_env
    from rl4co_b200.tensordict import TensorDict

    g = golden(name)
    inst = g.inst(DEV)
    B = inst["locs"].shape[0]
    env = get_env("pctsp", generator_params=dict(num_loc=inst["locs"].shape[1]), inplace=inplace)
    td = env.reset(TensorDict(inst, batch_size=[B]))
    assert torch.equal(td["action_mask"].cpu(), g["action_mask"][0])
    actions = g["actions"].to(DEV)
    for t in range(actions.shape[1]):
        td.set("action", actions[:, t].contiguous())
        td = env.step(td)["next"]
        assert torch.equal(td["action_mask"].cpu(), g["action_mask"][t + 1]), f"mask step {t}"
        assert torch.equal(td["done"].cpu(), g["done"][t])
        assert torch.equal(td["visited"].cpu(), g["visited"][t].bool())
        assert torch.equal(td["cur_total_prize"].cpu(), g["cur_total_prize"][t]), f"prize step {t}"
        # starts from penalty.sum(-1), a torch reduction whose order differs between the CPU (fixture) and CUDA
        torch.testing.assert_close(td["cur_total_penalty"].cpu(), g["cur_total_penalty"][t], rtol=1e-6, atol=1e-6)
        assert torch.equal(td["current_node"].cpu().reshape(-1), g["current_node"][t])
    r = env.get_reward(td, actions)  # includes check_solution_validity
    torch.testing.assert_close(r.cpu(), g["reward"], rtol=1e-5, atol=1e-5)
    dup = actions.clone()
    row = (dup != 0).sum(1).argmax()
    cust = dup[row][dup[row] != 0]
    if cust.numel() >= 2:  # visit a customer twice
        pos = (dup[row] != 0).nonzero().reshape(-1)
        dup[row, pos[1]] = dup[row, pos[0]]
        with pytest.raises(AssertionError):
            env.check_solution_validity(td, dup)


@pytest.mark.parametrize("name", ["am_pctsp20", "am_pctsp50"])
def test_pctsp_decoder_step_vs_reference_logits(golden, name):
    """decoder.forward with the OP context (budget left instead of capacity left), teacher-forced along the reference's
    greedy path: raw logits against the recorded ones, masks bit-exact; encoder (prize feature) against the recorded
    embeddings."""
    from rl4co_b200.envs import get_env
    from rl4co_b200.tensordict import TensorDict

    g = golden(name)
    pol = _policy(g.weights())
    inst = g.inst(DEV)
    B = inst["locs"].shape[0]
    env = get_env("pctsp", generator_params=dict(num_loc=inst["locs"].shape[1]))
    td = env.reset(TensorDict(inst, batch_size=[B]))
    with torch.inference_mode():
        h, _ = pol.encoder(td)
    torch.testing.assert_close(h.cpu(), g["h"], rtol=1e-4, atol=2e-5)
    td, env, cached = pol.decoder.pre_decoder_hook(td, env, g["h"].to(DEV))
    ref_logits, ref_actions = g["greedy_logits"], g["greedy_actions"]
    for t in range(ref_actions.shape[1]):
        logits, mask = pol.decoder(td, cached, 0)
        torch.testing.assert_close(logits.cpu(), ref_logits[t], rtol=1e-4, atol=2e-5)
        assert torch.equal(mask.cpu(), g["greedy_masks"][t])
        td.set("action", ref_actions[:, t].to(DEV).contiguous())
        td = env.step(td)["next"]


@pytest.mark.parametrize("name", ["am_pctsp20", "am_pctsp50"])
@pytest.mark.parametrize("mode", ["greedy", "sampling", "evaluate"])
@pytest.mark.parametrize("fused", [True, False])
def test_pctsp_policy_vs_golden(golden, name, mode, fused, monkeypatch):
    from rl4co_b200 import decoding
    from rl4co_b200.envs import get_env
    from rl4co_b200.tensordict import TensorDict

    g = golden(name)
    pol = _policy(g.weights())
    inst = g.inst(DEV)
    B = inst["locs"].shape[0]
    env = get_env("pctsp", generator_params=dict(num_loc=inst["locs"].shape[1]), check_solution=True)
    td = env.reset(TensorDict(inst, batch_size=[B]))
    N = inst["locs"].shape[1] + 1
    if mode == "sampling" and fused:  # recorded-noise protocol, padded to the kernel's step bound
        q = g["sampling_noise"]
        qpad = torch.ones(N + 1, q.shape[1], q.shape[2])
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
        assert same.float().mean() >= 0.75  # fp32 near-tie flips are checked against the oracle below
    T = ra.shape[1]
    torch.testing.assert_close(out["log_likelihood"].cpu()[:, :T][same], rl[same], rtol=RTOL, atol=ATOL_LP)
    torch.testing.assert_close(out["reward"].cpu()[same], rr[same], rtol=RTOL, atol=1e-6)


@pytest.mark.parametrize("n,batch", [(20, 64), (100, 32)])
def test_pctsp_policy_vs_oracle_on_fresh_instances(n, batch):
    """Seeded fresh instances (on-device generator off: the CPU call order): teacher-forced oracle log-probs / rewards of
    the GPU's own greedy and sampled actions, valid tours (check_solution=True); multistart decoding runs (its forced
    starts ignore the budget exactly like ops.py:128-149, so their validity is not asserted)."""
    from rl4co_b200.envs import get_env
    from rl4co_b200.policy import FusedAttentionModelPolicy

    torch.manual_seed(21 + n)
    env = get_env("pctsp", generator_params=dict(num_loc=n), check_solution=True)
    pol = FusedAttentionModelPolicy(env_name="pctsp", num_encoder_layers=2).to(DEV).eval()
    td_host = env.generator(batch)
    with torch.inference_mode():
        td = env.reset(td_host.to(DEV))
        out = pol(td, env, phase="test", decode_type="greedy")
        td = env.reset(td_host.to(DEV))  # the stepping path advances the state in place, like the reference's loop
        smp = pol(td, env, phase="train", decode_type="sampling")
        td = env.reset(td_host.to(DEV))
        env_nc = get_env("pctsp", generator_params=dict(num_loc=n), check_solution=False)
        ms = pol(td, env_nc, phase="test", decode_type="multistart_greedy", num_starts=4)
    assert ms["reward"].shape[0] == 4 * batch and torch.isfinite(ms["log_likelihood"]).all()
    assert (smp["actions"][:, -1] == 0).all()
    W = {k: v.detach().cpu() for k, v in pol.state_dict().items()}
    inst = {k: td_host[k] for k in td_host.keys()}
    with torch.inference_mode():
        ref = O.policy_forward(W, "pctsp", inst, num_layers=2, actions=out["actions"].cpu(), faithful_copies=False)
    torch.testing.assert_close(out["reward"].cpu(), ref["reward"], rtol=RTOL, atol=1e-6)
    torch.testing.assert_close(out["log_likelihood"].cpu(), ref["log_likelihood"], rtol=RTOL, atol=ATOL_LP * 2)
    with torch.inference_mode():
        ref = O.policy_forward(W, "pctsp", inst, num_layers=2, actions=smp["actions"].cpu(), faithful_copies=False)
    torch.testing.assert_close(smp["reward"].cpu(), ref["reward"], rtol=RTOL, atol=1e-6)
    torch.testing.assert_close(smp["log_likelihood"].cpu(), ref["log_likelihood"], rtol=RTOL, atol=ATOL_LP * 4)


def test_pctsp_fused_equals_stepping():
    """Persistent kernel == stepping kernels on the same instances (sampling with one shared noise tensor, so the
    trajectories are long), with check_solution=True validating every tour."""
    from rl4co_b200.envs import get_env
    from rl4co_b200.policy import FusedAttentionModelPolicy

    torch.manual_seed(5)
    n, B = 50, 256
    env = get_env("pctsp", generator_params=dict(num_loc=n), check_solution=True)
    pol = FusedAttentionModelPolicy(env_name="pctsp", num_encoder_layers=1).to(DEV).eval()
    pol.decoder.cache_gemm = "cublas"
    td_host = env.generator(B)
    with torch.inference_mode():
        a = pol(env.reset(td_host.to(DEV)), env, phase="test", decode_type="sampling", seed=3, return_sum_log_likelihood=False)
        b = pol(env.reset(td_host.to(DEV)), env, phase="test", actions=a["actions"], fused_rollout=False,
                return_sum_log_likelihood=False)
    assert (a["actions"][:, -1] == 0).all() and (a["actions"] != 0).any(1).float().mean() > 0.5
    T = min(a["log_likelihood"].shape[1], b["log_likelihood"].shape[1])
    torch.testing.assert_close(a["log_likelihood"][:, :T], b["log_likelihood"][:, :T], rtol=RTOL, atol=ATOL_LP)
    torch.testing.assert_close(a["reward"], b["reward"], rtol=RTOL, atol=1e-6)


def test_pctsp_under_the_reference_loop():
    """Drop-in: the reference's own ConstructivePolicy.forward + DecodingStrategy on its PCTSP env, as recorded in
    tests/golden/dropin.npz, reproduced by FusedPCTSPEnv and the CUDA decoder on the same weights, instances and
    sampling draws."""
    import os

    import numpy as np

    from test_gpu_dropin import check_forward_against_reference

    ref = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "dropin.npz"))
    *_, want = check_forward_against_reference(ref, "pctsp20_sampling", "pctsp", 20, 1, "sampling", sample_seed=11, phase="train")
    assert (want["actions"] != 0).any(1).float().mean() > 0.5  # the sampled tours are not trivial
