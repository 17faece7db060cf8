"""CPU: REINFORCE baselines that are host-side glue (SURVEY.md 8f-2) against what the reference's own classes
(rl4co/models/rl/reinforce/baselines.py) computed on the same fake policy / env and inputs, recorded in
tests/golden/ref_baselines.npz (tests/golden/make_golden.py): Warmup blending, the rollout baseline's epoch-end
paired t-test swap, the critic baseline's value / loss, registry names."""

import numpy as np
import pytest
import torch
import torch.nn as nn

from rl4co_b200 import reinforce as R
from rl4co_b200.data import TensorDictDataset
from rl4co_b200.tensordict import TensorDict


class FakePolicy(nn.Module):
    """reward = -(sum x) + bias + wobble * sin(40 x0): a policy whose quality is one number, so that candidate /
    baseline comparisons are controlled."""

    def __init__(self, bias=0.0, wobble=0.0):
        super().__init__()
        self.bias = nn.Parameter(torch.tensor(float(bias)))
        self.wobble = wobble

    def forward(self, td, env=None, phase=None, decode_type=None, **kw):
        x = td["x"]
        return {"reward": -(x.sum(-1)) + self.bias + self.wobble * torch.sin(40 * x[:, 0])}


class FakeEnv:
    name = "fake"

    def reset(self, td):
        return td

    def dataset(self, batch_size=[], **kw):
        g = torch.Generator().manual_seed(123)
        return TensorDictDataset(TensorDict({"x": torch.rand(batch_size[0], 5, generator=g)}, batch_size=batch_size))


class _Enc(nn.Module):
    def __init__(self):
        super().__init__()
        self.lin = nn.Linear(2, 128)

    def forward(self, td):
        h = self.lin(td["locs"])
        return h, h


class CriticPolicy(nn.Module):
    def __init__(self):
        super().__init__()
        self.encoder = _Enc()


def baseline_inputs():
    """The evaluation inputs of the tests below (a fixed generator, shared with the fixture's recorder)."""
    g = torch.Generator().manual_seed(0)
    return {"rollout_x": torch.rand(7, 5, generator=g).numpy(),
            "warmup_x": torch.rand(3, 2, 9, 5, generator=g).numpy(),
            "warmup_reward": (-torch.rand(3, 2, 9, generator=g) * 5).numpy(),
            "critic_locs": torch.rand(6, 10, 2, generator=g).numpy(),
            "critic_reward": (-torch.rand(6, generator=g) * 4).numpy()}


@pytest.fixture(scope="module")
def ref():
    import os

    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_baselines.npz"))


#: rollout-baseline candidates, in the order tests/golden/make_golden.py records them (ref_baselines.npz rollout<i>/)
ROLLOUT_CANDIDATES = [dict(bias=0.5, wobble=0.0), dict(bias=0.002, wobble=0.3), dict(bias=-0.3, wobble=0.0)]


@pytest.mark.parametrize("cand,expect_update", [(ROLLOUT_CANDIDATES[0], True),     # clearly better
                                                 (ROLLOUT_CANDIDATES[1], False),    # better on average, not significant
                                                 (ROLLOUT_CANDIDATES[2], False)])   # worse
def test_rollout_baseline_ttest_swap_matches_reference(ref, cand, expect_update):
    case = ROLLOUT_CANDIDATES.index(cand)
    base = FakePolicy(0.0)
    mine = R.RolloutBaseline(bl_alpha=0.05)
    mine.setup(base, FakeEnv(), batch_size=16, device="cpu", dataset_size=64)
    assert abs(float(mine.mean) - float(ref[f"rollout{case}/setup_mean"])) < 1e-6
    torch.testing.assert_close(torch.as_tensor(mine.bl_vals), torch.from_numpy(ref[f"rollout{case}/bl_vals"]))
    updated = mine.epoch_callback(FakePolicy(**cand), FakeEnv(), batch_size=16, device="cpu", epoch=0, dataset_size=64)
    assert updated == expect_update
    assert abs(float(mine.mean) - float(ref[f"rollout{case}/mean"])) < 1e-6   # both swapped, or both kept the old policy
    assert float(mine.policy.bias) == float(ref[f"rollout{case}/bias"])
    td = TensorDict({"x": torch.from_numpy(baseline_inputs()["rollout_x"])}, batch_size=[7])
    torch.testing.assert_close(mine.eval(td, None, FakeEnv())[0], torch.from_numpy(ref[f"rollout{case}/eval"]))


def test_warmup_baseline_blends_like_reference(ref, monkeypatch):
    # the exponential part's batch mean is `co_reward_stats` + all-reduce in the product (CUDA only, no CPU fallback);
    # this CPU test exercises the blending / epoch logic around it, so the mean is served by torch here
    monkeypatch.setattr(R, "global_mean_baseline", lambda r: r.double().mean().float())
    inp = baseline_inputs()
    mine = R.get_reinforce_baseline("rollout", n_epochs=2, exp_beta=0.8)
    assert isinstance(mine, R.WarmupBaseline) and isinstance(mine.baseline, R.RolloutBaseline)
    base = FakePolicy(0.1)
    mine.setup(base, FakeEnv(), batch_size=16, device="cpu", dataset_size=32)
    want_v, want_alpha = torch.from_numpy(ref["warmup/values"]), ref["warmup/alpha"]
    for epoch in range(3):
        for j in range(2):  # two batches per epoch: the exponential part has memory
            td = TensorDict({"x": torch.from_numpy(inp["warmup_x"][epoch, j])}, batch_size=[9])
            v_m, l_m = mine.eval(td, torch.from_numpy(inp["warmup_reward"][epoch, j]), FakeEnv())
            torch.testing.assert_close(torch.as_tensor(v_m).float().expand(9), want_v[2 * epoch + j])
            assert float(l_m) == 0.0
        mine.epoch_callback(base, FakeEnv(), batch_size=16, device="cpu", epoch=epoch, dataset_size=32)
        assert mine.alpha == want_alpha[epoch]
    assert mine.alpha == 1


def test_critic_baseline_matches_reference(ref):
    inp = baseline_inputs()
    torch.manual_seed(1)
    pol = CriticPolicy()
    mine = R.CriticBaseline()
    torch.manual_seed(2)
    mine.setup(pol, FakeEnv())
    assert list(mine.critic.state_dict().keys()) == [str(k) for k in ref["critic/keys"]]
    td = TensorDict({"locs": torch.from_numpy(inp["critic_locs"])}, batch_size=[6])
    v_m, l_m = mine.eval(td, torch.from_numpy(inp["critic_reward"]))
    torch.testing.assert_close(v_m, torch.from_numpy(ref["critic/value"]))
    torch.testing.assert_close(l_m, torch.from_numpy(ref["critic/loss"]))
    assert l_m.requires_grad and not v_m.requires_grad


def test_registry_names(ref):
    for name, theirs in zip(ref["registry/names"], ref["registry/types"]):
        mine = R.get_reinforce_baseline(str(name))
        assert type(mine).__name__ == str(theirs) or name == "mean"  # reference's Mean = Exponential(beta=0)
