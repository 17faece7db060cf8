"""CPU: oracle/am_rollout_oracle.py against what the unmodified reference computed on the same instances, weights
and seeds, recorded in tests/golden/ref_policy.npz (tests/golden/make_golden.py): policy forwards over every decode
type, top-k / top-p filters, beam search, the sibling envs, the instance generator."""

import os

import numpy as np
import pytest
import torch

from conftest import golden_case
from oracle import am_rollout_oracle as O


@pytest.fixture(scope="module")
def ref():
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_policy.npz"))


@pytest.mark.parametrize("name,n", [("tsp", 20), ("cvrp", 20), ("tsp", 37), ("cvrp", 33)])
@pytest.mark.parametrize("decode_type", ["greedy", "sampling", "multistart_greedy", "multistart_sampling"])
def test_policy_forward_matches_reference(ref, name, n, decode_type):
    inst, want, W = golden_case(ref, f"fwd_{name}{n}_{decode_type}")
    with torch.inference_mode():
        torch.manual_seed(5)
        o = O.policy_forward(W, name, inst, decode_type=decode_type, num_layers=2)
    assert torch.equal(want["actions"], o["actions"])
    torch.testing.assert_close(want["reward"], o["reward"], rtol=1e-6, atol=0)
    torch.testing.assert_close(want["ll"], o["log_likelihood"], rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("name", ["tsp", "cvrp"])
def test_multinomial_is_argmax_p_over_exp_noise(ref, name):
    """The recorded-noise protocol used for sampling parity: torch.multinomial(p,1) consumes
    exactly one empty_like(p).exponential_(1) draw per step."""
    inst, want, W = golden_case(ref, f"multinomial_{name}")
    with torch.inference_mode():
        torch.manual_seed(7)
        o = O.policy_forward(W, name, inst, decode_type="sampling", num_layers=1,
                             noise=lambda t, shape: torch.empty(shape).exponential_(1))
    assert torch.equal(want["actions"], o["actions"])


@pytest.mark.parametrize("top_k,top_p", [(3, 0.0), (0, 0.6), (4, 0.8), (50, 0.0), (0, 1.0)])
def test_top_k_top_p_process_logits_matches_reference(ref, top_k, top_p):
    """utils/decoding.py:109-188 with the filters on, bit for bit (same torch ops in the same order)."""
    _, case, _ = golden_case(ref, f"process_{top_k}_{top_p}")
    got = O.process_logits(case["logits"].clone(), case["mask"], temperature=1.3, tanh_clipping=10.0, top_k=top_k,
                           top_p=top_p)
    assert torch.equal(case["want"], got)


@pytest.mark.parametrize("name", ["tsp", "cvrp"])
def test_policy_forward_with_filters_matches_reference(ref, name):
    inst, want, W = golden_case(ref, f"filters_{name}")
    with torch.inference_mode():
        torch.manual_seed(9)
        o = O.policy_forward(W, name, inst, decode_type="sampling", num_layers=1, top_k=5, top_p=0.9)
    assert torch.equal(want["actions"], o["actions"])
    torch.testing.assert_close(want["ll"], o["log_likelihood"], rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("name,n", [("tsp", 12), ("cvrp", 11)])
@pytest.mark.parametrize("beam_width,select_best", [(3, True), (4, False), (None, True)])
def test_beam_search_matches_reference(ref, name, n, beam_width, select_best):
    """utils/decoding.py:464-600 through the reference's ConstructivePolicy loop."""
    inst, want, W = golden_case(ref, f"beam_{name}{n}_{beam_width}_{select_best}")
    kw = {} if beam_width is None else {"beam_width": beam_width}
    with torch.inference_mode():
        o = O.policy_forward(W, name, inst, decode_type="beam_search", num_layers=1, select_best=select_best, **kw)
    assert torch.equal(want["actions"], o["actions"])
    torch.testing.assert_close(want["reward"], o["reward"], rtol=1e-6, atol=0)
    torch.testing.assert_close(want["ll"], o["log_likelihood"], rtol=1e-5, atol=1e-5)


def test_generator_matches_reference(ref):
    for name, n in (("tsp", 50), ("cvrp", 50), ("cvrp", 100)):
        _, want, _ = golden_case(ref, f"gen_{name}{n}")
        torch.manual_seed(1234)
        inst = O.generate_instances(name, 5, n)
        assert want and set(inst) <= set(want), name
        for k in inst:
            assert torch.equal(want[k], inst[k]), (name, k)


@pytest.mark.parametrize("name,n", [("op", 20), ("op", 33), ("pctsp", 20), ("pctsp", 41), ("sdvrp", 20)])
@pytest.mark.parametrize("decode_type", ["greedy", "sampling"])
def test_sibling_env_policy_forward_matches_reference(ref, name, n, decode_type):
    """The sibling envs (SURVEY.md 8f-4): the reference policy (its own env, init / context / dynamic embeddings)
    against the oracle's restatement -- actions bit for bit, rewards and log-likelihoods to 1e-5."""
    inst, want, W = golden_case(ref, f"sibling_{name}{n}_{decode_type}")
    with torch.inference_mode():
        torch.manual_seed(5)
        o = O.policy_forward(W, name, inst, decode_type=decode_type, num_layers=2)
    assert torch.equal(want["actions"], o["actions"])
    torch.testing.assert_close(want["reward"], o["reward"], rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(want["ll"], o["log_likelihood"], rtol=1e-5, atol=1e-5)
