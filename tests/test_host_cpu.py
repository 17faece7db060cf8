"""CPU tests of the host side: the C-ABI library loads and exports every declared symbol,
TensorDict / layout helpers follow the reference conventions (golden layout fixture), envs
reset to the reference's keys / dtypes / shapes, parameter names match a reference
state_dict, and the product refuses to compute without CUDA."""

import ctypes
import os
import re

import pytest
import torch

from conftest import ROOT


@pytest.fixture(scope="module")
def libpath():
    from rl4co_b200 import native

    return native.build()


def test_library_exports_every_declared_symbol(libpath):
    L = ctypes.CDLL(libpath)
    header = open(os.path.join(ROOT, "include", "corollout.h")).read()
    declared = set(re.findall(r"\b(co_[a-z_0-9]+)\s*\(", header))
    declared -= {"co_rollout_args", "co_decoder_weights"}
    assert len(declared) >= 14
    for sym in declared:
        assert hasattr(L, sym), f"{sym} declared in include/corollout.h but not exported"
    from rl4co_b200 import native

    assert set(native.EXPORTS) == declared
    assert L.co_version() == 100
    assert L.co_cache_width(0) == 5 * 128 and L.co_cache_width(1) == 4 * 128
    assert L.co_rollout_max_nodes() == 128


def test_rollout_args_struct_matches_header():
    from rl4co_b200 import native

    header = open(os.path.join(ROOT, "include", "corollout.h")).read()
    body = header[header.index("typedef struct co_rollout_args {"):header.index("} co_rollout_args;")]
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = re.findall(r"[\s\*]([a-zA-Z_][a-zA-Z_0-9]*)\s*(?:,\s*([a-zA-Z_][a-zA-Z_0-9]*))?;", body)
    flat = [n for pair in names for n in pair if n]
    assert flat == [f[0] for f in native.RolloutArgs._fields_]


def test_bad_arguments_return_error_codes_without_a_gpu(libpath):
    L = ctypes.CDLL(libpath)
    L.co_last_error_string.restype = ctypes.c_char_p
    assert L.co_rollout(None, None) == -1
    assert b"null args" in L.co_last_error_string()
    assert L.co_tsp_step(None, None, None, None, None, None, None, 4, 10, None) == -1


def test_tensordict_batch_semantics():
    from rl4co_b200.tensordict import TensorDict

    td = TensorDict({"a": torch.arange(12.0).view(3, 4), "b": torch.arange(3)}, batch_size=[3])
    assert td.shape == (3,) and td.dim() == 1 and not td.is_empty()
    e = td.expand(2, 3).contiguous().view(6)
    assert e["a"].shape == (6, 4) and e["b"].shape == (6,)
    assert torch.equal(e["b"], torch.tensor([0, 1, 2, 0, 1, 2]))
    v = e.view(2, 3).permute(1, 0)
    assert v.batch_size == (3, 2) and v["a"].shape == (3, 2, 4)
    assert td[1:]["a"].shape == (2, 4) and td[1:].batch_size == (2,)
    c = td.clone()
    c["a"] += 1
    assert not torch.equal(c["a"], td["a"])
    td.update({"c": torch.zeros(3, 1)})
    assert set(td.keys()) == {"a", "b", "c"}
    assert td.get("zz", None) is None
    g = td.gather(0, torch.tensor([2, 0]))
    assert torch.equal(g["b"], torch.tensor([2, 0]))


def test_layout_helpers_match_reference_golden(golden):
    from rl4co_b200 import ops
    from rl4co_b200.envs import get_env
    from rl4co_b200.tensordict import TensorDict

    g = golden("layout")
    x = g["x"]
    assert torch.equal(ops.batchify(x, 4), g["batchify4"])
    assert torch.equal(ops.unbatchify(ops.batchify(x, 4), 4)[:, 0], x)  # reference tests/test_utils.py:12-28
    r = torch.arange(3 * 8 * 4, dtype=torch.float32)
    assert torch.equal(ops.unbatchify(r, (8, 4)), g["unbatchify_8_4"])
    assert torch.equal(ops.dihedral_8_augmentation(x), g["dihedral8"])
    td = TensorDict({"locs": x.clone()}, batch_size=[3])
    assert torch.equal(ops.StateAugmentation()(td)["locs"], g["state_aug"])
    tdb = ops.batchify(td, 4)
    assert torch.equal(tdb["locs"], g["batchify4"])
    assert torch.equal(ops.unbatchify(tdb, 4)["locs"][:, 0], x)
    for name, key in (("tsp", "tsp"), ("cvrp", "cvrp")):
        env = get_env(name, generator_params=dict(num_loc=5))
        fake = TensorDict({"action_mask": torch.ones(3, 5 + (name == "cvrp"), dtype=torch.bool)}, batch_size=[3])
        assert env.get_num_starts(fake) == int(g[f"{key}_num_starts"])
        assert torch.equal(env.select_start_nodes(fake, 5), g[f"{key}_starts"])


def test_env_reset_keys_dtypes_shapes_cpu():
    from rl4co_b200.envs import get_env

    env = get_env("tsp", generator_params=dict(num_loc=12))
    td = env.reset(batch_size=[5])
    assert td["locs"].shape == (5, 12, 2) and td["locs"].dtype == torch.float32
    assert td["first_node"].shape == (5,) and td["current_node"].dtype == torch.int64
    assert td["i"].shape == (5, 1) and td["action_mask"].dtype == torch.bool and td["action_mask"].all()
    assert td["done"].shape == (5, 1) and td["done"].dtype == torch.bool and td["reward"].shape == (5, 1)
    gen = get_env("cvrp", generator_params=dict(num_loc=50)).generator(7)
    assert gen["locs"].shape == (7, 50, 2) and gen["depot"].shape == (7, 2) and gen["demand"].shape == (7, 50)
    k = (gen["demand"] * 40.0).round()
    assert ((k >= 1) & (k <= 9)).all() and torch.allclose(gen["demand"], k / 40.0)


def test_generators_match_reference_call_order():
    """same torch RNG consumption as rl4co's generators (checked vs the live reference in
    tests/test_oracle_vs_reference.py through the oracle's generate_instances)."""
    from oracle import am_rollout_oracle as O
    from rl4co_b200.envs import get_env

    for name, n in (("tsp", 50), ("cvrp", 50), ("cvrp", 100), ("op", 20), ("op", 50), ("pctsp", 20), ("pctsp", 100)):
        env = get_env(name, generator_params=dict(num_loc=n))
        torch.manual_seed(1234)
        td = env.generator(6)
        torch.manual_seed(1234)
        inst = O.generate_instances(name, 6, n)
        for k in inst:
            assert torch.equal(td[k], inst[k]), (name, k)


@pytest.mark.parametrize("name", ["am_tsp20", "am_cvrp20", "enc_tsp20_batch", "enc_cvrp20_instance"])
def test_reference_state_dict_names_load(golden, name):
    from rl4co_b200.policy import FusedAttentionModelPolicy

    g = golden(name)
    env_name = "tsp" if "tsp" in name else "cvrp"
    norm = "instance" if "instance" in name else "batch"
    pol = FusedAttentionModelPolicy(env_name=env_name, num_encoder_layers=1, normalization=norm)
    sd = pol.state_dict()
    w = g.weights()
    for k, v in w.items():
        assert k in sd and sd[k].shape == v.shape, k
    missing, unexpected = pol.load_state_dict(w, strict=False)
    assert not unexpected


@pytest.mark.parametrize("name,norm", [("enc_tsp20_batch", "batch"), ("enc_cvrp20_instance", "instance")])
def test_encoder_matches_reference_golden_cpu(golden, name, norm):
    """the encoder is stock PyTorch (SURVEY.md 8f-1) and therefore runs on CPU too."""
    from rl4co_b200.envs import get_env
    from rl4co_b200.policy import FusedAttentionModelPolicy
    from rl4co_b200.tensordict import TensorDict

    g = golden(name)
    env_name = "tsp" if "tsp" in name else "cvrp"
    pol = FusedAttentionModelPolicy(env_name=env_name, num_encoder_layers=1, normalization=norm).eval()
    pol.load_state_dict(g.weights(), strict=False)
    inst = g.inst()
    env = get_env(env_name, generator_params=dict(num_loc=inst["locs"].shape[1]))
    td = env.reset(TensorDict(inst, batch_size=[inst["locs"].shape[0]])) if env_name == "tsp" else None
    if td is None:  # CVRP reset computes the action mask on the GPU; build the encoder inputs by hand
        td = TensorDict({"locs": torch.cat((inst["depot"][:, None], inst["locs"]), 1), "demand": inst["demand"]},
                        batch_size=[inst["locs"].shape[0]])
    with torch.inference_mode():
        h, init_h = pol.encoder(td)
    torch.testing.assert_close(init_h, g["init_h"], rtol=1e-6, atol=1e-6)
    torch.testing.assert_close(h, g["h"], rtol=1e-5, atol=1e-5)


def test_fused_weight_blocks_cpu(golden):
    """the single cache GEMM reproduces K / V and the folded logit key / context tables."""
    from rl4co_b200.decoder import FusedAttentionModelDecoder

    g = golden("am_tsp20")
    dec = FusedAttentionModelDecoder(env_name="tsp")
    w = {k[len("decoder."):]: v for k, v in g.weights().items()}
    dec.load_state_dict(w)
    h = g["h"]
    with torch.inference_mode():
        c = dec._precompute_cache(h)  # default layout: with the first-node table
        c4 = dec._precompute_cache(h, first_table=False)  # narrow layout (per-episode GEMV in the kernel)
    E = 128
    assert c.rollout_cache.shape[-1] == 5 * E and c4.rollout_cache.shape[-1] == 4 * E
    kvl = torch.nn.functional.linear(h, w["project_node_embeddings.weight"])
    torch.testing.assert_close(c.glimpse_key, kvl[..., :E], rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(c.glimpse_val, kvl[..., E:2 * E], rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(c.logit_key, kvl[..., 2 * E:], rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(c.logit_key_folded, kvl[..., 2 * E:] @ w["pointer.project_out.weight"], rtol=1e-4, atol=1e-4)
    wc = w["context_embedding.project_context.weight"]
    torch.testing.assert_close(c.rollout_cache[..., 3 * E:4 * E], h @ wc[:, :E].t(), rtol=1e-4, atol=1e-4)
    torch.testing.assert_close(c.rollout_cache[..., 4 * E:5 * E], h @ wc[:, E:].t(), rtol=1e-4, atol=1e-4)
    torch.testing.assert_close(c4.rollout_cache[..., :3 * E], c.rollout_cache[..., :3 * E])
    torch.testing.assert_close(c4.rollout_cache[..., 3 * E:], c.rollout_cache[..., 4 * E:])
    assert torch.equal(c4.w_first, wc[:, :E])
    # the concatenated weight is cached per weight version and refreshed when a parameter changes
    w0 = dec._fused_weight_cached(False)[0]
    assert dec._fused_weight_cached(False)[0] is w0
    with torch.no_grad():
        dec.pointer.project_out.weight.mul_(2.0)
    assert dec._fused_weight_cached(False)[0] is not w0
    torch.testing.assert_close(c.q_placeholder, wc @ w["context_embedding.W_placeholder"], rtol=1e-5, atol=1e-5)


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "rl4co_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert "oracle" not in src.replace("the oracle", "").replace("oracle's", "") or fn == "tensordict.py", fn


def test_no_cpu_fallback():
    from rl4co_b200 import native
    from rl4co_b200.envs import get_env

    env = get_env("cvrp", generator_params=dict(num_loc=10))
    td = env.reset(batch_size=[4])  # reset only allocates state: works on any device (ADVICE r1)
    assert td["action_mask"].shape == (4, 11) and not td["action_mask"][:, 0].any() and td["action_mask"][:, 1:].all()
    td.set("action", torch.ones(4, dtype=torch.int64))
    with pytest.raises(native.NativeLibraryError):
        env.step(td)  # every arithmetic entry point is CUDA-only
    with pytest.raises(native.NativeLibraryError):
        env.get_action_mask(td)
    with pytest.raises(native.NativeLibraryError):
        get_env("tsp", generator_params=dict(num_loc=5)).get_reward(
            get_env("tsp", generator_params=dict(num_loc=5)).reset(batch_size=[2]), torch.arange(5).repeat(2, 1))


def test_unsupported_options_are_rejected():
    from rl4co_b200.decoder import FusedAttentionModelDecoder
    from rl4co_b200.decoding import get_decoding_strategy

    with pytest.raises(NotImplementedError):
        FusedAttentionModelDecoder(embed_dim=256)
    with pytest.raises(NotImplementedError):
        FusedAttentionModelDecoder(env_name="cvrptw")
    with pytest.raises(NotImplementedError):
        get_decoding_strategy("lookahead")
    with pytest.raises(AssertionError):
        get_decoding_strategy("sampling", top_p=1.5)


@pytest.mark.parametrize("top_k,top_p", [(3, 0.0), (0, 0.7), (5, 0.9), (40, 0.0), (0, 1.0), (1, 0.5)])
def test_top_k_top_p_filters_match_oracle(top_k, top_p):
    """The host-side filters of the stepping path (library ops, device-agnostic) keep exactly the set the oracle's
    process_logits keeps -- including masked (-inf) entries, ties at the k-th value and a nucleus that ends mid-tie."""
    from oracle import am_rollout_oracle as O
    from rl4co_b200.decoding import keep_top_k, keep_top_p

    torch.manual_seed(top_k * 10 + int(top_p * 100))
    logits = torch.randn(64, 21) * 3
    logits[:, 5] = logits[:, 4]  # a tie
    mask = torch.rand(64, 21) > 0.3
    mask[:, 0] = True
    z = (torch.tanh(logits) * 10.0).masked_fill(~mask, float("-inf")) / 0.8
    if top_k > 0:
        z = keep_top_k(z, min(top_k, z.size(-1)))
    if top_p > 0:
        z = keep_top_p(z, top_p)
    ref = O.process_logits(logits.clone(), mask, temperature=0.8, tanh_clipping=10.0, top_k=top_k, top_p=top_p)
    assert torch.equal(torch.isfinite(z), torch.isfinite(ref))
    torch.testing.assert_close(torch.log_softmax(z, -1), ref, rtol=0, atol=0)
    if top_k > 0 and top_p == 0:
        assert (torch.isfinite(z).sum(-1) >= torch.minimum(mask.sum(-1), torch.tensor(min(top_k, 21)))).all()


@pytest.mark.parametrize("B,W,N", [(5, 3, 7), (1, 4, 4), (6, 2, 11)])
def test_beam_expand_and_backtrack(B, W, N):
    """Beam bookkeeping of the stepping path (device-agnostic index arithmetic): the expansion keeps the W best
    (parent, node) pairs per instance in the reference's row order, and back-tracking returns, for every final beam,
    the sequence obtained by following its parent pointers one step at a time."""
    from rl4co_b200.decoding import beam_backtrack, beam_expand

    torch.manual_seed(B * 100 + W * 10 + N)
    T = 6
    cum = torch.zeros(B * W, 1)
    acts, lps, pars = [torch.randint(0, N, (B * W,))], [torch.zeros(B * W, N)], [torch.zeros(B * W, dtype=torch.int32)]
    for _ in range(T - 1):
        lp = torch.log_softmax(torch.randn(B * W, N) * 2, -1)
        lp[torch.rand(B * W, N) < 0.2] = float("-inf")
        lp[:, 0] = torch.where(torch.isinf(lp).all(1), torch.zeros(()), lp[:, 0])
        node, parent, src, new_cum = beam_expand(lp, cum, W)
        # per-instance brute force: all (w, n) pairs ranked by cumulative log-prob
        for b in range(B):
            pairs = sorted(((float(lp[w * B + b, n] + cum[w * B + b, 0]), w, n) for w in range(W) for n in range(N)),
                           key=lambda x: -x[0])[:W]
            for k, (score, w, n) in enumerate(pairs):
                r = k * B + b
                assert abs(float(new_cum[r, 0]) - score) < 1e-6
                if sum(abs(p[0] - score) < 1e-9 for p in pairs) == 1:  # untied: the exact pair must match
                    assert (int(parent[r]), int(node[r]), int(src[r])) == (w, n, w * B + b)
        cum = new_cum
        acts.append(node), lps.append(lp[src]), pars.append(parent)
    A, L, P = torch.stack(acts, 1), torch.stack(lps, 1), torch.stack(pars, 1)
    out_a, out_lp = beam_backtrack(A, L, P, W)
    for r in range(B * W):
        cur, b = r, r % B
        for k in range(T - 1, -1, -1):
            assert out_a[r, k] == A[cur, k]
            assert torch.equal(out_lp[r, k], L[cur, k])
            cur = b + int(P[cur, k]) * B
    # a sequence's cumulative log-prob equals the beam score it ended with
    got = out_lp.gather(-1, out_a.unsqueeze(-1)).squeeze(-1).sum(1)
    torch.testing.assert_close(got, cum.squeeze(1), rtol=1e-5, atol=1e-5)


def test_bench_reference_arm_line_schema():
    """`bench.py --impl reference` (the CPU arm the driver times beside ours) runs without a GPU and prints one JSON
    line with the contract's keys."""
    import json
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "1", "--cpu-batch", "8", "--workload", "c2"], capture_output=True, text=True,
                         timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["higher_is_better"] is True and line["unit"] == "selections/s"
    for key in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "dtype", "data", "config",
                "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["value"] > 0 and line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    # the unmodified reference files (live tree or the staged oracle/_ref copy) when present, else the oracle port
    from oracle import ref_standin

    assert line["cpu_baseline"]["kind"] == ("reference" if ref_standin.reference_available() else "port")
    assert line["cpu_baseline"]["cores"] >= 1 and line["cpu_baseline"]["single_process"]["value"] > 0


def test_seeded_dataset_generation_matches_reference(tmp_path):
    """data/generate_data.py:37-76,213-317: the numpy-seeded validation / test sets are bit-identical to the
    reference's; `env.dataset(phase=...)` loads them (SURVEY.md 8f-3)."""
    import numpy as np

    from rl4co_b200 import data as D
    from rl4co_b200.envs import get_env

    files = D.generate_default_datasets(str(tmp_path), dataset_size=16, graph_sizes=(20, 50))
    assert len(files) == 8 and all(os.path.isfile(f) for f in files)
    assert os.path.basename(files[0]) == "tsp20_val_seed4321.npz" and os.path.basename(files[-1]) == "vrp50_test_seed1234.npz"
    # the reference's own sets, recorded by tests/golden/make_golden.py (ref_datasets.npz)
    ref = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_datasets.npz"))
    for prob, gs, seed, name in (("tsp", 20, 4321, "val"), ("vrp", 50, 1234, "test")):
        prefix = f"{prob}{gs}_{name}/"
        want = {k[len(prefix):]: ref[k] for k in ref.files if k.startswith(prefix)}
        got = np.load(D.dataset_filename(str(tmp_path), prob, gs, name, seed))
        assert want and set(got.files) == set(want)
        for k in want:
            assert np.array_equal(got[k], want[k]), (prob, k)
    env = get_env("cvrp", generator_params=dict(num_loc=20), data_dir=str(tmp_path), val_file="vrp/vrp20_val_seed4321.npz")
    ds = env.dataset(phase="val")
    assert len(ds) == 16
    raw = np.load(D.dataset_filename(str(tmp_path), "vrp", 20, "val", 4321))
    np.testing.assert_allclose(ds[0]["demand"].numpy(), raw["demand"][0] / raw["capacity"][0])  # cvrp/env.py:179-186
    assert len(env.dataset(batch_size=[5], phase="train")) == 5          # no train file: generated
    assert len(env.dataset(batch_size=[7], phase="test")) == 7           # test file unset: generated


@pytest.mark.parametrize("name", ["am_tsp20", "am_cvrp20", "am_tsp50", "am_cvrp50"])
def test_teacher_forced_pass_matches_reference_logprobs_cpu(golden, name):
    """The vectorised teacher-forced pass of the training step (replay of the MDP without a time loop + one batched
    attention over all decode steps) is plain torch off the GPU: its per-step log-probabilities along the reference's
    recorded trajectories equal the log-probabilities the reference recorded step by step
    (models/common/constructive/base.py:176-238 with `actions=`; multistart: decoding.py:300-345)."""
    from conftest import env_of
    from rl4co_b200.envs import get_env
    from rl4co_b200.policy import FusedAttentionModelPolicy
    from rl4co_b200.reinforce import evaluate_log_likelihood
    from rl4co_b200.tensordict import TensorDict

    g = golden(name)
    env_name = env_of(name)
    pol = FusedAttentionModelPolicy(env_name=env_name, num_encoder_layers=1).eval()
    pol.load_state_dict({**pol.state_dict(), **g.weights()})
    inst, h = g.inst(), g["h"]
    B = h.shape[0]
    env = get_env(env_name, generator_params=dict(num_loc=inst["locs"].shape[1]))
    td = env.reset(TensorDict(inst, batch_size=[B]))
    for mode in ("greedy", "sampling", "eval"):
        lp = evaluate_log_likelihood(pol, td, env, g[f"{mode}_actions"], hidden=h, return_sum=False)
        torch.testing.assert_close(lp, g[f"{mode}_logprobs"], rtol=1e-5, atol=2e-5)
        assert lp.requires_grad
    mb = int(g["ms_batch"])
    tdm = env.reset(TensorDict({k: v[:mb] for k, v in inst.items()}, batch_size=[mb]))
    lp = evaluate_log_likelihood(pol, tdm, env, g["ms_actions"], hidden=h[:mb], return_sum=False)
    torch.testing.assert_close(lp, g["ms_logprobs"], rtol=1e-5, atol=2e-5)
    assert (lp[:, 0] == 0).all()   # the forced start node carries no log-probability


@pytest.mark.parametrize("name", ["am_op20", "am_op50", "am_pctsp20", "am_pctsp50"])
def test_teacher_forced_pass_budget_envs_cpu(golden, name):
    """Orienteering / prize-collecting TSP: the replay of tour length / collected prize without the env (one fp32
    running total per instance) gives the reference's masks bit for bit, and the one-call teacher-forced pass the
    reference's recorded log-probabilities; longer near-uniform trajectories are checked against the oracle."""
    from conftest import env_of
    from oracle import am_rollout_oracle as O
    from rl4co_b200.envs import get_env
    from rl4co_b200.policy import FusedAttentionModelPolicy
    from rl4co_b200.reinforce import evaluate_log_likelihood, replay_budget_states
    from rl4co_b200.tensordict import TensorDict

    g = golden(name)
    env_name = env_of(name)
    pol = FusedAttentionModelPolicy(env_name=env_name, num_encoder_layers=1).eval()
    pol.load_state_dict({**pol.state_dict(), **g.weights()})
    inst, h = g.inst(), g["h"]
    B = h.shape[0]
    gp = dict(num_loc=inst["locs"].shape[1])
    if env_name == "op":
        gp["prize_type"] = "dist"
    env = get_env(env_name, generator_params=gp)
    td = env.reset(TensorDict(inst, batch_size=[B]))
    for mode in ("greedy", "sampling", "eval"):
        lp = evaluate_log_likelihood(pol, td, env, g[f"{mode}_actions"], hidden=h, return_sum=False)
        torch.testing.assert_close(lp, g[f"{mode}_logprobs"], rtol=1e-5, atol=2e-5)
    mask, _, _ = replay_budget_states(env_name, td, g["greedy_actions"])
    assert torch.equal(mask.transpose(0, 1), g["greedy_masks"].bool())
    # near-uniform random feasible tours from the oracle (temperature 50), many instances: every mask and log-prob
    gen = torch.Generator().manual_seed(11)
    inst2 = O.generate_instances(env_name, 96, gp["num_loc"], generator=gen)
    w = g.weights()
    h2 = torch.randn(96, gp["num_loc"] + 1, 128, generator=gen)   # any node embeddings do: the decoder is under test
    with torch.no_grad():
        ref = O.rollout(w, env_name, inst2, h2, decode_type="sampling", temperature=50.0, generator=gen, return_trace=True)
    assert ref["actions"].shape[1] > 5
    td2 = env.reset(TensorDict(inst2, batch_size=[96]))
    mask, _, _ = replay_budget_states(env_name, td2, ref["actions"])
    assert torch.equal(mask, torch.stack(ref["trace"]["mask"], 1))
    lp = evaluate_log_likelihood(pol, td2, env, ref["actions"], hidden=h2.clone().requires_grad_(), return_sum=False,
                                 temperature=50.0)
    torch.testing.assert_close(lp, ref["logprobs"], rtol=1e-5, atol=2e-5)
    lp.sum().backward()   # the graph reaches the decoder weights
    assert pol.decoder.context_embedding.project_context.weight.grad.abs().sum() > 0


@pytest.mark.parametrize("name", ["am_sdvrp20", "am_sdvrp50"])
def test_teacher_forced_pass_split_delivery_cpu(golden, name):
    """SDVRP: the per-step dynamic embedding applied as rank-one terms on scores / head outputs / logits (no per-step
    copies of K / V / L) reproduces the reference's recorded log-probabilities; masks bit for bit."""
    from oracle import am_rollout_oracle as O
    from rl4co_b200.envs import get_env
    from rl4co_b200.policy import FusedAttentionModelPolicy
    from rl4co_b200.reinforce import evaluate_log_likelihood, replay_split_delivery_states
    from rl4co_b200.tensordict import TensorDict

    g = golden(name)
    pol = FusedAttentionModelPolicy(env_name="sdvrp", num_encoder_layers=1).eval()
    pol.load_state_dict({**pol.state_dict(), **g.weights()})
    inst, h = g.inst(), g["h"]
    B = h.shape[0]
    env = get_env("sdvrp", generator_params=dict(num_loc=inst["locs"].shape[1]))
    td = env.reset(TensorDict(inst, batch_size=[B]))
    for mode in ("greedy", "sampling", "eval"):
        lp = evaluate_log_likelihood(pol, td, env, g[f"{mode}_actions"], hidden=h, return_sum=False)
        torch.testing.assert_close(lp, g[f"{mode}_logprobs"], rtol=1e-5, atol=2e-5)
    mask = replay_split_delivery_states(td, g["greedy_actions"])[0]
    assert torch.equal(mask.transpose(0, 1), g["greedy_masks"].bool())
    gen = torch.Generator().manual_seed(5)
    n = inst["locs"].shape[1]
    inst2 = O.generate_instances("sdvrp", 64, n, generator=gen)
    h2 = torch.randn(64, n + 1, 128, generator=gen)
    with torch.no_grad():
        ref = O.rollout(g.weights(), "sdvrp", inst2, h2, decode_type="sampling", temperature=20.0, generator=gen,
                        return_trace=True)
    td2 = env.reset(TensorDict(inst2, batch_size=[64]))
    assert torch.equal(replay_split_delivery_states(td2, ref["actions"])[0], torch.stack(ref["trace"]["mask"], 1))
    lp = evaluate_log_likelihood(pol, td2, env, ref["actions"], hidden=h2, return_sum=False, temperature=20.0)
    torch.testing.assert_close(lp, ref["logprobs"], rtol=1e-5, atol=2e-5)
    lp.sum().backward()
    assert pol.decoder.dynamic_embedding.projection.weight.grad.abs().sum() > 0


@pytest.mark.parametrize("name", ["am_tsp20", "am_cvrp20", "am_op20", "am_pctsp20"])
def test_teacher_forced_pass_multistart_cpu(golden, name):
    """POMO-style training: S forced start nodes per instance become S * T queries against one K / V; start-major
    [S * B, T] actions in, the oracle's multistart log-probabilities out (the start column carries 0)."""
    from conftest import env_of
    from oracle import am_rollout_oracle as O
    from rl4co_b200.envs import get_env
    from rl4co_b200.policy import FusedAttentionModelPolicy
    from rl4co_b200.reinforce import evaluate_log_likelihood
    from rl4co_b200.tensordict import TensorDict

    g = golden(name)
    env_name = env_of(name)
    pol = FusedAttentionModelPolicy(env_name=env_name, num_encoder_layers=1).eval()
    pol.load_state_dict({**pol.state_dict(), **g.weights()})
    gen = torch.Generator().manual_seed(3)
    n = g.inst()["locs"].shape[1]
    inst = O.generate_instances(env_name, 12, n, generator=gen)
    h = torch.randn(12, n + (0 if env_name == "tsp" else 1), 128, generator=gen)
    with torch.no_grad():
        ref = O.rollout(g.weights(), env_name, inst, h, decode_type="multistart_sampling", num_starts=5, temperature=20.0,
                        generator=gen)
    env = get_env(env_name, generator_params=dict(num_loc=n))
    td = env.reset(TensorDict(inst, batch_size=[12]))
    lp = evaluate_log_likelihood(pol, td, env, ref["actions"], hidden=h, return_sum=False, temperature=20.0)
    torch.testing.assert_close(lp, ref["logprobs"], rtol=1e-5, atol=2e-5)
    assert (lp[:, 0] == 0).all()
