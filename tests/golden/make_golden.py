"""Generate the golden vectors under tests/golden/ by executing rl4co's OWN, unmodified
hot-path files from /root/reference (through oracle/ref_standin.py -- container stubs for
tensordict/torchrl/lightning only, no arithmetic).

Run in the build container only (the GPU box has no /root/reference):

    python tests/golden/make_golden.py

Every array written here is produced by reference code + PyTorch CPU fp32.  The fixtures
pin (a) the env MDP (masks / visited / capacity / done / reward) under the reference's
``random_policy`` rollout, (b) the AM decoder path (raw logits per step, log-probs,
actions, reward, log-likelihood) for greedy, sampling-with-recorded-Exp(1)-noise,
multistart-greedy and teacher-forced evaluation, (c) the AM encoder, and (d) the
batchify / dihedral-8 layout conventions.
"""

from __future__ import annotations

import json
import os
import sys
import zlib

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import ref_standin  # noqa: E402

ref = ref_standin.load()
TensorDict = ref.TensorDict


def npy(x):
    return x.detach().cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)


def make_env(name, n, check=True):
    if name == "sdvrp":
        import importlib

        Env = importlib.import_module("rl4co.envs.routing.sdvrp.env").SDVRPEnv
    elif name == "op":
        import importlib

        Env = importlib.import_module("rl4co.envs.routing.op.env").OPEnv
    elif name == "pctsp":
        import importlib

        Env = importlib.import_module("rl4co.envs.routing.pctsp.env").PCTSPEnv
    else:
        Env = ref.TSPEnv if name == "tsp" else ref.CVRPEnv
    if name == "op":
        # the generator's default prize_distribution builds Uniform(1.0, 1.0), which current torch rejects at
        # construction; "dist" skips that sampler (it is unused: the prizes come from prize_type, op/generator.py:115-125)
        return Env(generator_params=dict(num_loc=n, prize_distribution="dist"), check_solution=check)
    return Env(generator_params=dict(num_loc=n), check_solution=check)


def env_fixture(name, n, batch, seed):
    """Reference env driven by the reference's random_policy (utils/decoding.py:78-106)."""
    torch.manual_seed(seed)
    env = make_env(name, n)
    td0 = env.generator(batch_size=[batch])
    out = {f"inst::{k}": npy(td0[k]) for k in td0.keys()}
    td = env.reset(td0.clone())
    masks, dones, visited, used, cur = [npy(td["action_mask"])], [], [], [], []
    actions = []
    while not td["done"].all():
        td = ref.decoding.random_policy(td)
        actions.append(td["action"].clone())
        td = env.step(td)["next"]
        masks.append(npy(td["action_mask"]))
        dones.append(npy(td["done"]))
        cur.append(npy(td["current_node"]).reshape(batch))
        if name == "cvrp":
            visited.append(npy(td["visited"]))
            used.append(npy(td["used_capacity"]))
        if name == "sdvrp":
            visited.append(npy(td["demand_with_depot"]))  # the dynamic state of the split-delivery env
            used.append(npy(td["used_capacity"]))
        if name == "op":
            visited.append(npy(td["visited"]))
            used.append(np.stack([npy(td["tour_length"]), npy(td["current_total_prize"])]))
        if name == "pctsp":
            visited.append(npy(td["visited"]))
            used.append(np.stack([npy(td["cur_total_prize"]), npy(td["cur_total_penalty"])]))
    actions = torch.stack(actions, 1)
    reward = env.get_reward(td, actions)  # runs check_solution_validity too
    out.update(actions=npy(actions), action_mask=np.stack(masks), done=np.stack(dones),
               current_node=np.stack(cur), reward=npy(reward))
    if name == "cvrp":
        out.update(visited=np.stack(visited), used_capacity=np.stack(used))
    elif name == "sdvrp":
        out.update(demand_with_depot=np.stack(visited), used_capacity=np.stack(used))
    elif name == "op":
        st = np.stack(used)  # [T, 2, B]
        out.update(visited=np.stack(visited), tour_length=st[:, 0], current_total_prize=st[:, 1])
    elif name == "pctsp":
        st = np.stack(used)
        out.update(visited=np.stack(visited), cur_total_prize=st[:, 0], cur_total_penalty=st[:, 1])
    else:
        out.update(first_node=npy(td["first_node"]), i=npy(td["i"]))
    return out


def sdvrp_am_fixture(n, batch, seed, name="sdvrp"):
    """A sibling env through the reference AttentionModelPolicy -- SDVRP (VRPContext + SDVRPDynamicEmbedding,
    dynamic.py:60-78) or OP (OPInitEmbedding init.py:254-280, OPContext context.py:201-213): greedy, sampling with
    recorded noise, teacher-forced evaluation -- single-start decoding."""
    torch.manual_seed(seed)
    env = make_env(name, n)
    pol = ref.AttentionModelPolicy(env_name=name, num_encoder_layers=1).eval()
    if name == "sdvrp":
        with torch.no_grad():  # the default init of a Linear(1, 3E) is small next to the static keys: make it count
            pol.decoder.dynamic_embedding.projection.weight.mul_(3.0)
    keep = ("decoder.",) if name == "sdvrp" else ("decoder.", "encoder.")
    out = {"w::" + k: npy(v) for k, v in pol.state_dict().items() if k.startswith(keep)}
    td0 = env.generator(batch_size=[batch])
    for k in td0.keys():
        out[f"inst::{k}"] = npy(td0[k])
    rec = Recorder(pol.decoder)
    with torch.inference_mode():
        td = env.reset(td0.clone())
        h, _ = pol.encoder(td)
        out["h"] = npy(h)
        o = pol(td.clone(), env, phase="test", decode_type="greedy", return_sum_log_likelihood=False)
        lg, mk = rec.pop()
        out.update(greedy_actions=npy(o["actions"]), greedy_logprobs=npy(o["log_likelihood"]),
                   greedy_reward=npy(o["reward"]), greedy_logits=lg, greedy_masks=mk)
        torch.manual_seed(seed + 1)
        o = pol(td.clone(), env, phase="train", decode_type="sampling", return_sum_log_likelihood=False)
        lg, mk = rec.pop()
        T = o["actions"].shape[1]
        torch.manual_seed(seed + 1)
        q = torch.stack([torch.empty(batch, lg.shape[-1]).exponential_(1) for _ in range(T)])
        out.update(sampling_actions=npy(o["actions"]), sampling_logprobs=npy(o["log_likelihood"]),
                   sampling_reward=npy(o["reward"]), sampling_noise=npy(q))
        torch.manual_seed(seed + 2)
        tdr = env.reset(td0.clone())
        acts = []
        while not tdr["done"].all():
            tdr = ref.decoding.random_policy(tdr)
            acts.append(tdr["action"].clone())
            tdr = env.step(tdr)["next"]
        acts = torch.stack(acts, 1)
        o = pol(td.clone(), env, phase="train", actions=acts, return_sum_log_likelihood=False)
        lg, mk = rec.pop()
        out.update(eval_actions=npy(acts), eval_logprobs=npy(o["log_likelihood"]), eval_reward=npy(o["reward"]),
                   eval_logits=lg)
    return out


class Recorder:
    """Forward hook on the reference decoder recording raw (logits, mask) per step."""

    def __init__(self, decoder):
        self.logits, self.masks = [], []
        self.h = decoder.register_forward_hook(self._hook)

    def _hook(self, mod, args, output):
        self.logits.append(output[0].detach().clone())
        self.masks.append(output[1].detach().clone())

    def pop(self):
        lg, mk = torch.stack(self.logits), torch.stack(self.masks)
        self.logits, self.masks = [], []
        return npy(lg), npy(mk)


def am_fixture(name, n, batch, seed, ms_batch=3, lean=False):
    """`lean` drops the recorded sampling / multistart logits (4 MB at N = 100); the greedy and
    teacher-forced logits, every action / log-prob / reward and the consumed noise stay."""
    torch.manual_seed(seed)
    env = make_env(name, n)
    pol = ref.AttentionModelPolicy(env_name=name, num_encoder_layers=1).eval()
    # make the decoder more "opinionated" than default init so that argmax margins are healthy
    out = {}
    for k, v in pol.state_dict().items():
        if k.startswith("decoder."):
            out["w::" + k] = npy(v)
    td0 = env.generator(batch_size=[batch])
    for k in td0.keys():
        out[f"inst::{k}"] = npy(td0[k])
    rec = Recorder(pol.decoder)
    with torch.inference_mode():
        td = env.reset(td0.clone())
        h, _ = pol.encoder(td)
        out["h"] = npy(h)
        # -- greedy
        o = pol(td.clone(), env, phase="test", decode_type="greedy", return_sum_log_likelihood=False)
        lg, mk = rec.pop()
        out.update(greedy_actions=npy(o["actions"]), greedy_logprobs=npy(o["log_likelihood"]),
                   greedy_reward=npy(o["reward"]), greedy_logits=lg, greedy_masks=mk)
        # -- sampling; the Exp(1) draws consumed by torch.multinomial are regenerated
        torch.manual_seed(seed + 1)
        o = pol(td.clone(), env, phase="train", decode_type="sampling", return_sum_log_likelihood=False)
        lg, mk = rec.pop()
        T = o["actions"].shape[1]
        torch.manual_seed(seed + 1)
        q = torch.stack([torch.empty(batch, lg.shape[-1]).exponential_(1) for _ in range(T)])
        out.update(sampling_actions=npy(o["actions"]), sampling_logprobs=npy(o["log_likelihood"]),
                   sampling_reward=npy(o["reward"]), sampling_noise=npy(q))
        if not lean:
            out.update(sampling_logits=lg)
        # -- teacher-forced evaluation of an independent (random-policy) action sequence
        torch.manual_seed(seed + 2)
        tdr = env.reset(td0.clone())
        acts = []
        while not tdr["done"].all():
            tdr = ref.decoding.random_policy(tdr)
            acts.append(tdr["action"].clone())
            tdr = env.step(tdr)["next"]
        acts = torch.stack(acts, 1)
        o = pol(td.clone(), env, phase="train", actions=acts, return_sum_log_likelihood=False)
        lg, mk = rec.pop()
        out.update(eval_actions=npy(acts), eval_logprobs=npy(o["log_likelihood"]), eval_reward=npy(o["reward"]),
                   eval_logits=lg)
        # -- multistart greedy on the first ms_batch instances (start-major layout)
        tdm = env.reset(td0[:ms_batch].clone())
        o = pol(tdm.clone(), env, phase="test", decode_type="multistart_greedy", return_sum_log_likelihood=False)
        lg, mk = rec.pop()
        out.update(ms_actions=npy(o["actions"]), ms_logprobs=npy(o["log_likelihood"]), ms_reward=npy(o["reward"]),
                   ms_batch=np.int64(ms_batch))
        if not lean:
            out.update(ms_logits=lg)
        # -- POMO-style: no graph context (pomo/model.py:59-63)
        polp = ref.AttentionModelPolicy(env_name=name, num_encoder_layers=1, use_graph_context=False).eval()
        polp.load_state_dict(pol.state_dict())
        o = polp(tdm.clone(), env, phase="test", decode_type="multistart_greedy", return_sum_log_likelihood=False)
        out.update(pomo_actions=npy(o["actions"]), pomo_logprobs=npy(o["log_likelihood"]), pomo_reward=npy(o["reward"]))
    return out


def decoding_fixture(name, n, batch, seed):
    """Beam search and top-k / top-p sampling (utils/decoding.py:109-188,464-600) on the SAME policy and instances
    as am_fixture(name, n, batch, seed): the seed sequence up to the generator call is replayed, weights and
    instances are not stored again (`h` is, as a guard)."""
    torch.manual_seed(seed)
    env = make_env(name, n)
    pol = ref.AttentionModelPolicy(env_name=name, num_encoder_layers=1).eval()
    td0 = env.generator(batch_size=[batch])
    out = {}
    with torch.inference_mode():
        td = env.reset(td0.clone())
        h, _ = pol.encoder(td)
        out["h"] = npy(h)
        for tag, kw in (("beam3_best", dict(beam_width=3, select_best=True)),
                        ("beam4_all", dict(beam_width=4, select_best=False)),
                        ("beamN_best", dict(select_best=True))):
            o = pol(td.clone(), env, phase="test", decode_type="beam_search", return_sum_log_likelihood=False, **kw)
            out.update({f"{tag}_actions": npy(o["actions"]), f"{tag}_logprobs": npy(o["log_likelihood"]),
                        f"{tag}_reward": npy(o["reward"])})
        for i, (tag, kw) in enumerate((("topk4", dict(top_k=4)), ("topp80", dict(top_p=0.8)),
                                       ("topk6_topp90", dict(top_k=6, top_p=0.9)))):
            torch.manual_seed(seed + 10 + i)
            o = pol(td.clone(), env, phase="train", decode_type="sampling", return_sum_log_likelihood=False, **kw)
            T = o["actions"].shape[1]
            torch.manual_seed(seed + 10 + i)  # the Exp(1) draws torch.multinomial consumed, one [B, N] block per step
            q = torch.stack([torch.empty(batch, td["action_mask"].shape[-1]).exponential_(1) for _ in range(T)])
            out.update({f"{tag}_actions": npy(o["actions"]), f"{tag}_logprobs": npy(o["log_likelihood"]),
                        f"{tag}_reward": npy(o["reward"]), f"{tag}_noise": npy(q)})
    return out


def encoder_fixture(name, n, batch, seed, normalization):
    torch.manual_seed(seed)
    env = make_env(name, n)
    pol = ref.AttentionModelPolicy(env_name=name, num_encoder_layers=1, normalization=normalization).eval()
    if normalization == "batch":  # non-trivial running stats
        for m in pol.modules():
            if isinstance(m, torch.nn.BatchNorm1d):
                m.running_mean.normal_(0, 0.1)
                m.running_var.uniform_(0.5, 1.5)
    out = {"w::" + k: npy(v) for k, v in pol.state_dict().items()
           if k.startswith("encoder.") and "num_batches" not in k}
    td0 = env.generator(batch_size=[batch])
    for k in td0.keys():
        out[f"inst::{k}"] = npy(td0[k])
    with torch.inference_mode():
        td = env.reset(td0.clone())
        h, init_h = pol.encoder(td)
    out.update(h=npy(h), init_h=npy(init_h))
    return out


def name_seeded_weights(module, seed):
    """Deterministic weights that depend only on (parameter name, shape, seed) -- not on module
    construction order -- so the consumer regenerates them instead of the fixture storing 5 MB:
    U(-1/sqrt(fan_in), 1/sqrt(fan_in)) for matrices (torch.nn.Linear's range), U(-.1,.1) for
    vectors, norm weights 1 + U(-.1,.1).  Mirrored by tests/conftest.py::name_seeded_weights."""
    import zlib

    sd = module.state_dict()
    new = {}
    for k in sorted(sd.keys()):
        v = sd[k]
        if not v.dtype.is_floating_point:
            new[k] = v.clone()
            continue
        gen = torch.Generator().manual_seed(seed * 1_000_003 + zlib.crc32(k.encode()))
        u = torch.rand(v.shape, generator=gen) * 2 - 1
        if v.dim() >= 2:
            new[k] = u / (v.shape[-1] ** 0.5)
        elif "W_placeholder" in k:
            new[k] = u
        elif "norm" in k and k.endswith("weight"):
            new[k] = 1 + 0.1 * u
        elif k.endswith("running_var"):
            new[k] = 1 + 0.25 * u
        else:
            new[k] = 0.1 * u
    module.load_state_dict(new)
    return new


def pomo_fixture(n, batch, seed, num_augment=8):
    """BASELINE config C4 at its own scale: TSP-n POMO = 6-layer instance-norm encoder, no graph
    context (zoo/pomo/model.py:59-63), dihedral-8 StateAugmentation (aug-major, data/transforms.py:
    16-38,118-151), multistart greedy with n starts (start-major), then POMO's reductions
    (pomo/model.py:103-136): max over starts, max over augmentations."""
    torch.manual_seed(seed)
    env = make_env("tsp", n, check=True)
    pol = ref.AttentionModelPolicy(env_name="tsp", num_encoder_layers=6, normalization="instance",
                                   use_graph_context=False).eval()
    name_seeded_weights(pol, seed)
    td0 = env.generator(batch_size=[batch])
    out = {"inst::locs": npy(td0["locs"]), "weight_seed": np.int64(seed), "num_augment": np.int64(num_augment)}
    with torch.inference_mode():
        td = env.reset(td0.clone())
        tda = ref.transforms.StateAugmentation(num_augment=num_augment, augment_fn="dihedral8")(td)
        out["aug_locs"] = npy(tda["locs"])
        h, _ = pol.encoder(tda)
        out["h_first_rows"] = npy(h[:2])  # encoder guard: aug 0 of the first two instances
        o = pol(tda.clone(), env, phase="test", decode_type="multistart_greedy", num_starts=n,
                return_sum_log_likelihood=False)
        acts, lp, rew = o["actions"], o["log_likelihood"], o["reward"]
        assert acts.max() < 256
        r = ref.ops.unbatchify(rew, (num_augment, n))            # [B, aug, start]
        max_r, _ = r.max(dim=-1)
        max_aug_r, _ = max_r.max(dim=1)
        out.update(actions=npy(acts).astype(np.uint8), logprobs_sum=npy(lp.sum(1)), reward=npy(rew),
                   logprobs_rows=npy(lp[: 2 * batch]),  # full per-step log-probs of the first rows
                   max_reward=npy(max_r), max_aug_reward=npy(max_aug_r), reward_b_aug_start=npy(r))
    return out


def layout_fixture():
    torch.manual_seed(11)
    x = torch.rand(3, 5, 2)
    aug = ref.transforms.dihedral_8_augmentation(x)
    td = TensorDict({"locs": x.clone()}, batch_size=[3])
    sa = ref.transforms.StateAugmentation(num_augment=8, augment_fn="dihedral8")(td)
    b = ref.ops.batchify(x, 4)
    r = torch.arange(3 * 8 * 4, dtype=torch.float32)
    ub = ref.ops.unbatchify(r, (8, 4))
    env = make_env("tsp", 5)
    envc = make_env("cvrp", 5)
    tdx = env.reset(batch_size=[3])
    tdc = envc.reset(batch_size=[3])
    return dict(x=npy(x), dihedral8=npy(aug), state_aug=npy(sa["locs"]), batchify4=npy(b),
                unbatchify_8_4=npy(ub), tsp_starts=npy(env.select_start_nodes(tdx, 5)),
                cvrp_starts=npy(envc.select_start_nodes(tdc, 5)),
                tsp_num_starts=np.int64(env.get_num_starts(tdx)), cvrp_num_starts=np.int64(envc.get_num_starts(tdc)))


def weight_meta(module):
    """Names / shapes / float flags of a state_dict: with the weight seed this is all a consumer needs to rebuild
    name_seeded_weights (tests/conftest.py::seeded_weights_from_meta)."""
    return np.array(json.dumps({k: [list(v.shape), bool(v.dtype.is_floating_point)]
                                for k, v in module.state_dict().items()}))


def seeded_instances(out, tag, name, n, batch, seed):
    """The reference generator's instances after torch.manual_seed(seed): a consumer regenerates them with the
    project's generator (tests/conftest.py::golden_case) and checks them against the stored CRC-32 of each array."""
    torch.manual_seed(seed)
    env = make_env(name, n)
    td0 = env.generator(batch_size=[batch])
    out[f"{tag}/gen"] = np.array(json.dumps({"env": name, "n": n, "batch": batch, "seed": seed}))
    out.update({f"{tag}/crc::{k}": np.int64(zlib.crc32(npy(td0[k]).tobytes())) for k in td0.keys()})
    return env, td0


def policy_case(out, tag, name, n, batch, seed, layers, decode_type, sample_seed=None, phase="test", evaluate=False,
                step_rows=0, **kw):
    """One reference policy forward on name-seeded weights: seeded instances, actions, log-likelihood, reward, the
    per-step log-probs of the first `step_rows` trajectories (and, with `evaluate`, the teacher-forced pass on its
    own actions).  `sample_seed` seeds the torch generator right before the forward, so a consumer regenerates the
    Exp(1) draws torch.multinomial took."""
    env, td0 = seeded_instances(out, tag, name, n, batch, seed)
    pol = ref.AttentionModelPolicy(env_name=name, num_encoder_layers=layers).eval()
    name_seeded_weights(pol, seed)
    with torch.inference_mode():
        if sample_seed is not None:
            torch.manual_seed(sample_seed)
        o = pol(env.reset(td0.clone()), env, phase=phase, decode_type=decode_type, return_sum_log_likelihood=False, **kw)
        if evaluate:
            e = pol(env.reset(td0.clone()), env, phase=phase, actions=o["actions"], return_sum_log_likelihood=False)
            out.update({f"{tag}/eval_ll": npy(e["log_likelihood"].sum(-1)), f"{tag}/eval_reward": npy(e["reward"]),
                        f"{tag}/eval_logprobs": npy(e["log_likelihood"][:step_rows])})
    acts = o["actions"]
    out.update({f"{tag}/actions": npy(acts).astype(np.uint8) if acts.max() < 256 else npy(acts),
                f"{tag}/ll": npy(o["log_likelihood"].sum(-1)), f"{tag}/reward": npy(o["reward"]),
                f"{tag}/w_meta": weight_meta(pol), f"{tag}/weight_seed": np.int64(seed)})
    if step_rows:
        out[f"{tag}/logprobs"] = npy(o["log_likelihood"][:step_rows])


def ref_policy_fixture():
    """tests/test_oracle_vs_reference.py: the reference's policy forward over decode types, filters, beam search and
    the sibling envs; its generator; process_logits with top-k / top-p."""
    out = {}
    for name, n in (("tsp", 20), ("cvrp", 20), ("tsp", 37), ("cvrp", 33)):
        for dt in ("greedy", "sampling", "multistart_greedy", "multistart_sampling"):
            policy_case(out, f"fwd_{name}{n}_{dt}", name, n, 6, 1000 + n, 2, dt, sample_seed=5)
    for name in ("tsp", "cvrp"):
        policy_case(out, f"multinomial_{name}", name, 20, 32, 3, 1, "sampling", sample_seed=7, phase="train")
        policy_case(out, f"filters_{name}", name, 20, 16, 21, 1, "sampling", sample_seed=9, phase="train", top_k=5,
                    top_p=0.9)
    for name, n in (("tsp", 12), ("cvrp", 11)):
        for bw, sb in ((3, True), (4, False), (None, True)):
            kw = {} if bw is None else {"beam_width": bw}
            policy_case(out, f"beam_{name}{n}_{bw}_{sb}", name, n, 5, 300 + n, 1, "beam_search", select_best=sb, **kw)
    for name, n in (("op", 20), ("op", 33), ("pctsp", 20), ("pctsp", 41), ("sdvrp", 20)):
        for dt in ("greedy", "sampling"):
            policy_case(out, f"sibling_{name}{n}_{dt}", name, n, 8, 2000 + n, 2, dt, sample_seed=5)
    for name, n in (("tsp", 50), ("cvrp", 50), ("cvrp", 100)):
        env = make_env(name, n)
        torch.manual_seed(1234)
        td = env.generator(batch_size=[5])
        out.update({f"gen_{name}{n}/{k}": npy(td[k]) for k in td.keys()})
    for top_k, top_p in ((3, 0.0), (0, 0.6), (4, 0.8), (50, 0.0), (0, 1.0)):
        torch.manual_seed(11 + top_k)
        logits = torch.randn(32, 20) * 2
        logits[:, 7] = logits[:, 3]
        mask = torch.rand(32, 20) > 0.4
        mask[:, 1] = True
        want = ref.decoding.process_logits(logits.clone(), mask, temperature=1.3, top_p=top_p, top_k=top_k,
                                           tanh_clipping=10.0)
        out.update({f"process_{top_k}_{top_p}/logits": npy(logits), f"process_{top_k}_{top_p}/mask": npy(mask),
                    f"process_{top_k}_{top_p}/want": npy(want)})
    return out


def ref_baselines_fixture():
    """tests/test_baselines_cpu.py: the reference's REINFORCE baselines (models/rl/reinforce/baselines.py) on the
    test's fake policy / env."""
    import copy
    import importlib

    sys.path.insert(0, os.path.dirname(HERE))
    from test_baselines_cpu import ROLLOUT_CANDIDATES, CriticPolicy, FakeEnv, FakePolicy, baseline_inputs

    class RefDataset(torch.utils.data.Dataset):
        """the reference's DataLoader path needs a dataset with `collate_fn` (data/dataset.py:41-78)."""

        def __init__(self, ds):
            self.ds, self.collate_fn = ds, ds.collate_fn

        def __len__(self):
            return len(self.ds)

        def __getitem__(self, i):
            return self.ds[i]

    class RefEnv(FakeEnv):
        def dataset(self, batch_size=[], **kw):
            return RefDataset(super().dataset(batch_size))

    bl = importlib.import_module("rl4co.models.rl.reinforce.baselines")
    inp = baseline_inputs()
    out = {}
    for i, cand in enumerate(ROLLOUT_CANDIDATES):
        theirs = bl.RolloutBaseline(bl_alpha=0.05)
        theirs.setup(FakePolicy(0.0), RefEnv(), batch_size=16, device="cpu", dataset_size=64)
        out[f"rollout{i}/setup_mean"], out[f"rollout{i}/bl_vals"] = npy(float(theirs.mean)), npy(theirs.bl_vals)
        theirs.epoch_callback(copy.deepcopy(FakePolicy(**cand)), RefEnv(), batch_size=16, device="cpu", epoch=0,
                              dataset_size=64)
        out[f"rollout{i}/mean"], out[f"rollout{i}/bias"] = npy(float(theirs.mean)), npy(float(theirs.policy.bias))
        td = TensorDict({"x": torch.from_numpy(inp["rollout_x"])}, batch_size=[7])
        out[f"rollout{i}/eval"] = npy(theirs.eval(td, None, RefEnv())[0])
    theirs = bl.get_reinforce_baseline("rollout", n_epochs=2, exp_beta=0.8)
    theirs.setup(FakePolicy(0.1), RefEnv(), batch_size=16, device="cpu", dataset_size=32)
    vals, alphas = [], []
    for epoch in range(3):
        for j in range(2):
            td = TensorDict({"x": torch.from_numpy(inp["warmup_x"][epoch, j])}, batch_size=[9])
            v, l = theirs.eval(td, torch.from_numpy(inp["warmup_reward"][epoch, j]), RefEnv())
            assert float(l) == 0.0
            vals.append(npy(torch.as_tensor(v).float().expand(9)))
        theirs.epoch_callback(FakePolicy(0.1), RefEnv(), batch_size=16, device="cpu", epoch=epoch, dataset_size=32)
        alphas.append(float(theirs.alpha))
    out["warmup/values"], out["warmup/alpha"] = np.stack(vals), np.array(alphas)
    torch.manual_seed(1)
    pol = CriticPolicy()
    theirs = bl.CriticBaseline()
    torch.manual_seed(2)
    theirs.setup(pol, FakeEnv())
    v, l = theirs.eval(TensorDict({"locs": torch.from_numpy(inp["critic_locs"])}, batch_size=[6]),
                       torch.from_numpy(inp["critic_reward"]))
    out["critic/keys"] = np.array(list(theirs.critic.state_dict().keys()))
    out["critic/value"], out["critic/loss"] = npy(v), npy(l)
    names = ("no", "shared", "exponential", "mean", "critic", "rollout_only", "rollout", "warmup")
    out["registry/names"] = np.array(names)
    out["registry/types"] = np.array([type(bl.get_reinforce_baseline(n)).__name__ for n in names])
    return out


def ref_datasets_fixture():
    """tests/test_host_cpu.py: the reference's numpy-seeded validation / test sets (data/generate_data.py)."""
    import importlib

    G = importlib.import_module("rl4co.data.generate_data")
    out = {}
    for prob, gs, seed, name in (("tsp", 20, 4321, "val"), ("vrp", 50, 1234, "test")):
        np.random.seed(seed)
        out.update({f"{prob}{gs}_{name}/{k}": v for k, v in G.generate_env_data(prob, 16, gs, None).items()})
    return out


def dropin_fixture():
    """tests/test_gpu_dropin.py and the sibling envs' drop-in tests: what the reference's own loop computes, to be
    matched by the CUDA env / decoder -- random-policy MDP traces (utils/decoding.py:85-106) and policy forwards
    on name-seeded weights (sampling: Exp(1) draws regenerated from the seed)."""
    out = {}
    for name, n in (("tsp", 20), ("cvrp", 20), ("tsp", 50), ("cvrp", 50)):
        seeded_instances(out, f"env_{name}{n}", name, n, 64, 11)  # the instances env_fixture draws first
        trace = env_fixture(name, n, 64, 11)
        out.update({f"env_{name}{n}/{k}": v for k, v in trace.items() if not k.startswith("inst::")})
        for dt in ("greedy", "sampling", "multistart_greedy"):
            policy_case(out, f"fwd_{name}{n}_{dt}", name, n, 32, 13, 2, dt, sample_seed=3,
                        evaluate="multistart" not in dt, step_rows=8)
    policy_case(out, "op20_sampling", "op", 20, 64, 3, 1, "sampling", sample_seed=11, phase="train", step_rows=8)
    policy_case(out, "pctsp20_sampling", "pctsp", 20, 64, 3, 1, "sampling", sample_seed=11, phase="train", step_rows=8)
    policy_case(out, "sdvrp20_greedy", "sdvrp", 20, 32, 3, 1, "greedy", step_rows=8)
    return out


def main():
    jobs = {
        "ref_policy": ref_policy_fixture,
        "ref_baselines": ref_baselines_fixture,
        "ref_datasets": ref_datasets_fixture,
        "dropin": dropin_fixture,
        "env_tsp20": lambda: env_fixture("tsp", 20, 16, 100),
        "env_tsp50": lambda: env_fixture("tsp", 50, 8, 101),
        "env_cvrp20": lambda: env_fixture("cvrp", 20, 16, 102),
        "env_cvrp50": lambda: env_fixture("cvrp", 50, 8, 103),
        "am_tsp20": lambda: am_fixture("tsp", 20, 8, 200),
        "am_cvrp20": lambda: am_fixture("cvrp", 20, 8, 201),
        "am_tsp50": lambda: am_fixture("tsp", 50, 4, 202, ms_batch=2),
        "am_cvrp50": lambda: am_fixture("cvrp", 50, 4, 203, ms_batch=2),
        "am_tsp100": lambda: am_fixture("tsp", 100, 4, 204, ms_batch=1, lean=True),
        "am_cvrp100": lambda: am_fixture("cvrp", 100, 4, 205, ms_batch=1, lean=True),
        "pomo_tsp100": lambda: pomo_fixture(100, 2, 400),
        "env_sdvrp20": lambda: env_fixture("sdvrp", 20, 16, 104),
        "env_sdvrp50": lambda: env_fixture("sdvrp", 50, 8, 105),
        "am_sdvrp20": lambda: sdvrp_am_fixture(20, 8, 206),
        "am_sdvrp50": lambda: sdvrp_am_fixture(50, 4, 207),
        "env_op20": lambda: env_fixture("op", 20, 16, 108),
        "env_op50": lambda: env_fixture("op", 50, 8, 109),
        "am_op20": lambda: sdvrp_am_fixture(20, 8, 210, name="op"),
        "am_op50": lambda: sdvrp_am_fixture(50, 4, 211, name="op"),
        "env_pctsp20": lambda: env_fixture("pctsp", 20, 16, 110),
        "env_pctsp50": lambda: env_fixture("pctsp", 50, 8, 111),
        "am_pctsp20": lambda: sdvrp_am_fixture(20, 8, 212, name="pctsp"),
        "am_pctsp50": lambda: sdvrp_am_fixture(50, 4, 213, name="pctsp"),
        "enc_tsp20_batch": lambda: encoder_fixture("tsp", 20, 4, 300, "batch"),
        "enc_cvrp20_instance": lambda: encoder_fixture("cvrp", 20, 4, 301, "instance"),
        "layout": layout_fixture,
        "dec_tsp20": lambda: decoding_fixture("tsp", 20, 8, 200),
        "dec_cvrp20": lambda: decoding_fixture("cvrp", 20, 8, 201),
    }
    only = set(sys.argv[1:])  # `python make_golden.py dec_tsp20 dec_cvrp20` regenerates just those files
    for name, fn in jobs.items():
        if only and name not in only:
            continue
        data = fn()
        path = os.path.join(HERE, name + ".npz")
        np.savez_compressed(path, **data)
        print(f"{name}: {len(data)} arrays, {os.path.getsize(path) / 1024:.0f} KiB")


if __name__ == "__main__":
    main()
