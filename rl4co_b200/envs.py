"""Drop-in TSP / CVRP environments whose step / mask / reward run as CUDA kernels.

Same plugin surface as rl4co's envs (SURVEY.md section 8b):
  RL4COEnvBase   rl4co/envs/common/base.py:19-333  (reset / step / get_reward / get_action_mask /
                 get_num_starts / select_start_nodes / check_solution_validity / generator / dataset)
  TSPEnv         rl4co/envs/routing/tsp/env.py:22-192
  CVRPEnv        rl4co/envs/routing/cvrp/env.py:22-256
TensorDict keys, dtypes and shapes are exactly the reference's, so the reference's context
embeddings / decoding strategies / REINFORCE loops can consume the state unchanged.

`reset` only allocates state (torch, any device).  `step`, `get_action_mask`, `get_reward`
and `check_solution_validity` call libcorollout and therefore require CUDA tensors: there
is deliberately no CPU fallback.
"""

from __future__ import annotations

import torch

from . import native
from .ops import get_num_starts, select_start_nodes
from .tensordict import TensorDict

# rl4co/envs/routing/cvrp/generator.py:15-30
CAPACITIES = {10: 20.0, 15: 25.0, 20: 30.0, 30: 33.0, 40: 37.0, 50: 40.0, 60: 43.0, 75: 45.0,
              100: 50.0, 125: 55.0, 150: 60.0, 200: 70.0, 500: 100.0, 1000: 150.0}


class Generator:
    """rl4co/envs/common/utils.py:19-32"""

    def __call__(self, batch_size) -> TensorDict:
        batch_size = [batch_size] if isinstance(batch_size, int) else list(batch_size)
        return self._generate(batch_size)


class _DeviceStream:
    """On-device generation state: `device="cuda"` makes a generator write instances straight into HBM with
    co_generate_uniform / co_generate_demand (Philox keyed by `seed`; every call advances `offset`, so successive
    batches differ and a (seed, call index) pair always reproduces the same batch).  Default: torch's CPU
    generator in the reference's call order (bit-identical to the reference under the same torch seed)."""

    def _init_stream(self, device, seed):
        self.device = None if device is None else torch.device(device)
        self.seed = 0 if seed is None else int(seed)
        self.calls = 0

    @property
    def on_device(self):
        return self.device is not None and self.device.type == "cuda"

    def _next_offset(self, streams: int) -> int:
        off = self.calls * streams
        self.calls += 1
        return off


class TSPGenerator(Generator, _DeviceStream):
    """rl4co/envs/routing/tsp/generator.py:14-58 (uniform locations)."""

    def __init__(self, num_loc: int = 20, min_loc: float = 0.0, max_loc: float = 1.0, device=None, seed=None, **_):
        self.num_loc, self.min_loc, self.max_loc = num_loc, min_loc, max_loc
        self._init_stream(device, seed)

    def _generate(self, batch_size) -> TensorDict:
        if self.on_device:
            locs = native.generate_uniform((*batch_size, self.num_loc, 2), self.device, self.seed, self._next_offset(1),
                                           self.min_loc, self.max_loc)
            return TensorDict({"locs": locs}, batch_size=batch_size, device=self.device)
        locs = torch.rand(*batch_size, self.num_loc, 2) * (self.max_loc - self.min_loc) + self.min_loc
        return TensorDict({"locs": locs}, batch_size=batch_size)


class CVRPGenerator(Generator, _DeviceStream):
    """rl4co/envs/routing/cvrp/generator.py:33-140 (uniform locations, integer demands 1..9
    over the Kool et al. capacity table, depot = first sampled point)."""

    def __init__(self, num_loc: int = 20, min_loc: float = 0.0, max_loc: float = 1.0, min_demand: int = 1,
                 max_demand: int = 10, vehicle_capacity: float = 1.0, capacity: float | None = None, device=None,
                 seed=None, **_):
        self._init_stream(device, seed)
        self.num_loc, self.min_loc, self.max_loc = num_loc, min_loc, max_loc
        self.min_demand, self.max_demand = min_demand, max_demand
        self.vehicle_capacity = vehicle_capacity
        if capacity is None:
            capacity = CAPACITIES.get(num_loc, None)
        if capacity is None:
            capacity = CAPACITIES[min(CAPACITIES.keys(), key=lambda x: abs(x - num_loc))]
        self.capacity = capacity

    def _generate(self, batch_size) -> TensorDict:
        if self.on_device:
            off = self._next_offset(2)
            locs = native.generate_uniform((*batch_size, self.num_loc + 1, 2), self.device, self.seed, off,
                                           self.min_loc, self.max_loc)
            demand = native.generate_demand((*batch_size, self.num_loc), self.device, self.seed, off + 1,
                                            self.min_demand, self.max_demand, self.capacity)
            return TensorDict(
                {"locs": locs[..., 1:, :], "depot": locs[..., 0, :], "demand": demand,
                 "capacity": torch.full((*batch_size, 1), self.capacity, device=self.device)},
                batch_size=batch_size, device=self.device)
        locs = torch.rand(*batch_size, self.num_loc + 1, 2) * (self.max_loc - self.min_loc) + self.min_loc
        lo, hi = self.min_demand - 1, self.max_demand - 1
        demand = torch.rand(*batch_size, self.num_loc) * (hi - lo) + lo
        demand = (demand.int() + 1).float()
        return TensorDict(
            {"locs": locs[..., 1:, :], "depot": locs[..., 0, :], "demand": demand / self.capacity,
             "capacity": torch.full((*batch_size, 1), self.capacity)},
            batch_size=batch_size,
        )


OP_MAX_LENGTHS = {20: 2.0, 50: 3.0, 100: 4.0}  # rl4co/envs/routing/op/generator.py:14


class OPGenerator(Generator, _DeviceStream):
    """rl4co/envs/routing/op/generator.py:19-139: uniform locations (depot = first sampled point); prize by type --
    "dist" (default, Fischetti et al. / Kool et al.: from the distance to the depot), "unif", "const"; max_length from
    the size table.  `device="cuda"`: locations from co_generate_uniform, prizes derived on the device."""

    def __init__(self, num_loc: int = 20, min_loc: float = 0.0, max_loc: float = 1.0, prize_type: str = "dist",
                 max_length: float | None = None, device=None, seed=None, **_):
        self._init_stream(device, seed)
        self.num_loc, self.min_loc, self.max_loc = num_loc, min_loc, max_loc
        if prize_type not in ("dist", "unif", "const"):
            raise ValueError(f"Invalid prize_type: {prize_type}")
        self.prize_type = prize_type
        if max_length is None:
            max_length = OP_MAX_LENGTHS.get(num_loc) or OP_MAX_LENGTHS[min(OP_MAX_LENGTHS, key=lambda x: abs(x - num_loc))]
        self.max_length = max_length

    def _generate(self, batch_size) -> TensorDict:
        dev = self.device if self.on_device else None
        if self.on_device:
            locs = native.generate_uniform((*batch_size, self.num_loc + 1, 2), self.device, self.seed,
                                           self._next_offset(2), self.min_loc, self.max_loc)
        else:
            locs = torch.rand(*batch_size, self.num_loc + 1, 2) * (self.max_loc - self.min_loc) + self.min_loc
        if self.prize_type == "const":
            prize = torch.ones(*batch_size, self.num_loc, device=dev)
        elif self.prize_type == "unif":
            prize = (1 + torch.randint(0, 100, (*batch_size, self.num_loc), device=dev).float()) / 100
        else:
            prize = (locs[..., 0:1, :] - locs[..., 1:, :]).norm(p=2, dim=-1)
            prize = (1 + (prize / prize.max(dim=-1, keepdim=True)[0] * 99).int()).float() / 100
        if isinstance(self.max_length, torch.Tensor):
            max_length = self.max_length
        else:
            max_length = torch.full((*batch_size,), self.max_length, device=dev)
        return TensorDict({"locs": locs[..., 1:, :], "depot": locs[..., 0, :], "prize": prize, "max_length": max_length},
                          batch_size=batch_size, device=dev)


class PCTSPGenerator(Generator, _DeviceStream):
    """rl4co/envs/routing/pctsp/generator.py:14-139: uniform locations (depot = first sampled point), penalties
    U(0, max_penalty * penalty_factor / num_loc), deterministic prizes U(0, 4 / num_loc), stochastic prizes U(0, 2) x
    deterministic -- sampled in that order.  `device="cuda"`: Philox streams of co_generate_uniform."""

    def __init__(self, num_loc: int = 20, min_loc: float = 0.0, max_loc: float = 1.0, penalty_factor: float = 3.0,
                 prize_required: float = 1.0, max_penalty: float | None = None, device=None, seed=None, **_):
        self._init_stream(device, seed)
        self.num_loc, self.min_loc, self.max_loc = num_loc, min_loc, max_loc
        self.prize_required = prize_required
        if max_penalty is None:
            max_penalty = OP_MAX_LENGTHS.get(num_loc) or OP_MAX_LENGTHS[min(OP_MAX_LENGTHS, key=lambda x: abs(x - num_loc))]
        self.max_penalty = max_penalty * penalty_factor / num_loc

    def _generate(self, batch_size) -> TensorDict:
        n = self.num_loc
        if self.on_device:
            off = self._next_offset(4)
            u = lambda shape, k, hi: native.generate_uniform(shape, self.device, self.seed, off + k, 0.0, hi)  # noqa: E731
            locs = native.generate_uniform((*batch_size, n + 1, 2), self.device, self.seed, off, self.min_loc, self.max_loc)
            penalty, det, sto = u((*batch_size, n), 1, self.max_penalty), u((*batch_size, n), 2, 4.0 / n), u((*batch_size, n), 3, 2.0)
            dev = self.device
        else:
            locs = torch.rand(*batch_size, n + 1, 2) * (self.max_loc - self.min_loc) + self.min_loc
            penalty = torch.rand(*batch_size, n) * self.max_penalty
            det = torch.rand(*batch_size, n) * (4.0 / n)
            sto = torch.rand(*batch_size, n) * 2.0
            dev = None
        return TensorDict({"locs": locs[..., 1:, :], "depot": locs[..., 0, :], "penalty": penalty, "deterministic_prize": det,
                           "stochastic_prize": sto * det}, batch_size=batch_size, device=dev)


class FusedEnvBase:
    """Host-side mirror of RL4COEnvBase (rl4co/envs/common/base.py:19-333)."""

    name = "base"
    batch_locked = False

    def __init__(self, *, check_solution: bool = True, seed: int | None = None, device: str = "cpu",
                 batch_size=None, inplace: bool = False, data_dir: str = "data/", train_file: str | None = None,
                 val_file: str | None = None, test_file: str | None = None, **kwargs):
        kwargs.pop("name", None)
        # rl4co/envs/common/base.py:45-79: optional dataset files per phase, relative to data_dir
        import os

        self.data_dir = data_dir
        self.train_file = os.path.join(data_dir, train_file) if train_file is not None else None
        self.val_file = os.path.join(data_dir, val_file) if val_file is not None else None
        self.test_file = os.path.join(data_dir, test_file) if test_file is not None else None
        self.check_solution = check_solution
        self.device = torch.device(device)
        self.batch_size = torch.Size([]) if batch_size is None else torch.Size(batch_size)
        self.inplace = inplace  # update mask / visited buffers in place instead of allocating per step
        if seed is None:
            seed = torch.empty((), dtype=torch.int64).random_().item()
        self.set_seed(seed)

    # -- torchrl-ish bookkeeping -------------------------------------------------
    def set_seed(self, seed):
        self.rng = torch.manual_seed(seed)
        return seed

    def to(self, device):
        if device is not None:
            self.device = torch.device(device)
        return self

    # -- public API ---------------------------------------------------------------
    def step(self, td: TensorDict) -> dict:
        """rl4co/envs/common/base.py:121-133 (fast path: {"next": td})"""
        return {"next": self._step(td)}

    def reset(self, td: TensorDict | None = None, batch_size=None) -> TensorDict:
        """rl4co/envs/common/base.py:135-143 (+ torchrl's done/terminated fill)"""
        if batch_size is None:
            batch_size = self.batch_size if td is None else td.batch_size
        if td is None or td.is_empty():
            td = self.generator(batch_size=batch_size)
        batch_size = [batch_size] if isinstance(batch_size, int) else batch_size
        self.to(td.device)
        out = self._reset(td, batch_size=batch_size)
        for key in ("done", "terminated"):
            if key not in out.keys():
                out.set(key, torch.zeros((*batch_size, 1), dtype=torch.bool, device=td.device))
        if td.device is not None:  # the reset state carries the device explicitly, like torchrl's
            out = out.to(td.device)
        return out

    def get_reward(self, td: TensorDict, actions: torch.Tensor, check_solution: bool | None = None) -> torch.Tensor:
        """rl4co/envs/common/base.py:180-190"""
        check_solution = self.check_solution if check_solution is None else check_solution
        if check_solution:
            self.check_solution_validity(td, actions)
        return self._get_reward(td, actions)

    def get_num_starts(self, td):
        return get_num_starts(td, self.name)

    def select_start_nodes(self, td, num_starts):
        return select_start_nodes(td, self, num_starts)

    def dataset(self, batch_size=[], phase="train", filename=None):
        """rl4co/envs/common/base.py:234-268: the phase's file (`{phase}_file`, or `filename`) when set -- e.g. the
        seeded validation / test sets of data.generate_default_datasets -- else freshly generated instances; a
        missing file falls back to generation like the reference."""
        from .data import TensorDictDataset

        f = getattr(self, f"{phase}_file", None) if filename is None else filename
        if f is None:
            td = self.generator(batch_size)
        else:
            try:
                td = self.load_data(f, batch_size)
            except FileNotFoundError:
                td = self.generator(batch_size)
        return TensorDictDataset(td)

    def local_search(self, td: TensorDict, actions: torch.Tensor, **kwargs) -> torch.Tensor:
        """rl4co/envs/common/base.py:228-232"""
        raise NotImplementedError(f"Local is not implemented yet for {self.name} environment")

    @staticmethod
    def load_data(fpath, batch_size=[]):
        from .data import load_npz_to_tensordict

        return load_npz_to_tensordict(fpath)


class FusedTSPEnv(FusedEnvBase):
    """CUDA drop-in for rl4co.envs.TSPEnv (rl4co/envs/routing/tsp/env.py:22-192)."""

    name = "tsp"

    def __init__(self, generator: TSPGenerator | None = None, generator_params: dict = {}, **kwargs):
        super().__init__(**kwargs)
        self.generator = TSPGenerator(**generator_params) if generator is None else generator

    def _reset(self, td: TensorDict, batch_size=None) -> TensorDict:
        """tsp/env.py:88-113"""
        device = td.device
        init_locs = td["locs"]
        num_loc = init_locs.shape[-2]
        current_node = torch.zeros((*batch_size,), dtype=torch.int64, device=device)
        available = torch.ones((*batch_size, num_loc), dtype=torch.bool, device=device)
        i = torch.zeros((*batch_size, 1), dtype=torch.int64, device=device)
        return TensorDict(
            {
                "locs": init_locs,
                "first_node": current_node,
                "current_node": current_node,
                "i": i,
                "action_mask": available,
                "reward": torch.zeros((*batch_size, 1), dtype=torch.float32, device=device),
            },
            batch_size=batch_size,
        )

    def _step(self, td: TensorDict) -> TensorDict:
        """tsp/env.py:60-86 in one kernel (co_tsp_step).  `first_node` follows the reference's
        "set on the first step" rule per instance (the reference tests `td["i"].all() == 0`
        batch-wide; identical whenever the batch advances in lock-step)."""
        action = td["action"].contiguous()
        mask_in = td["action_mask"]
        if not mask_in.is_contiguous():
            mask_in = mask_in.contiguous()
        B = action.shape[0]
        mask_out = mask_in if self.inplace else torch.empty_like(mask_in)
        # fresh int64 state tensors (the reference rebinds, never mutates, these keys)
        first_node = td["first_node"].clone()
        current_node = torch.empty_like(action)
        i = td["i"].clone()
        done = torch.empty(B, dtype=torch.bool, device=action.device)
        native.tsp_step(action, mask_in, mask_out, first_node, current_node, i.view(-1), done)
        td.update(
            {
                "first_node": first_node,
                "current_node": current_node,
                "i": i,
                "action_mask": mask_out,
                "reward": torch.zeros_like(done),  # bool zeros, as in the reference (tsp/env.py:74)
                "done": done,
            }
        )
        return td

    def _get_reward(self, td: TensorDict, actions: torch.Tensor) -> torch.Tensor:
        """tsp/env.py:150-156"""
        if self.check_solution:
            self.check_solution_validity(td, actions)
        return native.tour_length(td["locs"].contiguous(), actions.contiguous(), with_depot=False)

    @staticmethod
    def check_solution_validity(td: TensorDict, actions: torch.Tensor) -> None:
        """tsp/env.py:158-164"""
        bad = native.check_tours(actions.contiguous(), td["locs"].shape[-2])
        assert bad == 0, "Invalid tour"

    @staticmethod
    def local_search(td: TensorDict, actions: torch.Tensor, max_iterations: int = 1000,
                     num_threads: int | None = None) -> torch.Tensor:
        """tsp/env.py:184-188 -> tsp/local_search.py:16-81: 2-opt (best improvement per scan) on every tour, in one
        kernel (co_tsp_two_opt) on the tensors' GPU; the same tours as the reference, bit for bit.  Returns new int64
        tours [B, N]; `actions` is not modified.  `num_threads` (the reference's numba thread count) is ignored."""
        if "distances" in td.keys():
            raise NotImplementedError("local_search: a precomputed td['distances'] matrix is not supported; "
                                      "distances are computed from td['locs']")
        locs = td["locs"]
        if actions.dim() != 2 or locs.dim() != 3 or tuple(locs.shape) != (*actions.shape, 2):
            raise ValueError(f"local_search: actions must be [B, N] and td['locs'] [B, N, 2], got "
                             f"{tuple(actions.shape)} and {tuple(locs.shape)}")
        if actions.shape[1] > native.TWO_OPT_MAX_NODES:
            raise NotImplementedError(f"local_search: N={actions.shape[1]} above {native.TWO_OPT_MAX_NODES} nodes")
        return native.tsp_two_opt(locs.to(torch.float32).contiguous(), actions.to(torch.int64).contiguous(),
                                  max_iterations)


class FusedCVRPEnv(FusedEnvBase):
    """CUDA drop-in for rl4co.envs.CVRPEnv (rl4co/envs/routing/cvrp/env.py:22-256)."""

    name = "cvrp"

    def __init__(self, generator: CVRPGenerator | None = None, generator_params: dict = {}, **kwargs):
        super().__init__(**kwargs)
        self.generator = CVRPGenerator(**generator_params) if generator is None else generator

    def _reset(self, td: TensorDict, batch_size=None) -> TensorDict:
        """cvrp/env.py:98-124"""
        device = td.device
        td_reset = TensorDict(
            {
                "locs": torch.cat((td["depot"][:, None, :], td["locs"]), -2),
                "demand": td["demand"],
                "current_node": torch.zeros(*batch_size, 1, dtype=torch.long, device=device),
                "used_capacity": torch.zeros((*batch_size, 1), device=device),
                "vehicle_capacity": torch.full((*batch_size, 1), self.generator.vehicle_capacity, device=device),
                "visited": torch.zeros((*batch_size, td["locs"].shape[-2] + 1), dtype=torch.uint8, device=device),
            },
            batch_size=batch_size,
        )
        if td_reset["visited"].is_cuda:
            mask = self.get_action_mask(td_reset)
        else:
            # reset only allocates state and works on any device (module docstring): the initial mask of
            # cvrp/env.py:126-136 with nothing visited and the vehicle at the depot, in torch
            fits = ~(td_reset["demand"] + td_reset["used_capacity"] > td_reset["vehicle_capacity"] + 1e-5)
            mask = torch.cat((~fits.any(-1, keepdim=True), fits), -1)
        td_reset.set("action_mask", mask)
        return td_reset

    def _step(self, td: TensorDict) -> TensorDict:
        """cvrp/env.py:66-96 incl. the trailing get_action_mask, one kernel (co_cvrp_step)."""
        action = td["action"].contiguous()
        B = action.shape[0]
        visited_in = td["visited"].contiguous()
        used_in = td["used_capacity"].contiguous()
        visited_out = visited_in if self.inplace else torch.empty_like(visited_in)
        used_out = torch.empty_like(used_in)
        current_node = torch.empty(B, 1, dtype=torch.int64, device=action.device)
        done = torch.empty(B, dtype=torch.bool, device=action.device)
        mask_out = torch.empty(B, visited_in.shape[-1], dtype=torch.bool, device=action.device)
        native.cvrp_step(action, td["demand"].contiguous(), td["vehicle_capacity"].contiguous(), used_in, used_out,
                         visited_in, visited_out, current_node, done, mask_out)
        td.update(
            {
                "current_node": current_node,
                "used_capacity": used_out,
                "visited": visited_out,
                "reward": torch.zeros_like(done),
                "done": done,
            }
        )
        td.set("action_mask", mask_out)
        return td

    @staticmethod
    def get_action_mask(td: TensorDict) -> torch.Tensor:
        """cvrp/env.py:126-136 (co_cvrp_action_mask)"""
        visited = td["visited"].contiguous()
        mask = torch.empty(visited.shape, dtype=torch.bool, device=visited.device)
        native.cvrp_action_mask(td["demand"].contiguous(), td["used_capacity"].contiguous(),
                                td["vehicle_capacity"].contiguous(), visited,
                                td["current_node"].contiguous(), mask)
        return mask

    def _get_reward(self, td: TensorDict, actions: torch.Tensor) -> torch.Tensor:
        """cvrp/env.py:138-147"""
        return native.tour_length(td["locs"].contiguous(), actions.contiguous(), with_depot=True)

    @staticmethod
    def check_solution_validity(td: TensorDict, actions: torch.Tensor) -> None:
        """cvrp/env.py:149-177"""
        bad = native.check_tours(actions.contiguous(), td["locs"].shape[-2], td["demand"].contiguous(),
                                 td["vehicle_capacity"].contiguous().view(-1), B_inst=td["demand"].shape[0])
        assert bad == 0, "Invalid tour"

    @staticmethod
    def load_data(fpath, batch_size=[]):
        """cvrp/env.py:179-186: normalise demand by capacity."""
        from .data import load_npz_to_tensordict

        td_load = load_npz_to_tensordict(fpath)
        td_load.set("demand", td_load["demand"] / td_load["capacity"][:, None])
        return td_load


class FusedSDVRPEnv(FusedCVRPEnv):
    """CUDA drop-in for rl4co.envs.SDVRPEnv (rl4co/envs/routing/sdvrp/env.py:14-139): split deliveries -- a
    customer may be visited several times, each visit delivers min(remaining demand, remaining capacity).  The
    dynamic state is `demand_with_depot` [B, N]; it feeds the decoder's dynamic embedding
    (nn/env_embeddings/dynamic.py:60-78).  Runs on the stepping kernels (co_sdvrp_step / co_sdvrp_action_mask,
    co_pointer_logits with the dynamic term, co_select_action, co_tour_length)."""

    name = "sdvrp"

    def _reset(self, td: TensorDict, batch_size=None) -> TensorDict:
        """sdvrp/env.py:84-108"""
        device = td.device
        td_reset = TensorDict(
            {
                "locs": torch.cat((td["depot"][..., None, :], td["locs"]), -2),
                "demand": td["demand"],
                "demand_with_depot": torch.cat((torch.zeros_like(td["demand"][..., 0:1]), td["demand"]), -1),
                "current_node": torch.zeros(*batch_size, 1, dtype=torch.long, device=device),
                "used_capacity": torch.zeros((*batch_size, 1), device=device),
                "vehicle_capacity": torch.full((*batch_size, 1), self.generator.vehicle_capacity, device=device),
            },
            batch_size=batch_size,
        )
        if td_reset["demand"].is_cuda:
            mask = self.get_action_mask(td_reset)
        else:  # reset only allocates state: initial mask of sdvrp/env.py:110-116 (vehicle empty, at the depot)
            free = td_reset["demand"] != 0
            mask = torch.cat((~free.any(-1, keepdim=True), free), -1)
        td_reset.set("action_mask", mask)
        return td_reset

    def _step(self, td: TensorDict) -> TensorDict:
        """sdvrp/env.py:55-82 incl. the trailing get_action_mask, one kernel (co_sdvrp_step)."""
        action = td["action"].contiguous()
        B = action.shape[0]
        d_in = td["demand_with_depot"].contiguous()
        used_in = td["used_capacity"].contiguous()
        d_out = d_in if self.inplace else torch.empty_like(d_in)
        used_out = torch.empty_like(used_in)
        current_node = torch.empty(B, 1, dtype=torch.int64, device=action.device)
        done = torch.empty(B, dtype=torch.bool, device=action.device)
        mask_out = torch.empty(B, d_in.shape[-1], dtype=torch.bool, device=action.device)
        native.sdvrp_step(action, d_in, d_out, td["vehicle_capacity"].contiguous(), used_in, used_out, current_node,
                          done, mask_out)
        td.update({"demand_with_depot": d_out, "current_node": current_node, "used_capacity": used_out,
                   "reward": torch.zeros_like(done), "done": done})
        td.set("action_mask", mask_out)
        return td

    @staticmethod
    def get_action_mask(td: TensorDict) -> torch.Tensor:
        """sdvrp/env.py:110-116 (co_sdvrp_action_mask)"""
        d = td["demand_with_depot"].contiguous()
        mask = torch.empty(d.shape, dtype=torch.bool, device=d.device)
        return native.sdvrp_action_mask(d, td["used_capacity"].contiguous(), td["vehicle_capacity"].contiguous(),
                                        td["current_node"].contiguous(), mask)

    @staticmethod
    def check_solution_validity(td: TensorDict, actions: torch.Tensor) -> None:
        """sdvrp/env.py:118-139: replay the deliveries; all demand must be served, no idle depot-depot move while
        demand remains.  Validation path (host-synchronising asserts, like the reference); device tensors."""
        cap = td["vehicle_capacity"].reshape(-1)
        demands = torch.cat((-td["vehicle_capacity"].reshape(-1, 1), td["demand"]), 1).clone()
        rng = torch.arange(demands.shape[0], device=demands.device)
        used = torch.zeros_like(cap)
        a_prev = None
        for a in actions.transpose(0, 1):
            if a_prev is not None:
                assert (demands[(a_prev == 0) & (a == 0), :] == 0).all(), "Cannot visit depot twice if any nonzero demand"
            d = torch.min(demands[rng, a], cap - used)
            demands[rng, a] -= d
            used = used + d
            used[a == 0] = 0
            a_prev = a
        assert (demands == 0).all(), "All demand must be satisfied"


class FusedOPEnv(FusedEnvBase):
    """CUDA drop-in for rl4co.envs.OPEnv (rl4co/envs/routing/op/env.py:18-242, orienteering): collect prizes and be
    back at the depot within `max_length`.  State keys / dtypes as the reference's: `locs` [B,N,2] (depot at 0), `prize`
    [B,N] (depot 0), `tour_length` [B], `max_length` [B,N] (budget minus the way back per node), `current_node` [B,1],
    `visited` bool [B,N], `current_total_prize` [B], `i` [B].  Runs on the stepping kernels (co_op_step /
    co_op_action_mask / co_op_reward; the decoder shares the capacity-context arithmetic of co_pointer_logits)."""

    name = "op"

    def __init__(self, generator=None, generator_params: dict | None = None, prize_type: str = "dist", **kwargs):
        super().__init__(**kwargs)
        if generator is None:
            generator = OPGenerator(**{"prize_type": prize_type, **(generator_params or {})})
        self.generator = generator
        self.prize_type = prize_type

    def _reset(self, td: TensorDict, batch_size=None) -> TensorDict:
        """op/env.py:107-138"""
        device = td.device
        locs = torch.cat((td["depot"][:, None, :], td["locs"]), -2)
        td_reset = TensorDict(
            {
                "locs": locs,
                "prize": torch.nn.functional.pad(td["prize"], (1, 0), mode="constant", value=0),
                "tour_length": torch.zeros(*batch_size, device=device),
                "max_length": td["max_length"][..., None] - (td["depot"][..., None, :] - locs).norm(p=2, dim=-1) - 1e-6,
                "current_node": torch.zeros(*batch_size, 1, dtype=torch.long, device=device),
                "visited": torch.zeros((*batch_size, locs.shape[-2]), dtype=torch.bool, device=device),
                "current_total_prize": torch.zeros(*batch_size, dtype=torch.float, device=device),
                "i": torch.zeros((*batch_size,), dtype=torch.int64, device=device),
            },
            batch_size=batch_size,
        )
        if locs.is_cuda:
            mask = self.get_action_mask(td_reset)
        else:  # reset only allocates state: the initial mask of op/env.py:140-155 in torch
            exceeds = (locs - locs[..., 0:1, :]).norm(p=2, dim=-1) > td_reset["max_length"]
            mask = ~exceeds
            mask[..., 0] = True
        td_reset.set("action_mask", mask)
        return td_reset

    def _step(self, td: TensorDict) -> TensorDict:
        """op/env.py:72-105 incl. the trailing get_action_mask, one kernel (co_op_step)."""
        action = td["action"].contiguous()
        B = action.shape[0]
        vin = td["visited"].contiguous()
        vout = vin if self.inplace else torch.empty_like(vin)
        tour_length = td["tour_length"].clone()
        prize_sum = td["current_total_prize"].clone()
        current_node = td["current_node"].reshape(B).clone()
        i = td["i"].clone()
        done = torch.empty(B, dtype=torch.bool, device=action.device)
        mask_out = torch.empty(vin.shape, dtype=torch.bool, device=action.device)
        native.op_step(action, td["locs"].contiguous(), td["prize"].contiguous(), td["max_length"].contiguous(), vin, vout,
                       tour_length, prize_sum, current_node, i, done, mask_out)
        td.update({"tour_length": tour_length, "current_node": current_node[:, None], "visited": vout,
                   "current_total_prize": prize_sum, "i": i, "reward": torch.zeros_like(done), "done": done})
        td.set("action_mask", mask_out)
        return td

    @staticmethod
    def get_action_mask(td: TensorDict) -> torch.Tensor:
        """op/env.py:140-155 (co_op_action_mask)"""
        visited = td["visited"].contiguous()
        mask = torch.empty(visited.shape, dtype=torch.bool, device=visited.device)
        return native.op_action_mask(td["locs"].contiguous(), td["max_length"].contiguous(), visited,
                                     td["tour_length"].contiguous(), td["current_node"].reshape(-1).contiguous(), mask)

    def _get_reward(self, td: TensorDict, actions: torch.Tensor) -> torch.Tensor:
        """op/env.py:157-165 (co_op_reward)"""
        if actions.size(-1) == 1:
            assert (actions == 0).all(), "If all length 1 tours, they should be zero"
            return torch.zeros(actions.size(0), dtype=torch.float, device=actions.device)
        return native.op_reward(td["prize"].contiguous(), actions.contiguous())

    @staticmethod
    def check_solution_validity(td: TensorDict, actions: torch.Tensor, add_distance_to_depot: bool = True) -> None:
        """op/env.py:167-192: no customer twice, length within the budget.  Validation path (host-synchronising
        asserts like the reference)."""
        sorted_actions = actions.sort(1)[0]
        assert ((sorted_actions[:, 1:] == 0) | (sorted_actions[:, 1:] > sorted_actions[:, :-1])).all(), "Duplicates"
        length = -native.tour_length(td["locs"].contiguous(), actions.contiguous(), with_depot=False)
        max_length = td["max_length"]
        if add_distance_to_depot:
            max_length = max_length + (td["locs"][..., 0:1, :] - td["locs"]).norm(p=2, dim=-1) + 1e-6
        if max_length.shape[0] != length.shape[0]:
            max_length = max_length.repeat(length.shape[0] // max_length.shape[0], 1)
        assert (length[..., None] <= max_length + 1e-5).all(), "Max length exceeded"


class FusedPCTSPEnv(FusedEnvBase):
    """CUDA drop-in for rl4co.envs.PCTSPEnv (rl4co/envs/routing/pctsp/env.py:18-264, prize-collecting TSP, deterministic
    prizes): collect a total prize of at least 1 (or visit everything), then return to the depot; unvisited customers
    cost their penalty.  State keys / dtypes as the reference's: `locs` [B,N,2], `current_node` [B], `expected_prize`
    [B,N-1], `real_prize` / `penalty` [B,N] (depot 0), `cur_total_prize` / `cur_total_penalty` / `prize_required` [B],
    `visited` bool [B,N], `i` [B].  Stepping kernels: co_pctsp_step / co_pctsp_action_mask; reward = co_op_reward over the
    penalties + co_tour_length."""

    name = "pctsp"

    def __init__(self, generator=None, generator_params: dict | None = None, **kwargs):
        super().__init__(**kwargs)
        self.generator = PCTSPGenerator(**(generator_params or {})) if generator is None else generator

    def _reset(self, td: TensorDict, batch_size=None) -> TensorDict:
        """pctsp/env.py:95-141"""
        device = td.device
        prize, penalty = td["deterministic_prize"], td["penalty"]
        td_reset = TensorDict(
            {
                "locs": torch.cat([td["depot"][..., None, :], td["locs"]], dim=-2),
                "current_node": torch.zeros((*batch_size,), dtype=torch.int64, device=device),
                "expected_prize": prize,
                "real_prize": torch.cat([torch.zeros_like(prize[..., :1]), prize], dim=-1),
                "penalty": torch.nn.functional.pad(penalty, (1, 0), mode="constant", value=0),
                "cur_total_prize": torch.zeros(*batch_size, device=device),
                "cur_total_penalty": penalty.sum(-1),
                "visited": torch.zeros((*batch_size, td["locs"].shape[-2] + 1), dtype=torch.bool, device=device),
                "prize_required": torch.full((*batch_size,), self.generator.prize_required, device=device),
                "i": torch.zeros((*batch_size,), dtype=torch.int64, device=device),
            },
            batch_size=batch_size,
        )
        mask = torch.ones_like(td_reset["visited"])
        mask[..., 0] = False  # nothing collected yet and customers remain (pctsp/env.py:143-151 at reset)
        td_reset.set("action_mask", mask)
        return td_reset

    def _step(self, td: TensorDict) -> TensorDict:
        """pctsp/env.py:62-93 incl. the trailing get_action_mask, one kernel (co_pctsp_step)."""
        action = td["action"].contiguous()
        B = action.shape[0]
        vin = td["visited"].contiguous()
        vout = vin if self.inplace else torch.empty_like(vin)
        prize_sum, penalty_sum = td["cur_total_prize"].clone(), td["cur_total_penalty"].clone()
        current_node, i = td["current_node"].reshape(B).clone(), td["i"].clone()
        done = torch.empty(B, dtype=torch.bool, device=action.device)
        mask_out = torch.empty(vin.shape, dtype=torch.bool, device=action.device)
        native.pctsp_step(action, td["real_prize"].contiguous(), td["penalty"].contiguous(), vin, vout, prize_sum, penalty_sum,
                          current_node, i, done, mask_out)
        td.update({"current_node": current_node, "cur_total_prize": prize_sum, "cur_total_penalty": penalty_sum,
                   "visited": vout, "i": i, "reward": torch.zeros_like(done), "done": done})
        td.set("action_mask", mask_out)
        return td

    @staticmethod
    def get_action_mask(td: TensorDict) -> torch.Tensor:
        """pctsp/env.py:143-151 (co_pctsp_action_mask)"""
        visited = td["visited"].contiguous()
        mask = torch.empty(visited.shape, dtype=torch.bool, device=visited.device)
        return native.pctsp_action_mask(visited, td["cur_total_prize"].contiguous(), mask)

    def _get_reward(self, td: TensorDict, actions: torch.Tensor) -> torch.Tensor:
        """pctsp/env.py:153-172: saved penalties - (tour length from / to the depot + all penalties)."""
        if actions.size(-1) == 1:
            assert (actions == 0).all(), "If all length 1 tours, they should be zero"
            return torch.zeros(actions.size(0), dtype=torch.float, device=actions.device)
        actions = actions.contiguous()
        saved = native.op_reward(td["penalty"].contiguous(), actions)
        neg_length = native.tour_length(td["locs"].contiguous(), actions, with_depot=True)
        total = td["penalty"][..., 1:].sum(-1)
        if total.shape[0] != saved.shape[0]:
            total = total.repeat(saved.shape[0] // total.shape[0])
        return saved - (-neg_length + total)

    @staticmethod
    def check_solution_validity(td: TensorDict, actions: torch.Tensor) -> None:
        """pctsp/env.py:174-197: no customer twice; the prize constraint holds or every customer was visited."""
        sorted_actions = actions.sort(1)[0]
        assert ((sorted_actions[..., 1:] == 0) | (sorted_actions[..., 1:] > sorted_actions[..., :-1])).all(), "Duplicates"
        p = native.op_reward(td["real_prize"].contiguous(), actions.contiguous())
        all_visited = sorted_actions.size(-1) - (sorted_actions == 0).int().sum(-1) == (td["locs"].size(-2) - 1)
        assert ((p >= 1 - 1e-5) | all_visited).all(), "Total prize does not satisfy min total prize"


ENV_REGISTRY = {"tsp": FusedTSPEnv, "cvrp": FusedCVRPEnv, "sdvrp": FusedSDVRPEnv, "op": FusedOPEnv, "pctsp": FusedPCTSPEnv}


def _register_with_torchrl() -> bool:
    """When torchrl is importable, make the fused envs (virtual) subclasses of `torchrl.envs.EnvBase`, so
    `isinstance(env, EnvBase)` checks in user code hold.  Virtual (`ABCMeta.register`) on purpose: reset / step
    bookkeeping stays the few lines above instead of torchrl's spec machinery (rl4co's loops only use
    reset / step / get_reward, SURVEY.md 8b)."""
    try:
        from torchrl.envs import EnvBase
    except Exception:
        return False
    if hasattr(EnvBase, "register"):
        EnvBase.register(FusedEnvBase)
        return True
    return False


_register_with_torchrl()


def get_env(env_name: str, *args, **kwargs) -> FusedEnvBase:
    """rl4co/envs/__init__.py get_env for the two envs on the path."""
    if env_name not in ENV_REGISTRY:
        raise ValueError(f"Unknown environment {env_name}. Available: {list(ENV_REGISTRY)}")
    return ENV_REGISTRY[env_name](*args, **kwargs)
