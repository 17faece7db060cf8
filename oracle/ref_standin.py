"""TEST INFRASTRUCTURE ONLY -- never imported by the product package.

Runs rl4co's *own, unmodified* hot-path source files out of ``/root/reference``
so they can serve as the pinning oracle for ``oracle/am_rollout_oracle.py`` and
as the generator of the golden vectors under ``tests/golden/``.

rl4co cannot be imported as-is in this image: ``tensordict``, ``torchrl``,
``lightning``, ``matplotlib`` are not installed (no network) and the package
``__init__`` files pull in Hydra/Lightning and every env / zoo model
(SURVEY.md section 8c).  This module registers:

  * ``tensordict``           -> rl4co_b200.tensordict.TensorDict (container only,
                                no arithmetic)
  * ``torchrl.envs.EnvBase`` -> a bookkeeping-only base class whose ``reset``
                                calls ``_reset`` and fills ``done``/``terminated``
                                with zeros ``[B,1]`` bool, which is what torchrl
                                does from ``done_spec`` (rl4co relies on it:
                                rl4co/models/common/constructive/base.py:226)
  * ``torchrl.data``         -> inert spec holders
  * ``lightning...rank_zero_only`` -> identity
  * ``matplotlib``           -> empty modules (render.py is imported unguarded by
                                rl4co/envs/routing/{tsp,cvrp}/env.py:17)
  * synthetic *package* objects for ``rl4co`` and the sub-packages whose
    ``__init__`` is heavy, with ``__path__`` pointing into the reference tree so
    that the individual hot-path files import and execute verbatim.

Nothing here restates reference arithmetic: every number produced through this
module is computed by reference code + PyTorch.

``/root/reference`` does not exist on the GPU box.  ``oracle/make_ref.py`` (called by
``__graft_entry__.build()`` in the build container) stages the same unmodified files under the
git-ignored ``oracle/_ref/``, which travels with the snapshot; this module uses
the reference tree when present and ``oracle/_ref`` otherwise.  No test needs it: the tests compare
against fixtures recorded through it (tests/golden/make_golden.py).
"""

from __future__ import annotations

import importlib
import os
import sys
import types

_STAGED = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")


def _resolve_root() -> str:
    env = os.environ.get("RL4CO_REFERENCE_ROOT")
    if env:
        return env
    if os.path.isdir("/root/reference/rl4co"):
        return "/root/reference"
    return _STAGED


REFERENCE_ROOT = _resolve_root()


def reference_available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "rl4co"))


def reference_kind() -> str:
    """'reference' = live tree, 'staged' = oracle/_ref copy (same bytes, see MANIFEST.json)."""
    return "staged" if os.path.abspath(REFERENCE_ROOT) == os.path.abspath(_STAGED) else "reference"


def _mod(name: str, **attrs) -> types.ModuleType:
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    return m


def _pkg(name: str, relpath: str) -> types.ModuleType:
    m = types.ModuleType(name)
    m.__path__ = [os.path.join(REFERENCE_ROOT, relpath)]
    m.__package__ = name
    sys.modules[name] = m
    return m


_INSTALLED = False


def install() -> None:
    """Register the stand-ins (idempotent). Raises if the reference is absent."""
    global _INSTALLED
    if _INSTALLED:
        return
    if not reference_available():
        raise FileNotFoundError(f"reference tree not found at {REFERENCE_ROOT}")

    import torch

    repo_root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    if repo_root not in sys.path:
        sys.path.insert(0, repo_root)
    from rl4co_b200 import tensordict as td_mod

    # ---- tensordict ---------------------------------------------------------
    if "tensordict" not in sys.modules:
        t = _mod("tensordict", TensorDict=td_mod.TensorDict, __version__="0.6.0")
        t.__path__ = []  # mark as package so `tensordict.tensordict` resolves
        _mod("tensordict.tensordict", TensorDict=td_mod.TensorDict)
        t.tensordict = sys.modules["tensordict.tensordict"]
    TensorDict = sys.modules["tensordict"].TensorDict

    # ---- torchrl ------------------------------------------------------------
    class _Spec:
        def __init__(self, *a, **k):
            self.args, self.kwargs = a, k
            self.shape = k.get("shape", None)
            self.dtype = k.get("dtype", None)

    class Composite(_Spec):
        pass

    class EnvBase:
        """Bookkeeping-only stand-in for torchrl.envs.EnvBase."""

        batch_locked = False

        def __init__(self, device="cpu", batch_size=None, run_type_checks=False, allow_done_after_reset=False):
            self.device = torch.device(device) if device is not None else None
            self.batch_size = torch.Size([]) if batch_size is None else torch.Size(batch_size)

        def set_seed(self, seed=None, static_seed=False):
            self._set_seed(seed)
            return seed

        def to(self, device):
            self.device = torch.device(device)
            return self

        def reset(self, td=None, batch_size=None, **kwargs):
            out = self._reset(td, batch_size=batch_size)
            bs = out.batch_size
            dev = td.device if td is not None else self.device
            for key in ("done", "terminated"):
                if key not in out.keys():
                    out.set(key, torch.zeros((*bs, 1), dtype=torch.bool, device=dev))
            # torchrl returns the reset state on the env's device (RL4COEnvBase.reset moved the env to
            # td.device just before, envs/common/base.py:141): tensors `_reset` built without `device=`
            # (tsp/env.py:110) follow, and td.device is set -- select_start_nodes (utils/ops.py:141) relies on it
            if dev is not None:
                out = out.to(dev)
            return out

    tr = _mod("torchrl")
    tr.__path__ = []
    tr.envs = _mod("torchrl.envs", EnvBase=EnvBase)
    tr.data = _mod("torchrl.data", Bounded=_Spec, Composite=Composite, Unbounded=_Spec,
                   BoundedTensorSpec=_Spec, CompositeSpec=Composite, UnboundedContinuousTensorSpec=_Spec,
                   UnboundedDiscreteTensorSpec=_Spec)

    # ---- lightning (only rank_zero_only is touched, by utils/pylogger.py) ---
    lt = _mod("lightning"); lt.__path__ = []
    lp = _mod("lightning.pytorch"); lp.__path__ = []
    lu = _mod("lightning.pytorch.utilities"); lu.__path__ = []
    _mod("lightning.pytorch.utilities.rank_zero", rank_zero_only=lambda f: f)

    # ---- matplotlib (render.py imports, never called) -----------------------
    if "matplotlib" not in sys.modules:
        mpl = _mod("matplotlib", cm=types.SimpleNamespace(), colormaps={})
        mpl.__path__ = []
        _mod("matplotlib.pyplot")
        _mod("matplotlib.cm")
        _mod("matplotlib.axes", Axes=object)
        _mod("matplotlib.colors")
        mpl.pyplot = sys.modules["matplotlib.pyplot"]

    # ---- rl4co package skeleton (skips heavy __init__ files) ----------------
    rl = _pkg("rl4co", "rl4co")
    rl.__version__ = "0.6.0"
    _pkg("rl4co.utils", "rl4co/utils")
    pylogger = importlib.import_module("rl4co.utils.pylogger")
    sys.modules["rl4co.utils"].get_pylogger = pylogger.get_pylogger
    _pkg("rl4co.data", "rl4co/data")
    _pkg("rl4co.envs", "rl4co/envs")
    _pkg("rl4co.envs.common", "rl4co/envs/common")
    _pkg("rl4co.envs.routing", "rl4co/envs/routing")
    _pkg("rl4co.envs.routing.tsp", "rl4co/envs/routing/tsp")
    _pkg("rl4co.envs.routing.cvrp", "rl4co/envs/routing/cvrp")
    _pkg("rl4co.envs.routing.sdvrp", "rl4co/envs/routing/sdvrp")
    _pkg("rl4co.envs.routing.op", "rl4co/envs/routing/op")
    _pkg("rl4co.envs.routing.pctsp", "rl4co/envs/routing/pctsp")
    _pkg("rl4co.models", "rl4co/models")
    _pkg("rl4co.models.common", "rl4co/models/common")
    _pkg("rl4co.models.nn", "rl4co/models/nn")
    _pkg("rl4co.models.nn.graph", "rl4co/models/nn/graph")
    _pkg("rl4co.models.nn.env_embeddings", "rl4co/models/nn/env_embeddings")
    _pkg("rl4co.models.zoo", "rl4co/models/zoo")
    _pkg("rl4co.models.zoo.am", "rl4co/models/zoo/am")
    _pkg("rl4co.models.rl", "rl4co/models/rl")
    _pkg("rl4co.models.rl.common", "rl4co/models/rl/common")
    _pkg("rl4co.models.rl.reinforce", "rl4co/models/rl/reinforce")

    base = importlib.import_module("rl4co.envs.common.base")
    envs = sys.modules["rl4co.envs"]
    envs.RL4COEnvBase = base.RL4COEnvBase
    tsp_env = importlib.import_module("rl4co.envs.routing.tsp.env")
    cvrp_env = importlib.import_module("rl4co.envs.routing.cvrp.env")
    envs.TSPEnv, envs.CVRPEnv = tsp_env.TSPEnv, cvrp_env.CVRPEnv
    registry = {"tsp": tsp_env.TSPEnv, "cvrp": cvrp_env.CVRPEnv}
    envs.get_env = lambda name, *a, **k: registry[name](*a, **k)

    emb = sys.modules["rl4co.models.nn.env_embeddings"]
    emb.env_context_embedding = importlib.import_module("rl4co.models.nn.env_embeddings.context").env_context_embedding
    emb.env_dynamic_embedding = importlib.import_module("rl4co.models.nn.env_embeddings.dynamic").env_dynamic_embedding
    emb.env_init_embedding = importlib.import_module("rl4co.models.nn.env_embeddings.init").env_init_embedding

    # let rl4co.models.common.constructive/__init__.py run for real
    importlib.import_module("rl4co.models.common.constructive")
    _INSTALLED = True


def load():
    """Return a namespace with the reference classes / functions on the hot path."""
    install()
    ns = types.SimpleNamespace()
    ns.TensorDict = sys.modules["tensordict"].TensorDict
    ns.TSPEnv = sys.modules["rl4co.envs"].TSPEnv
    ns.CVRPEnv = sys.modules["rl4co.envs"].CVRPEnv
    ns.ops = importlib.import_module("rl4co.utils.ops")
    ns.decoding = importlib.import_module("rl4co.utils.decoding")
    ns.attention = importlib.import_module("rl4co.models.nn.attention")
    ns.am_decoder = importlib.import_module("rl4co.models.zoo.am.decoder")
    ns.am_encoder = importlib.import_module("rl4co.models.zoo.am.encoder")
    ns.am_policy = importlib.import_module("rl4co.models.zoo.am.policy")
    ns.AttentionModelPolicy = ns.am_policy.AttentionModelPolicy
    ns.AttentionModelDecoder = ns.am_decoder.AttentionModelDecoder
    ns.PrecomputedCache = ns.am_decoder.PrecomputedCache
    ns.transforms = importlib.import_module("rl4co.data.transforms")
    return ns
