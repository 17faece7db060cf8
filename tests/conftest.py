import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")

# the CPU oracle works on [B, N, 128]-sized tensors: torch's default of one thread per core is ~14x slower than 16
# threads on the 128-core GPU hosts (measured in bench.py's thread probe)
torch.set_num_threads(min(16, os.cpu_count() or 1))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def pytest_collection_modifyitems(config, items):
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


class Golden:
    """npz fixture produced by tests/golden/make_golden.py from the live reference."""

    def __init__(self, name):
        self.name = name
        self.z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))

    def __getitem__(self, k):
        return torch.from_numpy(self.z[k])

    def __contains__(self, k):
        return k in self.z.files

    def weights(self, device="cpu"):
        return {k[3:]: torch.from_numpy(self.z[k]).to(device) for k in self.z.files if k.startswith("w::")}

    def inst(self, device="cpu"):
        return {k[6:]: torch.from_numpy(self.z[k]).to(device) for k in self.z.files if k.startswith("inst::")}


@pytest.fixture(scope="session")
def golden():
    cache = {}

    def _get(name):
        if name not in cache:
            cache[name] = Golden(name)
        return cache[name]

    return _get


def env_of(name):
    for env in ("pctsp", "sdvrp", "cvrp"):
        if env in name:
            return env
    if "_op" in name:
        return "op"
    return "tsp" if "tsp" in name else "cvrp"


def name_seeded_weights(state_dict, seed):
    """Mirror of tests/golden/make_golden.py::name_seeded_weights: weights that depend only on
    (parameter name, shape, seed), so a fixture need not store them."""
    import zlib

    new = {}
    for k in sorted(state_dict.keys()):
        v = state_dict[k]
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
    return new


def seeded_weights_from_meta(meta, seed):
    """name_seeded_weights of a state_dict described by tests/golden/make_golden.py::weight_meta (names, shapes and
    float flags as JSON)."""
    import json

    spec = json.loads(str(meta))
    return name_seeded_weights({k: torch.zeros(shape, dtype=torch.float32 if is_float else torch.int64)
                                for k, (shape, is_float) in spec.items()}, int(seed))


def seeded_instances(spec, crcs):
    """The instances tests/golden/make_golden.py::seeded_instances drew from the reference's generator, regenerated
    by the project's generator under the same torch seed; every array must match the reference's CRC-32."""
    import json
    import zlib

    from rl4co_b200.envs import get_env

    spec = json.loads(str(spec))
    torch.manual_seed(spec["seed"])
    td = get_env(spec["env"], generator_params=dict(num_loc=spec["n"])).generator(spec["batch"])
    inst = {k: td[k] for k in td.keys()}
    assert set(inst) == set(crcs), (sorted(inst), sorted(crcs))
    for k, v in inst.items():
        assert zlib.crc32(v.numpy().tobytes()) == int(crcs[k]), f"regenerated {spec['env']} instances differ in {k}"
    return inst


def golden_case(z, tag):
    """One case `tag/...` of a multi-case fixture as tensors: (instances, outputs, weights); instances and weights
    are regenerated from their seeds when the fixture holds only those."""
    pre = tag + "/"
    arr = {k[len(pre):]: z[k] for k in z.files if k.startswith(pre)}
    outs = {k: torch.from_numpy(v.astype(np.int64) if v.dtype == np.uint8 else v) for k, v in arr.items()
            if "::" not in k and v.dtype.kind != "U"}
    inst = seeded_instances(arr["gen"], {k[5:]: v for k, v in arr.items() if k.startswith("crc::")}) \
        if "gen" in arr else None
    W = seeded_weights_from_meta(arr["w_meta"], arr["weight_seed"]) if "w_meta" in arr else None
    return inst, outs, W
