"""TEST / BENCH INFRASTRUCTURE ONLY -- recipe that stages the reference's hot-path files under
``oracle/_ref/`` so that the *unmodified* reference can run on the GPU box.

``/root/reference`` exists only in the build container.  The reference is Python, so there is
nothing to compile: this recipe copies exactly the files SURVEY.md section 8c lists (the ones
``oracle/ref_standin.py`` imports verbatim) to ``oracle/_ref/rl4co/...`` with their relative
paths.  ``oracle/_ref/`` is git-ignored (reference sources never enter the history) but NOT
gpurun-ignored, so it travels to the GPU box with the snapshot like a built ``.so`` does.
``__graft_entry__.build()`` calls :func:`make` whenever ``/root/reference`` is present.

Consumers (bench / fixture infrastructure; the product package never imports ``oracle/``):
  * ``bench.py --impl reference`` and ``bench.py``'s ``cpu_baseline`` leg  (kind "reference")
  * ``tests/golden/make_golden.py``, which records what the tests compare against; the tests themselves
    read only the recorded fixtures

    python oracle/make_ref.py            # (re)stage
    python oracle/make_ref.py --check    # verify staged files are byte-identical to the source
"""

from __future__ import annotations

import hashlib
import json
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SRC_ROOT = os.environ.get("RL4CO_REFERENCE_SRC", "/root/reference")
DST_ROOT = os.path.join(HERE, "_ref")

#: hot-path files of the reference (SURVEY.md 8c) + the next-row files of 8f whose parity tests use them
FILES = [
    "rl4co/data/dataset.py",
    "rl4co/data/generate_data.py",
    "rl4co/data/transforms.py",
    "rl4co/data/utils.py",
    "rl4co/envs/common/base.py",
    "rl4co/envs/common/distribution_utils.py",
    "rl4co/envs/common/utils.py",
    "rl4co/envs/routing/cvrp/env.py",
    "rl4co/envs/routing/cvrp/generator.py",
    "rl4co/envs/routing/cvrp/render.py",
    "rl4co/envs/routing/cvrp/local_search.py",
    "rl4co/envs/routing/tsp/env.py",
    "rl4co/envs/routing/tsp/generator.py",
    "rl4co/envs/routing/tsp/local_search.py",
    "rl4co/envs/routing/tsp/render.py",
    "rl4co/envs/routing/sdvrp/env.py",
    "rl4co/envs/routing/op/env.py",
    "rl4co/envs/routing/op/generator.py",
    "rl4co/envs/routing/op/render.py",
    "rl4co/envs/routing/pctsp/env.py",
    "rl4co/envs/routing/pctsp/generator.py",
    "rl4co/envs/routing/pctsp/render.py",
    "rl4co/models/common/constructive/__init__.py",
    "rl4co/models/common/constructive/base.py",
    "rl4co/models/common/constructive/autoregressive/__init__.py",
    "rl4co/models/common/constructive/autoregressive/decoder.py",
    "rl4co/models/common/constructive/autoregressive/encoder.py",
    "rl4co/models/common/constructive/autoregressive/policy.py",
    "rl4co/models/common/constructive/nonautoregressive/__init__.py",
    "rl4co/models/common/constructive/nonautoregressive/decoder.py",
    "rl4co/models/common/constructive/nonautoregressive/encoder.py",
    "rl4co/models/common/constructive/nonautoregressive/policy.py",
    "rl4co/models/nn/attention.py",
    "rl4co/models/nn/mlp.py",
    "rl4co/models/nn/moe.py",
    "rl4co/models/nn/ops.py",
    "rl4co/models/nn/env_embeddings/context.py",
    "rl4co/models/nn/env_embeddings/dynamic.py",
    "rl4co/models/nn/env_embeddings/init.py",
    "rl4co/models/nn/graph/attnnet.py",
    "rl4co/models/zoo/am/decoder.py",
    "rl4co/models/zoo/am/encoder.py",
    "rl4co/models/zoo/am/policy.py",
    "rl4co/models/rl/reinforce/baselines.py",
    "rl4co/models/rl/common/critic.py",
    "rl4co/utils/decoding.py",
    "rl4co/utils/ops.py",
    "rl4co/utils/pylogger.py",
]


def _sha(path: str) -> str:
    with open(path, "rb") as f:
        return hashlib.sha256(f.read()).hexdigest()


def source_available() -> bool:
    return os.path.isdir(os.path.join(SRC_ROOT, "rl4co"))


def make(verbose: bool = True) -> str:
    """Stage FILES from the read-only reference tree into oracle/_ref (idempotent)."""
    if not source_available():
        raise FileNotFoundError(f"reference tree not found at {SRC_ROOT}")
    manifest = {}
    for rel in FILES:
        src = os.path.join(SRC_ROOT, rel)
        if not os.path.exists(src):
            continue  # optional file (e.g. a local_search stub absent in some revisions)
        dst = os.path.join(DST_ROOT, rel)
        os.makedirs(os.path.dirname(dst), exist_ok=True)
        if not os.path.exists(dst) or _sha(dst) != _sha(src):
            shutil.copyfile(src, dst)
        manifest[rel] = _sha(dst)
    with open(os.path.join(DST_ROOT, "MANIFEST.json"), "w") as f:
        json.dump({"source": SRC_ROOT, "files": manifest}, f, indent=1, sort_keys=True)
    if verbose:
        print(f"oracle/_ref: {len(manifest)} reference files staged (unmodified copies, sha256 in MANIFEST.json)")
    return DST_ROOT


def check() -> bool:
    """True when every staged file is byte-identical to the reference source (or the manifest)."""
    mpath = os.path.join(DST_ROOT, "MANIFEST.json")
    if not os.path.exists(mpath):
        return False
    with open(mpath) as f:
        manifest = json.load(f)["files"]
    ok = True
    for rel, sha in manifest.items():
        dst = os.path.join(DST_ROOT, rel)
        if not os.path.exists(dst) or _sha(dst) != sha:
            print(f"MISMATCH vs manifest: {rel}")
            ok = False
        src = os.path.join(SRC_ROOT, rel)
        if os.path.exists(src) and _sha(src) != sha:
            print(f"MISMATCH vs source: {rel}")
            ok = False
    return ok


if __name__ == "__main__":
    if "--check" in sys.argv:
        sys.exit(0 if check() else 1)
    make()
