"""TEST / BASELINE INFRASTRUCTURE -- stages the reference's own Python tree for the GPU box.

    python oracle/build_ref.py [--force]

The reference (liupei101/AdvMIL) is a pure-Python script tree without an installer; `/root/reference` exists only in the
build container.  This recipe copies the packages the hot path and its caller need -- model/, loss/, optim/, eval/, utils/,
dataset/, config/ (Python sources and the yaml config only) -- from where they lie under /root/reference into
`oracle/_ref/`, which is git-ignored (never part of the history) but NOT gpurun-ignored, so it travels to the GPU box
next to the built `.so`.  Consumers (all of them checkers / baselines, never the product path):

  * `bench.py --impl reference` and the `cpu_baseline` leg: the reference's own modules, losses, optimiser factory and
    `MyHandler._update_disc/_update_gen` on the box's host cores (`cpu_baseline.kind = "reference"`);
  * `bench.py`'s `gpu_eager_baseline`: the same unmodified handler methods with the modules `.cuda()` on the same B200;
  * `bench.py`'s `dropin_handler`: the unmodified handler methods around the advmil_b200 modules (four-import swap of
    INTEGRATION.md §1).

Nothing under advmil_b200/ imports it (tests/test_host_cpu.py enforces that).
"""
from __future__ import annotations

import hashlib
import json
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.environ.get("ADVMIL_REFERENCE", "/root/reference")
DST = os.path.join(HERE, "_ref")
PACKAGES = ("model", "loss", "optim", "eval", "utils", "dataset", "config")
KEEP = (".py", ".yaml")


def source_available() -> bool:
    return os.path.isdir(os.path.join(SRC, "model"))


def staged() -> bool:
    return os.path.isfile(os.path.join(DST, "MANIFEST.json")) and os.path.isdir(os.path.join(DST, "model"))


def build_ref(force: bool = False) -> str | None:
    """Copies the reference packages to oracle/_ref (idempotent).  Returns the staged path, or None when neither the
    source tree nor an earlier staging exists (e.g. on a box that got neither)."""
    if not source_available():
        return DST if staged() else None
    files = []
    for pkg in PACKAGES:
        for root, _dirs, names in os.walk(os.path.join(SRC, pkg)):
            for n in sorted(names):
                if n.endswith(KEEP):
                    files.append(os.path.relpath(os.path.join(root, n), SRC))
    files.sort()
    hsh = hashlib.sha256()
    for rel in files:
        hsh.update(rel.encode())
        hsh.update(open(os.path.join(SRC, rel), "rb").read())
    digest = hsh.hexdigest()
    man = os.path.join(DST, "MANIFEST.json")
    if not force and os.path.isfile(man):
        try:
            if json.load(open(man)).get("sha256") == digest:
                return DST
        except Exception:
            pass
    if os.path.isdir(DST):
        shutil.rmtree(DST)
    for rel in files:
        out = os.path.join(DST, rel)
        os.makedirs(os.path.dirname(out), exist_ok=True)
        shutil.copyfile(os.path.join(SRC, rel), out)
    json.dump({"source": SRC, "sha256": digest, "files": files,
               "note": "verbatim copy of the reference's Python packages; git-ignored; baseline/checker use only"},
              open(man, "w"), indent=1)
    return DST


if __name__ == "__main__":
    print(build_ref(force="--force" in sys.argv))
