"""Recipe for oracle/_ref: a verbatim copy of the reference's own implementation of the hot path (TEST INFRASTRUCTURE).

    [VITB_REFERENCE_ROOT=<checkout of mahbodnr/ViT-CIFAR>] python oracle/make_ref.py     (also run by __graft_entry__.build())

The reference is pure Python (no build system, nothing to compile): the "build" is a byte-for-byte copy of the modules that
`import vit` pulls in — vit.py, layers.py, criterions.py and what layers.py imports at module level (autoencoders.py,
hamburger/, nnmf/) — from the checkout VITB_REFERENCE_ROOT names, else from an installed copy in baseline/_ref/, into
oracle/_ref/.  That directory is git-ignored (no reference source enters the history); where it exists, `bench.py --impl reference` / `--impl eager` and the cpu_baseline leg time the
reference ITSELF (kind "reference") instead of the oracle port, and the live-reference tests of tests/test_oracle.py run.
A manifest with the sha256 of every copied file is written next to them.
"""
from __future__ import annotations

import hashlib
import json
import os
import shutil
import sys

DST = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")
SRC = os.environ.get("VITB_REFERENCE_ROOT") or os.path.join(os.path.dirname(os.path.dirname(DST)), "baseline", "_ref")
FILES = ["vit.py", "layers.py", "criterions.py", "autoencoders.py"]
PACKAGES = ["hamburger", "nnmf"]


def make_ref(verbose: bool = True) -> bool:
    if os.path.abspath(SRC) == DST or not os.path.isfile(os.path.join(SRC, "vit.py")):
        if verbose:
            print(f"make_ref: no reference source at {SRC}; keeping whatever is in {DST}")
        return False
    os.makedirs(DST, exist_ok=True)
    manifest = {}
    todo = [(f, f) for f in FILES]
    for pkg in PACKAGES:
        for root, _, names in os.walk(os.path.join(SRC, pkg)):
            for n in names:
                if n.endswith(".py"):
                    rel = os.path.relpath(os.path.join(root, n), SRC)
                    todo.append((rel, rel))
    for src_rel, dst_rel in todo:
        s, d = os.path.join(SRC, src_rel), os.path.join(DST, dst_rel)
        os.makedirs(os.path.dirname(d), exist_ok=True)
        shutil.copyfile(s, d)
        manifest[dst_rel] = hashlib.sha256(open(d, "rb").read()).hexdigest()
    json.dump({"source": SRC, "files": manifest}, open(os.path.join(DST, "MANIFEST.json"), "w"), indent=1, sort_keys=True)
    if verbose:
        print(f"make_ref: copied {len(manifest)} files into {DST}")
    return True


if __name__ == "__main__":
    sys.exit(0 if make_ref() or os.path.isdir(DST) else 1)
