"""Import the UNMODIFIED reference modules (TEST INFRASTRUCTURE).

The first of these that holds the reference's ``vit.py``: the checkout of
mahbodnr/ViT-CIFAR named by ``VITB_REFERENCE_ROOT``; ``oracle/_ref``, the verbatim
copy ``oracle/make_ref.py`` makes; ``baseline/_ref``, where an installed copy of the
reference is placed beside a checkout.  Both directories are git-ignored: the
reference is not part of this repository.  Without it, the tests that run it live
skip, and the fixtures under tests/golden/ (its stored outputs) stand in for it.
Two shims are needed (SURVEY.md §0):
  * vit.py:3 imports ``torchsummary`` (unused, not installed);
  * layers.py:12 -> nnmf/optimizer.py:8 imports the private
    ``torch.optim.optimizer._dispatch_sqrt`` removed in torch 2.11.
"""
from __future__ import annotations

import math
import os
import sys
import types

_REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CANDIDATES = [os.path.abspath(p) for p in (os.environ.get("VITB_REFERENCE_ROOT"), os.path.join(_REPO, "oracle", "_ref"), os.path.join(_REPO, "baseline", "_ref")) if p]
REFERENCE_ROOT = next((p for p in CANDIDATES if os.path.isfile(os.path.join(p, "vit.py"))), CANDIDATES[0])
SKIP_REASON = "the reference's source is not available (VITB_REFERENCE_ROOT, oracle/_ref or baseline/_ref)"


def reference_available() -> bool:
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "vit.py"))


def import_reference():
    """Returns (vit, layers, criterions) reference modules."""
    if not reference_available():
        raise FileNotFoundError(f"no reference source at {REFERENCE_ROOT}")
    import torch
    import torch.optim.optimizer as opt_mod

    sys.modules.setdefault("torchsummary", types.ModuleType("torchsummary"))
    if not hasattr(opt_mod, "_dispatch_sqrt"):
        opt_mod._dispatch_sqrt = lambda x: x.sqrt() if torch.is_tensor(x) else math.sqrt(x)
    # The product package also ships modules called `vit`, `layers`, `criterions`
    # inside its own namespace; the reference's are top-level, so there is no clash.
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    import vit as ref_vit  # noqa: E402
    import layers as ref_layers  # noqa: E402
    import criterions as ref_criterions  # noqa: E402

    assert os.path.dirname(ref_vit.__file__) == REFERENCE_ROOT, ref_vit.__file__
    return ref_vit, ref_layers, ref_criterions
