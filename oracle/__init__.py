"""CPU oracle for the ViT-CIFAR training hot path.

TEST INFRASTRUCTURE ONLY.  Nothing under ``oracle/`` is part of the product:
only ``tests/``, ``__graft_entry__.smoke()`` and the ``cpu_baseline`` /
``--impl reference`` legs of ``bench.py`` may import it, and there only as the
checker (or as the timed CPU baseline), never as the thing shipped.  The
product path (``vit_cifar_b200``) never imports this package and fails loudly
when its CUDA library is missing.

Parity status: the reference ships no tests or golden vectors (SURVEY.md §4),
so the oracle is pinned against the reference itself: ``tests/golden/make_golden.py``
imports the unmodified reference modules from a checkout of it (two import
shims, see ``oracle/ref_shim.py``), runs them in fp32 on CPU and commits the
outputs as fixtures; ``tests/test_oracle.py`` checks this restatement against
those fixtures (and against the live reference whenever its source is available).
"""
from .vit_oracle import (  # noqa: F401
    ViTConfig,
    hash_init_,
    init_params,
    hash_inputs,
    vit_forward,
    to_words,
    mhsa_forward,
    encoder_forward,
    ls_ce_loss,
    ls_ce_dlogits,
    mixed_ls_ce_loss,
    cutmix_apply,
    mixup_apply,
    philox4x32_10,
    dropout_threshold,
    dropout_keep_mask,
    philox_drop,
    augment_crop_flip_normalize,
    adam_step,
    sgd_step,
    train_step,
    OracleViT,
)
