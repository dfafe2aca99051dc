"""The reference's AutoAugment policies (autoaugment.py, DeepVoltaire's implementation of the AutoAugment paper), restated as data
for the device kernel `vitb_augment_autoaugment` (csrc/augment.cu).

`SubPolicy(p1, op1, mag_idx1, p2, op2, mag_idx2)` applies op1 with probability p1, then op2 with probability p2; the policy picks one
of its 25 sub-policies uniformly per image.  Magnitudes are the reference's `ranges` (numpy float64, 10 bins).  Ops marked in SIGNED
draw their sign inside the op (`magnitude * random.choice([-1, 1])`); rotate does not (`rotate_with_fill(img, magnitude)`).
The reference also uses CIFAR10Policy for CIFAR-100 (utils.get_transform)."""
from __future__ import annotations

import numpy as np

# op codes of the kernel (include/vitb200.h): the order of the reference's `ranges`
OPS = ("shearX", "shearY", "translateX", "translateY", "rotate", "color", "posterize", "solarize", "contrast", "sharpness", "brightness",
       "autocontrast", "equalize", "invert")
OP_CODE = {name: i for i, name in enumerate(OPS)}
SIGNED = frozenset({"shearX", "shearY", "translateX", "translateY", "color", "contrast", "sharpness", "brightness"})

RANGES = {
    "shearX": np.linspace(0, 0.3, 10),
    "shearY": np.linspace(0, 0.3, 10),
    "translateX": np.linspace(0, 150 / 331, 10),   # a fraction of the image size: the op multiplies by img.size
    "translateY": np.linspace(0, 150 / 331, 10),
    "rotate": np.linspace(0, 30, 10),               # degrees
    "color": np.linspace(0.0, 0.9, 10),             # enhance factor 1 +- m
    "posterize": np.round(np.linspace(8, 4, 10), 0).astype(int),   # bits kept
    "solarize": np.linspace(256, 0, 10),            # threshold: i < t stays, the rest is inverted
    "contrast": np.linspace(0.0, 0.9, 10),
    "sharpness": np.linspace(0.0, 0.9, 10),
    "brightness": np.linspace(0.0, 0.9, 10),
    "autocontrast": [0] * 10,
    "equalize": [0] * 10,
    "invert": [0] * 10,
}

# ((op1, p1, magnitude_index1), (op2, p2, magnitude_index2)) per sub-policy, in the reference's order
CIFAR10_POLICY = (
    (("invert", 0.1, 7), ("contrast", 0.2, 6)),
    (("rotate", 0.7, 2), ("translateX", 0.3, 9)),
    (("sharpness", 0.8, 1), ("sharpness", 0.9, 3)),
    (("shearY", 0.5, 8), ("translateY", 0.7, 9)),
    (("autocontrast", 0.5, 8), ("equalize", 0.9, 2)),
    (("shearY", 0.2, 7), ("posterize", 0.3, 7)),
    (("color", 0.4, 3), ("brightness", 0.6, 7)),
    (("sharpness", 0.3, 9), ("brightness", 0.7, 9)),
    (("equalize", 0.6, 5), ("equalize", 0.5, 1)),
    (("contrast", 0.6, 7), ("sharpness", 0.6, 5)),
    (("color", 0.7, 7), ("translateX", 0.5, 8)),
    (("equalize", 0.3, 7), ("autocontrast", 0.4, 8)),
    (("translateY", 0.4, 3), ("sharpness", 0.2, 6)),
    (("brightness", 0.9, 6), ("color", 0.2, 8)),
    (("solarize", 0.5, 2), ("invert", 0.0, 3)),
    (("equalize", 0.2, 0), ("autocontrast", 0.6, 0)),
    (("equalize", 0.2, 8), ("equalize", 0.6, 4)),
    (("color", 0.9, 9), ("equalize", 0.6, 6)),
    (("autocontrast", 0.8, 4), ("solarize", 0.2, 8)),
    (("brightness", 0.1, 3), ("color", 0.7, 0)),
    (("solarize", 0.4, 5), ("autocontrast", 0.9, 3)),
    (("translateY", 0.9, 9), ("translateY", 0.7, 9)),
    (("autocontrast", 0.9, 2), ("solarize", 0.8, 3)),
    (("equalize", 0.8, 8), ("invert", 0.1, 3)),
    (("translateY", 0.7, 9), ("autocontrast", 0.9, 1)),
)

SVHN_POLICY = (
    (("shearX", 0.9, 4), ("invert", 0.2, 3)),
    (("shearY", 0.9, 8), ("invert", 0.7, 5)),
    (("equalize", 0.6, 5), ("solarize", 0.6, 6)),
    (("invert", 0.9, 3), ("equalize", 0.6, 3)),
    (("equalize", 0.6, 1), ("rotate", 0.9, 3)),
    (("shearX", 0.9, 4), ("autocontrast", 0.8, 3)),
    (("shearY", 0.9, 8), ("invert", 0.4, 5)),
    (("shearY", 0.9, 5), ("solarize", 0.2, 6)),
    (("invert", 0.9, 6), ("autocontrast", 0.8, 1)),
    (("equalize", 0.6, 3), ("rotate", 0.9, 3)),
    (("shearX", 0.9, 4), ("solarize", 0.3, 3)),
    (("shearY", 0.8, 8), ("invert", 0.7, 4)),
    (("equalize", 0.9, 5), ("translateY", 0.6, 6)),
    (("invert", 0.9, 4), ("equalize", 0.6, 7)),
    (("contrast", 0.3, 3), ("rotate", 0.8, 4)),
    (("invert", 0.8, 5), ("translateY", 0.0, 2)),
    (("shearY", 0.7, 6), ("solarize", 0.4, 8)),
    (("invert", 0.6, 4), ("rotate", 0.8, 4)),
    (("shearY", 0.3, 7), ("translateX", 0.9, 3)),
    (("shearX", 0.1, 6), ("invert", 0.6, 5)),
    (("solarize", 0.7, 2), ("translateY", 0.6, 7)),
    (("shearY", 0.8, 4), ("invert", 0.8, 8)),
    (("shearX", 0.7, 9), ("translateY", 0.8, 3)),
    (("shearY", 0.8, 5), ("autocontrast", 0.7, 3)),
    (("shearX", 0.7, 2), ("invert", 0.1, 5)),
)

POLICIES = {"cifar10": CIFAR10_POLICY, "svhn": SVHN_POLICY}


def kernel_table(policy):
    """(op_ids, mags, probs) of a policy (a name in POLICIES or a sequence of sub-policies) for `ops.augment_autoaugment`: two
    entries per sub-policy, op codes, raw reference magnitudes (float) and apply probabilities."""
    subs = POLICIES[policy] if isinstance(policy, str) else policy
    op_ids, mags, probs = [], [], []
    for sub in subs:
        for name, p, idx in sub:
            op_ids.append(OP_CODE[name])
            mags.append(float(RANGES[name][idx]))
            probs.append(float(p))
    return op_ids, mags, probs
