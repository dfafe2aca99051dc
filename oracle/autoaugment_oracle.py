"""CPU oracle for the device AutoAugment (TEST INFRASTRUCTURE): the reference's autoaugment.py ops written with the exact Pillow calls it
makes, and utils.get_transform's training pipeline for given random draws:
RandomCrop(S, padding) -> RandomHorizontalFlip -> sub-policy -> ToTensor -> Normalize (the first two and the last two as in
oracle.augment_crop_flip_normalize).

The reference's SubPolicy(p1, op1, mag_idx1, p2, op2, mag_idx2, fillcolor=(128, 128, 128)) applies op1 if random.random() < p1,
then op2 if random.random() < p2; the signed ops draw random.choice([-1, 1]) inside the op.  Here the gates and signs are arguments.
"""
from __future__ import annotations

import importlib.util
import os

import numpy as np
import torch
import torch.nn.functional as F
from PIL import Image, ImageEnhance, ImageOps


def _load_tables():
    # the restated tables (pure data), loaded by path: a top-level `autoaugment` would clash with the reference's own module
    path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "vit-cifar_b200", "autoaugment.py")
    spec = importlib.util.spec_from_file_location("_vitb_autoaugment_tables", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


tables = _load_tables()


def reference_autoaugment_path():
    """The reference's own autoaugment.py in the first of ref_shim's places that holds one (VITB_REFERENCE_ROOT, oracle/_ref,
    baseline/_ref), or None.  oracle/_ref holds only what `import vit` needs, so a full checkout or install is what provides it."""
    from .ref_shim import CANDIDATES
    return next((os.path.join(d, "autoaugment.py") for d in CANDIDATES if os.path.isfile(os.path.join(d, "autoaugment.py"))), None)


def import_reference_autoaugment():
    """The reference's autoaugment module (CIFAR10Policy, SVHNPolicy, SubPolicy), imported from its file under a private name (the
    product has a module of the same name).  It builds its posterize range with `.astype(np.int)`, an alias numpy 1.24 removed
    (`np.int` was the builtin `int`), so that alias is restored first."""
    path = reference_autoaugment_path()
    if path is None:
        raise FileNotFoundError("no reference autoaugment.py (VITB_REFERENCE_ROOT, oracle/_ref or baseline/_ref)")
    if not hasattr(np, "int"):
        np.int = int
    spec = importlib.util.spec_from_file_location("ref_autoaugment", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod

FILL = (128, 128, 128)


def _rotate_with_fill(img, magnitude):
    rot = img.convert("RGBA").rotate(magnitude)
    return Image.composite(rot, Image.new("RGBA", rot.size, (128,) * 4), rot).convert(img.mode)


def apply_op(img: Image.Image, op: str, magnitude, sign: int = 1) -> Image.Image:
    """One op of the reference on a PIL RGB image; `sign` is what random.choice([-1, 1]) returned (ignored by unsigned ops)."""
    if op == "shearX":
        return img.transform(img.size, Image.AFFINE, (1, magnitude * sign, 0, 0, 1, 0), Image.BICUBIC, fillcolor=FILL)
    if op == "shearY":
        return img.transform(img.size, Image.AFFINE, (1, 0, 0, magnitude * sign, 1, 0), Image.BICUBIC, fillcolor=FILL)
    if op == "translateX":
        return img.transform(img.size, Image.AFFINE, (1, 0, magnitude * img.size[0] * sign, 0, 1, 0), fillcolor=FILL)
    if op == "translateY":
        return img.transform(img.size, Image.AFFINE, (1, 0, 0, 0, 1, magnitude * img.size[1] * sign), fillcolor=FILL)
    if op == "rotate":
        return _rotate_with_fill(img, magnitude)
    if op == "color":
        return ImageEnhance.Color(img).enhance(1 + magnitude * sign)
    if op == "posterize":
        return ImageOps.posterize(img, magnitude)
    if op == "solarize":
        return ImageOps.solarize(img, magnitude)
    if op == "contrast":
        return ImageEnhance.Contrast(img).enhance(1 + magnitude * sign)
    if op == "sharpness":
        return ImageEnhance.Sharpness(img).enhance(1 + magnitude * sign)
    if op == "brightness":
        return ImageEnhance.Brightness(img).enhance(1 + magnitude * sign)
    if op == "autocontrast":
        return ImageOps.autocontrast(img)
    if op == "equalize":
        return ImageOps.equalize(img)
    if op == "invert":
        return ImageOps.invert(img)
    raise ValueError(op)


def sub_policy(img: Image.Image, sub, gates=(True, True), signs=(1, 1)) -> Image.Image:
    """SubPolicy.__call__ for given draws; sub = ((op1, p1, idx1), (op2, p2, idx2)) as in autoaugment.CIFAR10_POLICY."""
    for (op, _p, idx), g, s in zip(sub, gates, signs):
        if g:
            img = apply_op(img, op, tables.RANGES[op][idx], s)
    return img


def crop_flip(img_u8: torch.Tensor, dx: int, dy: int, flip: bool, pad: int) -> np.ndarray:
    """RandomCrop(S, padding=pad) at offset (dy, dx) of the zero-padded image and the flip: (S, S, 3) uint8 HWC."""
    S = img_u8.shape[0]
    crop = F.pad(img_u8.permute(2, 0, 1), (pad, pad, pad, pad))[:, dy:dy + S, dx:dx + S]
    if flip:
        crop = crop.flip(-1)
    return crop.permute(1, 2, 0).contiguous().numpy()


def decode(code: int):
    """The kernel's code word: (sub-policy index, (gate1, gate2), (sign1, sign2))."""
    return code & 0xFF, (bool(code >> 8 & 1), bool(code >> 9 & 1)), (-1 if code >> 10 & 1 else 1, -1 if code >> 11 & 1 else 1)


def autoaugment_bytes(img_u8: torch.Tensor, dx, dy, flip, code, policy, pad: int) -> torch.Tensor:
    """crop -> flip -> sub-policy for every image, as bytes: (B, S, S, 3) uint8.  policy: a sequence of sub-policies."""
    out = []
    for b in range(img_u8.shape[0]):
        x = crop_flip(img_u8[b], int(dx[b]), int(dy[b]), flip is not None and bool(flip[b]), pad)
        sub, gates, signs = decode(int(code[b]))
        out.append(np.asarray(sub_policy(Image.fromarray(x), policy[sub], gates, signs)))
    return torch.from_numpy(np.stack(out))


def autoaugment_normalize(img_u8, dx, dy, flip, code, policy, mean, std, pad: int) -> torch.Tensor:
    """The whole training transform for given draws: (B, 3, S, S) fp32 (ToTensor + Normalize of autoaugment_bytes)."""
    x = autoaugment_bytes(img_u8, dx, dy, flip, code, policy, pad).permute(0, 3, 1, 2).float() / 255.0
    return (x - torch.tensor(mean, dtype=torch.float32).view(1, 3, 1, 1)) / torch.tensor(std, dtype=torch.float32).view(1, 3, 1, 1)
