"""CPU oracle for the device RandomCropPaste (TEST INFRASTRUCTURE), imported by tests/test_crop_paste_host.py and
tests/test_gpu_crop_paste.py.

* `RandomCropPaste`: the reference's da.RandomCropPaste(size, alpha=1.0, flip_p=0.5) restated with its own numpy draws and torch
  calls (`np.int` restored, as oracle/autoaugment_oracle.py does for autoaugment.py).  `Scripted` replaces those draws by given
  values, so that any box, paste corner, flip and weight can be replayed.
* `closed_form`: the same transform for given per-image parameters, the form vitb_random_crop_paste takes, in fp64 torch ops:
  out = fp32(fp64(fp32(fp64(base) * a)) + fp64(front) * (1 - a)).  The GPU tests compare the kernel with it bit for bit; the CPU
  tests compare it with `RandomCropPaste`.
"""
from __future__ import annotations

from unittest import mock

import numpy as np
import torch

if not hasattr(np, "int"):
    np.int = int  # the reference's `np.int(...)`: the builtin int, an alias numpy 1.24 removed


class RandomCropPaste(object):
    """da.RandomCropPaste, as utils.get_transform appends it with --rcpaste: `RandomCropPaste(size=args.size)`."""

    def __init__(self, size, alpha=1.0, flip_p=0.5):
        self.size = size
        self.alpha = alpha
        self.flip_p = flip_p

    def __call__(self, img):
        lam = np.random.beta(self.alpha, self.alpha)
        front_bbx1, front_bby1, front_bbx2, front_bby2 = self._rand_bbox(lam)
        img_front = img[:, front_bby1:front_bby2, front_bbx1:front_bbx2].clone()
        front_w = front_bbx2 - front_bbx1
        front_h = front_bby2 - front_bby1

        img_x1 = np.random.randint(0, high=self.size - front_w)
        img_y1 = np.random.randint(0, high=self.size - front_h)
        img_x2 = img_x1 + front_w
        img_y2 = img_y1 + front_h

        if np.random.rand() <= self.flip_p:
            img_front = img_front.flip(-1)
        if np.random.rand() <= self.flip_p:
            img = img.flip(-1)

        mixup_alpha = np.random.rand(1)
        img[:, img_y1:img_y2, img_x1:img_x2] *= mixup_alpha
        img[:, img_y1:img_y2, img_x1:img_x2] += img_front * (1 - mixup_alpha)
        return img

    def _rand_bbox(self, lam):
        W = self.size
        H = self.size
        cut_rat = np.sqrt(1. - lam)
        cut_w = np.int(W * cut_rat)
        cut_h = np.int(H * cut_rat)

        cx = np.random.randint(W)
        cy = np.random.randint(H)

        bbx1 = np.clip(cx - cut_w // 2, 0, W)
        bby1 = np.clip(cy - cut_h // 2, 0, H)
        bbx2 = np.clip(cx + cut_w // 2, 0, W)
        bby2 = np.clip(cy + cut_h // 2, 0, H)
        return bbx1, bby1, bbx2, bby2


class Scripted:
    """np.random.beta / randint / rand return the given values, in the order RandomCropPaste draws them:
    lam, cx, cy, x1, y1, flip_front, flip_img (True = flip: rand returns 0.25, else 0.75), a.  A randint value outside the range the
    reference asks for raises, so a script cannot describe a draw the reference could not make."""

    def __init__(self, lam, cx, cy, x1, y1, flip_front, flip_img, a):
        self.beta = [float(lam)]
        self.ints = [int(cx), int(cy), int(x1), int(y1)]
        self.rands = [0.25 if flip_front else 0.75, 0.25 if flip_img else 0.75, np.array([float(a)])]

    def _beta(self, *args):
        return self.beta.pop(0)

    def _randint(self, low, high=None):
        lo, hi = (0, low) if high is None else (low, high)
        v = self.ints.pop(0)
        if not lo <= v < hi:
            raise ValueError(f"scripted randint {v} outside [{lo}, {hi})")
        return v

    def _rand(self, *shape):
        v = self.rands.pop(0)
        assert isinstance(v, np.ndarray) == (shape == (1,))
        return v

    def __enter__(self):
        self._patches = [mock.patch.object(np.random, "beta", self._beta), mock.patch.object(np.random, "randint", self._randint),
                         mock.patch.object(np.random, "rand", self._rand)]
        for p in self._patches:
            p.start()
        return self

    def __exit__(self, *exc):
        for p in self._patches:
            p.stop()
        assert exc[0] is not None or not (self.beta or self.ints or self.rands), "not every scripted draw was used"
        return False


def closed_form(img: torch.Tensor, params: torch.Tensor, a: torch.Tensor) -> torch.Tensor:
    """vitb_random_crop_paste's result on the CPU: img fp32 (B, 3, S, S), params int32 (B, 8) [fx1, fy1, fw, fh, x1, y1,
    flip_front, flip_img], a float64 (B,).  An image whose box does not lie inside it comes out as NaN."""
    img, params, a = img.cpu(), params.cpu().long(), a.cpu().double()
    B, _, S, _ = img.shape
    fx1, fy1, fw, fh, x1, y1, ff, fi = (params[:, k].view(B, 1, 1, 1) for k in range(8))
    ys = torch.arange(S).view(1, 1, S, 1)
    xs = torch.arange(S).view(1, 1, 1, S)
    bi = torch.arange(B).view(B, 1, 1, 1)
    ci = torch.arange(3).view(1, 3, 1, 1)
    base = img[bi, ci, ys, torch.where(fi != 0, S - 1 - xs, xs)]
    inside = (xs >= x1) & (xs < x1 + fw) & (ys >= y1) & (ys < y1 + fh)
    u = torch.where(ff != 0, fw - 1 - (xs - x1), xs - x1)
    fr = img[bi, ci, (fy1 + ys - y1).clamp(0, S - 1), (fx1 + u).clamp(0, S - 1)]
    av = a.view(B, 1, 1, 1)
    blend = ((base.double() * av).float().double() + fr.double() * (1.0 - av)).float()
    out = torch.where(inside, blend, base)
    ok = ((params[:, :6] >= 0).all(1) & (fx1 + fw <= S).flatten() & (fy1 + fh <= S).flatten() & (x1 + fw <= S).flatten()
          & (y1 + fh <= S).flatten())
    out[~ok] = float("nan")
    return out


def reference_params(S, lam, cx, cy, x1, y1, flip_front, flip_img):
    """params row [fx1, fy1, fw, fh, x1, y1, flip_front, flip_img] of a scripted reference call (its own _rand_bbox)."""
    with mock.patch.object(np.random, "randint", side_effect=[cx, cy]):
        bx1, by1, bx2, by2 = RandomCropPaste(S)._rand_bbox(lam)
    return [int(bx1), int(by1), int(bx2 - bx1), int(by2 - by1), int(x1), int(y1), int(flip_front), int(flip_img)]
