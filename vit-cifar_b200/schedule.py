"""Epoch-level pieces around the hot step (SURVEY.md §8f ranks 1-3): the reference's learning-rate schedule, its
validation step, its checkpoint format (host code only) and its training-time input transform on the device.

Learning rate — network.py:113-122: `CosineAnnealingLR(T_max=max_epochs, eta_min=min_lr)` wrapped in
`warmup_scheduler.GradualWarmupScheduler(multiplier=1.0, total_epoch=warmup_epoch)`, stepped once per epoch by Lightning.
The wrapper is the un-vendored dependency ildoonet/pytorch-gradual-warmup-lr (git HEAD, setup.sh:5); its published
algorithm with multiplier == 1.0 is restated here in closed form (tests/test_host_logic.py replays the library's class
against torch's real CosineAnnealingLR and compares):

    e = number of scheduler steps taken so far = index of the epoch about to be trained
    e <= W            lr = base * e / W              (epoch 0 trains with lr = 0, as upstream does)
    e == W + 1        lr = base                      (the cosine schedule's own epoch 0)
    e >  W + 1        lr = min_lr + (base - min_lr) * (1 + cos(pi * (e - W - 1) / T_max)) / 2
"""
from __future__ import annotations

import math
from typing import Dict, Optional

import torch


def warmup_cosine_lr(epoch: int, base_lr: float, min_lr: float, max_epochs: int, warmup_epoch: int) -> float:
    """Learning rate in force while epoch `epoch` (0-based) is trained."""
    if epoch < 0:
        raise ValueError("epoch must be >= 0")
    W = int(warmup_epoch)
    if W > 0 and epoch <= W:
        return base_lr * (float(epoch) / W)
    # upstream divides by zero for warmup_epoch == 0; here that simply means "no warm-up": the cosine schedule from epoch 0
    t = epoch - (W + 1) if W > 0 else epoch
    return min_lr + (base_lr - min_lr) * (1.0 + math.cos(math.pi * t / max_epochs)) / 2.0


class WarmupCosine:
    """`engine.set_lr(sched(epoch))` once per epoch reproduces network.py:113-122 for a TrainEngine / FusedAdam."""

    def __init__(self, base_lr: float = 1e-3, min_lr: float = 1e-5, max_epochs: int = 200, warmup_epoch: int = 5):
        self.base_lr, self.min_lr, self.max_epochs, self.warmup_epoch = float(base_lr), float(min_lr), int(max_epochs), int(warmup_epoch)

    def __call__(self, epoch: int) -> float:
        return warmup_cosine_lr(epoch, self.base_lr, self.min_lr, self.max_epochs, self.warmup_epoch)


@torch.no_grad()
def evaluate(model, criterion, batches) -> Dict[str, float]:
    """network.py:388-395 over an iterable of (img, label): mean loss and accuracy (each batch weighted by its size)."""
    was_training = model.training
    model.eval()
    dev = next(model.parameters()).device
    n, loss_sum, correct = 0, 0.0, 0
    for img, label in batches:
        img, label = img.to(dev, non_blocking=True), label.to(dev, non_blocking=True)
        out = model(img)
        loss_sum += float(criterion(out, label)) * img.shape[0]
        correct += int(torch.eq(out.argmax(-1), label).sum())
        n += img.shape[0]
    model.train(was_training)
    return {"val_loss": loss_sum / max(n, 1), "val_acc": correct / max(n, 1), "n": n}


# ---------------------------------------------------------------------------------------------
# checkpoints: what `trainer.save_checkpoint` writes (main.py:234-237) and run_model.py:12-37 reads — a dict with
# "state_dict" (keys prefixed by the LightningModule attribute, "model.") and "hyper_parameters"
# ---------------------------------------------------------------------------------------------
def to_lightning_checkpoint(model, hyper_parameters: Optional[dict] = None, prefix: str = "model.") -> dict:
    sd = {prefix + k: v.detach().to("cpu", copy=True) for k, v in model.state_dict().items()}
    return {"state_dict": sd, "hyper_parameters": dict(hyper_parameters or {})}


def save_checkpoint(model, path: str, hyper_parameters: Optional[dict] = None) -> None:
    torch.save(to_lightning_checkpoint(model, hyper_parameters), path)


def load_checkpoint(model, ckpt, strict: bool = False, prefix: str = "model."):
    """`ckpt`: a path or an already loaded dict in the reference's format (or a bare state_dict).  Keys are matched after
    stripping `prefix`; with strict=False (run_model.py:37) unknown / missing keys are reported, not fatal."""
    if isinstance(ckpt, (str, bytes)) or hasattr(ckpt, "__fspath__"):
        ckpt = torch.load(ckpt, map_location="cpu")
    sd = ckpt.get("state_dict", ckpt)
    sd = {(k[len(prefix):] if k.startswith(prefix) else k): v for k, v in sd.items()}
    return model.load_state_dict(sd, strict=strict)


# ---------------------------------------------------------------------------------------------
# training-time input transform on the device (utils.py:337-355)
# ---------------------------------------------------------------------------------------------
CIFAR10_MEAN, CIFAR10_STD = (0.4914, 0.4822, 0.4465), (0.2470, 0.2435, 0.2616)      # utils.py:380
CIFAR100_MEAN, CIFAR100_STD = (0.5071, 0.4867, 0.4408), (0.2675, 0.2565, 0.2761)    # utils.py:470
# utils.py, the svhn branch of get_dataloader: as remembered from the reference, not yet compared with its source
SVHN_MEAN, SVHN_STD = (0.4377, 0.4438, 0.4728), (0.1980, 0.2010, 0.1970)


def crop_paste_box(S: int, lam: torch.Tensor, cx: torch.Tensor, cy: torch.Tensor, ux: torch.Tensor, uy: torch.Tensor) -> torch.Tensor:
    """da.RandomCropPaste's box arithmetic for B images as int32 (B, 6) [fx1, fy1, fw, fh, x1, y1]: lam (float64) ~ Beta(1, 1),
    cx / cy the box centres (integers in [0, S)), ux / uy float64 uniforms in [0, 1) for the paste corner.
        cut = np.int(S * np.sqrt(1 - lam)); f?1, f?2 = clip(c? - cut // 2, 0, S), clip(c? + cut // 2, 0, S)   (_rand_bbox)
        x1 = randint(0, S - fw) = floor(ux * (S - fw)), y1 likewise
    fw == S (lam == 0 exactly) makes the reference's randint(0, 0) raise; here the paste starts at 0."""
    cut = torch.floor(S * torch.sqrt(1.0 - lam)).to(torch.int64)
    c = torch.stack((cx, cy), 1).to(torch.int64)
    half = (cut // 2)[:, None]
    lo, hi = (c - half).clamp(0, S), (c + half).clamp(0, S)
    w = hi - lo
    corner = torch.floor(torch.stack((ux, uy), 1) * (S - w)).to(torch.int64)
    return torch.cat((lo, w, corner), 1).to(torch.int32)


class GpuAugment:
    """get_transform's training pipeline — RandomCrop(size, padding) + RandomHorizontalFlip + [AutoAugment policy] + ToTensor +
    Normalize(mean, std) [+ RandomCropPaste] — on a raw uint8 (B, S, S, 3) batch that is already on the device: one kernel instead of a per-image PIL
    pipeline in DataLoader workers, and 4x fewer bytes over PCIe than normalised fp32 batches.
    The random draws use a torch.Generator on the device (torchvision and the reference draw them on the host, per image).

    policy: None (no AutoAugment), "cifar10" (CIFAR10Policy, which the reference also uses for CIFAR-100) or "svhn" (SVHNPolicy);
    the reference's recipes are
        c10 / c100   GpuAugment(32, 4, mean, std, policy="cifar10")
        svhn         GpuAugment(32, 4, mean, std, flip=False, policy="svhn")
    With a policy, each image also draws its sub-policy (uniform), the two gates (rand < p) and two signs (+-1, p = 1/2) after the
    crop and flip draws; every op reproduces the Pillow call of the reference's autoaugment.py (csrc/augment.cu).  The draws follow
    the reference's distribution, not Python's `random` stream.

    rcpaste=True (main.py --rcpaste) appends da.RandomCropPaste(size): a second kernel pass over `out`, in place
    (csrc/augment.cu), with its draws (draw_crop_paste) taken after all the others of the batch.  size <= 64."""

    def __init__(self, size: int = 32, padding: int = 4, mean=CIFAR10_MEAN, std=CIFAR10_STD, flip: bool = True, seed: int = 0,
                 device="cuda", policy: Optional[str] = None, rcpaste: bool = False):
        self.size, self.padding, self.mean, self.std, self.flip = int(size), int(padding), tuple(mean), tuple(std), bool(flip)
        self.gen = torch.Generator(device=device)
        self.gen.manual_seed(seed)
        self.policy = policy
        self.rcpaste = bool(rcpaste)
        if self.rcpaste:
            from .ops import CROP_PASTE_MAX_S
            if self.size > CROP_PASTE_MAX_S:
                raise ValueError(f"rcpaste=True takes images of at most {CROP_PASTE_MAX_S} x {CROP_PASTE_MAX_S} pixels, got size={self.size}")
        if policy is not None:
            from .autoaugment import POLICIES, kernel_table
            if policy not in POLICIES:
                raise ValueError(f"policy must be None or one of {sorted(POLICIES)}, got {policy!r}")
            self.op_ids, self.mags, probs = kernel_table(policy)
            self.n_sub = len(self.op_ids) // 2
            self.probs = torch.tensor(probs, dtype=torch.float64, device=device).view(self.n_sub, 2)

    def draw(self, B: int, device):
        """(dx, dy, flip) without a policy; (dx, dy, flip, code) with one (code as vitb_augment_autoaugment reads it)."""
        hi = 2 * self.padding + 1
        dx = torch.randint(0, hi, (B,), generator=self.gen, device=device, dtype=torch.int32)
        dy = torch.randint(0, hi, (B,), generator=self.gen, device=device, dtype=torch.int32)
        fl = (torch.rand((B,), generator=self.gen, device=device) < 0.5).to(torch.uint8) if self.flip else None  # p = 0.5
        if self.policy is None:
            return dx, dy, fl
        sub = torch.randint(0, self.n_sub, (B,), generator=self.gen, device=device, dtype=torch.int32)
        gate = torch.rand((B, 2), generator=self.gen, device=device, dtype=torch.float64) < self.probs[sub.long()]
        neg = torch.rand((B, 2), generator=self.gen, device=device) < 0.5
        g, s = gate.to(torch.int32), neg.to(torch.int32)
        code = sub | (g[:, 0] << 8) | (g[:, 1] << 9) | (s[:, 0] << 10) | (s[:, 1] << 11)
        return dx, dy, fl, code

    def draw_crop_paste(self, B: int, device):
        """(params, a) of da.RandomCropPaste(size) for B images, as vitb_random_crop_paste reads them: params int32 (B, 8) =
        [fx1, fy1, fw, fh, x1, y1, flip_front, flip_img], a float64 (B,).  lam ~ Beta(1, 1) = U[0, 1), the box centres uniform
        over [0, S), the paste corner uniform over [0, S - fw) x [0, S - fh), each flip rand <= 0.5 and a ~ U[0, 1), as the
        reference draws them (not numpy's stream).  On the device, without a host synchronisation."""
        u = torch.rand((B, 6), generator=self.gen, device=device, dtype=torch.float64)  # lam, ux, uy, two flips, a
        c = torch.randint(0, self.size, (B, 2), generator=self.gen, device=device)
        box = crop_paste_box(self.size, u[:, 0], c[:, 0], c[:, 1], u[:, 1], u[:, 2])
        params = torch.cat((box, (u[:, 3:5] <= 0.5).to(torch.int32)), 1)
        return params, u[:, 5].contiguous()

    def __call__(self, img_u8: torch.Tensor, out: Optional[torch.Tensor] = None, index: Optional[torch.Tensor] = None,
                 labels: Optional[torch.Tensor] = None, labels_out: Optional[torch.Tensor] = None):
        """Transform the uint8 (B, S, S, 3) batch `img_u8` into fp32 (B, 3, S, S) `out` (allocated when None) and return it.

        With `index` (int32 (B,) on the device), `img_u8` is a resident (N, S, S, 3) dataset and `labels` its int64 (N,) labels:
        the batch is rows index[0..B) of it, gathered inside the same kernel, with the same draws as for the contiguous batch
        img_u8[index].  Returns (out, labels_out), labels_out[i] = labels[index[i]] (allocated when None).  A row outside [0, N)
        comes out as a NaN image with label -1."""
        from . import ops
        if index is None:
            B = img_u8.shape[0]
            if out is None:
                out = torch.empty((B, 3, self.size, self.size), dtype=torch.float32, device=img_u8.device)
            if self.policy is None:
                dx, dy, fl = self.draw(B, img_u8.device)
                ops.augment(img_u8, dx, dy, fl, self.mean, self.std, out, self.padding)
            else:
                dx, dy, fl, code = self.draw(B, img_u8.device)
                ops.augment_autoaugment(img_u8, dx, dy, fl, code, self.op_ids, self.mags, self.mean, self.std, out, self.padding)
            if self.rcpaste:
                ops.random_crop_paste(out, *self.draw_crop_paste(B, img_u8.device))
            return out
        if labels is None:
            raise ValueError("index= gathers from a dataset: give its labels= too")
        B, dev = int(index.numel()), img_u8.device
        if out is None:
            out = torch.empty((B, 3, self.size, self.size), dtype=torch.float32, device=dev)
        if labels_out is None:
            labels_out = torch.empty((B,), dtype=torch.int64, device=dev)
        if self.policy is None:
            dx, dy, fl = self.draw(B, dev)
            ops.augment_gather(img_u8, labels, index, dx, dy, fl, self.mean, self.std, out, labels_out, self.padding)
        else:
            dx, dy, fl, code = self.draw(B, dev)
            ops.augment_autoaugment_gather(img_u8, labels, index, dx, dy, fl, code, self.op_ids, self.mags, self.mean, self.std, out, labels_out,
                                           self.padding)
        if self.rcpaste:
            ops.random_crop_paste(out, *self.draw_crop_paste(B, dev))
        return out, labels_out


# ---------------------------------------------------------------------------------------------
# batch-level CutMix / MixUp on the device (da.py:51-93; used at network.py:149-158)
# ---------------------------------------------------------------------------------------------
def cutmix_box(size: int, lambda_: float, r_x: float, r_y: float):
    """The box arithmetic of da.py:60-70: returns (x1, x2, y1, y2) and the area-corrected lambda."""
    import numpy as np
    r_w = size * np.sqrt(1 - lambda_)
    r_h = size * np.sqrt(1 - lambda_)
    x1 = int(np.clip(r_x - r_w // 2, a_min=0, a_max=size))
    x2 = int(np.clip(r_x + r_w // 2, a_min=0, a_max=size))
    y1 = int(np.clip(r_y - r_h // 2, a_min=0, a_max=size))
    y2 = int(np.clip(r_y + r_h // 2, a_min=0, a_max=size))
    return (x1, x2, y1, y2), 1 - (x2 - x1) * (y2 - y1) / (size * size)


class GpuCutMix:
    """da.CutMix (da.py:51-77) for a batch that is already on the device: same random draws in the same order from the same
    generators (torch.randperm, then np.random.beta / uniform), same return tuple (img, label, rand_label, lambda_); the paste is
    one kernel instead of a clone + fancy-index gather + slice assignment."""

    def __init__(self, size: int, beta: float):
        self.size, self.beta = size, beta

    def __call__(self, batch):
        import numpy as np
        from . import ops
        img, label = batch
        rand_idx = torch.randperm(img.size(0))
        lambda_ = np.random.beta(self.beta, self.beta)
        r_x = np.random.uniform(0, self.size)
        r_y = np.random.uniform(0, self.size)
        box, lambda_ = cutmix_box(self.size, lambda_, r_x, r_y)
        idx = rand_idx.pin_memory().to(img.device, non_blocking=True)  # from pageable memory the copy would wait for the device
        out = torch.empty_like(img)
        ops.batch_mix(img, idx.to(torch.int32), out, 0, 1.0, box)
        return out, label, label[idx], lambda_


class GpuMixUp:
    """da.MixUp (da.py:80-93) on the device: lam ~ Beta(alpha, alpha), index = randperm, lam * x + (1 - lam) * x[index]."""

    def __init__(self, alpha: float = 0.1):
        self.alpha = alpha

    def __call__(self, batch):
        import numpy as np
        from . import ops
        x, y = batch
        lam = np.random.beta(self.alpha, self.alpha)
        index = torch.randperm(x.size(0)).to(x.device)
        out = torch.empty_like(x)
        ops.batch_mix(x, index.to(torch.int32), out, 1, lam)
        return out, y, y[index], lam
