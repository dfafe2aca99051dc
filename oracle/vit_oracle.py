"""fp32 CPU restatement of the ViT-CIFAR training step (TEST INFRASTRUCTURE).

Every function cites the reference lines it follows (paths relative to the
root of a mahbodnr/ViT-CIFAR checkout).  The arithmetic is plain PyTorch fp32 on CPU, the same
library the reference itself computes with (SURVEY.md §8c: all arithmetic on
this path is ``torch``'s), written functionally over a ``dict`` of tensors that
uses the reference's ``state_dict`` names, so that weights interchange with the
reference ``vit.ViT`` unchanged.

Pinned by ``tests/golden/*.pt`` (generated from the unmodified reference by
``tests/golden/make_golden.py``) and ``tests/test_oracle.py``.
"""
from __future__ import annotations

import math
import zlib
from dataclasses import dataclass
from typing import Dict, Optional, Tuple

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

Params = Dict[str, torch.Tensor]


@dataclass(frozen=True)
class ViTConfig:
    """Constructor arguments of ``vit.ViT`` (vit.py:20-33), same names and meaning.

    ``patch`` is the NUMBER of patches per side (vit.py:37), not a pixel size.
    """

    in_c: int = 3
    num_classes: int = 10
    img_size: int = 32
    patch: int = 8
    dropout: float = 0.0
    num_layers: int = 7
    hidden: int = 384
    encoder_mlp: bool = True
    mlp_hidden: int = 384
    head: int = 12
    is_cls_token: bool = True

    @property
    def patch_size(self) -> int:  # vit.py:39
        return self.img_size // self.patch

    @property
    def patch_len(self) -> int:  # vit.py:41 (hard-codes 3 channels)
        return self.patch_size ** 2 * 3

    @property
    def num_tokens(self) -> int:  # vit.py:42
        return self.patch ** 2 + (1 if self.is_cls_token else 0)

    def param_shapes(self) -> Dict[str, Tuple[int, ...]]:
        """state_dict names and shapes in the reference's registration order (vit.py:44-63)."""
        H, M, K, T, C = self.hidden, self.mlp_hidden, self.patch_len, self.num_tokens, self.num_classes
        shapes: Dict[str, Tuple[int, ...]] = {}
        if self.is_cls_token:
            shapes["cls_token"] = (1, 1, H)
        shapes["pos_emb"] = (1, T, H)
        shapes["emb.weight"] = (H, K)
        shapes["emb.bias"] = (H,)
        for i in range(self.num_layers):
            p = f"enc.{i}."
            shapes[p + "la1.weight"] = (H,)
            shapes[p + "la1.bias"] = (H,)
            for w in ("Wq", "Wk", "Wv", "out_project"):
                shapes[p + f"attention.{w}.weight"] = (H, H)
                shapes[p + f"attention.{w}.bias"] = (H,)
            shapes[p + "la2.weight"] = (H,)
            shapes[p + "la2.bias"] = (H,)
            if self.encoder_mlp:
                shapes[p + "mlp.0.weight"] = (M, H)
                shapes[p + "mlp.0.bias"] = (M,)
                shapes[p + "mlp.3.weight"] = (H, M)
                shapes[p + "mlp.3.bias"] = (H,)
        shapes["fc.0.weight"] = (H,)
        shapes["fc.0.bias"] = (H,)
        shapes["fc.1.weight"] = (C, H)
        shapes["fc.1.bias"] = (C,)
        return shapes


# ---------------------------------------------------------------------------
# Deterministic, platform-independent initialisation (integer hash -> fp32).
# Used so that goldens need not store weights: the same bits are regenerated
# on any machine.  Not the reference's init (which is torch RNG dependent);
# numeric parity does not depend on the init distribution.
# ---------------------------------------------------------------------------

def _hash_uniform(n: int, seed: int) -> np.ndarray:
    """n values in [0, 1) with 24 significant bits (exact in fp32), splitmix64 of the index."""
    with np.errstate(over="ignore"):
        z = np.arange(n, dtype=np.uint64) + np.uint64(seed) * np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    return ((z >> np.uint64(40)).astype(np.float64) / float(1 << 24)).astype(np.float32)


def hash_init_(params: Params, seed: int = 0) -> Params:
    """Overwrite every tensor in ``params`` in place with hash-derived values."""
    for name, t in params.items():
        s = (zlib.crc32(name.encode()) + 7919 * seed) & 0x7FFFFFFF
        u = torch.from_numpy(_hash_uniform(t.numel(), s)).reshape(t.shape)
        if name.endswith("weight") and t.dim() == 2:
            v = (u - 0.5) * (2.0 / math.sqrt(t.shape[1]))
        elif name.endswith(("la1.weight", "la2.weight", "fc.0.weight")):
            v = 1.0 + (u - 0.5) * 0.2
        elif name in ("cls_token", "pos_emb"):
            v = (u - 0.5) * 1.0
        else:  # biases
            v = (u - 0.5) * 0.2
        with torch.no_grad():
            t.copy_(v.to(t.dtype))
    return params


def init_params(cfg: ViTConfig, seed: int = 0) -> Params:
    params = {k: torch.empty(s, dtype=torch.float32) for k, s in cfg.param_shapes().items()}
    return hash_init_(params, seed)


def hash_inputs(cfg: ViTConfig, batch: int, seed: int = 1) -> Tuple[torch.Tensor, torch.Tensor]:
    """Deterministic images in [-1.5, 1.5) and labels, from the same integer hash."""
    n = batch * 3 * cfg.img_size * cfg.img_size
    x = torch.from_numpy((_hash_uniform(n, 1000003 + seed) - 0.5) * 3.0).reshape(batch, 3, cfg.img_size, cfg.img_size)
    y = torch.from_numpy((_hash_uniform(batch, 2000003 + seed) * cfg.num_classes).astype(np.int64))
    return x.contiguous(), y.clamp_(0, cfg.num_classes - 1)


# ---------------------------------------------------------------------------
# Forward (follows the reference line by line)
# ---------------------------------------------------------------------------

def to_words(x: torch.Tensor, cfg: ViTConfig) -> torch.Tensor:
    """(B,C,H,W) -> (B, patch^2, ps*ps*C): vit.py:79-89.  Feature index (kh*ps+kw)*3+c."""
    ps = cfg.patch_size
    out = x.unfold(2, ps, ps).unfold(3, ps, ps).permute(0, 2, 3, 4, 5, 1)
    return out.reshape(x.size(0), cfg.patch ** 2, -1)


# ---------------------------------------------------------------------------
# nn.Dropout (layers.py:35, 38, 102).  The reference draws its masks from torch's generator; the build draws them from a
# counter-based generator (include/vitb200.h, vitb_dropout) restated here in numpy so that tests can replay the exact masks.
# `drop` arguments below are callables (site, tensor) -> tensor implementing `tensor * keep / (1 - p)`; None = eval / p = 0.
# ---------------------------------------------------------------------------
def philox4x32_10(counter: np.ndarray, key: Tuple[int, int]) -> np.ndarray:
    """Philox4x32 with 10 rounds (Salmon et al., "Parallel random numbers: as easy as 1, 2, 3", SC'11): counter (n,4) uint32,
    key two uint32 words -> (n,4) uint32."""
    c = [counter[:, i].astype(np.uint64) for i in range(4)]
    k0, k1 = np.uint64(key[0] & 0xFFFFFFFF), np.uint64(key[1] & 0xFFFFFFFF)
    m0, m1, mask = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57), np.uint64(0xFFFFFFFF)
    for _ in range(10):
        p0, p1 = m0 * c[0], m1 * c[2]
        hi0, lo0, hi1, lo1 = p0 >> np.uint64(32), p0 & mask, p1 >> np.uint64(32), p1 & mask
        c = [hi1 ^ c[1] ^ k0, lo1, hi0 ^ c[3] ^ k1, lo0]
        k0 = (k0 + np.uint64(0x9E3779B9)) & mask
        k1 = (k1 + np.uint64(0xBB67AE85)) & mask
    return np.stack(c, axis=1).astype(np.uint32)


def dropout_threshold(p: float) -> int:
    t = int(p * 65536.0 + 0.5)
    return min(max(t, 0), 65535)


def dropout_keep_mask(n: int, p: float, seed: int, site: int, step: int) -> np.ndarray:
    """The keep mask (bool, n) libvitb200 uses for (seed, site, step): one Philox call per group of 8 elements, counter =
    (group lo, group hi, site, step), key = seed; element j of a group takes 16-bit field j of the output and is kept iff it
    is >= round(p * 65536)."""
    assert n % 8 == 0
    g = np.arange(n // 8, dtype=np.uint64)
    ctr = np.stack([(g & np.uint64(0xFFFFFFFF)).astype(np.uint32), (g >> np.uint64(32)).astype(np.uint32),
                    np.full(g.shape, site, np.uint32), np.full(g.shape, step & 0xFFFFFFFF, np.uint32)], axis=1)
    r = philox4x32_10(ctr, (seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF))
    fields = np.stack([(r[:, j >> 1] >> np.uint32(16 * (j & 1))) & np.uint32(0xFFFF) for j in range(8)], axis=1)
    return (fields >= dropout_threshold(p)).reshape(-1)


def philox_drop(p: float, seed: int, step: int):
    """(site, tensor) -> tensor * keep / (1 - p) with libvitb200's mask for one encoder block's stream."""
    def drop(site: int, t: torch.Tensor) -> torch.Tensor:
        keep = torch.from_numpy(dropout_keep_mask(t.numel(), p, seed, site, step)).view(t.shape)
        return t * keep.to(t.dtype) / (1.0 - p)
    return drop


def mhsa_forward(p: Params, prefix: str, x: torch.Tensor, head: int,
                 return_attn: bool = False, drop=None):
    """layers.py:90-103.  Scale is 1/sqrt(features) (layers.py:79, 97), not 1/sqrt(head_dim)."""
    B, T, Fdim = x.shape
    d = Fdim // head
    q = F.linear(x, p[prefix + "Wq.weight"], p[prefix + "Wq.bias"]).view(B, T, head, d).transpose(1, 2)
    k = F.linear(x, p[prefix + "Wk.weight"], p[prefix + "Wk.bias"]).view(B, T, head, d).transpose(1, 2)
    v = F.linear(x, p[prefix + "Wv.weight"], p[prefix + "Wv.bias"]).view(B, T, head, d).transpose(1, 2)
    attn_map = F.softmax(torch.einsum("bhif,bhjf->bhij", q, k) / (Fdim ** 0.5), dim=-1)
    attn = torch.einsum("bhij,bhjf->bihf", attn_map, v)
    out = F.linear(attn.flatten(2), p[prefix + "out_project.weight"], p[prefix + "out_project.bias"])
    if drop is not None:
        out = drop(0, out)  # layers.py:102
    return (out, attn_map) if return_attn else out


def encoder_forward(p: Params, prefix: str, x: torch.Tensor, head: int, use_mlp: bool = True,
                    return_attn: bool = False, drop=None):
    """layers.py:44-48 (pre-LN residual wiring) and layers.py:32-39 (Linear-GELU-Linear-GELU)."""
    H = x.shape[-1]
    h1 = F.layer_norm(x, (H,), p[prefix + "la1.weight"], p[prefix + "la1.bias"], 1e-5)
    a = mhsa_forward(p, prefix + "attention.", h1, head, return_attn, drop)
    attn_map = None
    if return_attn:
        a, attn_map = a
    out = a + x
    if use_mlp:
        h2 = F.layer_norm(out, (H,), p[prefix + "la2.weight"], p[prefix + "la2.bias"], 1e-5)
        m = F.gelu(F.linear(h2, p[prefix + "mlp.0.weight"], p[prefix + "mlp.0.bias"]))
        if drop is not None:
            m = drop(1, m)  # layers.py:35
        m = F.gelu(F.linear(m, p[prefix + "mlp.3.weight"], p[prefix + "mlp.3.bias"]))
        if drop is not None:
            m = drop(2, m)  # layers.py:38
        out = m + out
    return (out, attn_map) if return_attn else out


def vit_forward(p: Params, x: torch.Tensor, cfg: ViTConfig, return_attn: bool = False, drops=None):
    """vit.py:65-77.  `drops`: None (eval, or dropout = 0: the reference default, main.py:87) or one (site, tensor) -> tensor
    callable per encoder block (training with dropout > 0)."""
    out = to_words(x, cfg)
    out = F.linear(out, p["emb.weight"], p["emb.bias"])  # vit.py:67
    if cfg.is_cls_token:
        out = torch.cat([p["cls_token"].repeat(out.size(0), 1, 1), out], dim=1)  # vit.py:69
    out = out + p["pos_emb"]  # vit.py:70
    maps = []
    for i in range(cfg.num_layers):  # vit.py:71
        out = encoder_forward(p, f"enc.{i}.", out, cfg.head, cfg.encoder_mlp, return_attn, drops[i] if drops is not None else None)
        if return_attn:
            out, am = out
            maps.append(am)
    out = out[:, 0] if cfg.is_cls_token else out.mean(1)  # vit.py:72-75
    out = F.layer_norm(out, (cfg.hidden,), p["fc.0.weight"], p["fc.0.bias"], 1e-5)
    out = F.linear(out, p["fc.1.weight"], p["fc.1.bias"])  # vit.py:76
    return (out, torch.stack(maps)) if return_attn else out


# ---------------------------------------------------------------------------
# Loss (criterions.py:13-19) and its closed-form gradient
# ---------------------------------------------------------------------------

def ls_ce_loss(logits: torch.Tensor, target: torch.Tensor, classes: int, smoothing: float) -> torch.Tensor:
    """Off-target mass is s/(C-1), target is exactly 1-s (criterions.py:16-18); mean over batch (:19)."""
    logp = logits.log_softmax(dim=-1)
    with torch.no_grad():
        q = torch.full_like(logp, smoothing / (classes - 1))
        q.scatter_(1, target.unsqueeze(1), 1.0 - smoothing)
    return torch.mean(torch.sum(-q * logp, dim=-1))


def ls_ce_dlogits(logits: torch.Tensor, target: torch.Tensor, classes: int, smoothing: float) -> torch.Tensor:
    """d loss / d logits = (softmax(z) - q) / B   (rows of q sum to 1)."""
    q = torch.full_like(logits, smoothing / (classes - 1))
    q.scatter_(1, target.unsqueeze(1), 1.0 - smoothing)
    return (logits.softmax(-1) - q) / logits.shape[0]


def augment_crop_flip_normalize(img_u8: torch.Tensor, dx: torch.Tensor, dy: torch.Tensor, flip: torch.Tensor, mean, std, pad: int) -> torch.Tensor:
    """utils.py:337-355 for given random draws: RandomCrop(S, padding=pad) at offset (dy, dx) of the zero-padded image, horizontal
    flip where flagged, ToTensor (/255, HWC -> CHW), Normalize(mean, std).  img_u8 (B,S,S,3) uint8 -> (B,3,S,S) fp32."""
    B, S = img_u8.shape[0], img_u8.shape[1]
    out = torch.empty((B, 3, S, S), dtype=torch.float32)
    m = torch.tensor(mean, dtype=torch.float32).view(3, 1, 1)
    sd = torch.tensor(std, dtype=torch.float32).view(3, 1, 1)
    for b in range(B):
        padded = F.pad(img_u8[b].permute(2, 0, 1), (pad, pad, pad, pad))              # RandomCrop pads with 0 first
        crop = padded[:, int(dy[b]):int(dy[b]) + S, int(dx[b]):int(dx[b]) + S]
        if bool(flip[b]):
            crop = crop.flip(-1)                                                       # RandomHorizontalFlip
        out[b] = (crop.float() / 255.0 - m) / sd                                       # ToTensor, Normalize
    return out


def cutmix_apply(img: torch.Tensor, perm: torch.Tensor, box) -> torch.Tensor:
    """da.py:57-68: rand_img = img[perm]; img[:, :, x1:x2, y1:y2] = rand_img[:, :, x1:x2, y1:y2] (on a copy)."""
    x1, x2, y1, y2 = box
    out = img.clone()
    out[:, :, x1:x2, y1:y2] = img[perm][:, :, x1:x2, y1:y2]
    return out


def mixup_apply(x: torch.Tensor, index: torch.Tensor, lam: float) -> torch.Tensor:
    """da.py:90: mixed_x = lam * x + (1 - lam) * x[index, :]."""
    return lam * x + (1 - lam) * x[index, :]


def mixed_ls_ce_loss(logits: torch.Tensor, target_a: torch.Tensor, target_b: torch.Tensor, lam: float, classes: int,
                     smoothing: float) -> torch.Tensor:
    """CutMix / MixUp objective, network.py:163-165: loss(out, label) * lambda + loss(out, rand_label) * (1 - lambda)."""
    return ls_ce_loss(logits, target_a, classes, smoothing) * lam + ls_ce_loss(logits, target_b, classes, smoothing) * (1.0 - lam)


# ---------------------------------------------------------------------------
# Adam with coupled L2 (torch.optim.Adam as configured at network.py:71-77)
# ---------------------------------------------------------------------------

def adam_step(params: Params, grads: Params, exp_avg: Params, exp_avg_sq: Params, step: int,
              lr: float = 1e-3, betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: float = 5e-5) -> None:
    """One in-place Adam step, ``step`` counted from 1.  Mirrors torch's single-tensor path:
    g += wd*p; m = lerp(m, g, 1-b1); v = b2*v + (1-b2) g^2;
    p -= (lr/(1-b1^t)) * m / (sqrt(v)/sqrt(1-b2^t) + eps).
    """
    b1, b2 = betas
    bc1 = 1.0 - b1 ** step
    bc2 = 1.0 - b2 ** step
    step_size = lr / bc1
    bc2_sqrt = math.sqrt(bc2)
    with torch.no_grad():
        for k, p in params.items():
            g = grads[k]
            if g is None:  # torch.optim.Adam skips parameters without a gradient
                continue
            if weight_decay != 0.0:
                g = g.add(p, alpha=weight_decay)
            exp_avg[k].lerp_(g, 1.0 - b1)
            exp_avg_sq[k].mul_(b2).addcmul_(g, g, value=1.0 - b2)
            denom = (exp_avg_sq[k].sqrt() / bc2_sqrt).add_(eps)
            p.addcdiv_(exp_avg[k], denom, value=-step_size)


def sgd_step(params: Params, grads: Params, bufs: Params, lr: float = 1e-3, momentum: float = 0.9, weight_decay: float = 5e-5) -> None:
    """In-place torch.optim.SGD step as network.py:78-84 configures it (momentum = beta1, dampening 0, no Nesterov, coupled weight
    decay); torch's single-tensor arithmetic: g += wd*p; buf = g on the first step (bufs[k] is None), else buf = momentum*buf + g;
    p -= lr*buf."""
    with torch.no_grad():
        for k, p in params.items():
            g = grads.get(k)
            if g is None:
                continue
            if weight_decay != 0.0:
                g = g.add(p, alpha=weight_decay)
            if bufs.get(k) is None:
                bufs[k] = g.clone()
            else:
                bufs[k].mul_(momentum).add_(g)
            p.add_(bufs[k], alpha=-lr)


def train_step(params: Params, x: torch.Tensor, y: torch.Tensor, cfg: ViTConfig, smoothing: float = 0.1,
               y_b: Optional[torch.Tensor] = None, lam: float = 1.0, drops=None):
    """forward + LS-CE (two-target form when y_b is given, network.py:149-167) + backward on leaf copies of ``params``;
    returns (logits, loss, grads)."""
    leaf = {k: v.detach().clone().requires_grad_(True) for k, v in params.items()}
    logits = vit_forward(leaf, x, cfg, drops=drops)
    if y_b is None:
        loss = ls_ce_loss(logits, y, cfg.num_classes, smoothing)
    else:
        loss = mixed_ls_ce_loss(logits, y, y_b, lam, cfg.num_classes, smoothing)
    loss.backward()
    # tensors the forward never touches (la2 when encoder_mlp=False) keep grad None, as in the reference
    grads = {k: (v.grad.detach() if v.grad is not None else None) for k, v in leaf.items()}
    return logits.detach(), loss.detach(), grads


# ---------------------------------------------------------------------------
# nn.Module wrapper (same state_dict names as vit.ViT) — used as the timed CPU
# baseline ("port") where the reference's source is not available (oracle/ref_shim.py).
# ---------------------------------------------------------------------------

class OracleViT(nn.Module):
    def __init__(self, cfg: ViTConfig, seed: Optional[int] = 0):
        super().__init__()
        self.cfg = cfg
        self._names = list(cfg.param_shapes().keys())
        init = init_params(cfg, seed if seed is not None else 0)
        self._p = nn.ParameterDict({k.replace(".", "__"): nn.Parameter(v) for k, v in init.items()})

    def params(self) -> Params:
        return {k: self._p[k.replace(".", "__")] for k in self._names}

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        return vit_forward(self.params(), x, self.cfg)
