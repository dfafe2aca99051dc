"""A dataset that stays in device memory and the per-epoch loader over it: what the reference gets from its DataLoader and
DistributedSampler (utils.py:452-470; main.py:220-231 hands the loaders to Lightning, which adds the sampler under DDP).

The whole CIFAR-10 training set is 50,000 x 3,072 bytes = 154 MB of uint8, so it is uploaded once and kept in HBM.  A training
batch is then a slice of the epoch's index order, and the gather of its rows happens inside the augmentation kernel
(``GpuAugment(..., index=)``): per step the host only slices a device tensor and launches.

* Training order (``shuffle=True``): the order of ``torch.utils.data.DistributedSampler(range(N), num_replicas=world,
  rank=rank, shuffle=True, seed=seed, drop_last=False)`` after ``set_epoch(e)``; one replica without a process group.  Every
  rank's shard is padded to ceil(N / world) indices, so every rank yields the same number of batches (the fused data-parallel
  step needs all ranks in ``step()`` the same number of times); the last batch keeps the remainder (no drop_last).
* Validation order (``shuffle=False``): contiguous uint8 slices of the resident set, which ``EvalEngine(mean=, std=)`` takes.
  With a process group each rank gets its own contiguous shard, unpadded: the union of the shards is the set, once.
"""
from __future__ import annotations

import math
from typing import Iterator, Optional

import numpy as np
import torch


def _as_tensor(a) -> torch.Tensor:
    return a if isinstance(a, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(a))


def to_hwc(images) -> torch.Tensor:
    """(N, S, S, 3) HWC uint8 as is, or (N, 3, S, S) CHW uint8 (torchvision's SVHN `.data`) converted to HWC."""
    t = _as_tensor(images)
    if t.dtype != torch.uint8 or t.dim() != 4:
        raise ValueError(f"images must be a uint8 (N, S, S, 3) or (N, 3, S, S) array, got {t.dtype} {tuple(t.shape)}")
    if t.shape[3] == 3 and t.shape[1] == t.shape[2]:
        return t
    if t.shape[1] == 3 and t.shape[2] == t.shape[3]:
        return t.permute(0, 2, 3, 1)
    raise ValueError(f"images must be square (N, S, S, 3) HWC or (N, 3, S, S) CHW, got {tuple(t.shape)}")


def distributed_order(n: int, world: int, rank: int, seed: int, epoch: int, shuffle: bool = True) -> torch.Tensor:
    """Rank `rank`'s indices for epoch `epoch`, as DistributedSampler(range(n), world, rank, shuffle, seed, drop_last=False) yields
    them after set_epoch(epoch): a permutation from torch.Generator seeded with seed + epoch, padded by repeating its head to a
    multiple of `world`, then every world-th index from `rank`.  int64 CPU tensor of ceil(n / world) entries."""
    if n < 1 or world < 1 or not 0 <= rank < world:
        raise ValueError(f"bad sampler arguments n={n} world={world} rank={rank}")
    if shuffle:
        g = torch.Generator()
        g.manual_seed(int(seed) + int(epoch))
        order = torch.randperm(n, generator=g)
    else:
        order = torch.arange(n)
    per_rank = math.ceil(n / world)
    total = per_rank * world
    if total > n:
        order = order.repeat(math.ceil(total / n))[:total]
    return order[rank:total:world]


def shard_bounds(n: int, world: int, rank: int):
    """[lo, hi) of rank `rank`'s contiguous validation shard: the shards are disjoint and cover range(n)."""
    return n * rank // world, n * (rank + 1) // world


class DeviceDataset:
    """A uint8 image set and its labels, uploaded to `device` once.

    images: (N, S, S, 3) HWC uint8, or (N, 3, S, S) CHW uint8 (converted to HWC once, here); numpy arrays or tensors.
    labels: N integer class labels."""

    def __init__(self, images_u8, labels, device="cuda"):
        hwc = to_hwc(images_u8)
        lab = _as_tensor(labels)
        if lab.dtype.is_floating_point or lab.dtype == torch.bool or lab.dim() != 1:
            raise ValueError(f"labels must be a vector of integers, got {lab.dtype} {tuple(lab.shape)}")
        if hwc.shape[0] < 1:
            raise ValueError("empty dataset: no images")
        if lab.shape[0] != hwc.shape[0]:
            raise ValueError(f"{hwc.shape[0]} images but {lab.shape[0]} labels")
        self.device = torch.device(device)
        self.images = hwc.contiguous().to(self.device)
        self.labels = lab.to(torch.int64).contiguous().to(self.device)
        self.N, self.S = int(self.images.shape[0]), int(self.images.shape[1])

    def __len__(self) -> int:
        return self.N


class DeviceLoader:
    """One epoch of batches over a DeviceDataset per iteration: ``loader.set_epoch(e)`` and then ``for batch in loader``.

    shuffle=True (training) needs `augment` (a GpuAugment; ``GpuAugment(S, padding=0, flip=False)`` is the bare ToTensor +
    Normalize) and yields ``(img, label)``, or ``(img, label, rand_label, lam)`` with `mix` (GpuCutMix / GpuMixUp): what
    ``TrainEngine.step`` takes.  `img` and `label` are views of buffers the loader reuses for the next batch, written on the
    current stream; hand them to the step before advancing the iterator.
    shuffle=False (validation) yields ``(img_u8, label)`` slices of the resident set for ``EvalEngine(mean=, std=)``.
    process_group: shard as DistributedSampler (training) or contiguously (validation) over its ranks."""

    def __init__(self, dataset: DeviceDataset, batch_size: int, shuffle: bool = True, seed: int = 0, augment=None, mix=None,
                 process_group=None):
        if not isinstance(dataset, DeviceDataset):
            raise TypeError(f"dataset must be a DeviceDataset, got {type(dataset).__name__}")
        if int(batch_size) < 1:
            raise ValueError(f"batch_size must be >= 1, got {batch_size}")
        if shuffle and augment is None:
            raise ValueError("shuffle=True builds batches inside the augmentation kernel: give augment= (GpuAugment(S, padding=0, "
                             "flip=False) for no augmentation)")
        if not shuffle and (augment is not None or mix is not None):
            raise ValueError("shuffle=False yields the validation set in order, unaugmented: augment= and mix= are for training")
        if augment is not None and augment.size != dataset.S:
            raise ValueError(f"augment is for {augment.size} x {augment.size} images, the dataset holds {dataset.S} x {dataset.S}")
        self.dataset, self.B, self.shuffle, self.seed = dataset, int(batch_size), bool(shuffle), int(seed)
        self.augment, self.mix = augment, mix
        self.world, self.rank = 1, 0
        if process_group is not None:
            import torch.distributed as dist
            self.world, self.rank = dist.get_world_size(process_group), dist.get_rank(process_group)
        self.epoch = 0
        if self.shuffle:
            self.num_samples = math.ceil(dataset.N / self.world)
            dev, S, B = dataset.device, dataset.S, min(self.B, self.num_samples)
            self._img = torch.empty((B, 3, S, S), dtype=torch.float32, device=dev)
            self._label = torch.empty((B,), dtype=torch.int64, device=dev)
        else:
            self.lo, self.hi = shard_bounds(dataset.N, self.world, self.rank)
            self.num_samples = self.hi - self.lo

    def set_epoch(self, epoch: int) -> None:
        """The epoch whose order the next iteration yields (DistributedSampler.set_epoch)."""
        self.epoch = int(epoch)

    def order(self) -> torch.Tensor:
        """This rank's dataset rows for the current epoch, in the order they are batched (int64, host)."""
        if self.shuffle:
            return distributed_order(self.dataset.N, self.world, self.rank, self.seed, self.epoch)
        return torch.arange(self.lo, self.hi)

    def __len__(self) -> int:
        return math.ceil(self.num_samples / self.B)

    def __iter__(self) -> Iterator[tuple]:
        ds, B = self.dataset, self.B
        if not self.shuffle:
            for s in range(self.lo, self.hi, B):
                e = min(s + B, self.hi)
                yield ds.images[s:e], ds.labels[s:e]
            return
        # the epoch's order crosses PCIe once (ceil(N / world) int32), asynchronously from pinned memory
        order_dev = self.order().to(torch.int32).pin_memory().to(ds.device, non_blocking=True)
        for s in range(0, self.num_samples, B):
            n = min(B, self.num_samples - s)
            img, label = self.augment(ds.images, out=self._img[:n], index=order_dev[s:s + n], labels=ds.labels, labels_out=self._label[:n])
            yield self.mix((img, label)) if self.mix is not None else (img, label)
