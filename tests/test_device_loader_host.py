"""CPU: DeviceLoader's epoch order and sharding (against torch's DistributedSampler), DeviceDataset's layouts, the host-side checks
of the gather kernels' wrappers, the C ABI entries, and tools/train.py's data reader and flags.  No device work."""
import os
import pickle
import re
import sys

import numpy as np
import pytest
import torch
from torch.utils.data import DistributedSampler

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))

import vit_cifar_b200 as vb  # noqa: E402
from vit_cifar_b200 import loader as L  # noqa: E402


class _Aug:
    """Stands in for GpuAugment where only the order is looked at."""
    size = 4


@pytest.fixture
def fake_group(monkeypatch):
    """A process-group stand-in: (world, rank) tuples answered by torch.distributed.get_world_size / get_rank."""
    import torch.distributed as dist
    monkeypatch.setattr(dist, "get_world_size", lambda g: g[0])
    monkeypatch.setattr(dist, "get_rank", lambda g: g[1])


def cpu_set(n, S=4):
    g = torch.Generator().manual_seed(n)
    return vb.DeviceDataset(torch.randint(0, 256, (n, S, S, 3), generator=g, dtype=torch.uint8), torch.arange(n) % 10, device="cpu")


@pytest.mark.parametrize("n,world,B", [(37, 1, 8), (37, 2, 8), (37, 3, 5), (2, 3, 4), (1, 2, 1), (64, 2, 16)])
def test_epoch_order_is_distributed_samplers(fake_group, n, world, B):
    ds = cpu_set(n)
    for rank in range(world):
        ld = vb.DeviceLoader(ds, B, shuffle=True, seed=9, augment=_Aug(), process_group=(world, rank) if world > 1 else None)
        for epoch in range(4):
            s = DistributedSampler(range(n), num_replicas=world, rank=rank, shuffle=True, seed=9, drop_last=False)
            s.set_epoch(epoch)
            ld.set_epoch(epoch)
            assert ld.order().tolist() == list(s), (rank, epoch)
        assert len(ld) == -(-(-(-n // world)) // B)  # every rank: ceil(ceil(n / world) / B) batches


def test_orders_differ_between_epochs_and_seeds():
    a, b, c = (L.distributed_order(100, 1, 0, s, e) for s, e in ((0, 0), (0, 1), (1, 0)))
    assert sorted(a.tolist()) == list(range(100))
    assert not torch.equal(a, b) and not torch.equal(a, c)


@pytest.mark.parametrize("n,world,B", [(10, 3, 4), (2, 3, 1), (1000, 8, 256), (7, 1, 3)])
def test_validation_shards_are_disjoint_and_cover_the_set(fake_group, n, world, B):
    ds = cpu_set(n)
    seen = []
    for rank in range(world):
        ld = vb.DeviceLoader(ds, B, shuffle=False, process_group=(world, rank) if world > 1 else None)
        rows = []
        for img, lab in ld:
            assert img.dtype == torch.uint8 and img.shape[1:] == (4, 4, 3) and 1 <= img.shape[0] <= B
            # each yielded slice is a view of the resident set: find its rows through the images
            lo = img.data_ptr() - ds.images.data_ptr()
            first = lo // (4 * 4 * 3)
            rows += list(range(first, first + img.shape[0]))
            assert torch.equal(lab, ds.labels[first:first + img.shape[0]])
        assert len(rows) == ld.num_samples and len(ld) == -(-len(rows) // B)
        seen += rows
    assert sorted(seen) == list(range(n)) and len(set(seen)) == n


def test_dataset_layouts():
    hwc = np.random.default_rng(0).integers(0, 256, (5, 6, 6, 3), dtype=np.uint8)
    chw = np.ascontiguousarray(hwc.transpose(0, 3, 1, 2))
    a, b = vb.DeviceDataset(hwc, [1, 2, 3, 4, 5], device="cpu"), vb.DeviceDataset(chw, np.arange(5), device="cpu")
    assert torch.equal(a.images, b.images) and a.images.is_contiguous() and a.images.shape == (5, 6, 6, 3)
    assert a.labels.dtype == torch.int64 and len(a) == 5 and a.S == 6
    with pytest.raises(ValueError, match="empty"):
        vb.DeviceDataset(np.zeros((0, 4, 4, 3), np.uint8), np.zeros(0, np.int64), device="cpu")
    with pytest.raises(ValueError, match="uint8"):
        vb.DeviceDataset(hwc.astype(np.float32), np.arange(5), device="cpu")
    with pytest.raises(ValueError, match="square"):
        vb.DeviceDataset(np.zeros((2, 4, 5, 3), np.uint8), np.arange(2), device="cpu")
    with pytest.raises(ValueError, match="labels"):
        vb.DeviceDataset(hwc, np.arange(4), device="cpu")
    with pytest.raises(ValueError, match="integers"):
        vb.DeviceDataset(hwc, np.zeros(5, np.float32), device="cpu")


def test_loader_argument_checks():
    ds = cpu_set(10)
    with pytest.raises(ValueError, match="augment"):
        vb.DeviceLoader(ds, 4, shuffle=True)
    with pytest.raises(ValueError, match="training"):
        vb.DeviceLoader(ds, 4, shuffle=False, augment=_Aug())
    with pytest.raises(ValueError, match="batch_size"):
        vb.DeviceLoader(ds, 0, shuffle=False)
    with pytest.raises(TypeError):
        vb.DeviceLoader(torch.zeros(3), 4, shuffle=False)
    big = _Aug()
    big.size = 32
    with pytest.raises(ValueError, match="32 x 32"):
        vb.DeviceLoader(ds, 4, augment=big)


def _gather_args(N=4, S=8, B=3):
    return dict(data_u8=torch.zeros((N, S, S, 3), dtype=torch.uint8), labels_src=torch.zeros(N, dtype=torch.int64),
                idx=torch.zeros(B, dtype=torch.int32), dx=None, dy=None, flip=None, mean=(0.5,) * 3, std=(0.5,) * 3,
                out=torch.zeros((B, 3, S, S)), labels_dst=torch.zeros(B, dtype=torch.int64), pad=4)


@pytest.mark.parametrize("change,match", [
    (dict(data_u8=torch.zeros((4, 8, 8, 3), dtype=torch.float32)), "uint8"),
    (dict(data_u8=torch.zeros((4, 3, 8, 8), dtype=torch.uint8)), "HWC"),
    (dict(data_u8=torch.zeros((0, 8, 8, 3), dtype=torch.uint8), labels_src=torch.zeros(0, dtype=torch.int64)), "empty"),
    (dict(idx=torch.zeros(3, dtype=torch.int64)), "int32"),
    (dict(idx=torch.zeros(0, dtype=torch.int32), out=torch.zeros((0, 3, 8, 8)), labels_dst=torch.zeros(0, dtype=torch.int64)), "non-empty"),
    (dict(labels_src=torch.zeros(4, dtype=torch.int32)), "labels_src"),
    (dict(out=torch.zeros((3, 3, 8, 8), dtype=torch.float16)), "out"),
    (dict(out=torch.zeros((3, 8, 8, 3))), "out"),
    (dict(labels_dst=torch.zeros(2, dtype=torch.int64)), "labels_dst"),
    (dict(dx=torch.zeros(3, dtype=torch.int64)), "dx"),
    (dict(flip=torch.zeros(3, dtype=torch.bool)), "flip"),
    ({}, "CUDA device"),  # CPU tensors: refused before any launch
])
def test_gather_wrappers_check_their_arguments(change, match):
    from vit_cifar_b200 import ops
    a = {**_gather_args(), **change}
    with pytest.raises(ValueError, match=match):
        ops.augment_gather(a["data_u8"], a["labels_src"], a["idx"], a["dx"], a["dy"], a["flip"], a["mean"], a["std"], a["out"], a["labels_dst"], a["pad"])
    code = torch.zeros(a["idx"].numel(), dtype=torch.int32)
    with pytest.raises(ValueError, match=match):
        ops.augment_autoaugment_gather(a["data_u8"], a["labels_src"], a["idx"], a["dx"], a["dy"], a["flip"], code, [0, 0], [0.1, 0.1],
                                       a["mean"], a["std"], a["out"], a["labels_dst"], a["pad"])


def test_policy_gather_refuses_images_over_64_pixels():
    from vit_cifar_b200 import ops
    a = _gather_args(N=2, S=65, B=1)
    with pytest.raises(ValueError, match="64"):
        ops.augment_autoaugment_gather(a["data_u8"], a["labels_src"], a["idx"], None, None, None, torch.zeros(1, dtype=torch.int32), [0, 0],
                                       [0.1, 0.1], a["mean"], a["std"], a["out"], a["labels_dst"], 4)
    with pytest.raises(ValueError, match="CUDA device"):  # the crop / flip form has no size limit: it gets as far as the device check
        ops.augment_gather(a["data_u8"], a["labels_src"], a["idx"], None, None, None, a["mean"], a["std"], a["out"], a["labels_dst"], 4)


def test_gpu_augment_index_needs_labels():
    aug = vb.GpuAugment(8, 4, device="cpu")
    with pytest.raises(ValueError, match="labels"):
        aug(torch.zeros((2, 8, 8, 3), dtype=torch.uint8), index=torch.zeros(1, dtype=torch.int32))


NEW = ("vitb_augment_crop_flip_normalize_gather", "vitb_augment_autoaugment_gather", "vitb_train_loss_accumulate")


def test_new_entry_points_are_declared_and_bound():
    from vit_cifar_b200 import _lib
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "vitb200.h")).read(), flags=re.S)
    for name in NEW:
        assert re.search(rf"\bint {name}\(", src), name
        assert name in _lib.SIGNATURES
    # argument counts of the ctypes table against the header's prototypes
    for name in NEW:
        proto = re.search(rf"\b{name}\((.*?)\);", src, flags=re.S).group(1)
        assert len(_lib.SIGNATURES[name][1]) == len(proto.split(",")), name


def _write_cifar(root, c100=False):
    rng = np.random.default_rng(1)
    d = os.path.join(root, "cifar-100-python" if c100 else "cifar-10-batches-py")
    os.makedirs(d)
    names = ["train", "test"] if c100 else [f"data_batch_{i}" for i in range(1, 6)] + ["test_batch"]
    key = b"fine_labels" if c100 else b"labels"
    expect = {}
    for f in names:
        x = rng.integers(0, 256, (3, 3072), dtype=np.uint8)
        y = list(rng.integers(0, 100 if c100 else 10, 3))
        with open(os.path.join(d, f), "wb") as fh:
            pickle.dump({b"data": x, key: y, b"coarse_labels": [0, 0, 0]}, fh)
        expect[f] = (x, y)
    return expect


@pytest.mark.parametrize("c100", [False, True])
def test_cifar_pickle_reader(tmp_path, c100):
    import train
    expect = _write_cifar(str(tmp_path), c100)
    (xtr, ytr), (xte, yte) = train.read_cifar(str(tmp_path), "c100" if c100 else "c10")
    tr_names = ["train"] if c100 else [f"data_batch_{i}" for i in range(1, 6)]
    assert xtr.shape == (3 * len(tr_names), 3, 32, 32) and xtr.dtype == np.uint8 and ytr.dtype == np.int64
    assert np.array_equal(xtr[:3].reshape(3, -1), expect[tr_names[0]][0]) and list(ytr[:3]) == expect[tr_names[0]][1]
    assert np.array_equal(xte.reshape(3, -1), expect["test" if c100 else "test_batch"][0])
    # the stored layout is CHW: the red plane comes first
    ds = vb.DeviceDataset(xte, yte, device="cpu")
    assert torch.equal(ds.images[0, :, :, 0].flatten(), torch.from_numpy(expect["test" if c100 else "test_batch"][0][0, :1024].copy()))


def test_cifar_reader_names_missing_files(tmp_path):
    import train
    with pytest.raises(FileNotFoundError, match="data_batch_1"):
        train.read_cifar(str(tmp_path), "c10")


def test_train_flags():
    import train
    a = train.parse_args([])
    assert (a.batch_size, a.eval_batch_size, a.lr, a.min_lr, a.max_epochs, a.warmup_epoch) == (128, 256, 1e-3, 1e-5, 200, 5)
    assert (a.beta1, a.beta2, a.weight_decay, a.smoothing, a.dropout, a.seed) == (0.9, 0.999, 5e-5, 0.1, 0.0, 2045)
    assert (a.patch, a.head, a.num_layers, a.hidden, a.mlp_hidden, a.encoder_mlp, a.is_cls_token) == (8, 12, 7, 384, 384, True, True)
    assert not (a.autoaugment or a.cutmix or a.mixup or a.label_smoothing) and a.num_classes == 10 and a.optimizer == "adam"
    b = train.parse_args(["--dataset", "c100", "--autoaugment", "--label-smoothing", "--cutmix", "--synthetic", "100", "--off-cls-token"])
    assert b.num_classes == 100 and b.autoaugment and b.cutmix and b.synthetic == 100 and not b.is_cls_token
    with pytest.raises(SystemExit):
        train.parse_args(["--cutmix", "--mixup"])
    with pytest.raises(SystemExit):
        train.parse_args(["--batch-size", "0"])


def test_train_help_runs():
    import subprocess
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "train.py"), "--help"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "--synthetic" in r.stdout and "--warmup-epoch" in r.stdout


def test_synthetic_set_is_seeded_and_learnable_shape():
    import train
    x1, y1 = train.synthetic_set(50, 10, 3)
    x2, y2 = train.synthetic_set(50, 10, 3)
    assert x1.dtype == np.uint8 and x1.shape == (50, 32, 32, 3) and np.array_equal(x1, x2) and np.array_equal(y1, y2)
    assert not np.array_equal(x1, train.synthetic_set(50, 10, 4)[0])
