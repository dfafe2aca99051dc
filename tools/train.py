"""Train the ViT on CIFAR-10 / CIFAR-100 with the reference's recipe (main.py + network.py), every step on the device.

    python tools/train.py --data-root DIR [--dataset c10|c100] [--autoaugment] [--label-smoothing] [--cutmix | --mixup] ...
    python tools/train.py --synthetic 5000 --max-epochs 2 ...            (a seeded, learnable uint8 set: tests, benchmarks)
    torchrun --nproc-per-node 8 tools/train.py ...                        (one process per GPU)

Data: the python-pickle batches from --data-root (cifar-10-batches-py/data_batch_1..5 + test_batch; cifar-100-python/train + test,
fine labels).  Nothing is downloaded.  Both sets are uploaded once (DeviceDataset); an epoch is one DeviceLoader pass (the
DistributedSampler order, batches gathered inside the augmentation kernel) through TrainEngine(metrics=True), then EvalEngine on
the resident test set.  Per epoch, as network.py does: the warm-up + cosine learning rate (network.py:113-122), the NaN check of
the parameters (network.py:226-228), the best-val_loss checkpoint (ModelCheckpoint(monitor="val_loss", save_top_k=1),
main.py:213-219) and one JSON line on stdout.  At the end the reference's checkpoint (main.py:234-237).  Flag names and defaults
are main.py's (SURVEY.md §5).
"""
from __future__ import annotations

import argparse
import json
import os
import pickle
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

NUM_CLASSES = {"c10": 10, "c100": 100}


def parse_args(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--dataset", default="c10", choices=sorted(NUM_CLASSES))
    ap.add_argument("--data-root", default="data")
    ap.add_argument("--synthetic", type=int, default=0, metavar="N", help="train on N seeded synthetic images (and N // 5 test images)")
    ap.add_argument("--batch-size", type=int, default=128)
    ap.add_argument("--eval-batch-size", type=int, default=256)
    ap.add_argument("--lr", type=float, default=1e-3)
    ap.add_argument("--min-lr", type=float, default=1e-5)
    ap.add_argument("--max-epochs", type=int, default=200)
    ap.add_argument("--warmup-epoch", type=int, default=5)
    ap.add_argument("--beta1", type=float, default=0.9)
    ap.add_argument("--beta2", type=float, default=0.999)
    ap.add_argument("--weight-decay", type=float, default=5e-5)
    ap.add_argument("--optimizer", default="adam", choices=["adam", "sgd"])
    ap.add_argument("--label-smoothing", action="store_true")
    ap.add_argument("--smoothing", type=float, default=0.1)
    ap.add_argument("--autoaugment", action="store_true")
    ap.add_argument("--cutmix", action="store_true")
    ap.add_argument("--mixup", action="store_true")
    ap.add_argument("--dropout", type=float, default=0.0)
    ap.add_argument("--patch", type=int, default=8)
    ap.add_argument("--head", type=int, default=12)
    ap.add_argument("--num-layers", type=int, default=7)
    ap.add_argument("--hidden", type=int, default=384)
    ap.add_argument("--mlp-hidden", type=int, default=384)
    ap.add_argument("--no-encoder-mlp", dest="encoder_mlp", action="store_false")
    ap.add_argument("--off-cls-token", dest="is_cls_token", action="store_false")
    ap.add_argument("--seed", type=int, default=2045)
    ap.add_argument("--out-dir", default="models", help="where the best-val_loss and the final checkpoint are written")
    ap.add_argument("--experiment-name", default=None, help="file name of the final checkpoint (default: vit_<dataset>)")
    args = ap.parse_args(argv)
    if args.batch_size < 1 or args.eval_batch_size < 1 or args.max_epochs < 1:
        ap.error("--batch-size, --eval-batch-size and --max-epochs must be >= 1")
    if args.cutmix and args.mixup:
        ap.error("choose one of --cutmix and --mixup")
    if args.synthetic < 0:
        ap.error("--synthetic must be >= 0")
    args.num_classes = NUM_CLASSES[args.dataset]
    args.experiment_name = args.experiment_name or f"vit_{args.dataset}"
    return args


def _unpickle(path):
    with open(path, "rb") as f:
        return pickle.load(f, encoding="bytes")


def read_cifar(root: str, dataset: str):
    """((train_images, train_labels), (test_images, test_labels)) from the python-pickle batches: images uint8 (N, 3, 32, 32) CHW as
    stored (DeviceDataset converts them), labels int64.  Raises FileNotFoundError naming what is missing."""
    if dataset == "c10":
        d = os.path.join(root, "cifar-10-batches-py")
        parts = {"train": [f"data_batch_{i}" for i in range(1, 6)], "test": ["test_batch"]}
        key = b"labels"
    else:
        d = os.path.join(root, "cifar-100-python")
        parts = {"train": ["train"], "test": ["test"]}
        key = b"fine_labels"
    missing = [os.path.join(d, f) for fs in parts.values() for f in fs if not os.path.isfile(os.path.join(d, f))]
    if missing:
        raise FileNotFoundError(f"CIFAR python batches not found (this tool downloads nothing): {', '.join(missing)}")
    out = []
    for split in ("train", "test"):
        xs, ys = [], []
        for f in parts[split]:
            b = _unpickle(os.path.join(d, f))
            xs.append(np.asarray(b[b"data"], dtype=np.uint8).reshape(-1, 3, 32, 32))
            ys.append(np.asarray(b[key], dtype=np.int64))
        out.append((np.concatenate(xs), np.concatenate(ys)))
    return tuple(out)


def synthetic_set(n: int, num_classes: int, seed: int, size: int = 32):
    """A seeded uint8 (n, size, size, 3) set a ViT can learn: each class is a fixed random colour pattern plus noise."""
    rng = np.random.default_rng(seed)
    protos = np.random.default_rng(12345).integers(0, 256, (num_classes, size, size, 3)).astype(np.int16)
    labels = rng.integers(0, num_classes, n).astype(np.int64)
    noise = rng.integers(-48, 49, (n, size, size, 3)).astype(np.int16)
    return np.clip(protos[labels] + noise, 0, 255).astype(np.uint8), labels


class MaybeMixUp:
    """network.py:149-167 with --mixup: MixUp (alpha = 1) on a batch with probability 0.8, else the batch as is (lambda = 1)."""

    def __init__(self, mixup):
        self.mixup = mixup

    def __call__(self, batch):
        if np.random.rand() <= 0.8:
            return self.mixup(batch)
        img, label = batch
        return img, label, label, 1.0


def main(argv=None):
    args = parse_args(argv)
    import torch
    import vit_cifar_b200 as vb
    from vit_cifar_b200.schedule import CIFAR10_MEAN, CIFAR10_STD, CIFAR100_MEAN, CIFAR100_STD

    pg, rank, world = None, 0, 1
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        import torch.distributed as dist
        local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        pg, rank, world = dist.group.WORLD, dist.get_rank(), dist.get_world_size()
    torch.manual_seed(args.seed)
    np.random.seed(args.seed)
    mean, std = (CIFAR10_MEAN, CIFAR10_STD) if args.dataset == "c10" else (CIFAR100_MEAN, CIFAR100_STD)

    if args.synthetic:
        train = synthetic_set(args.synthetic, args.num_classes, args.seed)
        test = synthetic_set(max(args.synthetic // 5, 1), args.num_classes, args.seed + 1)
    else:
        try:
            train, test = read_cifar(args.data_root, args.dataset)
        except FileNotFoundError as e:
            print(f"error: {e}", file=sys.stderr)
            return 2
    train_ds, test_ds = vb.DeviceDataset(*train, device="cuda"), vb.DeviceDataset(*test, device="cuda")
    S = train_ds.S

    model = vb.ViT(3, args.num_classes, img_size=S, patch=args.patch, dropout=args.dropout, num_layers=args.num_layers, hidden=args.hidden,
                   encoder_mlp=args.encoder_mlp, mlp_hidden=args.mlp_hidden, head=args.head, is_cls_token=args.is_cls_token).cuda()
    smoothing = args.smoothing if args.label_smoothing else 0.0
    mixed = args.cutmix or args.mixup
    engine = vb.TrainEngine(model, args.batch_size, smoothing=smoothing, lr=args.lr, betas=(args.beta1, args.beta2),
                            weight_decay=args.weight_decay, process_group=pg, mixed_targets=mixed, optimizer=args.optimizer, metrics=True)
    evaluator = vb.EvalEngine(model, batch_size=args.eval_batch_size, smoothing=smoothing, mean=mean, std=std, process_group=pg)
    aug = vb.GpuAugment(S, 4, mean, std, seed=args.seed + rank, policy="cifar10" if args.autoaugment else None)
    mix = vb.GpuCutMix(S, beta=1.0) if args.cutmix else MaybeMixUp(vb.GpuMixUp(alpha=1.0)) if args.mixup else None
    loader = vb.DeviceLoader(train_ds, args.batch_size, shuffle=True, seed=args.seed, augment=aug, mix=mix, process_group=pg)
    val_loader = vb.DeviceLoader(test_ds, args.eval_batch_size, shuffle=False, process_group=pg)
    sched = vb.WarmupCosine(args.lr, args.min_lr, args.max_epochs, args.warmup_epoch)
    hparams = {k: v for k, v in vars(args).items() if not k.startswith("_")}
    if rank == 0:
        os.makedirs(args.out_dir, exist_ok=True)

    best = float("inf")
    for epoch in range(args.max_epochs):
        lr = sched(epoch)
        engine.set_lr(lr)
        loader.set_epoch(epoch)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for batch in loader:
            if mixed:
                img, label, rand_label, lam = batch
                engine.step(img, label, rand_label, lam)
            else:
                engine.step(*batch)
        tr = engine.train_metrics()  # one host synchronisation
        t_train = time.perf_counter() - t0
        va = evaluator.run(val_loader)
        flat = engine.P[:engine.n]
        if bool(torch.isnan(flat).any()):  # network.py:226-228
            bad = [name for name, p in model.named_parameters() if bool(torch.isnan(p).any())]
            raise ValueError(f"NaN in parameters {bad} after epoch {epoch}")
        rec = {"epoch": epoch, "loss": tr["loss"], "acc": tr["acc"], "val_loss": va["val_loss"], "val_acc": va["val_acc"], "lr": lr,
               "epoch_s": round(time.perf_counter() - t0, 4), "train_s": round(t_train, 4), "img_per_s": round(tr["n"] / t_train, 1)}
        if va["val_loss"] < best:  # ModelCheckpoint(monitor="val_loss", save_top_k=1): one file, replaced on improvement
            best = va["val_loss"]
            ck = engine.checkpoint(hparams, epoch=epoch)  # (collective with several ranks)
            if rank == 0:
                torch.save(ck, os.path.join(args.out_dir, f"{args.experiment_name}-best.ckpt"))
        if rank == 0:
            print(json.dumps(rec), flush=True)

    ck = engine.checkpoint(hparams, epoch=args.max_epochs - 1)
    if rank == 0:
        torch.save(ck, os.path.join(args.out_dir, f"{args.experiment_name}.ckpt"))
    if pg is not None:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
