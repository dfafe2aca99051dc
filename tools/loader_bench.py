"""Cost of feeding an epoch: the host-fed loop against DeviceLoader over a dataset resident in device memory.

    python tools/loader_bench.py [--out profiles/r5_loader_bench.json] [--n 50000] [--reps 3]

1. Epochs: one epoch of N = 50,000 seeded uint8 32x32 images through TrainEngine for the headline model (bench.py's MODEL, T = 65)
   and t17c100 (patch 4, 100 classes, T = 17), at B = 128 and 1024, AutoAugment policy none and cifar10, without and with CutMix.
   Two feeds of the same engine, alternated (a, b, a, b, ...) after one warm-up epoch of each:
   (a) host-fed, as INTEGRATION.md described it before DeviceLoader: per batch a numpy fancy-index gather of the epoch's rows (the
       sampler order) into one of two pinned uint8 staging buffers, an H2D copy on a side stream that overlaps the previous step
       (the engine's `prefetch` pattern), GpuAugment on the device into the engine's batch, CutMix, step;
   (b) DeviceLoader: the epoch's order uploaded once, the gather inside the augmentation kernel, CutMix, step.
   Reported per run: wall time per epoch (host clock around the epoch, ending in a device synchronise), img/s, and host CPU
   seconds per epoch (time.process_time of this process).
2. Kernels: CUDA-event time of the gather kernels against the contiguous ones at B = 1024, reading random rows of the resident
   50,000-image set (154 MB: larger than the 126 MB L2) and, for the contiguous kernels, a contiguous 1024-image batch.
The card's name, power limit and max SM clock are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def gpu_context():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unavailable"


def kernel_times(vb, ops, data, labels, iters=200):
    """Kernel time alone: the draws are made once, outside the timed loop."""
    import torch
    B = 1024
    N = data.shape[0]
    rows = []
    g = torch.Generator().manual_seed(0)
    idx = torch.randperm(N, generator=g)[:B].to(torch.int32).cuda()
    contiguous = data[:B].clone()
    out = torch.empty((B, 3, 32, 32), device="cuda")
    lab = torch.empty((B,), dtype=torch.int64, device="cuda")
    for policy in (None, "cifar10", "svhn"):
        aug = vb.GpuAugment(32, 4, flip=policy != "svhn", seed=1, policy=policy)
        d = aug.draw(B, "cuda")
        if policy is None:
            fns = (("contiguous_us", lambda: ops.augment(contiguous, *d, aug.mean, aug.std, out, 4)),
                   ("gather_us", lambda: ops.augment_gather(data, labels, idx, *d, aug.mean, aug.std, out, lab, 4)))
        else:
            fns = (("contiguous_us", lambda: ops.augment_autoaugment(contiguous, *d, aug.op_ids, aug.mags, aug.mean, aug.std, out, 4)),
                   ("gather_us", lambda: ops.augment_autoaugment_gather(data, labels, idx, *d, aug.op_ids, aug.mags, aug.mean, aug.std, out, lab, 4)))
        res = {"policy": policy or "none", "B": B}
        for _ in range(3):  # alternated: the two kernels see the same clocks
            for name, fn in fns:
                for _ in range(10):
                    fn()
                torch.cuda.synchronize()
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                for _ in range(iters):
                    fn()
                e.record()
                torch.cuda.synchronize()
                res.setdefault(name, []).append(round(s.elapsed_time(e) * 1e3 / iters, 2))
        rows.append(res)
    return rows


class HostFed:
    """(a): numpy gather -> pinned staging (two slots) -> H2D on a side stream overlapping the previous step -> GpuAugment."""

    def __init__(self, x_np, y_np, B):
        import torch
        self.x, self.y, self.B = x_np, y_np, B
        self.pin_x = [torch.empty((B, 32, 32, 3), dtype=torch.uint8).pin_memory() for _ in range(2)]
        self.pin_y = [torch.empty((B,), dtype=torch.int64).pin_memory() for _ in range(2)]
        self.dev_x = [torch.empty((B, 32, 32, 3), dtype=torch.uint8, device="cuda") for _ in range(2)]
        self.dev_y = [torch.empty((B,), dtype=torch.int64, device="cuda") for _ in range(2)]
        self.copied = [torch.cuda.Event() for _ in range(2)]
        self.consumed = [torch.cuda.Event() for _ in range(2)]
        self.stream = torch.cuda.Stream()

    def epoch(self, order, aug, mix, engine):
        import numpy as np
        import torch
        B = self.B
        starts = list(range(0, len(order), B))
        main = torch.cuda.current_stream()

        def stage(k, s):
            rows = order[s:s + B]
            n = len(rows)
            self.copied[k].synchronize()  # the slot's previous H2D copy has finished reading the pinned buffer
            np.take(self.x, rows, axis=0, out=self.pin_x[k].numpy()[:n])
            np.take(self.y, rows, axis=0, out=self.pin_y[k].numpy()[:n])
            self.stream.wait_event(self.consumed[k])
            with torch.cuda.stream(self.stream):
                self.dev_x[k][:n].copy_(self.pin_x[k][:n], non_blocking=True)
                self.dev_y[k][:n].copy_(self.pin_y[k][:n], non_blocking=True)
                self.copied[k].record()
            return n

        n_next = stage(0, starts[0])
        for i, s in enumerate(starts):
            k, n = i & 1, n_next
            if i + 1 < len(starts):
                n_next = stage(k ^ 1, starts[i + 1])
            main.wait_event(self.copied[k])
            img = aug(self.dev_x[k][:n], out=engine.img[:n])
            batch = (img, self.dev_y[k][:n])
            self.consumed[k].record(main)
            if mix is not None:
                engine.step(*mix(batch))
            else:
                engine.step(*batch)


def epoch_runs(vb, x_np, y_np, ds, reps):
    import numpy as np
    import torch
    import bench
    runs = []
    N = len(ds)
    for model_name, mcfg in (("headline", bench.MODEL), ("t17c100", dict(bench.MODEL, patch=4, num_classes=100))):
        for B in (128, 1024):
            for policy in (None, "cifar10"):
                for cutmix in (False, True):
                    torch.manual_seed(2045)
                    np.random.seed(0)
                    model = vb.ViT(3, mcfg["num_classes"], img_size=32, patch=mcfg["patch"], num_layers=mcfg["num_layers"], hidden=mcfg["hidden"],
                                   mlp_hidden=mcfg["mlp_hidden"], head=mcfg["head"]).cuda()
                    eng = vb.TrainEngine(model, B, smoothing=bench.SMOOTHING, mixed_targets=cutmix, **bench.ADAM)
                    aug = vb.GpuAugment(32, 4, seed=1, policy=policy)
                    mix = vb.GpuCutMix(32, 1.0) if cutmix else None
                    loader = vb.DeviceLoader(ds, B, shuffle=True, seed=0, augment=aug, mix=mix)
                    host = HostFed(x_np, y_np, B)

                    def run_a(epoch):
                        loader.set_epoch(epoch)
                        host.epoch(loader.order().numpy(), aug, mix, eng)

                    def run_b(epoch):
                        loader.set_epoch(epoch)
                        for batch in loader:
                            eng.step(*batch)

                    def timed(fn, epoch):
                        torch.cuda.synchronize()
                        c0, t0 = time.process_time(), time.perf_counter()
                        fn(epoch)
                        torch.cuda.synchronize()
                        return time.perf_counter() - t0, time.process_time() - c0

                    timed(run_a, 0)
                    timed(run_b, 0)  # warm-up: graph capture, first launches
                    a, b = [], []
                    for r in range(reps):
                        a.append(timed(run_a, 1 + r))
                        b.append(timed(run_b, 1 + r))
                    med = lambda v: sorted(v)[len(v) // 2]  # noqa: E731
                    row = {"model": model_name, "B": B, "policy": policy or "none", "cutmix": cutmix, "images": N, "reps": reps}
                    for key, v in (("a_host_fed", a), ("b_device_loader", b)):
                        wall = med([w for w, _ in v])
                        row[key] = {"epoch_s": [round(w, 4) for w, _ in v], "img_per_s": round(N / wall, 1),
                                    "host_cpu_s": [round(c, 4) for _, c in v]}
                    row["b_over_a_img_per_s"] = round(row["b_device_loader"]["img_per_s"] / row["a_host_fed"]["img_per_s"], 4)
                    runs.append(row)
                    print(json.dumps(row), flush=True)
                    del eng, model, loader, host
                    torch.cuda.empty_cache()
    return runs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--n", type=int, default=50000)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    import numpy as np
    import torch
    import vit_cifar_b200 as vb
    from vit_cifar_b200 import ops
    ops.require_device()
    vb.set_precision("bf16")
    rng = np.random.default_rng(0)
    x_np = rng.integers(0, 256, (args.n, 32, 32, 3), dtype=np.uint8)
    y_np = rng.integers(0, 10, args.n).astype(np.int64)
    ds = vb.DeviceDataset(x_np, y_np)
    res = {"gpu(name, power.limit, clocks.max.sm)": gpu_context(), "cpu_count": os.cpu_count(), "torch": torch.__version__}
    res["kernel"] = kernel_times(vb, ops, ds.images, ds.labels)
    print(json.dumps(res["kernel"]), flush=True)
    res["epochs"] = epoch_runs(vb, x_np, y_np, ds, args.reps)
    text = json.dumps(res, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
