"""Cost of RandomCropPaste on the device (GpuAugment(rcpaste=True)).

    python tools/crop_paste_bench.py [--out profiles/r6_crop_paste_bench.json] [--n 50000] [--reps 3]

1. Kernel: CUDA-event time of vitb_random_crop_paste on fp32 (B, 3, 32, 32) batches at B = 1024 and 8192 (12 MB and 101 MB: the
   first stays in the 126 MB L2 between launches, the second mostly does not), with parameters drawn once by GpuAugment; beside it
   the draws (GpuAugment.draw_crop_paste) and the augmentation kernel without a policy at the same B, each alternated three times.
   Bytes: the kernel reads and writes every image once (2 x 12 B per pixel).
2. Epochs: one DeviceLoader epoch of N = 50,000 seeded uint8 32x32 images through TrainEngine for the headline model (bench.py's
   MODEL) at B = 128 and 1024, policy cifar10, without and with rcpaste, alternated (a, b, a, b, ...) after one warm-up epoch of
   each.  Wall time per epoch: a host clock around the epoch, ending in a device synchronise.
The card's name, power limit and max SM clock are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from loader_bench import gpu_context  # noqa: E402


def event_us(fn, iters):
    import torch
    for _ in range(10):
        fn()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(iters):
        fn()
    e.record()
    torch.cuda.synchronize()
    return round(s.elapsed_time(e) * 1e3 / iters, 2)


def kernel_times(vb, ops, iters=200):
    import torch
    rows = []
    for B in (1024, 8192):
        g = torch.Generator().manual_seed(B)
        img = torch.randn(B, 3, 32, 32, generator=g).cuda()
        u8 = torch.randint(0, 256, (B, 32, 32, 3), generator=g, dtype=torch.uint8).cuda()
        out = torch.empty_like(img)
        aug = vb.GpuAugment(32, 4, seed=1, rcpaste=True)
        params, a = aug.draw_crop_paste(B, "cuda")
        d = aug.draw(B, "cuda")
        fns = (("crop_paste_us", lambda: ops.random_crop_paste(img, params, a)),
               ("draw_crop_paste_us", lambda: aug.draw_crop_paste(B, "cuda")),
               ("augment_us", lambda: ops.augment(u8, *d, aug.mean, aug.std, out, 4)))
        res = {"B": B, "S": 32, "crop_paste_bytes": 2 * B * 3 * 32 * 32 * 4}
        for _ in range(3):
            for name, fn in fns:
                res.setdefault(name, []).append(event_us(fn, iters))
        best = min(res["crop_paste_us"])
        res["crop_paste_GB_per_s_at_best"] = round(res["crop_paste_bytes"] / (best * 1e-6) / 1e9, 1)
        rows.append(res)
        print(json.dumps(res), flush=True)
    return rows


def epoch_runs(vb, ds, reps):
    import numpy as np
    import torch
    import bench
    runs = []
    N = len(ds)
    m = bench.MODEL
    for B in (128, 1024):
        torch.manual_seed(2045)
        np.random.seed(0)
        model = vb.ViT(3, m["num_classes"], img_size=32, patch=m["patch"], num_layers=m["num_layers"], hidden=m["hidden"],
                       mlp_hidden=m["mlp_hidden"], head=m["head"]).cuda()
        eng = vb.TrainEngine(model, B, smoothing=bench.SMOOTHING, **bench.ADAM)
        loaders = {k: vb.DeviceLoader(ds, B, shuffle=True, seed=0, augment=vb.GpuAugment(32, 4, seed=1, policy="cifar10", rcpaste=k))
                   for k in (False, True)}

        def timed(rc, epoch):
            loader = loaders[rc]
            loader.set_epoch(epoch)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for batch in loader:
                eng.step(*batch)
            torch.cuda.synchronize()
            return time.perf_counter() - t0

        timed(False, 0)
        timed(True, 0)  # warm-up: graph capture, first launches
        t = {False: [], True: []}
        for r in range(reps):
            for rc in (False, True):
                t[rc].append(timed(rc, 1 + r))
        med = lambda v: sorted(v)[len(v) // 2]  # noqa: E731
        row = {"model": "headline", "B": B, "policy": "cifar10", "images": N, "reps": reps}
        for rc, key in ((False, "a_plain"), (True, "b_rcpaste")):
            row[key] = {"epoch_s": [round(v, 4) for v in t[rc]], "img_per_s": round(N / med(t[rc]), 1)}
        row["b_over_a_img_per_s"] = round(row["b_rcpaste"]["img_per_s"] / row["a_plain"]["img_per_s"], 4)
        runs.append(row)
        print(json.dumps(row), flush=True)
        del eng, model, loaders
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
    res = {"gpu(name, power.limit, clocks.max.sm)": gpu_context(), "torch": torch.__version__}
    res["kernel"] = kernel_times(vb, ops)
    rng = np.random.default_rng(0)
    ds = vb.DeviceDataset(rng.integers(0, 256, (args.n, 32, 32, 3), dtype=np.uint8), rng.integers(0, 10, args.n).astype(np.int64))
    res["epochs"] = epoch_runs(vb, ds, args.reps)
    text = json.dumps(res, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
