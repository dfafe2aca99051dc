"""Cost of the training transform with the reference's AutoAugment, on the device and on the host.

    python tools/augment_bench.py [--out FILE.json] [--cpu-images 2000] [--rounds 5] [--steps 40]

1. Kernel time (CUDA events, after warm-up) of vitb_augment_crop_flip_normalize (policy none) and vitb_augment_autoaugment
   (cifar10, svhn) at B = 1024 and 8192 on random 32x32 images and GpuAugment's own draws; bytes moved (3 B in, 12 B out per
   pixel) over kernel time as a share of 7.7 TB/s.  The working set fits in L2 (126 MB): this is the on-chip-resident rate.
2. The reference's host pipeline on one core: RandomCrop(32, 4) + RandomHorizontalFlip + CIFAR10Policy + ToTensor + Normalize on
   PIL images, with the reference's own autoaugment.py when its source is present (VITB_REFERENCE_ROOT, oracle/_ref or
   baseline/_ref), else torchvision's AutoAugment(CIFAR10) as a stand-in (the JSON says which).
3. End to end, TrainEngine at B = 1024, T = 65 (bench.py's model), alternated in one process:
   (a) steps on a resident fp32 batch (what bench.py times);
   (b) per step: a pinned uint8 host batch -> H2D -> GpuAugment(policy="cifar10") into the engine's input buffer -> step.
The card's name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import importlib.util
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

HBM_BYTES_PER_S = 7.7e12  # HGX B200 data sheet, one GPU


def gpu_context():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unavailable"


def cpu_context():
    model = "unknown"
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    except OSError:
        pass
    return {"cpu_model": model, "nproc": os.cpu_count()}


def kernel_times(vb, ops, iters=50):
    import torch
    from vit_cifar_b200.schedule import CIFAR10_MEAN, CIFAR10_STD
    rows = []
    for B in (1024, 8192):
        g = torch.Generator(device="cuda").manual_seed(B)
        img = torch.randint(0, 256, (B, 32, 32, 3), generator=g, device="cuda", dtype=torch.uint8)
        out = torch.empty((B, 3, 32, 32), device="cuda")
        for policy in (None, "cifar10", "svhn"):
            aug = vb.GpuAugment(32, 4, CIFAR10_MEAN, CIFAR10_STD, flip=policy != "svhn", seed=1, policy=policy)
            draws = aug.draw(B, "cuda")
            if policy is None:
                fn = lambda: ops.augment(img, *draws, aug.mean, aug.std, out, 4)  # noqa: E731
            else:
                fn = lambda: ops.augment_autoaugment(img, *draws, aug.op_ids, aug.mags, aug.mean, aug.std, out, 4)  # noqa: E731
            for _ in range(10):
                fn()
            torch.cuda.synchronize()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for _ in range(iters):
                fn()
            e.record()
            torch.cuda.synchronize()
            us = s.elapsed_time(e) * 1e3 / iters
            nbytes = B * 32 * 32 * 15
            rows.append({"policy": policy or "none", "B": B, "us_per_batch": round(us, 2), "bytes": nbytes,
                         "GB_per_s": round(nbytes / us / 1e3, 1), "share_of_hbm_peak": round(nbytes / (us * 1e-6) / HBM_BYTES_PER_S, 4)})
    return rows


def _reference_policy():
    cands = [os.environ.get("VITB_REFERENCE_ROOT"), os.path.join(ROOT, "oracle", "_ref"), os.path.join(ROOT, "baseline", "_ref")]
    for d in cands:
        if d and os.path.isfile(os.path.join(d, "autoaugment.py")):
            import numpy as np
            if not hasattr(np, "int"):
                np.int = int  # the reference's posterize range uses the alias numpy 1.24 removed
            spec = importlib.util.spec_from_file_location("ref_autoaugment", os.path.join(d, "autoaugment.py"))
            mod = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(mod)
            return mod.CIFAR10Policy(), "reference autoaugment.CIFAR10Policy"
    from torchvision.transforms import AutoAugment, AutoAugmentPolicy
    return AutoAugment(AutoAugmentPolicy.CIFAR10), "torchvision AutoAugment(CIFAR10) (stand-in: reference source not present)"


def cpu_pipeline(n):
    import numpy as np
    import torch
    import torchvision.transforms as tv
    from PIL import Image
    from vit_cifar_b200.schedule import CIFAR10_MEAN, CIFAR10_STD
    torch.set_num_threads(1)
    policy, which = _reference_policy()
    rng = np.random.default_rng(0)
    imgs = [Image.fromarray(rng.integers(0, 256, (32, 32, 3), dtype=np.uint8)) for _ in range(n)]
    res = {"policy_impl": which, "images": n}
    for name, tf in (("crop_flip_totensor_normalize", [tv.RandomCrop(32, padding=4), tv.RandomHorizontalFlip(), tv.ToTensor(), tv.Normalize(CIFAR10_MEAN, CIFAR10_STD)]),
                     ("with_autoaugment", [tv.RandomCrop(32, padding=4), tv.RandomHorizontalFlip(), policy, tv.ToTensor(), tv.Normalize(CIFAR10_MEAN, CIFAR10_STD)])):
        t = tv.Compose(tf)
        for im in imgs[:50]:
            t(im)
        t0 = time.perf_counter()
        for im in imgs:
            t(im)
        dt = time.perf_counter() - t0
        res[name] = {"us_per_image": round(dt / n * 1e6, 1), "images_per_s_one_core": round(n / dt, 1)}
    return res


def end_to_end(vb, rounds, steps):
    import torch
    sys.path.insert(0, ROOT)
    import bench
    vb.set_precision("bf16")
    torch.manual_seed(2045)
    M = bench.MODEL
    B = 1024
    model = vb.ViT(3, M["num_classes"], img_size=32, patch=M["patch"], num_layers=M["num_layers"], hidden=M["hidden"], mlp_hidden=M["mlp_hidden"],
                   head=M["head"]).cuda()
    eng = vb.TrainEngine(model, B, smoothing=bench.SMOOTHING, **bench.ADAM)
    g = torch.Generator().manual_seed(1)
    eng.load_batch(torch.randn(B, 3, 32, 32, generator=g).pin_memory(), torch.randint(0, 10, (B,), generator=g).pin_memory())
    host_u8 = [torch.randint(0, 256, (B, 32, 32, 3), generator=g, dtype=torch.uint8).pin_memory() for _ in range(4)]
    dev_u8 = torch.empty((B, 32, 32, 3), dtype=torch.uint8, device="cuda")
    aug = vb.GpuAugment(32, 4, policy="cifar10")

    def resident(i):
        eng.step()

    def augmented(i):
        dev_u8.copy_(host_u8[i % 4], non_blocking=True)
        aug(dev_u8, out=eng.img)
        eng.step()

    def timed(fn):
        for i in range(5):
            fn(i)
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for i in range(steps):
            fn(i)
        e.record()
        torch.cuda.synchronize()
        return s.elapsed_time(e) / steps

    a, b = [], []
    for _ in range(rounds):
        a.append(timed(resident))
        b.append(timed(augmented))
    med = lambda v: sorted(v)[len(v) // 2]  # noqa: E731
    return {"B": B, "T": 65, "rounds": rounds, "steps_per_round": steps,
            "a_resident_fp32": {"ms_per_step": [round(x, 4) for x in a], "img_per_s_median": round(B / med(a) * 1e3, 1)},
            "b_uint8_h2d_gpuaugment_cifar10": {"ms_per_step": [round(x, 4) for x in b], "img_per_s_median": round(B / med(b) * 1e3, 1)},
            "b_over_a": round(med(a) / med(b), 4)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--cpu-images", type=int, default=2000)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=40)
    args = ap.parse_args()
    import vit_cifar_b200 as vb
    from vit_cifar_b200 import ops
    ops.require_device()
    res = {"gpu": gpu_context(), **cpu_context()}
    res["kernel"] = kernel_times(vb, ops)
    res["cpu_pipeline"] = cpu_pipeline(args.cpu_images)
    per_core = res["cpu_pipeline"]["with_autoaugment"]["images_per_s_one_core"]
    res["end_to_end"] = end_to_end(vb, args.rounds, args.steps)
    step_rate = res["end_to_end"]["a_resident_fp32"]["img_per_s_median"]
    res["host_cores_to_feed_one_gpu"] = round(step_rate / per_core, 1)
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
