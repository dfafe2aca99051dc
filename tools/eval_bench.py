"""Cost of the validation pass (network.py:388-395) on the module path and through EvalEngine.

    python tools/eval_bench.py [--out FILE.json] [--rounds 5] [--images 10000]

1. One pass over 10,000 seeded synthetic test images for the headline model (7 layers, 384 wide, 12 heads, T = 65, C = 10) and
   t17c100 (T = 17, C = 100), bf16.  Four variants, each timed as the wall time of a full pass that ends with its result on the
   host, after one warm-up pass, repetitions alternated in one process:
   (a) schedule.evaluate at batch 256 from device-resident fp32 batches (the module path);
   (b) EvalEngine at batch 256, the same batches;
   (c) EvalEngine at batch 2,500 and 10,000;
   (d) EvalEngine at batch 256 from pinned uint8 host batches (H2D and ToTensor + Normalize on the device included).
   Reported: img/s and ms per pass (median, min, max), library launches per batch (ops.launch_count(); torch's own argmax / eq /
   sum kernels of (a) are not counted) and the engine's activation_bytes().
2. An epoch: 50,000 device-resident training images through TrainEngine at B = 1,024 (graph), then one validation pass with (a)
   and with (b); the share of the epoch spent in validation.
The card's name, power limit and maximum SM clock are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CIFAR10_MEAN, CIFAR10_STD = (0.4914, 0.4822, 0.4465), (0.2470, 0.2435, 0.2616)
MODELS = {"headline": dict(num_classes=10, patch=8), "t17c100": dict(num_classes=100, patch=4)}


def gpu_context():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unavailable"


def make_model(vb, num_classes, patch):
    import torch
    torch.manual_seed(0)
    return vb.ViT(3, num_classes, img_size=32, patch=patch, num_layers=7, hidden=384, mlp_hidden=384, head=12).cuda()


def timed(fn):
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = fn()  # ends with the result on the host
    return (time.perf_counter() - t0) * 1e3, res


def summary(ms, n):
    med = statistics.median(ms)
    return {"ms_per_pass_median": round(med, 3), "ms_min": round(min(ms), 3), "ms_max": round(max(ms), 3),
            "img_per_s_median": round(n / (med / 1e3), 1)}


def validation(vb, name, cfg, n_img, rounds):
    import torch
    from vit_cifar_b200 import ops
    C = cfg["num_classes"]
    model = make_model(vb, C, cfg["patch"])
    crit = vb.LabelSmoothingCrossEntropyLoss(C, smoothing=0.1)
    g = torch.Generator().manual_seed(1)
    u8 = torch.randint(0, 256, (n_img, 32, 32, 3), dtype=torch.uint8, generator=g)
    y = torch.randint(0, C, (n_img,), generator=g)
    x = torch.empty((n_img, 3, 32, 32), dtype=torch.float32, device="cuda")
    ops.augment(u8.cuda(), None, None, None, CIFAR10_MEAN, CIFAR10_STD, x, 0)  # the same images as fp32 test-transform output
    yd = y.cuda()
    dev = lambda bs: [(x[i:i + bs], yd[i:i + bs]) for i in range(0, n_img, bs)]  # noqa: E731
    host_u8 = [(u8[i:i + 256].pin_memory(), y[i:i + 256].pin_memory()) for i in range(0, n_img, 256)]
    variants = {"a_evaluate_b256": (None, dev(256)), "b_engine_b256": (vb.EvalEngine(model, 256), dev(256)),
                "c_engine_b2500": (vb.EvalEngine(model, 2500), dev(2500)), "c_engine_b10000": (vb.EvalEngine(model, 10000), dev(10000)),
                "d_engine_b256_pinned_uint8": (vb.EvalEngine(model, 256, mean=CIFAR10_MEAN, std=CIFAR10_STD), host_u8)}
    run = {k: ((lambda b=b: vb.evaluate(model, crit, b)) if ev is None else (lambda ev=ev, b=b: ev.run(b))) for k, (ev, b) in variants.items()}
    out = {}
    for k, fn in run.items():  # warm-up (the engines capture their graph here); launches of (a) per batch
        n0 = ops.launch_count()
        res = fn()
        ev, b = variants[k]
        out[k] = {"result": res, "batches_per_pass": len(b),
                  "launches_per_batch": round((ops.launch_count() - n0) / len(b), 2) if ev is None else ev.launches_per_batch,
                  "graph_replays_per_batch": 0 if ev is None else 1,
                  "activation_bytes": None if ev is None else ev.activation_bytes()}
    ms = {k: [] for k in run}
    for _ in range(rounds):
        for k, fn in run.items():
            t, res = timed(fn)
            ms[k].append(t)
            assert res == out[k]["result"], (k, res, out[k]["result"])  # every repetition computes the same metrics
    for k in run:
        out[k].update(summary(ms[k], n_img))
    a = out["a_evaluate_b256"]
    for k in run:
        out[k]["speedup_vs_a"] = round(a["ms_per_pass_median"] / out[k]["ms_per_pass_median"], 2)
    out["model"] = dict(name=name, layers=7, hidden=384, heads=12, tokens=cfg["patch"] ** 2 + 1, classes=C, images=n_img, precision="bf16")
    del model
    return out


def epoch(vb, rounds, n_val):
    import torch
    model = make_model(vb, 10, 8)
    crit = vb.LabelSmoothingCrossEntropyLoss(10, smoothing=0.1)
    g = torch.Generator().manual_seed(2)
    n_train, B = 50000, 1024
    xt = torch.randn(n_train, 3, 32, 32, generator=g).cuda()
    yt = torch.randint(0, 10, (n_train,), generator=g).cuda()
    xv = torch.randn(n_val, 3, 32, 32, generator=g).cuda()
    yv = torch.randint(0, 10, (n_val,), generator=g).cuda()
    val = [(xv[i:i + 256], yv[i:i + 256]) for i in range(0, n_val, 256)]
    eng = vb.TrainEngine(model, B, smoothing=0.1)
    ev = vb.EvalEngine(model, 256)

    def train():
        loss = None
        for i in range(0, n_train, B):
            loss = eng.step(xt[i:i + B], yt[i:i + B])
        return float(loss)

    fns = {"train_epoch": train, "val_a_evaluate": lambda: vb.evaluate(model, crit, val), "val_b_engine": lambda: ev.run(val)}
    for fn in fns.values():
        fn()
    ms = {k: [] for k in fns}
    for _ in range(rounds):
        for k, fn in fns.items():
            ms[k].append(timed(fn)[0])
    med = {k: statistics.median(v) for k, v in ms.items()}
    out = {"train_images": n_train, "train_batch": B, "val_images": n_val, "val_batch": 256,
           **{f"{k}_ms_median": round(v, 3) for k, v in med.items()}}
    for tag in ("a_evaluate", "b_engine"):
        v = med[f"val_{tag}"]
        out[f"epoch_ms_with_{tag}"] = round(med["train_epoch"] + v, 3)
        out[f"validation_share_with_{tag}"] = round(v / (med["train_epoch"] + v), 4)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--images", type=int, default=10000)
    args = ap.parse_args()
    import vit_cifar_b200 as vb
    vb.ops.require_device()
    vb.set_precision("bf16")
    res = {"gpu": gpu_context(), "timing": "wall time of a full pass ending with its metrics on the host; median over alternated rounds"}
    res["validation"] = {name: validation(vb, name, cfg, args.images, args.rounds) for name, cfg in MODELS.items()}
    res["epoch"] = epoch(vb, max(2, args.rounds // 2), args.images)
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
