"""Training speed at widths of 64 mod 128, and the partial-tile GEMMs next to the same GEMM at the next multiple of 128.

    python tools/width_bench.py [--out profiles/r6_width_bench.json] [--steps 40]

Reads the card's name, power limit and maximum SM clock in the same process.  Models: ViT-Tiny (12 layers, hidden 192, 3 heads,
MLP 768) and the reference recipe at width 192 (7 layers, hidden 192, 6 heads, MLP 192), T = 65, B = 1024 and 128, graph-captured
TrainEngine steps timed one by one with CUDA events.  GEMMs: 66,560 rows (B = 1024 at T = 65), 50 launches per shape between
two events, inputs of 26-100 MB (the 126 MB L2 holds part of them: times are L2-warm where they fit).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import vit_cifar_b200 as vb  # noqa: E402

MODELS = {
    "vit_tiny": dict(num_layers=12, hidden=192, head=3, mlp_hidden=768),
    "ref_width192": dict(num_layers=7, hidden=192, head=6, mlp_hidden=192),
}
ADAM = dict(lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=5e-5)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def pct(xs, q):
    s = sorted(xs)
    return s[min(len(s) - 1, int(round(q * (len(s) - 1))))]


def train_times(cfg, B, steps, warmup):
    vb.set_precision("bf16")
    torch.manual_seed(0)
    m = vb.ViT(3, 10, img_size=32, patch=8, dropout=0.0, **cfg).cuda()
    eng = vb.TrainEngine(m, B, smoothing=0.1, use_graph=True, **ADAM)
    g = torch.Generator().manual_seed(1)
    x = torch.randn(B, 3, 32, 32, generator=g).cuda()
    y = torch.randint(0, 10, (B,), generator=g).cuda()
    eng.step(x, y)
    for _ in range(warmup):
        eng.step()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    ev[0].record()
    for i in range(steps):
        eng.step()
        ev[i + 1].record()
    torch.cuda.synchronize()
    ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(steps)]
    p50 = pct(ms, 0.5)
    return {"B": B, "T": 65, "ms_p10": pct(ms, 0.1), "ms_p50": p50, "ms_p90": pct(ms, 0.9), "img_per_s_p50": B / p50 * 1e3}


def time_launches(fn, reps=50):
    for _ in range(5):
        fn()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) * 1e3 / reps


def gemm_times(M=66560):
    bf = torch.bfloat16
    rows = []
    for op, N, K in [("fwd", 192, 192), ("fwd", 192, 768), ("fwd", 576, 192), ("fwd", 768, 192),
                     ("dgrad", 192, 192), ("dgrad", 768, 192), ("dgrad", 192, 576),
                     ("wgrad", 192, 192), ("wgrad", 192, 768), ("wgrad", 768, 192), ("wgrad", 576, 192)]:
        pair = []
        up = lambda v: -(-v // 128) * 128  # noqa: E731
        nxt = {"fwd": (up(N), K), "dgrad": (N, up(K)), "wgrad": (up(N), up(K))}[op]
        for n_, k_ in ((N, K), nxt):
            a = torch.randn(M, k_, device="cuda").to(bf)
            if op == "fwd":
                w = torch.randn(n_, k_, device="cuda").to(bf)
                b = torch.randn(n_, device="cuda")
                c = torch.empty(M, n_, dtype=bf, device="cuda")
                fn = lambda: vb.ops.gemm_fwd(a, w, b, None, c, None, M, n_, k_)  # noqa: E731
                flops = 2.0 * M * n_ * k_
            elif op == "dgrad":  # dX[M, K] = dY[M, N] W[N, K]: output width K
                dy = torch.randn(M, n_, device="cuda").to(bf)
                w = torch.randn(n_, k_, device="cuda").to(bf)
                dx = torch.empty(M, k_, dtype=bf, device="cuda")
                fn = lambda: vb.ops.gemm_dgrad(dy, w, None, dx, M, n_, k_)  # noqa: E731
                flops = 2.0 * M * n_ * k_
            else:
                dy = torch.randn(M, n_, device="cuda").to(bf)
                dw = torch.empty(n_, k_, device="cuda")
                db = torch.empty(n_, device="cuda")
                fn = lambda: vb.ops.gemm_wgrad(dy, a, dw, db, M, n_, k_)  # noqa: E731
                flops = 2.0 * M * n_ * k_
            us = time_launches(fn)
            pair.append({"N": n_, "K": k_, "us": us, "tflops": flops / us * 1e-6})
            del fn
        rows.append({"op": op, "M": M, "shape": pair[0], "next_multiple_of_128": pair[1]})
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=10)
    args = ap.parse_args()
    vb.ops.require_device()
    res = {"gpu": gpu_info(), "train": {}, "gemm_us": None}
    for name, cfg in MODELS.items():
        res["train"][name] = [dict(cfg, **train_times(cfg, B, args.steps, args.warmup)) for B in (1024, 128)]
        print(json.dumps({name: res["train"][name]}), flush=True)
    res["gemm_us"] = gemm_times()
    for r in res["gemm_us"]:
        print(json.dumps(r), flush=True)
    print(json.dumps({"gpu": res["gpu"]}), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
