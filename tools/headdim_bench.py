"""Attention kernel times at every head dimension, and training speed at 3 / 4 / 6 / 12 heads of width 384.

    python tools/headdim_bench.py [--out profiles/r7_headdim_bench.json] [--reps 200] [--steps 40]

Reads the card's name, power limit and maximum SM clock in the same process.

Kernels: bf16 vitb_attn_fwd / vitb_attn_bwd at B = 1024, T = 17 and 65, H = 384 (12 / 6 / 4 / 3 heads: d = 32 / 64 / 96 / 128)
and H = 768 (24 / 12 / 8 / 6 heads).  Each is warmed up, then `--reps` launches run back to back between two CUDA events.  Bytes
are what the kernels must move (SURVEY §8(d)): forward 4E + LSE, backward 8E, with E = B·T·H·2.  At T = 65 the qkv tensor alone
is 153 MB (H = 384) or 307 MB (H = 768), larger than the 126 MB L2; at T = 17 the working set is 40-80 MB and stays partly
L2-resident across launches, so those rates are not HBM rates.

Steps: graph-captured TrainEngine steps of a 7-layer ViT, width 384, MLP 384, T = 65, at B = 1024 and 128, timed one by one
with CUDA events.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import vit_cifar_b200 as vb  # noqa: E402

HBM_TBPS = 7.7  # HGX B200 data sheet, one GPU
ADAM = dict(lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=5e-5)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def pct(xs, q):
    s = sorted(xs)
    return s[min(len(s) - 1, int(round(q * (len(s) - 1))))]


def time_launches(fn, reps, warmup=20):
    for _ in range(warmup):
        fn()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) * 1e3 / reps


def attention_times(reps, B=1024):
    bf = torch.bfloat16
    rows = []
    for T in (17, 65):
        for H in (384, 768):
            g = torch.Generator(device="cuda").manual_seed(T + H)
            qkv = torch.randn(B, T, 3 * H, device="cuda", generator=g).to(bf)
            do = torch.randn(B, T, H, device="cuda", generator=g).to(bf)
            o = torch.empty(B, T, H, dtype=bf, device="cuda")
            dqkv = torch.empty_like(qkv)
            E = B * T * H * 2
            for d in (32, 64, 96, 128):
                heads = H // d
                scale = 1.0 / math.sqrt(H)
                lse = torch.empty(B, heads, T, device="cuda")
                fwd = lambda: vb.ops.attn_fwd(qkv, o, lse, None, B, T, heads, d, scale)  # noqa: E731
                bwd = lambda: vb.ops.attn_bwd(qkv, o, do, lse, dqkv, B, T, heads, d, scale)  # noqa: E731
                fwd_us = time_launches(fwd, reps)
                bwd_us = time_launches(bwd, reps)
                fb, bb = 4 * E + B * heads * T * 4, 8 * E
                row = {"B": B, "T": T, "H": H, "heads": heads, "d": d, "fwd_us": fwd_us, "bwd_us": bwd_us,
                       "fwd_bytes": fb, "bwd_bytes": bb,
                       "fwd_GBps": fb / fwd_us * 1e-3, "bwd_GBps": bb / bwd_us * 1e-3,
                       "fwd_frac_hbm": fb / fwd_us * 1e-6 / HBM_TBPS, "bwd_frac_hbm": bb / bwd_us * 1e-6 / HBM_TBPS}
                rows.append(row)
                print(json.dumps(row), flush=True)
            ref = next(r for r in rows if r["T"] == T and r["H"] == H and r["d"] == 64)
            for r in rows:
                if r["T"] == T and r["H"] == H:
                    r["fwd_bwd_over_d64"] = (r["fwd_us"] + r["bwd_us"]) / (ref["fwd_us"] + ref["bwd_us"])
            del qkv, do, o, dqkv
    return rows


def train_times(heads, B, steps, warmup):
    vb.set_precision("bf16")
    torch.manual_seed(0)
    cfg = dict(num_layers=7, hidden=384, mlp_hidden=384, head=heads)
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
    return dict(cfg, d=384 // heads, B=B, T=65, ms_p10=pct(ms, 0.1), ms_p50=p50, ms_p90=pct(ms, 0.9), img_per_s_p50=B / p50 * 1e3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=10)
    args = ap.parse_args()
    vb.ops.require_device()
    res = {"gpu": gpu_info(), "attention": attention_times(args.reps), "train": []}
    for B in (1024, 128):
        for heads in (3, 4, 6, 12):
            r = train_times(heads, B, args.steps, args.warmup)
            res["train"].append(r)
            print(json.dumps(r), flush=True)
    print(json.dumps({"gpu": res["gpu"]}), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
