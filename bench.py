#!/usr/bin/env python
"""bench.py — train images/s (forward + LS-CE + backward + Adam) of the ViT-CIFAR hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

Workload (BASELINE.json configs[1]/[2]): ViT 7 layers / hidden 384 / 12 heads / MLP 384, `patch=8` patches per side
(T = 65 tokens, patch vector K = 48), 10 classes, label smoothing 0.1, Adam(lr 1e-3, wd 5e-5), bf16 storage with
fp32 accumulation, per-GPU batch 1024 (weak scaling: global batch = 1024 * N; 8192 at N = 8), synthetic
32x32x3 data.  One "step" = one optimisation step over one batch.

Prints ONE JSON line (rank 0).  `value` = steady-state img/s with the batch resident in HBM over `--steps` timed steps;
`e2e` = the same through the public API from pinned HOST buffers (H2D of every batch and D2H of every loss inside the timed
region); `step_ms` = per-step times of `--steps` more steps.  The side measurements after them have fixed sizes whatever
`--steps` says: the per-kernel probe (3 eager steps), `cpu_baseline` (3 steps of at most 128 images) and `gpu_eager_baseline`
(10 steps).  `--dump-outputs DIR` also writes what the last step of the first timed loop returned to its caller (loss, logits,
updated parameters, gradients) as DIR/<name>.npy in float32; the inputs depend on the arguments only, so two builds can be
compared output for output.
`cpu_baseline`, `gpu_eager_baseline`, `--impl reference` and `--impl eager` time the reference's own modules where their
source is available (VITB_REFERENCE_ROOT, oracle/_ref or baseline/_ref, see oracle/ref_shim.py; kind "reference"), else
the oracle's restatement of them (oracle/, kind "port").  `--impl reference` runs on the host cores over a bounded sample;
`--impl eager` times the same PyTorch modules on the B200 (eager ATen / cuBLAS: fp32
with matmul precision "medium" as main.py:173, bf16 and fp16 autocast as main.py:58, and torch.compile) — the
kernel-level bar the hand-written kernels have to beat, since the reference ships no GPU code of its own.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MODEL = dict(num_classes=10, img_size=32, patch=8, num_layers=7, hidden=384, mlp_hidden=384, head=12)
PER_GPU_BATCH = 1024
# --workload: the headline configuration (BASELINE.json configs[1], default — the only one the contract line is quoted on) and the
# other shapes SURVEY.md §8(d) lists, for DESIGN.md's tables.  `patch` is the number of patches per side (vit.py:37).
WORKLOADS = {
    "headline": (MODEL, PER_GPU_BATCH),
    "t17c100": (dict(MODEL, patch=4, num_classes=100), PER_GPU_BATCH),                                      # configs[3] as written (T = 17)
    "t65c100": (dict(MODEL, patch=8, num_classes=100), PER_GPU_BATCH),                                      # configs[3] at 65 tokens
    "scaled17": (dict(MODEL, patch=4, num_layers=12, hidden=768, mlp_hidden=3072, head=12), 512),           # configs[4] as written
    "scaled65": (dict(MODEL, patch=8, num_layers=12, hidden=768, mlp_hidden=3072, head=12), 512),           # configs[4] at 65 tokens
}
ADAM = dict(lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=5e-5)
SMOOTHING = 0.1
METRIC = "train images/s (fwd+bwd+Adam)"
UNIT = "img/s"


def train_flops_per_image(T=65, K=48, H=384, M=384, L=7, C=10):
    fwd = 2 * (T - 1) * K * H + L * (2 * T * H * (4 * H + 2 * M) + 4 * T * T * H) + 2 * H * C  # SURVEY.md §8(d)
    return 3 * fwd


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d.get("bf16_tflops_sustained", d["bf16_tflops"]), src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback")


# ---------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------
# CPU baseline / reference arm: the oracle port (same arithmetic as the reference, torch fp32 on host cores)
# ---------------------------------------------------------------------------------------------
def torch_reference_model():
    """(model, criterion, kind): the reference's own vit.ViT + LabelSmoothingCrossEntropyLoss when a copy of the reference is
    reachable (VITB_REFERENCE_ROOT, oracle/_ref or baseline/_ref, see oracle/ref_shim.py; kind "reference"), else the oracle's
    restatement with the same state_dict names (kind "port").  Same construction arguments as utils.get_model (utils.py:71-83)."""
    import torch
    import oracle
    from oracle import ref_shim
    torch.manual_seed(2045)  # main.py:150
    if ref_shim.reference_available():
        ref_vit, _, ref_crit = ref_shim.import_reference()
        model = ref_vit.ViT(3, MODEL["num_classes"], img_size=MODEL["img_size"], patch=MODEL["patch"], dropout=0.0, mlp_hidden=MODEL["mlp_hidden"],
                            num_layers=MODEL["num_layers"], hidden=MODEL["hidden"], head=MODEL["head"], is_cls_token=True)
        return model, ref_crit.LabelSmoothingCrossEntropyLoss(MODEL["num_classes"], smoothing=SMOOTHING), "reference"
    cfg = oracle.ViTConfig(**MODEL)
    model = oracle.OracleViT(cfg, seed=0)
    return model, (lambda out, y: oracle.ls_ce_loss(out, y, cfg.num_classes, SMOOTHING)), "port"


def cpu_port_images_per_s(batch: int, steps: int, warmup: int):
    import torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    model, crit, kind = torch_reference_model()
    opt = torch.optim.Adam(model.parameters(), **ADAM)
    g = torch.Generator().manual_seed(1234)
    x = torch.randn(batch, 3, 32, 32, generator=g)
    y = torch.randint(0, MODEL["num_classes"], (batch,), generator=g)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        opt.zero_grad(set_to_none=True)
        loss = crit(model(x), y)
        loss.backward()
        opt.step()
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    total = sum(times)
    return batch * len(times) / total, cores, 1e3 * total / len(times), kind


def pctl(xs, q):
    xs = sorted(xs)
    if not xs:
        return None
    k = (len(xs) - 1) * q
    lo, hi = int(k), min(int(k) + 1, len(xs) - 1)
    return xs[lo] + (xs[hi] - xs[lo]) * (k - lo)


def eager_gpu_images_per_s(mode: str, batch: int, steps: int, warmup: int, compile_: bool = False):
    """The PyTorch modules of the reference path on cuda:0, timed per step with CUDA events.  mode: "fp32-medium" (main.py:173),
    "bf16-autocast", "fp16-autocast" (main.py:58 "16-mixed": autocast + GradScaler)."""
    import torch
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.set_float32_matmul_precision("medium")  # main.py:139-144, 173
    model, crit, kind = torch_reference_model()
    model = model.to(dev)
    fwd = torch.compile(model) if compile_ else model
    opt = torch.optim.Adam(model.parameters(), **ADAM)
    g = torch.Generator().manual_seed(1234)
    x = torch.randn(batch, 3, 32, 32, generator=g).to(dev)
    y = torch.randint(0, MODEL["num_classes"], (batch,), generator=g).to(dev)
    scaler = torch.amp.GradScaler("cuda") if mode == "fp16-autocast" else None
    ac = {"fp32-medium": None, "bf16-autocast": torch.bfloat16, "fp16-autocast": torch.float16}[mode]
    ev = []
    for i in range(warmup + steps):
        s = torch.cuda.Event(enable_timing=True); e = torch.cuda.Event(enable_timing=True)
        s.record()
        opt.zero_grad(set_to_none=True)
        if ac is None:
            loss = crit(fwd(x), y)
        else:
            with torch.autocast("cuda", dtype=ac):
                loss = crit(fwd(x), y)
        if scaler is not None:
            scaler.scale(loss).backward()
            scaler.step(opt)
            scaler.update()
        else:
            loss.backward()
            opt.step()
        e.record()
        if i >= warmup:
            ev.append((s, e))
    torch.cuda.synchronize()
    ms = [a.elapsed_time(b) for a, b in ev]
    tot = sum(ms)
    return {"mode": mode + ("+compile" if compile_ else ""), "img_s": round(batch * len(ms) / (tot * 1e-3), 1), "ms_per_step": round(tot / len(ms), 4),
            "p10_ms": round(pctl(ms, 0.1), 4), "p50_ms": round(pctl(ms, 0.5), 4), "p90_ms": round(pctl(ms, 0.9), 4), "batch": batch, "kind": kind,
            "final_loss": float(loss.detach())}


def run_eager(args):
    """Extra arm (not part of the driver contract): the reference path in PyTorch eager on ONE B200."""
    if int(os.environ.get("RANK", "0")) != 0:
        return 0
    res = []
    for mode, comp in (("fp32-medium", False), ("bf16-autocast", False), ("fp16-autocast", False), ("bf16-autocast", True)):
        try:
            res.append(eager_gpu_images_per_s(mode, args.batch, args.steps, max(3, args.warmup), comp))
        except Exception as ex:  # torch.compile needs a working inductor tool chain on the box
            res.append({"mode": mode + ("+compile" if comp else ""), "error": f"{type(ex).__name__}: {str(ex)[:200]}"})
    best = max((r for r in res if "img_s" in r), key=lambda r: r["img_s"])
    out = {"impl": "eager", "metric": METRIC, "value": best["img_s"], "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": max(3, args.warmup),
           "ms_per_step": best["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": best["mode"],
           "data": "synthetic", "config": {"workload": workload_name(1, args.batch), "what": "PyTorch eager (ATen / cuBLAS) on the same B200"},
           "modes": res}
    print(json.dumps(out), flush=True)
    return 0


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    batch = min(128, args.batch)  # bounded sample of the step (the reference's own default batch, main.py:43): the CPU path is ~1e3x slower
    v, cores, ms, kind = cpu_port_images_per_s(batch, max(1, args.steps), max(1, min(args.warmup, 2)))
    what = "the reference's own vit.ViT / criterion" if kind == "reference" else "oracle port of the reference"
    out = {
        "impl": "reference", "metric": METRIC, "value": round(v, 2), "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(ms, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": model_name(), "per_step_batch": batch,
                   "sample": f"every step is a {batch}-image sample of the {args.batch}-image per-GPU batch, fp32 on {cores} host threads (one CPU process)"},
        "cpu_baseline": {"value": round(v, 2), "unit": UNIT, "cores": cores, "kind": kind,
                         "sample": f"{args.steps} steps of batch {batch} ({what}, torch fp32, {cores} threads)"},
        "e2e": {"value": round(v, 2), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(out), flush=True)
    return 0


def model_name():
    T = MODEL["patch"] ** 2 + 1
    K = 3 * (MODEL["img_size"] // MODEL["patch"]) ** 2
    return (f"ViT-CIFAR {MODEL['num_layers']}L/{MODEL['hidden']}h/{MODEL['head']}heads/MLP{MODEL['mlp_hidden']} patch={MODEL['patch']} "
            f"(T={T},K={K}) C={MODEL['num_classes']}, LS 0.1, Adam")


def workload_name(n, batch=None):
    b = PER_GPU_BATCH if batch is None else batch
    return f"{model_name()}, per-GPU batch {b} (global {b * n}), bf16"


# ---------------------------------------------------------------------------------------------
# per-kernel probe: CUDA-event time of every C-ABI call of an eager step, grouped by (op, shape)
# ---------------------------------------------------------------------------------------------
def probe_kernels(eng, steps=3):
    import torch
    from vit_cifar_b200 import ops
    names = ["patch_embed_fwd", "patch_embed_bwd", "layernorm_fwd", "layernorm_bwd", "layernorm_bwd_fused", "gemm_fwd", "gemm_dgrad", "gemm_wgrad",
             "attn_fwd", "attn_bwd", "gelu_bwd_colsum", "colsum", "pool_fwd", "pool_bwd", "ls_ce", "adam"]
    rec = []
    orig = {}

    def wrap(name, fn):
        def inner(*a, **k):
            s = torch.cuda.Event(enable_timing=True); e = torch.cuda.Event(enable_timing=True)
            s.record()
            r = fn(*a, **k)
            e.record()
            shape = tuple(x for x in a if isinstance(x, int))
            flags = tuple(sorted((kk, vv) for kk, vv in k.items() if isinstance(vv, bool) and vv))
            extra = ("res",) if name == "gemm_fwd" and a[3] is not None else ()
            extra += ("z",) if name == "gemm_dgrad" and a[2] is not None else ()
            extra += ("colsum",) if name == "layernorm_bwd" and a[11] is not None else ()
            rec.append((name, shape, flags + extra, s, e))
            return r
        return inner

    for n in names:
        orig[n] = getattr(ops, n)
        setattr(ops, n, wrap(n, orig[n]))
    try:
        saved_graph, eng.use_graph = eng.use_graph, False
        saved_side, eng._side = eng._side, None  # per-kernel times: everything on one stream, one kernel at a time
        for _ in range(steps):
            # Park the GPU (~25 ms spin) while the host enqueues the whole eager step: every kernel then starts the moment
            # its predecessor ends, so an event pair brackets device time only, not host launch latency.
            torch.cuda._sleep(50_000_000)
            eng.step()
            torch.cuda.synchronize()
        eng.use_graph = saved_graph
        eng._side = saved_side
    finally:
        for n in names:
            setattr(ops, n, orig[n])
    agg = {}
    for name, shape, flags, s, e in rec:
        key = (name, shape, flags)
        d = agg.setdefault(key, [0.0, 0])
        d[0] += s.elapsed_time(e)
        d[1] += 1
    table = []
    for (name, shape, flags), (ms, cnt) in agg.items():
        table.append({"op": name, "shape": list(shape), "flags": [str(f) for f in flags], "calls_per_step": cnt // steps,
                      "ms_per_call": ms / cnt, "ms_per_step": ms / steps})
    table.sort(key=lambda r: -r["ms_per_step"])
    return table


def ncu_traffic(kernel_name):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` capture of this round's final
    build (profiles/ncu_traffic.json, rows in profiles/r2_ncu_full_summary.csv), or None."""
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "ncu_traffic.json")
    try:
        with open(path) as f:
            return json.load(f).get("dram_bytes_per_launch", {}).get(kernel_name)
    except (OSError, ValueError):
        return None


def kernel_roofline(row, pk, B, T, H):
    r = _kernel_roofline(row, pk, B, T, H)
    if r is not None:
        r["traffic"] = ncu_traffic(r["kernel"])
    return r


def _kernel_roofline(row, pk, B, T, H):
    """Algorithmic FLOPs / bytes of one call (DESIGN.md §kernels) against the measured peaks."""
    op, sh = row["op"], row["shape"]
    sec = row["ms_per_call"] * 1e-3
    E = 2  # bytes per bf16 activation element
    if op in ("gemm_fwd", "gemm_dgrad", "gemm_wgrad"):
        M, N, K = sh[:3]
        fl = 2.0 * M * N * K
        r = {"bound": "tensor", "achieved": fl / sec / 1e12, "peak": pk["tf_sust"], "unit": "TFLOP/s", "frac": fl / sec / 1e12 / pk["tf_sust"],
             "traffic": None, "kernel": f"{op} M={M} N={N} K={K} {' '.join(row['flags'])}".strip(), "peak_kind": f"{pk['src']} sustained bf16"}
        if op == "gemm_wgrad":
            r["note"] = "split-K GEMM launch only: its fixed-order second pass runs in the step's deferred flush (vitb_defer_flush)"
        return r
    rows = B * T
    by = {
        "layernorm_fwd": 2 * rows * H * E, "layernorm_bwd": 4 * rows * H * E,
        "layernorm_bwd_fused": 6 * rows * H * E,  # + z2 read and dz2 written (the next block's GELU backward)
        "attn_fwd": 4 * rows * H * E, "attn_bwd": 8 * rows * H * E,
        "gelu_bwd_colsum": 3 * rows * H * E, "colsum": (sh[0] * sh[1] * E) if len(sh) >= 2 else 0,
        "patch_embed_fwd": B * 12288 + rows * H * E, "patch_embed_bwd": B * 12288 + rows * H * E,
    }.get(op)
    if op == "adam":
        by = 30 * eng_numel  # 28 B/param fp32 state + 2 B bf16 shadow
    if not by:
        return None
    return {"bound": "hbm", "achieved": by / sec / 1e9, "peak": pk["hbm"], "unit": "GB/s", "frac": by / sec / 1e9 / pk["hbm"], "traffic": None,
            "kernel": f"{op} {sh}", "peak_kind": f"{pk['src']} copy bandwidth"}


eng_numel = 0


# ---------------------------------------------------------------------------------------------
# data-parallel numerics (Lightning DDP semantics, main.py:220-231: every replica applies the MEAN of the ranks' gradients)
# ---------------------------------------------------------------------------------------------
def dp_verify(eng, vb, dist, pg, dev, rank, world):
    """(1) the replicas of the benchmarked engine are bit-identical after the timed loops; (2) a small fp32 model: one step of
    the data-parallel engine on rank-specific batches equals the oracle's Adam step on the gradient of the GLOBAL batch (= the
    mean of the ranks' gradients); (3) the benchmark model: two steps of the fused peer-memory path against NCCL all-reduce +
    the Adam kernel from the same weights and batches.  Returns a dict for `config`; `ok` False makes bench.py exit non-zero."""
    import torch
    res = {}
    # (1) replica identity: compare every rank's parameters with rank 0's
    mine = eng.P[:eng.n].clone()
    ref = mine.clone()
    dist.broadcast(ref, src=0, group=pg)
    same = torch.tensor([1 if torch.equal(mine, ref) else 0], device=dev)
    dist.all_reduce(same, op=dist.ReduceOp.MIN, group=pg)
    res["replicas_bit_identical"] = bool(same.item())
    # (2) oracle check on a small model (fp32 check mode, rank-specific batches)
    import oracle
    cfg = oracle.ViTConfig(num_classes=10, img_size=32, patch=8, num_layers=2, hidden=128, mlp_hidden=128, head=4)
    Bs = 4
    vb.set_precision("fp32")
    m = vb.ViT(3, 10, img_size=32, patch=8, num_layers=2, hidden=128, mlp_hidden=128, head=4)
    m.load_state_dict(oracle.init_params(cfg, 0))
    m = m.to(dev)
    e2 = vb.TrainEngine(m, Bs, smoothing=SMOOTHING, process_group=pg, use_graph=False, **ADAM)
    xs, ys = oracle.hash_inputs(cfg, Bs * world, seed=3)
    e2.step(xs[rank * Bs:(rank + 1) * Bs].to(dev), ys[rank * Bs:(rank + 1) * Bs].to(dev))
    torch.cuda.synchronize()
    err = 0.0
    if rank == 0:
        params = oracle.init_params(cfg, 0)
        p0 = {k: v.clone() for k, v in params.items()}
        _, _, grads = oracle.train_step(params, xs, ys, cfg, SMOOTHING)  # mean over the global batch = mean of the rank means
        mo = {k: torch.zeros_like(v) for k, v in params.items()}
        vo = {k: torch.zeros_like(v) for k, v in params.items()}
        oracle.adam_step(params, grads, mo, vo, 1, ADAM["lr"], ADAM["betas"], ADAM["eps"], ADAM["weight_decay"])
        sd = m.state_dict()
        num = den = 0.0
        for k in params:
            if "Wk.bias" in k:  # analytically zero gradient: Adam turns its rounding noise into +-lr updates
                continue
            num += float(((sd[k].cpu().double() - p0[k].double()) - (params[k].double() - p0[k].double())).pow(2).sum())
            den += float((params[k].double() - p0[k].double()).pow(2).sum())
        err = (num / max(den, 1e-300)) ** 0.5
    t = torch.tensor([err], device=dev, dtype=torch.float64)
    dist.broadcast(t, src=0, group=pg)
    res["adam_update_vs_oracle_global_batch_rel"] = float(t.item())
    vb.set_precision("bf16")
    # (3) fused peer-memory step vs NCCL all-reduce + Adam kernel on the benchmark model
    def two_steps(mode):
        prev = os.environ.get("VITB_DP_MODE")
        os.environ["VITB_DP_MODE"] = mode
        try:
            torch.manual_seed(2045)
            mm = vb.ViT(3, MODEL["num_classes"], img_size=32, patch=MODEL["patch"], dropout=0.0, num_layers=MODEL["num_layers"],
                        hidden=MODEL["hidden"], mlp_hidden=MODEL["mlp_hidden"], head=MODEL["head"]).to(dev)
            ee = vb.TrainEngine(mm, 64, smoothing=SMOOTHING, process_group=pg, use_graph=False, **ADAM)
            for st in range(2):
                g = torch.Generator().manual_seed(777 + 10 * st + rank)
                ee.step(torch.randn(64, 3, 32, 32, generator=g).to(dev), torch.randint(0, MODEL["num_classes"], (64,), generator=g).to(dev))
            torch.cuda.synchronize()
            return ee.P[:ee.n].clone(), ee._dp_mode
        finally:
            if prev is None:
                os.environ.pop("VITB_DP_MODE", None)
            else:
                os.environ["VITB_DP_MODE"] = prev
    p_nccl, _ = two_steps("single")
    p_fused, mode_used = two_steps("fused")
    d = ((p_fused - p_nccl).double().norm() / p_nccl.double().norm()).item()
    t = torch.tensor([d], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX, group=pg)
    res["fused_vs_nccl_params_rel_after_2_steps"] = float(t.item())
    res["fused_mode_active"] = mode_used == "fused"
    res["ok"] = bool(res["replicas_bit_identical"] and res["adam_update_vs_oracle_global_batch_rel"] < 1e-3
                     and res["fused_vs_nccl_params_rel_after_2_steps"] < 1e-3)
    return res


# ---------------------------------------------------------------------------------------------
# --dump-outputs: what one training step returns to its caller, for comparing two builds output for output
# ---------------------------------------------------------------------------------------------
DUMP_BYTES = 60 << 20  # all .npy files of one dump together stay below 64 MB, headers included


def step_outputs(eng):
    """Host float32 copies of what the engine's last step hands its caller: the loss, the logits, the updated parameters and the
    gradients they were updated with (both flattened and concatenated in state_dict order)."""
    import torch
    with torch.no_grad():
        params = torch.cat([t.detach().float().flatten() for t in eng.model.state_dict().values()])
        grads = torch.cat([g.float().flatten() for g in eng.grads().values()])
        return {"loss": eng.loss.float().cpu().numpy(), "logits": eng.logits.float().cpu().numpy(),
                "params": params.cpu().numpy(), "grads": grads.cpu().numpy()}


def dump_outputs(outdir, arrays, seed=0):
    """Writes every array as outdir/<name>.npy.  The smaller arrays are kept whole; an array that does not fit its share of
    DUMP_BYTES is replaced by its values at a fixed, seeded set of positions (sorted; the same on every run with the same shapes)."""
    import numpy as np
    os.makedirs(outdir, exist_ok=True)
    left = DUMP_BYTES // 4
    items = sorted(arrays.items(), key=lambda kv: kv[1].size)
    for i, (name, a) in enumerate(items):
        a = np.asarray(a, dtype=np.float32)
        share = left // (len(items) - i)
        if a.size > share:
            a = a.reshape(-1)[np.sort(np.random.default_rng(seed).choice(a.size, size=share, replace=False))]
        np.save(os.path.join(outdir, f"{name}.npy"), a)
        left -= a.size


# ---------------------------------------------------------------------------------------------
def run_ours(args):
    global eng_numel
    import torch
    import torch.distributed as dist
    import vit_cifar_b200 as vb

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit(f"--gpus {args.gpus} needs torchrun with {args.gpus} ranks (WORLD_SIZE=1 here)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    pg = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
        pg = dist.group.WORLD

    vb.set_precision("bf16")
    torch.manual_seed(2045)  # main.py:150
    model = vb.ViT(3, MODEL["num_classes"], img_size=32, patch=MODEL["patch"], dropout=args.dropout, num_layers=MODEL["num_layers"],
                   hidden=MODEL["hidden"], mlp_hidden=MODEL["mlp_hidden"], head=MODEL["head"]).to(dev)
    B = args.batch
    eng = vb.TrainEngine(model, B, smoothing=SMOOTHING, process_group=pg, use_graph=not args.no_graph, **ADAM)
    eng_numel = eng.n

    g = torch.Generator().manual_seed(1234 + rank)
    nbuf = 4  # rotating pinned host batches (different data every step)
    host_x = [torch.randn(B, 3, 32, 32, generator=g).pin_memory() for _ in range(nbuf)]
    host_y = [torch.randint(0, MODEL["num_classes"], (B,), generator=g).pin_memory() for _ in range(nbuf)]
    loss_host = torch.zeros(args.steps + args.warmup + 8, dtype=torch.float32).pin_memory()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(step_fn, steps, warmup):
        for i in range(warmup):
            step_fn(i)
        barrier()
        s = torch.cuda.Event(enable_timing=True); e = torch.cuda.Event(enable_timing=True)
        s.record()
        for i in range(steps):
            step_fn(warmup + i)
        e.record()
        barrier()
        ms = s.elapsed_time(e)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms

    # ---- device-resident arm: the batch is already in HBM -------------------------------------
    eng.load_batch(host_x[0], host_y[0])
    W = max(3, args.warmup)
    sampler = ClockSampler(local)
    for i in range(2):  # eager warm-up + graph capture happen here, outside any timed region
        eng.step()
    barrier()
    if rank == 0:
        sampler.start()
    ms_dev = timed(lambda i: eng.step(), args.steps, W)
    outputs = step_outputs(eng) if args.dump_outputs and rank == 0 else None  # taken now: the arms below keep training
    # ---- end-to-end arm: pinned host -> device every step, loss read back every step ----------
    # Public API as a training loop uses it: step() on the batch prefetched during the previous step, then prefetch() of the
    # next pinned host batch (its PCIe transfer overlaps this step's kernels).  One H2D batch copy and one D2H loss read per step.
    eng.prefetch(host_x[0], host_y[0])
    def e2e_step(i):
        loss = eng.step()
        eng.prefetch(host_x[(i + 1) % nbuf], host_y[(i + 1) % nbuf])
        loss_host[i % loss_host.numel()].copy_(loss, non_blocking=True)
    ms_e2e = timed(e2e_step, args.steps, W)
    clocks = sampler.stop() if rank == 0 else None
    # ---- per-step distribution (SURVEY.md §8d: median + p10/p90): one event pair per step, outside the two timed regions
    evs = []
    for i in range(args.steps):
        s_, e_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s_.record(); eng.step(); e_.record()
        evs.append((s_, e_))
    torch.cuda.synchronize()
    per_step = [a.elapsed_time(b) for a, b in evs]
    step_ms = {"p10": round(pctl(per_step, 0.1), 4), "p50": round(pctl(per_step, 0.5), 4), "p90": round(pctl(per_step, 0.9), 4), "n": len(per_step)}
    dp_check = dp_verify(eng, vb, dist, pg, dev, rank, world) if world > 1 else None
    final_loss = float(loss_host[(W + args.steps - 1) % loss_host.numel()])

    imgs = B * world * args.steps
    value = imgs / (ms_dev * 1e-3)
    e2e = imgs / (ms_e2e * 1e-3)
    pk = peaks()
    fl = train_flops_per_image(T=model.num_tokens, K=3 * (MODEL["img_size"] // MODEL["patch"]) ** 2, H=MODEL["hidden"], M=MODEL["mlp_hidden"],
                               L=MODEL["num_layers"], C=MODEL["num_classes"])

    # ---- per-kernel probe + roofline of the dominant kernel (rank 0, after the timed regions) ----
    act_bytes = eng.activation_bytes()
    launches_per_step = int(eng.launches_per_step)
    dp_mode = eng._dp_mode
    table = probe_kernels(eng, steps=3)
    roof = None
    for row in table:
        roof = kernel_roofline(row, pk, B, model.num_tokens, model.hidden)
        if roof:
            roof["share_of_step"] = row["ms_per_step"] / sum(r["ms_per_step"] for r in table)
            break
    cpu = None
    eager = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, cores, ms, kind = cpu_port_images_per_s(min(128, B), 3, 1)
        what = "the reference's own vit.ViT / criterion" if kind == "reference" else "oracle port of the reference"
        cpu = {"value": round(v, 2), "unit": UNIT, "cores": cores, "kind": kind,
               "sample": f"3 steps of batch {min(128, B)} of the same model ({what}, torch fp32, {cores} threads)"}
        try:  # the kernel-level bar: the same PyTorch modules on this GPU (eager ATen / cuBLAS under bf16 autocast)
            del eng
            torch.cuda.empty_cache()
            eager = eager_gpu_images_per_s("bf16-autocast", B, 10, 3)
        except Exception as ex:
            eager = {"error": f"{type(ex).__name__}: {str(ex)[:200]}"}
    if world > 1:
        dist.barrier()
    if rank == 0:
        out = {
            "metric": METRIC, "value": round(value, 1), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": W,
            "ms_per_step": round(ms_dev / args.steps, 4), "step_ms": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": workload_name(world, B) + (f", dropout {args.dropout}" if args.dropout else ""), "per_gpu_batch": B,
                       "cuda_graph": not args.no_graph,
                       "l2": "working set per step (>4 GB of activations) exceeds the 126 MB L2; no flush needed",
                       "parallelism": f"dp{world}",
                       "gradient_exchange": ("none (1 GPU)" if world == 1 else
                                             {"fused": "one peer-memory kernel: barrier + reduce-scatter (P2P loads) + Adam + all-gather (P2P stores)",
                                              "single": "NCCL all-reduce of the flat gradient buffer, then the Adam kernel",
                                              "overlap": "NCCL all-reduce per layer bucket on a side stream, then the Adam kernel"}.get(dp_mode, dp_mode))},
            "e2e": {"value": round(e2e, 1), "unit": UNIT, "ms_per_step": round(ms_e2e / args.steps, 4),
                    "h2d_bytes_per_step": B * (3 * 32 * 32 * 4 + 8) + 32, "d2h_bytes_per_step": 4},
            "gpu_launches": int(launches_per_step * args.steps),
            "launches_per_step": launches_per_step,
            "clocks": clocks,
            "tensor_pipe_frac": {"of_burst": value * fl / world / 1e12 / pk["tf_burst"], "of_sustained": value * fl / world / 1e12 / pk["tf_sust"],
                                 "train_flop_per_img": fl, "peaks": pk["src"]},
            "roofline": roof,
            "cpu_baseline": cpu,
            "gpu_eager_baseline": eager,
            "dp_check": dp_check,
            "final_loss": final_loss,
            "activation_bytes": act_bytes,
        }
        print(json.dumps(out), flush=True)
        if args.kernel_table:
            os.makedirs(os.path.dirname(os.path.abspath(args.kernel_table)), exist_ok=True)
            for row in table:
                r = kernel_roofline(row, pk, B, model.num_tokens, model.hidden)
                row["roofline"] = r
            json.dump({"ms_per_step_graph": ms_dev / args.steps, "img_per_s": value, "kernels": table}, open(args.kernel_table, "w"), indent=1)
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
    if world > 1 and dp_check is not None and not dp_check["ok"]:
        sys.stdout.flush()
        os._exit(3)  # a data-parallel numeric mismatch is a failed run, not a benchmark line
    if world > 1:
        # All ranks are done (barrier), results are printed.  Tearing NCCL down while captured CUDA graphs still reference
        # its communicator hung on B200 (observed at N=2), so leave without the interpreter/NCCL teardown.
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "eager"])
    ap.add_argument("--batch", type=int, default=None, help="per-GPU batch (default: the workload's, 1024 for the headline)")
    ap.add_argument("--workload", default="headline", choices=list(WORKLOADS), help="model shape (default: BASELINE.json's headline configuration)")
    ap.add_argument("--dropout", type=float, default=0.0, help="nn.Dropout probability of the encoder blocks (the reference's default and the headline: 0)")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--kernel-table", default=None, help="write the per-kernel CUDA-event table (JSON) here")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the loss, logits, parameters and gradients of the last timed step as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    global MODEL, PER_GPU_BATCH
    MODEL, PER_GPU_BATCH = WORKLOADS[args.workload]
    if args.batch is None:
        args.batch = PER_GPU_BATCH
    if args.impl == "reference":
        return run_reference(args)
    if args.impl == "eager":
        return run_eager(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
