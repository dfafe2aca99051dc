"""GPU: one training step under every execution plan of TrainEngine, bit for bit.

The engine can defer the second passes of its split reductions (VITB_DEFER), run the weight gradients on a side stream with the
critical path on a high-priority stream (VITB_WGRAD_STREAM), flush each layer's deferred reductions on the side stream as soon as
that layer's backward is issued (VITB_FLUSH_PER_LAYER) and, on one GPU, run that layer's optimiser step right behind the flush
(VITB_OPT_PER_LAYER).  These change where and when work runs, never what it computes: every plan must give the same losses,
logits, gradients, parameters, optimiser moments and bf16 weight copy, with no tolerance.  A reduction that misses a partial,
a flush ordered before the producer of its partials or an optimiser slice that reads a gradient before it is final changes bits
here, where the comparisons with the fp32 oracle (2e-2) would let it pass.

Each plan also asserts that the engine really runs it, so that a misspelt variable cannot make all plans equal by accident.
"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import oracle
from oracle import ViTConfig

pytestmark = pytest.mark.gpu

ADAM = dict(lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=5e-5)
TINY65 = ViTConfig(num_classes=10, patch=8, num_layers=2, hidden=128, mlp_hidden=128, head=4)
FULL65 = ViTConfig(num_classes=10, patch=8, num_layers=7, hidden=384, mlp_hidden=384, head=12)
FULL17C100 = ViTConfig(num_classes=100, patch=4, num_layers=7, hidden=384, mlp_hidden=384, head=12)
DEEP65 = ViTConfig(num_classes=10, patch=8, num_layers=32, hidden=128, mlp_hidden=128, head=4)
WIDE17 = ViTConfig(num_classes=10, patch=4, num_layers=3, hidden=768, mlp_hidden=3072, head=12)  # BASELINE.json's scaled ViT, 3 layers

# every switch the engine or the Python backward path reads; cleared before each build so that the plan alone decides
SWITCHES = ("VITB_DEFER", "VITB_WGRAD_STREAM", "VITB_FLUSH_PER_LAYER", "VITB_OPT_PER_LAYER", "VITB_BWD_FUSED", "VITB_LN_GELU_FUSED",
            "VITB_DROP_FUSED", "VITB_L2_PERSIST", "VITB_DP_MODE")

# plan -> (environment, what the engine must then run); flush / opt absent = the engine's default for the model's width
PLANS = {
    "P0": ({"VITB_DEFER": "0"}, dict(defer=False, side=False, main=False)),            # immediate second passes, one stream
    "P1": ({"VITB_WGRAD_STREAM": "0"}, dict(defer=True, side=False, main=False)),      # deferred, one flush, one stream
    "P2": ({"VITB_WGRAD_STREAM": "1", "VITB_FLUSH_PER_LAYER": "0"}, dict(defer=True, side=True, main=False, flush=False, opt=False)),
    "P3": ({"VITB_WGRAD_STREAM": "2", "VITB_FLUSH_PER_LAYER": "1", "VITB_OPT_PER_LAYER": "0"},
           dict(defer=True, side=True, main=True, flush=True, opt=False)),
    "P4": ({}, dict(defer=True, side=True, main=True)),                                # the default
    "P5": ({"VITB_FLUSH_PER_LAYER": "1"}, dict(defer=True, side=True, main=True, flush=True, opt=True)),
}
STATE = ("loss", "logits", "G", "P", "Mo", "V", "C")


@pytest.fixture()
def vb():
    import vit_cifar_b200 as v
    v.ops.require_device()
    yield v
    v.set_precision("bf16")


def batches(cfg, B, steps, seed=100):
    return [tuple(t.cuda() for t in oracle.hash_inputs(cfg, B, seed=seed + i)) for i in range(steps)]


def train(vb, monkeypatch, plan, cfg, B, data, use_graph, env=None, dropout=0.0, optimizer="adam"):
    """Build the model and engine under `plan` (+ `env`), train on `data`; returns the state after the last step, the gradient
    buffer after the first, and the parameter layout."""
    for k in SWITCHES:
        monkeypatch.delenv(k, raising=False)
    for k, v in {**(env or {}), **PLANS[plan][0]}.items():
        monkeypatch.setenv(k, v)
    vb.set_precision("bf16")
    torch.manual_seed(0)  # dropout mask seeds
    m = vb.ViT(3, cfg.num_classes, img_size=cfg.img_size, patch=cfg.patch, dropout=dropout, num_layers=cfg.num_layers, hidden=cfg.hidden,
               encoder_mlp=cfg.encoder_mlp, mlp_hidden=cfg.mlp_hidden, head=cfg.head, is_cls_token=cfg.is_cls_token)
    m.load_state_dict(oracle.init_params(cfg, seed=0))
    m = m.cuda()
    eng = vb.TrainEngine(m, B, smoothing=0.1, use_graph=use_graph, optimizer=optimizer, **ADAM)
    want = PLANS[plan][1]
    default = cfg.hidden * max(cfg.hidden, cfg.mlp_hidden) <= 384 * 1536
    got = dict(defer=eng._defer, side=eng._side is not None, main=eng._main_stream is not None, flush=eng._flush_per_layer, opt=eng._opt_per_layer)
    assert got == dict(want, flush=want.get("flush", default), opt=want.get("opt", default)), (plan, got)
    losses, g1 = [], None
    for i, (x, y) in enumerate(data):
        losses.append(eng.step(x, y).clone())
        if i == 0:
            g1 = eng.G.clone()
    torch.cuda.synchronize()
    out = dict(loss=torch.stack(losses), logits=eng.logits.clone(), G=eng.G.clone(), P=eng.P.clone(), Mo=eng.Mo.clone(), V=eng.V.clone(),
               C=eng.C.clone(), G1=g1)
    layout = eng.store.layout
    del eng, m
    torch.cuda.empty_cache()
    return out, layout


def first_difference(layout, a, b):
    for name, s in sorted(layout.slots.items(), key=lambda kv: kv[1].off):
        x, y = layout.view(a, name), layout.view(b, name)
        if not torch.equal(x, y):
            d = (x.double() - y.double()).abs()
            return f"first at {name}: {int((x != y).sum())} of {x.numel()} elements, max |diff| {d.max().item():.3g}"
    return "outside the parameter slots"


def assert_same(layout, a, b, what, names=STATE):
    for n in names:
        if torch.equal(a[n], b[n]):
            continue
        where = first_difference(layout, a[n], b[n]) if n in ("G", "P", "Mo", "V", "C") else \
            f"{int((a[n] != b[n]).sum())} of {a[n].numel()} elements"
        raise AssertionError(f"{what}: {n} differs, {where}")


# ---------------------------------------------------------------------------------------------
def test_tiny65_every_plan_eager_and_graph(vb, monkeypatch):
    cfg, B = TINY65, 8
    data = batches(cfg, B, 4)
    ref, layout = train(vb, monkeypatch, "P0", cfg, B, data, use_graph=False)
    for plan in ("P0", "P1", "P2", "P3", "P4"):
        for use_graph in (False, True):
            if plan == "P0" and not use_graph:
                continue
            out, _ = train(vb, monkeypatch, plan, cfg, B, data, use_graph)
            assert_same(layout, ref, out, f"P0 eager vs {plan} {'graph' if use_graph else 'eager'}")


@pytest.mark.parametrize("drop_fused", ["0", "1"])  # stand-alone dropout passes / masks inside the GEMM, GELU and LayerNorm kernels
def test_tiny65_dropout_and_sgd(vb, monkeypatch, drop_fused):
    cfg, B = TINY65, 8
    data = batches(cfg, B, 4, seed=200)
    env = {"VITB_DROP_FUSED": drop_fused}
    a, layout = train(vb, monkeypatch, "P0", cfg, B, data, True, env=env, dropout=0.1, optimizer="sgd")
    b, _ = train(vb, monkeypatch, "P4", cfg, B, data, True, env=env, dropout=0.1, optimizer="sgd")
    assert_same(layout, a, b, "P0 vs P4, dropout 0.1, SGD")


def test_deep_narrow_model_flushes_in_several_launches(vb, monkeypatch):
    """32 blocks of width 128: one flush holds several hundred plain jobs (four weight gradients of two jobs each per block alone
    make 256), more than one launch of 120; at 260 rows every partial set is plain (< 64 partials)."""
    cfg, B = DEEP65, 4
    lib = vb._lib.load()
    rows = B * cfg.num_tokens
    assert int(lib.vitb_layernorm_bwd_ws_bytes(rows, cfg.hidden)) // (12 * cfg.hidden) < 64
    assert int(lib.vitb_colsum_ws_bytes(rows, cfg.mlp_hidden)) // (4 * cfg.mlp_hidden) < 64
    flushes = []
    real = vb.ops.defer_flush

    def counted():
        n0 = vb.ops.launch_count()
        real()
        flushes.append(vb.ops.launch_count() - n0)
    monkeypatch.setattr(vb.ops, "defer_flush", counted)
    data = batches(cfg, B, 4, seed=300)
    a, layout = train(vb, monkeypatch, "P0", cfg, B, data, True)
    assert flushes == []
    b, _ = train(vb, monkeypatch, "P2", cfg, B, data, True)
    assert len(flushes) == 2 and min(flushes) >= 2, flushes  # the eager step and the capture, each >= 2 plain launches
    assert_same(layout, a, b, "P0 vs P2, 32 layers")


def test_full65_benchmark_configuration(vb, monkeypatch):
    cfg, B = FULL65, 1024
    data = batches(cfg, B, 3, seed=400)
    a, layout = train(vb, monkeypatch, "P0", cfg, B, data[:1], False)
    b, _ = train(vb, monkeypatch, "P4", cfg, B, data[:1], False)
    assert_same(layout, a, b, "P0 vs P4 eager, B = 1024", ("loss", "logits", "G"))
    a, _ = train(vb, monkeypatch, "P0", cfg, B, data, True)
    b, _ = train(vb, monkeypatch, "P4", cfg, B, data, True)
    assert_same(layout, a, b, "P0 vs P4 graph, B = 1024")


def test_full17c100_one_split_weight_gradients(vb, monkeypatch):
    """Two images of 17 tokens: 34 rows, so every tensor-core weight gradient has one split (dW and db written by the GEMM
    itself).  P0 and P4 agree bit for bit, and P4's first-step gradients match the fp32 oracle."""
    cfg, B = FULL17C100, 2
    lib = vb._lib.load()
    import ctypes as C
    f = lib.vitb_debug_wgrad_splits
    f.restype, f.argtypes = C.c_int, [C.c_int, C.c_int, C.c_int]
    H, M = cfg.hidden, cfg.mlp_hidden
    assert all(f(B * cfg.num_tokens, N, K) == 1 for N, K in ((3 * H, H), (H, H), (M, H), (H, M)))
    data = batches(cfg, B, 4, seed=500)
    a, layout = train(vb, monkeypatch, "P0", cfg, B, data, True)
    b, _ = train(vb, monkeypatch, "P4", cfg, B, data, True)
    assert_same(layout, a, b, "P0 vs P4, B = 2")
    x, y = data[0]
    _, loss_ref, grads_ref = oracle.train_step(oracle.init_params(cfg, 0), x.cpu(), y.cpu(), cfg, 0.1)
    assert abs(b["loss"][0].item() - loss_ref.item()) < 2e-2 * abs(loss_ref.item())
    gs = torch.cat([g.double().flatten() for g in grads_ref.values()]).pow(2).mean().sqrt().item()
    worst = ("", 0.0)
    for k, gr in grads_ref.items():
        g, gr = layout.view(b["G1"], k).double().cpu(), gr.double()
        if "Wk.bias" in k:  # analytically zero gradient: against the model's gradient scale
            e = ((g - gr).norm() / (gr.norm() + gs * gr.numel() ** 0.5)).item()
        else:
            e = ((g - gr).norm() / gr.norm().clamp_min(1e-30)).item()
        worst = max(worst, (k, e), key=lambda t: t[1])
    assert worst[1] < 2e-2, worst


def test_scaled_768_model_one_flush_and_per_layer_flush(vb, monkeypatch):
    cfg, B = WIDE17, 64
    data = batches(cfg, B, 3, seed=600)
    a, layout = train(vb, monkeypatch, "P0", cfg, B, data, True)
    b, _ = train(vb, monkeypatch, "P4", cfg, B, data, True)
    assert_same(layout, a, b, "P0 vs P4 (one flush), 768 / 3072")
    c, _ = train(vb, monkeypatch, "P5", cfg, B, data, True)
    assert_same(layout, a, c, "P0 vs P5 (per-layer flush and optimiser), 768 / 3072")


def test_fused_backward_does_not_depend_on_the_plan(vb, monkeypatch):
    cfg, B = FULL65, 64
    assert vb.ops.bwd_fused_ws_bytes(B * cfg.num_tokens, cfg.hidden, cfg.hidden) > 0  # the fused kernel really runs
    data = batches(cfg, B, 3, seed=700)
    env = {"VITB_BWD_FUSED": "1"}
    a, layout = train(vb, monkeypatch, "P0", cfg, B, data, True, env=env)
    b, _ = train(vb, monkeypatch, "P4", cfg, B, data, True, env=env)
    assert_same(layout, a, b, "P0 vs P4, VITB_BWD_FUSED=1")


# ---------------------------------------------------------------------------------------------
# switches the library caches in static variables (VITB_PDL) cannot change inside one process: bench.py runs, one per setting
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("workload", ["headline", "t17c100"])
def test_bench_outputs_do_not_depend_on_pdl_or_deferral(tmp_path, workload):
    """Programmatic dependent launch only lets kernels overlap: a difference here is a missing wait before a dependent access."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    names = ("loss", "logits", "params", "grads")

    def bench(tag, env):
        e = {k: v for k, v in os.environ.items() if k not in SWITCHES + ("VITB_PDL",)}
        e.update(env)
        outdir = tmp_path / tag
        r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--steps", "3", "--warmup", "1", "--batch", "128", "--workload", workload,
                            "--no-cpu-baseline", "--dump-outputs", str(outdir)], capture_output=True, text=True, timeout=900, env=e)
        assert r.returncode == 0, r.stderr[-3000:]
        json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
        return {n: np.load(outdir / f"{n}.npy") for n in names}

    ref = bench("default", {})
    assert ref["grads"].any()
    for tag, env in (("no_pdl", {"VITB_PDL": "0"}), ("immediate", {"VITB_DEFER": "0", "VITB_WGRAD_STREAM": "0"})):
        out = bench(tag, env)
        for n in names:
            np.testing.assert_array_equal(out[n], ref[n], err_msg=f"{workload}: {tag} vs default: {n}")
