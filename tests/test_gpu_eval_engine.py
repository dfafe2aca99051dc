"""GPU: the validation pass — vitb_eval_metrics against an fp64 torch reference, and EvalEngine (forward-only CUDA graph, metrics
on the device) against schedule.evaluate on the module path."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# (num_classes, patch, num_layers, encoder_mlp, is_cls_token): the headline model (T = 65, C = 10), t17c100 (T = 17, C = 100)
HEADLINE = dict(num_classes=10, patch=8, num_layers=7, encoder_mlp=True, is_cls_token=True)
T17C100 = dict(num_classes=100, patch=4, num_layers=7, encoder_mlp=True, is_cls_token=True)
NOCLS = dict(num_classes=10, patch=8, num_layers=3, encoder_mlp=True, is_cls_token=False)
NOMLP = dict(num_classes=10, patch=8, num_layers=3, encoder_mlp=False, is_cls_token=True)
CIFAR10_MEAN, CIFAR10_STD = (0.4914, 0.4822, 0.4465), (0.2470, 0.2435, 0.2616)


@pytest.fixture()
def vb():
    import vit_cifar_b200 as v
    v.ops.require_device()
    yield v
    v.set_precision("bf16")


def make_model(vb, cfg, precision="bf16", seed=0, num_layers=None):
    vb.set_precision(precision)
    torch.manual_seed(seed)
    m = vb.ViT(3, cfg["num_classes"], img_size=32, patch=cfg["patch"], dropout=0.0,
               num_layers=cfg["num_layers"] if num_layers is None else num_layers, hidden=384, encoder_mlp=cfg["encoder_mlp"],
               mlp_hidden=384, head=12, is_cls_token=cfg["is_cls_token"])
    return m.cuda()


def make_batches(n, bs, C, seed=1, device="cuda"):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n, 3, 32, 32, generator=g)
    y = torch.randint(0, C, (n,), generator=g)
    return [(x[i:i + bs].to(device), y[i:i + bs].to(device)) for i in range(0, n, bs)]


def assert_same_metrics(got, ref):
    assert got["n"] == ref["n"]
    assert got["val_acc"] == ref["val_acc"]
    assert abs(got["val_loss"] - ref["val_loss"]) <= 1e-6 * abs(ref["val_loss"]), (got, ref)


# ---------------------------------------------------------------------------------------------
# 1. the metrics kernel
# ---------------------------------------------------------------------------------------------
def metrics_ref(logits, labels, nv, smoothing):
    z = logits[:nv].double()
    y = labels[:nv]
    C = z.shape[1]
    lp = torch.log_softmax(z, dim=1)
    ok = (y >= 0) & (y < C)
    lpy = lp.gather(1, y.clamp(0, C - 1)[:, None])[:, 0]
    loss = -((1.0 - smoothing) * lpy + smoothing / (C - 1) * (lp.sum(1) - lpy))
    loss = torch.where(ok, loss, torch.full_like(loss, float("nan")))
    correct = ((z.argmax(1) == y) & ok).sum().item()
    return loss.sum().item(), correct, nv


def run_metrics(vb, logits, labels, smoothing, nv=None, totals=None, ws=None):
    dev = logits.device
    totals = torch.zeros(3, dtype=torch.float64, device=dev) if totals is None else totals
    ws = torch.zeros(vb.ops.eval_metrics_ws_bytes() // 8, dtype=torch.float64, device=dev) if ws is None else ws
    nvd = torch.tensor([nv], dtype=torch.int32, device=dev) if nv is not None else None
    vb.ops.eval_metrics(logits, labels, totals, ws, smoothing, n_valid_dev=nvd)
    return totals, ws


@pytest.mark.parametrize("smoothing", [0.0, 0.1])
@pytest.mark.parametrize("B", [1, 7, 1000, 4096])
@pytest.mark.parametrize("C", [3, 10, 100, 257])
def test_eval_metrics_vs_fp64_torch(vb, C, B, smoothing):
    g = torch.Generator().manual_seed(C * 7919 + B)
    logits = (3 * torch.randn(B, C, generator=g)).cuda()
    labels = torch.randint(0, C, (B,), generator=g).cuda()
    for nv in ([None] if B == 1 else [None, B - B // 3 - 1]):
        totals, ws = run_metrics(vb, logits, labels, smoothing, nv)
        ls, corr, cnt = metrics_ref(logits, labels, B if nv is None else nv, smoothing)
        t = totals.tolist()
        assert t[1] == corr and t[2] == cnt
        assert abs(t[0] - ls) <= 1e-6 * abs(ls), (t, ls)
        assert ws.view(torch.int32)[0].item() == 0  # the arrival counter is left at zero


@pytest.mark.parametrize("C", [3, 10, 100, 257])
def test_eval_metrics_ties_bad_labels_accumulation_determinism(vb, C):
    B = 600
    g = torch.Generator().manual_seed(C)
    logits = torch.randn(B, C, generator=g)
    labels = torch.randint(0, C, (B,), generator=g)
    # ties: rows 0..199 carry their maximum at two (or three) columns; the first one is torch's argmax
    for i in range(200):
        j1, j2 = sorted(torch.randperm(C, generator=g)[:2].tolist())
        logits[i, j1] = logits[i, j2] = logits[i].max() + 1.0
        if i % 3 == 0 and C > 2:
            logits[i, C - 1] = logits[i, j1]
        labels[i] = j1 if i % 2 == 0 else j2
    labels[200], labels[201], labels[202] = C, -1, C + 1000  # out of range: NaN loss, not correct, no fault
    logits, labels = logits.cuda(), labels.cuda()
    totals, ws = run_metrics(vb, logits, labels, 0.1)
    t = totals.tolist()
    assert t[0] != t[0]  # NaN
    ref_correct = ((logits.argmax(1) == labels).sum().item())
    assert t[1] == ref_correct and t[2] == B
    assert sum(1 for i in range(0, 200, 2) if logits[i].argmax().item() == labels[i].item()) == 100

    good = torch.ones(B, dtype=torch.bool)
    good[200:203] = False
    lg, lb = logits[good.cuda()].contiguous(), labels[good.cuda()].contiguous()
    a, ws = run_metrics(vb, lg, lb, 0.1)
    b, _ = run_metrics(vb, lg, lb, 0.1)
    assert torch.equal(a, b)                               # bit-identical runs
    run_metrics(vb, lg, lb, 0.1, totals=a, ws=ws)          # accumulates
    assert a[0].item() == 2 * b[0].item() and a[1].item() == 2 * b[1].item() and a[2].item() == 2 * (B - 3)
    assert ws.view(torch.int32)[0].item() == 0


@pytest.mark.parametrize("C", [3, 10, 100, 256])
def test_eval_row_loss_is_the_training_loss(vb, C):
    """Per image, the loss the metrics kernel adds is the value the training loss kernel averages (same per-row arithmetic)."""
    g = torch.Generator().manual_seed(C + 5)
    for r in range(6):
        z = (4 * torch.randn(1, C, generator=g)).cuda()
        y = torch.randint(0, C, (1,), generator=g).cuda()
        loss = torch.zeros((), dtype=torch.float32, device="cuda")
        vb.ops.ls_ce(z, y, loss, None, 0.1, 1.0)
        totals, _ = run_metrics(vb, z, y, 0.1)
        assert totals[0].item() == float(loss.item()), (r, totals[0].item(), loss.item())


# ---------------------------------------------------------------------------------------------
# 2-3. the engine against schedule.evaluate / model.eval()(x)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["bf16", "fp32"])
@pytest.mark.parametrize("cfg", [HEADLINE, T17C100, NOCLS, NOMLP], ids=["headline", "t17c100", "nocls", "nomlp"])
def test_run_matches_evaluate(vb, cfg, precision):
    model = make_model(vb, cfg, precision)
    batches = make_batches(600, 256, cfg["num_classes"])   # 256 + 256 + 88
    crit = vb.LabelSmoothingCrossEntropyLoss(cfg["num_classes"], smoothing=0.1)
    ref = vb.evaluate(model, crit, batches)
    for use_graph in ((False, True) if cfg is HEADLINE else (True,)):
        ev = vb.EvalEngine(model, batch_size=256, smoothing=0.1, use_graph=use_graph)
        got = ev.run(batches)
        assert_same_metrics(got, ref)
        assert_same_metrics(ev.run(batches), ref)          # second pass: graph replays only
        assert ev.launches_per_batch > 0


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
@pytest.mark.parametrize("cfg", [HEADLINE, T17C100], ids=["headline", "t17c100"])
def test_forward_is_bit_identical_to_module_path(vb, cfg, precision):
    model = make_model(vb, cfg, precision).eval()
    x = make_batches(256, 256, cfg["num_classes"], seed=3)[0][0]
    ev = vb.EvalEngine(model, batch_size=256)
    with torch.no_grad():
        ref = model(x)
    got = ev.forward(x)
    assert got.shape == ref.shape and torch.equal(got, ref)


def test_fresh_weights_after_training_and_load_state_dict(vb):
    model = make_model(vb, HEADLINE, "bf16")
    batches = make_batches(600, 256, 10, seed=4)
    crit = vb.LabelSmoothingCrossEntropyLoss(10, smoothing=0.1)
    ev = vb.EvalEngine(model, batch_size=256)
    r0 = ev.run(batches)
    eng = vb.TrainEngine(model, 128, smoothing=0.1)
    g = torch.Generator().manual_seed(9)
    for _ in range(4):
        eng.step(torch.randn(128, 3, 32, 32, generator=g).cuda(), torch.randint(0, 10, (128,), generator=g).cuda())
    r1 = ev.run(batches)
    assert_same_metrics(r1, vb.evaluate(model, crit, batches))
    assert r1["val_loss"] != r0["val_loss"]
    other = make_model(vb, HEADLINE, "bf16", seed=123)
    model.load_state_dict(other.state_dict())
    r2 = ev.run(batches)
    assert_same_metrics(r2, vb.evaluate(model, crit, batches))
    assert_same_metrics(r2, vb.evaluate(other, crit, batches))


# ---------------------------------------------------------------------------------------------
# 5. memory
# ---------------------------------------------------------------------------------------------
def test_activation_memory_does_not_grow_with_depth_and_full_test_set_batch(vb):
    sizes = []
    for L in (2, 7):
        model = make_model(vb, HEADLINE, "bf16", num_layers=L)
        ev = vb.EvalEngine(model, batch_size=64)
        ev.run(make_batches(64, 64, 10))
        sizes.append(ev.activation_bytes())
    assert sizes[0] == sizes[1] > 0
    model = make_model(vb, HEADLINE, "bf16")
    batches = make_batches(10000, 10000, 10, seed=6)
    ev = vb.EvalEngine(model, batch_size=10000)
    got = ev.run(batches)
    assert got["n"] == 10000
    assert_same_metrics(got, vb.evaluate(model, vb.LabelSmoothingCrossEntropyLoss(10, smoothing=0.1), batches))


# ---------------------------------------------------------------------------------------------
# 6. uint8 input
# ---------------------------------------------------------------------------------------------
def test_uint8_batches_match_normalised_fp32_batches(vb):
    model = make_model(vb, HEADLINE, "bf16")
    g = torch.Generator().manual_seed(8)
    u8 = torch.randint(0, 256, (600, 32, 32, 3), dtype=torch.uint8, generator=g)
    y = torch.randint(0, 10, (600,), generator=g)
    host = [(u8[i:i + 256].pin_memory(), y[i:i + 256].pin_memory()) for i in range(0, 600, 256)]
    ev_u8 = vb.EvalEngine(model, batch_size=256, mean=CIFAR10_MEAN, std=CIFAR10_STD)
    got = ev_u8.run(host)
    dev = []
    for xb, yb in host:
        xd = xb.cuda()
        out = torch.empty((xd.shape[0], 3, 32, 32), dtype=torch.float32, device="cuda")
        vb.ops.augment(xd, None, None, None, CIFAR10_MEAN, CIFAR10_STD, out, 0)
        ref_t = (xd.permute(0, 3, 1, 2).double() / 255 - torch.tensor(CIFAR10_MEAN, device="cuda", dtype=torch.float64)[:, None, None]) \
            / torch.tensor(CIFAR10_STD, device="cuda", dtype=torch.float64)[:, None, None]
        assert (out.double() - ref_t).abs().max().item() <= 1e-6 * max(1.0, ref_t.abs().max().item())
        dev.append((out, yb.cuda()))
    ref = vb.EvalEngine(model, batch_size=256).run(dev)
    assert got == ref
    assert_same_metrics(got, vb.evaluate(model, vb.LabelSmoothingCrossEntropyLoss(10, smoothing=0.1), dev))
    # device-resident uint8 batches go straight to the normalisation kernel
    assert ev_u8.run([(xb.cuda(), yb.cuda()) for xb, yb in host]) == ref


# ---------------------------------------------------------------------------------------------
# 7. host syncs and launches
# ---------------------------------------------------------------------------------------------
def test_add_does_not_synchronise_and_graph_launches_equal_eager(vb):
    model = make_model(vb, HEADLINE, "bf16")
    batches = make_batches(600, 256, 10, seed=10)
    ev = vb.EvalEngine(model, batch_size=256)
    ref = ev.run(batches)                       # builds the graph
    assert ev.captured_launches == ev.launches_per_batch > 0
    ev.reset()
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        for xb, yb in batches:
            ev.add(xb, yb)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert ev.result() == ref


def test_bad_inputs_raise(vb):
    model = make_model(vb, NOMLP, "bf16")
    ev = vb.EvalEngine(model, batch_size=16)
    with pytest.raises(ValueError):
        ev.add(torch.zeros(17, 3, 32, 32, device="cuda"), torch.zeros(17, dtype=torch.int64, device="cuda"))
    with pytest.raises(ValueError):
        ev.add(torch.zeros(4, 3, 16, 16, device="cuda"), torch.zeros(4, dtype=torch.int64, device="cuda"))
    with pytest.raises(ValueError):
        ev.add(torch.zeros(4, 3, 32, 32, device="cuda"), torch.zeros(5, dtype=torch.int64, device="cuda"))
    with pytest.raises(ValueError):  # uint8 without mean / std
        ev.add(torch.zeros(4, 32, 32, 3, dtype=torch.uint8, device="cuda"), torch.zeros(4, dtype=torch.int64, device="cuda"))
    model.enc[0].save_attn_map = True
    with pytest.raises(ValueError, match="model.eval"):
        ev.reset()
    model.enc[0].save_attn_map = False
    model.cls_token.data = model.cls_token.data.clone()  # the parameter leaves the flat buffer: the next model(x) re-packs
    with pytest.raises(RuntimeError, match="re-packed"):
        ev.reset()
    model._ensure_packed()
    with pytest.raises(RuntimeError, match="re-packed"):
        ev.reset()


# ---------------------------------------------------------------------------------------------
# 8. data parallel
# ---------------------------------------------------------------------------------------------
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs on one box")
def test_two_rank_sharded_evaluation_equals_single_gpu_union():
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29579", os.path.join(ROOT, "tools", "eval_dp_check.py")], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-3000:])
    assert "eval_dp_check PASSED" in r.stdout
