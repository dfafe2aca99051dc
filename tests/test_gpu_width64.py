"""GPU: hidden / MLP widths of 64 mod 128 (ViT-Tiny's 192 and friends).

Kernels against fp64 restatements of the same inputs (LayerNorm with two-element lane groups; the tensor-core GEMMs with a
partial last 128-column tile; the column sums), guard bands past the end of every output, deferred against immediate weight
gradients bit for bit, and whole models against the oracle, the graph against eager, EvalEngine against evaluate and
tools/train.py end to end.
"""
import json
import os
import subprocess
import sys

import pytest
import torch

import oracle
from oracle import ViTConfig

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ADAM = dict(lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=5e-5)
GUARD = 256


@pytest.fixture()
def vb():
    import vit_cifar_b200 as v
    v.ops.require_device()
    yield v
    v.set_precision("bf16")


def rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


def guarded(shape, dtype):
    """A tensor of `shape` followed by GUARD NaN elements in the same allocation; returns (view, guard view)."""
    n = 1
    for s in shape:
        n *= s
    buf = torch.full((n + GUARD,), float("nan"), dtype=dtype, device="cuda")
    return buf[:n].view(shape), buf[n:]


def untouched(g):
    return bool(torch.isnan(g.float()).all())


def gelu64(z):
    return 0.5 * z * (1.0 + torch.erf(z / 2 ** 0.5))


def gelu_grad64(z):
    return 0.5 * (1.0 + torch.erf(z / 2 ** 0.5)) + z * torch.exp(-0.5 * z * z) / (2 * torch.pi) ** 0.5


def kernel_names(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events()}


# ---------------------------------------------------------------------------------------------
# LayerNorm
# ---------------------------------------------------------------------------------------------
def ln_ref(x, w, b, eps=1e-5):
    x = x.double()
    mu = x.mean(-1, keepdim=True)
    var = ((x - mu) ** 2).mean(-1, keepdim=True)
    rs = 1.0 / torch.sqrt(var + eps)
    return (x - mu) * rs * w.double() + b.double(), mu.squeeze(-1), rs.squeeze(-1)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32], ids=["bf16", "fp32"])
@pytest.mark.parametrize("H", [64, 192, 320, 640, 960])
def test_layernorm_forward(vb, H, dtype):
    rows = 1037
    g = torch.Generator(device="cuda").manual_seed(H)
    x = (torch.randn(rows, H, device="cuda", generator=g) * 2 + 0.5).to(dtype)
    w = torch.randn(H, device="cuda", generator=g)
    b = torch.randn(H, device="cuda", generator=g)
    y, yg = guarded((rows, H), dtype)
    mean, mg = guarded((rows,), torch.float32)
    rstd, rg = guarded((rows,), torch.float32)
    vb.ops.layernorm_fwd(x, H, w, b, y, mean, rstd, rows, H)
    torch.cuda.synchronize()
    yr, mr, rr = ln_ref(x, w, b)
    tol = 1e-2 if dtype == torch.bfloat16 else 1e-5
    assert rel(y, yr) < tol
    assert rel(mean, mr) < 1e-5 and rel(rstd, rr) < 1e-5
    assert untouched(yg) and untouched(mg) and untouched(rg)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32], ids=["bf16", "fp32"])
@pytest.mark.parametrize("res,cs", [(False, False), (True, False), (False, True), (True, True)], ids=["plain", "res", "colsum", "res-colsum"])
@pytest.mark.parametrize("H", [64, 192, 320, 640, 960])
def test_layernorm_backward(vb, H, res, cs, dtype):
    rows = 2 * 1037 + 5
    g = torch.Generator(device="cuda").manual_seed(7 * H + 3)
    x = (torch.randn(rows, H, device="cuda", generator=g) + 0.3).to(dtype)
    dy = torch.randn(rows, H, device="cuda", generator=g).to(dtype)
    dres = torch.randn(rows, H, device="cuda", generator=g).to(dtype) if res else None
    w = torch.randn(H, device="cuda", generator=g)
    b = torch.zeros(H, device="cuda")
    y = torch.empty(rows, H, dtype=dtype, device="cuda")
    mean = torch.empty(rows, device="cuda")
    rstd = torch.empty(rows, device="cuda")
    vb.ops.layernorm_fwd(x, H, w, b, y, mean, rstd, rows, H)
    dx, dxg = guarded((rows, H), dtype)
    dw, dwg = guarded((H,), torch.float32)
    db, dbg = guarded((H,), torch.float32)
    csum, csg = guarded((H,), torch.float32) if cs else (None, None)
    vb.ops.layernorm_bwd(dy, x, H, w, mean, rstd, dres, dx, H, dw, db, csum, rows, H)
    torch.cuda.synchronize()
    xh = (x.double() - mean.double()[:, None]) * rstd.double()[:, None]
    gd = dy.double() * w.double()
    dx_ref = rstd.double()[:, None] * (gd - gd.mean(-1, keepdim=True) - xh * (gd * xh).mean(-1, keepdim=True))
    if res:
        dx_ref = dx_ref + dres.double()
    tol = 1e-2 if dtype == torch.bfloat16 else 1e-5
    assert rel(dx, dx_ref) < tol
    assert rel(dw, (dy.double() * xh).sum(0)) < 1e-4
    assert rel(db, dy.double().sum(0)) < 1e-4
    assert untouched(dxg) and untouched(dwg) and untouched(dbg)
    if cs:
        # (the kernel sums dx before its rounding to the storage type: compare with the exact values)
        assert rel(csum, dx_ref.sum(0)) < 1e-4
        assert untouched(csg)


@pytest.mark.parametrize("with_z", [False, True], ids=["drop", "drop-gelu"])
@pytest.mark.parametrize("H", [64, 192, 320, 640, 960])
def test_layernorm_backward_fused(vb, H, with_z):
    """The fused form also writes dx2 = dropout(dx) [* gelu'(z)] and its column sums; dx2 must equal what the stand-alone
    dropout / GELU-backward kernels make of dx."""
    rows = 1500
    dtype = torch.bfloat16
    g = torch.Generator(device="cuda").manual_seed(H + 11)
    x = torch.randn(rows, H, device="cuda", generator=g).to(dtype)
    dy = torch.randn(rows, H, device="cuda", generator=g).to(dtype)
    dres = torch.randn(rows, H, device="cuda", generator=g).to(dtype)
    z = torch.randn(rows, H, device="cuda", generator=g).to(dtype) if with_z else None
    w = torch.randn(H, device="cuda", generator=g)
    y = torch.empty(rows, H, dtype=dtype, device="cuda")
    mean = torch.empty(rows, device="cuda")
    rstd = torch.empty(rows, device="cuda")
    vb.ops.layernorm_fwd(x, H, w, torch.zeros(H, device="cuda"), y, mean, rstd, rows, H)
    dx = torch.empty(rows, H, dtype=dtype, device="cuda")
    dx2, dx2g = guarded((rows, H), dtype)
    dw = torch.empty(H, device="cuda")
    db = torch.empty(H, device="cuda")
    cs, csg = guarded((H,), torch.float32)
    drop = vb.ops.drop_desc(0.1, 1234, 2, 5)
    vb.ops.layernorm_bwd_fused(dy, x, H, w, mean, rstd, dres, dx, H, dw, db, z, dx2, cs, rows, H, drop=drop)
    ref = torch.empty_like(dx)
    if with_z:
        refcs = torch.empty(H, device="cuda")
        vb.ops.gelu_bwd_colsum(dx, z, ref, refcs, rows, H, drop=drop)
    else:
        vb.ops.dropout(dx, None, ref, 0.1, 1234, 2, 5)
    torch.cuda.synchronize()
    assert torch.equal(dx2, ref)
    # the column sums add dx2 before its rounding to bf16, as the stand-alone GELU backward does
    if with_z:
        assert rel(cs, refcs) < 1e-5
    else:
        assert rel(cs, dx2.double().sum(0)) < 1e-2
    assert untouched(dx2g) and untouched(csg)


@pytest.mark.parametrize("cols", [64, 192, 320, 576])
def test_column_sums_and_gelu_backward(vb, cols):
    rows = 8320 + 7
    g = torch.Generator(device="cuda").manual_seed(cols)
    a = torch.randn(rows, cols, device="cuda", generator=g).to(torch.bfloat16)
    z = torch.randn(rows, cols, device="cuda", generator=g).to(torch.bfloat16)
    s, sg = guarded((cols,), torch.float32)
    vb.ops.colsum(a, s, rows, cols)
    dz, dzg = guarded((rows, cols), torch.bfloat16)
    s2, s2g = guarded((cols,), torch.float32)
    vb.ops.gelu_bwd_colsum(a, z, dz, s2, rows, cols)
    torch.cuda.synchronize()
    assert rel(s, a.double().sum(0)) < 1e-5
    ref = a.double() * gelu_grad64(z.double())
    assert rel(dz, ref) < 1e-2
    assert rel(s2, ref.sum(0)) < 1e-2
    assert untouched(sg) and untouched(dzg) and untouched(s2g)


# ---------------------------------------------------------------------------------------------
# tensor-core GEMMs
# ---------------------------------------------------------------------------------------------
NS = [64, 192, 320, 576]
KS = [64, 192, 384, 768]


def bf(t):
    return t.to(torch.bfloat16)


@pytest.mark.parametrize("K", KS)
@pytest.mark.parametrize("N", NS)
@pytest.mark.parametrize("M", [77, 8320 + 45])
def test_gemm_forward_epilogues(vb, M, N, K):
    g = torch.Generator(device="cuda").manual_seed(M + N + K)
    a = bf(torch.randn(M, K, device="cuda", generator=g))
    w = bf(torch.randn(N, K, device="cuda", generator=g) / K ** 0.5)
    bias = torch.randn(N, device="cuda", generator=g)
    resid = bf(torch.randn(M, N, device="cuda", generator=g))
    z_ref = a.double() @ w.double().t() + bias.double()
    # bias only
    c, cg = guarded((M, N), torch.bfloat16)
    vb.ops.gemm_fwd(a, w, bias, None, c, None, M, N, K)
    # bias + GELU + pre-activation + residual
    c2, c2g = guarded((M, N), torch.bfloat16)
    pre, preg = guarded((M, N), torch.bfloat16)
    vb.ops.gemm_fwd(a, w, bias, resid, c2, pre, M, N, K, gelu=True)
    torch.cuda.synchronize()
    assert rel(c, z_ref) < 1e-2
    assert rel(pre, z_ref) < 1e-2
    assert rel(c2, gelu64(pre.double()) + resid.double()) < 1e-2
    assert untouched(cg) and untouched(c2g) and untouched(preg)


@pytest.mark.parametrize("N", NS)
def test_gemm_forward_dropout_epilogue_equals_the_standalone_mask(vb, N):
    M, K = 8320 + 45, 192
    g = torch.Generator(device="cuda").manual_seed(N)
    a = bf(torch.randn(M, K, device="cuda", generator=g))
    w = bf(torch.randn(N, K, device="cuda", generator=g) / K ** 0.5)
    bias = torch.randn(N, device="cuda", generator=g)
    resid = bf(torch.randn(M, N, device="cuda", generator=g))
    c, cg = guarded((M, N), torch.bfloat16)
    vb.ops.gemm_fwd(a, w, bias, resid, c, None, M, N, K, gelu=True, drop=vb.ops.drop_desc(0.1, 99, 1, 3))
    plain = torch.empty(M, N, dtype=torch.bfloat16, device="cuda")
    vb.ops.gemm_fwd(a, w, bias, None, plain, None, M, N, K, gelu=True)
    ref = torch.empty_like(plain)
    vb.ops.dropout(plain, resid, ref, 0.1, 99, 1, 3)
    torch.cuda.synchronize()
    assert rel(c, ref) < 1e-2     # (the epilogue adds the residual in fp32, the stand-alone pass after a bf16 round trip)
    assert untouched(cg)


@pytest.mark.parametrize("K", NS)
@pytest.mark.parametrize("N", KS)
@pytest.mark.parametrize("M", [77, 8320 + 45])
def test_gemm_dgrad(vb, M, N, K):
    """dX[M, K] = dY[M, N] W[N, K]: the output width is K."""
    g = torch.Generator(device="cuda").manual_seed(3 * M + N + K)
    dy = bf(torch.randn(M, N, device="cuda", generator=g))
    w = bf(torch.randn(N, K, device="cuda", generator=g) / N ** 0.5)
    z = bf(torch.randn(M, K, device="cuda", generator=g))
    dx, dxg = guarded((M, K), torch.bfloat16)
    vb.ops.gemm_dgrad(dy, w, None, dx, M, N, K)
    dx2, dx2g = guarded((M, K), torch.bfloat16)
    vb.ops.gemm_dgrad(dy, w, z, dx2, M, N, K)
    torch.cuda.synchronize()
    ref = dy.double() @ w.double()
    assert rel(dx, ref) < 1e-2
    assert rel(dx2, ref * gelu_grad64(z.double())) < 1e-2
    assert untouched(dxg) and untouched(dx2g)


@pytest.mark.parametrize("K", KS + [320])
@pytest.mark.parametrize("N", NS)
@pytest.mark.parametrize("M", [40, 1040 + 3, 8320 + 45])
def test_gemm_wgrad_deferred_equals_immediate(vb, M, N, K):
    """dW[N, K] = dYᵀ X and db = column sums of dY, in every split regime (M = 40: one split, written by the GEMM itself)."""
    from vit_cifar_b200 import _lib
    import ctypes as C
    lib = _lib.load()
    f = lib.vitb_debug_wgrad_splits
    f.restype, f.argtypes = C.c_int, [C.c_int, C.c_int, C.c_int]
    assert f(M, N, K) >= 1
    g = torch.Generator(device="cuda").manual_seed(M + 5 * N + K)
    dy = bf(torch.randn(M, N, device="cuda", generator=g))
    x = bf(torch.randn(M, K, device="cuda", generator=g))
    dw, dwg = guarded((N, K), torch.float32)
    db, dbg = guarded((N,), torch.float32)
    vb.ops.gemm_wgrad(dy, x, dw, db, M, N, K)
    arena = torch.empty(64 << 20, dtype=torch.uint8, device="cuda")
    dw2, dw2g = guarded((N, K), torch.float32)
    db2, db2g = guarded((N,), torch.float32)
    vb.ops.defer_begin(arena)
    vb.ops.gemm_wgrad(dy, x, dw2, db2, M, N, K)
    vb.ops.defer_flush()
    torch.cuda.synchronize()
    assert rel(dw, dy.double().t() @ x.double()) < 1e-5
    assert rel(db, dy.double().sum(0)) < 1e-5
    assert torch.equal(dw, dw2) and torch.equal(db, db2)
    assert untouched(dwg) and untouched(dbg) and untouched(dw2g) and untouched(db2g)


def test_partial_tiles_run_on_the_tensor_cores(vb):
    M = 4096
    a = bf(torch.randn(M, 192, device="cuda"))
    w = bf(torch.randn(768, 192, device="cuda"))
    w2 = bf(torch.randn(192, 768, device="cuda"))
    bias = torch.randn(768, device="cuda")
    out = torch.empty(M, 768, dtype=torch.bfloat16, device="cuda")
    out2 = torch.empty(M, 192, dtype=torch.bfloat16, device="cuda")
    dx = torch.empty(M, 192, dtype=torch.bfloat16, device="cuda")
    dw = torch.empty(192, 768, device="cuda")
    db = torch.empty(192, device="cuda")

    def run():
        vb.ops.gemm_fwd(a, w, bias, None, out, None, M, 768, 192)       # N % 128 == 0, K = 192
        vb.ops.gemm_fwd(out, w2, bias[:192], None, out2, None, M, 192, 768)   # N = 192: partial last column tile
        vb.ops.gemm_dgrad(out, w, None, dx, M, 768, 192)                # dX = dY W: output width 192
        vb.ops.gemm_wgrad(out2, out, dw, db, M, 192, 768)

    names = kernel_names(run)
    assert any("gemm_tc_tail_kernel" in n for n in names), names
    assert not any("simt" in n.lower() for n in names), names


# ---------------------------------------------------------------------------------------------
# whole models
# ---------------------------------------------------------------------------------------------
WIDTHS = {"tiny192": (192, 768, 3), "ref192": (192, 192, 6), "w320": (320, 320, 10), "w640": (640, 640, 10)}


def make_cfg(name, patch):
    H, M, heads = WIDTHS[name]
    return ViTConfig(num_classes=10, patch=patch, num_layers=2, hidden=H, mlp_hidden=M, head=heads)


def build(vb, cfg, precision):
    vb.set_precision(precision)
    m = vb.ViT(3, cfg.num_classes, img_size=cfg.img_size, patch=cfg.patch, dropout=0.0, num_layers=cfg.num_layers, hidden=cfg.hidden,
               encoder_mlp=cfg.encoder_mlp, mlp_hidden=cfg.mlp_hidden, head=cfg.head, is_cls_token=cfg.is_cls_token)
    m.load_state_dict(oracle.init_params(cfg, seed=0))
    return m.cuda()


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("patch", [8, 4], ids=["T65", "T17"])
@pytest.mark.parametrize("name", list(WIDTHS))
def test_module_forward_backward_vs_oracle(vb, name, patch, precision):
    cfg = make_cfg(name, patch)
    tol = 1e-4 if precision == "fp32" else 2e-2
    model = build(vb, cfg, precision)
    x, y = oracle.hash_inputs(cfg, 4, seed=1)
    logits_ref, loss_ref, grads_ref = oracle.train_step(oracle.init_params(cfg, 0), x, y, cfg, 0.1)
    logits = model(x.cuda())
    loss = vb.LabelSmoothingCrossEntropyLoss(cfg.num_classes, smoothing=0.1)(logits, y.cuda())
    loss.backward()
    assert rel(logits, logits_ref) < tol
    if precision == "fp32":
        assert torch.equal(logits.argmax(-1).cpu(), logits_ref.argmax(-1))
    scale = torch.cat([g.double().flatten() for g in grads_ref.values() if g is not None]).pow(2).mean().sqrt().item()
    for k, p in model.named_parameters():
        gr = grads_ref[k].double()
        # Wk.bias: analytically zero (softmax is shift invariant), measured against the model's typical gradient size
        e = ((p.grad.double().cpu() - gr).norm() / (gr.norm() + (scale * gr.numel() ** 0.5 if "Wk.bias" in k else 0.0))).item()
        assert e < tol, (k, e)


@pytest.mark.parametrize("name", ["tiny192", "w320"])
def test_engine_graph_equals_eager_and_tracks_the_oracle_for_30_adam_steps(vb, name):
    cfg = make_cfg(name, 8)
    B = 16
    res = []
    for use_graph in (False, True):
        model = build(vb, cfg, "bf16")
        eng = vb.TrainEngine(model, B, smoothing=0.1, use_graph=use_graph, **ADAM)
        ls = []
        for s in range(30):
            x, y = oracle.hash_inputs(cfg, B, seed=100 + s)
            ls.append(eng.step(x.cuda(), y.cuda()).item())
        res.append((ls, {k: v.clone() for k, v in model.state_dict().items()}))
    assert res[0][0] == res[1][0]
    for k in res[0][1]:
        assert torch.equal(res[0][1][k], res[1][1][k]), k
    params = oracle.init_params(cfg, 0)
    m = {k: torch.zeros_like(v) for k, v in params.items()}
    v = {k: torch.zeros_like(p) for k, p in params.items()}
    ref = []
    for s in range(30):
        x, y = oracle.hash_inputs(cfg, B, seed=100 + s)
        _, loss, grads = oracle.train_step(params, x, y, cfg, 0.1)
        ref.append(loss.item())
        oracle.adam_step(params, grads, m, v, s + 1, **ADAM)
    for s, (a, b) in enumerate(zip(res[0][0], ref)):
        assert abs(a - b) < 2e-2 * abs(b), (s, a, b)


@pytest.mark.parametrize("plan", [dict(VITB_DEFER="0"), dict(VITB_WGRAD_STREAM="0"), dict(VITB_FLUSH_PER_LAYER="1"),
                                  dict(VITB_OPT_PER_LAYER="1")], ids=["nodefer", "nostream", "flush-per-layer", "opt-per-layer"])
def test_execution_plans_give_bit_identical_steps(vb, plan, monkeypatch):
    cfg = make_cfg("tiny192", 8)
    B = 32

    def run():
        model = build(vb, cfg, "bf16")
        eng = vb.TrainEngine(model, B, smoothing=0.1, use_graph=True, **ADAM)
        ls = []
        for s in range(3):
            x, y = oracle.hash_inputs(cfg, B, seed=200 + s)
            ls.append(eng.step(x.cuda(), y.cuda()).item())
        return ls, {k: v.clone() for k, v in model.state_dict().items()}

    ref = run()
    for k, v in plan.items():
        monkeypatch.setenv(k, v)
    got = run()
    assert got[0] == ref[0]
    for k in ref[1]:
        assert torch.equal(got[1][k], ref[1][k]), k


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_eval_engine_matches_evaluate(vb, precision):
    cfg = make_cfg("tiny192", 8)
    model = build(vb, cfg, precision)
    g = torch.Generator().manual_seed(1)
    x = torch.randn(600, 3, 32, 32, generator=g)
    y = torch.randint(0, 10, (600,), generator=g)
    batches = [(x[i:i + 256].cuda(), y[i:i + 256].cuda()) for i in range(0, 600, 256)]
    ref = vb.evaluate(model, vb.LabelSmoothingCrossEntropyLoss(10, smoothing=0.1), batches)
    got = vb.EvalEngine(model, batch_size=256, smoothing=0.1, use_graph=True).run(batches)
    assert got["n"] == ref["n"] and got["val_acc"] == ref["val_acc"]
    assert abs(got["val_loss"] - ref["val_loss"]) <= 1e-6 * abs(ref["val_loss"])


def test_train_tool_trains_vit_tiny(vb, tmp_path):
    args = ["--synthetic", "4000", "--max-epochs", "2", "--warmup-epoch", "1", "--batch-size", "128", "--num-layers", "4", "--hidden", "192",
            "--mlp-hidden", "768", "--head", "3", "--seed", "5", "--out-dir", str(tmp_path)]
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "train.py"), *args], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-3000:])
    logs = [json.loads(line) for line in r.stdout.splitlines() if line.startswith("{")]
    assert len(logs) == 2
    assert logs[1]["loss"] < logs[0]["loss"] and logs[1]["val_loss"] < logs[0]["val_loss"]


def test_two_rank_data_parallel_step_at_width_192(vb):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29571", os.path.join(ROOT, "tools", "dp_check.py")], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-3000:])
    assert "[vit-tiny width 192 bf16 graph]" in r.stdout and "dp_check PASSED" in r.stdout
