"""CPU: host-side logic of the drop-in layer — constructor/state_dict compatibility with the reference,
flat parameter layout and gradient buckets, Adam hyper-parameter arithmetic, and the data-parallel bucket
all-reduce on a 2-rank gloo group."""
import math
import os

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import oracle
from oracle.ref_shim import SKIP_REASON, import_reference, reference_available

README = dict(num_classes=10, img_size=32, patch=8, num_layers=7, hidden=384, mlp_hidden=384, head=12)


def make(**kw):
    import vit_cifar_b200 as vb
    return vb.ViT(3, kw.pop("num_classes", 10), **kw)


def test_constructor_signature_and_state_dict_match_oracle_names():
    import inspect
    import vit_cifar_b200 as vb
    sig = inspect.signature(vb.ViT.__init__)
    assert list(sig.parameters)[1:] == ["in_c", "num_classes", "img_size", "patch", "dropout", "num_layers", "hidden", "encoder_mlp",
                                        "mlp_hidden", "head", "is_cls_token"]  # vit.py:20-33
    d = {k: v.default for k, v in sig.parameters.items() if k != "self"}
    assert d == dict(in_c=3, num_classes=10, img_size=224, patch=16, dropout=0.0, num_layers=12, hidden=768, encoder_mlp=True,
                     mlp_hidden=3072, head=8, is_cls_token=True)
    m = make(**README)
    cfg = oracle.ViTConfig(**README)
    sd = m.state_dict()
    assert {k: tuple(v.shape) for k, v in sd.items()} == cfg.param_shapes()
    assert list(sd.keys()) == list(cfg.param_shapes().keys())
    assert sum(p.numel() for p in m.parameters()) == 6_268_810 and len(list(m.parameters())) == 120
    with pytest.raises(AssertionError):
        make(img_size=32, patch=5)  # vit.py:40


@pytest.mark.skipif(not reference_available(), reason=SKIP_REASON)
def test_same_seed_gives_reference_initialisation_and_interchangeable_state_dict():
    ref_vit, _, _ = import_reference()
    kw = dict(img_size=32, patch=4, num_layers=2, hidden=128, mlp_hidden=256, head=4)
    torch.manual_seed(2045)
    ref = ref_vit.ViT(3, 100, **kw)
    torch.manual_seed(2045)
    ours = make(num_classes=100, **kw)
    rsd, osd = ref.state_dict(), ours.state_dict()
    assert list(rsd.keys()) == list(osd.keys())
    for k in rsd:
        assert torch.equal(rsd[k], osd[k]), k  # same construction order -> same RNG stream
    ours.load_state_dict(rsd)          # reference checkpoint -> ours
    ref.load_state_dict(ours.state_dict())  # and back
    # the block interfaces the reference's callers touch (network.py:411, run_model.py:45-47)
    assert hasattr(ours.enc[0], "save_attn_map") and hasattr(ours.enc[0].attention, "save_attn_map")
    ours.enc[0].save_attn_map = True
    assert ours.enc[0].attention.save_attn_map is True
    with pytest.raises(Exception):
        ours.enc[1].get_attention_map()


def test_flat_layout_and_buckets():
    from vit_cifar_b200.params import ALIGN
    m = make(**README)
    lay = m._layout()
    H = 384
    offs = [s.off for s in lay.slots.values()]
    assert all(o % ALIGN == 0 for o in offs)
    q, k, v = (lay.slots[f"enc.3.attention.{n}.weight"] for n in ("Wq", "Wk", "Wv"))
    assert k.off == q.off + H * H and v.off == k.off + H * H  # one (3H,H) operand for the fused QKV GEMM
    bq, bv = lay.slots["enc.3.attention.Wq.bias"], lay.slots["enc.3.attention.Wv.bias"]
    assert bv.off + bv.numel - bq.off == 3 * H
    b = m.bucket_bounds()
    assert len(b) == 7 + 2 and b[0][0] == 0 and b[-1][1] == lay.active_end
    assert all(b[i][1] == b[i + 1][0] for i in range(len(b) - 1))
    assert all(e - s == 888_576 for s, e in b[1:-1])  # SURVEY.md §8e: 888,576 parameters per encoder layer
    # a model without the MLP keeps la2 out of the optimised range (torch's Adam skips grad-less parameters)
    m2 = make(img_size=32, patch=4, num_layers=1, hidden=128, mlp_hidden=128, head=4, encoder_mlp=False)
    l2 = m2._layout()
    assert l2.slots["enc.0.la2.weight"].off >= l2.active_end


def test_adam_hyper_matches_torch_arithmetic():
    import vit_cifar_b200 as vb
    h = vb.adam_hyper(3, 1e-3, 0.9, 0.999, 1e-8, 5e-5, 0.5)
    assert h[0] == 1e-3 / (1 - 0.9 ** 3) and h[1] == math.sqrt(1 - 0.999 ** 3) and h[2:] == [0.9, 0.999, 1e-8, 5e-5, 0.5, 1.0 - 0.9, 1.0 - 0.999]


def test_dims_validation_messages():
    from vit_cifar_b200.functional import Dims
    Dims(B=2, T=65, H=384, heads=12, M=384).check()
    with pytest.raises(ValueError):
        Dims(B=2, T=65, H=100, heads=4, M=128).check()
    with pytest.raises(ValueError):
        Dims(B=2, T=65, H=384, heads=8, M=384).check()   # head_dim 48
    with pytest.raises(ValueError):
        Dims(B=2, T=197, H=384, heads=12, M=384).check()  # 14x14+1 tokens do not fit the short-sequence kernel


def test_dropout_stream_state_of_the_modules():
    """nn.Dropout(p) bookkeeping on the host: no mask stream in eval or at p = 0, a lazily drawn seed (torch.manual_seed makes it
    repeatable and it does not perturb the constructor's RNG stream), one step per training call, p validated like nn.Dropout."""
    import vit_cifar_b200 as vb
    torch.manual_seed(3)
    a = vb.TransformerEncoder(128, 128, head=4, dropout=0.25)
    torch.manual_seed(3)
    b = vb.TransformerEncoder(128, 128, head=4, dropout=0.0)
    assert all(torch.equal(x, y) for x, y in zip(a.state_dict().values(), b.state_dict().values()))
    assert a._drop_seed is None and a._next_drop(0.25, training=False) is None and b._next_drop(0.0, training=True) is None
    torch.manual_seed(9)
    d1, d2 = a._next_drop(0.25, True), a._next_drop(0.25, True)
    assert (d1.p, d1.step, d2.step) == (0.25, 1, 2) and d1.seed == d2.seed == a._drop_seed
    c = vb.TransformerEncoder(128, 128, head=4, dropout=0.25)
    torch.manual_seed(9)
    assert c._next_drop(0.25, True).seed == d1.seed
    with pytest.raises(ValueError):
        a._next_drop(1.0, True)
    assert isinstance(a.mlp[2], torch.nn.Dropout) and a.mlp[2].p == 0.25 and a.attention.dropout.p == 0.25  # reference structure


def _dp_worker(rank, world, port, outdir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from vit_cifar_b200.parallel import allreduce_all
        import vit_cifar_b200 as vb
        m = vb.ViT(3, 10, img_size=32, patch=4, num_layers=2, hidden=128, mlp_hidden=128, head=4)
        lay = m._layout()
        buckets = m.bucket_bounds()
        g = torch.Generator().manual_seed(100 + rank)
        flat = torch.randn(lay.total, generator=g)
        flat[lay.active_end:] = 0
        mine = flat.clone()
        allreduce_all(flat, buckets, None)
        torch.save((mine, flat), os.path.join(outdir, f"rank{rank}.pt"))
    finally:
        dist.destroy_process_group()


def test_bucket_allreduce_two_ranks_gloo():
    """world_size-2 data-parallel exchange on CPU: every bucket summed across ranks, identical on both, and
    Adam with grad_scale = 1/2 on the sum equals Adam on the mean (DDP semantics)."""
    import tempfile
    ctx = mp.get_context("spawn")
    port = 29500 + os.getpid() % 2000
    with tempfile.TemporaryDirectory() as outdir:
        procs = [ctx.Process(target=_dp_worker, args=(r, 2, port, outdir)) for r in range(2)]
        for p in procs:
            p.start()
        for p in procs:
            p.join(timeout=180)
            assert p.exitcode == 0
        got = {r: torch.load(os.path.join(outdir, f"rank{r}.pt")) for r in range(2)}
    total = got[0][0] + got[1][0]
    assert torch.equal(got[0][1], got[1][1])
    torch.testing.assert_close(got[0][1], total)
    # mean semantics through the optimiser scale
    p0 = torch.randn(64)
    a = {"p": p0.clone()}; b = {"p": p0.clone()}
    z = lambda: {"p": torch.zeros(64)}  # noqa: E731
    gsum = total[:64]
    oracle.adam_step(a, {"p": gsum / 2}, z(), z(), 1)
    oracle.adam_step(b, {"p": gsum * 0.5}, z(), z(), 1)
    assert torch.equal(a["p"], b["p"])


def _ipc_worker(rank, world, port, outdir, failing_rank, fail_at):
    """Handle exchange of the fused data-parallel step with the CUDA IPC calls replaced by fakes (no GPU here): what is tested is
    the collective choreography — one all_gather_object, failures stay local, every rank reaches the same verdict."""
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from vit_cifar_b200 import ops
        from vit_cifar_b200.parallel import exchange_peer_pointers

        class FakeTensor:
            def __init__(self, addr):
                self.addr = addr

            def data_ptr(self):
                return self.addr

        def fake_export(t):
            if rank == failing_rank and fail_at == "export":
                raise RuntimeError("cannot export")
            return (bytes([rank]) * 64, t.addr)

        def fake_open(handle, offset):
            if rank == failing_rank and fail_at == "open":
                raise RuntimeError("no peer access")
            return 1_000_000 * (handle[0] + 1) + offset

        ops.ipc_export, ops.ipc_open = fake_export, fake_open
        tensors = dict(g=FakeTensor(16 + rank), p=FakeTensor(32 + rank), c=None, flags=FakeTensor(48 + rank))
        peers, err = exchange_peer_pointers(tensors, None)
        ok = torch.tensor([0 if peers is None else 1])
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        res = dict(ok=int(ok.item()), err=None if err is None else str(err),
                   ptrs=None if peers is None else {k: (v.ptrs if v is not None else None) for k, v in peers.items()})
        torch.save(res, os.path.join(outdir, f"rank{rank}.pt"))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("fail_at", [None, "export", "open"])
def test_peer_pointer_exchange_two_ranks_gloo(fail_at):
    import tempfile
    ctx = mp.get_context("spawn")
    port = 31500 + os.getpid() % 2000 + {None: 0, "export": 1, "open": 2}[fail_at]
    with tempfile.TemporaryDirectory() as outdir:
        procs = [ctx.Process(target=_ipc_worker, args=(r, 2, port, outdir, 1, fail_at)) for r in range(2)]
        for p in procs:
            p.start()
        for p in procs:
            p.join(timeout=180)
            assert p.exitcode == 0  # in particular: nobody hangs when one rank fails
        got = {r: torch.load(os.path.join(outdir, f"rank{r}.pt")) for r in range(2)}
    if fail_at is None:
        assert got[0]["ok"] == got[1]["ok"] == 1
        # own address at [rank], the peer's mapped address (fake base of the OTHER rank + its offset) elsewhere; None passes through
        assert got[0]["ptrs"]["g"] == [16, 2_000_000 + 17] and got[1]["ptrs"]["g"] == [1_000_000 + 16, 17]
        assert got[0]["ptrs"]["flags"] == [48, 2_000_000 + 49] and got[0]["ptrs"]["c"] is None
    else:
        assert got[0]["ok"] == got[1]["ok"] == 0  # both fall back together
        assert got[1]["err"] is not None


# ---------------------------------------------------------------------------------------------
# SURVEY.md §8f rank 1-2: LR schedule, checkpoint format
# ---------------------------------------------------------------------------------------------
class _GradualWarmupRestated(torch.optim.lr_scheduler._LRScheduler):
    """Test-side restatement of ildoonet/pytorch-gradual-warmup-lr (git HEAD; the dependency the reference installs in
    setup.sh:5 and calls at network.py:116-121; not vendored, no network here): warmup_scheduler/scheduler.py's published
    algorithm, kept line by line so that torch's real CosineAnnealingLR is what runs after the warm-up."""

    def __init__(self, optimizer, multiplier, total_epoch, after_scheduler=None):
        self.multiplier = multiplier
        self.total_epoch = total_epoch
        self.after_scheduler = after_scheduler
        self.finished = False
        super().__init__(optimizer)

    def get_lr(self):
        if self.last_epoch > self.total_epoch:
            if self.after_scheduler:
                if not self.finished:
                    self.after_scheduler.base_lrs = [base_lr * self.multiplier for base_lr in self.base_lrs]
                    self.finished = True
                return self.after_scheduler.get_last_lr()
            return [base_lr * self.multiplier for base_lr in self.base_lrs]
        if self.multiplier == 1.0:
            return [base_lr * (float(self.last_epoch) / self.total_epoch) for base_lr in self.base_lrs]
        return [base_lr * ((self.multiplier - 1.0) * self.last_epoch / self.total_epoch + 1.0) for base_lr in self.base_lrs]

    def step(self, epoch=None, metrics=None):
        if self.finished and self.after_scheduler:
            self.after_scheduler.step(None)
            self._last_lr = self.after_scheduler.get_last_lr()
        else:
            return super().step(epoch)


@pytest.mark.parametrize("base_lr,min_lr,max_epochs,warmup", [(1e-3, 1e-5, 100, 5), (5e-4, 0.0, 30, 1), (1e-3, 1e-5, 12, 3)])
def test_warmup_cosine_matches_the_reference_schedulers(base_lr, min_lr, max_epochs, warmup):
    import warnings
    import vit_cifar_b200 as vb
    p = torch.nn.Parameter(torch.zeros(1))
    opt = torch.optim.Adam([p], lr=base_lr)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        base = torch.optim.lr_scheduler.CosineAnnealingLR(opt, T_max=max_epochs, eta_min=min_lr)      # network.py:113-115
        sched = _GradualWarmupRestated(opt, multiplier=1.0, total_epoch=warmup, after_scheduler=base)  # network.py:116-121
        ours = vb.WarmupCosine(base_lr, min_lr, max_epochs, warmup)
        for epoch in range(max_epochs):
            lr_ref = opt.param_groups[0]["lr"]            # the LR Lightning trains epoch `epoch` with
            assert ours(epoch) == pytest.approx(lr_ref, rel=1e-9, abs=1e-15), epoch
            opt.step()
            sched.step()                                  # Lightning: once per epoch


def test_checkpoint_format_round_trip(tmp_path):
    """main.py:234-237 writes {'state_dict': {'model.<name>': tensor}, 'hyper_parameters': {...}}; run_model.py:12-37 reads it
    with strict=False.  Same keys as the reference model -> interchangeable both ways."""
    import vit_cifar_b200 as vb
    kw = dict(img_size=32, patch=4, num_layers=2, hidden=128, mlp_hidden=128, head=4)
    torch.manual_seed(3)
    a = vb.ViT(3, 10, **kw)
    hp = {"model_name": "vit", "lr": 1e-3, **kw}
    path = tmp_path / "m.ckpt"
    vb.save_checkpoint(a, str(path), hp)
    raw = torch.load(str(path), map_location="cpu")
    assert set(raw) == {"state_dict", "hyper_parameters"} and raw["hyper_parameters"] == hp
    assert all(k.startswith("model.") for k in raw["state_dict"])
    if reference_available():  # a reference ViT accepts the stripped keys, strictly
        ref_vit, _, _ = import_reference()
        ref = ref_vit.ViT(3, 10, **kw)
        ref.load_state_dict({k[len("model."):]: v for k, v in raw["state_dict"].items()}, strict=True)
    torch.manual_seed(4)
    b = vb.ViT(3, 10, **kw)
    res = vb.load_checkpoint(b, str(path))
    assert not res.missing_keys and not res.unexpected_keys
    for (ka, va), (kb, vb_) in zip(a.state_dict().items(), b.state_dict().items()):
        assert ka == kb and torch.equal(va, vb_)
    # extra keys of a larger LightningModule (criterion buffers, ...) are ignored with strict=False
    raw["state_dict"]["criterion.weight"] = torch.zeros(3)
    res = vb.load_checkpoint(b, raw, strict=False)
    assert res.unexpected_keys == ["criterion.weight"]


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the arm the driver runs beside ours): one JSON line with the contract's keys, the reference's CPU
    path timed on a bounded sample; rank != 0 exits silently."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1]
    d = json.loads(line)
    assert d["impl"] == "reference" and d["unit"] == "img/s" and d["higher_is_better"] is True and d["value"] > 0
    for k in ("metric", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    # "reference" when a copy of the reference's own modules is reachable (VITB_REFERENCE_ROOT or oracle/_ref), else the port
    from oracle import ref_shim
    assert d["cpu_baseline"]["kind"] == ("reference" if ref_shim.reference_available() else "port")
    assert d["cpu_baseline"]["cores"] >= 1 and "sample" in d["cpu_baseline"]
    assert "bf16" not in d["config"]["workload"] and d["config"]["per_step_batch"] == 128  # the arm says what it actually ran
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    r2 = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1"],
                        capture_output=True, text=True, timeout=600, env=env)
    assert r2.returncode == 0 and not [ln for ln in r2.stdout.splitlines() if ln.startswith("{")]


def test_fused_dp_slices_partition_the_flat_buffer():
    """vitb_dp_reduce_adam's ownership rule (parallel.owned_slice mirrors the C side): float4-aligned, disjoint, covering, in rank order."""
    from vit_cifar_b200.parallel import owned_slice
    import vit_cifar_b200 as vb
    n_model = vb.ViT(3, 10, img_size=32, patch=8, num_layers=7, hidden=384, mlp_hidden=384, head=12)._layout().active_end
    for n in (n_model, 64, 4, 6_268_864):
        assert n % 4 == 0
        for world in (1, 2, 3, 4, 8):
            edges = [owned_slice(n, r, world) for r in range(world)]
            assert edges[0][0] == 0 and edges[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(edges, edges[1:]))
            assert all(lo % 4 == 0 and hi % 4 == 0 and lo <= hi for lo, hi in edges)
            assert max(hi - lo for lo, hi in edges) - min(hi - lo for lo, hi in edges[:-1] or edges) <= 4 * world or world == 1 or n < 64


def test_weight_gradient_split_plan_follows_the_measured_rule():
    """Host-side plan of the tensor-core weight gradients (csrc/gemm_tc.cu: wgrad_tc_plan): short reductions get 8-12 splits per
    output tile (profiles/r2_wgrad_splits_ab.md), the benchmark size keeps one work item per SM."""
    import ctypes
    import vit_cifar_b200  # noqa: F401
    from vit_cifar_b200 import _lib
    lib = ctypes.CDLL(_lib.LIB_PATH)
    f = lib.vitb_debug_wgrad_splits
    f.restype = ctypes.c_int
    f.argtypes = [ctypes.c_int] * 3
    rows = lambda B, T: B * T  # noqa: E731
    assert f(rows(128, 65), 384, 384) == 8          # 130 k-blocks of 64 rows
    assert f(rows(256, 65), 384, 384) == 10         # 260
    assert f(rows(1024, 17), 384, 384) == 11        # 272
    assert f(rows(512, 65), 384, 384) == 12         # 520
    assert f(rows(1024, 65), 384, 384) == 24        # 1040: 148 SMs / 6 tiles
    assert f(rows(128, 17), 384, 384) == 7          # 34 k-blocks: 8 asked for, 5 k-blocks each -> 7 items
    assert f(100, 384, 384) == 2                    # never more splits than k-blocks
    assert 1 <= f(rows(1024, 65), 1152, 384) <= 12  # wide output (27 tiles of 128 x 128, two streams): 148 * 2 / 27
    assert f(rows(128, 65), 100, 384) == 0          # not a tensor-core shape (N % 128 != 0)


def test_committed_evidence_lines_carry_the_bench_contract():
    """The bench lines committed under profiles/ (what DESIGN.md quotes) have every key of the bench.py contract, with sane values:
    a kernel-only number, an end-to-end number below it with real host<->device bytes, a measured roofline and clean clocks."""
    import glob
    import json
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    files = sorted(glob.glob(os.path.join(root, "profiles", "r2_evidence_bench*.json")))
    assert len(files) >= 6
    for f in files:
        d = json.load(open(f))
        if d.get("impl") == "reference":
            assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["e2e"]["h2d_bytes_per_step"] == 0 and d["value"] > 0
            continue
        for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
                  "data", "config", "e2e", "gpu_launches", "clocks", "roofline", "step_ms"):
            assert k in d, (f, k)
        assert d["unit"] == "img/s" and d["dtype"] == "bf16" and d["higher_is_better"] is True and d["data"] == "synthetic"
        assert d["warmup"] >= 3 and "workload" in d["config"] and "model" not in d["config"]
        e = d["e2e"]
        assert 0 < e["value"] <= d["value"] * 1.02 and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0
        assert d["gpu_launches"] >= 100 * d["steps"]          # > 100 of our kernels per step, counted by the library
        r = d["roofline"]
        assert r["bound"] in ("hbm", "tensor") and 0 < r["frac"] < 1 and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-6
        bad = {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
        assert not bad & set(d["clocks"]["reasons"]), (f, d["clocks"])
        assert d["step_ms"]["p10"] <= d["step_ms"]["p50"] <= d["step_ms"]["p90"]


def test_bench_output_dump_fits_its_budget_with_a_fixed_sample(tmp_path):
    """bench.py --dump-outputs: small arrays are written whole, large ones as the values at seeded positions that are the same on
    every run, and the files together stay below 64 MB."""
    import numpy as np
    import bench
    rng = np.random.default_rng(1)
    arrays = {"loss": np.float32(2.5), "logits": rng.standard_normal((1024, 10)),
              "params": rng.standard_normal(12_000_000, dtype=np.float32), "grads": rng.standard_normal(12_000_000, dtype=np.float32)}
    bench.dump_outputs(str(tmp_path / "a"), arrays)
    bench.dump_outputs(str(tmp_path / "b"), arrays)
    sizes = 0
    for name, a in arrays.items():
        got, again = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")
        assert got.dtype == np.float32 and np.array_equal(got, again)
        sizes += os.path.getsize(tmp_path / "a" / f"{name}.npy")
        if name in ("loss", "logits"):
            assert np.array_equal(got, np.asarray(a, dtype=np.float32))
        else:
            assert 0 < got.size < a.size and np.isin(got, a).all()
    assert 50_000_000 < sizes <= 64_000_000
