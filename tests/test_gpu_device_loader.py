"""GPU: the index-gathered augmentation kernels against the contiguous ones on data[idx]; DeviceLoader-fed training against
host-gathered batches; TrainEngine(metrics=True) against fp64 torch; no host sync in an epoch of steps; tools/train.py end to end;
two-rank sharding (on machines with two GPUs)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MEAN, STD = (0.4914, 0.4822, 0.4465), (0.2470, 0.2435, 0.2616)


@pytest.fixture(scope="module")
def vb():
    import vit_cifar_b200 as m
    from vit_cifar_b200 import ops
    ops.require_device()
    m.set_precision("bf16")
    return m


def dataset(N, S, seed=0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randint(0, 256, (N, S, S, 3), generator=g, dtype=torch.uint8).cuda(),
            torch.randint(0, 10, (N,), generator=g, dtype=torch.int64).cuda())


def bits(t):
    return t.contiguous().view(torch.int32)


# ---------------------------------------------------------------------------------------------
# 1. gather kernels
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("policy", [None, "cifar10", "svhn"])
@pytest.mark.parametrize("flip", [True, False])
@pytest.mark.parametrize("S", [32, 17])
@pytest.mark.parametrize("kind", ["full", "one", "partial", "repeats"])
def test_gather_is_bit_exact_against_the_contiguous_kernel(vb, policy, flip, S, kind):
    N = 300
    data, labels = dataset(N, S, seed=S)
    g = torch.Generator().manual_seed(len(kind) + S)
    idx = {"full": torch.randperm(N, generator=g)[:256], "one": torch.tensor([N - 1]), "partial": torch.randperm(N, generator=g)[:77],
           "repeats": torch.tensor([5, 5, 0, 5, N - 1, 0, 17, 17])}[kind].to(torch.int32).cuda()
    a = vb.GpuAugment(S, 4, MEAN, STD, flip=flip, seed=3, policy=policy)
    b = vb.GpuAugment(S, 4, MEAN, STD, flip=flip, seed=3, policy=policy)
    ref = a(data[idx.long()])
    out, lab = b(data, index=idx, labels=labels)
    torch.cuda.synchronize()
    assert torch.equal(bits(out), bits(ref))
    assert torch.equal(lab, labels[idx.long()])


@pytest.mark.parametrize("policy", [None, "cifar10"])
def test_out_of_range_rows_are_nan_with_label_minus_one(vb, policy):
    N, S = 50, 32
    data, labels = dataset(N, S, seed=1)
    idx = torch.tensor([3, -1, 7, N, 2 ** 31 - 1, 9], dtype=torch.int32, device="cuda")
    ok = torch.tensor([0, 2, 5])
    a = vb.GpuAugment(S, 4, MEAN, STD, seed=5, policy=policy)
    b = vb.GpuAugment(S, 4, MEAN, STD, seed=5, policy=policy)
    safe = torch.where((idx >= 0) & (idx < N), idx, 0).long()
    ref = a(data[safe])
    out = torch.full((6, 3, S, S), 7.0, device="cuda")
    lab = torch.full((6,), 99, dtype=torch.int64, device="cuda")
    b(data, index=idx, labels=labels, out=out, labels_out=lab)
    torch.cuda.synchronize()
    assert torch.isnan(out[[1, 3, 4]]).all()
    assert lab[[1, 3, 4]].tolist() == [-1, -1, -1]
    assert torch.equal(bits(out[ok]), bits(ref[ok])) and torch.equal(lab[ok], labels[idx[ok].long()])


# ---------------------------------------------------------------------------------------------
# 2. DeviceLoader-fed training == host-gathered batches with the same indices and draws
# ---------------------------------------------------------------------------------------------
def small_model(vb, seed=2045, dropout=0.0):
    torch.manual_seed(seed)
    return vb.ViT(3, 10, img_size=32, patch=8, num_layers=2, hidden=128, mlp_hidden=128, head=4, dropout=dropout).cuda()


def _mix(vb, kind):
    return {"none": None, "cutmix": vb.GpuCutMix(32, 1.0), "mixup": vb.GpuMixUp(1.0)}[kind]


@pytest.mark.parametrize("use_graph", [False, True])
@pytest.mark.parametrize("mix", ["none", "cutmix", "mixup"])
def test_loader_training_equals_host_gathered_training(vb, use_graph, mix):
    N, B, policy = 300, 64, "cifar10"  # 300 = 4 * 64 + 44: the last batch is partial
    data, labels = dataset(N, 32, seed=4)
    ds = vb.DeviceDataset(data, labels)
    mixed = mix != "none"

    def engine():
        return vb.TrainEngine(small_model(vb), B, use_graph=use_graph, mixed_targets=mixed)

    # (a) DeviceLoader, two epochs
    ea = engine()
    loader = vb.DeviceLoader(ds, B, shuffle=True, seed=1, augment=vb.GpuAugment(32, 4, MEAN, STD, seed=9, policy=policy), mix=_mix(vb, mix))
    torch.manual_seed(11); np.random.seed(11)
    orders = []
    for epoch in range(2):
        loader.set_epoch(epoch)
        orders.append(loader.order())
        for batch in loader:
            ea.step(*batch)
    # (b) the same rows gathered on the host, H2D, GpuAugment on the contiguous batch, the same mix draws
    eb = engine()
    aug = vb.GpuAugment(32, 4, MEAN, STD, seed=9, policy=policy)
    mixer = _mix(vb, mix)
    host_x, host_y = data.cpu().numpy(), labels.cpu()
    torch.manual_seed(11); np.random.seed(11)
    for order in orders:
        for s in range(0, N, B):
            rows = order[s:s + B].numpy()
            x = torch.from_numpy(host_x[rows]).pin_memory().cuda(non_blocking=True)
            y = host_y[rows].pin_memory().cuda(non_blocking=True)
            img = aug(x)
            eb.step(*(mixer((img, y)) if mixer else (img, y)))
    torch.cuda.synchronize()
    assert ea.step_count == eb.step_count == 2 * 5
    for name, ta, tb in (("params", ea.P, eb.P), ("exp_avg", ea.Mo, eb.Mo), ("exp_avg_sq", ea.V, eb.V)):
        assert torch.equal(bits(ta[:ea.n]), bits(tb[:eb.n])), name


# ---------------------------------------------------------------------------------------------
# 3. the epoch record
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mix", ["none", "cutmix"])
def test_train_metrics_equal_fp64_torch(vb, mix):
    N, B = 300, 64
    data, labels = dataset(N, 32, seed=6)
    ds = vb.DeviceDataset(data, labels)
    eng = vb.TrainEngine(small_model(vb), B, use_graph=True, mixed_targets=mix != "none", metrics=True)
    loader = vb.DeviceLoader(ds, B, shuffle=True, seed=2, augment=vb.GpuAugment(32, 4, MEAN, STD, seed=1), mix=_mix(vb, mix))
    for epoch in range(2):
        loader.set_epoch(epoch)
        correct, loss_sum, n_all = 0, 0.0, 0
        for batch in loader:
            loss = eng.step(*batch)
            n = batch[0].shape[0]
            logits = eng.logits[:n].double()
            correct += int((logits.argmax(-1) == batch[1]).sum())
            loss_sum += float(loss.double()) * n
            n_all += n
        m = eng.train_metrics()
        assert m["n"] == n_all == N
        assert m["acc"] == correct / N
        assert m["loss"] == loss_sum / N
    assert eng.train_metrics()["n"] == 0  # reset by the previous call


def test_metrics_cost_two_launches_and_leave_the_default_step_alone(vb):
    B = 32
    data, labels = dataset(40, 32, seed=7)
    counts = {}
    for metrics in (False, True):
        eng = vb.TrainEngine(small_model(vb), B, use_graph=False, metrics=metrics)
        eng.step(vb.GpuAugment(32, 4, seed=1)(data[:B]), labels[:B])
        counts[metrics] = eng.launches_per_step
        if not metrics:
            with pytest.raises(RuntimeError, match="metrics=True"):
                eng.train_metrics()
        else:
            assert eng.train_metrics()["n"] == B
    assert counts[True] == counts[False] + 2


# ---------------------------------------------------------------------------------------------
# 4. no host synchronisation in an epoch of steps
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("policy", [None, "cifar10"])
def test_an_epoch_of_loader_steps_never_synchronises(vb, policy):
    N, B = 500, 128
    data, labels = dataset(N, 32, seed=8)
    ds = vb.DeviceDataset(data, labels)
    eng = vb.TrainEngine(small_model(vb), B, metrics=True)
    loader = vb.DeviceLoader(ds, B, shuffle=True, seed=0, augment=vb.GpuAugment(32, 4, MEAN, STD, seed=0, policy=policy))
    loader.set_epoch(0)
    for batch in loader:  # epoch 0: the first step captures the graph (which synchronises once)
        eng.step(*batch)
    eng.train_metrics()
    loader.set_epoch(1)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        for batch in loader:
            eng.step(*batch)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    assert eng.train_metrics()["n"] == N


# ---------------------------------------------------------------------------------------------
# 5. tools/train.py end to end
# ---------------------------------------------------------------------------------------------
TRAIN_ARGS = ["--synthetic", "2000", "--max-epochs", "2", "--warmup-epoch", "1", "--batch-size", "128", "--num-layers", "2", "--hidden", "128",
              "--mlp-hidden", "128", "--head", "4", "--label-smoothing", "--autoaugment", "--cutmix", "--seed", "3"]


def _train(out_dir):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "train.py"), *TRAIN_ARGS, "--out-dir", str(out_dir)],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-3000:])
    return [json.loads(line) for line in r.stdout.splitlines() if line.startswith("{")]


def test_train_tool_runs_reproduces_and_its_checkpoint_evaluates_as_logged(vb, tmp_path):
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import train
    logs = _train(tmp_path / "a")
    assert [r["epoch"] for r in logs] == [0, 1]
    for r in logs:
        assert all(np.isfinite(r[k]) for k in ("loss", "acc", "val_loss", "val_acc", "lr", "img_per_s"))
    assert logs[0]["lr"] == 0.0 and logs[1]["lr"] == 1e-3  # warm-up epoch 0, then the cosine schedule's first epoch
    ck_a = torch.load(tmp_path / "a" / "vit_c10.ckpt", map_location="cpu")
    assert os.path.isfile(tmp_path / "a" / "vit_c10-best.ckpt")
    model = vb.ViT(3, 10, img_size=32, patch=8, num_layers=2, hidden=128, mlp_hidden=128, head=4)
    res = vb.load_checkpoint(model, str(tmp_path / "a" / "vit_c10.ckpt"), strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    model = model.cuda()
    x, y = train.synthetic_set(400, 10, 3 + 1)
    val = vb.EvalEngine(model, 256, smoothing=0.1, mean=MEAN, std=STD).run(vb.DeviceLoader(vb.DeviceDataset(x, y), 256, shuffle=False))
    assert val["val_loss"] == logs[-1]["val_loss"] and val["val_acc"] == logs[-1]["val_acc"]
    # the same seed: the same checkpoint
    _train(tmp_path / "b")
    ck_b = torch.load(tmp_path / "b" / "vit_c10.ckpt", map_location="cpu")
    assert ck_a["state_dict"].keys() == ck_b["state_dict"].keys()
    for k in ck_a["state_dict"]:
        assert torch.equal(ck_a["state_dict"][k], ck_b["state_dict"][k]), k
    for k in ("exp_avg", "exp_avg_sq"):
        assert torch.equal(ck_a["optimizer_states"][0][k], ck_b["optimizer_states"][0][k]), k


# ---------------------------------------------------------------------------------------------
# 6. two ranks
# ---------------------------------------------------------------------------------------------
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs on one box")
def test_two_rank_loader_takes_equal_steps_and_keeps_replicas_identical():
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29581", os.path.join(ROOT, "tools", "loader_dp_check.py")], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-3000:])
    assert "loader_dp_check PASSED" in r.stdout
