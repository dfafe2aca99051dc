"""GPU: vitb_random_crop_paste bit for bit against the fp64 closed form (tests/crop_paste_ref.py), NaN images, the size bound,
GpuAugment(rcpaste=True) against GpuAugment(rcpaste=False) followed by the closed form on the parameters it drew, the statistics of
the draws, DeviceLoader epochs without host synchronisation, and tools/train.py with --rcpaste and --dataset svhn end to end."""
import itertools
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import crop_paste_ref as R  # noqa: E402

MEAN, STD = (0.4914, 0.4822, 0.4465), (0.2470, 0.2435, 0.2616)


@pytest.fixture(scope="module")
def vb():
    import vit_cifar_b200 as m
    from vit_cifar_b200 import ops
    ops.require_device()
    m.set_precision("bf16")
    return m


def same(a, b):
    """Bit-identical, except that any NaN equals any NaN (the payload of a propagated NaN is not part of the contract)."""
    a, b = a.cpu().contiguous(), b.cpu().contiguous()
    na, nb = torch.isnan(a), torch.isnan(b)
    return torch.equal(na, nb) and torch.equal(a.view(torch.int32)[~na], b.view(torch.int32)[~nb])


def crafted(S):
    """Edge, empty, full and overlapping boxes with every flip combination: int32 rows of vitb_random_crop_paste's params."""
    h = S // 2
    boxes = [
        (0, 0, 0, 0, 0, 0),                  # empty
        (2, 1, 0, h, 1, 2),                  # fw = 0
        (1, 2, h, 0, 3, 1),                  # fh = 0
        (0, 0, S, S, 0, 0),                  # the whole image (lam = 0: the reference raises, here it pastes at 0)
        (S - h, S - h, h, h, 0, 0),          # front at the bottom-right corner, pasted at the top-left
        (0, 0, h, h, S - h, S - h),          # and the other way round
        (0, S - h, h, h, S - h, 0),
        (1, 1, h, h, 2, 3),                  # overlapping
        (3, 2, h, h, 3, 2),                  # pasted where it was taken
        (S - 1, S - 1, 1, 1, S - 1, 0),      # one pixel in a corner
        (0, 0, S, 1, 0, S - 1),              # a full-width row, pasted at the bottom
        (0, 3, 1, S - 3, S - 1, 0),          # a column, pasted at the right edge
    ]
    return [list(b) + [ff, fi] for b in boxes for ff, fi in itertools.product((0, 1), repeat=2)]


def make_inputs(vb, B, S, seed):
    """img (B, 3, S, S), params (B, 8) and a (B,) on the device: crafted rows first (from an offset that depends on the seed), then
    GpuAugment's own draws; a cycles through 0, 1 and uniform values."""
    g = torch.Generator().manual_seed(seed)
    img = (torch.randn(B, 3, S, S, generator=g) * 1.5).cuda()
    rows = crafted(S)
    k = seed % len(rows)
    rows = (rows[k:] + rows[:k])[:B]
    drawn, _ = vb.GpuAugment(S, 4, seed=seed, rcpaste=True).draw_crop_paste(B, "cuda")
    params = torch.cat((torch.tensor(rows, dtype=torch.int32).view(-1, 8), drawn[len(rows):].cpu())).cuda()
    a = torch.rand(B, generator=g, dtype=torch.float64)
    a[0::3], a[1::3] = 0.0, 1.0
    return img, params.contiguous(), a.cuda()


@pytest.mark.parametrize("S", [17, 32, 64])
@pytest.mark.parametrize("B,seed", [(1, 0), (1, 13), (5, 1), (5, 22), (5, 37), (1024, 3)])
def test_kernel_is_bit_exact_against_the_closed_form(vb, B, S, seed):
    from vit_cifar_b200 import ops
    img, params, a = make_inputs(vb, B, S, seed)
    out = img.clone()
    ops.random_crop_paste(out, params, a)
    torch.cuda.synchronize()
    expect = R.closed_form(img, params, a)
    assert not torch.isnan(expect).any()
    assert same(out, expect)
    if B == 1024:  # every crafted row with every flip went through, and not every image is unchanged
        assert len(crafted(S)) < B and not torch.equal(out, img)


def test_nan_images_stay_nan_and_bad_boxes_give_nan(vb):
    from vit_cifar_b200 import ops
    S = 32
    img, params, a = make_inputs(vb, 96, S, 5)
    img[7] = float("nan")   # what the gather kernels write for a row outside the dataset
    img[50] = float("nan")
    bad = [[-1, 0, 4, 4, 0, 0, 0, 0], [0, -1, 4, 4, 0, 0, 0, 0], [30, 0, 4, 4, 0, 0, 0, 0], [0, 0, 4, 4, 29, 0, 0, 0],
           [0, 0, 4, 4, 0, 29, 0, 0], [0, 0, -2, 4, 0, 0, 0, 0], [0, 0, 4, 33, 0, 0, 0, 0], [0, 0, 4, 4, -1, 0, 1, 1]]
    params[60:60 + len(bad)] = torch.tensor(bad, dtype=torch.int32, device="cuda")
    out = img.clone()
    ops.random_crop_paste(out, params, a)
    torch.cuda.synchronize()
    nan_rows = torch.isnan(out).flatten(1).all(1).cpu()
    assert nan_rows.tolist() == [i in (7, 50) or 60 <= i < 60 + len(bad) for i in range(96)]
    assert same(out, R.closed_form(img, params, a))


def test_the_size_bound_is_enforced(vb):
    from vit_cifar_b200 import _lib, ops
    img = torch.zeros((2, 3, 65, 65), device="cuda")
    params = torch.zeros((2, 8), dtype=torch.int32, device="cuda")
    a = torch.zeros(2, dtype=torch.float64, device="cuda")
    n0 = ops.launch_count()
    with pytest.raises(ValueError, match="64"):
        ops.random_crop_paste(img, params, a)
    lib = _lib.load()
    stream = torch.cuda.current_stream().cuda_stream

    def call():  # in a thread of its own: the last-error message is per thread
        return lib.vitb_random_crop_paste(img.data_ptr(), params.data_ptr(), a.data_ptr(), 2, 65, stream), lib.vitb_last_error()

    from concurrent.futures import ThreadPoolExecutor
    with ThreadPoolExecutor(1) as ex:
        rc, err = ex.submit(call).result()
    assert rc < 0 and b"S <= 64" in err
    assert ops.launch_count() == n0
    with pytest.raises(ValueError, match="64"):
        vb.GpuAugment(65, 4, rcpaste=True)
    torch.cuda.synchronize()
    assert torch.count_nonzero(img) == 0


def dataset(N, S, seed=0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randint(0, 256, (N, S, S, 3), generator=g, dtype=torch.uint8).cuda(),
            torch.randint(0, 10, (N,), generator=g, dtype=torch.int64).cuda())


@pytest.mark.parametrize("policy", [None, "cifar10", "svhn"])
@pytest.mark.parametrize("path", ["contiguous", "gather", "gather_out_of_range"])
def test_gpu_augment_rcpaste_is_the_plain_pipeline_then_crop_paste(vb, policy, path):
    N, S, B = 300, 32, 200
    data, labels = dataset(N, S, seed=2)
    flip = policy != "svhn"
    plain = vb.GpuAugment(S, 4, MEAN, STD, flip=flip, seed=11, policy=policy)
    paste = vb.GpuAugment(S, 4, MEAN, STD, flip=flip, seed=11, policy=policy, rcpaste=True)
    if path == "contiguous":
        base = plain(data[:B])
        params, a = plain.draw_crop_paste(B, "cuda")  # the generator is where `paste` takes its crop-paste draws from
        out = paste(data[:B])
    else:
        idx = torch.randperm(N, generator=torch.Generator().manual_seed(1))[:B].to(torch.int32)
        if path == "gather_out_of_range":
            idx[[0, 17, 199]] = torch.tensor([-1, N, 2 ** 31 - 1], dtype=torch.int32)
        idx = idx.cuda()
        base, lab_a = plain(data, index=idx, labels=labels)
        params, a = plain.draw_crop_paste(B, "cuda")
        out, lab_b = paste(data, index=idx, labels=labels)
        assert torch.equal(lab_a, lab_b)
        if path == "gather_out_of_range":
            assert torch.isnan(out[[0, 17, 199]]).all() and lab_b[[0, 17, 199]].tolist() == [-1, -1, -1]
    torch.cuda.synchronize()
    expect = R.closed_form(base, params, a)
    assert same(out, expect)
    assert not same(out, base)


def test_draw_statistics(vb):
    from scipy import stats
    from vit_cifar_b200.schedule import crop_paste_box
    S, B = 32, 200_000
    aug = vb.GpuAugment(S, 4, seed=7, rcpaste=True)
    replay = torch.Generator(device="cuda")
    replay.set_state(aug.gen.get_state())
    params, a = aug.draw_crop_paste(B, "cuda")
    # the raw draws, replayed: lam, the paste-corner uniforms, the two flips and a in one float64 (B, 6) draw, then the centres
    u = torch.rand((B, 6), generator=replay, device="cuda", dtype=torch.float64)
    c = torch.randint(0, S, (B, 2), generator=replay, device="cuda")
    assert torch.equal(crop_paste_box(S, u[:, 0], c[:, 0], c[:, 1], u[:, 1], u[:, 2]), params[:, :6])
    assert torch.equal(u[:, 5], a)
    assert stats.kstest(u[:, 0].cpu().numpy(), "uniform").pvalue > 1e-4   # lam ~ Beta(1, 1)
    assert stats.kstest(a.cpu().numpy(), "uniform").pvalue > 1e-4
    assert set(c[:, 0].tolist()) == set(range(S)) and set(c[:, 1].tolist()) == set(range(S))
    p = params.cpu().long()
    fx1, fy1, fw, fh, x1, y1, ff, fi = p.T
    assert ((x1 >= 0) & (y1 >= 0)).all()
    assert (x1[fw < S] < (S - fw)[fw < S]).all() and (y1[fh < S] < (S - fh)[fh < S]).all()   # randint(0, high=S - fw)
    assert set(x1[fw == 0].tolist()) == set(range(S)) and set(y1[fh == 0].tolist()) == set(range(S))
    for flips in (ff, fi):
        assert abs(flips.double().mean().item() - 0.5) < 0.01
    # the widths follow from lam ~ U[0, 1): P(cut <= k) = ((k + 1) / S)^2, seen through unclipped boxes (fx1 > 0, fx1 + fw < S)
    cut_half = (torch.floor(S * torch.sqrt(1 - u[:, 0])).long() // 2).cpu()
    free = (fx1 > 0) & (fx1 + fw < S)
    assert torch.equal(fw[free], 2 * cut_half[free])


def small_model(vb, seed=2045):
    torch.manual_seed(seed)
    return vb.ViT(3, 10, img_size=32, patch=8, num_layers=2, hidden=128, mlp_hidden=128, head=4).cuda()


@pytest.mark.parametrize("cutmix", [False, True])
def test_an_epoch_of_rcpaste_loader_steps_never_synchronises(vb, cutmix):
    N, B = 500, 128
    data, labels = dataset(N, 32, seed=8)
    ds = vb.DeviceDataset(data, labels)
    eng = vb.TrainEngine(small_model(vb), B, metrics=True, mixed_targets=cutmix)
    aug = vb.GpuAugment(32, 4, MEAN, STD, seed=0, policy="cifar10", rcpaste=True)
    loader = vb.DeviceLoader(ds, B, shuffle=True, seed=0, augment=aug, mix=vb.GpuCutMix(32, 1.0) if cutmix else None)
    np.random.seed(0)
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
    m = eng.train_metrics()
    assert m["n"] == N and np.isfinite(m["loss"])


# ---------------------------------------------------------------------------------------------
# tools/train.py end to end
# ---------------------------------------------------------------------------------------------
SMALL = ["--max-epochs", "2", "--warmup-epoch", "1", "--batch-size", "128", "--num-layers", "2", "--hidden", "128", "--mlp-hidden", "128",
         "--head", "4", "--seed", "3"]
TIMING = ("epoch_s", "train_s", "img_per_s")


def _train(args, out_dir):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "train.py"), *args, *SMALL, "--out-dir", str(out_dir)],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-3000:])
    return [json.loads(line) for line in r.stdout.splitlines() if line.startswith("{")]


def test_train_tool_with_rcpaste_reproduces_its_runs(vb, tmp_path):
    args = ["--synthetic", "2000", "--rcpaste", "--label-smoothing"]
    a, b = _train(args, tmp_path / "a"), _train(args, tmp_path / "b")
    assert [r["epoch"] for r in a] == [0, 1]
    for r in a:
        assert all(np.isfinite(r[k]) for k in ("loss", "acc", "val_loss", "val_acc"))
    strip = lambda rs: [{k: v for k, v in r.items() if k not in TIMING} for r in rs]  # noqa: E731
    assert strip(a) == strip(b)
    ck_a = torch.load(tmp_path / "a" / "vit_c10.ckpt", map_location="cpu")
    ck_b = torch.load(tmp_path / "b" / "vit_c10.ckpt", map_location="cpu")
    assert ck_a["hyper_parameters"]["rcpaste"] is True
    for k in ck_a["state_dict"]:
        assert torch.equal(ck_a["state_dict"][k], ck_b["state_dict"][k]), k


def test_train_tool_trains_svhn_and_its_checkpoint_evaluates_as_logged(vb, tmp_path):
    from scipy.io import savemat
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import train
    from vit_cifar_b200.schedule import SVHN_MEAN, SVHN_STD
    data = tmp_path / "svhn"
    data.mkdir()
    for split, n, seed in (("train", 1500, 3), ("test", 300, 4)):
        x, y = train.synthetic_set(n, 10, seed)
        y = np.where(y == 0, 10, y).astype(np.uint8)  # SVHN stores the digit 0 as label 10
        savemat(str(data / f"{split}_32x32.mat"), {"X": np.ascontiguousarray(x.transpose(1, 2, 3, 0)), "y": y[:, None]})
    logs = _train(["--dataset", "svhn", "--data-root", str(data), "--autoaugment", "--rcpaste"], tmp_path / "out")
    assert [r["epoch"] for r in logs] == [0, 1] and all(np.isfinite(r["val_loss"]) for r in logs)
    ck = torch.load(tmp_path / "out" / "vit_svhn.ckpt", map_location="cpu")
    assert ck["hyper_parameters"]["dataset"] == "svhn"
    model = vb.ViT(3, 10, img_size=32, patch=8, num_layers=2, hidden=128, mlp_hidden=128, head=4)
    res = vb.load_checkpoint(model, ck, strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    (_, _), (xte, yte) = train.read_svhn(str(data))
    val = vb.EvalEngine(model.cuda(), 256, smoothing=0.0, mean=SVHN_MEAN, std=SVHN_STD).run(
        vb.DeviceLoader(vb.DeviceDataset(xte, yte), 256, shuffle=False))
    assert val["val_loss"] == logs[-1]["val_loss"] and val["val_acc"] == logs[-1]["val_acc"]
