"""CPU: RandomCropPaste's fp64 closed form against the reference's code run on real torch tensors with scripted draws (and against the
live reference where its source is present), the torch box derivation of GpuAugment.draw_crop_paste against the reference's
_rand_bbox, the C ABI entry and its wrapper's checks, GpuAugment's generator use, and tools/train.py's SVHN reader and flags.
No device work."""
import itertools
import os
import re
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import crop_paste_ref as R  # noqa: E402
import vit_cifar_b200 as vb  # noqa: E402
from oracle.ref_shim import SKIP_REASON, import_reference, reference_available  # noqa: E402
from vit_cifar_b200.schedule import crop_paste_box  # noqa: E402

# the reference's `img[...] *= float64 array` goes through numpy's __array_wrap__, which numpy 2 warns about
pytestmark = pytest.mark.filterwarnings("ignore:__array_wrap__:DeprecationWarning")


def image(S, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(3, S, S, generator=g) * 1.7 + 0.3


def box_cases(S):
    """(lam, cx, cy, x1, y1) scripts covering empty boxes, boxes on every edge, full-width boxes and overlapping front / paste boxes;
    x1 / y1 = None picks the last legal corner (S - fw - 1)."""
    lam_half = 1 - 0.5 ** 2  # cut = S / 2 (rounded down)
    cases = [
        (0.999999, S // 2, S // 2, 0, 0),          # cut <= 1: empty box, only the flip
        (1 - 2.0 ** -53, 0, S - 1, 3, S - 1),      # empty
        (lam_half, 0, 0, 0, 0),                    # top-left corner, clipped; paste over the front box
        (lam_half, S - 1, S - 1, None, None),      # bottom-right corner, clipped; paste at the last legal corner
        (lam_half, 0, S - 1, None, 0),             # left / bottom edges
        (lam_half, S - 1, 0, 0, None),             # right / top edges
        (0.0, 1, S - 2, 0, 0),                     # lam = 0: the largest cut, clipped on one side
        (0.3, S // 2, S // 3, S // 5, S // 4),     # overlapping, shifted
        (0.75, S // 2 - 1, S // 2 + 1, None, 1),
        (0.97, 3, S - 4, 1, None),                 # small box
    ]
    out = []
    for lam, cx, cy, x1, y1 in cases:
        p = R.reference_params(S, lam, cx, cy, 0, 0, 0, 0)
        fw, fh = p[2], p[3]
        if fw == S or fh == S:
            continue
        out.append((lam, cx, cy, S - fw - 1 if x1 is None else min(x1, S - fw - 1), S - fh - 1 if y1 is None else min(y1, S - fh - 1)))
    return out


@pytest.mark.parametrize("S", [17, 32, 64])
@pytest.mark.parametrize("flip_front,flip_img", list(itertools.product([False, True], repeat=2)))
@pytest.mark.parametrize("a_kind", ["zero", "one", "random"])
def test_closed_form_equals_the_reference_code_with_scripted_draws(S, flip_front, flip_img, a_kind):
    rng = np.random.default_rng(S * 7 + flip_front * 2 + flip_img)
    cases = box_cases(S)
    assert len(cases) >= 8
    for k, (lam, cx, cy, x1, y1) in enumerate(cases):
        a = {"zero": 0.0, "one": 1.0, "random": float(rng.random())}[a_kind]
        img = image(S, k)
        with R.Scripted(lam, cx, cy, x1, y1, flip_front, flip_img, a):
            ref = R.RandomCropPaste(S)(img.clone())
        params = torch.tensor([R.reference_params(S, lam, cx, cy, x1, y1, flip_front, flip_img)], dtype=torch.int32)
        got = R.closed_form(img[None], params, torch.tensor([a], dtype=torch.float64))[0]
        assert ref.dtype == torch.float32 and torch.equal(got.view(torch.int32), ref.view(torch.int32)), (S, k)


def test_scripted_cases_cover_what_they_claim():
    for S in (17, 32, 64):
        rows = [R.reference_params(S, lam, cx, cy, x1, y1, 0, 0) for lam, cx, cy, x1, y1 in box_cases(S)]
        assert any(r[2] == 0 or r[3] == 0 for r in rows)                                   # empty
        assert any(r[0] == 0 for r in rows) and any(r[1] == 0 for r in rows)               # left / top edges
        assert any(r[0] + r[2] == S for r in rows) and any(r[1] + r[3] == S for r in rows)  # right / bottom edges
        assert any(r[4] + r[2] == S - 1 for r in rows) and any(r[4] == 0 for r in rows)    # last and first paste corners
        assert any(r[2] and r[3] and max(r[0], r[4]) < min(r[0], r[4]) + r[2] and max(r[1], r[5]) < min(r[1], r[5]) + r[3] for r in rows)


def test_the_fp64_blend_is_not_the_fp32_one():
    """The closed form's fp64 arithmetic matters: the fp32 blend differs in the last bit for some pixels."""
    S = 32
    img = image(S, 3)[None]
    params = torch.tensor([[0, 0, S // 2, S // 2, 3, 5, 0, 0]], dtype=torch.int32)
    a = 0.3141592653589793
    got = R.closed_form(img, params, torch.tensor([a], dtype=torch.float64))
    region = img[:, :, 5:5 + S // 2, 3:3 + S // 2]
    f32 = region * np.float32(a) + img[:, :, :S // 2, :S // 2] * np.float32(1 - a)
    assert not torch.equal(got[:, :, 5:5 + S // 2, 3:3 + S // 2], f32)


def test_lam_zero_full_box_is_the_documented_deviation():
    """fw == S: the reference's randint(0, 0) raises; the device derivation pastes at 0."""
    S = 32
    with pytest.raises(ValueError):
        with R.Scripted(0.0, S // 2, S // 2, 0, 0, False, False, 0.5):
            R.RandomCropPaste(S)(image(S, 0))
    box = crop_paste_box(S, torch.tensor([0.0], dtype=torch.float64), torch.tensor([S // 2]), torch.tensor([S // 2]),
                         torch.tensor([1 - 2.0 ** -53], dtype=torch.float64), torch.tensor([0.5], dtype=torch.float64))
    assert box.tolist() == [[0, 0, S, S, 0, 0]]


@pytest.mark.skipif(not reference_available(), reason=SKIP_REASON)
@pytest.mark.parametrize("S", [17, 32])
def test_restatement_matches_live_reference(S):
    """da.RandomCropPaste with seeded numpy / torch against the restatement with the same seeds, bit for bit."""
    import_reference()
    import da as ref_da  # the reference's module (sys.path set by import_reference)
    for seed in range(20):
        img = image(S, seed)
        np.random.seed(seed); torch.manual_seed(seed)
        ref = ref_da.RandomCropPaste(size=S)(img.clone())
        np.random.seed(seed); torch.manual_seed(seed)
        ours = R.RandomCropPaste(S)(img.clone())
        assert torch.equal(ref.view(torch.int32), ours.view(torch.int32)), seed


def lam_grid(S):
    """0, 1 - 2^-53, and the lam of every cut step k (S sqrt(1 - lam) = k) with its two neighbouring doubles."""
    out = [0.0, 1 - 2.0 ** -53, 0.5, 0.123456789]
    for k in range(S + 1):
        lam = 1.0 - (k / S) ** 2
        out += [lam, np.nextafter(lam, 0.0), np.nextafter(lam, 1.0)]
    return [v for v in out if 0.0 <= v < 1.0]


@pytest.mark.parametrize("S", [17, 32, 64])
def test_torch_box_derivation_equals_rand_bbox_and_the_randint_ranges(S):
    lams = lam_grid(S)
    cs = [0, 1, S // 2, S - 2, S - 1]
    rows = [(lam, cx, cy) for lam in lams for cx in cs for cy in cs[::2]]
    lam_t = torch.tensor([r[0] for r in rows], dtype=torch.float64)
    cx_t, cy_t = torch.tensor([r[1] for r in rows]), torch.tensor([r[2] for r in rows])
    n = len(rows)
    for u in (0.0, 0.5, 1 - 2.0 ** -53):
        ux = torch.full((n,), u, dtype=torch.float64)
        box = crop_paste_box(S, lam_t, cx_t, cy_t, ux, ux.flip(0))
        assert box.dtype == torch.int32 and box.shape == (n, 6)
        for i, (lam, cx, cy) in enumerate(rows):
            ref = R.reference_params(S, lam, cx, cy, 0, 0, 0, 0)
            assert box[i, :4].tolist() == ref[:4], (lam, cx, cy)
            for corner, width in ((int(box[i, 4]), ref[2]), (int(box[i, 5]), ref[3])):
                if width == S:
                    assert corner == 0  # the documented deviation
                else:
                    assert 0 <= corner < S - width  # randint(0, high=S - width)
        if u == 1 - 2.0 ** -53:  # the largest uniform reaches the last corner the reference can draw
            w = box[:, 2]
            assert torch.equal(box[:, 4][w < S], (S - 1 - w)[w < S])
    # the cut steps are really crossed: every width 0..S occurs for a centred box
    widths = crop_paste_box(S, torch.tensor(lams, dtype=torch.float64), torch.full((len(lams),), S // 2), torch.full((len(lams),), S // 2),
                            torch.zeros(len(lams), dtype=torch.float64), torch.zeros(len(lams), dtype=torch.float64))[:, 2]
    assert set(widths.tolist()) == {min(S // 2 + k // 2, S) - max(S // 2 - k // 2, 0) for k in range(S + 1)}


def test_new_entry_point_is_declared_and_bound():
    from vit_cifar_b200 import _lib
    name = "vitb_random_crop_paste"
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "vitb200.h")).read(), flags=re.S)
    proto = re.search(rf"\bint {name}\((.*?)\);", src, flags=re.S).group(1)
    assert name in _lib.SIGNATURES and len(_lib.SIGNATURES[name][1]) == len(proto.split(",")) == 6


def _cp_args(B=3, S=8):
    return dict(img=torch.zeros((B, 3, S, S)), params=torch.zeros((B, 8), dtype=torch.int32), alpha=torch.zeros(B, dtype=torch.float64))


@pytest.mark.parametrize("change,match", [
    (dict(img=torch.zeros((3, 3, 8, 8), dtype=torch.float64)), "float32"),
    (dict(img=torch.zeros((3, 1, 8, 8))), "float32"),
    (dict(img=torch.zeros((3, 3, 8, 7))), "float32"),
    (dict(img=torch.zeros((0, 3, 8, 8)), params=torch.zeros((0, 8), dtype=torch.int32), alpha=torch.zeros(0, dtype=torch.float64)), "non-empty"),
    (dict(img=torch.zeros((1, 3, 65, 65)), params=torch.zeros((1, 8), dtype=torch.int32), alpha=torch.zeros(1, dtype=torch.float64)), "64"),
    (dict(params=torch.zeros((3, 8), dtype=torch.int64)), "params"),
    (dict(params=torch.zeros((3, 6), dtype=torch.int32)), "params"),
    (dict(alpha=torch.zeros(3, dtype=torch.float32)), "alpha"),
    (dict(alpha=torch.zeros(4, dtype=torch.float64)), "alpha"),
    ({}, "CUDA device"),  # CPU tensors: refused before any launch
])
def test_wrapper_checks_its_arguments_before_any_launch(change, match):
    from vit_cifar_b200 import ops
    a = {**_cp_args(), **change}
    n0 = ops.launch_count()
    with pytest.raises(ValueError, match=match):
        ops.random_crop_paste(a["img"], a["params"], a["alpha"])
    assert ops.launch_count() == n0


def test_library_refuses_bad_shapes_without_launching():
    """(In a thread of its own: the library's last-error message is per thread, and other tests expect this one's to be empty.)"""
    from concurrent.futures import ThreadPoolExecutor
    from vit_cifar_b200 import _lib, ops
    lib = _lib.load()
    n0 = ops.launch_count()

    def calls():
        errors = []
        for args in ((None, 1, 1, 4, 32), (1, None, 1, 4, 32), (1, 1, None, 4, 32), (1, 1, 1, 0, 32), (1, 1, 1, 4, 0), (1, 1, 1, 4, 65)):
            assert lib.vitb_random_crop_paste(*args, None) < 0
            errors.append(lib.vitb_last_error())
        return errors

    with ThreadPoolExecutor(1) as ex:
        errors = ex.submit(calls).result()
    assert all(b"random_crop_paste" in e for e in errors) and b"S <= 64" in errors[-1]
    assert ops.launch_count() == n0


class _Recorder:
    def __init__(self, monkeypatch):
        from vit_cifar_b200 import ops
        self.calls = []
        for name in ("augment", "augment_autoaugment", "augment_gather", "augment_autoaugment_gather", "random_crop_paste"):
            monkeypatch.setattr(ops, name, lambda *a, _n=name, **k: self.calls.append(_n))


def _parent_draws(gen, B, pad, flip):
    """GpuAugment.draw without a policy, as it has always consumed its generator."""
    torch.randint(0, 2 * pad + 1, (B,), generator=gen, dtype=torch.int32)
    torch.randint(0, 2 * pad + 1, (B,), generator=gen, dtype=torch.int32)
    if flip:
        torch.rand((B,), generator=gen)


@pytest.mark.parametrize("gather", [False, True])
def test_rcpaste_false_consumes_the_generator_as_before_and_true_draws_after(monkeypatch, gather):
    rec = _Recorder(monkeypatch)
    B, S = 6, 8
    data = torch.zeros((10, S, S, 3), dtype=torch.uint8)
    kw = dict(index=torch.arange(B, dtype=torch.int32), labels=torch.zeros(10, dtype=torch.int64)) if gather else {}
    x = data if gather else data[:B]
    expect = torch.Generator().manual_seed(4)
    _parent_draws(expect, B, 4, True)
    off = vb.GpuAugment(S, 4, seed=4, device="cpu")
    off(x, **kw)
    assert torch.equal(off.gen.get_state(), expect.get_state()) and rec.calls[-1] != "random_crop_paste"
    on = vb.GpuAugment(S, 4, seed=4, device="cpu", rcpaste=True)
    on(x, **kw)
    assert rec.calls[-1] == "random_crop_paste"
    off.draw_crop_paste(B, "cpu")  # the crop-paste draws come after all the others
    assert torch.equal(on.gen.get_state(), off.gen.get_state())


def test_draw_crop_paste_shapes_and_ranges():
    S, B = 17, 4000
    aug = vb.GpuAugment(S, 4, seed=1, device="cpu", rcpaste=True)
    params, a = aug.draw_crop_paste(B, "cpu")
    assert params.dtype == torch.int32 and params.shape == (B, 8) and a.dtype == torch.float64 and a.shape == (B,) and a.is_contiguous()
    fx1, fy1, fw, fh, x1, y1, ff, fi = params.T
    assert ((fx1 >= 0) & (fw >= 0) & (fx1 + fw <= S) & (fy1 >= 0) & (fh >= 0) & (fy1 + fh <= S)).all()
    assert ((x1 >= 0) & (x1 + fw <= S) & (y1 >= 0) & (y1 + fh <= S)).all()
    assert set(ff.tolist()) == {0, 1} and set(fi.tolist()) == {0, 1} and ((a >= 0) & (a < 1)).all()


def test_rcpaste_refuses_images_over_64_pixels():
    with pytest.raises(ValueError, match="64"):
        vb.GpuAugment(65, 4, device="cpu", rcpaste=True)
    vb.GpuAugment(65, 4, device="cpu")  # without it there is no such limit


# ---------------------------------------------------------------------------------------------
# tools/train.py: the SVHN reader and the new flags
# ---------------------------------------------------------------------------------------------
def _write_svhn(root, n_train=7, n_test=5, seed=0):
    from scipy.io import savemat
    rng = np.random.default_rng(seed)
    out = {}
    for split, n in (("train", n_train), ("test", n_test)):
        X = rng.integers(0, 256, (32, 32, 3, n), dtype=np.uint8)
        y = rng.integers(1, 11, (n, 1)).astype(np.uint8)
        y[0, 0] = 10
        savemat(os.path.join(root, f"{split}_32x32.mat"), {"X": X, "y": y})
        out[split] = (X, y)
    return out


def test_svhn_reader_equals_torchvision(tmp_path, monkeypatch):
    import train
    from torchvision.datasets import SVHN
    monkeypatch.setattr(SVHN, "_check_integrity", lambda self: True)
    raw = _write_svhn(str(tmp_path))
    (xtr, ytr), (xte, yte) = train.read_svhn(str(tmp_path))
    for (x, y), split in (((xtr, ytr), "train"), ((xte, yte), "test")):
        tv = SVHN(str(tmp_path), split=split, download=False)
        assert x.dtype == np.uint8 and x.shape == (len(tv), 32, 32, 3) and x.flags.c_contiguous
        assert np.array_equal(x, tv.data.transpose(0, 2, 3, 1))
        assert y.dtype == np.int64 and np.array_equal(y, tv.labels)
        assert y[0] == 0 and set(y.tolist()) <= set(range(10))
        assert np.array_equal(y[raw[split][1][:, 0] != 10], raw[split][1][raw[split][1][:, 0] != 10, 0])
        ds = vb.DeviceDataset(tv.data, tv.labels, device="cpu")  # torchvision's CHW layout converts to the same images
        assert torch.equal(ds.images, torch.from_numpy(x))


def test_svhn_reader_names_missing_files(tmp_path):
    import train
    with pytest.raises(FileNotFoundError, match="train_32x32.mat.*test_32x32.mat"):
        train.read_svhn(str(tmp_path))
    _write_svhn(str(tmp_path))
    os.remove(tmp_path / "test_32x32.mat")
    with pytest.raises(FileNotFoundError, match="test_32x32.mat") as e:
        train.read_svhn(str(tmp_path))
    assert "train_32x32" not in str(e.value)


def test_new_train_flags_and_recipes():
    import train
    from vit_cifar_b200.schedule import CIFAR10_MEAN, CIFAR10_STD, CIFAR100_MEAN, CIFAR100_STD, SVHN_MEAN, SVHN_STD
    a = train.parse_args([])
    assert not a.rcpaste and a.dataset == "c10"
    b = train.parse_args(["--dataset", "svhn", "--rcpaste", "--autoaugment"])
    assert b.rcpaste and b.dataset == "svhn" and b.num_classes == 10 and b.experiment_name == "vit_svhn"
    assert train.augment_recipe("svhn", True) == dict(mean=SVHN_MEAN, std=SVHN_STD, flip=False, policy="svhn")
    assert train.augment_recipe("svhn", False) == dict(mean=SVHN_MEAN, std=SVHN_STD, flip=False, policy=None)
    assert train.augment_recipe("c10", True) == dict(mean=CIFAR10_MEAN, std=CIFAR10_STD, flip=True, policy="cifar10")
    assert train.augment_recipe("c100", True) == dict(mean=CIFAR100_MEAN, std=CIFAR100_STD, flip=True, policy="cifar10")
    assert train.augment_recipe("c10", False)["policy"] is None
    assert SVHN_MEAN == (0.4377, 0.4438, 0.4728) and SVHN_STD == (0.1980, 0.2010, 0.1970)
    with pytest.raises(SystemExit):
        train.parse_args(["--dataset", "svhn-extra"])
