"""CPU: the restated AutoAugment tables (vit-cifar_b200/autoaugment.py), GpuAugment's random draws, the host-side argument checks of
vitb_augment_autoaugment, and the oracle (oracle/autoaugment_oracle.py) against the reference's own autoaugment.py when its source
is available."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import autoaugment_oracle as aao

T = aao.tables

# torchvision's names for the reference's ops (torchvision/transforms/autoaugment.py, AutoAugment._get_policies)
TV_NAME = {"shearX": "ShearX", "shearY": "ShearY", "translateX": "TranslateX", "translateY": "TranslateY", "rotate": "Rotate", "color": "Color",
           "posterize": "Posterize", "solarize": "Solarize", "contrast": "Contrast", "sharpness": "Sharpness", "brightness": "Brightness",
           "autocontrast": "AutoContrast", "equalize": "Equalize", "invert": "Invert"}
NO_MAGNITUDE = {"autocontrast", "equalize", "invert"}


@pytest.mark.parametrize("name,tv", [("cifar10", "CIFAR10"), ("svhn", "SVHN")])
def test_policy_tables_match_torchvision(name, tv):
    """Both come from the AutoAugment paper: same ops, probabilities and magnitude bins (torchvision has no bin for magnitude-free ops)."""
    from torchvision.transforms import autoaugment as tva
    want = tva.AutoAugment(getattr(tva.AutoAugmentPolicy, tv))._get_policies(getattr(tva.AutoAugmentPolicy, tv))
    got = T.POLICIES[name]
    assert len(got) == len(want) == 25
    for sub_got, sub_want in zip(got, want):
        for (op, p, idx), (tv_op, tv_p, tv_idx) in zip(sub_got, sub_want):
            assert TV_NAME[op] == tv_op and p == tv_p
            assert (tv_idx is None) if op in NO_MAGNITUDE else (idx == tv_idx)


def test_ranges_are_the_reference_formulas():
    lin = lambda a, b: [a + (b - a) * k / 9 for k in range(10)]  # noqa: E731
    for op in ("shearX", "shearY"):
        np.testing.assert_allclose(T.RANGES[op], lin(0, 0.3), rtol=0, atol=1e-15)
    for op in ("translateX", "translateY"):
        np.testing.assert_allclose(T.RANGES[op], lin(0, 150 / 331), rtol=0, atol=1e-15)
    np.testing.assert_allclose(T.RANGES["rotate"], lin(0, 30), rtol=0, atol=1e-13)
    for op in ("color", "contrast", "sharpness", "brightness"):
        np.testing.assert_allclose(T.RANGES[op], lin(0, 0.9), rtol=0, atol=1e-15)
    assert list(T.RANGES["posterize"]) == [8, 8, 7, 7, 6, 6, 5, 5, 4, 4]
    assert T.RANGES["solarize"][0] == 256.0 and T.RANGES["solarize"][-1] == 0.0
    np.testing.assert_allclose(T.RANGES["solarize"], lin(256, 0), rtol=0, atol=1e-12)
    assert [T.OP_CODE[o] for o in T.OPS] == list(range(14)) and set(T.RANGES) == set(T.OPS)
    assert T.SIGNED == {"shearX", "shearY", "translateX", "translateY", "color", "contrast", "sharpness", "brightness"}


def test_kernel_table_layout():
    ids, mags, probs = T.kernel_table("cifar10")
    assert len(ids) == len(mags) == len(probs) == 50
    assert (ids[2], mags[2], probs[2]) == (T.OP_CODE["rotate"], float(T.RANGES["rotate"][2]), 0.7)
    assert (ids[3], probs[3]) == (T.OP_CODE["translateX"], 0.3)


def _draw_before_policies(gen, B, padding, flip):
    """GpuAugment.draw as it was before AutoAugment (pinned: the draws of policy=None must not change)."""
    hi = 2 * padding + 1
    dx = torch.randint(0, hi, (B,), generator=gen, dtype=torch.int32)
    dy = torch.randint(0, hi, (B,), generator=gen, dtype=torch.int32)
    fl = (torch.rand((B,), generator=gen) < 0.5).to(torch.uint8) if flip else None
    return dx, dy, fl


@pytest.mark.parametrize("flip", [True, False])
def test_no_policy_draws_are_unchanged(flip):
    from vit_cifar_b200.schedule import GpuAugment
    aug = GpuAugment(32, 4, flip=flip, seed=7, device="cpu")
    ref = torch.Generator().manual_seed(7)
    for B in (5, 300):
        got, want = aug.draw(B, "cpu"), _draw_before_policies(ref, B, 4, flip)
        assert len(got) == 3
        for g, w in zip(got, want):
            assert (g is None and w is None) or torch.equal(g, w)


def test_policy_draws_extend_the_crop_draws():
    """With a policy, dx / dy / flip are the same draws as without one; the code follows them."""
    from vit_cifar_b200.schedule import GpuAugment
    a0 = GpuAugment(32, 4, seed=3, device="cpu")
    a1 = GpuAugment(32, 4, seed=3, device="cpu", policy="cifar10")
    dx0, dy0, fl0 = a0.draw(4000, "cpu")
    dx1, dy1, fl1, code = a1.draw(4000, "cpu")
    assert torch.equal(dx0, dx1) and torch.equal(dy0, dy1) and torch.equal(fl0, fl1)
    assert code.dtype == torch.int32 and int(code.min()) >= 0 and int(code.max()) < 1 << 12
    sub = code & 0xFF
    assert int(sub.max()) == 24 and int(sub.min()) == 0
    # sub-policy 14 has p2 = 0.0 (invert): its second gate never opens
    assert not bool(((code >> 9) & 1)[sub == 14].any())
    with pytest.raises(ValueError):
        GpuAugment(device="cpu", policy="imagenet")


def test_augment_autoaugment_rejects_bad_arguments_on_the_host():
    """The argument checks run before any device work (no GPU needed): table size, op codes, posterize bits, image size."""
    import vit_cifar_b200 as vb
    from vit_cifar_b200 import _lib
    if not __import__("os").path.exists(_lib.LIB_PATH):
        pytest.skip("library not built")
    lib = vb.load_library()
    f3 = (C.c_float * 3)(0.5, 0.5, 0.5)
    fake = 256  # never dereferenced: every call below fails its checks before the launch

    def call(ids, mags, n_sub, S=32, std=f3):
        n = max(len(ids), 1)
        return lib.vitb_augment_autoaugment(fake, None, None, None, fake, (C.c_int32 * n)(*ids), (C.c_double * n)(*mags), n_sub, f3, std,
                                            fake, 4, S, 4, None)

    assert call([0, 1], [0.1, 0.1], 0) < 0 and b"n_sub" in lib.vitb_last_error()
    assert call([0] * 66, [0.1] * 66, 33) < 0 and b"n_sub" in lib.vitb_last_error()
    assert call([0, 14], [0.1, 0.0], 1) < 0 and b"unknown op code 14" in lib.vitb_last_error()
    assert call([-1, 0], [0.1, 0.0], 1) < 0 and b"unknown op code" in lib.vitb_last_error()
    assert call([6, 0], [9.0, 0.0], 1) < 0 and b"posterize" in lib.vitb_last_error()
    assert call([0, 0], [float("nan"), 0.0], 1) < 0 and b"finite" in lib.vitb_last_error()
    assert call([0, 0], [0.1, 0.1], 1, S=65) < 0 and b"S <= 64" in lib.vitb_last_error()
    assert call([0, 0], [0.1, 0.1], 1, std=(C.c_float * 3)(0.5, 0.0, 0.5)) < 0 and b"zero std" in lib.vitb_last_error()


def test_oracle_crop_flip_is_the_existing_oracles():
    """autoaugment_oracle with no op applied is oracle.augment_crop_flip_normalize."""
    import oracle
    g = torch.Generator().manual_seed(0)
    img = torch.randint(0, 256, (6, 32, 32, 3), generator=g, dtype=torch.uint8)
    dx = torch.randint(0, 9, (6,), generator=g); dy = torch.randint(0, 9, (6,), generator=g); fl = torch.randint(0, 2, (6,), generator=g)
    mean, std = (0.4914, 0.4822, 0.4465), (0.2470, 0.2435, 0.2616)
    code = torch.arange(6) % 25
    got = aao.autoaugment_normalize(img, dx, dy, fl, code, T.CIFAR10_POLICY, mean, std, 4)
    want = oracle.augment_crop_flip_normalize(img, dx, dy, fl, mean, std, 4)
    assert torch.equal(got, want)


# ---------------------------------------------------------------------------------------------
# live reference: the reference's CIFAR10Policy / SVHNPolicy with scripted random draws vs the oracle, bit for bit
# ---------------------------------------------------------------------------------------------
class _Script:
    """Stands in for the `random` module inside the reference's autoaugment.py: returns the scripted values in order."""

    def __init__(self, randoms=(), choices=(), randints=()):
        self.randoms, self.choices, self.randints = list(randoms), list(choices), list(randints)

    def random(self):
        return self.randoms.pop(0)

    def choice(self, seq):
        assert list(seq) == [-1, 1]
        return self.choices.pop(0)

    def randint(self, a, b):
        return self.randints.pop(0)


def _gate_value(p, on):
    """A random.random() value that opens (on) or closes the gate `random.random() < p`, just either side of p."""
    return float(np.nextafter(p, -1.0)) if on else float(p)


@pytest.mark.skipif(aao.reference_autoaugment_path() is None, reason="the reference's autoaugment.py is not available (VITB_REFERENCE_ROOT, oracle/_ref or baseline/_ref)")
@pytest.mark.parametrize("name", ["cifar10", "svhn"])
def test_oracle_matches_live_reference_policies(name, monkeypatch):
    from PIL import Image
    ref = aao.import_reference_autoaugment()
    policy = (ref.CIFAR10Policy if name == "cifar10" else ref.SVHNPolicy)()
    table = T.POLICIES[name]
    assert len(policy.policies) == len(table)
    rng = np.random.default_rng(0)
    images = [rng.integers(0, 256, (32, 32, 3), dtype=np.uint8) for _ in range(2)]
    images.append(np.full((32, 32, 3), 77, np.uint8))
    images.append(np.where(rng.random((32, 32, 1)) < 0.5, 40, 200).astype(np.uint8).repeat(3, -1))
    checked = 0
    for i, sub in enumerate(table):
        (op1, p1, _), (op2, p2, _) = sub
        for g1 in (False, True):
            for g2 in (False, True):
                if (g1 and p1 == 0.0) or (g2 and p2 == 0.0):
                    continue   # a gate with p = 0 never opens
                for s1 in (-1, 1):
                    for s2 in (-1, 1):
                        choices = ([s1] if g1 and op1 in T.SIGNED else []) + ([s2] if g2 and op2 in T.SIGNED else [])
                        for img in images:
                            script = _Script([_gate_value(p1, g1), _gate_value(p2, g2)], choices, [i])
                            monkeypatch.setattr(ref, "random", script)
                            got = np.asarray(policy(Image.fromarray(img)))
                            assert not script.randoms and not script.choices and not script.randints
                            want = np.asarray(aao.sub_policy(Image.fromarray(img), sub, (g1, g2), (s1, s2)))
                            assert np.array_equal(got, want), (name, i, sub, g1, g2, s1, s2)
                            checked += 1
    assert checked > 25 * 4
