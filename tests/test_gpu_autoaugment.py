"""GPU: vitb_augment_autoaugment (csrc/augment.cu) against the Pillow oracle (oracle/autoaugment_oracle.py), op by op and policy by
policy, bit for bit on the bytes before ToTensor; the unchanged crop / flip path; GpuAugment(policy=...) draw statistics."""
import math

import numpy as np
import pytest
import torch

from oracle import autoaugment_oracle as aao

pytestmark = pytest.mark.gpu

T = aao.tables
MEAN, STD = (0.4914, 0.4822, 0.4465), (0.2470, 0.2435, 0.2616)
PAD = 4


@pytest.fixture(scope="module")
def ops():
    import vit_cifar_b200  # noqa: F401
    from vit_cifar_b200 import ops as o
    o.require_device()
    return o


def sample_images(n_random=6, S=32):
    """Random images, a constant one, a two-level one and narrow-range ones (the identity branches of equalize / autocontrast)."""
    g = torch.Generator().manual_seed(0)
    imgs = [torch.randint(0, 256, (S, S, 3), generator=g, dtype=torch.uint8) for _ in range(n_random)]
    imgs.append(torch.full((S, S, 3), 93, dtype=torch.uint8))
    imgs.append(torch.where(torch.rand((S, S, 1), generator=g) < 0.3, 30, 220).to(torch.uint8).expand(S, S, 3).contiguous())
    imgs.append(torch.randint(120, 123, (S, S, 3), generator=g, dtype=torch.uint8))
    imgs.append(torch.randint(250, 256, (S, S, 3), generator=g, dtype=torch.uint8))
    return torch.stack(imgs)


def to_bytes(out):
    """The bytes before ToTensor: round((out * std + mean) * 255); one byte step is >= 0.015 after normalisation."""
    m = torch.tensor(MEAN, device=out.device).view(1, 3, 1, 1)
    s = torch.tensor(STD, device=out.device).view(1, 3, 1, 1)
    return torch.round((out * s + m) * 255).clamp(0, 255).to(torch.uint8).permute(0, 2, 3, 1).cpu()


def run(ops, img, dx, dy, fl, code, op_ids, mags):
    out = torch.empty((img.shape[0], 3, img.shape[1], img.shape[1]), device="cuda")
    ops.augment_autoaugment(img.cuda(), dx.cuda(), dy.cuda(), None if fl is None else fl.cuda(), code.cuda(), op_ids, mags, MEAN, STD, out, PAD)
    torch.cuda.synchronize()
    return out


@pytest.mark.parametrize("op", T.OPS)
def test_every_op_every_bin_both_signs_bit_exact(ops, op):
    """One-op sub-policies: table entry 2k = (op, bin k), entry 2k + 1 = invert (never gated on).  Every image of the test set x 10 bins x
    2 signs, with crop offsets and flips, against Pillow."""
    base = sample_images()
    n = base.shape[0]
    op_ids, mags, subs = [], [], []
    for k in range(10):
        op_ids += [T.OP_CODE[op], T.OP_CODE["invert"]]
        mags += [float(T.RANGES[op][k]), 0.0]
        subs.append(((op, 1.0, k), ("invert", 0.0, 0)))
    rows = [(i, k, neg) for k in range(10) for neg in (0, 1) for i in range(n)]
    B = len(rows)
    img = base[[r[0] for r in rows]]
    g = torch.Generator().manual_seed(1)
    dx = torch.randint(0, 2 * PAD + 1, (B,), generator=g, dtype=torch.int32)
    dy = torch.randint(0, 2 * PAD + 1, (B,), generator=g, dtype=torch.int32)
    fl = torch.randint(0, 2, (B,), generator=g, dtype=torch.uint8)
    code = torch.tensor([k | (1 << 8) | (neg << 10) for _, k, neg in rows], dtype=torch.int32)
    got = to_bytes(run(ops, img, dx, dy, fl, code, op_ids, mags))
    want = aao.autoaugment_bytes(img, dx, dy, fl, code, subs, PAD)
    diff = (got.int() - want.int()).abs()
    bad = [(rows[b], int(diff[b].max()), int((diff[b] > 0).sum())) for b in range(B) if diff[b].max() > 0]
    assert not bad, f"{op}: {len(bad)} of {B} images differ (row, max |d|, pixels): {bad[:8]}"


@pytest.mark.parametrize("name", ["cifar10", "svhn"])
def test_policies_bit_exact(ops, name):
    """All 25 sub-policies x 4 gate combinations x 4 sign combinations, crop offsets and flips, B = 1024; the first 400 images (every
    combination once) are checked against Pillow, and all 1024 must be finite."""
    policy = T.POLICIES[name]
    op_ids, mags, _ = T.kernel_table(name)
    B = 1024
    combos = [s | (g << 8) | (n << 10) for s in range(25) for g in range(4) for n in range(4)]
    code = torch.tensor([combos[b % len(combos)] for b in range(B)], dtype=torch.int32)
    g = torch.Generator().manual_seed(2)
    img = torch.randint(0, 256, (B, 32, 32, 3), generator=g, dtype=torch.uint8)
    img[1::7] = sample_images()[-4:].repeat(math.ceil(B / 7 / 4), 1, 1, 1)[: len(range(1, B, 7))]
    dx = torch.randint(0, 2 * PAD + 1, (B,), generator=g, dtype=torch.int32)
    dy = torch.randint(0, 2 * PAD + 1, (B,), generator=g, dtype=torch.int32)
    fl = torch.randint(0, 2, (B,), generator=g, dtype=torch.uint8)
    out = run(ops, img, dx, dy, fl, code, op_ids, mags)
    assert torch.isfinite(out).all()
    nb = len(combos)
    got = to_bytes(out[:nb])
    want = aao.autoaugment_bytes(img[:nb], dx[:nb], dy[:nb], fl[:nb], code[:nb], policy, PAD)
    bad = [(int(code[b]) & 0xFF, hex(int(code[b]))) for b in range(nb) if not torch.equal(got[b], want[b])]
    assert not bad, f"{name}: {len(bad)} of {nb} images differ: {bad[:10]}"
    # the fp32 output itself is the oracle's ToTensor + Normalize of those bytes up to one rounding
    ref = aao.autoaugment_normalize(img[:64], dx[:64], dy[:64], fl[:64], code[:64], policy, MEAN, STD, PAD)
    assert (out[:64].cpu() - ref).abs().max().item() < 1e-6


def test_gates_off_is_the_crop_flip_kernel(ops):
    """Codes with both gates off give exactly vitb_augment_crop_flip_normalize's output for the same crop / flip draws."""
    B = 777
    g = torch.Generator().manual_seed(3)
    img = torch.randint(0, 256, (B, 32, 32, 3), generator=g, dtype=torch.uint8).cuda()
    dx = torch.randint(0, 9, (B,), generator=g, dtype=torch.int32).cuda()
    dy = torch.randint(0, 9, (B,), generator=g, dtype=torch.int32).cuda()
    fl = torch.randint(0, 2, (B,), generator=g, dtype=torch.uint8).cuda()
    code = (torch.randint(0, 25, (B,), generator=g, dtype=torch.int32) | (torch.randint(0, 4, (B,), generator=g, dtype=torch.int32) << 10)).cuda()
    op_ids, mags, _ = T.kernel_table("cifar10")
    a = torch.empty((B, 3, 32, 32), device="cuda")
    b = torch.empty_like(a)
    ops.augment_autoaugment(img, dx, dy, fl, code, op_ids, mags, MEAN, STD, a, PAD)
    ops.augment(img, dx, dy, fl, MEAN, STD, b, PAD)
    assert torch.equal(a, b)
    ops.augment_autoaugment(img, None, None, None, code, op_ids, mags, MEAN, STD, a, PAD)   # no draws = centre crop, no flip
    ops.augment(img, None, None, None, MEAN, STD, b, PAD)
    assert torch.equal(a, b)


def test_other_image_sizes(ops):
    """S = 17 (odd; the rotation centre is not a pixel corner) and S = 64 (the largest accepted) against Pillow."""
    for S in (17, 64):
        g = torch.Generator().manual_seed(S)
        policy = T.CIFAR10_POLICY + T.SVHN_POLICY[:7]
        op_ids, mags, _ = T.kernel_table(policy)
        B = 128
        img = torch.randint(0, 256, (B, S, S, 3), generator=g, dtype=torch.uint8)
        dx = torch.randint(0, 9, (B,), generator=g, dtype=torch.int32)
        dy = torch.randint(0, 9, (B,), generator=g, dtype=torch.int32)
        code = torch.randint(0, 32, (B,), generator=g, dtype=torch.int32) | (torch.randint(0, 16, (B,), generator=g, dtype=torch.int32) << 8)
        out = torch.empty((B, 3, S, S), device="cuda")
        ops.augment_autoaugment(img.cuda(), dx.cuda(), dy.cuda(), None, code.cuda(), op_ids, mags, MEAN, STD, out, PAD)
        want = aao.autoaugment_bytes(img, dx, dy, None, code, policy, PAD)
        assert torch.equal(to_bytes(out), want), S


def test_gpu_augment_policy_replays_and_statistics(ops):
    """GpuAugment(policy=...) launches the kernel on its own draws (replayed through the oracle), and over 65,536 draws the sub-policy
    frequencies, gate rates and sign rates are within 5 sigma of the policy's."""
    import vit_cifar_b200 as vb
    aug = vb.GpuAugment(32, 4, MEAN, STD, flip=False, seed=5, policy="svhn")
    B = 96
    img = sample_images().repeat(10, 1, 1, 1)[:B].cuda()
    state = aug.gen.get_state()
    out = aug(img)
    aug.gen.set_state(state)
    dx, dy, fl, code = aug.draw(B, "cuda")
    assert fl is None
    want = aao.autoaugment_bytes(img.cpu(), dx.cpu(), dy.cpu(), None, code.cpu(), T.SVHN_POLICY, PAD)
    assert torch.equal(to_bytes(out), want)

    aug = vb.GpuAugment(32, 4, seed=6, policy="cifar10")
    N = 65536
    _, _, _, code = aug.draw(N, "cuda")
    code = code.cpu().long()
    sub, g1, g2, n1, n2 = code & 0xFF, code >> 8 & 1, code >> 9 & 1, code >> 10 & 1, code >> 11 & 1
    counts = torch.bincount(sub, minlength=25)
    p = 1 / 25
    assert counts.numel() == 25 and ((counts - N * p).abs() <= 5 * math.sqrt(N * p * (1 - p))).all(), counts
    for i, ((_, p1, _), (_, p2, _)) in enumerate(T.CIFAR10_POLICY):
        m = sub == i
        k = int(m.sum())
        for gate, pk in ((g1, p1), (g2, p2)):
            rate = gate[m].float().mean().item()
            assert abs(rate - pk) <= 5 * math.sqrt(pk * (1 - pk) / k) + 1e-12, (i, rate, pk)
    for s in (n1, n2):
        assert abs(s.float().mean().item() - 0.5) <= 5 * math.sqrt(0.25 / N)


def test_bad_arguments_raise(ops):
    from vit_cifar_b200 import VitbError
    img = torch.zeros((4, 32, 32, 3), dtype=torch.uint8, device="cuda")
    code = torch.zeros((4,), dtype=torch.int32, device="cuda")
    out = torch.empty((4, 3, 32, 32), device="cuda")
    with pytest.raises(VitbError, match="unknown op code"):
        ops.augment_autoaugment(img, None, None, None, code, [14, 0], [0.0, 0.0], MEAN, STD, out, PAD)
    with pytest.raises(VitbError, match="n_sub"):
        ops.augment_autoaugment(img, None, None, None, code, [0, 0] * 33, [0.1, 0.1] * 33, MEAN, STD, out, PAD)
    with pytest.raises(VitbError, match="posterize"):
        ops.augment_autoaugment(img, None, None, None, code, [6, 0], [9.0, 0.0], MEAN, STD, out, PAD)
    big = torch.zeros((2, 65, 65, 3), dtype=torch.uint8, device="cuda")
    with pytest.raises(VitbError, match="S <= 64"):
        ops.augment_autoaugment(big, None, None, None, code[:2], [0, 0], [0.1, 0.1], MEAN, STD, torch.empty((2, 3, 65, 65), device="cuda"), PAD)
    # an index past the table cannot be reported without a device round trip: that image comes out as NaN, the others do not
    code[2] = 1 | (1 << 8)
    ops.augment_autoaugment(img, None, None, None, code, [0, 0], [0.1, 0.1], MEAN, STD, out, PAD)
    nan = torch.isnan(out).flatten(1).all(1).cpu()
    assert nan.tolist() == [False, False, True, False]
