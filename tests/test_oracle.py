"""CPU: pin the oracle restatement against the fixtures generated from the unmodified reference
(tests/golden/make_golden.py) and, where the reference's source is available, against the live reference."""
import math
import os

import pytest
import torch

import oracle
from oracle import ViTConfig
from oracle.ref_shim import SKIP_REASON, import_reference, reference_available

FULL = ["tiny65", "tiny17c100", "nocls_nomlp"]
SUMMARY = ["full65", "full17c100"]


def _load(golden_dir, name):
    return torch.load(os.path.join(golden_dir, f"{name}.pt"), weights_only=False)


def _run_oracle(g, steps=3):
    torch.set_num_threads(1)
    cfg = ViTConfig(**g["cfg"])
    params = oracle.init_params(cfg, seed=0)
    x, y = oracle.hash_inputs(cfg, g["batch"], seed=1)
    logits, loss, grads = oracle.train_step(params, x, y, cfg, g["smoothing"])
    m = {k: torch.zeros_like(v) for k, v in params.items()}
    v = {k: torch.zeros_like(p) for k, p in params.items()}
    a = g["adam"]
    losses = [loss.item()]
    g_step = grads
    for t in range(1, steps + 1):
        oracle.adam_step(params, g_step, m, v, t, a["lr"], a["betas"], a["eps"], a["weight_decay"])
        if t < steps:
            _, l2, g_step = oracle.train_step(params, x, y, cfg, g["smoothing"])
            losses.append(l2.item())
    return cfg, logits, losses, grads, params


@pytest.mark.parametrize("name", FULL)
def test_oracle_matches_reference_golden_full(golden_dir, name):
    g = _load(golden_dir, name)
    cfg, logits, losses, grads, params3 = _run_oracle(g)
    torch.testing.assert_close(logits, g["logits"], rtol=1e-5, atol=1e-6)
    assert losses == pytest.approx(g["losses"], rel=1e-5)
    for k, ref in g["grads"].items():
        got = grads[k] if grads[k] is not None else torch.zeros_like(ref)
        torch.testing.assert_close(got, ref, rtol=1e-4, atol=1e-6, msg=lambda m, k=k: f"grad {k}: {m}")
    for k, ref in g["params3"].items():
        torch.testing.assert_close(params3[k], ref, rtol=1e-5, atol=2e-6, msg=lambda m, k=k: f"param {k}: {m}")
    # attention maps (save_attn_map protocol, layers.py:99-100)
    x, _ = oracle.hash_inputs(cfg, g["batch"], seed=1)
    _, attn = oracle.vit_forward(oracle.init_params(cfg, 0), x, cfg, return_attn=True)
    torch.testing.assert_close(attn, g["attn"], rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("name", SUMMARY)
def test_oracle_matches_reference_golden_summary(golden_dir, name):
    g = _load(golden_dir, name)
    cfg, logits, losses, grads, params3 = _run_oracle(g)
    torch.testing.assert_close(logits, g["logits"], rtol=1e-4, atol=1e-5)
    assert losses == pytest.approx(g["losses"], rel=1e-4)
    for k, ref in g["grads"].items():
        assert grads[k].double().norm().item() == pytest.approx(ref["norm"], rel=1e-4, abs=1e-9), k
        torch.testing.assert_close(grads[k].flatten()[:16], ref["head"], rtol=1e-3, atol=1e-6)
    for k, ref in g["params3"].items():
        assert params3[k].double().norm().item() == pytest.approx(ref["norm"], rel=1e-5), k
        torch.testing.assert_close(params3[k].flatten()[:16], ref["head"], rtol=1e-4, atol=1e-5)


def test_param_count_matches_reference_readme():
    # README.md:37 "6.3 M"; exact count probed from the reference (SURVEY.md §0)
    cfg = ViTConfig(num_classes=10, img_size=32, patch=8, num_layers=7, hidden=384, mlp_hidden=384, head=12)
    shapes = cfg.param_shapes()
    assert len(shapes) == 120
    assert sum(math.prod(s) for s in shapes.values()) == 6_268_810
    cfg = ViTConfig(num_classes=100, img_size=32, patch=4, num_layers=7, hidden=384, mlp_hidden=384, head=12)
    assert sum(math.prod(s) for s in cfg.param_shapes().values()) == 6_340_324


def test_patch_layout_identity():
    # words[b, ph*P+pw, (kh*ps+kw)*3+c] == x[b, c, ph*ps+kh, pw*ps+kw]   (vit.py:83-88)
    cfg = ViTConfig(patch=4)
    x, _ = oracle.hash_inputs(cfg, 2)
    w = oracle.to_words(x, cfg)
    ps, P = cfg.patch_size, cfg.patch
    for (b, ph, pw, kh, kw, c) in [(0, 0, 0, 0, 0, 0), (1, 3, 2, 7, 5, 2), (0, 1, 3, 4, 0, 1)]:
        assert w[b, ph * P + pw, (kh * ps + kw) * 3 + c] == x[b, c, ph * ps + kh, pw * ps + kw]


def test_ls_ce_closed_form_gradient():
    torch.manual_seed(0)
    z = torch.randn(5, 10, requires_grad=True)
    y = torch.randint(0, 10, (5,))
    loss = oracle.ls_ce_loss(z, y, 10, 0.1)
    loss.backward()
    torch.testing.assert_close(z.grad, oracle.ls_ce_dlogits(z.detach(), y, 10, 0.1), rtol=1e-5, atol=1e-7)


def test_adam_restatement_matches_torch_adam():
    torch.manual_seed(0)
    p0 = {"a": torch.randn(7, 5), "b": torch.randn(11)}
    ours = {k: v.clone() for k, v in p0.items()}
    theirs = [torch.nn.Parameter(v.clone()) for v in p0.values()]
    opt = torch.optim.Adam(theirs, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=5e-5)
    m = {k: torch.zeros_like(v) for k, v in p0.items()}
    v = {k: torch.zeros_like(x) for k, x in p0.items()}
    for t in range(1, 6):
        g = {k: torch.randn_like(x) for k, x in p0.items()}
        for p, gg in zip(theirs, g.values()):
            p.grad = gg.clone()
        opt.step()
        oracle.adam_step(ours, g, m, v, t)
    for p, k in zip(theirs, ours):
        torch.testing.assert_close(ours[k], p.detach(), rtol=1e-6, atol=1e-7)


@pytest.mark.skipif(not reference_available(), reason=SKIP_REASON)
@pytest.mark.parametrize("kw", [
    dict(num_classes=10, img_size=32, patch=8, num_layers=2, hidden=64, mlp_hidden=96, head=4),
    dict(num_classes=100, img_size=32, patch=4, num_layers=1, hidden=64, mlp_hidden=64, head=2, is_cls_token=False),
])
def test_oracle_matches_live_reference(kw):
    ref_vit, _, ref_crit = import_reference()
    cfg = ViTConfig(**kw)
    torch.manual_seed(2045)  # main.py:150
    model = ref_vit.ViT(3, cfg.num_classes, img_size=cfg.img_size, patch=cfg.patch, num_layers=cfg.num_layers,
                        hidden=cfg.hidden, mlp_hidden=cfg.mlp_hidden, head=cfg.head, is_cls_token=cfg.is_cls_token)
    params = {k: v.detach().clone() for k, v in model.state_dict().items()}  # reference's own init
    x = torch.randn(3, 3, 32, 32)
    y = torch.randint(0, cfg.num_classes, (3,))
    loss_ref = ref_crit.LabelSmoothingCrossEntropyLoss(cfg.num_classes, 0.1)(model(x), y)
    loss_ref.backward()
    logits, loss, grads = oracle.train_step(params, x, y, cfg, 0.1)
    torch.testing.assert_close(logits, model(x).detach(), rtol=1e-5, atol=1e-6)
    assert loss.item() == pytest.approx(loss_ref.item(), rel=1e-6)
    for k, p in model.named_parameters():
        torch.testing.assert_close(grads[k], p.grad, rtol=1e-4, atol=1e-6)


def test_two_target_loss_is_the_reference_expression():
    """network.py:163-165: loss(out, label) * lambda + loss(out, rand_label) * (1 - lambda), with the reference criterion when mounted."""
    g = torch.Generator().manual_seed(7)
    z = torch.randn(9, 10, generator=g); ya = torch.randint(0, 10, (9,), generator=g); yb = torch.randint(0, 10, (9,), generator=g)
    lam = 0.37
    ours = oracle.mixed_ls_ce_loss(z, ya, yb, lam, 10, 0.1)
    manual = oracle.ls_ce_loss(z, ya, 10, 0.1) * lam + oracle.ls_ce_loss(z, yb, 10, 0.1) * (1 - lam)
    torch.testing.assert_close(ours, manual)
    if reference_available():
        _, _, ref_crit = import_reference()
        crit = ref_crit.LabelSmoothingCrossEntropyLoss(10, smoothing=0.1)
        torch.testing.assert_close(ours, crit(z, ya) * lam + crit(z, yb) * (1 - lam), rtol=1e-6, atol=1e-7)


def test_augment_oracle_equals_torchvision_semantics_for_given_draws():
    """The oracle's crop/flip/normalize against the definition spelled out with plain indexing (torchvision's RandomCrop pads with
    zeros, crops at (top, left); flip reverses the width axis; ToTensor divides by 255; Normalize is per channel)."""
    g = torch.Generator().manual_seed(0)
    img = torch.randint(0, 256, (5, 32, 32, 3), generator=g, dtype=torch.uint8)
    dx = torch.tensor([0, 8, 4, 3, 7]); dy = torch.tensor([8, 0, 4, 5, 1]); fl = torch.tensor([0, 1, 0, 1, 1])
    mean, std = (0.4914, 0.4822, 0.4465), (0.2470, 0.2435, 0.2616)
    out = oracle.augment_crop_flip_normalize(img, dx, dy, fl, mean, std, 4)
    for b in range(5):
        for (c, y, x) in [(0, 0, 0), (1, 31, 31), (2, 10, 20), (0, 3, 29)]:
            xs = 31 - x if fl[b] else x
            sy, sx = y + int(dy[b]) - 4, xs + int(dx[b]) - 4
            v = float(img[b, sy, sx, c]) / 255.0 if (0 <= sy < 32 and 0 <= sx < 32) else 0.0
            assert abs(out[b, c, y, x].item() - (v - mean[c]) / std[c]) < 1e-6
    ident = oracle.augment_crop_flip_normalize(img, torch.full((5,), 4), torch.full((5,), 4), torch.zeros(5), (0, 0, 0), (1, 1, 1), 4)
    torch.testing.assert_close(ident, img.permute(0, 3, 1, 2).float() / 255.0)


def test_philox_restatement_known_answers():
    """Random123's published known-answer vectors for philox4x32-10 (kat_vectors): the generator behind libvitb200's dropout masks."""
    import numpy as np
    kat = [((0, 0, 0, 0), (0, 0), "6627e8d5 e169c58d bc57ac4c 9b00dbd8"),
           ((0xffffffff,) * 4, (0xffffffff,) * 2, "408f276d 41c83b0e a20bc7c6 6d5451fd"),
           ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0), "d16cfe09 94fdcceb 5001e420 24126ea1")]
    for ctr, key, want in kat:
        r = oracle.philox4x32_10(np.array([ctr], dtype=np.uint32), key)
        assert " ".join("%08x" % v for v in r[0]) == want
    keep = oracle.dropout_keep_mask(1 << 18, 0.25, seed=0x1234567890ABCDEF, site=2, step=5)
    assert abs(keep.mean() - 0.75) < 4 * math.sqrt(0.25 * 0.75 / (1 << 18))
    assert not (keep == oracle.dropout_keep_mask(1 << 18, 0.25, seed=0x1234567890ABCDEF, site=1, step=5)).all()
    assert oracle.dropout_threshold(0.0) == 0 and oracle.dropout_keep_mask(64, 0.0, 1, 0, 0).all()


@pytest.mark.skipif(not reference_available(), reason=SKIP_REASON)
@pytest.mark.parametrize("use_mlp", [True, False])
def test_oracle_dropout_sites_match_live_reference(use_mlp):
    """The three nn.Dropout sites of the reference block (layers.py:35, 38, 102) in training mode: replay the masks torch drew
    (captured by forward hooks) through the oracle's `drop` hook and compare output and every gradient."""
    import torch.nn as nn
    _, ref_layers, _ = import_reference()
    p_drop = 0.3
    torch.manual_seed(11)
    blk = ref_layers.TransformerEncoder(64, 96, head=4, dropout=p_drop, use_mlp=use_mlp)
    blk.train()
    x = torch.randn(3, 17, 64, requires_grad=True)
    masks = {}
    sites = {blk.attention.dropout: 0}
    if use_mlp:
        sites[blk.mlp[2]] = 1
        sites[blk.mlp[5]] = 2
    hooks = [m.register_forward_hook(lambda mod, inp, out, s=s: masks.__setitem__(s, (out != 0) | (inp[0] == 0))) for m, s in sites.items()]
    y_ref = blk(x)
    for h in hooks:
        h.remove()
    assert all(isinstance(m, nn.Dropout) for m in sites) and len(masks) == len(sites)
    w = torch.randn_like(y_ref)
    (y_ref * w).sum().backward()

    params = {k: v.detach().clone().requires_grad_(True) for k, v in blk.state_dict().items()}
    xo = x.detach().clone().requires_grad_(True)
    y = oracle.encoder_forward(params, "", xo, 4, use_mlp, drop=lambda site, t: t * masks[site].to(t.dtype) / (1.0 - p_drop))
    torch.testing.assert_close(y, y_ref.detach(), rtol=1e-5, atol=1e-6)
    (y * w).sum().backward()
    torch.testing.assert_close(xo.grad, x.grad, rtol=1e-4, atol=1e-6)
    for k, v in blk.named_parameters():
        if params[k].grad is None:
            assert v.grad is None
            continue
        torch.testing.assert_close(params[k].grad, v.grad, rtol=1e-4, atol=1e-6)
    # eval mode: identity (the oracle's drop=None path)
    blk.eval()
    torch.testing.assert_close(oracle.encoder_forward({k: v.detach() for k, v in params.items()}, "", x.detach(), 4, use_mlp), blk(x).detach(),
                               rtol=1e-5, atol=1e-6)


def test_oracle_dropout_block_matches_reference_golden(golden_dir):
    """Committed fixture of the reference block in training mode with dropout 0.2 (tests/golden/make_golden.py dropout_block):
    replaying the stored masks through the oracle reproduces the reference's output and gradients."""
    g = _load(golden_dir, "dropout_block")
    torch.set_num_threads(1)
    params = {k: v.clone().requires_grad_(True) for k, v in g["state_dict"].items()}
    x = g["x"].clone().requires_grad_(True)
    y = oracle.encoder_forward(params, "", x, g["head"], True, drop=lambda site, t: t * g["masks"][site].to(t.dtype) / (1.0 - g["p"]))
    torch.testing.assert_close(y, g["y"], rtol=1e-5, atol=1e-6)
    (y * g["w"]).sum().backward()
    torch.testing.assert_close(x.grad, g["dx"], rtol=1e-4, atol=1e-6)
    for k, v in g["grads"].items():
        torch.testing.assert_close(params[k].grad, v, rtol=1e-4, atol=1e-6)


def test_sgd_restatement_matches_torch_sgd():
    """network.py:78-84: torch.optim.SGD(lr, momentum=beta1, weight_decay)."""
    torch.manual_seed(0)
    p0 = {"a": torch.randn(7, 5), "b": torch.randn(11)}
    ours = {k: v.clone() for k, v in p0.items()}
    theirs = [torch.nn.Parameter(v.clone()) for v in p0.values()]
    opt = torch.optim.SGD(theirs, lr=1e-2, momentum=0.9, weight_decay=5e-5)
    bufs = {}
    for _ in range(5):
        g = {k: torch.randn_like(x) for k, x in p0.items()}
        for p, gg in zip(theirs, g.values()):
            p.grad = gg.clone()
        opt.step()
        oracle.sgd_step(ours, g, bufs, 1e-2, 0.9, 5e-5)
    for p, k in zip(theirs, ours):
        torch.testing.assert_close(ours[k], p.detach(), rtol=1e-6, atol=1e-7)


@pytest.mark.skipif(not reference_available(), reason=SKIP_REASON)
def test_cutmix_mixup_restatements_match_live_reference():
    """da.CutMix / da.MixUp (da.py:51-93) with seeded generators vs the oracle's paste / blend and the product's host-side box
    arithmetic (vit_cifar_b200.cutmix_box draws nothing itself: same numbers in, same box out)."""
    import numpy as np
    import_reference()
    import da as ref_da  # the reference's module (sys.path set by import_reference)
    import vit_cifar_b200 as vb
    g = torch.Generator().manual_seed(3)
    img = torch.randn(16, 3, 32, 32, generator=g)
    label = torch.randint(0, 10, (16,), generator=g)
    for seed in range(6):
        np.random.seed(seed); torch.manual_seed(seed)
        out_ref, l_ref, rl_ref, lam_ref = ref_da.CutMix(32, 1.0)((img.clone(), label.clone()))
        np.random.seed(seed); torch.manual_seed(seed)
        perm = torch.randperm(16)
        lam0 = np.random.beta(1.0, 1.0); r_x = np.random.uniform(0, 32); r_y = np.random.uniform(0, 32)
        box, lam = vb.cutmix_box(32, lam0, r_x, r_y)
        assert lam == lam_ref and torch.equal(label[perm], rl_ref) and torch.equal(l_ref, label)
        assert torch.equal(oracle.cutmix_apply(img, perm, box), out_ref)
        np.random.seed(seed); torch.manual_seed(seed)
        mx_ref, ya, yb, lam_m = ref_da.MixUp(0.1)((img, label))
        np.random.seed(seed); torch.manual_seed(seed)
        lam2 = np.random.beta(0.1, 0.1); index = torch.randperm(16)
        assert lam2 == lam_m and torch.equal(label[index], yb)
        assert torch.equal(oracle.mixup_apply(img, index, lam2), mx_ref)
