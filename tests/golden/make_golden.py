"""Generate golden fixtures from the UNMODIFIED reference.

    VITB_REFERENCE_ROOT=<checkout of mahbodnr/ViT-CIFAR> python tests/golden/make_golden.py

Imports ``vit.ViT`` / ``criterions.LabelSmoothingCrossEntropyLoss`` from
that checkout (via oracle/ref_shim.py), loads hash-derived weights and inputs
(oracle.hash_init_ / oracle.hash_inputs: integer arithmetic, reproducible bit for
bit anywhere), runs forward + LS-CE + backward + torch.optim.Adam (the optimiser
network.py:71-77 configures) in fp32 on CPU and stores the results.

"full" fixtures store every tensor; "summary" fixtures (the 6.3 M-parameter
model) store logits, loss and per-tensor norms + leading elements to stay small.
"""
from __future__ import annotations

import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import ViTConfig, hash_init_, hash_inputs  # noqa: E402
from oracle.ref_shim import import_reference  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))

ADAM = dict(lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=5e-5)  # main.py:48-56
SMOOTHING = 0.1  # main.py:62

CASES = {
    # name: (cfg kwargs, batch, mode)
    "tiny65": (dict(num_classes=10, img_size=32, patch=8, num_layers=2, hidden=128, mlp_hidden=128, head=4), 4, "full"),
    "tiny17c100": (dict(num_classes=100, img_size=32, patch=4, num_layers=1, hidden=128, mlp_hidden=256, head=2), 3, "full"),
    "nocls_nomlp": (dict(num_classes=10, img_size=32, patch=4, num_layers=1, hidden=128, mlp_hidden=128, head=4,
                         is_cls_token=False, encoder_mlp=False), 2, "full"),
    "full65": (dict(num_classes=10, img_size=32, patch=8, num_layers=7, hidden=384, mlp_hidden=384, head=12), 4, "summary"),
    "full17c100": (dict(num_classes=100, img_size=32, patch=4, num_layers=7, hidden=384, mlp_hidden=384, head=12), 4, "summary"),
}


def summarize(d):
    return {k: dict(norm=v.double().norm().item(), sum=v.double().sum().item(), head=v.flatten()[:16].clone())
            for k, v in d.items()}


def main():
    ref_vit, ref_layers, ref_crit = import_reference()
    torch.set_num_threads(1)  # fixed reduction order
    for name, (kw, batch, mode) in CASES.items():
        cfg = ViTConfig(**kw)
        model = ref_vit.ViT(
            3, cfg.num_classes, img_size=cfg.img_size, patch=cfg.patch, dropout=0.0,
            num_layers=cfg.num_layers, hidden=cfg.hidden, encoder_mlp=cfg.encoder_mlp,
            mlp_hidden=cfg.mlp_hidden, head=cfg.head, is_cls_token=cfg.is_cls_token)
        sd = model.state_dict()
        assert list(sd.keys()) == list(cfg.param_shapes().keys()), (list(sd.keys()), list(cfg.param_shapes().keys()))
        hash_init_(sd, seed=0)  # in place -> model weights
        x, y = hash_inputs(cfg, batch, seed=1)
        crit = ref_crit.LabelSmoothingCrossEntropyLoss(cfg.num_classes, smoothing=SMOOTHING)
        opt = torch.optim.Adam(model.parameters(), **ADAM)

        # attention maps via the reference's own save_attn_map protocol (layers.py:50-65)
        for m in model.modules():
            if hasattr(m, "save_attn_map"):
                m.save_attn_map = True
        logits = model(x)
        attn = torch.stack([blk.get_attention_map().detach() for blk in model.enc])
        loss = crit(logits, y)
        opt.zero_grad()
        loss.backward()
        # parameters the forward never touches (la2 when encoder_mlp=False, layers.py:30,46) keep grad None
        # and torch's Adam skips them; stored as zeros.
        grads = {k: (p.grad.detach().clone() if p.grad is not None else torch.zeros_like(p))
                 for k, p in model.named_parameters()}
        losses = [loss.item()]
        opt.step()
        for _ in range(2):  # two more steps on the same batch -> params after 3 Adam steps
            opt.zero_grad()
            l2 = crit(model(x), y)
            l2.backward()
            losses.append(l2.item())
            opt.step()
        params3 = {k: v.detach().clone() for k, v in model.state_dict().items()}

        out = dict(cfg=kw, batch=batch, mode=mode, smoothing=SMOOTHING, adam=ADAM,
                   logits=logits.detach().clone(), loss=losses[0], losses=losses,
                   torch_version=torch.__version__)
        if mode == "full":
            out.update(grads=grads, params3=params3, attn=attn)
        else:
            out.update(grads=summarize(grads), params3=summarize(params3),
                       attn=dict(norm=attn.double().norm().item(), head=attn[0, 0, 0, :2].clone(),
                                 shape=tuple(attn.shape)))
        path = os.path.join(HERE, f"{name}.pt")
        torch.save(out, path)
        print(f"{name}: loss={losses} logits[0,:3]={logits[0, :3].tolist()} -> {path} "
              f"({os.path.getsize(path) / 1e6:.2f} MB)")


def dropout_block():
    """One reference TransformerEncoder in TRAINING mode with dropout 0.2 (layers.py:35, 38, 102): the masks torch drew at the three
    nn.Dropout sites (captured by forward hooks), the output, and every gradient for a fixed cotangent."""
    _, ref_layers, _ = import_reference()
    torch.set_num_threads(1)
    p_drop, F_, M, head, B, T = 0.2, 128, 256, 4, 2, 17
    torch.manual_seed(5)
    blk = ref_layers.TransformerEncoder(F_, M, head=head, dropout=p_drop)
    sd = blk.state_dict()
    hash_init_(sd, seed=3)
    blk.train()
    x = torch.randn(B, T, F_, requires_grad=True)
    w = torch.randn(B, T, F_)
    masks = {}
    sites = {blk.attention.dropout: 0, blk.mlp[2]: 1, blk.mlp[5]: 2}
    hooks = [m.register_forward_hook(lambda mod, inp, out, s=s: masks.__setitem__(s, ((out != 0) | (inp[0] == 0)).clone()))
             for m, s in sites.items()]
    y = blk(x)
    for h in hooks:
        h.remove()
    (y * w).sum().backward()
    out = dict(p=p_drop, features=F_, mlp_hidden=M, head=head, state_dict={k: v.detach().clone() for k, v in blk.state_dict().items()},
               x=x.detach().clone(), w=w, masks=masks, y=y.detach().clone(), dx=x.grad.clone(),
               grads={k: v.grad.detach().clone() for k, v in blk.named_parameters()}, torch_version=torch.__version__)
    path = os.path.join(HERE, "dropout_block.pt")
    torch.save(out, path)
    print(f"dropout_block: keep rates {[round(m.float().mean().item(), 3) for m in masks.values()]} -> {path} ({os.path.getsize(path) / 1e6:.2f} MB)")


# the configurations of tests/test_oracle.py::test_oracle_matches_live_reference
SEEDED = {
    "seeded_cls": dict(num_classes=10, img_size=32, patch=8, num_layers=2, hidden=64, mlp_hidden=96, head=4),
    "seeded_nocls": dict(num_classes=100, img_size=32, patch=4, num_layers=1, hidden=64, mlp_hidden=64, head=2, is_cls_token=False),
}
# the model of tests/test_host_logic.py::test_checkpoint_format_round_trip
CHECKPOINT_KW = dict(img_size=32, patch=4, num_layers=2, hidden=128, mlp_hidden=128, head=4)


def seeded_reference():
    """The reference's OWN initialisation (torch.manual_seed(2045), main.py:150) and one LS-CE forward + backward on torch.randn
    inputs drawn right after it, for the two configurations the live comparison uses; plus the state_dict names and shapes of
    the checkpoint test's model.  Same draws, in the same order, as the live tests."""
    ref_vit, _, ref_crit = import_reference()
    torch.set_num_threads(1)
    for name, kw in SEEDED.items():
        cfg = ViTConfig(**kw)
        torch.manual_seed(2045)
        model = ref_vit.ViT(3, cfg.num_classes, img_size=cfg.img_size, patch=cfg.patch, num_layers=cfg.num_layers,
                            hidden=cfg.hidden, mlp_hidden=cfg.mlp_hidden, head=cfg.head, is_cls_token=cfg.is_cls_token)
        state_dict = {k: v.detach().clone() for k, v in model.state_dict().items()}
        x = torch.randn(3, 3, 32, 32)
        y = torch.randint(0, cfg.num_classes, (3,))
        logits = model(x)
        loss = ref_crit.LabelSmoothingCrossEntropyLoss(cfg.num_classes, 0.1)(logits, y)
        loss.backward()
        out = dict(cfg=kw, state_dict=state_dict, x=x, y=y, logits=logits.detach().clone(), loss=loss.item(),
                   grads={k: p.grad.detach().clone() for k, p in model.named_parameters()}, torch_version=torch.__version__)
        if name == "seeded_cls":
            out["checkpoint_shapes"] = {k: tuple(v.shape) for k, v in ref_vit.ViT(3, 10, **CHECKPOINT_KW).state_dict().items()}
        _save(out, name)


def dropout_sites():
    """The reference block in training mode at p = 0.3 with and without its MLP (layers.py:35, 38, 102), as the live test
    builds it: the masks torch drew (forward hooks), the output, every gradient for a random cotangent, and the eval output."""
    _, ref_layers, _ = import_reference()
    torch.set_num_threads(1)
    out = {}
    for use_mlp in (True, False):
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
        hooks = [m.register_forward_hook(lambda mod, inp, o, s=s: masks.__setitem__(s, ((o != 0) | (inp[0] == 0)).clone()))
                 for m, s in sites.items()]
        y = blk(x)
        for h in hooks:
            h.remove()
        w = torch.randn_like(y)
        (y * w).sum().backward()
        blk.eval()
        out[use_mlp] = dict(p=p_drop, head=4, state_dict={k: v.detach().clone() for k, v in blk.state_dict().items()},
                            x=x.detach().clone(), w=w, masks=masks, y=y.detach().clone(), dx=x.grad.clone(),
                            grads={k: (v.grad.detach().clone() if v.grad is not None else None) for k, v in blk.named_parameters()},
                            y_eval=blk(x.detach()).detach().clone())
    _save(dict(cases=out, torch_version=torch.__version__), "dropout_sites")


def batch_mixing():
    """da.CutMix(32, 1.0) and da.MixUp(0.1) (da.py:51-93) on a seeded 4-image batch for seeds 0..5, and the reference
    criterion's two-target loss (network.py:163-165) on seeded logits."""
    import numpy as np
    _, _, ref_crit = import_reference()
    import da as ref_da  # the reference's module (sys.path set by import_reference)
    g = torch.Generator().manual_seed(3)
    img = torch.randn(4, 3, 32, 32, generator=g)
    label = torch.randint(0, 10, (4,), generator=g)
    cutmix, mixup = [], []
    for seed in range(6):
        np.random.seed(seed); torch.manual_seed(seed)
        o, la, lb, lam = ref_da.CutMix(32, 1.0)((img.clone(), label.clone()))
        cutmix.append(dict(out=o, label=la, rand_label=lb, lam=lam))
        np.random.seed(seed); torch.manual_seed(seed)
        o, la, lb, lam = ref_da.MixUp(0.1)((img, label))
        mixup.append(dict(out=o, label=la, rand_label=lb, lam=lam))
    g = torch.Generator().manual_seed(7)
    z = torch.randn(9, 10, generator=g); ya = torch.randint(0, 10, (9,), generator=g); yb = torch.randint(0, 10, (9,), generator=g)
    crit = ref_crit.LabelSmoothingCrossEntropyLoss(10, smoothing=0.1)
    two_target = (crit(z, ya) * 0.37 + crit(z, yb) * (1 - 0.37)).item()
    _save(dict(img=img, label=label, cutmix=cutmix, mixup=mixup, two_target_loss=two_target, torch_version=torch.__version__),
          "batch_mixing")


def _save(obj, name):
    path = os.path.join(HERE, f"{name}.pt")
    torch.save(obj, path)
    size = os.path.getsize(path)
    assert size < 1_000_000, (path, size)
    print(f"{name} -> {path} ({size / 1e6:.2f} MB)")


if __name__ == "__main__":
    which = sys.argv[1] if len(sys.argv) > 1 else "all"
    if which == "dropout":  # only the newer fixture; the others stay byte-identical
        dropout_block()
    elif which == "seeded":  # the fixtures of the live-reference tests only
        seeded_reference()
        dropout_sites()
        batch_mixing()
    else:
        main()
        dropout_block()
        seeded_reference()
        dropout_sites()
        batch_mixing()
