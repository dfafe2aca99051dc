"""CPU: head dimensions 96 and 128 pass the shape check (the attention kernels run them as 32- / 64-column panels); the other
head dimensions stay rejected."""
import pytest

from vit_cifar_b200.functional import Dims


def test_dims_accepts_head_dims_96_and_128():
    n = 0
    for H in range(64, 1025, 64):
        for d in (96, 128):
            if H % d == 0:
                Dims(B=4, T=65, H=H, heads=H // d, M=H).check()
                n += 1
    assert n == 5 + 8  # d = 96: H = 192 .. 960 in steps of 192; d = 128: H = 128 .. 1024 in steps of 128


@pytest.mark.parametrize("H,heads", [(384, 24), (384, 8), (640, 8), (768, 4), (384, 1)], ids=["d16", "d48", "d80", "d192", "d384"])
def test_dims_still_rejects_other_head_dims(H, heads):
    with pytest.raises(ValueError, match="32, 64, 96 or 128"):
        Dims(B=4, T=65, H=H, heads=heads, M=H).check()


def test_vit_constructs_at_head_dim_96():
    import vit_cifar_b200 as vb
    m = vb.ViT(3, 10, img_size=32, patch=8, hidden=384, mlp_hidden=384, head=4)
    assert sum(p.numel() for p in m.parameters()) > 0
