"""CPU: the width rule of the model (hidden and MLP widths multiples of 64) and the library's workspace queries at those widths."""
import ctypes as C

import pytest

from vit_cifar_b200.functional import Dims


@pytest.mark.parametrize("H", [64 * k for k in range(1, 17)])
def test_dims_accepts_every_multiple_of_64_up_to_1024(H):
    for d in (32, 64):
        if H % d == 0:
            Dims(B=2, T=65, H=H, heads=H // d, M=H, use_mlp=True).check()
            Dims(B=2, T=17, H=H, heads=H // d, M=4 * H).check()


@pytest.mark.parametrize("kw", [
    dict(H=1088, heads=17, M=1088),   # wider than one warp's LayerNorm row
    dict(H=100, heads=4, M=128),      # not a multiple of 64
    dict(H=192, heads=3, M=96),       # MLP width not a multiple of 64
    dict(H=192, heads=4, M=192),      # head_dim 48
    dict(H=192, heads=12, M=192),     # head_dim 16
    dict(H=320, heads=4, M=320),      # head_dim 80
])
def test_dims_rejects(kw):
    with pytest.raises(ValueError):
        Dims(B=2, T=65, **kw).check()


def test_dims_without_mlp_ignores_the_mlp_width():
    Dims(B=2, T=65, H=192, heads=3, M=96, use_mlp=False).check()


def test_vit_tiny_module_is_accepted():
    import vit_cifar_b200 as vb
    vb.ViT(3, 10, img_size=32, patch=8, num_layers=12, hidden=192, mlp_hidden=768, head=3)


def _lib_with_debug_queries():
    from vit_cifar_b200 import _lib
    lib = _lib.load()
    f = lib.vitb_debug_wgrad_splits  # exported for tools and tests, not declared in the header
    f.restype, f.argtypes = C.c_int, [C.c_int, C.c_int, C.c_int]
    return lib


@pytest.mark.parametrize("cols", [64, 192, 320, 576, 640, 960])
@pytest.mark.parametrize("rows", [17, 1040, 66560])
def test_workspace_queries_at_the_new_widths(cols, rows):
    lib = _lib_with_debug_queries()
    cs = lib.vitb_colsum_ws_bytes(rows, cols)
    assert cs > 0 and cs % (cols * 4) == 0              # [row parts][cols] fp32 partials
    ln = lib.vitb_layernorm_bwd_ws_bytes(rows, cols)
    assert ln > 0 and ln % (3 * cols * 4) == 0          # [3][blocks][H] fp32 partials
    for K in (64, 192, 384, 768):
        wg = lib.vitb_gemm_wgrad_ws_bytes(rows, cols, K, 1)
        assert wg >= cols * 4                           # at least the bias-gradient partials
        splits = lib.vitb_debug_wgrad_splits(rows, cols, K)
        assert splits >= 1, (rows, cols, K)            # the tensor-core weight gradient takes this shape
        if splits > 1:
            assert wg >= splits * cols * K * 4


def test_workspace_queries_keep_rejecting_widths_off_the_64_grid():
    lib = _lib_with_debug_queries()
    assert lib.vitb_colsum_ws_bytes(100, 96) == 0
    assert lib.vitb_debug_wgrad_splits(1000, 96, 128) == 0
