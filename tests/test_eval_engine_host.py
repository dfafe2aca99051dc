"""CPU: host side of the validation pass — the vitb_eval_metrics ABI entry, its argument checks (they return before any
device work), the forward-only switch of functional.encoder_fwd, and EvalEngine's refusal to run without a device."""
import inspect

import pytest
import torch


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    import vit_cifar_b200 as vb
    return vb.load_library()


def test_eval_metrics_is_in_the_abi(lib):
    from vit_cifar_b200 import _lib
    assert "vitb_eval_metrics" in _lib.SIGNATURES and "vitb_eval_metrics_ws_bytes" in _lib.SIGNATURES
    # one 8-byte counter word + (loss, correct) fp64 partials of up to 256 blocks
    assert lib.vitb_eval_metrics_ws_bytes() == (1 + 2 * 256) * 8


def test_eval_metrics_host_argument_checks(lib):
    ws_bytes = lib.vitb_eval_metrics_ws_bytes()
    p = 4096  # never dereferenced: every call below is refused before a launch
    cases = [
        ((None, p, None, 8, 10, 0.1, p, p, ws_bytes), b"null pointer"),
        ((p, None, None, 8, 10, 0.1, p, p, ws_bytes), b"null pointer"),
        ((p, p, None, 8, 10, 0.1, None, p, ws_bytes), b"null pointer"),
        ((p, p, None, 8, 10, 0.1, p, None, ws_bytes), b"null pointer"),
        ((p, p, None, 0, 10, 0.1, p, p, ws_bytes), b"bad shape"),
        ((p, p, None, -3, 10, 0.1, p, p, ws_bytes), b"bad shape"),
        ((p, p, None, 8, 1, 0.1, p, p, ws_bytes), b"bad shape"),
        ((p, p, None, 8, 10, 0.1, p, p, ws_bytes - 1), b"workspace too small"),
        ((p, p, None, 8, 10, 0.1, p, p + 4, ws_bytes), b"aligned"),
    ]
    for args, msg in cases:
        assert lib.vitb_eval_metrics(*args, None) < 0, args
        assert msg in lib.vitb_last_error(), (args, lib.vitb_last_error())


def test_encoder_fwd_saves_preactivations_by_default():
    from vit_cifar_b200 import functional as Fn
    sig = inspect.signature(Fn.encoder_fwd)
    assert sig.parameters["save_preact"].default is True


def test_eval_engine_is_exported_and_needs_a_device(lib):
    import vit_cifar_b200 as vb
    assert "EvalEngine" in vb.__doc__
    assert vb.EvalEngine.__module__ == "vit_cifar_b200.evaluator"
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    m = vb.ViT(3, 10, img_size=32, patch=8, num_layers=1, hidden=128, mlp_hidden=128, head=4)
    with pytest.raises(vb.VitbError):
        vb.EvalEngine(m, batch_size=4)
