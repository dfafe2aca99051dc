"""vit_cifar_b200 — B200-native training hot path of mahbodnr/ViT-CIFAR.

The sources live in the directory ``vit-cifar_b200/`` (the project's layout name, not importable as written);
this package makes them importable as ``vit_cifar_b200`` by extending its ``__path__``.

Public surface (mirrors the reference's module/class names for this path):
  ViT, TransformerEncoder, MultiHeadSelfAttention      (vit.py / layers.py of the reference)
  LabelSmoothingCrossEntropyLoss                        (criterions.py)
  FusedAdam                                             (torch.optim.Adam as configured in network.py:71-77)
  TrainEngine                                           (the per-batch hot loop, CUDA-graphed, data-parallel)
  EvalEngine                                            (the validation pass, network.py:388-395: forward-only CUDA graph,
                                                         loss / accuracy summed on the device, one host sync per pass)
  DeviceDataset, DeviceLoader                           (the DataLoader / DistributedSampler of utils.py:452-470 over a
                                                         dataset resident in device memory)
  set_precision / get_precision                         ('bf16' tensor-core path or 'fp32' check mode)
  WarmupCosine, evaluate, save_checkpoint, load_checkpoint   (network.py:113-122, 388-395; main.py:234-237, run_model.py:12-37)
"""
import os as _os

__path__.append(_os.path.join(_os.path.dirname(_os.path.dirname(_os.path.abspath(__file__))), "vit-cifar_b200"))

from ._lib import VitbError, LIB_PATH, load as load_library  # noqa: E402,F401
from .layers import MultiHeadSelfAttention, TransformerEncoder, get_precision, set_precision  # noqa: E402,F401
from .vit import ViT  # noqa: E402,F401
from .criterions import LabelSmoothingCrossEntropyLoss  # noqa: E402,F401
from .optim import FusedAdam, adam_hyper, sgd_hyper  # noqa: E402,F401
from .engine import TrainEngine  # noqa: E402,F401
from .evaluator import EvalEngine  # noqa: E402,F401
from .loader import DeviceDataset, DeviceLoader  # noqa: E402,F401
from .schedule import (WarmupCosine, warmup_cosine_lr, evaluate, save_checkpoint, load_checkpoint, to_lightning_checkpoint,  # noqa: E402,F401
                       GpuAugment, GpuCutMix, GpuMixUp, cutmix_box)
