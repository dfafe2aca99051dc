"""``EvalEngine``: the reference's validation step (network.py:388-395, run once per epoch over the test set) as ONE static,
forward-only kernel sequence, captured into a CUDA graph, with the loss and accuracy summed on the device.

``schedule.evaluate`` goes through the module path once per batch: a weight cast, ~50 launches issued one by one, fresh
allocations for every intermediate (the MLP pre-activations included) and two host synchronisations.  Here a batch is
one graph replay and a whole pass one host synchronisation:

* Batches of 1..batch_size images: the number of valid rows travels in a device word (like ``TrainEngine``'s), so the partial
  last batch of the test set goes through the same graph.
* Forward only: no dropout (``model.eval()``), no pre-activation saves, and the activation buffers of the encoder blocks
  ping-pong between two scopes, so activation memory does not grow with the depth.
* ``vitb_eval_metrics`` (csrc/loss_adam.cu) adds each batch's [loss_sum, correct, count] to a 3-double device record;
  ``result()`` reads it once (after one all-reduce of the record when a process group is given).
* Weights: the engine reads the model's packed fp32 master and its bf16 shadow in place; ``reset()`` / ``run()`` refresh the
  shadow with one cast, as ``model(x)`` does per call, so weights written by ``TrainEngine`` steps or ``load_state_dict`` are
  evaluated without further calls.
"""
from __future__ import annotations

from typing import Dict, Iterable, Optional, Tuple

import torch

from . import functional as Fn
from . import ops
from .layers import act_dtype
from .params import LayerViews
from .vit import ViT


class EvalEngine:
    def __init__(self, model: ViT, batch_size: int = 256, smoothing: float = 0.1, mean=None, std=None, process_group=None,
                 use_graph: bool = True):
        """`mean` / `std` (3 floats each): also accept raw uint8 (n, S, S, 3) batches, normalised on the device (ToTensor +
        Normalize, the reference's test transform).  `process_group`: `result()` returns the metrics of the union of the ranks'
        batches on every rank."""
        ops.require_device()
        if (mean is None) != (std is None):
            raise ValueError("give both mean and std (uint8 input) or neither")
        if int(batch_size) < 1:
            raise ValueError(f"batch_size must be >= 1, got {batch_size}")
        self.model = model
        self.B = int(batch_size)
        self.smoothing = float(smoothing)
        self.mean = tuple(float(v) for v in mean) if mean is not None else None
        self.std = tuple(float(v) for v in std) if std is not None else None
        self.pg = process_group
        self.world = 1
        if process_group is not None:
            import torch.distributed as dist
            self.world = dist.get_world_size(process_group)
        self.use_graph = bool(use_graph)

        st = model._ensure_packed()
        self.store = st
        self.dev = st.device
        self.act = act_dtype()
        self.P = st.flat
        self.C = st.shadow() if self.act == torch.bfloat16 else self.P
        H, M = model.hidden, model.mlp_hidden
        self.dm = Fn.Dims(B=self.B, T=model.num_tokens, H=H, heads=model.head, M=M, use_mlp=model.encoder_mlp)
        self.dm.check()
        L = st.layout
        mk = lambda buf, i: LayerViews(L, buf, f"enc.{i}.", H, M, model.encoder_mlp)  # noqa: E731
        self.lp = [mk(self.P, i) for i in range(model.num_layers)]
        self.lc = [mk(self.C, i) for i in range(model.num_layers)]
        v = L.view
        self.stem_p = (v(self.P, "emb.weight"), v(self.P, "emb.bias"),
                       v(self.P, "cls_token").view(-1) if model.is_cls_token else None, v(self.P, "pos_emb").view(model.num_tokens, H))
        self.emb_w_c = v(self.C, "emb.weight") if self.C is not self.P else None
        self.head_p = (v(self.P, "fc.0.weight"), v(self.P, "fc.0.bias"), v(self.C, "fc.1.weight"), v(self.P, "fc.1.bias"))

        S = model.img_size
        self.img = torch.zeros((self.B, 3, S, S), dtype=torch.float32, device=self.dev)
        self.img_u8 = torch.zeros((self.B, S, S, 3), dtype=torch.uint8, device=self.dev) if mean is not None else None
        self.labels = torch.zeros((self.B,), dtype=torch.int64, device=self.dev)
        # number of valid rows of the current batch: a device-to-device copy from this table (no host memory the next batch could
        # overwrite before the copy has run)
        self._nv_table = torch.arange(self.B + 1, dtype=torch.int32, device=self.dev)
        self.n_valid = self._nv_table[self.B:].clone()
        self.totals = torch.zeros(3, dtype=torch.float64, device=self.dev)  # [loss_sum, correct, count]
        self._ws = torch.zeros(ops.eval_metrics_ws_bytes() // 8, dtype=torch.float64, device=self.dev)
        self.logits: Optional[torch.Tensor] = None
        self._bufs: Dict[str, torch.Tensor] = {}
        self._graph: Optional[torch.cuda.CUDAGraph] = None
        self.launches_per_batch = 0   # kernels of one batch, counted on the eager (warm-up) run
        self.captured_launches = 0    # kernels recorded into the graph
        self._check_model()
        if self.C is not self.P:
            ops.cast_f32_to_bf16(self.P, self.C)

    # -- static buffers ---------------------------------------------------------------------------
    def _alloc(self, scope: str):
        def alloc(name: str, shape: tuple, dtype: torch.dtype) -> torch.Tensor:
            key = f"{scope}.{name}"
            t = self._bufs.get(key)
            if t is None:
                t = torch.empty(shape, dtype=dtype, device=self.dev)
                self._bufs[key] = t
            return t
        return alloc

    def activation_bytes(self) -> int:
        """Bytes of the static intermediate buffers (stem, the two block scopes, head)."""
        return sum(t.numel() * t.element_size() for t in self._bufs.values())

    # -- the kernel sequence ----------------------------------------------------------------------
    def _forward(self) -> torch.Tensor:
        m, dm = self.model, self.dm
        emb_w, emb_b, cls, pos = self.stem_p
        x, _ = Fn.stem_fwd(self.img, emb_w, self.emb_w_c, emb_b, cls, pos, m.patch, self.act, self._alloc("stem"))
        for i in range(m.num_layers):
            # block i writes scope i % 2 and reads only its input x, the output of block i - 1 in the other scope; block i + 1
            # reads only block i's output, so block i + 2 may overwrite everything of block i (one stream: strictly in order)
            x_in = x
            x, _ = Fn.encoder_fwd(x, self.lc[i], self.lp[i], dm, self._alloc(f"l{i % 2}"), save_preact=False)
            self._check_scopes(x_in, x, i)
        ln_w, ln_b, fc_w_c, fc_b = self.head_p
        logits, _ = Fn.head_fwd(x, ln_w, ln_b, fc_w_c, fc_b, self.B, m.num_tokens, m.hidden, m.num_classes, m.is_cls_token,
                                self._alloc("head"))
        self.logits = logits
        return logits

    def _body(self) -> None:
        logits = self._forward()
        ops.eval_metrics(logits, self.labels, self.totals, self._ws, self.smoothing, n_valid_dev=self.n_valid)

    # -- checks -----------------------------------------------------------------------------------
    def _check_scopes(self, x_in: torch.Tensor, x_out: torch.Tensor, i: int) -> None:
        """Host-side proof of the ping-pong: block i's input is no buffer of the scope block i writes, and its output is one."""
        mine = [t for k, t in self._bufs.items() if k.startswith(f"l{i % 2}.")]
        if any(t.data_ptr() == x_in.data_ptr() for t in mine) or not any(t.data_ptr() == x_out.data_ptr() for t in mine):
            raise AssertionError(f"encoder block {i}: activation scopes overlap (engine bug)")

    def _check_model(self) -> None:
        m = self.model
        if getattr(m, "_store", None) is not self.store or not self.store.consistent():
            raise RuntimeError("the model's parameters no longer live in the flat buffer this EvalEngine was built on (re-packed by "
                               ".to() / .cuda() / parameter re-assignment): build a new EvalEngine")
        if act_dtype() != self.act:
            raise RuntimeError(f"precision changed to {act_dtype()} after this EvalEngine was built for {self.act}: build a new one")
        if any(blk.save_attn_map for blk in m.enc):
            raise ValueError("save_attn_map is set on an encoder block: attention maps come from the module path, "
                             "run model.eval()(x) for them")

    def _load(self, img: torch.Tensor, labels: Optional[torch.Tensor]) -> int:
        S = self.model.img_size
        if not isinstance(img, torch.Tensor) or img.dim() != 4:
            raise ValueError(f"expected a 4-d image batch, got {type(img).__name__} {tuple(getattr(img, 'shape', ()))}")
        n = int(img.shape[0])
        if not 1 <= n <= self.B:
            raise ValueError(f"batch of {n} images: this engine was built for batches of 1..{self.B} (batch_size={self.B})")
        if labels is not None:
            if labels.dim() != 1 or labels.shape[0] != n or labels.dtype.is_floating_point or labels.dtype == torch.bool:
                raise ValueError(f"expected {n} integer labels, got {labels.dtype} {tuple(labels.shape)}")
        if img.dtype == torch.uint8:
            if self.img_u8 is None:
                raise ValueError("uint8 batches need an EvalEngine built with mean and std")
            if tuple(img.shape[1:]) != (S, S, 3):
                raise ValueError(f"expected uint8 images of shape (n, {S}, {S}, 3), got {tuple(img.shape)}")
            if img.is_cuda:
                src = img.contiguous()
            else:
                self.img_u8[:n].copy_(img, non_blocking=True)
                src = self.img_u8[:n]
            ops.augment(src, None, None, None, self.mean, self.std, self.img[:n], 0)  # ToTensor + Normalize
        elif img.dtype == torch.float32:
            if tuple(img.shape[1:]) != (3, S, S):
                raise ValueError(f"expected float32 images of shape (n, 3, {S}, {S}), got {tuple(img.shape)}")
            self.img[:n].copy_(img, non_blocking=True)
        else:
            raise ValueError(f"images must be float32 (n, 3, S, S) or uint8 (n, S, S, 3), got {img.dtype}")
        if labels is not None:
            self.labels[:n].copy_(labels, non_blocking=True)
        self.n_valid.copy_(self._nv_table[n:n + 1], non_blocking=True)
        return n

    # -- public API -------------------------------------------------------------------------------
    def reset(self) -> None:
        """Start a pass: zero the metric record and refresh the bf16 weight copy from the fp32 master (one cast kernel)."""
        self._check_model()
        self.totals.zero_()
        if self.C is not self.P:
            ops.cast_f32_to_bf16(self.P, self.C)

    def add(self, img: torch.Tensor, labels: torch.Tensor) -> None:
        """Add one batch of 1..batch_size images to the pass.  No host synchronisation (host tensors should be pinned).  The first
        batch an engine sees runs the sequence eagerly and captures it; every later one is a graph replay."""
        self._check_model()
        self._load(img, labels)
        if not self.use_graph:
            n0 = ops.launch_count()
            self._body()
            self.launches_per_batch = ops.launch_count() - n0
        elif self._graph is None:
            n0 = ops.launch_count()
            self._body()                                  # warm-up: allocates every static buffer, counts this batch
            self.launches_per_batch = ops.launch_count() - n0
            g = torch.cuda.CUDAGraph()
            n0 = ops.launch_count()
            with torch.cuda.graph(g):
                self._body()                              # recorded, not executed
            self.captured_launches = ops.launch_count() - n0
            self._graph = g
        else:
            self._graph.replay()

    def result(self) -> Dict[str, float]:
        """{"val_loss", "val_acc", "n"} of the batches added since reset(), as schedule.evaluate returns them: one host
        synchronisation (and, with a process group, one all-reduce of the 3-double record first)."""
        t = self.totals
        if self.pg is not None and self.world > 1:
            import torch.distributed as dist
            t = t.clone()
            dist.all_reduce(t, group=self.pg)
        loss_sum, correct, n = t.tolist()
        n, correct = int(n), int(correct)
        return {"val_loss": loss_sum / max(n, 1), "val_acc": correct / max(n, 1), "n": n}

    def run(self, batches: Iterable[Tuple[torch.Tensor, torch.Tensor]]) -> Dict[str, float]:
        """One validation pass over an iterable of (img, label): reset(), add() per batch, result()."""
        self.reset()
        for img, label in batches:
            self.add(img, label)
        return self.result()

    @torch.no_grad()
    def forward(self, img: torch.Tensor) -> torch.Tensor:
        """(n, C) fp32 logits of one batch of n <= batch_size images: the inference forward (run_model.py:50-57), the same kernels
        in the same order as model.eval()(img) at batch size batch_size.  Like model(x) it refreshes the bf16 weight copy first;
        it runs the sequence directly (not the graph) and leaves the metric record alone."""
        self._check_model()
        if self.C is not self.P:
            ops.cast_f32_to_bf16(self.P, self.C)
        n = self._load(img, None)
        return self._forward()[:n].clone()
