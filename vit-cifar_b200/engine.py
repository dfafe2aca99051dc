"""``TrainEngine``: the whole training step (forward + LS-CE + backward + gradient averaging + Adam) of a packed
``ViT`` as ONE static kernel sequence, captured into a CUDA graph.

This is the caller the reference gets from Lightning (network.py:149-208 + automatic optimisation + DDP,
SURVEY.md §3.1) reduced to the hot loop: no autograd, no allocation, no host sync inside a step.

* Batches of 1..batch_size images (the reference's DataLoader keeps the partial last batch of an epoch): the loss kernel reads
  the number of valid rows from device memory.
* Backward: the weight-gradient GEMMs run on a second stream (nothing reads dW before the optimiser), the critical path on a
  high-priority stream; the second passes of all split reductions are deferred to one flush before the optimiser
  (``vitb_defer_begin`` / ``vitb_defer_flush``), every call owning its slice of a partial-sum arena.
* Data parallel (one process per GPU): by default gradient averaging and the optimiser are one peer-memory kernel
  (csrc/dp.cu; ``VITB_DP_MODE=fused``); ``single`` = one NCCL all-reduce of the flat gradient buffer after backward, ``overlap`` =
  per-layer buckets on a side stream as soon as that layer's backward has been issued.  The 1/world_size of DDP's mean is folded
  into the optimiser's gradient scale.
* ``checkpoint()`` / ``load_checkpoint()`` / ``sync_weights()``: Lightning-format checkpoints with optimiser state, and the hook
  to call after writing weights from outside the step.
"""
from __future__ import annotations

import os
from typing import Dict, Optional, Tuple

import torch

from . import functional as Fn
from . import ops
from .layers import act_dtype
from .optim import adam_hyper, sgd_hyper
from .parallel import allreduce_bucket
from .params import LayerViews
from .vit import ViT


class TrainEngine:
    def __init__(self, model: ViT, batch_size: int, smoothing: float = 0.1, lr: float = 1e-3, betas=(0.9, 0.999),
                 eps: float = 1e-8, weight_decay: float = 5e-5, process_group=None, use_graph: bool = True,
                 overlap_comm: bool = False, mixed_targets: bool = False, optimizer: str = "adam", momentum: Optional[float] = None,
                 metrics: bool = False):
        """optimizer: "adam" (network.py:71-77) or "sgd" (network.py:78-84: torch.optim.SGD with momentum = beta1 unless `momentum`
        is given, coupled weight decay).  metrics: each step also adds to an epoch record on the device (the correct count of the
        logits against `labels`, the batch-size-weighted step loss), read by `train_metrics()`; off, the step is unchanged."""
        ops.require_device()
        if optimizer not in ("adam", "sgd"):
            raise NotImplementedError(f"Unknown optimizer: {optimizer}")  # the reference's message (network.py:110)
        self.optimizer = optimizer
        self.momentum = float(betas[0] if momentum is None else momentum)
        self.model = model
        self.B = int(batch_size)
        self.smoothing = float(smoothing)
        self.lr, self.betas, self.eps, self.weight_decay = float(lr), betas, float(eps), float(weight_decay)
        self.pg = process_group
        self.world, self._rank = 1, 0
        if process_group is not None:
            import torch.distributed as dist
            self.world, self._rank = dist.get_world_size(process_group), dist.get_rank(process_group)
        self.use_graph = use_graph
        # two-target loss lam*L(out,y) + (1-lam)*L(out,y') for CutMix / MixUp batches (network.py:149-167); lam travels in the
        # per-step hyper-parameter block so the captured graph reads a fresh value every step
        self.mixed_targets = bool(mixed_targets)
        self._l2_persist = os.environ.get("VITB_L2_PERSIST", "0") != "0"
        self._lam = 1.0
        self._next_lam = 1.0
        # "overlap": per-layer buckets on a side stream while backward continues; "single": one all-reduce of the whole flat
        # gradient buffer after backward (no SM contention between NCCL's CTAs and the persistent GEMM kernels); "fused": no NCCL
        # in the step at all — one kernel does barrier + reduce-scatter over NVLink peer memory + Adam + all-gather (csrc/dp.cu)
        mode = os.environ.get("VITB_DP_MODE", "overlap" if overlap_comm else "fused")
        if mode not in ("single", "overlap", "fused", "none"):
            raise ValueError(f"VITB_DP_MODE={mode!r}: expected single, overlap or fused")
        self._dp_mode = mode
        self.overlap_comm = (mode == "overlap") and self.world > 1
        if not 0.0 <= model.p_drop < 1.0:
            raise ValueError(f"dropout probability has to be in [0, 1), got {model.p_drop}")

        st = model._ensure_packed()
        self.store = st
        self.dev = st.device
        self.act = act_dtype()
        L = st.layout
        self.n = L.active_end
        self.P = st.flat
        self.G = torch.zeros_like(self.P)
        self.Mo = torch.zeros_like(self.P)
        self.V = torch.zeros_like(self.P)
        if self.act == torch.bfloat16:
            self.C = st.shadow()
            ops.cast_f32_to_bf16(self.P, self.C)
        else:
            self.C = self.P
        if self.world > 1:
            import torch.distributed as dist
            dist.broadcast(self.P, src=0, group=self.pg)  # identical replicas
            if self.C is not self.P:
                ops.cast_f32_to_bf16(self.P, self.C)

        self._fused_dp = None
        if self.world > 1 and mode == "fused":
            import torch.distributed as dist
            from .parallel import exchange_peer_pointers
            flags = torch.zeros(64, dtype=torch.int32, device=self.dev)
            sync = torch.zeros(4, dtype=torch.int32, device=self.dev)
            torch.cuda.synchronize(self.dev)
            if self.world > 8 or self.n % 4 != 0:  # the same on every rank
                peers, err = None, ValueError("at most 8 ranks of one node and a flat buffer that is a multiple of 4 elements")
            else:
                peers, err = exchange_peer_pointers(dict(g=self.G, p=self.P, c=self.C if self.C is not self.P else None, flags=flags), self.pg)
            ok = torch.tensor([0 if peers is None else 1], device=self.dev)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=self.pg)  # also: every rank has mapped every peer before the first step
            if int(ok.item()) == 1:
                self._fused_dp = dict(peers, flags_t=flags, sync=sync, rank=dist.get_rank(self.pg))
            else:
                import warnings
                warnings.warn(f"fused data-parallel step unavailable ({err}); using one NCCL all-reduce + the Adam kernel")
                self._dp_mode = mode = "single"

        H, M = model.hidden, model.mlp_hidden
        self.dm = Fn.Dims(B=self.B, T=model.num_tokens, H=H, heads=model.head, M=M, use_mlp=model.encoder_mlp)
        self.dm.check()
        mk = lambda buf, i: LayerViews(L, buf, f"enc.{i}.", H, M, model.encoder_mlp)  # noqa: E731
        self.lp = [mk(self.P, i) for i in range(model.num_layers)]
        self.lc = [mk(self.C, i) for i in range(model.num_layers)]
        self.lg = [mk(self.G, i) for i in range(model.num_layers)]
        v = L.view
        self.has_cls = model.is_cls_token
        self.stem_p = (v(self.P, "emb.weight"), v(self.P, "emb.bias"),
                       v(self.P, "cls_token").view(-1) if self.has_cls else None, v(self.P, "pos_emb").view(model.num_tokens, H))
        self.stem_g = (v(self.G, "emb.weight"), v(self.G, "emb.bias"),
                       v(self.G, "cls_token").view(-1) if self.has_cls else None, v(self.G, "pos_emb").view(model.num_tokens, H))
        self.head_p = (v(self.P, "fc.0.weight"), v(self.P, "fc.0.bias"), v(self.C, "fc.1.weight"), v(self.P, "fc.1.bias"))
        self.head_g = (v(self.G, "fc.0.weight"), v(self.G, "fc.0.bias"), v(self.G, "fc.1.weight"), v(self.G, "fc.1.bias"))
        self.buckets = model.bucket_bounds()  # [stem, layer0..layerL-1, head]

        S = model.img_size
        self.img = torch.zeros((self.B, 3, S, S), dtype=torch.float32, device=self.dev)
        self.labels = torch.zeros((self.B,), dtype=torch.int64, device=self.dev)
        self.labels_b = torch.zeros_like(self.labels)
        self._labels_b_stage = torch.zeros_like(self.labels)
        self.loss = torch.zeros((), dtype=torch.float32, device=self.dev)
        from . import _lib
        self._ls_ws = torch.zeros(int(_lib.load().vitb_ls_ce_ws_bytes()) // 4, dtype=torch.float32, device=self.dev)  # loss kernel: partials + counter
        # input staging for `prefetch`: the next batch crosses PCIe on a copy stream while the current step computes
        self._img_stage = torch.zeros_like(self.img)
        self._labels_stage = torch.zeros_like(self.labels)
        self._copy_stream = torch.cuda.Stream(device=self.dev)
        self._staged = torch.cuda.Event()
        self._consumed = torch.cuda.Event()
        self._consumed.record()
        self._pending = False
        # number of real images in the static batch buffers (a partial last batch of an epoch: the reference's DataLoader does
        # not drop it, main.py:43 / utils.py:452-470); word 11 of the per-step block, read by the loss kernel
        self._n_valid = self.B
        self._next_n_valid = self.B
        self.dlogits = torch.zeros((self.B, model.num_classes), dtype=torch.float32, device=self.dev)
        # epoch record (metrics=True): [loss_sum, correct, count] of vitb_eval_metrics (its unmixed loss_sum is not reported), then the
        # sum of step loss * n_valid (vitb_train_loss_accumulate)
        self.metrics = bool(metrics)
        self._record = torch.zeros(4, dtype=torch.float64, device=self.dev) if self.metrics else None
        self._record_ws = torch.zeros(ops.eval_metrics_ws_bytes() // 8, dtype=torch.float64, device=self.dev) if self.metrics else None
        self.logits: Optional[torch.Tensor] = None
        self.hyper_dev = torch.zeros(16, dtype=torch.float32, device=self.dev)
        # nn.Dropout(p) of the blocks (layers.py:35, 38, 102): each block owns a mask stream (seed), the step index is word 10 of
        # the per-step block (as an integer), so that graph replays draw fresh masks
        self.drops = None
        if model.p_drop > 0.0:
            from .layers import _new_drop_seed
            step_dev = self.hyper_dev.view(torch.int32)[10:11]
            self.drops = []
            for blk in model.enc:
                if blk._drop_seed is None:
                    blk._drop_seed = _new_drop_seed()
                # data parallel: every rank draws its own masks (per-rank offset of the stream seed, SURVEY.md §8e)
                seed = (blk._drop_seed + 0x9E3779B97F4A7C15 * self._rank) & 0xFFFFFFFFFFFFFFFF
                self.drops.append(Fn.Drop(p=float(model.p_drop), seed=seed, step_dev=step_dev))
        # ring of pinned slots: the async H2D of step k must not see the host writing step k+1's values
        self.hyper_host = torch.zeros((1024, 16), dtype=torch.float32).pin_memory()
        self.step_count = 0
        self._bufs: Dict[str, torch.Tensor] = {}
        self._graph: Optional[torch.cuda.CUDAGraph] = None
        self._comm_stream = torch.cuda.Stream(device=self.dev) if self.overlap_comm else None
        self.launches_per_step = 0  # filled by the first (eager) step
        # Deferred second passes of the split reductions (one flush launch before the optimiser instead of ~7 per layer) and weight
        # gradients on a second stream (they are off the critical path of backward).  Both need every wgrad / LayerNorm-backward
        # call to own its partial-sum workspace: an arena sized from the library's workspace queries.  bf16 path only; with
        # per-layer NCCL buckets ("overlap") the gradients must be final layer by layer, so neither applies there.
        self._defer = (self.act == torch.bfloat16 and not self.overlap_comm and os.environ.get("VITB_DEFER", "1") != "0")
        self._arena = torch.empty(self._arena_bytes(), dtype=torch.uint8, device=self.dev) if self._defer else None
        self.defer_bytes_used = 0
        ws_mode = int(os.environ.get("VITB_WGRAD_STREAM", "2")) if self._defer else 0
        self._side = None
        self._main_stream = None
        # second passes of a layer's reductions on the side stream right after that layer's backward (instead of all at the end):
        # +0.4-1.1 % on the 384-wide models (B = 1024 / 128, T = 65 / 17), -1.4 % on the 768 / 3072 model, whose flushes are large
        # enough to compete with the critical path (profiles/r2_flush_per_layer_ab.md) -> on for small weight matrices only
        env = os.environ.get("VITB_FLUSH_PER_LAYER")
        self._flush_per_layer = (env != "0") if env is not None else (model.hidden * max(model.hidden, model.mlp_hidden) <= 384 * 1536)
        # ... and, on one GPU, the optimiser step of that layer's parameters right behind it (with several GPUs the exchange comes first)
        self._opt_per_layer = self._flush_per_layer and self.world == 1 and os.environ.get("VITB_OPT_PER_LAYER", "1") != "0"
        self._opt_done_from = 0
        if ws_mode >= 1:
            if ws_mode >= 2:  # critical path on a high-priority stream: its pending CTAs get the SMs first
                self._main_stream = torch.cuda.Stream(device=self.dev, priority=-1)
            self._side = Fn.SideStream(torch.cuda.Stream(device=self.dev))

    # -- static buffers ---------------------------------------------------------------------------
    def _alloc(self, scope: str):
        def alloc(name: str, shape: tuple, dtype: torch.dtype) -> torch.Tensor:
            key = f"{scope}.{name}"
            t = self._bufs.get(key)
            if t is None:
                # "dxL" (gradient of the last block's output): only its cls rows are ever written, the rest must read as zero
                t = (torch.zeros if name == "dxL" else torch.empty)(shape, dtype=dtype, device=self.dev)
                self._bufs[key] = t
            return t
        return alloc

    def _arena_bytes(self) -> int:
        from . import _lib
        lib, dm, m = _lib.load(), self.dm, self.model
        rows, H, M = dm.rows, dm.H, dm.M
        ln = int(lib.vitb_layernorm_bwd_ws_bytes(rows, H))
        pair = lambda N, K: max(ops.wgrad_ws_bytes(rows, N, K), ops.bwd_fused_ws_bytes(rows, N, K))  # noqa: E731  (whichever path runs)
        per_layer = pair(H, H) + ops.wgrad_ws_bytes(rows, 3 * H, H) + ln
        if dm.use_mlp:
            per_layer += pair(H, M) + pair(M, H) + ln + int(lib.vitb_colsum_ws_bytes(rows, H))
        per_layer += 8 * 256  # alignment of every piece
        return m.num_layers * per_layer + int(lib.vitb_layernorm_bwd_ws_bytes(self.B, H)) + (1 << 20)

    def activation_bytes(self) -> int:
        return sum(t.numel() * t.element_size() for t in self._bufs.values())

    # -- the kernel sequence ----------------------------------------------------------------------
    def _allreduce(self, bucket: Tuple[int, int], last: bool = False) -> None:
        if self.world == 1:
            return
        if self._dp_mode in ("none", "fused"):  # none: diagnostic only (replicas drift apart); fused: the optimiser kernel does it
            return
        if self.overlap_comm:
            allreduce_bucket(self.G, bucket, self.pg, self._comm_stream)
        elif last:
            allreduce_bucket(self.G, (0, self.n), self.pg, None)

    def _body(self) -> None:
        m, dm = self.model, self.dm
        B, T, H, Cn = self.B, m.num_tokens, m.hidden, m.num_classes
        emb_w, emb_b, cls, pos = self.stem_p
        emb_w_c = self.store.layout.view(self.C, "emb.weight") if self.C is not self.P else None
        x, words = Fn.stem_fwd(self.img, emb_w, emb_w_c, emb_b, cls, pos, m.patch, self.act, self._alloc("stem"))
        saved = []
        for i in range(m.num_layers):
            x, sv = Fn.encoder_fwd(x, self.lc[i], self.lp[i], dm, self._alloc(f"l{i}"), drop=self.drops[i] if self.drops else None)
            saved.append(sv)
        ln_w, ln_b, fc_w_c, fc_b = self.head_p
        self.logits, hsaved = Fn.head_fwd(x, ln_w, ln_b, fc_w_c, fc_b, B, T, H, Cn, m.is_cls_token, self._alloc("head"))
        n_valid_dev = self.hyper_dev.view(torch.int32)[11:12]
        if self.mixed_targets:
            ops.ls_ce(self.logits, self.labels, self.loss, self.dlogits, self.smoothing, 1.0, labels_b=self.labels_b, lam_dev=self.hyper_dev[9:10],
                      n_valid_dev=n_valid_dev, ws=self._ls_ws)
        else:
            ops.ls_ce(self.logits, self.labels, self.loss, self.dlogits, self.smoothing, 1.0, n_valid_dev=n_valid_dev, ws=self._ls_ws)
        if self.metrics:  # training accuracy is against the first target (network.py:206)
            ops.eval_metrics(self.logits, self.labels, self._record[:3], self._record_ws, self.smoothing, n_valid_dev=n_valid_dev)
            ops.train_loss_accumulate(self.loss, self._record[3:], self.B, n_valid_dev=n_valid_dev)

        self._opt_done_from = self.n  # elements [_opt_done_from, n) have had their optimiser step on the side stream
        self._backward(hsaved, saved, words)
        n = self.n
        if self._fused_dp is not None:
            f = self._fused_dp
            ops.dp_reduce_adam(f["g"], f["p"], f["c"], f["flags"], self.Mo, self.V, f["sync"], n, f["rank"], self.world, hyper_dev=self.hyper_dev,
                               optimizer=0 if self.optimizer == "adam" else 1)
        else:
            self._optimizer_slice(0, self._opt_done_from)

    def _optimizer_slice(self, lo: int, hi: int) -> None:
        """Optimiser step on elements [lo, hi) of the flat buffers (slot boundaries: 64-element aligned)."""
        if hi <= lo:
            return
        shadow = self.C[lo:hi] if self.C is not self.P else None
        if self.optimizer == "adam":
            ops.adam(self.P[lo:hi], self.G[lo:hi], self.Mo[lo:hi], self.V[lo:hi], shadow, hyper_dev=self.hyper_dev)
        else:
            ops.sgd(self.P[lo:hi], self.G[lo:hi], self.Mo[lo:hi], shadow, hyper_dev=self.hyper_dev)

    def _backward(self, hsaved, saved, words) -> None:
        m, dm = self.model, self.dm
        B, T, H, Cn = self.B, m.num_tokens, m.hidden, m.num_classes
        ln_w, ln_b, fc_w_c, fc_b = self.head_p
        if self._main_stream is not None:  # run the critical path on the high-priority stream
            outer = torch.cuda.current_stream()
            self._main_stream.wait_stream(outer)
            with torch.cuda.stream(self._main_stream):
                self._backward_kernels(hsaved, saved, words, B, T, H, Cn, ln_w, fc_w_c)
            outer.wait_stream(self._main_stream)
        else:
            self._backward_kernels(hsaved, saved, words, B, T, H, Cn, ln_w, fc_w_c)

    def _backward_kernels(self, hsaved, saved, words, B, T, H, Cn, ln_w, fc_w_c) -> None:
        m, dm, side = self.model, self.dm, self._side
        if self._defer:
            ops.defer_begin(self._arena)
        g_ln_w, g_ln_b, g_fc_w, g_fc_b = self.head_g
        dx = Fn.head_bwd(self.dlogits, hsaved, ln_w, fc_w_c, g_ln_w, g_ln_b, g_fc_w, g_fc_b, B, T, H, Cn, m.is_cls_token, self.act,
                         self._alloc("headb"), dx_prezeroed=True, side=side)
        self._allreduce(self.buckets[-1])
        done = {}
        # (bf16 only: the fp32 check mode keeps the module path's kernel chain, with which it is compared bit for bit)
        fuse_below = (Fn.ln_gelu_fused() and dm.use_mlp and self.act == torch.bfloat16 and (not self.drops or Fn._drop_fused(dm.rows)))
        dz2_in = None
        for i in reversed(range(m.num_layers)):
            # backward scratch ping-pongs between two sets; with weight gradients on the side stream a set may only be rewritten
            # once the side-stream kernels of the layer that used it last (i + 2) have read it
            if side is not None and (i + 2) in done:
                torch.cuda.current_stream().wait_event(done[i + 2])
            # block i's last kernel (LayerNorm-1 backward) also writes block i - 1's dz2 and b2 gradient; that buffer rotates over
            # three, not two: block i + 1's side-stream wgrad may still be reading its dz2 (the wait above covers i + 2 only)
            below = None
            if fuse_below and i > 0:
                dz2_b = self._alloc(f"bwd_dz2_{(i - 1) % 3}")("dz2", (dm.rows, dm.H), self.act)
                below = (saved[i - 1][4][6], dz2_b, self.lg[i - 1].b2, self.drops[i - 1] if self.drops else None)
            dx = Fn.encoder_bwd(dx, saved[i], self.lc[i], self.lp[i], self.lg[i], dm, self._bwd_alloc(i),
                                drop=self.drops[i] if self.drops else None, side=side, dz2_in=dz2_in, below=below)
            dz2_in = below[1] if below is not None else None
            if side is not None:
                if self._defer and self._flush_per_layer:
                    # this layer's second passes on the side stream (ordered after everything issued so far on both streams),
                    # while the main stream goes on with the next layer's backward; on one GPU the optimiser step of the
                    # layer's slice of the flat buffers follows at once (its gradients are final, its weights no longer read)
                    side.run(ops.defer_flush_partial)
                    if self._opt_per_layer:
                        lo = self.buckets[1 + i][0]
                        hi = self._opt_done_from
                        side.run(lambda lo=lo, hi=hi: self._optimizer_slice(lo, hi))
                        self._opt_done_from = lo
                done[i] = side.done_event()
            self._allreduce(self.buckets[1 + i])
        g_emb_w, g_emb_b, g_cls, g_pos = self.stem_g
        Fn.stem_bwd(self.img, words, dx, g_emb_w, g_emb_b, g_cls, g_pos, m.patch)
        if side is not None:
            side.join()
        if self._defer:
            ops.defer_flush()
            used = ops.defer_used()
            if used > self._arena.numel():
                raise RuntimeError(f"deferred-reduction arena too small ({self._arena.numel()} < {used} bytes): engine sizing bug")
            self.defer_bytes_used = used
        self._allreduce(self.buckets[0], last=True)
        if self._comm_stream is not None:
            torch.cuda.current_stream().wait_stream(self._comm_stream)

    def _bwd_alloc(self, i: int):
        shared = self._alloc("bwd")
        pp = self._alloc(f"bwd{i & 1}")
        if self._side is not None:  # everything ping-pongs: side-stream wgrads of layer i + 1 still read that layer's scratch
            return pp

        def alloc(name: str, shape: tuple, dtype: torch.dtype) -> torch.Tensor:
            return pp(name, shape, dtype) if name == "dx" else shared(name, shape, dtype)
        return alloc

    # -- public API -------------------------------------------------------------------------------
    def set_lr(self, lr: float) -> None:
        self.lr = float(lr)

    def _check_batch(self, img: torch.Tensor, labels: torch.Tensor, labels_b: Optional[torch.Tensor]) -> int:
        """Number of images of a batch for the fixed-size step: 1..B.  The step is a static kernel sequence over B rows (a CUDA
        graph); a smaller batch — the last one of an epoch, the reference's DataLoader has no drop_last — occupies the first n
        rows, the loss kernel averages over n and zeroes the gradient of the other rows."""
        if img.dim() != 4 or tuple(img.shape[1:]) != tuple(self.img.shape[1:]):
            raise ValueError(f"expected images of shape (n, {', '.join(str(d) for d in self.img.shape[1:])}) with n <= {self.B}, got {tuple(img.shape)}")
        n = int(img.shape[0])
        if not 1 <= n <= self.B:
            raise ValueError(f"batch of {n} images: this engine was built for batches of 1..{self.B} (batch_size={self.B})")
        if labels.dim() != 1 or labels.shape[0] != n or (labels_b is not None and tuple(labels_b.shape) != (n,)):
            raise ValueError(f"expected {n} labels, got {tuple(labels.shape)}" + (f" / {tuple(labels_b.shape)}" if labels_b is not None else ""))
        if labels_b is not None and not self.mixed_targets:
            raise ValueError("construct the engine with mixed_targets=True to train on (label, rand_label, lambda) batches")
        return n

    @staticmethod
    def _copy_rows(dst: torch.Tensor, src: torch.Tensor, n: int) -> None:
        if n == dst.shape[0]:
            dst.copy_(src, non_blocking=True)
        else:  # rows >= n: defined, finite values (their gradient is zeroed by the loss kernel)
            dst[:n].copy_(src, non_blocking=True)
            dst[n:].zero_()

    def load_batch(self, img: torch.Tensor, labels: torch.Tensor, labels_b: Optional[torch.Tensor] = None) -> None:
        """Copy a batch of n <= batch_size images (pinned host or device tensors) into the static input buffers on the current stream."""
        n = self._check_batch(img, labels, labels_b)
        self._copy_rows(self.img, img, n)
        self._copy_rows(self.labels, labels, n)
        if self.mixed_targets:
            self._copy_rows(self.labels_b, labels if labels_b is None else labels_b, n)
        self._n_valid = n

    def prefetch(self, img: torch.Tensor, labels: torch.Tensor, labels_b: Optional[torch.Tensor] = None, lam: float = 1.0) -> None:
        """Start copying the NEXT batch (pinned host tensors) to the device on a side stream; the following `step()` (called
        without arguments) trains on it.  Called right after `step()` returns, the host-to-device transfer overlaps that step's
        kernels — the role the DataLoader's pinned-memory prefetch plays for the reference (main.py:175)."""
        n = self._check_batch(img, labels, labels_b)
        cs = self._copy_stream
        cs.wait_event(self._consumed)  # the previously staged batch has been moved into the input buffers
        with torch.cuda.stream(cs):
            self._copy_rows(self._img_stage, img, n)
            self._copy_rows(self._labels_stage, labels, n)
            if self.mixed_targets:
                self._copy_rows(self._labels_b_stage, labels if labels_b is None else labels_b, n)
            self._staged.record(cs)
        self._next_n_valid = n
        self._next_lam = float(lam) if labels_b is not None else 1.0
        self._pending = True

    def step(self, img: Optional[torch.Tensor] = None, labels: Optional[torch.Tensor] = None, labels_b: Optional[torch.Tensor] = None,
             lam: float = 1.0) -> torch.Tensor:
        """One optimisation step.  Returns the (device) loss tensor of this step; no host synchronisation.
        `labels_b`, `lam`: the second targets and the mixing weight of a CutMix / MixUp batch (engine built with mixed_targets)."""
        if img is not None:
            self.load_batch(img, labels, labels_b)
            self._lam = float(lam) if labels_b is not None else 1.0
        elif self._pending:
            cur = torch.cuda.current_stream()
            cur.wait_event(self._staged)
            self.img.copy_(self._img_stage, non_blocking=True)
            self.labels.copy_(self._labels_stage, non_blocking=True)
            if self.mixed_targets:
                self.labels_b.copy_(self._labels_b_stage, non_blocking=True)
            self._lam = self._next_lam
            self._n_valid = self._next_n_valid
            self._consumed.record(cur)
            self._pending = False
        self.step_count += 1
        if self.optimizer == "adam":
            h = adam_hyper(self.step_count, self.lr, self.betas[0], self.betas[1], self.eps, self.weight_decay, 1.0 / self.world)
        else:
            h = sgd_hyper(self.lr, self.momentum, self.weight_decay, 1.0 / self.world)
        slot = self.hyper_host[self.step_count % self.hyper_host.shape[0]]
        slot[:9] = torch.tensor(h, dtype=torch.float32)
        slot[9] = self._lam
        slot.view(torch.int32)[10] = self.step_count & 0x7FFFFFFF  # dropout mask step
        slot.view(torch.int32)[11] = self._n_valid
        self.hyper_dev.copy_(slot, non_blocking=True)
        if self._l2_persist and self.step_count == 1 and self.C is not self.P:
            # bf16 weights stay in a persisting carve-out of L2 (16 MB of 126): the resident GEMMs' weight blocks are L2 hits
            ops.set_l2_persisting_window(self.C[:self.n], max(16 << 20, self.n * 2))
        if not self.use_graph:
            n0 = ops.launch_count()
            self._body()
            self.launches_per_step = ops.launch_count() - n0
        elif self._graph is None:
            # warm-up run (allocates every static buffer, primes NCCL), then capture
            n0 = ops.launch_count()
            self._body()
            self.launches_per_step = ops.launch_count() - n0
            torch.cuda.current_stream().synchronize()
            # the warm-up already applied this step's update; capture for the following ones
            g = torch.cuda.CUDAGraph()
            snapshot = (self.P.clone(), self.Mo.clone(), self.V.clone(), self.loss.clone())
            with torch.cuda.graph(g):
                self._body()
            # capture does not execute, but restore state anyway in case a backend ran work eagerly
            self.P.copy_(snapshot[0]); self.Mo.copy_(snapshot[1]); self.V.copy_(snapshot[2]); self.loss.copy_(snapshot[3])
            if self.C is not self.P:
                ops.cast_f32_to_bf16(self.P, self.C)
            self._graph = g
        else:
            self._graph.replay()
        return self.loss

    def train_metrics(self, reset: bool = True) -> Dict[str, float]:
        """{"loss", "acc", "n"} of the steps since the last reset: the n-weighted mean of the step losses (for CutMix / MixUp batches
        the mixed objective, network.py:149-167), the accuracy of the logits against the first labels, and the number of images.  One
        host synchronisation; with a process group the record is first summed over the ranks (a collective: call on all ranks)."""
        if not self.metrics:
            raise RuntimeError("construct the engine with metrics=True to keep an epoch record")
        t = self._record
        if self.pg is not None and self.world > 1:
            import torch.distributed as dist
            t = t.clone()
            dist.all_reduce(t, group=self.pg)
        _, correct, n, loss_sum = t.tolist()
        if reset:
            self._record.zero_()
        n = int(n)
        return {"loss": loss_sum / max(n, 1), "acc": correct / max(n, 1), "n": n}

    def sync_weights(self) -> None:
        """Call after writing parameters from outside the step (load_state_dict / load_checkpoint / manual edits on the packed
        model): re-derives the bf16 weight copy the kernels read from the fp32 master and, with world > 1, makes rank 0's
        parameters those of every replica.  The step itself keeps both in sync (the optimiser kernel writes both)."""
        if self.world > 1:
            import torch.distributed as dist
            dist.broadcast(self.P, src=0, group=self.pg)
        if self.C is not self.P:
            ops.cast_f32_to_bf16(self.P, self.C)

    def load_checkpoint(self, ckpt, strict: bool = False):
        """schedule.load_checkpoint into the engine's model, followed by sync_weights(); restores the optimiser state too when the
        checkpoint carries one (`optimizer_states` as written by `checkpoint()`)."""
        from .schedule import load_checkpoint
        if isinstance(ckpt, (str, bytes)) or hasattr(ckpt, "__fspath__"):
            ckpt = torch.load(ckpt, map_location="cpu")
        res = load_checkpoint(self.model, ckpt, strict=strict)
        self.sync_weights()
        if isinstance(ckpt, dict) and ckpt.get("optimizer_states"):
            self.load_optimizer_state(ckpt["optimizer_states"][0], ckpt.get("global_step"))
        return res

    def optimizer_state(self) -> dict:
        """torch.optim-style optimiser state of the flat parameter buffer: {"step", "exp_avg", "exp_avg_sq"} (Adam) or
        {"step", "momentum_buffer"} (SGD) as CPU tensors of `n` elements.  In the fused data-parallel mode every rank maintains
        the moments of its owned slice only (parallel.owned_slice): the slices are gathered here (a collective: call on all ranks)."""
        from .parallel import owned_slice
        bufs = {"exp_avg": self.Mo, "exp_avg_sq": self.V} if self.optimizer == "adam" else {"momentum_buffer": self.Mo}
        out = {"step": int(self.step_count)}
        for name, t in bufs.items():
            full = t[:self.n].clone()
            if self._fused_dp is not None:
                import torch.distributed as dist
                lo, hi = owned_slice(self.n, self._rank, self.world)
                full[:lo].zero_()
                full[hi:].zero_()
                dist.all_reduce(full, op=dist.ReduceOp.SUM, group=self.pg)
            out[name] = full.cpu()
        return out

    def load_optimizer_state(self, state: dict, step: Optional[int] = None) -> None:
        self.step_count = int(state.get("step", 0) if step is None else step)
        pairs = (("exp_avg", self.Mo), ("exp_avg_sq", self.V)) if self.optimizer == "adam" else (("momentum_buffer", self.Mo),)
        for name, t in pairs:
            src = state[name]
            if src.numel() != self.n:
                raise ValueError(f"optimizer state {name}: {src.numel()} elements, this model has {self.n}")
            t[:self.n].copy_(src.to(self.dev, torch.float32).flatten())

    def checkpoint(self, hyper_parameters: Optional[dict] = None, epoch: int = 0) -> dict:
        """The reference's checkpoint dict (main.py:234-237: "state_dict" with "model." keys + "hyper_parameters") extended with
        what Lightning also stores for resuming: "optimizer_states", "global_step", "epoch".  Collective when world > 1."""
        from .schedule import to_lightning_checkpoint
        ck = to_lightning_checkpoint(self.model, hyper_parameters)
        ck["optimizer_states"] = [self.optimizer_state()]
        ck["global_step"] = int(self.step_count)
        ck["epoch"] = int(epoch)
        return ck

    def grads(self) -> Dict[str, torch.Tensor]:
        """Views of the flat gradient buffer by state_dict name (of the LAST step; summed over ranks when world > 1)."""
        L = self.store.layout
        return {k: L.view(self.G, k) for k in L.slots if L.slots[k].off < self.n}
