"""Forward / backward of the ViT training step as explicit kernel sequences over libvitb200.

No autograd in here: each function launches the kernels of one block in order and returns what the
matching backward needs.  The module layer (layers.py / vit.py) wraps these in ``autograd.Function``s;
the training engine (engine.py) calls them directly on static buffers inside a CUDA graph.

`alloc(name, shape, dtype)` supplies output/scratch tensors: fresh ones under autograd, fixed ones in
the engine.  Activations are (rows, H) row-major with rows = B*T.
"""
from __future__ import annotations

import os
from dataclasses import dataclass
from typing import Callable, Optional

import torch

from . import ops
from .params import LayerViews

Alloc = Callable[[str, tuple, torch.dtype], torch.Tensor]


def default_alloc(device: torch.device) -> Alloc:
    def alloc(name: str, shape: tuple, dtype: torch.dtype) -> torch.Tensor:
        return torch.empty(shape, dtype=dtype, device=device)
    return alloc


@dataclass
class Dims:
    B: int
    T: int
    H: int
    heads: int
    M: int          # mlp_hidden
    use_mlp: bool = True

    @property
    def rows(self) -> int:
        return self.B * self.T

    @property
    def d(self) -> int:
        return self.H // self.heads

    @property
    def scale(self) -> float:  # layers.py:79,97: 1/sqrt(features), NOT 1/sqrt(head_dim)
        return 1.0 / (self.H ** 0.5)

    def check(self) -> None:
        if self.H % 128 != 0:
            raise ValueError(f"hidden={self.H} must be a multiple of 128 for the vectorised LayerNorm kernels")
        if self.H % self.heads != 0 or self.d not in (32, 64):
            raise ValueError(f"head_dim={self.H}/{self.heads} must be 32 or 64 for the fused attention kernel")
        if self.T > 128:
            raise ValueError(f"{self.T} tokens > 128: the fused short-sequence attention kernel keeps (T x T) on chip")
        if self.use_mlp and self.M % 128 != 0:
            raise ValueError(f"mlp_hidden={self.M} must be a multiple of 128")


class SideStream:
    """Weight-gradient GEMMs are off the backward pass's critical path (nothing reads dW before the optimiser): `run(fn)` issues
    fn's kernels on a second stream once everything issued so far on the current stream has been ordered before them, so they
    fill the SMs that the tails / prologues of the critical-path kernels leave idle.  The caller joins with `join()` before the
    gradients are read and keeps every buffer such a kernel reads untouched until then (or until `done_event()` of that point)."""

    def __init__(self, stream: "torch.cuda.Stream"):
        self.stream = stream

    def run(self, fn) -> None:
        self.stream.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(self.stream):
            fn()

    def done_event(self) -> "torch.cuda.Event":
        ev = torch.cuda.Event()
        ev.record(self.stream)
        return ev

    def join(self) -> None:
        torch.cuda.current_stream().wait_stream(self.stream)


def _bwd_fused_ok(rows: int, N: int, K: int, t: torch.Tensor) -> bool:
    """Use the one-pass backward of a Linear (ops.gemm_bwd_fused) for this shape / dtype (bf16, N <= 384)?  Opt-in
    (VITB_BWD_FUSED=1): measured on B200 it only equals dgrad + wgrad (66.5 vs 67.4 us at 66560 x 384 x 384; DESIGN.md 3c) — with the
    weight slice resident, 131 KB of shared memory are left to stream 128 KB of operands per row block, too little to cover the
    load latency — and it is slower at 8,320 rows, where its 29 MB of per-CTA dW partials dominate."""
    if os.environ.get("VITB_BWD_FUSED", "0") == "0":
        return False
    return ops.bwd_fused_ws_bytes(rows, N, K, ops.dt_of(t)) > 0


def _wgrad(side: Optional["SideStream"], *args, **kw) -> None:
    if side is None:
        ops.gemm_wgrad(*args, **kw)
    else:
        side.run(lambda: ops.gemm_wgrad(*args, **kw))


@dataclass
class Drop:
    """Training-mode nn.Dropout(p) of one encoder block (layers.py:35, 38, 102).  Its three sites (0: after out_project, 1: after the
    first GELU, 2: after the second GELU) draw their keep masks from (seed, site, step); nothing is stored for the backward pass,
    which regenerates them.  `step_dev` (1-element int32 device tensor) replaces `step` inside a captured CUDA graph."""
    p: float
    seed: int
    step: int = 0
    step_dev: Optional[torch.Tensor] = None

    def __call__(self, x: torch.Tensor, residual: Optional[torch.Tensor], out: torch.Tensor, site: int) -> None:
        ops.dropout(x, residual, out, self.p, self.seed, site, self.step, self.step_dev)

    def desc(self, site: int):
        """The site's descriptor for the kernels that apply the mask themselves (GEMM epilogues, GELU / LayerNorm backward)."""
        return ops.drop_desc(self.p, self.seed, site, self.step, self.step_dev)


# rows from which the in-kernel masks win: measured on B200 with dropout 0.1, 66,560 rows 6.644 vs 6.736 ms per step (+1.4 %),
# 8,320 rows 1.585 vs 1.520 ms (-4 %): ten Philox rounds per eight elements cost the eight epilogue warps of a GEMM tile about as much
# as the GELU does, which a large problem hides behind the other stream's MMAs and a single-wave problem does not, and the
# stand-alone pass over a small tensor is a 4 us launch
DROP_FUSED_MIN_ROWS = 16384


def _drop_fused(rows: int = 1 << 30) -> bool:
    """Dropout masks inside the producing / consuming kernels, or as separate elementwise passes (the round-1 path, kept as the
    A/B and as what the fused path is tested against).  VITB_DROP_FUSED=1 / 0 forces one of them; default: by problem size."""
    v = os.environ.get("VITB_DROP_FUSED", "auto")
    if v in ("0", "1"):
        return v == "1"
    return rows >= DROP_FUSED_MIN_ROWS


def ln_gelu_fused() -> bool:
    """LayerNorm-1 backward of block i + 1 also writes dz2 of block i (the GELU backward of its second MLP Linear and that Linear's
    bias gradient): one launch and one read of the block-output gradient less per block.  Opt-in (VITB_LN_GELU_FUSED=1): measured
    on B200 the fused kernel is faster than its two parts in isolation (76 vs 46 + 41 us at 66,560 rows) but the step is not
    (6.19 vs 6.17 ms at B = 1024, 1.391 vs 1.375 ms at B = 128, 2.211 vs 2.225 ms at T = 17): the GELU arithmetic moves from a
    78-register kernel that shares SMs with the side-stream weight-gradient GEMMs into a 128-register one that does not."""
    return os.environ.get("VITB_LN_GELU_FUSED", "0") != "0"


# ---------------------------------------------------------------------------------------------
# attention block: layers.py:90-103  (x -> out_project(attn(QKV(x))))
# ---------------------------------------------------------------------------------------------
def mhsa_fwd(x: torch.Tensor, c: LayerViews, p: LayerViews, dm: Dims, alloc: Alloc, residual: Optional[torch.Tensor],
             attn_map: Optional[torch.Tensor] = None, drop: Optional[Drop] = None):
    """x (rows,H) act -> y (rows,H) = dropout(out_project(attention(x))) (+ residual).  Returns (y, saved)."""
    rows, H, act = dm.rows, dm.H, x.dtype
    qkv = alloc("qkv", (rows, 3 * H), act)
    ops.gemm_fwd(x, c.wqkv, p.bqkv, None, qkv, None, rows, 3 * H, H)
    o = alloc("o", (rows, H), act)
    lse = alloc("lse", (dm.B, dm.heads, dm.T), torch.float32)
    ops.attn_fwd(qkv, o, lse, attn_map, dm.B, dm.T, dm.heads, dm.d, dm.scale)
    y = alloc("x1", (rows, H), act)
    if drop is None or _drop_fused(rows):                                           # layers.py:102, then "+ x" of layers.py:45
        ops.gemm_fwd(o, c.wo, p.bo, residual, y, None, rows, H, H, drop=drop.desc(0) if drop is not None else None)
    else:
        ops.gemm_fwd(o, c.wo, p.bo, None, y, None, rows, H, H)
        drop(y, residual, y, 0)
    return y, (x, qkv, o, lse)


def mhsa_bwd(dy: torch.Tensor, saved, c: LayerViews, g: LayerViews, dm: Dims, alloc: Alloc, bo_done: bool = False,
             drop: Optional[Drop] = None, side: Optional[SideStream] = None, dy_masked: Optional[torch.Tensor] = None):
    """dy (rows,H) = grad of the block's attention branch output.  Fills g.wqkv,g.bqkv,g.wo,(g.bo); returns grad of x.
    `dy_masked`: dy already taken through the out_project Dropout's mask (by the LayerNorm backward that produced dy)."""
    x, qkv, o, lse = saved
    rows, H, act = dm.rows, dm.H, dy.dtype
    if dy_masked is not None:
        dy = dy_masked
    elif drop is not None:  # gradient of the out_project output = dy through the same mask (dy itself is still needed by the caller)
        dya = alloc("dao", (rows, H), act)
        drop(dy, None, dya, 0)
        dy = dya
    do = alloc("do", (rows, H), act)
    if bo_done and _bwd_fused_ok(rows, H, H, dy):
        ops.gemm_bwd_fused(dy, o, c.wo, None, do, g.wo, None, rows, H, H)            # out_project: dgrad + wgrad in one pass over dy
    else:
        _wgrad(side, dy, o, g.wo, None if bo_done else g.bo, rows, H, H)
        ops.gemm_dgrad(dy, c.wo, None, do, rows, H, H)
    dqkv = alloc("dqkv", (rows, 3 * H), act)
    ops.attn_bwd(qkv, o, do, lse, dqkv, dm.B, dm.T, dm.heads, dm.d, dm.scale)
    _wgrad(side, dqkv, x, g.wqkv, g.bqkv, rows, 3 * H, H)
    dx = alloc("dxn", (rows, H), act)
    ops.gemm_dgrad(dqkv, c.wqkv, None, dx, rows, 3 * H, H)
    return dx


# ---------------------------------------------------------------------------------------------
# encoder block: layers.py:44-48
# ---------------------------------------------------------------------------------------------
def encoder_fwd(x: torch.Tensor, c: LayerViews, p: LayerViews, dm: Dims, alloc: Alloc, attn_map: Optional[torch.Tensor] = None,
                drop: Optional[Drop] = None, save_preact: bool = True):
    """`save_preact=False` (forward only, no backward will follow): the two MLP GEMMs do not store their pre-GELU values z1 / z2,
    which then come back as None in the saved tuple."""
    rows, H, M, act = dm.rows, dm.H, dm.M, x.dtype
    xn = alloc("xn", (rows, H), act)
    mean1 = alloc("mean1", (rows,), torch.float32)
    rstd1 = alloc("rstd1", (rows,), torch.float32)
    ops.layernorm_fwd(x, H, p.ln1_w, p.ln1_b, xn, mean1, rstd1, rows, H)
    x1, att_saved = mhsa_fwd(xn, c, p, dm, alloc, residual=x, attn_map=attn_map, drop=drop)  # out = attention(la1(x)) + x
    if not dm.use_mlp:
        return x1, (x, mean1, rstd1, att_saved, None)
    x1n = alloc("x1n", (rows, H), act)
    mean2 = alloc("mean2", (rows,), torch.float32)
    rstd2 = alloc("rstd2", (rows,), torch.float32)
    ops.layernorm_fwd(x1, H, p.ln2_w, p.ln2_b, x1n, mean2, rstd2, rows, H)
    z1 = alloc("z1", (rows, M), act) if save_preact else None
    a1 = alloc("a1", (rows, M), act)
    z2 = alloc("z2", (rows, H), act) if save_preact else None
    x2 = alloc("x2", (rows, H), act)
    if drop is not None and _drop_fused(rows):                                     # mlp[0..2]: the mask in the epilogue, after the GELU
        ops.gemm_fwd(x1n, c.w1, p.b1, None, a1, z1, rows, M, H, gelu=True, drop=drop.desc(1))
        ops.gemm_fwd(a1, c.w2, p.b2, x1, x2, z2, rows, H, M, gelu=True, drop=drop.desc(2))   # mlp[3..5], + out
        return x2, (x, mean1, rstd1, att_saved, (x1, x1n, mean2, rstd2, z1, a1, z2))
    ops.gemm_fwd(x1n, c.w1, p.b1, None, a1, z1, rows, M, H, gelu=True)            # mlp[0], mlp[1]
    if drop is None:
        ops.gemm_fwd(a1, c.w2, p.b2, x1, x2, z2, rows, H, M, gelu=True)            # mlp[3], mlp[4], + out
    else:
        drop(a1, None, a1, 1)                                                      # mlp[2]
        ops.gemm_fwd(a1, c.w2, p.b2, None, x2, z2, rows, H, M, gelu=True)          # mlp[3], mlp[4]
        drop(x2, x1, x2, 2)                                                        # mlp[5], + out
    return x2, (x, mean1, rstd1, att_saved, (x1, x1n, mean2, rstd2, z1, a1, z2))


def encoder_bwd(dout: torch.Tensor, saved, c: LayerViews, p: LayerViews, g: LayerViews, dm: Dims, alloc: Alloc,
                drop: Optional[Drop] = None, side: Optional[SideStream] = None, dz2_in: Optional[torch.Tensor] = None,
                below: Optional[tuple] = None):
    """dout = grad of the block output; fills every field of g; returns grad of the block input.  `drop`: the same Drop the
    forward ran with (masks are regenerated, not stored).

    Cross-block fusion (both optional, bf16 or fp32): `dz2_in` = this block's dz2 (gradient entering its second MLP Linear) and
    g.b2, already produced by the block above; `below` = (z2, dz2, g_b2, drop) of the block BELOW: this block's last kernel, the
    LayerNorm-1 backward that forms the block-input gradient, then also writes that block's dz2 = dropout(dx) * gelu'(z2) and its
    column sums g_b2 (ops.layernorm_bwd_fused), which replaces that block's GELU-backward launch."""
    x, mean1, rstd1, att_saved, mlp_saved = saved
    rows, H, M, act = dm.rows, dm.H, dm.M, dout.dtype
    fused_drop = drop is not None and _drop_fused(rows)
    dya = None
    if dm.use_mlp:
        x1, x1n, mean2, rstd2, z1, a1, z2 = mlp_saved
        if dz2_in is not None:
            dz2 = dz2_in
        else:
            dz2 = alloc("dz2", (rows, H), act)
            if drop is None or fused_drop:                               # second GELU (layers.py:37) + db2, mlp[5]'s mask on the way in
                ops.gelu_bwd_colsum(dout, z2, dz2, g.b2, rows, H, drop=drop.desc(2) if drop is not None else None)
            else:
                dg2 = alloc("dg2", (rows, H), act)
                drop(dout, None, dg2, 2)                                 # mlp[5] backward
                ops.gelu_bwd_colsum(dg2, z2, dz2, g.b2, rows, H)
        dz1 = alloc("dz1", (rows, M), act)
        b1_done = False
        if drop is None and _bwd_fused_ok(rows, H, M, dz2):
            # mlp[3]: dgrad (first GELU's backward in the epilogue) + wgrad in one pass over dz2; the column sums of dz1 are db1
            ops.gemm_bwd_fused(dz2, a1, c.w2, z1, dz1, g.w2, g.b1, rows, H, M)
            b1_done = True
        else:
            _wgrad(side, dz2, a1, g.w2, None, rows, H, M)
            # first GELU's backward — and mlp[2]'s mask: the two commute — fused in the epilogue
            ops.gemm_dgrad(dz2, c.w2, z1, dz1, rows, H, M, drop=drop.desc(1) if fused_drop else None)
            if drop is not None and not fused_drop:
                drop(dz1, None, dz1, 1)
        dx1n = alloc("dx1n", (rows, H), act)
        if b1_done and _bwd_fused_ok(rows, M, H, dz1):
            ops.gemm_bwd_fused(dz1, x1n, c.w1, None, dx1n, g.w1, None, rows, M, H)   # mlp[0]
        else:
            _wgrad(side, dz1, x1n, g.w1, None if b1_done else g.b1, rows, M, H)
            ops.gemm_dgrad(dz1, c.w1, None, dx1n, rows, M, H)
        dx1 = alloc("dx1", (rows, H), act)
        # grad of x1 = residual branch (dout) + LN2 backward; its column sums are out_project's bias grad.  With dropout the
        # out_project output gradient is the MASKED dx1: the fused kernel writes it as a second output and sums THAT; the
        # unfused path masks it in mhsa_bwd and takes the bias gradient from the wgrad instead
        if fused_drop:
            dya = alloc("dao", (rows, H), act)
            ops.layernorm_bwd_fused(dx1n, x1, H, p.ln2_w, mean2, rstd2, dout, dx1, H, g.ln2_w, g.ln2_b, None, dya, g.bo, rows, H,
                                    drop=drop.desc(0))
            bo_done = True
        else:
            bo_done = drop is None
            ops.layernorm_bwd(dx1n, x1, H, p.ln2_w, mean2, rstd2, dout, dx1, H, g.ln2_w, g.ln2_b, g.bo if bo_done else None, rows, H)
    else:
        dx1 = dout
        bo_done = False
    dxn = mhsa_bwd(dx1, att_saved, c, g, dm, alloc, bo_done=bo_done, drop=drop, side=side, dy_masked=dya)
    dx = alloc("dx", (rows, H), act)
    if below is not None:
        z2_b, dz2_b, g_b2_b, drop_b = below
        ops.layernorm_bwd_fused(dxn, x, H, p.ln1_w, mean1, rstd1, dx1, dx, H, g.ln1_w, g.ln1_b, z2_b, dz2_b, g_b2_b, rows, H,
                                drop=drop_b.desc(2) if drop_b is not None else None)
    else:
        ops.layernorm_bwd(dxn, x, H, p.ln1_w, mean1, rstd1, dx1, dx, H, g.ln1_w, g.ln1_b, None, rows, H)
    return dx


# ---------------------------------------------------------------------------------------------
# stem: vit.py:66-70   and   head: vit.py:72-76
# ---------------------------------------------------------------------------------------------
def stem_fwd(img: torch.Tensor, emb_w, emb_w_c, emb_b, cls, pos, P: int, act: torch.dtype, alloc: Alloc):
    """emb_w: fp32 master; emb_w_c: the same weight in the activation dtype (bf16 shadow) or None.  Returns (x0, words)."""
    B, _, S, _ = img.shape
    has_cls = cls is not None
    T = P * P + (1 if has_cls else 0)
    H, K = emb_w.shape
    x0 = alloc("x0", (B * T, H), act)
    words = alloc("words", (B * P * P, K), act) if (act == torch.bfloat16 and emb_w_c is not None) else None
    ops.patch_embed_fwd(img, emb_w, emb_w_c if words is not None else None, emb_b, cls, pos, x0, words, P, has_cls)
    return x0, words


def stem_bwd(img: torch.Tensor, words, dx0: torch.Tensor, g_emb_w, g_emb_b, g_cls, g_pos, P: int) -> None:
    ops.patch_embed_bwd(img, words, dx0, g_emb_w, g_emb_b, g_cls, g_pos, P, g_cls is not None)


def head_fwd(x: torch.Tensor, ln_w, ln_b, fc_w_c, fc_b, B: int, T: int, H: int, C: int, is_cls: bool, alloc: Alloc):
    """x (B*T,H) act -> logits (B,C) fp32."""
    act = x.dtype
    if is_cls:
        src, stride = x, T * H          # LayerNorm reads out[:,0] in place (vit.py:73)
    else:
        src = alloc("pooled", (B, H), act)
        ops.pool_fwd(x, src, B, T, H, 1)  # out.mean(1), vit.py:75
        stride = H
    hn = alloc("hn", (B, H), act)
    mean = alloc("hmean", (B,), torch.float32)
    rstd = alloc("hrstd", (B,), torch.float32)
    ops.layernorm_fwd(src, stride, ln_w, ln_b, hn, mean, rstd, B, H)
    logits = alloc("logits", (B, C), torch.float32)
    ops.gemm_fwd(hn, fc_w_c, fc_b, None, logits, None, B, C, H, out_f32=True)
    return logits, (src, stride, hn, mean, rstd)


def head_bwd(dlogits: torch.Tensor, saved, ln_w, fc_w_c, g_ln_w, g_ln_b, g_fc_w, g_fc_b, B: int, T: int, H: int, C: int,
             is_cls: bool, act: torch.dtype, alloc: Alloc, dx_prezeroed: bool = False, side: Optional[SideStream] = None) -> torch.Tensor:
    """dlogits (B,C) fp32 -> grad of the encoder output (B*T,H) act (zeros where nothing flows).  `side`: stream for the weight
    gradient (off the critical path, like the encoder's)."""
    src, stride, hn, mean, rstd = saved
    _wgrad(side, dlogits, hn, g_fc_w, g_fc_b, B, C, H, dy_f32=True)
    dhn = alloc("dhn", (B, H), act)
    ops.gemm_dgrad(dlogits, fc_w_c, None, dhn, B, C, H, dy_f32=True)
    dx = alloc("dxL", (B * T, H), act)
    if is_cls and dx_prezeroed:
        # `alloc` hands out a static buffer whose non-cls rows are zero and stay zero (TrainEngine): the LayerNorm backward writes
        # its B rows straight into the cls rows of dx (row stride T * H) — no pooled gradient, no scatter launch
        ops.layernorm_bwd(dhn, src, stride, ln_w, mean, rstd, None, dx, T * H, g_ln_w, g_ln_b, None, B, H)
        return dx
    dpool = alloc("dpool", (B, H), act)
    ops.layernorm_bwd(dhn, src, stride, ln_w, mean, rstd, None, dpool, H, g_ln_w, g_ln_b, None, B, H)
    ops.pool_bwd(dpool, dx, B, T, H, 0 if is_cls else 1)
    return dx
