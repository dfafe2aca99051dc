"""GPU: the deferred second passes of the split reductions (vitb_defer_begin / vitb_defer_flush / vitb_defer_flush_partial), producer
by producer, and the fp32 -> bf16 weight-copy cast.

Between begin and flush, a wgrad's dW / db, a LayerNorm backward's dgamma / dbeta / column sums, a GELU backward's column sums and
gemm_bwd_fused's dW / column sums leave their fp32 partials in the caller's arena and record a job; the flush reduces the jobs in
launches of at most 120 (kMaxReduceJobs) per class ("plain": few partials, "tall": >= 64 partials of <= 8192 columns).  The flush
sums every column in the order of the producer's own second pass, so deferred results must equal immediate ones bit for bit: a
missing partial, a job reduced into the wrong destination or a lost launch shows up here, where a tolerance against fp32 would hide
it.  Each producer is also checked against an fp64 restatement of the same bf16 inputs, at the tolerances of test_gpu_kernels.py,
so that an error common to both paths is caught as well.

Partial counts come from the library's own queries, so the cases follow the geometry when it changes: LayerNorm
vitb_layernorm_bwd_ws_bytes / (12 H), column sums vitb_colsum_ws_bytes / (4 cols) (the row-streaming geometry, cols = 3072 here),
wgrad vitb_debug_wgrad_splits (exported for tools and tests, not declared in the header).
"""
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import oracle

pytestmark = pytest.mark.gpu

F32, BF16 = torch.float32, torch.bfloat16
MAX_JOBS = 120  # kMaxReduceJobs (common.cuh): jobs of one class per flush launch
GUARD = 4096    # guard-band elements on each side of a destination (as test_gpu_round2.py (e))
DROP = dict(p=0.2, seed=0x1234ABCD5678EF01, step=7)


@pytest.fixture(scope="module")
def ops():
    import vit_cifar_b200  # noqa: F401
    from vit_cifar_b200 import ops as o
    o.require_device()
    return o


@pytest.fixture(scope="module")
def lib(ops):
    from vit_cifar_b200 import _lib
    h = _lib.load()
    f = h.vitb_debug_wgrad_splits
    f.restype, f.argtypes = C.c_int, [C.c_int, C.c_int, C.c_int]
    return h


_spare = []


@pytest.fixture(autouse=True)
def no_open_window(ops):
    """No test leaves a deferral window open, not even one that fails inside it: later calls would put their partials into a freed
    arena.  A begin over a spare arena drops whatever was recorded, and a flush of no jobs launches nothing."""
    yield
    if not _spare:
        _spare.append(torch.empty(256, dtype=torch.uint8, device="cuda"))
    ops.defer_begin(_spare[0])
    ops.defer_flush()
    torch.cuda.synchronize()


def align(n):
    return (int(n) + 255) // 256 * 256


def is_tall(nparts, cols):  # finalize_is_tall (common.cuh)
    return cols % 4 == 0 and nparts >= 64 and cols <= 8192


def rnd(shape, seed, scale=1.0, dtype=BF16):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.randn(shape, generator=g, device="cuda") * scale).to(dtype)


def rel(a, b):
    a, b = a.double(), b.double()
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


def keep_scale(rows, cols, site):
    keep = oracle.dropout_keep_mask(rows * cols, DROP["p"], DROP["seed"], site, DROP["step"])
    return torch.from_numpy(keep.astype(np.float64)).view(rows, cols).cuda() / (1 - DROP["p"])


def gelu_grad64(z):
    zz = z.double().requires_grad_(True)
    F.gelu(zz).sum().backward()
    return zz.grad


def arena(nbytes):
    a = torch.empty(max(align(nbytes), 256), dtype=torch.uint8, device="cuda")
    assert a.data_ptr() % 256 == 0
    return a


# ---------------------------------------------------------------------------------------------
# producers: one library call with its inputs, its outputs, the arena bytes it reserves and the jobs it records
# ---------------------------------------------------------------------------------------------
class Producer:
    def __init__(self, name, outs, deferred, ws, jobs, call, ref, tol, refill):
        self.name = name
        self.outs = outs          # output name -> (shape, dtype)
        self.deferred = deferred  # outputs written by the flush (hold the sentinel until then)
        self.ws = ws              # bytes reserved in the arena (before alignment)
        self.jobs = jobs          # [(nparts, cols)] recorded
        self.call = call          # call(outs): the library call
        self.ref = ref            # ref(outs) -> output name -> fp64 reference
        self.tol = tol            # output name -> relative tolerance
        self.refill = refill      # refill(seed): new input values, in place

    def fresh(self, guard=False):
        """Outputs filled with NaN; with guard, each inside its own allocation with -77 bands ({name: band buffer} second)."""
        outs, bands = {}, {}
        for k, (shape, dt) in self.outs.items():
            n = int(np.prod(shape))
            if guard:
                buf = torch.full((n + 2 * GUARD,), -77.0, dtype=dt, device="cuda")
                buf[GUARD:GUARD + n] = float("nan")
                outs[k], bands[k] = buf[GUARD:GUARD + n].view(*shape), buf
            else:
                outs[k] = torch.full(shape, float("nan"), dtype=dt, device="cuda")
        return (outs, bands) if guard else outs

    def plain_tall(self):
        t = sum(1 for n, c in self.jobs if is_tall(n, c))
        return len(self.jobs) - t, t


def intact(buf):
    return bool((buf[:GUARD] == -77.0).all() and (buf[-GUARD:] == -77.0).all())


def wgrad(ops, lib, M, N, K, dbias, seed):
    dy, x = rnd((M, N), seed), rnd((M, K), seed + 1)
    splits = lib.vitb_debug_wgrad_splits(M, N, K)
    assert splits >= 1
    outs = {"dw": ((N, K), F32)}
    if dbias:
        outs["db"] = ((N,), F32)
    jobs = ([(splits, N * K)] + ([(splits, N)] if dbias else [])) if splits > 1 else []

    def call(o):
        ops.gemm_wgrad(dy, x, o["dw"], o.get("db"), M, N, K)

    def ref(o):
        r = {"dw": dy.double().t() @ x.double()}
        if dbias:
            r["db"] = dy.double().sum(0)
        return r

    def refill(s):
        dy.copy_(rnd((M, N), s)); x.copy_(rnd((M, K), s + 1))
    p = Producer(f"wgrad{M}x{N}x{K}{'+db' if dbias else ''}", outs, list(outs) if splits > 1 else [], ops.wgrad_ws_bytes(M, N, K), jobs,
                 call, ref, {"dw": 1e-4, "db": 1e-4}, refill)
    p.splits = splits
    return p


def ln_nparts(lib, rows, H):
    return int(lib.vitb_layernorm_bwd_ws_bytes(rows, H)) // (12 * H)


def layernorm(ops, lib, rows, H, res, colsum, seed, fused=None):
    """layernorm_bwd, or with fused = (use_z, use_drop) layernorm_bwd_fused (dres, dx2 and its column sums always present)."""
    x, dy = rnd((rows, H), seed, 2.0), rnd((rows, H), seed + 1)
    dres = rnd((rows, H), seed + 2) if (res or fused) else None
    z = rnd((rows, H), seed + 3, 1.5) if fused and fused[0] else None
    drop = ops.drop_desc(DROP["p"], DROP["seed"], 0, DROP["step"]) if fused and fused[1] else None
    gamma = 1 + 0.2 * rnd((H,), seed + 4, dtype=F32)
    beta = 0.2 * rnd((H,), seed + 5, dtype=F32)
    mean, rstd = torch.empty(rows, device="cuda"), torch.empty(rows, device="cuda")
    y = torch.empty_like(x)

    def stats():
        ops.layernorm_fwd(x, H, gamma, beta, y, mean, rstd, rows, H)
    stats()
    nparts = ln_nparts(lib, rows, H)
    outs = {"dx": ((rows, H), BF16), "dg": ((H,), F32), "db": ((H,), F32)}
    if fused:
        outs["dx2"] = ((rows, H), BF16)
        outs["dc"] = ((H,), F32)
    elif colsum:
        outs["dc"] = ((H,), F32)
    deferred = [k for k in ("dg", "db", "dc") if k in outs]

    def call(o):
        if fused:
            ops.layernorm_bwd_fused(dy, x, H, gamma, mean, rstd, dres, o["dx"], H, o["dg"], o["db"], z, o["dx2"], o["dc"], rows, H, drop=drop)
        else:
            ops.layernorm_bwd(dy, x, H, gamma, mean, rstd, dres, o["dx"], H, o["dg"], o["db"], o.get("dc"), rows, H)

    def ref(o):
        xr = x.double().requires_grad_(True)
        gr, br = gamma.double().requires_grad_(True), beta.double().requires_grad_(True)
        F.layer_norm(xr, (H,), gr, br, 1e-5).backward(dy.double())
        dx = xr.grad + (dres.double() if dres is not None else 0.0)
        r = {"dx": dx, "dg": gr.grad, "db": br.grad}
        if fused:  # dx2 is computed from dx as stored (bf16)
            dx2 = o["dx"].double()
            if drop is not None:
                dx2 = dx2 * keep_scale(rows, H, 0)
            if z is not None:
                dx2 = dx2 * gelu_grad64(z)
            r["dx2"], r["dc"] = dx2, dx2.sum(0)
        elif colsum:
            r["dc"] = dx.sum(0)
        return r

    def refill(s):
        x.copy_(rnd((rows, H), s, 2.0)); dy.copy_(rnd((rows, H), s + 1))
        if dres is not None:
            dres.copy_(rnd((rows, H), s + 2))
        stats()
    name = f"ln{rows}x{H}" + (f"fused(z={fused[0]},drop={fused[1]})" if fused else f"(res={res},colsum={colsum})")
    tol = {"dx": 2e-2, "dg": 2e-2, "db": 2e-2, "dc": 5e-3, "dx2": 6e-3}
    p = Producer(name, outs, deferred, lib.vitb_layernorm_bwd_ws_bytes(rows, H), [(nparts, H)] * len(deferred), call, ref, tol, refill)
    p.nparts = nparts
    return p


def gelu(ops, lib, rows, cols, use_drop, seed):
    dy, z = rnd((rows, cols), seed), rnd((rows, cols), seed + 1, 1.5)
    drop = ops.drop_desc(DROP["p"], DROP["seed"], 2, DROP["step"]) if use_drop else None
    ws = int(lib.vitb_colsum_ws_bytes(rows, cols))

    def call(o):
        ops.gelu_bwd_colsum(dy, z, o["dz"], o["cs"], rows, cols, drop=drop)

    def ref(o):
        dz = dy.double() * gelu_grad64(z)
        if use_drop:
            dz = dz * keep_scale(rows, cols, 2)
        return {"dz": dz, "cs": dz.sum(0)}

    def refill(s):
        dy.copy_(rnd((rows, cols), s)); z.copy_(rnd((rows, cols), s + 1, 1.5))
    # (ws / (4 cols) is the partial count of the row-streaming geometry; the 16-byte bf16 path, cols <= 1024, uses fewer)
    return Producer(f"gelu{rows}x{cols}(drop={use_drop})", {"dz": ((rows, cols), BF16), "cs": ((cols,), F32)}, ["cs"], ws,
                    [(ws // (4 * cols), cols)], call, ref, {"dz": 2e-2, "cs": 6e-3 if use_drop else 5e-3}, refill)


def bwd_fused(ops, M, N, K, seed):
    dy, x = rnd((M, N), seed), rnd((M, K), seed + 1)
    w, z = rnd((N, K), seed + 2, N ** -0.5), rnd((M, K), seed + 3)
    ws = ops.bwd_fused_ws_bytes(M, N, K)
    assert ws > 0
    # members (dW partial sets): ws = align(members N K 4) + align(members 4 K 4) + 256
    members = next(m for m in range(1, 4096) if align(m * N * K * 4) + align(m * 16 * K) + 256 == ws)

    def call(o):
        ops.gemm_bwd_fused(dy, x, w, z, o["dx"], o["dw"], o["cs"], M, N, K)

    def ref(o):
        return {"dx": (dy.double() @ w.double()) * gelu_grad64(z), "dw": dy.double().t() @ x.double(), "cs": o["dx"].double().sum(0)}

    def refill(s):
        dy.copy_(rnd((M, N), s)); x.copy_(rnd((M, K), s + 1))
    jobs = ([(members, N * K)] if members > 1 else []) + [(members * 4, K)]
    return Producer(f"bwd_fused{M}x{N}x{K}", {"dx": ((M, K), BF16), "dw": ((N, K), F32), "cs": ((K,), F32)},
                    (["dw"] if members > 1 else []) + ["cs"], ws, jobs, call, ref, {"dx": 2e-2, "dw": 1e-3, "cs": 1e-3}, refill)


# ---------------------------------------------------------------------------------------------
def immediate(prods):
    outs = [p.fresh() for p in prods]
    for p, o in zip(prods, outs):
        p.call(o)
    return outs


def assert_equal(p, got, want, what):
    for k in p.outs:
        assert torch.equal(got[k], want[k]), f"{p.name}.{k}: {what} differs from the immediate call"


def assert_correct(p, outs):
    ref = p.ref(outs)
    for k, r in ref.items():
        e = rel(outs[k], r)
        assert e < p.tol[k], f"{p.name}.{k}: {e:.3g} from the fp64 reference (tolerance {p.tol[k]})"


def assert_sentinel(p, outs):
    for k in p.deferred:
        assert bool(torch.isnan(outs[k]).all()), f"{p.name}.{k}: written before the flush (the call did not defer)"


def deferred_vs_immediate(ops, prods):
    imm = immediate(prods)
    ar = arena(sum(align(p.ws) for p in prods))
    dfr = [p.fresh() for p in prods]
    ops.defer_begin(ar)
    for p, o in zip(prods, dfr):
        p.call(o)
    torch.cuda.synchronize()
    for p, o in zip(prods, dfr):
        assert_sentinel(p, o)
    assert ops.defer_used() == sum(align(p.ws) for p in prods)
    ops.defer_flush()
    torch.cuda.synchronize()
    for p, o, i in zip(prods, dfr, imm):
        assert_equal(p, o, i, "deferred")
        assert_correct(p, i)


# ---------------------------------------------------------------------------------------------
# 1. deferred == immediate, bit for bit, producer by producer
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,K", [(384, 384), (1152, 384), (3072, 768)])
@pytest.mark.parametrize("M", [17, 51, 64, 8320, 20000, 66560])
def test_wgrad_deferred_equals_immediate(ops, lib, M, N, K):
    """Every split regime of wgrad_tc_plan: one split (M <= 64: dW / db written by the GEMM itself, nothing deferred), the 8-12
    rule (8,320 and 20,000 rows) and the uncapped plan (66,560 rows), with and without the bias gradient."""
    prods = [wgrad(ops, lib, M, N, K, dbias, 10 * M + N) for dbias in (True, False)]
    splits = prods[0].splits
    if M <= 64:
        assert splits == 1
    else:
        assert splits > 1
    deferred_vs_immediate(ops, prods)


@pytest.mark.parametrize("H", [128, 384, 768])
@pytest.mark.parametrize("res,colsum", [(False, False), (True, False), (False, True), (True, True)])
def test_layernorm_bwd_deferred_equals_immediate(ops, lib, H, res, colsum):
    deferred_vs_immediate(ops, [layernorm(ops, lib, rows, H, res, colsum, rows + H) for rows in (77, 4133)])


@pytest.mark.parametrize("use_z,use_drop", [(True, False), (False, True), (True, True)])
def test_layernorm_bwd_fused_deferred_equals_immediate(ops, lib, use_z, use_drop):
    deferred_vs_immediate(ops, [layernorm(ops, lib, rows, 384, True, True, rows, fused=(use_z, use_drop)) for rows in (130, 4133)])


@pytest.mark.parametrize("cols", [384, 3072])   # the 16-byte bf16 kernel / the row-streaming kernel
@pytest.mark.parametrize("use_drop", [False, True])
def test_gelu_bwd_colsum_deferred_equals_immediate(ops, lib, cols, use_drop):
    deferred_vs_immediate(ops, [gelu(ops, lib, rows, cols, use_drop, rows + cols) for rows in (1000, 4133)])


def test_gemm_bwd_fused_deferred_equals_immediate(ops):
    deferred_vs_immediate(ops, [bwd_fused(ops, 8320, 384, 384, 3)])


# ---------------------------------------------------------------------------------------------
# 2. the plain / tall boundary of the LayerNorm partials
# ---------------------------------------------------------------------------------------------
def test_layernorm_partials_at_the_plain_tall_boundary(ops, lib):
    """The smallest row count whose LayerNorm backward has 64 partials (tall jobs) and the one below it (63: plain jobs)."""
    H = 384
    r64 = next(r for r in range(1, 1 << 16) if ln_nparts(lib, r, H) >= 64)
    assert ln_nparts(lib, r64 - 1, H) == 63 and ln_nparts(lib, r64, H) == 64  # (rows 504 / 505 at kLnBwdWarps = 8)
    prods = [layernorm(ops, lib, r, H, True, True, r) for r in (r64 - 1, r64)]
    assert prods[0].plain_tall() == (3, 0) and prods[1].plain_tall() == (0, 3)
    deferred_vs_immediate(ops, prods)


# ---------------------------------------------------------------------------------------------
# 3. more than 120 jobs of a class: several launches, find_job over full tables
# ---------------------------------------------------------------------------------------------
def job_mix(ops, lib, n_plain, n_tall):
    """Producers recording exactly n_plain plain and n_tall tall jobs, interleaved, large jobs next to tiny ones:
    plain: a 1152 x 384 dW (hundreds of blocks) and LayerNorm at 40 rows (one block per job);
    tall:  GELU column sums over 3072 columns (96 blocks) and LayerNorm at 600 rows (4 blocks per job)."""
    def big_plain(i):
        return wgrad(ops, lib, 128, 1152, 384, False, 1000 + i)

    def tiny_plain(i, cs):
        return layernorm(ops, lib, 40, 128, i % 3 == 0, cs, 2000 + i)

    def big_tall(i):
        return gelu(ops, lib, 520, 3072, False, 3000 + i)

    def tiny_tall(i, cs):
        return layernorm(ops, lib, 600, 128, i % 3 == 1, cs, 4000 + i)

    def chain(n, big, tiny):
        out, left, i = [], n, 0
        while left > 0:
            if i % 2 == 0 or left == 1:
                out.append(big(i)); left -= 1
            else:
                cs = left >= 3 and i % 4 == 1
                out.append(tiny(i, cs)); left -= 3 if cs else 2
            i += 1
        return out
    plain, tall = chain(n_plain, big_plain, tiny_plain), chain(n_tall, big_tall, tiny_tall)
    prods = [p for pair in zip(plain + [None] * len(tall), tall + [None] * len(plain)) for p in pair if p is not None]
    counts = [p.plain_tall() for p in prods]
    assert (sum(c[0] for c in counts), sum(c[1] for c in counts)) == (n_plain, n_tall)
    return prods


@pytest.mark.parametrize("n", [119, 120, 121, 240, 241])
def test_flush_of_more_than_120_jobs_per_class(ops, lib, n):
    prods = job_mix(ops, lib, n, n)
    assert prods[0].splits > 1
    imm = immediate(prods)
    ar = arena(sum(align(p.ws) for p in prods))
    dfr = [p.fresh(guard=True) for p in prods]
    ops.defer_begin(ar)
    for p, (o, _) in zip(prods, dfr):
        p.call(o)
    n0 = ops.launch_count()
    ops.defer_flush()
    launches = ops.launch_count() - n0
    torch.cuda.synchronize()
    assert launches == 2 * -(-n // MAX_JOBS)
    for p, (o, bands), i in zip(prods, dfr, imm):
        assert_equal(p, o, i, "deferred")
        for k, b in bands.items():
            assert intact(b), f"{p.name}.{k}: guard band overwritten"
    for p, i in list(zip(prods, imm))[:8]:
        assert_correct(p, i)


# ---------------------------------------------------------------------------------------------
# 4. flush_partial: flushed jobs are not flushed again, the arena keeps growing
# ---------------------------------------------------------------------------------------------
def test_flush_partial_then_flush(ops, lib):
    A = [layernorm(ops, lib, 40, 128, True, True, 1), wgrad(ops, lib, 8320, 384, 384, True, 2), layernorm(ops, lib, 4133, 384, False, True, 3)]
    B = [gelu(ops, lib, 4133, 384, False, 4), wgrad(ops, lib, 20000, 1152, 384, True, 5), layernorm(ops, lib, 999, 768, True, False, 6),
         layernorm(ops, lib, 77, 384, True, True, 7)]
    imm_a, imm_b = immediate(A), immediate(B)
    ar = arena(sum(align(p.ws) for p in A + B))
    out_a, out_b = [p.fresh() for p in A], [p.fresh() for p in B]
    ops.defer_begin(ar)
    for p, o in zip(A, out_a):
        p.call(o)
    used_a = ops.defer_used()
    assert used_a == sum(align(p.ws) for p in A)
    ops.defer_flush_partial()
    torch.cuda.synchronize()
    for p, o, i in zip(A, out_a, imm_a):
        assert_equal(p, o, i, "after flush_partial")
        for k in p.deferred:
            o[k].fill_(float("nan"))
    for p, o in zip(B, out_b):
        p.call(o)
    assert ops.defer_used() == used_a + sum(align(p.ws) for p in B)  # B's partials lie behind A's
    ops.defer_flush()
    torch.cuda.synchronize()
    for p, o in zip(A, out_a):
        assert_sentinel(p, o)  # flushed once only
    for p, o, i in zip(B, out_b, imm_b):
        assert_equal(p, o, i, "deferred after a partial flush")
        assert_correct(p, i)


# ---------------------------------------------------------------------------------------------
# 5. arena exhaustion, accounting, host-side errors
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [1, 3])
def test_arena_exhaustion_falls_back_to_the_immediate_second_pass(ops, lib, k):
    prods = [wgrad(ops, lib, 8320, 384, 384, True, 11), layernorm(ops, lib, 4133, 384, True, True, 12), gelu(ops, lib, 4133, 384, True, 13),
             layernorm(ops, lib, 40, 128, False, False, 14), bwd_fused(ops, 8320, 384, 384, 15), wgrad(ops, lib, 20000, 1152, 384, False, 16),
             gelu(ops, lib, 1000, 3072, False, 17)]
    imm = immediate(prods)
    ar = arena(sum(align(p.ws) for p in prods[:k]))  # holds exactly the first k producers' partials
    outs = [p.fresh() for p in prods]
    ops.defer_begin(ar)
    for p, o in zip(prods, outs):
        p.call(o)
    torch.cuda.synchronize()
    for p, o, i in zip(prods[k:], outs[k:], imm[k:]):
        assert_equal(p, o, i, "immediate fallback")  # final before the flush
    for p, o in zip(prods[:k], outs[:k]):
        assert_sentinel(p, o)
    # what a large enough arena would have held: every call of the window, the ones that did not fit included
    assert ops.defer_used() == sum(align(p.ws) for p in prods)
    ops.defer_flush()
    torch.cuda.synchronize()
    for p, o, i in zip(prods, outs, imm):
        assert_equal(p, o, i, "deferred")
        assert_correct(p, i)


def test_defer_host_side_errors_launch_nothing(ops):
    from vit_cifar_b200._lib import VitbError
    big = torch.empty(4096, dtype=torch.uint8, device="cuda")
    assert big.data_ptr() % 256 == 0
    n0 = ops.launch_count()
    with pytest.raises(VitbError):
        ops.defer_begin(torch.empty(128, dtype=torch.uint8, device="cuda"))  # smaller than 256 bytes
    for off in (1, 16, 128):
        with pytest.raises(VitbError):
            ops.defer_begin(big[off:])  # not 256-byte aligned
    with pytest.raises(VitbError):
        ops.defer_flush()  # no window open (the failed begins opened none)
    with pytest.raises(VitbError):
        ops.defer_flush_partial()
    assert ops.launch_count() == n0


def test_second_begin_drops_the_first_windows_jobs(ops, lib):
    A = [wgrad(ops, lib, 8320, 384, 384, True, 21), layernorm(ops, lib, 4133, 384, True, True, 22)]
    B = [gelu(ops, lib, 4133, 384, False, 23)]
    imm_b = immediate(B)
    ar1, ar2 = arena(sum(align(p.ws) for p in A)), arena(sum(align(p.ws) for p in B))
    out_a, out_b = [p.fresh() for p in A], [p.fresh() for p in B]
    ops.defer_begin(ar1)
    for p, o in zip(A, out_a):
        p.call(o)
    ops.defer_begin(ar2)
    for p, o in zip(B, out_b):
        p.call(o)
    assert ops.defer_used() == sum(align(p.ws) for p in B)
    ops.defer_flush()
    torch.cuda.synchronize()
    for p, o in zip(A, out_a):
        assert_sentinel(p, o)
    for p, o, i in zip(B, out_b, imm_b):
        assert_equal(p, o, i, "deferred")


# ---------------------------------------------------------------------------------------------
# 6. under CUDA graph capture: the job table travels by value in the kernel parameters
# ---------------------------------------------------------------------------------------------
def test_captured_window_with_more_than_120_plain_jobs(ops, lib):
    prods = job_mix(ops, lib, 130, 7)
    outs = [p.fresh() for p in prods]
    ar = arena(sum(align(p.ws) for p in prods))

    def window():
        ops.defer_begin(ar)
        for p, o in zip(prods, outs):
            p.call(o)
        n0 = ops.launch_count()
        ops.defer_flush()
        return ops.launch_count() - n0
    assert window() == 3  # eager once: the workspace reaches its size before the capture
    torch.cuda.synchronize()
    before = [{k: t.clone() for k, t in o.items()} for o in outs]
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        assert window() == 3  # two plain launches, one tall
    for i, p in enumerate(prods):
        p.refill(7000 + 10 * i)
    for o in outs:
        for t in o.values():
            t.fill_(float("nan"))
    g.replay()
    torch.cuda.synchronize()
    imm = immediate(prods)
    torch.cuda.synchronize()
    for p, o, i, b in zip(prods, outs, imm, before):
        assert_equal(p, o, i, "graph replay")
        assert not any(torch.equal(o[k], b[k]) for k in p.deferred), p.name  # new inputs, new results
    del g


# ---------------------------------------------------------------------------------------------
# 7. vitb_cast_f32_to_bf16 (the bf16 weight copy) against torch's round-to-nearest-even
# ---------------------------------------------------------------------------------------------
def _bits(*words):
    return torch.tensor(np.array(words, dtype=np.uint32).view(np.int32)).view(torch.float32)


SPECIALS = _bits(
    0x00000000, 0x80000000,              # +-0
    0x7F800000, 0xFF800000,              # +-inf
    0x7FC00000, 0xFFC00001, 0x7F800001,  # NaNs (quiet, negative, signalling)
    0x00000001, 0x80000001, 0x00007FFF, 0x00008000, 0x00018000, 0x007FFFFF, 0x807F8000,  # fp32 subnormals, ties among them
    0x3F808000, 0x3F818000, 0xBF808000, 0xBF818000,  # exact ties: even below rounds down, odd below rounds up
    0x3F808001, 0x3F807FFF,              # just above / below a tie
    0x7F7FFFFF, 0xFF7FFFFF, 0x7F7F8000,  # round up to +-inf (the last an exact tie with an odd bf16 below)
    0x7F7F7FFF, 0x00800000, 0x80800000)  # largest that stays finite, smallest normals


def _cast_case(ops, n, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    src = torch.randn(n, generator=g, device="cuda") * torch.exp2(torch.randint(-130, 128, (n,), generator=g, device="cuda").float())
    sp = SPECIALS.cuda()
    m = min(n, sp.numel())
    src[:m] = sp[:m]
    if n > 2 * sp.numel():
        src[-sp.numel():] = sp
    return src


def _assert_cast(src, dst):
    want = src.to(BF16)
    nan = torch.isnan(want)
    assert torch.equal(torch.isnan(dst), nan)
    d, w = dst.view(torch.int16)[~nan], want.view(torch.int16)[~nan]
    bad = (d != w).nonzero()
    assert bad.numel() == 0, f"{bad.numel()} elements differ, first at {int(bad[0])}: src bits {hex(int(src[~nan].view(torch.int32)[bad[0]]))}"


@pytest.mark.parametrize("n", [1, 2, 3, 4, 5, 1023, 6_268_810])
def test_cast_f32_to_bf16_matches_torch_bit_for_bit(ops, n):
    src = _cast_case(ops, n, n)
    dst = torch.full((n,), float("nan"), dtype=BF16, device="cuda")
    ops.cast_f32_to_bf16(src, dst)
    _assert_cast(src, dst)
    # 16-byte aligned sub-views at an offset, with the neighbours untouched
    sbuf = torch.zeros(n + 12, device="cuda")
    sbuf[4:4 + n] = src
    dbuf = torch.full((n + 12,), -77.0, dtype=BF16, device="cuda")
    ops.cast_f32_to_bf16(sbuf[4:4 + n], dbuf[4:4 + n])
    _assert_cast(src, dbuf[4:4 + n])
    assert bool((dbuf[:4] == -77.0).all() and (dbuf[4 + n:] == -77.0).all())


def test_cast_f32_to_bf16_rejects_misaligned_views(ops):
    """The entry checks alignment before it launches (16 bytes for the source, 8 for the copy): nothing runs."""
    from vit_cifar_b200._lib import VitbError
    sbuf = torch.zeros(64, device="cuda")
    dbuf = torch.zeros(64, dtype=BF16, device="cuda")
    n0 = ops.launch_count()
    with pytest.raises(VitbError):
        ops.cast_f32_to_bf16(sbuf[1:33], dbuf[:32])
    with pytest.raises(VitbError):
        ops.cast_f32_to_bf16(sbuf[:32], dbuf[1:33])
    assert ops.launch_count() == n0
