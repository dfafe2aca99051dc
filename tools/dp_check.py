"""2+ GPU check of the fused data-parallel step (csrc/dp.cu) against the NCCL path.  Run under torchrun:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29533 tools/dp_check.py

For a small and the benchmark model: same initial weights, rank-specific batches, K steps with VITB_DP_MODE=single (NCCL all-reduce +
Adam kernel) and =fused (one peer-memory kernel); prints the parameter difference between the two paths (bit-exact at 2 ranks: a+b has
one association), checks that all replicas of the fused path are bit-identical, and times both.
"""
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import vit_cifar_b200 as vb  # noqa: E402

local = int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
rank, world = dist.get_rank(), dist.get_world_size()
ADAM = dict(lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=5e-5)


def run(cfg, B, mode, steps, use_graph, precision, optimizer="adam"):
    os.environ["VITB_DP_MODE"] = mode
    vb.set_precision(precision)
    torch.manual_seed(2045)  # same initial weights for both paths and all ranks
    m = vb.ViT(3, cfg["num_classes"], img_size=32, patch=cfg["patch"], num_layers=cfg["num_layers"], hidden=cfg["hidden"],
               mlp_hidden=cfg["mlp_hidden"], head=cfg["head"]).cuda()
    eng = vb.TrainEngine(m, B, use_graph=use_graph, process_group=dist.group.WORLD, optimizer=optimizer, **ADAM)
    losses = []
    for t in range(steps):
        g = torch.Generator().manual_seed(100 * t + rank)  # rank-specific batches
        x, y = torch.randn(B, 3, 32, 32, generator=g), torch.randint(0, cfg["num_classes"], (B,), generator=g)
        losses.append(eng.step(x.cuda(), y.cuda()).item())
    torch.cuda.synchronize()
    # timing: same batch again and again
    dist.barrier()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(10):
        eng.step()
    e.record()
    torch.cuda.synchronize()
    ms = torch.tensor([s.elapsed_time(e) / 10], device="cuda")
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return eng.P[:eng.n].clone(), losses, ms.item()


def main():
    ok = True
    tiny = dict(num_classes=10, patch=8, num_layers=2, hidden=128, mlp_hidden=128, head=4)
    cases = [("tiny fp32", tiny, 8, "fp32", False, "adam"), ("tiny fp32 sgd graph", tiny, 8, "fp32", True, "sgd"),
             ("bench bf16 graph", dict(num_classes=10, patch=8, num_layers=7, hidden=384, mlp_hidden=384, head=12), 1024, "bf16", True, "adam"),
             ("vit-tiny width 192 bf16 graph", dict(num_classes=10, patch=8, num_layers=2, hidden=192, mlp_hidden=768, head=3), 256, "bf16", True,
              "adam")]
    for name, cfg, B, precision, graph, optimizer in cases:
        p_ref, l_ref, ms_ref = run(cfg, B, "single", 4, graph, precision, optimizer)
        p_fus, l_fus, ms_fus = run(cfg, B, "fused", 4, graph, precision, optimizer)
        diff = ((p_fus - p_ref).double().norm() / p_ref.double().norm()).item()
        gathered = [torch.empty_like(p_fus) for _ in range(world)]
        dist.all_gather(gathered, p_fus)
        same = all(torch.equal(gathered[0], g) for g in gathered)
        exact = torch.equal(p_fus, p_ref)
        # (bf16: a last-bit difference in one parameter is amplified by the bf16 rounding of activations over the following steps)
        good = same and diff < (1e-5 if precision == "fp32" else 1e-3) and all(abs(a - b) <= 1e-4 * abs(b) for a, b in zip(l_fus, l_ref))
        ok = ok and good
        if rank == 0:
            print(f"[{name}] world={world}: fused vs NCCL params rel diff {diff:.3e} (bit-exact: {exact}); replicas identical: {same}; "
                  f"losses fused {[round(v, 6) for v in l_fus]} nccl {[round(v, 6) for v in l_ref]}; "
                  f"ms/step NCCL {ms_ref:.3f} fused {ms_fus:.3f}  -> {'OK' if good else 'MISMATCH'}", flush=True)
    dist.barrier()
    torch.cuda.synchronize()
    if rank == 0:
        print("dp_check", "PASSED" if ok else "FAILED", flush=True)
    os._exit(0 if ok else 1)


main()
