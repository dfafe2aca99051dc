"""2+ GPU check of EvalEngine's sharded validation pass.  Run under torchrun:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29579 tools/eval_dp_check.py

Every rank builds the same model, evaluates its own shard of one seeded set of 1,000 images (rank r takes batches r, r + world, ...,
the last one partial) under the process group, and must return the single-GPU result of the whole set: n and val_acc equal,
val_loss within 1e-6 relative, identical on every rank.
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


def main():
    torch.manual_seed(2045)  # same weights on every rank
    m = vb.ViT(3, 10, img_size=32, patch=8, num_layers=7, hidden=384, mlp_hidden=384, head=12).cuda()
    g = torch.Generator().manual_seed(7)
    x, y = torch.randn(1000, 3, 32, 32, generator=g), torch.randint(0, 10, (1000,), generator=g)
    batches = [(x[i:i + 256].cuda(), y[i:i + 256].cuda()) for i in range(0, 1000, 256)]
    single = vb.EvalEngine(m, batch_size=256).run(batches)
    sharded = vb.EvalEngine(m, batch_size=256, process_group=dist.group.WORLD).run(batches[rank::world])
    gathered = [None] * world
    dist.all_gather_object(gathered, sharded)
    ok = (all(r == gathered[0] for r in gathered) and sharded["n"] == single["n"] == 1000 and sharded["val_acc"] == single["val_acc"]
          and abs(sharded["val_loss"] - single["val_loss"]) <= 1e-6 * abs(single["val_loss"]))
    if rank == 0:
        print(f"world={world}: single {single} sharded {gathered}", flush=True)
        print("eval_dp_check", "PASSED" if ok else "FAILED", flush=True)
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


main()
