"""2+ GPU check of DeviceLoader's sharding.  Run under torchrun:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29581 tools/loader_dp_check.py

Every rank holds the same seeded set of 1,001 images (1,001 % 2 != 0: DistributedSampler pads one rank's shard), trains one epoch
through DeviceLoader(process_group=WORLD) at batch 96 (the last batch partial) with CutMix, and must
  * take as many steps as every other rank (ceil(ceil(1001 / world) / 96)),
  * end with bit-identical parameters on every rank (the replicas of one data-parallel model),
  * report from the sharded validation pass (DeviceLoader(shuffle=False) + EvalEngine) what one GPU reports for the whole set.
"""
import os
import sys

import numpy as np
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
    np.random.seed(7)
    m = vb.ViT(3, 10, img_size=32, patch=8, num_layers=2, hidden=128, mlp_hidden=128, head=4).cuda()
    rng = np.random.default_rng(3)
    N, B = 1001, 96
    ds = vb.DeviceDataset(rng.integers(0, 256, (N, 32, 32, 3), dtype=np.uint8), rng.integers(0, 10, N), device="cuda")
    eng = vb.TrainEngine(m, B, mixed_targets=True, process_group=dist.group.WORLD, metrics=True)
    aug = vb.GpuAugment(32, 4, seed=11 + rank, policy="cifar10")
    loader = vb.DeviceLoader(ds, B, shuffle=True, seed=5, augment=aug, mix=vb.GpuCutMix(32, 1.0), process_group=dist.group.WORLD)
    loader.set_epoch(1)
    steps = 0
    for img, label, rand_label, lam in loader:
        eng.step(img, label, rand_label, lam)
        steps += 1
    tr = eng.train_metrics()
    counts = [None] * world
    dist.all_gather_object(counts, steps)
    p = eng.P[:eng.n].clone()
    p0 = p.clone()
    dist.broadcast(p0, src=0)
    same_params = bool(torch.equal(p, p0))
    per_rank = -(-N // world)
    expect = -(-per_rank // B)
    sharded = vb.EvalEngine(m, 256, mean=aug.mean, std=aug.std, process_group=dist.group.WORLD).run(
        vb.DeviceLoader(ds, 256, shuffle=False, process_group=dist.group.WORLD))
    single = vb.EvalEngine(m, 256, mean=aug.mean, std=aug.std).run(vb.DeviceLoader(ds, 256, shuffle=False))
    ok = (all(c == expect for c in counts) and same_params and tr["n"] == world * per_rank
          and sharded["n"] == single["n"] == N and sharded["val_acc"] == single["val_acc"]
          and abs(sharded["val_loss"] - single["val_loss"]) <= 1e-6 * abs(single["val_loss"]))
    flags = torch.tensor([1 if ok else 0], device="cuda")
    dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    ok = int(flags.item()) == 1
    if rank == 0:
        print(f"world={world}: steps {counts} (expected {expect}), replicas identical {same_params}, train {tr}, "
              f"single {single} sharded {sharded}", flush=True)
        print("loader_dp_check", "PASSED" if ok else "FAILED", flush=True)
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


main()
