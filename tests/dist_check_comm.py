"""Peer-memory all-reduce check (run under torchrun, one rank per GPU):

    torchrun --nproc-per-node 2 --master-addr 127.0.0.1 tests/dist_check_comm.py [--time]

1. exactness: integer-valued inputs f(rank, call, i) whose sum is known in closed form, 2000 back-to-back calls with a different
   input every call (a stale or half-written slot would show up as a wrong sum);
2. random fp32 inputs: result within 1e-6 relative of NCCL's all-reduce and BIT-IDENTICAL across ranks (fixed rank order);
3. --time: device time per all-reduce of the PPO gradient size, next to NCCL's.
"""
import argparse
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--time", action="store_true")
    ap.add_argument("--n", type=int, default=329_259)  # the Humanoid PPO gradient + 8 metric sums: not a multiple of 4
    args = ap.parse_args()
    from rl_x_b200.algorithms.ppo.b200.kernels import PeerComm
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    dist.init_process_group("nccl", device_id=dev)
    n = args.n
    comm = PeerComm(dist, n, dev)
    out = torch.empty(n, device=dev)
    idx = torch.arange(n, device=dev, dtype=torch.float32) % 97.0
    # 1. exact sums, many calls in flight
    calls = 2000
    bad = torch.zeros(1, device=dev)
    rank_sum = world * (world - 1) / 2.0
    for c in range(calls):
        src = idx * float(rank + 1) + float((c % 13) * (rank + 2))
        comm.stage(src)
        comm.allreduce_sum(out)
        expect = idx * float(rank_sum + world) + float((c % 13) * (rank_sum + 2 * world))
        bad += (out != expect).sum()
    assert int(bad.item()) == 0, f"rank {rank}: {int(bad.item())} wrong elements over {calls} calls"

    # 2. random inputs: against NCCL, and identical bits everywhere
    g = torch.Generator(device=dev).manual_seed(100 + rank)
    src = torch.randn(n, device=dev, generator=g)
    comm.stage(src)
    comm.allreduce_sum(out)
    ref = src.clone()
    dist.all_reduce(ref)
    rel = float((out - ref).norm() / ref.norm())
    assert rel < 1e-6, rel
    gathered = [torch.empty_like(out) for _ in range(world)]
    dist.all_gather(gathered, out)
    for r in range(world):
        assert torch.equal(gathered[r], gathered[0]), f"rank {r} differs from rank 0"

    if args.time:
        timed = [("peer", lambda: comm.allreduce_sum(out)), ("nccl", lambda: dist.all_reduce(ref))]
        for name, fn in timed:
            for _ in range(50):
                fn()
            dist.barrier()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(500):
                fn()
            e1.record()
            torch.cuda.synchronize()
            t = torch.tensor([e0.elapsed_time(e1) / 500 * 1e3], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            if rank == 0:
                print(f"{name}: {t.item():.1f} us per all-reduce of {n} floats over {world} GPUs (back to back, host launch included)")
    comm.close()
    if rank == 0:
        print(f"peer all-reduce over {world} ranks: OK (vs NCCL rel {rel:.2e})")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
