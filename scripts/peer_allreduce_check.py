"""torchrun check of the fused statistics + peer-memory all-reduce + weight kernel against the NCCL path.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29531 scripts/peer_allreduce_check.py
"""
import json
import os
import sys
import time

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from retinex_image_enhancement_b200.losses import loss as L  # noqa: E402


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    nccl = L.DynamicSmoothWeight(1.0, True, "tv")
    fused = L.DynamicSmoothWeight(1.0, True, "tv", fused_collective=True)
    ok = True          # every rank derives the same weight, bit for bit
    close = True       # ... and it agrees with the NCCL path (identical for 2 ranks; NCCL's summation order differs beyond that)
    exact_vs_nccl = True
    for step in range(40):
        b = 8 if step % 3 else 5 + rank            # unequal local batches on some steps
        x = torch.rand((b, 3, 256, 256), device=dev, generator=torch.Generator(device=dev).manual_seed(100 * step + rank))
        if step % 2:
            x *= 0.3
        w_ref = nccl(x)
        w_fused = fused(x)
        exact_vs_nccl = exact_vs_nccl and torch.equal(w_ref, w_fused)
        close = close and bool(torch.allclose(w_ref, w_fused, rtol=1e-6, atol=0))
        gathered = [torch.empty_like(w_fused) for _ in range(world)]
        dist.all_gather(gathered, w_fused)
        ok = ok and all(torch.equal(g, gathered[0]) for g in gathered)
    for name, obj in (("edge_nccl", L.DynamicSmoothWeight(1.0, True, "edge_density")),
                      ("edge_fused", L.DynamicSmoothWeight(1.0, True, "edge_density", fused_collective=True))):
        x = torch.rand((4, 3, 128, 128), device=dev, generator=torch.Generator(device=dev).manual_seed(7 + rank))
        v = obj(x)
        if name == "edge_nccl":
            ref = v
        else:
            close = close and bool(torch.allclose(ref, v, rtol=1e-6, atol=0))
    # timing: CUDA events around 200 calls
    x = torch.rand((8, 3, 256, 256), device=dev)
    res = {}
    for name, obj in (("nccl", nccl), ("fused", fused)):
        for _ in range(20):
            obj(x)
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(200):
            obj(x)
        e.record()
        torch.cuda.synchronize()
        res[name] = {"us_per_step_device": s.elapsed_time(e) * 1e3 / 200, "us_per_step_wall": (time.perf_counter() - t0) * 1e6 / 200}
    # a peer that skips a step: the waiting rank gets NaN after the time-out and an exception from check_peers() -- no hang, no trap
    from retinex_image_enhancement_b200 import native
    fused.check_peers()                                   # nothing failed so far
    native.peer_set_timeout_ms(150.0)
    torch.cuda.synchronize()
    dist.barrier()
    timeout_ok = True
    if rank == 0:
        w_late = fused(x)                                 # the other ranks never make this call
        torch.cuda.synchronize()
        timeout_ok = bool(torch.isnan(w_late).item())
        try:
            fused.check_peers()
            timeout_ok = False
        except native.UprError as e:
            timeout_ok = timeout_ok and "timed out waiting for rank" in str(e)
    dist.barrier()
    flag = torch.tensor([1.0 if ok else 0.0, 1.0 if close else 0.0, 1.0 if exact_vs_nccl else 0.0, 1.0 if timeout_ok else 0.0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    good = bool(flag[0].item() == 1.0 and flag[1].item() == 1.0 and flag[3].item() == 1.0)
    if rank == 0:
        print(json.dumps({"world": world, "weights_identical_across_ranks": bool(flag[0].item() == 1.0),
                          "within_1e-6_of_nccl_path": bool(flag[1].item() == 1.0), "bit_equal_to_nccl_path": bool(flag[2].item() == 1.0),
                          "late_peer_times_out_with_nan_and_status": bool(flag[3].item() == 1.0), **res}))
    dist.destroy_process_group()
    return 0 if good else 1


if __name__ == "__main__":
    sys.exit(main())
