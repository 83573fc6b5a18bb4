#!/usr/bin/env python
"""Kernel timeline of ONE training step (torch.profiler / CUPTI, run on the GPU box): start, duration,
stream and the idle gap before every kernel, so launch gaps on the critical path are visible.
Not a bench number (profiler overhead); use it to see ordering and overlap."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import bigcn_b200  # noqa: E402
from bigcn_b200.data import Batch, make_batch_shard  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402


def main():
    world, rank = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    pg = None
    if world > 1:      # torchrun: the data-parallel step (rank 0 prints its own timeline)
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
        pg = dist.group.WORLD
    import ctypes as C
    from bigcn_b200 import _lib as L
    lib = L.lib()
    lib.bigcn_debug_set.argtypes = [C.c_int, C.c_int]
    lib.bigcn_debug_set.restype = None
    for spec in sys.argv[1:]:               # "key:value" pairs (bigcn_debug_set), e.g. 10:9
        k, v = spec.split(":")
        lib.bigcn_debug_set(int(k), int(v))
    batches = []
    for i in range(3):
        b = make_batch_shard("twitter16", 128 * world, 1000 + i, rank=rank, world=world)[0]
        batches.append(Batch(**{k: getattr(b, k).to(dev) for k in Batch._tensor_keys}))
    torch.manual_seed(0)
    model = bigcn_b200.BiGCN(5000, 64, 64, dev, gemm_mode="sparse", validate="off").to(dev).train()
    tr = bigcn_b200.FusedTrainer(model, process_group=pg, world_size=world)
    prefetch = os.environ.get("BIGCN_PREFETCH", "1") != "0"
    nxt = lambda i: batches[(i + 1) % 3] if prefetch else None  # noqa: E731
    for i in range(24):
        tr.step(batches[i % 3], b_global=128 * world, next_data=nxt(i))
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(24, 28):
            tr.step(batches[i % 3], b_global=128 * world, next_data=nxt(i))
        torch.cuda.synchronize()
    if rank != 0:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()
        return
    ev = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    ev.sort(key=lambda e: e.time_range.start)
    # last step = from the last k_transpose_jobs on
    starts = [i for i, e in enumerate(ev) if "k_transpose_jobs" in e.name]
    ev = ev[starts[-1]:]
    t0 = ev[0].time_range.start
    end_by_stream = {}
    last_end = t0
    print(f"{'start':>8} {'dur':>7} {'gap_any':>7} {'gap_str':>7}  stream  kernel")
    for e in ev:
        s, d = e.time_range.start - t0, e.time_range.end - e.time_range.start
        stream = getattr(e, "stream", None)
        if stream is None:
            stream = -1
        gap_any = e.time_range.start - last_end
        gap_s = e.time_range.start - end_by_stream.get(stream, e.time_range.start)
        print(f"{s:8.1f} {d:7.1f} {gap_any:7.1f} {gap_s:7.1f}  {stream:>6}  {e.name[:70]}")
        last_end = max(last_end, e.time_range.end)
        end_by_stream[stream] = e.time_range.end
    print("step span us", last_end - t0)
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
