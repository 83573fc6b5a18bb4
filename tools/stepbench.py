#!/usr/bin/env python
"""Step-level A/B through the bigcn_debug_set keys (needs the GPU): times FusedTrainer.step on three resident
Twitter16-shaped batches with CUDA events.  `python tools/stepbench.py 10:0,9` compares the two forms of the background
capture pass over x (0 = TMA-fed, the shipped one; 9 = LDG)."""
import ctypes as C
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import bigcn_b200  # noqa: E402
from bigcn_b200 import _lib as L  # noqa: E402
from bigcn_b200.data import Batch, make_batch_shard  # noqa: E402
from bigcn_b200.ops import GraphCache  # noqa: E402


def main():
    dev = torch.device("cuda", 0)
    lib = L.lib()
    lib.bigcn_debug_set.argtypes = [C.c_int, C.c_int]
    lib.bigcn_debug_set.restype = None
    batches = []
    for i in range(3):
        b = make_batch_shard("twitter16", 128, 1000 + i)[0]
        batches.append(Batch(**{k: getattr(b, k).to(dev) for k in Batch._tensor_keys}))
    torch.manual_seed(0)
    model = bigcn_b200.BiGCN(5000, 64, 64, dev, gemm_mode="sparse", validate="off").to(dev).train()
    tr = bigcn_b200.FusedTrainer(model)      # CUDA graphs (host enqueue would hide the differences): re-captured per knob value
    prefetch = os.environ.get("BIGCN_PREFETCH", "1") != "0"
    nxt = lambda i: batches[(i + 1) % 3] if prefetch else None  # noqa: E731

    def run(steps=60):
        # knobs are read at enqueue / capture time: start from no captures and no sightings
        tr._graphs = GraphCache(tr._graphs.max_graphs, tr._graphs.max_seen)
        for i in range(18):
            tr.step(batches[i % 3], next_data=nxt(i))
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(18, 18 + steps):
            tr.step(batches[i % 3], next_data=nxt(i))
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps
    for a in [a for a in sys.argv[1:] if a.startswith("set:")]:      # "set:15=1": holds for the whole run (combinations)
        key, v = a[4:].split("=")
        lib.bigcn_debug_set(int(key), int(v))
    spec = [a for a in sys.argv[1:] if not a.startswith("set:")] or ["10:0,9"]
    print(f"baseline {run():.4f} ms/step", flush=True)
    for s in spec:
        key, vals = s.split(":")
        for v in vals.split(","):
            lib.bigcn_debug_set(int(key), int(v))
            print(f"knob {key} = {v}: {run():.4f} ms/step", flush=True)
        lib.bigcn_debug_set(int(key), 0)      # 0: the shipped value of every key
    tr.check_inputs()


if __name__ == "__main__":
    main()
