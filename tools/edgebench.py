#!/usr/bin/env python
"""Cost of edge weights on the module path, in one GPU call (prints JSON lines, and writes them to the file given
as the first argument when there is one):

  step    one module-path training step (BiGCN(data) forward, nll_loss, backward: what train_GCN runs before the
          optimiser) on three rotating batches, three variants alternated over five repeats of 30 steps:
          'none' (no weights), 'weights' (data.edge_weight / data.BU_edge_weight, no gradient) and 'weights_grad'
          (both require grad: the edge-gradient pass runs too).  Median ms per step (CUDA events) and the spread
          (max - min over the repeats).  Cases: Twitter16-shaped 128 trees at K = 5000 ('sparse') and PHEME-shaped
          4096 trees at K = 768 ('tf32x3').
  kernels torch.profiler (CUDA activity) over 10 'weights_grad' steps in a run of its own: device time per step of
          every kernel the weighted path adds or swaps in, beside the unweighted sweeps of a 'none' run.
  gpu     card name, power limit and max SM clock (nvidia-smi), read in the same call.
"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402
import bigcn_b200  # noqa: E402
from bigcn_b200.data import Batch, make_batch_shard  # noqa: E402

LINES = []
# kernels the weighted path adds (k_wf_*, k_w_*) or swaps in for the unweighted sweeps (*_w)
WATCH = ("k_wf_", "k_w_", "k_propagate", "k_prop1_mix")


def out(**kw):
    line = json.dumps(kw)
    LINES.append(line)
    print(line, flush=True)


def timed(fn, iters, warm):
    for i in range(warm):
        fn(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(iters):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def batches(dev, shape, trees, k):
    res = []
    for i in range(3):
        b = make_batch_shard(shape, trees, seed=5000 + i, train=True, in_feats=k)[0]
        d = Batch(**{f: getattr(b, f).to(dev) for f in Batch._tensor_keys})
        g = torch.Generator(device="cpu").manual_seed(i)
        tw = torch.rand(d.edge_index.shape[1], generator=g).to(dev) + 0.5
        bw = torch.rand(d.BU_edge_index.shape[1], generator=g).to(dev) + 0.5
        res.append((d, tw, bw))
    return res


def runner(m, data, variant):
    def one(i):
        d, tw, bw = data[i % 3]
        if variant == "none":
            d.edge_weight = d.BU_edge_weight = None
        else:
            grad = variant == "weights_grad"
            d.edge_weight = tw.detach().requires_grad_(grad)
            d.BU_edge_weight = bw.detach().requires_grad_(grad)
        m.zero_grad(set_to_none=True)
        F.nll_loss(m(d), d.y).backward()
    return one


def kernel_times(m, data, variant, steps=10):
    one = runner(m, data, variant)
    for i in range(3):
        one(i)
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for i in range(steps):
            one(i)
        torch.cuda.synchronize()
    tot = {}
    for ev in prof.key_averages():
        name = ev.key
        if any(w in name for w in WATCH):
            us = getattr(ev, "device_time_total", None)
            if us is None:
                us = ev.cuda_time_total
            short = name.split("(")[0].replace("void ", "").replace("bigcn::", "")
            tot[short] = tot.get(short, 0.0) + us
    return {k: round(v / steps, 2) for k, v in sorted(tot.items())}


def main():
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    out(part="gpu", nvidia_smi=smi, torch_name=torch.cuda.get_device_name(dev))
    variants = ("none", "weights", "weights_grad")
    for shape, trees, k, mode in (("twitter16", 128, 5000, "sparse"), ("pheme", 4096, 768, "tf32x3")):
        torch.cuda.empty_cache()
        data = batches(dev, shape, trees, k)
        torch.manual_seed(0)
        m = bigcn_b200.BiGCN(k, 64, 64, dev, gemm_mode=mode, validate="off").to(dev).train()
        runs = {v: runner(m, data, v) for v in variants}
        res = {v: [] for v in variants}
        for rep in range(5):
            for v in variants:
                res[v].append(timed(runs[v], 30, warm=10 if rep == 0 else 3))
        nodes = [int(d.x.shape[0]) for d, _, _ in data]
        edges = [int(d.edge_index.shape[1] + d.BU_edge_index.shape[1]) for d, _, _ in data]
        for v in variants:
            s = sorted(res[v])
            out(part="step", shape=shape, trees=trees, K=k, mode=mode, variant=v, ms_runs=[round(a, 4) for a in res[v]],
                ms_median=round(s[len(s) // 2], 4), spread=round(s[-1] - s[0], 4), nodes_per_batch=nodes,
                edges_per_batch_td_plus_bu=edges)
        for v in ("none", "weights_grad"):
            out(part="kernels", shape=shape, trees=trees, K=k, mode=mode, variant=v, us_per_step=kernel_times(m, data, v))
        del m, runs, data
    if len(sys.argv) > 1:
        os.makedirs(os.path.dirname(os.path.abspath(sys.argv[1])), exist_ok=True)
        with open(sys.argv[1], "w") as f:
            f.write("\n".join(LINES) + "\n")


if __name__ == "__main__":
    main()
