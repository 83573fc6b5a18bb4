#!/usr/bin/env python
"""Edge-weighted training on the fused path, in one GPU call (prints JSON lines, and writes them to the file given as
the first argument when there is one; the profiler trace of `timeline` goes beside it):

  step      ms per training step, four variants alternated within the call over three repeats (median and spread):
              a  FusedTrainer, no weights, pipelined (next_data) and replayed from CUDA graphs
              b  FusedTrainer(edge_weights=True), weighted batches, pipelined and replayed
              c  FusedTrainer(edge_weights=True), weighted batches without next_data: the normalisation runs inline
              d  the module path (BiGCN(data), nll_loss, backward) plus torch.optim.Adam in the reference's lr groups
              e  FusedTrainer(edge_grad=True), weighted batches whose weights are leaves that require grad (the step
                 forms d loss / d weight and accumulates it into .grad), pipelined and replayed
              f  as e without next_data
              g  as d with weights that require grad (the modules form the edge gradient)
            Cases: Twitter16-shaped 128 trees K = 5000 'sparse' (3 batches of ~625 MB dense x in rotation, > L2);
            PHEME-shaped 24 and 4,096 trees K = 768 in 'auto' (tf32x3 + dense_roots) and 'bf16' (4,096 trees: 3 batches
            of ~125 / 63 MB; 24 trees: 32 batches in rotation, which together still fit in L2).
  forest    DeviceForest epoch loop (batches assembled on the device with DropEdge 0.2, FusedTrainer with next_data):
            ms per step, weighted forest against the same forest without weights, alternated over three repeats.
  asm       torch.profiler, a run of its own: device time of k_asm_edges<false> / <true> per batch.
  timeline  torch.profiler trace of pipelined weighted steps: the stream every kernel ran on, so that the
            normalisation kernels (k_w_*, k_wf_*) show on the prepare streams and not on the step's chain; then a
            pipelined edge_grad step: where k_w_ddeg / k_w_dweight ran against the T1 propagate and dW1.
  gpu       card name, power limit and max SM clock (nvidia-smi), read in the same call.
"""
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402
import bigcn_b200  # noqa: E402
from bigcn_b200.data import Batch, forest_slice_batch, make_batch_shard, synth_forest_device  # noqa: E402

LINES = []


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


def twitter_batches(dev, trees, k, n):
    res = []
    for i in range(n):
        b = make_batch_shard("twitter16", trees, seed=5000 + i, train=True, in_feats=k)[0]
        d = Batch(**{f: getattr(b, f).to(dev) for f in Batch._tensor_keys})
        g = torch.Generator(device="cpu").manual_seed(i)
        d.edge_weight = (1.0 - torch.rand(d.edge_index.shape[1], generator=g)).to(dev)
        d.BU_edge_weight = (1.0 - torch.rand(d.BU_edge_index.shape[1], generator=g)).to(dev)
        res.append(d)
    return res


def pheme_batches(dev, trees, n, dtype):
    f = synth_forest_device("pheme", trees * n, dev, seed=11, edge_weights=True)
    if dtype == torch.bfloat16:
        f["x"] = f["x"].to(torch.bfloat16)
    return [forest_slice_batch(f, i * trees, (i + 1) * trees) for i in range(n)]


def unweighted(d):
    return Batch(**{f: getattr(d, f) for f in Batch._tensor_keys})


def ref_adam(m, lr=5e-4, wd=1e-4):
    bu = {id(p) for p in list(m.BUrumorGCN.conv1.parameters()) + list(m.BUrumorGCN.conv2.parameters())}
    return torch.optim.Adam([{"params": [p for p in m.parameters() if id(p) not in bu]},
                             {"params": m.BUrumorGCN.conv1.parameters(), "lr": lr / 5},
                             {"params": m.BUrumorGCN.conv2.parameters(), "lr": lr / 5}], lr=lr, weight_decay=wd)


def with_leaf_weights(d):
    w = Batch(**{f: getattr(d, f) for f in Batch._tensor_keys})
    w.edge_weight = d.edge_weight.detach().clone().requires_grad_()
    w.BU_edge_weight = d.BU_edge_weight.detach().clone().requires_grad_()
    return w


def step_case(dev, name, batches, k, mode):
    r = len(batches)
    plain = [unweighted(d) for d in batches]
    learnt = [with_leaf_weights(d) for d in batches]
    models = {}
    for v in "abcdefg":
        torch.manual_seed(0)
        models[v] = bigcn_b200.BiGCN(k, 64, 64, dev, gemm_mode=mode, validate="off").to(dev).train()
    trs = {v: bigcn_b200.FusedTrainer(models[v], lr=5e-4, weight_decay=1e-4, edge_weights=v != "a", edge_grad=v in "ef",
                                      max_graphs=2 * r + 2)
           for v in "abcef"}
    opts = {v: ref_adam(models[v]) for v in "dg"}

    def fused(v, data, pipelined):
        tr = trs[v]
        return lambda i: tr.step(data[i % r], next_data=data[(i + 1) % r] if pipelined else None)

    def module(v, data):
        def run(i):
            m, d, opt = models[v], data[i % r], opts[v]
            opt.zero_grad(set_to_none=True)
            F.nll_loss(m(d), d.y).backward()
            opt.step()
        return run

    runs = {"a": fused("a", plain, True), "b": fused("b", batches, True), "c": fused("c", batches, False),
            "d": module("d", batches), "e": fused("e", learnt, True), "f": fused("f", learnt, False),
            "g": module("g", learnt)}
    iters = max(30, 3 * r)
    res = {v: [] for v in runs}
    for rep in range(3):
        for v, fn in runs.items():
            res[v].append(timed(fn, iters, warm=2 * r + 4 if rep == 0 else r))
    for v in trs:
        trs[v].check_inputs()
    assert all(d.edge_weight.grad is not None and d.BU_edge_weight.grad is not None for d in learnt)
    nodes = [int(d.batch.numel()) for d in batches]
    x_mb = [round(d.x.numel() * d.x.element_size() / 2 ** 20, 1) for d in batches]
    for v in runs:
        s = sorted(res[v])
        extra = {"graph_replays": trs[v].graph_replays} if v in trs else {}
        out(part="step", case=name, K=k, mode=mode, variant=v, ms_runs=[round(a, 4) for a in res[v]],
            ms_median=round(s[len(s) // 2], 4), spread=round(s[-1] - s[0], 4), iters=iters, batches_in_rotation=r,
            nodes_per_batch_mean=round(float(np.mean(nodes)), 1), x_mb_per_batch_mean=round(float(np.mean(x_mb)), 1),
            **extra)


def forest_case(dev, steps_per_epoch=12, trees=128):
    f = synth_forest_device("twitter16", steps_per_epoch * trees, dev, seed=3, edge_weights=True)
    g = {k: v for k, v in f.items() if k != "edge_weight"}
    forests = {"unweighted": bigcn_b200.DeviceForest.from_device_arrays(g),
               "weighted": bigcn_b200.DeviceForest.from_device_arrays(f)}
    trs = {}
    for v, fo in forests.items():
        torch.manual_seed(0)
        m = bigcn_b200.BiGCN(5000, 64, 64, dev, gemm_mode="sparse", validate="off").to(dev).train()
        trs[v] = bigcn_b200.FusedTrainer(m, lr=5e-4, weight_decay=1e-4, edge_weights=v == "weighted")
    ids = np.arange(steps_per_epoch * trees)
    lists = [ids[i * trees:(i + 1) * trees] for i in range(steps_per_epoch)]

    def epoch(v, e):
        for d, nxt in forests[v].batches(lists, 0.2, 0.2, seeds=[e * 4096 + i for i in range(len(lists))]):
            trs[v].step(d, next_data=nxt)

    res = {v: [] for v in forests}
    for v in forests:
        epoch(v, 0)
    for rep in range(3):
        for v in forests:
            res[v].append(timed(lambda i, v=v: epoch(v, i + 1), 3, warm=0) / steps_per_epoch)
    for v in forests:
        s = sorted(res[v])
        out(part="forest", variant=v, trees_per_batch=trees, steps_per_epoch=steps_per_epoch,
            ms_per_step_runs=[round(a, 4) for a in res[v]], ms_per_step_median=round(s[1], 4),
            spread=round(s[-1] - s[0], 4))
    # k_asm_edges with and without weights, in a profiler run of its own
    for v, fo in forests.items():
        for i in range(3):
            fo.batch(lists[i], 0.2, 0.2, seed=i)
    torch.cuda.synchronize()
    n = 20
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for i in range(n):
            for fo in forests.values():
                fo.batch(lists[i % len(lists)], 0.2, 0.2, seed=100 + i)
        torch.cuda.synchronize()
    tot = {}
    for ev in prof.key_averages():
        if "k_asm_" in ev.key:
            us = getattr(ev, "device_time_total", None)
            tot[ev.key.split("(")[0].replace("void ", "").replace("bigcn::", "")] = \
                round((us if us is not None else ev.cuda_time_total) / n, 2)
    out(part="asm", trees_per_batch=trees, droprate=0.2, us_per_batch=tot)


def timeline(dev, trace_path):
    batches = twitter_batches(dev, 128, 5000, 3)
    torch.manual_seed(0)
    m = bigcn_b200.BiGCN(5000, 64, 64, dev, gemm_mode="sparse", validate="off").to(dev).train()
    tr = bigcn_b200.FusedTrainer(m, lr=5e-4, weight_decay=1e-4, edge_weights=True, graphs=False)
    for i in range(4):
        tr.step(batches[i % 3], next_data=batches[(i + 1) % 3])
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        tr.step(batches[1], next_data=batches[2])
        torch.cuda.synchronize()
    prof.export_chrome_trace(trace_path)
    with open(trace_path) as fh:
        ev = json.load(fh)["traceEvents"]
    kern = [e for e in ev if e.get("cat") == "kernel"]
    streams = {}
    for e in kern:
        short = e["name"].split("(")[0].replace("void ", "").replace("bigcn::", "")
        short = short.split("<")[0]
        streams.setdefault(short, set()).add(e.get("args", {}).get("stream", e.get("tid")))
    step_streams = streams.get("k_prop1_mix_w", set())
    norm = {k: sorted(v) for k, v in streams.items() if k.startswith(("k_w_", "k_wf_"))}
    out(part="timeline", steps=1, step_chain_streams=sorted(step_streams), normalisation_streams=norm,
        normalisation_on_step_chain=any(set(v) & step_streams for v in norm.values()),
        all_kernel_streams={k: sorted(v) for k, v in sorted(streams.items())}, trace=os.path.basename(trace_path))
    # edge_grad: the chain through the normalisation forks after k_wf_edge_dot; where it ran against T1 and dW1
    learnt = [with_leaf_weights(d) for d in batches]
    torch.manual_seed(0)
    m = bigcn_b200.BiGCN(5000, 64, 64, dev, gemm_mode="sparse", validate="off").to(dev).train()
    tr = bigcn_b200.FusedTrainer(m, lr=5e-4, weight_decay=1e-4, edge_grad=True, graphs=False)
    for i in range(4):
        tr.step(learnt[i % 3], next_data=learnt[(i + 1) % 3])
    torch.cuda.synchronize()
    eg_path = trace_path.replace("timeline", "timeline_edge_grad")
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        tr.step(learnt[1], next_data=learnt[2])
        torch.cuda.synchronize()
    prof.export_chrome_trace(eg_path)
    with open(eg_path) as fh:
        kern = sorted((e for e in json.load(fh)["traceEvents"] if e.get("cat") == "kernel"), key=lambda e: e["ts"])

    def short(e):
        return e["name"].split("(")[0].replace("void ", "").replace("bigcn::", "").split("<")[0]

    t0 = kern[0]["ts"]
    dot = next(e for e in kern if short(e) == "k_wf_edge_dot")
    chain = dot.get("args", {}).get("stream", dot.get("tid"))
    after = [e for e in kern if e["ts"] >= dot["ts"] + dot["dur"]]
    t1 = next(e for e in after if short(e) == "k_propagate_w" and e.get("args", {}).get("stream", e.get("tid")) == chain)
    dw1 = next(e for e in after if short(e) == "k_dw_sweep")
    adam = next(e for e in after if "adam" in short(e))

    def span(e):
        return {"stream": e.get("args", {}).get("stream", e.get("tid")), "start_us": round(e["ts"] - t0, 2),
                "end_us": round(e["ts"] + e["dur"] - t0, 2)}
    eg = {short(e): span(e) for e in kern if short(e) in ("k_w_ddeg", "k_w_dweight")}
    eg_end = max(v["end_us"] for v in eg.values())
    out(part="timeline_edge_grad", step_chain_stream=chain, k_wf_edge_dot=span(dot), t1_propagate=span(t1),
        dw1=span(dw1), adam=span(adam), edge_chain=eg, edge_chain_ends_before_dw1_ends=eg_end <= span(dw1)["end_us"],
        adam_start_after_dw1_end_us=round(span(adam)["start_us"] - span(dw1)["end_us"], 2),
        trace=os.path.basename(eg_path))


def main():
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    dest = sys.argv[1] if len(sys.argv) > 1 else None
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    out(part="gpu", nvidia_smi=smi, torch_name=torch.cuda.get_device_name(dev), gpus=torch.cuda.device_count())
    step_case(dev, "twitter16_128", twitter_batches(dev, 128, 5000, 3), 5000, "sparse")
    torch.cuda.empty_cache()
    for trees, n in ((24, 32), (4096, 3)):
        for mode, dt in (("auto", torch.float32), ("bf16", torch.bfloat16)):
            step_case(dev, f"pheme_{trees}", pheme_batches(dev, trees, n, dt), 768, mode)
            torch.cuda.empty_cache()
    forest_case(dev)
    torch.cuda.empty_cache()
    trace = os.path.join(os.path.dirname(os.path.abspath(dest)) if dest else tempfile.gettempdir(), "r09_timeline.pt.trace.json")
    os.makedirs(os.path.dirname(trace), exist_ok=True)
    timeline(dev, trace)
    if dest:
        os.makedirs(os.path.dirname(os.path.abspath(dest)), exist_ok=True)
        with open(dest, "w") as f:
            f.write("\n".join(LINES) + "\n")


if __name__ == "__main__":
    main()
