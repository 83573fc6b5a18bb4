#!/usr/bin/env python
"""bench.py -- BiGCN training throughput (trees/s) on B200, the metric of BASELINE.json.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

A step = one pass of the hot path over one batch: graph prep + forward + nll_loss + backward
+ Adam on a Twitter16-shaped synthetic batch of 128 reply trees per GPU (BASELINE.json
configs[1]; K = 5000 bag-of-words, 4 classes, DropEdge 0.2/0.2, train mode, fp32).
`value` times the steps with the batches resident in HBM (three batches in rotation, each
~600 MB of features >> the 126 MB L2); `e2e` times the same steps fed from pinned HOST
buffers (H2D of every input inside the timed region, loss read back).  `roofline` is the
dominant kernel (the X stream) timed alone with CUDA events; `cpu_baseline` is the oracle's
restatement of the reference module -- including its Python max()/mask loops, which is what
the reference executes -- on this host's cores, on a bounded sample of the same workload.
Multi-GPU: trees are sharded per rank (weak scaling, 128 trees per GPU); the gradient exchange is the fused
peer-memory reduce-scatter + Adam + all-gather kernel (or two NCCL all-reduces with --comm nccl).  Under torchrun
the line also carries `dp_parity`: three fixed-seed steps whose parameters must be bit-identical on every rank and
within 2e-6 of a single-process replay of the same global batches on rank 0.
`configs` holds the other BASELINE.json configurations (bench_configs.py): the Twitter16 epoch, Weibo training in
the fp32-class and tensor-core modes, PHEME 9-fold inference, the 1 M-tree power-law stream.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

T0 = time.time()


def log(msg):
    """Progress on stderr (stdout carries the one JSON line)."""
    sys.stderr.write(f"[bench {time.time() - T0:7.1f}s] {msg}\n")
    sys.stderr.flush()

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SHAPE = "twitter16"
TREES_PER_GPU = 128
K_FEATS, N_CLASSES = 5000, 4
N_ROTATE = 3


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="bigcn_b200", choices=["bigcn_b200", "reference"])
    ap.add_argument("--gemm-mode", default="sparse", choices=["fp32", "tf32", "tf32x3", "mixed", "sparse"])
    ap.add_argument("--no-graphs", action="store_true", help="enqueue every launch instead of replaying CUDA graphs")
    ap.add_argument("--no-prefetch", action="store_true",
                    help="do not prepare the next batch (graph prep, pass over x, column sort) beside the current step")
    ap.add_argument("--no-configs", action="store_true", help="skip the other BASELINE.json configurations (c2..c5)")
    ap.add_argument("--configs", default="c2,c3,c4,c5", help="which of c2,c3,c4,c5 to run")
    ap.add_argument("--no-fused-sync", action="store_true", help="symm: torch symmetric-memory barriers around the optimiser kernel")
    ap.add_argument("--comm", default="auto", choices=["auto", "symm", "nccl"],
                    help="N > 1: fused peer-memory optimiser step (symm) or NCCL all-reduce + Adam")
    ap.add_argument("--cpu-sample-trees", type=int, default=TREES_PER_GPU)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-kernels", action="store_true", help="skip the large-N propagate micro-benchmark")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (loss, log-probs, the parameters "
                         "Adam wrote and the gradients it used) as DIR/<name>.npy, float32 (rank 0)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "bigcn_b200":
        ap.error("--dump-outputs applies to --impl bigcn_b200")
    return args


def dump_outputs(out_dir, tr, loss):
    """The arrays a caller of FusedTrainer.step holds after the last timed step: the loss, the batch's log-probs,
    every parameter as Adam left it and the gradient it was updated with (about 10 MB in all)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"loss": loss.reshape(1), "logp": tr.last_logp}
    arrays.update({"param." + k: v for k, v in tr.views.items()})
    arrays.update({"grad." + k: v for k, v in tr.gviews.items()})
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())
    log(f"dumped {len(arrays)} arrays to {out_dir}")


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------- clocks
class ClockSampler:
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:  # noqa: BLE001
            self.nv = None
            self.err = repr(e)

    def _run(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40,
                 "sw_thermal_slowdown": 0x20, "hw_power_brake_slowdown": 0x80,
                 "applications_clocks_setting": 0x2}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(
                    nv, "nvmlDeviceGetCurrentClocksEventReasons") else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.002)     # the timed region lasts ~13 ms: a few samples inside it

    def __enter__(self):
        if self.nv is not None:
            self._thr = threading.Thread(target=self._run, daemon=True)
            self._thr.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thr is not None:
            self._thr.join()

    def summary(self):
        if self.nv is None or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "note": "nvml unavailable"}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ------------------------------------------------------------------------------- reference arm / cpu baseline
def _load_data_module():
    """bigcn_b200/data.py loaded BY PATH: the synthetic generators without importing the package (whose __init__
    dlopens libbigcn_b200.so) -- the reference arm must not map the product's library."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bigcn_b200_data_standalone", os.path.join(ROOT, "bigcn_b200", "data.py"))
    mod = importlib.util.module_from_spec(spec)
    sys.modules[spec.name] = mod
    spec.loader.exec_module(mod)
    return mod


def cpu_reference_run(steps, warmup, sample_trees, seed=1000, shape=SHAPE, optimizer=True):
    """The reference's own CPU implementation of the path (oracle restatement of BiGCN_Twitter.py:26-131 with the
    reference's Python max()/mask loops), train mode, fwd + nll_loss + bwd (+ Adam), all host threads."""
    import torch
    from oracle import bigcn_oracle
    data = _load_data_module()
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    torch.manual_seed(0)
    b = data.make_batch(shape, sample_trees, seed=seed, train=True)
    model = bigcn_oracle.BiGCN(K_FEATS, 64, 64, num_classes=N_CLASSES, reference_loops=True).train()
    opt = bigcn_oracle.make_optimizer(model)
    times, opt_times = [], []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        out = model(b)
        loss = torch.nn.functional.nll_loss(out, b.y)
        opt.zero_grad()
        loss.backward()
        float(loss.item())
        t1 = time.perf_counter()
        opt.step()
        t2 = time.perf_counter()
        if i >= warmup:
            times.append((t2 - t0) if optimizer else (t1 - t0))
            opt_times.append(t2 - t1)
    times.sort()
    opt_times.sort()
    med = times[len(times) // 2]
    return {"value": sample_trees / med, "unit": "trees/s", "cores": cores, "kind": "port",
            "sample": f"{sample_trees} {shape}-shaped trees ({int(b.x.shape[0])} nodes) per step, {steps} timed steps "
                      f"after {warmup} warm-up, median; oracle restatement incl. the reference's Python loops; "
                      + ("fwd+nll+bwd+Adam" if optimizer else "fwd+nll+bwd (optimizer step reported separately)"),
            "ms_per_step": med * 1e3, "optimizer_ms": opt_times[len(opt_times) // 2] * 1e3, "nodes": int(b.x.shape[0]),
            "torch_threads": cores}


def cpu_config1():
    """BASELINE.md section 4, to the letter: config 1 = Twitter15-shaped, 128 trees, seed 0, fwd + nll_loss + bwd,
    1 warm-up + 3 timed steps, median."""
    r = cpu_reference_run(3, 1, 128, seed=0, shape="twitter15", optimizer=False)
    return {k: r[k] for k in ("value", "unit", "cores", "kind", "sample", "ms_per_step", "optimizer_ms", "nodes")}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = max(1, min(args.steps, 3))
    warm = max(1, min(args.warmup, 1))
    r = cpu_reference_run(steps, warm, args.cpu_sample_trees)
    line = {"impl": "reference", "metric": "BiGCN train trees/sec", "value": r["value"], "unit": "trees/s",
            "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": r["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp32",
            "data": "synthetic",
            "config": {"workload": f"{SHAPE}-shaped BiGCN training step (graph prep+fwd+nll+bwd+Adam), "
                                   f"{TREES_PER_GPU} trees/GPU, K={K_FEATS}, C={N_CLASSES}, DropEdge 0.2/0.2, dropout 0.5",
                       "trees_per_step": args.cpu_sample_trees, "trees_per_gpu": TREES_PER_GPU,
                       "note": "CPU arm: the same batch shape as the GPU arm (seed 1000), one process, all host threads"},
            "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": r["value"], "unit": "trees/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    if not args.no_configs:
        line["configs"] = {"c1_cpu_twitter15": cpu_config1()}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------- our arm
def time_kernel(fn, iters, torch):
    """CUDA-event time of `iters` back-to-back launches on the current stream (ms per launch)."""
    for _ in range(3):
        fn(0)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(iters):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def run_ours(args):
    import torch
    import bigcn_b200
    from bigcn_b200 import _lib as L, ops
    from bigcn_b200.data import make_batch, make_batch_shard, make_trees_shard, Batch
    from bigcn_b200.trainer import launches_per_step

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    pg = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
        pg = dist.group.WORLD
    L.require_device()

    # ---- data: N_ROTATE distinct GLOBAL batches of 128 trees per GPU; every rank builds its
    # contiguous, node-balanced range of trees (SURVEY 8e), pinned on the host and resident in HBM
    shards = [make_batch_shard(SHAPE, TREES_PER_GPU * world, seed=1000 + i, rank=rank, world=world, train=True)
              for i in range(N_ROTATE)]
    host = [sh[0].pin_memory() for sh in shards]
    id_base = [sh[1] for sh in shards]
    resident = [Batch(**{k: getattr(b, k).to(dev) for k in Batch._tensor_keys}) for b in host]
    nodes = [int(b.x.shape[0]) for b in host]
    h2d_bytes = sum(getattr(host[0], k).numel() * getattr(host[0], k).element_size() for k in Batch._tensor_keys)

    torch.manual_seed(0)
    model = bigcn_b200.BiGCN(K_FEATS, 64, 64, dev, num_classes=N_CLASSES, gemm_mode=args.gemm_mode,
                             validate="off").to(dev).train()
    tr = bigcn_b200.FusedTrainer(model, lr=5e-4, weight_decay=1e-4, process_group=pg, world_size=world,
                                 comm=args.comm, graphs=False if args.no_graphs else "auto",
                                 fused_sync=not args.no_fused_sync)
    log(f"data + model ready ({nodes} nodes), comm={tr.comm}, graphs={tr.graphs}")
    b_global = TREES_PER_GPU * world
    sparse_ok = args.gemm_mode == "sparse"
    tr_comm, tr_comm_note = tr.comm, tr.comm_note

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident timing ------------------------------------------------------
    # The loader loop: step i is handed batch i+1 as well, whose weight-independent half (graph prep, the HBM-bound
    # pass over its x, the column sort) runs on low-priority streams beside step i.  CUDA graphs: a (batch, next
    # batch, buffer) combination is enqueued at its first sighting and captured at its second; prime them all
    # before the W warm-up steps so that the timed region only replays.
    prefetch = not args.no_prefetch
    step_no = [0]

    def run_step():
        i = step_no[0]
        step_no[0] = i + 1
        nxt = resident[(i + 1) % N_ROTATE] if prefetch else None
        return tr.step(resident[i % N_ROTATE], b_global=b_global, node_id_base=id_base[i % N_ROTATE], next_data=nxt)

    for _ in range(6 * N_ROTATE if tr.graphs else 0):
        run_step()
    for _ in range(args.warmup):
        run_step()
    tr.check_inputs()
    sampler = ClockSampler(local)          # NVML init before the barrier: its duration differs per rank
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    align = torch.zeros(1, device=dev)
    with sampler:
        barrier()
        if world > 1:                      # a collective on the stream right before e0: the timed
            torch.distributed.all_reduce(align)   # regions of all ranks start together on the devices
        t_cpu0 = time.perf_counter()
        e0.record()
        captures0, replays0 = tr.graph_captures, tr.graph_replays
        for i in range(args.steps):
            loss = run_step()
        e1.record()
        cpu_enqueue_ms = (time.perf_counter() - t_cpu0) * 1e3 / args.steps
        barrier()
    my_ms = e0.elapsed_time(e1)
    ms = max_over_ranks(my_ms)
    per_rank = [my_ms / args.steps]
    per_rank_cpu = [cpu_enqueue_ms]
    if world > 1:
        t = torch.tensor([my_ms / args.steps, cpu_enqueue_ms], dtype=torch.float64, device=dev)
        g = [torch.empty_like(t) for _ in range(world)]
        torch.distributed.all_gather(g, t)
        per_rank = [float(x[0]) for x in g]
        per_rank_cpu = [float(x[1]) for x in g]
    value = TREES_PER_GPU * world * args.steps / (ms * 1e-3)
    final_loss = float(loss.item())
    graph_info = {"enabled": bool(tr.graphs), "captures": tr.graph_captures, "replays": tr.graph_replays,
                  "captures_in_timed_region": tr.graph_captures - captures0,
                  "replays_in_timed_region": tr.graph_replays - replays0, "prefetch_next_batch": prefetch}
    log(f"resident: {ms / args.steps:.4f} ms/step, cpu enqueue {cpu_enqueue_ms:.4f} ms/step, graphs {graph_info}")
    if args.dump_outputs and rank == 0:      # before dp_parity_check, which resets the trainer's parameters
        dump_outputs(args.dump_outputs, tr, loss)
    dp_parity = dp_parity_check(torch, bigcn_b200, tr, dev, rank, world, args) if world > 1 else None

    # ---- end to end: host buffers in, loss out ---------------------------------------
    # Every step starts from the PINNED HOST tensors of a batch (the dense fp32 data.x the
    # reference's loader produces, edge lists, batch vector, labels) and ends with the loss on
    # the host.  Two routes for the dense matrix, both through the public API:
    #   "dense_h2d"    : copy the dense [N,5000] matrix to the device (644 MB over PCIe)
    #   "host_compact" : bigcn_b200.host_dense_to_csr -- one threaded pass over the host
    #                    matrix keeps the non-zero entries -- then copy the CSR (a few MB)
    #   "hybrid_feed"  : bigcn_b200.HostFeeder -- the copy engine DMAs the last rows dense (compacted on the
    #                    device) while the host threads compact the first rows; batch i+1 is fed on a side
    #                    stream while step i runs (a prefetching loader loop)
    # and, separately, the loader-native sparse route ("e2e_sparse_loader": the batch is already
    # CSR on the host, as a loader that keeps the reference's index:count pairs would hand it).
    small_keys = [k for k in Batch._tensor_keys if k != "x"]
    stage = [Batch(**{k: torch.empty_like(getattr(b, k), device=dev) for k in Batch._tensor_keys}) for b in host[:2]]

    def copy_small(src, dst):
        for k in small_keys:
            s, d = getattr(src, k), getattr(dst, k)
            if d.shape != s.shape:
                d = torch.empty_like(s, device=dev)
                setattr(dst, k, d)
            d.copy_(s, non_blocking=True)

    def e2e_dense(i):
        src, dst = host[i % N_ROTATE], stage[i % 2]
        copy_small(src, dst)
        if not isinstance(dst.x, torch.Tensor) or dst.x.shape != src.x.shape:
            dst.x = torch.empty_like(src.x, device=dev)
        dst.x.copy_(src.x, non_blocking=True)
        return float(tr.step(dst, b_global=b_global, node_id_base=id_base[i % N_ROTATE]).item())   # device -> host read of the step's result

    host_csr = [None, None]
    cap = max(nodes) * 48
    dev_csr = [ops.SparseX(torch.empty(max(nodes) + 1, dtype=torch.int32, device=dev),
                           torch.empty(cap, dtype=torch.int32, device=dev),
                           torch.empty(cap, dtype=torch.float32, device=dev), (0, K_FEATS)) for _ in range(2)]

    def ship_csr(sx, slot):
        d = dev_csr[slot]
        n, nnz = sx.shape[0], int(sx.col.numel())
        d.ptr[:n + 1].copy_(sx.ptr, non_blocking=True)
        d.col[:nnz].copy_(sx.col, non_blocking=True)
        d.val[:nnz].copy_(sx.val, non_blocking=True)
        return ops.SparseX(d.ptr[:n + 1], d.col[:nnz], d.val[:nnz], sx.shape)

    def e2e_compact(i):
        src, dst = host[i % N_ROTATE], stage[i % 2]
        host_csr[i % 2] = bigcn_b200.host_dense_to_csr(src.x, out=host_csr[i % 2], cap=cap,
                                                       n_threads=host_threads)   # threaded pass over the dense host x
        copy_small(src, dst)
        dst.x = ship_csr(host_csr[i % 2], i % 2)
        return float(tr.step(dst, b_global=b_global, node_id_base=id_base[i % N_ROTATE]).item())

    host_threads = max(1, (os.cpu_count() or 1) // max(1, int(os.environ.get("LOCAL_WORLD_SIZE", world))))
    loader_csr = [bigcn_b200.host_dense_to_csr(b.x, cap=cap) for b in host] if sparse_ok else None

    class LateRead:
        """Every step's loss crosses to pinned host memory right behind the step (non-blocking copy + event); the host
        reads it one step LATER, waiting on that event only -- so it enqueues step i while the device runs step i-1
        (a plain .item() would wait for everything enqueued so far, step i included)."""

        def __init__(self):
            self.pin = [torch.zeros(1, dtype=torch.float32).pin_memory() for _ in range(2)]
            self.ev = [torch.cuda.Event() for _ in range(2)]
            self.n = 0

        def __call__(self, loss):
            k = self.n % 2
            self.pin[k].copy_(loss, non_blocking=True)
            self.ev[k].record()
            self.n += 1
            if self.n == 1:
                return 0.0
            self.ev[1 - k].synchronize()
            return float(self.pin[1 - k][0])

    late_loader, late_forest = LateRead(), LateRead()

    def e2e_loader(i):
        src, dst = host[i % N_ROTATE], stage[i % 2]
        copy_small(src, dst)
        dst.x = ship_csr(loader_csr[i % N_ROTATE], i % 2)
        return late_loader(tr.step(dst, b_global=b_global, node_id_base=id_base[i % N_ROTATE]))

    feeder = bigcn_b200.HostFeeder(dev, K_FEATS, max(nodes), n_threads=host_threads) if sparse_ok else None

    feed_stream = torch.cuda.Stream(device=dev)
    hyb_cpu = {}
    fed = {"i": None, "ready": None}

    def feed_begin(i):
        with torch.cuda.stream(feed_stream):
            return (i, feeder.begin(host[i % N_ROTATE].x))      # the DMA of the last rows starts now

    def feed_finish(tk):
        i, ticket = tk
        src, dst = host[i % N_ROTATE], stage[i % 2]
        with torch.cuda.stream(feed_stream):
            ta = time.perf_counter()
            dst.x = feeder.finish(ticket)                        # host threads compact the first rows
            tb = time.perf_counter()
            copy_small(src, dst)
            hyb_cpu["finish.ship"] = (tb - ta) * 1e3
            hyb_cpu["finish.small"] = (time.perf_counter() - tb) * 1e3
            hyb_cpu.update({"ship." + k: v for k, v in feeder.last_cpu.items()})
            ev = torch.cuda.Event()
            ev.record()
        fed["i"], fed["ready"] = i, ev

    def e2e_hybrid(i):
        """Prefetching loader loop: batch i+1 is fed (HostFeeder, on its own stream) while the device runs
        step i; every step still ends with the device -> host read of its loss."""
        if fed["i"] != i:
            feed_finish(feed_begin(i))
        t0 = time.perf_counter()
        tk = feed_begin(i + 1)
        t1 = time.perf_counter()
        torch.cuda.current_stream().wait_event(fed["ready"])
        loss = tr.step(stage[i % 2], b_global=b_global, node_id_base=id_base[i % N_ROTATE])
        t2 = time.perf_counter()
        feed_finish(tk)
        t3 = time.perf_counter()
        out = float(loss.item())
        t4 = time.perf_counter()
        for k, v in (("begin", t1 - t0), ("step_enqueue", t2 - t1), ("finish", t3 - t2), ("loss_read", t4 - t3)):
            hyb_cpu[k] = hyb_cpu.get(k, 0.0) * 0.7 + 0.3 * v * 1e3      # running mean, ms
        return out

    def time_e2e(fn, warm=None, n_steps=None):
        warm = warm or max(1, min(args.warmup, 3))
        for i in range(warm):
            fn(i)
        barrier()
        n_steps = n_steps or max(3, min(args.steps, 12))
        t0 = time.perf_counter()
        for i in range(warm, warm + n_steps):      # the step index keeps counting: a prefetching route stays primed
            fn(i)
        torch.cuda.synchronize()
        wall = (time.perf_counter() - t0) * 1e3
        barrier()
        ms = max_over_ranks(wall)           # host work is part of this path: wall clock, max over ranks
        return TREES_PER_GPU * world * n_steps / (ms * 1e-3), ms / n_steps, n_steps

    # SURVEY 8f N2: the dataset (here: the trees of the three global batches) packed once in HBM, features as
    # CSR; every step assembles its batch on the device (collate + fresh DropEdge 0.2/0.2) from the tree
    # ids the host sampler hands over
    forest = ids_of = None
    if sparse_ok:
        all_trees, ids_of = [], []
        for i in range(N_ROTATE):
            trs = make_trees_shard(SHAPE, TREES_PER_GPU * world, seed=1000 + i, rank=rank, world=world)[0]
            ids_of.append(list(range(len(all_trees), len(all_trees) + len(trs))))
            all_trees += trs
        forest = bigcn_b200.DeviceForest.from_data_list(all_trees, dev)

    def e2e_forest(i):
        """A loader loop over the device-resident dataset: every step assembles its batch on the device (collate + a
        fresh DropEdge) and enqueues the step; the loss read back every step is the PREVIOUS step's, so the host
        enqueues step i while the device still runs step i-1 (these batches are new objects every step: no CUDA-graph
        replay; batch i+1 is assembled before step i is enqueued and handed to it as next_data, so its graph prep,
        root columns and CSR build run underneath step i)."""
        j = i % N_ROTATE
        if forest_it["i"] != i:             # (re)start the loader at step i
            forest_it["gen"] = forest.batches([ids_of[k % N_ROTATE] for k in range(i, i + 4096)], 0.2, 0.2, seeds=range(i, i + 4096))
        bd, nxt = next(forest_it["gen"])
        forest_it["i"] = i + 1
        return late_forest(tr.step(bd, b_global=b_global, node_id_base=id_base[j], next_data=nxt))
    forest_it = {"i": -1, "gen": None}

    small_bytes = sum(getattr(host[0], k).numel() * getattr(host[0], k).element_size() for k in small_keys)
    routes = {}
    v, ms_, n_ = time_e2e(e2e_dense)
    routes["dense_h2d"] = {"value": v, "ms_per_step": ms_, "h2d_bytes_per_step": h2d_bytes}
    if sparse_ok:
        v, ms_, n_ = time_e2e(e2e_compact)
        routes["host_compact"] = {"value": v, "ms_per_step": ms_,
                                  "h2d_bytes_per_step": small_bytes + host_csr[0].nbytes(),
                                  "host_threads": host_threads}
        v, ms_, n_ = time_e2e(e2e_hybrid, warm=30 if args.steps >= 10 else 3)      # the split settles over the first calls
        feeder.check()
        routes["hybrid_feed"] = {"value": v, "ms_per_step": ms_, "host_threads": host_threads,
                                 "dma_fraction": round(feeder.frac, 3), "host_loop_ms": {k: round(v, 3) for k, v in hyb_cpu.items()}, "last": {k: round(float(x), 3) for k, x in feeder.last.items()},
                                 "h2d_bytes_per_step": int(small_bytes + feeder.last.get("n_dma", 0) * K_FEATS * 4
                                                           + (1 - feeder.frac) * host_csr[0].nbytes())}
        v, ms_, _ = time_e2e(e2e_loader, warm=6, n_steps=max(12, 2 * args.steps))     # sub-millisecond steps: a longer window
        routes["sparse_loader"] = {"value": v, "ms_per_step": ms_,
                                   "h2d_bytes_per_step": small_bytes + loader_csr[0].nbytes()}
        v, ms_, _ = time_e2e(e2e_forest, warm=6, n_steps=max(12, 2 * args.steps))
        routes["device_dataset"] = {"value": v, "ms_per_step": ms_,
                                    "h2d_bytes_per_step": 5 * 8 * (len(ids_of[0]) + 1)}
    best = max((k for k in routes if k in ("dense_h2d", "host_compact", "hybrid_feed")), key=lambda k: routes[k]["value"])
    e2e_value, e2e_ms, e2e_steps = routes[best]["value"], routes[best]["ms_per_step"], n_
    e2e_h2d = routes[best]["h2d_bytes_per_step"]

    # what bounds the dense-host routes: host-memory read bandwidth of this rank's threads, all ranks probing at once
    barrier()
    hx = host[0].x
    my_gbs = float(L.lib().bigcn_host_read_gbs(hx.data_ptr(), hx.numel() * 4, host_threads, 3))
    host_gbs = [my_gbs]
    if world > 1:
        t = torch.tensor([my_gbs], dtype=torch.float64, device=dev)
        g = [torch.empty_like(t) for _ in range(world)]
        torch.distributed.all_gather(g, t)
        host_gbs = [float(v[0]) for v in g]
    log(f"e2e routes done: {({k: round(v['ms_per_step'], 3) for k, v in routes.items()})}; host read GB/s per rank {host_gbs}")
    loader_nnz = [int(c.col.numel()) for c in loader_csr] if loader_csr is not None else [0] * N_ROTATE
    del feeder, forest, stage, dev_csr, loader_csr
    configs = {}
    if not args.no_configs:
        import bench_configs as bc
        want = set(args.configs.split(","))
        try:
            if world == 1 and "c2" in want:
                configs["c2_epoch"] = bc.c2_epoch(torch, bigcn_b200, dev)
                log("c2 done")
            if world == 1 and "c3" in want:
                configs["c3_weibo"] = bc.c3_weibo(torch, bigcn_b200, dev)
                log("c3 done")
            if "c4" in want:
                configs["c4_pheme_infer"] = bc.c4_pheme_infer(torch, bigcn_b200, dev, rank, world, max_over_ranks)
                log("c4 done")
            if "c5" in want:
                configs["c5_powerlaw"] = bc.c5_powerlaw(torch, bigcn_b200, dev, rank, world, pg, max_over_ranks)
                log("c5 done")
        except Exception as e:  # noqa: BLE001  (a failing side configuration must not lose the headline line)
            if world > 1:
                raise
            configs["error"] = f"{type(e).__name__}: {e}"
            log(f"configs failed: {configs['error']}")
        torch.cuda.empty_cache()

    if rank != 0:
        if world > 1:
            torch.distributed.destroy_process_group()
        return

    # ---- roofline of the dominant kernels (rank 0, timed alone, inputs >> L2) ---------
    hbm_peak, peak_src = peaks()
    import ctypes as C
    lib = L.lib()
    st = torch.cuda.current_stream().cuda_stream
    n0 = nodes[0]
    w0 = torch.randn(64, K_FEATS, device=dev) * 0.02
    w1 = torch.randn(64, K_FEATS, device=dev) * 0.02
    scr = torch.empty(lib.bigcn_xw_scratch_floats(K_FEATS, 2), device=dev)
    ys = [torch.empty(n, 128, device=dev) for n in nodes]
    sparse = args.gemm_mode == "sparse"
    if sparse:
        xs_ws = [torch.empty(lib.bigcn_xsparse_workspace_bytes(n, K_FEATS), dtype=torch.uint8, device=dev) for n in nodes]
        xs_flags = torch.zeros(1, dtype=torch.int32, device=dev)

    def xw_fn(i):
        j = i % N_ROTATE
        if sparse:      # weight re-layout + the scan that also captures the non-zeros (no CSR/CSC build)
            L.check(lib.bigcn_xw_sparse(resident[j].x.data_ptr(), nodes[j], K_FEATS, w0.data_ptr(), w1.data_ptr(), K_FEATS,
                                        ys[j].data_ptr(), 128, 0, xs_flags.data_ptr(), xs_ws[j].data_ptr(),
                                        xs_ws[j].numel(), st))
        else:
            L.check(lib.bigcn_xw(resident[j].x.data_ptr(), nodes[j], K_FEATS, w0.data_ptr(), w1.data_ptr(), K_FEATS,
                                 ys[j].data_ptr(), 128, L.GEMM_MODE[args.gemm_mode], scr.data_ptr(), st))
    xw_ms = time_kernel(xw_fn, 12, torch)
    mean_nodes = sum(nodes[i % N_ROTATE] for i in range(12)) / 12
    # SURVEY 8(d): conv1 GEMM (TD|BU fused) bytes = N*K*4 + 128*K*4 + N*128*4
    xw_bytes = mean_nodes * K_FEATS * 4 + K_FEATS * 128 * 4 + mean_nodes * 128 * 4
    xw_gbs = xw_bytes / (xw_ms * 1e-3) / 1e9
    fwd_kernel = {"fp32": "k_xw_scan<128>", "mixed": "k_xw_scan<128>", "tf32": "k_xw_tc<1> (tcgen05 kind::tf32)",
                  "tf32x3": "k_xw_tc<2,true> (tcgen05 kind::tf32, X and W split hi+lo)",
                  "sparse": "k_transpose_jobs + k_xw_scan<128, capture>"}[args.gemm_mode]
    roof_fwd = {"kernel": fwd_kernel + ": X * [W1_td;W1_bu]^T, conv1.lin of both directions in one pass over X",
                "bound": "hbm", "achieved": xw_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": xw_gbs / hbm_peak,
                "traffic": None, "peak_source": peak_src, "ms": xw_ms, "algorithmic_bytes": xw_bytes,
                "frac_of_8TBs_nominal": xw_gbs / 8000.0}
    # the pipelined step (prefetch) reads x in bigcn_batch_prepare instead: the same pass without the product
    roof_cap = None
    if sparse:
        nnz_mean = sum(int(loader_nnz[i % N_ROTATE]) for i in range(12)) / 12

        def cap_fn(i):
            j = i % N_ROTATE
            L.check(lib.bigcn_x_capture(resident[j].x.data_ptr(), nodes[j], K_FEATS, 0, xs_flags.data_ptr(), xs_ws[j].data_ptr(),
                                        xs_ws[j].numel(), st))
        cap_ms = time_kernel(cap_fn, 12, torch)
        cap_bytes = mean_nodes * K_FEATS * 4 + nnz_mean * 8 + mean_nodes * 4      # x once; (col, val) per non-zero + a count per row
        cap_gbs = cap_bytes / (cap_ms * 1e-3) / 1e9
        # the same pass as an UNPACED kernel (LDG form, all the bytes in flight the SMs can hold): what the pass can do alone
        lib.bigcn_debug_set.argtypes = [C.c_int, C.c_int]
        lib.bigcn_debug_set.restype = None
        lib.bigcn_debug_set(10, 9)
        unp_ms = time_kernel(cap_fn, 12, torch)
        lib.bigcn_debug_set(10, 0)
        unp_gbs = cap_bytes / (unp_ms * 1e-3) / 1e9
        roof_cap = {"kernel": "k_x_capture_tma<4,3> (bigcn_batch_prepare: the one pass over the dense x of a step, run a step ahead "
                              "beside the current step's chain; TMA-fed, persistent, PACED: at most 48 KB in flight per SM)",
                    "bound": "hbm", "achieved": cap_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": cap_gbs / hbm_peak,
                    "traffic": None, "peak_source": peak_src, "ms": cap_ms, "algorithmic_bytes": cap_bytes,
                    "frac_of_8TBs_nominal": cap_gbs / 8000.0,
                    "paced_by_design": "the pass has a whole step (~0.33 ms) to read 625 MB, i.e. needs ~1.9 TB/s; it keeps 4 warps x 3 x 4 KB "
                                       "of bulk copies in flight per SM (128 threads, 48 KB of shared memory): what it must not take from "
                                       "the step's latency-bound kernels is SM slots, registers and shared memory (the same pass fed from "
                                       "L2-resident rows leaves the step time unchanged, so HBM contention is not what the chain feels).  "
                                       "`unpaced` below is the same pass as a kernel that takes the whole machine: faster alone, but the "
                                       "step is 10 % slower with it (tools/stepbench.py 10:0,9: 0.326 vs 0.362 ms)",
                    "unpaced": {"kernel": "k_xw_scan<64, capture, no product> (LDG form, 3.9 k short CTAs)", "ms": unp_ms,
                                "achieved": unp_gbs, "frac": unp_gbs / hbm_peak, "frac_of_8TBs_nominal": unp_gbs / 8000.0,
                                "note": "a read-only stream: `peak` is the measured COPY bandwidth (read + write traffic), which a "
                                        "pure read stream can exceed slightly"},
                    "note": "timed alone (CUDA events, 12 launches over the 3 batches in rotation, each 625 MB >> L2); inside the "
                            "step it runs the whole length of the step underneath the chain (~320 us)"}
    # the weight gradient dW1 = T1^T X
    ts = [torch.randn(n, 128, device=dev) for n in nodes]
    dws = [torch.empty(64, K_FEATS, device=dev) for _ in range(2)]
    if sparse:
        for j in range(N_ROTATE):    # build the column-sorted copies once (in a step: on the side stream)
            L.check(lib.bigcn_xw_sparse(resident[j].x.data_ptr(), nodes[j], K_FEATS, w0.data_ptr(), w1.data_ptr(), K_FEATS,
                                        ys[j].data_ptr(), 128, 1, xs_flags.data_ptr(), xs_ws[j].data_ptr(),
                                        xs_ws[j].numel(), st))

        def dw_fn(i):
            j = i % N_ROTATE
            L.check(lib.bigcn_xw_wgrad_sparse(nodes[j], K_FEATS, ts[j].data_ptr(), 2, dws[0].data_ptr(), dws[1].data_ptr(),
                                              K_FEATS, xs_ws[j].data_ptr(), xs_ws[j].numel(), st))
    else:
        wscr = torch.empty(max(lib.bigcn_xw_wgrad_scratch_floats(n, K_FEATS, 2) for n in nodes), device=dev)

        def dw_fn(i):
            j = i % N_ROTATE
            L.check(lib.bigcn_xw_wgrad(resident[j].x.data_ptr(), nodes[j], K_FEATS, ts[j].data_ptr(), 2, dws[0].data_ptr(),
                                       dws[1].data_ptr(), K_FEATS, L.GEMM_MODE[args.gemm_mode], wscr.data_ptr(), st))
    dw_ms = time_kernel(dw_fn, 12, torch)
    # same algorithmic bytes: X once, T [N,128] once, dW [128,K] once
    dw_gbs = xw_bytes / (dw_ms * 1e-3) / 1e9
    bwd_kernel = {"fp32": "k_dw_slab<128> + k_dw_reduce", "tf32": "k_dw_tc<1> (tcgen05 kind::tf32, MN-major) + k_dw_reduce",
                  "tf32x3": "k_split + k_dw_tc<2> (tcgen05 kind::tf32, MN-major, T hi+lo) + k_dw_reduce",
                  "mixed": "k_split + k_dw_tc<2> (tcgen05 kind::tf32, MN-major, T hi+lo) + k_dw_reduce",
                  "sparse": "k_dw_sweep (CSR sweep over the column-sorted non-zeros of X)"}[args.gemm_mode]
    roof_bwd = {"kernel": bwd_kernel + ": dW1 = T1^T X for both directions" + ("" if sparse else ", second pass over X"),
                "bound": "hbm", "achieved": dw_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": dw_gbs / hbm_peak,
                "traffic": None, "peak_source": peak_src, "ms": dw_ms, "algorithmic_bytes": xw_bytes,
                "frac_of_8TBs_nominal": dw_gbs / 8000.0,
                "note": "ms covers the split-K reduce (and the T split) launched with the GEMM"}
    if sparse:
        nnz = int((resident[0].x != 0).sum().item())
        sw_bytes = nnz * (8 + 512) + K_FEATS * 128 * 4 + (K_FEATS + 1) * 4     # entries + gathered T rows + dW
        roof_bwd.update({"bound": "l2 (gathers of L2-resident T1 rows; X is not read again)",
                         "achieved": sw_bytes / (dw_ms * 1e-3) / 1e9, "frac": None, "peak": None,
                         "algorithmic_bytes": sw_bytes, "nnz": nnz, "frac_of_8TBs_nominal": None,
                         "note": "the dense-mode second pass over X (%.0f MB) is gone" % (nodes[0] * K_FEATS * 4 / 1e6)})
    # the tcgen05 / TMA / TMEM GEMMs on the same matrices (gemm_mode tf32 / tf32x3; what 'auto' picks for dense features)
    tc = {}
    wscr_tc = torch.empty(max(lib.bigcn_xw_wgrad_scratch_floats(n, K_FEATS, 2) for n in nodes), device=dev)
    for mode, kname in (("tf32", "k_xw_tc<1> (tcgen05.mma kind::tf32, TMA, TMEM)"),
                        ("tf32x3", "k_xw_tc<2,true> (tcgen05.mma kind::tf32 x3: X split hi/lo in shared memory, W hi/lo; fp32-class)")):
        def fn(i, mode=mode):
            j = i % N_ROTATE
            L.check(lib.bigcn_xw(resident[j].x.data_ptr(), nodes[j], K_FEATS, w0.data_ptr(), w1.data_ptr(), K_FEATS,
                                 ys[j].data_ptr(), 128, L.GEMM_MODE[mode], scr.data_ptr(), st))
        t_ms = time_kernel(fn, 12, torch)
        g = xw_bytes / (t_ms * 1e-3) / 1e9
        tc["xw_" + mode] = {"kernel": kname, "bound": "hbm", "achieved": g, "peak": hbm_peak, "unit": "GB/s", "frac": g / hbm_peak,
                            "ms": t_ms, "algorithmic_bytes": xw_bytes, "tflops": 2 * mean_nodes * K_FEATS * 128 / (t_ms * 1e-3) / 1e12,
                            "note": "ms includes the weight hi/lo split kernel of the mode"}

    def dw_tc_fn(i):
        j = i % N_ROTATE
        L.check(lib.bigcn_xw_wgrad(resident[j].x.data_ptr(), nodes[j], K_FEATS, ts[j].data_ptr(), 2, dws[0].data_ptr(),
                                   dws[1].data_ptr(), K_FEATS, L.GEMM_MODE["tf32x3"], wscr_tc.data_ptr(), st))
    t_ms = time_kernel(dw_tc_fn, 12, torch)
    g = xw_bytes / (t_ms * 1e-3) / 1e9
    tc["dw_tf32x3"] = {"kernel": "k_split + k_dw_tc<2> (tcgen05 kind::tf32, MN-major, T hi+lo) + k_dw_reduce", "bound": "hbm",
                       "achieved": g, "peak": hbm_peak, "unit": "GB/s", "frac": g / hbm_peak, "ms": t_ms,
                       "algorithmic_bytes": xw_bytes}
    del wscr_tc
    log("kernel rooflines done")
    # DRAM bytes per launch from the committed `ncu --set full` captures (profiles/traffic.json)
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        if args.gemm_mode in ("fp32", "mixed", "sparse"):
            key = "k_xw_scan_capture" if sparse and "k_xw_scan_capture" in traffic else "k_xw_scan"
            roof_fwd["traffic"] = traffic[key]["bytes"]
            roof_fwd["traffic_note"] = f"ncu capture of {key} at N = {traffic[key]['nodes']} nodes; algorithmic bytes above are the mean over the rotation"
            if roof_cap is not None and "k_x_capture" in traffic:
                key = "k_x_capture_tma" if "k_x_capture_tma" in traffic else "k_x_capture"
                roof_cap["traffic"] = traffic[key]["bytes"]
                roof_cap["traffic_note"] = (f"ncu --set full capture of {key} at N = {traffic[key]['nodes']} nodes "
                                            "(profiles/); algorithmic bytes above are the mean over the rotation")
        if args.gemm_mode in ("tf32x3", "mixed"):
            roof_bwd["traffic"] = traffic["k_dw_tc"]["bytes"]
            roof_bwd["traffic_note"] = f"GEMM kernel only, ncu capture at N = {traffic['k_dw_tc']['nodes']} nodes"
    except Exception:  # noqa: BLE001
        pass
    roof, other_gemm = (roof_bwd, roof_fwd) if (dw_ms >= xw_ms and not sparse) else (roof_fwd, roof_bwd)
    others = {"weight_gradient_dW1" if sparse else "other_x_stream": other_gemm, "xw_tcgen05": tc}
    if roof_cap is not None and prefetch:      # the dominant kernel of the step as it is timed: the background pass over x
        others["xw_scan_fused_product"] = roof
        roof = roof_cap
    if not args.no_kernels:
        others.update(kernel_microbench(torch, L, ops, dev, hbm_peak))

    cpu = None
    if not args.no_cpu_baseline:
        cpu = cpu_reference_run(3, 1, args.cpu_sample_trees)
        log("cpu baseline done")
        if not args.no_configs:
            configs["c1_cpu_twitter15"] = cpu_config1()
            log("cpu config 1 done")

    line = {"metric": "BiGCN train trees/sec", "value": value, "unit": "trees/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp32",
            "data": "synthetic",
            "config": {"workload": f"{SHAPE}-shaped BiGCN training step (graph prep+fwd+nll+bwd+Adam), "
                                   f"{TREES_PER_GPU} trees/GPU, K={K_FEATS}, C={N_CLASSES}, DropEdge 0.2/0.2, dropout 0.5",
                       "trees_per_gpu": TREES_PER_GPU, "nodes_per_batch": nodes, "gemm_mode": args.gemm_mode,
                       "sharding": "global batch of 128 trees per GPU, contiguous tree ranges balanced by node count",
                       "pipeline": ("step i also prepares batch i+1 (graph prep, pass over x, column sort) on low-priority streams"
                                    if prefetch else "every step prepares its own batch") + ("; CUDA-graph replay" if graph_info["enabled"] else ""),
                       "l2": f"{N_ROTATE} batches in rotation, {nodes[0] * K_FEATS * 4 / 1e6:.0f} MB of features each (> 126 MB L2)",
                       "parallelism": (f"dp{world} (trees sharded; " + (
                           "gradient reduce-scatter + Adam + parameter all-gather fused in one kernel over NVLink peer memory"
                           if tr_comm == "symm" else "two bucketed NCCL all-reduces of the flat gradient + Adam on every rank")
                           + ")") if world > 1 else "single GPU", "comm": tr_comm, "comm_note": tr_comm_note},
            "clocks": sampler.summary(),
            "e2e": {"value": e2e_value, "unit": "trees/s", "h2d_bytes_per_step": e2e_h2d, "d2h_bytes_per_step": 4,
                    "steps": e2e_steps, "ms_per_step": e2e_ms, "route": best,
                    "note": "dense fp32 data.x in pinned host memory -> loss on the host, wall clock; routes timed: "
                            "dense_h2d = the matrix crosses PCIe as is, host_compact = host_dense_to_csr keeps the "
                            "non-zeros on the host and the CSR crosses PCIe, hybrid_feed = HostFeeder.ship: the copy "
                            "engine DMAs the last rows dense (compacted on the device) while the host threads compact "
                            "the first rows, split adapted so both finish together; the fastest one is reported",
                    "routes": {k: v for k, v in routes.items() if k in ("dense_h2d", "host_compact", "hybrid_feed")},
                    "host_read_gbs": {"per_rank": [round(v, 1) for v in host_gbs], "sum": round(sum(host_gbs), 1),
                                      "threads_per_rank": host_threads,
                                      "note": "STREAM-style read probe (bigcn_host_read_gbs) run by every rank at the same "
                                              "time over its pinned feature matrix: the dense-host routes read "
                                              f"{nodes[0] * K_FEATS * 4 / 1e6:.0f} MB of host memory per step and rank, so "
                                              "trees/s <= trees_per_step x (this + PCIe share) / that size"}},
            "gpu_launches": args.steps * (launches_per_step(nodes[0], 2, True, args.gemm_mode, K_FEATS)
                                          + (1 if prefetch and sparse_ok else 0)),
            "roofline": roof, "final_loss": final_loss, "cuda_graphs": graph_info,
            "step_vs_hbm_floor": {"floor_ms": nodes[0] * K_FEATS * 4 / (hbm_peak * 1e9) * 1e3, "step_ms": ms / args.steps,
                                  "frac": nodes[0] * K_FEATS * 4 / (hbm_peak * 1e9) * 1e3 / (ms / args.steps),
                                  "note": "x read once at the measured HBM peak vs the whole step (graph prep + fwd + bwd + Adam)"},
            "per_rank": {"gpu_ms_per_step": [round(v, 4) for v in per_rank],
                         "cpu_enqueue_ms_per_step": [round(v, 4) for v in per_rank_cpu],
                         "nodes_per_step_mean": sum(nodes) / len(nodes)}}
    if "device_dataset" in routes:
        line["e2e_device_dataset"] = dict(routes["device_dataset"], unit="trees/s", d2h_bytes_per_step=4,
                                          note="dataset packed once in HBM (features as CSR); per step the host sends the "
                                               "tree ids, bigcn_assemble_batch collates and applies a fresh DropEdge 0.2/0.2 "
                                               "on the device (SURVEY 8f N2, stands in for BiGraphDataset + PyG collate)")
    if "sparse_loader" in routes:
        line["e2e_sparse_loader"] = dict(routes["sparse_loader"], unit="trees/s", d2h_bytes_per_step=4,
                                         note="data.x already CSR on the host (a loader that keeps the reference's "
                                              "index:count pairs): SURVEY 8f N1, an API extension, not the dense contract")
    if others:
        line["roofline_others"] = others
    if configs:
        line["configs"] = configs
    if dp_parity is not None:
        line["dp_parity"] = dp_parity["status"]
        line["dp_parity_detail"] = dp_parity
    if cpu is not None:
        line["cpu_baseline"] = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")}
    print(json.dumps(line), flush=True)
    if world > 1:
        torch.distributed.destroy_process_group()


def dp_parity_check(torch, bigcn_b200, tr, dev, rank, world, args, n_steps=3, trees_per_rank=16):
    """Multi-GPU correctness under the driver's own launch: from a common fixed state, three fixed-seed steps on
    a sharded global batch; then (a) the flat parameters must be BIT-IDENTICAL on every rank, (b) rank 0 replays
    the same global batches in a single-process trainer and the result must agree within 2e-6 of the parameter
    scale (only the summation order of the gradient differs)."""
    import torch.distributed as dist
    from bigcn_b200.data import Batch, make_batch_shard
    torch.manual_seed(1234)
    ref_model = bigcn_b200.BiGCN(K_FEATS, 64, 64, dev, num_classes=N_CLASSES, gemm_mode=args.gemm_mode,
                                 validate="off").to(dev).train()
    ref_tr = bigcn_b200.FusedTrainer(ref_model, lr=5e-4, weight_decay=1e-4, graphs=False)   # same seed on every rank
    init = ref_tr.flat.detach().clone()
    torch.cuda.synchronize()
    dist.barrier()
    tr.flat.copy_(init)
    tr.exp_avg.zero_()
    tr.exp_avg_sq.zero_()
    tr.step_count[0] = 0                 # the Adam step; [2] (calls counter = barrier epoch, dropout seed offset) never rewinds
    tr._graphs.clear()
    torch.cuda.synchronize()
    dist.barrier()
    glob = trees_per_rank * world
    for i in range(n_steps):
        b, base, _ = make_batch_shard(SHAPE, glob, seed=7000 + i, rank=rank, world=world, train=True)
        bd = Batch(**{k: getattr(b, k).to(dev) for k in Batch._tensor_keys})
        tr.step(bd, b_global=glob, node_id_base=base, seed=4242 + i)
    tr.check_inputs()
    torch.cuda.synchronize()
    mine = tr.flat.detach().clone()
    gathered = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(gathered, mine)
    identical = all(torch.equal(g, gathered[0]) for g in gathered)
    res = {"status": "n/a", "ranks_bit_identical": bool(identical), "steps": n_steps, "global_trees_per_step": glob}
    if rank == 0:
        for i in range(n_steps):
            b, base, _ = make_batch_shard(SHAPE, glob, seed=7000 + i, rank=0, world=1, train=True)
            bd = Batch(**{k: getattr(b, k).to(dev) for k in Batch._tensor_keys})
            ref_tr.step(bd, b_global=glob, node_id_base=base, seed=4242 + i)
        ref_tr.check_inputs()
        torch.cuda.synchronize()
        diff = float((ref_tr.flat.double() - mine.double()).abs().max())
        scale = float(ref_tr.flat.abs().max())
        moved = float((ref_tr.flat.double() - init.double()).abs().max())
        ok = identical and diff <= 2e-6 * scale
        res.update(status="ok" if ok else "FAIL", max_abs_diff_vs_single_process=diff, param_scale=scale,
                   max_abs_update=moved, tolerance=2e-6 * scale)
    dist.barrier()
    return res


def kernel_microbench(torch, L, ops, dev, hbm_peak):
    """propagate (both CSR orientations) and readout on a forest far larger than L2
    (16384 trees x 256 nodes = 4.2 M rows, 1.07 GB per [N,64] panel)."""
    from bigcn_b200.data import make_device_forest
    out = {}
    n_trees, per = 16384, 256
    n = n_trees * per
    f = make_device_forest(n_trees, per, dev, seed=3)
    graphs, node_ptr, flags = ops.graph_prep([f.edge_index, f.BU_edge_index], n, f.batch, n_trees, rowsum=False)
    e = int(f.edge_index.shape[1])
    hs = [torch.randn(n, 64, device=dev) for _ in range(2)]
    outb = torch.empty(n, 64, device=dev)
    lib = L.lib()
    st = torch.cuda.current_stream().cuda_stream
    bias = torch.zeros(64, device=dev)
    for name, g in (("propagate_td_parent_gather", graphs[0]), ("propagate_bu_child_segment_sum", graphs[1])):
        ptr, idx = g["in_ptr"], g["in_idx"]

        def fn(i, ptr=ptr, idx=idx, g=g):
            L.check(lib.bigcn_propagate(ptr.data_ptr(), idx.data_ptr(), g["dis"].data_ptr(), n, g["E"],
                                        g["in_long"].data_ptr(), hs[i % 2].data_ptr(), 64,
                                        bias.data_ptr(), 1, outb.data_ptr(), 64, st))
        ms = time_kernel(fn, 10, torch)
        # SURVEY 8(d): N*(2*256 + 8) + 4E + 260 bytes (each source row counted once)
        byt = n * (2 * 256 + 8) + 4 * e + 260
        gbs = byt / (ms * 1e-3) / 1e9
        out[name] = {"kernel": "k_propagate (CSR sweep, cp.async stage)", "bound": "hbm", "achieved": gbs, "peak": hbm_peak,
                     "unit": "GB/s", "frac": gbs / hbm_peak, "frac_of_8TBs_nominal": gbs / 8000.0, "ms": ms,
                     "nodes": n, "edges": e, "algorithmic_bytes": byt}
    scr = torch.empty(lib.bigcn_readout_scratch_floats(n, n_trees), device=dev)
    feat = torch.empty(n_trees, 128, device=dev)

    def ro(i):
        L.check(lib.bigcn_readout(hs[i % 2].data_ptr(), hs[(i + 1) % 2].data_ptr(), node_ptr.data_ptr(),
                                  f.rootindex.data_ptr(), n, n_trees, feat.data_ptr(), 128, None, scr.data_ptr(),
                                  flags.data_ptr(), st))
    ms = time_kernel(ro, 10, torch)
    # SURVEY 8(d): read N*256 (h2) + B*256 (root h1) + 4(B+1), write B*512
    byt = n * 256 + n_trees * 256 + 4 * (n_trees + 1) + n_trees * 512
    gbs = byt / (ms * 1e-3) / 1e9
    out["readout_scatter_mean"] = {"kernel": "k_readout_part + k_readout_final", "bound": "hbm", "achieved": gbs,
                                   "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak,
                                   "frac_of_8TBs_nominal": gbs / 8000.0, "ms": ms, "nodes": n, "trees": n_trees,
                                   "algorithmic_bytes": byt}
    return out


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
