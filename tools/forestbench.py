#!/usr/bin/env python
"""DeviceForest with dense features (PHEME), in one GPU call (JSON lines on stdout and in --out, by default
profiles/r06_forestbench.jsonl):

  gpu       card name, power limit and max SM clock (nvidia-smi) and the device-to-device copy peak (tools/dxbench.py's
            probe: 1 GiB copied, 2 GiB moved), read in the same call.
  assembly  the row gather alone (k_asm_dense_rows) on a 6,425-tree PHEME-shaped data.synth_forest_device forest: fp32
            and bf16 storage, random id lists of 24 and 4,096 trees, and 24 trees at K = 196,608 in bf16 (a 300-tree
            forest: the 6,425-tree one would be 40 GB).  Kernel time from torch.profiler (a run of its own), each call
            after a 256 MB write that evicts L2, so both the forest rows and the batch start cold; algorithmic bytes
            2 n K s over that time, and the fraction of the copy peak.  Beside it, CUDA events over back-to-back
            DeviceForest.batch calls (all three assembly kernels and the host work, L2 not flushed).
  loop      ms per step of DeviceForest.batches + FusedTrainer.step(next_data=...) over PHEME training epochs (all
            6,425 trees shuffled, batch 24 and 4,096, DropEdge 0.2 / 0.2), host clock around whole epochs ending in a
            device synchronise, one warm-up epoch, three timed repeats, for four routes:
              dense_fp32_auto   dense fp32 storage, gemm_mode 'auto' (-> tf32x3 with dense_roots)
              dense_bf16_bf16   dense bf16 storage, gemm_mode 'bf16'
              csr_auto          the same features stored as CSR (every entry), 'auto' (-> sparse); errors recorded
              slice_views       data.forest_slice_batch views of contiguous trees: no shuffle, no DropEdge, no gather,
                                batches built before the timed loop (the no-gather reference)
  share     torch.profiler over one epoch of dense_fp32_auto and dense_bf16_bf16 (a run of its own): device time of the
            assembly kernels per step and their share of all kernel time.
Default: every part; name parts to run fewer (python tools/forestbench.py assembly).
"""
import argparse
import json
import os
import subprocess
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import numpy as np  # noqa: E402
import torch  # noqa: E402
import bigcn_b200  # noqa: E402
from bigcn_b200.data import forest_slice_batch, synth_forest_device  # noqa: E402
from dxbench import copy_peak  # noqa: E402

N_TREES = 6425            # PHEME's threads (bench_configs.PHEME_EVENT_SIZES)
ASM_KERNELS = ("k_asm_dense_rows", "k_asm_nodes", "k_asm_edges")
_out = None


def out(**kw):
    line = json.dumps(kw)
    print(line, flush=True)
    if _out:
        with open(_out, "a") as f:
            f.write(line + "\n")


def kernel_times(prof, names):
    """{name: (total device ms, launches)} of the kernels whose name contains one of ``names``"""
    res = {}
    for e in prof.key_averages():
        for k in names:
            if k in e.key:
                t = getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0)) / 1e3
                a, c = res.get(k, (0.0, 0))
                res[k] = (a + t, c + e.count)
    return res


def all_kernel_ms(prof):
    tot = 0.0
    for e in prof.key_averages():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            tot += getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0)) / 1e3
    return tot


def pheme_dict(dev, dtype, n_trees=N_TREES, k=None, seed=9):
    f = synth_forest_device("pheme", n_trees, dev, seed=seed, in_feats=k)
    f["x"] = f["x"].to(dtype)
    return f


def assembly(dev, peak):
    rng = np.random.default_rng(0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    cases = [(torch.float32, None, N_TREES, 24), (torch.float32, None, N_TREES, 4096),
             (torch.bfloat16, None, N_TREES, 24), (torch.bfloat16, None, N_TREES, 4096),
             (torch.bfloat16, 196608, 300, 24)]
    for dtype, k, n_trees, bsz in cases:
        torch.cuda.empty_cache()
        f = pheme_dict(dev, dtype, n_trees, k)
        forest = bigcn_b200.DeviceForest.from_device_arrays(f)
        kk, s = forest.in_feats, forest.x.element_size()
        lists = [rng.choice(n_trees, bsz, replace=False) for _ in range(8)]
        nodes = [int((forest.h_node_ptr[ids + 1] - forest.h_node_ptr[ids]).sum()) for ids in lists]
        calls = 40 if bsz == 24 else 16
        for i in range(4):
            forest.batch(lists[i % 8], 0.2, 0.2, seed=i)
        torch.cuda.synchronize()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for i in range(calls):
                flush.zero_()
                forest.batch(lists[i % 8], 0.2, 0.2, seed=i)
            torch.cuda.synchronize()
        kt = kernel_times(prof, ASM_KERNELS)
        ms_gather = kt["k_asm_dense_rows"][0] / kt["k_asm_dense_rows"][1]
        by = np.mean([2 * nodes[i % 8] * kk * s for i in range(calls)])
        # back to back, no flush: what a loader loop pays per batch (device events; host work included if it is slower)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(calls):
            forest.batch(lists[i % 8], 0.2, 0.2, seed=i)
        e1.record()
        torch.cuda.synchronize()
        out(part="assembly", dtype=str(dtype)[6:], K=kk, forest_trees=n_trees, forest_bytes=int(forest.x.numel() * s),
            trees=bsz, nodes_mean=round(float(np.mean(nodes)), 1), alg_bytes_mean=int(by), calls=calls,
            ms_gather_cold=round(ms_gather, 5), gbs_gather=round(by / (ms_gather * 1e-3) / 1e9, 1),
            frac_copy_peak=round(by / (ms_gather * 1e-3) / peak, 3),
            ms_asm_nodes=round(kt["k_asm_nodes"][0] / kt["k_asm_nodes"][1], 5),
            ms_asm_edges=round(kt["k_asm_edges"][0] / kt["k_asm_edges"][1], 5),
            ms_batch_call_back_to_back=round(e0.elapsed_time(e1) / calls, 5))
        del forest, f


def csr_dict(f):
    """the same dataset with its dense rows stored as CSR: every entry (tanh of a normal is never 0)"""
    x = f["x"]
    n, k = x.shape
    g = dict(f)
    del g["x"]
    g["x_ptr"] = torch.arange(0, n * k + 1, k, dtype=torch.int64, device=x.device)
    g["x_col"] = torch.arange(k, dtype=torch.int32, device=x.device).repeat(n)
    g["x_val"] = x.reshape(-1).float().contiguous()
    return g


def epoch_lists(order, bsz):
    return [order[lo:lo + bsz] for lo in range(0, len(order), bsz)]


def loop(dev):
    f32 = pheme_dict(dev, torch.float32)
    routes = {}
    routes["dense_fp32_auto"] = (lambda: bigcn_b200.DeviceForest.from_device_arrays(f32), "auto")
    routes["dense_bf16_bf16"] = (lambda: bigcn_b200.DeviceForest.from_device_arrays(
        dict(f32, x=f32["x"].to(torch.bfloat16))), "bf16")
    routes["csr_auto"] = (lambda: bigcn_b200.DeviceForest.from_device_arrays(csr_dict(f32)), "auto")
    routes["slice_views"] = (None, "auto")
    # the CSR route last: it runs gemm_mode='sparse' at 768 non-zeros per row, far outside what that path is built for
    order = [(b, r) for r in ("dense_fp32_auto", "dense_bf16_bf16", "slice_views", "csr_auto") for b in (24, 4096)]
    for bsz, name in order:
        make, mode = routes[name]
        epochs = 4 if bsz == 24 else 8          # 268 or 2 steps per epoch
        torch.cuda.empty_cache()
        rec = dict(part="loop", route=name, trees=bsz, gemm_mode=mode)
        try:
            torch.manual_seed(0)
            m = bigcn_b200.BiGCN(768, 64, 64, dev, num_classes=4, gemm_mode=mode, validate="off").to(dev).train()
            tr = bigcn_b200.FusedTrainer(m, lr=5e-4, weight_decay=1e-4)
            rng = np.random.default_rng(1)
            if make is None:
                views = [forest_slice_batch(f32, int(ids[0]), int(ids[-1]) + 1)
                         for ids in epoch_lists(np.arange(N_TREES), bsz)]
                probe = views[0].x

                def run_epoch(ep):
                    for i, b in enumerate(views):
                        tr.step(b, next_data=views[i + 1] if i + 1 < len(views) else None)
                    return len(views)
            else:
                forest = make()
                probe = forest.batch([0, 1]).x

                def run_epoch(ep):
                    lists = epoch_lists(rng.permutation(N_TREES), bsz)
                    seeds = [ep * 4096 + i for i in range(len(lists))]
                    for b, nxt in forest.batches(lists, 0.2, 0.2, seeds):
                        tr.step(b, next_data=nxt)
                    return len(lists)
            for ep in range(epochs):
                run_epoch(ep)
            torch.cuda.synchronize()
            tr.check_inputs()
            runs = []
            for rep in range(3):
                torch.cuda.synchronize()
                t0, steps = time.perf_counter(), 0
                for ep in range(epochs):
                    steps += run_epoch(1 + rep * epochs + ep)
                torch.cuda.synchronize()
                runs.append((time.perf_counter() - t0) * 1e3 / steps)
            tr.check_inputs()
            v = sorted(runs)
            rec.update(resolved=m.TDrumorGCN.resolved_gemm_mode(probe),
                       dense_roots=bool(m.TDrumorGCN.resolved_dense_roots(probe)), steps_per_repeat=steps,
                       ms_per_step_runs=[round(a, 4) for a in runs], ms_per_step_median=round(v[1], 4), spread=round(v[-1] - v[0], 4))
        except Exception as e:     # the CSR route at full density: record what happens
            rec["error"] = f"{type(e).__name__}: {e}"[:400]
        out(**rec)


def share(dev):
    f32 = pheme_dict(dev, torch.float32)
    for name, dtype, mode in (("dense_fp32_auto", torch.float32, "auto"), ("dense_bf16_bf16", torch.bfloat16, "bf16")):
        forest = bigcn_b200.DeviceForest.from_device_arrays(dict(f32, x=f32["x"].to(dtype)))
        for bsz in (24, 4096):
            torch.cuda.empty_cache()
            torch.manual_seed(0)
            m = bigcn_b200.BiGCN(768, 64, 64, dev, num_classes=4, gemm_mode=mode, validate="off").to(dev).train()
            tr = bigcn_b200.FusedTrainer(m, lr=5e-4, weight_decay=1e-4)
            rng = np.random.default_rng(2)
            reps = 1 if bsz == 24 else 4

            def epoch(ep):
                n = 0
                for r in range(reps):
                    lists = epoch_lists(rng.permutation(N_TREES), bsz)
                    for b, nxt in forest.batches(lists, 0.2, 0.2, [ep * 4096 + r * 64 + i for i in range(len(lists))]):
                        tr.step(b, next_data=nxt)
                        n += 1
                return n
            epoch(0)
            torch.cuda.synchronize()
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                steps = epoch(1)
                torch.cuda.synchronize()
            kt = kernel_times(prof, ASM_KERNELS)
            tot = all_kernel_ms(prof)
            g = kt["k_asm_dense_rows"][0]
            asm = sum(v[0] for v in kt.values())
            out(part="share", route=name, trees=bsz, steps=steps, us_gather_per_step=round(g * 1e3 / steps, 2),
                us_assembly_per_step=round(asm * 1e3 / steps, 2), us_all_kernels_per_step=round(tot * 1e3 / steps, 2),
                gather_share_of_kernel_time=round(g / tot, 4), assembly_share_of_kernel_time=round(asm / tot, 4))
            del m, tr


def main():
    global _out
    ap = argparse.ArgumentParser()
    ap.add_argument("parts", nargs="*", default=["assembly", "loop", "share"])
    ap.add_argument("--out", default=os.path.join(os.path.dirname(HERE), "profiles", "r06_forestbench.jsonl"),
                    help="the JSON lines also go to this file, rewritten by every run (default: profiles/r06_forestbench.jsonl)")
    a = ap.parse_args()
    _out = a.out
    open(_out, "w").close()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    peak = copy_peak(dev)
    out(part="gpu", nvidia_smi=smi, torch_name=torch.cuda.get_device_name(dev), copy_peak_gbs=round(peak / 1e9, 1))
    if "assembly" in a.parts:
        assembly(dev, peak)
    if "share" in a.parts:
        share(dev)
    if "loop" in a.parts:
        loop(dev)


if __name__ == "__main__":
    main()
