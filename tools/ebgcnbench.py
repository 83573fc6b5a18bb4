#!/usr/bin/env python
"""EBGCN: bigcn_b200.EBGCN (bn1 + conv2 per tree, csrc/ebgcn.cu) against the materialising harness
(tests/ebgcn_harness.py: root_extend, cat and torch's BatchNorm1d over N x (64 + K)), in one GPU call.  Prints JSON
lines, and writes them to the file given with --out.

  step   ms for forward + nll_loss + backward in training mode, the two models alternated step by step (CUDA events
         around each step, median and min/max over the timed steps), edge inference off ("plain": the path this library
         replaces) and on ("infer": the reference's edge-inference sub-networks, plain torch, run in both).
  mem    torch.cuda.max_memory_allocated above what is allocated before the step (the batch and the model), for one
         training step of each model, and one fp32 copy of x (N x K x 4 bytes) for scale.
  gpu    card name, power limit and max SM clock (nvidia-smi), read in the same call.

Cases: Twitter16-shaped 128 trees with K = 5000 (bag-of-words), PHEME-shaped 24 and 4,096 trees with K = 768 (dense
tanh features).  --sparse instead alternates two library models with the same weights, one fed data.x dense and one
fed the same batch as a SparseX (CSR, what DeviceForest and forest_from_raw hand over): Twitter16- and Twitter15-shaped
128 trees at K = 5000.  --tiny runs every path once at a toy size (a rehearsal, not a measurement)."""
import argparse
import copy
import json
import os
import subprocess
import sys
from types import SimpleNamespace

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402
import bigcn_b200  # noqa: E402
import ebgcn_harness  # noqa: E402
from bigcn_b200.data import make_batch  # noqa: E402

LINES = []


def emit(**kw):
    line = json.dumps(kw)
    LINES.append(line)
    print(line, flush=True)


def step(m, bd):
    out, tdl, bul = m(bd)
    loss = F.nll_loss(out, bd.y)
    for el in (tdl, bul):
        if el is not None:
            loss = loss + 0.2 * el
    loss.backward()


def peak_above(m, bd):
    m.zero_grad(set_to_none=True)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    step(m, bd)
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() - base


def run_case(name, shape, n_trees, k, infer, steps, warmup, sparse=False):
    dev = torch.device("cuda:0")
    args = SimpleNamespace(input_features=k, hidden_features=64, output_features=64, edge_num=2, dropout=0.5,
                           num_class=4, edge_infer_td=infer, edge_infer_bu=infer, device=dev)
    torch.manual_seed(0)
    ref = (bigcn_b200.EBGCN if sparse else ebgcn_harness.EBGCN)(args).to(dev).train()
    new = bigcn_b200.EBGCN(args).to(dev).train()
    new.load_state_dict(ref.state_dict())
    bd = make_batch(shape, n_trees, seed=1, train=True, in_feats=k).to(dev)
    n = int(bd.x.shape[0])
    if sparse:
        sb = copy.copy(bd)
        sb.x = bigcn_b200.SparseX.from_torch_csr(bd.x.to_sparse_csr())
        models = {"sparse_x": (new, sb), "dense_x": (ref, bd)}
    else:
        models = {"library": (new, bd), "harness": (ref, bd)}
    for _ in range(warmup):
        for m, b in models.values():
            m.zero_grad(set_to_none=True)
            step(m, b)
    times = {key: [] for key in models}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for i in range(steps):
        order = list(models) if i % 2 == 0 else list(models)[::-1]
        for key in order:
            m, b = models[key]
            m.zero_grad(set_to_none=True)
            torch.cuda.synchronize()
            ev[0].record()
            step(m, b)
            ev[1].record()
            torch.cuda.synchronize()
            times[key].append(ev[0].elapsed_time(ev[1]))
    for key, t in times.items():
        t = sorted(t)
        emit(kind="step", case=name, edge_infer=infer, model=key, N=n, B=n_trees, K=k, E=int(bd.edge_index.shape[1]),
             ms_median=t[len(t) // 2], ms_min=t[0], ms_max=t[-1], steps=steps)
    if not infer:
        for key, (m, b) in models.items():
            p = peak_above(m, b)
            extra = {"x_csr_mib": b.x.nbytes() / 2**20} if key == "sparse_x" else {}
            emit(kind="mem", case=name, model=key, N=n, B=n_trees, K=k, peak_above_inputs_mib=p / 2**20,
                 x_fp32_mib=n * k * 4 / 2**20, ratio_to_x=p / (n * k * 4), **extra)
    del ref, new, models
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--tiny", action="store_true")
    ap.add_argument("--sparse", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    emit(kind="gpu", nvidia_smi=smi[0] if smi else None, torch_name=torch.cuda.get_device_name(0))
    if a.tiny:
        cases = [("tiny", "twitter15", 4, 40)] if a.sparse else [("tiny", "twitter15", 4, 40), ("tiny-dense", "pheme", 6, 96)]
        steps, warmup = 2, 1
    elif a.sparse:
        cases = [("twitter16-128-K5000", "twitter16", 128, 5000), ("twitter15-128-K5000", "twitter15", 128, 5000)]
        steps, warmup = a.steps, a.warmup
    else:
        cases = [("twitter16-128-K5000", "twitter16", 128, 5000), ("pheme-24-K768", "pheme", 24, 768),
                 ("pheme-4096-K768", "pheme", 4096, 768)]
        steps, warmup = a.steps, a.warmup
    for infer in (False, True):
        for name, shape, b, k in cases:
            run_case(name, shape, b, k, infer, steps, warmup, a.sparse)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(LINES) + "\n")


if __name__ == "__main__":
    main()
