#!/usr/bin/env python
"""gemm_mode='bf16' against the fp32-x tensor-core modes, in one GPU call (prints JSON lines):

  kernel  X * W (both directions, n_out = 128) and dW1 = T^T X alone on a Twitter-sized dense matrix (31 k x 5000,
          bag-of-words counts) and on PHEME at 4096 trees (41 k x 768): tf32 / tf32x3 on fp32 x, bf16 on bf16 x (three
          weight terms).  Inputs rotate over enough copies to exceed the 126 MB L2.  ms per call
          (CUDA events), algorithmic bytes (x read once + y / dW written), fraction of the copy peak measured in the
          same call, tensor TFLOP/s of the MMAs issued, and the error against fp64.
  step    whole steps replayed from CUDA graphs (FusedTrainer with next_data for training), three rotating batches,
          the modes of a case alternated, three repeats: PHEME inference / training at 24 and 4096 trees ('auto' on
          fp32 x against bf16), Weibo training at 128 trees, and PHEME v1 width (in_feats = 196,608) at 24 trees.
  gpu     card name, power limit and max SM clock (nvidia-smi), read in the same call.
"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import bigcn_b200  # noqa: E402
from bigcn_b200 import _lib as L  # noqa: E402
from bigcn_b200.data import Batch, make_batch_shard  # noqa: E402

L2_BYTES = 126 << 20


def out(**kw):
    print(json.dumps(kw), flush=True)


def timed(fn, iters, warm=3):
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


def copy_peak(dev):
    a = torch.empty(1 << 30, dtype=torch.uint8, device=dev)
    b = torch.empty_like(a)
    ms = timed(lambda i: b.copy_(a), 20)
    return 2 * a.numel() / (ms * 1e-3)


def kernels(dev, peak):
    lib = L.lib()
    st = torch.cuda.current_stream().cuda_stream
    for name, n, k, dense in (("twitter_dense", 31000, 5000, False), ("pheme4096", 41000, 768, True)):
        g = torch.Generator(device=dev).manual_seed(0)
        if dense:
            x32 = torch.tanh(torch.randn(n, k, device=dev, generator=g))
        else:   # bag-of-words counts, ~14 non-zeros per row
            x32 = torch.zeros(n, k, device=dev)
            cols = torch.randint(0, k, (n, 14), device=dev, generator=g)
            x32.scatter_(1, cols, torch.randint(1, 4, (n, 14), device=dev, generator=g).float())
        x16 = x32.to(torch.bfloat16)
        w = [torch.randn(64, k, device=dev, generator=g) * 0.05 for _ in range(2)]
        t = torch.randn(n, 128, device=dev, generator=g)
        ref_y = (x16.double() @ torch.cat(w).double().t())
        ref_dw = t.double().t() @ x16.double()                              # [128, K]
        ref_y32 = (x32.double() @ torch.cat(w).double().t())
        ref_dw32 = t.double().t() @ x32.double()
        for mode, terms in (("tf32", 1), ("tf32x3", 3), ("bf16", 3)):
            xb = x16 if mode == "bf16" else x32
            copies = max(2, -(-2 * L2_BYTES // (xb.numel() * xb.element_size())))
            xs = [xb] + [xb.clone() for _ in range(copies - 1)]
            y = torch.empty(n, 128, device=dev)
            dw = [torch.empty(64, k, device=dev) for _ in range(2)]
            scr_x = torch.empty(lib.bigcn_xw_scratch_floats(k, 2), device=dev)
            nscr = lib.bigcn_xw_wgrad_scratch_floats(n, k, 2)
            scr_d = torch.empty(nscr, device=dev)
            m = L.GEMM_MODE[mode]

            def fwd(i):
                L.check(lib.bigcn_xw(xs[i % copies].data_ptr(), n, k, w[0].data_ptr(), w[1].data_ptr(), k, y.data_ptr(),
                                     128, m, scr_x.data_ptr(), st), "xw")

            def bwd(i):
                L.check(lib.bigcn_xw_wgrad(xs[i % copies].data_ptr(), n, k, t.data_ptr(), 2, dw[0].data_ptr(),
                                           dw[1].data_ptr(), k, m, scr_d.data_ptr(), st), "xw_wgrad")
            xbytes = xb.numel() * xb.element_size()
            for op, fn, ybytes, ref in (("xw", fwd, n * 128 * 4, ref_y if mode == "bf16" else ref_y32),
                                        ("dw1", bwd, n * 128 * 4 + k * 128 * 4, ref_dw if mode == "bf16" else ref_dw32)):
                ms = timed(fn, 20)
                got = y if op == "xw" else torch.cat(dw)
                err = float((got.double() - ref).abs().max() / ref.abs().max())
                by = xbytes + ybytes
                out(part="kernel", matrix=name, N=n, K=k, op=op, mode=mode, terms=terms, x_dtype=str(xb.dtype)[6:],
                    ms=round(ms, 4), alg_bytes=by, frac_copy_peak=round(by / (ms * 1e-3) / peak, 3),
                    tensor_tflops=round(2 * n * k * 128 * terms / (ms * 1e-3) / 1e12, 1), rel_err_fp64=float(f"{err:.3e}"),
                    x_copies_rotated=copies)
            del xs


def steps(dev):
    # PHEME's fp32 baseline is 'auto' (tf32x3 with dense_roots on, what a user gets for dense features; an explicit
    # 'tf32x3' leaves dense_roots off); bf16 turns dense_roots on by its own probe
    pheme = [("auto", "auto"), ("bf16x3", "bf16")]
    cases = [  # (shape, trees, in_feats, phases, [(label, gemm_mode)])
        ("pheme", 24, 768, ("infer", "train"), pheme),
        ("pheme", 4096, 768, ("infer", "train"), pheme),
        ("weibo", 128, 5000, ("train",), [("sparse", "sparse"), ("tf32", "tf32"), ("tf32x3", "tf32x3"), ("bf16x3", "bf16")]),
        ("pheme", 24, 196608, ("infer", "train"), pheme),
    ]
    for shape, trees, k, phases, modes in cases:
        torch.cuda.empty_cache()
        cfg = bigcn_b200.data.SHAPES[shape]
        cpu = [make_batch_shard(shape, trees, seed=3000 + i, train=True, in_feats=k)[0] for i in range(3)]
        b32 = [Batch(**{f: getattr(b, f).to(dev) for f in Batch._tensor_keys}) for b in cpu]
        for b in b32:
            b.x = b.x.to(torch.bfloat16).float()          # the same values in both forms
        b16 = []
        for b in b32:
            c = Batch(**{f: getattr(b, f) for f in Batch._tensor_keys})
            c.x = b.x.to(torch.bfloat16)
            b16.append(c)
        del cpu
        nodes = [int(b.x.shape[0]) for b in b32]
        for phase in phases:
            runners = {}
            for label, mode in modes:
                torch.manual_seed(0)
                m = bigcn_b200.BiGCN(k, 64, 64, dev, num_classes=cfg["num_classes"], gemm_mode=mode, validate="off",
                                     graphs=True).to(dev)
                m.train(phase == "train")
                tr = bigcn_b200.FusedTrainer(m) if phase == "train" else None
                data = b16 if mode == "bf16" else b32

                def one(i, m=m, tr=tr, data=data):
                    if tr is not None:
                        return tr.step(data[i % 3], next_data=data[(i + 1) % 3])
                    with torch.no_grad():
                        return m(data[i % 3])
                runners[label] = one
            res = {label: [] for label, _ in modes}
            for rep in range(3):
                for label, _ in modes:
                    res[label].append(timed(runners[label], 30, warm=24 if rep == 0 else 6))
            for label, mode in modes:
                v = sorted(res[label])
                out(part="step", shape=shape, trees=trees, K=k, phase=phase, mode=label, ms_runs=[round(a, 4) for a in res[label]],
                    ms_median=round(v[1], 4), spread=round(v[-1] - v[0], 4), nodes_per_batch=nodes,
                    x_bytes_per_batch=int(sum(nodes) / 3 * k * (2 if mode == "bf16" else 4)))
            del runners


def main():
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    peak = copy_peak(dev)
    out(part="gpu", nvidia_smi=smi, torch_name=torch.cuda.get_device_name(dev), copy_peak_gbs=round(peak / 1e9, 1))
    which = sys.argv[1:] or ["kernel", "step"]
    if "kernel" in which:
        kernels(dev, peak)
    if "step" in which:
        steps(dev)


if __name__ == "__main__":
    main()
