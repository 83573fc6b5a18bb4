#!/usr/bin/env python
"""The gradient w.r.t. data.x (k_dx_tc), in one GPU call (prints JSON lines):

  kernel  dX[N, K] = T[N, 128] [W_TD; W_BU] alone through bigcn_x_dgrad: Twitter-sized (31 k x 5000, fp32 out) and
          PHEME at 4096 trees (41 k x 768, fp32 and bf16 out).  T and dX rotate over enough copies to exceed the
          126 MB L2.  ms per call (CUDA events), algorithmic bytes (N K s + N 128 4 + 128 K 4: the three split kernels
          and the scratch traffic are not counted), fraction of the copy peak measured in the same call, tensor TFLOP/s
          of the MMAs issued (three per K step), the error against fp64 and whether two calls are bit-identical.
  step    the autograd training step of the module path (forward, nll_loss, backward), with and without
          data.x.requires_grad, alternated, three repeats: PHEME 24 / 4096 trees (K = 768, 'auto' = tf32x3) and Twitter
          128 trees (K = 5000, 'auto' = sparse on the dense x).
  csr     dval[nnz] = T[i] . W^T[col] at the stored entries of a CSR x (k_dx_csr, n_w = 2) through bigcn_x_dgrad_csr, on
          a 128-tree Twitter16-shaped and a 128-tree Weibo-shaped batch (K = 5000, data.synth_forest_device): T, ptr,
          col and dval cold (rotated over copies larger than L2) and warm (one copy, as in the step; W^T stays in L2
          either way).  ms per call (CUDA events, W's transpose included) and per k_dx_csr launch alone
          (torch.profiler, a run of its own), nnz, the L2 bytes the entries pull (nnz 4 NOUT of W^T rows), error
          against fp64, bit-identical rerun; beside it k_dx_tc (bigcn_x_dgrad) on the same batch made dense.
  csrstep the autograd training step of the module path on DeviceForest batches of those two shapes (SparseX x,
          gemm_mode 'sparse'), with and without val.requires_grad, alternated, three repeats.
  gpu     card name, power limit and max SM clock (nvidia-smi), read in the same call.
Default: kernel step; name the parts to run others (python tools/dxbench.py csr csrstep).
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
    for name, n, k, dtypes in (("twitter", 31000, 5000, (torch.float32,)),
                               ("pheme4096", 41000, 768, (torch.float32, torch.bfloat16))):
        g = torch.Generator(device=dev).manual_seed(0)
        w = [torch.randn(64, k, device=dev, generator=g) * 0.05 for _ in range(2)]
        t0 = torch.randn(n, 128, device=dev, generator=g)
        ref = t0.double() @ torch.cat(w).double()
        scr = torch.empty(lib.bigcn_x_dgrad_scratch_floats(n, k, 2), device=dev)
        for dt in dtypes:
            s = 2 if dt == torch.bfloat16 else 4
            copies = max(2, -(-2 * L2_BYTES // (n * k * s + n * 128 * 4)))
            ts = [t0] + [t0.clone() for _ in range(copies - 1)]
            dxs = [torch.empty(n, k, dtype=dt, device=dev) for _ in range(copies)]
            bf = dt == torch.bfloat16

            def fn(i):
                dx = dxs[i % copies]
                L.check(lib.bigcn_x_dgrad(ts[i % copies].data_ptr(), 2, w[0].data_ptr(), w[1].data_ptr(), k, n, k,
                                          None if bf else dx.data_ptr(), dx.data_ptr() if bf else None, scr.data_ptr(),
                                          st), "x_dgrad")
            ms = timed(fn, 30)
            fn(0)
            a = dxs[0].clone()
            fn(0)
            torch.cuda.synchronize()
            same = bool(torch.equal(a, dxs[0]))
            err = float((a.double() - ref).abs().max() / ref.abs().max())
            by = n * k * s + n * 128 * 4 + 128 * k * 4
            out(part="kernel", shape=name, N=n, K=k, out_dtype=str(dt)[6:], ms=round(ms, 4), alg_bytes=by,
                frac_copy_peak=round(by / (ms * 1e-3) / peak, 3),
                tensor_tflops=round(3 * 2 * n * k * 128 / (ms * 1e-3) / 1e12, 1), rel_err_fp64=float(f"{err:.3e}"),
                bit_identical_rerun=same, copies_rotated=copies)
            del ts, dxs


def steps(dev):
    for shape, trees, k in (("pheme", 24, 768), ("pheme", 4096, 768), ("twitter15", 128, 5000)):
        torch.cuda.empty_cache()
        cfg = bigcn_b200.data.SHAPES[shape]
        cpu = [make_batch_shard(shape, trees, seed=3000 + i, train=True, in_feats=k)[0] for i in range(3)]
        data = [Batch(**{f: getattr(b, f).to(dev) for f in Batch._tensor_keys}) for b in cpu]
        torch.manual_seed(0)
        m = bigcn_b200.BiGCN(k, 64, 64, dev, num_classes=cfg["num_classes"], gemm_mode="auto", validate="off").to(dev)
        m.train()

        def one(i, xg):
            d = data[i % 3]
            x = d.x.detach().requires_grad_(xg)
            b = Batch(**{f: getattr(d, f) for f in Batch._tensor_keys})
            b.x = x
            m.zero_grad(set_to_none=True)
            F.nll_loss(m(b), b.y).backward()
        res = {False: [], True: []}
        for rep in range(3):
            for xg in (False, True):
                res[xg].append(timed(lambda i: one(i, xg), 30, warm=10 if rep == 0 else 3))
        for xg in (False, True):
            v = sorted(res[xg])
            out(part="step", shape=shape, trees=trees, K=k, mode=m.TDrumorGCN.resolved_gemm_mode(data[0].x),
                x_requires_grad=xg, ms_runs=[round(a, 4) for a in res[xg]], ms_median=round(v[1], 4),
                spread=round(v[-1] - v[0], 4), nodes_per_batch=[int(d.x.shape[0]) for d in data])
        del m, data


def _sparse_batch(shape, dev, seed=0):
    """128 trees of `shape` from data.synth_forest_device as a DeviceForest batch: data.x is a SparseX"""
    f = bigcn_b200.data.synth_forest_device(shape, 128, dev, seed=seed)
    return bigcn_b200.DeviceForest.from_device_arrays(f).batch(list(range(128)))


def csr_kernels(dev, peak):
    lib = L.lib()
    st = torch.cuda.current_stream().cuda_stream
    k = 5000
    for shape in ("twitter16", "weibo"):
        xs = _sparse_batch(shape, dev).x
        n, nnz = xs.shape[0], xs.val.numel()
        g = torch.Generator(device=dev).manual_seed(1)
        w = [torch.randn(64, k, device=dev, generator=g) * 0.05 for _ in range(2)]
        t0 = torch.randn(n, 128, device=dev, generator=g)
        rows = torch.repeat_interleave(torch.arange(n, device=dev), (xs.ptr[1:] - xs.ptr[:-1]).long())
        ref = (t0.double()[rows] * torch.cat(w).double()[:, xs.col.long()].t()).sum(1)
        scr = torch.empty(lib.bigcn_x_dgrad_csr_scratch_floats(k, 2), device=dev)
        per_copy = n * 128 * 4 + (n + 1) * 4 + nnz * 8
        res = {}
        for temp, copies in (("cold", max(2, -(-2 * L2_BYTES // per_copy))), ("warm", 1)):
            sets = [(t0, xs.ptr, xs.col)] + [(t0.clone(), xs.ptr.clone(), xs.col.clone()) for _ in range(copies - 1)]
            dvs = [torch.empty(nnz, device=dev) for _ in range(copies)]

            def fn(i):
                t, ptr, col = sets[i % copies]
                L.check(lib.bigcn_x_dgrad_csr(ptr.data_ptr(), col.data_ptr(), n, k, nnz, t.data_ptr(), 2, w[0].data_ptr(),
                                              w[1].data_ptr(), k, dvs[i % copies].data_ptr(), scr.data_ptr(), st),
                        "x_dgrad_csr")
            ms = timed(fn, 200, warm=10)
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                for i in range(50):
                    fn(i)
                torch.cuda.synchronize()
            kern = {}
            for e in prof.key_averages():
                for key in ("k_dx_csr", "k_transpose_jobs"):
                    if key in e.key:
                        kern[key] = round(getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0)) / e.count / 1e3, 5)
            fn(0)
            a = dvs[0].clone()
            fn(0)
            torch.cuda.synchronize()
            res[temp] = dict(ms_call=round(ms, 5), ms_k_dx_csr=kern.get("k_dx_csr"),
                             ms_transpose=kern.get("k_transpose_jobs"), copies_rotated=copies,
                             bit_identical_rerun=bool(torch.equal(a, dvs[0])),
                             rel_err_fp64=float(f"{float((a.double() - ref).abs().max() / ref.abs().max()):.3e}"))
            del sets, dvs
        l2 = nnz * 4 * 128
        kd = res["warm"]["ms_k_dx_csr"]
        # the dense gradient of the same batch (k_dx_tc, fp32 out), T and dX one copy each (dX alone is > L2)
        dx = torch.empty(n, k, device=dev)
        dscr = torch.empty(lib.bigcn_x_dgrad_scratch_floats(n, k, 2), device=dev)
        ms_tc = timed(lambda i: L.check(lib.bigcn_x_dgrad(t0.data_ptr(), 2, w[0].data_ptr(), w[1].data_ptr(), k, n, k,
                                                          dx.data_ptr(), None, dscr.data_ptr(), st), "x_dgrad"), 20)
        out(part="csr", shape=shape, trees=128, N=n, K=k, nnz=nnz, l2_bytes_w_rows=l2,
            l2_tbs_warm=round(l2 / (kd * 1e-3) / 1e12, 2) if kd else None, cold=res["cold"], warm=res["warm"],
            k_dx_tc_dense_ms=round(ms_tc, 4), dense_dx_bytes=n * k * 4)
        del dx, dscr


def csr_steps(dev):
    from bigcn_b200.ops import SparseX
    for shape in ("twitter16", "weibo"):
        torch.cuda.empty_cache()
        cfg = bigcn_b200.data.SHAPES[shape]
        data = [_sparse_batch(shape, dev, seed=4000 + i) for i in range(3)]
        torch.manual_seed(0)
        m = bigcn_b200.BiGCN(5000, 64, 64, dev, num_classes=cfg["num_classes"], validate="off").to(dev)
        m.train()
        ys = [torch.randint(0, cfg["num_classes"], (128,), device=dev) for _ in range(3)]

        def one(i, vg):
            d = data[i % 3]
            b = Batch(**{f: getattr(d, f) for f in Batch._tensor_keys})
            b.x = SparseX(d.x.ptr, d.x.col, d.x.val.detach().requires_grad_(vg), d.x.shape)
            m.zero_grad(set_to_none=True)
            F.nll_loss(m(b), ys[i % 3]).backward()
        res = {False: [], True: []}
        for rep in range(3):
            for vg in (False, True):
                res[vg].append(timed(lambda i: one(i, vg), 30, warm=10 if rep == 0 else 3))
        for vg in (False, True):
            v = sorted(res[vg])
            out(part="csrstep", shape=shape, trees=128, K=5000, mode=m.TDrumorGCN.resolved_gemm_mode(data[0].x),
                val_requires_grad=vg, ms_runs=[round(a, 4) for a in res[vg]], ms_median=round(v[1], 4),
                spread=round(v[-1] - v[0], 4), nodes_per_batch=[int(d.x.shape[0]) for d in data],
                nnz_per_batch=[int(d.x.val.numel()) for d in data])
        del m, data


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
    if "csr" in which:
        csr_kernels(dev, peak)
    if "csrstep" in which:
        csr_steps(dev)


if __name__ == "__main__":
    main()
