#!/usr/bin/env python
"""bigcn_x_capture (the TMA-fed pass over x of bigcn_batch_prepare) against torch.to_sparse_csr, several shapes
(needs the GPU): the same entries per row, and -- between the two forms bigcn_debug_set key 10 selects, 9 being the
LDG scan whose slot order the product is defined by, 0 the TMA-fed pass -- the same slot order.
`python tools/capture_check.py 9 0`."""
import ctypes as C
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
from bigcn_b200 import _lib as L  # noqa: E402
from bigcn_b200.ops import _p, _stream, check  # noqa: E402


def capture_csr(lib, x):
    n, k = x.shape
    ws = torch.zeros(lib.bigcn_xsparse_workspace_bytes(n, k), dtype=torch.uint8, device=x.device)
    flags = torch.zeros(1, dtype=torch.int32, device=x.device)
    check(lib.bigcn_x_capture(_p(x), n, k, 1, _p(flags), _p(ws), ws.numel(), _stream()), "x_capture")
    ptrs = [C.c_void_p() for _ in range(7)]
    check(lib.bigcn_xsparse_view(n, k, _p(ws), ws.numel(), *[C.byref(p) for p in ptrs]), "view")
    base = ws.data_ptr()

    def arr(p, count, dtype):
        off = p.value - base
        return ws[off:off + count * 4].view(dtype)
    torch.cuda.synchronize()
    nnz = int(arr(ptrs[0], 4, torch.int32)[0].item())
    return arr(ptrs[1], n + 1, torch.int32), arr(ptrs[2], nnz, torch.int32), arr(ptrs[3], nnz, torch.float32), int(flags.item())


def main():
    dev = torch.device("cuda", 0)
    lib = L.lib()
    lib.bigcn_debug_set.argtypes = [C.c_int, C.c_int]
    lib.bigcn_debug_set.restype = None
    bad = 0
    first = {}
    for knob in [int(a) for a in sys.argv[1:]] or [9, 0]:
        lib.bigcn_debug_set(10, knob)
        g = torch.Generator(device="cpu").manual_seed(3)      # every variant sees the same matrices
        for n, k, per_row in ((1, 4, 2), (37, 24, 3), (300, 1000, 11), (2000, 5000, 20), (513, 5000, 1), (64, 4096, 20), (100, 1028, 5)):
            x = torch.zeros(n, k)
            for r in range(n):
                cols = torch.randperm(k, generator=g)[:min(k, int(torch.randint(0, 2 * per_row + 1, (1,), generator=g)))]
                x[r, cols] = torch.randint(1, 5, (len(cols),), generator=g).float()
            x[0, k - 1] = 7.0
            x[n - 1, 0] = -3.0
            want = x.to_sparse_csr()
            ptr, col, val, fl = capture_csr(lib, x.to(dev))
            ptr, col, val = ptr.cpu().long(), col.cpu().long(), val.cpu()
            ok = fl == 0 and torch.equal(ptr, want.crow_indices()) and len(col) == want.values().numel()
            if ok:      # rows hold the same (col, val) set; the order inside a row is the scan's, not ascending
                rowid = torch.repeat_interleave(torch.arange(n), ptr[1:] - ptr[:-1])
                order = torch.argsort(rowid * k + col, stable=True)
                ok = torch.equal(col[order], want.col_indices()) and torch.equal(val[order], want.values())
            same = first.setdefault((n, k), col)
            ok_order = torch.equal(same, col)
            print(f"knob {knob} N={n} K={k}: {'ok' if ok else 'MISMATCH'} (nnz {want.values().numel()}, flags {fl}); slot order "
                  f"{'as the first variant' if ok_order else 'DIFFERS from the first variant'}", flush=True)
            bad += (not ok) + (not ok_order)
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
