"""Host-side wrappers over the C-ABI: torch supplies device memory, streams and
autograd plumbing; every arithmetic step runs in libbigcn_b200.so."""
from __future__ import annotations

import ctypes as C
import operator
import weakref
from types import SimpleNamespace

import torch

from . import _lib as L
from ._lib import H, Dims, BatchPtrs, Params, Graph, Opts, check, lib


def _stream():
    # the raw handle of torch's current stream on the current device (what torch.cuda.current_stream().cuda_stream
    # returns, without building a Stream object: this runs on every library call)
    return torch._C._cuda_getCurrentRawStream(torch._C._cuda_getDevice())


def _p(t):
    return None if t is None else t.data_ptr()


_capture_streams = {}
_step_streams = {}


def _priority_stream(table, dev):
    """``table``'s stream on device ``dev``, two priority levels above the default one (levels: csrc/api.cu)"""
    s = table.get(dev)
    if s is None:
        try:
            lo, hi = torch.cuda.Stream.priority_range()
        except Exception:  # noqa: BLE001
            lo, hi = 0, -1
        s = table[dev] = torch.cuda.Stream(device=dev, priority=max(hi, lo - 2) if hi < lo else lo)
    return s


def step_stream(device=None):
    """A stream two priority levels above the default one, per device: FusedTrainer runs (and captures) its steps
    on it so that bigcn_batch_prepare's lowest-priority streams -- the next batch's preparation -- really yield
    to the step's own kernels (the caller's default stream already has the lowest priority there is)."""
    return _priority_stream(_step_streams, torch.cuda.current_device() if device is None else torch.device(device).index)


def capture_graph(enqueue):
    """Stream-capture ``enqueue()`` (C-ABI launches only: nothing allocates, nothing synchronises) into a
    torch.cuda.CUDAGraph on a side stream.  The bare capture_begin / capture_end pair instead of the
    ``torch.cuda.graph`` context manager: no device synchronise, gc.collect or empty_cache per capture, so a
    capture costs about one enqueue plus the instantiation."""
    # kernel nodes inherit the capturing stream's priority: the step stream's level
    s = _priority_stream(_capture_streams, torch.cuda.current_device())
    cur = torch.cuda.current_stream()
    s.wait_stream(cur)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        g.capture_begin(capture_error_mode="thread_local")
        try:
            enqueue()
        finally:
            g.capture_end()
    cur.wait_stream(s)
    return g


class GraphCache:
    """CUDA graphs by batch key: a batch object's first sighting is enqueued (which also warms the library's lazy
    state), its second is captured, later ones replay.  Keeps at most ``max_graphs`` captures (the oldest goes first)
    and ``max_seen`` first sightings; ``clear()`` drops the captures only."""

    def __init__(self, max_graphs, max_seen, capture=capture_graph):
        self.max_graphs, self.max_seen, self._capture = int(max_graphs), int(max_seen), capture
        self._entries, self._seen = {}, {}     # key -> (graph, plan, pins, batch); key -> weakref to the batch
        self.captures = self.replays = 0

    def __len__(self):
        return len(self._entries)

    def clear(self):
        self._entries.clear()

    def replay(self, key, pins=()):
        """Replay ``key``'s capture and return its plan if ``pins`` are the objects they were at capture, else None"""
        e = self._entries.get(key)
        if e is None or len(e[2]) != len(pins) or not all(map(operator.is_, e[2], pins)):
            return None
        e[0].replay()
        self.replays += 1
        return e[1]

    def first_sighting(self, key, data):
        """True (and remembered, weakly) the first time ``data`` comes under ``key``"""
        ref = self._seen.get(key)
        if ref is not None and ref() is data:
            return False
        if len(self._seen) >= self.max_seen:
            self._seen.clear()
        self._seen[key] = weakref.ref(data)
        return True

    def capture(self, key, enqueue, plan, pins=(), data=None):
        """Capture ``enqueue()`` as the graph of ``key`` and replay it.  The entry keeps ``plan`` (what the launches
        point at) and ``data``: the strong reference pins id(data)."""
        g = self._capture(enqueue)
        while len(self._entries) >= self.max_graphs:
            self._entries.pop(next(iter(self._entries)))
        self._entries[key] = (g, plan, tuple(pins), data)
        self.captures += 1
        self.replay(key, pins)


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise L.BigcnError("bigcn_b200 ops take CUDA tensors only (no CPU fallback)")


def _i64(t):
    if t.dtype != torch.int64:
        t = t.to(torch.int64)
    return t.contiguous()


def _f32(t):
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


# ----------------------------------------------------------------------------- sparse data.x
class SparseX:
    """``data.x`` as CSR (int32 ``ptr [N+1]``, int32 ``col``, fp32 ``val``): what the
    ``gemm_mode='sparse'`` path consumes when the dense [N, K] matrix is never shipped to the
    device (a loader that keeps the reference's ``index:count`` pairs,
    Process/getTwittergraph.py:16-24, or :func:`host_dense_to_csr` on a dense host matrix).
    Quacks enough like a tensor for ``forward(data)``: ``shape``, ``device``, ``to``."""

    def __init__(self, ptr, col, val, shape):
        self.ptr, self.col, self.val = ptr, col, val
        self.shape = (int(shape[0]), int(shape[1]))

    @property
    def device(self):
        return self.val.device

    @property
    def is_cuda(self):
        return self.val.is_cuda

    def to(self, device, non_blocking=False):
        return SparseX(self.ptr.to(device, non_blocking=non_blocking), self.col.to(device, non_blocking=non_blocking),
                       self.val.to(device, non_blocking=non_blocking), self.shape)

    def pin_memory(self):
        return SparseX(self.ptr.pin_memory(), self.col.pin_memory(), self.val.pin_memory(), self.shape)

    def nbytes(self):
        return sum(t.numel() * t.element_size() for t in (self.ptr, self.col, self.val))

    @staticmethod
    def from_torch_csr(t):
        t = t.coalesce() if t.layout == torch.sparse_coo else t
        if t.layout != torch.sparse_csr:
            t = t.to_sparse_csr()
        return SparseX(t.crow_indices().to(torch.int32), t.col_indices().to(torch.int32),
                       t.values().to(torch.float32), t.shape)

    def to_dense(self):
        n, k = self.shape
        rows = torch.repeat_interleave(torch.arange(n, device=self.ptr.device),
                                       (self.ptr[1:] - self.ptr[:-1]).long())
        out = torch.zeros(n, k, dtype=torch.float32, device=self.val.device)
        out[rows, self.col.long()] = self.val
        return out


def host_dense_to_csr(x, n_threads=0, out=None, cap=None):
    """One threaded pass over a dense HOST matrix -> :class:`SparseX` in (pinned) host memory
    (bigcn_host_dense_to_csr, csrc/host_compact.cpp: data movement only).  ``out`` may be a
    SparseX whose buffers are reused when large enough."""
    if x.is_cuda or x.dtype != torch.float32 or not x.is_contiguous():
        raise L.BigcnError("host_dense_to_csr: expects a contiguous fp32 CPU tensor")
    n, k = x.shape
    cap = int(cap if cap is not None else n * min(k, 48))
    if out is not None and out.ptr.numel() >= n + 1 and out.col.numel() >= cap:
        ptr, col, val = out.ptr, out.col, out.val
    else:
        pin = torch.cuda.is_available()
        ptr = torch.empty(n + 1, dtype=torch.int32, pin_memory=pin)
        col = torch.empty(cap, dtype=torch.int32, pin_memory=pin)
        val = torch.empty(cap, dtype=torch.float32, pin_memory=pin)
    nnz = lib().bigcn_host_dense_to_csr(x.data_ptr(), n, k, ptr.data_ptr(), col.data_ptr(), val.data_ptr(),
                                        col.numel(), int(n_threads))
    if nnz < 0:
        raise L.BigcnError(f"host_dense_to_csr: {-nnz} non-zeros do not fit the sparse layout (capacity {col.numel()}): "
                           "the features are not row-sparse, ship them dense")
    return SparseX(ptr[:n + 1], col[:nnz], val[:nnz], (n, k))


def sparse_x(xs, who):
    """A :class:`SparseX` checked for the CSR ops (GCNConv on a SparseX, EBGCN): on a CUDA device, int32 ``ptr [N+1]``,
    int32 ``col`` and fp32 ``val`` of one length, shape (N, K); returned with contiguous buffers.  These ops form no
    gradient for x, so a ``val`` that requires grad raises."""
    n, k = xs.shape
    _need_cuda(xs.ptr, xs.col, xs.val)
    if not xs.ptr.device == xs.col.device == xs.val.device:
        raise L.BigcnError(f"{who}: a SparseX's ptr, col and val must be on one device, got {xs.ptr.device}, "
                           f"{xs.col.device}, {xs.val.device}")
    if xs.ptr.dtype != torch.int32 or xs.col.dtype != torch.int32 or xs.val.dtype != torch.float32:
        raise L.BigcnError(f"{who}: a SparseX needs int32 ptr, int32 col and fp32 val, got {xs.ptr.dtype}, "
                           f"{xs.col.dtype}, {xs.val.dtype}")
    if n < 0 or k < 1 or tuple(xs.ptr.shape) != (n + 1,) or xs.col.dim() != 1 or xs.col.shape != xs.val.shape:
        raise L.BigcnError(f"{who}: a SparseX of shape {xs.shape} needs ptr [{n + 1}] and col / val of one length, got "
                           f"ptr {tuple(xs.ptr.shape)}, col {tuple(xs.col.shape)}, val {tuple(xs.val.shape)}")
    if xs.val.requires_grad:
        raise L.BigcnError(f"{who} forms no gradient w.r.t. data.x: pass SparseX(ptr, col, val.detach(), shape) (a "
                           "SparseX whose val requires grad is not supported)")
    return SparseX(xs.ptr.contiguous(), xs.col.contiguous(), xs.val.contiguous(), xs.shape)


def check_bf16_width(k):
    """bf16 features reach the tensor cores through TMA, which needs 16-byte rows"""
    if k % 8:
        raise L.BigcnError(f"gemm_mode='bf16': in_feats must be a multiple of 8 (16-byte rows for TMA), got "
                           f"{k}: pad the features with zero columns (and the weights to match)")


def bf16_x(x):
    """data.x for ``gemm_mode='bf16'``: a dense, contiguous CUDA bfloat16 matrix whose rows the TMA can address,
    passed through as it is.  Anything else raises (never a silent cast)."""
    if not isinstance(x, torch.Tensor) or x.layout != torch.strided:
        raise L.BigcnError("gemm_mode='bf16' needs a dense torch.bfloat16 data.x; a sparse x takes gemm_mode='sparse'")
    if x.dtype != torch.bfloat16:
        raise L.BigcnError(f"gemm_mode='bf16' needs data.x in torch.bfloat16, got {x.dtype}: convert the features once "
                           "with x.to(torch.bfloat16), or keep fp32 features with gemm_mode='tf32x3'")
    _need_cuda(x)
    if x.dim() != 2:
        raise L.BigcnError(f"gemm_mode='bf16': data.x must be [N, in_feats], got shape {tuple(x.shape)}")
    if not x.is_contiguous():
        raise L.BigcnError("gemm_mode='bf16': data.x must be contiguous (row pitch = in_feats): pass x.contiguous()")
    check_bf16_width(x.shape[1])
    if x.data_ptr() % 16:
        raise L.BigcnError("gemm_mode='bf16': data.x must start on a 16-byte boundary: pass x.clone()")
    return x


def _as_x(x, gemm_mode=None):
    """dense fp32 tensor | SparseX | torch sparse tensor -> (dense or None, SparseX or None); with
    ``gemm_mode='bf16'`` the dense bf16 x as it is (bf16_x)"""
    if gemm_mode == "bf16":
        return bf16_x(x), None
    if isinstance(x, SparseX):
        return None, x
    if isinstance(x, torch.Tensor) and x.layout != torch.strided:
        return None, SparseX.from_torch_csr(x)
    return _f32(x), None


def _x_for(x, gemm_mode):
    """a dense x for one of the ops below: bf16 as it is in ``gemm_mode='bf16'``, fp32 otherwise"""
    return bf16_x(x) if gemm_mode == "bf16" else _f32(x)


def pick_gemm_mode(x, sample_rows=4096):
    """``gemm_mode='auto'``: which conv1 product suits this feature matrix.  Counts the non-zeros of (up to)
    the first ``sample_rows`` rows on the device (bigcn_dense_row_counts) and reads the counts back ONCE per
    model: row-sparse bag-of-words features (Twitter / Weibo: ~14 of 5000 columns) take 'sparse' (exact fp32
    scan that also captures the non-zeros, X read once per step); dense features (PHEME's 768-d BERT
    embeddings) take 'tf32x3' (tcgen05 kind::tf32 with the hi/lo weight split, fp32-class accuracy)."""
    L.require_device()
    x = _f32(x)
    _need_cuda(x)
    n, k = x.shape
    m = min(int(n), int(sample_rows))
    if m == 0:
        return "sparse"
    tma_ok = k % 4 == 0 and x.data_ptr() % 16 == 0       # TMA needs 16 B aligned rows; otherwise the exact FFMA scan
    cnt = torch.empty(m, dtype=torch.int32, device=x.device)
    check(lib().bigcn_dense_row_counts(_p(x), m, k, _p(cnt), _stream()), "dense_row_counts")
    if _rows_look_sparse(cnt, k):
        return "sparse"
    return "tf32x3" if tma_ok else "fp32"


def _rows_look_sparse(cnt, k):
    """the row-density threshold of pick_gemm_mode over per-row non-zero counts (one device -> host read)"""
    c = cnt.cpu().numpy()
    cap = min(int(k), 48)
    return float(c.mean()) <= cap / 2 and int(c.max()) <= 4 * cap


def bf16_features_dense(x, sample_rows=4096):
    """``gemm_mode='bf16'``: whether a bf16 feature matrix has dense rows (PHEME's embeddings) rather than
    bag-of-words rows -- the same probe and threshold as pick_gemm_mode, counted on the bf16 values
    (bigcn_dense_row_counts_bf16).  Decides ``dense_roots='auto'`` in that mode."""
    L.require_device()
    x = bf16_x(x)
    n, k = x.shape
    m = min(int(n), int(sample_rows))
    if m == 0:
        return False
    cnt = torch.empty(m, dtype=torch.int32, device=x.device)
    check(lib().bigcn_dense_row_counts_bf16(_p(x), m, k, _p(cnt), _stream()), "dense_row_counts_bf16")
    return not _rows_look_sparse(cnt, k)


# ----------------------------------------------------------------------------- graph prep
def graph_prep(edge_indexes, num_nodes, batch=None, num_graphs=0, deg_by="target", rowsum=True, long_rows=True):
    """gcn_norm structure for 1 or 2 edge lists.  Returns (graphs, node_ptr, flags) where each
    graph is a dict of device tensors (see include/bigcn_b200.h: bigcn_graph_t).
    ``long_rows=False`` leaves the hub-row lists out: propagate then walks every row
    sequentially (exact COO' order even for rows with more than 32 in-edges)."""
    L.require_device()
    eis = [_i64(e) for e in edge_indexes]
    _need_cuda(*eis)
    dev = eis[0].device
    n = int(num_nodes)
    nd = len(eis)
    graphs, structs = [], (Graph * nd)()
    for d, ei in enumerate(eis):
        e = int(ei.shape[1])
        g = dict(in_ptr=torch.empty(n + 1, dtype=torch.int32, device=dev),
                 in_idx=torch.empty(max(e, 1), dtype=torch.int32, device=dev),
                 out_ptr=torch.empty(n + 1, dtype=torch.int32, device=dev),
                 out_idx=torch.empty(max(e, 1), dtype=torch.int32, device=dev),
                 deg=torch.empty(max(n, 1), dtype=torch.int32, device=dev),
                 dis=torch.empty(max(n, 1), dtype=torch.float32, device=dev),
                 rowsum=torch.empty(max(n, 1), dtype=torch.float32, device=dev) if rowsum else None)
        nl = lib().bigcn_long_ws_ints(e)
        g["in_long"] = torch.empty(nl, dtype=torch.int32, device=dev) if long_rows else None
        g["out_long"] = torch.empty(nl, dtype=torch.int32, device=dev) if long_rows else None
        for k, v in g.items():
            setattr(structs[d], k, _p(v))
        g["E"] = e
        graphs.append(g)
    node_ptr = None
    if batch is not None:
        batch = _i64(batch)
        node_ptr = torch.empty(int(num_graphs) + 1, dtype=torch.int32, device=dev)
    flags = torch.zeros(1, dtype=torch.int32, device=dev)
    emax = max(int(e.shape[1]) for e in eis)
    ws_bytes = lib().bigcn_graph_prep_workspace_bytes(n, emax, nd)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    ei_ptrs = (C.c_void_p * nd)(*[e.data_ptr() for e in eis])
    e_arr = (C.c_int64 * nd)(*[int(e.shape[1]) for e in eis])
    check(lib().bigcn_graph_prep(nd, ei_ptrs, e_arr, n, _p(batch), int(num_graphs), L.DEG_BY[deg_by],
                                 structs, _p(node_ptr), _p(flags), _p(ws), ws_bytes, _stream()),
          "graph_prep")
    for g in graphs:
        g["_keep"] = (ws,)
    return graphs, node_ptr, flags


def transpose_weight(w, k0, k, wt, col0):
    check(lib().bigcn_transpose_weight(_p(w), w.stride(0), k0, k, _p(wt), wt.stride(0), col0, _stream()),
          "transpose_weight")


def xw(x, weights, gemm_mode="fp32"):
    """y[N, 64*len(weights)] = x @ cat(weights).T with one pass over x (weights: [64,K] each).  ``gemm_mode='bf16'``
    takes a bf16 x as it is; y is fp32 in every mode."""
    L.require_device()
    x = _x_for(x, gemm_mode)
    _need_cuda(x, *weights)
    n, k = x.shape
    n_out = H * len(weights)
    ws = [_f32(w) for w in weights]
    if len(ws) == 2 and ws[0].stride(0) != ws[1].stride(0):
        raise L.BigcnError("xw: the two weight matrices must share a row pitch")
    nscr = lib().bigcn_xw_scratch_floats(k, len(ws))
    scr = torch.empty(nscr, dtype=torch.float32, device=x.device)
    y = torch.empty(n, n_out, dtype=torch.float32, device=x.device)
    check(lib().bigcn_xw(_p(x), n, k, _p(ws[0]), _p(ws[1]) if len(ws) == 2 else None, ws[0].stride(0), _p(y),
                         n_out, L.GEMM_MODE[gemm_mode], _p(scr), _stream()), "xw")
    return y


def x_dgrad(t, weights, out_dtype=torch.float32):
    """dx[N,K] = t @ cat(weights) with t [N, 64*len(weights)] and weights [64,K] each: the input gradient of ``xw``
    (tcgen05 kind::tf32, 3xTF32: fp32-class).  ``out_dtype`` float32, or bfloat16 (rounded once to nearest even)."""
    L.require_device()
    t = _f32(t)
    ws = [_f32(w) for w in weights]
    _need_cuda(t, *ws)
    n, k = t.shape[0], ws[0].shape[1]
    if t.shape[1] != H * len(ws) or any(w.shape != (H, k) for w in ws):
        raise L.BigcnError(f"x_dgrad: t must be [N,{H * len(ws)}] and every weight [64,{k}]")
    if len(ws) == 2 and ws[0].stride(0) != ws[1].stride(0):
        raise L.BigcnError("x_dgrad: the two weight matrices must share a row pitch")
    if out_dtype not in (torch.float32, torch.bfloat16):
        raise L.BigcnError(f"x_dgrad: out_dtype must be float32 or bfloat16, got {out_dtype}")
    dx = torch.empty(n, k, dtype=out_dtype, device=t.device)
    scr = torch.empty(lib().bigcn_x_dgrad_scratch_floats(n, k, len(ws)), dtype=torch.float32, device=t.device)
    bf = out_dtype == torch.bfloat16
    check(lib().bigcn_x_dgrad(_p(t), len(ws), _p(ws[0]), _p(ws[1]) if len(ws) == 2 else None, ws[0].stride(0), n, k,
                              None if bf else _p(dx), _p(dx) if bf else None, _p(scr), _stream()), "x_dgrad")
    return dx


def x_dgrad_csr(xs, t, weights):
    """dval[e] = t[i] . cat(weights)[:, col[e]] for every stored entry e = (i, col[e]) of the SparseX ``xs``: the input
    gradient of ``xs @ cat(weights).T`` sampled at x's pattern (the gradient of ``xs.val``; plain fp32 FMAs,
    deterministic).  t [N, 64*len(weights)], weights [64,K] each.  Returns fp32 [xs.val.numel()]: an entry whose column
    is outside [0, K), and every entry past ptr[N], gets 0."""
    L.require_device()
    t = _f32(t)
    ws = [_f32(w) for w in weights]
    _need_cuda(t, xs.ptr, xs.col, *ws)
    n, k = xs.shape
    if t.shape != (n, H * len(ws)) or any(w.shape != (H, k) for w in ws):
        raise L.BigcnError(f"x_dgrad_csr: t must be [{n},{H * len(ws)}] and every weight [64,{k}]")
    if len(ws) == 2 and ws[0].stride(0) != ws[1].stride(0):
        raise L.BigcnError("x_dgrad_csr: the two weight matrices must share a row pitch")
    if xs.ptr.dtype != torch.int32 or xs.col.dtype != torch.int32 or xs.ptr.numel() != n + 1:
        raise L.BigcnError("x_dgrad_csr: ptr must be int32 [N+1] and col int32")
    nnz = xs.val.numel()
    if xs.col.numel() < nnz:
        raise L.BigcnError(f"x_dgrad_csr: col holds {xs.col.numel()} entries, val {nnz}")
    dval = torch.empty(nnz, dtype=torch.float32, device=t.device)
    scr = torch.empty(lib().bigcn_x_dgrad_csr_scratch_floats(k, len(ws)), dtype=torch.float32, device=t.device)
    check(lib().bigcn_x_dgrad_csr(_p(xs.ptr.contiguous()), _p(xs.col.contiguous()), n, k, nnz, _p(t), len(ws),
                                  _p(ws[0]), _p(ws[1]) if len(ws) == 2 else None, ws[0].stride(0), _p(dval), _p(scr),
                                  _stream()), "x_dgrad_csr")
    return dval


class XSparseProduct:
    """y = x @ cat(weights).T through the exact scan that also captures the non-zeros of x
    (``gemm_mode='sparse'`` on its own).  ``wgrad(t)`` returns the weight gradients from the
    column-sorted copy; ``csr()`` / ``csc()`` expose the structures built on the device."""

    def __init__(self, x, weights):
        L.require_device()
        x = _f32(x)
        ws_ = [_f32(w) for w in weights]
        _need_cuda(x, *ws_)
        self.n, self.k, self.n_w = x.shape[0], x.shape[1], len(ws_)
        self.ws = torch.empty(lib().bigcn_xsparse_workspace_bytes(self.n, self.k), dtype=torch.uint8, device=x.device)
        self.flags = torch.zeros(1, dtype=torch.int32, device=x.device)
        self.y = torch.empty(self.n, H * self.n_w, dtype=torch.float32, device=x.device)
        check(lib().bigcn_xw_sparse(_p(x), self.n, self.k, _p(ws_[0]), _p(ws_[1]) if self.n_w == 2 else None,
                                    ws_[0].stride(0), _p(self.y), H * self.n_w, 1, _p(self.flags), _p(self.ws),
                                    self.ws.numel(), _stream()), "xw_sparse")

    def wgrad(self, t):
        t = _f32(t)
        dev = t.device
        dws = [torch.empty(H, self.k, dtype=torch.float32, device=dev) for _ in range(self.n_w)]
        check(lib().bigcn_xw_wgrad_sparse(self.n, self.k, _p(t), self.n_w, _p(dws[0]),
                                          _p(dws[1]) if self.n_w == 2 else None, self.k, _p(self.ws),
                                          self.ws.numel(), _stream()), "xw_wgrad_sparse")
        return dws

    def _view(self):
        ptrs = [C.c_void_p() for _ in range(7)]
        check(lib().bigcn_xsparse_view(self.n, self.k, _p(self.ws), self.ws.numel(), *[C.byref(p) for p in ptrs]),
              "xsparse_view")
        base = self.ws.data_ptr()

        def arr(p, count, dtype):
            off = p.value - base
            return self.ws[off:off + count * 4].view(dtype)
        state = arr(ptrs[0], 4, torch.int32)
        nnz = int(state[0].item())
        return dict(state=state, nnz=nnz, ptr=arr(ptrs[1], self.n + 1, torch.int32), col=arr(ptrs[2], nnz, torch.int32),
                    val=arr(ptrs[3], nnz, torch.float32), cptr=arr(ptrs[4], self.k + 1, torch.int32),
                    crow=arr(ptrs[5], nnz, torch.int32), cval=arr(ptrs[6], nnz, torch.float32))

    def csr(self):
        v = self._view()
        return v["ptr"], v["col"], v["val"]

    def csc(self):
        v = self._view()
        return v["cptr"], v["crow"], v["cval"]


def propagate(graph, h, bias=None, relu=False, transpose=False):
    """out = A-hat h (+bias)(relu), or A-hat^T h with transpose=True."""
    L.require_device()
    h = _f32(h)
    n = h.shape[0]
    out = torch.empty(n, H, dtype=torch.float32, device=h.device)
    ptr, idx, lng = (graph["out_ptr"], graph["out_idx"], graph.get("out_long")) if transpose else \
        (graph["in_ptr"], graph["in_idx"], graph.get("in_long"))
    check(lib().bigcn_propagate(_p(ptr), _p(idx), _p(graph["dis"]), n, graph["E"], _p(lng), _p(h), h.stride(0),
                                _p(bias), int(relu), _p(out), H, _stream()), "propagate")
    return out


def readout(h2, h1, node_ptr, rootindex, want_pos=False):
    """[mean over each tree of h2 | h1[rootindex]] -> [B,128] (scatter_mean + second root-extend)."""
    L.require_device()
    h2, h1 = _f32(h2), _f32(h1)
    rootindex = _i64(rootindex)
    n, b = h2.shape[0], int(rootindex.numel())
    feat = torch.empty(b, 2 * H, dtype=torch.float32, device=h2.device)
    pos = torch.empty(b, H, dtype=torch.float32, device=h2.device) if want_pos else None
    scr = torch.empty(lib().bigcn_readout_scratch_floats(n, b), dtype=torch.float32, device=h2.device)
    flags = torch.zeros(1, dtype=torch.int32, device=h2.device)
    check(lib().bigcn_readout(_p(h2), _p(h1), _p(node_ptr), _p(rootindex), n, b, _p(feat), 2 * H, _p(pos), _p(scr),
                              _p(flags), _stream()), "readout")
    return (feat, pos) if want_pos else feat


def dropout_mask(seed, stream_id, node_id_base, n, n_cols, p, device):
    L.require_device()
    keep = torch.empty(n, n_cols, dtype=torch.uint8, device=device)
    check(lib().bigcn_dropout_mask(seed, stream_id, node_id_base, n, n_cols, p, _p(keep), _stream()),
          "dropout_mask")
    return keep


def raise_on_flags(flags: torch.Tensor):
    """Host read of the device-side violation word (synchronises the stream)."""
    v = int(flags.item())
    if v == 0:
        return
    msgs = []
    if v & L.FLAG_EDGE_RANGE:
        msgs.append("an edge endpoint is outside [0, N)")
    if v & L.FLAG_BATCH_ORDER:
        msgs.append("data.batch is not sorted ascending within [0, B)")
    if v & L.FLAG_ROOT_RANGE:
        msgs.append("data.rootindex has an entry outside [0, N)")
    if v & L.FLAG_EDGE_WEIGHT:
        msgs.append("an edge weight is not finite, or a node's weighted degree is negative")
    if v & L.FLAG_X_CSR_RANGE:
        msgs.append("sparse data.x has a column index outside [0, in_feats)")
    if v & L.FLAG_X_NOT_SPARSE:
        msgs.append("gemm_mode='sparse' needs at most N*min(K,48) non-zeros in data.x (the conv1 weight "
                    "gradient of this batch is NaN): use 'tf32x3' / 'fp32' for dense features; a SparseX data.x "
                    "that dense (EBGCN, GCNConv) is better passed dense (x.to_dense())")
    raise IndexError("bigcn_b200: invalid graph input: " + "; ".join(msgs))


# ----------------------------------------------------------------------------- GCNConv
class GCNConvFunction(torch.autograd.Function):
    """conv(x, edge_index) -> [N,64]; gradients for weight and bias (x is treated as data)."""

    @staticmethod
    def forward(ctx, x, edge_index, weight, bias, deg_by, gemm_mode):
        L.require_device()
        x, weight, bias = _x_for(x, gemm_mode), _f32(weight), _f32(bias)
        ei = _i64(edge_index)
        _need_cuda(x, ei, weight, bias)
        n, k = x.shape
        e = int(ei.shape[1])
        if weight.shape != (H, k):
            raise L.BigcnError(f"GCNConv: out_channels must be {H} and weight [64,{k}], got {tuple(weight.shape)}")
        ws_bytes = lib().bigcn_gcnconv_workspace_bytes(n, e, k)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device)
        flags = torch.zeros(1, dtype=torch.int32, device=x.device)
        out = torch.empty(n, H, dtype=torch.float32, device=x.device)
        check(lib().bigcn_gcnconv_forward(_p(x), n, k, _p(ei), e, _p(weight), _p(bias), L.DEG_BY[deg_by],
                                          L.GEMM_MODE[gemm_mode], _p(out), _p(flags), _p(ws), ws_bytes,
                                          _stream()), "gcnconv_forward")
        ctx.save_for_backward(x, ws)
        ctx.dims = (n, k, e)
        ctx.flags = flags
        ctx.gemm_mode = gemm_mode
        return out

    @staticmethod
    def backward(ctx, grad_out):
        x, ws = ctx.saved_tensors
        n, k, e = ctx.dims
        g = _f32(grad_out)
        dw = torch.empty(H, k, dtype=torch.float32, device=x.device)
        db = torch.empty(H, dtype=torch.float32, device=x.device)
        check(lib().bigcn_gcnconv_backward(_p(x), n, k, e, _p(g), _p(dw), _p(db), L.GEMM_MODE[ctx.gemm_mode],
                                           _p(ws), ws.numel(), _stream()), "gcnconv_backward")
        return None, None, dw, db, None, None


def _csr_scratch(n, k, device):
    # dropped when the call returns: the caching allocator hands it out again only behind this stream's queued work
    return torch.empty(lib().bigcn_gcnconv_csr_scratch_bytes(n, k), dtype=torch.uint8, device=device)


class GCNConvCSRFunction(torch.autograd.Function):
    """conv(x, edge_index) -> [N,64] for a SparseX x (bigcn_gcnconv_csr_*, given as its ``val``, ``ptr``, ``col`` and
    ``shape``): the CSR product forward, dW as a sweep over x's columns; gradients for weight and bias.  ``flags``
    receives an out-of-range column and a batch past the sparse capacity (its dW is then NaN).  Only the structure,
    W^T and X W^T are kept for the backward; each call allocates the per-non-zero scratch it needs and drops it."""

    @staticmethod
    def forward(ctx, val, ptr, col, shape, edge_index, weight, bias, deg_by, flags):
        L.require_device()
        weight, bias = _f32(weight), _f32(bias)
        ei = _i64(edge_index)
        _need_cuda(val, ei, weight, bias)
        if weight.device != val.device:
            raise L.BigcnError(f"GCNConv: the SparseX x is on {val.device}, the conv's weight on {weight.device}")
        n, k = shape
        e = int(ei.shape[1])
        if weight.shape != (H, k):
            raise L.BigcnError(f"GCNConv: out_channels must be {H} and weight [64,{k}], got {tuple(weight.shape)}")
        ws_bytes = lib().bigcn_gcnconv_csr_workspace_bytes(n, e, k)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=val.device)
        out = torch.empty(n, H, dtype=torch.float32, device=val.device)
        sc = _csr_scratch(n, k, val.device)
        check(lib().bigcn_gcnconv_csr_forward(_p(ptr), _p(col), _p(val), n, k, _p(ei), e, _p(weight), _p(bias),
                                              L.DEG_BY[deg_by], _p(out), _p(flags), _p(ws), ws_bytes, _p(sc), sc.numel(),
                                              _stream()), "gcnconv_csr_forward")
        ctx.save_for_backward(ptr, col, val, ws)
        ctx.dims = (n, k, e)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        ptr, col, val, ws = ctx.saved_tensors
        n, k, e = ctx.dims
        g = _f32(grad_out)
        dw = torch.empty(H, k, dtype=torch.float32, device=val.device)
        db = torch.empty(H, dtype=torch.float32, device=val.device)
        sc = _csr_scratch(n, k, val.device)
        check(lib().bigcn_gcnconv_csr_backward(_p(ptr), _p(col), _p(val), n, k, e, _p(g), _p(dw), _p(db), _p(ws),
                                               ws.numel(), _p(sc), sc.numel(), _stream()), "gcnconv_csr_backward")
        return None, None, None, None, None, dw, db, None, None


class GCNConvWeightedFunction(torch.autograd.Function):
    """conv(x, edge_index, edge_weight) -> [N,64] (EBGCN.py:84,181); gradients for the conv's weight and
    bias, the edge weights (directly and through the degree normalisation) and x."""

    @staticmethod
    def forward(ctx, x, edge_index, edge_weight, weight, bias, deg_by, gemm_mode):
        L.require_device()
        x, weight, bias, ew = _f32(x), _f32(weight), _f32(bias), _f32(edge_weight)
        ei = _i64(edge_index)
        _need_cuda(x, ei, ew, weight, bias)
        n, k = x.shape
        e = int(ei.shape[1])
        if weight.shape != (H, k):
            raise L.BigcnError(f"GCNConv: out_channels must be {H} and weight [64,{k}], got {tuple(weight.shape)}")
        if ew.shape != (e,):
            raise L.BigcnError(f"GCNConv: edge_weight must be [{e}], got {tuple(ew.shape)}")
        ws_bytes = lib().bigcn_gcnconv_weighted_workspace_bytes(n, e, k)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device)
        flags = torch.zeros(1, dtype=torch.int32, device=x.device)
        out = torch.empty(n, H, dtype=torch.float32, device=x.device)
        check(lib().bigcn_gcnconv_weighted_forward(_p(x), n, k, _p(ei), e, _p(ew), _p(weight), _p(bias),
                                                   L.DEG_BY[deg_by], L.GEMM_MODE[gemm_mode], _p(out), _p(flags),
                                                   _p(ws), ws_bytes, _stream()), "gcnconv_weighted_forward")
        ctx.save_for_backward(x, ei, ew, weight, ws)
        ctx.flags = flags
        ctx.deg_by, ctx.gemm_mode = deg_by, gemm_mode
        return out

    @staticmethod
    def backward(ctx, grad_out):
        x, ei, ew, weight, ws = ctx.saved_tensors
        n, k = x.shape
        e = int(ei.shape[1])
        g = _f32(grad_out)
        dw = torch.empty(H, k, dtype=torch.float32, device=x.device)
        db = torch.empty(H, dtype=torch.float32, device=x.device)
        dew = torch.empty(e, dtype=torch.float32, device=x.device) if ctx.needs_input_grad[2] else None
        dx = torch.empty(n, k, dtype=torch.float32, device=x.device) if ctx.needs_input_grad[0] else None
        check(lib().bigcn_gcnconv_weighted_backward(_p(x), n, k, _p(ei), e, _p(ew), _p(weight), _p(g), _p(dw), _p(db),
                                                    _p(dew), _p(dx), L.DEG_BY[ctx.deg_by], L.GEMM_MODE[ctx.gemm_mode],
                                                    _p(ws), ws.numel(), _stream()), "gcnconv_weighted_backward")
        return dx, None, dew, dw, db, None, None


def ebgcn_x(x):
    """EBGCN's data.x for :class:`EBGCNConv2Function`: dense, widened to contiguous fp32 as the reference's ``.float()``
    does, or a :class:`SparseX` (checked by :func:`sparse_x`; conv1 then runs on the CSR and conv2's op reads the root
    rows from it).  A torch sparse tensor, or an x that requires grad, raises: the op reads x only at the tree roots
    and forms no gradient for it."""
    if isinstance(x, SparseX):
        return sparse_x(x, "EBGCN")
    if not torch.is_tensor(x) or x.layout != torch.strided:
        raise L.BigcnError("EBGCN takes a dense data.x or a bigcn_b200.SparseX (a torch sparse x is not supported); "
                           "pass bigcn_b200.SparseX.from_torch_csr(x)")
    if x.requires_grad:
        raise L.BigcnError("EBGCN forms no gradient w.r.t. data.x: pass data.x.detach() (a data.x that requires grad "
                           "is not supported)")
    if x.dim() != 2:
        raise L.BigcnError(f"EBGCN: data.x must be [N, input_features], got shape {tuple(x.shape)}")
    return _f32(x)


class EBGCNConv2Function(torch.autograd.Function):
    """EBGCN's ``relu(conv2(relu(bn1(cat(h1, x[rootindex[batch]]))), edge_index, edge_weight))`` for one direction
    (EBGCN.py:71-85) without the N x (64 + K) concatenation (bigcn_ebgcn_conv2_*, csrc/ebgcn.cu).  ``bn`` is the
    module's ``torch.nn.BatchNorm1d(64 + K)``: the op reads its parameters and buffers (updating the running statistics
    and ``num_batches_tracked`` in training, as its forward would) and does not run it.  Gradients for h1, edge_weight,
    bn.weight, bn.bias, w2 and b2; ``x`` (dense fp32 or a :class:`SparseX`) is data.  ``node_ptr`` ([B+1] int32)
    receives the tree offsets."""

    @staticmethod
    def forward(ctx, h1, edge_weight_, bn_weight, bn_bias, w2, b2, x, edge_index, batch, rootindex, bn, deg_by, node_ptr,
                flags):
        L.require_device()
        h1, w2, b2 = _f32(h1), _f32(w2), _f32(b2)
        ei, batch, rootindex = _i64(edge_index), _i64(batch), _i64(rootindex)
        xs = x if isinstance(x, SparseX) else None
        xd = None if xs is not None else x
        n, k = x.shape
        e, b = int(ei.shape[1]), int(rootindex.numel())
        ew = edge_weight(edge_weight_, e, "edge_weight")
        _need_cuda(h1, xd, ei, batch, rootindex, w2, b2, *((xs.ptr, xs.col, xs.val) if xs is not None else ()))
        if xs is not None and xs.val.device != h1.device:
            raise L.BigcnError(f"EBGCN: the SparseX x is on {xs.val.device}, the model on {h1.device}")
        if tuple(h1.shape) != (n, H):
            raise L.BigcnError(f"EBGCN: conv1's output must be [{n},{H}], got {tuple(h1.shape)}")
        if tuple(w2.shape) != (H, H + k) or tuple(b2.shape) != (H,):
            raise L.BigcnError(f"EBGCN: conv2 must be GCNConv({H + k}, {H}), got weight {tuple(w2.shape)}")
        if bn.num_features != H + k:
            raise L.BigcnError(f"EBGCN: bn1 must be BatchNorm1d({H + k}), got {bn.num_features}")
        gw = None if bn_weight is None else _f32(bn_weight)
        gb = None if bn_bias is None else _f32(bn_bias)
        rm, rv, nbt = bn.running_mean, bn.running_var, bn.num_batches_tracked
        for t in (rm, rv):
            if t is not None and (t.dtype != torch.float32 or not t.is_contiguous() or not t.is_cuda):
                raise L.BigcnError("EBGCN: bn1's running statistics must be contiguous fp32 CUDA tensors")
        a = L.Ebgcn(N=n, B=b, K=k, E=e, h1=_p(h1), x=_p(xd), edge_index=_p(ei), edge_weight=_p(ew), batch=_p(batch),
                    rootindex=_p(rootindex), node_ptr=_p(node_ptr), bn_weight=_p(gw), bn_bias=_p(gb), running_mean=_p(rm),
                    running_var=_p(rv), num_batches_tracked=_p(nbt),
                    momentum=-1.0 if bn.momentum is None else float(bn.momentum), eps=float(bn.eps),
                    training=int(bn.training), deg_by=L.DEG_BY[deg_by], w2=_p(w2), b2=_p(b2))
        if xs is not None:
            a.x_ptr, a.x_col, a.x_val = _p(xs.ptr), _p(xs.col), _p(xs.val)
        ws_bytes = (lib().bigcn_ebgcn_conv2_workspace_bytes if xs is None else
                    lib().bigcn_ebgcn_conv2_csr_workspace_bytes)(n, b, k, e)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=h1.device)
        out = torch.empty(n, H, dtype=torch.float32, device=h1.device)
        check(lib().bigcn_ebgcn_conv2_forward(C.byref(a), _p(out), _p(flags), _p(ws), ws_bytes, _stream()),
              "ebgcn_conv2_forward")
        # the backward reads the same arguments: keep every tensor they point at
        ctx.save_for_backward(h1, xd if xs is None else xs.val, ei, batch, rootindex, node_ptr, w2, b2, ws, out,
                              *[t for t in (ew, gw, gb) if t is not None], *((xs.ptr, xs.col) if xs is not None else ()))
        ctx.a, ctx.has = a, (ew is not None, gw is not None, gb is not None)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        saved = ctx.saved_tensors
        ws, out = saved[8], saved[9]
        a = ctx.a
        n, k, e = a.N, a.K, a.E
        dev = out.device
        g = _f32(grad_out)
        dh1 = torch.empty(n, H, dtype=torch.float32, device=dev)
        dw2 = torch.empty(H, H + k, dtype=torch.float32, device=dev)
        db2 = torch.empty(H, dtype=torch.float32, device=dev)
        bn_on = n != 1          # EBGCN.py:79: bn1 is skipped for a one-node batch
        dgw = torch.empty(H + k, dtype=torch.float32, device=dev) if bn_on and ctx.needs_input_grad[2] else None
        dgb = torch.empty(H + k, dtype=torch.float32, device=dev) if bn_on and ctx.needs_input_grad[3] else None
        dew = torch.empty(e, dtype=torch.float32, device=dev) if ctx.has[0] and ctx.needs_input_grad[1] else None
        check(lib().bigcn_ebgcn_conv2_backward(C.byref(a), _p(out), _p(g), _p(dh1), _p(dgw), _p(dgb), _p(dw2), _p(db2),
                                               _p(dew), _p(ws), ws.numel(), _stream()), "ebgcn_conv2_backward")
        return (dh1, dew, dgw, dgb, dw2, db2) + (None,) * 8


def gcn_norm(edge_index, edge_weight=None, num_nodes=None, improved=False, add_self_loops=True, deg_by="target"):
    """``torch_geometric.nn.conv.gcn_conv.gcn_norm`` as explain_PHEME.py:62-63 calls it
    (``gcn_norm(edge_index, edge_weight, N, False, True)``): returns (edge_index', norm) with
    edge_index' = [non-loop edges in order | (i, i) for every node].  No gradient (the explain
    script uses it on constants); the differentiable form lives inside GCNConv."""
    L.require_device()
    if improved or not add_self_loops:
        raise NotImplementedError("gcn_norm: only improved=False, add_self_loops=True (the reference's call)")
    ei = _i64(edge_index)
    _need_cuda(ei)
    dev = ei.device
    e = int(ei.shape[1])
    n = int(num_nodes) if num_nodes is not None else (int(ei.max().item()) + 1 if e else 0)
    ew = torch.ones(e, dtype=torch.float32, device=dev) if edge_weight is None else _f32(edge_weight.detach())
    norm_e = torch.empty(max(e, 1), dtype=torch.float32, device=dev)
    norm_self = torch.empty(max(n, 1), dtype=torch.float32, device=dev)
    dis = torch.empty(max(n, 1), dtype=torch.float32, device=dev)
    flags = torch.zeros(1, dtype=torch.int32, device=dev)
    ws_bytes = lib().bigcn_gcn_norm_weighted_workspace_bytes(n, e)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    check(lib().bigcn_gcn_norm_weighted(_p(ei), e, _p(ew), n, L.DEG_BY[deg_by], _p(norm_e), _p(norm_self), _p(dis),
                                        _p(flags), _p(ws), ws_bytes, _stream()), "gcn_norm_weighted")
    raise_on_flags(flags)
    keep = ei[0] != ei[1]
    loops = torch.arange(n, dtype=ei.dtype, device=dev)
    return (torch.cat([ei[:, keep], torch.stack([loops, loops])], dim=1),
            torch.cat([norm_e[:e][keep], norm_self[:n]]))


# ----------------------------------------------------------------------------- feature path
_PNAMES = ("td_w1", "td_b1", "td_w2", "td_b2", "bu_w1", "bu_b1", "bu_w2", "bu_b2")


def edge_weight(w, e, name):
    """A BiGCN edge weight checked and laid out for the library: None stays None; otherwise a CUDA tensor of shape
    [e] with a floating dtype, returned as contiguous fp32.  A non-finite value is reported by the device flags
    (raise_on_flags), with a negative weighted degree."""
    if w is None:
        return None
    if not torch.is_tensor(w):
        raise L.BigcnError(f"{name} must be a tensor, got {type(w).__name__}")
    if not w.is_cuda:
        raise L.BigcnError(f"{name}: bigcn_b200 ops take CUDA tensors only (no CPU fallback)")
    if not w.is_floating_point():
        raise L.BigcnError(f"{name} must have a floating dtype, got {w.dtype}")
    if tuple(w.shape) != (e,):
        raise L.BigcnError(f"{name} must be [{e}] (one weight per column of its edge index), got {tuple(w.shape)}")
    return w.to(torch.float32).contiguous()


def _make_structs(x, ei, bu_ei, batch, rootindex, params, num_classes, node_id_base, xs=None, ew=(None, None)):
    n, k = xs.shape if xs is not None else x.shape
    dims = Dims(N=n, B=int(rootindex.numel()), K=k, C=num_classes, E_td=int(ei.shape[1]),
                E_bu=int(bu_ei.shape[1]))
    bt = BatchPtrs(x=_p(x), edge_index=_p(ei), bu_edge_index=_p(bu_ei), batch=_p(batch), rootindex=_p(rootindex),
                   node_id_base=int(node_id_base), td_edge_weight=_p(ew[0]), bu_edge_weight=_p(ew[1]))
    if xs is not None:
        bt.x_ptr, bt.x_col, bt.x_val = _p(xs.ptr), _p(xs.col), _p(xs.val)
    pr = Params()
    for name, t in zip(_PNAMES, params):
        if t is not None:
            want = {"w1": (H, k), "b1": (H,), "w2": (H, H + k), "b2": (H,)}[name[3:]]
            if tuple(t.shape) != want:
                raise L.BigcnError(f"{name}: expected shape {want} (hid_feats = out_feats = 64), got {tuple(t.shape)}")
        setattr(pr, name, _p(t))
    return dims, bt, pr


def batch_args(x, edge_index, bu_edge_index, batch, rootindex, td_ew=None, bu_ew=None, *, gemm_mode, num_classes=0,
               node_id_base=0, params=()):
    """Check a batch and lay it out for the feature path: data.x as ``gemm_mode`` reads it, the index tensors as
    int64, the edge weights as fp32 [E], all on a CUDA device; ``params`` (``_PNAMES`` order, None for a direction
    left out) shape-checked.  Returns the structs ``dims``, ``bt``, ``pr`` (null pointers without params), the tensors
    they point at, which the caller keeps until the launches are done (``x`` or ``xs`` (SparseX), ``ei``, ``bu``,
    ``batch``, ``root``, ``ew`` = (TD, BU)), ``dev`` and ``weighted``."""
    x, xs = _as_x(x, gemm_mode)
    if xs is not None and gemm_mode != "sparse":
        raise L.BigcnError("a sparse data.x needs gemm_mode='sparse'")
    ei, bu, batch, root = _i64(edge_index), _i64(bu_edge_index), _i64(batch), _i64(rootindex)
    _need_cuda(x, ei, bu, batch, root, *params)
    if xs is not None:
        _need_cuda(xs.ptr, xs.col, xs.val)
    ew = (edge_weight(td_ew, int(ei.shape[1]), "edge_weight"), edge_weight(bu_ew, int(bu.shape[1]), "BU_edge_weight"))
    dims, bt, pr = _make_structs(x, ei, bu, batch, root, params, num_classes, node_id_base, xs, ew)
    return SimpleNamespace(dims=dims, bt=bt, pr=pr, x=x, xs=xs, ei=ei, bu=bu, batch=batch, root=root, ew=ew,
                           dev=xs.device if xs is not None else x.device, weighted=any(w is not None for w in ew))


def features_workspace_bytes(dims, weighted, edge_grad=False):
    return lib().bigcn_features_edge_workspace_bytes(C.byref(dims), int(edge_grad)) if weighted else \
        lib().bigcn_features_workspace_bytes(C.byref(dims))


def batch_prepare_bytes(dims, weighted):
    return (lib().bigcn_batch_prepare_edge_bytes if weighted else lib().bigcn_batch_prepare_bytes)(C.byref(dims))


def batch_key(data, *extra):
    """What a captured CUDA graph or a prepared buffer read of a batch: the object, and where its tensors (data.x, the
    two edge indices, batch, rootindex, then ``extra``) live, with their shapes and dtypes -- not their values"""
    x = data.x
    xk = (x.ptr.data_ptr(), x.col.data_ptr(), x.val.data_ptr(), x.shape) if hasattr(x, "ptr") else \
        (x.data_ptr(), tuple(x.shape), x.dtype, x.layout)
    # built on every replayed step: a list comprehension costs less host time than a generator here
    return (id(data), xk, tuple([(t.data_ptr(), tuple(t.shape), t.dtype) for t in
                                 (data.edge_index, data.BU_edge_index, data.batch, data.rootindex, *extra)]))


def edge_weight_key(data):
    """batch_key's counterpart for the batch's edge weights (data.edge_weight, data.BU_edge_weight)"""
    return tuple([(w.data_ptr(), tuple(w.shape), w.dtype) if torch.is_tensor(w) else id(w)
                  for w in (getattr(data, "edge_weight", None), getattr(data, "BU_edge_weight", None))])


def x_val(x):
    """The autograd input that carries a SparseX's gradient (its ``val``), None for any other data.x:
    FeaturesFunction takes it beside x, which autograd cannot see into."""
    return x.val if isinstance(x, SparseX) else None


class FeaturesFunction(torch.autograd.Function):
    """TDrumorGCN / BUrumorGCN forward for the directions in dir_mask -> feat [B,256]
    laid out [BU mean | BU root | TD mean | TD root] (cat order of BiGCN_Twitter.py:128).

    Gradient w.r.t. data.x (conv1's input) when it requires one: a dense x gets dX = T1cat [W1_TD; W1_BU]; a sparse
    x gets that gradient sampled at its stored entries -- ``val`` (= ``x_val(x)``, a SparseX's values) gets fp32 [nnz],
    a torch sparse COO x a COO gradient on ``x.coalesce()``'s indices (the ``torch.sparse.mm`` convention), a
    torch sparse CSR x a CSR gradient on its own ``crow_indices`` / ``col_indices`` (torch's ``csr @ dense``
    returns a dense one instead: the masked form keeps the gradient as small as x).

    ``td_ew`` / ``bu_ew`` (None, or [E_td] / [E_bu]): edge weights of both convs of that direction, as
    ``GCNConv(x, edge_index, edge_weight)``; their gradients are formed only when they require one."""

    @staticmethod
    def forward(ctx, x, val, ei, bu_ei, batch, rootindex, td_ew, bu_ew, opts, *params):
        L.require_device()
        ctx.x_layout = x.layout if isinstance(x, torch.Tensor) else None
        if ctx.needs_input_grad[0] and x.layout == torch.sparse_coo:
            x = x.coalesce()     # the CSR below keeps this order: its gradient values map onto these indices
        if ctx.needs_input_grad[0] and x.layout in (torch.sparse_coo, torch.sparse_csr):
            ctx.x_pattern = (x.indices(),) if x.layout == torch.sparse_coo else (x.crow_indices(), x.col_indices())
        elif ctx.needs_input_grad[0] and x.layout != torch.strided:
            raise L.BigcnError(f"a gradient w.r.t. a {x.layout} data.x is not produced: pass it as sparse COO or CSR")
        params = tuple(None if p is None else _f32(p) for p in params)
        a = batch_args(x, ei, bu_ei, batch, rootindex, td_ew, bu_ew, gemm_mode=opts["gemm_mode"],
                       node_id_base=opts["node_id_base"], params=params)
        x, xs, dims, dev = a.x, a.xs, a.dims, a.dev
        want_grad = opts.get("want_grad", True)
        edge_grad = want_grad and (ctx.needs_input_grad[6] or ctx.needs_input_grad[7])
        o = Opts(training=int(opts["training"]), p_drop=float(opts["p"]), seed=int(opts["seed"]),
                 deg_by=L.DEG_BY[opts["deg_by"]], gemm_mode=L.GEMM_MODE[opts["gemm_mode"]],
                 dir_mask=int(opts["dir_mask"]), dense_roots=int(bool(opts.get("dense_roots", False))),
                 # inference (torch.no_grad() or no parameter wants a gradient): no column sort of x
                 skip_wgrad_prep=int(not (want_grad and any(ctx.needs_input_grad))), edge_grad=int(edge_grad))
        ws_bytes = features_workspace_bytes(dims, a.weighted, o.edge_grad)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        flags = opts.get("flags")
        if flags is None:
            flags = torch.zeros(1, dtype=torch.int32, device=dev)
        feat = torch.empty(dims.B, 4 * H, dtype=torch.float32, device=dev)
        check(lib().bigcn_features_forward(C.byref(dims), C.byref(a.bt), C.byref(a.pr), C.byref(o), _p(feat),
                                           _p(flags), _p(ws), ws_bytes, _stream()), "features_forward")
        if o.gemm_mode == L.GEMM_MODE["sparse"] and not o.skip_wgrad_prep:
            # the column sort of x is still running on the library's low-priority stream: keep the
            # caching allocator from recycling the workspace (or x) under it
            h = lib().bigcn_internal_stream()
            if h:
                side = torch.cuda.ExternalStream(h, device=dev)
                for t in (ws, x) if xs is None else (ws, xs.ptr, xs.col, xs.val):
                    t.record_stream(side)
        xt = (x,) if xs is None else (xs.ptr, xs.col, xs.val)
        ctx.x_sparse_shape = None if xs is None else xs.shape
        # the backward reuses the structs: the saved tensors are the ones they point at
        ctx.save_for_backward(*xt, a.ei, a.bu, a.batch, a.root, ws, *[p for p in params if p is not None])
        ctx.present = [p is not None for p in params]
        ctx.o = o
        ctx.ew = a.ew
        ctx.structs = (dims, a.bt, a.pr)
        ctx.flags = flags
        return feat

    @staticmethod
    def backward(ctx, grad_feat):
        saved = ctx.saved_tensors      # unpacked all the same: autograd's check that none was modified in place
        x, xs = saved[0], None
        if ctx.x_sparse_shape is not None:
            x, xs = None, SparseX(saved[0], saved[1], saved[2], ctx.x_sparse_shape)
            saved = saved[2:]
        ws = saved[5]
        it = iter(saved[6:])
        params = tuple(next(it) if pres else None for pres in ctx.present)
        dims, bt, pr = ctx.structs
        grads = tuple(None if p is None else torch.empty_like(p) for p in params)
        gs = Params()
        for name, t in zip(_PNAMES, grads):
            setattr(gs, name, _p(t))
        g = _f32(grad_feat)
        check(lib().bigcn_features_backward(C.byref(dims), C.byref(bt), C.byref(pr), C.byref(ctx.o), _p(g),
                                            C.byref(gs), _p(ws), ws.numel(), _stream()),
              "features_backward")
        dew = [None, None]
        if ctx.o.edge_grad:
            # dL/dnorm of every edge was taken by the backward; the chain through the normalisation runs here
            for q, e in ((0, dims.E_td), (1, dims.E_bu)):
                if ctx.needs_input_grad[6 + q] and ctx.ew[q] is not None:
                    dew[q] = torch.empty(e, dtype=torch.float32, device=ctx.ew[q].device)
            check(lib().bigcn_features_edge_grad(C.byref(dims), C.byref(bt), C.byref(ctx.o), _p(dew[0]), _p(dew[1]),
                                                 _p(ws), ws.numel(), _stream()), "features_edge_grad")
        dx = dval = None
        if (ctx.needs_input_grad[0] or ctx.needs_input_grad[1]) and xs is not None:
            # the dense gradient below sampled at the stored entries of x, in CSR order; T1cat and W1^T come from ws
            nnz = xs.val.numel()
            g = torch.empty(nnz, dtype=torch.float32, device=xs.val.device)
            check(lib().bigcn_features_x_grad_csr(C.byref(dims), C.byref(bt), C.byref(ctx.o), _p(g), nnz, _p(ws),
                                                  ws.numel(), _stream()), "features_x_grad_csr")
            if ctx.needs_input_grad[1]:
                dval = g
            elif ctx.x_layout == torch.sparse_coo:
                dx = torch.sparse_coo_tensor(ctx.x_pattern[0], g, xs.shape, is_coalesced=True)
            else:
                dx = torch.sparse_csr_tensor(*ctx.x_pattern, g, xs.shape)
        elif ctx.needs_input_grad[0] and x is not None:
            # only conv1 carries a gradient to x: the root-extend reads the detached copy.copy (BiGCN_Twitter.py:28).
            # dX = T1cat [W1_TD; W1_BU], T1cat left in the workspace by features_backward.  Same dtype as the x the
            # forward read: bf16 in gemm_mode='bf16', fp32 otherwise (autograd casts it to a widened x's dtype)
            n, k = x.shape
            dx = torch.empty(n, k, dtype=x.dtype, device=x.device)
            bf = x.dtype == torch.bfloat16
            nscr = lib().bigcn_x_dgrad_scratch_floats(n, k, bin(ctx.o.dir_mask).count("1"))
            scr = torch.empty(nscr, dtype=torch.float32, device=x.device)
            check(lib().bigcn_features_x_grad(C.byref(dims), C.byref(pr), C.byref(ctx.o), None if bf else _p(dx),
                                              _p(dx) if bf else None, _p(scr), _p(ws), ws.numel(), _stream()),
                  "features_x_grad")
        return (dx, dval, None, None, None, None, dew[0], dew[1], None) + grads


class HeadFunction(torch.autograd.Function):
    """log_softmax(feat @ fc_w.T + fc_b) (BiGCN_Twitter.py:129-130)."""

    @staticmethod
    def forward(ctx, feat, fc_w, fc_b):
        L.require_device()
        feat, fc_w, fc_b = _f32(feat), _f32(fc_w), _f32(fc_b)
        b, c = feat.shape[0], fc_w.shape[0]
        if fc_w.shape[1] != 4 * H or feat.shape[1] != 4 * H:
            raise L.BigcnError("head: fc.weight must be [C,256]")
        logp = torch.empty(b, c, dtype=torch.float32, device=feat.device)
        check(lib().bigcn_head_forward(_p(feat), b, c, _p(fc_w), _p(fc_b), _p(logp), _stream()), "head_forward")
        ctx.save_for_backward(feat, fc_w, logp)
        return logp

    @staticmethod
    def backward(ctx, grad_logp):
        feat, fc_w, logp = ctx.saved_tensors
        b, c = logp.shape
        g = _f32(grad_logp)
        gfeat = torch.empty_like(feat)
        dw = torch.empty_like(fc_w)
        db = torch.empty(c, dtype=torch.float32, device=feat.device)
        nscr = lib().bigcn_head_backward_scratch_floats(b, c)
        scr = torch.empty(nscr, dtype=torch.float32, device=feat.device)
        check(lib().bigcn_head_backward(_p(g), _p(logp), _p(feat), b, c, _p(fc_w), _p(gfeat), _p(dw), _p(db),
                                        _p(scr), nscr, _stream()), "head_backward")
        return gfeat, dw, db


# ----------------------------------------------------------------------------- loss / optimiser
def nll_loss(logp, y, b_global=None, want_grad=False):
    """F.nll_loss(logp, y) with mean over b_global trees (BiGCN_Twitter.py:184)."""
    L.require_device()
    b, c = logp.shape
    y = _i64(y)
    loss = torch.empty(1, dtype=torch.float32, device=logp.device)
    grad = torch.empty_like(logp) if want_grad else None
    check(lib().bigcn_nll_loss(_p(logp), _p(y), b, c, int(b_global or b), _p(loss), _p(grad), _stream()),
          "nll_loss")
    return (loss, grad) if want_grad else loss
