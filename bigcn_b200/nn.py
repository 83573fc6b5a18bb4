"""Drop-in modules for the reference's hot path.

Same class names, constructor signatures, sub-module names and state_dict keys as
/root/reference/model/Twitter/BiGCN_Twitter.py:19-131 (``TDrumorGCN``, ``BUrumorGCN``,
``BiGCN``) and /root/reference/model/Weibo/BiGCN_Weibo.py:16-89 (``Net``), and a
``GCNConv`` that stands in for ``torch_geometric.nn.GCNConv`` on this path
(``conv(x, edge_index)`` as called at explain_PHEME.py:95,132).  ``forward(data)``
is duck-typed on ``data.x, data.edge_index, data.BU_edge_index, data.batch,
data.rootindex`` and the optional ``data.edge_weight`` / ``data.BU_edge_weight`` (the edge weights of
both convs of that direction, as ``GCNConv(x, edge_index, edge_weight)``).  All arithmetic runs in libbigcn_b200.so; nothing here falls back
to PyTorch or the CPU.
"""
from __future__ import annotations

import math

import torch

from . import _lib as L
import ctypes as C
import weakref

from .ops import (FeaturesFunction, GCNConvFunction, GCNConvWeightedFunction, HeadFunction, raise_on_flags,
                  capture_graph, pick_gemm_mode, bf16_features_dense, edge_weight, x_val, _as_x, _i64, _make_structs, _p,
                  _stream)

H = L.H


class _Lin(torch.nn.Module):
    """``GCNConv.lin`` of PyG 2.x: Linear(in, out, bias=False), glorot-uniform weight [out,in]."""

    def __init__(self, in_channels, out_channels):
        super().__init__()
        self.weight = torch.nn.Parameter(torch.empty(out_channels, in_channels))
        a = math.sqrt(6.0 / (in_channels + out_channels))
        with torch.no_grad():
            self.weight.uniform_(-a, a)


class GCNConv(torch.nn.Module):
    """GCNConv(in, 64): state_dict keys ``lin.weight`` [64,in] and ``bias`` [64] (PyG 2.x);
    PyG-1.3.2 checkpoints (``weight`` [in,64]) are accepted on load."""

    def __init__(self, in_channels, out_channels, deg_by="target", gemm_mode="auto"):
        super().__init__()
        if out_channels != H:
            raise L.BigcnError(f"bigcn_b200 kernels are specialised for out_channels = {H} "
                               f"(the reference's only configuration), got {out_channels}")
        self.in_channels, self.out_channels = in_channels, out_channels
        self.lin = _Lin(in_channels, out_channels)
        self.bias = torch.nn.Parameter(torch.zeros(out_channels))
        self.deg_by, self.gemm_mode = deg_by, gemm_mode
        self._auto_mode = None

    def _mode(self, x):
        if self.gemm_mode != "auto":
            return self.gemm_mode
        if self._auto_mode is None:         # decided once, on the first feature matrix this conv sees
            self._auto_mode = pick_gemm_mode(x.detach())
        return self._auto_mode

    def forward(self, x, edge_index, edge_weight=None):
        if edge_weight is None and torch.is_tensor(x) and x.requires_grad:
            # x is an activation (EBGCN's conv2 input is batch-normalised): the generic form returns dx
            edge_weight = torch.ones(edge_index.shape[1], dtype=torch.float32, device=x.device)
        if edge_weight is not None:      # EBGCN.py:84,181
            return GCNConvWeightedFunction.apply(x, edge_index, edge_weight, self.lin.weight, self.bias, self.deg_by,
                                                 self._mode(x))
        return GCNConvFunction.apply(x, edge_index, self.lin.weight, self.bias, self.deg_by, self._mode(x))

    def _load_from_state_dict(self, state_dict, prefix, *args, **kw):
        old = prefix + "weight"      # torch_geometric 1.3.2: weight [in,out]
        if old in state_dict and prefix + "lin.weight" not in state_dict:
            state_dict[prefix + "lin.weight"] = state_dict.pop(old).t().contiguous()
        super()._load_from_state_dict(state_dict, prefix, *args, **kw)


class _RumorGCN(torch.nn.Module):
    _dir = L.DIR_TD

    def __init__(self, in_feats, hid_feats, out_feats, device=None, deg_by="target", gemm_mode="auto"):
        super().__init__()
        if hid_feats != H or out_feats != H:
            raise L.BigcnError(f"bigcn_b200 kernels are specialised for hid_feats = out_feats = {H}")
        self.conv1 = GCNConv(in_feats, hid_feats, deg_by, gemm_mode)
        self.conv2 = GCNConv(hid_feats + in_feats, out_feats, deg_by, gemm_mode)
        self.device = device
        self.p = 0.5                        # F.dropout default (BiGCN_Twitter.py:54)
        self.deg_by, self.gemm_mode = deg_by, gemm_mode
        self.seed = torch.initial_seed() & ((1 << 63) - 1)
        self._calls = 0
        self.node_id_base = 0
        self.last_flags = None
        self._auto_mode = None
        self._bf16_dense = None
        self.dense_roots = "auto"           # see resolved_dense_roots

    def resolved_gemm_mode(self, x):
        """``gemm_mode`` with 'auto' resolved: a sparse ``data.x`` -> 'sparse'; a dense one -> 'sparse' for
        row-sparse bag-of-words features, 'tf32x3' for dense features (ops.pick_gemm_mode; decided on the
        first batch, one small device -> host read, then cached for the life of the module)."""
        if self.gemm_mode != "auto":
            return self.gemm_mode
        if not (isinstance(x, torch.Tensor) and x.layout == torch.strided):
            return "sparse"
        if self._auto_mode is None:
            self._auto_mode = pick_gemm_mode(x.detach())
        return self._auto_mode

    def resolved_dense_roots(self, x):
        """``opts.dense_roots`` (training only): the root half of conv2.lin as a tiled masked product instead of a walk
        over each tree's positive root columns.  ``self.dense_roots`` = True / False forces it; 'auto' (default) turns
        it on when ``gemm_mode='auto'`` measured DENSE features (PHEME's sentence embeddings), or when ``gemm_mode='bf16'``
        finds dense rows with the same probe on the bf16 values -- bag-of-words roots (~20 columns) keep the list walk.
        Same forward sums in the same order either way."""
        if self.dense_roots != "auto":
            return bool(self.dense_roots) and isinstance(x, torch.Tensor) and x.layout == torch.strided
        if self.gemm_mode == "bf16":
            if self._bf16_dense is None:     # decided once, on the first feature matrix, like gemm_mode='auto'
                self._bf16_dense = bf16_features_dense(x.detach())
            return self._bf16_dense
        return self.gemm_mode == "auto" and self.resolved_gemm_mode(x) != "sparse"

    def _conv_params(self):
        return (self.conv1.lin.weight, self.conv1.bias, self.conv2.lin.weight, self.conv2.bias)

    def _opts(self, dir_mask, x=None):
        seed = (self.seed + self._calls) & ((1 << 64) - 1)
        if self.training:
            self._calls += 1
        self.last_seed = seed
        # want_grad: autograd.Function.forward cannot see torch.no_grad() (needs_input_grad is True for
        # parameters either way); inference then skips the capture / column sort of x that only dW1 needs
        return dict(training=self.training, p=self.p, seed=seed, deg_by=self.deg_by,
                    gemm_mode=self.resolved_gemm_mode(x), dense_roots=self.resolved_dense_roots(x),
                    dir_mask=dir_mask, node_id_base=self.node_id_base,
                    want_grad=torch.is_grad_enabled())

    def forward(self, data):
        none4 = (None,) * 4
        td = self._dir == L.DIR_TD
        params = self._conv_params() + none4 if td else none4 + self._conv_params()
        ew = (getattr(data, "edge_weight", None), None) if td else (None, getattr(data, "BU_edge_weight", None))
        feat = FeaturesFunction.apply(data.x, x_val(data.x), data.edge_index, data.BU_edge_index, data.batch,
                                      data.rootindex, *ew, self._opts(self._dir, data.x), *params)
        return feat[:, 2 * H:] if self._dir == L.DIR_TD else feat[:, :2 * H]


class TDrumorGCN(_RumorGCN):
    """BiGCN_Twitter.py:19-67."""
    _dir = L.DIR_TD


class BUrumorGCN(_RumorGCN):
    """BiGCN_Twitter.py:70-114."""
    _dir = L.DIR_BU


class BiGCN(torch.nn.Module):
    """BiGCN_Twitter.py:117-131: ``BiGCN(in_feats, hid_feats, out_feats, device)`` -> log-probs [B,4]."""

    def __init__(self, in_feats, hid_feats, out_feats, device=None, num_classes=4, deg_by="target",
                 gemm_mode="auto", validate="lazy", graphs=False, max_graphs=8):
        super().__init__()
        self.TDrumorGCN = TDrumorGCN(in_feats, hid_feats, out_feats, device, deg_by, gemm_mode)
        self.BUrumorGCN = BUrumorGCN(in_feats, hid_feats, out_feats, device, deg_by, gemm_mode)
        self.fc = torch.nn.Linear((out_feats + hid_feats) * 2, num_classes)
        self.device = device
        self.validate = validate            # "lazy": check the previous call's flags; "sync"; "off"
        self.last_flags = None
        self.graphs = bool(graphs)          # inference under torch.no_grad(): replay a CUDA graph for a batch seen before
        self.max_graphs = int(max_graphs)
        self._graphs, self._seen = {}, {}

    @property
    def gemm_mode(self):
        return self.TDrumorGCN.gemm_mode

    @gemm_mode.setter
    def gemm_mode(self, mode):
        for m in (self.TDrumorGCN, self.BUrumorGCN):
            m.gemm_mode = mode

    def check_inputs(self):
        """Raise if the last forward saw an invalid graph (synchronises)."""
        if self.last_flags is not None:
            flags, self.last_flags = self.last_flags, None
            raise_on_flags(flags)

    def forward(self, data):
        if self.validate == "lazy":
            self.check_inputs()
        if not torch.is_grad_enabled():
            return self._forward_nograd(data)
        td = self.TDrumorGCN
        opts = td._opts(L.DIR_TD | L.DIR_BU, data.x)
        flags = torch.zeros(1, dtype=torch.int32, device=data.x.device)
        opts["flags"] = flags
        feat = FeaturesFunction.apply(data.x, x_val(data.x), data.edge_index, data.BU_edge_index, data.batch,
                                      data.rootindex, getattr(data, "edge_weight", None),
                                      getattr(data, "BU_edge_weight", None), opts, *td._conv_params(),
                                      *self.BUrumorGCN._conv_params())
        out = HeadFunction.apply(feat, self.fc.weight, self.fc.bias)
        self.last_flags = flags
        if self.validate == "sync":
            self.check_inputs()
        return out

    # ---- inference (torch.no_grad()): two C-ABI calls, no autograd nodes; a batch seen before replays a CUDA graph
    def _infer_plan(self, data):
        L.require_device()
        td, bu = self.TDrumorGCN, self.BUrumorGCN
        mode = td.resolved_gemm_mode(data.x)
        x, xs = _as_x(data.x, mode)
        ei, bue, batch, root = _i64(data.edge_index), _i64(data.BU_edge_index), _i64(data.batch), _i64(data.rootindex)
        params = tuple(p.detach() for p in td._conv_params() + bu._conv_params())
        for t in (x, ei, bue, batch, root) + params:
            if t is not None and not t.is_cuda:
                raise L.BigcnError("bigcn_b200 ops take CUDA tensors only (no CPU fallback)")
        c = self.fc.weight.shape[0]
        if xs is not None and mode != "sparse":
            raise L.BigcnError("a sparse data.x needs gemm_mode='sparse'")
        ew = (edge_weight(getattr(data, "edge_weight", None), int(ei.shape[1]), "edge_weight"),
              edge_weight(getattr(data, "BU_edge_weight", None), int(bue.shape[1]), "BU_edge_weight"))
        dims, bt, pr = _make_structs(x, ei, bue, batch, root, params, c, td.node_id_base, xs, ew)
        opts = td._opts(L.DIR_TD | L.DIR_BU, data.x)
        o = L.Opts(training=int(self.training), p_drop=float(td.p), seed=int(opts["seed"]), deg_by=L.DEG_BY[td.deg_by],
                   gemm_mode=L.GEMM_MODE[mode], dir_mask=L.DIR_TD | L.DIR_BU, skip_wgrad_prep=1)
        dev = xs.device if xs is not None else x.device
        nbytes = L.lib().bigcn_features_workspace_bytes(C.byref(dims)) if ew == (None, None) else \
            L.lib().bigcn_features_edge_workspace_bytes(C.byref(dims), 0)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        return {"dims": dims, "bt": bt, "pr": pr, "o": o, "ws": ws, "c": c,
                "keep": (x, xs, ei, bue, batch, root, params, ew, self.fc.weight, self.fc.bias),
                "flags": torch.zeros(1, dtype=torch.int32, device=dev),
                "feat": torch.empty(dims.B, 4 * H, dtype=torch.float32, device=dev),
                "logp": torch.empty(dims.B, c, dtype=torch.float32, device=dev)}

    def _infer_enqueue(self, p):
        l, st = L.lib(), _stream()
        L.check(l.bigcn_features_forward(C.byref(p["dims"]), C.byref(p["bt"]), C.byref(p["pr"]), C.byref(p["o"]),
                                         _p(p["feat"]), _p(p["flags"]), _p(p["ws"]), p["ws"].numel(), st), "features_forward")
        L.check(l.bigcn_head_forward(_p(p["feat"]), p["dims"].B, p["c"], _p(self.fc.weight), _p(self.fc.bias),
                                     _p(p["logp"]), st), "head_forward")

    def _forward_nograd(self, data):
        use_graph = self.graphs and not (self.training and self.TDrumorGCN.p > 0)   # train-mode masks need a fresh seed
        if not use_graph:
            p = self._infer_plan(data)
            self._infer_enqueue(p)
        else:
            x = data.x
            xk = (x.ptr.data_ptr(), x.col.data_ptr(), x.val.data_ptr(), x.shape) if hasattr(x, "ptr") else \
                (x.data_ptr(), tuple(x.shape), x.dtype, x.layout)
            ews = (getattr(data, "edge_weight", None), getattr(data, "BU_edge_weight", None))
            key = (id(data), xk, tuple((t.data_ptr(), tuple(t.shape), t.dtype) for t in
                             (data.edge_index, data.BU_edge_index, data.batch, data.rootindex)),
                   tuple(None if t is None else (t.data_ptr(), tuple(t.shape), t.dtype) for t in ews),
                   tuple(q.data_ptr() for q in self.parameters()), self.training, self.TDrumorGCN.deg_by,
                   self.TDrumorGCN.gemm_mode)
            p = self._graphs.get(key)
            if p is not None:
                p["graph"].replay()
            elif self._seen.get(key) is None or self._seen[key]() is not data:   # first sighting of this batch object
                if len(self._seen) >= 4096:
                    self._seen.clear()
                self._seen[key] = weakref.ref(data)
                p = self._infer_plan(data)
                self._infer_enqueue(p)
            else:                               # seen before: capture, then replay
                p = self._infer_plan(data)
                g = capture_graph(lambda: self._infer_enqueue(p))
                p["graph"], p["data"] = g, data        # the strong reference pins id(data)
                while len(self._graphs) >= self.max_graphs:
                    self._graphs.pop(next(iter(self._graphs)))
                self._graphs[key] = p
                g.replay()
        self.last_flags = p["flags"]
        if self.validate == "sync":
            self.check_inputs()
        return p["logp"]


class Net(BiGCN):
    """BiGCN_Weibo.py:76-89: ``Net(in_feats, hid_feats, out_feats)`` -> log-probs [B,2]."""

    def __init__(self, in_feats, hid_feats, out_feats, num_classes=2, **kw):
        super().__init__(in_feats, hid_feats, out_feats, None, num_classes=num_classes, **kw)
