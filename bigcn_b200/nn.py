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

from .ops import (FeaturesFunction, GCNConvCSRFunction, GCNConvFunction, GCNConvWeightedFunction, GraphCache,
                  HeadFunction, SparseX, raise_on_flags, pick_gemm_mode, bf16_features_dense, batch_args, batch_key,
                  edge_weight_key, features_workspace_bytes, sparse_x, x_val, _p, _stream)

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
    PyG-1.3.2 checkpoints (``weight`` [in,64]) are accepted on load.

    ``x`` may be a :class:`~bigcn_b200.SparseX` (bag-of-words rows as CSR, never densified): the product then runs
    from the CSR and dW as a sweep over x's columns, with ``gemm_mode`` 'auto' or 'sparse' and no ``edge_weight``.
    Its violation word (an out-of-range column, more non-zeros than N*min(K,48)) is ``last_flags``; pass it to
    ``ops.raise_on_flags`` to check."""

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
        self.last_flags = None

    def _mode(self, x):
        if self.gemm_mode != "auto":
            return self.gemm_mode
        if self._auto_mode is None:         # decided once, on the first feature matrix this conv sees
            self._auto_mode = pick_gemm_mode(x.detach())
        return self._auto_mode

    def forward(self, x, edge_index, edge_weight=None):
        if isinstance(x, SparseX):
            if edge_weight is not None:
                raise L.BigcnError("GCNConv: edge_weight is not supported with a SparseX x (the edge-weighted conv has "
                                   "no CSR form); pass a dense x")
            if self.gemm_mode not in ("auto", "sparse"):
                raise L.BigcnError(f"a sparse data.x needs gemm_mode='sparse' (or 'auto'), got {self.gemm_mode!r}")
            xs = sparse_x(x, "GCNConv")
            self.last_flags = torch.zeros(1, dtype=torch.int32, device=xs.device)
            return GCNConvCSRFunction.apply(xs.val, xs.ptr, xs.col, xs.shape, edge_index, self.lin.weight, self.bias,
                                            self.deg_by, self.last_flags)
        self.last_flags = None             # the dense paths report nothing here: no stale flags from a SparseX batch
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
        self._graphs = GraphCache(max_graphs, 4096)

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
        c = self.fc.weight.shape[0]
        params = tuple(p.detach() for p in td._conv_params() + bu._conv_params())
        a = batch_args(data.x, data.edge_index, data.BU_edge_index, data.batch, data.rootindex,
                       getattr(data, "edge_weight", None), getattr(data, "BU_edge_weight", None), gemm_mode=mode,
                       num_classes=c, node_id_base=td.node_id_base, params=params)
        opts = td._opts(L.DIR_TD | L.DIR_BU, data.x)
        o = L.Opts(training=int(self.training), p_drop=float(td.p), seed=int(opts["seed"]), deg_by=L.DEG_BY[td.deg_by],
                   gemm_mode=L.GEMM_MODE[mode], dir_mask=L.DIR_TD | L.DIR_BU, skip_wgrad_prep=1)
        ws = torch.empty(features_workspace_bytes(a.dims, a.weighted), dtype=torch.uint8, device=a.dev)
        return {"dims": a.dims, "bt": a.bt, "pr": a.pr, "o": o, "ws": ws, "c": c,
                "keep": (a, params, self.fc.weight, self.fc.bias),
                "flags": torch.zeros(1, dtype=torch.int32, device=a.dev),
                "feat": torch.empty(a.dims.B, 4 * H, dtype=torch.float32, device=a.dev),
                "logp": torch.empty(a.dims.B, c, dtype=torch.float32, device=a.dev)}

    def _infer_enqueue(self, p):
        l, st = L.lib(), _stream()
        L.check(l.bigcn_features_forward(C.byref(p["dims"]), C.byref(p["bt"]), C.byref(p["pr"]), C.byref(p["o"]),
                                         _p(p["feat"]), _p(p["flags"]), _p(p["ws"]), p["ws"].numel(), st), "features_forward")
        L.check(l.bigcn_head_forward(_p(p["feat"]), p["dims"].B, p["c"], _p(self.fc.weight), _p(self.fc.bias),
                                     _p(p["logp"]), st), "head_forward")

    def _forward_nograd(self, data):
        use_graph = self.graphs and not (self.training and self.TDrumorGCN.p > 0)   # train-mode masks need a fresh seed
        p = key = None
        if use_graph:
            key = batch_key(data) + (edge_weight_key(data), tuple(q.data_ptr() for q in self.parameters()),
                                     self.training, self.TDrumorGCN.deg_by, self.TDrumorGCN.gemm_mode)
            p = self._graphs.replay(key)
        if p is None:
            p = self._infer_plan(data)
            if not use_graph or self._graphs.first_sighting(key, data):
                self._infer_enqueue(p)
            else:
                self._graphs.capture(key, lambda: self._infer_enqueue(p), p, data=data)
        self.last_flags = p["flags"]
        if self.validate == "sync":
            self.check_inputs()
        return p["logp"]


class Net(BiGCN):
    """BiGCN_Weibo.py:76-89: ``Net(in_feats, hid_feats, out_feats)`` -> log-probs [B,2]."""

    def __init__(self, in_feats, hid_feats, out_feats, num_classes=2, **kw):
        super().__init__(in_feats, hid_feats, out_feats, None, num_classes=num_classes, **kw)
