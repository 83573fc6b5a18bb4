"""EBGCN (the fork's second GCN model, model/Twitter/EBGCN.py) on this library.

Same class names, constructor (``args`` with ``input_features``, ``hidden_features``, ``output_features``,
``edge_num``, ``dropout``, ``num_class``, ``edge_infer_td``, ``edge_infer_bu``), sub-module names and ``state_dict``
keys as the reference, and the same ``forward(data) -> (log-probs [B, num_class], TD_edge_loss, BU_edge_loss)``, so
a reference checkpoint loads unchanged.

What runs where:
  conv1 (EBGCN.py:64)                                   -> bigcn_b200.GCNConv
  root-extend, cat, bn1, relu, conv2 with the inferred edge weights, relu (:71-85)
                                                        -> EBGCNConv2Function (csrc/ebgcn.cu): the N x (64 + K)
                                                           concatenation is never formed; bn1's statistics over the
                                                           K root columns come from the B root rows, weighted by tree size
  second root-extend + scatter_mean (:86-92)            -> torch.ops.bigcn_b200.readout
  fc + log_softmax (:230-232)                           -> the BiGCN head (HeadFunction)
  edge-inference sub-networks and their KL loss (:29-59, :95-117): the reference's torch modules, unchanged (including
  the ``row - 1`` / ``col - 1`` indexing and the ``torch.normal`` draw; the library op draws nothing from torch's
  generator, so the random stream is the reference's).

``bn1`` is a real ``torch.nn.BatchNorm1d(hidden + input)``: its parameters, buffers, ``train()`` / ``eval()`` and
momentum behave as users expect; the op reads and updates them as its forward would.  data.x is dense (widened to
fp32) or a ``SparseX``, as ``DeviceForest`` batches and ``forest_from_raw`` forests hand it over: conv1 then runs on
the CSR and conv2's op reads the root rows from it, so nothing N x K is formed.  A torch sparse data.x, or one that
requires grad, raises BigcnError.
"""
from __future__ import annotations

from collections import OrderedDict

import torch
import torch.nn.functional as F

from . import _lib as L
from .nn import GCNConv
from .ops import EBGCNConv2Function, HeadFunction, ebgcn_x, raise_on_flags


def _create_network(hidden, name):
    """EBGCN.py:33-48: Conv1d(k=1, no bias) -> BatchNorm1d -> LeakyReLU, then Conv1d(hidden -> 1, k=1)."""
    layers = OrderedDict()
    layers[name + "conv0"] = torch.nn.Conv1d(hidden, hidden, kernel_size=1, bias=False)
    layers[name + "norm0"] = torch.nn.BatchNorm1d(num_features=hidden)
    layers[name + "relu0"] = torch.nn.LeakyReLU()
    layers[name + "conv_out"] = torch.nn.Conv1d(hidden, 1, kernel_size=1)
    return layers


class _EdgeRumorGCN(torch.nn.Module):
    _edge_key = "edge_index"
    _flag = "edge_infer_td"

    def __init__(self, args):
        super().__init__()
        self.args = args
        hid = args.hidden_features
        if hid != L.H or args.output_features != L.H:
            raise L.BigcnError(f"bigcn_b200 kernels are specialised for hidden_features = output_features = {L.H}")
        self.conv1 = GCNConv(args.input_features, hid)
        self.conv2 = GCNConv(args.input_features + hid, args.output_features)
        self.device = getattr(args, "device", None)
        self.sim_network = torch.nn.Sequential(_create_network(hid, "sim_val"))
        self.W_mean = torch.nn.Sequential(_create_network(hid, "W_mean"))
        self.W_bias = torch.nn.Sequential(_create_network(hid, "W_bias"))
        self.B_mean = torch.nn.Sequential(_create_network(hid, "B_mean"))
        self.B_bias = torch.nn.Sequential(_create_network(hid, "B_bias"))
        self.fc1 = torch.nn.Linear(hid, args.edge_num, bias=False)
        self.fc2 = torch.nn.Linear(hid, args.edge_num, bias=False)
        self.dropout = torch.nn.Dropout(args.dropout)
        self.eval_loss = torch.nn.KLDivLoss(reduction="batchmean")
        self.bn1 = torch.nn.BatchNorm1d(hid + args.input_features)
        self.last_flags = None

    def check_inputs(self):
        """Raise if the last forward saw an invalid graph, or a SparseX x that conv1 flagged (synchronises)."""
        pending = [f for f in (self.conv1.last_flags, self.last_flags) if f is not None]
        self.conv1.last_flags = self.last_flags = None
        for flags in pending:
            raise_on_flags(flags)

    def forward(self, data):
        x1 = ebgcn_x(data.x)                                            # :62-63
        edge_index = getattr(data, self._edge_key)
        x = self.conv1(x1, edge_index)                                  # :64
        if getattr(self.args, self._flag, False):
            edge_loss, edge_pred = self.edge_infer(x, edge_index)       # :67-70
        else:
            edge_loss, edge_pred = None, None
        num_graphs = int(data.rootindex.numel())
        node_ptr = torch.empty(num_graphs + 1, dtype=torch.int32, device=x1.device)
        flags = torch.zeros(1, dtype=torch.int32, device=x1.device)
        bn = self.bn1
        h = EBGCNConv2Function.apply(x, edge_pred, bn.weight, bn.bias, self.conv2.lin.weight, self.conv2.bias, x1,
                                     edge_index, data.batch, data.rootindex, bn, self.conv2.deg_by, node_ptr, flags)
        self.last_flags = flags
        # cat(h, x[root]) + scatter_mean (:86-92); x[root] is the detached copy.copy of :65
        return torch.ops.bigcn_b200.readout(h, x.detach(), node_ptr, data.rootindex, data.batch), edge_loss

    def edge_infer(self, x, edge_index):
        """EBGCN.py:95-117, unchanged (including its ``row - 1`` / ``col - 1`` indexing)."""
        row, col = edge_index[0], edge_index[1]
        x_i = x[row - 1].unsqueeze(2)
        x_j = x[col - 1].unsqueeze(1)
        x_ij = torch.abs(x_i - x_j)
        sim_val = self.sim_network(x_ij)
        edge_pred = torch.sigmoid(self.fc1(sim_val))
        w_mean, w_bias = self.W_mean(x_ij), self.W_bias(x_ij)
        b_mean, b_bias = self.B_mean(x_ij), self.B_bias(x_ij)
        logit_mean = w_mean * sim_val + b_mean
        logit_var = torch.relu(torch.log((sim_val ** 2) * torch.exp(w_bias) + torch.exp(b_bias)))
        edge_y = torch.sigmoid(torch.normal(logit_mean, logit_var))
        edge_y = self.fc2(edge_y)
        logp_x = F.log_softmax(edge_pred, dim=-1)
        p_y = F.softmax(edge_y, dim=-1)
        return self.eval_loss(logp_x, p_y), torch.mean(edge_pred, dim=-1).squeeze(1)


class TDrumorGCN(_EdgeRumorGCN):
    """EBGCN.py:23-117."""
    _edge_key, _flag = "edge_index", "edge_infer_td"


class BUrumorGCN(_EdgeRumorGCN):
    """EBGCN.py:120-214."""
    _edge_key, _flag = "BU_edge_index", "edge_infer_bu"


class EBGCN(torch.nn.Module):
    """EBGCN.py:217-233: ``EBGCN(args)``, ``forward(data) -> (log-probs [B, num_class], TD_edge_loss, BU_edge_loss)``
    (the edge losses are None when that direction's edge inference is off)."""

    def __init__(self, args):
        super().__init__()
        self.args = args
        self.TDrumorGCN = TDrumorGCN(args)
        self.BUrumorGCN = BUrumorGCN(args)
        self.fc = torch.nn.Linear((args.hidden_features + args.output_features) * 2, args.num_class)

    def check_inputs(self):
        """Raise if the last forward saw an invalid graph (synchronises)."""
        self.TDrumorGCN.check_inputs()
        self.BUrumorGCN.check_inputs()

    def forward(self, data):
        TD_x, TD_edge_loss = self.TDrumorGCN(data)
        BU_x, BU_edge_loss = self.BUrumorGCN(data)
        self.x = torch.cat((BU_x, TD_x), 1)
        out = HeadFunction.apply(self.x, self.fc.weight, self.fc.bias)
        return out, TD_edge_loss, BU_edge_loss
