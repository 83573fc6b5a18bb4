"""The building blocks of the path as ``torch.library`` operators, namespace ``bigcn_b200::``
(SURVEY.md 8b: "what a native replacement must export").  CUDA only: there is no CPU kernel behind
any of them, so a CPU tensor fails in the dispatcher (NotImplementedError) -- no fallback.  Each op
is a thin call into libbigcn_b200.so on the current stream; outputs come from torch's allocator.

  graph_prep(edge_index, num_nodes, batch?, num_graphs, deg_by)
        -> (in_ptr, in_idx, out_ptr, out_idx, deg, dis, rowsum, node_ptr, flags, in_long, out_long)
        gcn_norm / add_remaining_self_loops structure [torch_geometric], BiGCN_Twitter.py:42,56,92,105
  xw(x, w, mode) -> [N,64]            GCNConv.lin;  backward: xw_wgrad(x, t, mode) -> [64,K] and, when x wants a
        gradient, xw_dgrad(t, w, mode) -> [N,K]
  propagate(h, in_ptr, in_idx, out_ptr, out_idx, dis, num_edges, in_long?, out_long?, bias?, relu) -> [N,64]
        MessagePassing.propagate + bias (+ relu); backward: the transposed CSR for dh, column sums for dbias
  readout(h2, h1, node_ptr, rootindex, batch) -> [B,128]   second root-extend + scatter_mean (:58-65);
        backward: readout_backward (the mean's gradient to h2; h1[root] is detached as in the reference)

``torch.ops.bigcn_b200.xw(x, w, "fp32")`` etc.; ``conv(x, edge_index)`` of torch_geometric is
``propagate(xw(x, W), *graph_prep(...))``, which is how tests/test_gpu_torch_ops.py checks them
against the oracle with autograd."""
from __future__ import annotations

from typing import Optional, Tuple

import torch
from torch import Tensor
from torch.library import custom_op

from . import _lib as L
from . import ops
from ._lib import H, check, lib
from .ops import _p, _stream, _f32, _i64, _x_for

T11 = Tuple[Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, Tensor]


@custom_op("bigcn_b200::graph_prep", mutates_args=(), device_types="cuda")
def graph_prep(edge_index: Tensor, num_nodes: int, batch: Optional[Tensor], num_graphs: int, deg_by: str) -> T11:
    graphs, node_ptr, flags = ops.graph_prep([edge_index], num_nodes, batch, num_graphs, deg_by)
    g = graphs[0]
    if node_ptr is None:
        node_ptr = torch.empty(0, dtype=torch.int32, device=edge_index.device)
    return (g["in_ptr"], g["in_idx"], g["out_ptr"], g["out_idx"], g["deg"], g["dis"], g["rowsum"], node_ptr, flags,
            g["in_long"], g["out_long"])


@graph_prep.register_fake
def _(edge_index, num_nodes, batch, num_graphs, deg_by):
    e = edge_index.shape[1]
    i32 = dict(dtype=torch.int32, device=edge_index.device)
    f32 = dict(dtype=torch.float32, device=edge_index.device)
    nl = lib().bigcn_long_ws_ints(int(e)) if isinstance(e, int) else e
    return (torch.empty(num_nodes + 1, **i32), torch.empty(e, **i32), torch.empty(num_nodes + 1, **i32),
            torch.empty(e, **i32), torch.empty(num_nodes, **i32), torch.empty(num_nodes, **f32),
            torch.empty(num_nodes, **f32), torch.empty(num_graphs + 1 if batch is not None else 0, **i32),
            torch.empty(1, **i32), torch.empty(nl, **i32), torch.empty(nl, **i32))


# ---------------------------------------------------------------------------------- X W^T
@custom_op("bigcn_b200::xw", mutates_args=(), device_types="cuda")
def xw(x: Tensor, w: Tensor, mode: str) -> Tensor:
    return ops.xw(x, [w], mode)


@xw.register_fake
def _(x, w, mode):
    return x.new_empty(x.shape[0], H, dtype=torch.float32)   # fp32 whatever x is (bf16 in mode 'bf16')


@custom_op("bigcn_b200::xw_wgrad", mutates_args=(), device_types="cuda")
def xw_wgrad(x: Tensor, t: Tensor, mode: str) -> Tensor:
    L.require_device()
    x, t = _x_for(x, mode), _f32(t)
    n, k = x.shape
    m = L.GEMM_MODE["fp32" if mode == "sparse" else mode]
    dw = torch.empty(H, k, dtype=torch.float32, device=x.device)
    nscr = lib().bigcn_xw_wgrad_scratch_floats(n, k, 1)
    scr = torch.empty(nscr, dtype=torch.float32, device=x.device)
    check(lib().bigcn_xw_wgrad(_p(x), n, k, _p(t), 1, _p(dw), None, k, m, _p(scr), _stream()), "xw_wgrad")
    return dw


@xw_wgrad.register_fake
def _(x, t, mode):
    return x.new_empty(H, x.shape[1], dtype=torch.float32)


@custom_op("bigcn_b200::xw_dgrad", mutates_args=(), device_types="cuda")
def xw_dgrad(g: Tensor, w: Tensor, mode: str) -> Tensor:
    # the input gradient g @ w of xw: bf16 in mode 'bf16' (the dtype xw reads there), fp32 otherwise
    return ops.x_dgrad(g, [w], torch.bfloat16 if mode == "bf16" else torch.float32)


@xw_dgrad.register_fake
def _(g, w, mode):
    return g.new_empty(g.shape[0], w.shape[1], dtype=torch.bfloat16 if mode == "bf16" else torch.float32)


def _xw_setup(ctx, inputs, output):
    x, w, mode = inputs
    ctx.save_for_backward(x, w)
    ctx.mode = mode


def _xw_backward(ctx, g):
    x, w = ctx.saved_tensors
    g = g.contiguous()
    dx = torch.ops.bigcn_b200.xw_dgrad(g, w, ctx.mode) if ctx.needs_input_grad[0] else None
    return dx, torch.ops.bigcn_b200.xw_wgrad(x, g, ctx.mode), None


xw.register_autograd(_xw_backward, setup_context=_xw_setup)


# ---------------------------------------------------------------------------------- propagate
@custom_op("bigcn_b200::propagate", mutates_args=(), device_types="cuda")
def propagate(h: Tensor, in_ptr: Tensor, in_idx: Tensor, out_ptr: Tensor, out_idx: Tensor, dis: Tensor, num_edges: int,
              in_long: Optional[Tensor], out_long: Optional[Tensor], bias: Optional[Tensor], relu: bool) -> Tensor:
    g = dict(in_ptr=in_ptr, in_idx=in_idx, in_long=in_long, dis=dis, E=int(num_edges))
    return ops.propagate(g, h, bias, relu)


@propagate.register_fake
def _(h, in_ptr, in_idx, out_ptr, out_idx, dis, num_edges, in_long, out_long, bias, relu):
    return h.new_empty(h.shape[0], H)


@custom_op("bigcn_b200::propagate_transposed", mutates_args=(), device_types="cuda")
def propagate_transposed(g: Tensor, out_ptr: Tensor, out_idx: Tensor, dis: Tensor, num_edges: int,
                         out_long: Optional[Tensor]) -> Tensor:
    gr = dict(out_ptr=out_ptr, out_idx=out_idx, out_long=out_long, dis=dis, E=int(num_edges))
    return ops.propagate(gr, g, None, False, transpose=True)


@propagate_transposed.register_fake
def _(g, out_ptr, out_idx, dis, num_edges, out_long):
    return g.new_empty(g.shape[0], H)


@custom_op("bigcn_b200::colsum64", mutates_args=(), device_types="cuda")
def colsum64(g: Tensor) -> Tensor:
    L.require_device()
    g = _f32(g)
    n = g.shape[0]
    out = torch.empty(H, dtype=torch.float32, device=g.device)
    scr = torch.empty(lib().bigcn_colsum64_scratch_floats(n), dtype=torch.float32, device=g.device)
    check(lib().bigcn_colsum64(_p(g), n, _p(out), _p(scr), _stream()), "colsum64")
    return out


@colsum64.register_fake
def _(g):
    return g.new_empty(H)


def _prop_setup(ctx, inputs, output):
    h, in_ptr, in_idx, out_ptr, out_idx, dis, num_edges, in_long, out_long, bias, relu = inputs
    ctx.save_for_backward(out_ptr, out_idx, dis, out_long, output if relu else None)
    ctx.num_edges, ctx.has_bias = num_edges, bias is not None


def _prop_backward(ctx, g):
    out_ptr, out_idx, dis, out_long, out = ctx.saved_tensors
    g = g.contiguous()
    if out is not None:
        g = g * (out > 0)                          # relu'
    dh = torch.ops.bigcn_b200.propagate_transposed(g, out_ptr, out_idx, dis, ctx.num_edges, out_long)
    db = torch.ops.bigcn_b200.colsum64(g) if ctx.has_bias else None
    return dh, None, None, None, None, None, None, None, None, db, None


propagate.register_autograd(_prop_backward, setup_context=_prop_setup)


# ---------------------------------------------------------------------------------- readout
@custom_op("bigcn_b200::readout", mutates_args=(), device_types="cuda")
def readout(h2: Tensor, h1: Tensor, node_ptr: Tensor, rootindex: Tensor, batch: Tensor) -> Tensor:
    return ops.readout(h2, h1, node_ptr, rootindex)


@readout.register_fake
def _(h2, h1, node_ptr, rootindex, batch):
    return h2.new_empty(rootindex.shape[0], 2 * H)


@custom_op("bigcn_b200::readout_backward", mutates_args=(), device_types="cuda")
def readout_backward(grad_feat: Tensor, node_ptr: Tensor, batch: Tensor) -> Tensor:
    L.require_device()
    g, batch = _f32(grad_feat), _i64(batch)
    n, b = batch.shape[0], g.shape[0]
    out = torch.empty(n, H, dtype=torch.float32, device=g.device)
    check(lib().bigcn_readout_backward(_p(g), g.stride(0), _p(node_ptr), _p(batch), n, b, _p(out), _stream()),
          "readout_backward")
    return out


@readout_backward.register_fake
def _(grad_feat, node_ptr, batch):
    return grad_feat.new_empty(batch.shape[0], H)


def _readout_setup(ctx, inputs, output):
    h2, h1, node_ptr, rootindex, batch = inputs
    ctx.save_for_backward(node_ptr, batch)


def _readout_backward(ctx, g):
    node_ptr, batch = ctx.saved_tensors
    # only the scatter_mean half carries a gradient: the reference's copy.copy detaches h1[root] (:44,58-63)
    return torch.ops.bigcn_b200.readout_backward(g.contiguous(), node_ptr, batch), None, None, None, None


readout.register_autograd(_readout_backward, setup_context=_readout_setup)
