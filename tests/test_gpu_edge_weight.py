"""Edge weights in the BiGCN modules: ``data.edge_weight`` (TD) and ``data.BU_edge_weight`` (BU) go to both convs of
their direction as ``GCNConv(x, edge_index, edge_weight)``, and autograd returns their gradients from the fused path.
The reference for every value is the fp64 oracle: oracle.bigcn_oracle's modules with the direction's weights passed to
both of its GCNConvs (``weighted_oracle`` below), the Philox dropout mask injected in train mode."""
import copy
import types

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import bigcn_oracle, gcn_oracle
from bigcn_b200.data import make_batch

K = 64


class Data(types.SimpleNamespace):
    """A duck-typed batch (the modules read attributes); unlike SimpleNamespace itself it takes weak references, which
    the inference path's graph cache keeps to the batches it has seen."""


def rel_err(got, want):
    want = want.detach().cpu().double()
    got = got.detach().cpu().double()
    return float((got - want).abs().max()) / max(float(want.abs().max()), 1e-30)


def masks_for(seed, n, k):
    return [torch.from_numpy(gcn_oracle.dropout_keep_mask(seed, d, np.arange(n), 64 + k, 0.5)) for d in (0, 1)]


def edge_case_batch(seed, train, k=K):
    """Trees chosen for the corners of the weighted path: single-node trees, a 60-node star (its root is a BU hub row
    with more than 32 in-edges), random trees; in train mode TD and BU lose different edges (DropEdge); each list gets
    a self-loop edge and a duplicate of an existing edge.  Weights: uniform in [0.1, 2) with every tenth set to 0."""
    rng = np.random.default_rng(seed)
    sizes = [1, 60, 12, 7, 20, 1, 9, 33]
    td, off = [], 0
    for t, n in enumerate(sizes):
        for i in range(1, n):
            p = 0 if t == 1 else int(rng.integers(0, i))
            td.append((off + p, off + i))
        off += n
    n_nodes = off
    td = np.array(td, dtype=np.int64).T
    bu = td[::-1].copy()
    if train:
        td = td[:, rng.random(td.shape[1]) >= 0.2]
        bu = bu[:, rng.random(bu.shape[1]) >= 0.2]
    extra_node = sizes[0] + sizes[1] + 3       # a node of the third tree
    lists = []
    for ei in (td, bu):
        ei = np.concatenate([ei, [[extra_node], [extra_node]], ei[:, 2:3]], axis=1)
        lists.append(ei)
    x = np.zeros((n_nodes, k), dtype=np.float32)
    for i in range(n_nodes):
        cols = rng.choice(k, 5, replace=False)
        x[i, cols] = rng.integers(1, 4, 5)
    batch = np.repeat(np.arange(len(sizes)), sizes)
    root = np.concatenate([[0], np.cumsum(sizes)[:-1]])
    ws = []
    for ei in lists:
        w = rng.uniform(0.1, 2.0, ei.shape[1]).astype(np.float32)
        w[::10] = 0.0
        w[-2] = 1.5                             # the self-loop edge: the node's loop weight
        ws.append(w)
    return types.SimpleNamespace(
        x=torch.from_numpy(x), edge_index=torch.from_numpy(lists[0]), BU_edge_index=torch.from_numpy(lists[1]),
        batch=torch.from_numpy(batch), rootindex=torch.from_numpy(root.astype(np.int64)),
        y=torch.from_numpy(rng.integers(0, 4, len(sizes))), w=ws)


def _weighted_forward(self, data, keep=None):
    """bigcn_oracle._RumorGCN.forward statement by statement, with ``getattr(data, self.weight_attr, None)`` handed to
    conv1 and conv2 as PyG's ``GCNConv(x, edge_index, edge_weight)`` takes it (the oracle's GCNConv already does);
    absent means unweighted."""
    x, edge_index = data.x, getattr(data, self.edge_attr)
    dtype = self.conv1.lin.weight.dtype
    ew = getattr(data, self.weight_attr, None)
    if ew is not None:
        ew = ew.to(dtype)
    x1 = copy.copy(x.to(dtype))
    h = self.conv1(x1, edge_index, ew)
    h2 = h.detach()                                                # copy.copy at :44 cuts this root-extend
    h = torch.cat((h, self._root_extend(x1, data)), 1)
    h = F.relu(h)
    h = bigcn_oracle._dropout(h, self.p, self.training, keep)
    h = self.conv2(h, edge_index, ew)
    h = F.relu(h)
    h = torch.cat((h, self._root_extend(h2, data)), 1)
    return gcn_oracle.scatter_mean(h, data.batch, int(data.rootindex.numel()))


class WeightedTD(bigcn_oracle.TDrumorGCN):
    weight_attr = "edge_weight"
    forward = _weighted_forward


class WeightedBU(bigcn_oracle.BUrumorGCN):
    weight_attr = "BU_edge_weight"
    forward = _weighted_forward


def oracle(k, seed, deg_by="target"):
    torch.manual_seed(seed)
    ref = bigcn_oracle.BiGCN(k, 64, 64, deg_by=deg_by)
    with torch.no_grad():
        for p in ref.parameters():
            if p.dim() == 1:
                p.uniform_(-0.1, 0.1)
    ref.TDrumorGCN.__class__ = WeightedTD
    ref.BUrumorGCN.__class__ = WeightedBU
    return ref.double()


def test_weighted_oracle_without_weights_is_the_oracle():
    """CPU: with no weight attribute, and with all-ones weights, the weighted restatement gives the packaged oracle's
    log-probs exactly (eval and train with an explicit mask)."""
    for train in (False, True):
        b = edge_case_batch(7, train)
        ref = oracle(K, 2)
        plain = bigcn_oracle.BiGCN(K, 64, 64).double()
        plain.load_state_dict(ref.state_dict())
        keep = masks_for(11, b.x.shape[0], K) if train else [None, None]
        ref.train(train)
        plain.train(train)
        d = types.SimpleNamespace(**vars(b))
        with torch.no_grad():
            want = plain(d, keep_td=keep[0], keep_bu=keep[1])
            assert torch.equal(ref(d, keep_td=keep[0], keep_bu=keep[1]), want)
            d.edge_weight, d.BU_edge_weight = (torch.ones(len(w), dtype=torch.float64) for w in b.w)
            assert torch.equal(ref(d, keep_td=keep[0], keep_bu=keep[1]), want)


def on_device(b, dev, td_w=None, bu_w=None):
    d = Data(**{k: getattr(b, k).to(dev) for k in ("x", "edge_index", "BU_edge_index", "batch", "rootindex", "y")})
    if td_w is not None:
        d.edge_weight = td_w
    if bu_w is not None:
        d.BU_edge_weight = bu_w
    return d


def run_model(m, d, train):
    for mod in (m.TDrumorGCN, m.BUrumorGCN):
        mod._calls = 0                          # the same dropout seed in every run
    m.zero_grad(set_to_none=True)
    out = m(d)
    loss = F.nll_loss(out, d.y)
    loss.backward()
    m.check_inputs()
    return out.detach().clone(), loss.detach().clone(), [p.grad.clone() for p in m.parameters()]


def ref_run(ref, b, train, seed, td_w, bu_w):
    d = types.SimpleNamespace(**vars(b))
    if td_w is not None:
        d.edge_weight = td_w
    if bu_w is not None:
        d.BU_edge_weight = bu_w
    keep = masks_for(seed, b.x.shape[0], b.x.shape[1]) if train else [None, None]
    ref.train(train)
    ref.zero_grad(set_to_none=True)
    out = ref(d, keep_td=keep[0], keep_bu=keep[1])
    F.nll_loss(out, b.y).backward()
    return out


# ---------------------------------------------------------------------------------------------- all-ones weights
@pytest.mark.gpu
@pytest.mark.parametrize("train", [False, True])
@pytest.mark.parametrize("mode", ["sparse", "tf32x3", "bf16"])
def test_ones_equal_unweighted(dev, mode, train):
    """Weights of 1 on both directions give the unweighted path's log-probs, loss and ten parameter gradients bit for
    bit: (dis_r * 1) * dis_c = dis_r * dis_c, and the weighted degree is a float sum of exact integers.  With the
    weights requiring a gradient too (the backward then keeps X W1^T and conv2's input apart)."""
    import bigcn_b200
    k = 5000 if mode == "sparse" else 256
    b = make_batch("twitter15", 16, seed=3, train=train, in_feats=k)
    m = bigcn_b200.BiGCN(k, 64, 64, dev, gemm_mode=mode).to(dev)
    m.load_state_dict(oracle(k, 1).float().state_dict())
    m.train(train)
    d0 = on_device(b, dev)
    if mode == "bf16":
        d0.x = d0.x.to(torch.bfloat16).contiguous()
    base = run_model(m, d0, train)
    for grad in (False, True):
        ones = [torch.ones(e.shape[1], device=dev, requires_grad=grad) for e in (b.edge_index, b.BU_edge_index)]
        d1 = on_device(b, dev, *ones)
        d1.x = d0.x
        got = run_model(m, d1, train)
        assert torch.equal(base[0], got[0]) and torch.equal(base[1], got[1])
        for (name, _), g0, g1 in zip(m.named_parameters(), base[2], got[2]):
            assert torch.equal(g0, g1), (name, grad)
        if grad:
            assert all(w.grad is not None and bool(torch.isfinite(w.grad).all()) for w in ones)


# ---------------------------------------------------------------------------------------------- oracle parity
@pytest.mark.gpu
@pytest.mark.parametrize("train", [False, True])
@pytest.mark.parametrize("deg_by", ["target", "source"])
@pytest.mark.parametrize("mode", ["sparse", "tf32x3"])
def test_weighted_matches_oracle(dev, mode, deg_by, train):
    """Random non-negative weights (zeros, a self-loop and a duplicate edge in each list, asymmetric DropEdge in train
    mode, a BU hub row, single-node trees) against the fp64 oracle's autograd: log-probs 1e-5, parameter gradients
    1e-4 and both weight gradients 1e-4 of max|ref|."""
    import bigcn_b200
    b = edge_case_batch(7, train)
    ref = oracle(K, 2, deg_by)
    m = bigcn_b200.BiGCN(K, 64, 64, dev, gemm_mode=mode, deg_by=deg_by).to(dev)
    m.load_state_dict(ref.state_dict())
    m.train(train)
    tw, bw = (torch.tensor(w, device=dev, requires_grad=True) for w in b.w)
    assert int((b.BU_edge_index[1] == 1).sum()) > 32      # the star's root: a hub row of the by-target BU CSR
    out, _, grads = run_model(m, on_device(b, dev, tw, bw), train)
    rtw, rbw = (torch.tensor(w, dtype=torch.float64, requires_grad=True) for w in b.w)
    want = ref_run(ref, b, train, m.TDrumorGCN.last_seed, rtw, rbw)
    assert rel_err(out, want) <= 1e-5
    for (name, _), g, q in zip(m.named_parameters(), grads, ref.parameters()):
        assert rel_err(g, q.grad) <= 1e-4, name
    assert rel_err(tw.grad, rtw.grad) <= 1e-4
    assert rel_err(bw.grad, rbw.grad) <= 1e-4
    # the self-loop edge (second to last) receives its node's loop gradient, the duplicate its own
    assert float(rtw.grad[-2].abs()) > 0 and float(tw.grad[-2].abs()) > 0


@pytest.mark.gpu
def test_edge_grad_deterministic(dev):
    """Two backward passes on one batch give bit-identical weight gradients."""
    import bigcn_b200
    b = edge_case_batch(11, True)
    m = bigcn_b200.BiGCN(K, 64, 64, dev, gemm_mode="sparse").to(dev)
    m.load_state_dict(oracle(K, 4).float().state_dict())
    m.train()
    res = []
    for _ in range(2):
        tw, bw = (torch.tensor(w, device=dev, requires_grad=True) for w in b.w)
        run_model(m, on_device(b, dev, tw, bw), True)
        res.append((tw.grad, bw.grad))
    assert torch.equal(res[0][0], res[1][0]) and torch.equal(res[0][1], res[1][1])


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["td", "bu"])
def test_one_direction_weighted(dev, which):
    """A weight on one direction only: that direction weighted, the other unweighted, against the oracle; and the
    direction modules on their own (TDrumorGCN with data.edge_weight, BUrumorGCN with data.BU_edge_weight)."""
    import bigcn_b200
    b = edge_case_batch(5, False)
    ref = oracle(K, 6)
    m = bigcn_b200.BiGCN(K, 64, 64, dev, gemm_mode="tf32x3").to(dev).eval()
    m.load_state_dict(ref.state_dict())
    w = torch.tensor(b.w[0 if which == "td" else 1], device=dev, requires_grad=True)
    args = (w, None) if which == "td" else (None, w)
    out, _, grads = run_model(m, on_device(b, dev, *args), False)
    rw = torch.tensor(b.w[0 if which == "td" else 1], dtype=torch.float64, requires_grad=True)
    want = ref_run(ref, b, False, 0, *((rw, None) if which == "td" else (None, rw)))
    assert rel_err(out, want) <= 1e-5
    for (name, _), g, q in zip(m.named_parameters(), grads, ref.parameters()):
        assert rel_err(g, q.grad) <= 1e-4, name
    assert rel_err(w.grad, rw.grad) <= 1e-4
    # the direction module alone
    mod = m.TDrumorGCN if which == "td" else m.BUrumorGCN
    rmod = ref.TDrumorGCN if which == "td" else ref.BUrumorGCN
    w.grad = None
    rw.grad = None
    feat = mod(on_device(b, dev, *args))
    feat.square().sum().backward()
    d = types.SimpleNamespace(**vars(b))
    setattr(d, "edge_weight" if which == "td" else "BU_edge_weight", rw)
    rfeat = rmod(d)
    rfeat.square().sum().backward()
    assert rel_err(feat, rfeat) <= 1e-5
    assert rel_err(w.grad, rw.grad) <= 1e-4


@pytest.mark.gpu
@pytest.mark.parametrize("train", [False, True])
def test_nograd_and_replay_equal_autograd(dev, train):
    """torch.no_grad() inference with weights (a plain run, then a captured CUDA graph and its replay) gives the
    autograd forward's log-probs bit for bit; a new weight tensor is a new graph key."""
    import bigcn_b200
    b = edge_case_batch(9, False)
    m = bigcn_b200.BiGCN(K, 64, 64, dev, gemm_mode="tf32x3", graphs=True).to(dev)
    m.load_state_dict(oracle(K, 8).float().state_dict())
    m.train(train)
    m.TDrumorGCN.p = m.BUrumorGCN.p = 0.0 if train else 0.5   # graphs replay train mode only without dropout
    tw, bw = (torch.tensor(w, device=dev) for w in b.w)
    d = on_device(b, dev, tw, bw)
    want = m(d).detach().clone()
    with torch.no_grad():
        outs = [m(d).clone() for _ in range(3)]
    m.check_inputs()
    assert len(m._graphs) == 1
    for o in outs:
        assert torch.equal(o, want)
    d.BU_edge_weight = bw * 2
    with torch.no_grad():
        other = m(d).clone()
    assert not torch.equal(other, want)


@pytest.mark.gpu
def test_bad_weights_raise(dev):
    """Wrong shape, non-floating dtype or a CPU tensor raise BigcnError; a NaN weight is reported by the device flags;
    other floating dtypes are cast; FusedTrainer refuses a weighted batch."""
    import bigcn_b200
    b = edge_case_batch(3, False)
    m = bigcn_b200.BiGCN(K, 64, 64, dev, gemm_mode="sparse").to(dev).eval()
    e = b.edge_index.shape[1]
    for bad in (torch.ones(e + 1, device=dev), torch.ones(e, 1, device=dev), torch.ones(e, dtype=torch.int64, device=dev),
                torch.ones(e)):
        with pytest.raises(bigcn_b200.BigcnError):
            m(on_device(b, dev, bad))
        with torch.no_grad(), pytest.raises(bigcn_b200.BigcnError):
            m(on_device(b, dev, bad))
    nan = torch.ones(e, device=dev)
    nan[3] = float("nan")
    m(on_device(b, dev, nan))
    with pytest.raises(IndexError, match="edge weight"):
        m.check_inputs()
    w64 = torch.tensor(b.w[0], dtype=torch.float64, device=dev, requires_grad=True)
    w32 = torch.tensor(b.w[0], device=dev, requires_grad=True)
    o64 = m(on_device(b, dev, w64))
    o32 = m(on_device(b, dev, w32))
    assert torch.equal(o64, o32)
    o64.sum().backward()
    assert w64.grad.dtype == torch.float64
    m.train()
    tr = bigcn_b200.FusedTrainer(m, lr=5e-4, weight_decay=1e-4)
    with pytest.raises(bigcn_b200.BigcnError, match="edge-weighted"):
        tr.step(on_device(b, dev, w32.detach()), seed=1)
