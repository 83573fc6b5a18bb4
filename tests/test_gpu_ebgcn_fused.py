"""bigcn_b200.EBGCN (bn1 + conv2 per tree on the device, csrc/ebgcn.cu) against the materialising harness
(tests/ebgcn_harness.py: the same modules with root_extend, cat and torch's BatchNorm1d over N x (64 + K)), against
the fp64 oracle module of test_gpu_ebgcn.py, and on its own (memory, determinism, training)."""
import copy
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from test_gpu_ebgcn import OracleDir

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")
TIGHT = ("conv1.lin.weight", "conv2.lin.weight", "conv2.bias", "bn1.weight", "bn1.bias", "conv_out.weight",
         "fc1.weight", "fc.weight", "fc.bias")


@pytest.fixture(autouse=True)
def _no_tf32(monkeypatch):
    # the edge-inference sub-networks are plain torch modules: keep cuDNN / cuBLAS from running them in TF32
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)
    monkeypatch.setattr(torch.backends.cuda.matmul, "allow_tf32", False)


def _args(k, infer):
    return SimpleNamespace(input_features=k, hidden_features=64, output_features=64, edge_num=2, dropout=0.5,
                           num_class=4, edge_infer_td=infer, edge_infer_bu=infer, device=DEV)


def _pair(k, infer, seed=4):
    import bigcn_b200
    import ebgcn_harness
    torch.manual_seed(seed)
    ref = ebgcn_harness.EBGCN(_args(k, infer)).to(DEV)
    new = bigcn_b200.EBGCN(_args(k, infer)).to(DEV)
    new.load_state_dict(ref.state_dict())
    # the harness's conv2 takes its N x (64 + K) input with the exact fp32 product: in 'auto' it would pick tf32x3 for
    # the dense BatchNorm output, and at K = 5000 that alone puts BU conv1's weight gradient 5e-4 away from the fp64
    # result (the fp32 product: 5e-6), so the harness would not be a reference at the tight bar
    for d in (ref.TDrumorGCN, ref.BUrumorGCN):
        d.conv2.gemm_mode = "fp32"
    return ref, new


def _batch(shape, n_trees, seed, k, sizes=None):
    from bigcn_b200.data import make_batch
    return make_batch(shape, n_trees, seed=seed, train=True, in_feats=k, sizes=sizes).to(DEV)


def _step(m, bd, seed, edge_w=0.2):
    """one forward + nll (+ the edge losses) + backward from a fixed torch seed; returns (log-probs, losses)"""
    torch.manual_seed(seed)
    out, tdl, bul = m(bd)
    loss = F.nll_loss(out, bd.y)
    for el in (tdl, bul):
        if el is not None:
            loss = loss + edge_w * el
    loss.backward()
    return out.detach(), (tdl, bul), loss.detach()


def _grad_errors(ref, new):
    theirs = dict(ref.named_parameters())
    gmax = max(float(p.grad.abs().max()) for p in ref.parameters() if p.grad is not None)
    errs = {}
    for name, p in new.named_parameters():
        q = theirs[name]
        if q.grad is None:
            assert p.grad is None or float(p.grad.abs().max()) == 0.0, name
            continue
        assert p.grad is not None, name
        scale = max(float(q.grad.abs().max()), 1e-3 * gmax)
        errs[name] = float((p.grad - q.grad).abs().max()) / scale
    return errs


def _check_grads(ref, new, min_count):
    errs = _grad_errors(ref, new)
    assert len(errs) >= min_count, sorted(errs)
    bad = {k: v for k, v in errs.items() if v >= (5e-4 if k.endswith(TIGHT) else 5e-3)}
    assert not bad, bad


def _check_bn_buffers(ref, new):
    for d in ("TDrumorGCN", "BUrumorGCN"):
        a, b = getattr(ref, d).bn1, getattr(new, d).bn1
        assert int(a.num_batches_tracked) == int(b.num_batches_tracked)
        torch.testing.assert_close(b.running_mean, a.running_mean, rtol=1e-5, atol=1e-6)
        torch.testing.assert_close(b.running_var, a.running_var, rtol=1e-5, atol=1e-6)


CASES = [("twitter15", 5, 40), ("pheme", 24, 768), ("twitter16", 128, 5000)]


@pytest.mark.parametrize("shape,n_trees,k", CASES, ids=["K40", "K768", "K5000"])
@pytest.mark.parametrize("infer", [True, False], ids=["infer", "plain"])
@pytest.mark.parametrize("train", [True, False], ids=["train", "eval"])
def test_matches_harness(shape, n_trees, k, infer, train):
    ref, new = _pair(k, infer)
    bd = _batch(shape, n_trees, 21, k)
    for m in (ref, new):
        m.train(train)
    want, wl, _ = _step(ref, bd, 7)
    got, gl, _ = _step(new, bd, 7)
    assert float((got - want).abs().max()) <= 5e-5 * float(want.abs().max())
    for a, b in zip(wl, gl):
        if infer:
            assert abs(float(a) - float(b)) <= 1e-5 * max(1.0, abs(float(a)))
        else:
            assert a is None and b is None
    _check_grads(ref, new, 20 if infer else 12)
    _check_bn_buffers(ref, new)
    new.check_inputs()


def test_eval_uses_running_statistics():
    """a few training steps move the running statistics; eval mode then normalises with them, as torch does"""
    ref, new = _pair(768, False)
    for m in (ref, new):
        m.train()
    for s in range(3):
        bd = _batch("pheme", 24, 30 + s, 768)
        for m in (ref, new):
            m.zero_grad()
            _step(m, bd, s)
    _check_bn_buffers(ref, new)
    assert int(new.TDrumorGCN.bn1.num_batches_tracked) == 3
    for m in (ref, new):
        m.eval()
        m.zero_grad()
    bd = _batch("pheme", 24, 99, 768)
    want, _, _ = _step(ref, bd, 5)
    got, _, _ = _step(new, bd, 5)
    assert float((got - want).abs().max()) <= 5e-5 * float(want.abs().max())
    _check_grads(ref, new, 12)
    before = new.TDrumorGCN.bn1.running_mean.clone()
    _step(new, bd, 5)
    assert torch.equal(before, new.TDrumorGCN.bn1.running_mean)      # eval leaves the buffers alone
    assert int(new.TDrumorGCN.bn1.num_batches_tracked) == 3


@pytest.mark.parametrize("infer", [True, False])
def test_matches_fp64_oracle(infer):
    """test_gpu_ebgcn.py's fp64 oracle module (reference loops, oracle GCNConv) with the library model, same bars"""
    import bigcn_b200
    from bigcn_b200.data import make_batch
    k = 40
    torch.manual_seed(4)
    m = bigcn_b200.EBGCN(_args(k, infer))
    ref_td = OracleDir(m.TDrumorGCN, "edge_index", "edge_infer_td")
    ref_bu = OracleDir(m.BUrumorGCN, "BU_edge_index", "edge_infer_bu")
    ref_fc = copy.deepcopy(m.fc)
    for r, d in ((ref_td, m.TDrumorGCN), (ref_bu, m.BUrumorGCN)):
        r.conv1.load_state_dict(d.conv1.state_dict())
        r.conv2.load_state_dict(d.conv2.state_dict())
    m = m.to(DEV).train()
    ref_td, ref_bu, ref_fc = ref_td.double(), ref_bu.double(), ref_fc.double()
    b = make_batch("twitter15", 5, seed=21, train=True, in_feats=k)
    b.x = b.x.double()
    bd = make_batch("twitter15", 5, seed=21, train=True, in_feats=k).to(DEV)
    out, tdl, bul = m(bd)
    want = F.log_softmax(ref_fc(torch.cat((ref_bu(b), ref_td(b)), 1)), dim=1)
    assert float((out.detach().cpu().double() - want.detach()).abs().max()) <= 5e-5 * float(want.abs().max())
    F.nll_loss(want, b.y).backward()
    F.nll_loss(out, bd.y).backward()
    gmax = max(float(p.grad.abs().max()) for p in list(ref_td.parameters()) + list(ref_bu.parameters()) if p.grad is not None)
    errs = {}
    for tag, ours, ref in (("TD", m.TDrumorGCN, ref_td), ("BU", m.BUrumorGCN, ref_bu)):
        theirs = dict(ref.named_parameters())
        for name, p in ours.named_parameters():
            q = theirs.get(name)
            if q is None or q.grad is None:
                continue
            scale = max(float(q.grad.abs().max()), 1e-3 * gmax)
            errs[f"{tag}.{name}"] = float((p.grad.cpu().double() - q.grad).abs().max()) / scale
    assert len(errs) >= (12 if not infer else 20)
    tight = ("conv1.lin.weight", "conv2.lin.weight", "conv2.bias", "bn1.weight", "bn1.bias", "conv_out.weight", "fc1.weight")
    bad = {k_: v for k_, v in errs.items() if v >= (5e-4 if k_.endswith(tight) else 5e-3)}
    assert not bad, bad



def test_k5000_training_matches_fp64_oracle():
    """128 Twitter16-shaped trees at K = 5000 in training mode against the fp64 oracle module: bn1's statistics and its
    dbeta / dgamma over ~31 k rows are where fp32 partial sums would show (the centred output turns a shifted mean into
    a coherent error in dW2), so every gradient is held to the tight bar"""
    import bigcn_b200
    from bigcn_b200.data import make_batch
    k = 5000
    torch.manual_seed(4)
    m = bigcn_b200.EBGCN(_args(k, False))
    ref_td = OracleDir(m.TDrumorGCN, "edge_index", "edge_infer_td")
    ref_bu = OracleDir(m.BUrumorGCN, "BU_edge_index", "edge_infer_bu")
    ref_fc = copy.deepcopy(m.fc)
    for r, d in ((ref_td, m.TDrumorGCN), (ref_bu, m.BUrumorGCN)):
        r.conv1.load_state_dict(d.conv1.state_dict())
        r.conv2.load_state_dict(d.conv2.state_dict())
    m = m.to(DEV).train()
    ref_td, ref_bu, ref_fc = ref_td.double().train(), ref_bu.double().train(), ref_fc.double()
    b = make_batch("twitter16", 128, seed=21, train=True, in_feats=k)
    b.x = b.x.double()
    bd = make_batch("twitter16", 128, seed=21, train=True, in_feats=k).to(DEV)
    want = F.log_softmax(ref_fc(torch.cat((ref_bu(b), ref_td(b)), 1)), dim=1)
    out, _, _ = m(bd)
    assert float((out.detach().cpu().double() - want.detach()).abs().max()) <= 5e-5 * float(want.abs().max())
    F.nll_loss(want, b.y).backward()
    F.nll_loss(out, bd.y).backward()
    theirs = {f"{tag}.{n}": q.grad for tag, r in (("TDrumorGCN", ref_td), ("BUrumorGCN", ref_bu))
              for n, q in r.named_parameters() if q.grad is not None}
    theirs.update({"fc.weight": ref_fc.weight.grad, "fc.bias": ref_fc.bias.grad})
    gmax = max(float(g.abs().max()) for g in theirs.values())
    errs = {n: float((p.grad.cpu().double() - theirs[n]).abs().max()) / max(float(theirs[n].abs().max()), 1e-3 * gmax)
            for n, p in m.named_parameters() if n in theirs}
    assert len(errs) >= 14
    bad = {n: v for n, v in errs.items() if v >= 5e-4}
    assert not bad, bad

# ---- the op on its own against the harness's composition, on batches built for the edge cases ----------------------
def _tree(n, k, rng, star=False):
    from bigcn_b200.data import Data, make_tree
    if not star:
        return make_tree("twitter15", n, rng, k)
    ch = np.arange(1, n)
    ei = np.stack([np.zeros(n - 1, np.int64), ch])
    x = rng.integers(0, 3, (n, k)).astype(np.float32)
    return Data(x=torch.from_numpy(x), edge_index=torch.from_numpy(ei), BU_edge_index=torch.from_numpy(ei[::-1].copy()),
                rootindex=torch.tensor([0]), y=torch.tensor([0]))


def _forest(sizes, k, seed=3, star=()):
    from bigcn_b200.data import collate
    rng = np.random.default_rng(seed)
    return collate([_tree(int(n), k, rng, i in star) for i, n in enumerate(sizes)]).to(DEV)


def _op_vs_composition(bd, k, weights, train=True, momentum=0.1, steps=1):
    """EBGCNConv2Function against relu(conv2(relu(bn1(cat(h1, x[root[batch]]))), ei, w)) built from the library's
    GCNConv and torch's BatchNorm1d (the harness's code path); every gradient, the buffers"""
    from bigcn_b200.nn import GCNConv
    from bigcn_b200.ops import EBGCNConv2Function
    torch.manual_seed(11)
    n, e = bd.x.shape[0], bd.edge_index.shape[1]
    conv_r = GCNConv(64 + k, 64, gemm_mode="fp32").to(DEV)
    conv_n = copy.deepcopy(conv_r)
    bn_r = torch.nn.BatchNorm1d(64 + k, momentum=momentum).to(DEV)
    with torch.no_grad():
        bn_r.weight.uniform_(0.5, 1.5)
        bn_r.bias.uniform_(-0.2, 0.2)
    bn_r.train(train)
    bn_n = copy.deepcopy(bn_r)
    h_base = torch.randn(n, 64, device=DEV)
    for step in range(steps):
        h_r = h_base.clone().requires_grad_(True)
        h_n = h_base.clone().requires_grad_(True)
        w_r = None if weights is None else weights.clone().requires_grad_(True)
        w_n = None if weights is None else weights.clone().requires_grad_(True)
        u = torch.cat((h_r, bd.x[bd.rootindex[bd.batch]]), 1)
        if n != 1:
            u = bn_r(u)
        want = F.relu(conv_r(F.relu(u), bd.edge_index, edge_weight=w_r))
        node_ptr = torch.empty(bd.rootindex.numel() + 1, dtype=torch.int32, device=DEV)
        flags = torch.zeros(1, dtype=torch.int32, device=DEV)
        got = EBGCNConv2Function.apply(h_n, w_n, bn_n.weight, bn_n.bias, conv_n.lin.weight, conv_n.bias, bd.x,
                                       bd.edge_index, bd.batch, bd.rootindex, bn_n, "target", node_ptr, flags)
        assert int(flags.item()) == 0
        assert torch.equal(node_ptr.long(), torch.searchsorted(bd.batch, torch.arange(node_ptr.numel(), device=DEV)))
        assert float((got - want).abs().max()) <= 5e-5 * max(float(want.abs().max()), 1e-6)
        r = torch.randn(n, 64, device=DEV)
        (want * r).sum().backward()
        (got * r).sum().backward()
        pairs = [("h1", h_n.grad, h_r.grad), ("w2", conv_n.lin.weight.grad, conv_r.lin.weight.grad),
                 ("b2", conv_n.bias.grad, conv_r.bias.grad)]
        if weights is not None:
            pairs.append(("edge_weight", w_n.grad, w_r.grad))
        if n != 1:
            pairs += [("bn.weight", bn_n.weight.grad, bn_r.weight.grad), ("bn.bias", bn_n.bias.grad, bn_r.bias.grad)]
        else:
            assert bn_n.weight.grad is None and bn_r.weight.grad is None
        gmax = max(float(b.abs().max()) for _, _, b in pairs)
        for name, a, b in pairs:
            scale = max(float(b.abs().max()), 1e-3 * gmax, 1e-12)
            assert float((a - b).abs().max()) <= 5e-4 * scale, (name, step, float((a - b).abs().max()), scale)
        for m in (conv_r, conv_n, bn_r, bn_n):
            m.zero_grad()
        assert int(bn_n.num_batches_tracked) == int(bn_r.num_batches_tracked)
        torch.testing.assert_close(bn_n.running_mean, bn_r.running_mean, rtol=1e-5, atol=1e-6)
        torch.testing.assert_close(bn_n.running_var, bn_r.running_var, rtol=1e-5, atol=1e-6)
    return bn_n


@pytest.mark.parametrize("train", [True, False])
def test_single_node_batch_skips_bn1(train):
    bd = _forest([1], 40)
    bn = _op_vs_composition(bd, 40, None, train=train)
    assert int(bn.num_batches_tracked) == 0 and float(bn.running_mean.abs().max()) == 0.0


def test_single_node_trees_among_larger_ones():
    bd = _forest([1, 30, 1, 1, 12, 1, 57, 1], 40)
    _op_vs_composition(bd, 40, torch.rand(bd.edge_index.shape[1], device=DEV), steps=2)


@pytest.mark.parametrize("train", [True, False])
def test_one_tree(train):
    bd = _forest([45], 40)
    _op_vs_composition(bd, 40, None, train=train)


def test_momentum_none_cumulative_average():
    bd = _forest([20, 33, 7, 64], 40)
    bn = _op_vs_composition(bd, 40, None, momentum=None, steps=3)
    assert int(bn.num_batches_tracked) == 3


def test_zero_edge_weights():
    bd = _forest([20, 33, 7, 64], 40)
    e = bd.edge_index.shape[1]
    w = torch.rand(e, device=DEV)
    w[::3] = 0.0
    _op_vs_composition(bd, 40, w)
    _op_vs_composition(bd, 40, torch.zeros(e, device=DEV))


def test_hub_root():
    bd = _forest([12, 601, 5, 300], 40, star=(1, 3))
    _op_vs_composition(bd, 40, torch.rand(bd.edge_index.shape[1], device=DEV) + 0.05, steps=2)


def test_out_of_range_root_is_flagged():
    import bigcn_b200
    _, new = _pair(40, False)
    bd = _batch("twitter15", 3, 5, 40)
    bd.rootindex = bd.rootindex.clone()
    bd.rootindex[1] = bd.x.shape[0] + 7
    new(bd)
    with pytest.raises(IndexError, match="rootindex"):
        new.check_inputs()


def test_rejects_sparse_or_grad_x():
    import bigcn_b200
    _, new = _pair(40, False)
    bd = _batch("twitter15", 3, 5, 40)
    xd = bd.x
    bd.x = xd.to_sparse()
    with pytest.raises(bigcn_b200.BigcnError, match="sparse"):
        new(bd)
    bd.x = xd.clone().requires_grad_(True)
    with pytest.raises(bigcn_b200.BigcnError, match="requires grad"):
        new(bd)


# ---- not materialised, deterministic, trains --------------------------------------------------------------------------
def _peak_above(m, bd):
    m.zero_grad(set_to_none=True)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    out, _, _ = m(bd)
    F.nll_loss(out, bd.y).backward()
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() - base


def test_root_half_not_materialised():
    ref, new = _pair(5000, False)
    bd = _batch("twitter16", 128, 21, 5000)
    n, k = bd.x.shape
    one_x = n * k * 4
    for m in (ref, new):
        m.train()
        _peak_above(m, bd)                                 # first calls: auto gemm modes, allocator pools
    peak_new, peak_ref = _peak_above(new, bd), _peak_above(ref, bd)
    print(f"N={n} K={k}: one fp32 x = {one_x / 2**20:.0f} MiB, peak above inputs: library {peak_new / 2**20:.0f} MiB, "
          f"harness {peak_ref / 2**20:.0f} MiB")
    assert peak_new < one_x
    assert peak_ref > 2 * one_x


def test_deterministic():
    from bigcn_b200.ops import EBGCNConv2Function
    _, new = _pair(768, False)
    bd = _batch("pheme", 64, 8, 768)
    new.train()

    def run():
        new.zero_grad(set_to_none=True)
        torch.manual_seed(1)
        out, _, _ = new(bd)
        F.nll_loss(out, bd.y).backward()
        return [out.detach().clone()] + [p.grad.clone() for p in new.parameters() if p.grad is not None]
    a, b = run(), run()
    assert len(a) >= 8 and all(torch.equal(x, y) for x, y in zip(a, b))
    # the op with learnt edge weights: d edge_weight too
    m = new.TDrumorGCN
    h = torch.randn(bd.x.shape[0], 64, device=DEV)
    w = torch.rand(bd.edge_index.shape[1], device=DEV)

    def op():
        hh, ww = h.clone().requires_grad_(True), w.clone().requires_grad_(True)
        node_ptr = torch.empty(bd.rootindex.numel() + 1, dtype=torch.int32, device=DEV)
        out = EBGCNConv2Function.apply(hh, ww, m.bn1.weight, m.bn1.bias, m.conv2.lin.weight, m.conv2.bias, bd.x,
                                       bd.edge_index, bd.batch, bd.rootindex, m.bn1, "target", node_ptr,
                                       torch.zeros(1, dtype=torch.int32, device=DEV))
        out.square().sum().backward()
        return out.detach(), hh.grad, ww.grad
    assert all(torch.equal(x, y) for x, y in zip(op(), op()))


def test_trains_like_harness():
    ref, new = _pair(40, True)
    opts = [torch.optim.Adam(m.parameters(), lr=5e-4, weight_decay=1e-4) for m in (ref, new)]
    for m in (ref, new):
        m.train()
    for s in range(10):
        bd = _batch("twitter15", 8, 100 + s, 40)
        losses = []
        for m, o in zip((ref, new), opts):
            o.zero_grad()
            _, _, loss = _step(m, bd, 1000 + s)
            o.step()
            losses.append(float(loss))
        assert abs(losses[0] - losses[1]) <= 1e-4, (s, losses)
