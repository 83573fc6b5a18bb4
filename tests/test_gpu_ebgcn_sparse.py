"""EBGCN and GCNConv on a SparseX data.x (bag-of-words rows as CSR, never densified): GCNConv through the CSR product
and the column sweep (bigcn_gcnconv_csr_*), EBGCN's conv2 op through the dense block of root rows it forms from the CSR
(csrc/ebgcn.cu, k_eb_root_csr).  Compared with the same models on the same values dense, with the fp64 oracle, on
DeviceForest batches of both storages, and on the edge cases, refusals, memory and determinism."""
import copy
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from test_gpu_ebgcn import OracleDir
from test_gpu_ebgcn_fused import TIGHT, _args, _grad_errors, _peak_above, _step

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")
GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(autouse=True)
def _no_tf32(monkeypatch):
    # the edge-inference sub-networks are plain torch modules: keep cuDNN / cuBLAS from running them in TF32
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)
    monkeypatch.setattr(torch.backends.cuda.matmul, "allow_tf32", False)


def _sx(x):
    """the dense CUDA matrix x as a SparseX (columns ascending in every row)"""
    from bigcn_b200 import SparseX
    return SparseX.from_torch_csr(x.to_sparse_csr())


def _sparse_batch(bd):
    sb = copy.copy(bd)
    sb.x = _sx(bd.x)
    return sb


def _csr(n, k, counts, rng):
    """a SparseX [n, k] with counts[i] distinct columns in row i, in random (unsorted) order, values in [-2, 2)"""
    from bigcn_b200 import SparseX
    cols = [rng.choice(k, int(c), replace=False) for c in counts]
    ptr = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    col = np.concatenate(cols).astype(np.int32) if n else np.zeros(0, np.int32)
    val = rng.uniform(-2, 2, int(ptr[-1])).astype(np.float32)
    return SparseX(torch.from_numpy(ptr).to(DEV), torch.from_numpy(col).to(DEV), torch.from_numpy(val).to(DEV), (n, k))


def _tree_edges(n, rng):
    par = np.array([rng.integers(0, i) for i in range(1, n)], np.int64)
    return torch.from_numpy(np.stack([par, np.arange(1, n)])).to(DEV)


# ---- GCNConv on a SparseX ---------------------------------------------------------------------------------------------
def _counts(case, n, k, rng):
    if case == "empty":
        return np.zeros(n, np.int64)
    if case == "one":
        return np.array([min(k, 9)])
    c = np.minimum(rng.poisson(12, n), k)
    c[::7] = 0                                   # empty rows
    c[5] = 60 if k > 60 else k                   # a row longer than 48 entries where K allows one
    return c


@pytest.mark.parametrize("case,n", [("mixed", 300), ("empty", 20), ("one", 1)])
@pytest.mark.parametrize("k", [40, 5000])
def test_gcnconv_on_sparse_x(case, n, k):
    """the CSR conv against the same conv on the dense x (exact fp32 scan) and the fp64 oracle: output, dW, db"""
    import bigcn_b200
    from bigcn_b200.ops import raise_on_flags
    from oracle import gcn_oracle
    rng = np.random.default_rng(k + n)
    xs = _csr(n, k, _counts(case, n, k, rng), rng)
    xd = xs.to_dense()
    ei = _tree_edges(n, rng)
    torch.manual_seed(3)
    sp = bigcn_b200.GCNConv(k, 64).to(DEV)
    with torch.no_grad():
        sp.bias.uniform_(-0.5, 0.5)
    de = copy.deepcopy(sp)
    de.gemm_mode = "fp32"
    orc = gcn_oracle.GCNConv(k, 64).double()
    orc.load_state_dict({k_: v.detach().cpu().double() for k_, v in sp.state_dict().items()})
    r = torch.randn(n, 64, device=DEV)
    got = sp(xs, ei)
    want = de(xd, ei)
    ref = orc(xd.cpu().double(), ei.cpu())
    (got * r).sum().backward()
    (want * r).sum().backward()
    (ref * r.cpu().double()).sum().backward()
    raise_on_flags(sp.last_flags)
    scale = max(float(ref.abs().max()), 1e-6)
    assert float((got - want).abs().max()) <= 1e-5 * scale
    assert float((got.detach().cpu().double() - ref.detach()).abs().max()) <= 1e-5 * scale
    for name, a, b, c in (("dW", sp.lin.weight.grad, de.lin.weight.grad, orc.lin.weight.grad),
                          ("db", sp.bias.grad, de.bias.grad, orc.bias.grad)):
        s = max(float(c.abs().max()), 1e-6)
        assert float((a - b).abs().max()) <= 5e-5 * s, name
        assert float((a.cpu().double() - c).abs().max()) <= 5e-5 * s, name
    if case == "empty":
        assert float(sp.lin.weight.grad.abs().max()) == 0.0


# ---- EBGCN: SparseX model against the dense-x model --------------------------------------------------------------------
def _pair(k, infer, seed=4):
    import bigcn_b200
    torch.manual_seed(seed)
    dense = bigcn_b200.EBGCN(_args(k, infer)).to(DEV)
    sparse = bigcn_b200.EBGCN(_args(k, infer)).to(DEV)
    sparse.load_state_dict(dense.state_dict())
    return dense, sparse


def _batch(shape, n_trees, seed, k):
    from bigcn_b200.data import make_batch
    return make_batch(shape, n_trees, seed=seed, train=True, in_feats=k).to(DEV)


def _check_bn(dense, sparse, k):
    for d in ("TDrumorGCN", "BUrumorGCN"):
        a, b = getattr(dense, d).bn1, getattr(sparse, d).bn1
        assert int(a.num_batches_tracked) == int(b.num_batches_tracked)
        # the root columns see the same root rows: bit for bit; the h1 columns see conv1's output
        assert torch.equal(a.running_mean[64:], b.running_mean[64:]) and torch.equal(a.running_var[64:], b.running_var[64:])
        torch.testing.assert_close(b.running_mean, a.running_mean, rtol=1e-5, atol=1e-6)
        torch.testing.assert_close(b.running_var, a.running_var, rtol=1e-5, atol=1e-6)


def _compare(dense, sparse, bd, infer, min_grads, seed=7):
    sb = _sparse_batch(bd)
    want, wl, _ = _step(dense, bd, seed)
    got, gl, _ = _step(sparse, sb, seed)
    assert float((got - want).abs().max()) <= 5e-5 * float(want.abs().max())
    for a, b in zip(wl, gl):
        if infer:
            assert abs(float(a) - float(b)) <= 1e-5 * max(1.0, abs(float(a)))
        else:
            assert a is None and b is None
    errs = _grad_errors(dense, sparse)
    assert len(errs) >= min_grads, sorted(errs)
    bad = {n: v for n, v in errs.items() if v >= (5e-4 if n.endswith(TIGHT) else 5e-3)}
    assert not bad, bad
    sparse.check_inputs()


@pytest.mark.parametrize("k", [40, 5000])
@pytest.mark.parametrize("infer", [True, False], ids=["infer", "plain"])
@pytest.mark.parametrize("train", [True, False], ids=["train", "eval"])
def test_matches_dense_model(k, infer, train):
    dense, sparse = _pair(k, infer)
    bd = _batch("twitter16", 128, 21, k)
    for m in (dense, sparse):
        m.train(train)
    _compare(dense, sparse, bd, infer, 20 if infer else 12)
    _check_bn(dense, sparse, k)


def test_k5000_training_matches_fp64_oracle():
    """128 Twitter16-shaped trees at K = 5000, data.x a SparseX, against the fp64 oracle module: every gradient at the
    tight bar of test_gpu_ebgcn_fused.py"""
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
    bd = _sparse_batch(make_batch("twitter16", 128, seed=21, train=True, in_feats=k).to(DEV))
    want = F.log_softmax(ref_fc(torch.cat((ref_bu(b), ref_td(b)), 1)), dim=1)
    out, _, _ = m(bd)
    assert float((out.detach().cpu().double() - want.detach()).abs().max()) <= 5e-5 * float(want.abs().max())
    F.nll_loss(want, b.y).backward()
    F.nll_loss(out, bd.y).backward()
    m.check_inputs()
    theirs = {f"{tag}.{n}": q.grad for tag, r in (("TDrumorGCN", ref_td), ("BUrumorGCN", ref_bu))
              for n, q in r.named_parameters() if q.grad is not None}
    theirs.update({"fc.weight": ref_fc.weight.grad, "fc.bias": ref_fc.bias.grad})
    gmax = max(float(g.abs().max()) for g in theirs.values())
    errs = {n: float((p.grad.cpu().double() - theirs[n]).abs().max()) / max(float(theirs[n].abs().max()), 1e-3 * gmax)
            for n, p in m.named_parameters() if n in theirs}
    assert len(errs) >= 14
    bad = {n: v for n, v in errs.items() if v >= 5e-4}
    assert not bad, bad


# ---- the op on a CSR x against the op on the same x dense: the same root rows, so bit-identical ------------------------
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


def _op_dense_vs_csr(bd, k, weights, train=True, steps=2, xs=None, csr_flags=0):
    """the op on bd.x dense and on ``xs`` (default: bd.x as CSR), every output, gradient and buffer bit for bit; the
    CSR run's flags must be ``csr_flags``"""
    from bigcn_b200.ops import EBGCNConv2Function
    torch.manual_seed(11)
    n = bd.x.shape[0]
    w2 = (torch.randn(64, 64 + k, device=DEV) * 0.05).requires_grad_(True)
    b2 = torch.randn(64, device=DEV).requires_grad_(True)
    bns = [torch.nn.BatchNorm1d(64 + k).to(DEV) for _ in range(2)]
    with torch.no_grad():
        bns[0].weight.uniform_(0.5, 1.5)
        bns[0].bias.uniform_(-0.2, 0.2)
    bns[1].load_state_dict(bns[0].state_dict())
    xs = _sx(bd.x) if xs is None else xs
    h = torch.randn(n, 64, device=DEV)
    r = torch.randn(n, 64, device=DEV)
    for _ in range(steps):
        res = []
        for x, bn, want_flags in ((bd.x, bns[0], 0), (xs, bns[1], csr_flags)):
            bn.train(train)
            bn.zero_grad(set_to_none=True)
            hh = h.clone().requires_grad_(True)
            ww = None if weights is None else weights.clone().requires_grad_(True)
            w2.grad = b2.grad = None
            node_ptr = torch.empty(bd.rootindex.numel() + 1, dtype=torch.int32, device=DEV)
            flags = torch.zeros(1, dtype=torch.int32, device=DEV)
            out = EBGCNConv2Function.apply(hh, ww, bn.weight, bn.bias, w2, b2, x, bd.edge_index, bd.batch,
                                           bd.rootindex, bn, "target", node_ptr, flags)
            (out * r).sum().backward()
            assert int(flags.item()) == want_flags
            res.append([out.detach(), hh.grad, w2.grad, b2.grad, bn.weight.grad, bn.bias.grad,
                        None if ww is None else ww.grad, bn.running_mean.clone(), bn.running_var.clone(),
                        bn.num_batches_tracked.clone()])
        for i, (a, b) in enumerate(zip(*res)):
            assert (a is None and b is None) or torch.equal(a, b), i


@pytest.mark.parametrize("train", [True, False])
def test_op_single_node_batch(train):
    _op_dense_vs_csr(_forest([1], 40), 40, None, train=train)


def test_op_single_node_trees_among_larger_ones():
    bd = _forest([1, 30, 1, 1, 12, 1, 57, 1], 40)
    _op_dense_vs_csr(bd, 40, torch.rand(bd.edge_index.shape[1], device=DEV))


@pytest.mark.parametrize("train", [True, False])
def test_op_one_tree(train):
    _op_dense_vs_csr(_forest([45], 5000), 5000, None, train=train)


def test_op_hub_roots():
    bd = _forest([12, 601, 5, 300], 40, star=(1, 3))
    _op_dense_vs_csr(bd, 40, torch.rand(bd.edge_index.shape[1], device=DEV) + 0.05)


def test_op_empty_root_row():
    bd = _forest([20, 33, 7, 64], 40)
    bd.x = bd.x.clone()
    bd.x[bd.rootindex[1]] = 0.0
    bd.x[bd.rootindex[3]] = 0.0
    _op_dense_vs_csr(bd, 40, None)
    _op_dense_vs_csr(bd, 40, None, train=False)


def test_op_out_of_range_root_column():
    """a root row's entry with column K + 3: conv2's op skips and flags it (the dense op sees that row without the
    entry), and the next tree's root row is left alone"""
    from bigcn_b200 import SparseX
    from bigcn_b200._lib import FLAG_X_CSR_RANGE
    bd = _forest([20, 33, 7, 64], 40)
    xs = _sx(bd.x)
    r = int(bd.rootindex[1])
    p = int(xs.ptr[r])
    col = xs.col.clone()
    col[p] = 40 + 3
    bd.x = bd.x.clone()
    bd.x[r, int(xs.col[p])] = 0.0
    _op_dense_vs_csr(bd, 40, None, xs=SparseX(xs.ptr, col, xs.val, xs.shape), csr_flags=FLAG_X_CSR_RANGE)


def test_model_edge_cases():
    """the library model on the same batches as SparseX and dense: one-node batch, one-node trees, one tree, hub roots,
    a root whose feature row is empty"""
    for sizes, star in (([1], ()), ([1, 30, 1, 1, 12, 1, 57, 1], ()), ([45], ()), ([12, 601, 5, 300], (1, 3))):
        dense, sparse = _pair(40, False)
        bd = _forest(sizes, 40, star=star)
        bd.y = torch.zeros(len(sizes), dtype=torch.long, device=DEV)
        _compare(dense, sparse, bd, False, 10)          # bn1 has no gradient in a one-node batch
    dense, sparse = _pair(40, False)
    bd = _forest([20, 33, 7, 64], 40)
    bd.y = torch.zeros(4, dtype=torch.long, device=DEV)
    bd.x = bd.x.clone()
    bd.x[bd.rootindex[2]] = 0.0
    _compare(dense, sparse, bd, False, 12)
    _check_bn(dense, sparse, 40)


# ---- flags ------------------------------------------------------------------------------------------------------------
def test_out_of_range_root_is_flagged():
    _, m = _pair(40, False)
    bd = _sparse_batch(_batch("twitter15", 3, 5, 40))
    bd.rootindex = bd.rootindex.clone()
    bd.rootindex[1] = bd.x.shape[0] + 7
    m(bd)
    with pytest.raises(IndexError, match="rootindex"):
        m.check_inputs()


def test_out_of_range_column_is_flagged():
    from bigcn_b200 import SparseX
    _, m = _pair(40, False)
    bd = _sparse_batch(_batch("twitter15", 3, 5, 40))
    col = bd.x.col.clone()
    col[int(bd.x.ptr[int(bd.rootindex[1])])] = 40 + 3          # an entry of a root row
    bd.x = SparseX(bd.x.ptr, col, bd.x.val, bd.x.shape)
    out, _, _ = m(bd)
    assert bool(torch.isfinite(out).all())
    with pytest.raises(IndexError, match="column index"):
        m.check_inputs()


def test_more_nonzeros_than_capacity_is_flagged():
    """60 entries per row at K = 5000: past N * min(K, 48); conv1's dW is NaN and the flag says so"""
    from bigcn_b200 import SparseX
    _, m = _pair(5000, False)
    bd = _batch("twitter15", 2, 5, 5000)
    n = bd.x.shape[0]
    rng = np.random.default_rng(0)
    xs = _csr(n, 5000, np.full(n, 60), rng)
    bd.x = SparseX(xs.ptr, xs.col, xs.val.abs(), xs.shape)
    out, _, _ = m(bd)
    F.nll_loss(out, bd.y).backward()
    assert bool(torch.isnan(m.TDrumorGCN.conv1.lin.weight.grad).any())
    with pytest.raises(IndexError, match="N\\*min"):
        m.check_inputs()


# ---- determinism, memory ----------------------------------------------------------------------------------------------
def test_deterministic():
    # edge inference off: its sub-networks are torch / cuDNN modules, outside what the library makes deterministic
    _, m = _pair(5000, False)
    bd = _sparse_batch(_batch("twitter16", 32, 8, 5000))
    m.train()

    def run():
        m.zero_grad(set_to_none=True)
        torch.manual_seed(1)
        out, _, _ = m(bd)
        F.nll_loss(out, bd.y).backward()
        return [out.detach().clone()] + [p.grad.clone() for p in m.parameters() if p.grad is not None]
    a, b = run(), run()
    assert len(a) >= 15 and all(torch.equal(x, y) for x, y in zip(a, b))


def test_peak_memory_below_dense_x():
    """peak memory above the inputs for one training step at 128 Twitter16 trees, K = 5000: the SparseX model keeps
    no per-non-zero buffer from conv1's forward to its backward, and stays below the dense-x model"""
    dense, sparse = _pair(5000, False)
    bd = _batch("twitter16", 128, 21, 5000)
    sb = _sparse_batch(bd)
    for m in (dense, sparse):
        m.train()
    _peak_above(dense, bd)
    _peak_above(sparse, sb)
    peak_d, peak_s = _peak_above(dense, bd), _peak_above(sparse, sb)
    print(f"peak above inputs: dense x {peak_d / 2**20:.0f} MiB, SparseX {peak_s / 2**20:.0f} MiB")
    assert peak_s < peak_d


# ---- DeviceForest and raw files ----------------------------------------------------------------------------------------
def _forests(k=5000, n_trees=40, seed=6):
    import bigcn_b200
    from bigcn_b200.data import make_tree, tree_sizes
    rng = np.random.default_rng(seed)
    trees = [make_tree("twitter16", int(n), rng, in_feats=k) for n in tree_sizes("twitter16", n_trees, rng)]
    return (bigcn_b200.DeviceForest.from_data_list(trees, DEV, features="csr"),
            bigcn_b200.DeviceForest.from_data_list(trees, DEV, features="dense"))


def test_device_forest_csr_and_dense_batches_agree():
    csr, dense_f = _forests()
    ids = [3, 0, 17, 1, 1, 25, 39, 8, 12]
    a = csr.batch(ids, 0.2, 0.3, seed=5)
    b = dense_f.batch(ids, 0.2, 0.3, seed=5)
    assert isinstance(a.x, __import__("bigcn_b200").SparseX) and torch.equal(a.x.to_dense(), b.x)
    for infer in (False, True):
        dm, sm = _pair(5000, infer)
        for m in (dm, sm):
            m.train()
        want, wl, _ = _step(dm, b, 3)
        got, gl, _ = _step(sm, a, 3)
        assert float((got - want).abs().max()) <= 5e-5 * float(want.abs().max())
        errs = _grad_errors(dm, sm)
        bad = {n: v for n, v in errs.items() if v >= (5e-4 if n.endswith(TIGHT) else 5e-3)}
        assert not bad, bad
        sm.check_inputs()


def test_device_forest_adam_steps_agree():
    """five Adam steps with edge inference on, from the same torch seeds, on batches of a CSR and a dense forest"""
    csr, dense_f = _forests()
    dm, sm = _pair(5000, True)
    opts = [torch.optim.Adam(m.parameters(), lr=5e-4, weight_decay=1e-4) for m in (dm, sm)]
    for m in (dm, sm):
        m.train()
    ids = [[0, 5, 9, 13], [2, 4, 6, 8, 10], [1, 3], [20, 21, 22, 39], [7, 30]]
    seeds = [1, 2, 3, 4, 5]
    for s, ((a, _), (b, _)) in enumerate(zip(csr.batches(ids, 0.2, 0.2, seeds=seeds),
                                             dense_f.batches(ids, 0.2, 0.2, seeds=seeds))):
        losses = []
        for m, o, bd in zip((dm, sm), opts, (b, a)):
            o.zero_grad()
            _, _, loss = _step(m, bd, 100 + s)
            o.step()
            losses.append(float(loss))
        assert abs(losses[0] - losses[1]) <= 1e-4, (s, losses)
    sm.check_inputs()
    for (name, p), q in zip(sm.named_parameters(), dm.parameters()):
        assert float((p - q).abs().max()) <= 1e-4, name


def test_forest_from_raw():
    from bigcn_b200 import ingest
    raw = os.path.join(GOLD, "ref_ingest", "data", "Twitter15")
    forest = ingest.forest_from_raw(os.path.join(raw, "data.TD_RvNN.vol_5000.txt"),
                                    os.path.join(raw, "Twitter15_label_All.txt"), "Twitter15", DEV)
    bd = forest.batch(list(range(len(forest.ids))), 0.2, 0.2, seed=1)
    _, m = _pair(5000, True)
    m.train()
    out, tdl, bul = m(bd)
    (F.nll_loss(out, bd.y) + 0.2 * (tdl + bul)).backward()
    assert bool(torch.isfinite(out).all()) and bool(torch.isfinite(tdl)) and bool(torch.isfinite(bul))
    assert all(bool(torch.isfinite(p.grad).all()) for p in m.parameters() if p.grad is not None)
    m.check_inputs()


# ---- refusals ---------------------------------------------------------------------------------------------------------
def test_refusals():
    import bigcn_b200
    from bigcn_b200 import SparseX
    _, m = _pair(40, False)
    bd = _sparse_batch(_batch("twitter15", 3, 5, 40))
    xs = bd.x
    bd.x = SparseX(xs.ptr, xs.col, xs.val.clone().requires_grad_(True), xs.shape)
    with pytest.raises(bigcn_b200.BigcnError, match="requires grad"):
        m(bd)
    bd.x = xs.to("cpu")
    with pytest.raises(bigcn_b200.BigcnError, match="CUDA"):
        m(bd)
    bd.x = SparseX(xs.ptr, xs.col.long(), xs.val, xs.shape)
    with pytest.raises(bigcn_b200.BigcnError, match="int32"):
        m(bd)
    conv = bigcn_b200.GCNConv(40, 64, gemm_mode="tf32x3").to(DEV)
    with pytest.raises(bigcn_b200.BigcnError, match="gemm_mode='sparse'"):
        conv(xs, bd.edge_index)
    conv.gemm_mode = "sparse"
    with pytest.raises(bigcn_b200.BigcnError, match="edge_weight"):
        conv(xs, bd.edge_index, torch.ones(bd.edge_index.shape[1], device=DEV))
    conv(xs, bd.edge_index)            # 'sparse' and 'auto' take it


def test_dense_batch_after_flagged_sparse_batch():
    """conv1's flags belong to its last forward: a flagged SparseX batch followed by a clean dense one raises nothing"""
    from bigcn_b200 import SparseX
    _, m = _pair(40, False)
    bd = _batch("twitter15", 3, 5, 40)
    sb = _sparse_batch(bd)
    col = sb.x.col.clone()
    col[0] = 40 + 3
    sb.x = SparseX(sb.x.ptr, col, sb.x.val, sb.x.shape)
    m(sb)
    assert m.TDrumorGCN.conv1.last_flags is not None
    m(bd)
    assert m.TDrumorGCN.conv1.last_flags is None and m.BUrumorGCN.conv1.last_flags is None
    m.check_inputs()
