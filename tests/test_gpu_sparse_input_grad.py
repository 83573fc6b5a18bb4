"""Gradient w.r.t. a sparse data.x.  The gradient a sparse x receives is the dense one (data.x.grad = T1_TD W1_TD +
T1_BU W1_BU, see test_gpu_input_grad.py) sampled at x's stored entries -- the convention of torch.sparse.mm.  The
fused path returns it from k_dx_csr (an SDDMM over the CSR): into ``val.grad`` for an ops.SparseX, as a COO gradient
on ``x.coalesce()``'s indices for a torch sparse COO x and as a CSR gradient on x's own pattern for a torch sparse
CSR x.  The reference is the fixed fp64 oracle's dense x.grad gathered at the stored (row, col) entries."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from bigcn_b200.data import make_batch, make_tree
from test_gpu_input_grad import fixed_oracle, masks_for, rel_err, with_x


def rows_of(ptr):
    ptr = torch.as_tensor(ptr).long().cpu()
    return torch.repeat_interleave(torch.arange(ptr.numel() - 1), ptr[1:] - ptr[:-1])


def gathered(dense, ptr, col):
    """dense[i, col[e]] for every entry e of row i"""
    return dense.detach().cpu()[rows_of(ptr), torch.as_tensor(col).long().cpu()]


def coo_with_duplicates(x, split=7):
    """an uncoalesced COO of the dense x: every `split`-th stored value is cut in two entries at the same (row, col),
    the second half placed at the end; plus one explicit zero entry"""
    idx = torch.nonzero(x).t()
    vals = x[idx[0], idx[1]].clone()
    dup = torch.arange(0, idx.shape[1], split)
    half = vals[dup] * 0.25
    vals[dup] -= half
    zero = torch.tensor([[0], [int((idx[1, :].max() + 1) % x.shape[1])]])
    while bool(((idx[0] == zero[0, 0]) & (idx[1] == zero[1, 0])).any()):
        zero[1, 0] = (zero[1, 0] + 1) % x.shape[1]
    idx = torch.cat([idx, idx[:, dup], zero], 1)
    vals = torch.cat([vals, half, torch.zeros(1, dtype=vals.dtype)])
    return torch.sparse_coo_tensor(idx, vals, x.shape)


# ---------------------------------------------------------------------------------------------- CPU: the convention
def _oracle_through_sparse_mm(ref, b, x_coo):
    """the fixed oracle with conv1's input formed by torch.sparse.mm(x_coo, I): its gradient w.r.t. x_coo is torch's"""
    eye = torch.eye(x_coo.shape[1], dtype=x_coo.dtype)
    return ref(with_x(b, torch.sparse.mm(x_coo, eye)))


def test_sampled_gradient_is_torch_sparse_mm_convention():
    """fp64, eval: the oracle's dense x.grad gathered at x.coalesce()'s entries equals the COO gradient torch.sparse.mm
    gives an uncoalesced x with duplicates and an explicit zero; each duplicate's own derivative is that full value."""
    b = make_batch("twitter15", 3, seed=5, train=False, in_feats=16)
    ref = fixed_oracle(16, seed=2).double().eval()
    x0 = b.x.double()
    xr = x0.clone().requires_grad_(True)
    F.nll_loss(ref(with_x(b, xr)), b.y).backward()
    x_coo = coo_with_duplicates(x0).requires_grad_(True)
    F.nll_loss(_oracle_through_sparse_mm(ref, b, x_coo), b.y).backward()
    g = x_coo.grad.coalesce()
    xc = x_coo.detach().coalesce()
    assert x_coo.grad.layout == torch.sparse_coo
    assert torch.equal(g.indices(), xc.indices())
    want = xr.grad[xc.indices()[0], xc.indices()[1]]
    assert torch.allclose(g.values(), want, rtol=0, atol=1e-14 * float(want.abs().max()))
    # the values of an uncoalesced x: every stored entry, duplicates included, gets the sampled value in full
    vals = x_coo.detach()._values().clone().requires_grad_(True)
    xv = torch.sparse_coo_tensor(x_coo.detach()._indices(), vals, x0.shape)
    F.nll_loss(_oracle_through_sparse_mm(ref, b, xv), b.y).backward()
    idx = x_coo.detach()._indices()
    assert torch.allclose(vals.grad, xr.grad[idx[0], idx[1]], rtol=0, atol=1e-14 * float(want.abs().max()))


def test_sampled_gradient_central_difference():
    """fp64: the sampled gradient of a few stored values (a duplicate and the explicit zero among them) equals a
    central difference of the loss in that value, through conv1 only (the root-extend inputs held fixed)."""
    b = make_batch("twitter15", 3, seed=6, train=False, in_feats=16)
    ref = fixed_oracle(16, seed=4).double().eval()
    x_coo = coo_with_duplicates(b.x.double())
    idx, v0 = x_coo._indices(), x_coo._values()
    xr = b.x.double().clone().requires_grad_(True)
    F.nll_loss(ref(with_x(b, xr)), b.y).backward()
    for mod in (ref.TDrumorGCN, ref.BUrumorGCN):
        mod.pinned = mod.detached
    m = v0.numel()
    picks = [0, 5, m // 2, m - 3, m - 2, m - 1]        # m - 2: a duplicate's second half; m - 1: the explicit zero
    eps = 1e-6
    with torch.no_grad():
        for e in picks:
            vp, vm = v0.clone(), v0.clone()
            vp[e] += eps
            vm[e] -= eps
            lp = F.nll_loss(_oracle_through_sparse_mm(ref, b, torch.sparse_coo_tensor(idx, vp, x_coo.shape)), b.y)
            lm = F.nll_loss(_oracle_through_sparse_mm(ref, b, torch.sparse_coo_tensor(idx, vm, x_coo.shape)), b.y)
            fd = float((lp - lm) / (2 * eps))
            want = float(xr.grad[idx[0, e], idx[1, e]])
            assert abs(fd - want) <= 1e-7 * max(1.0, float(xr.grad.abs().max())), e


# ---------------------------------------------------------------------------------------------- the kernel alone
def edge_case_csr(k, seed):
    """bag-of-words rows of make_batch, then: empty rows, a row with all K columns, duplicate columns in a row,
    explicit zero values, out-of-range columns (k + 3 and -1)"""
    rng = np.random.default_rng(seed)
    x = make_batch("twitter15", 6, seed=seed, train=False, in_feats=k).x.numpy()
    rows = []
    for i in range(x.shape[0]):
        c = np.nonzero(x[i])[0]
        rows.append([c.astype(np.int64), x[i, c].astype(np.float32)])
    rows[1] = rows[2] = [np.zeros(0, np.int64), np.zeros(0, np.float32)]
    rows[5] = [rng.permutation(k), rng.normal(size=k).astype(np.float32)]
    c, v = rows[7]
    rows[7] = [np.concatenate([c, c[:3], c[:1]]), np.concatenate([v, v[:3] * 2, v[:1]])]
    rows[9][1] = rows[9][1].copy()
    rows[9][1][0] = 0.0
    rows[11][0] = np.concatenate([rows[11][0], [k + 3, -1]])
    rows[11][1] = np.concatenate([rows[11][1], [1.0, 2.0]]).astype(np.float32)
    ptr = np.concatenate([[0], np.cumsum([len(r[0]) for r in rows])]).astype(np.int32)
    col = np.concatenate([r[0] for r in rows]).astype(np.int32)
    val = np.concatenate([r[1] for r in rows]).astype(np.float32)
    return torch.from_numpy(ptr), torch.from_numpy(col), torch.from_numpy(val)


def sddmm_ref(ptr, col, t, ws, k):
    """fp64 dval[e] = t[i] . cat(ws)[:, col[e]], 0 outside [0, K)"""
    wcat = torch.cat(ws).double()
    rows, col = rows_of(ptr), col.long()
    ok = (col >= 0) & (col < k)
    out = torch.zeros(col.numel(), dtype=torch.float64)
    out[ok] = (t.double()[rows[ok]] * wcat[:, col[ok]].t()).sum(1)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("k", [5000, 776, 64, 5003])
@pytest.mark.parametrize("n_w", [1, 2])
def test_x_dgrad_csr_kernel(dev, k, n_w):
    """ops.x_dgrad_csr against fp64: max|d| <= 2e-6 max|ref| with the edge cases of edge_case_csr; two calls
    bit-identical; a CSR handed over at capacity (col / val longer than ptr[N]) gets 0 past ptr[N]; nnz = 0."""
    from bigcn_b200 import ops
    ptr, col, val = edge_case_csr(k, seed=k + n_w)
    n = ptr.numel() - 1
    torch.manual_seed(k + n_w)
    t = torch.randn(n, 64 * n_w)
    ws = [torch.randn(64, k) * 0.05 for _ in range(n_w)]
    want = sddmm_ref(ptr, col, t, ws, k)
    td, wd = t.to(dev), [w.to(dev) for w in ws]
    xs = ops.SparseX(ptr, col, val, (n, k)).to(dev)
    got = ops.x_dgrad_csr(xs, td, wd)
    assert got.dtype == torch.float32 and got.shape == val.shape
    assert rel_err(got, want) <= 2e-6
    oor = (col < 0) | (col >= k)
    assert bool(oor.any()) and bool((got.cpu()[oor] == 0).all())
    assert torch.equal(got, ops.x_dgrad_csr(xs, td, wd))
    cap = ops.SparseX(xs.ptr, torch.cat([xs.col, torch.full((37,), 1, dtype=torch.int32, device=dev)]),
                      torch.cat([xs.val, torch.ones(37, device=dev)]), (n, k))
    got_cap = ops.x_dgrad_csr(cap, td, wd)
    assert torch.equal(got_cap[:col.numel()], got) and bool((got_cap[col.numel():] == 0).all())
    empty = ops.SparseX(torch.zeros(n + 1, dtype=torch.int32), torch.zeros(0, dtype=torch.int32), torch.zeros(0),
                        (n, k)).to(dev)
    assert ops.x_dgrad_csr(empty, td, wd).shape == (0,)


# ---------------------------------------------------------------------------------------------- the model
def sparse_x(x, dev):
    from bigcn_b200 import ops
    return ops.SparseX.from_torch_csr(x.to_sparse_csr()).to(dev)


def _run(m, bd, xs, need, seed=777):
    from bigcn_b200 import ops
    for mod in (m.TDrumorGCN, m.BUrumorGCN):
        mod.seed, mod._calls = seed, 0
    m.zero_grad(set_to_none=True)
    val = xs.val.detach().clone().requires_grad_(need)
    out = m(with_x(bd, ops.SparseX(xs.ptr, xs.col, val, xs.shape)))
    F.nll_loss(out, bd.y).backward()
    m.check_inputs()
    return out.detach().clone(), [p.grad.clone() for p in m.parameters()], val.grad


def oracle_x_grad(ref, b, train, seed, k):
    """fp64 log-probs and dense x.grad of the fixed oracle, with the kernel's dropout masks in train mode"""
    n = b.x.shape[0]
    keep = masks_for(seed, n, k) if train else [None, None]
    ref.train(train)
    xr = b.x.double().requires_grad_(True)
    want = ref(with_x(b, xr), keep_td=keep[0], keep_bu=keep[1])
    F.nll_loss(want, b.y).backward()
    return want, xr.grad


@pytest.mark.gpu
@pytest.mark.parametrize("train", [False, True])
def test_model_sparse_x_val_grad(dev, train):
    """BiGCN on a SparseX whose val requires grad: val.grad within 1e-4 of the gathered oracle gradient; log-probs and
    all ten parameter gradients bit-identical to the run without val.requires_grad."""
    import bigcn_b200
    k = 5000
    b = make_batch("twitter15", 10, seed=4, train=train, in_feats=k)
    ref = fixed_oracle(k, seed=3).double()
    m = bigcn_b200.BiGCN(k, 64, 64, dev).to(dev).train(train)
    m.load_state_dict(ref.state_dict())
    bd = with_x(b, b.x).to(dev)
    xs = sparse_x(b.x, dev)
    out0, grads0, none = _run(m, bd, xs, False)
    assert none is None
    out1, grads1, vg = _run(m, bd, xs, True)
    assert torch.equal(out0, out1)
    for (name, _), g0, g1 in zip(m.named_parameters(), grads0, grads1):
        assert torch.equal(g0, g1), name
    assert vg.dtype == torch.float32 and vg.shape == xs.val.shape
    want, xgrad = oracle_x_grad(ref, b, train, m.TDrumorGCN.last_seed, k)
    assert rel_err(out1, want) < 2.2e-5
    assert rel_err(vg, gathered(xgrad, xs.ptr, xs.col)) < 1e-4
    for (name, p), q in zip(m.named_parameters(), ref.parameters()):
        assert rel_err(p.grad, q.grad) < 1e-4, name


@pytest.mark.gpu
def test_single_direction_sparse_x(dev):
    """TDrumorGCN alone, BUrumorGCN alone (n_w = 1) and both on one val (autograd sums the two)."""
    import bigcn_b200
    from bigcn_b200 import ops
    b = make_batch("twitter15", 8, seed=9, train=False, in_feats=5000)
    ref = fixed_oracle(5000, seed=8).double().eval()
    bd = with_x(b, b.x).to(dev)
    xs = sparse_x(b.x, dev)
    td = bigcn_b200.TDrumorGCN(5000, 64, 64, dev).to(dev).eval()
    bu = bigcn_b200.BUrumorGCN(5000, 64, 64, dev).to(dev).eval()
    td.load_state_dict(ref.TDrumorGCN.state_dict())
    bu.load_state_dict(ref.BUrumorGCN.state_dict())
    torch.manual_seed(1)
    gt, gb = torch.randn(b.rootindex.numel(), 128), torch.randn(b.rootindex.numel(), 128)
    for mods in ((td,), (bu,), (td, bu)):
        val = xs.val.detach().clone().requires_grad_(True)
        x = ops.SparseX(xs.ptr, xs.col, val, xs.shape)
        xr = b.x.double().requires_grad_(True)
        loss, want = 0, 0
        for mod in mods:
            r = ref.TDrumorGCN if mod is td else ref.BUrumorGCN
            g = gt if mod is td else gb
            loss = loss + (mod(with_x(bd, x)) * g.to(dev)).sum()
            want = want + (r(with_x(b, xr)) * g.double()).sum()
        loss.backward()
        want.backward()
        assert rel_err(val.grad, gathered(xr.grad, xs.ptr, xs.col)) < 1e-4, [type(q).__name__ for q in mods]


@pytest.mark.gpu
def test_torch_sparse_x_grad_layouts(dev):
    """An uncoalesced COO x with duplicates and an explicit zero gets a COO gradient on x.coalesce()'s indices; a CSR
    x gets a CSR gradient on its own crow / col indices; values = the gathered oracle gradient (1e-4)."""
    import bigcn_b200
    k = 5000
    b = make_batch("twitter15", 8, seed=14, train=True, in_feats=k)
    ref = fixed_oracle(k, seed=15).double()
    m = bigcn_b200.BiGCN(k, 64, 64, dev).to(dev).train()
    m.load_state_dict(ref.state_dict())
    bd = with_x(b, b.x).to(dev)
    for layout in (torch.sparse_coo, torch.sparse_csr):
        for mod in (m.TDrumorGCN, m.BUrumorGCN):
            mod.seed, mod._calls = 31, 0
        coo = coo_with_duplicates(b.x)
        x = (coo if layout == torch.sparse_coo else coo.coalesce().to_sparse_csr()).to(dev).requires_grad_(True)
        F.nll_loss(m(with_x(bd, x)), bd.y).backward()
        m.check_inputs()
        _, xgrad = oracle_x_grad(ref, b, True, m.TDrumorGCN.last_seed, k)
        assert x.grad.layout == layout and x.grad.dtype == torch.float32 and x.grad.shape == x.shape
        if layout == torch.sparse_coo:
            xc, g = x.detach().coalesce(), x.grad.coalesce()
            assert g.values().numel() == xc.values().numel() and torch.equal(g.indices(), xc.indices())
            got, idx = g.values(), xc.indices().cpu()
            want = xgrad[idx[0], idx[1]]
        else:
            assert torch.equal(x.grad.crow_indices(), x.crow_indices())
            assert torch.equal(x.grad.col_indices(), x.col_indices())
            got, want = x.grad.values(), gathered(xgrad, x.crow_indices(), x.col_indices())
        assert rel_err(got, want) < 1e-4, layout


@pytest.mark.gpu
def test_upstream_per_column_weight(dev):
    """x = torch.sparse_coo_tensor(idx, counts * w[col]): w.grad against the oracle run on the densified equivalent."""
    import bigcn_b200
    k = 5000
    b = make_batch("twitter15", 8, seed=16, train=False, in_feats=k)
    ref = fixed_oracle(k, seed=17).double().eval()
    m = bigcn_b200.BiGCN(k, 64, 64, dev).to(dev).eval()
    m.load_state_dict(ref.state_dict())
    coo = coo_with_duplicates(b.x)
    idx, counts = coo._indices(), coo._values()
    torch.manual_seed(18)
    w0 = 0.5 + torch.rand(k)
    w = w0.to(dev).requires_grad_(True)
    x = torch.sparse_coo_tensor(idx.to(dev), counts.to(dev) * w[idx[1].to(dev)], b.x.shape)
    bd = with_x(b, b.x).to(dev)
    F.nll_loss(m(with_x(bd, x)), bd.y).backward()
    m.check_inputs()
    wr = w0.double().requires_grad_(True)
    xr = torch.zeros(b.x.shape, dtype=torch.float64).index_put((idx[0], idx[1]), counts.double() * wr[idx[1]],
                                                                accumulate=True)
    F.nll_loss(ref(with_x(b, xr)), b.y).backward()
    assert rel_err(w.grad, wr.grad) < 1e-4


@pytest.mark.gpu
def test_sparse_grad_equals_dense_grad_gathered(dev):
    """On one batch: the SparseX val.grad equals the dense-x x.grad (gemm_mode='sparse', k_dx_tc) gathered at the
    pattern, within 1e-5 of max|ref|."""
    import bigcn_b200
    k = 5000
    b = make_batch("twitter16", 16, seed=19, train=True, in_feats=k)
    m = bigcn_b200.BiGCN(k, 64, 64, dev, gemm_mode="sparse").to(dev).train()
    bd = with_x(b, b.x).to(dev)
    xs = sparse_x(b.x, dev)
    _, _, vg = _run(m, bd, xs, True)
    for mod in (m.TDrumorGCN, m.BUrumorGCN):
        mod.seed, mod._calls = 777, 0
    x = bd.x.detach().clone().requires_grad_(True)
    F.nll_loss(m(with_x(bd, x)), bd.y).backward()
    want = gathered(x.grad, xs.ptr, xs.col)
    assert rel_err(vg, want) < 1e-5


@pytest.mark.gpu
def test_device_forest_batch_and_saliency(dev):
    """A DeviceForest batch (its val cloned with requires_grad_()) gives the same val.grad as the torch sparse CSR form
    of that batch, bit for bit; a frozen model used for saliency still fills val.grad, against the oracle."""
    import bigcn_b200
    from bigcn_b200 import ops
    k = 3000
    rng = np.random.default_rng(20)
    trees = [make_tree("twitter15", int(n), rng, in_feats=k) for n in (60, 1, 350, 17, 90, 5, 200)]
    forest = bigcn_b200.DeviceForest.from_data_list(trees, dev)
    fb = forest.batch([3, 0, 6, 2, 2, 5])
    ref = fixed_oracle(k, seed=21).double().eval()
    m = bigcn_b200.BiGCN(k, 64, 64, dev).to(dev).eval()
    m.load_state_dict(ref.state_dict())
    m.requires_grad_(False)
    xs = fb.x
    val = xs.val.clone().requires_grad_()
    out = m(with_x(fb, ops.SparseX(xs.ptr, xs.col, val, xs.shape)))
    out.gather(1, fb.y.view(-1, 1)).sum().backward()
    m.check_inputs()
    assert val.grad is not None and all(p.grad is None for p in m.parameters())
    x = torch.sparse_csr_tensor(xs.ptr.long(), xs.col.long(), xs.val.clone(), xs.shape).requires_grad_(True)
    m(with_x(fb, x)).gather(1, fb.y.view(-1, 1)).sum().backward()
    assert torch.equal(x.grad.values(), val.grad)
    # saliency against the oracle on the host copy of the batch
    hb = with_x(fb, xs.to_dense()).to("cpu")
    xr = hb.x.double().requires_grad_(True)
    ref(with_x(hb, xr)).gather(1, hb.y.view(-1, 1)).sum().backward()
    assert rel_err(val.grad, gathered(xr.grad, xs.ptr, xs.col)) < 1e-4
