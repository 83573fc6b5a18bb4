"""Gradient w.r.t. data.x.  The reference's conv1 reads x itself (BiGCN_Twitter.py:42) while the first root-extend
reads ``x1 = copy.copy(x.float())`` (:28,45-50), a detached leaf: only conv1 sends a gradient back, and
data.x.grad = T1_TD W1_TD + T1_BU W1_BU.  The fused path returns it from k_dx_tc (tcgen05 kind::tf32, 3xTF32).

The oracle here is oracle.bigcn_oracle with that data flow restated (``fixed_oracle``): conv1 reads x and only the
root-extend reads the detached copy.  Its forward values equal the packaged oracle's; only the gradient differs
(the packaged one feeds conv1 from the copy as well, so its data.x never receives a gradient)."""
import copy

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import bigcn_oracle, gcn_oracle
from bigcn_b200.data import Batch, make_batch


def rel_err(got, want):
    want = want.detach().cpu().double()
    got = got.detach().cpu().double()
    return float((got - want).abs().max()) / max(float(want.abs().max()), 1e-30)


def assert_bf16_close(got, want, atol=1e-5):
    """each element within 2^-8 |ref| + atol max|ref|: one bf16 rounding of a value that is fp32-class (atol = 1e-5,
    the kernel alone) or within the gradient bar of the model (atol = 1e-4)"""
    got, want = got.detach().cpu().double(), want.detach().cpu().double()
    bar = 2.0 ** -8 * want.abs() + atol * float(want.abs().max())
    assert bool(((got - want).abs() <= bar).all()), float(((got - want).abs() - bar).max())


# ---------------------------------------------------------------------------------------------- the fixed oracle
def _fixed_forward(self, data, keep=None):
    """bigcn_oracle._RumorGCN.forward with the reference's data flow for x: conv1 reads x.to(dtype) (:42), only the
    root-extend reads the detached copy x1 (:28).  ``self.pinned`` (tests) replaces the two detached copies, x1 and
    x2 = conv1's output (:44), by given tensors: the forward then depends on x through conv1 alone."""
    x, edge_index = data.x, getattr(data, self.edge_attr)
    dtype = self.conv1.lin.weight.dtype
    x1 = copy.copy(x.to(dtype).detach())
    h = self.conv1(x.to(dtype), edge_index)
    h2 = h.detach()
    if getattr(self, "pinned", None) is not None:
        x1, h2 = self.pinned
    self.detached = (x1, h2)
    h = torch.cat((h, self._root_extend(x1, data)), 1)
    h = F.relu(h)
    h = bigcn_oracle._dropout(h, self.p, self.training, keep)
    h = self.conv2(h, edge_index)
    h = F.relu(h)
    h = torch.cat((h, self._root_extend(h2, data)), 1)
    return gcn_oracle.scatter_mean(h, data.batch, int(data.rootindex.numel()))


class FixedTD(bigcn_oracle.TDrumorGCN):
    forward = _fixed_forward


class FixedBU(bigcn_oracle.BUrumorGCN):
    forward = _fixed_forward


def fixed_oracle(k, seed):
    torch.manual_seed(seed)
    ref = bigcn_oracle.BiGCN(k, 64, 64)
    with torch.no_grad():
        for p in ref.parameters():
            if p.dim() == 1:
                p.uniform_(-0.1, 0.1)
    ref.TDrumorGCN.__class__ = FixedTD
    ref.BUrumorGCN.__class__ = FixedBU
    return ref


def with_x(b, x):
    d = Batch(**{k: getattr(b, k) for k in Batch._tensor_keys})
    d.x = x
    return d


def masks_for(seed, n, k):
    return [torch.from_numpy(gcn_oracle.dropout_keep_mask(seed, d, np.arange(n), 64 + k, 0.5)) for d in (0, 1)]


# ---------------------------------------------------------------------------------------------- CPU: the oracle
def test_fixed_oracle_x_grad_is_conv1_derivative():
    """fp64, eval: the oracle's x.grad equals a central difference taken through conv1's input only, with the inputs
    of both root-extends held fixed (the reference's copy.copy cuts those paths); the full derivative differs."""
    b = make_batch("twitter15", 3, seed=5, train=False, in_feats=16)
    ref = fixed_oracle(16, seed=2).double().eval()
    x0 = b.x.double()
    x = x0.clone().requires_grad_(True)
    F.nll_loss(ref(with_x(b, x)), b.y).backward()
    # the packaged oracle gives the same forward values
    plain = bigcn_oracle.BiGCN(16, 64, 64).double().eval()
    plain.load_state_dict(ref.state_dict())
    with torch.no_grad():
        assert torch.allclose(plain(with_x(b, x0)), ref(with_x(b, x0)), rtol=0, atol=1e-14)
    for mod in (ref.TDrumorGCN, ref.BUrumorGCN):
        mod.pinned = mod.detached
    rng = np.random.default_rng(0)
    nz = torch.nonzero(x0).tolist()
    picks = [tuple(nz[i]) for i in rng.choice(len(nz), 12, replace=False)]
    picks += [(int(rng.integers(x0.shape[0])), int(rng.integers(16))) for _ in range(12)]
    eps = 1e-6
    with torch.no_grad():
        for i, j in picks:
            xp, xm = x0.clone(), x0.clone()
            xp[i, j] += eps
            xm[i, j] -= eps
            fd = (F.nll_loss(ref(with_x(b, xp)), b.y) - F.nll_loss(ref(with_x(b, xm)), b.y)) / (2 * eps)
            assert abs(float(fd) - float(x.grad[i, j])) <= 1e-7 * max(1.0, float(x.grad.abs().max())), (i, j)
    # the root path is not zero: the full derivative (nothing pinned) differs from x.grad
    for mod in (ref.TDrumorGCN, ref.BUrumorGCN):
        mod.pinned = None
    r = int(b.rootindex[0])
    j = int(torch.nonzero(x0[r])[0])
    with torch.no_grad():
        xp, xm = x0.clone(), x0.clone()
        xp[r, j] += eps
        xm[r, j] -= eps
        full = (F.nll_loss(ref(with_x(b, xp)), b.y) - F.nll_loss(ref(with_x(b, xm)), b.y)) / (2 * eps)
    assert abs(float(full) - float(x.grad[r, j])) > 1e-6


# ---------------------------------------------------------------------------------------------- the kernel alone
@pytest.mark.gpu
@pytest.mark.parametrize("k", [5000, 776, 64, 5003])
@pytest.mark.parametrize("n_w", [1, 2])
def test_x_dgrad_kernel(dev, k, n_w):
    """dx = g @ cat(W) against fp64, N = 1000 (off the 128-row tile); fp32 output at 1e-5 of max|ref|, bf16 output
    per element; two calls bit-identical.  K = 5003: the column tail without 16 B stores (fp32 output only)."""
    from bigcn_b200 import ops
    torch.manual_seed(k + n_w)
    n = 1000
    g = torch.randn(n, 64 * n_w)
    ws = [torch.randn(64, k) * 0.05 for _ in range(n_w)]
    want = g.double() @ torch.cat(ws).double()
    gd, wd = g.to(dev), [w.to(dev) for w in ws]
    got = ops.x_dgrad(gd, wd)
    assert got.dtype == torch.float32 and got.shape == (n, k)
    assert rel_err(got, want) <= 1e-5
    assert torch.equal(got, ops.x_dgrad(gd, wd))
    if k % 8 == 0:
        gb = ops.x_dgrad(gd, wd, torch.bfloat16)
        assert gb.dtype == torch.bfloat16
        assert_bf16_close(gb, want)
        assert torch.equal(gb, ops.x_dgrad(gd, wd, torch.bfloat16))
    if k == 5003:   # a weight with a row pitch larger than K
        wide = torch.randn(64, k + 5)
        got = ops.x_dgrad(gd[:, :64].contiguous(), [wide.to(dev)[:, :k]])
        assert rel_err(got, g[:, :64].double() @ wide[:, :k].double()) <= 1e-5


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["tf32x3", "bf16", "fp32"])
def test_xw_op_input_grad(dev, mode):
    """torch.ops.bigcn_b200.xw: autograd returns x.grad through xw_dgrad (bf16 in mode 'bf16'); FakeTensorMode."""
    import bigcn_b200.torch_ops  # noqa: F401  (registers the ops)
    from torch._subclasses.fake_tensor import FakeTensorMode
    torch.manual_seed(3)
    n, k = 777, 776
    dt = torch.bfloat16 if mode == "bf16" else torch.float32
    x = torch.randn(n, k).to(dt)
    w = torch.randn(64, k) * 0.05
    g = torch.randn(n, 64)
    xd = x.to(dev).requires_grad_(True)
    wd = w.to(dev).requires_grad_(True)
    torch.ops.bigcn_b200.xw(xd, wd, mode).backward(g.to(dev))
    want = g.double() @ w.double()
    assert xd.grad.dtype == dt
    if mode == "bf16":
        assert_bf16_close(xd.grad, want)
    else:
        assert rel_err(xd.grad, want) <= 1e-5
    assert rel_err(wd.grad, g.double().t() @ x.double()) < 1e-4
    direct = torch.ops.bigcn_b200.xw_dgrad(g.to(dev), w.to(dev), mode)
    assert torch.equal(direct, xd.grad)
    with FakeTensorMode():
        fg = torch.ops.bigcn_b200.xw_dgrad(torch.empty(n, 64, device=dev), torch.empty(64, k, device=dev), mode)
        assert fg.dtype == dt and tuple(fg.shape) == (n, k)


# ---------------------------------------------------------------------------------------------- the model
CASES = [("twitter15", 5000, 10, m) for m in ("sparse", "fp32", "tf32x3", "bf16", "tf32")] + \
        [("pheme", 768, 40, m) for m in ("fp32", "tf32x3", "bf16", "tf32")]


def _run(m, bd, x_grad, train, seed=777):
    for mod in (m.TDrumorGCN, m.BUrumorGCN):
        mod.seed, mod._calls = seed, 0
    m.zero_grad(set_to_none=True)
    x = bd.x.detach().clone().requires_grad_(x_grad)
    out = m(with_x(bd, x))
    F.nll_loss(out, bd.y).backward()
    m.check_inputs()
    return out.detach().clone(), [p.grad.clone() for p in m.parameters()], x.grad


@pytest.mark.gpu
@pytest.mark.parametrize("train", [False, True])
@pytest.mark.parametrize("shape,k,trees,mode", CASES)
def test_model_x_grad(dev, shape, k, trees, mode, train):
    """data.x.grad against the fp64 fixed oracle (Philox mask injected in train mode): 1e-4 of max|ref|, per element
    in bf16; tf32 1e-2 on bag-of-words x and 3e-2 on dense x (plain TF32 rounds a dense x itself in conv1's forward,
    and T1 inherits that; dX itself is 3xTF32).  Log-probs and all ten parameter gradients bit-identical to the run
    without x.grad."""
    import bigcn_b200
    b = make_batch(shape, trees, seed=4, train=train, in_feats=k)
    x_dt = torch.bfloat16 if mode == "bf16" else torch.float32
    b.x = b.x.to(x_dt).float()
    ref = fixed_oracle(k, seed=3).double()
    m = bigcn_b200.BiGCN(k, 64, 64, dev, gemm_mode=mode).to(dev)
    m.load_state_dict(ref.state_dict())
    ref.train(train); m.train(train)
    bd = with_x(b, b.x).to(dev)
    bd.x = bd.x.to(x_dt).contiguous()
    out0, grads0, none = _run(m, bd, False, train)
    assert none is None
    out1, grads1, xg = _run(m, bd, True, train)
    assert torch.equal(out0, out1)
    for (name, _), g0, g1 in zip(m.named_parameters(), grads0, grads1):
        assert torch.equal(g0, g1), name
    assert xg.dtype == x_dt and xg.shape == bd.x.shape
    gtol = 1e-4 if mode != "tf32" else (1e-2 if shape == "twitter15" else 3e-2)
    n = b.x.shape[0]
    keep = masks_for(m.TDrumorGCN.last_seed, n, k) if train else [None, None]
    xr = b.x.double().requires_grad_(True)
    want = ref(with_x(b, xr), keep_td=keep[0], keep_bu=keep[1])
    F.nll_loss(want, b.y).backward()
    assert rel_err(out1, want) < (1e-2 if mode == "tf32" else 2.2e-5)
    if mode == "bf16":
        assert_bf16_close(xg, xr.grad, 1e-4)
    else:
        assert rel_err(xg, xr.grad) < gtol
    for (name, p), q in zip(m.named_parameters(), ref.parameters()):
        assert rel_err(p.grad, q.grad) < gtol, name


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["tf32x3", "sparse"])
def test_single_direction_x_grad(dev, mode):
    """TDrumorGCN alone, BUrumorGCN alone (one weight, n_w = 1) and both called on one x (autograd sums the two)."""
    import bigcn_b200
    b = make_batch("twitter15", 8, seed=9, train=False, in_feats=5000)
    ref = fixed_oracle(5000, seed=8).double().eval()
    bd = with_x(b, b.x).to(dev)
    td = bigcn_b200.TDrumorGCN(5000, 64, 64, dev, gemm_mode=mode).to(dev).eval()
    bu = bigcn_b200.BUrumorGCN(5000, 64, 64, dev, gemm_mode=mode).to(dev).eval()
    td.load_state_dict(ref.TDrumorGCN.state_dict())
    bu.load_state_dict(ref.BUrumorGCN.state_dict())
    torch.manual_seed(1)
    gt, gb = torch.randn(b.rootindex.numel(), 128), torch.randn(b.rootindex.numel(), 128)
    for mods in ((td,), (bu,), (td, bu)):
        x = bd.x.detach().clone().requires_grad_(True)
        xr = b.x.double().requires_grad_(True)
        loss, want = 0, 0
        for mod in mods:
            r = ref.TDrumorGCN if mod is td else ref.BUrumorGCN
            g = gt if mod is td else gb
            loss = loss + (mod(with_x(bd, x)) * g.to(dev)).sum()
            want = want + (r(with_x(b, xr)) * g.double()).sum()
        loss.backward()
        want.backward()
        assert rel_err(x.grad, xr.grad) < 1e-4, [type(q).__name__ for q in mods]


@pytest.mark.gpu
def test_upstream_module_gets_gradient(dev):
    """x = Linear(emb): the upstream weight's gradient flows through the fused model and matches the oracle."""
    import bigcn_b200
    b = make_batch("pheme", 30, seed=12, train=False, in_feats=768)
    torch.manual_seed(13)
    emb = torch.randn(b.x.shape[0], 32)
    proj = torch.nn.Linear(32, 768)
    ref = fixed_oracle(768, seed=14).double().eval()
    m = bigcn_b200.BiGCN(768, 64, 64, dev, gemm_mode="tf32x3").to(dev).eval()
    m.load_state_dict(ref.state_dict())
    proj_d = copy.deepcopy(proj).to(dev)
    proj_r = copy.deepcopy(proj).double()
    bd = with_x(b, b.x).to(dev)
    F.nll_loss(m(with_x(bd, proj_d(emb.to(dev)))), bd.y).backward()
    F.nll_loss(ref(with_x(b, proj_r(emb.double()))), b.y).backward()
    assert proj_d.weight.grad is not None
    assert rel_err(proj_d.weight.grad, proj_r.weight.grad) < 1e-4
    assert rel_err(proj_d.bias.grad, proj_r.bias.grad) < 1e-4


@pytest.mark.gpu
def test_saliency_frozen_model(dev):
    """All parameters frozen, only x requires grad: x.grad is right; a bf16 x under tf32x3 gets a bf16 x.grad."""
    import bigcn_b200
    b = make_batch("pheme", 24, seed=21, train=False, in_feats=768)
    b.x = b.x.to(torch.bfloat16).float()
    ref = fixed_oracle(768, seed=22).double().eval()
    m = bigcn_b200.BiGCN(768, 64, 64, dev, gemm_mode="tf32x3").to(dev).eval()
    m.load_state_dict(ref.state_dict())
    m.requires_grad_(False)
    xr = b.x.double().requires_grad_(True)
    want = ref(with_x(b, xr))
    want.gather(1, b.y.view(-1, 1)).sum().backward()
    bd = with_x(b, b.x).to(dev)
    for dt in (torch.float32, torch.bfloat16):
        x = bd.x.detach().to(dt).clone().requires_grad_(True)
        m(with_x(bd, x)).gather(1, bd.y.view(-1, 1)).sum().backward()
        assert x.grad is not None and x.grad.dtype == dt
        assert all(p.grad is None for p in m.parameters())
        if dt == torch.float32:
            assert rel_err(x.grad, xr.grad) < 1e-4
        else:
            assert_bf16_close(x.grad, xr.grad, 1e-4)
