"""gemm_mode='bf16': data.x stored in bfloat16, X * W and dW1 on tcgen05 kind::f16 with the small operand split into
bf16 terms.  Every check is against the fp64 / fp32 oracle evaluated on x.float() (a bf16 x widens exactly), at the
fp32-class bars of the tf32x3 mode; plus the input contract of the mode and what it leaves unchanged."""
import copy
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import bigcn_oracle, gcn_oracle
from bigcn_b200.data import Batch, make_batch

pytestmark = pytest.mark.gpu


def rel_err(got, want):
    want = want.detach().cpu().double()
    got = got.detach().cpu().double()
    return float((got - want).abs().max()) / max(float(want.abs().max()), 1e-30)


def bf16_batch(shape, n_trees, seed, train, in_feats=None):
    """(CPU batch whose x is the fp32 widening of a bf16 x, the same batch on the device with x in bf16)"""
    b = make_batch(shape, n_trees, seed=seed, train=train, in_feats=in_feats)
    b.x = b.x.to(torch.bfloat16).float()
    return b, device_batch(b, "cuda", torch.bfloat16)


def device_batch(b, dev, x_dtype=torch.float32):
    d = Batch(**{k: getattr(b, k).to(dev) for k in Batch._tensor_keys})
    d.x = d.x.to(x_dtype).contiguous()
    return d


def make_pair(k, dev, seed, mode="bf16"):
    import bigcn_b200
    torch.manual_seed(seed)
    ref = bigcn_oracle.BiGCN(k, 64, 64)
    with torch.no_grad():
        for p in ref.parameters():
            if p.dim() == 1:
                p.uniform_(-0.1, 0.1)
    m = bigcn_b200.BiGCN(k, 64, 64, dev, gemm_mode=mode).to(dev)
    m.load_state_dict(ref.state_dict())
    return ref, m


def masks_for(m, n, k):
    seed = m.TDrumorGCN.last_seed
    ktd = torch.from_numpy(gcn_oracle.dropout_keep_mask(seed, 0, np.arange(n), 64 + k, 0.5))
    kbu = torch.from_numpy(gcn_oracle.dropout_keep_mask(seed, 1, np.arange(n), 64 + k, 0.5))
    return ktd, kbu


def debug_set(key, value):
    import bigcn_b200
    lib = bigcn_b200.lib()
    lib.bigcn_debug_set.argtypes = [C.c_int, C.c_int]
    lib.bigcn_debug_set.restype = None
    lib.bigcn_debug_set(key, value)


# ---------------------------------------------------------------------------------------------- X * W alone
@pytest.mark.parametrize("shape,n_trees,k", [("twitter15", 3, 5000), ("twitter15", 9, 5000), ("twitter15", 2, 64),
                                              ("pheme", 5, 768), ("pheme", 2, 768), ("pheme", 7, 776)])
def test_xw_bf16_matches_fp64(dev, shape, n_trees, k):
    """K = 776: not a multiple of the 32-element K block; every batch here has N off the 256-row tile."""
    from bigcn_b200 import ops
    torch.manual_seed(0)
    b = make_batch(shape, n_trees, seed=11, train=False, in_feats=k)
    x = b.x.to(torch.bfloat16)
    w_td, w_bu = torch.randn(64, k) * 0.05, torch.randn(64, k) * 0.05
    want = x.double() @ torch.cat([w_td, w_bu]).double().t()
    tol = 2e-6 if shape != "pheme" else 1e-5
    xd = x.to(dev)
    got = ops.xw(xd, [w_td.to(dev), w_bu.to(dev)], "bf16")
    assert got.dtype == torch.float32 and got.shape == want.shape
    assert rel_err(got, want) < tol
    one = ops.xw(xd, [w_bu.to(dev)], "bf16")            # single direction, N = 64 MMA
    assert rel_err(one, want[:, 64:]) < tol


def test_torch_ops_bf16(dev):
    import bigcn_b200.torch_ops  # noqa: F401  (registers the ops)
    from torch._subclasses.fake_tensor import FakeTensorMode
    torch.manual_seed(1)
    b = make_batch("pheme", 6, seed=3, train=False)
    x = b.x.to(torch.bfloat16)
    n, k = x.shape
    w = torch.randn(64, k) * 0.05
    t = torch.randn(n, 64)
    xd = x.to(dev)
    y = torch.ops.bigcn_b200.xw(xd, w.to(dev), "bf16")
    assert y.dtype == torch.float32
    assert rel_err(y, x.double() @ w.double().t()) < 1e-5
    dw = torch.ops.bigcn_b200.xw_wgrad(xd, t.to(dev), "bf16")
    assert dw.dtype == torch.float32 and dw.shape == (64, k)
    assert rel_err(dw, t.double().t() @ x.double()) < 1e-5
    wd = w.to(dev).requires_grad_(True)
    g = torch.randn(n, 64)
    torch.ops.bigcn_b200.xw(xd, wd, "bf16").backward(g.to(dev))
    assert rel_err(wd.grad, g.double().t() @ x.double()) < 1e-5
    with FakeTensorMode():
        fx = torch.empty(n, k, dtype=torch.bfloat16, device=dev)
        fy = torch.ops.bigcn_b200.xw(fx, torch.empty(64, k, device=dev), "bf16")
        fg = torch.ops.bigcn_b200.xw_wgrad(fx, torch.empty(n, 64, device=dev), "bf16")
        assert fy.dtype == torch.float32 and tuple(fy.shape) == (n, 64)
        assert fg.dtype == torch.float32 and tuple(fg.shape) == (64, k)


# ---------------------------------------------------------------------------------------------- the model
@pytest.mark.parametrize("shape,k,trees", [("twitter15", 5000, 16), ("pheme", 768, 24)])
def test_model_bf16_eval(dev, shape, k, trees):
    """The bars of the tf32x3 row of test_model_in_tf32_mode; the same model in tf32x3 on x.float() alongside."""
    b, bd = bf16_batch(shape, trees, seed=2, train=False, in_feats=k)
    ref, m = make_pair(k, dev, seed=1)
    ref.eval(); m.eval()
    want = ref(b)
    got = m(bd)
    m.check_inputs()
    assert rel_err(got, want) < 2.2e-5
    assert torch.equal(got.argmax(1).cpu(), want.argmax(1))
    with torch.no_grad():                                 # the inference path (two C-ABI calls)
        assert rel_err(m(bd), want) < 2.2e-5
    m3 = copy.deepcopy(m)
    m3.gemm_mode = "tf32x3"
    got3 = m3(device_batch(b, dev))
    assert rel_err(got3, want) < 2.2e-5
    assert torch.equal(got3.argmax(1).cpu(), want.argmax(1))


@pytest.mark.parametrize("shape,k,trees", [("twitter15", 5000, 10), ("pheme", 768, 40)])
def test_training_bf16(dev, shape, k, trees):
    """Train mode with the kernel's Philox mask injected into the oracle: log-probs 1e-5 (2.2e-5 for dense K = 768),
    all ten gradients 1e-4, with dense_roots on and off.  With one column split of the dense-root product (knob 15)
    the two forwards are the same sums in the same order: bit-identical log-probs."""
    b, bd = bf16_batch(shape, trees, seed=4, train=True, in_feats=k)
    n = b.x.shape[0]
    ltol = 1e-5 if k == 5000 else 2.2e-5
    outs = {}
    debug_set(15, 1)
    try:
        for dense in (False, True):
            ref, m = make_pair(k, dev, seed=3)
            ref.train(); m.train()
            for mod in (m.TDrumorGCN, m.BUrumorGCN):
                mod.dense_roots = dense
                mod.seed, mod._calls = 777, 0
            got = m(bd)
            m.check_inputs()
            ktd, kbu = masks_for(m, n, k)
            want = ref(b, keep_td=ktd, keep_bu=kbu)
            assert rel_err(got, want) < ltol, dense
            torch.nn.functional.nll_loss(want, b.y).backward()
            torch.nn.functional.nll_loss(got, bd.y).backward()
            for (name, p), (_, q) in zip(m.named_parameters(), ref.named_parameters()):
                e = rel_err(p.grad, q.grad)
                assert e < 1e-4, f"dense_roots={dense} {name}: {e:.3e}"
            outs[dense] = got.detach().clone()
    finally:
        debug_set(15, 0)
    assert torch.equal(outs[False], outs[True])


def test_fused_trainer_bf16(dev):
    """Three rotating bf16 batches: parameters bit-identical with and without CUDA-graph replay and between
    prefetched (next_data) and self-contained steps; the first step's loss within 1e-5 of the module path."""
    import bigcn_b200
    cpu = [bf16_batch("pheme", 60, seed=50 + i, train=True) for i in range(3)]
    batches = [d for _, d in cpu]
    out = {}
    for name, graphs, prefetch in (("plain", False, False), ("prefetch", False, True), ("prefetch+graphs", True, True)):
        _, m = make_pair(768, dev, seed=6)
        m.train()
        tr = bigcn_b200.FusedTrainer(m, lr=5e-4, weight_decay=1e-4, graphs=graphs)
        losses = [tr.step(batches[i % 3], next_data=batches[(i + 1) % 3] if prefetch else None).clone() for i in range(9)]
        tr.check_inputs()
        out[name] = (tr.flat.clone(), tr.exp_avg.clone(), torch.cat(losses), tr)
    assert out["prefetch+graphs"][3].graph_replays >= 2
    for name in ("prefetch", "prefetch+graphs"):
        for a, c in zip(out["plain"][:3], out[name][:3]):
            assert torch.equal(a, c), name
    # the first step against the module path with the same dropout seed
    _, m = make_pair(768, dev, seed=6)
    m.train()
    for mod in (m.TDrumorGCN, m.BUrumorGCN):
        mod.seed, mod._calls = 4242, 0
    want = float(torch.nn.functional.nll_loss(m(batches[0]), batches[0].y).detach())
    _, m2 = make_pair(768, dev, seed=6)
    m2.train()
    tr = bigcn_b200.FusedTrainer(m2, lr=5e-4, weight_decay=1e-4, graphs=False)
    got = float(tr.step(batches[0], seed=4242))
    assert abs(got - want) <= 1e-5 * max(1.0, abs(want))


@pytest.mark.parametrize("shape,k", [("twitter16", 520), ("pheme", 768)])
def test_gcnconv_bf16(dev, shape, k):
    import bigcn_b200
    torch.manual_seed(5)
    b = make_batch(shape, 7 if shape != "pheme" else 60, seed=6, train=True, in_feats=k)
    x = b.x.to(torch.bfloat16)
    ref = gcn_oracle.GCNConv(k, 64)
    conv = bigcn_b200.GCNConv(k, 64, gemm_mode="bf16").to(dev)
    conv.load_state_dict(ref.state_dict())
    want = ref(x.float(), b.edge_index)
    got = conv(x.to(dev), b.edge_index.to(dev))
    assert rel_err(got, want) < 1e-5
    g = torch.randn_like(want)
    want.backward(g); got.backward(g.to(dev))
    assert rel_err(conv.lin.weight.grad, ref.lin.weight.grad) < 1e-4
    assert rel_err(conv.bias.grad, ref.bias.grad) < 1e-4


# ---------------------------------------------------------------------------------------------- input contract
def test_bf16_input_contract(dev):
    import bigcn_b200
    from bigcn_b200 import ops
    b, bd = bf16_batch("pheme", 6, seed=8, train=False)
    _, m = make_pair(768, dev, seed=9)
    m.eval()
    with torch.no_grad():
        m(bd)
        bad = device_batch(b, dev)                              # fp32 x: never cast silently
        with pytest.raises(bigcn_b200.BigcnError, match="bfloat16"):
            m(bad)
        bad.x = ops.SparseX.from_torch_csr(b.x.to_sparse_csr().to(dev))
        with pytest.raises(bigcn_b200.BigcnError):
            m(bad)
        flat = torch.zeros(bd.x.numel() + 8, dtype=torch.bfloat16, device=dev)
        bad.x = flat[1:1 + bd.x.numel()].view(bd.x.shape)      # contiguous, 2 bytes off the 16-byte boundary
        bad.x.copy_(bd.x)
        with pytest.raises(bigcn_b200.BigcnError, match="16-byte"):
            m(bad)
        with pytest.raises(bigcn_b200.BigcnError, match="contiguous"):
            ops.xw(bd.x.t(), [torch.zeros(64, bd.x.shape[0], device=dev)], "bf16")
    b2, bd2 = bf16_batch("twitter15", 3, seed=8, train=False, in_feats=5004)
    _, m2 = make_pair(5004, dev, seed=9)
    with torch.no_grad(), pytest.raises(bigcn_b200.BigcnError, match="multiple of 8"):
        m2.eval()(bd2)
    with pytest.raises(bigcn_b200.BigcnError):                  # the edge-weighted GCNConv has no bf16 form
        conv = bigcn_b200.GCNConv(768, 64, gemm_mode="bf16").to(dev)
        conv(bd.x, bd.edge_index, torch.ones(bd.edge_index.shape[1], device=dev))


@pytest.mark.parametrize("mode", ["tf32x3", "sparse"])
def test_bf16_x_in_other_modes_is_upcast(dev, mode):
    """Unchanged behaviour: a bf16 x under any other mode is widened to fp32 first; same result bit for bit."""
    b, bd = bf16_batch("twitter15", 5, seed=12, train=False)
    _, m = make_pair(5000, dev, seed=13, mode=mode)
    m.eval()
    got = m(bd)
    want = m(device_batch(b, dev))
    assert torch.equal(got, want)


def test_bf16_dense_roots_auto(dev):
    _, bow = bf16_batch("twitter15", 3, seed=1, train=True)
    _, dense = bf16_batch("pheme", 24, seed=1, train=True)
    _, m = make_pair(5000, dev, seed=1)
    assert m.TDrumorGCN.resolved_dense_roots(bow.x) is False
    _, m = make_pair(768, dev, seed=1)
    assert m.TDrumorGCN.resolved_dense_roots(dense.x) is True
    # 'auto' never picks bf16
    import bigcn_b200
    a = bigcn_b200.BiGCN(768, 64, 64, dev).to(dev)
    assert a.TDrumorGCN.resolved_gemm_mode(dense.x) == "tf32x3"


# ---------------------------------------------------------------------------------------------- PHEME v1 width
def test_pheme_v1_width(dev):
    """in_feats = 256 * 768 = 196,608 (BiGCN_Twitter.py:140-144 with PHEME's v1 features), four trees: eval and one
    training step at the fp32 bars."""
    k = 196608
    b, bd = bf16_batch("pheme", 4, seed=14, train=True, in_feats=k)
    n = b.x.shape[0]
    ref, m = make_pair(k, dev, seed=15)
    ref.eval(); m.eval()
    assert rel_err(m(bd), ref(b)) < 2.2e-5
    ref.train(); m.train()
    got = m(bd)
    m.check_inputs()
    ktd, kbu = masks_for(m, n, k)
    want = ref(b, keep_td=ktd, keep_bu=kbu)
    assert rel_err(got, want) < 2.2e-5
    torch.nn.functional.nll_loss(want, b.y).backward()
    torch.nn.functional.nll_loss(got, bd.y).backward()
    for (name, p), (_, q) in zip(m.named_parameters(), ref.named_parameters()):
        e = rel_err(p.grad, q.grad)
        assert e < 1e-4, f"{name}: {e:.3e}"
