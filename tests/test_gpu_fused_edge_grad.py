"""Learnt edge weights on the fused step: ``FusedTrainer(..., edge_grad=True)`` forms d loss / d edge_weight of every
direction whose weight requires grad and hands it to autograd as ``loss.backward()`` would.  References: the module
path (``BiGCN(data)`` + ``F.nll_loss`` + ``backward``), the fp64 oracle, and ``edge_weights=True`` on detached copies
for everything that is not an edge gradient.  Batch and oracle helpers are those of test_gpu_fused_edge_weight.py."""
import copy
import ctypes as C
import types

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from bigcn_b200.data import make_batch
from test_gpu_fused_edge_weight import (K, MODES, Data, assert_same_state, edge_case_batch, mode_batches, on_device,
                                        oracle)

gpu = pytest.mark.gpu


def leaf(w, dev):
    return torch.as_tensor(w, dtype=torch.float32).to(dev).requires_grad_()


def rand_weights(d, seed):
    g = torch.Generator().manual_seed(seed)
    return [torch.rand(ei.shape[1], generator=g) * 1.9 + 0.1 for ei in (d.edge_index, d.BU_edge_index)]


def with_weights(d, td, bu):
    out = Data(**{k: v for k, v in vars(d).items() if k not in ("edge_weight", "BU_edge_weight")})
    if td is not None:
        out.edge_weight = td
    if bu is not None:
        out.BU_edge_weight = bu
    return out


def max_rel(got, want):
    return float((got.double() - want.double()).abs().max()) / max(float(want.double().abs().max()), 1e-30)


# ---------------------------------------------------------------------------------------------- module path, oracle
@gpu
@pytest.mark.parametrize("which", ["both", "td", "bu"])
@pytest.mark.parametrize("mode", list(MODES))
def test_edge_grad_equals_module_path(dev, mode, which):
    """Train mode, the same Philox seed: the fused step's edge gradients against the module path's .grad on the same
    weighted batch, within 1e-6 of max|g|; the test reports whether they are bit-identical."""
    import bigcn_b200
    _, k, gm, _ = MODES[mode]
    d = mode_batches(mode, dev, 1)[0]
    tw, bw = rand_weights(d, 11)
    torch.manual_seed(5)
    m = bigcn_b200.BiGCN(k, 64, 64, dev, gemm_mode=gm).to(dev).train()
    tr = bigcn_b200.FusedTrainer(m, lr=5e-3, weight_decay=1e-4, edge_grad=True, graphs=False)
    use = (which != "bu", which != "td")
    mod_w = [leaf(w, dev) if u else None for w, u in zip((tw, bw), use)]
    fus_w = [leaf(w, dev) if u else None for w, u in zip((tw, bw), use)]
    for mod in (m.TDrumorGCN, m.BUrumorGCN):
        mod._calls = 0
    F.nll_loss(m(with_weights(d, *mod_w)), d.y).backward()
    seed = m.TDrumorGCN.last_seed
    tr.step(with_weights(d, *fus_w), seed=seed)
    tr.check_inputs()
    identical = True
    for a, b in zip(fus_w, mod_w):
        if a is None:
            continue
        assert a.grad is not None and a.grad.dtype == torch.float32
        assert float((a.grad - b.grad).abs().max()) <= 1e-6 * float(b.grad.abs().max())
        identical &= bool(torch.equal(a.grad, b.grad))
    print(f"fused vs module edge gradient ({mode}, {which}): {'bit-identical' if identical else 'within 1e-6 of max|g|'}")


@gpu
@pytest.mark.parametrize("which", ["both", "td", "bu"])
@pytest.mark.parametrize("gemm", ["sparse", "tf32x3"])
def test_edge_grad_matches_oracle(dev, gemm, which):
    """edge_case_batch (self-loop edge, duplicate edge, zero weights, a BU hub row, asymmetric DropEdge) in eval mode:
    the edge gradients within 1e-4 of max|g| of the fp64 oracle's autograd."""
    import bigcn_b200
    b = edge_case_batch(17, train=True)
    ref = oracle(K, 6).eval()
    m = bigcn_b200.BiGCN(K, 64, 64, dev, gemm_mode=gemm).to(dev).eval()
    m.load_state_dict(ref.state_dict())
    tr = bigcn_b200.FusedTrainer(m, lr=5e-4, weight_decay=1e-4, edge_grad=True, graphs=False)
    use = (which != "bu", which != "td")
    rw = [torch.tensor(w, dtype=torch.float64, requires_grad=True) if u else None for w, u in zip(b.w, use)]
    dref = types.SimpleNamespace(**vars(b))
    dref.edge_weight, dref.BU_edge_weight = rw
    F.nll_loss(ref(dref), b.y).backward()
    fw = [leaf(w, dev) if u else None for w, u in zip(b.w, use)]
    tr.step(on_device(b, dev, *fw))
    tr.check_inputs()
    for a, r in zip(fw, rw):
        if a is not None:
            assert max_rel(a.grad.cpu(), r.grad) <= 1e-4


# ---------------------------------------------------------------------------------------------- parameters untouched
@gpu
@pytest.mark.parametrize("mode", list(MODES))
def test_parameters_equal_detached_weights(dev, mode):
    """Pipelined and replayed steps: loss, log-probs, parameters and both Adam moments bit-identical to an
    edge_weights=True trainer fed detached copies of the same weights."""
    import bigcn_b200
    _, k, gm, _ = MODES[mode]
    torch.manual_seed(5)
    m0 = bigcn_b200.BiGCN(k, 64, 64, dev, gemm_mode=gm).to(dev).train()
    m1 = copy.deepcopy(m0)
    eg = bigcn_b200.FusedTrainer(m0, lr=5e-3, weight_decay=1e-4, edge_grad=True)
    ew = bigcn_b200.FusedTrainer(m1, lr=5e-3, weight_decay=1e-4, edge_weights=True)
    bs = mode_batches(mode, dev)
    ws = [rand_weights(d, 20 + i) for i, d in enumerate(bs)]
    grad_b = [with_weights(d, leaf(t, dev), leaf(u, dev)) for d, (t, u) in zip(bs, ws)]
    det_b = [with_weights(d, t.to(dev), u.to(dev)) for d, (t, u) in zip(bs, ws)]
    order = [0, 1, 2] * 3 + [0]
    for j, i in enumerate(order):
        nx = order[j + 1] if j + 1 < len(order) else None
        l0 = eg.step(grad_b[i], next_data=None if nx is None else grad_b[nx])
        l1 = ew.step(det_b[i], next_data=None if nx is None else det_b[nx])
        assert torch.equal(l0, l1), j
        assert torch.equal(eg.last_logp, ew.last_logp), j
        assert_same_state(eg, ew)
    assert eg.graph_replays > 0
    for d in grad_b:
        assert d.edge_weight.grad is not None and d.BU_edge_weight.grad is not None
    eg.check_inputs()


# ---------------------------------------------------------------------------------------------- non-leaf weights
class EdgeScorer(torch.nn.Module):
    """sigmoid(MLP(edge features)): a learnt edge mask upstream of BiGCN."""

    def __init__(self, f):
        super().__init__()
        self.mlp = torch.nn.Sequential(torch.nn.Linear(f, 16), torch.nn.Tanh(), torch.nn.Linear(16, 1))

    def forward(self, feats):
        return torch.sigmoid(self.mlp(feats)).squeeze(1)


@gpu
@pytest.mark.parametrize("case", ["scorer", "shared", "fp16"])
def test_non_leaf_shared_and_cast_weights(dev, case):
    """scorer: TD and BU weights from an edge-scoring module; its parameters' .grad after one fused step within 1e-5
    of the module path's.  shared: one tensor for both directions gets the sum of the two gradients.  fp16: the
    gradient passes back through the cast (within fp16 rounding of the module path's)."""
    import bigcn_b200
    b = edge_case_batch(23, train=False)       # TD and BU lists of the same length (BU = TD reversed)
    m = bigcn_b200.BiGCN(K, 64, 64, dev, gemm_mode="sparse").to(dev).eval()
    m.load_state_dict(oracle(K, 8).float().state_dict())
    tr = bigcn_b200.FusedTrainer(m, lr=5e-4, weight_decay=1e-4, edge_grad=True)
    d = on_device(b, dev)
    e = d.edge_index.shape[1]
    assert d.BU_edge_index.shape[1] == e

    def make():
        if case == "scorer":
            torch.manual_seed(1)
            sc = EdgeScorer(8).to(dev)
            g = torch.Generator().manual_seed(2)
            f_td, f_bu = (torch.randn(e, 8, generator=g).to(dev) for _ in range(2))
            return sc, list(sc.parameters()), lambda: (sc(f_td), sc(f_bu))
        w = torch.tensor(b.w[0], device=dev, dtype=torch.float16 if case == "fp16" else torch.float32).requires_grad_()
        return None, [w], lambda: (w, w) if case == "shared" else (w, None)

    _, pm, fm = make()
    F.nll_loss(m(with_weights(d, *fm())), d.y).backward()        # module path (reads the parameters before the step)
    _, pf, ff = make()
    tr.step(with_weights(d, *ff()))
    tr.check_inputs()
    for a, r in zip(pf, pm):
        assert a.grad is not None and a.grad.dtype == r.dtype and a.grad.shape == r.shape
        assert max_rel(a.grad, r.grad) <= (1e-3 if case == "fp16" else 1e-5), case
    if case == "shared":                       # against the sum of the two single-direction gradients
        tw, bw = leaf(b.w[0], dev), leaf(b.w[0], dev)
        m2 = bigcn_b200.BiGCN(K, 64, 64, dev, gemm_mode="sparse").to(dev).eval()
        m2.load_state_dict(oracle(K, 8).float().state_dict())
        tr2 = bigcn_b200.FusedTrainer(m2, lr=5e-4, weight_decay=1e-4, edge_grad=True)
        tr2.step(with_weights(d, tw, bw))
        assert torch.equal(pf[0].grad, tw.grad + bw.grad)


# ---------------------------------------------------------------------------------------------- prepared == inline
def _rotation(dev, copies):
    """The same batches `copies` times over, each copy with weight tensors of its own: weighted with grad (both, TD
    only), weighted without grad, unweighted."""
    base = [edge_case_batch(70 + i, train=True) for i in range(3)]
    small = [on_device(make_batch("twitter15", 2, seed=60 + i, train=True, in_feats=K, sizes=np.array([3, 4])), dev)
             for i in range(2)]
    out = []
    for _ in range(copies):
        bs = [on_device(base[0], dev, leaf(base[0].w[0], dev), leaf(base[0].w[1], dev)),
              on_device(base[1], dev, leaf(base[1].w[0], dev), None),
              on_device(base[2], dev, torch.tensor(base[2].w[0], device=dev), torch.tensor(base[2].w[1], device=dev))]
        out.append(small[:1] + bs + [small[1]])
    return out


def _grads(d):
    return [None if w is None or w.grad is None else w.grad.clone()
            for w in (getattr(d, "edge_weight", None), getattr(d, "BU_edge_weight", None))]


def _clear(d):
    for w in (getattr(d, "edge_weight", None), getattr(d, "BU_edge_weight", None)):
        if w is not None:
            w.grad = None


def _same_grads(a, b, tag):
    for x, y in zip(_grads(a), _grads(b)):
        assert (x is None) == (y is None), tag
        if x is not None:
            assert torch.equal(x, y), tag


@gpu
@pytest.mark.parametrize("graphs", [False, True])
def test_prepared_equals_inline(dev, graphs):
    """step(b_i, next_data=b_i+1) over a rotation of weighted-with-grad, weighted-without and unweighted batches equals
    the same steps without next_data bit for bit: loss, parameters, Adam moments and edge gradients.  Then a weight
    written in place after it was prepared, and one replaced by a new tensor (at a recycled address when the caching
    allocator hands the old block back), give the inline result on the new values."""
    import bigcn_b200
    torch.manual_seed(2)
    m0 = bigcn_b200.BiGCN(K, 64, 64, dev, gemm_mode="sparse").to(dev).train()
    m1 = copy.deepcopy(m0)
    pipe = bigcn_b200.FusedTrainer(m0, lr=5e-3, weight_decay=1e-4, edge_grad=True, graphs=graphs)
    inline = bigcn_b200.FusedTrainer(m1, lr=5e-3, weight_decay=1e-4, edge_grad=True, graphs=graphs)
    rp, ri = _rotation(dev, 2)
    order = [0, 1, 2, 3, 4, 1, 2, 0, 3, 1, 2, 4, 1]

    def both(i, nx, tag):
        l0 = pipe.step(rp[i], next_data=None if nx is None else rp[nx])
        l1 = inline.step(ri[i])
        assert torch.equal(l0, l1), tag
        assert torch.equal(pipe.last_logp, inline.last_logp), tag
        assert_same_state(pipe, inline)
        _same_grads(rp[i], ri[i], tag)
        _clear(rp[i])
        _clear(ri[i])

    for j, i in enumerate(order):
        both(i, order[j + 1] if j + 1 < len(order) else None, j)
    if graphs:
        assert pipe.graph_replays > 0
    # written in place after it was prepared
    both(0, 1, "before in-place")
    with torch.no_grad():
        for d in (rp[1], ri[1]):
            d.edge_weight.mul_(0.5)
            d.BU_edge_weight[:5] = 3.0
    both(1, None, "in place")
    # replaced by another tensor after it was prepared
    both(0, 2, "before replace")
    old = rp[2].edge_weight.data_ptr()
    e = rp[2].edge_index.shape[1]
    rp[2].edge_weight = ri[2].edge_weight = None
    new_vals = torch.linspace(0.2, 1.7, e, device=dev)
    rp[2].edge_weight = torch.empty(e, device=dev).copy_(new_vals).requires_grad_()
    ri[2].edge_weight = new_vals.clone().requires_grad_()
    print(f"replacement weight at a recycled address: {rp[2].edge_weight.data_ptr() == old}")
    both(2, None, "replaced")
    pipe.check_inputs()
    inline.check_inputs()


# ---------------------------------------------------------------------------------------------- accumulation
@gpu
def test_accumulation_and_no_aliasing(dev):
    """Two steps accumulate .grad as autograd does (g1 + g2, against a trainer whose .grad is cleared after each step),
    and a gradient taken from .grad does not change when a later step or replay runs."""
    import bigcn_b200
    torch.manual_seed(4)
    m0 = bigcn_b200.BiGCN(K, 64, 64, dev, gemm_mode="sparse").to(dev).train()
    m1 = copy.deepcopy(m0)
    acc = bigcn_b200.FusedTrainer(m0, lr=5e-3, weight_decay=1e-4, edge_grad=True, graphs=True)
    ref = bigcn_b200.FusedTrainer(m1, lr=5e-3, weight_decay=1e-4, edge_grad=True, graphs=False)
    b = edge_case_batch(31, train=True)
    da = on_device(b, dev, leaf(b.w[0], dev), leaf(b.w[1], dev))
    dr = on_device(b, dev, leaf(b.w[0], dev), leaf(b.w[1], dev))
    gs = []
    for _ in range(2):
        acc.step(da)
        ref.step(dr)
        gs.append(_grads(dr))
        _clear(dr)
    for q, w in enumerate((da.edge_weight, da.BU_edge_weight)):
        assert torch.equal(w.grad, gs[0][q] + gs[1][q])
    taken = [da.edge_weight.grad, da.BU_edge_weight.grad]
    snap = [t.clone() for t in taken]
    _clear(da)
    for _ in range(3):                        # the second sighting is captured, then replayed
        acc.step(da)
        ref.step(dr)
        _same_grads(da, dr, "replay")
        _clear(da)
        _clear(dr)
    other = on_device(edge_case_batch(32, train=True), dev)
    acc.step(other)
    torch.cuda.synchronize()
    assert acc.graph_replays >= 2
    for t, s in zip(taken, snap):
        assert torch.equal(t, s)


# ---------------------------------------------------------------------------------------------- no extra work
def _kernel_names(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events()}


@gpu
def test_no_edge_work_without_grad(dev):
    """On an edge_grad=True trainer, weights that do not require grad give results bit-identical to edge_weights=True,
    the same workspace, and no edge-gradient kernel (torch.profiler; a batch with grad shows them); edge_grad=True
    with world_size=2 raises at construction."""
    import bigcn_b200
    torch.manual_seed(6)
    m0 = bigcn_b200.BiGCN(K, 64, 64, dev, gemm_mode="sparse").to(dev).train()
    m1 = copy.deepcopy(m0)
    eg = bigcn_b200.FusedTrainer(m0, lr=5e-3, weight_decay=1e-4, edge_grad=True, graphs=False)
    ew = bigcn_b200.FusedTrainer(m1, lr=5e-3, weight_decay=1e-4, edge_weights=True, graphs=False)
    b = edge_case_batch(41, train=True)
    d = on_device(b, dev, torch.tensor(b.w[0], device=dev), torch.tensor(b.w[1], device=dev))
    names = _kernel_names(lambda: [eg.step(d), ew.step(d)])
    assert torch.equal(eg.last_logp, ew.last_logp)
    assert_same_state(eg, ew)
    assert eg._ws.numel() == ew._ws.numel()
    assert not any("k_wf_edge_dot" in n or "k_w_dweight" in n or "k_w_ddeg" in n for n in names)
    dg = on_device(b, dev, leaf(b.w[0], dev), None)
    names = _kernel_names(lambda: eg.step(dg))
    assert any("k_wf_edge_dot" in n for n in names) and any("k_w_dweight" in n for n in names)
    assert eg._ws.numel() > ew._ws.numel()
    with pytest.raises(bigcn_b200.BigcnError, match="one GPU"):
        bigcn_b200.FusedTrainer(copy.deepcopy(m1), edge_grad=True, world_size=2)


# ---------------------------------------------------------------------------------------------- the C-ABI
def _abi_edge_grad(d, m, prepared):
    """bigcn_batch_prepare (optional) -> features_forward -> features_backward -> features_edge_grad, directly."""
    from bigcn_b200 import _lib as L
    from bigcn_b200.ops import _PNAMES, _as_x, _i64, _make_structs, _p, _stream, edge_weight
    lib = L.lib()
    x, xs = _as_x(d.x, "sparse")
    ei, bu, batch, root = _i64(d.edge_index), _i64(d.BU_edge_index), _i64(d.batch), _i64(d.rootindex)
    ew = (edge_weight(d.edge_weight, ei.shape[1], "edge_weight"), edge_weight(d.BU_edge_weight, bu.shape[1], "BU"))
    mods = {"td": m.TDrumorGCN, "bu": m.BUrumorGCN}
    params = []
    for n in _PNAMES:
        conv = getattr(mods[n[:2]], "conv" + n[4])
        params.append((conv.lin.weight if n[3] == "w" else conv.bias).detach())
    dims, bt, pr = _make_structs(x, ei, bu, batch, root, params, 0, 0, xs, ew)
    o = L.Opts(training=1, p_drop=0.2, seed=9, deg_by=L.DEG_BY["target"], gemm_mode=L.GEMM_MODE["sparse"],
               dir_mask=L.DIR_TD | L.DIR_BU, edge_grad=1)
    st = _stream()
    flags = torch.zeros(1, dtype=torch.int32, device=x.device)
    keep = []
    if prepared:
        nb = lib.bigcn_batch_prepare_edge_bytes(C.byref(dims))
        buf = torch.empty(nb, dtype=torch.uint8, device=x.device)
        keep.append(buf)
        bt.prepared = buf.data_ptr()
        L.check(lib.bigcn_batch_prepare(C.byref(dims), C.byref(bt), C.byref(o), _p(flags), _p(buf), nb, st), "prepare")
        L.check(lib.bigcn_batch_prepare_join(st), "prepare_join")
    nws = lib.bigcn_features_edge_workspace_bytes(C.byref(dims), 1)
    ws = torch.empty(nws, dtype=torch.uint8, device=x.device)
    feat = torch.empty(dims.B, 256, device=x.device)
    L.check(lib.bigcn_features_forward(C.byref(dims), C.byref(bt), C.byref(pr), C.byref(o), _p(feat), _p(flags), _p(ws),
                                       nws, st), "forward")
    gfeat = torch.randn(dims.B, 256, generator=torch.Generator().manual_seed(3)).to(x.device)
    grads = [torch.empty_like(p) for p in params]
    gr = L.Params()
    for n, t in zip(_PNAMES, grads):
        setattr(gr, n, _p(t))
    L.check(lib.bigcn_features_backward(C.byref(dims), C.byref(bt), C.byref(pr), C.byref(o), _p(gfeat), C.byref(gr),
                                        _p(ws), nws, st), "backward")
    dew = [torch.empty(dims.E_td, device=x.device), torch.empty(dims.E_bu, device=x.device)]
    L.check(lib.bigcn_features_edge_grad(C.byref(dims), C.byref(bt), C.byref(o), _p(dew[0]), _p(dew[1]), _p(ws), nws,
                                         st), "edge_grad")
    torch.cuda.synchronize()
    assert int(flags.item()) == 0
    return feat, grads, dew


@gpu
def test_abi_prepared_equals_inline(dev):
    """bigcn_features_edge_grad on a prepared batch equals the same call on the inline batch bit for bit (and so do
    the features and the parameter gradients)."""
    import bigcn_b200
    b = edge_case_batch(51, train=True)
    m = bigcn_b200.BiGCN(K, 64, 64, dev, gemm_mode="sparse").to(dev)
    m.load_state_dict(oracle(K, 2).float().state_dict())
    d = on_device(b, dev, torch.tensor(b.w[0], device=dev), torch.tensor(b.w[1], device=dev))
    fa, ga, ea = _abi_edge_grad(d, m, False)
    fb, gb, eb = _abi_edge_grad(d, m, True)
    assert torch.equal(fa, fb)
    for x, y in zip(ga, gb):
        assert torch.equal(x, y)
    for x, y in zip(ea, eb):
        assert torch.equal(x, y)
    assert float(ea[0].abs().max()) > 0 and float(ea[1].abs().max()) > 0
