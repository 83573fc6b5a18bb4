"""Edge-weighted training on the fused path: ``FusedTrainer(..., edge_weights=True)`` steps batches that carry
``data.edge_weight`` / ``data.BU_edge_weight``, their normalisation prepared a step ahead with ``next_data``; and
``DeviceForest`` keeps one weight per tree edge and hands every batch the weights of the edges each direction kept.
The reference for weighted values is the fp64 oracle with the direction's weights passed to both of its GCNConvs
(``WeightedTD`` / ``WeightedBU`` below, as in test_gpu_edge_weight.py) and torch.optim.Adam in the reference's lr groups."""
import copy
import types

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import bigcn_oracle, gcn_oracle
from bigcn_b200.data import make_batch

gpu = pytest.mark.gpu
K = 64


class Data(types.SimpleNamespace):
    """A duck-typed batch that takes weak references (the trainer keeps them to the batches it has seen)."""


def rel_err(got, want):
    want = want.detach().cpu().double()
    got = got.detach().cpu().double()
    return float((got - want).abs().max()) / max(float(want.abs().max()), 1e-30)


def edge_case_batch(seed, train, k=K):
    """Single-node trees, a 60-node star (its root is a BU hub row with more than 32 in-edges), random trees; with
    ``train`` TD and BU lose different edges (DropEdge); each list gets a self-loop edge and a duplicate edge.  Weights:
    uniform in [0.1, 2) with every tenth set to 0."""
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
    extra_node = sizes[0] + sizes[1] + 3
    lists = [np.concatenate([ei, [[extra_node], [extra_node]], ei[:, 2:3]], axis=1) for ei in (td, bu)]
    x = np.zeros((n_nodes, k), dtype=np.float32)
    for i in range(n_nodes):
        x[i, rng.choice(k, 5, replace=False)] = rng.integers(1, 4, 5)
    ws = []
    for ei in lists:
        w = rng.uniform(0.1, 2.0, ei.shape[1]).astype(np.float32)
        w[::10] = 0.0
        w[-2] = 1.5
        ws.append(w)
    return types.SimpleNamespace(
        x=torch.from_numpy(x), edge_index=torch.from_numpy(lists[0]), BU_edge_index=torch.from_numpy(lists[1]),
        batch=torch.from_numpy(np.repeat(np.arange(len(sizes)), sizes)),
        rootindex=torch.from_numpy(np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(np.int64)),
        y=torch.from_numpy(rng.integers(0, 4, len(sizes))), w=ws)


def _weighted_forward(self, data, keep=None):
    """bigcn_oracle._RumorGCN.forward with ``getattr(data, self.weight_attr, None)`` handed to conv1 and conv2."""
    x, edge_index = data.x, getattr(data, self.edge_attr)
    dtype = self.conv1.lin.weight.dtype
    ew = getattr(data, self.weight_attr, None)
    if ew is not None:
        ew = ew.to(dtype)
    x1 = copy.copy(x.to(dtype))
    h = self.conv1(x1, edge_index, ew)
    h2 = h.detach()
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


def on_device(b, dev, td_w=None, bu_w=None):
    d = Data(**{k: getattr(b, k).to(dev) for k in ("x", "edge_index", "BU_edge_index", "batch", "rootindex", "y")})
    if td_w is not None:
        d.edge_weight = td_w
    if bu_w is not None:
        d.BU_edge_weight = bu_w
    return d


def state(tr):
    return [t.clone() for t in (tr.flat, tr.exp_avg, tr.exp_avg_sq)]


def assert_same_state(a, b):
    for x, y, name in zip(state(a), state(b), ("params", "exp_avg", "exp_avg_sq")):
        assert torch.equal(x, y), name


# ---------------------------------------------------------------------------------------------- all-ones weights
MODES = {   # mode -> (batch shape, in_feats, gemm_mode of the model, x dtype)
    "sparse": ("twitter15", 5000, "sparse", torch.float32),
    "tf32x3_dense_roots": ("pheme", 256, "auto", torch.float32),
    "bf16": ("pheme", 256, "bf16", torch.bfloat16),
}


def mode_batches(mode, dev, n=3):
    shape, k, _, dt = MODES[mode]
    out = []
    for i in range(n):
        b = make_batch(shape, 6 + 2 * i, seed=30 + i, train=True, in_feats=k)
        if shape == "pheme":
            b.x = torch.tanh(torch.randn(b.x.shape[0], k, generator=torch.Generator().manual_seed(i)))
        d = on_device(b, dev)
        d.x = d.x.to(dt).contiguous()
        out.append(d)
    return out


def with_ones(d):
    w = Data(**vars(d))
    w.edge_weight = torch.ones(d.edge_index.shape[1], device=d.x.device)
    w.BU_edge_weight = torch.ones(d.BU_edge_index.shape[1], device=d.x.device)
    return w


def trainer_pair(mode, dev, **kw):
    import bigcn_b200
    _, k, gm, _ = MODES[mode]
    torch.manual_seed(5)
    m0 = bigcn_b200.BiGCN(k, 64, 64, dev, gemm_mode=gm).to(dev).train()
    m1 = copy.deepcopy(m0)
    return (bigcn_b200.FusedTrainer(m0, lr=5e-3, weight_decay=1e-4, **kw),
            bigcn_b200.FusedTrainer(m1, lr=5e-3, weight_decay=1e-4, edge_weights=True, **kw))


@gpu
@pytest.mark.parametrize("how", ["enqueued", "replayed", "pipelined"])
@pytest.mark.parametrize("mode", list(MODES))
def test_ones_equal_unweighted(dev, mode, how):
    """Weights of 1 on both directions give the unweighted trainer's loss, log-probs, parameters and both Adam moments
    bit for bit after every step: enqueued (graphs off), one batch replayed from a captured graph, and pipelined with
    next_data (prepared weighted batches, captured once seen)."""
    plain, wtd = trainer_pair(mode, dev, graphs=(how != "enqueued"))
    bs = mode_batches(mode, dev)
    ws = [with_ones(d) for d in bs]
    if how == "replayed":
        seq = [(0, None)] * 4
    elif how == "pipelined":
        order = [0, 1, 2] * 3 + [0]          # prepared slots alternate: a (batch, slot, next) repeats every 6 steps
        seq = [(order[i], order[i + 1] if i + 1 < len(order) else None) for i in range(len(order))]
    else:
        seq = [(0, None), (1, None), (2, None)]
    for i, nx in seq:
        l0 = plain.step(bs[i], next_data=None if nx is None else bs[nx])
        l1 = wtd.step(ws[i], next_data=None if nx is None else ws[nx])
        assert torch.equal(l0, l1)
        assert torch.equal(plain.last_logp, wtd.last_logp)
        assert_same_state(plain, wtd)
    plain.check_inputs()
    wtd.check_inputs()
    if how != "enqueued":
        assert wtd.graph_replays > 0


# ---------------------------------------------------------------------------------------------- oracle parity
@gpu
@pytest.mark.parametrize("deg_by", ["target", "source"])
@pytest.mark.parametrize("which", ["both", "td", "bu"])
def test_weighted_steps_match_reference_adam(dev, which, deg_by):
    """Three eval-mode steps on random weights (zeros, self-loops, duplicates, a BU hub row, single-node trees,
    asymmetric DropEdge) against the fp64 oracle with the same weights and torch.optim.Adam in the reference's lr
    groups: loss 1e-5, parameters 2e-5 relative (the bars of test_fused_trainer_matches_reference_adam)."""
    import bigcn_b200
    ref = oracle(K, 3, deg_by)
    m = bigcn_b200.BiGCN(K, 64, 64, dev, gemm_mode="sparse", deg_by=deg_by).to(dev).eval()
    m.load_state_dict(ref.state_dict())
    ref.eval()
    opt = bigcn_oracle.make_optimizer(ref, lr=5e-4, weight_decay=1e-4)
    tr = bigcn_b200.FusedTrainer(m, lr=5e-4, weight_decay=1e-4, edge_weights=True)
    for step in range(3):
        b = edge_case_batch(40 + step, train=True)
        tw = b.w[0] if which in ("both", "td") else None
        bw = b.w[1] if which in ("both", "bu") else None
        d = types.SimpleNamespace(**vars(b))
        if tw is not None:
            d.edge_weight = torch.tensor(tw, dtype=torch.float64)
        if bw is not None:
            d.BU_edge_weight = torch.tensor(bw, dtype=torch.float64)
        loss_ref = F.nll_loss(ref(d), b.y)
        opt.zero_grad()
        loss_ref.backward()
        opt.step()
        loss = tr.step(on_device(b, dev, None if tw is None else torch.tensor(tw, device=dev),
                                 None if bw is None else torch.tensor(bw, device=dev)))
        tr.check_inputs()
        assert abs(float(loss) - float(loss_ref.detach())) <= 1e-5 * max(1.0, abs(float(loss_ref.detach()))), step
    for (name, p), (_, q) in zip(m.named_parameters(), ref.named_parameters()):
        assert rel_err(p, q) < 2e-5, name


@gpu
@pytest.mark.parametrize("mode", ["sparse", "tf32x3"])
def test_train_step_gradient_equals_module_path(dev, mode):
    """Train mode, the same Philox seed: one fused step's flat gradient against the module path's .grad on the same
    weighted batch.  Equal within 1e-6 of max|grad| (the fused tail may order its sums differently from the modules'
    separate head); the test reports whether they were bit-identical."""
    import bigcn_b200
    b = edge_case_batch(13, train=True)
    m = bigcn_b200.BiGCN(K, 64, 64, dev, gemm_mode=mode).to(dev).train()
    m.load_state_dict(oracle(K, 4).float().state_dict())
    tr = bigcn_b200.FusedTrainer(m, lr=5e-4, weight_decay=1e-4, edge_weights=True, graphs=False)
    tw, bw = (torch.tensor(w, device=dev) for w in b.w)
    d = on_device(b, dev, tw, bw)
    for mod in (m.TDrumorGCN, m.BUrumorGCN):
        mod._calls = 0
    m.zero_grad(set_to_none=True)
    out = m(d)
    loss_mod = F.nll_loss(out, d.y)
    loss_mod.backward()
    seed = m.TDrumorGCN.last_seed
    loss = tr.step(d, seed=seed)
    tr.check_inputs()
    identical = True
    for name, p in m.named_parameters():
        g = tr.gviews[name]
        scale = float(p.grad.abs().max())
        assert float((g - p.grad).abs().max()) <= 1e-6 * max(scale, 1e-30), name
        identical &= bool(torch.equal(g, p.grad))
    assert abs(float(loss) - float(loss_mod)) <= 1e-6 * max(1.0, abs(float(loss_mod)))
    print(f"fused vs module gradient ({mode}): {'bit-identical' if identical else 'within 1e-6 of max|grad|'}")


# ---------------------------------------------------------------------------------------------- prepared == inline
@gpu
@pytest.mark.parametrize("mode", ["sparse", "tf32x3"])
def test_prepared_equals_inline(dev, mode):
    """step(b_i, next_data=b_i+1) over a rotation of weighted and unweighted batches equals the same steps without
    next_data bit for bit; the rotation starts with unweighted batches, so the prepared buffers grow mid-run."""
    import bigcn_b200
    torch.manual_seed(2)
    m0 = bigcn_b200.BiGCN(K, 64, 64, dev, gemm_mode=mode).to(dev).train()
    m1 = copy.deepcopy(m0)
    pipe = bigcn_b200.FusedTrainer(m0, lr=5e-3, weight_decay=1e-4, edge_weights=True)
    inline = bigcn_b200.FusedTrainer(m1, lr=5e-3, weight_decay=1e-4, edge_weights=True)
    small = [on_device(make_batch("twitter15", 2, seed=60 + i, train=True, in_feats=K, sizes=np.array([3, 4])), dev)
             for i in range(2)]
    big = []
    for i, which in enumerate(("both", "td", "bu")):
        b = edge_case_batch(70 + i, train=True)
        big.append(on_device(b, dev, torch.tensor(b.w[0], device=dev) if which != "bu" else None,
                             torch.tensor(b.w[1], device=dev) if which != "td" else None))
    order = small + big + [small[0], big[0], big[1], small[1], big[2], big[0]]
    first_buf = None
    for i, d in enumerate(order):
        nx = order[i + 1] if i + 1 < len(order) else None
        l0 = pipe.step(d, next_data=nx)
        l1 = inline.step(d)
        if i == 0:
            first_buf = pipe._prep_buf[0].numel()
        assert torch.equal(l0, l1), i
        assert torch.equal(pipe.last_logp, inline.last_logp), i
        assert_same_state(pipe, inline)
    assert pipe._prep_buf[0].numel() > first_buf        # grew for the weighted batches
    pipe.check_inputs()
    inline.check_inputs()


# ---------------------------------------------------------------------------------------------- graph replays
@gpu
def test_replays_read_current_weights(dev):
    """A captured step replays with the weights' current values (same storage, changed in place), and a new weight
    tensor builds a new plan instead of replaying the old graph; against a trainer that never captures."""
    import bigcn_b200
    torch.manual_seed(3)
    m0 = bigcn_b200.BiGCN(K, 64, 64, dev, gemm_mode="sparse").to(dev).train()
    m1 = copy.deepcopy(m0)
    rep = bigcn_b200.FusedTrainer(m0, lr=5e-3, weight_decay=1e-4, edge_weights=True, graphs=True)
    ref = bigcn_b200.FusedTrainer(m1, lr=5e-3, weight_decay=1e-4, edge_weights=True, graphs=False)
    b = edge_case_batch(21, train=True)
    d = on_device(b, dev, torch.tensor(b.w[0], device=dev), torch.tensor(b.w[1], device=dev))

    def both():
        assert torch.equal(rep.step(d), ref.step(d))
        assert_same_state(rep, ref)

    for _ in range(3):
        both()
    assert rep.graph_captures == 1 and rep.graph_replays == 2
    d.edge_weight.mul_(0.5)                  # in place: the captured graph reads the same storage
    d.BU_edge_weight[:5] = 3.0
    both()
    assert rep.graph_captures == 1 and rep.graph_replays == 3
    d.edge_weight = d.edge_weight * 2.0      # a new tensor: a new plan, captured again when seen twice
    for _ in range(3):
        both()
    assert rep.graph_captures == 2 and rep.graph_replays == 5
    rep.check_inputs()


# ---------------------------------------------------------------------------------------------- errors
@gpu
def test_weight_errors(dev):
    """A weight that requires grad, a bad shape, dtype or device raise BigcnError; a NaN weight in a batch prepared
    ahead is reported by check_inputs(); a default trainer still refuses weights."""
    import bigcn_b200
    b = edge_case_batch(3, train=False)
    m = bigcn_b200.BiGCN(K, 64, 64, dev, gemm_mode="sparse").to(dev).train()
    m.load_state_dict(oracle(K, 1).float().state_dict())
    tr = bigcn_b200.FusedTrainer(m, lr=5e-4, weight_decay=1e-4, edge_weights=True)
    e = b.edge_index.shape[1]
    with pytest.raises(bigcn_b200.BigcnError, match="gradient"):
        tr.step(on_device(b, dev, torch.ones(e, device=dev, requires_grad=True)), seed=1)
    for bad in (torch.ones(e + 1, device=dev), torch.ones(e, 1, device=dev), torch.ones(e, dtype=torch.int64, device=dev),
                torch.ones(e)):
        with pytest.raises(bigcn_b200.BigcnError):
            tr.step(on_device(b, dev, bad), seed=1)
        with pytest.raises(bigcn_b200.BigcnError):      # on BU, as the next batch: refused before anything is enqueued
            tr.step(on_device(b, dev), next_data=on_device(b, dev, None, bad), seed=1)
    tr.check_inputs()
    nan = torch.ones(e, device=dev)
    nan[3] = float("nan")
    good, bad = on_device(b, dev, torch.ones(e, device=dev)), on_device(b, dev, nan)
    tr.step(good, next_data=bad, seed=2)
    tr.step(bad, seed=3)                     # from the prepared buffer
    with pytest.raises(IndexError, match="edge weight"):
        tr.check_inputs()
    plain = bigcn_b200.FusedTrainer(m, lr=5e-4, weight_decay=1e-4)
    with pytest.raises(bigcn_b200.BigcnError, match="edge-weighted"):
        plain.step(good, seed=1)


# ---------------------------------------------------------------------------------------------- DeviceForest
def _forests(dev, shape, n_trees, dense, bu_own):
    """(dataset dict, unweighted forest, forest with weight = position + 1 (TD) and, with bu_own, -(position + 1) (BU))"""
    import bigcn_b200
    from bigcn_b200.data import synth_forest_device
    f = synth_forest_device(shape, n_trees, dev, seed=4, in_feats=64 if shape != "pheme" else 32)
    assert dense == ("x" in f)
    e_all = int(f["edge_ptr"][-1])
    assert e_all < (1 << 24)                  # position + 1 is exact in fp32
    td = torch.arange(1, e_all + 1, dtype=torch.float32, device=dev)
    bu = -td if bu_own else None
    plain = bigcn_b200.DeviceForest.from_device_arrays(f)
    g = dict(f)
    g["edge_weight"] = td
    wf = bigcn_b200.DeviceForest.from_device_arrays(g)
    if bu_own:
        wf = bigcn_b200.DeviceForest(f["node_ptr"], f["edge_ptr"], f["edge_src"].cpu().numpy(),
                                     f["edge_dst"].cpu().numpy(), None if dense else f["x_ptr"].cpu().numpy(),
                                     None if dense else f["x_col"].cpu().numpy(),
                                     None if dense else f["x_val"].cpu().numpy(), f["root_local"].cpu().numpy(),
                                     f["y"].cpu().numpy(), f["in_feats"], dev, x=f["x"] if dense else None,
                                     edge_weight=td, bu_edge_weight=bu)
    return f, plain, wf


@gpu
@pytest.mark.parametrize("bu_own", [False, True])
@pytest.mark.parametrize("rate", [0.0, 0.2])
@pytest.mark.parametrize("shape", ["twitter16", "weibo", "pheme"])
def test_forest_weights_follow_kept_edges(dev, shape, rate, bu_own):
    """Weight = the edge's position in the forest + 1, so a batch's weights name the edges kept.  Each direction's
    weights are exactly the kept edges' forest weights in kept order (BU: its own array, or the TD one); the edges are
    bit-identical to an unweighted forest's for the same ids and seed; an unweighted forest's batch has no weights.
    Weibo: a tree of more than 8192 edges (the single-thread selection sampling); PHEME: dense storage."""
    dense = shape == "pheme"
    n_trees = {"twitter16": 40, "weibo": 1000, "pheme": 60}[shape]
    f, plain, wf = _forests(dev, shape, n_trees, dense, bu_own)
    sizes = f["sizes"]
    if shape == "weibo":
        big = np.argsort(sizes)[-2:]
        assert sizes[big].max() - 1 > 8192
        ids = np.concatenate([big, [t for t in range(6) if t not in big][:5]])
    else:
        ids = np.random.default_rng(1).permutation(n_trees)[:16]
    for seed in (0, 9):
        a = plain.batch(ids, rate, rate, seed=seed)
        w = wf.batch(ids, rate, rate, seed=seed)
        assert not hasattr(a, "edge_weight") and not hasattr(a, "BU_edge_weight")
        assert torch.equal(a.edge_index, w.edge_index) and torch.equal(a.BU_edge_index, w.BU_edge_index)
        assert torch.equal(a.batch, w.batch) and torch.equal(a.rootindex, w.rootindex)
        if dense:
            assert torch.equal(a.x, w.x)
        else:
            assert torch.equal(a.x.ptr, w.x.ptr) and torch.equal(a.x.col, w.x.col) and torch.equal(a.x.val, w.x.val)
        src, dst = f["edge_src"].long().cpu(), f["edge_dst"].long().cpu()
        eptr = torch.from_numpy(f["edge_ptr"])
        node_off = torch.from_numpy(np.concatenate([[0], np.cumsum(sizes[ids])]))
        slot_of = {int(t): i for i, t in enumerate(ids)}
        for ei, wt, sign, flip in ((w.edge_index, w.edge_weight, 1, False),
                                   (w.BU_edge_index, w.BU_edge_weight, -1 if bu_own else 1, True)):
            assert wt.dtype == torch.float32 and wt.shape == (ei.shape[1],)
            pos = (wt.cpu() * sign).long() - 1                       # forest position of each kept edge
            tree = torch.searchsorted(eptr, pos, right=True) - 1     # its tree
            slot = torch.tensor([slot_of[int(t)] for t in tree], dtype=torch.int64)
            off = node_off[slot]
            want = torch.stack([src[pos] + off, dst[pos] + off])
            if flip:
                want = want.flip(0)
            assert torch.equal(ei.cpu(), want)
            # kept order: slots in batch order, positions ascending within a slot
            key = slot * (1 << 40) + pos
            assert bool((key[1:] > key[:-1]).all())
            kept = torch.bincount(slot, minlength=len(ids))
            e_t = torch.from_numpy(sizes[ids] - 1).clamp(min=0)
            want_k = e_t if rate <= 0 else torch.floor(e_t.double() * (1.0 - rate)).long()
            assert torch.equal(kept, want_k)


@gpu
def test_unweighted_forest_batches_unchanged(dev):
    """A forest without weights returns exactly the batch attributes it always did."""
    import bigcn_b200
    from bigcn_b200.data import synth_forest_device
    f = synth_forest_device("twitter16", 20, dev, seed=2, in_feats=64)
    fw = synth_forest_device("twitter16", 20, dev, seed=2, in_feats=64, edge_weights=True)
    for k in ("edge_src", "edge_dst", "root_local", "y", "x_ptr", "x_col", "x_val"):
        assert torch.equal(f[k], fw[k]), k
    w = fw["edge_weight"]
    assert w.dtype == torch.float32 and bool(((w > 0) & (w <= 1)).all())
    b = bigcn_b200.DeviceForest.from_device_arrays(f).batch(np.arange(8), 0.2, 0.2, seed=3)
    assert set(vars(b)) == {"x", "edge_index", "BU_edge_index", "batch", "rootindex", "y"}


# ---------------------------------------------------------------------------------------------- train_GCN
@gpu
def test_train_gcn_weighted_forest(tmp_path, monkeypatch, dev):
    """train_GCN on a weighted synthetic forest: finite losses, the checkpoint is written, and the first epoch's
    training loss equals a manual loop of FusedTrainer(edge_weights=True) over forest.batches with the same seeds."""
    import bigcn_b200
    from bigcn_b200.data import synth_forest_device
    from bigcn_b200.metrics import EvalCounts
    monkeypatch.chdir(tmp_path)
    f = synth_forest_device("twitter16", 48, dev, seed=5, in_feats=64, edge_weights=True)
    forest = bigcn_b200.DeviceForest.from_device_arrays(f)
    ids = np.arange(48)
    torch.manual_seed(0)
    model = bigcn_b200.BiGCN(64, 64, 64, dev, gemm_mode="sparse").to(dev)
    m2 = copy.deepcopy(model)
    out = bigcn_b200.train_GCN(model, forest, ids[:40], ids[40:], 0.2, 0.2, lr=5e-4, weight_decay=1e-4, patience=100,
                               n_epochs=3, batchsize=8, seed=7, log=lambda s: None, checkpoint_dir=str(tmp_path / "ck"))
    assert len(out[0]) == 3 and all(np.isfinite(v).all() for v in out[:4])
    assert bigcn_b200.train_GCN.last_final_checkpoint is not None
    assert torch.load(bigcn_b200.train_GCN.last_final_checkpoint, weights_only=False)
    # the first epoch by hand
    tr = bigcn_b200.FusedTrainer(m2, lr=5e-4, weight_decay=1e-4, edge_weights=True)
    ev = EvalCounts(4, dev)
    order = np.random.default_rng(7).permutation(ids[:40])
    lists = [order[lo:lo + 8] for lo in range(0, 40, 8)]
    seeds = [(7 << 20) + bi for bi in range(len(lists))]
    m2.train()
    for data, nxt in forest.batches(lists, 0.2, 0.2, seeds):
        assert data.edge_weight is not None and data.BU_edge_weight is not None
        tr.step(data, next_data=nxt)
        ev.update(tr.last_logp, data.y)
    assert ev.epoch_means()[0] == out[0][0]
