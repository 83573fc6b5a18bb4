"""Input contract of the hot path and deterministic synthetic reply trees.

The reference feeds ``model(Batch_data)`` with a torch_geometric ``Batch`` built
by ``BiGraphDataset.__getitem__`` (/root/reference/Process/dataset.py:64-99) and
PyG's DataLoader collate (/root/reference/model/Twitter/BiGCN_Twitter.py:168).
PyG is not on this path here: ``Data`` / ``Batch`` below are minimal duck-typed
containers with the same attribute names and the same collate offset rules
(keys containing "index" are offset by the cumulative node count and
concatenated on the last dim; ``batch`` is the sorted tree id per node).

Real ``.npz`` trees are missing from the reference checkout, so shapes follow
SURVEY.md section 8(d): log-normal tree sizes per dataset, preferential-attachment
topology, permuted local node ids, BoW features with small integer counts.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np
import torch

# name -> (in_feats, num_classes, reference batch size, DropEdge rate)
SHAPES = {
    "twitter15": dict(in_feats=5000, num_classes=4, batch=128, droprate=0.2),
    "twitter16": dict(in_feats=5000, num_classes=4, batch=128, droprate=0.2),
    "weibo": dict(in_feats=5000, num_classes=2, batch=16, droprate=0.0),
    "pheme": dict(in_feats=768, num_classes=4, batch=24, droprate=0.2),
    "powerlaw": dict(in_feats=5000, num_classes=4, batch=128, droprate=0.2),
}


class Data:
    """One reply tree (attribute names of dataset.py:91-98)."""

    def __init__(self, **kw):
        for k, v in kw.items():
            setattr(self, k, v)

    @property
    def num_nodes(self):
        return int(self.x.shape[0])


class Batch(Data):
    """Concatenated trees; ``forward(data)`` reads x, edge_index, BU_edge_index,
    batch, rootindex (BiGCN_Twitter.py:27,45-47,78)."""

    _tensor_keys = ("x", "edge_index", "BU_edge_index", "batch", "rootindex", "y")

    def to(self, device, non_blocking=False):
        for k in self._tensor_keys:
            v = getattr(self, k, None)
            if isinstance(v, torch.Tensor) or hasattr(v, "ptr"):      # tensors and ops.SparseX
                setattr(self, k, v.to(device, non_blocking=non_blocking))
        return self

    def pin_memory(self):
        for k in self._tensor_keys:
            v = getattr(self, k, None)
            if isinstance(v, torch.Tensor) or hasattr(v, "ptr"):
                setattr(self, k, v.pin_memory())
        return self

    @property
    def num_graphs(self):
        return int(self.rootindex.numel())


def collate(trees) -> Batch:
    """PyG ``Batch.from_data_list`` offset rules for the five attributes used."""
    xs, eis, bus, roots, ys, bs = [], [], [], [], [], []
    off = 0
    for t, d in enumerate(trees):
        n = d.num_nodes
        xs.append(d.x)
        eis.append(d.edge_index + off)
        bus.append(d.BU_edge_index + off)
        roots.append(d.rootindex + off)
        ys.append(d.y)
        bs.append(torch.full((n,), t, dtype=torch.int64))
        off += n
    return Batch(x=torch.cat(xs, 0), edge_index=torch.cat(eis, 1), BU_edge_index=torch.cat(bus, 1),
                 rootindex=torch.cat(roots, 0), y=torch.cat(ys, 0), batch=torch.cat(bs, 0))


# --------------------------------------------------------------------------
# synthetic generators
# --------------------------------------------------------------------------
def tree_sizes(shape: str, n_trees: int, rng: np.random.Generator) -> np.ndarray:
    if shape == "twitter15":
        n = np.clip(np.rint(np.exp(rng.normal(5.2, 0.6, n_trees))), 55, 1768)
    elif shape == "twitter16":
        n = np.clip(np.rint(np.exp(rng.normal(5.3, 0.65, n_trees))), 81, 2765)
    elif shape == "weibo":
        n = np.clip(np.rint(np.exp(rng.normal(5.9, 1.25, n_trees))), 10, 59318)
    elif shape == "pheme":
        single = rng.random(n_trees) < 0.21
        n = np.where(single, 1, np.minimum(1 + np.ceil(rng.exponential(11.0, n_trees)), 108))
    elif shape == "powerlaw":
        n = np.clip(np.floor(2.0 * (1.0 + rng.pareto(2.0, n_trees))), 2, 10000)
    else:
        raise ValueError(f"unknown shape {shape!r}")
    return n.astype(np.int64)


def _parents_pref_attach(n: int, rng: np.random.Generator, max_depth: int = 50) -> np.ndarray:
    """parent[c] for c=1..n-1 chosen with probability ~ 1 + #children among earlier
    nodes (urn trick, O(n)); node 0 is the root."""
    parent = np.full(n, -1, np.int64)
    if n == 1:
        return parent
    depth = np.zeros(n, np.int64)
    urn = np.empty(2 * n, np.int64)
    urn[0] = 0
    m = 1
    draws = rng.random(n)
    for c in range(1, n):
        p = int(urn[int(draws[c] * m)])
        while depth[p] >= max_depth:
            p = int(parent[p])
        parent[c] = p
        depth[c] = depth[p] + 1
        urn[m] = p
        urn[m + 1] = c
        m += 2
    return parent


def _bow_features(n: int, k: int, rng: np.random.Generator) -> np.ndarray:
    """1+Poisson(12) distinct Zipf-distributed columns per node, counts in 1..3."""
    x = np.zeros((n, k), np.float32)
    nnz = 1 + rng.poisson(12.0, n)
    tot = int(nnz.sum())
    cols = np.minimum(rng.zipf(1.3, tot) - 1, k - 1) if k > 1 else np.zeros(tot, np.int64)
    # spread the Zipf head over the vocabulary so the hot columns are not all < 10
    cols = (cols * 2654435761 % k).astype(np.int64)
    vals = rng.integers(1, 4, tot).astype(np.float32)
    rows = np.repeat(np.arange(n), nnz)
    x[rows, cols] = vals
    return x


def make_tree(shape: str, n: int, rng: np.random.Generator, in_feats: int | None = None,
              num_classes: int | None = None) -> Data:
    """One synthetic tree with the attribute layout of dataset.py:91-98 (no DropEdge)."""
    spec = SHAPES[shape]
    k = spec["in_feats"] if in_feats is None else in_feats
    c = spec["num_classes"] if num_classes is None else num_classes
    parent = _parents_pref_attach(n, rng)
    if shape == "pheme":          # getPHEMEgraph.py:29 keeps the root at local index 0
        perm = np.arange(n)
    else:                         # getTwittergraph.py:45: root sits at an arbitrary local index
        perm = rng.permutation(n)
    child = np.arange(1, n)
    row = perm[parent[1:]]
    col = perm[child]
    order = np.lexsort((col, row))  # sorted by (parent, child), getTwittergraph.py:56-63
    ei = np.stack([row[order], col[order]]).astype(np.int64).reshape(2, -1)
    if shape == "pheme":
        x = np.tanh(rng.normal(0.0, 1.0, (n, k))).astype(np.float32)
    else:
        x = _bow_features(n, k, rng)
    return Data(x=torch.from_numpy(x), edge_index=torch.from_numpy(ei),
                BU_edge_index=torch.from_numpy(ei[::-1].copy()),
                rootindex=torch.tensor([int(perm[0])], dtype=torch.int64),
                y=torch.tensor([int(rng.integers(0, c))], dtype=torch.int64))


def drop_edge(d: Data, td_rate: float, bu_rate: float, rng: np.random.Generator) -> Data:
    """dataset.py:68-90: keep int(e*(1-rate)) positions, order preserved,
    sampled independently for the TD and the BU list."""
    ei = d.edge_index.numpy()
    e = ei.shape[1]

    def keep(rate):
        if rate <= 0 or e == 0:
            return np.arange(e)
        return np.sort(rng.choice(e, int(e * (1 - rate)), replace=False))
    ktd, kbu = keep(td_rate), keep(bu_rate)
    td = ei[:, ktd]
    bu = ei[::-1][:, kbu]
    return Data(x=d.x, edge_index=torch.from_numpy(np.ascontiguousarray(td)),
                BU_edge_index=torch.from_numpy(np.ascontiguousarray(bu)),
                rootindex=d.rootindex, y=d.y)


def make_batch(shape: str, n_trees: int, seed: int = 0, train: bool = True,
               in_feats: int | None = None, num_classes: int | None = None,
               sizes: np.ndarray | None = None) -> Batch:
    """A collated synthetic batch.  ``train=True`` applies the dataset's DropEdge
    rates independently per direction (BiGCN_Twitter.py:358-359); eval batches
    keep BU_edge_index == flip(edge_index) (Process/process.py:63)."""
    rng = np.random.default_rng(seed)
    if sizes is None:
        sizes = tree_sizes(shape, n_trees, rng)
    rate = SHAPES[shape]["droprate"] if train else 0.0
    trees = []
    for n in sizes:
        t = make_tree(shape, int(n), rng, in_feats, num_classes)
        if rate > 0:
            t = drop_edge(t, rate, rate, rng)
        trees.append(t)
    return collate(trees)


def make_batch_shard(shape: str, n_trees_global: int, seed: int, rank: int = 0, world: int = 1,
                     train: bool = True, in_feats: int | None = None, num_classes: int | None = None):
    """Rank `rank`'s share of a GLOBAL batch of n_trees_global trees (SURVEY.md 8e): tree sizes
    come from one generator every rank replays, trees are assigned as contiguous ranges balanced
    by NODE count (dist.shard_trees) and each tree is generated from its own (seed, tree index)
    stream, so any rank can build any tree and the global batch does not depend on the world
    size.  Returns (Batch, node_id_base, (lo, hi))."""
    trees, base, rng_of, (lo, hi) = make_trees_shard(shape, n_trees_global, seed, rank, world, in_feats, num_classes)
    rate = SHAPES[shape]["droprate"] if train else 0.0
    if rate > 0:
        trees = [drop_edge(t, rate, rate, rng_of(lo + j)) for j, t in enumerate(trees)]
    return collate(trees), base, (lo, hi)


def make_trees_shard(shape: str, n_trees_global: int, seed: int, rank: int = 0, world: int = 1,
                     in_feats: int | None = None, num_classes: int | None = None):
    """The trees (no DropEdge) of rank `rank`'s node-balanced range of a global batch; returns
    (trees, node_id_base, rng_of(tree index) -> the tree's generator after make_tree, (lo, hi))."""
    from .dist import shard_trees, node_id_base
    sizes = tree_sizes(shape, n_trees_global, np.random.default_rng(seed))
    lo, hi = shard_trees(sizes, world)[rank]
    rngs = {}
    trees = []
    for t in range(lo, hi):
        rng = np.random.default_rng([seed, t])
        trees.append(make_tree(shape, int(sizes[t]), rng, in_feats, num_classes))
        rngs[t] = rng
    return trees, node_id_base(sizes, lo), (lambda t: rngs[t]), (lo, hi)


@dataclass
class DeviceTrees:
    """Large synthetic forest built directly on the device (kernel micro-benchmarks
    and the power-law scale-out config): uniform random recursive trees."""
    edge_index: torch.Tensor
    BU_edge_index: torch.Tensor
    batch: torch.Tensor
    rootindex: torch.Tensor


def make_device_forest(n_trees: int, nodes_per_tree: int, device, seed: int = 0, skew: float = 1.0) -> DeviceTrees:
    """``skew`` = 1: uniform random recursive trees (parent of node i uniform in [0, i));
    > 1 biases parents towards the early nodes (u**skew), i.e. hub-heavy reply trees whose root
    collects O(n**(1-1/skew)) children."""
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    n = n_trees * nodes_per_tree
    local = torch.arange(n, device=device, dtype=torch.int64) % nodes_per_tree
    base = torch.arange(n, device=device, dtype=torch.int64) - local
    u = torch.rand(n, device=device, generator=g, dtype=torch.float64)
    if skew != 1.0:
        u = u ** skew
    par_local = (u * local.to(torch.float64)).to(torch.int64).clamp_(min=0)
    is_child = local > 0
    child = torch.arange(n, device=device, dtype=torch.int64)[is_child]
    par = (base + par_local)[is_child]
    order = torch.argsort(par * n + child)
    ei = torch.stack([par[order], child[order]])
    batch = torch.arange(n, device=device, dtype=torch.int64) // nodes_per_tree
    root = torch.arange(n_trees, device=device, dtype=torch.int64) * nodes_per_tree
    return DeviceTrees(ei, ei.flip(0).contiguous(), batch, root)


def synth_forest_device(shape: str, n_trees: int, device, seed: int = 0, in_feats: int | None = None,
                        num_classes: int | None = None, edge_weights: bool = False):
    """A whole synthetic DATASET generated on the device in a few vectorised passes (the per-tree Python
    generators above take minutes for Weibo's 3.7 M nodes or the 1 M-tree scale-out config): tree sizes of
    SURVEY.md 8(d), hub-heavy random recursive topology (parent of local node i = floor(u^2 * i)), the root at a
    random local index (a per-tree rotation of the local ids; PHEME keeps it at 0), TD edges sorted by
    (parent, child), BoW rows of 1+Poisson(12) distinct Zipf-ish columns with counts 1..3 (kept as CSR) or,
    for PHEME, dense tanh(N(0,1)) rows.  Returns a dict of device tensors + host size arrays:
    node_ptr / edge_ptr (host int64 [T+1]), edge_src / edge_dst (int32, local ids), root_local, y, and either
    x_ptr / x_col / x_val (CSR over all nodes) or x (dense [N, K]).  ``edge_weights``: also ``edge_weight``, one fp32
    weight in (0, 1] per tree edge (drawn after everything else: the other arrays are those of the unweighted call)."""
    spec = SHAPES[shape]
    k = spec["in_feats"] if in_feats is None else in_feats
    c = spec["num_classes"] if num_classes is None else num_classes
    sizes = tree_sizes(shape, n_trees, np.random.default_rng(seed))
    node_ptr = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    edge_ptr = node_ptr - np.arange(n_trees + 1, dtype=np.int64)
    n = int(node_ptr[-1])
    g = torch.Generator(device=device)
    g.manual_seed(int(seed) * 7919 + 17)
    d_sizes = torch.from_numpy(sizes).to(device)
    d_ptr = torch.from_numpy(node_ptr).to(device)
    tree = torch.repeat_interleave(torch.arange(n_trees, device=device), d_sizes)
    local = torch.arange(n, device=device) - d_ptr[tree]
    nt = d_sizes[tree]
    u = torch.rand(n, device=device, generator=g, dtype=torch.float64)
    par = (u * u * local.to(torch.float64)).to(torch.int64)
    if shape == "pheme":
        shift = torch.zeros(n_trees, dtype=torch.int64, device=device)
    else:
        shift = (torch.rand(n_trees, device=device, generator=g, dtype=torch.float64) * d_sizes.to(torch.float64)).to(torch.int64)
        shift = torch.minimum(shift, d_sizes - 1)
    sh = shift[tree]
    is_child = local > 0
    ch = ((local + sh) % nt)[is_child]
    pa = ((par + sh) % nt)[is_child]
    tr = tree[is_child]
    order = torch.argsort((tr << 40) | (pa << 20) | ch)       # (tree, parent, child); local ids < 2^20
    out = dict(node_ptr=node_ptr, edge_ptr=edge_ptr, edge_src=pa[order].to(torch.int32), edge_dst=ch[order].to(torch.int32),
               root_local=shift.to(torch.int32), y=torch.randint(0, c, (n_trees,), device=device, generator=g),
               in_feats=k, num_classes=c, sizes=sizes)
    if shape == "pheme":
        out["x"] = torch.tanh(torch.randn(n, k, device=device, generator=g))
        return _synth_edge_weights(out, g, device) if edge_weights else out
    nnz = 1 + torch.poisson(torch.full((n,), 12.0, device=device), generator=g).to(torch.int64)
    rows = torch.repeat_interleave(torch.arange(n, device=device), nnz)
    uz = torch.rand(rows.numel(), device=device, generator=g, dtype=torch.float64).clamp_(min=1e-12)
    z = torch.clamp(torch.floor(uz ** (-1.0 / 0.3)), max=float(1 << 40)).to(torch.int64)     # Zipf(1.3)-like head
    cols = ((z - 1).clamp_(max=k - 1) * 2654435761) % k
    key = torch.unique(rows * k + cols)                        # distinct columns per row, ascending
    rows, cols = key // k, key % k
    x_ptr = torch.zeros(n + 1, dtype=torch.int64, device=device)
    x_ptr[1:] = torch.cumsum(torch.bincount(rows, minlength=n), 0)
    out.update(x_ptr=x_ptr, x_col=cols.to(torch.int32),
               x_val=torch.randint(1, 4, (cols.numel(),), device=device, generator=g).to(torch.float32))
    return _synth_edge_weights(out, g, device) if edge_weights else out


def _synth_edge_weights(out, g, device):
    e_all = int(out["edge_ptr"][-1])
    out["edge_weight"] = 1.0 - torch.rand(e_all, device=device, generator=g)     # (0, 1]
    return out


def forest_slice_batch(f: dict, t0: int, t1: int) -> Batch:
    """Trees [t0, t1) of a ``synth_forest_device`` dataset with DENSE features as one collated batch on the device
    (no DropEdge: the test split of Process/process.py:63); x is a view of the dataset's rows.  A weighted dataset's
    batch carries the trees' ``edge_weight`` (a view) on both directions."""
    node_ptr, edge_ptr = f["node_ptr"], f["edge_ptr"]
    n0, n1, e0, e1 = int(node_ptr[t0]), int(node_ptr[t1]), int(edge_ptr[t0]), int(edge_ptr[t1])
    dev = f["edge_src"].device
    sizes = torch.from_numpy(f["sizes"][t0:t1]).to(dev)
    starts = torch.from_numpy(node_ptr[t0:t1] - n0).to(dev)
    etree = torch.repeat_interleave(torch.arange(t1 - t0, device=dev), torch.clamp(sizes - 1, min=0))
    off = starts[etree]
    ei = torch.stack([f["edge_src"][e0:e1].to(torch.int64) + off, f["edge_dst"][e0:e1].to(torch.int64) + off])
    extra = {}
    if "edge_weight" in f:
        extra = {"edge_weight": f["edge_weight"][e0:e1], "BU_edge_weight": f["edge_weight"][e0:e1]}
    return Batch(x=f["x"][n0:n1], edge_index=ei, BU_edge_index=ei.flip(0).contiguous(),
                 batch=torch.repeat_interleave(torch.arange(t1 - t0, device=dev), sizes),
                 rootindex=starts + f["root_local"][t0:t1].to(torch.int64), y=f["y"][t0:t1], **extra)
