"""A dataset resident on the device and batch assembly there (SURVEY.md 8f, N2).

Stands in for ``BiGraphDataset`` (/root/reference/Process/dataset.py:45-99: one ``.npz`` per tree
loaded per epoch, DropEdge per direction) plus PyG's ``DataLoader`` collate
(/root/reference/model/Twitter/BiGCN_Twitter.py:162-169) when the whole dataset fits in HBM --
at ~14 non-zeros per node even the 1 M-tree synthetic scale-out config does.  Trees are packed
once, with the features in one of two forms: CSR (bag-of-words rows, never densified; ``data.x`` is a
SparseX for ``gemm_mode='sparse'``) or dense fp32 / bf16 rows (PHEME's sentence embeddings; ``data.x``
is a dense tensor for the tensor-core modes).  ``batch(ids)`` builds the batch on the device with one
call into libbigcn_b200.so.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib as L
from ._lib import check, lib
from .data import Batch
from .ops import SparseX, _p, _stream, check_bf16_width


def _dense_storage(x, n, k):
    """dense feature rows kept as they are: [n, k], fp32 or bf16, contiguous, on a CUDA device"""
    if not isinstance(x, torch.Tensor) or x.layout != torch.strided or x.dtype not in (torch.float32, torch.bfloat16):
        raise L.BigcnError(f"DeviceForest: dense features must be a torch.float32 or torch.bfloat16 tensor, got "
                           f"{getattr(x, 'dtype', type(x))}")
    if tuple(x.shape) != (n, k):
        raise L.BigcnError(f"DeviceForest: dense features must be [{n}, {k}] (all nodes x in_feats), got {tuple(x.shape)}")
    if x.dtype == torch.bfloat16:
        check_bf16_width(k)
    if not x.is_cuda:
        raise L.BigcnError("DeviceForest: dense features must be on the CUDA device")
    return x.contiguous()


def _weight_storage(w, e_all, name, dev):
    """per-tree-edge weights kept as they are: fp32 [e_all] on the device, or None"""
    if w is None:
        return None
    w = torch.as_tensor(w)
    if w.dtype != torch.float32 or tuple(w.shape) != (e_all,):
        raise L.BigcnError(f"DeviceForest: {name} must be torch.float32 [{e_all}] (one weight per tree edge), got "
                           f"{w.dtype} {tuple(w.shape)}")
    return w.to(dev).contiguous()


class DeviceForest:
    def __init__(self, node_ptr, edge_ptr, edge_src, edge_dst, x_ptr, x_col, x_val, root_local, y, in_feats, device,
                 x=None, edge_weight=None, bu_edge_weight=None):
        """Trees packed back to back: node_ptr / edge_ptr [T+1], the local edge lists edge_src / edge_dst
        ([parent; child]), root_local and y per tree, and the features of all nodes, either as CSR (x_ptr [N_all+1],
        x_col, x_val) or -- ``x`` given, the CSR arguments None -- as dense rows [N_all, in_feats] of torch.float32
        or torch.bfloat16 on the device, which ``batch()`` gathers into a dense ``data.x`` of the same dtype.
        ``edge_weight``: None, or one torch.float32 weight per tree edge [E_all], aligned with edge_src / edge_dst; a
        batch then carries ``edge_weight`` / ``BU_edge_weight`` for the edges each direction kept.  ``bu_edge_weight``:
        the BU list's own weights for the same tree edges (default: ``edge_weight``, one weight seen from either end)."""
        # host copies of the (small) size arrays: batch offsets are computed without touching the device
        self.h_node_ptr = np.asarray(node_ptr, np.int64)
        self.h_edge_ptr = np.asarray(edge_ptr, np.int64)
        self.in_feats = int(in_feats)
        self.device = torch.device(device)
        dev = self.device
        t = lambda a, dt: torch.as_tensor(np.ascontiguousarray(a), dtype=dt).to(dev)  # noqa: E731
        self.node_ptr, self.edge_ptr = t(node_ptr, torch.int64), t(edge_ptr, torch.int64)
        self.edge_src, self.edge_dst = t(edge_src, torch.int32), t(edge_dst, torch.int32)
        if x is None:
            self.h_x_ptr_at_tree = np.asarray(x_ptr, np.int64)[self.h_node_ptr]   # nnz offset of each tree's first node
            self.x_ptr, self.x_col, self.x_val = t(x_ptr, torch.int64), t(x_col, torch.int32), t(x_val, torch.float32)
            self.x = None
        else:
            self.x_ptr = self.x_col = self.x_val = None
            self.x = _dense_storage(x, int(self.h_node_ptr[-1]), self.in_feats)
        self.root_local, self.y = t(root_local, torch.int32), t(y, torch.int64)
        self.num_trees = len(self.h_node_ptr) - 1
        self._set_weights(edge_weight, bu_edge_weight)
        self._stage, self._turn = None, 0
        self._cache_ptrs()

    def _set_weights(self, edge_weight, bu_edge_weight):
        e_all = int(self.h_edge_ptr[-1])
        self.edge_weight = _weight_storage(edge_weight, e_all, "edge_weight", self.device)
        self.bu_edge_weight = _weight_storage(bu_edge_weight, e_all, "bu_edge_weight", self.device)
        if self.edge_weight is None and self.bu_edge_weight is not None:
            raise L.BigcnError("DeviceForest: bu_edge_weight needs edge_weight (the TD weights of the same edges)")

    def _cache_ptrs(self):
        # the dataset arrays never move: their addresses are looked up once, not on every batch
        for k in ("node_ptr", "edge_ptr", "edge_src", "edge_dst", "x_ptr", "x_col", "x_val", "x", "root_local", "y",
                  "edge_weight", "bu_edge_weight"):
            setattr(self, "_p_" + k, _p(getattr(self, k)))

    @staticmethod
    def from_device_arrays(f):
        """From ``data.synth_forest_device``: everything already sits on the device; only the size arrays live on the
        host.  Features stay in the form ``f`` holds them: dense rows when it has ``"x"`` (PHEME; fp32, or bf16 after
        ``f["x"] = f["x"].to(torch.bfloat16)``), CSR otherwise.  ``f["edge_weight"]`` (optional): the per-tree-edge
        weights (``synth_forest_device(..., edge_weights=True)``)."""
        self = DeviceForest.__new__(DeviceForest)
        dev = f["edge_src"].device
        self.h_node_ptr = np.asarray(f["node_ptr"], np.int64)
        self.h_edge_ptr = np.asarray(f["edge_ptr"], np.int64)
        self.node_ptr = torch.from_numpy(self.h_node_ptr).to(dev)
        self.edge_ptr = torch.from_numpy(self.h_edge_ptr).to(dev)
        self.in_feats, self.device = int(f["in_feats"]), dev
        self.edge_src, self.edge_dst = f["edge_src"], f["edge_dst"]
        if "x" in f:
            self.x_ptr = self.x_col = self.x_val = None
            self.x = _dense_storage(f["x"], int(self.h_node_ptr[-1]), self.in_feats)
        else:
            self.h_x_ptr_at_tree = f["x_ptr"][self.node_ptr].cpu().numpy()
            self.x_ptr, self.x_col, self.x_val = f["x_ptr"], f["x_col"], f["x_val"]
            self.x = None
        self.root_local, self.y = f["root_local"], f["y"].to(torch.int64)
        self.num_trees = len(self.h_node_ptr) - 1
        self._set_weights(f.get("edge_weight"), None)
        self._stage, self._turn = None, 0
        self._cache_ptrs()
        return self

    @staticmethod
    def from_data_list(trees, device, features="csr", dtype=torch.float32):
        """Pack ``Data`` objects with the attribute layout of dataset.py:91-98 (x dense or SparseX,
        edge_index [2,e] = [parent; child] WITHOUT DropEdge, rootindex, y).  ``features``: 'csr' keeps the non-zeros
        of every row (bag-of-words features; ``data.x`` of a batch is a SparseX); 'dense' keeps the rows as they are,
        in ``dtype`` (torch.float32 or torch.bfloat16; a SparseX tree is densified here, once), and a batch's
        ``data.x`` is a dense tensor of that dtype.  ``d.edge_weight`` (one weight per column of ``d.edge_index``), on
        every tree or on none, is kept as the forest's ``edge_weight``."""
        if features not in ("csr", "dense"):
            raise L.BigcnError(f"DeviceForest: features must be 'csr' or 'dense', got {features!r}")
        dense = features == "dense"
        if dense and dtype not in (torch.float32, torch.bfloat16):
            raise L.BigcnError(f"DeviceForest: dense features are stored as torch.float32 or torch.bfloat16, got {dtype}")
        node_ptr, edge_ptr, x_ptr = [0], [0], [0]
        es, ed, xc, xv, xd, roots, ys = [], [], [], [], [], [], []
        trees = list(trees)
        ws = [getattr(d, "edge_weight", None) for d in trees]
        weighted = any(w is not None for w in ws)
        if weighted and any(w is None for w in ws):
            raise L.BigcnError("DeviceForest: edge_weight must be given on every tree or on none")
        for i, (d, w) in enumerate(zip(trees, ws)):
            if weighted and tuple(torch.as_tensor(w).shape) != (int(d.edge_index.shape[1]),):
                raise L.BigcnError(f"DeviceForest: tree {i}: edge_weight must be [{int(d.edge_index.shape[1])}] (one weight "
                                   f"per edge), got {tuple(torch.as_tensor(w).shape)}")
        ew = torch.cat([torch.as_tensor(w).detach().cpu().to(torch.float32).reshape(-1) for w in ws]) \
            if weighted and trees else (torch.zeros(0, dtype=torch.float32) if weighted else None)
        k = None
        for d in trees:
            x = d.x
            if dense:
                xn = (x.to_dense() if isinstance(x, SparseX) else x).to(dtype)
                n, k = xn.shape
                if dtype == torch.bfloat16:
                    check_bf16_width(k)      # before anything is copied to the device
                xd.append(xn)
            elif isinstance(x, SparseX):
                ptr, col, val, n = x.ptr.numpy().astype(np.int64), x.col.numpy(), x.val.numpy(), x.shape[0]
                k = x.shape[1]
            else:
                xn = x.numpy()
                n, k = xn.shape
                r, c = np.nonzero(xn)
                col, val = c.astype(np.int32), xn[r, c]
                ptr = np.concatenate([[0], np.cumsum(np.bincount(r, minlength=n))]).astype(np.int64)
            ei = d.edge_index.numpy()
            es.append(ei[0].astype(np.int32)); ed.append(ei[1].astype(np.int32))
            if not dense:
                xc.append(col); xv.append(val)
                x_ptr.extend((x_ptr[-1] + ptr[1:]).tolist())
            node_ptr.append(node_ptr[-1] + n)
            edge_ptr.append(edge_ptr[-1] + ei.shape[1])
            roots.append(int(d.rootindex)); ys.append(int(d.y))
        cat = lambda xs, dt: np.concatenate(xs).astype(dt) if xs else np.zeros(0, dt)  # noqa: E731
        if dense:
            return DeviceForest(node_ptr, edge_ptr, cat(es, np.int32), cat(ed, np.int32), None, None, None, roots, ys, k,
                                device, x=torch.cat(xd).to(device), edge_weight=ew)
        return DeviceForest(node_ptr, edge_ptr, cat(es, np.int32), cat(ed, np.int32), x_ptr, cat(xc, np.int32),
                            cat(xv, np.float32), roots, ys, k, device, edge_weight=ew)

    @staticmethod
    def from_npz_dir(fold_x, data_path, device, treeDic=None, lower=2, upper=100000, features="csr",
                     dtype=torch.float32):
        """Pack the reference's preprocessed dataset: one ``<id>.npz`` per tree under ``data_path`` with ``x`` [n, K],
        ``edgeindex`` [2, e] = [parent; child], ``rootindex`` and ``y`` (written by Process/getTwittergraph.py:67-72,
        read per item and per epoch by ``BiGraphDataset.__getitem__``, Process/dataset.py:64-99 -- here once).  The id
        filter is ``BiGraphDataset.__init__``'s (dataset.py:48-59): PHEME paths take ``fold_x`` as is, the others keep
        the ids found in ``treeDic`` whose tree has ``lower .. upper`` nodes.  ``self.ids`` holds the kept ids in
        order: tree t of the forest is ``ids[t]``.  ``features`` / ``dtype``: as in ``from_data_list``."""
        import os
        from .data import Data
        if str(data_path).find("PHEME") == -1 and treeDic is not None:
            fold_x = [i for i in fold_x if i in treeDic and lower <= len(treeDic[i]) <= upper]
        trees = []
        for i in fold_x:
            z = np.load(os.path.join(data_path, str(i) + ".npz"), allow_pickle=True)
            ei = np.asarray(z["edgeindex"], np.int64).reshape(2, -1)
            trees.append(Data(x=torch.tensor(np.asarray(z["x"]), dtype=torch.float32), edge_index=torch.from_numpy(ei),
                              rootindex=torch.tensor([int(z["rootindex"])]), y=torch.tensor([int(z["y"])])))
        forest = DeviceForest.from_data_list(trees, device, features, dtype)
        forest.ids = list(fold_x)
        return forest

    def batches(self, id_lists, td_droprate=0.0, bu_droprate=0.0, seeds=None):
        """The loader loop (the reference's ``DataLoader`` over ``BiGraphDataset``, BiGCN_Twitter.py:168): yields
        ``(batch_i, batch_i+1)`` -- the second one already assembled (None after the last) so that
        ``FusedTrainer.step(batch_i, next_data=batch_i+1)`` can run batch i+1's weight-independent half (graph prep,
        root columns, CSR of x) underneath step i.  ``seeds[i]``: DropEdge seed of batch i (default i)."""
        id_lists = list(id_lists)
        seeds = list(range(len(id_lists))) if seeds is None else list(seeds)
        nxt = self.batch(id_lists[0], td_droprate, bu_droprate, seed=seeds[0]) if id_lists else None
        for i in range(len(id_lists)):
            cur = nxt
            nxt = self.batch(id_lists[i + 1], td_droprate, bu_droprate, seed=seeds[i + 1]) if i + 1 < len(id_lists) else None
            yield cur, nxt

    def batch(self, tree_ids, td_droprate=0.0, bu_droprate=0.0, seed=0) -> Batch:
        """The collated batch of ``tree_ids`` (host sequence, in batch order) with DropEdge at the
        given rates, on the device; ``data.x`` is a SparseX for CSR storage, a fresh contiguous [n, in_feats] tensor
        of the storage dtype for dense storage.  DropEdge draws depend only on the seed, the tree id, the direction and
        the edge position: both storage forms give the same edges for the same ids and seed, and so does a weighted
        forest, whose batches also carry ``edge_weight`` / ``BU_edge_weight`` (fp32, the kept edges' weights in order)."""
        L.require_device()
        ids = np.asarray(tree_ids, np.int64)
        b = len(ids)
        dev = self.device
        dense = self.x is not None
        # The per-tree offsets live in a ring of pinned staging buffers which the assembly kernels read IN PLACE
        # (pinned memory is device-addressable: 5 (b + 1) int64 cross PCIe inside the kernels, no copy, no device
        # buffer).  A slot is rewritten only after the kernels that last read it have completed: the epoch loop never
        # synchronises the host, so the device may lag many batches.
        need = 5 * (b + 1)
        if self._stage is None or self._stage[0][0].numel() < need:
            if self._stage is not None:
                for _, ev, _ in self._stage:
                    if ev is not None:
                        ev.synchronize()
            self._stage = []
            for _ in range(4):
                t = torch.empty(max(need, 4096), dtype=torch.int64).pin_memory()
                self._stage.append([t, None, t.numpy()])
        self._turn = (self._turn + 1) % len(self._stage)
        slot = self._stage[self._turn]
        if slot[1] is not None:
            slot[1].synchronize()
        offs = slot[2][:need].reshape(5, b + 1)
        ids1 = ids + 1
        e_t = self.h_edge_ptr[ids1] - self.h_edge_ptr[ids]
        offs[0, :b] = ids
        offs[1:, 0] = 0
        np.cumsum(self.h_node_ptr[ids1] - self.h_node_ptr[ids], out=offs[1, 1:])
        # int(length * (1 - droprate)), dataset.py:72,84 (Python float arithmetic = IEEE double)
        for row, rate in ((2, td_droprate), (3, bu_droprate)):
            np.cumsum(e_t if rate <= 0 else np.floor(e_t.astype(np.float64) * (1.0 - rate)).astype(np.int64), out=offs[row, 1:])
        if dense:
            offs[4, 1:] = 0
        else:
            np.cumsum(self.h_x_ptr_at_tree[ids1] - self.h_x_ptr_at_tree[ids], out=offs[4, 1:])
        n, e_td, e_bu, nnz = (int(v) for v in offs[1:, b])
        # one int64 block [edge_index | BU_edge_index | batch | rootindex | y], one 32-bit block [x ptr | x col | x val]
        # (CSR) or a dense x of its own
        blk = torch.empty(2 * e_td + 2 * e_bu + n + 2 * b, dtype=torch.int64, device=dev)
        o = 0
        ei = blk[o:o + 2 * e_td].view(2, e_td); o += 2 * e_td
        bu = blk[o:o + 2 * e_bu].view(2, e_bu); o += 2 * e_bu
        batch = blk[o:o + n]; o += n
        root = blk[o:o + b]; o += b
        y = blk[o:o + b]
        cur = torch.cuda.current_stream(dev)
        base, pitch = slot[0].data_ptr(), 8 * (b + 1)
        seed = int(seed) & ((1 << 64) - 1)
        extra = {}
        aw = None
        if self.edge_weight is not None:      # the kept edges' weights: one fp32 block [TD | BU]
            wblk = torch.empty(e_td + e_bu, dtype=torch.float32, device=dev)
            extra = {"edge_weight": wblk[:e_td], "BU_edge_weight": wblk[e_td:]}
            aw = L.AsmWeights(td_weight=self._p_edge_weight, bu_weight=self._p_bu_edge_weight,
                              edge_weight=_p(extra["edge_weight"]), bu_edge_weight=_p(extra["BU_edge_weight"]))
        if dense:
            x = torch.empty(n, self.in_feats, dtype=self.x.dtype, device=dev)
            args = (self._p_node_ptr, self._p_edge_ptr, self._p_edge_src, self._p_edge_dst, self._p_root_local, self._p_y,
                    base, base + pitch, base + 2 * pitch, base + 3 * pitch, b, e_td, e_bu, seed, _p(ei), _p(bu), _p(batch),
                    _p(root), _p(y), self._p_x, self.in_feats, self.x.element_size(), _p(x))
            if aw is None:
                check(lib().bigcn_assemble_batch_dense(*args, cur.cuda_stream), "assemble_batch_dense")
            else:
                check(lib().bigcn_assemble_batch_dense_weighted(*args, C.byref(aw), cur.cuda_stream),
                      "assemble_batch_dense_weighted")
        else:
            iblk = torch.empty(n + 1 + 2 * nnz, dtype=torch.int32, device=dev)
            if b == 0:
                iblk.zero_()
            ox_ptr, ox_col = iblk[:n + 1], iblk[n + 1:n + 1 + nnz]
            ox_val = iblk[n + 1 + nnz:].view(torch.float32)
            args = (self._p_node_ptr, self._p_edge_ptr, self._p_edge_src, self._p_edge_dst, self._p_x_ptr, self._p_x_col,
                    self._p_x_val, self._p_root_local, self._p_y, base, base + pitch, base + 2 * pitch, base + 3 * pitch,
                    base + 4 * pitch, b, e_td, e_bu, seed, _p(ei), _p(bu), _p(batch), _p(root), _p(y), _p(ox_ptr),
                    _p(ox_col), _p(ox_val))
            if aw is None:
                check(lib().bigcn_assemble_batch(*args, cur.cuda_stream), "assemble_batch")
            else:
                check(lib().bigcn_assemble_batch_weighted(*args, C.byref(aw), cur.cuda_stream), "assemble_batch_weighted")
            x = SparseX(ox_ptr, ox_col, ox_val, (n, self.in_feats))
        if slot[1] is None:
            slot[1] = torch.cuda.Event()
        slot[1].record(cur)
        return Batch(x=x, edge_index=ei, BU_edge_index=bu, batch=batch, rootindex=root, y=y, **extra)
