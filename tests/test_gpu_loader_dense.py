"""DeviceForest with dense feature rows (fp32 or bf16 in HBM): the batch's x is gathered on the device
(k_asm_dense_rows, bigcn_assemble_batch_dense) in the same call that builds the edges, DropEdge, batch, rootindex
and y.  The gather is checked bit for bit on random bit patterns, the rest against the CSR forest, the model on such
batches against the oracle, and train_GCN end to end.  The argument checks at the bottom run without a GPU."""
import os

import numpy as np
import pytest
import torch

from oracle import bigcn_oracle, gcn_oracle
from bigcn_b200.data import Batch, collate, make_tree

gpu = pytest.mark.gpu
INT_OF = {torch.float32: torch.int32, torch.bfloat16: torch.int16}


def random_bits(n, k, dtype, gen=None, device="cpu"):
    """[n, k] of random 32- or 16-bit patterns (NaNs with arbitrary payloads included) plus -0.0 and a quiet NaN"""
    it = INT_OF[dtype]
    info = torch.iinfo(it)
    x = torch.randint(info.min, info.max + 1, (n, k), dtype=it, generator=gen, device=device).view(dtype)
    if n * k >= 2:
        x.view(-1)[0] = -0.0
        x.view(-1)[-1] = float("nan")
    return x


def bit_trees(k, sizes, dtype, seed=0):
    rng = np.random.default_rng(seed)
    g = torch.Generator().manual_seed(seed)
    trees = [make_tree("pheme", int(n), rng, in_feats=1) for n in sizes]
    for t in trees:
        t.x = random_bits(t.num_nodes, k, dtype, g)
    return trees


def forest_rows(forest, ids):
    """torch.cat of the chosen trees' rows of the forest's own storage"""
    p = forest.h_node_ptr
    return torch.cat([forest.x[p[t]:p[t + 1]] for t in ids]) if len(ids) else forest.x[:0]


def same_bits(a, b):
    return a.dtype == b.dtype and a.shape == b.shape and torch.equal(a.view(INT_OF[a.dtype]), b.view(INT_OF[b.dtype]))


def raw_dense_gather(forest, x_all, ids):
    """bigcn_assemble_batch_dense called directly (offsets in device memory), for storage DeviceForest refuses: bf16
    rows whose width is not a multiple of 8 still take the kernel's 2-byte path"""
    from bigcn_b200 import _lib as L
    dev = forest.device
    ids = np.asarray(ids, np.int64)
    sizes = forest.h_node_ptr[ids + 1] - forest.h_node_ptr[ids]
    node_off = np.concatenate([[0], np.cumsum(sizes)])
    e_off = np.concatenate([[0], np.cumsum(forest.h_edge_ptr[ids + 1] - forest.h_edge_ptr[ids])])
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a, np.int64)).to(dev)  # noqa: E731
    tid, noff, eoff = d(ids), d(node_off), d(e_off)
    n, e, b = int(node_off[-1]), int(e_off[-1]), len(ids)
    ei, bu = torch.empty(2, e, dtype=torch.int64, device=dev), torch.empty(2, e, dtype=torch.int64, device=dev)
    bt, root, y = (torch.empty(m, dtype=torch.int64, device=dev) for m in (n, b, b))
    ox = torch.empty(n, x_all.shape[1], dtype=x_all.dtype, device=dev)
    p = lambda t: t.data_ptr()  # noqa: E731
    L.check(L.lib().bigcn_assemble_batch_dense(p(forest.node_ptr), p(forest.edge_ptr), p(forest.edge_src),
                                               p(forest.edge_dst), p(forest.root_local), p(forest.y), p(tid), p(noff),
                                               p(eoff), p(eoff), b, e, e, 0, p(ei), p(bu), p(bt), p(root), p(y),
                                               p(x_all), x_all.shape[1], x_all.element_size(), p(ox),
                                               torch.cuda.current_stream().cuda_stream), "assemble_batch_dense")
    return ox


# ---------------------------------------------------------------------------------------------- 1. the gather
@gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("k", [768, 5000, 7, 13])
def test_dense_gather_is_bit_exact(dev, dtype, k):
    """Random bit patterns, NaN payloads and -0.0 included: 16-byte units (768, 5000) and the 4- or 2-byte element
    path (7, 13); arbitrary order, repeated ids, single-node trees and a 300-node tree beside them."""
    import bigcn_b200
    sizes = (1, 60, 2, 300, 17, 1, 1, 5)
    ids = [3, 0, 7, 1, 1, 5, 2, 3, 6, 4]
    trees = bit_trees(k, sizes, dtype, seed=k)
    if dtype == torch.bfloat16 and k % 8:
        forest = bigcn_b200.DeviceForest.from_data_list(bit_trees(k, sizes, torch.float32, seed=k), dev,
                                                        features="dense")
        x_all = torch.cat([t.x for t in trees]).to(dev)
        got = raw_dense_gather(forest, x_all, ids)
        p = forest.h_node_ptr
        assert same_bits(got, torch.cat([x_all[p[t]:p[t + 1]] for t in ids]))
        return
    forest = bigcn_b200.DeviceForest.from_data_list(trees, dev, features="dense", dtype=dtype)
    assert forest.x.dtype == dtype and same_bits(forest.x.cpu(), torch.cat([t.x for t in trees]))
    got = forest.batch(ids, 0.2, 0.2, seed=1)
    assert got.x.is_contiguous() and got.x.data_ptr() % 16 == 0
    assert same_bits(got.x, forest_rows(forest, ids))
    assert same_bits(got.x.cpu(), torch.cat([trees[i].x for i in ids]))
    empty = forest.batch([])
    assert empty.x.shape == (0, k) and empty.x.dtype == dtype and empty.batch.numel() == 0


@gpu
@pytest.mark.parametrize("k", [1, 3])
def test_dense_gather_many_small_trees(dev, k):
    """Thousands of one- to three-node trees at a few columns: one CTA's run of rows spans more trees than it stages
    at once, so it walks them in several rounds; the fp32 forest through DeviceForest, bf16 through the C entry."""
    import bigcn_b200
    rng = np.random.default_rng(k)
    sizes = rng.integers(1, 4, 3000)
    trees = bit_trees(k, sizes, torch.float32, seed=10 + k)
    forest = bigcn_b200.DeviceForest.from_data_list(trees, dev, features="dense")
    ids = rng.integers(0, len(trees), 6000)
    assert same_bits(forest.batch(ids).x, forest_rows(forest, ids))
    xb = random_bits(forest.x.shape[0], k, torch.bfloat16, device=dev)
    p = forest.h_node_ptr
    assert same_bits(raw_dense_gather(forest, xb, ids), torch.cat([xb[p[t]:p[t + 1]] for t in ids]))


@gpu
def test_dense_gather_past_2_31_elements(dev):
    """One bf16 batch at PHEME's v1 width (K = 196,608) with 11,295 nodes: 2.2e9 elements (4.4 GB), past 2^31."""
    import bigcn_b200
    k = 196608
    sizes = np.array([300, 1, 250, 1, 1, 200] * 15, np.int64)
    node_ptr = np.concatenate([[0], np.cumsum(sizes)])
    edge_ptr = node_ptr - np.arange(len(sizes) + 1)
    src = np.concatenate([np.arange(n - 1) for n in sizes]).astype(np.int32)
    n_all = int(node_ptr[-1])
    g = torch.Generator(device=dev).manual_seed(0)
    x = random_bits(n_all, k, torch.bfloat16, g, dev)
    forest = bigcn_b200.DeviceForest(node_ptr, edge_ptr, src, src + 1, None, None, None, np.zeros(len(sizes)),
                                     np.zeros(len(sizes)), k, dev, x=x)
    ids = np.random.default_rng(1).permutation(len(sizes))
    got = forest.batch(ids)
    assert got.x.numel() > 2 ** 31
    want = forest_rows(forest, ids)
    assert same_bits(got.x, want)
    del got, want, forest, x
    torch.cuda.empty_cache()
    # an odd width takes the 2-byte unit path, so the batch is past 2^31 UNITS too: source and destination unit
    # indices and (row + delta) * row_units overflow 32 bits here (the forest's own storage only gives the structure)
    k = 196607
    x = random_bits(n_all, k, torch.bfloat16, g, dev)
    forest = bigcn_b200.DeviceForest(node_ptr, edge_ptr, src, src + 1, None, None, None, np.zeros(len(sizes)),
                                     np.zeros(len(sizes)), 8, dev, x=torch.zeros(n_all, 8, dtype=torch.bfloat16, device=dev))
    got = raw_dense_gather(forest, x, ids)
    assert got.numel() > 2 ** 31
    assert same_bits(got, torch.cat([x[node_ptr[t]:node_ptr[t + 1]] for t in ids]))


# ---------------------------------------------------------------------------------------------- 2. same batch as CSR
@gpu
@pytest.mark.parametrize("shape,k", [("twitter15", 300), ("pheme", 64)])
def test_dense_batch_equals_csr_batch(dev, shape, k):
    """Same trees, ids, rates and seed: the dense and the CSR forest give equal edges, batch, rootindex and y, and x
    equals the CSR batch's to_dense(); a CSR tree (SparseX) is densified when packed."""
    import bigcn_b200
    from bigcn_b200.ops import host_dense_to_csr
    rng = np.random.default_rng(4)
    trees = [make_tree(shape, int(n), rng, in_feats=k) for n in (1, 60, 2, 300, 17, 90, 1, 5)]
    csr = bigcn_b200.DeviceForest.from_data_list(trees, dev)
    trees[2].x = host_dense_to_csr(trees[2].x, cap=trees[2].x.numel())
    dense = bigcn_b200.DeviceForest.from_data_list(trees, dev, features="dense")
    for ids, rates, seed in (([3, 0, 7, 1, 1, 5, 2], (0.0, 0.0), 0), ([3, 5, 6, 3, 1], (0.2, 0.35), 7),
                             (list(range(8)), (0.5, 0.1), 2 ** 40 + 3)):
        a, b = dense.batch(ids, *rates, seed=seed), csr.batch(ids, *rates, seed=seed)
        for key in ("edge_index", "BU_edge_index", "batch", "rootindex", "y"):
            assert torch.equal(getattr(a, key), getattr(b, key)), key
        assert a.x.dtype == torch.float32 and torch.equal(a.x, b.x.to_dense())


@gpu
def test_dense_npz_dir_against_the_reference_dataset_class(dev):
    """from_npz_dir(features='dense') on the reference's own .npz trees: the PyG collate of what
    BiGraphDataset.__getitem__ returned (tests/golden/ref_dataset.npz), bit for bit, in fp32."""
    import bigcn_b200
    gold = os.path.join(os.path.dirname(__file__), "golden")
    ref = np.load(os.path.join(gold, "ref_dataset.npz"))
    fold_x = [str(i) for i in ref["fold_x"]]
    sizes = {"1001": 9, "1002": 1, "1003": 14, "1004": 5, "1005": 2, "1006": 23, "1007": 7}
    tree_dic = {i: {j: {} for j in range(n)} for i, n in sizes.items()}
    forest = bigcn_b200.DeviceForest.from_npz_dir(fold_x, os.path.join(gold, "ref_dataset"), dev, treeDic=tree_dic,
                                                  lower=2, features="dense")
    assert forest.ids == [str(i) for i in ref["nodrop/kept_ids"]]
    from bigcn_b200.data import Data
    items = [Data(**{k: torch.from_numpy(ref[f"nodrop/{j}/{k}"]) for k in ("x", "edge_index", "BU_edge_index",
                                                                          "rootindex", "y")})
             for j in range(len(forest.ids))]
    order = [4, 0, 5, 2]
    got, want = forest.batch(order), collate([items[i] for i in order])
    for key in ("x", "edge_index", "BU_edge_index", "batch", "rootindex", "y"):
        assert torch.equal(getattr(got, key).cpu(), getattr(want, key)), key


@gpu
def test_from_device_arrays_dense_pheme(dev):
    """The PHEME dict of data.synth_forest_device (dense x): contiguous ids without DropEdge give forest_slice_batch's
    batch; bf16 storage is the same dict with x converted once."""
    import bigcn_b200
    from bigcn_b200.data import forest_slice_batch, synth_forest_device
    f = synth_forest_device("pheme", 200, dev, seed=5)
    forest = bigcn_b200.DeviceForest.from_device_arrays(f)
    got, want = forest.batch(list(range(17, 60))), forest_slice_batch(f, 17, 60)
    for key in ("x", "edge_index", "BU_edge_index", "batch", "rootindex", "y"):
        assert torch.equal(getattr(got, key), getattr(want, key)), key
    f["x"] = f["x"].to(torch.bfloat16)
    fb = bigcn_b200.DeviceForest.from_device_arrays(f)
    xb = fb.batch([5, 199, 0, 5]).x
    p = fb.h_node_ptr
    assert same_bits(xb, torch.cat([f["x"][p[t]:p[t + 1]] for t in (5, 199, 0, 5)]))


# ---------------------------------------------------------------------------------------------- 3. the model
def _pheme_forest(dev, dtype, n_trees=200, seed=5):
    import bigcn_b200
    from bigcn_b200.data import synth_forest_device
    f = synth_forest_device("pheme", n_trees, dev, seed=seed)
    f["x"] = f["x"].to(dtype)
    return bigcn_b200.DeviceForest.from_device_arrays(f)


def _host_copy(bd):
    return Batch(x=bd.x.float().cpu(), edge_index=bd.edge_index.cpu(), BU_edge_index=bd.BU_edge_index.cpu(),
                 batch=bd.batch.cpu(), rootindex=bd.rootindex.cpu(), y=bd.y.cpu())


@gpu
@pytest.mark.parametrize("dtype,mode", [(torch.float32, "auto"), (torch.bfloat16, "bf16")])
def test_model_on_dense_assembled_batch_matches_oracle(dev, dtype, mode):
    """Train-mode step on a DropEdge'd PHEME-shaped dense batch, the kernel's Philox mask injected into the oracle run
    on the same kept edges (read back) and x.float(): 'auto' resolves to tf32x3 with dense_roots."""
    import bigcn_b200
    K = 768
    forest = _pheme_forest(dev, dtype)
    ids = np.random.default_rng(0).choice(200, 24, replace=False)
    bd = forest.batch(ids, 0.2, 0.2, seed=3)
    assert bd.x.dtype == dtype
    torch.manual_seed(1)
    ref = bigcn_oracle.BiGCN(K, 64, 64).train()
    with torch.no_grad():
        for p in ref.parameters():
            if p.dim() == 1:
                p.uniform_(-0.1, 0.1)
    m = bigcn_b200.BiGCN(K, 64, 64, dev, gemm_mode=mode).to(dev).train()
    m.load_state_dict(ref.state_dict())
    if mode == "auto":
        assert m.TDrumorGCN.resolved_gemm_mode(bd.x) == "tf32x3"
    assert m.TDrumorGCN.resolved_dense_roots(bd.x) and m.BUrumorGCN.resolved_dense_roots(bd.x)
    got = m(bd)
    m.check_inputs()
    host = _host_copy(bd)
    n = host.x.shape[0]
    s = m.TDrumorGCN.last_seed
    ktd = torch.from_numpy(gcn_oracle.dropout_keep_mask(s, 0, np.arange(n), 64 + K, 0.5))
    kbu = torch.from_numpy(gcn_oracle.dropout_keep_mask(s, 1, np.arange(n), 64 + K, 0.5))
    want = ref(host, keep_td=ktd, keep_bu=kbu)
    err = float((got.detach().cpu().double() - want.detach().double()).abs().max() / want.detach().abs().max())
    assert err < 1e-5, err
    torch.nn.functional.nll_loss(want, host.y).backward()
    torch.nn.functional.nll_loss(got, bd.y).backward()
    for (name, p), (_, q) in zip(m.named_parameters(), ref.named_parameters()):
        e = float((p.grad.cpu().double() - q.grad.double()).abs().max() / max(float(q.grad.abs().max()), 1e-30))
        assert e < 1e-4, (name, e)


@gpu
@pytest.mark.parametrize("dtype,mode", [(torch.float32, "auto"), (torch.bfloat16, "bf16")])
def test_fused_trainer_on_dense_assembled_batches(dev, dtype, mode):
    """FusedTrainer steps on assembled batches give parameters bit-identical to steps on Batches built by hand from the
    torch-concatenated rows and the edges read back, with and without next_data."""
    import bigcn_b200
    forest = _pheme_forest(dev, dtype)
    rng = np.random.default_rng(3)
    lists = [rng.choice(200, 24, replace=False) for _ in range(3)]
    assembled = [forest.batch(ids, 0.2, 0.2, seed=40 + i) for i, ids in enumerate(lists)]
    by_hand = [Batch(x=forest_rows(forest, ids).clone(), edge_index=b.edge_index.clone(),
                     BU_edge_index=b.BU_edge_index.clone(), batch=b.batch.clone(), rootindex=b.rootindex.clone(),
                     y=b.y.clone()) for ids, b in zip(lists, assembled)]
    for look in (False, True):
        res = []
        for batches in (assembled, by_hand):
            torch.manual_seed(3)
            m = bigcn_b200.BiGCN(768, 64, 64, dev, gemm_mode=mode, validate="off").to(dev).train()
            tr = bigcn_b200.FusedTrainer(m, lr=5e-4, weight_decay=1e-4)
            for i, b in enumerate(batches):
                nxt = batches[i + 1] if look and i + 1 < len(batches) else None
                tr.step(b, next_data=nxt)
            tr.check_inputs()
            res.append((tr.flat.clone(), tr.exp_avg.clone()))
        for a, b in zip(*res):
            assert torch.equal(a, b), look


# ---------------------------------------------------------------------------------------------- 4. the loop
@gpu
@pytest.mark.parametrize("dtype,mode", [(torch.float32, "auto"), (torch.bfloat16, "bf16")])
def test_train_gcn_on_dense_forest(tmp_path, monkeypatch, dev, dtype, mode):
    """train_GCN on a 200-tree PHEME-shaped dense forest, 3 epochs, DropEdge 0.2: finite losses and metrics, the same
    seed twice gives bit-identical losses, and the final checkpoint has the keys of the CSR route's."""
    import bigcn_b200
    from bigcn_b200.data import make_trees_shard
    monkeypatch.chdir(tmp_path)
    forest = _pheme_forest(dev, dtype)
    ids = np.arange(200)
    runs = []
    for r in range(2):
        torch.manual_seed(0)
        model = bigcn_b200.BiGCN(768, 64, 64, dev, gemm_mode=mode).to(dev)
        out = bigcn_b200.train_GCN(model, forest, ids[:160], ids[160:], 0.2, 0.2, lr=5e-4, weight_decay=1e-4,
                                   patience=100, n_epochs=3, batchsize=24, datasetname="PHEME", fold=r, seed=7,
                                   log=lambda s: None)
        assert len(out[0]) == 3
        assert all(np.isfinite(v).all() for v in out[:4]) and all(np.isfinite(v) for v in out[4:])
        runs.append((out, torch.load(bigcn_b200.train_GCN.last_final_checkpoint, weights_only=False)))
    assert runs[0][0][0] == runs[1][0][0] and runs[0][0][1] == runs[1][0][1]
    trees = make_trees_shard("twitter16", 24, seed=6, in_feats=64)[0]
    csr = bigcn_b200.DeviceForest.from_data_list(trees, dev)
    torch.manual_seed(0)
    model = bigcn_b200.BiGCN(64, 64, 64, dev, gemm_mode="sparse").to(dev)
    bigcn_b200.train_GCN(model, csr, np.arange(16), np.arange(16, 24), 0.2, 0.2, lr=5e-4, weight_decay=1e-4,
                         patience=100, n_epochs=1, batchsize=8, fold=9, log=lambda s: None)
    want = torch.load(bigcn_b200.train_GCN.last_final_checkpoint, weights_only=False)
    got = runs[0][1]
    assert set(got) == set(want)
    assert set(got["model_state_dict"]) == set(want["model_state_dict"])
    assert set(got["optimizer_state_dict"]) == set(want["optimizer_state_dict"])


# ---------------------------------------------------------------------------------------------- 5. errors (no GPU)
def test_bf16_storage_width_is_checked_when_packing(built_lib):
    """bf16 rows must be a multiple of 8 wide (what gemm_mode='bf16' reads): refused before anything reaches the
    device; so is an unknown storage form."""
    import bigcn_b200
    trees = bit_trees(12, (3, 1), torch.float32)
    with pytest.raises(bigcn_b200.BigcnError, match="multiple of 8"):
        bigcn_b200.DeviceForest.from_data_list(trees, "cuda", features="dense", dtype=torch.bfloat16)
    with pytest.raises(bigcn_b200.BigcnError, match="'csr' or 'dense'"):
        bigcn_b200.DeviceForest.from_data_list(trees, "cuda", features="rows")
    with pytest.raises(bigcn_b200.BigcnError, match="float32 or torch.bfloat16"):
        bigcn_b200.DeviceForest.from_data_list(trees, "cuda", features="dense", dtype=torch.float16)


@pytest.mark.parametrize("k,elem_bytes,b,what", [(768, 3, 1, "elem_bytes"), (768, 8, 0, "elem_bytes"),
                                                 (0, 4, 1, "K = 0"), (-5, 2, 1, "K = -5"), (1 << 29, 2, 1, "K = "),
                                                 (768, 4, 1, "NULL")])
def test_assemble_batch_dense_rejects_bad_arguments(built_lib, k, elem_bytes, b, what):
    """Checked before any launch: an error code and a message, never a fault (NULL pointers throughout)."""
    from bigcn_b200 import _lib as L
    rc = L.lib().bigcn_assemble_batch_dense(*([None] * 10), b, 0, 0, 0, *([None] * 6), k, elem_bytes, None, None)
    assert rc != 0 and what in L.lib().bigcn_last_error().decode()


def test_assemble_batch_dense_rejects_misaligned_rows(built_lib):
    """An x_all or ox not aligned to its element size is an error before any launch (non-NULL stand-in pointers)."""
    from bigcn_b200 import _lib as L
    for x_all, ox, elem_bytes in ((18, 16, 4), (16, 17, 2), (16, 14, 4)):
        rc = L.lib().bigcn_assemble_batch_dense(*([16] * 10), 1, 0, 0, 0, *([16] * 5), x_all, 768, elem_bytes, ox, None)
        assert rc != 0 and "aligned" in L.lib().bigcn_last_error().decode()


def test_assemble_batch_dense_empty_batch_is_a_no_op(built_lib):
    from bigcn_b200 import _lib as L
    assert L.lib().bigcn_assemble_batch_dense(*([None] * 10), 0, 0, 0, 0, *([None] * 6), 768, 2, None, None) == 0
