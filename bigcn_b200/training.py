"""The caller of the path: the reference's ``train_GCN`` loop (model/Twitter/BiGCN_Twitter.py:134-275)
with this library's pieces in place of the host-side ones -- same structure, same bookkeeping,
no per-batch host synchronisation:

  loadBiData + DataLoader(shuffle=True) per epoch (:160-169)  -> DeviceForest.batches(id lists, droprates, seeds)
  forward / nll_loss / backward / optimizer.step (:183-189)    -> FusedTrainer.step
  loss.item(), pred.eq(y).sum().item() per batch (:188-191)    -> EvalCounts.update (device), read once per epoch
  evaluation4class per validation batch + np.mean (:217-246)   -> EvalCounts.epoch_means
  checkpoint dict (:253-261), EarlyStopping (:269-275)         -> make_checkpoint, EarlyStopping

Returns what train_GCN returns: (train_losses, val_losses, train_accs, val_accs, accs, F1, F2, F3, F4).
"""
from __future__ import annotations

import numpy as np
import torch

from .checkpoint import EarlyStopping, make_checkpoint
from .metrics import EvalCounts
from .trainer import FusedTrainer


def train_GCN(model, forest, train_ids, test_ids, TDdroprate, BUdroprate, lr, weight_decay, patience, n_epochs,
              batchsize, datasetname="Twitter16", iter=0, fold=0, modelname="BiGCN", seed=0, log=print,
              trainer=None, save=True, checkpoint_dir="checkpoints"):
    """``model``: a bigcn_b200.BiGCN / Net on the device; ``forest``: a DeviceForest holding every tree;
    ``train_ids`` / ``test_ids``: tree indices of the fold (the reference's x_train / x_test).  A forest with edge
    weights trains them (``FusedTrainer(..., edge_weights=True)`` unless ``trainer`` is given) and validates with them."""
    dev = forest.device
    c = model.fc.weight.shape[0]
    tr = trainer or FusedTrainer(model, lr=lr, weight_decay=weight_decay,
                                 edge_weights=getattr(forest, "edge_weight", None) is not None)
    train_ev, val_ev = EvalCounts(c, dev), EvalCounts(c, dev)
    early_stopping = EarlyStopping(patience=patience, verbose=True)
    rng = np.random.default_rng(seed)
    train_losses, val_losses, train_accs, val_accs = [], [], [], []
    train_ids, test_ids = np.asarray(train_ids, np.int64), np.asarray(test_ids, np.int64)
    accs = F1 = F2 = F3 = F4 = 0
    checkpoint, epoch, final_path = None, -1, None

    def save_final(tag):
        """BiGCN_Twitter.py:311-325 (for/else: n_epochs ran out without early stopping ->
        final_bigcn_f{fold}_i{iter}_e{epoch}_l{loss}.pt) and :326-340 (KeyboardInterrupt ->
        interrupt_bigcn_f{fold}_i{iter}_e{epoch}_last.pt), in ``checkpoint_dir``."""
        if not save:
            return None
        import os
        ck = checkpoint if checkpoint is not None else make_checkpoint(model, tr, fold, iter, max(epoch, 0),
                                                                        train_losses[-1] if train_losses else float("nan"), [])
        os.makedirs(checkpoint_dir, exist_ok=True)
        name = ("final_bigcn_f{}_i{}_e{:05d}_l{:.5f}.pt".format(fold, iter, epoch, train_losses[-1]) if tag == "final"
                else "interrupt_bigcn_f{}_i{}_e{:05d}_last.pt".format(fold, iter, max(epoch, 0)))
        path = os.path.join(checkpoint_dir, name)
        torch.save(ck, path)
        return path

    try:
        for epoch in range(n_epochs):
            model.train()
            train_ev.reset()
            order = rng.permutation(train_ids)                        # DataLoader(shuffle=True), :168
            lists = [order[lo:lo + batchsize] for lo in range(0, len(order), batchsize)]
            seeds = [(seed << 20) + epoch * 4096 + bi for bi in range(len(lists))]
            for data, nxt in forest.batches(lists, TDdroprate, BUdroprate, seeds):   # batch i+1 is prepared under step i
                tr.step(data, next_data=nxt)                           # :183-189
                train_ev.update(tr.last_logp, data.y)                  # :188-191, no .item()
            # np.mean over batches of the per-batch loss / accuracy (:199-200): one read per epoch
            tl, ta, _ = train_ev.epoch_means()
            train_losses.append(tl)
            train_accs.append(ta)
            model.eval()
            val_ev.reset()
            order = rng.permutation(test_ids)
            with torch.no_grad():
                for lo in range(0, len(order), batchsize):
                    data = forest.batch(order[lo:lo + batchsize], 0.0, 0.0)   # test trees: no DropEdge (Process/dataset.py)
                    val_ev.update(model(data), data.y)                 # :217-225
            vl, va, m = val_ev.epoch_means()
            val_losses.append(vl)
            val_accs.append(va)
            log("Fold {} | Epoch {:05d} | Val_Loss {:.4f}| Val_Accuracy {:.4f}".format(fold, epoch, vl, va))
            res = ["acc:{:.4f}".format(m[0])] + ["C{}:{:.4f},{:.4f},{:.4f},{:.4f}".format(k + 1, *m[1 + 4 * k:5 + 4 * k])
                                                 for k in range(c)]   # :236-245
            checkpoint = make_checkpoint(model, tr, fold, iter, epoch, train_losses[-1], res)
            f = [m[4 + 4 * k] if k < c else 0 for k in range(4)]      # F1 of each class (two classes: F3 = F4 = 0)
            early_stopping(vl, va, f[0], f[1], f[2], f[3], model, modelname, datasetname, checkpoint=checkpoint)
            accs, F1, F2, F3, F4 = va, f[0], f[1], f[2], f[3]
            tr.check_inputs()     # the epoch's reads above synchronised anyway: a bad batch (e.g. features too dense for
            #                       gemm_mode='sparse', NaN dW1) is reported now, not after all epochs
            if early_stopping.early_stop:
                log("Early stopping")
                accs, F1, F2, F3, F4 = (early_stopping.accs, early_stopping.F1, early_stopping.F2, early_stopping.F3,
                                        early_stopping.F4)
                break
        else:
            final_path = save_final("final")
    except KeyboardInterrupt:
        final_path = save_final("interrupt")
        raise
    train_GCN.last_final_checkpoint = final_path
    if not save and early_stopping.saved_path:
        import os
        os.remove(early_stopping.saved_path)
    tr.check_inputs()
    return train_losses, val_losses, train_accs, val_accs, accs, F1, F2, F3, F4
