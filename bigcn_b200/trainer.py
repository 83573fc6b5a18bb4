"""The training step around the path (BiGCN_Twitter.py:146-153 optimizer, :183-189 step).

``FusedTrainer`` keeps the ten parameter tensors as views of ONE flat fp32 buffer (and one
flat gradient buffer), so a step is: features forward -> head -> nll -> head backward ->
features backward written straight into the flat gradient -> (data-parallel: one NCCL
all-reduce of that 5 MB buffer) -> one fused Adam kernel with the reference's three lr
groups (BU convs at lr/5).  Nothing in a step synchronises the host.
"""
from __future__ import annotations

import ctypes as C
import weakref

import torch
import torch.utils.weak

from . import _lib as L
from ._lib import H, Opts, Params, check, lib
from .ops import _make_structs, _p, _stream, _i64, _f32, _as_x, capture_graph, edge_weight, raise_on_flags, step_stream

# flat layout: the two conv1 weights (the gradients the second X stream produces LAST) first, so
# the gradient splits into two contiguous all-reduce buckets: [W1_td | W1_bu] and [everything else]
_ORDER = ("TDrumorGCN.conv1.lin.weight", "BUrumorGCN.conv1.lin.weight",
          "TDrumorGCN.conv1.bias", "TDrumorGCN.conv2.lin.weight", "TDrumorGCN.conv2.bias", "fc.weight", "fc.bias",
          "BUrumorGCN.conv1.bias", "BUrumorGCN.conv2.lin.weight", "BUrumorGCN.conv2.bias")
_LR_DIV = (1, 5, 1, 1, 1, 1, 1, 5, 5, 5)     # BU conv1 / conv2 at lr/5 (BiGCN_Twitter.py:146-153)
_STRUCT = {"TDrumorGCN.conv1.lin.weight": "td_w1", "TDrumorGCN.conv1.bias": "td_b1",
           "TDrumorGCN.conv2.lin.weight": "td_w2", "TDrumorGCN.conv2.bias": "td_b2",
           "BUrumorGCN.conv1.lin.weight": "bu_w1", "BUrumorGCN.conv1.bias": "bu_b1",
           "BUrumorGCN.conv2.lin.weight": "bu_w2", "BUrumorGCN.conv2.bias": "bu_b2",
           "fc.weight": "fc_w", "fc.bias": "fc_b"}


class FusedTrainer:
    """Adam(lr, weight_decay) with BU conv1/conv2 at lr/5 over a flat parameter buffer."""

    def __init__(self, model, lr=5e-4, weight_decay=1e-4, betas=(0.9, 0.999), eps=1e-8,
                 process_group=None, world_size=1, validate=False, comm="auto", graphs="auto", max_graphs=16,
                 fused_sync=True, dp_push=True, edge_weights=False, edge_grad=False):
        """``comm`` (world_size > 1): "symm" = one fused kernel over NVLink peer memory
        (reduce-scatter of the gradients in rank order + Adam on the owned shard + all-gather of
        the parameters, bigcn_dp_reduce_adam) between two symmetric-memory barriers; "nccl" = two
        bucketed NCCL all-reduces overlapping the last backward kernels + Adam on every rank;
        "auto" = symm when the symmetric-memory rendezvous succeeds, else nccl.
        ``graphs``: replay a CUDA graph of the whole step for batches seen before (True / False;
        "auto" = on for a single GPU and for comm="symm", off for the NCCL path whose collectives
        run on NCCL's own stream); at most ``max_graphs`` batches are kept captured.
        ``fused_sync`` (comm="symm"): the two cross-rank barriers around the optimiser kernel happen inside it
        (release / acquire on signal words in symmetric memory) instead of as two more launches.
        ``edge_weights``: True = ``step`` takes batches that carry ``data.edge_weight`` (TD) and / or
        ``data.BU_edge_weight`` (BU), both convs of a direction weighted as ``GCNConv(x, edge_index, edge_weight)``; their
        normalisation is prepared a step ahead with the rest of ``next_data``.  Unless ``edge_grad`` is set the weights get
        no gradient here (one that requires grad is refused: train it through the modules).  False = such a batch is
        refused.
        ``edge_grad`` (implies ``edge_weights``; single GPU only): a weight that requires grad gets the gradient of the
        step's loss (the mean nll over ``b_global`` trees), handed to autograd as ``loss.backward()`` would -- a leaf
        accumulates it into ``.grad``, a non-leaf passes it on to whatever produced it.  A batch prepared a step ahead is
        matched to its weights by tensor identity and ``_version``: a weight written in place or replaced after it was
        prepared is prepared again inline."""
        L.require_device()
        if edge_grad and world_size > 1:
            raise L.BigcnError("FusedTrainer(edge_grad=True) runs on one GPU: data-parallel edge-weight gradients are not "
                               "supported")
        self.model = model
        self.lr, self.wd, self.betas, self.eps = lr, weight_decay, betas, eps
        self.pg, self.world = process_group, world_size
        self.validate = validate
        self.edge_grad = bool(edge_grad)
        self.edge_weights = bool(edge_weights) or self.edge_grad
        self._wserial, self._wnext = torch.utils.weak.WeakIdKeyDictionary(), 0   # edge_grad: weight tensor -> serial
        self.fused_sync = bool(fused_sync)     # comm="symm": cross-rank barriers inside the optimiser kernel
        self.dp_push = bool(dp_push)           # ... and gradient slices pushed to their owners (peer stores) instead of pulled
        self.raise_priority = False            # enqueued (not replayed) steps without a prepared batch: stay on the caller's stream
        self.comm, self.comm_note = "single", ""
        named = dict(model.named_parameters())
        dev = named[_ORDER[0]].device
        if dev.type != "cuda":
            raise L.BigcnError("FusedTrainer needs the model on a CUDA device")
        sizes = [named[n].numel() for n in _ORDER]
        offs = [0]
        for s in sizes:
            offs.append(offs[-1] + (s + 3) // 4 * 4)   # keep every tensor 16 B aligned
        self.n = offs[-1]
        self.flat = self.grad = None
        if world_size > 1:
            self.comm = "nccl"
            if comm in ("auto", "symm"):
                try:
                    self._setup_symm(dev)
                    self.comm = "symm"
                except Exception as e:  # noqa: BLE001
                    if comm == "symm":
                        raise
                    self.comm_note = f"symmetric memory unavailable ({type(e).__name__}: {e}); using NCCL all-reduce"
        if self.flat is None:
            self.flat = torch.zeros(self.n, dtype=torch.float32, device=dev)
            self.grad = torch.zeros(self.n, dtype=torch.float32, device=dev)
        self.exp_avg = torch.zeros_like(self.flat)
        self.exp_avg_sq = torch.zeros_like(self.flat)
        self.views, self.gviews = {}, {}
        with torch.no_grad():
            for name, o, s in zip(_ORDER, offs, sizes):
                p = named[name]
                v = self.flat[o:o + s].view(p.shape)
                v.copy_(p)
                p.data = v                         # the module now reads the flat buffer
                self.views[name] = v
                self.gviews[name] = self.grad[o:o + s].view(p.shape)
        if self.world > 1:                         # identical start on every rank
            torch.distributed.broadcast(self.flat, src=0, group=self.pg)
        # lr groups: TD convs + fc at lr, BU convs at lr/5  (BiGCN_Twitter.py:146-153)
        self.seg_end = torch.tensor(offs[1:], dtype=torch.int64, device=dev)
        self.seg_lr_host = [lr / d for d in _LR_DIV]
        self.seg_lr = torch.tensor(self.seg_lr_host, dtype=torch.float32, device=dev)
        self.n_seg = len(_LR_DIV)
        self.w1_end = offs[2]                    # [0, w1_end) = the two conv1 weight gradients
        self.step_count = torch.zeros(4, dtype=torch.int64, device=dev)   # [step, arrival counter, calls, spare]
        self.flags = torch.zeros(1, dtype=torch.int32, device=dev)
        self._pr, self._gr = Params(), Params()
        for name in _ORDER:
            setattr(self._pr, _STRUCT[name], _p(self.views[name]))
            setattr(self._gr, _STRUCT[name], _p(self.gviews[name]))
        self._ws = None
        self._calls = 0
        self.launches_per_step = None
        self.graphs = (self.comm in ("single", "symm")) if graphs == "auto" else bool(graphs)
        self.max_graphs = int(max_graphs)
        self._graphs, self._seen = {}, {}   # captured steps by batch identity; batch identities seen once
        self._prep_buf, self._prep_owner = None, [None, None]   # two prepared-batch buffers and what they hold
        self.graph_captures = self.graph_replays = 0

    # -------------------------------------------------------------------------------
    def _setup_symm(self, dev):
        """Flat parameter / gradient buffers in symmetric memory: every rank's buffers mapped into
        every process over NVLink (torch.distributed._symmetric_memory: allocation, rendezvous and
        the cross-rank barrier; the data path is this library's kernel)."""
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm
        group = self.pg if self.pg is not None else dist.group.WORLD
        try:
            symm.enable_symm_mem_for_group(group.group_name)
        except Exception:  # noqa: BLE001  (not needed / deprecated on recent torch)
            pass
        flat = symm.empty(self.n, dtype=torch.float32, device=dev)
        grad = symm.empty(self.n, dtype=torch.float32, device=dev)
        hf, hg = symm.rendezvous(flat, group), symm.rendezvous(grad, group)
        if hf.world_size != self.world or len(hg.buffer_ptrs) != self.world:
            raise RuntimeError("symmetric memory world size mismatch")
        flat.zero_()
        grad.zero_()
        self.flat, self.grad, self._hf, self._hg = flat, grad, hf, hg
        self._rank = hf.rank
        self._pptrs = (C.c_void_p * self.world)(*[int(p) for p in hf.buffer_ptrs])
        self._gptrs = (C.c_void_p * self.world)(*[int(p) for p in hg.buffer_ptrs])
        # signal blocks of the in-kernel barriers of bigcn_dp_reduce_adam (64 uint64 per rank: 2 x 16 epoch words, never reset, + time stamps)
        self._sptrs = self._stptrs = None
        if self.fused_sync:
            sig = symm.empty(64, dtype=torch.int64, device=dev)
            hs = symm.rendezvous(sig, group)
            sig.zero_()
            torch.cuda.synchronize()
            dist.barrier(group=group)          # every rank's block is zero before anyone signals
            self._sig, self._hs = sig, hs
            self._sptrs = (C.c_void_p * self.world)(*[int(p) for p in hs.buffer_ptrs])
            # staging rows for the PUSH form: rank r writes its gradient slice q into rank q's row r before the barrier
            self._stptrs = None
            if self.dp_push:
                chunk = lib().bigcn_dp_stage_chunk(self.n, self.world)
                stage = symm.empty(self.world * chunk, dtype=torch.float32, device=dev)
                hst = symm.rendezvous(stage, group)
                self._stage, self._hst = stage, hst
                self._stptrs = (C.c_void_p * self.world)(*[int(p) for p in hst.buffer_ptrs])

    def _workspace(self, dims, dev, weighted=False, edge_grad=False):
        need = lib().bigcn_features_edge_workspace_bytes(C.byref(dims), int(edge_grad)) if weighted else \
            lib().bigcn_features_workspace_bytes(C.byref(dims))
        if self._ws is None or self._ws.numel() < need:
            # head room: captured graphs hold pointers into the workspace, a slightly larger batch should not move it
            self._ws = torch.empty(need + need // 4 if self.graphs else need, dtype=torch.uint8, device=dev)
        return self._ws

    def _plan(self, data, b_global, node_id_base, seed):
        """Everything one step needs besides the launches: argument structs, output buffers, workspace."""
        m = self.model
        x, xs = _as_x(data.x, m.TDrumorGCN.resolved_gemm_mode(data.x))
        ei, bu, batch, root = _i64(data.edge_index), _i64(data.BU_edge_index), _i64(data.batch), \
            _i64(data.rootindex)
        y = _i64(data.y)
        td = m.TDrumorGCN
        c = m.fc.weight.shape[0]
        ew = self._weights(data, ei, bu)
        # edge_grad: d loss / d weight of each direction whose weight requires grad (ew keeps the autograd link of a cast)
        dew = [torch.empty(w.numel(), dtype=torch.float32, device=w.device) if w is not None and w.requires_grad else None
               for w in ew]
        eg = self.edge_grad and any(d is not None for d in dew)
        dims, bt, _ = _make_structs(x, ei, bu, batch, root, (None,) * 8, c, node_id_base, xs, ew)
        # seed=None: the module's seed plus the device-side calls counter (step_count[2], advanced by the
        # optimiser kernel) -- the same value whether the step is enqueued or replayed from a CUDA graph
        o = Opts(training=int(m.training), p_drop=float(td.p), seed=int(td.seed if seed is None else seed) & ((1 << 64) - 1),
                 deg_by=L.DEG_BY[td.deg_by], gemm_mode=L.GEMM_MODE[td.resolved_gemm_mode(data.x)], dir_mask=L.DIR_TD | L.DIR_BU,
                 fused_tail=1, seed_dev=self.step_count[2:].data_ptr() if seed is None else None,
                 dense_roots=int(td.resolved_dense_roots(data.x)), edge_grad=int(eg))
        dev = xs.device if xs is not None else x.device
        b = dims.B
        p = {"dims": dims, "bt": bt, "o": o, "b": b, "c": c, "dev": dev, "y": y, "b_global": int(b_global or b),
             "keep": (x, xs, ei, bu, batch, root, y, ew), "weighted": any(w is not None for w in ew),
             "edge_grad": eg, "ew": ew, "dew": dew,
             "feat": torch.empty(b, 4 * H, dtype=torch.float32, device=dev),
             "logp": torch.empty(b, c, dtype=torch.float32, device=dev),
             "gfeat": torch.empty(b, 4 * H, dtype=torch.float32, device=dev),
             "loss": torch.empty(1, dtype=torch.float32, device=dev)}
        p["nscr"] = lib().bigcn_head_train_scratch_floats(b, c)
        p["scr"] = torch.empty(p["nscr"], dtype=torch.float32, device=dev)
        return p

    def _enqueue(self, p):
        """The launches of one step on the current stream (nothing allocates, nothing synchronises)."""
        dims, bt, o = p["dims"], p["bt"], p["o"]
        feat, logp, gfeat, loss, scr = p["feat"], p["logp"], p["gfeat"], p["loss"], p["scr"]
        ws = self._ws
        st = _stream()
        l = lib()
        if p.get("prep_inline"):     # this batch was not prepared a step ahead: do it now, on the critical path
            buf = self._prep_buf[p["slot"]]
            check(l.bigcn_batch_prepare(C.byref(dims), C.byref(bt), C.byref(o), _p(self.flags), _p(buf), buf.numel(), st),
                  "batch_prepare")
            check(l.bigcn_batch_prepare_join(st), "batch_prepare_join")
        nxt = p.get("next")
        if nxt is not None:          # the NEXT batch's weight-independent half, beside everything below
            buf = self._prep_buf[nxt["slot"]]
            check(l.bigcn_batch_prepare(C.byref(nxt["dims"]), C.byref(nxt["bt"]), C.byref(o), _p(self.flags), _p(buf),
                                        buf.numel(), st), "batch_prepare")
        check(l.bigcn_features_forward(C.byref(dims), C.byref(bt), C.byref(self._pr), C.byref(o), _p(feat),
                                       _p(self.flags), _p(ws), ws.numel(), st), "features_forward")
        # readout's second pass + fc / log_softmax / nll and their backward + the per-tree gradient scaling: one launch
        check(l.bigcn_train_tail(C.byref(dims), C.byref(bt), C.byref(o), _p(feat), _p(p["y"]), p["b_global"],
                                 self._pr.fc_w, self._pr.fc_b, _p(logp), _p(loss), _p(gfeat), self._gr.fc_w,
                                 self._gr.fc_b, _p(scr), p["nscr"], _p(self.flags), _p(ws), ws.numel(), st), "train_tail")
        if self.comm == "symm":
            check(l.bigcn_features_backward(C.byref(dims), C.byref(bt), C.byref(self._pr), C.byref(o), _p(gfeat),
                                            C.byref(self._gr), _p(ws), ws.numel(), st), "features_backward")
            if self._sptrs is None:
                self._hg.barrier(channel=0)    # every rank's gradient is complete
            # with signal blocks both cross-rank barriers happen inside the kernel (one launch instead of three)
            check(l.bigcn_dp_reduce_adam(self._gptrs, self._pptrs, self.world, self._rank, _p(self.exp_avg),
                                         _p(self.exp_avg_sq), self.n, _p(self.seg_end), _p(self.seg_lr), self.n_seg,
                                         self.betas[0], self.betas[1], self.eps, self.wd, 1.0, _p(self.step_count),
                                         self._sptrs, self._stptrs if self._sptrs is not None else None, st), "dp_reduce_adam")
            if self._sptrs is None:
                self._hf.barrier(channel=1)    # every rank's parameters are written; gradients are free again
        else:
            if self.world > 1:
                # everything but dW1, then its all-reduce runs (on NCCL's stream) under the second X stream
                o.bwd_phase = 1
                check(l.bigcn_features_backward(C.byref(dims), C.byref(bt), C.byref(self._pr), C.byref(o), _p(gfeat),
                                                C.byref(self._gr), _p(ws), ws.numel(), st), "features_backward")
                h_rest = torch.distributed.all_reduce(self.grad[self.w1_end:], group=self.pg, async_op=True)
                o.bwd_phase = 2
                check(l.bigcn_features_backward(C.byref(dims), C.byref(bt), C.byref(self._pr), C.byref(o), _p(gfeat),
                                                C.byref(self._gr), _p(ws), ws.numel(), st), "features_backward")
                o.bwd_phase = 0
                h_w1 = torch.distributed.all_reduce(self.grad[:self.w1_end], group=self.pg, async_op=True)
                h_rest.wait()
                h_w1.wait()
            else:
                check(l.bigcn_features_backward(C.byref(dims), C.byref(bt), C.byref(self._pr), C.byref(o), _p(gfeat),
                                                C.byref(self._gr), _p(ws), ws.numel(), st), "features_backward")
            check(l.bigcn_adam_step(_p(self.flat), _p(self.grad), _p(self.exp_avg), _p(self.exp_avg_sq), self.n,
                                    _p(self.seg_end), _p(self.seg_lr), self.n_seg, self.betas[0], self.betas[1],
                                    self.eps, self.wd, 1.0, _p(self.step_count), st), "adam_step")
            if p["edge_grad"]:       # forks from inside the backward (it runs under T1 / dW1), joins here
                dew = p["dew"]
                check(l.bigcn_features_edge_grad(C.byref(dims), C.byref(bt), C.byref(o), _p(dew[0]), _p(dew[1]), _p(ws),
                                                 ws.numel(), st), "features_edge_grad")
        if nxt is not None:          # the next step may start: its batch is prepared
            check(l.bigcn_batch_prepare_join(st), "batch_prepare_join")

    def _enqueue_prio(self, p, raised):
        """_enqueue on a stream one priority level above the caller's (the default stream has the lowest priority
        there is): the library's lowest-priority streams -- the next batch's preparation, the backward's dW2 / db
        chains -- then really yield SM slots to the step's critical chain."""
        if not (raised or self.raise_priority):
            return self._enqueue(p)
        cur = torch.cuda.current_stream()
        s = step_stream(p["dev"])
        s.wait_stream(cur)
        with torch.cuda.stream(s):
            self._enqueue(p)
        cur.wait_stream(s)
        for t in (p["feat"], p["logp"], p["gfeat"], p["loss"], p["scr"], *(d for d in p["dew"] if d is not None)):
            t.record_stream(s)

    # ---- batches prepared one step ahead (bigcn_batch_prepare) ---------------------------------------------
    def _prep_key(self, data):
        td = self.model.TDrumorGCN
        x = data.x
        xk = (x.ptr.data_ptr(), x.col.data_ptr(), x.val.data_ptr(), x.shape) if hasattr(x, "ptr") else \
            (x.data_ptr(), tuple(x.shape), x.dtype, x.layout)
        small = tuple((t.data_ptr(), tuple(t.shape), t.dtype) for t in
                      (data.edge_index, data.BU_edge_index, data.batch, data.rootindex))
        return (id(data), xk, small, self._weight_key(data, True), td.deg_by, td.resolved_gemm_mode(data.x))

    def _prep_setup(self, p, data, next_data, node_id_base):
        """Decide which prepared buffer this step reads (or prepares inline) and which one the next batch's
        preparation writes; returns the part of the CUDA-graph key that pins those decisions."""
        l = lib()
        pk = self._prep_key(data)

        def prep_bytes(dims, weighted):
            return (l.bigcn_batch_prepare_edge_bytes if weighted else l.bigcn_batch_prepare_bytes)(C.byref(dims))
        need = prep_bytes(p["dims"], p["weighted"])
        nxt = None
        if next_data is not None:
            nx, nxs = _as_x(next_data.x, self.model.TDrumorGCN.resolved_gemm_mode(next_data.x))
            nei, nbu = _i64(next_data.edge_index), _i64(next_data.BU_edge_index)
            new = self._weights(next_data, nei, nbu)
            nd, nbt, _ = _make_structs(nx, nei, nbu, _i64(next_data.batch), _i64(next_data.rootindex), (None,) * 8, p["c"],
                                       0, nxs, new)
            need = max(need, prep_bytes(nd, any(w is not None for w in new)))
            nxt = {"dims": nd, "bt": nbt, "keep": (nx, nxs, nei, nbu, new, next_data), "key": self._prep_key(next_data)}
        if self._prep_buf is None or self._prep_buf[0].numel() < need:
            self._prep_buf = [torch.empty(need + need // 4, dtype=torch.uint8, device=p["dev"]) for _ in range(2)]
            self._prep_owner = [None, None]
            self._graphs.clear()               # captured pointers into the old buffers are stale
        slot = next((i for i in (0, 1) if self._prep_owner[i] is not None and self._prep_owner[i][0] == pk
                     and self._prep_owner[i][1]() is data), None)
        p["prep_inline"] = slot is None
        if slot is None:
            slot = 0
        p["slot"] = slot
        p["bt"].prepared = self._prep_buf[slot].data_ptr()
        if nxt is not None:
            nxt["slot"] = 1 - slot
            p["next"] = nxt
        return (slot, p["prep_inline"], None if nxt is None else nxt["key"])

    def _prep_peek(self, data, next_data):
        """(slot, inline, key of the next batch) as _prep_setup would decide them, without building anything."""
        slot = None
        if self._prep_buf is not None:
            pk = self._prep_key(data)
            slot = next((i for i in (0, 1) if self._prep_owner[i] is not None and self._prep_owner[i][0] == pk
                         and self._prep_owner[i][1]() is data), None)
        return (0 if slot is None else slot, slot is None, None if next_data is None else self._prep_key(next_data))

    def _prep_commit(self, p, data, next_data):
        """Host-side record of what the prepared buffers hold after this step (enqueued or replayed)."""
        self._prep_owner[p["slot"]] = (self._prep_key(data), weakref.ref(data))
        if p.get("next") is not None:
            self._prep_owner[p["next"]["slot"]] = (p["next"]["key"], weakref.ref(next_data))

    def _graph_key(self, data, b_global, node_id_base):
        m, td = self.model, self.model.TDrumorGCN
        x = data.x
        xk = (x.ptr.data_ptr(), x.col.data_ptr(), x.val.data_ptr(), x.shape) if hasattr(x, "ptr") else \
            (x.data_ptr(), tuple(x.shape), x.dtype, x.layout)
        small = tuple((t.data_ptr(), tuple(t.shape), t.dtype) for t in
                      (data.edge_index, data.BU_edge_index, data.batch, data.rootindex, data.y))
        return (id(data), xk, small, self._weight_key(data, False), b_global, node_id_base, m.training, td.p, td.deg_by,
                td.gemm_mode, td.dense_roots, td.seed)

    # ---- edge weights (edge_weights=True) ------------------------------------------------------------------
    def _weight_key(self, data, prepared):
        """what a captured step or a prepared buffer read of the batch's weights: the tensors, not their values.  With
        edge_grad the tensors are told apart by identity (a serial per live tensor, so one at a recycled address is
        another) and, for a prepared buffer (``prepared``), by ``_version``: learnt weights change between steps, and a
        normalisation prepared from older values must not be used"""
        ws = (getattr(data, "edge_weight", None), getattr(data, "BU_edge_weight", None))
        if not self.edge_grad:
            return tuple((w.data_ptr(), tuple(w.shape), w.dtype) if torch.is_tensor(w) else id(w) for w in ws)
        return tuple((w.data_ptr(), self._serial(w), w._version if prepared else None, tuple(w.shape), w.dtype,
                      w.requires_grad) if torch.is_tensor(w) else id(w) for w in ws)

    def _serial(self, w):
        s = self._wserial.get(w)
        if s is None:
            self._wnext += 1
            s = self._wserial[w] = self._wnext
        return s

    def _check_weights(self, data):
        ws = (getattr(data, "edge_weight", None), getattr(data, "BU_edge_weight", None))
        if all(w is None for w in ws):
            return
        if not self.edge_weights:
            raise L.BigcnError("FusedTrainer does not take edge-weighted batches (data.edge_weight / data.BU_edge_weight) "
                               "unless built with edge_weights=True; or train them through the modules (BiGCN(data))")
        if not self.edge_grad and any(torch.is_tensor(w) and w.requires_grad for w in ws):
            raise L.BigcnError("FusedTrainer forms no edge-weight gradient: a weight that requires grad trains through "
                               "the modules (BiGCN(data)); pass it detached here")

    @staticmethod
    def _weights_copied(data):
        return any(torch.is_tensor(w) and (w.dtype != torch.float32 or not w.is_contiguous())
                   for w in (getattr(data, "edge_weight", None), getattr(data, "BU_edge_weight", None)))

    @staticmethod
    def _weights(data, ei, bu):
        """(TD, BU) weights checked and laid out as fp32 [E] (or None); a cast copy is kept by the plan that reads it
        (and, for a weight that requires grad, carries the gradient back through the cast)"""
        with torch.enable_grad():
            return (edge_weight(getattr(data, "edge_weight", None), int(ei.shape[1]), "edge_weight"),
                    edge_weight(getattr(data, "BU_edge_weight", None), int(bu.shape[1]), "BU_edge_weight"))

    @staticmethod
    def _deliver(p):
        """edge_grad: hand the step's weight gradients to autograd, on the caller's stream.  Clones: ``.grad`` must not
        alias the plan's buffers, which the next replay overwrites."""
        roots, grads = [], []
        for w, g in zip(p["ew"], p["dew"]):
            if g is None:
                continue
            if roots and roots[0] is w:       # one tensor for both directions: the sum of the two
                grads[0] = grads[0] + g
            else:
                roots.append(w)
                grads.append(g.clone())
        torch.autograd.backward(roots, grads)

    def step(self, data, b_global=None, node_id_base=0, seed=None, next_data=None):
        """One optimisation step on a device-resident batch; returns the loss (device scalar).

        ``next_data``: the batch of the NEXT step, if the caller knows it (a loader loop does).  Its
        weight-independent half -- graph prep, root columns, the HBM-bound pass over its ``x`` and the
        column sort -- is then enqueued on low-priority streams beside this step (bigcn_batch_prepare), and
        the next ``step(next_data, ...)`` finds it done: the step's chain shrinks to the latency-bound
        kernels, with the memory-bound work of the following batch hidden underneath.

        With ``graphs`` on, a batch OBJECT stepped on for the second time (the same ``data``, same device
        buffers, same shapes -- a resident batch, not a freshly assembled one that happens to reuse freed
        memory) has its whole step captured into a CUDA graph: ~45 launches over four streams become one
        ``cudaGraphLaunch``, and every later step on it is a replay.  The dropout seed of a replay comes
        from the device-side calls counter, so replays draw fresh masks exactly as enqueued steps do."""
        for d in (data, next_data):
            if d is not None:
                self._check_weights(d)
        self._calls += 1
        # a weight that needs an fp32 copy is read through that copy: a replay would not see the caller's later writes
        use_graph = self.graphs and seed is None and not self.validate and not self._weights_copied(data)
        pk_any = next_data is not None or (self._prep_buf is not None and any(
            o is not None and o[1]() is data for o in self._prep_owner))
        key = None
        if use_graph:
            key = self._graph_key(data, b_global, node_id_base)
            if pk_any:                          # which prepared buffer holds this batch, what the next batch is
                key = key + self._prep_peek(data, next_data)
            ent = self._graphs.get(key)
            if ent is not None and ent["ws"] is self._ws and (not pk_any or ent["prep"] is self._prep_buf):
                ent["graph"].replay()
                self.graph_replays += 1
                if pk_any:
                    self._prep_commit(ent["plan"], data, next_data)
                if ent["plan"]["edge_grad"]:
                    self._deliver(ent["plan"])
                self.last_logp = ent["plan"]["logp"]
                return ent["plan"]["loss"]
        p = self._plan(data, b_global, node_id_base, seed)
        ws_before = self._ws
        self._workspace(p["dims"], p["dev"], p["weighted"], p["edge_grad"])
        if self._ws is not ws_before:
            self._graphs.clear()               # the workspace moved: every captured pointer into it is stale
        if pk_any:
            pkey = self._prep_setup(p, data, next_data, node_id_base)
            if use_graph:
                key = self._graph_key(data, b_global, node_id_base) + pkey   # (the buffers may just have moved)
        if not use_graph:
            self._enqueue_prio(p, pk_any)
        else:
            ref = self._seen.get(key)
            if ref is None or ref() is not data:   # first sighting: enqueue (also warms the library's lazy state)
                if len(self._seen) >= 256:
                    self._seen.clear()
                self._seen[key] = weakref.ref(data)
                self._enqueue_prio(p, pk_any)
            else:                                   # seen before: capture, then replay
                g = capture_graph(lambda: self._enqueue(p))
                while len(self._graphs) >= self.max_graphs:
                    self._graphs.pop(next(iter(self._graphs)))
                self._graphs[key] = {"ws": self._ws, "prep": self._prep_buf, "graph": g, "plan": p,
                                     "data": (data, next_data)}   # the strong references pin id(data)
                self.graph_captures += 1
                g.replay()
                self.graph_replays += 1
        if pk_any:
            self._prep_commit(p, data, next_data)
        if p["edge_grad"]:
            self._deliver(p)
        self.last_logp = p["logp"]
        if self.validate:
            raise_on_flags(self.flags)
        return p["loss"]

    def check_inputs(self):
        raise_on_flags(self.flags)

    # ---- checkpoint interchange with the reference's torch.optim.Adam (BiGCN_Twitter.py:146-153,253-261)
    def _ref_groups(self):
        """Parameter names in the reference optimizer's order: group 0 = model.parameters() minus the
        BU convs, group 1 = BUrumorGCN.conv1, group 2 = BUrumorGCN.conv2."""
        names = [n for n, _ in self.model.named_parameters()]
        g1 = [n for n in names if n.startswith("BUrumorGCN.conv1.")]
        g2 = [n for n in names if n.startswith("BUrumorGCN.conv2.")]
        g0 = [n for n in names if n not in g1 and n not in g2]
        return [g0, g1, g2]

    def _own_slice(self):
        lo, hi = C.c_int64(), C.c_int64()
        check(lib().bigcn_dp_slice(self.n, self.world, self._rank, C.byref(lo), C.byref(hi)), "dp_slice")
        return lo.value, hi.value

    def _full_moments(self):
        """comm="symm" shards the Adam moments (rank r owns bigcn_dp_slice(r)); a checkpoint needs all
        of them: every rank contributes its slice to a sum (a collective -- call on every rank)."""
        if self.comm != "symm":
            return self.exp_avg, self.exp_avg_sq
        lo, hi = self._own_slice()
        both = torch.zeros(2, self.n, dtype=torch.float32, device=self.flat.device)
        both[0, lo:hi] = self.exp_avg[lo:hi]
        both[1, lo:hi] = self.exp_avg_sq[lo:hi]
        torch.distributed.all_reduce(both, group=self.pg)
        return both[0], both[1]

    def optimizer_state_dict(self):
        """The state a ``torch.optim.Adam`` built as the reference builds it (:149-153) would hold
        after the same steps; its ``load_state_dict`` accepts the result.  Reads the device."""
        step = float(self.step_count[0].item())
        m_all, v_all = self._full_moments()
        seg_lr_host = self.seg_lr_host
        groups, state, i = [], {}, 0
        for gi, names in enumerate(self._ref_groups()):
            ids = []
            for n in names:
                v = self.views[n]
                off = (v.data_ptr() - self.flat.data_ptr()) // 4
                sl = slice(off, off + v.numel())
                if step > 0:
                    state[i] = {"step": torch.tensor(step), "exp_avg": m_all[sl].view(v.shape).clone(),
                                "exp_avg_sq": v_all[sl].view(v.shape).clone()}
                ids.append(i)
                i += 1
            lrs = {float(seg_lr_host[_ORDER.index(n)]) for n in names}
            groups.append({"lr": lrs.pop() if len(lrs) == 1 else (self.lr if gi == 0 else self.lr / 5),
                           "betas": tuple(self.betas), "eps": self.eps,
                           "weight_decay": self.wd, "amsgrad": False, "maximize": False, "foreach": None,
                           "capturable": False, "differentiable": False, "fused": None,
                           "decoupled_weight_decay": False, "params": ids})
        return {"state": state, "param_groups": groups}

    def load_optimizer_state_dict(self, sd):
        """Inverse of ``optimizer_state_dict`` (also takes the reference optimizer's own state_dict).
        All parameters must be at the same step, as they are under the reference's loop."""
        names = [n for g in self._ref_groups() for n in g]
        ids = [i for g in sd["param_groups"] for i in g["params"]]
        if len(ids) != len(names):
            raise L.BigcnError(f"optimizer state has {len(ids)} parameters, this model has {len(names)}")
        steps = set()
        self.exp_avg.zero_()
        self.exp_avg_sq.zero_()
        for n, i in zip(names, ids):
            st = sd["state"].get(i)
            if st is None:
                steps.add(0)
                continue
            v = self.views[n]
            if tuple(st["exp_avg"].shape) != tuple(v.shape):
                raise L.BigcnError(f"optimizer state of {n}: shape {tuple(st['exp_avg'].shape)} != {tuple(v.shape)}")
            off = (v.data_ptr() - self.flat.data_ptr()) // 4
            self.exp_avg[off:off + v.numel()].copy_(st["exp_avg"].reshape(-1))
            self.exp_avg_sq[off:off + v.numel()].copy_(st["exp_avg_sq"].reshape(-1))
            steps.add(int(float(st["step"])))
        if len(steps) != 1:
            raise L.BigcnError(f"optimizer state mixes step counts {sorted(steps)}")
        self.step_count[0] = steps.pop()
        # hyper-parameters travel with the state (torch.optim.Adam.load_state_dict restores them too)
        groups = sd["param_groups"]
        g0 = groups[0]
        for g in groups[1:]:
            for k in ("betas", "eps", "weight_decay"):
                if k in g and k in g0 and (tuple(g[k]) != tuple(g0[k]) if k == "betas" else g[k] != g0[k]):
                    raise L.BigcnError(f"optimizer state: param groups disagree on {k}; the fused Adam kernel takes one value")
        self.lr = float(g0["lr"])
        if "betas" in g0:
            self.betas = (float(g0["betas"][0]), float(g0["betas"][1]))
        self.eps = float(g0.get("eps", self.eps))
        self.wd = float(g0.get("weight_decay", self.wd))
        if g0.get("amsgrad") or g0.get("maximize") or g0.get("decoupled_weight_decay"):
            raise L.BigcnError("optimizer state: amsgrad / maximize / decoupled weight decay are not what the reference uses")
        # per-tensor lr from the group each tensor sits in (reference: group 0 at lr, BU conv1 / conv2 at lr/5)
        lr_of = {}
        for g, gnames in zip(groups, self._ref_groups()):
            for n in gnames:
                lr_of[n] = float(g["lr"])
        self.seg_lr_host = [lr_of[n] for n in _ORDER]
        self.seg_lr.copy_(torch.tensor(self.seg_lr_host, dtype=torch.float32))
        self._graphs.clear()      # betas / eps / weight decay are baked into captured launches


def launches_per_step(n_nodes: int, n_dirs: int = 2, training: bool = True, gemm_mode: str = "fp32",
                      in_feats: int = 5000, comm: str = "single", sparse_input: bool = False) -> int:
    """How many kernels of this library one FusedTrainer.step enqueues (for bench.py's
    gpu_launches claim); mirrors the launch sequence in csrc/api.cu, graph_prep.cu, xsparse.cu
    (checked against the ncu launch list in profiles/)."""
    def radix_passes(n):
        bits = 1
        while (1 << bits) <= n:
            bits += 1
        return (bits + 7) // 8
    prep = 1 + 2 + 3 * radix_passes(n_nodes) + 1 + 1   # count, scan x2, radix passes, deg, hub lists
    sparse = gemm_mode == "sparse"
    xw = 1 + (n_dirs if gemm_mode in ("tf32x3", "bf16") else 0)     # [W hi/lo or bf16-term split per direction], X*W
    csc = 0
    if sparse:      # row scan x2 + compaction (or CSR ingest), radix passes over the column keys, finish, hub columns
        kbits = max(1, (in_feats - 1).bit_length())
        csc = (1 if sparse_input else 3) + 3 * ((kbits + 7) // 8) + 2
    # transposes, prep, root_nz, [root_proj], xw, [csc build], mix, prop2, readout x2  (the W2a hi/lo split is only launched
    # when the tcgen05 forms of the 64 x 64 products are selected: BIGCN_MIX_TC)
    fwd = 1 + prep + 1 + (0 if training else 1) + xw + csc + 1 + 1 + 2
    head = 1 + 1 + 3                           # head fwd, nll, head bwd (feat, w partial, w reduce)
    if sparse:
        dw = 1                                 # sweep over the column-sorted non-zeros
    else:
        dw = 1 + (1 if gemm_mode in ("tf32x3", "mixed", "bf16") else 0) + n_dirs   # [T split], dW GEMM/scan, reduce x dirs
    # gscale+colsum, propT(g2), outer x2, [segsum | dw2b part], dw2b reduce + dense fallback,
    # bwdmix+colsum, propT, dW
    bwd = 2 + 1 + 2 + 1 + 2 + 2 + 1 + dw
    head = 1 + 3 - 2                           # fused tail (readout final + head + gscale in one launch), then dW / db / loss sum
    adam = 1                                   # Adam (or the fused peer-memory reduce + Adam) incl. the step counter
    return fwd + head + bwd + adam
